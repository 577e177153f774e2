// BERT encoder model object (declarations shared by fl_bert.cu and fl_lib.cu).
#pragma once
#include <cuda.h>

#include <mutex>
#include <vector>

#include "../../include/fastllm_b200.h"
#include "runtime.cuh"
#include "tensor_table.hpp"

namespace fl {

struct BertLayerW {
    uint16_t *wqkv = nullptr, *wo = nullptr, *wi = nullptr, *wo2 = nullptr;   // [3H,H] (q|k|v rows), [H,H], [I,H], [H,I] bf16
    float *bqkv = nullptr, *bo = nullptr, *bi = nullptr, *bo2 = nullptr;
    float *ln1w = nullptr, *ln1b = nullptr, *ln2w = nullptr, *ln2b = nullptr;
    CUtensorMap tm_wqkv, tm_wo, tm_wi, tm_wo2;
};

struct BertModel {
    fl_config cfg{};
    int H = 0, I = 0, V = 0, L = 0, nh = 0, d = 0, maxpos = 0;
    TensorTable table;
    uint16_t *wemb = nullptr, *pemb = nullptr;
    float *lnw = nullptr, *lnb = nullptr;
    std::vector<BertLayerW> layers;
    cudaStream_t stream = nullptr;
    std::mutex mu;
    // workspace (grown on demand)
    size_t cap_tokens = 0, cap_batch = 0, cap_words = 0;
    DevBuf<uint16_t> x, x1, ctx, qkv, hbuf;
    DevBuf<float> pre, out;
    DevBuf<uint32_t> ids;             // one upload (u32 words): ids [T] | mask [T] (if any) | token positions [T] | sentence starts [n + 1] |
                                      // attention items
    PinnedBuf<uint32_t> h_ids;        // its pinned staging copy
    PinnedBuf<float> h_out;
    struct Batch {                    // layout of the last upload, reused by bert_repeat
        int T = 0, n = 0, nshort = 0, nlong = 0;
        bool mask = false;
        size_t o_pos = 0, o_starts = 0, o_short = 0, o_long = 0;
    } batch;
    ~BertModel() {
        if (stream) cudaStreamDestroy(stream);
    }
};

void finalize(BertModel& m);
void bert_embed(BertModel& m, const uint32_t* ids, const uint32_t* mask, int b, int t, float* out);
void bert_embed_packed(BertModel& m, const uint32_t* ids, const int32_t* lengths, int n, float* out);
void bert_repeat(BertModel& m, int b, int t, int iters, float* elapsed_ms);
CUtensorMap make_tmap_bf16(const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows);
CUtensorMap make_tmap_pk(const void* ptr, uint64_t N, uint64_t K);
CUtensorMap make_tmap_kv(const void* ptr, uint64_t rows, uint32_t head_dim, uint32_t elem_bytes = 2);

}  // namespace fl
