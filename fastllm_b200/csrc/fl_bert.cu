// BERT / MiniLM sentence-encoder path behind fl_embed (host orchestration), sm_100a.
// Reference: MiniLMModel::{new, embed_tokens, forward, mean_pooling, normalize_l2, embed} src/models/embeddings.rs:245-447.
#include <algorithm>
#include <cmath>
#include <cstring>

#include "bert.cuh"
#include "bert_model.cuh"
#include "gemm_tc.cuh"

namespace fl {

// ---- TMA descriptors (driver entry point fetched through the runtime: no link-time libcuda dependency) -----------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        FL_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
        FL_CHECK(p != nullptr && qres == cudaDriverEntryPointSuccess, -2, "cuTensorMapEncodeTiled not available from the driver");
        fn = (EncodeTiledFn)p;
    }
    return fn;
}

// 2-D bf16 tensor [rows, cols] row-major (row stride ld elements), box [box_rows, 64 cols], 128-byte swizzle.
// Output-tile width of the encoder GEMMs.  With hidden = 384 every GEMM of the model has K-major operands of equal depth, so a
// 128 x BN tile moves (128 + BN) * K * 2 bytes from L2 for 2 * 128 * BN * K FLOP: 64 FLOP/B at BN = 128 -- L2->SM bound
// (~7 TB/s chip-wide => ~450 TFLOP/s) long before the tensor pipe.  BN = 192 divides all three widths (1152, 384, 1536), lifts
// the intensity to 77 FLOP/B and still fits two TMEM accumulator stages (2 x 256 columns).  It also divides every width at hidden
// 768 (2304, 768, 3072); at hidden 1024, N = 1024 and 4096 end in a partial tile (TMA zero-fills the dead weight rows, the epilogue
// stores col < N only).  One width for every model, no split-K: a row's sums never depend on the other rows in the batch.
constexpr int kBertBN = 192;

CUtensorMap make_tmap_bf16(const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
    CUtensorMap m;
    const cuuint64_t dims[2] = {cols, rows};
    const cuuint64_t strides[1] = {ld * 2};
    const cuuint32_t box[2] = {(cuuint32_t)kGemmBK, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode_tiled_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FL_CHECK(r == CUDA_SUCCESS, -2, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
    return m;
}

// Weight matrix [N, K] bf16 (K % 64 == 0) as the persistent decode kernel streams it: a 3-D view {64 columns, N rows, K/64
// column blocks} whose box {64, 16, 16} is ONE 32 KB request = 16 rows x 1024 columns, landing in shared memory as
// [column block][row][128 bytes] with the 128-byte swizzle keyed by the row: conflict-free ldmatrix of 16 x 16 tiles.
// Out-of-range rows / column blocks are zero-filled by the TMA engine (no tail handling in the kernel).
CUtensorMap make_tmap_pk(const void* ptr, uint64_t N, uint64_t K) {
    CUtensorMap m;
    const cuuint64_t dims[3] = {64, N, K / 64};
    const cuuint64_t strides[2] = {K * 2, 128};
    const cuuint32_t box[3] = {64, 16, 16};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = encode_tiled_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FL_CHECK(r == CUDA_SUCCESS, -2, "cuTensorMapEncodeTiled (3-D weight stream) failed (" + std::to_string((int)r) + ")");
    return m;
}

// K or V pool of a cache seen as one [rows, head_dim] matrix (rows = layers x pages x kv heads x 64 tokens) of bf16 (elem_bytes 2) or
// e4m3 (elem_bytes 1) elements: the stream-K decode attention fetches a page of one kv head as 64-row boxes of 128 bytes with the
// 128-byte swizzle (bf16: 64 columns per box; e4m3: the 128-byte row of head_dim 128), or as one [64, head_dim] box of 64-byte rows
// with the 64-byte swizzle (e4m3, head_dim 64); test-size heads (< 64) as one unswizzled [64, head_dim] box.
CUtensorMap make_tmap_kv(const void* ptr, uint64_t rows, uint32_t head_dim, uint32_t elem_bytes) {
    CUtensorMap m;
    const cuuint64_t dims[2] = {head_dim, rows};
    const cuuint64_t strides[1] = {(cuuint64_t)head_dim * elem_bytes};
    const uint32_t row_bytes = head_dim * elem_bytes;
    const cuuint32_t box[2] = {row_bytes >= 128 ? 128u / elem_bytes : head_dim, 64u};
    const cuuint32_t estr[2] = {1, 1};
    const CUtensorMapSwizzle swz = row_bytes >= 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (row_bytes == 64 && elem_bytes == 1 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                                                                                      : CU_TENSOR_MAP_SWIZZLE_NONE);
    const CUresult r = encode_tiled_fn()(&m, elem_bytes == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr),
                                         dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FL_CHECK(r == CUDA_SUCCESS, -2, "cuTensorMapEncodeTiled (KV pool) failed (" + std::to_string((int)r) + ")");
    return m;
}

// Every kernel of the encoder is launched with programmatic stream serialization: each calls griddepcontrol.launch_dependents at
// entry and griddepcontrol.wait before it touches anything the previous kernel wrote, so a kernel's prologue (barrier / TMEM
// set-up, descriptor fetch, block scheduling) overlaps its predecessor's tail instead of following it.
template <int EPI>
static void launch_gemm(LaunchCtx& lc, const char* tag, const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmArgs& g) {
    constexpr int BN = kBertBN;
    const size_t smem = gemm_smem_bytes(BN, DUAL_NONE) + (gemm_epi_staged(EPI) ? kEpiStageBytes : 0);
    const int tiles = ((g.M + kGemmBM - 1) / kGemmBM) * ((g.N + BN - 1) / BN);
    launch(lc, tag, (uint64_t)g.N * g.K * 2, gemm_tc_kernel<BN, EPI>, dim3(std::min(tiles, kNumSMs)), dim3(kGemmThreads), smem, tmA, tmA, tmB,
           g);
}

void finalize(BertModel& m) {
    m.table.check_complete();
    for (BertLayerW& w : m.layers) {   // weight-side TMA descriptors ([out, in] row-major == K-major B operand)
        w.tm_wqkv = make_tmap_bf16(w.wqkv, 3 * m.H, m.H, m.H, kBertBN);
        w.tm_wo = make_tmap_bf16(w.wo, m.H, m.H, m.H, kBertBN);
        w.tm_wi = make_tmap_bf16(w.wi, m.I, m.H, m.H, kBertBN);
        w.tm_wo2 = make_tmap_bf16(w.wo2, m.H, m.I, m.I, kBertBN);
    }
    m.table.finalized = true;
}

static void bert_reserve(BertModel& m, size_t T, size_t n, size_t words) {
    const size_t H = m.H, I = m.I;
    if (T > m.cap_tokens) {
        m.cap_tokens = T;
        m.x.alloc(T * H); m.x1.alloc(T * H); m.ctx.alloc(T * H); m.qkv.alloc(T * 3 * H); m.hbuf.alloc(T * I); m.pre.alloc(T * H);
    }
    if (n > m.cap_batch) {
        m.cap_batch = n;
        m.out.alloc(n * H); m.h_out.alloc(n * H);
    }
    if (words > m.cap_words) {
        m.cap_words = words;
        m.ids.alloc(words); m.h_ids.alloc(words);
    }
}

// Enqueue the encoder on m.stream over the batch m.batch describes: B1 -> L x (B2..B7) -> B8 (SURVEY.md section 2.4)
static void bert_enqueue(BertModel& m, bool use_mask) {
    const BertModel::Batch& bb = m.batch;
    const int T = bb.T, H = m.H, I = m.I;
    const int* positions = (const int*)(m.ids.p + bb.o_pos);
    const int* starts = (const int*)(m.ids.p + bb.o_starts);
    const BertItem* shorts = (const BertItem*)(m.ids.p + bb.o_short);
    const BertItem* longs = (const BertItem*)(m.ids.p + bb.o_long);
    LaunchCtx lc{m.stream};
    // the model's kernel instantiations (bert_plan admits head_dim 32 / 64 and hidden <= 1024); rows of up to 512 columns take the
    // narrow LayerNorm kernels, which hold 16 values per lane instead of 32
    const bool wide = H > 512;
    const auto embed_ln = wide ? embed_ln_kernel<32> : embed_ln_kernel<16>;
    const auto layernorm = wide ? layernorm_kernel<8> : layernorm_kernel<4>;
    const auto attn = m.d == 64 ? bert_attn_kernel<64> : bert_attn_kernel<32>;
    const auto attn_long = m.d == 64 ? bert_attn_long_kernel<64> : bert_attn_long_kernel<32>;
    const size_t attn_smem = bert_attn_dyn_smem(m.d);
    const int rows_per_cta = 8;
    const dim3 row_grid((T + rows_per_cta - 1) / rows_per_cta), row_block(rows_per_cta * 32);
    launch(lc, "bert_embed_ln", 0, embed_ln, row_grid, row_block, 0, (const uint16_t*)m.wemb, (const uint16_t*)m.pemb, (const float*)m.lnw,
           (const float*)m.lnb, (const uint32_t*)m.ids.p, positions, T, H, m.V, m.maxpos, 1e-12f, m.x.p);
    const CUtensorMap tm_x = make_tmap_bf16(m.x.p, T, H, H, kGemmBM), tm_x1 = make_tmap_bf16(m.x1.p, T, H, H, kGemmBM),
                      tm_ctx = make_tmap_bf16(m.ctx.p, T, H, H, kGemmBM), tm_h = make_tmap_bf16(m.hbuf.p, T, I, I, kGemmBM);
    const float eps = m.cfg.norm_eps;
    const float scale = (float)std::sqrt((double)m.d);
    for (int l = 0; l < m.L; ++l) {
        const BertLayerW& w = m.layers[l];
        // B2: fused q|k|v projection + bias -> bf16 [T, 3H]
        launch_gemm<GEPI_BIAS_BF16>(lc, "bert_gemm_qkv", tm_x, w.tm_wqkv, GemmArgs{T, 3 * H, H, w.bqkv, nullptr, 0, m.qkv.p, 3 * H, 1, 0});
        // B3+B4: per (sentence, head) softmax(QK^T / sqrt(d)) V, no mask; sentences of <= 128 tokens in one tile, longer ones key-tiled
        if (bb.nshort)
            launch(lc, "bert_attn", 0, attn, dim3(m.nh * bb.nshort), dim3(128), attn_smem, (const uint16_t*)m.qkv.p, shorts, m.nh, H, scale,
                   m.ctx.p);
        if (bb.nlong)
            launch(lc, "bert_attn", 0, attn_long, dim3(m.nh * bb.nlong), dim3(128), attn_smem, (const uint16_t*)m.qkv.p, longs, m.nh, H,
                   scale, m.ctx.p);
        // B5: attention output dense + bias + residual -> f32, then LayerNorm -> bf16
        launch_gemm<GEPI_BIAS_RESID_F32>(lc, "bert_gemm_o", tm_ctx, w.tm_wo, GemmArgs{T, H, H, w.bo, m.x.p, H, m.pre.p, H, 1, 0});
        launch(lc, "bert_layernorm", 0, layernorm, row_grid, row_block, 0, (const float*)m.pre.p, (const float*)w.ln1w, (const float*)w.ln1b,
               T, H, eps, m.x1.p);
        // B6: intermediate dense + bias + GELU(tanh) -> bf16 [T, I]
        launch_gemm<GEPI_BIAS_GELU_BF16>(lc, "bert_gemm_up_gelu", tm_x1, w.tm_wi, GemmArgs{T, I, H, w.bi, nullptr, 0, m.hbuf.p, I, 1, 0});
        // B7: output dense + bias + residual -> f32, LayerNorm -> bf16
        launch_gemm<GEPI_BIAS_RESID_F32>(lc, "bert_gemm_down", tm_h, w.tm_wo2, GemmArgs{T, H, I, w.bo2, m.x1.p, H, m.pre.p, H, 1, 0});
        launch(lc, "bert_layernorm", 0, layernorm, row_grid, row_block, 0, (const float*)m.pre.p, (const float*)w.ln2w, (const float*)w.ln2b,
               T, H, eps, m.x.p);
    }
    // B8: masked mean pooling + L2 normalise -> f32 [n, H]
    launch(lc, "bert_pool_l2", 0, pool_l2_kernel, dim3(bb.n), dim3((H + 31) / 32 * 32), 0, (const uint16_t*)m.x.p,
           use_mask && bb.mask ? (const uint32_t*)m.ids.p + T : (const uint32_t*)nullptr, starts, H, m.out.p);
}

// The total token count T of a batch, checked: GemmArgs and the kernels' index arithmetic are int, so T x max(3H, I) must fit in int32.
static int bert_total_tokens(const BertModel& m, int64_t T) {
    FL_CHECK(T * std::max(3 * m.H, m.I) <= (int64_t)INT32_MAX, FL_ERR_INVALID,
             "batch too large: total tokens x max(3 x hidden, intermediate) must fit in int32");
    return (int)T;
}

// One encoder pass over n packed sentences (lengths already checked, T = their sum): stage ids | mask | token positions | sentence
// starts | attention work lists in the pinned buffer, upload them in one copy, run, read back f32 [n, H].  The work lists: a sentence of <= 128 tokens
// is one bert_attn_kernel item, a longer one is one bert_attn_long_kernel item per 128-row query tile -- the kernel its lone fl_embed
// uses, so its rows get the same arithmetic.  Both lists hold the sentences in order of decreasing length (most key tiles first), so
// the longest sentences start first instead of running alone at the end of the launch.
static void bert_run(BertModel& m, const uint32_t* ids, const uint32_t* mask, const int32_t* lengths, int n, int T, float* out) {
    std::vector<int> order(n);
    for (int i = 0; i < n; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return lengths[a] > lengths[b]; });
    int nshort = 0, nlong = 0;
    for (int i = 0; i < n; ++i) {
        if (lengths[i] <= kBertS) ++nshort;
        else nlong += (lengths[i] + kBertS - 1) / kBertS;
    }
    BertModel::Batch bb;
    bb.T = T; bb.n = n; bb.nshort = nshort; bb.nlong = nlong; bb.mask = mask != nullptr;
    bb.o_pos = (size_t)T * (mask ? 2 : 1);
    bb.o_starts = bb.o_pos + T;
    bb.o_short = align_up(bb.o_starts + n + 1, 4);      // BertItem: 16-byte aligned
    bb.o_long = bb.o_short + 4 * (size_t)nshort;
    const size_t words = bb.o_long + 4 * (size_t)nlong;
    std::lock_guard<std::mutex> lock(m.mu);      // embed(&self) may be called from several threads: one workspace
    bert_reserve(m, T, n, words);
    m.batch = bb;
    uint32_t* h = m.h_ids.p;
    std::memcpy(h, ids, (size_t)T * 4);
    if (mask) std::memcpy(h + T, mask, (size_t)T * 4);
    int32_t* positions = (int32_t*)(h + bb.o_pos);
    int32_t* starts = (int32_t*)(h + bb.o_starts);
    starts[0] = 0;
    for (int i = 0; i < n; ++i) {
        starts[i + 1] = starts[i] + lengths[i];
        for (int p = 0; p < lengths[i]; ++p) positions[starts[i] + p] = p;
    }
    BertItem* shorts = (BertItem*)(h + bb.o_short);
    BertItem* longs = (BertItem*)(h + bb.o_long);
    for (int s : order) {
        if (lengths[s] <= kBertS) *shorts++ = BertItem{starts[s], lengths[s], 0, 0};
        else for (int q0 = 0; q0 < lengths[s]; q0 += kBertS) *longs++ = BertItem{starts[s], lengths[s], q0, 0};
    }
    FL_CUDA(cudaMemcpyAsync(m.ids.p, h, words * 4, cudaMemcpyHostToDevice, m.stream));
    bert_enqueue(m, true);
    FL_CUDA(cudaGetLastError());
    FL_CUDA(cudaMemcpyAsync(m.h_out.p, m.out.p, (size_t)n * m.H * 4, cudaMemcpyDeviceToHost, m.stream));
    FL_CUDA(cudaStreamSynchronize(m.stream));
    std::memcpy(out, m.h_out.p, (size_t)n * m.H * 4);
}

void bert_embed(BertModel& m, const uint32_t* ids, const uint32_t* mask, int b, int t, float* out) {
    FL_CHECK(m.table.finalized, FL_ERR_STATE, "model not finalized");
    FL_CHECK(ids && out && b >= 1 && t >= 1, FL_ERR_INVALID, "bad arguments");
    // the reference enforces no max_seq_length (embeddings.rs:285-286); what bounds a sentence is its position table: position ids
    // 0..n index a [max_position_embeddings, H] embedding (embeddings.rs:416, 370-378), and candle's index_select fails past it
    FL_CHECK(t <= m.maxpos, FL_ERR_INVALID, "sentence longer than max_position_embeddings (the position-embedding lookup fails in the reference too)");
    const int T = bert_total_tokens(m, (int64_t)b * t);
    for (int i = 0; i < T; ++i) FL_CHECK(ids[i] < (uint32_t)m.V, FL_ERR_INVALID, "token id out of range");
    const std::vector<int32_t> lengths(b, t);
    bert_run(m, ids, mask, lengths.data(), b, T, out);
}

void bert_embed_packed(BertModel& m, const uint32_t* ids, const int32_t* lengths, int n, float* out) {
    FL_CHECK(m.table.finalized, FL_ERR_STATE, "model not finalized");
    FL_CHECK(ids && lengths && out && n >= 1, FL_ERR_INVALID, "bad arguments");
    int64_t total = 0;
    for (int i = 0; i < n; ++i) {
        FL_CHECK(lengths[i] >= 1, FL_ERR_INVALID, "bad arguments");
        FL_CHECK(lengths[i] <= m.maxpos, FL_ERR_INVALID, "sentence longer than max_position_embeddings (the position-embedding lookup fails in the reference too)");
        total += lengths[i];
    }
    const int T = bert_total_tokens(m, total);
    for (int i = 0; i < T; ++i) FL_CHECK(ids[i] < (uint32_t)m.V, FL_ERR_INVALID, "token id out of range");
    bert_run(m, ids, nullptr, lengths, n, T, out);
}

// Device-resident repeat of the encoder on the batch the last bert_embed uploaded (benchmark `value`).
void bert_repeat(BertModel& m, int b, int t, int iters, float* elapsed_ms) {
    std::lock_guard<std::mutex> lock(m.mu);
    FL_CHECK(m.batch.n == b && m.batch.T == (int64_t)b * t, FL_ERR_STATE, "call fl_embed with this shape first");
    EventPair ev;
    FL_CUDA(cudaEventRecord(ev.e0, m.stream));
    for (int i = 0; i < iters; ++i) bert_enqueue(m, false);
    FL_CUDA(cudaEventRecord(ev.e1, m.stream));
    FL_CUDA(cudaStreamSynchronize(m.stream));
    FL_CUDA(cudaGetLastError());
    FL_CUDA(cudaEventElapsedTime(elapsed_ms, ev.e0, ev.e1));
}

}  // namespace fl
