// One table per model: every HuggingFace tensor the model reads, where this rank keeps it in the weight slab and how it is
// initialised.  A model's plan step registers the slots and lays out the slab in one pass (no CUDA call); alloc() then makes
// the slab, and put / random_init / check_complete serve fl_model_put_tensor, fl_model_random_init and fl_model_finalize.
#pragma once
#include <cstdint>
#include <functional>
#include <map>
#include <set>
#include <string>
#include <vector>

#include "../../include/fastllm_b200.h"
#include "row_map.cuh"
#include "runtime.cuh"

namespace fl {

struct TensorSlot {
    std::string name;               // exact HF name
    bool mat;                       // bf16 matrix; else f32 vector
    size_t off;                     // slab byte offset of the destination buffer
    int64_t rows, cols, ld;         // local block this rank keeps (a vector: [rows], cols = ld = 1); ld > cols: zero-padded columns
    RowMap map;                     // local row -> destination row
    int64_t full_rows, full_cols;   // shape the caller hands over (the full HF tensor)
    int64_t row0, col0;             // window of the full tensor this rank keeps
    bool ones;                      // synthetic init: 1.0 (norm weights); else tensor_seed values of the full-tensor index
    bool round;                     // f32 vector stored bf16-rounded (causal LMs) or as uploaded (BERT)
    bool required;                  // finalize fails without it
};

struct TensorTable {
    bool f32_only = false;          // dtype policy: f32 uploads only (BERT), else f32 / f16 / bf16
    std::vector<TensorSlot> slots;  // registration order
    std::map<std::string, size_t> index;
    std::set<std::string> have;     // names that arrived
    bool finalized = false;
    size_t size = 0;                // slab bytes laid out so far
    DevBuf<uint8_t> slab;           // every weight of the model lives in this one allocation
    std::vector<std::function<void(uint8_t*)>> binds;

    // `bytes` of the slab, 256-byte aligned; returns their offset.  With `p`: alloc() points p at them.
    size_t take(size_t bytes) {
        const size_t o = size;
        size = align_up(size + bytes, 256);
        return o;
    }
    template <typename T>
    size_t take(size_t bytes, T*& p) {
        const size_t o = take(bytes);
        bind(o, p);
        return o;
    }
    template <typename T>
    void bind(size_t off, T*& p) {
        binds.push_back([off, &p](uint8_t* base) { p = (T*)(base + off); });
    }
    void add(TensorSlot s) {
        index[s.name] = slots.size();
        slots.push_back(std::move(s));
    }
    void alloc() {
        slab.alloc(size, /*zero=*/true);
        for (auto& b : binds) b(slab.p);
    }
    // Upload one tensor (names outside the table are accepted and ignored) / synthesise every slot / the start of finalize.
    void put(const char* name, int dtype, const int64_t* shape, int rank, const void* host);
    void random_init(uint64_t seed, float stdv);
    void check_complete() const {
        FL_CHECK(!finalized, FL_ERR_STATE, "model already finalized");
        for (const TensorSlot& s : slots) FL_CHECK(!s.required || have.count(s.name), FL_ERR_STATE, "missing tensor: " + s.name);
    }
};

}  // namespace fl
