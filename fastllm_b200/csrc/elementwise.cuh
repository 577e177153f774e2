// Small glue kernels of the decode step (token gather, arg-max finalisation, step-state advance), sm_100a.
#pragma once
#include "common.cuh"
#include "gemv.cuh"

namespace fl {

// K1: Embedding::forward = index_select.  resid[m, :] = f32(embed[ids[row_base + m], :])   (bf16 table, f32 residual stream)
static __global__ void embed_gather_kernel(const uint16_t* __restrict__ table, const uint32_t* __restrict__ ids, int row_base, int H,
                                    int vocab, float* __restrict__ resid) {
    pdl_launch_dependents();
    pdl_wait();
    const int m = blockIdx.y;
    uint32_t id = ids[row_base + m];
    if (id >= (uint32_t)vocab) id = vocab - 1;   // candle would raise; ids are validated on the host before launch
    const uint4* src = reinterpret_cast<const uint4*>(table + (size_t)id * H);
    float* dst = resid + (size_t)m * H;
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < H / 8; c += gridDim.x * blockDim.x) {
        const uint4 w = src[c];
        float4 a = make_float4(bf16lo(w.x), bf16hi(w.x), bf16lo(w.y), bf16hi(w.y));
        float4 b = make_float4(bf16lo(w.z), bf16hi(w.z), bf16lo(w.w), bf16hi(w.w));
        reinterpret_cast<float4*>(dst + c * 8)[0] = a;
        reinterpret_cast<float4*>(dst + c * 8)[1] = b;
    }
}

// K18 on device: merge the per-CTA arg-max partials of the lm_head GEMV (last index wins ties, like candle's
// LogitsProcessor::sample_argmax) and write next_ids[seq] for rows that are the last token of their sequence.
static __global__ void argmax_finalize_kernel(const float* __restrict__ val, const int* __restrict__ idx, int nparts, int M, int row_base,
                                       int t, uint32_t* __restrict__ next_ids) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float sv[32];
    __shared__ int si[32];
    for (int m = 0; m < M; ++m) {
        float v = -INFINITY;
        int i = -1;
        for (int p = threadIdx.x; p < nparts; p += blockDim.x) {
            const float ov = val[m * nparts + p];
            const int oi = idx[m * nparts + p];
            if (ov > v || (ov == v && oi > i)) { v = ov; i = oi; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xFFFFFFFFu, v, o);
            const int oi = __shfl_xor_sync(0xFFFFFFFFu, i, o);
            if (ov > v || (ov == v && oi > i)) { v = ov; i = oi; }
        }
        if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = v; si[threadIdx.x >> 5] = i; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
                if (sv[w] > v || (sv[w] == v && si[w] > i)) { v = sv[w]; i = si[w]; }
            const int rg = row_base + m;
            if (rg % t == t - 1) next_ids[rg / t] = (uint32_t)i;
        }
        __syncthreads();
    }
}

// End of a forward call: kv_base[seq] += t (packed calls: lens[seq]).  In the device-resident greedy loop also rope_pos += 1 and
// ids <- next_ids.
static __global__ void advance_state_kernel(StepState* st, int b, int t, int rope_inc, uint32_t* ids, const uint32_t* next_ids, int feedback,
                                     uint32_t* trace, int* trace_pos, const int* lens) {
    pdl_launch_dependents();
    pdl_wait();
    const int i = threadIdx.x;
    if (i < b) {
        st->kv_base[st_slot(st, i)] += lens ? lens[i] : t;       // distinct slots per row (checked on the host)
        if (feedback) ids[i] = next_ids[i];
        if (trace != nullptr) trace[(size_t)(*trace_pos) * b + i] = next_ids[i];
    }
    __syncthreads();
    if (i == 0) {
        st->rope_pos += rope_inc;
        st->ragged = 0;                         // the slot / position tables are valid for ONE call
        if (trace != nullptr) *trace_pos += 1;
    }
}

// ---- tensor-parallel glue -------------------------------------------------------------------------------------------------
// out = sum over split-K slices (fixed order)
static __global__ void sum_slices_kernel(const float* __restrict__ y, int nsl, long long stride, int n, float* __restrict__ out) {
    pdl_launch_dependents();
    pdl_wait();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int k = 0; k < nsl; ++k) s += y[(size_t)k * stride + i];
        out[i] = s;
    }
}
// vocab-parallel logits gathered rank-major [tp][rows][Vl] -> row-major [rows][tp * Vl]
static __global__ void tp_logits_kernel(const float* __restrict__ g, int tp, int rows, int Vl, float* __restrict__ logits) {
    pdl_launch_dependents();
    pdl_wait();
    const int n = tp * rows * Vl;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int r = i / (rows * Vl), rem = i % (rows * Vl), row = rem / Vl, c = rem % Vl;
        logits[(size_t)row * tp * Vl + (size_t)r * Vl + c] = g[i];
    }
}

// ---- opt-in device-side temperature sampling (fl_forward_sample_device; the parity path stays the host sampler) --------------
// candle's LogitsProcessor with a temperature: prs = softmax(logits / T); WeightedIndex::new(prs).sample(rng) = the first index
// whose cumulative weight exceeds x = u * total, u being ONE draw of the request's StdRng.  The host sampler object keeps the
// generator and hands over u (so the random stream of a request is the same as on the host path); the soft-max weights, their
// prefix sums and the search run here, on the logits row that is already in HBM: 4 bytes travel back instead of vocab * 4.
// Difference to the host path: the prefix sums are built by a block scan (1024 partial sums) instead of one sequential f32 loop,
// so a draw that lands within rounding distance (~1e-6 relative) of a boundary between two tokens may pick the neighbour.
static __global__ void __launch_bounds__(1024) sample_softmax_kernel(const float* __restrict__ logits, int V, float mul, float u01,
                                                                    uint32_t* __restrict__ out) {
    __shared__ float red[32];
    __shared__ float wtot[32];
    __shared__ int s_pick;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (V + 1023) / 1024, i0 = min(tid * per, V), i1 = min(i0 + per, V);
    float mx = -INFINITY;
    for (int i = i0; i < i1; ++i) mx = fmaxf(mx, logits[i] * mul);
    mx = warp_max(mx);
    if (lane == 0) red[warp] = mx;
    if (tid == 0) s_pick = -1;
    __syncthreads();
    mx = red[0];
    for (int w = 1; w < 32; ++w) mx = fmaxf(mx, red[w]);
    float sum = 0.f;
    for (int i = i0; i < i1; ++i) sum += expf(logits[i] * mul - mx);
    float inc = sum;                                   // inclusive scan over the 1024 chunk sums
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) wtot[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        float v = wtot[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float t = __shfl_up_sync(0xFFFFFFFFu, v, o);
            if (lane >= o) v += t;
        }
        wtot[lane] = v;
    }
    __syncthreads();
    const float base = warp ? wtot[warp - 1] : 0.f;
    float excl = __shfl_up_sync(0xFFFFFFFFu, inc, 1);  // the intervals [excl, inc) of consecutive threads tile [0, total) exactly
    excl = (lane ? excl : 0.f) + base;
    inc += base;
    const float chosen = u01 * wtot[31];
    if (i0 < i1 && excl <= chosen && chosen < inc) {
        float run = excl;
        int pick = -1, last = i0;
        for (int i = i0; i < i1 && pick < 0; ++i) {
            const float wgt = expf(logits[i] * mul - mx);
            if (wgt > 0.f) last = i;
            run += wgt;
            if (run > chosen) pick = i;
        }
        s_pick = pick >= 0 ? pick : last;
    }
    __syncthreads();
    if (tid == 0) out[0] = (uint32_t)(s_pick >= 0 ? s_pick : V - 1);
}

static __global__ void set_state_kernel(StepState* st, int rope_pos) { st->rope_pos = rope_pos; }
static __global__ void reset_state_kernel(StepState* st, int kv_len) {
    for (int i = threadIdx.x; i < kMaxBatch; i += blockDim.x) st->kv_base[i] = kv_len;
    if (threadIdx.x == 0) { st->rope_pos = 0; st->ragged = 0; }
}
// fl_forward_slots: batch row i runs on cache slot tab[i] at RoPE position tab[n + i]
static __global__ void set_slots_kernel(StepState* st, const int* __restrict__ tab, int n) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        st->slot[i] = tab[i];
        st->rope_seq[i] = tab[n + i];
    }
    if (threadIdx.x == 0) st->ragged = 1;
}
static __global__ void reset_slot_kernel(StepState* st, int slot) { st->kv_base[slot] = 0; }
// fl_cache_slot_fork: the forked slot's length
static __global__ void set_slot_len_kernel(StepState* st, int slot, int len) { st->kv_base[slot] = len; }
// Page-table entries a call changed: table[upd[i].x] = upd[i].y
static __global__ void page_table_scatter_kernel(int* __restrict__ table, const int2* __restrict__ upd, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) table[upd[i].x] = upd[i].y;
}
// fl_cache_slot_fork: copy one K or V page (blockIdx.z) of every layer (blockIdx.y) from page src to page dst, in bytes (any element
// type); page_bytes = nkv * 64 * d * element size, a multiple of 16
static __global__ void kv_page_copy_kernel(uint8_t* kpool, uint8_t* vpool, size_t layer_bytes, int src, int dst, int page_bytes) {
    uint8_t* pool = (blockIdx.z ? vpool : kpool) + (size_t)blockIdx.y * layer_bytes;
    const uint4* s = reinterpret_cast<const uint4*>(pool + (size_t)src * page_bytes);
    uint4* d = reinterpret_cast<uint4*>(pool + (size_t)dst * page_bytes);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < page_bytes / 16; i += gridDim.x * blockDim.x) d[i] = s[i];
}

}  // namespace fl
