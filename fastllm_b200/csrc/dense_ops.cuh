// Element-wise kernels of the dense (tensor-core) causal-LM path: prefill and batched decode (3+ activation rows), sm_100a.
// The GEMMs run on tcgen05 (gemm_tc.cuh) with bf16 operands; to stay within parity tolerance of the f32 oracle every f32
// activation x is split as x = hi + lo (hi = bf16(x), lo = bf16(x - hi)) and BOTH halves are multiplied with the same
// staged weight tile (DUAL mode), i.e. ~16 mantissa bits on the activation side at no extra weight traffic.
// These kernels implement the same fused steps as the GEMV epilogues in gemv.cuh (SURVEY.md section 2.4 K1-K18).
#pragma once
#include "common.cuh"
#include "gemm_tc.cuh"
#include "gemv.cuh"

namespace fl {

__device__ __forceinline__ void split_hi_lo(float x, uint16_t& hi, uint16_t& lo) {
    hi = f32_to_bf16_rne(x);
    lo = f32_to_bf16_rne(x - __uint_as_float((uint32_t)hi << 16));
}

__device__ __forceinline__ float block_sum_256(float v, float* red) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    __syncthreads();
    return s;
}

// Sum of the split-K slices of one element / pair, in slice order (deterministic), with the loads of up to eight slices in flight
// at once.  Measured per kernel (Mistral-7B batch 8): the q|k|v epilogue gains (8.1 -> 6.9 us), the RMSNorm / SiLU / arg-max kernels
// lose with eight (their plain loops already overlap across the threads' elements), so only the former and the MoE combine use it;
// the RMSNorm prologue keeps FOUR slice loads in flight (same-box A/B at batch 8: 1951 -> 1964-1970 tok/s, batch 64 unchanged).
__device__ __forceinline__ float sum_slices1(const float* p, long long stride, int nsl) {
    float acc = 0.f;
    for (int s0 = 0; s0 < nsl; s0 += 8) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = s0 + j < nsl ? p[(size_t)(s0 + j) * stride] : 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) if (s0 + j < nsl) acc += v[j];
    }
    return acc;
}
__device__ __forceinline__ float2 sum_slices2(const float* p, long long stride, int nsl) {
    float2 acc = make_float2(0.f, 0.f);
    for (int s0 = 0; s0 < nsl; s0 += 8) {
        float2 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = s0 + j < nsl ? *reinterpret_cast<const float2*>(p + (size_t)(s0 + j) * stride) : make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < 8; ++j) if (s0 + j < nsl) { acc.x += v[j].x; acc.y += v[j].y; }
    }
    return acc;
}
struct PrepArgs {
    const uint16_t* embed;      // non-null: resid[row] = f32(embed[ids[row]])  (K1)
    const uint32_t* ids;
    int vocab;
    float* resid;               // [R, K] residual stream (read, optionally updated)
    const float* delta;         // non-null: resid[row] += sum over slices of delta[row]  (K13 / K16 residual add), ldd floats per row
    int ldd;
    int nsl;                    // split-K slices of delta (>= 1), summed in order: deterministic
    long long sl_stride;
    const float* norm_w;        // non-null: x = rms_norm(resid) * norm_w, else x = src row
    float eps;
    const float* src;           // plain split source [R, K] (norm_w == null, embed == null)
    int K;
    int t;                      // last_only: output row j takes input row (j + 1) * t - 1
    int last_only;
    uint16_t* xhi;              // [R_out, K]
    uint16_t* xlo;
    const int* last_rows;       // optional (packed calls, dense_prep_kernel): output row j takes input row last_rows[j]
};

// one CTA per output row, float4-vectorised (K % 4 == 0); up to 1024 threads so a 4096-wide row is one load per thread
static __global__ void __launch_bounds__(1024) dense_prep_kernel(const PrepArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float red[32];
    const int orow = blockIdx.x;
    const int row = a.last_rows ? a.last_rows[orow] : (a.last_only ? (orow + 1) * a.t - 1 : orow);
    const int K = a.K, K4 = K >> 2;
    uint2* xh = reinterpret_cast<uint2*>(a.xhi + (size_t)orow * K);
    uint2* xl = reinterpret_cast<uint2*>(a.xlo + (size_t)orow * K);
    auto emit = [&](int i, const float4& x) {
        uint16_t h0, l0, h1, l1, h2, l2, h3, l3;
        split_hi_lo(x.x, h0, l0); split_hi_lo(x.y, h1, l1); split_hi_lo(x.z, h2, l2); split_hi_lo(x.w, h3, l3);
        xh[i] = make_uint2((uint32_t)h0 | ((uint32_t)h1 << 16), (uint32_t)h2 | ((uint32_t)h3 << 16));
        xl[i] = make_uint2((uint32_t)l0 | ((uint32_t)l1 << 16), (uint32_t)l2 | ((uint32_t)l3 << 16));
    };
    if (a.norm_w == nullptr && a.embed == nullptr) {      // plain hi/lo split of an f32 row
        const float4* s = reinterpret_cast<const float4*>(a.src + (size_t)row * K);
        for (int i = threadIdx.x; i < K4; i += blockDim.x) emit(i, s[i]);
        return;
    }
    float4* r = reinterpret_cast<float4*>(a.resid + (size_t)row * K);
    float ss = 0.f;
    for (int i = threadIdx.x; i < K4; i += blockDim.x) {
        float4 v;
        if (a.embed) {
            uint32_t id = a.ids[row];
            if (id >= (uint32_t)a.vocab) id = a.vocab - 1;
            const uint2 e = reinterpret_cast<const uint2*>(a.embed + (size_t)id * K)[i];
            v = make_float4(bf16lo(e.x), bf16hi(e.x), bf16lo(e.y), bf16hi(e.y));
            r[i] = v;
        } else {
            v = r[i];
            if (a.delta) {
                float4 ds = make_float4(0.f, 0.f, 0.f, 0.f);
                const float4* dp = reinterpret_cast<const float4*>(a.delta + (size_t)row * a.ldd) + i;
                const size_t st4 = (size_t)a.sl_stride / 4;
                int s = 0;
                for (; s + 4 <= a.nsl; s += 4) {          // four slice loads in flight, added in slice order (deterministic)
                    const float4 p0 = dp[(size_t)s * st4], p1 = dp[(size_t)(s + 1) * st4], p2 = dp[(size_t)(s + 2) * st4], p3 = dp[(size_t)(s + 3) * st4];
                    ds.x += p0.x; ds.y += p0.y; ds.z += p0.z; ds.w += p0.w;
                    ds.x += p1.x; ds.y += p1.y; ds.z += p1.z; ds.w += p1.w;
                    ds.x += p2.x; ds.y += p2.y; ds.z += p2.z; ds.w += p2.w;
                    ds.x += p3.x; ds.y += p3.y; ds.z += p3.z; ds.w += p3.w;
                }
                for (; s < a.nsl; ++s) {
                    const float4 p = dp[(size_t)s * st4];
                    ds.x += p.x; ds.y += p.y; ds.z += p.z; ds.w += p.w;
                }
                v.x += ds.x; v.y += ds.y; v.z += ds.z; v.w += ds.w;
                r[i] = v;
            }
        }
        ss = fmaf(v.x, v.x, ss); ss = fmaf(v.y, v.y, ss); ss = fmaf(v.z, v.z, ss); ss = fmaf(v.w, v.w, ss);
    }
    __syncthreads();
    const float tot = block_sum_256(ss, red);
    const float m = sqrtf(tot / (float)K + a.eps);       // candle rms_norm: x / sqrt(mean(x^2) + eps) * w
    for (int i = threadIdx.x; i < K4; i += blockDim.x) {
        const float4 v = r[i];
        const float4 wv = reinterpret_cast<const float4*>(a.norm_w)[i];
        emit(i, make_float4(v.x / m * wv.x, v.y / m * wv.y, v.z / m * wv.z, v.w / m * wv.w));
    }
}

// Many-row variant (prefill): 256 threads per row with the row held in registers between the sum-of-squares and the scaling pass
// (NV float4 per thread: K <= 1024 NV), so a row is read once and more rows are resident per SM.  Same arithmetic as
// dense_prep_kernel (slices summed in order, then added to the residual); only the residual-add + RMSNorm form.
constexpr int kPrepRowsThreads = 256;
template <int NV>
static __global__ void __launch_bounds__(kPrepRowsThreads) dense_prep_rows_kernel(const PrepArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float red[32];
    const int orow = blockIdx.x;
    const int row = a.last_only ? (orow + 1) * a.t - 1 : orow;
    const int K = a.K, K4 = K >> 2;
    uint2* xh = reinterpret_cast<uint2*>(a.xhi + (size_t)orow * K);
    uint2* xl = reinterpret_cast<uint2*>(a.xlo + (size_t)orow * K);
    float4* r = reinterpret_cast<float4*>(a.resid + (size_t)row * K);
    float4 v[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int i = threadIdx.x + j * kPrepRowsThreads;
        v[j] = i < K4 ? r[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (a.delta) {
        float4 ds[NV];
#pragma unroll
        for (int j = 0; j < NV; ++j) ds[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int s = 0; s < a.nsl; ++s) {         // fixed order: deterministic split-K reduction
            const float4* dp = reinterpret_cast<const float4*>(a.delta + (size_t)s * a.sl_stride + (size_t)row * a.ldd);
#pragma unroll
            for (int j = 0; j < NV; ++j) {
                const int i = threadIdx.x + j * kPrepRowsThreads;
                if (i < K4) {
                    const float4 p = dp[i];
                    ds[j].x += p.x; ds[j].y += p.y; ds[j].z += p.z; ds[j].w += p.w;
                }
            }
        }
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int i = threadIdx.x + j * kPrepRowsThreads;
            v[j].x += ds[j].x; v[j].y += ds[j].y; v[j].z += ds[j].z; v[j].w += ds[j].w;
            if (i < K4) r[i] = v[j];
        }
    }
    float ss = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {      // elements past K are zeros
        ss = fmaf(v[j].x, v[j].x, ss); ss = fmaf(v[j].y, v[j].y, ss); ss = fmaf(v[j].z, v[j].z, ss); ss = fmaf(v[j].w, v[j].w, ss);
    }
    const float tot = block_sum_256(ss, red);
    const float m = sqrtf(tot / (float)K + a.eps);       // candle rms_norm: x / sqrt(mean(x^2) + eps) * w
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int i = threadIdx.x + j * kPrepRowsThreads;
        if (i < K4) {
            const float4 wv = __ldg(reinterpret_cast<const float4*>(a.norm_w) + i);
            const float4 x = make_float4(v[j].x / m * wv.x, v[j].y / m * wv.y, v[j].z / m * wv.z, v[j].w / m * wv.w);
            uint16_t h0, l0, h1, l1, h2, l2, h3, l3;
            split_hi_lo(x.x, h0, l0); split_hi_lo(x.y, h1, l1); split_hi_lo(x.z, h2, l2); split_hi_lo(x.w, h3, l3);
            xh[i] = make_uint2((uint32_t)h0 | ((uint32_t)h1 << 16), (uint32_t)h2 | ((uint32_t)h3 << 16));
            xl[i] = make_uint2((uint32_t)l0 | ((uint32_t)l1 << 16), (uint32_t)l2 | ((uint32_t)l3 << 16));
        }
    }
}

struct QkvEpiArgs {
    int nsl;                   // split-K slices of y
    long long sl_stride;
    const float* y;            // [nsl][R, nqkv] GEMM output in the permuted row order of wqkv
    const float* bias;         // [nqkv] or null
    float* q_out;              // [R, nh*d]
    void* kpool;               // this layer's K / V pages, elements of the kernel's KV type (bf16 or e4m3)
    void* vpool;
    const int* page_table;
    int pt_stride;
    const StepState* state;
    const float* rope_cos;
    const float* rope_sin;
    int nh, nkv, d, max_pos, t, nqkv;
    uint16_t* vt;              // optional (prefill on the tcgen05 attention kernel): V of this call TRANSPOSED per 64-token page,
    int vt_pages;              // [sequence][kv head][vt_pages][d][64 tokens] -- the K-major B operand of O += P . V
    // packed calls (sequences of different lengths; dense_qkv_epi_kernel<true> only):
    int rows;                  // R: the kernel walks rows blockIdx.y, + gridDim.y, ...
    const int2* row_tab;       // [R] (sequence, position in the sequence) of every row
    const int* seq_len;        // [sequences] tokens each sequence is fed
    const int* vt_tile0;       // [sequences] first [d][64] tile of the sequence's V^T pages ([kv head][its pages]), or -1: none
    uint16_t* kt;              // FP8 caches with vt: K of this call as bf16 (the e4m3-rounded values) in pages [tile][64 tokens][d], the
                               // tiles numbered as the V^T tiles (the K operand of the tcgen05 prefill, which needs bf16 K)
};

// The V^T / K scratch tile of (sequence, kv head hkv, position irel), or -1 when the sequence's attention does not read the scratch.
template <bool PACKED>
__device__ __forceinline__ long long qkv_scratch_tile(const QkvEpiArgs& a, int seq, int irel, int hkv) {
    if constexpr (PACKED) {
        const int t0 = a.vt_tile0[seq];
        if (t0 < 0) return -1;
        return (long long)t0 + (long long)hkv * ((a.seq_len[seq] + kKvPage - 1) / kKvPage) + irel / kKvPage;
    } else {
        return ((long long)seq * a.nkv + hkv) * a.vt_pages + irel / kKvPage;
    }
}

// bias + RoPE (rotate-half) + q store + paged KV append of one row and column pair.  PACKED (packed calls): the row's sequence and
// position come from row_tab, its V^T tile from vt_tile0.  KV: element type of the pages (uint16_t = bf16, uint8_t = e4m3, each
// value rounded once from f32); the scratch copies for the tcgen05 prefill carry the stored value as bf16.
template <bool PACKED, typename KV>
__device__ __forceinline__ void qkv_epi_row(const QkvEpiArgs& a, int row, int pair) {
    const int ra = pair * 2;
    const int d = a.d, half = d >> 1;
    const int hh = ra / d, j = (ra % d) >> 1;
    const float2 vab = sum_slices2(a.y + (size_t)row * a.nqkv + ra, a.sl_stride, a.nsl);
    float va = vab.x, vb = vab.y;
    if (a.bias) { va += a.bias[ra]; vb += a.bias[ra + 1]; }
    int seq, irel;
    if constexpr (PACKED) {
        const int2 rt = a.row_tab[row];
        seq = rt.x;
        irel = rt.y;
    } else {
        seq = row / a.t;
        irel = row % a.t;
    }
    const int cslot = st_slot(a.state, seq);                    // cache slot of this sequence (its own index unless the call is ragged)
    const int slot = a.state->kv_base[cslot] + irel;
    const int page = a.page_table[cslot * a.pt_stride + slot / kKvPage];
    if (hh < a.nh + a.nkv) {
        int pos = st_rope(a.state, seq) + irel;
        pos = pos < a.max_pos ? pos : a.max_pos - 1;
        const float cs = a.rope_cos[(size_t)pos * half + j], sn = a.rope_sin[(size_t)pos * half + j];
        const float o1 = va * cs - vb * sn, o2 = va * sn + vb * cs;
        if (hh < a.nh) {
            float* q = a.q_out + ((size_t)row * a.nh + hh) * d;
            q[j] = o1;
            q[j + half] = o2;
        } else {
            KV* kp = static_cast<KV*>(a.kpool) + (((size_t)page * a.nkv + (hh - a.nh)) * kKvPage + slot % kKvPage) * d;
            if constexpr (kv_is_fp8<KV>) {
                const uint16_t e = f32x2_to_e4m3x2(o1, o2);
                kp[j] = (uint8_t)(e & 0xFFu);
                kp[j + half] = (uint8_t)(e >> 8);
                if (a.kt != nullptr) {
                    const long long tile = qkv_scratch_tile<PACKED>(a, seq, irel, hh - a.nh);
                    if (tile < 0) return;
                    uint16_t* tk = a.kt + ((size_t)tile * kKvPage + irel % kKvPage) * d;
                    const uint32_t b = e4m3x2_to_bf16x2(e);
                    tk[j] = (uint16_t)(b & 0xFFFFu);
                    tk[j + half] = (uint16_t)(b >> 16);
                }
            } else {
                kp[j] = f32_to_bf16_rne(o1);
                kp[j + half] = f32_to_bf16_rne(o2);
            }
        }
    } else {
        KV* vp = static_cast<KV*>(a.vpool) + (((size_t)page * a.nkv + (hh - a.nh - a.nkv)) * kKvPage + slot % kKvPage) * d;
        if constexpr (kv_is_fp8<KV>)
            *reinterpret_cast<uint16_t*>(vp + 2 * j) = f32x2_to_e4m3x2(va, vb);
        else
            *reinterpret_cast<uint32_t*>(vp + 2 * j) = (uint32_t)f32_to_bf16_rne(va) | ((uint32_t)f32_to_bf16_rne(vb) << 16);
        if (a.vt != nullptr) {
            const long long tile = qkv_scratch_tile<PACKED>(a, seq, irel, hh - a.nh - a.nkv);      // the [d][64] V^T tile
            if (tile < 0) return;       // this sequence's attention does not read the scratch
            uint16_t* tp = a.vt + ((size_t)tile * d + 2 * j) * kKvPage + irel % kKvPage;
            tp[0] = kv_round_bf16<KV>(va);
            tp[kKvPage] = kv_round_bf16<KV>(vb);
        }
    }
}

// thread per column pair, grid.y = row (PACKED: grid.y strides over the rows, which may be more than a grid dimension holds)
template <bool PACKED, typename KV>
static __global__ void dense_qkv_epi_kernel(const QkvEpiArgs a) {
    // the dependent (attention) kernel is released only AFTER this kernel's own wait: when it starts, the q|k|v GEMM -- and by
    // induction every earlier kernel of the stream -- has completed, so its preamble may read the step state, the page table and
    // every K/V page except the rows appended here before its own griddepcontrol.wait (attn_sk_decode_kernel streams them early)
    pdl_wait();
    pdl_launch_dependents();
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair * 2 >= a.nqkv) return;
    if constexpr (PACKED) {
        for (int row = blockIdx.y; row < a.rows; row += gridDim.y) qkv_epi_row<true, KV>(a, row, pair);
    } else {
        qkv_epi_row<false, KV>(a, blockIdx.y, pair);
    }
}

// Prefill variant (t % 8 == 0): one thread takes a column pair of EIGHT consecutive rows (tokens) of one sequence.  The one-row kernel
// is a chain of dependent small loads per thread (step state -> KV length -> page table -> store address, RoPE position -> cos / sin)
// repeated by 36 k CTAs of a 4096-token call, and its V^T scratch writes are 2-byte stores 128 bytes apart (126 us per layer against a
// 25 us memory floor on Qwen2.5-7B); here the chain is paid once per eight rows, their loads travel together, and the eight tokens of
// a V^T row are one 16-byte store.  Same arithmetic per element.
constexpr int kQkvRowsPerThread = 8;
template <typename KV>
static __global__ void __launch_bounds__(256) dense_qkv_epi_rows_kernel(const QkvEpiArgs a) {
    pdl_wait();
    pdl_launch_dependents();
    constexpr int RPT = kQkvRowsPerThread;
    const int row0 = blockIdx.y * RPT;
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair * 2 >= a.nqkv) return;
    const int ra = pair * 2;
    const int d = a.d, half = d >> 1;
    const int hh = ra / d, j = (ra % d) >> 1;
    float2 y[RPT];
#pragma unroll
    for (int r = 0; r < RPT; ++r) {      // (0 + first slice: the same additions as sum_slices2, so a -0.0 comes out the same way)
        const float2 p = *reinterpret_cast<const float2*>(a.y + (size_t)(row0 + r) * a.nqkv + ra);
        y[r] = make_float2(0.f + p.x, 0.f + p.y);
    }
    for (int s = 1; s < a.nsl; ++s) {      // further split-K slices, in slice order
#pragma unroll
        for (int r = 0; r < RPT; ++r) {
            const float2 p = *reinterpret_cast<const float2*>(a.y + (size_t)s * a.sl_stride + (size_t)(row0 + r) * a.nqkv + ra);
            y[r].x += p.x;
            y[r].y += p.y;
        }
    }
    if (a.bias) {
        const float b0 = a.bias[ra], b1 = a.bias[ra + 1];
#pragma unroll
        for (int r = 0; r < RPT; ++r) { y[r].x += b0; y[r].y += b1; }
    }
    const int seq = row0 / a.t, irel0 = row0 % a.t;             // t % 8 == 0: the eight rows belong to one sequence
    const int cslot = st_slot(a.state, seq);
    const int slot0 = a.state->kv_base[cslot] + irel0;
    if (hh < a.nh + a.nkv) {
        const int pos0 = st_rope(a.state, seq) + irel0;
        float cs[RPT], sn[RPT];
#pragma unroll
        for (int r = 0; r < RPT; ++r) {
            const int pos = min(pos0 + r, a.max_pos - 1);
            cs[r] = a.rope_cos[(size_t)pos * half + j];
            sn[r] = a.rope_sin[(size_t)pos * half + j];
        }
#pragma unroll
        for (int r = 0; r < RPT; ++r) {
            const float o1 = y[r].x * cs[r] - y[r].y * sn[r], o2 = y[r].x * sn[r] + y[r].y * cs[r];
            if (hh < a.nh) {
                float* q = a.q_out + ((size_t)(row0 + r) * a.nh + hh) * d;
                q[j] = o1;
                q[j + half] = o2;
            } else {
                const int slot = slot0 + r;
                const int page = a.page_table[cslot * a.pt_stride + slot / kKvPage];
                KV* kp = static_cast<KV*>(a.kpool) + (((size_t)page * a.nkv + (hh - a.nh)) * kKvPage + slot % kKvPage) * d;
                if constexpr (kv_is_fp8<KV>) {
                    const uint16_t e = f32x2_to_e4m3x2(o1, o2);
                    kp[j] = (uint8_t)(e & 0xFFu);
                    kp[j + half] = (uint8_t)(e >> 8);
                    if (a.kt != nullptr) {      // the eight rows lie in one page: irel0 % 8 == 0
                        uint16_t* tk = a.kt + ((size_t)qkv_scratch_tile<false>(a, seq, irel0, hh - a.nh) * kKvPage + (irel0 + r) % kKvPage) * d;
                        const uint32_t b = e4m3x2_to_bf16x2(e);
                        tk[j] = (uint16_t)(b & 0xFFFFu);
                        tk[j + half] = (uint16_t)(b >> 16);
                    }
                } else {
                    kp[j] = f32_to_bf16_rne(o1);
                    kp[j + half] = f32_to_bf16_rne(o2);
                }
            }
        }
    } else {
        const int hv = hh - a.nh - a.nkv;
        uint32_t va[RPT / 2], vb[RPT / 2];      // bf16 of column 2j / 2j + 1 for the eight tokens, packed in token order
#pragma unroll
        for (int r = 0; r < RPT; ++r) {
            const int slot = slot0 + r;
            const int page = a.page_table[cslot * a.pt_stride + slot / kKvPage];
            KV* vp = static_cast<KV*>(a.vpool) + (((size_t)page * a.nkv + hv) * kKvPage + slot % kKvPage) * d;
            uint32_t ba, bb;
            if constexpr (kv_is_fp8<KV>) {
                const uint16_t e = f32x2_to_e4m3x2(y[r].x, y[r].y);
                *reinterpret_cast<uint16_t*>(vp + 2 * j) = e;
                const uint32_t b = e4m3x2_to_bf16x2(e);
                ba = b & 0xFFFFu;
                bb = b >> 16;
            } else {
                ba = f32_to_bf16_rne(y[r].x);
                bb = f32_to_bf16_rne(y[r].y);
                *reinterpret_cast<uint32_t*>(vp + 2 * j) = ba | (bb << 16);
            }
            if (r & 1) { va[r >> 1] |= ba << 16; vb[r >> 1] |= bb << 16; } else { va[r >> 1] = ba; vb[r >> 1] = bb; }
        }
        if (a.vt != nullptr) {      // irel0 % 8 == 0: the eight tokens are 16 aligned bytes of one V^T row
            uint16_t* tp = a.vt + ((((size_t)seq * a.nkv + hv) * a.vt_pages + irel0 / kKvPage) * d + 2 * j) * kKvPage + irel0 % kKvPage;
            *reinterpret_cast<uint4*>(tp) = make_uint4(va[0], va[1], va[2], va[3]);
            *reinterpret_cast<uint4*>(tp + kKvPage) = make_uint4(vb[0], vb[1], vb[2], vb[3]);
        }
    }
}

// act = silu(gate) * up from the interleaved gate|up GEMM output, written directly as the hi/lo split the down GEMM reads
// (grouped expert GEMMs: rows are blocks of `grp_cap` per expert, of which grp_cnt[block] are valid; the rest is skipped)
static __global__ void dense_silu_split_kernel(const float* __restrict__ y, int nsl, long long sl_stride, int I, uint16_t* __restrict__ xhi,
                                               uint16_t* __restrict__ xlo, const int* __restrict__ grp_cnt = nullptr, int grp_cap = 0) {
    pdl_launch_dependents();
    pdl_wait();
    const int row = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= I) return;
    if (grp_cnt != nullptr && (row % grp_cap) >= grp_cnt[row / grp_cap]) return;
    float2 gu = make_float2(0.f, 0.f);
    for (int s = 0; s < nsl; ++s) {
        const float2 p = *reinterpret_cast<const float2*>(y + (size_t)s * sl_stride + (size_t)row * 2 * I + 2 * j);
        gu.x += p.x;
        gu.y += p.y;
    }
    const float act = gu.x / (1.f + expf(-gu.x)) * gu.y;
    uint16_t h, l;
    split_hi_lo(act, h, l);
    xhi[(size_t)row * I + j] = h;
    xlo[(size_t)row * I + j] = l;
}

// ---- Mixtral sparse-MoE (candle-transformers models::mixtral::SparseMoeBlock; SURVEY.md section 8a row 7) ----------------
// router: logits = x . W_gate^T, softmax over ALL experts (f32), stable descending sort (ties keep the LOWER expert index),
// take top_k, renormalise by their sum; route_w[row][e] = weight or 0.  One CTA per row, one WARP per expert (128-bit loads,
// one shuffle reduction each): the eight dot products of a Mixtral row run side by side instead of as eight block reductions.
static __global__ void __launch_bounds__(256) moe_router_kernel(const uint16_t* __restrict__ xhi, const uint16_t* __restrict__ xlo, int H,
                                                                const float* __restrict__ wgate, int E, int top_k, float* __restrict__ route_w,
                                                                int* __restrict__ sel_log, float* __restrict__ margin_log) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float logit[64];
    const int row = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint2* h4 = reinterpret_cast<const uint2*>(xhi + (size_t)row * H);      // 4 bf16 per load (H % 8 == 0 on the dense path)
    const uint2* l4 = reinterpret_cast<const uint2*>(xlo + (size_t)row * H);
    for (int e = warp; e < E; e += 8) {
        const float4* wg = reinterpret_cast<const float4*>(wgate + (size_t)e * H);
        float acc = 0.f;
        for (int i = lane; i < H / 4; i += 32) {
            const uint2 a = h4[i], b = l4[i];
            const float4 w = wg[i];
            acc = fmaf(bf16lo(a.x) + bf16lo(b.x), w.x, acc);
            acc = fmaf(bf16hi(a.x) + bf16hi(b.x), w.y, acc);
            acc = fmaf(bf16lo(a.y) + bf16lo(b.y), w.z, acc);
            acc = fmaf(bf16hi(a.y) + bf16hi(b.y), w.w, acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) logit[e] = acc;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float mx = -INFINITY;
        for (int e = 0; e < E; ++e) mx = fmaxf(mx, logit[e]);
        float sum = 0.f;
        for (int e = 0; e < E; ++e) { logit[e] = expf(logit[e] - mx); sum += logit[e]; }
        for (int e = 0; e < E; ++e) logit[e] /= sum;                 // softmax_last_dim
        float* rw = route_w + (size_t)row * E;
        for (int e = 0; e < E; ++e) rw[e] = 0.f;
        float picked_sum = 0.f;
        unsigned long long taken = 0ull;
        int picked[8];
        for (int k = 0; k < top_k; ++k) {                            // k-th largest, lowest index among equals
            int best = -1;
            for (int e = 0; e < E; ++e)
                if (!((taken >> e) & 1ull) && (best < 0 || logit[e] > logit[best])) best = e;
            taken |= 1ull << best;
            picked[k] = best;
            picked_sum += logit[best];                               // sum::<f32>() in rank order
        }
        for (int k = 0; k < top_k; ++k) rw[picked[k]] = logit[picked[k]] / picked_sum;
        // routing record for the sharded-vs-single-GPU checks (fl_cache_moe_routing): the picked experts in rank order and how far
        // the last pick was from not being picked (softmax-probability gap to the best expert left out)
        if (sel_log != nullptr) {
            float next = -INFINITY;
            for (int e = 0; e < E; ++e)
                if (!((taken >> e) & 1ull)) next = fmaxf(next, logit[e]);
            for (int k = 0; k < top_k; ++k) sel_log[(size_t)row * top_k + k] = picked[k];
            margin_log[row] = logit[picked[top_k - 1]] - next;
        }
    }
}

// Grouped expert GEMMs (decode batches): the rows routed to each LOCAL expert are gathered into that expert's block of a
// stacked activation buffer (candle: index_select of the rows per expert), in ascending row order.
//   gx_hi / gx_lo [E_local * cap, H] : block j holds the hi / lo halves of the rows routed to expert e0 + j
//   cnt [E_local]                    : rows in block j (read by the grouped GEMM, the SiLU kernel and nobody else)
//   pos [Rm, E_local]                : slot (j * cap + p) of row r in block j, or -1: the combine kernel's scatter map
// grid (E_local, copy CTAs), 256 threads; every CTA of an expert rebuilds the (<= 256-entry) list, then copies its share of rows.
struct MoeGatherArgs {
    const uint16_t* xhi;
    const uint16_t* xlo;
    const float* route;      // [Rm, E]
    int Rm, H, E, e0, E_local, cap;
    uint16_t* gx_hi;
    uint16_t* gx_lo;
    int* cnt;
    int* pos;
};
static __global__ void moe_gather_kernel(const MoeGatherArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ int s_list[256];
    __shared__ int s_cnt;
    const int j = blockIdx.x, e = a.e0 + j, tid = threadIdx.x, lane = tid & 31;
    if (tid < 32) {
        int n = 0;
        for (int r0 = 0; r0 < a.Rm; r0 += 32) {
            const int r = r0 + lane;
            const bool sel = r < a.Rm && a.route[(size_t)r * a.E + e] != 0.f;
            const unsigned m = __ballot_sync(0xFFFFFFFFu, sel);
            if (sel) s_list[n + __popc(m & ((1u << lane) - 1u))] = r;
            n += __popc(m);
        }
        if (lane == 0) s_cnt = n;
    }
    __syncthreads();
    const int n = s_cnt;
    if (blockIdx.y == 0) {
        if (tid == 0) a.cnt[j] = n;
        for (int r = tid; r < a.Rm; r += blockDim.x) a.pos[(size_t)r * a.E_local + j] = -1;
        __syncthreads();
        for (int p = tid; p < n; p += blockDim.x) a.pos[(size_t)s_list[p] * a.E_local + j] = j * a.cap + p;
    }
    const int H8 = a.H / 8;
    for (int p = blockIdx.y; p < n; p += gridDim.y) {
        const uint4* sh = reinterpret_cast<const uint4*>(a.xhi + (size_t)s_list[p] * a.H);
        const uint4* sl = reinterpret_cast<const uint4*>(a.xlo + (size_t)s_list[p] * a.H);
        uint4* dh = reinterpret_cast<uint4*>(a.gx_hi + ((size_t)j * a.cap + p) * a.H);
        uint4* dl = reinterpret_cast<uint4*>(a.gx_lo + ((size_t)j * a.cap + p) * a.H);
        for (int i = tid; i < H8; i += blockDim.x) {
            dh[i] = sh[i];
            dl[i] = sl[i];
        }
    }
}

// index_add of the weighted expert outputs: moe_out[row] = sum over this rank's experts j (ascending: a fixed order) that
// selected the row of route[row][e0 + j] * (sum over split-K slices of y[slot of the row in block j])
static __global__ void moe_combine_kernel(const float* __restrict__ y, int nsl, long long sl_stride, int H, const float* __restrict__ route, int E,
                                          int e0, int E_local, const int* __restrict__ pos, float* __restrict__ moe_out) {
    pdl_launch_dependents();
    pdl_wait();
    const int row = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= H) return;
    float v = 0.f;
    for (int j = 0; j < E_local; ++j) {
        const int p = pos[(size_t)row * E_local + j];
        if (p < 0) continue;
        v += route[(size_t)row * E + e0 + j] * sum_slices1(y + (size_t)p * H + i, sl_stride, nsl);
    }
    moe_out[(size_t)row * H + i] = v;
}

// moe_out[row] (=|+=) route_w[row][e] * sum over split-K slices of y[row]   (index_add of the weighted expert output)
static __global__ void moe_accum_kernel(const float* __restrict__ y, int nsl, long long sl_stride, int H, const float* __restrict__ route_w,
                                        int E, int e, int first, float* __restrict__ moe_out) {
    pdl_launch_dependents();
    pdl_wait();
    const int row = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= H) return;
    const float v = route_w[(size_t)row * E + e] * sum_slices1(y + (size_t)row * H + i, sl_stride, nsl);
    float* o = moe_out + (size_t)row * H + i;
    *o = first ? v : (*o + v);
}

// arg-max over the vocabulary, one CTA per row, last index wins ties (candle LogitsProcessor::sample_argmax)
// (also folds the split-K slices of the lm_head GEMM into the f32 logits buffer the caller reads)
static __global__ void __launch_bounds__(1024) dense_argmax_kernel(const float* __restrict__ y, int nsl, long long sl_stride, int V,
                                                                  float* __restrict__ logits, uint32_t* __restrict__ next_ids) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float sv[32];
    __shared__ int si[32];
    float* l = logits + (size_t)blockIdx.x * V;
    float v = -INFINITY;
    int idx = -1;
    for (int i = threadIdx.x; i < V; i += blockDim.x) {
        float x = 0.f;
        for (int s = 0; s < nsl; ++s) x += y[(size_t)s * sl_stride + (size_t)blockIdx.x * V + i];
        l[i] = x;
        if (x >= v) { v = x; idx = i; }      // i ascends per thread: >= keeps the last
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xFFFFFFFFu, v, o);
        const int oi = __shfl_xor_sync(0xFFFFFFFFu, idx, o);
        if (ov > v || (ov == v && oi > idx)) { v = ov; idx = oi; }
    }
    if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = v; si[threadIdx.x >> 5] = idx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
            if (sv[w] > v || (sv[w] == v && si[w] > idx)) { v = sv[w]; idx = si[w]; }
        next_ids[blockIdx.x] = (uint32_t)idx;
    }
}

// Scoring: one warp per row merges the row's nparts soft-max partials (the lm_head's GEPI_LOGPROB epilogue) -- lane l takes
// partials l, l + 32, ... in order, then a fixed butterfly -- so the result does not depend on the grid.
// logprob[row] = z[target] - (m + log s); argmax[row] = the last index among equal maxima (a NaN never wins).
constexpr int kLogprobRowsPerCta = 8;
static __global__ void __launch_bounds__(32 * kLogprobRowsPerCta) logprob_combine_kernel(const LogprobPart* __restrict__ part, int nparts,
                                                                                       const float* __restrict__ target_logit, int R,
                                                                                       float* __restrict__ logprob, uint32_t* __restrict__ argmax) {
    pdl_launch_dependents();
    pdl_wait();
    const int row = blockIdx.x * kLogprobRowsPerCta + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= R) return;
    const LogprobPart* p = part + (size_t)row * nparts;
    float m = -INFINITY, s = 0.f;
    int idx = -1;
    for (int i = lane; i < nparts; i += 32) {
        const LogprobPart q = p[i];
        logprob_merge(m, s, idx, q.m, q.s, q.idx);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float m2 = __shfl_xor_sync(0xFFFFFFFFu, m, o), s2 = __shfl_xor_sync(0xFFFFFFFFu, s, o);
        const int i2 = __shfl_xor_sync(0xFFFFFFFFu, idx, o);
        logprob_merge(m, s, idx, m2, s2, i2);
    }
    if (lane == 0) {
        logprob[row] = target_logit[row] - (m + logf(s));
        argmax[row] = (uint32_t)idx;
    }
}

}  // namespace fl
