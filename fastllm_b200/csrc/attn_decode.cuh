// Paged-KV decode attention, split-K over the sequence, bulk-copy (TMA engine) staging in shared memory, sm_100a.
//
// Replaces the reference's K6-K11 chain (SURVEY.md section 2.4): whole-cache `cat`, `repeat_kv` materialisation,
// q.k^T matmul, scale, mask, softmax_last_dim, att.v matmul, transpose.  Here:
//   * the KV cache is paged ([page][kv_head][64 tokens][d] bf16) and appended in place by the QKV GEMV epilogue;
//   * one CTA owns (split, kv_head, row): it streams its pages' K and V chunks (contiguous 64*d*2 bytes each) into a
//     2-stage shared-memory ring with cp.async.bulk + mbarrier, and serves ALL n_rep query heads of the GQA group from
//     the staged copy, so K/V are read from HBM exactly once (no repeat_kv);
//   * online softmax in f32 (running max / sum per head), partial (acc, m, l) per split, and the LAST CTA of each
//     (row, kv_head) -- elected with an atomic ticket -- merges the splits and writes the normalised output, so no
//     separate combine launch is needed;
//   * rows of a multi-token call (prefill chunks) are causal: row r sees kv_base + i_rel + 1 keys, and the
//     Mistral/Qwen2 sliding-window prefill rule (key j banned when j + sw < i, among the NEW tokens only: cached keys stay
//     visible, as candle concatenates zeros for the cached columns of its mask) is applied.
#pragma once
#include "common.cuh"
#include "gemv.cuh"

namespace fl {

constexpr int kAttnThreads = 128;
constexpr int kAttnMaxRep = 8;

struct AttnArgs {
    const float* q;        // [rows, nh, d] f32 (bias + RoPE applied)
    const uint16_t* kpool; // layer base, [page][nkv][kKvPage][d]
    const uint16_t* vpool;
    const int* page_table;
    int pt_stride;
    const StepState* state;
    float* part_acc;       // [rows, nh, nsplit, d]
    float* part_ml;        // [rows, nh, nsplit, 2]
    int* counters;         // [rows, nkv], zero between launches
    float* out;            // [rows, nh*d]
    uint16_t* out_hi;      // attn_mma.cuh kernels, optional: write the output as the hi/lo bf16 pair the o_proj GEMM consumes
    uint16_t* out_lo;      // (instead of `out`)
    int nh, nkv, t, row_base;
    int sliding_window;    // <= 0: none
    float qscale;          // q is multiplied by this (1/sqrt(d))
    // prefill kernels of attn_mma.cuh, packed calls: blockIdx.x is work item items[blockIdx.x] = (sequence, its first row, its
    // length, query tile) instead of a query tile of the uniform [b, t] grid (null)
    const int4* items;
};

template <int D>
__global__ void __launch_bounds__(kAttnThreads) attn_decode_kernel(const AttnArgs a) {
    constexpr int LPT = D / 8;                // lanes per token row (16-byte chunk each)
    constexpr int TPW = 32 / LPT;             // token rows per warp instruction
    constexpr int G = (kAttnThreads / 32) * TPW;   // token groups per CTA
    constexpr uint32_t kChunkBytes = kKvPage * D * 2;

    extern __shared__ __align__(128) uint8_t dsm[];
    uint16_t* kbuf = reinterpret_cast<uint16_t*>(dsm);                      // [2][kKvPage*D]
    uint16_t* vbuf = reinterpret_cast<uint16_t*>(dsm + 2 * kChunkBytes);    // [2][kKvPage*D]
    __shared__ __align__(16) float qs[kAttnMaxRep][D];
    __shared__ float sc[kAttnMaxRep][kKvPage];
    __shared__ float alpha_s[kAttnMaxRep], mrun[kAttnMaxRep], lrun[kAttnMaxRep];
    __shared__ __align__(8) uint64_t full[2];
    __shared__ int s_last;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int grp = lane / LPT, gl = lane % LPT;
    const int split = blockIdx.x, nsplit = gridDim.x, kvh = blockIdx.y, row = blockIdx.z;
    const int n_rep = a.nh / a.nkv;

    if (tid == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        mbar_fence_init();
    }
    pdl_launch_dependents();
    pdl_wait();

    const int rg = a.row_base + row;
    const int seq = rg / a.t, irel = rg % a.t;
    const int kv_base = a.state->kv_base[seq];
    const int len = kv_base + irel + 1;
    // candle's Mistral/Qwen2 mask is [t, t] over the NEW tokens (key j banned when j + sw < i) with ZEROS concatenated for the
    // cached columns: every cached key (< kv_base) stays visible, the window only thins out the new tokens
    const int start = (a.sliding_window > 0 && irel - a.sliding_window > 0) ? kv_base + irel - a.sliding_window : 0;
    const int first_page = kv_base > 0 ? 0 : start / kKvPage;
    const int npages = (len + kKvPage - 1) / kKvPage;
    const int per = (npages - first_page + nsplit - 1) / nsplit;
    const int p0 = first_page + split * per;
    const int p1 = min(p0 + per, npages);
    const int* pt = a.page_table + (size_t)seq * a.pt_stride;

    for (int i = tid; i < n_rep * D; i += kAttnThreads) {
        // stored as [half][chunk][4] so that the LPT lanes of a token row read contiguous 16-byte pieces (no bank conflicts)
        const int h = i / D, dd = i % D;
        qs[h][((dd >> 2) & 1) * (D / 2) + (dd >> 3) * 4 + (dd & 3)] =
            a.q[((size_t)row * a.nh + kvh * n_rep + h) * D + dd] * a.qscale;
    }
    if (tid < kAttnMaxRep) {
        mrun[tid] = -INFINITY;
        lrun[tid] = 0.f;
    }

    auto issue = [&](int p) {   // thread 0 only
        const int st = (p - p0) & 1;
        const size_t off = ((size_t)pt[p] * a.nkv + kvh) * (size_t)(kKvPage * D);
        mbar_expect_tx(&full[st], 2 * kChunkBytes);
        bulk_g2s(kbuf + st * (kKvPage * D), a.kpool + off, kChunkBytes, &full[st]);
        bulk_g2s(vbuf + st * (kKvPage * D), a.vpool + off, kChunkBytes, &full[st]);
    };
    __syncthreads();   // barrier init + qs visible
    if (tid == 0) {
        if (p0 < p1) issue(p0);
        if (p0 + 1 < p1) issue(p0 + 1);
    }

    float acc[kAttnMaxRep][8];
#pragma unroll
    for (int h = 0; h < kAttnMaxRep; ++h)
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[h][i] = 0.f;

    for (int p = p0; p < p1; ++p) {
        const int it = p - p0, st = it & 1;
        mbar_wait(&full[st], (it >> 1) & 1);
        const uint16_t* kb = kbuf + st * (kKvPage * D);
        const uint16_t* vb = vbuf + st * (kKvPage * D);

        // (1) scores for all heads of the group: LPT lanes per token, shuffle-reduce inside the lane group
#pragma unroll 2
        for (int tok = warp * TPW + grp; tok < kKvPage; tok += G) {
            const uint4 kw = *reinterpret_cast<const uint4*>(kb + tok * D + gl * 8);
            const float kf[8] = {bf16lo(kw.x), bf16hi(kw.x), bf16lo(kw.y), bf16hi(kw.y),
                                 bf16lo(kw.z), bf16hi(kw.z), bf16lo(kw.w), bf16hi(kw.w)};
            const int tok_abs = p * kKvPage + tok;
            const bool valid = (tok_abs >= start || tok_abs < kv_base) && tok_abs < len;
#pragma unroll
            for (int h = 0; h < kAttnMaxRep; ++h) {
                if (h < n_rep) {
                    const float4 q0 = *reinterpret_cast<const float4*>(&qs[h][gl * 4]);
                    const float4 q1 = *reinterpret_cast<const float4*>(&qs[h][D / 2 + gl * 4]);
                    float s = kf[0] * q0.x;
                    s = fmaf(kf[1], q0.y, s); s = fmaf(kf[2], q0.z, s); s = fmaf(kf[3], q0.w, s);
                    s = fmaf(kf[4], q1.x, s); s = fmaf(kf[5], q1.y, s); s = fmaf(kf[6], q1.z, s); s = fmaf(kf[7], q1.w, s);
#pragma unroll
                    for (int o = LPT / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
                    if (gl == 0) sc[h][tok] = valid ? s : -INFINITY;
                }
            }
        }
        __syncthreads();

        // (2) online-softmax statistics: warp w owns heads w, w+4
        for (int h = warp; h < n_rep; h += kAttnThreads / 32) {
            const float s0 = sc[h][lane], s1 = sc[h][lane + 32];
            const float m_old = mrun[h];
            const float m_new = fmaxf(m_old, warp_max(fmaxf(s0, s1)));
            float e0 = 0.f, e1 = 0.f, al = 1.f;
            if (m_new != -INFINITY) {
                e0 = expf(s0 - m_new);
                e1 = expf(s1 - m_new);
                al = expf(m_old - m_new);
            }
            const float sum = warp_sum(e0 + e1);
            sc[h][lane] = e0;
            sc[h][lane + 32] = e1;
            if (lane == 0) {
                alpha_s[h] = al;
                mrun[h] = m_new;
                lrun[h] = lrun[h] * al + sum;
            }
        }
        __syncthreads();

        // (3) acc = acc * alpha + P . V ; each lane group walks its share of the page's tokens
#pragma unroll
        for (int h = 0; h < kAttnMaxRep; ++h)
            if (h < n_rep) {
                const float al = alpha_s[h];
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[h][i] *= al;
            }
#pragma unroll 2
        for (int tok = warp * TPW + grp; tok < kKvPage; tok += G) {
            const uint4 vw = *reinterpret_cast<const uint4*>(vb + tok * D + gl * 8);
            const float vf[8] = {bf16lo(vw.x), bf16hi(vw.x), bf16lo(vw.y), bf16hi(vw.y),
                                 bf16lo(vw.z), bf16hi(vw.z), bf16lo(vw.w), bf16hi(vw.w)};
#pragma unroll
            for (int h = 0; h < kAttnMaxRep; ++h)
                if (h < n_rep) {
                    const float pr = sc[h][tok];
#pragma unroll
                    for (int i = 0; i < 8; ++i) acc[h][i] = fmaf(pr, vf[i], acc[h][i]);
                }
        }
        __syncthreads();   // everyone is done with stage st and with sc[]
        if (tid == 0 && p + 2 < p1) issue(p + 2);
    }

    // ---- cross-group reduction of acc (reuses the K staging buffer), partial write ----
    float* redbuf = reinterpret_cast<float*>(dsm);   // [G][n_rep][D] f32 <= 8*8*128*4 = 32 KB
#pragma unroll
    for (int h = 0; h < kAttnMaxRep; ++h)
        if (h < n_rep) {
            float* dst = redbuf + ((size_t)(warp * TPW + grp) * n_rep + h) * D + gl * 8;
#pragma unroll
            for (int i = 0; i < 8; ++i) dst[i] = acc[h][i];
        }
    __syncthreads();
    if (tid < D) {
        for (int h = 0; h < n_rep; ++h) {
            float s = 0.f;
#pragma unroll
            for (int g = 0; g < G; ++g) s += redbuf[((size_t)g * n_rep + h) * D + tid];
            a.part_acc[(((size_t)row * a.nh + kvh * n_rep + h) * nsplit + split) * D + tid] = s;
        }
    }
    if (tid < n_rep) {
        float* ml = a.part_ml + (((size_t)row * a.nh + kvh * n_rep + tid) * nsplit + split) * 2;
        ml[0] = mrun[tid];
        ml[1] = lrun[tid];
    }

    // ---- last CTA of this (row, kv head) merges the splits ----
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const int ticket = atomicAdd(&a.counters[row * a.nkv + kvh], 1);
        s_last = (ticket == nsplit - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // The merge is latency-bound (one CTA, L2 reads): spread it over all threads and keep many loads in flight.
    float* cm = reinterpret_cast<float*>(dsm);            // [n_rep][nsplit] split weights, reusing the staging buffer
    float* cden = cm + kAttnMaxRep * nsplit;              // [n_rep]
    __syncthreads();
    for (int h = warp; h < n_rep; h += kAttnThreads / 32) {
        const size_t base = ((size_t)row * a.nh + kvh * n_rep + h) * nsplit;
        float mstar = -INFINITY;
        for (int s = lane; s < nsplit; s += 32) mstar = fmaxf(mstar, __ldcg(a.part_ml + (base + s) * 2));
        mstar = warp_max(mstar);
        float den = 0.f;
        for (int s = lane; s < nsplit; s += 32) {
            const float ms = __ldcg(a.part_ml + (base + s) * 2);
            const float w = (ms == -INFINITY) ? 0.f : expf(ms - mstar);
            cm[h * nsplit + s] = w;
            den = fmaf(w, __ldcg(a.part_ml + (base + s) * 2 + 1), den);
        }
        den = warp_sum(den);
        if (lane == 0) cden[h] = den;
    }
    __syncthreads();
    constexpr int D4 = D / 4;
    for (int i = tid; i < n_rep * D4; i += kAttnThreads) {
        const int h = i / D4, c4 = i % D4;
        const float4* src = reinterpret_cast<const float4*>(a.part_acc + ((size_t)row * a.nh + kvh * n_rep + h) * nsplit * D) + c4;
        float4 num = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
        for (int s = 0; s < nsplit; ++s) {
            const float w = cm[h * nsplit + s];
            if (w != 0.f) {                                // empty splits hold unwritten (possibly non-finite) partials
                const float4 v = __ldcg(src + (size_t)s * D4);
                num.x = fmaf(w, v.x, num.x); num.y = fmaf(w, v.y, num.y); num.z = fmaf(w, v.z, num.z); num.w = fmaf(w, v.w, num.w);
            }
        }
        const float den = cden[h];
        float4 o = make_float4(num.x / den, num.y / den, num.z / den, num.w / den);
        reinterpret_cast<float4*>(a.out + (size_t)row * a.nh * D + (size_t)(kvh * n_rep + h) * D)[c4] = o;
    }
    if (tid == 0) a.counters[row * a.nkv + kvh] = 0;
}

}  // namespace fl
