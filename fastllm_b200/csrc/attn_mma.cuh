// Tensor-core attention over the paged bf16 KV cache for the dense path (3+ activation rows), sm_100a.
//
//   attn_sk_decode_kernel<D>   : batched decode (one new token per sequence), stream-K: a fixed grid of resident CTAs cuts the
//       step's whole K|V page stream into equal ranges; a producer warp streams the range through a 2-D TMA ring, 4 consumer
//       warps fold 16 keys of every page each into an online softmax (mma.sync m16n8k16, the GQA group's heads are the M rows),
//       pairs that straddle ranges are merged by the last-arriving CTA.  HBM-bound.  Details at the kernel.
//   attn_prefill_kernel<D>     : multi-token calls (prefill).  One CTA per (64-query tile, q head, sequence): FlashAttention-
//       style loop over the causal range of 64-key pages, S = Q K^T and O += P V on mma.sync, online softmax in registers.
//       Replaces the row-per-CTA decode kernel in prefill (84 % of the Qwen2.5-7B 4k prefill before).
//
// Precision: q and the softmax probabilities are f32 in the oracle.  Both are split hi + lo into two bf16 operands and
// multiplied against the same K / V fragments (as the dense GEMMs do with their activations), K/V are bf16 in the cache
// already, accumulation is f32: results stay inside the kernel tolerance of the f32 oracle.
// Semantics (SURVEY.md section 8a rows 1, 3, 4): scores * 1/sqrt(d) after the matmul, causal rows for multi-token calls,
// Mistral/Qwen2 sliding-window rule inside the prefill only (key j banned when j + sw < i, new tokens only; cached keys stay visible), softmax max-subtract/exp/sum/div.
#pragma once
#include "attn_decode.cuh"
#include "dense_ops.cuh"
#include "gemm_tc.cuh"
#include "mma.cuh"

namespace fl {

constexpr int kMmaAttnThreads = 128;
constexpr int kPrefillBM = 64;       // query rows per CTA of the prefill kernel (4 warps x 16)

// element offset of (row, col) in a [rows][D] bf16 tile whose 16-byte chunks are XOR-swizzled by the row (conflict-free ldmatrix)
template <int D>
__device__ __forceinline__ int swz(int row, int col) {
    constexpr int CH = D / 8;
    constexpr int MASK = (CH < 8 ? CH : 8) - 1;
    return row * D + ((((col >> 3) ^ (row & MASK))) << 3) + (col & 7);
}

template <int D>
__device__ __forceinline__ void stage_kv_tile(uint16_t* kd, uint16_t* vd, const uint16_t* ksrc, const uint16_t* vsrc, int tid) {
    constexpr int CH = D / 8;
#pragma unroll
    for (int i = tid; i < kKvPage * CH; i += kMmaAttnThreads) {
        const int r = i / CH, c = i % CH;
        cp_async16(kd + swz<D>(r, c * 8), ksrc + r * D + c * 8);
        cp_async16(vd + swz<D>(r, c * 8), vsrc + r * D + c * 8);
    }
    cp_async_commit();
}

// f32 q rows -> hi/lo bf16 tiles [NR][D] (rows >= valid rows are zero)
__device__ __forceinline__ void store_hi_lo(uint16_t* hi, uint16_t* lo, int off, float x) {
    uint16_t h, l;
    split_hi_lo(x, h, l);
    hi[off] = h;
    lo[off] = l;
}

// writes one output element either as f32 or as the hi/lo bf16 pair the next GEMM consumes
__device__ __forceinline__ void store_out2(const AttnArgs& a, size_t idx, float x0, float x1) {
    if (a.out_hi) {
        uint16_t h0, l0, h1, l1;
        split_hi_lo(x0, h0, l0);
        split_hi_lo(x1, h1, l1);
        *reinterpret_cast<uint32_t*>(a.out_hi + idx) = (uint32_t)h0 | ((uint32_t)h1 << 16);
        *reinterpret_cast<uint32_t*>(a.out_lo + idx) = (uint32_t)l0 | ((uint32_t)l1 << 16);
    } else {
        *reinterpret_cast<float2*>(a.out + idx) = make_float2(x0, x1);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// batched decode, stream-K: a fixed grid of resident CTAs splits the batch's whole K|V page stream evenly
// ---------------------------------------------------------------------------------------------------------------------
// A kernel that hands each (split, kv head, sequence) to a CTA (round 1): the number of CTAs is a multiple of the pairs, not of
// the machine (batch 64 x 8 kv heads x 3 splits = 1536 CTAs on 444 slots = 3.46 waves; Mixtral's batch 32 = 256 CTAs on 444
// slots), every CTA re-pays set-up, q conversion and merge, and its cp.async ring drains at every CTA boundary.  Here the pages
// of all (sequence, kv head) pairs form ONE list (pair-major) cut into gridDim.x equal ranges:
//   * the producer warp streams the range's pages through a ring of K|V stages with 2-D TMA (one 64-row x 128-byte box per
//     half tile, 128-byte swizzle = the conflict-free ldmatrix layout; SASS UTMALDG) and never stops at a pair boundary;
//   * 4 consumer warps (16 keys of every page each, mma.sync m16n8k16, heads of the GQA group = the M rows) wait on the stage's
//     mbarrier, fold the page into their online softmax, release the stage -- no CTA-wide barrier per page;
//   * a pair that lies inside one range is finished by that CTA alone; a pair that straddles ranges leaves one partial per CTA
//     (at most two per CTA: its first and its last pair) and the last-arriving CTA of the pair merges them in CTA order, so
//     the result is deterministic for a given batch composition.
// Ragged batches (continuous batching) balance the same way: the split is by pages, not by sequences.
constexpr int kSkConsumerWarps = 4;
constexpr int kSkConsumers = kSkConsumerWarps * 32;
constexpr int kSkThreads = kSkConsumers + 32;
// K|V stages of the ring; with up to 3 resident CTAs per SM (attn_sk_plan in fl_lib.cu).  Measured on Mistral-7B at 2k context:
// batch 64 is the same with 3 stages x 2 CTAs (6.83 vs 6.84 ms/step), batch 8 is better with more, smaller ranges (4.07 vs
// 4.17 ms/step); 4 stages x 1 CTA loses 14 %.
constexpr int kSkStages = 2;

// element offset of (row, col) inside a staged 64 x D K or V page.  D >= 64: [D / 64 halves][64 rows][128 bytes] with the TMA
// engine's 128-byte swizzle (16-byte chunk index XOR row & 7); D < 64 (test-size heads): the plain [64][D] box, no swizzle.
template <int D>
__device__ __forceinline__ int kv_off(int row, int col) {
    if constexpr (D >= 64) return (col >> 6) * (kKvPage * 64) + row * 64 + (((((col >> 3) & 7) ^ (row & 7))) << 3) + (col & 7);
    else return row * D + col;
}

struct SkArgs {
    AttnArgs a;
    float* sk_acc;        // [gridDim.x][2][n_rep][D] partial numerators of the pairs a CTA shares with its neighbours
    float* sk_ml;         // [gridDim.x][2][n_rep][2] their running max / denominator
    int b;                // sequences in the step
    int layer_row0;       // row of this layer's page 0 / kv head 0 in the pool-wide tensor maps
};

template <int D>
__global__ void __launch_bounds__(kSkThreads) attn_sk_decode_kernel(const __grid_constant__ CUtensorMap tmk, const __grid_constant__ CUtensorMap tmv,
                                                                    const SkArgs k) {
    const AttnArgs& a = k.a;
    constexpr int TILE = kKvPage * D;
    constexpr int NW = kSkConsumerWarps;
    extern __shared__ __align__(1024) uint8_t sksm[];
    const int n_rep = a.nh / a.nkv;
    // q tiles (hi | lo, [16][D] each) and the cross-warp merge scratch ([NW][n_rep][D] f32) share the front region: the scratch is
    // written when a pair's last page is done, the q tiles are rewritten before the next pair starts
    const int front = max(2 * 16 * D * 2, NW * n_rep * D * 4);
    uint16_t* qhi = reinterpret_cast<uint16_t*>(sksm);
    uint16_t* qlo = qhi + 16 * D;
    float* red_o = reinterpret_cast<float*>(sksm);
    uint16_t* ring = reinterpret_cast<uint16_t*>(sksm + ((front + 1023) & ~1023));
    __shared__ __align__(8) uint64_t full[kSkStages];
    __shared__ __align__(8) uint64_t empty[kSkStages];
    __shared__ float red_m[NW][16], red_l[NW][16], mrg_w[NW][16], mrg_den[16], mrg_star[16];
    __shared__ int prefix[kMaxBatch + 1];        // pages of the sequences before s
    __shared__ int s_len[kMaxBatch], s_slot[kMaxBatch];
    __shared__ int s_last, s_i0, s_i1;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, tq = lane & 3;
    if (tid == 0) {
        for (int s = 0; s < kSkStages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], NW);
        }
        mbar_fence_init();
    }
    pdl_launch_dependents();
    // No griddepcontrol.wait yet: the step state, the page table and every K/V row except the one the preceding kernel
    // (dense_qkv_epi_kernel) appends were written by kernels that completed before this one could start (that kernel releases its
    // dependents only after its own wait).  The producer streams all pages that cannot hold the new token right away; q, the new
    // K/V row and the output buffers are touched only after the wait.
    for (int i = tid; i < k.b; i += kSkThreads) {
        const int slot = st_slot(a.state, i);
        const int len = a.state->kv_base[slot] + 1;
        s_slot[i] = slot;
        s_len[i] = len;
        prefix[i + 1] = (len + kKvPage - 1) / kKvPage;
    }
    if (tid == 0) prefix[0] = 0;
    __syncthreads();
    if (warp == 0) {      // inclusive scan of the page counts
        int carry = 0;
        for (int base = 0; base < k.b; base += 32) {
            int v = base + lane < k.b ? prefix[base + lane + 1] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xFFFFFFFFu, v, o);
                if (lane >= o) v += t;
            }
            if (base + lane < k.b) prefix[base + lane + 1] = v + carry;
            carry += __shfl_sync(0xFFFFFFFFu, v, 31);
        }
    }
    __syncthreads();
    const long long P = (long long)a.nkv * prefix[k.b];          // pages of the whole step (K and V of a page travel together)
    const int G = (int)min((long long)gridDim.x, P);              // every participating CTA owns at least one page
    const int cta = blockIdx.x;
    if (cta >= G) return;
    const long long flat0 = (long long)cta * P / G, flat1 = (long long)(cta + 1) * P / G;
    // flat index -> (sequence, kv head, page): pair-major, a sequence's nkv pairs are adjacent
    auto locate = [&](long long n, int& s, int& h, int& p) {
        int lo = 0, hi = k.b - 1;
        while (lo < hi) {      // largest s with nkv * prefix[s] <= n
            const int mid = (lo + hi + 1) >> 1;
            if ((long long)a.nkv * prefix[mid] <= n) lo = mid; else hi = mid - 1;
        }
        s = lo;
        const int np = prefix[s + 1] - prefix[s];
        const int rem = (int)(n - (long long)a.nkv * prefix[s]);
        h = rem / np;
        p = rem - h * np;
    };

    // =================================================================================================================
    // producer warp: page-table entries are fetched 32 pages at a time (one per lane), lane 0 issues the TMA requests
    // =================================================================================================================
    if (warp == NW) {
        unsigned int c = 0;
        bool waited = false;
        for (long long base = flat0; base < flat1; base += 32) {
            const long long n = base + lane;
            int row = 0;
            if (n < flat1) {
                int s, h, p;
                locate(n, s, h, p);
                const int pg = a.page_table[(size_t)s_slot[s] * a.pt_stride + p];
                row = k.layer_row0 + (pg * a.nkv + h) * kKvPage;
                if (p == prefix[s + 1] - prefix[s] - 1) row |= 1 << 31;      // the sequence's last page: holds the token appended in this step
            }
            const int cnt = (int)min(32LL, flat1 - base);
            for (int j = 0; j < cnt; ++j, ++c) {
                int r = __shfl_sync(0xFFFFFFFFu, row, j);
                if (r < 0 && !waited) {
                    pdl_wait();
                    waited = true;
                }
                r &= 0x7FFFFFFF;
                if (lane == 0) {
                    const int st = c % kSkStages;
                    mbar_wait(&empty[st], ((c / kSkStages) & 1) ^ 1);
                    mbar_expect_tx(&full[st], 2u * TILE * 2u);
                    uint16_t* kd = ring + (size_t)st * 2 * TILE;
                    if constexpr (D >= 64) {
#pragma unroll
                        for (int hf = 0; hf < D / 64; ++hf) {
                            tma_load_2d(kd + hf * (kKvPage * 64), &tmk, hf * 64, r, &full[st]);
                            tma_load_2d(kd + TILE + hf * (kKvPage * 64), &tmv, hf * 64, r, &full[st]);
                        }
                    } else {
                        tma_load_2d(kd, &tmk, 0, r, &full[st]);
                        tma_load_2d(kd + TILE, &tmv, 0, r, &full[st]);
                    }
                }
            }
        }
        return;
    }

    // =================================================================================================================
    // consumers
    // =================================================================================================================
    auto csync = [] { asm volatile("bar.sync 1, %0;" ::"n"(kSkConsumers) : "memory"); };
    pdl_wait();
    int s, h, p;
    locate(flat0, s, h, p);
    float o[D / 8][4];
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
    bool open = false, from_start = false;
    unsigned int c = 0;
    for (long long n = flat0; n < flat1; ++n, ++c) {
        const int np = prefix[s + 1] - prefix[s], len = s_len[s];
        if (!open) {       // first page of this CTA's share of pair (s, h): stage q, reset the running softmax
            csync();       // the previous pair's readers of the merge scratch are done
            for (int i = tid; i < 16 * D; i += kSkConsumers) {
                const int hh = i / D, dd = i % D;
                const float q = hh < n_rep ? a.q[((size_t)s * a.nh + h * n_rep + hh) * D + dd] : 0.f;
                store_hi_lo(qhi, qlo, swz<D>(hh, dd), q);
            }
            csync();
#pragma unroll
            for (int i = 0; i < D / 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
            m0 = m1 = -INFINITY;
            l0 = l1 = 0.f;
            open = true;
            from_start = (p == 0);
        }
        const int st = c % kSkStages;
        mbar_wait(&full[st], (c / kSkStages) & 1);
        const uint16_t* kt = ring + (size_t)st * 2 * TILE;
        const uint16_t* vt = kt + TILE;
        const int key0 = p * kKvPage + warp * 16;
        if (key0 < len) {
            float sc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
            for (int ks = 0; ks < D / 16; ++ks) {
                uint32_t ah[4], al[4], kb[4];
                ldmatrix_x4(ah, qhi + swz<D>(lane & 15, ks * 16 + (lane >> 4) * 8));
                ldmatrix_x4(al, qlo + swz<D>(lane & 15, ks * 16 + (lane >> 4) * 8));
                ldmatrix_x4(kb, kt + kv_off<D>(warp * 16 + (lane & 7) + ((lane >> 4) << 3), ks * 16 + ((lane >> 3) & 1) * 8));
                mma_bf16_16816(sc[0], ah, kb[0], kb[1]);
                mma_bf16_16816(sc[0], al, kb[0], kb[1]);
                mma_bf16_16816(sc[1], ah, kb[2], kb[3]);
                mma_bf16_16816(sc[1], al, kb[2], kb[3]);
            }
            float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int key = key0 + nt * 8 + tq * 2 + (e & 1);
                    sc[nt][e] = key < len ? sc[nt][e] * a.qscale : -INFINITY;
                    if (e < 2) mx0 = fmaxf(mx0, sc[nt][e]); else mx1 = fmaxf(mx1, sc[nt][e]);
                }
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xFFFFFFFFu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xFFFFFFFFu, mx0, 2));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xFFFFFFFFu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xFFFFFFFFu, mx1, 2));
            const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);       // finite: key0 < len is valid for every row
            const float al0 = expf(m0 - mn0), al1 = expf(m1 - mn1);
            m0 = mn0; m1 = mn1;
            float ps0 = 0.f, ps1 = 0.f;
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                sc[nt][0] = expf(sc[nt][0] - mn0); sc[nt][1] = expf(sc[nt][1] - mn0);
                sc[nt][2] = expf(sc[nt][2] - mn1); sc[nt][3] = expf(sc[nt][3] - mn1);
                ps0 += sc[nt][0] + sc[nt][1];
                ps1 += sc[nt][2] + sc[nt][3];
            }
            l0 = l0 * al0 + ps0;       // per-thread partial row sums; the quad is reduced when the pair is emitted
            l1 = l1 * al1 + ps1;
            uint32_t ph[4], pl[4];
            ph[0] = pack_bf16x2(sc[0][0], sc[0][1]); ph[1] = pack_bf16x2(sc[0][2], sc[0][3]);
            ph[2] = pack_bf16x2(sc[1][0], sc[1][1]); ph[3] = pack_bf16x2(sc[1][2], sc[1][3]);
            pl[0] = pack_bf16x2(sc[0][0] - bf16lo(ph[0]), sc[0][1] - bf16hi(ph[0]));
            pl[1] = pack_bf16x2(sc[0][2] - bf16lo(ph[1]), sc[0][3] - bf16hi(ph[1]));
            pl[2] = pack_bf16x2(sc[1][0] - bf16lo(ph[2]), sc[1][1] - bf16hi(ph[2]));
            pl[3] = pack_bf16x2(sc[1][2] - bf16lo(ph[3]), sc[1][3] - bf16hi(ph[3]));
#pragma unroll
            for (int dt = 0; dt < D / 16; ++dt) {
                uint32_t vb[4];
                ldmatrix_x4_trans(vb, vt + kv_off<D>(warp * 16 + (lane & 15), dt * 16 + (lane >> 4) * 8));
                float(&oa)[4] = o[2 * dt];
                float(&ob)[4] = o[2 * dt + 1];
                oa[0] *= al0; oa[1] *= al0; oa[2] *= al1; oa[3] *= al1;
                ob[0] *= al0; ob[1] *= al0; ob[2] *= al1; ob[3] *= al1;
                mma_bf16_16816(oa, ph, vb[0], vb[1]);
                mma_bf16_16816(oa, pl, vb[0], vb[1]);
                mma_bf16_16816(ob, ph, vb[2], vb[3]);
                mma_bf16_16816(ob, pl, vb[2], vb[3]);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[st]);

        const bool pair_done = (p == np - 1);
        if (pair_done || n == flat1 - 1) {
            // ---- emit: merge the 4 warps (each saw a different quarter of every page) ----
            const bool whole = from_start && pair_done;       // nobody else holds a piece of this pair
            l0 += __shfl_xor_sync(0xFFFFFFFFu, l0, 1); l0 += __shfl_xor_sync(0xFFFFFFFFu, l0, 2);
            l1 += __shfl_xor_sync(0xFFFFFFFFu, l1, 1); l1 += __shfl_xor_sync(0xFFFFFFFFu, l1, 2);
            csync();       // every warp is past its last read of the q tiles (the scratch overlays them)
            if (tq == 0) {
                red_m[warp][g] = m0; red_m[warp][g + 8] = m1;
                red_l[warp][g] = l0; red_l[warp][g + 8] = l1;
            }
#pragma unroll
            for (int nt = 0; nt < D / 8; ++nt) {
                if (g < n_rep) *reinterpret_cast<float2*>(red_o + ((size_t)warp * n_rep + g) * D + nt * 8 + tq * 2) = make_float2(o[nt][0], o[nt][1]);
                if (g + 8 < n_rep) *reinterpret_cast<float2*>(red_o + ((size_t)warp * n_rep + g + 8) * D + nt * 8 + tq * 2) = make_float2(o[nt][2], o[nt][3]);
            }
            csync();
            const int part = cta * 2 + (from_start ? 1 : 0);      // this CTA's partial slot for the pair
            if (tid < 16) {
                float ms = -INFINITY;
#pragma unroll
                for (int w = 0; w < NW; ++w) ms = fmaxf(ms, red_m[w][tid]);
                float den = 0.f;
#pragma unroll
                for (int w = 0; w < NW; ++w) {
                    const float wt = red_m[w][tid] == -INFINITY ? 0.f : expf(red_m[w][tid] - ms);
                    mrg_w[w][tid] = wt;
                    den = fmaf(wt, red_l[w][tid], den);
                }
                mrg_den[tid] = den;
                if (!whole && tid < n_rep) {
                    float* ml = k.sk_ml + ((size_t)part * n_rep + tid) * 2;
                    ml[0] = ms;
                    ml[1] = den;
                }
            }
            csync();
            for (int i = tid; i < n_rep * (D / 2); i += kSkConsumers) {
                const int hh = i / (D / 2), cc = (i % (D / 2)) * 2;
                float x0 = 0.f, x1 = 0.f;
#pragma unroll
                for (int w = 0; w < NW; ++w) {
                    const float2 v = *reinterpret_cast<const float2*>(red_o + ((size_t)w * n_rep + hh) * D + cc);
                    x0 = fmaf(mrg_w[w][hh], v.x, x0);
                    x1 = fmaf(mrg_w[w][hh], v.y, x1);
                }
                if (whole) {
                    const float den = mrg_den[hh];
                    store_out2(a, (size_t)s * a.nh * D + (size_t)(h * n_rep + hh) * D + cc, x0 / den, x1 / den);
                } else {
                    *reinterpret_cast<float2*>(k.sk_acc + ((size_t)part * n_rep + hh) * D + cc) = make_float2(x0, x1);
                }
            }
            if (!whole) {
                // ---- the pair straddles ranges: the last CTA to arrive merges the partials in CTA order ----
                __threadfence();
                csync();
                if (tid == 0) {
                    const long long ps = (long long)a.nkv * prefix[s] + (long long)h * np, pe = ps + np;
                    const int i0 = (int)(((ps + 1) * G - 1) / P), i1 = (int)((pe * G - 1) / P);      // CTAs holding the first / last page
                    const int ticket = atomicAdd(&a.counters[s * a.nkv + h], 1);
                    s_last = (ticket == i1 - i0);
                    s_i0 = i0;
                    s_i1 = i1;
                }
                csync();
                if (s_last) {
                    __threadfence();
                    const int i0 = s_i0, i1 = s_i1;
                    // partial of CTA j: slot 1 in the CTA where the pair starts (i0), slot 0 in the others
                    for (int hh = warp; hh < n_rep; hh += NW) {
                        float mstar = -INFINITY;
                        for (int j = i0 + lane; j <= i1; j += 32)
                            mstar = fmaxf(mstar, __ldcg(k.sk_ml + ((size_t)(j * 2 + (j == i0)) * n_rep + hh) * 2));
                        mstar = warp_max(mstar);
                        float den = 0.f;
                        for (int j = i0 + lane; j <= i1; j += 32) {
                            const float* ml = k.sk_ml + ((size_t)(j * 2 + (j == i0)) * n_rep + hh) * 2;
                            den = fmaf(expf(__ldcg(ml) - mstar), __ldcg(ml + 1), den);
                        }
                        den = warp_sum(den);
                        if (lane == 0) { mrg_star[hh] = mstar; mrg_den[hh] = den; }
                    }
                    csync();
                    for (int i = tid; i < n_rep * (D / 2); i += kSkConsumers) {
                        const int hh = i / (D / 2), cc = (i % (D / 2)) * 2;
                        float x0 = 0.f, x1 = 0.f;
                        for (int j = i0; j <= i1; ++j) {
                            const size_t pj = (size_t)(j * 2 + (j == i0)) * n_rep + hh;
                            const float w = expf(__ldcg(k.sk_ml + pj * 2) - mrg_star[hh]);
                            const float2 v = __ldcg(reinterpret_cast<const float2*>(k.sk_acc + pj * D + cc));
                            x0 = fmaf(w, v.x, x0);
                            x1 = fmaf(w, v.y, x1);
                        }
                        const float den = mrg_den[hh];
                        store_out2(a, (size_t)s * a.nh * D + (size_t)(h * n_rep + hh) * D + cc, x0 / den, x1 / den);
                    }
                    if (tid == 0) a.counters[s * a.nkv + h] = 0;
                }
            }
            open = false;
        }
        if (++p == np) {
            p = 0;
            if (++h == a.nkv) { h = 0; ++s; }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// prefill: grid (ceil(t / 64), nh, b), 128 threads; warp w owns query rows [16w, 16w+16) of the tile
// ---------------------------------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(kMmaAttnThreads) attn_prefill_kernel(const AttnArgs a) {
    constexpr int TILE = kKvPage * D;
    extern __shared__ __align__(128) uint8_t dsm[];
    uint16_t* qhi = reinterpret_cast<uint16_t*>(dsm);   // [64][D]
    uint16_t* qlo = qhi + kPrefillBM * D;
    uint16_t* kv = qlo + kPrefillBM * D;                // [2 stages][K tile | V tile]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, tq = lane & 3;
    // heaviest (latest) query tiles first: the causal range grows with the tile index
    const int qt = gridDim.x - 1 - blockIdx.x, head = blockIdx.y, seq = blockIdx.z;
    const int n_rep = a.nh / a.nkv, kvh = head / n_rep;
    pdl_launch_dependents();
    pdl_wait();
    const int i0 = qt * kPrefillBM;
    const int cslot = st_slot(a.state, seq);
    const int kv_base = a.state->kv_base[cslot];
    const int sw = a.sliding_window;
    const int* pt = a.page_table + (size_t)cslot * a.pt_stride;

    // key range of the whole tile
    const int ilast = min(i0 + kPrefillBM, a.t) - 1;
    const int len_tile = kv_base + ilast + 1;
    // the window thins out the NEW tokens only: candle concatenates zeros for the cached columns of its [t, t] mask, so every
    // cached key (< kv_base) stays visible and a call on a non-empty cache walks all pages
    const int start_tile = (sw > 0 && i0 - sw > 0 && kv_base == 0) ? i0 - sw : 0;
    const int p0 = start_tile / kKvPage, p1 = (len_tile + kKvPage - 1) / kKvPage;

    auto load = [&](int p, int st) {
        const size_t off = ((size_t)pt[p] * a.nkv + kvh) * (size_t)TILE;
        stage_kv_tile<D>(kv + st * 2 * TILE, kv + st * 2 * TILE + TILE, a.kpool + off, a.vpool + off, tid);
    };
    if (p0 < p1) load(p0, 0);
    for (int i = tid; i < kPrefillBM * (D / 4); i += kMmaAttnThreads) {
        const int r = i / (D / 4), c = (i % (D / 4)) * 4;
        float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i0 + r < a.t) q = *reinterpret_cast<const float4*>(a.q + (((size_t)seq * a.t + i0 + r) * a.nh + head) * D + c);
        const int off = swz<D>(r, c);
        store_hi_lo(qhi, qlo, off, q.x); store_hi_lo(qhi, qlo, off + 1, q.y);
        store_hi_lo(qhi, qlo, off + 2, q.z); store_hi_lo(qhi, qlo, off + 3, q.w);
    }

    // per-thread rows: g and g + 8 of the warp's 16 (rows past t are clamped: computed, never stored)
    const int ir0 = min(i0 + warp * 16 + g, a.t - 1), ir1 = min(i0 + warp * 16 + g + 8, a.t - 1);
    const int len0 = kv_base + ir0 + 1, len1 = kv_base + ir1 + 1;
    const int st0 = (sw > 0 && ir0 - sw > 0) ? kv_base + ir0 - sw : 0;
    const int st1 = (sw > 0 && ir1 - sw > 0) ? kv_base + ir1 - sw : 0;
    const int warp_len = kv_base + min(i0 + warp * 16 + 15, a.t - 1) + 1;    // keys >= this are masked for the whole warp

    float o[D / 8][4];
#pragma unroll
    for (int i = 0; i < D / 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

    for (int p = p0; p < p1; ++p) {
        const int st = (p - p0) & 1;
        if (p + 1 < p1) {
            load(p + 1, st ^ 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const uint16_t* kt = kv + st * 2 * TILE;
        const uint16_t* vt = kt + TILE;
        const int key0 = p * kKvPage;
        if (key0 < warp_len) {
            float s[8][4];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
            for (int ks = 0; ks < D / 16; ++ks) {
                uint32_t ah[4], al[4];
                ldmatrix_x4(ah, qhi + swz<D>(warp * 16 + (lane & 15), ks * 16 + (lane >> 4) * 8));
                ldmatrix_x4(al, qlo + swz<D>(warp * 16 + (lane & 15), ks * 16 + (lane >> 4) * 8));
#pragma unroll
                for (int n2 = 0; n2 < 4; ++n2) {
                    uint32_t kb[4];
                    ldmatrix_x4(kb, kt + swz<D>(n2 * 16 + (lane & 7) + ((lane >> 4) << 3), ks * 16 + ((lane >> 3) & 1) * 8));
                    mma_bf16_16816(s[2 * n2], ah, kb[0], kb[1]);
                    mma_bf16_16816(s[2 * n2], al, kb[0], kb[1]);
                    mma_bf16_16816(s[2 * n2 + 1], ah, kb[2], kb[3]);
                    mma_bf16_16816(s[2 * n2 + 1], al, kb[2], kb[3]);
                }
            }
            float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int key = key0 + nt * 8 + tq * 2 + (e & 1);
                    if (e < 2) {
                        s[nt][e] = ((key >= st0 || key < kv_base) && key < len0) ? s[nt][e] * a.qscale : -INFINITY;
                        mx0 = fmaxf(mx0, s[nt][e]);
                    } else {
                        s[nt][e] = ((key >= st1 || key < kv_base) && key < len1) ? s[nt][e] * a.qscale : -INFINITY;
                        mx1 = fmaxf(mx1, s[nt][e]);
                    }
                }
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xFFFFFFFFu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xFFFFFFFFu, mx0, 2));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xFFFFFFFFu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xFFFFFFFFu, mx1, 2));
            const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
            // a row may not have seen a visible key yet (window start inside a later page): keep exp() finite
            const float mu0 = mn0 == -INFINITY ? 0.f : mn0, mu1 = mn1 == -INFINITY ? 0.f : mn1;
            const float al0 = expf(m0 - mu0), al1 = expf(m1 - mu1);
            m0 = mn0; m1 = mn1;
            float ps0 = 0.f, ps1 = 0.f;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                s[nt][0] = expf(s[nt][0] - mu0); s[nt][1] = expf(s[nt][1] - mu0);
                s[nt][2] = expf(s[nt][2] - mu1); s[nt][3] = expf(s[nt][3] - mu1);
                ps0 += s[nt][0] + s[nt][1];
                ps1 += s[nt][2] + s[nt][3];
            }
            l0 = l0 * al0 + ps0;
            l1 = l1 * al1 + ps1;
#pragma unroll
            for (int nt = 0; nt < D / 8; ++nt) {
                o[nt][0] *= al0; o[nt][1] *= al0; o[nt][2] *= al1; o[nt][3] *= al1;
            }
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                uint32_t ph[4], pl[4];
                ph[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]); ph[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
                ph[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]); ph[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
                pl[0] = pack_bf16x2(s[2 * kk][0] - bf16lo(ph[0]), s[2 * kk][1] - bf16hi(ph[0]));
                pl[1] = pack_bf16x2(s[2 * kk][2] - bf16lo(ph[1]), s[2 * kk][3] - bf16hi(ph[1]));
                pl[2] = pack_bf16x2(s[2 * kk + 1][0] - bf16lo(ph[2]), s[2 * kk + 1][1] - bf16hi(ph[2]));
                pl[3] = pack_bf16x2(s[2 * kk + 1][2] - bf16lo(ph[3]), s[2 * kk + 1][3] - bf16hi(ph[3]));
#pragma unroll
                for (int dt = 0; dt < D / 16; ++dt) {
                    uint32_t vb[4];
                    ldmatrix_x4_trans(vb, vt + swz<D>(kk * 16 + (lane & 15), dt * 16 + (lane >> 4) * 8));
                    mma_bf16_16816(o[2 * dt], ph, vb[0], vb[1]);
                    mma_bf16_16816(o[2 * dt], pl, vb[0], vb[1]);
                    mma_bf16_16816(o[2 * dt + 1], ph, vb[2], vb[3]);
                    mma_bf16_16816(o[2 * dt + 1], pl, vb[2], vb[3]);
                }
            }
        }
        __syncthreads();
    }

    l0 += __shfl_xor_sync(0xFFFFFFFFu, l0, 1); l0 += __shfl_xor_sync(0xFFFFFFFFu, l0, 2);
    l1 += __shfl_xor_sync(0xFFFFFFFFu, l1, 1); l1 += __shfl_xor_sync(0xFFFFFFFFu, l1, 2);
    const float inv0 = 1.f / l0, inv1 = 1.f / l1;
    const int r0 = i0 + warp * 16 + g, r1 = r0 + 8;
#pragma unroll
    for (int nt = 0; nt < D / 8; ++nt) {
        const int c = nt * 8 + tq * 2;
        if (r0 < a.t) store_out2(a, (((size_t)seq * a.t + r0) * a.nh + head) * D + c, o[nt][0] * inv0, o[nt][1] * inv0);
        if (r1 < a.t) store_out2(a, (((size_t)seq * a.t + r1) * a.nh + head) * D + c, o[nt][2] * inv1, o[nt][3] * inv1);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// prefill on the 5th-gen tensor cores: grid (ceil(t / 128), nh, b), 192 threads, head_dim 64 / 128, calls that start on empty caches
// ---------------------------------------------------------------------------------------------------------------------
// One CTA owns 128 query rows of one head (M = 128 of tcgen05.mma) and walks the causal range of 64-key pages:
//   warp 0      producer: K page (the pool's own rows, 2-D TMA, 128-byte swizzle) + the page of V^T that dense_qkv_epi_kernel wrote
//               for this call ([d][64 keys]: K-major, so O += P.V is the same operand form as every GEMM of the library);
//   warp 1      allocates TMEM (S double-buffered 2 x 64 columns, O d columns), one thread issues S = Q.K^T (q = hi + lo: two
//               accumulating MMA groups against the same K tile) and, one tile behind, O += P.V (P = hi + lo likewise);
//   warps 2-9   softmax: thread == query row and half of a page's keys (tcgen05.ld 32x32b), scale / causal + window mask / running max and sum in the
//               exp2 domain, P written hi | lo into shared memory in the swizzled operand layout; when a row's max moved, the warp
//               rescales its 32 TMEM lanes of O in place (tcgen05.ld / st) after the previous P.V has completed.
// Same arithmetic contract as attn_prefill_kernel (f32 scores and probabilities carried as hi + lo bf16 pairs, f32 accumulation).
constexpr int kTcQ = 128;
constexpr int kTcThreads = 352;

struct TcPrefillArgs {
    AttnArgs a;
    int layer_row0;      // row of this layer's page 0 / kv head 0 in the pool-wide K tensor map
    int vt_pages;        // pages per (sequence, kv head) in the V^T scratch
    float tau;           // a row's reference max moves only when the tile's max exceeds it by more than this (exp2 domain)
};

// K and V^T pages travel through separate rings: a K page is free again as soon as its S = Q.K^T has completed, a V^T page only after
// the O += P.V a whole softmax later, so with one shared ring the K loads could run only ~1.5 tiles ahead and the MMA warp waited for
// them (ncu: the softmax warps stalled 25 % of their time on S).  Three K stages + two (d = 128) or three V^T stages sit next to Q
// (hi | lo) and the two P buffers.
constexpr int kTcKStages = 3;
constexpr int kTcSBufs = 4;          // S accumulators in TMEM (64 columns each): S = Q.K^T runs up to four pages ahead of the softmax
__host__ __device__ constexpr int attn_prefill_tc_vstages(int d) { return d == 128 ? 2 : 3; }
inline size_t attn_prefill_tc_smem_bytes(int d) {
    return (size_t)2 * (d / 64) * 16384 + 65536 + (size_t)(kTcKStages + attn_prefill_tc_vstages(d)) * d * 128 + 1024;
}

__device__ __forceinline__ float ex2_approx(float x) {      // one MUFU op; -inf -> 0
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

template <int D>
__global__ void __launch_bounds__(kTcThreads, 1) attn_prefill_tc_kernel(const __grid_constant__ CUtensorMap tmk, const __grid_constant__ CUtensorMap tmvt,
                                                                        const TcPrefillArgs k) {
    static_assert(D == 64 || D == 128, "head_dim 64 or 128");
    const AttnArgs& a = k.a;
    constexpr int HALF = D / 64;
    constexpr uint32_t kQBytes = HALF * 16384;              // one of q_hi / q_lo: HALF k-blocks of [128 rows][128 B]
    constexpr uint32_t kPOff = 2 * kQBytes;                 // P: [2 buffers][hi | lo][128 rows][128 B]
    constexpr int NK = kTcKStages, NV = attn_prefill_tc_vstages(D);
    constexpr uint32_t kTile = D * 128;                    // a K page (HALF boxes of [64 keys][128 B]) or a V^T page ([D][128 B])
    constexpr uint32_t kKOff = kPOff + 65536, kVOff = kKOff + NK * kTile;
    extern __shared__ __align__(1024) uint8_t tcsm_raw[];
    uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(tcsm_raw) + 1023) & ~(uintptr_t)1023);
    __shared__ __align__(8) uint64_t k_full[NK], k_empty[NK], v_full[NV], v_empty[NV], s_full[kTcSBufs], s_free[kTcSBufs], p_ready[2], p_free[2], o_done, q_ready;
    __shared__ uint32_t s_tmem;
    __shared__ float xmax[2][2][kTcQ];      // [page parity][column half][row]: page maxima of the two halves of a row
    __shared__ float xsum[2][kTcQ];         // their row sums (epilogue)

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int qt = gridDim.x - 1 - blockIdx.x, head = blockIdx.y, seq = blockIdx.z;      // heaviest (latest) query tiles first
    const int n_rep = a.nh / a.nkv, kvh = head / n_rep;
    const int q0 = qt * kTcQ, sw = a.sliding_window;
    const int kend = min(a.t, q0 + kTcQ);                            // keys [0, kend) can be visible to this tile
    const int kt0 = (sw > 0 && q0 - sw > 0) ? (q0 - sw) / kKvPage : 0;
    const int nkt = (kend + kKvPage - 1) / kKvPage - kt0;

    if (tid == 0) {
        for (int i = 0; i < NK; ++i) { mbar_init(&k_full[i], 1); mbar_init(&k_empty[i], 1); }
        for (int i = 0; i < NV; ++i) { mbar_init(&v_full[i], 1); mbar_init(&v_empty[i], 1); }
        for (int i = 0; i < kTcSBufs; ++i) { mbar_init(&s_full[i], 1); mbar_init(&s_free[i], 8); }
        for (int i = 0; i < 2; ++i) { mbar_init(&p_ready[i], 8); mbar_init(&p_free[i], 1); }
        mbar_init(&o_done, 1);
        mbar_init(&q_ready, 8);
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc(&s_tmem, 512);
    pdl_launch_dependents();
    pdl_wait();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    const uint32_t sm_s = smem_u32(sm);
    const uint32_t tO = tmem + kTcSBufs * 64;

    if (warp == 0) {
        if (lane == 0) {      // K pages: the pool's own rows
            const int cslot = st_slot(a.state, seq);
            const int* pt = a.page_table + (size_t)cslot * a.pt_stride;
            for (int j = 0; j < nkt; ++j) {
                const int st = j % NK;
                const int row = k.layer_row0 + (pt[kt0 + j] * a.nkv + kvh) * kKvPage;
                mbar_wait(&k_empty[st], ((j / NK) & 1) ^ 1);
                mbar_expect_tx(&k_full[st], kTile);
#pragma unroll
                for (int hf = 0; hf < HALF; ++hf) tma_load_2d(sm + kKOff + st * kTile + hf * 8192, &tmk, hf * 64, row, &k_full[st]);
            }
        }
    } else if (warp == 10) {
        if (lane == 0) {      // V^T pages of this call (written by dense_qkv_epi_kernel)
            for (int j = 0; j < nkt; ++j) {
                const int st = j % NV;
                mbar_wait(&v_empty[st], ((j / NV) & 1) ^ 1);
                mbar_expect_tx(&v_full[st], kTile);
                tma_load_2d(sm + kVOff + st * kTile, &tmvt, 0, ((seq * a.nkv + kvh) * k.vt_pages + kt0 + j) * D, &v_full[st]);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc_s = umma_idesc_bf16(128, 64), idesc_o = umma_idesc_bf16(128, D);
            // S = Q.K^T is issued as far ahead as K pages and free S buffers allow, O += P.V as soon as a page's probabilities are
            // in shared memory: neither waits for the other (in lock step the issue -> commit -> softmax -> issue round trip of a
            // page was the critical path: ~3100 clocks per page against ~700 of tensor work).
            int qi = 0, pi = 0;
            mbar_wait(&q_ready, 0);
            tc_fence_after();
            while (pi < nkt) {
                if (pi < qi && mbar_test(&p_ready[pi & 1], (pi >> 1) & 1) && mbar_test(&v_full[pi % NV], (pi / NV) & 1)) {
                    const int b = pi & 1;
                    tc_fence_after();
                    const uint64_t vdesc = umma_smem_desc_sw128(sm + kVOff + (pi % NV) * kTile);
#pragma unroll
                    for (int hl = 0; hl < 2; ++hl) {
                        const uint64_t pdesc = umma_smem_desc_sw128(sm + kPOff + (b * 2 + hl) * 16384);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) umma_bf16(tO, pdesc + 2 * kk, vdesc + 2 * kk, idesc_o, (pi > 0 || hl > 0 || kk > 0) ? 1u : 0u);
                    }
                    umma_commit(&v_empty[pi % NV]);
                    umma_commit(&p_free[b]);
                    umma_commit(&o_done);
                    ++pi;
                } else if (qi < nkt && mbar_test(&k_full[qi % NK], (qi / NK) & 1) &&
                           mbar_test(&s_free[qi % kTcSBufs], ((qi / kTcSBufs) & 1) ^ 1)) {
                    const int st = qi % NK, sb = qi % kTcSBufs;
                    tc_fence_after();
                    const uint32_t tS = tmem + sb * 64;
#pragma unroll
                    for (int hl = 0; hl < 2; ++hl)
#pragma unroll
                        for (int hf = 0; hf < HALF; ++hf) {
                            const uint64_t qdesc = umma_smem_desc_sw128(sm + hl * kQBytes + hf * 16384);
                            const uint64_t kdesc = umma_smem_desc_sw128(sm + kKOff + st * kTile + hf * 8192);
#pragma unroll
                            for (int kk = 0; kk < 4; ++kk) umma_bf16(tS, qdesc + 2 * kk, kdesc + 2 * kk, idesc_s, (hl > 0 || hf > 0 || kk > 0) ? 1u : 0u);
                        }
                    umma_commit(&s_full[sb]);
                    umma_commit(&k_empty[st]);
                    ++qi;
                }
            }
        }
    } else if (warp < 10) {
        // softmax: warps 2-5 own key columns 0-31 of every page, warps 6-9 columns 32-63 (same TMEM lanes: warp & 3 selects the
        // quarter).  One warp per scheduler could not hide its own issue latencies (ncu: ~0.4 instructions per clock, the softmax
        // warps were the critical path at ~3400 clocks per page); two per scheduler overlap one's MUFU / TMEM waits with the other's
        // arithmetic.  The halves of a row exchange their page maxima through shared memory (one 256-thread named barrier per page).
        const int grp = (warp - 2) >> 2, quarter = warp & 3, r = quarter * 32 + lane;
        const int irow = min(q0 + r, a.t - 1);               // rows past t are clamped: computed, never stored
        const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
        auto gsync = [] { asm volatile("bar.sync 2, 256;" ::: "memory"); };
        // ---- q row -> hi / lo bf16, swizzled operand layout: 16-byte chunk c of row r at chunk (c & 7) ^ (r & 7) of k-block c >> 3 ----
        {
            const float* qsrc = a.q + (((size_t)seq * a.t + irow) * a.nh + head) * D;
#pragma unroll
            for (int cc = 0; cc < D / 16; ++cc) {
                const int c = grp * (D / 16) + cc;
                const float4 x = *reinterpret_cast<const float4*>(qsrc + c * 8), y = *reinterpret_cast<const float4*>(qsrc + c * 8 + 4);
                uint4 h, l;
                h.x = pack_bf16x2(x.x, x.y); h.y = pack_bf16x2(x.z, x.w); h.z = pack_bf16x2(y.x, y.y); h.w = pack_bf16x2(y.z, y.w);
                l.x = pack_bf16x2(x.x - bf16lo(h.x), x.y - bf16hi(h.x)); l.y = pack_bf16x2(x.z - bf16lo(h.y), x.w - bf16hi(h.y));
                l.z = pack_bf16x2(y.x - bf16lo(h.z), y.y - bf16hi(h.z)); l.w = pack_bf16x2(y.z - bf16lo(h.w), y.w - bf16hi(h.w));
                const uint32_t off = (uint32_t)(c >> 3) * 16384u + (uint32_t)r * 128u + (uint32_t)(((c & 7) ^ (r & 7)) << 4);
                sts128(sm_s + off, h);
                sts128(sm_s + kQBytes + off, l);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&q_ready);
        }
        const float c2 = a.qscale * 1.4426950408889634f;      // scores are carried in the exp2 domain
        const int lo_key = (sw > 0 && irow - sw > 0) ? irow - sw : 0;
        float m = -INFINITY, l = 0.f;                         // l: this thread's half of the row sum
        for (int j = 0; j < nkt; ++j) {
            const int b = j & 1, sb = j % kTcSBufs, key0 = (kt0 + j) * kKvPage + grp * 32;
            mbar_wait(&s_full[sb], (j / kTcSBufs) & 1);
            tc_fence_after();
            float sc[32];
            {
                uint32_t r0[32];
                tmem_ld32(tmem + lane_addr + sb * 64 + grp * 32, r0);
#pragma unroll
                for (int e = 0; e < 32; ++e) sc[e] = __uint_as_float(r0[e]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&s_free[sb]);
            float mx = -INFINITY;
            if (key0 + 31 <= q0 && (sw <= 0 || key0 + sw >= q0 + kTcQ - 1)) {      // every key of this half page is visible to every row
#pragma unroll
                for (int e = 0; e < 32; ++e) mx = fmaxf(mx, sc[e]);
            } else {
#pragma unroll
                for (int e = 0; e < 32; ++e) {
                    const int key = key0 + e;
                    sc[e] = (key <= irow && key >= lo_key) ? sc[e] : -INFINITY;
                    mx = fmaxf(mx, sc[e]);
                }
            }
            xmax[b][grp][r] = mx;
            gsync();
            mx = fmaxf(mx, xmax[b][grp ^ 1][r]) * c2;
            // The exponent offset m follows the running max lazily: it moves only when a page's max exceeds it by more than tau, so
            // probabilities reach at most 2^tau (the final O / l does not depend on the offset) and the O accumulator in TMEM needs
            // a rescale only on such a jump -- rare after the first pages -- instead of in every page.  Both halves of a row see
            // the same maxima, so they take the same decisions.
            const bool bump = mx > m + k.tau;              // m = -inf until the row has seen a visible key
            const float mn = bump ? mx : m;
            const float mu = mn == -INFINITY ? 0.f : mn;
            const float alpha = bump ? ex2_approx(m - mu) : 1.f;
            m = mn;
            float ps = 0.f;
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                sc[e] = ex2_approx(fmaf(sc[e], c2, -mu));
                ps += sc[e];
            }
            l = l * alpha + ps;
            if (j > 0 && __any_sync(0xFFFFFFFFu, bump)) {
                // O may be touched only when the previous P.V has completed; the warp rescales its half of the columns of its 32 lanes
                mbar_wait(&o_done, (j - 1) & 1);
                tc_fence_after();
#pragma unroll 1
                for (int c4 = 0; c4 < D / 64; ++c4) {
                    uint32_t o[32];
                    tmem_ld32(tO + lane_addr + grp * (D / 2) + c4 * 32, o);
#pragma unroll
                    for (int e = 0; e < 32; ++e) o[e] = __float_as_uint(__uint_as_float(o[e]) * alpha);
                    tmem_st32(tO + lane_addr + grp * (D / 2) + c4 * 32, o);
                }
            }
            mbar_wait(&p_free[b], ((j >> 1) & 1) ^ 1);       // the P.V two pages back has finished reading this P buffer
            const uint32_t ph = sm_s + kPOff + (b * 2) * 16384 + (uint32_t)r * 128u;
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
                uint4 h, lo4;
                h.x = pack_bf16x2(sc[8 * cc], sc[8 * cc + 1]); h.y = pack_bf16x2(sc[8 * cc + 2], sc[8 * cc + 3]);
                h.z = pack_bf16x2(sc[8 * cc + 4], sc[8 * cc + 5]); h.w = pack_bf16x2(sc[8 * cc + 6], sc[8 * cc + 7]);
                lo4.x = pack_bf16x2(sc[8 * cc] - bf16lo(h.x), sc[8 * cc + 1] - bf16hi(h.x));
                lo4.y = pack_bf16x2(sc[8 * cc + 2] - bf16lo(h.y), sc[8 * cc + 3] - bf16hi(h.y));
                lo4.z = pack_bf16x2(sc[8 * cc + 4] - bf16lo(h.z), sc[8 * cc + 5] - bf16hi(h.z));
                lo4.w = pack_bf16x2(sc[8 * cc + 6] - bf16lo(h.w), sc[8 * cc + 7] - bf16hi(h.w));
                const uint32_t off = (uint32_t)(((grp * 4 + cc) ^ (r & 7)) << 4);
                sts128(ph + off, h);
                sts128(ph + 16384 + off, lo4);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&p_ready[b]);
        }
        // ---- epilogue: O / l -> hi | lo bf16 operands of the o_proj GEMM; each half writes its half of the head's columns ----
        xsum[grp][r] = l;
        gsync();
        const float inv = 1.f / (l + xsum[grp ^ 1][r]);
        mbar_wait(&o_done, (nkt - 1) & 1);
        tc_fence_after();
        const size_t obase = (((size_t)seq * a.t + irow) * a.nh + head) * D + grp * (D / 2);
#pragma unroll 1
        for (int c4 = 0; c4 < D / 64; ++c4) {
            uint32_t o[32];
            tmem_ld32(tO + lane_addr + grp * (D / 2) + c4 * 32, o);
            if (q0 + r < a.t) {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    float v[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) v[e] = __uint_as_float(o[8 * c + e]) * inv;
                    uint4 h, lo4;
                    h.x = pack_bf16x2(v[0], v[1]); h.y = pack_bf16x2(v[2], v[3]); h.z = pack_bf16x2(v[4], v[5]); h.w = pack_bf16x2(v[6], v[7]);
                    lo4.x = pack_bf16x2(v[0] - bf16lo(h.x), v[1] - bf16hi(h.x)); lo4.y = pack_bf16x2(v[2] - bf16lo(h.y), v[3] - bf16hi(h.y));
                    lo4.z = pack_bf16x2(v[4] - bf16lo(h.z), v[5] - bf16hi(h.z)); lo4.w = pack_bf16x2(v[6] - bf16lo(h.w), v[7] - bf16hi(h.w));
                    *reinterpret_cast<uint4*>(a.out_hi + obase + c4 * 32 + c * 8) = h;
                    *reinterpret_cast<uint4*>(a.out_lo + obase + c4 * 32 + c * 8) = lo4;
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
}

}  // namespace fl
