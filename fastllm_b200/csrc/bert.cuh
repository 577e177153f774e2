// BERT / MiniLM encoder glue kernels around the tcgen05 GEMM (gemm_tc.cuh), sm_100a.
// Semantics follow the reference's hand-written encoder line by line (src/models/embeddings.rs):
//   embed_ln_kernel   : word + position embedding gather, add, LayerNorm eps = 1e-12 literal, NO token-type (:370-378, :315-318)
//   bert_attn_kernel  : per (sentence, head): softmax(Q K^T / sqrt(d)) V, NO attention / padding mask (:130-166); sentences of
//                       more than 128 tokens go through bert_attn_long_kernel (key tiles + online softmax)
//   layernorm_kernel  : post-LN over (x + f(x)), eps = config.layer_norm_eps (:185-190, :236-241); one-pass var = E[x^2]-mean^2
//   pool_l2_kernel    : masked mean pooling (divisor = mask_count * hidden [sic], :346-368) + L2 normalise (:341-344)
// Token rows are packed: sentence s is rows [starts[s], starts[s + 1]) of every [T, .] activation, with no padding between
// sentences.  A uniform [b, t] batch is the case starts[s] = s * t.  The attention kernels take a work list of BertItem.
// The sentence tables (positions, starts, items) are written by the host upload that precedes the encoder's first kernel and by
// no kernel, so every kernel reads them BEFORE pdl_wait: their load latency overlaps the previous kernel's tail.
// Shapes: head_dim 32 or 64 (the attention kernels' template parameter), hidden a multiple of 64 and <= 1024.
#pragma once
#include "common.cuh"
#include "mma.cuh"

namespace fl {

// One attention work item: the sentence's first token row and length, and the first query row q0 of the item within the sentence
// (a multiple of 128; always 0 for bert_attn_kernel, whose sentences are one tile).
struct __align__(16) BertItem {
    int row0, len, q0, pad;
};

// One warp per token row, PER values per lane: H <= 32 * PER (PER = 16 up to hidden 512, 32 up to 1024).  out bf16 [T, H].
template <int PER>
static __global__ void embed_ln_kernel(const uint16_t* __restrict__ wemb, const uint16_t* __restrict__ pemb, const float* __restrict__ lnw,
                                const float* __restrict__ lnb, const uint32_t* __restrict__ ids, const int* __restrict__ positions, int T,
                                int H, int vocab, int maxpos, float eps, uint16_t* __restrict__ out) {
    pdl_launch_dependents();      // programmatic dependent launch: the next kernel may start its prologue now ...
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    int pos = row < T ? positions[row] : 0;  // position ids 0..n-1 of each sentence (embeddings.rs:416); a sentence table
    pdl_wait();                   // ... and nothing below runs before the previous kernel has completed
    if (row >= T) return;
    uint32_t id = ids[row];
    if (id >= (uint32_t)vocab) id = vocab - 1;
    if (pos >= maxpos) pos = maxpos - 1;
    const uint16_t* w = wemb + (size_t)id * H;
    const uint16_t* p = pemb + (size_t)pos * H;
    float v[PER];
    float s = 0.f, s2 = 0.f;
    const int per = (H + 31) / 32;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        const int c = lane + 32 * j;
        v[j] = 0.f;
        if (j < per && c < H) {
            v[j] = __uint_as_float((uint32_t)w[c] << 16) + __uint_as_float((uint32_t)p[c] << 16);
            s += v[j];
            s2 = fmaf(v[j], v[j], s2);
        }
    }
    s = warp_sum(s);
    s2 = warp_sum(s2);
    const float mean = s / (float)H;
    const float inv = 1.f / sqrtf(s2 / (float)H - mean * mean + eps);
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        const int c = lane + 32 * j;
        if (j < per && c < H) out[(size_t)row * H + c] = f32_to_bf16_rne((v[j] - mean) * inv * lnw[c] + lnb[c]);
    }
}

// LayerNorm over f32 rows [T, H] -> bf16 [T, H]; one warp per row, V4 float4 per lane, 128-bit loads / 64-bit stores
// (H % 4 == 0, H <= 128 * V4: V4 = 4 up to hidden 512, 8 up to 1024).
template <int V4>
static __global__ void layernorm_kernel(const float* __restrict__ x, const float* __restrict__ lnw, const float* __restrict__ lnb, int T, int H,
                                 float eps, uint16_t* __restrict__ out) {
    pdl_launch_dependents();      // programmatic dependent launch: the next kernel may start its prologue now ...
    pdl_wait();                   // ... and nothing below runs before the previous kernel has completed
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= T) return;
    const float4* xr = reinterpret_cast<const float4*>(x + (size_t)row * H);
    const int H4 = H >> 2;
    float4 v[V4];
    float s = 0.f, s2 = 0.f;
#pragma unroll
    for (int j = 0; j < V4; ++j) {
        const int c = lane + 32 * j;
        v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c < H4) {
            v[j] = xr[c];
            s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
            s2 = fmaf(v[j].x, v[j].x, s2); s2 = fmaf(v[j].y, v[j].y, s2); s2 = fmaf(v[j].z, v[j].z, s2); s2 = fmaf(v[j].w, v[j].w, s2);
        }
    }
    s = warp_sum(s);
    s2 = warp_sum(s2);
    const float mean = s / (float)H;
    const float inv = 1.f / sqrtf(s2 / (float)H - mean * mean + eps);
    uint2* orow = reinterpret_cast<uint2*>(out + (size_t)row * H);
#pragma unroll
    for (int j = 0; j < V4; ++j) {
        const int c = lane + 32 * j;
        if (c < H4) {
            const float4 w4 = reinterpret_cast<const float4*>(lnw)[c], b4 = reinterpret_cast<const float4*>(lnb)[c];
            orow[c] = make_uint2(pack_bf16x2((v[j].x - mean) * inv * w4.x + b4.x, (v[j].y - mean) * inv * w4.y + b4.y),
                                 pack_bf16x2((v[j].z - mean) * inv * w4.z + b4.z, (v[j].w - mean) * inv * w4.w + b4.w));
        }
    }
}

// ---- fused attention (head_dim D = 32 or 64) on mma.sync m16n8k16 bf16 ----------------------------------------------------
constexpr int kBertS = 128;      // query / key rows per tile (a sentence of <= 128 tokens is ONE tile: bert_attn_kernel)

// Q | K | V staging of one attention CTA: 3 x 128 rows of D + 8 bf16.  The 8-element pad makes the row 80 bytes (D = 32) or 144
// bytes (D = 64), so the 8 rows one ldmatrix phase reads fall in distinct bank groups.  30 720 bytes at D = 32 are three static
// arrays; 55 296 bytes at D = 64 exceed the 48 KB static limit and are dynamic (launched with bert_attn_dyn_smem(64) bytes).
template <int D>
constexpr int bert_attn_ld() { return D + 8; }
constexpr size_t bert_attn_dyn_smem(int d) { return d == 32 ? 0 : (size_t)3 * kBertS * (d + 8) * 2; }

struct BertAttnStage {
    uint16_t *q, *k, *v;
};
template <int D>
static __device__ __forceinline__ BertAttnStage bert_attn_stage() {
    static_assert(D == 32 || D == 64, "BERT attention is built for head_dim 32 and 64");
    constexpr int n = kBertS * bert_attn_ld<D>();
    if constexpr (D == 32) {
        __shared__ __align__(16) uint16_t sq[n], sk[n], sv[n];
        return {sq, sk, sv};
    } else {
        extern __shared__ __align__(16) uint16_t bert_attn_dyn[];
        return {bert_attn_dyn, bert_attn_dyn + n, bert_attn_dyn + 2 * n};
    }
}

// grid (heads x items), head fastest; 128 threads: warp w owns query rows [32w, 32w+32).  qkv bf16 [T, 3H] (q | k | v), ctx bf16 [T, H].
template <int D>
static __global__ void __launch_bounds__(128) bert_attn_kernel(const uint16_t* __restrict__ qkv, const BertItem* __restrict__ items, int nh,
                                                               int H, float scale, uint16_t* __restrict__ ctx) {
    constexpr int LD = bert_attn_ld<D>(), KS = D / 16, DT = D / 8;      // row pitch; k16 steps of Q K^T; 8-column output tiles of P V
    pdl_launch_dependents();      // programmatic dependent launch: the next kernel may start its prologue now ...
    const BertItem it = items[blockIdx.x / nh];      // a sentence table
    pdl_wait();                   // ... and nothing below runs before the previous kernel has completed
    const auto [sq, sk, sv] = bert_attn_stage<D>();
    const int head = blockIdx.x % nh, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t row0 = (size_t)it.row0;
    const int t = it.len;
    const int ld = 3 * H;
    // stage Q, K, V of this (sentence, head): 128 rows x D bf16 each, in 16-byte chunks; rows >= t are zero
    for (int i = tid; i < kBertS * DT; i += 128) {
        const int r = i / DT, c = (i % DT) * 8;
        uint4 q = make_uint4(0, 0, 0, 0), k = q, v = q;
        if (r < t) {
            const uint16_t* src = qkv + (row0 + r) * ld + head * D + c;
            q = *reinterpret_cast<const uint4*>(src);
            k = *reinterpret_cast<const uint4*>(src + H);
            v = *reinterpret_cast<const uint4*>(src + 2 * H);
        }
        *reinterpret_cast<uint4*>(sq + r * LD + c) = q;
        *reinterpret_cast<uint4*>(sk + r * LD + c) = k;
        *reinterpret_cast<uint4*>(sv + r * LD + c) = v;
    }
    __syncthreads();
    const int g = lane >> 2, tq = lane & 3;
#pragma unroll 1
    for (int mt = 0; mt < 2; ++mt) {
        const int m0 = warp * 32 + mt * 16;
        if (m0 >= t) break;
        // A fragments of Q: 16 rows x D (KS k16 steps)
        uint32_t qa[KS][4];
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) ldmatrix_x4(qa[ks], sq + (m0 + (lane & 15)) * LD + ks * 16 + (lane >> 4) * 8);
        // S = Q K^T : 16 key tiles of 8
        float s[16][4];
#pragma unroll
        for (int nt = 0; nt < 16; ++nt) {
            s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                uint32_t kb[2];
                ldmatrix_x2(kb, sk + (nt * 8 + (lane & 7)) * LD + ks * 16 + ((lane >> 3) & 1) * 8);
                mma_bf16_16816(s[nt], qa[ks], kb);
            }
        }
        // scores / sqrt(d) (after the matmul, embeddings.rs:155-159), softmax over keys < t; rows g and g+8
        // (the reference divides by sqrt(d); sqrt(32) is not a power of two, so x * (1/sqrt(d)) differs by <= 1 ulp; at d = 64 it is exact)
        const float inv_scale = 1.f / scale;
        float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
        for (int nt = 0; nt < 16; ++nt) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int key = nt * 8 + tq * 2 + (e & 1);
                s[nt][e] = key < t ? s[nt][e] * inv_scale : -INFINITY;
            }
            mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
            mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xFFFFFFFFu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xFFFFFFFFu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xFFFFFFFFu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xFFFFFFFFu, mx1, 2));
        float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
        for (int nt = 0; nt < 16; ++nt) {
            s[nt][0] = __expf(s[nt][0] - mx0); s[nt][1] = __expf(s[nt][1] - mx0);
            s[nt][2] = __expf(s[nt][2] - mx1); s[nt][3] = __expf(s[nt][3] - mx1);
            sum0 += s[nt][0] + s[nt][1];
            sum1 += s[nt][2] + s[nt][3];
        }
        sum0 += __shfl_xor_sync(0xFFFFFFFFu, sum0, 1); sum0 += __shfl_xor_sync(0xFFFFFFFFu, sum0, 2);
        sum1 += __shfl_xor_sync(0xFFFFFFFFu, sum1, 1); sum1 += __shfl_xor_sync(0xFFFFFFFFu, sum1, 2);
        // O = P V : the S accumulator layout of key tiles (2j, 2j+1) is exactly the A fragment of k16 step j
        float o[DT][4];
#pragma unroll
        for (int dt = 0; dt < DT; ++dt) o[dt][0] = o[dt][1] = o[dt][2] = o[dt][3] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {
            uint32_t pa[4];
            pa[0] = pack_bf16(s[2 * ks][0], s[2 * ks][1]);
            pa[1] = pack_bf16(s[2 * ks][2], s[2 * ks][3]);
            pa[2] = pack_bf16(s[2 * ks + 1][0], s[2 * ks + 1][1]);
            pa[3] = pack_bf16(s[2 * ks + 1][2], s[2 * ks + 1][3]);
#pragma unroll
            for (int dt = 0; dt < DT; ++dt) {
                uint32_t vb[2];
                ldmatrix_x2_trans(vb, sv + (ks * 16 + (lane & 15)) * LD + dt * 8);
                mma_bf16_16816(o[dt], pa, vb);
            }
        }
        const float i0 = 1.f / sum0, i1 = 1.f / sum1;
        const int r0 = m0 + g, r1 = m0 + g + 8;
#pragma unroll
        for (int dt = 0; dt < DT; ++dt) {
            const int c = head * D + dt * 8 + tq * 2;
            if (r0 < t) *reinterpret_cast<uint32_t*>(ctx + (row0 + r0) * H + c) = pack_bf16(o[dt][0] * i0, o[dt][1] * i0);
            if (r1 < t) *reinterpret_cast<uint32_t*>(ctx + (row0 + r1) * H + c) = pack_bf16(o[dt][2] * i1, o[dt][3] * i1);
        }
    }
}

// Sentences longer than one 128-row tile (up to max_position_embeddings, 512 for MiniLM: the reference enforces no limit,
// embeddings.rs:285-286): the same attention, FlashAttention-style.  grid (heads x (sentence, query tile) items), 128 threads;
// a CTA stages its 128 query rows once and walks the sentence's keys in 128-row tiles with an online softmax (running max / sum per
// row, accumulator rescaled when the max moves) -- algebraically the reference's max-subtract / exp / sum / div over all keys.
template <int D>
static __global__ void __launch_bounds__(128) bert_attn_long_kernel(const uint16_t* __restrict__ qkv, const BertItem* __restrict__ items,
                                                                    int nh, int H, float scale, uint16_t* __restrict__ ctx) {
    constexpr int LD = bert_attn_ld<D>(), KS = D / 16, DT = D / 8;
    pdl_launch_dependents();      // programmatic dependent launch: the next kernel may start its prologue now ...
    const BertItem it = items[blockIdx.x / nh];      // a sentence table
    pdl_wait();                   // ... and nothing below runs before the previous kernel has completed
    const auto [sq, sk, sv] = bert_attn_stage<D>();
    const int head = blockIdx.x % nh, q0 = it.q0, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t row0 = (size_t)it.row0;
    const int t = it.len;
    const int ld = 3 * H;
    for (int i = tid; i < kBertS * DT; i += 128) {
        const int r = i / DT, c = (i % DT) * 8;
        uint4 q = make_uint4(0, 0, 0, 0);
        if (q0 + r < t) q = *reinterpret_cast<const uint4*>(qkv + (row0 + q0 + r) * ld + head * D + c);
        *reinterpret_cast<uint4*>(sq + r * LD + c) = q;
    }
    __syncthreads();
    const int g = lane >> 2, tq = lane & 3;
    const float inv_scale = 1.f / scale;
    uint32_t qa[2][KS][4];
    float o[2][DT][4], mrun[2][2], lrun[2][2];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) ldmatrix_x4(qa[mt][ks], sq + (warp * 32 + mt * 16 + (lane & 15)) * LD + ks * 16 + (lane >> 4) * 8);
#pragma unroll
        for (int dt = 0; dt < DT; ++dt) o[mt][dt][0] = o[mt][dt][1] = o[mt][dt][2] = o[mt][dt][3] = 0.f;
        mrun[mt][0] = mrun[mt][1] = -INFINITY;
        lrun[mt][0] = lrun[mt][1] = 0.f;
    }
    for (int k0 = 0; k0 < t; k0 += kBertS) {
        __syncthreads();      // the previous key tile is no longer being read
        for (int i = tid; i < kBertS * DT; i += 128) {
            const int r = i / DT, c = (i % DT) * 8;
            uint4 k = make_uint4(0, 0, 0, 0), v = k;
            if (k0 + r < t) {
                const uint16_t* src = qkv + (row0 + k0 + r) * ld + head * D + c;
                k = *reinterpret_cast<const uint4*>(src + H);
                v = *reinterpret_cast<const uint4*>(src + 2 * H);
            }
            *reinterpret_cast<uint4*>(sk + r * LD + c) = k;
            *reinterpret_cast<uint4*>(sv + r * LD + c) = v;
        }
        __syncthreads();
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            if (q0 + warp * 32 + mt * 16 >= t) continue;
            float s[16][4];
#pragma unroll
            for (int nt = 0; nt < 16; ++nt) {
                s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
                for (int ks = 0; ks < KS; ++ks) {
                    uint32_t kb[2];
                    ldmatrix_x2(kb, sk + (nt * 8 + (lane & 7)) * LD + ks * 16 + ((lane >> 3) & 1) * 8);
                    mma_bf16_16816(s[nt], qa[mt][ks], kb);
                }
            }
            float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
            for (int nt = 0; nt < 16; ++nt) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int key = k0 + nt * 8 + tq * 2 + (e & 1);
                    s[nt][e] = key < t ? s[nt][e] * inv_scale : -INFINITY;
                }
                mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
                mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
            }
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xFFFFFFFFu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xFFFFFFFFu, mx0, 2));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xFFFFFFFFu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xFFFFFFFFu, mx1, 2));
            const float mn0 = fmaxf(mrun[mt][0], mx0), mn1 = fmaxf(mrun[mt][1], mx1);      // finite: the tile holds key k0 < t
            const float al0 = __expf(mrun[mt][0] - mn0), al1 = __expf(mrun[mt][1] - mn1);
            mrun[mt][0] = mn0; mrun[mt][1] = mn1;
            float ps0 = 0.f, ps1 = 0.f;
#pragma unroll
            for (int nt = 0; nt < 16; ++nt) {
                s[nt][0] = __expf(s[nt][0] - mn0); s[nt][1] = __expf(s[nt][1] - mn0);
                s[nt][2] = __expf(s[nt][2] - mn1); s[nt][3] = __expf(s[nt][3] - mn1);
                ps0 += s[nt][0] + s[nt][1];
                ps1 += s[nt][2] + s[nt][3];
            }
            lrun[mt][0] = lrun[mt][0] * al0 + ps0;      // per-thread partial row sums; the quad is reduced once at the end
            lrun[mt][1] = lrun[mt][1] * al1 + ps1;
#pragma unroll
            for (int dt = 0; dt < DT; ++dt) {
                o[mt][dt][0] *= al0; o[mt][dt][1] *= al0; o[mt][dt][2] *= al1; o[mt][dt][3] *= al1;
            }
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) {
                uint32_t pa[4];
                pa[0] = pack_bf16(s[2 * ks][0], s[2 * ks][1]);
                pa[1] = pack_bf16(s[2 * ks][2], s[2 * ks][3]);
                pa[2] = pack_bf16(s[2 * ks + 1][0], s[2 * ks + 1][1]);
                pa[3] = pack_bf16(s[2 * ks + 1][2], s[2 * ks + 1][3]);
#pragma unroll
                for (int dt = 0; dt < DT; ++dt) {
                    uint32_t vb[2];
                    ldmatrix_x2_trans(vb, sv + (ks * 16 + (lane & 15)) * LD + dt * 8);
                    mma_bf16_16816(o[mt][dt], pa, vb);
                }
            }
        }
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        const int m0 = q0 + warp * 32 + mt * 16;
        if (m0 >= t) continue;
        float l0 = lrun[mt][0], l1 = lrun[mt][1];
        l0 += __shfl_xor_sync(0xFFFFFFFFu, l0, 1); l0 += __shfl_xor_sync(0xFFFFFFFFu, l0, 2);
        l1 += __shfl_xor_sync(0xFFFFFFFFu, l1, 1); l1 += __shfl_xor_sync(0xFFFFFFFFu, l1, 2);
        const float i0 = 1.f / l0, i1 = 1.f / l1;
        const int r0 = m0 + g, r1 = m0 + g + 8;
#pragma unroll
        for (int dt = 0; dt < DT; ++dt) {
            const int c = head * D + dt * 8 + tq * 2;
            if (r0 < t) *reinterpret_cast<uint32_t*>(ctx + (row0 + r0) * H + c) = pack_bf16(o[mt][dt][0] * i0, o[mt][dt][1] * i0);
            if (r1 < t) *reinterpret_cast<uint32_t*>(ctx + (row0 + r1) * H + c) = pack_bf16(o[mt][dt][2] * i1, o[mt][dt][3] * i1);
        }
    }
}

// mean_pooling + normalize_l2: one CTA per sentence, thread per hidden column (H <= 1024); mask (per token row) may be NULL = all ones.
static __global__ void pool_l2_kernel(const uint16_t* __restrict__ x, const uint32_t* __restrict__ mask, const int* __restrict__ starts, int H,
                                      float* __restrict__ out) {
    pdl_launch_dependents();      // programmatic dependent launch: the next kernel may start its prologue now ...
    const int sent = blockIdx.x, c = threadIdx.x;
    const int r0 = starts[sent], r1 = starts[sent + 1];      // a sentence table
    pdl_wait();                   // ... and nothing below runs before the previous kernel has completed
    __shared__ float red[32];
    float acc = 0.f, cnt = 0.f;
    for (int r = r0; r < r1; ++r) {
        const float m = mask ? (float)mask[r] : 1.f;
        cnt += m;
        if (c < H) acc = fmaf(__uint_as_float((uint32_t)x[(size_t)r * H + c] << 16), m, acc);
    }
    const float pooled = acc / (cnt * (float)H);      // divisor = mask_count * hidden (embeddings.rs:359-365); cancelled below
    float sq = (c < H) ? pooled * pooled : 0.f;
    sq = warp_sum(sq);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sq;
    __syncthreads();
    float tot = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
    if (c < H) out[(size_t)sent * H + c] = pooled / sqrtf(tot);
}

}  // namespace fl
