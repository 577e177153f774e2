// Dense bf16 GEMM on the 5th-gen tensor cores: D[M,N] = A[M,K] . B[N,K]^T (+ fused epilogue), sm_100a only.
//
// Hand-written tcgen05 / TMEM / TMA (inline PTX, no CUTLASS):
//   * operands are K-major bf16 in global memory ([rows, K] row-major: activations [tokens, K], weights [out, K] exactly as
//     HF stores them), fetched by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle) into a 4-stage shared-memory ring;
//   * one elected thread issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16) with shared-memory descriptors,
//     accumulating f32 in TMEM; tcgen05.commit releases ring slots / signals the epilogue through mbarriers;
//   * warp roles: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2-5 = epilogue (tcgen05.ld
//     32x32b: thread == accumulator row), which applies bias / GELU-tanh / residual and stores bf16 or f32.
// Replaces the reference's cuBLAS-through-candle matmuls + separate bias/activation kernels (SURVEY.md section 2.4 B2, B5,
// B6, B7 and K3/K12/K15/K16 for prefill).
#pragma once
#include <cuda.h>

#include <algorithm>

#include "common.cuh"

namespace fl {

enum : int { GEPI_BIAS_BF16 = 0, GEPI_BIAS_GELU_BF16 = 1, GEPI_BIAS_RESID_F32 = 2, GEPI_F32 = 3, GEPI_F32_T = 5, GEPI_SILU_HL = 6 };
enum : int { DUAL_NONE = 0, DUAL_A = 1, DUAL_B = 2 };

constexpr int kGemmBM = 128;
constexpr int kGemmBK = 64;          // 64 bf16 = 128 bytes = one swizzle row
constexpr int kGemmEpiWarps = 16;      // four per TMEM lane quarter; each takes BN/4 columns of the tile
constexpr int kGemmThreads = 64 + 32 * kGemmEpiWarps;

struct GemmArgs {
    int M, N, K;
    const float* bias;          // [N] or null
    const uint16_t* resid;      // bf16 [M, ldr] residual (GEPI_BIAS_RESID_F32) or null
    int ldr;
    void* out;                  // bf16 or f32 [M, ldo]
    int ldo;
    int ksplit;                 // >1: K is cut into ksplit ranges handled by different work items (GEPI_F32)
    long long split_stride;     // GEPI_F32 with ksplit > 1: split s writes its partial sums to out + s * split_stride (deterministic)
    void* out2 = nullptr;       // GEPI_SILU_HL: the lo half ([M, ldo] bf16, like `out` = the hi half)
    // GROUPED swap-AB GEMM (DUAL_B + GEPI_F32_T; the Mixtral experts): A stacks `M / grp_m` weight matrices of grp_m rows each,
    // B stacks one block of grp_cap (<= BN) activation rows per group -- the rows routed to that expert, gathered -- and group j
    // multiplies ITS rows with ITS matrix: out[slice][j * grp_cap + n][row within the group].  grp_cnt[j] (device memory, written
    // by the gather kernel) is the number of valid rows: a group without rows is skipped entirely (no weight traffic), columns
    // past the count are not stored.
    int grp_m = 0;
    int grp_cap = 0;
    const int* grp_cnt = nullptr;
};

// ---- PTX wrappers ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on the mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// thread i of the warp receives columns [col, col+32) of TMEM lane (32*quarter + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// thread i of the warp writes columns [col, col+32) of TMEM lane (32*quarter + i)
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
        "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]),
        "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// 16-column variant (register pressure: the hi | lo halves of a DUAL_B accumulator are added 16 columns at a time)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptor for a K-major bf16 tile stored as rows of 128 bytes with the 128-byte swizzle
// (exactly what TMA SWIZZLE_128B writes): start address >> 4, LBO = 1 (ignored for swizzled K-major), SBO = 1024 B >> 4
// (stride between 8-row groups), version = 1 (Blackwell), layout type 2 = SWIZZLE_128B.
__device__ __forceinline__ uint64_t umma_smem_desc_sw128(const void* smem_ptr) {
    const uint64_t addr = (uint64_t)((smem_u32(smem_ptr) & 0x3FFFF) >> 4);
    return addr | ((uint64_t)1 << 16) | ((uint64_t)64 << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// Instruction descriptor, kind::f16: D=f32 (bits 4-5 = 1), A=B=bf16 (bits 7-9 = 1, 10-12 = 1), both K-major, N>>3 at 17, M>>4 at 24.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// dynamic shared memory of gemm_tc_kernel<BN, *, DUAL> (ring + 1 KB alignment slack); mirrors the constants in the kernel
// The encoder's epilogues (GEPI_BIAS_BF16 / GEPI_BIAS_GELU_BF16: 32 bf16 columns per pass; GEPI_BIAS_RESID_F32: 16 f32 columns per
// pass, its bf16 residual rows read through the same buffer) stage every warp's 32 rows x 64 bytes in shared memory (rows padded
// to 80 bytes: conflict-free 16-byte accesses) and move them 8 rows x 64 bytes per instruction.  thread == accumulator row is
// what tcgen05.ld hands out, and storing that way scatters every 16-byte store of a warp over 32 lines: ncu had the encoder's GEMMs
// at 27 % tensor activity with the LSU as the busiest unit.
constexpr int kEpiStageRow = 80;
constexpr int kEpiStageBytes = kGemmEpiWarps * 32 * kEpiStageRow;      // 40 KB
__host__ __device__ constexpr bool gemm_epi_staged(int epi) { return epi == GEPI_BIAS_BF16 || epi == GEPI_BIAS_GELU_BF16 || epi == GEPI_BIAS_RESID_F32; }

inline size_t gemm_smem_bytes(int BN, int dual) {
    const size_t stage = (size_t)(dual == DUAL_A ? 2 : 1) * kGemmBM * kGemmBK * 2 + (size_t)(dual == DUAL_B ? 2 : 1) * BN * kGemmBK * 2;
    const size_t stages = std::min<size_t>(196608 / stage, 8);
    return stages * stage + 1024;
}

__device__ __forceinline__ float gelu_tanh_f(float x) {
    // candle Tensor::gelu(): 0.5 x (1 + tanh(u)), u = sqrt(2/pi) x (1 + 0.044715 x^2)   (models/embeddings.rs:229-231)
    // ONE MUFU op per element (tanh.approx.f32, |error| ~ 5e-4, far inside the bf16 rounding of the output): the intermediate GEMM's
    // epilogue handles 50 M elements per 256 x 128 batch and the special-function unit issues 16 per clock per SM -- the two-MUFU
    // sigmoid form (ex2 + rcp) this replaces spent ~20 of the GEMM's 72 us there.
    const float u = x * fmaf(0.7978845608028654f * 0.044715f, x * x, 0.7978845608028654f);
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
    const float hx = 0.5f * x;
    return fmaf(hx, t, hx);
}

// Persistent, warp-specialised: grid = min(#SMs, #tiles); each CTA walks tiles t = blockIdx.x, +gridDim.x, ... (n fastest, so
// the CTAs running concurrently share activation rows through L2).  Three pipelines: shared-memory ring (TMA -> MMA),
// two TMEM accumulator stages (MMA -> epilogue: the epilogue of tile i overlaps the MMAs of tile i+1), and the tile walk.
// DUAL_A / DUAL_B: that operand is the sum of two bf16 tensors (hi + lo split of an f32 activation); both halves are
// multiplied with the same staged tile of the other operand: ~16 mantissa bits on the activations at no extra weight traffic.
//   DUAL_A: prefill orientation, A = activations [tokens, K] (hi, lo), B = weights [out, K].
//   DUAL_B: swap-AB decode orientation (<= 128 activation rows): A = weights [out, K] (the 128-row MMA operand, the only
//           large tile), B = activations [rows <= BN, K] (hi, lo); D[out, rows] is stored transposed (GEPI_F32_T) so that
//           a warp writes 32 consecutive floats of one activation row.
template <int BN, int EPI, int DUAL = DUAL_NONE>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB,
               const GemmArgs g) {
    static_assert(BN % 16 == 0 && BN >= 16 && BN <= 256, "UMMA N for M=128 must be a multiple of 16 in [16, 256]");
    constexpr uint32_t kABytes = kGemmBM * kGemmBK * 2;   // 16 KB
    constexpr uint32_t kBBytes = BN * kGemmBK * 2;
    constexpr uint32_t kStageBytes = (DUAL == DUAL_A ? 2 : 1) * kABytes + (DUAL == DUAL_B ? 2 : 1) * kBBytes;
    constexpr int kStages = (196608 / kStageBytes) < 8 ? (196608 / kStageBytes) : 8;   // <= 192 KB of ring, <= 8 stages
    constexpr uint32_t kBOff = (DUAL == DUAL_A ? 2 : 1) * kABytes;
    // DUAL_B: the hi and lo activation tiles sit back to back in a stage ([BN rows x 128 B] each, same swizzle), so ONE MMA of
    // N = 2 BN multiplies the weight tile with both -- half the tcgen05.mma instructions per staged byte (at N = 16 the issue rate
    // of these tiny MMAs, not the weight stream, was the limit, measured in round 2) -- into two accumulator column blocks
    // [W.hi | W.lo] that the epilogue adds.
    constexpr int kMmaN = (DUAL == DUAL_B) ? 2 * BN : BN;
    static_assert(kMmaN <= 256, "UMMA N <= 256");
    constexpr uint32_t kAccCols = kMmaN <= 32 ? 32 : (kMmaN <= 64 ? 64 : (kMmaN <= 128 ? 128 : 256));
    constexpr uint32_t kTmemCols = 2 * kAccCols;          // two accumulator stages

    extern __shared__ uint8_t gsm_raw[];
    // SWIZZLE_128B tiles need 1024-byte alignment; the launch adds 1024 bytes of slack for this round-up
    uint8_t* gsm = gsm_raw + ((1024u - (smem_u32(gsm_raw) & 1023u)) & 1023u);
    __shared__ __align__(8) uint64_t full[kStages], empty[kStages], acc_full[2], acc_empty[2];
    __shared__ uint32_t tmem_base_s;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nk = (g.K + kGemmBK - 1) / kGemmBK;
    const bool grouped = (DUAL == DUAL_B) && g.grp_m > 0;
    const int mt_e = grouped ? (g.grp_m + kGemmBM - 1) / kGemmBM : 0;      // m tiles per group
    const int mt = grouped ? (g.M / g.grp_m) * mt_e : (g.M + kGemmBM - 1) / kGemmBM, nt = grouped ? 1 : (g.N + BN - 1) / BN;
    const int ksplit = g.ksplit > 1 ? g.ksplit : 1;
    // tile -> (first row of the A box, first row of the B box, group, first row inside the group)
    auto coords = [&](int tile, int& m0, int& n0, int& grp, int& mrow0) {
        if (grouped) {
            grp = tile / mt_e;
            mrow0 = (tile % mt_e) * kGemmBM;
            m0 = grp * g.grp_m + mrow0;
            n0 = grp * g.grp_cap;
        } else {
            grp = 0;
            m0 = mrow0 = (tile / nt) * kGemmBM;
            n0 = (tile % nt) * BN;
        }
    };
    const int nkps = (nk + ksplit - 1) / ksplit;          // k-blocks per split
    const int ntiles = mt * nt * ksplit;                  // work items: (m tile, n tile, k split), k split fastest

    // programmatic dependent launch: the next kernel's prologue may start now; our own prologue (barriers, TMEM, descriptor
    // fetch) overlaps the previous kernel's tail.  Everything that touches dependent memory is ordered behind the producer's
    // griddepcontrol.wait below (MMA waits for TMA, the epilogue waits for MMA).
    pdl_launch_dependents();
    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&acc_full[s], 1);
            mbar_init(&acc_empty[s], kGemmEpiWarps);      // one arrive per epilogue warp
        }
        mbar_fence_init();
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
    }
    if (warp == 1) tmem_alloc(&tmem_base_s, kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            pdl_wait();
            asm volatile("fence.proxy.async;" ::: "memory");      // the previous kernel's generic-proxy stores -> TMA reads
            uint32_t c = 0;
            for (int item = blockIdx.x; item < ntiles; item += gridDim.x) {
                const int tile = item / ksplit, ks = item % ksplit;
                int m0, n0, grp, mrow0;
                coords(tile, m0, n0, grp, mrow0);
                if (grouped && g.grp_cnt[grp] == 0) continue;      // no row was routed to this expert: its weights are not read
                const int kb1 = min((ks + 1) * nkps, nk);
                for (int kb = ks * nkps; kb < kb1; ++kb, ++c) {
                    const int st = c % kStages;
                    uint8_t* sa = gsm + (size_t)st * kStageBytes;
                    mbar_wait(&empty[st], ((c / kStages) & 1) ^ 1);
                    mbar_expect_tx(&full[st], kStageBytes);
                    if (DUAL == DUAL_B) {       // tmA = weights, tmA2 / tmB = activation hi / lo
                        tma_load_2d(sa, &tmA, kb * kGemmBK, m0, &full[st]);
                        tma_load_2d(sa + kBOff, &tmA2, kb * kGemmBK, n0, &full[st]);
                        tma_load_2d(sa + kBOff + kBBytes, &tmB, kb * kGemmBK, n0, &full[st]);
                    } else {
                        tma_load_2d(sa, &tmA, kb * kGemmBK, m0, &full[st]);
                        if (DUAL == DUAL_A) tma_load_2d(sa + kABytes, &tmA2, kb * kGemmBK, m0, &full[st]);
                        tma_load_2d(sa + kBOff, &tmB, kb * kGemmBK, n0, &full[st]);
                        // DUAL_A with a 256-row weight tile: the weight descriptors carry a 128-row box (the swap-AB decode GEMMs'
                        // A operand), so the tile arrives as two boxes; rows past the matrix are zero-filled by the TMA engine
                        if (DUAL == DUAL_A && BN == 256) tma_load_2d(sa + kBOff + kBBytes / 2, &tmB, kb * kGemmBK, n0 + 128, &full[st]);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (single thread) =====
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(kGemmBM, kMmaN);
            uint32_t c = 0, ti = 0;
            if (grouped) pdl_wait();      // grp_cnt is written by the preceding kernel
            for (int item = blockIdx.x; item < ntiles; item += gridDim.x) {
                if (grouped && g.grp_cnt[(item / ksplit) / mt_e] == 0) continue;
                const uint32_t ti_now = ti++;
                const int ks = item % ksplit;
                const int kb0 = ks * nkps, kb1 = min((ks + 1) * nkps, nk);
                const uint32_t as = ti_now & 1;
                mbar_wait(&acc_empty[as], ((ti_now >> 1) & 1) ^ 1);     // epilogue has drained this accumulator stage
                tc_fence_after();
                const uint32_t tacc = tmem_base + as * kAccCols;
                for (int kb = kb0; kb < kb1; ++kb, ++c) {
                    const int st = c % kStages;
                    mbar_wait(&full[st], (c / kStages) & 1);
                    tc_fence_after();
                    const uint8_t* sa = gsm + (size_t)st * kStageBytes;
                    const uint64_t adesc = umma_smem_desc_sw128(sa), bdesc = umma_smem_desc_sw128(sa + kBOff);
#pragma unroll
                    for (int k = 0; k < kGemmBK / 16; ++k)   // advance 16 elements = 32 bytes inside the swizzle row: +2 in the (>>4) address field
                        umma_bf16(tacc, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, ((kb - kb0) | k) ? 1u : 0u);
                    if (DUAL == DUAL_A) {
                        const uint64_t a2desc = umma_smem_desc_sw128(sa + kABytes);
#pragma unroll
                        for (int k = 0; k < kGemmBK / 16; ++k) umma_bf16(tacc, a2desc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, 1u);
                    }       // DUAL_B: the first loop already covered hi | lo (N = 2 BN)
                    umma_commit(&empty[st]);                 // slot reusable once these MMAs have read it
                }
                umma_commit(&acc_full[as]);                  // accumulator of this tile complete
            }
        }
    } else {
        // ===== epilogue: warps 2..17; TMEM lane quarter = warp % 4 (hardware rule), column slice = (warp - 2) / 4; thread == output row =====
        const int q = warp & 3;
        const int cslice = (warp - 2) >> 2;
        uint32_t ti = 0;
        if (grouped) pdl_wait();          // grp_cnt is written by the preceding kernel
        for (int item = blockIdx.x; item < ntiles; item += gridDim.x) {
            const int tile = item / ksplit, ksi = item % ksplit;
            int m0, n0, grp, mrow0;
            coords(tile, m0, n0, grp, mrow0);
            const int gcnt = grouped ? g.grp_cnt[grp] : 0;
            if (grouped && gcnt == 0) continue;
            const uint32_t ti_now = ti++;
            const uint32_t as = ti_now & 1;
            // grouped: `row` counts inside the group's matrix and the columns are the group's block of the stacked output
            const int row = mrow0 + q * 32 + lane;
            const int row_lim = grouped ? g.grp_m : g.M, col_lim = grouped ? gcnt : g.N;
            if (grouped) n0 = 0;
            mbar_wait(&acc_full[as], (ti_now >> 1) & 1);
            tc_fence_after();
#pragma unroll 1
            for (int c0 = cslice * 32; c0 < BN; c0 += 128) {      // 32-column chunks dealt round-robin to the 4 warps of a lane quarter
                uint32_t r[32];
                tmem_ld32(tmem_base + as * kAccCols + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, r);
                if (DUAL == DUAL_B) {       // accumulator columns [0, BN) = W . hi, [BN, 2 BN) = W . lo
                    if (BN >= 32) {
#pragma unroll
                        for (int hlf = 0; hlf < 2; ++hlf) {
                            uint32_t r2[16];
                            tmem_ld16(tmem_base + as * kAccCols + ((uint32_t)(q * 32) << 16) + (uint32_t)(BN + c0 + 16 * hlf), r2);
#pragma unroll
                            for (int j = 0; j < 16; ++j) r[16 * hlf + j] = __float_as_uint(__uint_as_float(r[16 * hlf + j]) + __uint_as_float(r2[j]));
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(r[j + 16]));
                    }
                }
                if (EPI == GEPI_BIAS_RESID_F32) {
                    // f32 out = acc + bias + bf16 residual, 16 columns (64 bytes of f32) per pass: the residual rows (32 bytes each) come
                    // in through the staging buffer two rows per lane, the results leave through it 8 rows x 64 bytes per instruction
                    uint8_t* stg = gsm + (size_t)kStages * kStageBytes + (size_t)(warp - 2) * (32 * kEpiStageRow);
                    float* obase = reinterpret_cast<float*>(g.out);
#pragma unroll
                    for (int hc = 0; hc < 32; hc += 16) {
                        const int col = n0 + c0 + hc;
                        if (g.resid != nullptr) {
#pragma unroll
                            for (int p = lane; p < 64; p += 32) {
                                const int rr = p >> 1, part = p & 1;
                                const int grow = m0 + q * 32 + rr, gcol = col + part * 8;
                                uint4 rv = make_uint4(0u, 0u, 0u, 0u);
                                if (grow < g.M && gcol < g.N) rv = *reinterpret_cast<const uint4*>(g.resid + (size_t)grow * g.ldr + gcol);
                                *reinterpret_cast<uint4*>(stg + rr * kEpiStageRow + part * 16) = rv;
                            }
                            __syncwarp();
                        }
                        uint4 r0 = make_uint4(0u, 0u, 0u, 0u), r1 = r0;
                        if (g.resid != nullptr) {
                            r0 = *reinterpret_cast<const uint4*>(stg + lane * kEpiStageRow);
                            r1 = *reinterpret_cast<const uint4*>(stg + lane * kEpiStageRow + 16);
                            __syncwarp();
                        }
                        const uint32_t rw[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
                        for (int j = 0; j < 16; j += 4) {
                            float4 v = make_float4(__uint_as_float(r[hc + j]), __uint_as_float(r[hc + j + 1]), __uint_as_float(r[hc + j + 2]),
                                                   __uint_as_float(r[hc + j + 3]));
                            if (g.bias != nullptr && col + j < g.N) {
                                const float4 bv = *reinterpret_cast<const float4*>(g.bias + col + j);
                                v.x += bv.x; v.y += bv.y; v.z += bv.z; v.w += bv.w;
                            }
                            v.x += bf16lo(rw[j >> 1]); v.y += bf16hi(rw[j >> 1]); v.z += bf16lo(rw[(j >> 1) + 1]); v.w += bf16hi(rw[(j >> 1) + 1]);
                            *reinterpret_cast<float4*>(stg + lane * kEpiStageRow + j * 4) = v;
                        }
                        __syncwarp();
#pragma unroll
                        for (int p = lane; p < 128; p += 32) {
                            const int rr = p >> 2, part = p & 3;
                            const int grow = m0 + q * 32 + rr, gcol = col + part * 4;
                            if (grow < g.M && gcol < g.N)
                                *reinterpret_cast<uint4*>(obase + (size_t)grow * g.ldo + gcol) = *reinterpret_cast<const uint4*>(stg + rr * kEpiStageRow + part * 16);
                        }
                        __syncwarp();
                    }
                    continue;
                }
                if (gemm_epi_staged(EPI)) {
                    // stage this lane's row (32 columns = 64 bytes), then the warp stores 8 rows x 64 bytes per instruction
                    uint8_t* stg = gsm + (size_t)kStages * kStageBytes + (size_t)(warp - 2) * (32 * kEpiStageRow);
                    const int col = n0 + c0;
#pragma unroll
                    for (int j = 0; j < 32; j += 8) {
                        uint32_t pk[4] = {0u, 0u, 0u, 0u};
                        if (col + j < g.N) {
                            const float4 b0 = g.bias ? *reinterpret_cast<const float4*>(g.bias + col + j) : make_float4(0.f, 0.f, 0.f, 0.f);
                            const float4 b1 = g.bias ? *reinterpret_cast<const float4*>(g.bias + col + j + 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                            for (int e = 0; e < 8; e += 2) {
                                float v0 = __uint_as_float(r[j + e]) + bb[e];
                                float v1 = __uint_as_float(r[j + e + 1]) + bb[e + 1];
                                if (EPI == GEPI_BIAS_GELU_BF16) { v0 = gelu_tanh_f(v0); v1 = gelu_tanh_f(v1); }
                                pk[e >> 1] = pack_bf16x2(v0, v1);
                            }
                        }
                        *reinterpret_cast<uint4*>(stg + lane * kEpiStageRow + (j >> 3) * 16) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    }
                    __syncwarp();
                    uint16_t* obase = reinterpret_cast<uint16_t*>(g.out);
#pragma unroll
                    for (int p = lane; p < 128; p += 32) {
                        const int rr = p >> 2, part = p & 3;
                        const int grow = m0 + q * 32 + rr, gcol = col + part * 8;
                        if (grow < g.M && gcol < g.N)
                            *reinterpret_cast<uint4*>(obase + (size_t)grow * g.ldo + gcol) = *reinterpret_cast<const uint4*>(stg + rr * kEpiStageRow + part * 16);
                    }
                    __syncwarp();
                    continue;
                }
                if (row < row_lim) {
                    const int col = n0 + c0;
                    if (EPI == GEPI_SILU_HL) {
                        // gate|up GEMM of the prefill: columns interleave gate_j (even) and up_j (odd); act_j = silu(gate_j) * up_j
                        // is written straight as the hi/lo bf16 operand of the down_proj GEMM ([M, N/2] each)
                        uint16_t* oh = reinterpret_cast<uint16_t*>(g.out) + (size_t)row * g.ldo + (col >> 1);
                        uint16_t* ol = reinterpret_cast<uint16_t*>(g.out2) + (size_t)row * g.ldo + (col >> 1);
#pragma unroll
                        for (int j = 0; j < 32; j += 16) {
                            if (col + j < g.N) {
                                uint32_t ph[4], pl[4];
#pragma unroll
                                for (int e = 0; e < 4; ++e) {
                                    const float g0 = __uint_as_float(r[j + 4 * e]), u0 = __uint_as_float(r[j + 4 * e + 1]);
                                    const float g1 = __uint_as_float(r[j + 4 * e + 2]), u1 = __uint_as_float(r[j + 4 * e + 3]);
                                    const float a0 = g0 / (1.f + expf(-g0)) * u0, a1 = g1 / (1.f + expf(-g1)) * u1;
                                    ph[e] = pack_bf16x2(a0, a1);
                                    pl[e] = pack_bf16x2(a0 - bf16lo(ph[e]), a1 - bf16hi(ph[e]));
                                }
                                *reinterpret_cast<uint4*>(oh + (j >> 1)) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
                                *reinterpret_cast<uint4*>(ol + (j >> 1)) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
                            }
                        }
                    } else if (EPI == GEPI_F32_T) {
                        // transposed store: D[row = weight row, col = activation row] -> out[slice][col, row]; for a fixed col the
                        // 32 lanes of the warp write 32 consecutive floats
                        float* o = reinterpret_cast<float*>(g.out) + (size_t)ksi * (size_t)g.split_stride + (size_t)grp * g.grp_cap * g.ldo + row;
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (col + j < col_lim) o[(size_t)(col + j) * g.ldo] = __uint_as_float(r[j]);
                    } else {      // GEPI_F32
                        float* o = reinterpret_cast<float*>(g.out) + (size_t)ksi * (size_t)g.split_stride + (size_t)row * g.ldo + col;
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            if (col + j < g.N) {
                                float4 v;
                                v.x = __uint_as_float(r[j]); v.y = __uint_as_float(r[j + 1]); v.z = __uint_as_float(r[j + 2]); v.w = __uint_as_float(r[j + 3]);
                                *reinterpret_cast<float4*>(o + j) = v;
                            }
                        }
                    }
                }
            }
            // all TMEM reads of this warp are complete (tcgen05.wait::ld inside tmem_ld32): hand the stage back
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[as]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, kTmemCols);
    }
}

}  // namespace fl
