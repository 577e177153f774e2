// Persistent batch-1 decode kernel: ONE cooperative launch runs whole decode steps (all layers + lm_head + arg-max),
// sm_100a.  This is the B200-first answer to "every small kernel pays a ramp and a tail": at batch 1 a decoder layer of
// Mistral-7B is five kernels of 5-36 us of HBM time each, and launch/ramp/tail costs as much as the streaming.
//
//   * grid = one CTA per SM (148), all resident (cooperative launch), 8 consumer warps + 1 producer warp.
//   * WEIGHT STREAM: the producer thread feeds a ring of shared-memory stages with the weight chunks this CTA will consume
//     -- per phase its static share of 16-row blocks, then blocks drawn from the phase's ticketed pool -- one 3-D TMA
//     request (32 KB, swizzled) per chunk, completion on the stage's mbarrier, plus a small per-stage message telling the
//     consumers which block / chunk arrived.  The stream is decoupled from the compute phases: while consumers sit in a
//     grid barrier, an epilogue or the attention phase, the ring is already filling with the NEXT phase's weights.
//   * consumers: a chunk is a 16-row x 1024-column block of the weight matrix: ONE 3-D TMA request that lands as
//     [column block][row][128 B] with the 128-byte swizzle keyed by the row (bank-conflict-free ldmatrix).  The 8 warps split its 64 k-steps; each k-step is ONE mma.sync m16n8k16: A = the bf16 weight tile
//     straight from shared memory (ldmatrix, no unpack instructions), B = the activation vector split hi + lo into two bf16
//     columns (~16 mantissa bits, products exact, f32 accumulate; the other six columns are don't-care), so
//     y[row] = D[row][0] + D[row][1] falls out of the
//     accumulator fragment without a single shuffle.  ~35 instructions per warp per 32 KB chunk (the CUDA-core version
//     needed ~170 and was the bottleneck: measured 1030 clk/chunk against the 770 clk/chunk the L2 can deliver).
//     Per-warp partials land in shared memory, one cross-warp sum per phase, then the same fused epilogues as gemv.cuh
//     (RMSNorm prologue; bias+RoPE+KV append; residual add; SiLU*up; logits+arg-max).
//   * phases of a layer are separated by a grid barrier (monotonic atomic counter, release/acquire fences); data that
//     crosses CTAs is read with ld.global.cg (L2) because L1 is not coherent across SMs.
//   * attention: split-K over the sequence, (kv_head, split) items spread over the CTAs, K/V read straight from the paged
//     cache with 128-bit ld.global.cg, online softmax, last-arriver merge (same algorithm as attn_decode.cuh).
//   * `nsteps` decode steps can run inside one launch (greedy feedback on device), so the device-resident loop has no
//     launch gaps at all.
#pragma once
#include "attn_decode.cuh"
#include "common.cuh"
#include "dense_ops.cuh"
#include "gemm_tc.cuh"
#include "gemv.cuh"
#include "mma.cuh"

namespace fl {

constexpr int kPkConsumerWarps = 8;
constexpr int kPkConsumers = kPkConsumerWarps * 32;
constexpr int kPkThreads = kPkConsumers + 32;
constexpr int kPkBlockRows = 16;                       // rows per chunk = M of the MMA
constexpr int kPkChunkCols = 1024;                     // columns per chunk
constexpr int kPkStageBytes = kPkBlockRows * kPkChunkCols * 2;     // 32 KB: ONE 3-D TMA request (see make_tmap_pk)
constexpr int kPkMaxStages = 6;
constexpr int kPkMaxSlots = 96;                        // blocks one CTA can process per phase (static share + pool cap)
constexpr int kPkMaxNormK = 8192;                      // RMSNorm prologue keeps the row in registers (hidden size limit)

struct PkLayer {
    const uint16_t* wqkv;
    const float* bqkv;
    const uint16_t* wo;
    const uint16_t* wgu;
    const uint16_t* wdown;
    const float* ln1;
    const float* ln2;
};

struct PkArgs {
    const PkLayer* layers;
    int L;
    const uint16_t* embed;
    const uint16_t* lm_head;
    const float* final_norm;
    int H, I, V, nh, nkv, d, nqkv, max_pos;
    float eps, qscale;
    const float* rope_cos;
    const float* rope_sin;
    uint16_t* kpool;
    uint16_t* vpool;
    size_t layer_pool_elems;
    const int* page_table;
    StepState* state;
    float* resid;      // [H]
    float* q;          // [nh*d]
    float* attn_out;   // [nh*d]   (unused by this kernel since the hi/lo hand-over below)
    uint16_t* xhl;     // hi/lo bf16 hand-over of the two plain activation vectors, written by their producers so the consumers'
                       // x-load is a straight copy: attn hi [nq] | attn lo [nq] | act hi [I] | act lo [I]
    float* act;        // [I]
    float* logits;     // [V]
    float* part_acc;   // [nh, nsplit, d]
    float* part_ml;    // [nh, nsplit, 2]
    int* counters;     // [nkv]
    int nsplit;
    float* amax_val;   // [gridDim.x]
    int* amax_idx;
    uint32_t* ids;
    uint32_t* next_ids;
    uint32_t* trace;
    int* trace_pos;
    unsigned int* gbar;   // grid-barrier counter, zero at launch
    int nsteps, feedback;
    int nstages;
    int xs_floats;        // shared-memory activation / scratch region capacity (floats)
    int kcap;             // largest K of any phase rounded up to whole chunks (x_hi at xs, x_lo at xs + (kcap + 8) bf16)
    const CUtensorMap* tmaps;   // [4 L + 1] weight-stream descriptors, indexed by the phase id g
    unsigned int* pool;         // [4 L + 1] ticket counters of the phases' dynamic block pools (zero between uses)
    int partial_rows;     // rows of the per-warp partial buffer
    // ---- tensor parallelism inside the kernel: all-reduce over NVLink peer memory (no NCCL call, no extra launch) ----
    int tp, rank;                    // tp == 1: single GPU
    float* peer_part[8];             // rank r's receive area [2 parities][tp sources][H] f32   (peer-mapped, r == rank: local)
    unsigned int* peer_flag[8];      // rank r's flags [tp sources][gridDim.x + 1] u32, monotone exchange epochs
    float* peer_amax[8];             // rank r's arg-max exchange slots [tp sources][2] (value, index bits)
    float* peer_logits[8];           // rank r's full-vocabulary logits [Vfull]
    unsigned int ar_epoch0;          // exchanges completed on this communicator before this launch
    int* comm_err;                   // set to 1 when a peer did not show up within the spin budget
    long long* dbg;       // optional: CTA 0 writes %globaltimer at the phase boundaries of layer L/2 (FL_PK_DEBUG=1)
};

// ---- block schedule ---------------------------------------------------------------------------------------------------
// A phase's weight matrix is cut into 16-row blocks.  Every CTA owns a STATIC share of contiguous blocks; the remaining
// ~16 % form a pool that the producers drain one block at a time through an atomic ticket counter: a CTA whose stream runs
// ahead (the L2->SM delivery rate differs by +-13 % between SMs, reproducibly) frees its ring slots sooner, reaches the pool
// sooner and takes more of it, so all CTAs reach the phase's grid barrier together.  Which CTA computes a row never changes
// its value (the whole dot product of a row lives in one CTA, summed in a fixed order), so results stay bit-reproducible.
// Tensor parallelism keeps the split static (no pool): the in-kernel all-reduce pairs the same CTA on every rank.
struct PkSplit {
    int s0, s1;        // static block range of this CTA
    int pool0, npool;  // pool = blocks [pool0, pool0 + npool)
    int ncc;           // column chunks per block
};
constexpr int kPkStaticNum = 30;      // static share of a phase's blocks, in 32nds (the rest is the pool)
constexpr int kPkPoolCap = 8;      // pool blocks one CTA may take per phase (bounds the per-CTA partial-sum buffer)

__device__ __forceinline__ PkSplit pk_split(int N, int K, int cta, int ncta, bool dynamic) {
    PkSplit p;
    const int nblk = N / kPkBlockRows;
    p.ncc = (K + kPkChunkCols - 1) / kPkChunkCols;
    if (dynamic) {
        const int S = (int)((long long)nblk * kPkStaticNum / 32) / ncta;
        p.s0 = cta * S; p.s1 = p.s0 + S;
        p.pool0 = ncta * S; p.npool = nblk - p.pool0;
    } else {
        p.s0 = (int)((long long)nblk * cta / ncta); p.s1 = (int)((long long)nblk * (cta + 1) / ncta);
        p.pool0 = nblk; p.npool = 0;
    }
    return p;
}

// per-stage message from the producer to the consumers (shared memory, published by the stage's mbarrier)
constexpr int kPkMetaEnd = 1 << 30;      // no data in this stage: the phase is over for this CTA

__device__ __forceinline__ void pk_named_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kPkConsumers) : "memory"); }

__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ uint4 ldcg_u4(const void* p) {
    uint4 r;
    asm volatile("ld.global.cg.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// L2 eviction-priority hint of the weight stream: weights are read exactly once per step and are dead once they are in shared
// memory, so the demand loads carry evict_first and leave the L2 to the KV cache and the activations.
// Prefetching the NEXT phase's weights into the L2 while the consumers sit between two weight phases (HBM idles there, and the L2
// feeds these boxes at 14.3 TB/s against 6.4-7.5 TB/s from HBM, tools/tma_stream_bench.cu) was built twice in round 2 -- a
// prefetch warp walking the CTA's static share N chunks ahead of the producer, with `cp.async.bulk.prefetch.tensor` and with
// plain `prefetch.global.L2`, all the time or only inside the gaps -- and measured SLOWER every time (N = 4: -4 %, 8: -10 %,
// 16: -15 %; DRAM bytes +1.4 %, only a third of the demand sectors turned into L2 hits): profiles/r02_persistent_limits.md.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
// Weight matrix of global phase g of a step: g = 4*layer + {0:qkv, 1:o, 2:gate|up, 3:down}, g = 4*L: lm_head.
__device__ __forceinline__ void pk_phase(const PkArgs& a, int g, const uint16_t*& W, int& N, int& K) {
    if (g == 4 * a.L) { W = a.lm_head; N = a.V; K = a.H; return; }
    const PkLayer& lw = a.layers[g >> 2];
    switch (g & 3) {
        case 0: W = lw.wqkv; N = a.nqkv; K = a.H; break;
        case 1: W = lw.wo; N = a.H; K = a.nh * a.d; break;
        case 2: W = lw.wgu; N = 2 * a.I; K = a.H; break;
        default: W = lw.wdown; N = a.H; K = a.I; break;
    }
}

// Grid barrier among the consumer threads of all CTAs (the producer warp never takes part and keeps streaming).
__device__ __forceinline__ void pk_grid_barrier(unsigned int* ctr, unsigned int& epoch, int tid) {
    pk_named_sync();
    epoch += 1;
    if (tid == 0) {
        // arrive: a release-reduction (no return value, so no round trip before the poll starts); the CTA barrier above
        // orders every consumer thread's writes before it (cumulativity), the acquire loads below order the reads after it
        asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(ctr), "r"(1u) : "memory");
        const unsigned int target = epoch * gridDim.x;
        while (ld_acquire_gpu(ctr) < target) { }
    }
    pk_named_sync();
}

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// wait until the peer's flag reaches `epoch`; bounded (about 2 s) so that a missing peer becomes an error, not a hang
__device__ __forceinline__ void pk_wait_flag(const unsigned int* flag, unsigned int epoch, int* err) {
    const long long t0 = clock64();
    while ((int)(ld_acquire_sys(flag) - epoch) < 0) {
        if (clock64() - t0 > 4000000000LL) {
            *err = 1;
            break;
        }
    }
}

template <int D>
__global__ void __launch_bounds__(kPkThreads, 1) decode_persistent_kernel(const PkArgs a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    // layout: [ring: nstages * 32 KB][xs: xs_floats f32][partial: partial_rows * 8 f32][sc: 8 * 64 f32][small]
    uint8_t* ring = smem;
    float* xs = reinterpret_cast<float*>(smem + (size_t)a.nstages * kPkStageBytes);
    float* partial = xs + a.xs_floats;
    float* sc = partial + (size_t)a.partial_rows * kPkConsumerWarps;      // [kAttnMaxRep][kKvPage]
    float* red = sc + kAttnMaxRep * kKvPage;                              // [32] block-reduce scratch
    float* alpha_s = red + 32;                                            // [8]
    float* mrun = alpha_s + 8;
    float* lrun = mrun + 8;
    int* s_flag = reinterpret_cast<int*>(lrun + 8);
    __shared__ __align__(8) uint64_t full[kPkMaxStages];
    __shared__ __align__(8) uint64_t empty[kPkMaxStages];
    __shared__ __align__(8) uint64_t xbar;      // completion of the bulk copies that bring a phase's hi/lo activation vector in
    __shared__ int2 meta[kPkMaxStages];      // per stage: {first row of the block, column chunk | last-chunk flag | end-of-phase flag}
    __shared__ int blk_rows[kPkMaxSlots];    // first rows of the blocks processed in the current phase

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cta = blockIdx.x, ncta = gridDim.x;
    const int NS = a.nstages;
    const int nq = a.nh * a.d;

    if (tid == 0) {
        for (int s = 0; s < NS; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kPkConsumerWarps);
        }
        mbar_init(&xbar, 1);
        mbar_fence_init();
    }
    __syncthreads();

    // =================================================================================================================
    // PRODUCER: one thread streams every weight chunk this CTA will ever need, in consumption order.
    // =================================================================================================================
    if (warp == kPkConsumerWarps) {
        if (lane != 0) return;
        unsigned int c = 0;   // running stage counter -> stage = c % NS, use = c / NS
        const uint64_t pol_first = l2_policy_evict_first();
        const bool dynamic = a.tp == 1 && a.pool != nullptr;
        for (int step = 0; step < a.nsteps; ++step) {
            for (int g = 0; g <= 4 * a.L; ++g) {
                const uint16_t* W;
                int N, K;
                pk_phase(a, g, W, N, K);
                const PkSplit sp = pk_split(N, K, cta, ncta, dynamic);
                const bool pdbg = a.dbg != nullptr && cta == 0 && g < 4 * a.L && (g >> 2) == a.L / 2;
                int pn = 0;
                auto fetch_block = [&](int blk) {
                    for (int cc = 0; cc < sp.ncc; ++cc) {
                        const int st = c % NS;
                        mbar_wait(&empty[st], ((c / NS) & 1) ^ 1);
                        ++c;
                        meta[st] = make_int2(blk * kPkBlockRows, cc | (cc == sp.ncc - 1 ? 1 << 16 : 0));
                        if (pdbg) {      // issue times of this phase's first 8 chunks and of its last one (FL_PK_DEBUG)
                            long long t;
                            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
                            if (pn < 8) a.dbg[660 + (g & 3) * 10 + pn] = t;
                            a.dbg[660 + (g & 3) * 10 + 8] = t;
                            a.dbg[660 + (g & 3) * 10 + 9] = ++pn;
                        }
                        mbar_expect_tx(&full[st], kPkStageBytes);      // the whole box always arrives (out-of-range columns as zeros)
                        // weights are dead once staged: evict_first keeps the L2 for the KV cache and the activations
                        asm volatile(
                            "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, %4}], [%5], %6;" ::"r"(
                                smem_u32(ring + (size_t)st * kPkStageBytes)),
                            "l"(a.tmaps + g), "r"(0), "r"(blk * kPkBlockRows), "r"(cc * (kPkChunkCols / 64)), "r"(smem_u32(&full[st])), "l"(pol_first)
                            : "memory");
                    }
                };
                for (int blk = sp.s0; blk < sp.s1; ++blk) fetch_block(blk);
                // tickets are taken lazily, only when this CTA is ready to stream another block (taking them ahead of time hands
                // the tail of the phase to CTAs that may turn out slow: measured slower); the ring hides the atomic's round trip
                for (int taken = 0; sp.npool > 0 && taken < kPkPoolCap; ++taken) {
                    const int t = (int)atomicAdd(a.pool + g, 1u);
                    if (t >= sp.npool) break;
                    fetch_block(sp.pool0 + t);
                }
                const int st = c % NS;          // end-of-phase message (no data)
                mbar_wait(&empty[st], ((c / NS) & 1) ^ 1);
                meta[st] = make_int2(0, kPkMetaEnd);
                mbar_arrive(&full[st]);
                ++c;
            }
        }
        return;
    }

    // =================================================================================================================
    // CONSUMERS
    // =================================================================================================================
    unsigned int c = 0;       // chunk counter, in lock-step with the producer's
    unsigned int epoch = 0;   // grid-barrier epoch

    // activation vector of the current phase as two bf16 vectors (x = hi + lo), the B operand of the MMAs
    uint16_t* xh = reinterpret_cast<uint16_t*>(xs);
    uint16_t* xl = xh + a.kcap + 8;          // +16 bytes: x_hi[k] and x_lo[k] sit in different bank groups
    const int g = lane >> 2, tq = lane & 3;

    // y = W_slice . x for this CTA's rows.  Chunk = 16 rows x <= 1024 columns; warp w takes k-steps w, w+8, ...; the f32
    // accumulator fragment lives in registers across the column chunks of a row block, and at the block's last chunk the
    // lanes with tq == 0 hold y[row g] = D[g][0] + D[g][1] (hi + lo column) and y[row g+8]: no shuffles.  Per-warp partial
    // sums land in partial[(row - row_begin) * 8 + warp] and are added up in the phase epilogue.
    long long dbg_wait = 0;
    int dbg_layer = -1, dbg_phase = 0;
    auto consume = [&](int K) -> int {      // -> number of 16-row blocks this CTA processed (their first rows in blk_rows[])
        dbg_wait = 0;
        // ldmatrix row addresses of this lane: A = weight tile rows (lane & 15), +8 columns for lanes 16-31;
        // B = [n = lane & 7][8 consecutive k]: n == 1 -> x_lo, every other n -> x_hi (columns 2-7 of D are never read, so those
        // rows need not be zero: re-reading x_hi is a broadcast and keeps the load bank-conflict-free); lanes 8-15 take k + 8
        // staged tile: [column block kb][row r][128 B], 16-byte piece p of a row stored at p ^ (r & 7) (TMA SWIZZLE_128B).
        // k-step ks = warp + 8 j covers pieces 2 (ks & 3) + {0, 1} of column block ks >> 2, so for a given lane the piece is
        // the same for every j and the k-steps of a warp are 4096 bytes apart.
        const int ar = lane & 15;
        const uint32_t a_off = (uint32_t)(warp >> 2) * 2048u + (uint32_t)ar * 128u + (uint32_t)(((((warp & 3) << 1) | (lane >> 4)) ^ (ar & 7)) << 4);
        const int bn = lane & 7, bk = ((lane >> 3) & 1) * 8;
        const uint16_t* xrow = bn == 1 ? xl : xh;
        float acc[2][4];
        int nslots = 0, nch = 0;
        while (true) {
            const int st = c % NS;
            const long long tw0 = a.dbg ? clock64() : 0;
            mbar_wait(&full[st], (c / NS) & 1);
            if (a.dbg) dbg_wait += clock64() - tw0;
            const int2 m = meta[st];
            ++c;
            if (m.y & kPkMetaEnd) {
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[st]);
                break;
            }
            const int cc = m.y & 0xFFFF;
            if (cc == 0) {
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[0][q] = acc[1][q] = 0.f;
            }
            const uint8_t* tile = ring + (size_t)st * kPkStageBytes + a_off;
            const int col0 = cc * kPkChunkCols;
            // all fragment loads of a half chunk first (independent, in flight together), then the MMAs (two accumulator chains).
            // (Round 2 tried the whole chunk's 16 loads ahead of four chains, with the stage index kept incrementally instead of
            // c % NS: faster with the weight traffic switched off, 0.8-3.6 % SLOWER in the real run on all three models: dropped.)
            constexpr int KPW = kPkChunkCols / 16 / kPkConsumerWarps;      // k-steps per warp per full chunk (8)
            const uint16_t* xcol = xrow + (col0 + bk + warp * 16);
#pragma unroll
            for (int h = 0; h < KPW; h += 4) {
                uint32_t af[4][4], bf[4][2];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    ldmatrix_x4(af[j], tile + (h + j) * 4096);
                    ldmatrix_x2(bf[j], xcol + (h + j) * kPkConsumerWarps * 16);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) mma_bf16_16816(acc[j & 1], af[j], bf[j]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[st]);
            ++nch;
            if (m.y & (1 << 16)) {      // last column chunk of the block: the row sums are complete
                if (tq == 0) {
                    float* pr = partial + (size_t)(nslots * kPkBlockRows + g) * kPkConsumerWarps + warp;
                    pr[0] = (acc[0][0] + acc[0][1]) + (acc[1][0] + acc[1][1]);
                    pr[8 * kPkConsumerWarps] = (acc[0][2] + acc[0][3]) + (acc[1][2] + acc[1][3]);
                }
                if (tid == 0) blk_rows[nslots] = m.x;
                ++nslots;
            }
        }
        if (a.dbg != nullptr && cta == 0 && tid == 0 && dbg_layer == a.L / 2) a.dbg[32 + (dbg_phase++ & 3)] = dbg_wait * 1000 + nch;
        pk_named_sync();   // partial[] and blk_rows[] complete
        return nslots;
    };
    // local row (slot * 16 + r) of the blocks this CTA processed in the current phase -> row of the weight matrix
    auto grow = [&](int local_row) { return blk_rows[local_row >> 4] + (local_row & 15); };
    // sum of the 8 per-warp partials of one row
    auto row_sum = [&](int local_row) {
        const float* pr = partial + (size_t)local_row * kPkConsumerWarps;
        float v = pr[0];
#pragma unroll
        for (int k = 1; k < kPkConsumerWarps; ++k) v += pr[k];
        return v;
    };
    // Row-parallel epilogue under tensor parallelism: resid[slice] += sum over ranks of this rank-local partial output.
    // One-shot exchange over NVLink peer memory: every CTA PUSHES its partial row slice into every rank's receive area
    // (tp x ~100 bytes), publishes a per-CTA flag with release.sys, waits for the same CTA of every peer, then sums the tp
    // partials in rank order (identical on every rank, so the replicas stay bit-identical) and adds them to the residual.
    unsigned int ar_epoch = a.ar_epoch0;
    auto allreduce_resid_add = [&](int nslots) {
        ar_epoch += 1;
        const int par = ar_epoch & 1;
        const int npair = nslots * (kPkBlockRows / 2);
        for (int e = tid; e < npair; e += kPkConsumers) {
            const float2 v = make_float2(row_sum(2 * e), row_sum(2 * e + 1));
            const size_t off = (size_t)(par * a.tp + a.rank) * a.H + grow(2 * e);
            for (int r = 0; r < a.tp; ++r) *reinterpret_cast<float2*>(a.peer_part[r] + off) = v;
        }
        // no per-thread system fence: the CTA barrier orders every thread's pushes before the flag writers' st.release.sys,
        // which is cumulative at system scope (PTX memory model), so one release per peer publishes the whole slice
        pk_named_sync();
        if (tid < a.tp) {
            st_release_sys(a.peer_flag[tid] + (size_t)a.rank * (ncta + 1) + cta, ar_epoch);
            pk_wait_flag(a.peer_flag[a.rank] + (size_t)tid * (ncta + 1) + cta, ar_epoch, a.comm_err);
        }
        pk_named_sync();
        const float* mine = a.peer_part[a.rank];
        for (int e = tid; e < npair; e += kPkConsumers) {
            const int gr = grow(2 * e);
            float2* p = reinterpret_cast<float2*>(a.resid + gr);
            float2 v = __ldcg(p);
            for (int r = 0; r < a.tp; ++r) {
                const float2 y = __ldcg(reinterpret_cast<const float2*>(mine + (size_t)(par * a.tp + r) * a.H + gr));
                v.x += y.x;
                v.y += y.y;
            }
            *p = v;
        }
    };
    auto block_sum = [&](float v) {   // sum over the 256 consumer threads
        v = warp_sum(v);
        if (lane == 0) red[warp] = v;
        pk_named_sync();
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kPkConsumerWarps; ++w) s += red[w];
        pk_named_sync();
        return s;
    };
    // x = hi + lo with two packed conversions per pair (cvt.rn.bf16x2.f32: the same round-to-nearest-even as split_hi_lo)
    auto split2 = [](float x0, float x1, uint32_t& hi2, uint32_t& lo2) {
        hi2 = pack_bf16x2(x0, x1);
        lo2 = pack_bf16x2(x0 - bf16lo(hi2), x1 - bf16hi(hi2));
    };
    auto store_x4 = [&](int i, const float4& v) {      // x[4i .. 4i+3] -> hi / lo bf16
        uint32_t h0, l0, h1, l1;
        split2(v.x, v.y, h0, l0);
        split2(v.z, v.w, h1, l1);
        reinterpret_cast<uint2*>(xh)[i] = make_uint2(h0, h1);
        reinterpret_cast<uint2*>(xl)[i] = make_uint2(l0, l1);
    };
    auto zero_x_tail = [&](int K) {     // columns [K, next multiple of 1024): the weight side is zero-filled, x must be finite
        const int kpad = (K + kPkChunkCols - 1) / kPkChunkCols * kPkChunkCols;
        for (int i = K / 4 + tid; i < kpad / 4; i += kPkConsumers) {
            reinterpret_cast<uint2*>(xh)[i] = make_uint2(0u, 0u);
            reinterpret_cast<uint2*>(xl)[i] = make_uint2(0u, 0u);
        }
    };
    // x = rms_norm(src) * norm_w      (candle_nn::ops::rms_norm, as in gemv.cuh); the row stays in registers between the passes
    auto load_x_rmsnorm = [&](const float* src, bool src_is_embed_row, const uint16_t* erow, const float* norm_w, int K,
                              float* resid_out) {
        constexpr int NV = kPkMaxNormK / 4 / kPkConsumers;      // float4 per thread
        float4 v[NV], wv[NV];
        float ss = 0.f;
        // the norm weights do not depend on the previous phase: their loads go out first and travel together with the row's, so the
        // scaling pass below finds them in registers instead of paying a second L2 round trip after the block reduction
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int i = tid + j * kPkConsumers;
            wv[j] = i < K / 4 ? __ldg(reinterpret_cast<const float4*>(norm_w) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int i = tid + j * kPkConsumers;
            v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < K / 4) {
                if (src_is_embed_row) {
                    const uint2 e = __ldg(reinterpret_cast<const uint2*>(erow) + i);
                    v[j] = make_float4(bf16lo(e.x), bf16hi(e.x), bf16lo(e.y), bf16hi(e.y));
                    if (resid_out) reinterpret_cast<float4*>(resid_out)[i] = v[j];
                } else {
                    v[j] = __ldcg(reinterpret_cast<const float4*>(src) + i);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < NV; ++j) {      // rows past K hold zeros
            ss = fmaf(v[j].x, v[j].x, ss); ss = fmaf(v[j].y, v[j].y, ss); ss = fmaf(v[j].z, v[j].z, ss); ss = fmaf(v[j].w, v[j].w, ss);
        }
        const float tot = block_sum(ss);
        const float m = sqrtf(tot / (float)K + a.eps);
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int i = tid + j * kPkConsumers;
            const float4 x = v[j];
            if (i < K / 4) store_x4(i, make_float4(x.x / m * wv[j].x, x.y / m * wv[j].y, x.z / m * wv[j].z, x.w / m * wv[j].w));
        }
        zero_x_tail(K);
        pk_named_sync();
    };
    // plain activation vectors arrive already split (written hi | lo by their producers): a straight L2 -> shared copy, issued as
    // two bulk copies (TMA engine, 1-D) by one thread -- one request per half instead of 14 load / store pairs per thread
    unsigned int xphase = 0;
    auto load_x_plain = [&](const uint16_t* hi, int K) {
        if (tid == 0) {
            asm volatile("fence.proxy.async;" ::: "memory");      // other CTAs' generic-proxy stores (ordered by the grid barrier) -> bulk reads
            mbar_expect_tx(&xbar, (uint32_t)K * 4u);
            bulk_g2s(xh, hi, (uint32_t)K * 2u, &xbar);
            bulk_g2s(xl, hi + K, (uint32_t)K * 2u, &xbar);
        }
        zero_x_tail(K);
        mbar_wait(&xbar, xphase & 1u);
        xphase ^= 1u;
        pk_named_sync();
    };

    // pull a small f32 vector (norm weights of an upcoming phase) towards L2 well before its prologue needs it
    auto prefetch_vec = [&](const float* p, int n) {
        for (int i = tid * 32; i < n; i += kPkConsumers * 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + i));
    };
    int dbg_i = 0;
    auto stamp = [&](int l) {
        if (a.dbg != nullptr && cta == 0 && tid == 0 && l == a.L / 2) {
            long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            a.dbg[dbg_i] = t;
        }
        ++dbg_i;
    };
    const int n_rep = a.nh / a.nkv;
    constexpr int LPT = D / 8, TPW = 32 / LPT;
    const int grp = lane / LPT, gl = lane % LPT;
    // this CTA's first attention item, opaque to the optimiser: starting the item loop at `cta` itself lets the compiler keep values
    // derived from it live across every weight phase, and the q|k|v phase then spills its MMA accumulators (ptxas at 168 registers;
    // Mistral-7B and TinyLlama batch 1 measured 0.9 % and 1.7 % slower per step)
    int item0 = cta;
    asm volatile("" : "+r"(item0));

    for (int step = 0; step < a.nsteps; ++step) {
        const uint32_t tok_id = __ldcg(a.ids);
        const int rope_pos = min(__ldcg(&a.state->rope_pos), a.max_pos - 1);
        const int kv_base = __ldcg(&a.state->kv_base[0]);
        const int slot = kv_base;                       // cache slot of the token being decoded
        const int len = kv_base + 1;
        const int page_of_slot = __ldg(a.page_table + slot / kKvPage);

        for (int l = 0; l < a.L; ++l) {
            const PkLayer& lw = a.layers[l];
            uint16_t* kpool = a.kpool + (size_t)l * a.layer_pool_elems;
            uint16_t* vpool = a.vpool + (size_t)l * a.layer_pool_elems;

            // ---------------- P1: RMSNorm -> q|k|v (+bias) -> RoPE -> q store + KV append ----------------
            prefetch_vec(lw.ln2, a.H);                                         // needed by P4, ~25 us from now
            dbg_i = 0;
            dbg_layer = l;
            stamp(l);
            if (l == 0) {      // page-table entries of this CTA's attention items (constant during the launch): towards L1, off the
                               // load -> load dependency chain of every layer's attention phase
                const int npages = (len + kKvPage - 1) / kKvPage;
                for (int i = tid * 32; i < npages; i += kPkConsumers * 32) asm volatile("prefetch.global.L1 [%0];" ::"l"(a.page_table + i));
            }
            if (l == 0)
                load_x_rmsnorm(nullptr, true, a.embed + (size_t)tok_id * a.H, lw.ln1, a.H, cta == 0 ? a.resid : nullptr);
            else
                load_x_rmsnorm(a.resid, false, nullptr, lw.ln1, a.H, nullptr);
            stamp(l);
            {
                const int nslots = consume(a.H);
                stamp(l);
                const int d = a.d, half = d >> 1;
                for (int e = tid; e < nslots * (kPkBlockRows / 2); e += kPkConsumers) {
                    const int ra = grow(2 * e);
                    float va = row_sum(2 * e), vb = row_sum(2 * e + 1);
                    if (lw.bqkv) { va += lw.bqkv[ra]; vb += lw.bqkv[ra + 1]; }
                    const int hh = ra / d, j = (ra % d) >> 1;
                    if (hh < a.nh + a.nkv) {
                        const float cs = a.rope_cos[(size_t)rope_pos * half + j], sn = a.rope_sin[(size_t)rope_pos * half + j];
                        const float o1 = va * cs - vb * sn, o2 = va * sn + vb * cs;
                        if (hh < a.nh) {
                            a.q[(size_t)hh * d + j] = o1;
                            a.q[(size_t)hh * d + j + half] = o2;
                        } else {
                            uint16_t* kp = kpool + (((size_t)page_of_slot * a.nkv + (hh - a.nh)) * kKvPage + slot % kKvPage) * d;
                            kp[j] = f32_to_bf16_rne(o1);
                            kp[j + half] = f32_to_bf16_rne(o2);
                        }
                    } else {
                        uint16_t* vp = vpool + (((size_t)page_of_slot * a.nkv + (hh - a.nh - a.nkv)) * kKvPage + slot % kKvPage) * d;
                        *reinterpret_cast<uint32_t*>(vp + 2 * j) = (uint32_t)f32_to_bf16_rne(va) | ((uint32_t)f32_to_bf16_rne(vb) << 16);
                    }
                }
            }
            stamp(l);
            pk_grid_barrier(a.gbar, epoch, tid);
            if (cta == 0 && tid == 0 && a.pool != nullptr) atomicExch(a.pool + (4 * l), 0u);      // every producer is past this phase: re-arm its pool
            stamp(l);

            // ---------------- P2: split-K attention over (kv head, split) items + last-arriver merge ----------------
            // Latency-optimised: every 16-lane group (two per warp, 16 per CTA) runs its OWN online softmax over a strided
            // subset of the item's tokens with all of its K/V loads in flight at once and q held in registers (loaded from L2
            // concurrently with K/V); the 16 partial states meet in shared memory after ONE block sync.
            {
                constexpr int HG = 4;                       // query heads per pass (register budget)
                constexpr int NG = kPkConsumerWarps * TPW;  // lane groups per CTA
                constexpr int BATCH = 4;                    // tokens in flight per lane group
                const int npages = (len + kKvPage - 1) / kKvPage;
                const int per = (npages + a.nsplit - 1) / a.nsplit;
                float* gacc = xs;                            // [NG][HG][D]
                float* gml = xs + NG * HG * D;               // [NG][HG][2]
                for (int item = item0; item < a.nkv * a.nsplit; item += ncta) {
                    const int kvh = item / a.nsplit, split = item % a.nsplit;
                    const int tok0 = split * per * kKvPage, tok1 = min(min((split + 1) * per, npages) * kKvPage, len);
                    const int gidx = warp * TPW + grp;
                    for (int h0 = 0; h0 < n_rep; h0 += HG) {
                        float qv[HG][8], acc[HG][8], mr[HG], lr[HG];
#pragma unroll
                        for (int h = 0; h < HG; ++h) {
                            mr[h] = -INFINITY;
                            lr[h] = 0.f;
#pragma unroll
                            for (int i = 0; i < 8; ++i) acc[h][i] = 0.f;
                            if (h0 + h < n_rep) {
                                const float4* qp = reinterpret_cast<const float4*>(a.q + (size_t)(kvh * n_rep + h0 + h) * D + gl * 8);
                                const float4 q0 = __ldcg(qp), q1 = __ldcg(qp + 1);
                                qv[h][0] = q0.x * a.qscale; qv[h][1] = q0.y * a.qscale; qv[h][2] = q0.z * a.qscale; qv[h][3] = q0.w * a.qscale;
                                qv[h][4] = q1.x * a.qscale; qv[h][5] = q1.y * a.qscale; qv[h][6] = q1.z * a.qscale; qv[h][7] = q1.w * a.qscale;
                            } else {
#pragma unroll
                                for (int i = 0; i < 8; ++i) qv[h][i] = 0.f;
                            }
                        }
                        // trip count is uniform across the CTA (the shuffles below use the full mask); validity is per lane group
                        for (int tb0 = tok0; tb0 < tok1; tb0 += NG * BATCH) {
                            const int tb = tb0 + gidx;
                            uint4 kw[BATCH], vw[BATCH];
#pragma unroll
                            for (int it = 0; it < BATCH; ++it) {
                                const int tk = tb + it * NG;
                                if (tk < tok1) {
                                    const size_t base = (((size_t)__ldg(a.page_table + tk / kKvPage) * a.nkv + kvh) * kKvPage + tk % kKvPage) * D + gl * 8;
                                    kw[it] = ldcg_u4(kpool + base);
                                    vw[it] = ldcg_u4(vpool + base);
                                } else {
                                    kw[it] = make_uint4(0u, 0u, 0u, 0u);
                                    vw[it] = kw[it];
                                }
                            }
#pragma unroll
                            for (int it = 0; it < BATCH; ++it) {
                                const bool valid = tb + it * NG < tok1;
                                const float kf[8] = {bf16lo(kw[it].x), bf16hi(kw[it].x), bf16lo(kw[it].y), bf16hi(kw[it].y),
                                                     bf16lo(kw[it].z), bf16hi(kw[it].z), bf16lo(kw[it].w), bf16hi(kw[it].w)};
                                const float vf[8] = {bf16lo(vw[it].x), bf16hi(vw[it].x), bf16lo(vw[it].y), bf16hi(vw[it].y),
                                                     bf16lo(vw[it].z), bf16hi(vw[it].z), bf16lo(vw[it].w), bf16hi(vw[it].w)};
#pragma unroll
                                for (int h = 0; h < HG; ++h) {
                                    float sv = kf[0] * qv[h][0];
#pragma unroll
                                    for (int i = 1; i < 8; ++i) sv = fmaf(kf[i], qv[h][i], sv);
#pragma unroll
                                    for (int o = LPT / 2; o > 0; o >>= 1) sv += __shfl_xor_sync(0xFFFFFFFFu, sv, o);
                                    if (valid) {      // uniform inside the lane group
                                        const float m_new = fmaxf(mr[h], sv);
                                        const float al = expf(mr[h] - m_new), pr = expf(sv - m_new);
                                        lr[h] = lr[h] * al + pr;
                                        mr[h] = m_new;
#pragma unroll
                                        for (int i = 0; i < 8; ++i) acc[h][i] = fmaf(acc[h][i], al, pr * vf[i]);
                                    }
                                }
                            }
                        }
                        // the NG partial states meet in shared memory
#pragma unroll
                        for (int h = 0; h < HG; ++h) {
                            float* dst = gacc + ((size_t)gidx * HG + h) * D + gl * 8;
#pragma unroll
                            for (int i = 0; i < 8; ++i) dst[i] = acc[h][i];
                            if (gl == 0) {
                                gml[(gidx * HG + h) * 2] = mr[h];
                                gml[(gidx * HG + h) * 2 + 1] = lr[h];
                            }
                        }
                        pk_named_sync();
                        for (int i = tid; i < HG * D; i += kPkConsumers) {
                            const int h = i / D, dd = i % D;
                            if (h0 + h < n_rep) {
                                float M = -INFINITY;
#pragma unroll
                                for (int g = 0; g < NG; ++g) M = fmaxf(M, gml[(g * HG + h) * 2]);
                                float num = 0.f, den = 0.f;
                                if (M != -INFINITY) {
#pragma unroll
                                    for (int g = 0; g < NG; ++g) {
                                        const float wg = expf(gml[(g * HG + h) * 2] - M);      // exp(-inf) = 0 for idle groups
                                        num = fmaf(wg, gacc[((size_t)g * HG + h) * D + dd], num);
                                        den = fmaf(wg, gml[(g * HG + h) * 2 + 1], den);
                                    }
                                }
                                const size_t pidx = (size_t)(kvh * n_rep + h0 + h) * a.nsplit + split;
                                a.part_acc[pidx * D + dd] = num;
                                if (dd == 0) {
                                    a.part_ml[pidx * 2] = M;
                                    a.part_ml[pidx * 2 + 1] = den;
                                }
                            }
                        }
                        pk_named_sync();      // gacc / gml are reused by the next head group
                    }
                    __threadfence();
                    pk_named_sync();
                    if (tid == 0) *s_flag = (atomicAdd(&a.counters[kvh], 1) == a.nsplit - 1);
                    pk_named_sync();
                    if (*s_flag) {
                        __threadfence();
                        float* cm = xs;                      // [n_rep][nsplit] weights
                        float* cden = cm + kAttnMaxRep * a.nsplit;
                        if (warp < n_rep) {
                            const int h = warp;
                            const size_t base = (size_t)(kvh * n_rep + h) * a.nsplit;
                            float mstar = -INFINITY;
                            for (int s = lane; s < a.nsplit; s += 32) mstar = fmaxf(mstar, __ldcg(a.part_ml + (base + s) * 2));
                            mstar = warp_max(mstar);
                            float den = 0.f;
                            for (int s = lane; s < a.nsplit; s += 32) {
                                const float ms = __ldcg(a.part_ml + (base + s) * 2);
                                const float w = (ms == -INFINITY) ? 0.f : expf(ms - mstar);
                                cm[h * a.nsplit + s] = w;
                                den = fmaf(w, __ldcg(a.part_ml + (base + s) * 2 + 1), den);
                            }
                            den = warp_sum(den);
                            if (lane == 0) cden[h] = den;
                        }
                        pk_named_sync();
                        constexpr int D4 = D / 4;
                        for (int i = tid; i < n_rep * D4; i += kPkConsumers) {
                            const int h = i / D4, c4 = i % D4;
                            const float4* src = reinterpret_cast<const float4*>(a.part_acc + (size_t)(kvh * n_rep + h) * a.nsplit * D) + c4;
                            float4 num = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
                            for (int s = 0; s < a.nsplit; ++s) {
                                const float w = cm[h * a.nsplit + s];
                                if (w != 0.f) {
                                    const float4 v = __ldcg(src + (size_t)s * D4);
                                    num.x = fmaf(w, v.x, num.x); num.y = fmaf(w, v.y, num.y); num.z = fmaf(w, v.z, num.z); num.w = fmaf(w, v.w, num.w);
                                }
                            }
                            const float den = cden[h];
                            uint32_t h0, l0, h1, l1;
                            split2(num.x / den, num.y / den, h0, l0);
                            split2(num.z / den, num.w / den, h1, l1);
                            const size_t oi = (size_t)(kvh * n_rep + h) * D + c4 * 4;
                            *reinterpret_cast<uint2*>(a.xhl + oi) = make_uint2(h0, h1);
                            *reinterpret_cast<uint2*>(a.xhl + nq + oi) = make_uint2(l0, l1);
                        }
                        if (tid == 0) a.counters[kvh] = 0;
                    }
                    pk_named_sync();
                }
            }
            stamp(l);
            pk_grid_barrier(a.gbar, epoch, tid);
            stamp(l);

            // ---------------- P3: o_proj + residual add ----------------
            prefetch_vec(l + 1 < a.L ? a.layers[l + 1].ln1 : a.final_norm, a.H);   // needed by the next P1 / the head
            load_x_plain(a.xhl, nq);
            stamp(l);
            {
                const int nslots = consume(nq);
                stamp(l);
                if (a.tp > 1) {
                    allreduce_resid_add(nslots);
                } else {
                    for (int e = tid; e < nslots * (kPkBlockRows / 2); e += kPkConsumers) {
                        float2* p = reinterpret_cast<float2*>(a.resid + grow(2 * e));
                        float2 v = __ldcg(p);
                        v.x += row_sum(2 * e);
                        v.y += row_sum(2 * e + 1);
                        *p = v;
                    }
                }
            }
            stamp(l);
            pk_grid_barrier(a.gbar, epoch, tid);
            if (cta == 0 && tid == 0 && a.pool != nullptr) atomicExch(a.pool + (4 * l + 1), 0u);      // every producer is past this phase: re-arm its pool
            stamp(l);

            // ---------------- P4: RMSNorm -> gate|up -> SiLU(gate) * up ----------------
            load_x_rmsnorm(a.resid, false, nullptr, lw.ln2, a.H, nullptr);
            stamp(l);
            {
                long long t0c = 0;
                if (a.dbg != nullptr && tid == 0 && l == a.L / 2) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0c));
                const int nslots = consume(a.H);
                if (a.dbg != nullptr && tid == 0 && l == a.L / 2) {
                    long long t1c;
                    unsigned int smid;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1c));
                    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
                    a.dbg[64 + cta * 4] = t0c; a.dbg[64 + cta * 4 + 1] = t1c; a.dbg[64 + cta * 4 + 2] = smid; a.dbg[64 + cta * 4 + 3] = nslots;
                }
                stamp(l);
                for (int e = tid; e < nslots * (kPkBlockRows / 2); e += kPkConsumers) {
                    const float g = row_sum(2 * e), u = row_sum(2 * e + 1);
                    const float av = g / (1.f + expf(-g)) * u;
                    uint16_t ah, al;
                    split_hi_lo(av, ah, al);
                    const int aj = grow(2 * e) >> 1;
                    a.xhl[2 * nq + aj] = ah;
                    a.xhl[2 * nq + a.I + aj] = al;
                }
            }
            stamp(l);
            pk_grid_barrier(a.gbar, epoch, tid);
            if (cta == 0 && tid == 0 && a.pool != nullptr) atomicExch(a.pool + (4 * l + 2), 0u);      // every producer is past this phase: re-arm its pool
            stamp(l);

            // ---------------- P5: down_proj + residual add ----------------
            load_x_plain(a.xhl + 2 * nq, a.I);
            stamp(l);
            {
                const int nslots = consume(a.I);
                stamp(l);
                if (a.tp > 1) {
                    allreduce_resid_add(nslots);
                } else {
                    for (int e = tid; e < nslots * (kPkBlockRows / 2); e += kPkConsumers) {
                        float2* p = reinterpret_cast<float2*>(a.resid + grow(2 * e));
                        float2 v = __ldcg(p);
                        v.x += row_sum(2 * e);
                        v.y += row_sum(2 * e + 1);
                        *p = v;
                    }
                }
            }
            stamp(l);
            pk_grid_barrier(a.gbar, epoch, tid);
            if (cta == 0 && tid == 0 && a.pool != nullptr) atomicExch(a.pool + (4 * l + 3), 0u);      // every producer is past this phase: re-arm its pool
            stamp(l);
        }

        // ---------------- final RMSNorm -> lm_head -> f32 logits + arg-max (last index wins ties) ----------------
        load_x_rmsnorm(a.resid, false, nullptr, a.final_norm, a.H, nullptr);
        {
            const int nslots = consume(a.H);
            float bv = -INFINITY;
            int bi = -1;
            for (int e = tid; e < nslots * (kPkBlockRows / 2); e += kPkConsumers) {
                const int ra = a.rank * a.V + grow(2 * e);      // index in the FULL vocabulary (vocab-parallel head)
                const float va = row_sum(2 * e), vb = row_sum(2 * e + 1);
                if (a.tp > 1) {
                    for (int r = 0; r < a.tp; ++r) *reinterpret_cast<float2*>(a.peer_logits[r] + ra) = make_float2(va, vb);
                } else {
                    *reinterpret_cast<float2*>(a.logits + ra) = make_float2(va, vb);
                }
                if (va >= bv) { bv = va; bi = ra; }
                if (vb >= bv) { bv = vb; bi = ra + 1; }
            }
            if (a.tp > 1) __threadfence_system();
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(0xFFFFFFFFu, bv, o);
                const int oi = __shfl_xor_sync(0xFFFFFFFFu, bi, o);
                if (ov > bv || (ov == bv && oi > bi)) { bv = ov; bi = oi; }
            }
            if (lane == 0) { red[warp] = bv; reinterpret_cast<int*>(red)[8 + warp] = bi; }
            pk_named_sync();
            if (tid == 0) {
                for (int w = 1; w < kPkConsumerWarps; ++w) {
                    const float ov = red[w];
                    const int oi = reinterpret_cast<int*>(red)[8 + w];
                    if (ov > bv || (ov == bv && oi > bi)) { bv = ov; bi = oi; }
                }
                a.amax_val[cta] = bv;
                a.amax_idx[cta] = bi;
            }
        }
        pk_grid_barrier(a.gbar, epoch, tid);
        if (cta == 0 && tid == 0 && a.pool != nullptr) atomicExch(a.pool + (4 * a.L), 0u);      // every producer is past this phase: re-arm its pool
        if (a.tp > 1) ar_epoch += 1;      // the arg-max exchange below is exchange number 2L+1 of the step (uniform in every thread)
        if (cta == 0 && warp == 0) {
            float bv = -INFINITY;
            int bi = -1;
            for (int p = lane; p < ncta; p += 32) {
                const float ov = __ldcg(a.amax_val + p);
                const int oi = __ldcg(a.amax_idx + p);
                if (ov > bv || (ov == bv && oi > bi)) { bv = ov; bi = oi; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(0xFFFFFFFFu, bv, o);
                const int oi = __shfl_xor_sync(0xFFFFFFFFu, bi, o);
                if (ov > bv || (ov == bv && oi > bi)) { bv = ov; bi = oi; }
            }
            if (a.tp > 1) {   // exchange the per-rank winners (and, by cumulativity, make every rank's logits slice visible)
                if (lane == 0) {
                    for (int r = 0; r < a.tp; ++r) {
                        a.peer_amax[r][a.rank * 2] = bv;
                        a.peer_amax[r][a.rank * 2 + 1] = __int_as_float(bi);
                    }
                    __threadfence_system();
                }
                __syncwarp();
                if (lane < a.tp) {
                    st_release_sys(a.peer_flag[lane] + (size_t)a.rank * (ncta + 1) + ncta, ar_epoch);
                    pk_wait_flag(a.peer_flag[a.rank] + (size_t)lane * (ncta + 1) + ncta, ar_epoch, a.comm_err);
                }
                __syncwarp();
                bv = -INFINITY;
                bi = -1;
                for (int r = 0; r < a.tp; ++r) {
                    const float ov = __ldcg(a.peer_amax[a.rank] + r * 2);
                    const int oi = __float_as_int(__ldcg(a.peer_amax[a.rank] + r * 2 + 1));
                    if (ov > bv || (ov == bv && oi > bi)) { bv = ov; bi = oi; }
                }
            }
            if (lane == 0) {
                a.next_ids[0] = (uint32_t)bi;
                a.state->kv_base[0] = kv_base + 1;
                if (a.feedback) {
                    a.ids[0] = (uint32_t)bi;
                    a.state->rope_pos = rope_pos + 1;
                    if (a.trace != nullptr) {
                        const int tp = *a.trace_pos;
                        a.trace[tp] = (uint32_t)bi;
                        *a.trace_pos = tp + 1;
                    }
                }
            }
        }
        if (step + 1 < a.nsteps) pk_grid_barrier(a.gbar, epoch, tid);
    }
}

}  // namespace fl
