// fastllm_b200: C-ABI entry points + causal-LM decode/prefill orchestration (sm_100a).
// See include/fastllm_b200.h for the reference interface each entry point replaces.
#include <cmath>
#include <sstream>
#include <thread>

#include "attn_decode.cuh"
#include "attn_mma.cuh"
#include "comm.cuh"
#include "decode_persistent.cuh"
#include "dense_ops.cuh"
#include "gemm_tc.cuh"
#include "elementwise.cuh"
#include "gemv.cuh"
#include "model.cuh"
#include "sampler.hpp"
#include "synth.cuh"

namespace fl {

thread_local std::string g_last_error;
std::atomic<uint64_t> g_launches{0};
Profiler g_prof;
NcclApi g_nccl;
PeerComm g_peer;
static std::atomic<int> g_device{-1};

static float host_f16_to_f32(uint16_t h) {
    const uint32_t sign = (uint32_t)(h >> 15) << 31;
    int exp = (h >> 10) & 0x1F;
    uint32_t man = h & 0x3FF;
    uint32_t bits;
    if (exp == 0) {
        if (man == 0) {
            bits = sign;
        } else {
            exp = 1;
            while (!(man & 0x400)) { man <<= 1; --exp; }
            man &= 0x3FF;
            bits = sign | ((uint32_t)(exp + 112) << 23) | (man << 13);
        }
    } else if (exp == 31) {
        bits = sign | 0x7F800000u | (man << 13);
    } else {
        bits = sign | ((uint32_t)(exp + 112) << 23) | (man << 13);
    }
    float f;
    std::memcpy(&f, &bits, 4);
    return f;
}

// Calls f(std::integral_constant<int, D>{}) for head size d: the one place a runtime head_dim becomes the kernels' template
// parameter D.  (Kernels built for 64 / 128 only are guarded with `if constexpr` at the call.)
template <typename F>
static decltype(auto) with_head_dim(int d, F&& f) {
    switch (d) {
        case 16: return f(std::integral_constant<int, 16>{});
        case 32: return f(std::integral_constant<int, 32>{});
        case 64: return f(std::integral_constant<int, 64>{});
        case 128: return f(std::integral_constant<int, 128>{});
    }
    throw Error(FL_ERR_UNSUPPORTED, "head_dim must be 16, 32, 64 or 128");
}

// The same for the N tile (activation rows) of the swap-AB GEMMs.
template <typename F>
static decltype(auto) with_tile_n(int bn, F&& f) {
    switch (bn) {
        case 16: return f(std::integral_constant<int, 16>{});
        case 32: return f(std::integral_constant<int, 32>{});
        case 64: return f(std::integral_constant<int, 64>{});
        case 128: return f(std::integral_constant<int, 128>{});
    }
    throw Error(FL_ERR_INVALID, "internal: GEMM N tile must be 16, 32, 64 or 128");
}

// ------------------------------------------------------------------------------------------------------------------
// GEMV dispatch
// ------------------------------------------------------------------------------------------------------------------
struct GemvPlan {
    int cpt, threads, grid;
};

static GemvPlan plan_gemv(int N, int K) {
    FL_CHECK(K % 8 == 0 && N % 2 == 0, FL_ERR_INVALID, "GEMV needs K % 8 == 0 and N % 2 == 0");
    const int K8 = K / 8;
    GemvPlan p;
    p.cpt = (K8 + 511) / 512;
    FL_CHECK(p.cpt <= 5, FL_ERR_UNSUPPORTED, "GEMV K too large (K <= 20480)");
    p.threads = (int)align_up((size_t)(K8 + p.cpt - 1) / p.cpt, 32);
    int cps = 512 / p.threads;   // CTAs per SM so that 512 threads stream on every SM
    if (cps < 1) cps = 1;
    if (cps > 4) cps = 4;
    p.grid = kNumSMs * cps;
    if (p.grid > N / 2) p.grid = N / 2;
    return p;
}

template <int M, int PRO, int EPI>
static void launch_gemv_cpt(LaunchCtx& lc, const char* tag, const GemvPlan& p, const GemvArgs& a) {
    const uint64_t bytes = (uint64_t)a.N * a.K * 2;
    dim3 g(p.grid), b(p.threads);
    switch (p.cpt) {
        case 1: launch(lc, tag, bytes, gemv_kernel<M, 1, PRO, EPI>, g, b, 0, a); break;
        case 2: launch(lc, tag, bytes, gemv_kernel<M, 2, PRO, EPI>, g, b, 0, a); break;
        case 3: launch(lc, tag, bytes, gemv_kernel<M, 3, PRO, EPI>, g, b, 0, a); break;
        case 4: launch(lc, tag, bytes, gemv_kernel<M, 4, PRO, EPI>, g, b, 0, a); break;
        default: launch(lc, tag, bytes, gemv_kernel<M, 5, PRO, EPI>, g, b, 0, a); break;
    }
}

template <int PRO, int EPI>
static void launch_gemv(LaunchCtx& lc, const char* tag, int M, const GemvPlan& p, const GemvArgs& a) {
    if (M == 1)
        launch_gemv_cpt<1, PRO, EPI>(lc, tag, p, a);
    else
        launch_gemv_cpt<2, PRO, EPI>(lc, tag, p, a);
}

static size_t attn_smem_bytes(int d, int n_rep) {
    const size_t ring = (size_t)4 * kKvPage * d * 2;
    const size_t red = (size_t)1024 * n_rep * 4;
    return ring > red ? ring : red;
}

static void launch_attn(LaunchCtx& lc, int d, int nsplit, int nkv, int rows, size_t smem, uint64_t bytes, const AttnArgs& a) {
    with_head_dim(d, [&](auto D) {
        launch(lc, "attn_decode", bytes, attn_decode_kernel<D>, dim3(nsplit, nkv, rows), dim3(kAttnThreads), smem, a);
    });
}

// mma.sync prefill attention of the dense path (attn_prefill_kernel, attn_mma.cuh): one CTA per 64-query tile x q head x sequence,
// for the multi-token calls that the tcgen05 kernel (attn_prefill_tc_kernel) does not take
static size_t attn_prefill_smem_bytes(int d) {
    return (size_t)(2 * kPrefillBM + 4 * kKvPage) * d * 2;
}

// stream-K batched decode (attn_sk_decode_kernel): q tiles / merge scratch in front, then the K|V ring
static size_t attn_sk_smem_bytes(int d, int n_rep) {
    const size_t front = std::max<size_t>((size_t)2 * 16 * d * 2, (size_t)kSkConsumerWarps * n_rep * d * 4);
    return ((front + 1023) & ~(size_t)1023) + (size_t)kSkStages * 2 * kKvPage * d * 2;
}
struct SkPlan { int ctas = 0; size_t smem = 0; };
// resident CTAs per SM: 3, capped by the runtime's occupancy answer (the ring depth and why: kSkStages in attn_mma.cuh)
template <int D>
static SkPlan attn_sk_plan(int n_rep) {
    static std::map<int, SkPlan> memo;
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    auto it = memo.find(n_rep);
    if (it != memo.end()) return it->second;
    SkPlan p;
    p.smem = attn_sk_smem_bytes(D, n_rep);
    ensure_smem_optin((const void*)attn_sk_decode_kernel<D>, p.smem);    // the occupancy answer is 0 above the opt-in limit
    int fit = 0;
    FL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, attn_sk_decode_kernel<D>, kSkThreads, p.smem));
    p.ctas = std::min(3, fit);
    FL_CHECK(p.ctas >= 1, FL_ERR_UNSUPPORTED, "stream-K attention does not fit an SM");
    memo[n_rep] = p;
    return p;
}
// ------------------------------------------------------------------------------------------------------------------
// Weights
// ------------------------------------------------------------------------------------------------------------------
static void validate_config(const fl_config& c) {
    FL_CHECK(c.arch >= FL_ARCH_LLAMA && c.arch <= FL_ARCH_BERT, FL_ERR_INVALID, "unknown arch");
    FL_CHECK(c.hidden_size > 0 && c.num_attention_heads > 0 && c.num_hidden_layers > 0 && c.vocab_size > 0 &&
                 c.intermediate_size > 0,
             FL_ERR_INVALID, "config sizes must be positive");
    const int d = c.hidden_size / c.num_attention_heads;
    // the reference panics on these: mistral.rs:109-127, models/config.rs:20-54
    FL_CHECK(d * c.num_attention_heads == c.hidden_size, FL_ERR_INVALID, "hidden_size must be divisible by num_attention_heads");
    FL_CHECK(d % 2 == 0, FL_ERR_INVALID, "head_dim must be even for RoPE embeddings");
    const int nkv = c.num_key_value_heads > 0 ? c.num_key_value_heads : c.num_attention_heads;
    if (c.arch == FL_ARCH_BERT) return;   // remaining checks are causal-LM specific; bert_build has its own
    FL_CHECK(c.num_attention_heads % nkv == 0, FL_ERR_INVALID, "num_attention_heads must be divisible by num_key_value_heads");
    FL_CHECK(c.num_attention_heads / nkv <= kAttnMaxRep, FL_ERR_UNSUPPORTED, "GQA group size > 8 not supported");
    FL_CHECK(c.hidden_size % 8 == 0 && c.intermediate_size % 8 == 0, FL_ERR_UNSUPPORTED, "hidden/intermediate size must be a multiple of 8");
    FL_CHECK(c.max_position_embeddings > 0, FL_ERR_INVALID, "max_position_embeddings must be positive");
}

static void build_weights(Weights& w) {
    const fl_config& c = w.cfg;
    const int nh_f = c.num_attention_heads, nkv_f = c.num_key_value_heads > 0 ? c.num_key_value_heads : c.num_attention_heads;
    const bool moe = c.arch == FL_ARCH_MIXTRAL;
    // Mixtral shards by EXPERT (attention, router and head replicated); the dense models shard by tensor
    w.ep = (moe && c.tp_size > 1) ? c.tp_size : 1;
    w.tp = (!moe && c.tp_size > 1) ? c.tp_size : 1;
    w.rank = c.tp_size > 1 ? c.tp_rank : 0;
    if (moe) {
        w.E = c.num_local_experts; w.top_k = c.num_experts_per_tok > 0 ? c.num_experts_per_tok : 2;
        FL_CHECK(w.E >= 1 && w.E <= 64 && w.top_k >= 1 && w.top_k <= 8 && w.top_k <= w.E, FL_ERR_INVALID, "bad Mixtral expert counts");
        FL_CHECK(w.E % w.ep == 0, FL_ERR_UNSUPPORTED, "expert parallelism needs num_local_experts divisible by the world size");
        w.E_local = w.E / w.ep;
        w.ep_dp = w.ep > 1 && c.ep_dp_attention != 0;
    }
    FL_CHECK(w.rank >= 0 && w.rank < std::max(w.tp, w.ep), FL_ERR_INVALID, "tp_rank out of range");
    if (w.tp > 1) {
        // column-parallel q/k/v (by head) and gate/up, row-parallel o_proj and down_proj, vocab-parallel lm_head
        FL_CHECK((nkv_f % w.tp == 0 && nh_f % w.tp == 0) || (w.tp > nkv_f && w.tp % nkv_f == 0), FL_ERR_UNSUPPORTED,
                 "tensor parallelism needs heads and kv heads divisible by tp_size, or tp_size a multiple of the kv heads");
        FL_CHECK(c.intermediate_size % (8 * w.tp) == 0 && c.vocab_size % (2 * w.tp) == 0, FL_ERR_UNSUPPORTED,
                 "tensor parallelism needs intermediate_size % (8 tp) == 0 and vocab_size % (2 tp) == 0");
    }
    w.H = c.hidden_size; w.L = c.num_hidden_layers;
    w.I = c.intermediate_size / w.tp; w.Vfull = c.vocab_size; w.V = c.vocab_size / w.tp;
    const int trank = w.tp > 1 ? w.rank : 0;       // under expert parallelism (tp == 1) the attention weights are replicated
    if (w.tp <= nkv_f) {
        w.nh = nh_f / w.tp; w.nkv = nkv_f / w.tp;
        w.q_head0 = trank * w.nh; w.q_real = w.nh; w.kv_head0 = trank * w.nkv;
    } else {
        // more ranks than kv heads (Qwen2.5-7B at TP-8: 28 q / 4 kv heads): every kv head lives on rep = tp / nkv ranks, and the
        // group's query heads are dealt out ceil(group / rep) per rank; the last rank of a group pads with zero heads
        // (zero q rows and zero o_proj columns contribute nothing)
        const int rep = w.tp / nkv_f, group = nh_f / nkv_f, hpr = (group + rep - 1) / rep;
        const int kvh = trank / rep, sub = trank % rep;
        w.nh = hpr; w.nkv = 1;
        w.q_head0 = kvh * group + sub * hpr;
        w.q_real = std::max(0, std::min(hpr, group - sub * hpr));
        w.kv_head0 = kvh;
    }
    w.d = w.H / nh_f;
    w.max_pos = c.max_position_embeddings;
    w.nqkv = (w.nh + 2 * w.nkv) * w.d;
    with_head_dim(w.d, [](auto) {});
    FL_CHECK(c.arch != FL_ARCH_BERT, FL_ERR_INVALID, "internal: BERT goes through bert_build");

    const size_t A = 256;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, A); return o; };
    const size_t H = w.H, I = w.I, V = w.V, nq = (size_t)w.nh * w.d;
    const size_t o_embed = take((size_t)w.Vfull * H * 2), o_head = take(V * H * 2), o_fnorm = take(H * 4);
    struct LO { size_t wqkv, bqkv, wo, wgu, wdown, ln1, ln2, wgate; std::vector<size_t> ewgu, ewdown; };
    std::vector<LO> lo(w.L);
    for (int l = 0; l < w.L; ++l) {
        lo[l].wqkv = take((size_t)w.nqkv * H * 2);
        lo[l].bqkv = c.qkv_bias ? take((size_t)w.nqkv * 4) : (size_t)-1;
        lo[l].wo = take(H * nq * 2);
        if (moe) {
            lo[l].wgate = take((size_t)w.E * H * 4);
            // a layer's w1|w3 matrices back to back, then its w2 matrices back to back: each set is also ONE stacked matrix
            // ([E_local * 2I, H] / [E_local * H, I]), the A operand of the grouped expert GEMMs
            const size_t gu0 = take((size_t)w.E_local * 2 * I * H * 2), dn0 = take((size_t)w.E_local * H * I * 2);
            for (int e = 0; e < w.E_local; ++e) {
                lo[l].ewgu.push_back(gu0 + (size_t)e * 2 * I * H * 2);
                lo[l].ewdown.push_back(dn0 + (size_t)e * H * I * 2);
            }
            lo[l].wgu = lo[l].wdown = 0;
        } else {
            lo[l].wgu = take(2 * I * H * 2);
            lo[l].wdown = take(H * I * 2);
        }
        lo[l].ln1 = take(H * 4);
        lo[l].ln2 = take(H * 4);
    }
    const size_t o_cos = take((size_t)w.max_pos * (w.d / 2) * 4), o_sin = take((size_t)w.max_pos * (w.d / 2) * 4);
    w.slab.alloc(off, /*zero=*/true);
    uint8_t* base = w.slab.p;
    w.embed = (uint16_t*)(base + o_embed);
    w.lm_head = (uint16_t*)(base + o_head);
    w.final_norm = (float*)(base + o_fnorm);
    w.layers.resize(w.L);
    for (int l = 0; l < w.L; ++l) {
        w.layers[l].wqkv = (uint16_t*)(base + lo[l].wqkv);
        w.layers[l].bqkv = c.qkv_bias ? (float*)(base + lo[l].bqkv) : nullptr;
        w.layers[l].wo = (uint16_t*)(base + lo[l].wo);
        if (moe) {
            w.layers[l].wgate = (float*)(base + lo[l].wgate);
            for (int e = 0; e < w.E_local; ++e) {
                w.layers[l].ewgu.push_back((uint16_t*)(base + lo[l].ewgu[e]));
                w.layers[l].ewdown.push_back((uint16_t*)(base + lo[l].ewdown[e]));
            }
        } else {
            w.layers[l].wgu = (uint16_t*)(base + lo[l].wgu);
            w.layers[l].wdown = (uint16_t*)(base + lo[l].wdown);
        }
        w.layers[l].ln1 = (float*)(base + lo[l].ln1);
        w.layers[l].ln2 = (float*)(base + lo[l].ln2);
    }
    w.rope_cos = (float*)(base + o_cos);
    w.rope_sin = (float*)(base + o_sin);
    // bytes one decode step must stream: every parameter except the embedding table (SURVEY.md section 8d)
    const uint64_t mlp = moe ? (uint64_t)w.E_local * 3 * I * H : 3 * I * H;     // every local expert is streamed each step
    w.streamed_bytes = 2 * ((uint64_t)w.L * ((uint64_t)w.nqkv * H + H * nq + mlp) + V * H) +
                       4 * ((uint64_t)w.L * (2 * H + (c.qkv_bias ? w.nqkv : 0) + (moe ? (uint64_t)w.E * H : 0)) + H);
}

struct TensorRoute {
    enum Kind { BF16_MAT, F32_VEC } kind;
    void* base;
    int64_t rows, cols;             // LOCAL block held by this rank ([rows, cols] or [rows])
    int64_t ld;                     // leading dimension of the local matrix in elements (>= cols; > cols: zero-padded heads)
    RowMap map;
    int64_t full_rows, full_cols;   // shape the caller hands over (the full HF tensor)
    int64_t src_row0, src_col0;     // window of the full tensor this rank keeps
};

static bool route_tensor(Weights& w, const std::string& name, TensorRoute& r) {
    const int64_t H = w.H, I = w.I, d = w.d, nq = (int64_t)w.nh * d, nk = (int64_t)w.nkv * d, tp = w.tp,
                  rk = w.tp > 1 ? w.rank : 0;   // under expert parallelism (tp == 1) every dense tensor is replicated
    // row-sharded matrix: local rows [rk*rows, (rk+1)*rows) of a [tp*rows, cols] tensor; col-sharded: the same along columns
    auto mat_rows = [&](uint16_t* base, int64_t rows, int64_t cols, RowMap m, bool sharded) {
        r = {TensorRoute::BF16_MAT, base, rows, cols, cols, m, sharded ? rows * tp : rows, cols, sharded ? rk * rows : 0, 0};
        return true;
    };
    auto mat_cols = [&](uint16_t* base, int64_t rows, int64_t cols, RowMap m) {
        r = {TensorRoute::BF16_MAT, base, rows, cols, cols, m, rows, cols * tp, 0, rk * cols};
        return true;
    };
    auto vec = [&](float* base, int64_t rows, RowMap m, bool sharded) {
        r = {TensorRoute::F32_VEC, base, rows, 1, 1, m, sharded ? rows * tp : rows, 1, sharded ? rk * rows : 0, 0};
        return true;
    };
    // attention projections: head windows of the full tensors (w.q_head0 / w.q_real / w.kv_head0, see build_weights)
    const int64_t nh_f = w.cfg.num_attention_heads, nkv_f = w.cfg.num_key_value_heads > 0 ? w.cfg.num_key_value_heads : nh_f;
    const int64_t qreal = (int64_t)w.q_real * d, q0 = (int64_t)w.q_head0 * d, k0 = (int64_t)w.kv_head0 * d;
    auto head_rows = [&](uint16_t* base, int64_t rows, RowMap m, int64_t full_heads, int64_t row0) {
        r = {TensorRoute::BF16_MAT, base, rows, H, H, m, full_heads * d, H, row0, 0};
        return true;
    };
    auto head_vec = [&](float* base, int64_t rows, RowMap m, int64_t full_heads, int64_t row0) {
        r = {TensorRoute::F32_VEC, base, rows, 1, 1, m, full_heads * d, 1, row0, 0};
        return true;
    };
    const RowMap ident{0, 0, 0, 0};
    if (name == "model.embed_tokens.weight") return mat_rows(w.embed, w.Vfull, H, ident, false);
    if (name == "lm_head.weight") return mat_rows(w.lm_head, w.V, H, ident, true);
    if (name == "model.norm.weight") return vec(w.final_norm, H, ident, false);
    const std::string pre = "model.layers.";
    if (name.compare(0, pre.size(), pre) != 0) return false;
    size_t dot = name.find('.', pre.size());
    if (dot == std::string::npos) return false;
    int li = -1;
    try { li = std::stoi(name.substr(pre.size(), dot - pre.size())); } catch (...) { return false; }
    if (li < 0 || li >= w.L) return false;
    LayerW& lw = w.layers[li];
    const std::string rest = name.substr(dot + 1);
    const RowMap ropeq{0, 1, (int32_t)d, 0}, ropek{nq, 1, (int32_t)d, 0}, vmap{nq + nk, 0, 0, 0};
    if (rest == "input_layernorm.weight") return vec(lw.ln1, H, ident, false);
    if (rest == "post_attention_layernorm.weight") return vec(lw.ln2, H, ident, false);
    if (rest == "self_attn.q_proj.weight") return head_rows(lw.wqkv, qreal, ropeq, nh_f, q0);
    if (rest == "self_attn.k_proj.weight") return head_rows(lw.wqkv, nk, ropek, nkv_f, k0);
    if (rest == "self_attn.v_proj.weight") return head_rows(lw.wqkv, nk, vmap, nkv_f, k0);
    if (w.cfg.qkv_bias) {
        if (rest == "self_attn.q_proj.bias") return head_vec(lw.bqkv, qreal, ropeq, nh_f, q0);
        if (rest == "self_attn.k_proj.bias") return head_vec(lw.bqkv, nk, ropek, nkv_f, k0);
        if (rest == "self_attn.v_proj.bias") return head_vec(lw.bqkv, nk, vmap, nkv_f, k0);
    }
    if (rest == "self_attn.o_proj.weight") {
        r = {TensorRoute::BF16_MAT, lw.wo, H, qreal, nq, ident, H, nh_f * d, 0, q0};
        return true;
    }
    if (w.cfg.arch == FL_ARCH_MIXTRAL) {
        if (rest == "block_sparse_moe.gate.weight") return vec(lw.wgate, (int64_t)w.E * H, ident, false);   // [E, H] kept in f32
        const std::string ep = "block_sparse_moe.experts.";
        if (rest.compare(0, ep.size(), ep) != 0) return false;
        const size_t d2 = rest.find('.', ep.size());
        if (d2 == std::string::npos) return false;
        int e = -1;
        try { e = std::stoi(rest.substr(ep.size(), d2 - ep.size())); } catch (...) { return false; }
        if (e < 0 || e >= w.E) return false;
        const std::string tail = rest.substr(d2 + 1);
        const int el = e - w.rank * w.E_local;                  // local slot, or outside this rank's range
        const bool mine = el >= 0 && el < w.E_local;
        uint16_t* gu = mine ? lw.ewgu[el] : nullptr;
        uint16_t* dn = mine ? lw.ewdown[el] : nullptr;
        bool ok = false;
        if (tail == "w1.weight") ok = mat_rows(gu, I, H, RowMap{0, 2, 0, 0}, false);
        else if (tail == "w3.weight") ok = mat_rows(gu, I, H, RowMap{0, 2, 0, 1}, false);
        else if (tail == "w2.weight") ok = mat_rows(dn, H, I, ident, false);
        return ok;      // r.base == nullptr: a valid tensor that belongs to another expert-parallel rank
    }
    if (rest == "mlp.gate_proj.weight") return mat_rows(lw.wgu, I, H, RowMap{0, 2, 0, 0}, true);
    if (rest == "mlp.up_proj.weight") return mat_rows(lw.wgu, I, H, RowMap{0, 2, 0, 1}, true);
    if (rest == "mlp.down_proj.weight") return mat_cols(lw.wdown, H, I, ident);
    return false;
}

static std::vector<std::string> expected_tensors(const Weights& w) {
    std::vector<std::string> v = {"model.embed_tokens.weight", "model.norm.weight"};
    for (int l = 0; l < w.L; ++l) {
        const std::string p = "model.layers." + std::to_string(l) + ".";
        for (const char* s : {"input_layernorm.weight", "post_attention_layernorm.weight", "self_attn.q_proj.weight",
                              "self_attn.k_proj.weight", "self_attn.v_proj.weight", "self_attn.o_proj.weight"})
            v.push_back(p + s);
        if (w.cfg.arch == FL_ARCH_MIXTRAL) {
            v.push_back(p + "block_sparse_moe.gate.weight");
            for (int e = w.rank * w.E_local; e < (w.rank + 1) * w.E_local; ++e)
                for (const char* s : {"w1.weight", "w2.weight", "w3.weight"})
                    v.push_back(p + "block_sparse_moe.experts." + std::to_string(e) + "." + s);
        } else {
            for (const char* s : {"mlp.gate_proj.weight", "mlp.up_proj.weight", "mlp.down_proj.weight"}) v.push_back(p + s);
        }
        if (w.cfg.qkv_bias)
            for (const char* s : {"self_attn.q_proj.bias", "self_attn.k_proj.bias", "self_attn.v_proj.bias"}) v.push_back(p + s);
    }
    return v;
}

static void put_tensor(Weights& w, const char* name, int dtype, const int64_t* shape, int rank, const void* host) {
    FL_CHECK(!w.finalized, FL_ERR_STATE, "model already finalized");
    TensorRoute r;
    // Names the model does not read are skipped, as candle's VarBuilder ignores the extra entries of the HashMap the loader hands
    // over (huggingface.rs:81-130 loads EVERY tensor of the checkpoint: `self_attn.rotary_emb.inv_freq` in older Llama exports,
    // `visual.*` in Qwen2_5_VLForConditionalGeneration, ...).  finalize() stays the strict gate: a MISSING tensor is an error.
    if (!route_tensor(w, name, r)) return;
    if (r.base == nullptr) return;       // an expert that lives on another expert-parallel rank
    int64_t numel = 1;
    for (int i = 0; i < rank; ++i) numel *= shape[i];
    const bool shape_ok = (r.kind == TensorRoute::BF16_MAT) ? (rank == 2 && shape[0] == r.full_rows && shape[1] == r.full_cols)
                                                            : ((rank == 1 && shape[0] == r.full_rows) || (rank == 2 && shape[0] * shape[1] == r.full_rows));
    FL_CHECK(shape_ok, FL_ERR_INVALID, std::string("shape mismatch for ") + name);
    FL_CHECK(dtype == FL_DTYPE_F32 || dtype == FL_DTYPE_BF16 || dtype == FL_DTYPE_F16, FL_ERR_INVALID, "bad dtype");
    // keep this rank's window of the full tensor, converted to bf16 bit patterns (round-to-nearest-even), the dtype the
    // reference server loads into (main.rs:120)
    numel = r.rows * r.cols;
    std::vector<uint16_t> bits((size_t)numel);
    for (int64_t lr = 0; lr < r.rows; ++lr) {
        const int64_t src = (lr + r.src_row0) * r.full_cols + r.src_col0;
        uint16_t* dstp = bits.data() + (size_t)lr * r.cols;
        if (dtype == FL_DTYPE_BF16) {
            std::memcpy(dstp, (const uint16_t*)host + src, (size_t)r.cols * 2);
        } else if (dtype == FL_DTYPE_F32) {
            const float* f = (const float*)host + src;
            for (int64_t i = 0; i < r.cols; ++i) dstp[i] = host_f32_to_bf16(f[i]);
        } else {
            const uint16_t* h = (const uint16_t*)host + src;
            for (int64_t i = 0; i < r.cols; ++i) dstp[i] = host_f32_to_bf16(host_f16_to_f32(h[i]));
        }
    }
    if (r.kind == TensorRoute::BF16_MAT) {
        uint16_t* dst = (uint16_t*)r.base;
        const size_t rowb = (size_t)r.cols * 2;
        if (numel == 0) {
            // a rank that holds only padding heads of this tensor
        } else if (r.map.mode == 0) {
            FL_CUDA(cudaMemcpy2D(dst + r.map.dst_row0 * r.ld, (size_t)r.ld * 2, bits.data(), rowb, rowb, (size_t)r.rows, cudaMemcpyHostToDevice));
        } else if (r.map.mode == 2) {
            FL_CUDA(cudaMemcpy2D(dst + (size_t)r.map.lane * r.cols, 2 * rowb, bits.data(), rowb, rowb, (size_t)r.rows,
                                 cudaMemcpyHostToDevice));
        } else {
            std::vector<uint16_t> perm((size_t)numel);
            for (int64_t row = 0; row < r.rows; ++row)
                std::memcpy(perm.data() + (size_t)(r.map.map(row) - r.map.dst_row0) * r.cols, bits.data() + (size_t)row * r.cols, rowb);
            FL_CUDA(cudaMemcpy(dst + r.map.dst_row0 * r.cols, perm.data(), (size_t)numel * 2, cudaMemcpyHostToDevice));
        }
    } else {
        std::vector<float> vals((size_t)r.rows);
        for (int64_t row = 0; row < r.rows; ++row) {
            const uint32_t b = (uint32_t)bits[row] << 16;
            float f;
            std::memcpy(&f, &b, 4);
            vals[(size_t)(r.map.map(row) - r.map.dst_row0)] = f;
        }
        FL_CUDA(cudaMemcpy((float*)r.base + r.map.dst_row0, vals.data(), (size_t)r.rows * 4, cudaMemcpyHostToDevice));
    }
    w.have.insert(name);
    if (std::string(name) == "lm_head.weight") w.lm_head_loaded = true;
}

static void random_init(Weights& w, uint64_t seed, float stdv) {
    FL_CHECK(!w.finalized, FL_ERR_STATE, "model already finalized");
    std::vector<std::string> names = expected_tensors(w);
    names.push_back("lm_head.weight");
    for (const std::string& n : names) {
        TensorRoute r;
        FL_CHECK(route_tensor(w, n, r), FL_ERR_INVALID, "internal: unroutable " + n);
        const bool is_norm = n.size() >= 11 && n.compare(n.size() - 11, 11, "norm.weight") == 0;
        const uint64_t ts = tensor_seed(seed, n.c_str());
        if (r.kind == TensorRoute::BF16_MAT) {
            synth_fill_bf16_kernel<<<kNumSMs * 8, 256>>>((uint16_t*)r.base, r.rows, r.cols, r.ld, ts, stdv, r.map,
                                                         SrcWin{r.src_row0, r.src_col0, r.full_cols});
        } else if (is_norm) {
            fill_f32_kernel<<<8, 256>>>((float*)r.base, r.rows, 1.0f);
        } else {
            synth_fill_f32_kernel<<<8, 256>>>((float*)r.base, r.rows, ts, stdv, r.map, r.src_row0);
        }
        g_launches.fetch_add(1);
        w.have.insert(n);
    }
    w.lm_head_loaded = true;
    FL_CUDA(cudaGetLastError());
    FL_CUDA(cudaDeviceSynchronize());
}

static void finalize(Weights& w) {
    FL_CHECK(!w.finalized, FL_ERR_STATE, "model already finalized");
    for (const std::string& n : expected_tensors(w))
        FL_CHECK(w.have.count(n), FL_ERR_STATE, "missing tensor: " + n);
    if (!w.lm_head_loaded) w.lm_head = w.embed;   // candle qwen2: tied embeddings when lm_head.weight is absent
    // RoPE tables (see oracle/candle_ops.py rope_tables for the candle rule being followed)
    const int half = w.d / 2;
    std::vector<float> cs((size_t)w.max_pos * half), sn((size_t)w.max_pos * half);
    std::vector<float> inv(half);
    for (int i = 0; i < half; ++i) {
        float p;
        if (w.cfg.arch == FL_ARCH_LLAMA) {
            const float e = (float)(2 * i) / (float)w.d;
            p = (float)std::pow((double)(float)w.cfg.rope_theta, (double)e);
        } else {
            p = (float)std::pow(w.cfg.rope_theta, (double)(2 * i) / (double)w.d);
        }
        inv[i] = 1.0f / p;
    }
    for (int pos = 0; pos < w.max_pos; ++pos)
        for (int i = 0; i < half; ++i) {
            const float f = (float)pos * inv[i];
            cs[(size_t)pos * half + i] = (float)std::cos((double)f);
            sn[(size_t)pos * half + i] = (float)std::sin((double)f);
        }
    FL_CUDA(cudaMemcpy(w.rope_cos, cs.data(), cs.size() * 4, cudaMemcpyHostToDevice));
    FL_CUDA(cudaMemcpy(w.rope_sin, sn.data(), sn.size() * 4, cudaMemcpyHostToDevice));
    w.dense_ok = !env_flag("FL_NO_DENSE") && (w.nh * w.d) % 8 == 0 && w.H % 8 == 0 && w.I % 8 == 0 && w.nqkv % 4 == 0 && w.V % 4 == 0 && w.H % 4 == 0;
    FL_CHECK(w.dense_ok || w.cfg.arch != FL_ARCH_MIXTRAL, FL_ERR_UNSUPPORTED, "Mixtral runs on the dense path only: shapes must be multiples of 8");
    if (w.dense_ok) {
        const uint64_t nq = (uint64_t)w.nh * w.d;
        for (LayerW& lw : w.layers) {
            lw.tm_wqkv = make_tmap_bf16(lw.wqkv, w.nqkv, w.H, w.H, 128);
            lw.tm_wo = make_tmap_bf16(lw.wo, w.H, nq, nq, 128);
            if (w.cfg.arch == FL_ARCH_MIXTRAL) {
                for (int e = 0; e < w.E_local; ++e) {
                    lw.tm_ewgu.push_back(make_tmap_bf16(lw.ewgu[e], 2 * (uint64_t)w.I, w.H, w.H, 128));
                    lw.tm_ewdown.push_back(make_tmap_bf16(lw.ewdown[e], w.H, w.I, w.I, 128));
                }
                lw.tm_ewgu_all = make_tmap_bf16(lw.ewgu[0], (uint64_t)w.E_local * 2 * w.I, w.H, w.H, 128);
                lw.tm_ewdown_all = make_tmap_bf16(lw.ewdown[0], (uint64_t)w.E_local * w.H, w.I, w.I, 128);
            } else {
                lw.tm_wgu = make_tmap_bf16(lw.wgu, 2 * (uint64_t)w.I, w.H, w.H, 128);
                lw.tm_wdown = make_tmap_bf16(lw.wdown, w.H, w.I, w.I, 128);
            }
        }
        w.tm_head = make_tmap_bf16(w.lm_head, w.V, w.H, w.H, 128);
    }
    std::vector<PkLayer> pk(w.L);
    for (int l = 0; l < w.L; ++l)
        pk[l] = PkLayer{w.layers[l].wqkv, w.layers[l].bqkv, w.layers[l].wo, w.layers[l].wgu, w.layers[l].wdown, w.layers[l].ln1, w.layers[l].ln2};
    w.pk_layers.alloc(w.L);
    FL_CUDA(cudaMemcpy(w.pk_layers.p, pk.data(), pk.size() * sizeof(PkLayer), cudaMemcpyHostToDevice));
    const uint64_t nqk = (uint64_t)w.nh * w.d;
    if (w.cfg.arch != FL_ARCH_MIXTRAL && w.H % 64 == 0 && nqk % 64 == 0 && w.I % 64 == 0) {
        std::vector<CUtensorMap> tm;
        for (int l = 0; l < w.L; ++l) {
            tm.push_back(make_tmap_pk(w.layers[l].wqkv, w.nqkv, w.H));
            tm.push_back(make_tmap_pk(w.layers[l].wo, w.H, nqk));
            tm.push_back(make_tmap_pk(w.layers[l].wgu, 2 * (uint64_t)w.I, w.H));
            tm.push_back(make_tmap_pk(w.layers[l].wdown, w.H, w.I));
        }
        tm.push_back(make_tmap_pk(w.lm_head, w.V, w.H));
        w.pk_tmaps.alloc(tm.size());
        FL_CUDA(cudaMemcpy(w.pk_tmaps.p, tm.data(), tm.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice));
    }
    w.finalized = true;
}

// ------------------------------------------------------------------------------------------------------------------
// Tensor-parallel collectives (NCCL over NVLink 5 / NVSwitch; captured into the CUDA graph with the rest of the step)
// ------------------------------------------------------------------------------------------------------------------
static void tp_allreduce_sum(LaunchCtx& lc, float* buf, size_t count) {
    FL_CHECK(g_nccl.comm != nullptr, FL_ERR_STATE, "tensor parallelism: fl_comm_init has not been called");
    g_nccl.check(g_nccl.AllReduce(buf, buf, count, ncclFloat32, ncclSum, g_nccl.comm, lc.stream), "ncclAllReduce");
    count_launch(lc);
}
static void tp_allgather(LaunchCtx& lc, const float* send, float* recv, size_t count) {
    FL_CHECK(g_nccl.comm != nullptr, FL_ERR_STATE, "tensor parallelism: fl_comm_init has not been called");
    g_nccl.check(g_nccl.AllGather(send, recv, count, ncclFloat32, g_nccl.comm, lc.stream), "ncclAllGather");
    count_launch(lc);
}
// All-to-all over the communicator (grouped ncclSend / ncclRecv, ONE fused NCCL launch for all segments): for every segment,
// rank r receives block `r` of every peer's send buffer into recv[src * bytes ...].  `replicate`: every peer gets the SAME
// block (send holds one block: the expert-parallel dispatch, where a token's row goes to the expert ranks), else send holds
// `world` blocks (the expert-parallel combine, where expert outputs travel back to the rank that owns the sequence).
struct A2aSeg {
    const void* send;
    void* recv;
    size_t bytes;       // per peer
    bool replicate;
};
static void ep_alltoall(LaunchCtx& lc, const A2aSeg* segs, int nseg) {
    FL_CHECK(g_nccl.comm != nullptr, FL_ERR_STATE, "expert parallelism: fl_comm_init has not been called");
    g_nccl.check(g_nccl.GroupStart(), "ncclGroupStart");
    for (int i = 0; i < nseg; ++i) {
        const A2aSeg& sg = segs[i];
        for (int p = 0; p < g_nccl.world; ++p) {
            const uint8_t* sp = (const uint8_t*)sg.send + (sg.replicate ? 0 : (size_t)p * sg.bytes);
            g_nccl.check(g_nccl.Send(sp, sg.bytes, ncclUint8, p, g_nccl.comm, lc.stream), "ncclSend");
            g_nccl.check(g_nccl.Recv((uint8_t*)sg.recv + (size_t)p * sg.bytes, sg.bytes, ncclUint8, p, g_nccl.comm, lc.stream), "ncclRecv");
        }
    }
    g_nccl.check(g_nccl.GroupEnd(), "ncclGroupEnd");
    count_launch(lc);
}

// ------------------------------------------------------------------------------------------------------------------
// Cache + forward
// ------------------------------------------------------------------------------------------------------------------
constexpr int kPassRows = 2;   // activation rows per CUDA-core GEMV pass

// ------------------------------------------------------------------------------------------------------------------
// Persistent batch-1 decode kernel: plan + launch
// ------------------------------------------------------------------------------------------------------------------
static void plan_persistent(fl_cache& c) {
    const Weights& w = *c.w;
    PkPlan& p = c.pk;
    p.ok = false;
    if (env_flag("FL_NO_PERSISTENT")) return;
    // tensor parallelism: the kernel all-reduces over peer-mapped memory, which needs the CUDA-IPC exchange area
    if (w.tp > 1 && (!g_peer.ready || w.H > PeerComm::kMaxH || (size_t)w.Vfull > PeerComm::kMaxVocab || w.tp > PeerComm::kMaxTp)) return;
    if (w.cfg.arch == FL_ARCH_MIXTRAL) return;   // MoE runs on the dense path
    const int nq = w.nh * w.d;
    if (!(w.d == 64 || w.d == 128)) return;
    if (w.H < 2048 || nq < 256 || w.I < 256) return;        // small models stay on the multi-kernel path
    // MMA weight stream: row slices in units of 8 rows, k-steps of 16 columns; the RMSNorm prologue keeps a row in registers
    // whole 16-row blocks in every phase; the RMSNorm prologue keeps a row in registers
    if (w.pk_tmaps.p == nullptr || w.nqkv % 16 || w.H % 16 || (2 * w.I) % 16 || w.V % 16 || w.H > kPkMaxNormK) return;
    // x_hi / x_lo are zero-padded to whole 1024-column chunks (the weight tail of the last chunk is zero-filled by TMA)
    int kmax = (std::max(w.H, std::max(nq, w.I)) + kPkChunkCols - 1) / kPkChunkCols * kPkChunkCols;
    // attention scratch in the same region: [lane groups = 8 warps * 32/(d/8)][4 heads][d] + (m, l) pairs = 8192 + 512 floats,
    // and the split-merge weights [8][nsplit] + 8
    p.xs_floats = (int)align_up((size_t)std::max(std::max(kmax + 16, 8192 + 512), 8 * kNumSMs + 16), 4);
    int slots = 0;      // blocks one CTA can process in a phase: its static share + the pool cap (see pk_split)
    for (int N : {w.nqkv, w.H, 2 * w.I, w.V}) {
        const int nblk = N / kPkBlockRows;
        slots = std::max(slots, w.tp == 1 ? nblk / kNumSMs + kPkPoolCap : (nblk + kNumSMs - 1) / kNumSMs + 1);
    }
    if (slots > kPkMaxSlots) return;
    p.partial_rows = slots * kPkBlockRows;
    const size_t fixed = (size_t)p.xs_floats * 4 + (size_t)p.partial_rows * kPkConsumerWarps * 4 + (size_t)kAttnMaxRep * kKvPage * 4 + 64 * 4;
    const size_t avail = 232448 - 2048;   // 227 KB opt-in limit minus static shared memory and slack
    if (fixed + 2 * (size_t)kPkStageBytes > avail) return;
    p.nstages = (int)std::min<size_t>(kPkMaxStages, (avail - fixed) / kPkStageBytes);
    p.smem = (size_t)p.nstages * kPkStageBytes + fixed;
    p.nsplit = std::max(1, std::min(c.pages_per_seq, kNumSMs / w.nkv));
    if (p.nsplit > c.nsplit) p.nsplit = c.nsplit;            // partial buffers are sized for c.nsplit
    int coop = 0;
    FL_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, w.device));
    if (!coop) return;
    c.gbar.alloc(1, true);
    p.ok = true;
}

// Enqueue `nsteps` batch-1 decode steps as ONE cooperative launch on the cache's stream.
static void launch_persistent(fl_cache& c, int nsteps, bool feedback) {
    const Weights& w = *c.w;
    PkArgs a{};
    a.layers = w.pk_layers.p; a.L = w.L; a.embed = w.embed; a.lm_head = w.lm_head; a.final_norm = w.final_norm;
    a.H = w.H; a.I = w.I; a.V = w.V; a.nh = w.nh; a.nkv = w.nkv; a.d = w.d; a.nqkv = w.nqkv; a.max_pos = w.max_pos;
    a.eps = w.cfg.norm_eps; a.qscale = (float)(1.0 / std::sqrt((double)w.d));
    a.rope_cos = w.rope_cos; a.rope_sin = w.rope_sin;
    a.kpool = c.kpool.p; a.vpool = c.vpool.p; a.layer_pool_elems = c.layer_pool_elems; a.page_table = c.page_table.p;
    a.state = c.state.p; a.resid = c.resid.p; a.q = c.q.p; a.attn_out = c.attn_out.p; a.act = c.act.p; a.logits = c.logits.p;
    a.part_acc = c.part_acc.p; a.part_ml = c.part_ml.p; a.counters = c.counters.p; a.nsplit = c.pk.nsplit;
    a.amax_val = c.amax_val.p; a.amax_idx = c.amax_idx.p; a.ids = c.ids.p; a.next_ids = c.next_ids.p;
    a.trace = feedback ? c.trace.p : nullptr; a.trace_pos = c.trace_pos.p; a.gbar = c.gbar.p;
    a.nsteps = nsteps; a.feedback = feedback ? 1 : 0; a.nstages = c.pk.nstages; a.xs_floats = c.pk.xs_floats;
    a.partial_rows = c.pk.partial_rows;
    if (c.pk_xhl.p == nullptr) c.pk_xhl.alloc(2 * ((size_t)w.nh * w.d + w.I) + 64, true);
    a.xhl = c.pk_xhl.p;
    a.kcap = (std::max(w.H, std::max(w.nh * w.d, w.I)) + kPkChunkCols - 1) / kPkChunkCols * kPkChunkCols;
    a.tmaps = w.pk_tmaps.p;
    if (c.pk_pool.p == nullptr) c.pk_pool.alloc(4 * (size_t)w.L + 1, true);
    a.pool = c.pk_pool.p;
    a.tp = w.tp; a.rank = w.rank;
    if (w.tp > 1) {
        for (int r = 0; r < w.tp; ++r) {
            uint8_t* base = (uint8_t*)g_peer.peer[r];
            a.peer_part[r] = (float*)(base + PeerComm::kPartOff);
            a.peer_flag[r] = (unsigned int*)(base + PeerComm::kFlagOff);
            a.peer_amax[r] = (float*)(base + PeerComm::kAmaxOff);
            a.peer_logits[r] = (float*)(base + PeerComm::kLogitsOff);
        }
        a.comm_err = (int*)((uint8_t*)g_peer.local + PeerComm::kErrOff);
        a.ar_epoch0 = g_peer.ar_epoch;
        g_peer.ar_epoch += (unsigned int)nsteps * (2u * (unsigned int)w.L + 1u);
    }
    static long long* dbg_buf = nullptr;
    const bool dbg = env_flag("FL_PK_DEBUG");
    if (dbg && !dbg_buf) {
        FL_CUDA(cudaMalloc(&dbg_buf, (64 + 4 * kNumSMs + 64) * sizeof(long long)));
        FL_CUDA(cudaMemset(dbg_buf, 0, (64 + 4 * kNumSMs + 64) * sizeof(long long)));
    }
    a.dbg = dbg ? dbg_buf : nullptr;
    FL_CUDA(cudaMemsetAsync(c.gbar.p, 0, sizeof(unsigned int), c.stream));
    FL_CUDA(cudaMemsetAsync(c.pk_pool.p, 0, (4 * (size_t)w.L + 1) * sizeof(unsigned int), c.stream));   // the kernel re-arms them itself; this covers an aborted launch
    LaunchCtx lc{c.stream, /*pdl=*/false};
    lc.cooperative = true;
    const uint64_t bytes = (uint64_t)nsteps * (w.streamed_bytes + (uint64_t)c.kv_len * w.L * w.nkv * w.d * 2 * 2);
    with_head_dim(w.d, [&](auto D) {     // plan_persistent admits head_dim 64 / 128 only
        if constexpr (D == 64 || D == 128)
            launch(lc, "decode_persistent", bytes, decode_persistent_kernel<D>, dim3(kNumSMs), dim3(kPkThreads), c.pk.smem, a);
    });
    if (w.tp > 1)   // every rank received every logits slice in its exchange area: hand them to the usual logits buffer
        FL_CUDA(cudaMemcpyAsync(c.logits.p, (uint8_t*)g_peer.local + PeerComm::kLogitsOff, (size_t)w.Vfull * 4, cudaMemcpyDeviceToDevice, c.stream));
    if (dbg) {
        static const char* names[] = {"P1 x(rmsnorm)", "P1 consume qkv", "P1 epilogue", "P1 grid barrier", "P2 attention", "P2 grid barrier",
                                      "P3 x", "P3 consume o", "P3 epilogue", "P3 grid barrier", "P4 x(rmsnorm)", "P4 consume gate/up",
                                      "P4 epilogue", "P4 grid barrier", "P5 x", "P5 consume down", "P5 epilogue", "P5 grid barrier"};
        long long h[40];
        FL_CUDA(cudaStreamSynchronize(c.stream));
        FL_CUDA(cudaMemcpy(h, dbg_buf, sizeof(h), cudaMemcpyDeviceToHost));
        fprintf(stderr, "[FL_PK_DEBUG] warp 0 of CTA 0, clocks waiting for weights / chunks per phase: qkv %lld/%lld o %lld/%lld gateup %lld/%lld down %lld/%lld\n",
                h[32] / 1000, h[32] % 1000, h[33] / 1000, h[33] % 1000, h[34] / 1000, h[34] % 1000, h[35] / 1000, h[35] % 1000);
        fprintf(stderr, "[FL_PK_DEBUG] layer %d, CTA 0 phase times (us):", w.L / 2);
        for (int i = 0; i < 18; ++i) fprintf(stderr, " %s=%.2f;", names[i], (h[i + 1] - h[i]) / 1000.0);
        fprintf(stderr, " layer total=%.2f\n", (h[18] - h[0]) / 1000.0);
        {      // the producer's view: when (relative to the consumers' phase boundaries) it issued the first chunks of each phase
            long long pr[40];
            FL_CUDA(cudaMemcpy(pr, dbg_buf + 660, sizeof(pr), cudaMemcpyDeviceToHost));
            static const char* pn[] = {"qkv", "o", "gate|up", "down"};
            const int cons_start[] = {1, 7, 11, 15};      // stamp index at which the consumers start consuming the phase
            for (int ph = 0; ph < 4; ++ph) {
                fprintf(stderr, "[FL_PK_DEBUG] producer, %s: chunk issue times relative to the consumers' start of the phase (us):", pn[ph]);
                for (int i = 0; i < 8 && i < pr[ph * 10 + 9]; ++i) fprintf(stderr, " %.2f", (pr[ph * 10 + i] - h[cons_start[ph]]) / 1000.0);
                fprintf(stderr, " ... last of %lld at %.2f (consume ends at %.2f)\n", pr[ph * 10 + 9], (pr[ph * 10 + 8] - h[cons_start[ph]]) / 1000.0,
                        (h[cons_start[ph] + 1] - h[cons_start[ph]]) / 1000.0);
            }
        }
        if (env_flag("FL_PK_DEBUG_CTAS")) {      // per-CTA start / end of the gate|up weight phase: who is the barrier waiting for?
            std::vector<long long> pc(4 * kNumSMs);
            FL_CUDA(cudaMemcpy(pc.data(), dbg_buf + 64, pc.size() * sizeof(long long), cudaMemcpyDeviceToHost));
            long long tmin = pc[0];
            for (int i = 0; i < kNumSMs; ++i) tmin = std::min(tmin, pc[4 * i]);
            for (int i = 0; i < kNumSMs; ++i)
                fprintf(stderr, "[FL_PK_CTA] cta %d sm %lld chunks %lld start %.2f end %.2f\n", i, pc[4 * i + 2], pc[4 * i + 3], (pc[4 * i] - tmin) / 1000.0,
                        (pc[4 * i + 1] - tmin) / 1000.0);
        }
    }
}

static void cache_create(fl_cache& c, int max_batch, int max_seq) {
    const Weights& w = *c.w;
    FL_CHECK(w.finalized, FL_ERR_STATE, "model not finalized");
    FL_CHECK(max_batch >= 1 && max_batch <= kMaxBatch && max_seq >= 1, FL_ERR_INVALID, "bad cache dimensions");
    c.max_batch = max_batch;
    c.max_seq = max_seq;
    c.pages_per_seq = (max_seq + kKvPage - 1) / kKvPage;
    FL_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    c.state.alloc(1, true);
    std::vector<int> pt((size_t)max_batch * c.pages_per_seq);
    for (size_t i = 0; i < pt.size(); ++i) pt[i] = (int)i;   // static page assignment; the layout stays paged
    c.page_table.alloc(pt.size());
    FL_CUDA(cudaMemcpy(c.page_table.p, pt.data(), pt.size() * 4, cudaMemcpyHostToDevice));
    c.layer_pool_elems = (size_t)max_batch * c.pages_per_seq * w.nkv * kKvPage * w.d;
    c.kpool.alloc(c.layer_pool_elems * w.L, true);
    c.vpool.alloc(c.layer_pool_elems * w.L, true);
    {
        const uint64_t rows = (uint64_t)c.layer_pool_elems / w.d * w.L;
        c.kv_tmaps = rows < (1ull << 31) && (w.d == 16 || w.d == 32 || w.d == 64 || w.d == 128);
        if (c.kv_tmaps) {
            c.tm_kpool = make_tmap_kv(c.kpool.p, rows, (uint32_t)w.d);
            c.tm_vpool = make_tmap_kv(c.vpool.p, rows, (uint32_t)w.d);
        }
    }
    int ns = (2 * kNumSMs + w.nkv * kPassRows - 1) / (w.nkv * kPassRows);
    if (ns > c.pages_per_seq) ns = c.pages_per_seq;
    if (ns < 1) ns = 1;
    c.nsplit = ns;
    const size_t nq = (size_t)w.nh * w.d;
    c.ids.alloc((size_t)max_batch * max_seq);
    c.next_ids.alloc(max_batch, true);
    c.trace_pos.alloc(1, true);
    c.resid.alloc(kPassRows * w.H);
    c.q.alloc(kPassRows * nq);
    c.attn_out.alloc(kPassRows * nq);
    c.act.alloc((size_t)kPassRows * w.I);
    c.logits.alloc((size_t)max_batch * w.Vfull, true);
    if (w.tp > 1) {
        c.tp_buf.alloc((size_t)kPassRows * w.H);
        c.resid2.alloc((size_t)kPassRows * w.H);
        c.tp_local.alloc((size_t)max_batch * w.V, true);
        c.tp_gather.alloc((size_t)w.tp * max_batch * w.V);
    }
    c.part_acc.alloc((size_t)kPassRows * w.nh * c.nsplit * w.d);
    c.part_ml.alloc((size_t)kPassRows * w.nh * c.nsplit * 2);
    c.counters.alloc((size_t)kPassRows * w.nkv, true);
    c.amax_parts = kNumSMs * 4;
    c.amax_val.alloc((size_t)kPassRows * c.amax_parts);
    c.amax_idx.alloc((size_t)kPassRows * c.amax_parts);
    c.h_ids.alloc((size_t)max_batch * max_seq);
    c.h_logits.alloc((size_t)max_batch * w.Vfull);
    c.slot_len.assign(max_batch, 0);
    c.slot_tab.alloc(2 * (size_t)max_batch);
    c.h_slot_tab.alloc(2 * (size_t)max_batch);
    c.sample_out.alloc(1, true);
    plan_persistent(c);
    FL_CUDA(cudaDeviceSynchronize());
}

static void cache_destroy_graphs(fl_cache& c) {
    for (auto& kv : c.graphs)
        if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    c.graphs.clear();
}

// Enqueue the whole forward for the flattened [b, t] call on lc.stream.  Rows are processed in passes of kPassRows,
// pass-major / layer-minor: a token's layer-l attention only needs the layer-l K/V of EARLIER tokens, which earlier
// passes already appended, so the order is causal-correct.
static void enqueue_forward_dense(fl_cache& c, LaunchCtx& lc, int b, int t, bool loop_mode);

// A uniform call of `rows` activation rows runs on the dense (tcgen05) path: 3+ rows, or any Mixtral call.
static bool uses_dense(const fl_cache& c, int rows) {
    return (rows >= 3 || c.w->cfg.arch == FL_ARCH_MIXTRAL) && c.w->dense_ok;
}

static void enqueue_forward(fl_cache& c, LaunchCtx& lc, int b, int t, bool loop_mode) {
    const Weights& w = *c.w;
    const int rows = b * t;
    FL_CHECK(w.cfg.arch != FL_ARCH_MIXTRAL || c.dw.rows >= (size_t)rows, FL_ERR_STATE, "internal: Mixtral needs the dense workspace");
    if (uses_dense(c, rows) && c.dw.rows >= (size_t)rows) {   // workspace is reserved by the caller (never during capture)
        enqueue_forward_dense(c, lc, b, t, loop_mode);
        return;
    }
    const size_t nq = (size_t)w.nh * w.d;
    const GemvPlan p_qkv = plan_gemv(w.nqkv, w.H), p_o = plan_gemv(w.H, (int)nq), p_gu = plan_gemv(2 * w.I, w.H),
                   p_down = plan_gemv(w.H, w.I), p_head = plan_gemv(w.V, w.H);
    FL_CHECK(p_head.grid <= c.amax_parts, FL_ERR_STATE, "internal: arg-max partial buffer too small");
    const size_t attn_smem = attn_smem_bytes(w.d, w.nh / w.nkv);
    const float qscale = (float)(1.0 / std::sqrt((double)w.d));
    const bool windowed = (w.cfg.arch != FL_ARCH_LLAMA) && w.cfg.sliding_window > 0 && t > 1;

    for (int row_base = 0; row_base < rows; row_base += kPassRows) {
        const int M = std::min(kPassRows, rows - row_base);
        bool has_last = false;
        for (int m = 0; m < M; ++m) has_last |= ((row_base + m) % t == t - 1);

        launch(lc, "embed_gather", (uint64_t)M * w.H * 2, embed_gather_kernel, dim3((w.H / 8 + 255) / 256, M), dim3(256), 0,
               (const uint16_t*)w.embed, (const uint32_t*)c.ids.p, row_base, w.H, w.Vfull, c.resid.p);
        // tensor parallelism: the all-reduced o_proj / down_proj output is added to the residual stream inside the NEXT
        // RMSNorm prologue (which writes the advanced stream to the other of two buffers), not by a separate kernel
        float* rcur = c.resid.p;
        float* roth = c.resid2.p;
        const float* pending = nullptr;
        auto take_pending = [&](GemvArgs& ga) {
            ga.x = rcur;
            if (pending) {
                ga.delta = pending; ga.resid_out = roth;
                std::swap(rcur, roth);
                pending = nullptr;
            }
        };

        for (int l = 0; l < w.L; ++l) {
            const LayerW& lw = w.layers[l];
            GemvArgs a{};
            a.row_base = row_base; a.t = t; a.eps = w.cfg.norm_eps;
            // K2+K3+K4+K5+K6: RMSNorm -> fused q|k|v GEMV (+bias) -> RoPE -> q store + in-place paged KV append
            a.W = lw.wqkv; a.N = w.nqkv; a.K = w.H; a.norm_w = lw.ln1; a.bias = lw.bqkv;
            take_pending(a);
            a.q_out = c.q.p; a.kpool = c.kpool.p + (size_t)l * c.layer_pool_elems; a.vpool = c.vpool.p + (size_t)l * c.layer_pool_elems;
            a.page_table = c.page_table.p; a.pt_stride = c.pages_per_seq; a.state = c.state.p;
            a.rope_cos = w.rope_cos; a.rope_sin = w.rope_sin; a.nh = w.nh; a.nkv = w.nkv; a.d = w.d; a.max_pos = w.max_pos;
            launch_gemv<PRO_RMSNORM, EPI_QKV>(lc, "gemv_qkv_rope", M, p_qkv, a);

            // K7-K11: split-K paged decode attention
            AttnArgs at{};
            at.q = c.q.p; at.kpool = a.kpool; at.vpool = a.vpool; at.page_table = c.page_table.p; at.pt_stride = c.pages_per_seq;
            at.state = c.state.p; at.part_acc = c.part_acc.p; at.part_ml = c.part_ml.p; at.counters = c.counters.p; at.out = c.attn_out.p;
            at.nh = w.nh; at.nkv = w.nkv; at.t = t; at.row_base = row_base;
            at.sliding_window = windowed ? w.cfg.sliding_window : 0;
            at.qscale = qscale;
            const uint64_t kv_bytes = (uint64_t)M * (c.kv_len + t) * w.nkv * w.d * 2 * 2;
            launch_attn(lc, w.d, c.nsplit, w.nkv, M, attn_smem, kv_bytes, at);

            // K12+K13: o_proj + residual add
            GemvArgs o{};
            o.row_base = row_base; o.t = t;
            o.W = lw.wo; o.N = w.H; o.K = (int)nq; o.x = c.attn_out.p; o.out = c.resid.p;
            if (w.tp > 1) {   // row-parallel: partial sums -> all-reduce -> residual add
                o.out = c.tp_buf.p; o.ldo = w.H;
                launch_gemv<PRO_PLAIN, EPI_STORE>(lc, "gemv_o_partial", M, p_o, o);
                tp_allreduce_sum(lc, c.tp_buf.p, (size_t)M * w.H);
                pending = c.tp_buf.p;
            } else {
                launch_gemv<PRO_PLAIN, EPI_RESID>(lc, "gemv_o_resid", M, p_o, o);
            }

            // K14+K15: RMSNorm -> fused gate|up GEMV -> SiLU(gate) * up
            GemvArgs g{};
            g.row_base = row_base; g.t = t; g.eps = w.cfg.norm_eps;
            g.W = lw.wgu; g.N = 2 * w.I; g.K = w.H; g.norm_w = lw.ln2; g.out = c.act.p;
            take_pending(g);
            launch_gemv<PRO_RMSNORM, EPI_SILU>(lc, "gemv_gateup_silu", M, p_gu, g);

            // K16: down_proj + residual add
            GemvArgs dn{};
            dn.row_base = row_base; dn.t = t;
            dn.W = lw.wdown; dn.N = w.H; dn.K = w.I; dn.x = c.act.p; dn.out = c.resid.p;
            if (w.tp > 1) {
                dn.out = c.tp_buf.p; dn.ldo = w.H;
                launch_gemv<PRO_PLAIN, EPI_STORE>(lc, "gemv_down_partial", M, p_down, dn);
                tp_allreduce_sum(lc, c.tp_buf.p, (size_t)M * w.H);
                pending = c.tp_buf.p;
            } else {
                launch_gemv<PRO_PLAIN, EPI_RESID>(lc, "gemv_down_resid", M, p_down, dn);
            }
        }
        if (has_last) {
            // K17 (+K18): final RMSNorm -> lm_head -> f32 logits of the last position + arg-max partials
            GemvArgs h{};
            h.row_base = row_base; h.t = t; h.eps = w.cfg.norm_eps;
            h.W = w.lm_head; h.N = w.V; h.K = w.H; h.norm_w = w.final_norm;
            take_pending(h);
            h.out = c.logits.p; h.ldo = w.V; h.last_only = 1; h.amax_val = c.amax_val.p; h.amax_idx = c.amax_idx.p;
            if (w.tp > 1) {   // vocab-parallel head: this rank's slice; gathered + arg-maxed after the pass loop
                h.out = c.tp_local.p; h.amax_val = nullptr; h.amax_idx = nullptr;
                launch_gemv<PRO_RMSNORM, EPI_STORE>(lc, "gemv_lm_head", M, p_head, h);
            } else {
                launch_gemv<PRO_RMSNORM, EPI_STORE>(lc, "gemv_lm_head", M, p_head, h);
                launch(lc, "argmax_finalize", 0, argmax_finalize_kernel, dim3(1), dim3(256), 0, (const float*)c.amax_val.p,
                       (const int*)c.amax_idx.p, p_head.grid, M, row_base, t, c.next_ids.p);
            }
        }
    }
    if (w.tp > 1) {   // gather the vocab slices of every rank, lay them out as [b, Vfull], arg-max (last index wins ties)
        tp_allgather(lc, c.tp_local.p, c.tp_gather.p, (size_t)b * w.V);
        launch(lc, "tp_logits", 0, tp_logits_kernel, dim3(kNumSMs), dim3(256), 0, (const float*)c.tp_gather.p, w.tp, b, w.V, c.logits.p);
        launch(lc, "dense_argmax", 0, dense_argmax_kernel, dim3(b), dim3(1024), 0, (const float*)c.logits.p, 1, (long long)0, w.Vfull,
               c.logits.p, c.next_ids.p);
    }
    launch(lc, "advance_state", 0, advance_state_kernel, dim3(1), dim3(kMaxBatch), 0, c.state.p, b, t, loop_mode ? 1 : 0, c.ids.p,
           (const uint32_t*)c.next_ids.p, loop_mode ? 1 : 0, loop_mode ? c.trace.p : (uint32_t*)nullptr,
           loop_mode ? c.trace_pos.p : (int*)nullptr);
}


// ------------------------------------------------------------------------------------------------------------------
// Dense (tcgen05) path: prefill and batched decode with 3+ activation rows
// ------------------------------------------------------------------------------------------------------------------
constexpr int kDenseMaxSplit = 16;    // upper bound on the split-K slices of a decode GEMM (see pick_ksplit)

static int pick_ksplit(int tiles, int nk, int R);
// N tile of a swap-AB GEMM over `rows` (<= 128) activation rows: the smallest of 16 / 32 / 64 / 128 that holds every row; for the
// grouped expert GEMMs also the rows per expert block
static int swap_tile_n(int rows) { return rows <= 16 ? 16 : (rows <= 32 ? 32 : (rows <= 64 ? 64 : 128)); }

static void ensure_dense_ws(fl_cache& c, int rows) {
    DenseWs& d = c.dw;
    if ((size_t)rows <= d.rows) return;
    const Weights& w = *c.w;
    FL_CUDA(cudaStreamSynchronize(c.stream));
    cache_destroy_graphs(c);             // captured graphs hold the old workspace pointers
    const size_t R = rows, nq = (size_t)w.nh * w.d;
    const size_t kmax = std::max<size_t>(std::max<size_t>(w.H, nq), w.I);
    const size_t nmax = std::max<size_t>(std::max<size_t>(w.nqkv, 2 * (size_t)w.I), std::max<size_t>(w.H, w.V));
    d.xhi.alloc(R * kmax); d.xlo.alloc(R * kmax);
    const size_t Rm = w.ep_dp ? R * (size_t)w.ep : R;        // rows the expert GEMMs see
    {   // GEMM output: [ks][rows, N] for the largest N * ks over the model's GEMM shapes at this row count
        size_t need = Rm * nmax;
        auto consider = [&](size_t rows, size_t N, size_t K) {
            const int ks = rows <= 128 ? pick_ksplit((int)((N + 127) / 128), (int)((K + kGemmBK - 1) / kGemmBK), (int)rows) : 1;
            need = std::max(need, rows * N * (size_t)ks);
        };
        consider(R, w.nqkv, w.H); consider(R, w.H, nq); consider(R, w.V, w.H);
        consider(Rm, 2 * (size_t)w.I, w.H); consider(Rm, w.H, w.I);
        if (w.cfg.arch == FL_ARCH_MIXTRAL) {      // grouped expert GEMMs: E_local stacked matrices x one block of `cap` rows each
            for (size_t cap = 16; cap <= (size_t)swap_tile_n((int)std::min<size_t>(Rm, 128)); cap *= 2) {
                const size_t Rg = (size_t)w.E_local * cap;
                for (size_t NK : {(size_t)0, (size_t)1}) {
                    const size_t N = NK == 0 ? 2 * (size_t)w.I : w.H, K = NK == 0 ? w.H : w.I;
                    const int ksg = pick_ksplit((int)(w.E_local * ((N + 127) / 128)), (int)((K + kGemmBK - 1) / kGemmBK), (int)cap);
                    need = std::max(need, Rg * N * (size_t)ksg);
                }
            }
        }
        for (size_t r = 1; r <= std::min<size_t>(R, kMaxBatch); ++r) consider(r, w.V, w.H);     // the lm_head runs on one row per sequence
        d.y.alloc(need);
    }
    d.resid.alloc(R * w.H); d.q.alloc(R * nq);      // the attention output goes straight into xhi / xlo (hi/lo operand of o_proj)
    if (w.tp > 1) d.tp_buf.alloc(R * w.H);
    if (w.cfg.arch != FL_ARCH_MIXTRAL && R > 128) { d.xhi2.alloc(R * (size_t)w.I); d.xlo2.alloc(R * (size_t)w.I); }
    if (w.cfg.arch == FL_ARCH_MIXTRAL) {
        // grouped path (calls with <= 128 expert rows): E_local blocks of up to grp_cap rows; masked path (prefill): Rm rows
        const size_t grp_cap = swap_tile_n((int)std::min<size_t>(Rm, 128));
        const size_t Rg = (size_t)w.E_local * grp_cap;
        d.xhi2.alloc(std::max(Rm, Rg) * kmax); d.xlo2.alloc(std::max(Rm, Rg) * kmax);
        d.gx_hi.alloc(Rg * w.H, true); d.gx_lo.alloc(Rg * w.H, true);
        d.grp_cnt.alloc(w.E_local, true); d.grp_pos.alloc(Rm * w.E_local);
        d.moe_out.alloc(Rm * w.H); d.route_w.alloc(R * w.E);
        d.route_sel.alloc((size_t)w.L * R * w.top_k, true); d.route_margin.alloc((size_t)w.L * R, true);
        if (w.ep_dp) {
            d.g_xhi.alloc(Rm * w.H); d.g_xlo.alloc(Rm * w.H); d.g_route.alloc(Rm * w.E);
            d.comb.alloc(Rm * w.H);
        }
    }
    const int chunk = std::min(rows, kMaxBatch);    // split partials of the batched-decode attention: one row per sequence
    d.counters.alloc((size_t)chunk * w.nkv, true);
    d.sk_acc.alloc((size_t)4 * kNumSMs * 2 * (w.nh / w.nkv) * w.d);
    d.sk_ml.alloc((size_t)4 * kNumSMs * 2 * (w.nh / w.nkv) * 2);
    d.vt_pages_cap = 0;
    if ((w.d == 64 || w.d == 128) && R > (size_t)kKvPage) {
        d.vt_pages_cap = R / kKvPage + std::min<size_t>(R, kMaxBatch);
        d.vt.alloc(d.vt_pages_cap * w.nkv * w.d * kKvPage, true);        // zero: the last page's tail multiplies P = 0 and must stay finite
        d.tm_vt = make_tmap_bf16(d.vt.p, d.vt_pages_cap * w.nkv * w.d, kKvPage, kKvPage, (uint32_t)w.d);
    }
    d.rows = R;
}

// Split-K factor of a swap-AB (decode) GEMM: the one whose work items (output tiles x k slices) fill whole waves of the 148
// persistent CTAs best, counting the padding of the last k slice; fewer, longer items win ties (pipeline fill / epilogue per item).
// The consumer sums the slices in a fixed order, so a row's bytes read grow with ks: capped by the row count.
static int pick_ksplit(int tiles, int nk, int R) {
    const int maxks = std::max(1, std::min(std::min(kDenseMaxSplit, std::max(2, 256 / std::max(R, 1))), nk / 4));
    int best = 1;
    double best_eff = 0.0;
    for (int ks = 1; ks <= maxks; ++ks) {
        const long long items = (long long)tiles * ks;
        const long long waves = (items + kNumSMs - 1) / kNumSMs;
        const int nkps = (nk + ks - 1) / ks;
        const double eff = (double)items / (double)(waves * kNumSMs) * (double)nk / (double)(ks * nkps);
        if (eff > best_eff * 1.03) { best_eff = eff; best = ks; }
    }
    return best;
}

// out[ks][R, N] (f32, row stride N, slice stride R*N) = (xhi + xlo)[R, K] . W[N, K]^T; returns the number of split-K slices,
// which the consumer kernel sums in a fixed order (deterministic, no atomics, no memset).
//   R <= 128 (decode batches, short prefills): swap-AB -- the weights are the 128-row MMA operand, the activations a tiny
//             N = R tile, the result is stored transposed; the only large shared-memory traffic is the weight stream.
//   R  > 128 (prefill): tokens are the M dimension, 128 x 256 output tiles.
static int dense_gemm(fl_cache& c, LaunchCtx& lc, const char* tag, int R, int N, int K, const CUtensorMap& tmW, float* out,
                      const uint16_t* xhi = nullptr, const uint16_t* xlo = nullptr, uint16_t* silu_hi = nullptr, uint16_t* silu_lo = nullptr) {
    if (!xhi) { xhi = c.dw.xhi.p; xlo = c.dw.xlo.p; }
    const int nk = (K + kGemmBK - 1) / kGemmBK;
    const bool swap = R <= 128;
    // prefill: 128 tokens x 256 weight rows per tile.  The hi/lo activation pair makes a k-block 2 x 16 KB of A next to the weight
    // tile, and the GEMM is bound by the shared-memory fill rate (L2 -> SM), not by the tensor pipe: a 256-row weight tile is
    // 64 KB per 2 x 128 x 256 x 64 MACs where the 128-row one is 48 KB per half of that -- 1.5x the arithmetic per staged byte.
    const int tiles = swap ? (N + 127) / 128 : ((R + kGemmBM - 1) / kGemmBM) * ((N + 255) / 256);
    const int ks = swap ? pick_ksplit(tiles, nk, R) : 1;
    const uint64_t bytes = (uint64_t)N * K * 2;
    const dim3 block(kGemmThreads);
    if (swap) {
        const int bn = swap_tile_n(R);
        const CUtensorMap hi = make_tmap_bf16(xhi, R, K, K, bn), lo = make_tmap_bf16(xlo, R, K, K, bn);
        GemmArgs g{N, R, K, nullptr, nullptr, 0, out, N, ks, (long long)R * N};     // M = weight rows, N = activation rows
        with_tile_n(bn, [&](auto BN) {
            launch(lc, tag, bytes, gemm_tc_kernel<BN, GEPI_F32_T, DUAL_B>, dim3(std::min(tiles * ks, kNumSMs)), block, gemm_smem_bytes(BN, DUAL_B),
                   tmW, hi, lo, g);
        });
    } else {
        const CUtensorMap hi = make_tmap_bf16(xhi, R, K, K, kGemmBM), lo = make_tmap_bf16(xlo, R, K, K, kGemmBM);
        const dim3 grid(std::min(tiles, kNumSMs));
        if (silu_hi != nullptr) {       // prefill gate|up: SiLU(gate) * up + hi/lo split fused into the epilogue
            GemmArgs g{R, N, K, nullptr, nullptr, 0, silu_hi, N / 2, 1, 0, silu_lo};
            launch(lc, tag, bytes, gemm_tc_kernel<256, GEPI_SILU_HL, DUAL_A>, grid, block, gemm_smem_bytes(256, DUAL_A), hi, lo, tmW, g);
        } else {
            GemmArgs g{R, N, K, nullptr, nullptr, 0, out, N, 1, (long long)R * N};
            launch(lc, tag, bytes, gemm_tc_kernel<256, GEPI_F32, DUAL_A>, grid, block, gemm_smem_bytes(256, DUAL_A), hi, lo, tmW, g);
        }
    }
    return ks;
}

// Grouped swap-AB GEMM over this rank's experts (decode batches): group j multiplies ITS gathered rows (block j of xhi / xlo,
// `cap` rows, cnt[j] valid) with ITS matrix (block j of the stacked weights, Ne rows): out[ks][j * cap + n][Ne].  ONE launch over
// (expert, weight tile, k slice) work items; an expert without rows costs nothing.  Returns the split-K factor.
static int dense_gemm_grouped(fl_cache& c, LaunchCtx& lc, const char* tag, int groups, int cap, int Ne, int K, const CUtensorMap& tmWall,
                              float* out, const uint16_t* xhi, const uint16_t* xlo, const int* cnt) {
    const int nk = (K + kGemmBK - 1) / kGemmBK;
    const int tiles = groups * ((Ne + kGemmBM - 1) / kGemmBM);
    const int ks = pick_ksplit(tiles, nk, cap);
    const CUtensorMap hi = make_tmap_bf16(xhi, (uint64_t)groups * cap, K, K, cap), lo = make_tmap_bf16(xlo, (uint64_t)groups * cap, K, K, cap);
    GemmArgs g{groups * Ne, cap, K, nullptr, nullptr, 0, out, Ne, ks, (long long)groups * cap * Ne};
    g.grp_m = Ne; g.grp_cap = cap; g.grp_cnt = cnt;
    with_tile_n(cap, [&](auto BN) {
        launch(lc, tag, (uint64_t)groups * Ne * K * 2, gemm_tc_kernel<BN, GEPI_F32_T, DUAL_B>, dim3(std::min(tiles * ks, kNumSMs)), dim3(kGemmThreads),
               gemm_smem_bytes(BN, DUAL_B), tmWall, hi, lo, g);
    });
    return ks;
}

static void enqueue_forward_dense(fl_cache& c, LaunchCtx& lc, int b, int t, bool loop_mode) {
    const Weights& w = *c.w;
    DenseWs& d = c.dw;
    const int R = b * t;
    const int nq = w.nh * w.d;
    const float qscale = (float)(1.0 / std::sqrt((double)w.d));
    const bool windowed = (w.cfg.arch != FL_ARCH_LLAMA) && w.cfg.sliding_window > 0 && t > 1;
    // multi-token calls on empty sequences with head_dim 64 / 128 and more than one page of keys: attention on tcgen05
    // (attn_prefill_tc_kernel; FL_ATTN_PREFILL_MMA=1 keeps the mma.sync kernel, the A/B knob)
    const int vt_pages = (t + kKvPage - 1) / kKvPage;
    const bool prefill_mma = env_flag("FL_ATTN_PREFILL_MMA");
    const bool tc_prefill = t > kKvPage && (w.d == 64 || w.d == 128) && c.kv_tmaps && c.fresh_call && !prefill_mma &&
                            (size_t)b * vt_pages <= d.vt_pages_cap;

    auto prep = [&](const char* tag, PrepArgs pa, int rows_out) {
        pa.xhi = d.xhi.p; pa.xlo = d.xlo.p; pa.eps = w.cfg.norm_eps; pa.t = t;
        // many rows (prefill): the register-resident 256-thread kernel (dense_prep_rows_kernel)
        if (rows_out >= 512 && pa.norm_w != nullptr && pa.embed == nullptr && pa.K <= 8192 && pa.K % 4 == 0) {
            if (pa.K <= 4096)
                launch(lc, tag, 0, dense_prep_rows_kernel<4>, dim3(rows_out), dim3(kPrepRowsThreads), 0, pa);
            else
                launch(lc, tag, 0, dense_prep_rows_kernel<8>, dim3(rows_out), dim3(kPrepRowsThreads), 0, pa);
            return;
        }
        const int threads = std::min(1024, std::max(32, (pa.K / 4 + 31) / 32 * 32));
        launch(lc, tag, 0, dense_prep_kernel, dim3(rows_out), dim3(threads), 0, pa);
    };
    {   // K1 + K2 of layer 0
        PrepArgs pa{};
        pa.embed = w.embed; pa.ids = c.ids.p; pa.vocab = w.Vfull; pa.resid = d.resid.p; pa.norm_w = w.layers[0].ln1; pa.K = w.H;
        prep("dense_embed_rmsnorm", pa, R);
    }
    for (int l = 0; l < w.L; ++l) {
        const LayerW& lw = w.layers[l];
        uint16_t* kpool = c.kpool.p + (size_t)l * c.layer_pool_elems;
        uint16_t* vpool = c.vpool.p + (size_t)l * c.layer_pool_elems;
        int ks = dense_gemm(c, lc, "gemm_tc_qkv", R, w.nqkv, w.H, lw.tm_wqkv, d.y.p);
        QkvEpiArgs qa{ks, (long long)R * w.nqkv, d.y.p, lw.bqkv, d.q.p, kpool, vpool, c.page_table.p, c.pages_per_seq, c.state.p, w.rope_cos,
                      w.rope_sin, w.nh, w.nkv, w.d, w.max_pos, t, w.nqkv, tc_prefill ? d.vt.p : nullptr, vt_pages};
        if (t >= 64 && t % kQkvRowsPerThread == 0)      // prefill: eight rows per thread (dense_qkv_epi_rows_kernel)
            launch(lc, "dense_qkv_rope_append", 0, dense_qkv_epi_rows_kernel, dim3((w.nqkv / 2 + 255) / 256, R / kQkvRowsPerThread), dim3(256), 0, qa);
        else
            launch(lc, "dense_qkv_rope_append", 0, dense_qkv_epi_kernel, dim3((w.nqkv / 2 + 255) / 256, R), dim3(256), 0, qa);
        {   // K7-K11 on tensor cores; the output lands as the hi/lo bf16 operands of the o_proj GEMM
            AttnArgs at{};
            at.q = d.q.p; at.kpool = kpool; at.vpool = vpool; at.page_table = c.page_table.p; at.pt_stride = c.pages_per_seq;
            at.state = c.state.p; at.counters = d.counters.p;
            at.out_hi = d.xhi.p; at.out_lo = d.xlo.p; at.nh = w.nh; at.nkv = w.nkv; at.t = t; at.row_base = 0;
            at.sliding_window = windowed ? w.cfg.sliding_window : 0; at.qscale = qscale;
            const uint64_t kv_bytes = (uint64_t)b * (c.kv_len + t) * w.nkv * w.d * 4;
            const int layer_row0 = (int)((size_t)l * (c.layer_pool_elems / w.d));
            with_head_dim(w.d, [&](auto D) {
                if (t == 1) {
                    // stream-K: a fixed grid of resident CTAs, each an equal share of the step's page stream.  The grid does NOT
                    // depend on the KV length: this launch is captured into the step's CUDA graph, which is keyed by (batch, mode)
                    // only and replayed as the context grows.
                    FL_CHECK(c.kv_tmaps && w.nh / w.nkv <= 16, FL_ERR_UNSUPPORTED, "batched decode attention: GQA group > 16 heads or KV pool beyond 2^31 rows");
                    const SkPlan pl = attn_sk_plan<D>(w.nh / w.nkv);
                    SkArgs sk{};
                    sk.a = at; sk.sk_acc = d.sk_acc.p; sk.sk_ml = d.sk_ml.p; sk.b = b; sk.layer_row0 = layer_row0;
                    launch(lc, "attn_sk_decode", kv_bytes, attn_sk_decode_kernel<D>, dim3(pl.ctas * kNumSMs), dim3(kSkThreads), pl.smem, c.tm_kpool,
                           c.tm_vpool, sk);
                } else if (tc_prefill) {
                    if constexpr (D == 64 || D == 128) {
                        TcPrefillArgs tp{};
                        tp.a = at; tp.layer_row0 = layer_row0; tp.vt_pages = vt_pages;
                        tp.tau = std::getenv("FL_ATTN_TC_TAU") ? (float)std::atof(std::getenv("FL_ATTN_TC_TAU")) : 8.f;      // 0: O is rescaled on every new row max (tests)
                        launch(lc, "attn_prefill_tc", kv_bytes, attn_prefill_tc_kernel<D>, dim3((t + kTcQ - 1) / kTcQ, w.nh, b), dim3(kTcThreads),
                               attn_prefill_tc_smem_bytes(D), c.tm_kpool, d.tm_vt, tp);
                    }
                } else {
                    launch(lc, "attn_prefill", kv_bytes, attn_prefill_kernel<D>, dim3((t + kPrefillBM - 1) / kPrefillBM, w.nh, b), dim3(kMmaAttnThreads),
                           attn_prefill_smem_bytes(D), at);
                }
            });
        }
        ks = dense_gemm(c, lc, "gemm_tc_o", R, w.H, nq, lw.tm_wo, d.y.p);
        const float* delta = d.y.p;
        auto tp_reduce = [&]() {   // row-parallel GEMM: fold the split-K slices, then all-reduce the partial sums across ranks
            if (w.tp <= 1) return;
            float* buf = d.tp_buf.p;
            if (ks == 1)        // one slice (every prefill GEMM): the GEMM output is all-reduced in place, no copy pass over [R, H]
                buf = d.y.p;
            else
                launch(lc, "tp_sum_slices", 0, sum_slices_kernel, dim3(kNumSMs), dim3(256), 0, (const float*)d.y.p, ks, (long long)R * w.H, R * w.H,
                       d.tp_buf.p);
            tp_allreduce_sum(lc, buf, (size_t)R * w.H);
            delta = buf;
            ks = 1;
        };
        tp_reduce();
        {   // K13 + K14: resid += o_proj; x = rms_norm(resid) * ln2
            PrepArgs pa{};
            pa.resid = d.resid.p; pa.delta = delta; pa.ldd = w.H; pa.nsl = ks; pa.sl_stride = (long long)R * w.H; pa.norm_w = lw.ln2; pa.K = w.H;
            prep("dense_resid_rmsnorm", pa, R);
        }
        if (w.cfg.arch == FL_ARCH_MIXTRAL) {
            // sparse MoE: route, then (decode batches) gather each local expert's rows and run ONE grouped GEMM pair over all
            // experts, or (prefill, > 128 rows) stream every local expert over all rows with the routing weight as a mask (zero
            // when not selected).  No host sync either way, and a fixed summation order (experts ascending).
            launch(lc, "moe_router", 0, moe_router_kernel, dim3(R), dim3(256), 0, (const uint16_t*)d.xhi.p, (const uint16_t*)d.xlo.p, w.H,
                   (const float*)lw.wgate, w.E, w.top_k, d.route_w.p, d.route_sel.p + (size_t)l * R * w.top_k, d.route_margin.p + (size_t)l * R);
            // expert parallelism with data-parallel attention: DISPATCH -- this rank's rows (hi/lo halves + routing weights)
            // travel to the expert ranks, which then see the rows of all ranks in rank-major order
            const int Rm = w.ep_dp ? R * w.ep : R;
            const uint16_t* ex_hi = d.xhi.p;
            const uint16_t* ex_lo = d.xlo.p;
            const float* ex_route = d.route_w.p;
            if (w.ep_dp) {
                const A2aSeg segs[3] = {{d.xhi.p, d.g_xhi.p, (size_t)R * w.H * 2, true}, {d.xlo.p, d.g_xlo.p, (size_t)R * w.H * 2, true},
                                        {d.route_w.p, d.g_route.p, (size_t)R * w.E * 4, true}};
                ep_alltoall(lc, segs, 3);
                ex_hi = d.g_xhi.p; ex_lo = d.g_xlo.p; ex_route = d.g_route.p;
            }
            if (Rm <= 128 && !env_flag("FL_MOE_MASKED")) {
                // decode batches: per-expert row lists + ONE grouped GEMM pair over (expert, weight tile, k slice) work items
                const int cap = swap_tile_n(Rm), Rg = w.E_local * cap, e0 = w.rank * w.E_local;
                MoeGatherArgs ga{ex_hi, ex_lo, ex_route, Rm, w.H, w.E, e0, w.E_local, cap, d.gx_hi.p, d.gx_lo.p, d.grp_cnt.p, d.grp_pos.p};
                launch(lc, "moe_gather", 0, moe_gather_kernel, dim3(w.E_local, std::max(1, std::min(Rm, 2 * kNumSMs / w.E_local))), dim3(256), 0, ga);
                int ke = dense_gemm_grouped(c, lc, "gemm_tc_moe_w13", w.E_local, cap, 2 * w.I, w.H, lw.tm_ewgu_all, d.y.p, d.gx_hi.p, d.gx_lo.p,
                                            d.grp_cnt.p);
                launch(lc, "dense_silu_split", 0, dense_silu_split_kernel, dim3((w.I + 255) / 256, Rg), dim3(256), 0, (const float*)d.y.p, ke,
                       (long long)Rg * 2 * w.I, w.I, d.xhi2.p, d.xlo2.p, (const int*)d.grp_cnt.p, cap);
                ke = dense_gemm_grouped(c, lc, "gemm_tc_moe_w2", w.E_local, cap, w.H, w.I, lw.tm_ewdown_all, d.y.p, d.xhi2.p, d.xlo2.p, d.grp_cnt.p);
                launch(lc, "moe_combine", 0, moe_combine_kernel, dim3((w.H + 255) / 256, Rm), dim3(256), 0, (const float*)d.y.p, ke,
                       (long long)Rg * w.H, w.H, ex_route, w.E, e0, w.E_local, (const int*)d.grp_pos.p, d.moe_out.p);
            } else
            for (int j = 0; j < w.E_local; ++j) {
                const int e = w.rank * w.E_local + j;
                int ke = dense_gemm(c, lc, "gemm_tc_moe_w13", Rm, 2 * w.I, w.H, lw.tm_ewgu[j], d.y.p, ex_hi, ex_lo);
                launch(lc, "dense_silu_split", 0, dense_silu_split_kernel, dim3((w.I + 255) / 256, Rm), dim3(256), 0, (const float*)d.y.p, ke,
                       (long long)Rm * 2 * w.I, w.I, d.xhi2.p, d.xlo2.p, (const int*)nullptr, 0);
                ke = dense_gemm(c, lc, "gemm_tc_moe_w2", Rm, w.H, w.I, lw.tm_ewdown[j], d.y.p, d.xhi2.p, d.xlo2.p);
                launch(lc, "moe_accum", 0, moe_accum_kernel, dim3((w.H + 255) / 256, Rm), dim3(256), 0, (const float*)d.y.p, ke,
                       (long long)Rm * w.H, w.H, ex_route, w.E, e, j == 0 ? 1 : 0, d.moe_out.p);
            }
            delta = d.moe_out.p;
            ks = 1;
            if (w.ep_dp) {
                // COMBINE: the weighted expert outputs of rank p's rows travel back to rank p; the owner sums the ep partial
                // outputs in rank order inside the next residual-add prologue (fixed order: deterministic)
                const A2aSeg seg{d.moe_out.p, d.comb.p, (size_t)R * w.H * 4, false};
                ep_alltoall(lc, &seg, 1);
                delta = d.comb.p;
                ks = w.ep;
            } else if (w.ep > 1) {
                tp_allreduce_sum(lc, d.moe_out.p, (size_t)R * w.H);    // attention replicated: combine = sum over ranks
            }
        } else {
            if (R > 128) {      // prefill: the gate|up epilogue writes the down_proj operand directly
                dense_gemm(c, lc, "gemm_tc_gateup", R, 2 * w.I, w.H, lw.tm_wgu, d.y.p, nullptr, nullptr, d.xhi2.p, d.xlo2.p);
                ks = dense_gemm(c, lc, "gemm_tc_down", R, w.H, w.I, lw.tm_wdown, d.y.p, d.xhi2.p, d.xlo2.p);
            } else {
                ks = dense_gemm(c, lc, "gemm_tc_gateup", R, 2 * w.I, w.H, lw.tm_wgu, d.y.p);
                launch(lc, "dense_silu_split", 0, dense_silu_split_kernel, dim3((w.I + 255) / 256, R), dim3(256), 0, (const float*)d.y.p, ks,
                       (long long)R * 2 * w.I, w.I, d.xhi.p, d.xlo.p, (const int*)nullptr, 0);
                ks = dense_gemm(c, lc, "gemm_tc_down", R, w.H, w.I, lw.tm_wdown, d.y.p);
            }
            delta = d.y.p;
            tp_reduce();
        }
        PrepArgs pa{};
        pa.resid = d.resid.p; pa.delta = delta; pa.ldd = w.H; pa.nsl = ks; pa.sl_stride = (long long)R * w.H; pa.K = w.H;
        if (l + 1 < w.L) {   // K16 + next layer's K2
            pa.norm_w = w.layers[l + 1].ln1;
            prep("dense_resid_rmsnorm", pa, R);
        } else {             // K16 + K17: only the last token of every sequence goes on to the lm_head
            pa.norm_w = w.final_norm; pa.last_only = 1;
            prep("dense_final_rmsnorm", pa, b);
        }
    }
    const int ksh = dense_gemm(c, lc, "gemm_tc_lm_head", b, w.V, w.H, w.tm_head, d.y.p);
    if (w.tp > 1) {   // vocab-parallel head
        launch(lc, "tp_sum_slices", 0, sum_slices_kernel, dim3(kNumSMs), dim3(256), 0, (const float*)d.y.p, ksh, (long long)b * w.V, b * w.V,
               c.tp_local.p);
        tp_allgather(lc, c.tp_local.p, c.tp_gather.p, (size_t)b * w.V);
        launch(lc, "tp_logits", 0, tp_logits_kernel, dim3(kNumSMs), dim3(256), 0, (const float*)c.tp_gather.p, w.tp, b, w.V, c.logits.p);
        launch(lc, "dense_argmax", 0, dense_argmax_kernel, dim3(b), dim3(1024), 0, (const float*)c.logits.p, 1, (long long)0, w.Vfull, c.logits.p,
               c.next_ids.p);
    } else {
        launch(lc, "dense_argmax", 0, dense_argmax_kernel, dim3(b), dim3(1024), 0, (const float*)d.y.p, ksh, (long long)b * w.V, w.V, c.logits.p,
               c.next_ids.p);
    }
    launch(lc, "advance_state", 0, advance_state_kernel, dim3(1), dim3(kMaxBatch), 0, c.state.p, b, t, loop_mode ? 1 : 0, c.ids.p,
           (const uint32_t*)c.next_ids.p, loop_mode ? 1 : 0, loop_mode ? c.trace.p : (uint32_t*)nullptr,
           loop_mode ? c.trace_pos.p : (int*)nullptr);
}

// mode 0: one decode step of a uniform batch; 1: the same inside the device-resident greedy loop; 2: one decode step of a ragged
// batch (fl_forward_slots: always the dense path, whatever the row count)
static void enqueue_step(fl_cache& c, LaunchCtx& lc, int b, int t, int mode) {
    if (mode == 2) enqueue_forward_dense(c, lc, b, t, false);
    else enqueue_forward(c, lc, b, t, mode == 1);
}

static GraphEntry& get_graph(fl_cache& c, int b, int mode) {
    const GraphKey key{b, mode};
    auto it = c.graphs.find(key);
    if (it != c.graphs.end()) return it->second;
    LaunchCtx lc{c.stream};
    lc.capturing = true;
    cudaGraph_t graph = nullptr;
    FL_CUDA(cudaStreamBeginCapture(c.stream, cudaStreamCaptureModeThreadLocal));
    try {
        enqueue_step(c, lc, b, 1, mode);
    } catch (...) {
        cudaStreamEndCapture(c.stream, &graph);
        if (graph) cudaGraphDestroy(graph);
        throw;
    }
    FL_CUDA(cudaStreamEndCapture(c.stream, &graph));
    GraphEntry e;
    FL_CUDA(cudaGraphInstantiate(&e.exec, graph, 0));
    FL_CUDA(cudaGraphDestroy(graph));
    e.kernels = lc.captured;
    return c.graphs[key] = e;
}

// Enqueues `steps` forward steps of b x t rows on the cache's stream (mode as in enqueue_step; several steps only in the greedy
// loop) and advances kv_len by t per step (not in mode 2: ragged calls keep per-slot lengths).  Batch-1 decode runs in the
// persistent kernel, all steps in one launch.  Other single-token steps replay the step's CUDA graph, except inside a profile
// window, whose per-kernel events a graph cannot record.  Everything else is enqueued kernel by kernel.  `ev`, if given, brackets
// the enqueued work; a graph is captured before it.
static void run_steps(fl_cache& c, int b, int t, int mode, int steps, const EventPair* ev = nullptr) {
    const bool persistent = mode != 2 && b == 1 && t == 1 && c.pk.ok;
    const bool use_graph = !persistent && t == 1 && !g_prof.on && !env_flag("FL_NO_GRAPH");
    const GraphEntry* g = use_graph ? &get_graph(c, b, mode) : nullptr;
    if (ev) FL_CUDA(cudaEventRecord(ev->e0, c.stream));
    if (persistent) {
        launch_persistent(c, steps, mode == 1);
        c.kv_len += steps;
    } else {
        for (int s = 0; s < steps; ++s) {
            if (g) {
                FL_CUDA(cudaGraphLaunch(g->exec, c.stream));
                g_launches.fetch_add(g->kernels);
            } else {
                LaunchCtx lc{c.stream};
                enqueue_step(c, lc, b, t, mode);
            }
            if (mode != 2) c.kv_len += t;
        }
    }
    if (ev) FL_CUDA(cudaEventRecord(ev->e1, c.stream));
}

static void check_call(fl_cache& c, const uint32_t* ids, int b, int t, size_t rope_offset, int extra_steps) {
    const Weights& w = *c.w;
    FL_CHECK(!c.poisoned, FL_ERR_CUDA, "cache poisoned by an earlier CUDA error");
    FL_CHECK(!c.slots_used, FL_ERR_STATE, "this cache is driven by sequence slots (fl_forward_slots): call fl_cache_reset before a uniform call");
    FL_CHECK(ids != nullptr, FL_ERR_INVALID, "ids is NULL");
    FL_CHECK(b >= 1 && b <= c.max_batch && t >= 1, FL_ERR_INVALID, "bad batch / sequence length");
    FL_CHECK(c.kv_len + t + extra_steps <= c.max_seq, FL_ERR_STATE, "KV cache full (kv_len + t > max_seq)");
    FL_CHECK((int64_t)rope_offset + t + extra_steps <= w.max_pos, FL_ERR_INVALID, "RoPE position beyond max_position_embeddings");
    // candle's Llama mask is t x t: a multi-token call on a non-empty cache is a shape error there
    FL_CHECK(!(w.cfg.arch == FL_ARCH_LLAMA && t > 1 && c.kv_len != 0), FL_ERR_INVALID,
             "Llama: multi-token forward needs an empty cache (candle builds a t x t mask)");
    for (int i = 0; i < b * t; ++i) FL_CHECK(ids[i] < (uint32_t)w.Vfull, FL_ERR_INVALID, "token id out of range");
}

static void run_forward(fl_cache& c, const uint32_t* ids, int b, int t, size_t rope_offset) {
    check_call(c, ids, b, t, rope_offset, 0);
    if (uses_dense(c, b * t)) ensure_dense_ws(c, b * t);
    std::memcpy(c.h_ids.p, ids, (size_t)b * t * 4);
    FL_CUDA(cudaMemcpyAsync(c.ids.p, c.h_ids.p, (size_t)b * t * 4, cudaMemcpyHostToDevice, c.stream));
    set_state_kernel<<<1, 1, 0, c.stream>>>(c.state.p, (int)rope_offset);
    g_launches.fetch_add(1);
    c.dw.route_rows = b * t;
    c.fresh_call = c.kv_len == 0 && !c.slots_used;
    run_steps(c, b, t, 0, 1);
}

// Ragged forward (continuous batching): batch row i is the sequence in cache slot slots[i], which holds slot_len[slots[i]]
// tokens and is fed t new ones at RoPE position rope_offsets[i].  Every kernel of the dense path reads the per-row slot / position
// from the step state, so sequences of different lengths share one step; the call always takes the dense (tcgen05) path.
static void run_forward_slots(fl_cache& c, const int* slots, const uint32_t* ids, int n, int t, const size_t* rope_offsets) {
    const Weights& w = *c.w;
    FL_CHECK(!c.poisoned, FL_ERR_CUDA, "cache poisoned by an earlier CUDA error");
    FL_CHECK(slots && ids && rope_offsets, FL_ERR_INVALID, "NULL argument");
    FL_CHECK(n >= 1 && n <= c.max_batch && t >= 1, FL_ERR_INVALID, "bad batch / sequence length");
    FL_CHECK(w.dense_ok, FL_ERR_UNSUPPORTED, "ragged batches run on the dense path: shapes must be multiples of 8");
    FL_CHECK(c.slots_used || c.kv_len == 0, FL_ERR_STATE, "the cache holds tokens of uniform calls: fl_cache_reset before driving it by slots");
    std::vector<char> seen(c.max_batch, 0);
    for (int i = 0; i < n; ++i) {
        const int sl = slots[i];
        FL_CHECK(sl >= 0 && sl < c.max_batch, FL_ERR_INVALID, "slot index out of range");
        FL_CHECK(!seen[sl], FL_ERR_INVALID, "a slot appears twice in one call");
        seen[sl] = 1;
        FL_CHECK(c.slot_len[sl] + t <= c.max_seq, FL_ERR_STATE, "KV cache full (slot length + t > max_seq)");
        FL_CHECK((int64_t)rope_offsets[i] + t <= w.max_pos, FL_ERR_INVALID, "RoPE position beyond max_position_embeddings");
        FL_CHECK(!(w.cfg.arch == FL_ARCH_LLAMA && t > 1 && c.slot_len[sl] != 0), FL_ERR_INVALID,
                 "Llama: multi-token forward needs an empty cache (candle builds a t x t mask)");
    }
    for (int i = 0; i < n * t; ++i) FL_CHECK(ids[i] < (uint32_t)w.Vfull, FL_ERR_INVALID, "token id out of range");
    ensure_dense_ws(c, n * t);
    c.dw.route_rows = n * t;
    c.fresh_call = true;
    for (int i = 0; i < n; ++i) c.fresh_call = c.fresh_call && c.slot_len[slots[i]] == 0;
    c.slots_used = true;
    std::memcpy(c.h_ids.p, ids, (size_t)n * t * 4);
    for (int i = 0; i < n; ++i) {
        c.h_slot_tab.p[i] = slots[i];
        c.h_slot_tab.p[n + i] = (int)rope_offsets[i];
    }
    FL_CUDA(cudaMemcpyAsync(c.ids.p, c.h_ids.p, (size_t)n * t * 4, cudaMemcpyHostToDevice, c.stream));
    FL_CUDA(cudaMemcpyAsync(c.slot_tab.p, c.h_slot_tab.p, (size_t)2 * n * 4, cudaMemcpyHostToDevice, c.stream));
    set_slots_kernel<<<1, 256, 0, c.stream>>>(c.state.p, c.slot_tab.p, n);
    g_launches.fetch_add(1);
    run_steps(c, n, t, 2, 1);
    for (int i = 0; i < n; ++i) c.slot_len[slots[i]] += t;
}

}  // namespace fl

// ------------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------------
using namespace fl;

#define FL_API_BEGIN try {
#define FL_API_END                                                 \
    return FL_OK;                                                  \
    }                                                              \
    catch (const fl::Error& e) {                                   \
        fl::g_last_error = e.what();                               \
        return e.code;                                             \
    }                                                              \
    catch (const std::exception& e) {                              \
        fl::g_last_error = std::string("internal: ") + e.what();   \
        return FL_ERR_INVALID;                                     \
    }

static void check_peer_error() {
    if (!g_peer.ready) return;
    int err = 0;
    FL_CUDA(cudaMemcpy(&err, (uint8_t*)g_peer.local + PeerComm::kErrOff, 4, cudaMemcpyDeviceToHost));
    FL_CHECK(err == 0, FL_ERR_NCCL, "tensor-parallel exchange timed out: a peer rank did not reach the same decode step");
}

static void use_device() {
    const int dev = g_device.load();
    FL_CHECK(dev >= 0, FL_ERR_STATE, "fl_init has not been called");
    FL_CUDA(cudaSetDevice(dev));   // no thread-affine state: callers may hop OS threads between calls (SURVEY.md section 8b)
}

// Body of a forward entry point on model m and its cache c (`args_ok`: the entry point's other pointer arguments are set).
// A CUDA or NCCL error poisons the cache: a missed peer leaves kv_len / exchange epochs out of step.
template <typename F>
static void forward_guard(fl_model* m, fl_cache* c, bool args_ok, F&& body) {
    FL_CHECK(m && c && args_ok, FL_ERR_INVALID, "NULL argument");
    FL_CHECK(m->w != nullptr && m->w.get() == c->w.get(), FL_ERR_INVALID, "cache belongs to a different model");
    use_device();
    try {
        body(*c);
    } catch (const fl::Error& e) {
        if (e.code == FL_ERR_CUDA || e.code == FL_ERR_NCCL) c->poisoned = true;
        throw;
    }
}

extern "C" {

FL_EXPORT const char* fl_last_error(void) { return g_last_error.c_str(); }
FL_EXPORT int fl_version(void) { return 100; }

FL_EXPORT int fl_init(int device) {
    FL_API_BEGIN
    int n = 0;
    FL_CUDA(cudaGetDeviceCount(&n));
    FL_CHECK(n > 0, FL_ERR_CUDA, "no CUDA device visible (this library has no CPU fallback)");
    FL_CHECK(device >= 0 && device < n, FL_ERR_INVALID, "device index out of range");
    cudaDeviceProp prop;
    FL_CUDA(cudaGetDeviceProperties(&prop, device));
    FL_CHECK(prop.major == 10, FL_ERR_UNSUPPORTED,
             std::string("fastllm_b200 is built for sm_100a (B200) only; found ") + prop.name);
    // one process drives ONE GPU (SURVEY.md section 8e: a process per GPU); per-process state -- the opt-in shared-memory
    // attributes of the kernels, the exchange area, the communicator -- is bound to the first device
    const int cur = g_device.load();
    FL_CHECK(cur < 0 || cur == device, FL_ERR_STATE, "fl_init: this process is already bound to device " + std::to_string(cur));
    FL_CUDA(cudaSetDevice(device));
    g_device.store(device);
    FL_API_END
}

FL_EXPORT int fl_device_synchronize(void) {
    FL_API_BEGIN
    use_device();
    FL_CUDA(cudaDeviceSynchronize());
    FL_API_END
}

FL_EXPORT int fl_model_create(const fl_config* cfg, fl_model** out) {
    FL_API_BEGIN
    FL_CHECK(cfg != nullptr && out != nullptr, FL_ERR_INVALID, "NULL argument");
    validate_config(*cfg);   // host logic first: the reference panics on a bad config before anything touches the device (mistral.rs:109-127)
    use_device();
    if (cfg->arch == FL_ARCH_BERT) {
        auto bm = std::make_shared<BertModel>();
        bm->cfg = *cfg;
        bert_build(*bm);
        *out = new fl_model{nullptr, bm};
        return FL_OK;
    }
    if (cfg->tp_size > 1)   // tensor parallel (dense models) or expert parallel (Mixtral)
        FL_CHECK(g_nccl.comm != nullptr && g_nccl.world == cfg->tp_size && g_nccl.rank == cfg->tp_rank, FL_ERR_STATE,
                 "tensor-parallel model: call fl_comm_init(rank, world, id) with world == tp_size first");
    auto w = std::make_shared<Weights>();
    w->cfg = *cfg;
    w->device = g_device.load();
    build_weights(*w);
    *out = new fl_model{w, nullptr};
    FL_API_END
}

FL_EXPORT int fl_model_put_tensor(fl_model* m, const char* name, int dtype, const int64_t* shape, int rank, const void* host_ptr) {
    FL_API_BEGIN
    FL_CHECK(m && name && shape && host_ptr, FL_ERR_INVALID, "NULL argument");
    use_device();
    if (m->bert) {
        std::lock_guard<std::mutex> g(m->bert->mu);
        bert_put_tensor(*m->bert, name, dtype, shape, rank, host_ptr);
        return FL_OK;
    }
    std::lock_guard<std::mutex> g(m->w->mu);
    put_tensor(*m->w, name, dtype, shape, rank, host_ptr);
    FL_API_END
}

FL_EXPORT int fl_model_random_init(fl_model* m, uint64_t seed, float stdv) {
    FL_API_BEGIN
    FL_CHECK(m, FL_ERR_INVALID, "NULL argument");
    use_device();
    if (m->bert) {
        std::lock_guard<std::mutex> g(m->bert->mu);
        bert_random_init(*m->bert, seed, stdv);
        return FL_OK;
    }
    std::lock_guard<std::mutex> g(m->w->mu);
    random_init(*m->w, seed, stdv);
    FL_API_END
}

FL_EXPORT int fl_model_finalize(fl_model* m) {
    FL_API_BEGIN
    FL_CHECK(m, FL_ERR_INVALID, "NULL argument");
    use_device();
    if (m->bert) {
        std::lock_guard<std::mutex> g(m->bert->mu);
        bert_finalize(*m->bert);
        return FL_OK;
    }
    std::lock_guard<std::mutex> g(m->w->mu);
    finalize(*m->w);
    FL_API_END
}

FL_EXPORT int fl_model_clone(fl_model* m, fl_model** out) {
    FL_API_BEGIN
    FL_CHECK(m && out, FL_ERR_INVALID, "NULL argument");
    *out = new fl_model{m->w, m->bert};
    FL_API_END
}

FL_EXPORT int fl_model_destroy(fl_model* m) {
    FL_API_BEGIN
    if (m) {
        use_device();
        delete m;
    }
    FL_API_END
}

FL_EXPORT int fl_model_weight_bytes(fl_model* m, uint64_t* streamed_bytes) {
    FL_API_BEGIN
    FL_CHECK(m && streamed_bytes, FL_ERR_INVALID, "NULL argument");
    FL_CHECK(m->w != nullptr, FL_ERR_INVALID, "not a causal LM");
    *streamed_bytes = m->w->streamed_bytes;
    FL_API_END
}

FL_EXPORT int fl_cache_create(fl_model* m, int max_batch, int max_seq, fl_cache** out) {
    FL_API_BEGIN
    FL_CHECK(m && out, FL_ERR_INVALID, "NULL argument");
    FL_CHECK(m->w != nullptr, FL_ERR_INVALID, "BERT models have no KV cache");
    use_device();
    std::unique_ptr<fl_cache> c(new fl_cache);
    c->w = m->w;
    cache_create(*c, max_batch, max_seq);
    *out = c.release();
    FL_API_END
}

FL_EXPORT int fl_cache_reset(fl_cache* c) {
    FL_API_BEGIN
    FL_CHECK(c, FL_ERR_INVALID, "NULL argument");
    use_device();
    reset_state_kernel<<<1, 256, 0, c->stream>>>(c->state.p, 0);
    g_launches.fetch_add(1);
    FL_CUDA(cudaStreamSynchronize(c->stream));
    c->kv_len = 0;
    c->slots_used = false;
    std::fill(c->slot_len.begin(), c->slot_len.end(), 0);
    FL_API_END
}

FL_EXPORT int fl_cache_slot_reset(fl_cache* c, int slot) {
    FL_API_BEGIN
    FL_CHECK(c, FL_ERR_INVALID, "NULL argument");
    FL_CHECK(slot >= 0 && slot < c->max_batch, FL_ERR_INVALID, "slot index out of range");
    use_device();
    reset_slot_kernel<<<1, 1, 0, c->stream>>>(c->state.p, slot);
    g_launches.fetch_add(1);
    c->slot_len[slot] = 0;
    FL_API_END
}

FL_EXPORT int fl_cache_slot_len(fl_cache* c, int slot, int* out) {
    FL_API_BEGIN
    FL_CHECK(c && out, FL_ERR_INVALID, "NULL argument");
    FL_CHECK(slot >= 0 && slot < c->max_batch, FL_ERR_INVALID, "slot index out of range");
    *out = c->slot_len[slot];
    FL_API_END
}

FL_EXPORT int fl_cache_moe_routing(fl_cache* c, int rows, int32_t* experts, float* margins) {
    FL_API_BEGIN
    FL_CHECK(c && experts && margins, FL_ERR_INVALID, "NULL argument");
    const Weights& w = *c->w;
    FL_CHECK(w.cfg.arch == FL_ARCH_MIXTRAL, FL_ERR_UNSUPPORTED, "routing records exist for the MoE architecture only");
    FL_CHECK(!c->poisoned, FL_ERR_CUDA, "cache poisoned by an earlier CUDA error");
    FL_CHECK(rows >= 1 && rows == c->dw.route_rows, FL_ERR_INVALID, "rows must equal batch x t of the last forward on this cache");
    FL_CUDA(cudaStreamSynchronize(c->stream));
    FL_CUDA(cudaMemcpy(experts, c->dw.route_sel.p, (size_t)w.L * rows * w.top_k * 4, cudaMemcpyDeviceToHost));
    FL_CUDA(cudaMemcpy(margins, c->dw.route_margin.p, (size_t)w.L * rows * 4, cudaMemcpyDeviceToHost));
    FL_API_END
}

FL_EXPORT int fl_cache_kv_len(fl_cache* c, int* out) {
    FL_API_BEGIN
    FL_CHECK(c && out, FL_ERR_INVALID, "NULL argument");
    *out = c->kv_len;
    FL_API_END
}

FL_EXPORT int fl_cache_fill_synthetic(fl_cache* c, int batch, int kv_len, uint64_t seed) {
    FL_API_BEGIN
    FL_CHECK(c, FL_ERR_INVALID, "NULL argument");
    FL_CHECK(batch >= 1 && batch <= c->max_batch && kv_len >= 0 && kv_len <= c->max_seq, FL_ERR_INVALID, "bad synthetic fill size");
    use_device();
    const RowMap ident{0, 0, 0, 0};
    synth_fill_bf16_kernel<<<kNumSMs * 8, 256, 0, c->stream>>>(c->kpool.p, 1, (int64_t)c->kpool.n, (int64_t)c->kpool.n, tensor_seed(seed, "kv.k"), 0.5f, ident);
    synth_fill_bf16_kernel<<<kNumSMs * 8, 256, 0, c->stream>>>(c->vpool.p, 1, (int64_t)c->vpool.n, (int64_t)c->vpool.n, tensor_seed(seed, "kv.v"), 0.5f, ident);
    reset_state_kernel<<<1, 256, 0, c->stream>>>(c->state.p, kv_len);
    g_launches.fetch_add(3);
    FL_CUDA(cudaStreamSynchronize(c->stream));
    c->kv_len = kv_len;
    FL_API_END
}

FL_EXPORT int fl_cache_destroy(fl_cache* c) {
    FL_API_BEGIN
    if (c) {
        use_device();
        if (c->stream) cudaStreamSynchronize(c->stream);
        cache_destroy_graphs(*c);
        if (c->stream) cudaStreamDestroy(c->stream);
        delete c;
    }
    FL_API_END
}

FL_EXPORT int fl_forward(fl_model* m, fl_cache* c, const uint32_t* ids, int b, int t, size_t rope_offset, float* logits_host) {
    FL_API_BEGIN
    forward_guard(m, c, logits_host, [&](fl_cache& c) {
        run_forward(c, ids, b, t, rope_offset);
        const size_t n = (size_t)b * c.w->Vfull;
        FL_CUDA(cudaMemcpyAsync(c.h_logits.p, c.logits.p, n * 4, cudaMemcpyDeviceToHost, c.stream));
        FL_CUDA(cudaStreamSynchronize(c.stream));
        check_peer_error();
        std::memcpy(logits_host, c.h_logits.p, n * 4);
    });
    FL_API_END
}

FL_EXPORT int fl_forward_greedy(fl_model* m, fl_cache* c, const uint32_t* ids, int b, int t, size_t rope_offset, uint32_t* next_ids) {
    FL_API_BEGIN
    forward_guard(m, c, next_ids, [&](fl_cache& c) {
        run_forward(c, ids, b, t, rope_offset);
        FL_CUDA(cudaMemcpyAsync(c.h_ids.p, c.next_ids.p, (size_t)b * 4, cudaMemcpyDeviceToHost, c.stream));
        FL_CUDA(cudaStreamSynchronize(c.stream));
        check_peer_error();
        std::memcpy(next_ids, c.h_ids.p, (size_t)b * 4);
    });
    FL_API_END
}

FL_EXPORT int fl_decode_greedy_loop(fl_model* m, fl_cache* c, const uint32_t* first_ids, int b, size_t rope_offset, int steps,
                          uint32_t* out_ids, float* elapsed_ms) {
    FL_API_BEGIN
    forward_guard(m, c, true, [&](fl_cache& c) {
        FL_CHECK(steps >= 1, FL_ERR_INVALID, "steps must be >= 1");
        check_call(c, first_ids, b, 1, rope_offset, steps - 1);
        if (uses_dense(c, b)) ensure_dense_ws(c, b);
        if (c.trace_cap < (size_t)steps * b) {
            c.trace.alloc((size_t)steps * b);
            c.trace_cap = (size_t)steps * b;
            cache_destroy_graphs(c);   // captured graphs hold the old trace pointer
        }
        std::memcpy(c.h_ids.p, first_ids, (size_t)b * 4);
        FL_CUDA(cudaMemcpyAsync(c.ids.p, c.h_ids.p, (size_t)b * 4, cudaMemcpyHostToDevice, c.stream));
        FL_CUDA(cudaMemsetAsync(c.trace_pos.p, 0, 4, c.stream));
        set_state_kernel<<<1, 1, 0, c.stream>>>(c.state.p, (int)rope_offset);
        g_launches.fetch_add(1);
        EventPair ev;
        run_steps(c, b, 1, 1, steps, &ev);     // batch 1: all steps inside one persistent launch
        FL_CUDA(cudaStreamSynchronize(c.stream));
        check_peer_error();
        float ms = 0.f;
        FL_CUDA(cudaEventElapsedTime(&ms, ev.e0, ev.e1));
        if (elapsed_ms) *elapsed_ms = ms;
        if (out_ids) FL_CUDA(cudaMemcpy(out_ids, c.trace.p, (size_t)steps * b * 4, cudaMemcpyDeviceToHost));
    });
    FL_API_END
}

// ---- sampling (host code; the reference samples on the host from the logits of every forward, models/mod.rs:425-428) ----
struct fl_sampler {
    fl::LogitsProcessor lp;
    fl_sampler(uint64_t seed, double temperature) : lp(seed, temperature) {}
};

// One host-side sample; a sampler error (e.g. logits that are all NaN) is an invalid argument at the C ABI.
static uint32_t sample_host(fl_sampler* s, const float* logits_host, size_t n) {
    try {
        return s->lp.sample(logits_host, n);
    } catch (const fl::SamplerError& e) {
        throw fl::Error(FL_ERR_INVALID, e.what());
    }
}

FL_EXPORT int fl_sampler_create(uint64_t seed, double temperature, fl_sampler** out) {
    FL_API_BEGIN
    FL_CHECK(out, FL_ERR_INVALID, "NULL argument");
    FL_CHECK(!std::isnan(temperature), FL_ERR_INVALID, "temperature is NaN");
    *out = new fl_sampler(seed, temperature);
    FL_API_END
}

FL_EXPORT int fl_sampler_sample(fl_sampler* s, const float* logits_host, size_t n, uint32_t* token) {
    FL_API_BEGIN
    FL_CHECK(s && logits_host && token, FL_ERR_INVALID, "NULL argument");
    *token = sample_host(s, logits_host, n);
    FL_API_END
}

FL_EXPORT int fl_argmax_rows(const float* logits_host, int rows, size_t n, uint32_t* tokens) {
    FL_API_BEGIN
    FL_CHECK(logits_host && tokens && rows >= 0 && n > 0, FL_ERR_INVALID, "bad argument");
    // a batch of rows is a memory-bound scan of rows * n * 4 bytes: fan it out over a few host threads
    const int nthr = (size_t)rows * n >= ((size_t)1 << 20) ? std::min(rows, 8) : 1;
    auto scan = [&](int r0, int r1) {
        for (int r = r0; r < r1; ++r) tokens[r] = fl::sample_argmax(logits_host + (size_t)r * n, n);
    };
    if (nthr <= 1) {
        scan(0, rows);
    } else {
        std::vector<std::thread> pool;
        for (int i = 1; i < nthr; ++i) pool.emplace_back(scan, (int)((long long)rows * i / nthr), (int)((long long)rows * (i + 1) / nthr));
        scan(0, rows / nthr);
        for (std::thread& th : pool) th.join();
    }
    FL_API_END
}

FL_EXPORT int fl_sampler_next_u32(fl_sampler* s, uint32_t* out) {
    FL_API_BEGIN
    FL_CHECK(s && out, FL_ERR_INVALID, "NULL argument");
    *out = s->lp.next_u32();
    FL_API_END
}

FL_EXPORT int fl_sampler_destroy(fl_sampler* s) {
    FL_API_BEGIN
    delete s;
    FL_API_END
}

FL_EXPORT int fl_forward_sample(fl_model* m, fl_cache* c, const uint32_t* ids, int b, int t, size_t rope_offset, fl_sampler* s,
                                uint32_t* next_id) {
    FL_API_BEGIN
    forward_guard(m, c, s && next_id, [&](fl_cache& c) {
        run_forward(c, ids, b, t, rope_offset);
        // only row 0 is sampled (logits.get(0)?.flatten_all()?, models/mod.rs:421): one V*4-byte read-back into the pinned staging row
        const size_t n = c.w->Vfull;
        FL_CUDA(cudaMemcpyAsync(c.h_logits.p, c.logits.p, n * 4, cudaMemcpyDeviceToHost, c.stream));
        FL_CUDA(cudaStreamSynchronize(c.stream));
        check_peer_error();
        *next_id = sample_host(s, c.h_logits.p, n);
    });
    FL_API_END
}

FL_EXPORT int fl_forward_slots(fl_model* m, fl_cache* c, const int* slots, const uint32_t* ids, int n, int t, const size_t* rope_offsets,
                               float* logits_host) {
    FL_API_BEGIN
    forward_guard(m, c, logits_host, [&](fl_cache& c) {
        run_forward_slots(c, slots, ids, n, t, rope_offsets);
        const size_t cnt = (size_t)n * c.w->Vfull;
        FL_CUDA(cudaMemcpyAsync(c.h_logits.p, c.logits.p, cnt * 4, cudaMemcpyDeviceToHost, c.stream));
        FL_CUDA(cudaStreamSynchronize(c.stream));
        check_peer_error();
        std::memcpy(logits_host, c.h_logits.p, cnt * 4);
    });
    FL_API_END
}

FL_EXPORT int fl_forward_sample_device(fl_model* m, fl_cache* c, const uint32_t* ids, int b, int t, size_t rope_offset, fl_sampler* s,
                                       uint32_t* next_id) {
    FL_API_BEGIN
    forward_guard(m, c, s && next_id, [&](fl_cache& c) {
        run_forward(c, ids, b, t, rope_offset);
        const uint32_t* src = c.next_ids.p;                       // temperature below 1e-7: the arg-max the forward already computed
        if (!s->lp.is_argmax()) {
            // row 0 only (logits.get(0)?, models/mod.rs:421); ONE generator draw per sample, exactly as on the host path
            const float u = s->lp.draw_unit();
            sample_softmax_kernel<<<1, 1024, 0, c.stream>>>(c.logits.p, c.w->Vfull, s->lp.inv_temperature(), u, c.sample_out.p);
            g_launches.fetch_add(1);
            src = c.sample_out.p;
        }
        FL_CUDA(cudaMemcpyAsync(c.h_ids.p, src, 4, cudaMemcpyDeviceToHost, c.stream));
        FL_CUDA(cudaStreamSynchronize(c.stream));
        check_peer_error();
        *next_id = c.h_ids.p[0];
    });
    FL_API_END
}

FL_EXPORT int fl_embed(fl_model* m, const uint32_t* ids, const uint32_t* mask, int b, int t, float* out) {
    FL_API_BEGIN
    FL_CHECK(m && ids && out, FL_ERR_INVALID, "NULL argument");
    FL_CHECK(m->bert != nullptr, FL_ERR_INVALID, "fl_embed needs a BERT-family model (the reference panics on embedding_size() of chat models, models/mod.rs:97-106)");
    use_device();
    bert_embed(*m->bert, ids, mask, b, t, out);
    FL_API_END
}

FL_EXPORT int fl_embed_packed(fl_model* m, const uint32_t* ids, const int32_t* lengths, int n, float* out) {
    FL_API_BEGIN
    FL_CHECK(m && ids && lengths && out, FL_ERR_INVALID, "NULL argument");
    FL_CHECK(m->bert != nullptr, FL_ERR_INVALID, "fl_embed_packed needs a BERT-family model (the reference panics on embedding_size() of chat models, models/mod.rs:97-106)");
    use_device();
    bert_embed_packed(*m->bert, ids, lengths, n, out);
    FL_API_END
}

FL_EXPORT int fl_embed_timed(fl_model* m, const uint32_t* ids, const uint32_t* mask, int b, int t, float* out, int repeats, float* device_ms) {
    FL_API_BEGIN
    FL_CHECK(m && ids && out && device_ms, FL_ERR_INVALID, "NULL argument");
    FL_CHECK(m->bert != nullptr, FL_ERR_INVALID, "fl_embed_timed needs a BERT-family model");
    use_device();
    bert_embed(*m->bert, ids, mask, b, t, out);
    bert_repeat(*m->bert, b, t, repeats < 1 ? 1 : repeats, device_ms);
    FL_API_END
}

FL_EXPORT int fl_comm_unique_id(void* out) {
    FL_API_BEGIN
    FL_CHECK(out != nullptr, FL_ERR_INVALID, "NULL argument");
    g_nccl.load();
    ncclUniqueId id;
    g_nccl.check(g_nccl.GetUniqueId(&id), "ncclGetUniqueId");
    static_assert(sizeof(id) == 128, "ncclUniqueId is 128 bytes");
    std::memcpy(out, &id, sizeof(id));
    FL_API_END
}
FL_EXPORT int fl_comm_init(int rank, int world, const void* id_bytes) {
    FL_API_BEGIN
    FL_CHECK(id_bytes != nullptr && world >= 1 && rank >= 0 && rank < world, FL_ERR_INVALID, "bad communicator arguments");
    use_device();
    g_nccl.load();
    FL_CHECK(g_nccl.comm == nullptr, FL_ERR_STATE, "communicator already initialised");
    ncclUniqueId id;
    std::memcpy(&id, id_bytes, sizeof(id));
    g_nccl.check(g_nccl.CommInitRank(&g_nccl.comm, world, id, rank), "ncclCommInitRank");
    g_nccl.rank = rank;
    g_nccl.world = world;
    FL_API_END
}
FL_EXPORT int fl_comm_ipc_export(void* handle_64_bytes) {
    FL_API_BEGIN
    FL_CHECK(handle_64_bytes != nullptr, FL_ERR_INVALID, "NULL argument");
    use_device();
    if (!g_peer.local) {
        FL_CUDA(cudaMalloc(&g_peer.local, PeerComm::kBytes));
        FL_CUDA(cudaMemset(g_peer.local, 0, PeerComm::kBytes));
        FL_CUDA(cudaDeviceSynchronize());
    }
    cudaIpcMemHandle_t h;
    FL_CUDA(cudaIpcGetMemHandle(&h, g_peer.local));
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    std::memcpy(handle_64_bytes, &h, sizeof(h));
    FL_API_END
}
FL_EXPORT int fl_comm_ipc_import(const void* handles, int world, int rank) {
    FL_API_BEGIN
    FL_CHECK(handles != nullptr && world >= 1 && world <= PeerComm::kMaxTp && rank >= 0 && rank < world, FL_ERR_INVALID, "bad arguments");
    FL_CHECK(g_peer.local != nullptr, FL_ERR_STATE, "call fl_comm_ipc_export first");
    use_device();
    for (int r = 0; r < world; ++r) {
        if (r == rank) {
            g_peer.peer[r] = g_peer.local;
        } else {
            cudaIpcMemHandle_t h;
            std::memcpy(&h, (const uint8_t*)handles + (size_t)r * 64, 64);
            FL_CUDA(cudaIpcOpenMemHandle(&g_peer.peer[r], h, cudaIpcMemLazyEnablePeerAccess));
        }
    }
    g_peer.ready = true;
    FL_API_END
}
FL_EXPORT int fl_comm_destroy(void) {
    FL_API_BEGIN
    if (g_nccl.comm) {
        use_device();
        FL_CUDA(cudaDeviceSynchronize());
        g_nccl.CommDestroy(g_nccl.comm);
        g_nccl.comm = nullptr;
    }
    FL_API_END
}

FL_EXPORT int fl_prof_begin(void) {
    FL_API_BEGIN
    use_device();
    FL_CUDA(cudaDeviceSynchronize());
    g_prof.entries.clear();
    g_prof.on = true;
    FL_API_END
}

FL_EXPORT int fl_prof_end(char* json_out, size_t cap) {
    FL_API_BEGIN
    use_device();
    FL_CUDA(cudaDeviceSynchronize());
    g_prof.on = false;
    struct Agg { uint64_t n = 0, bytes = 0; double ms = 0; };
    std::map<std::string, Agg> agg;
    std::vector<std::string> order;
    for (auto& e : g_prof.entries) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e.e0, e.e1);
        cudaEventDestroy(e.e0);
        cudaEventDestroy(e.e1);
        if (!agg.count(e.tag)) order.push_back(e.tag);
        Agg& a = agg[e.tag];
        a.n++; a.bytes += e.bytes; a.ms += ms;
    }
    g_prof.entries.clear();
    std::ostringstream os;
    os << "[";
    for (size_t i = 0; i < order.size(); ++i) {
        const Agg& a = agg[order[i]];
        os << (i ? "," : "") << "{\"kernel\":\"" << order[i] << "\",\"launches\":" << a.n << ",\"ms\":" << a.ms << ",\"bytes\":" << a.bytes << "}";
    }
    os << "]";
    const std::string s = os.str();
    FL_CHECK(json_out && cap > s.size(), FL_ERR_INVALID, "profile buffer too small");
    std::memcpy(json_out, s.c_str(), s.size() + 1);
    FL_API_END
}

FL_EXPORT int fl_launch_count(uint64_t* n) {
    FL_API_BEGIN
    FL_CHECK(n, FL_ERR_INVALID, "NULL argument");
    *n = g_launches.load();
    FL_API_END
}

}  // extern "C"
