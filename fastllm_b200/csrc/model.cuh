// Model / cache objects behind the C ABI (declarations).
#pragma once
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/fastllm_b200.h"
#include "bert_model.cuh"
#include "decode_persistent.cuh"
#include "gemv.cuh"
#include "kv_pool.hpp"
#include "runtime.cuh"
#include "tensor_table.hpp"

namespace fl {

struct LayerW {
    uint16_t* wqkv = nullptr;   // [(nh + 2 nkv) d, H]  q | k | v rows; q/k rows pair-permuted per head for RoPE
    float* bqkv = nullptr;      // [(nh + 2 nkv) d] or null (same permutation)
    uint16_t* wo = nullptr;     // [H, nh d]
    uint16_t* wgu = nullptr;    // [2 I, H]  row 2j = gate_j, row 2j+1 = up_j
    uint16_t* wdown = nullptr;  // [H, I]
    float* ln1 = nullptr;       // [H]
    float* ln2 = nullptr;       // [H]
    CUtensorMap tm_wqkv, tm_wo, tm_wgu, tm_wdown;   // TMA descriptors of the weights (dense tcgen05 path)
    // Mixtral sparse-MoE: router + this rank's experts (w1|w3 interleaved like wgu, w2 like wdown)
    float* wgate = nullptr;                         // [E, H] f32 (bf16-rounded values)
    std::vector<uint16_t*> ewgu, ewdown;
    std::vector<CUtensorMap> tm_ewgu, tm_ewdown;
    // the same expert matrices as ONE stacked tensor each (they are allocated back to back): [E_local * 2I, H] and
    // [E_local * H, I], the A operands of the grouped expert GEMMs
    CUtensorMap tm_ewgu_all, tm_ewdown_all;
};

// Immutable after finalize; shared (ref-counted) between fl_model clones and their caches.
struct Weights {
    fl_config cfg{};
    int H = 0, I = 0, V = 0, L = 0, nh = 0, nkv = 0, d = 0, max_pos = 0;
    int nqkv = 0;               // (nh + 2 nkv) * d   (nh, nkv, I, V, nqkv are LOCAL to this tensor-parallel rank)
    int tp = 1, rank = 0;       // tensor-parallel size / rank of this process
    // this rank's attention heads: full-model q heads [q_head0, q_head0 + q_real) (nh - q_real trailing local heads are zero
    // padding: tp > kv heads replicates a kv head on tp / nkv ranks and splits its query group between them), kv heads
    // [kv_head0, kv_head0 + nkv)
    int q_head0 = 0, q_real = 0, kv_head0 = 0;
    int E = 0, top_k = 0;       // Mixtral: experts / experts per token
    int ep = 1, E_local = 0;    // expert parallelism: this rank holds experts [rank * E_local, (rank + 1) * E_local)
    bool ep_dp = false;         // expert parallelism with data-parallel attention (fl_config.ep_dp_attention)
    int Vfull = 0;              // full vocabulary (embedding table rows, logits length); V = Vfull / tp rows of lm_head live here
    int device = 0;
    TensorTable table;
    uint16_t* embed = nullptr;  // [V, H]
    uint16_t* lm_head = nullptr;
    float* final_norm = nullptr;
    std::vector<LayerW> layers;
    DevBuf<PkLayer> pk_layers;  // device copy of the per-layer pointers for the persistent decode kernel
    DevBuf<CUtensorMap> pk_tmaps; // [4 L + 1] 3-D TMA descriptors of the weight stream (phase g = 4 layer + {qkv, o, gate|up, down}; lm_head last)
    float* rope_cos = nullptr;  // [max_pos, d/2]
    float* rope_sin = nullptr;
    uint64_t streamed_bytes = 0;
    CUtensorMap tm_head;
    bool dense_ok = false;      // shapes admit the dense (tcgen05) path for 3+ rows
    std::mutex mu;
};

// Shared-memory plan of the persistent decode kernel for one (model, cache) pair.
struct PkPlan {
    bool ok = false;
    int nstages = 0, xs_floats = 0, partial_rows = 0, nsplit = 1;
    size_t smem = 0;
};

// Workspace of the dense (tensor-core) path, sized for the largest row count seen so far.
struct DenseWs {
    size_t rows = 0;
    DevBuf<uint16_t> xhi, xlo;  // [rows, Kmax] hi/lo bf16 split of the activations fed to the next GEMM
    DevBuf<float> y;            // [rows, Nmax] GEMM output
    DevBuf<float> resid, q;
    DevBuf<float> tp_buf;       // [rows, H] reduced partial sums awaiting the all-reduce (tp > 1)
    DevBuf<uint16_t> xhi2, xlo2; // Mixtral: expert activations (the block input xhi/xlo is shared by all experts)
    DevBuf<uint16_t> vt;            // V of the current multi-token call transposed per page: [seq][kv head][page][d][64] (tcgen05 prefill attention)
    size_t vt_pages_cap = 0;        // pages the scratch holds (over all sequences of a call)
    CUtensorMap tm_vt{};
    DevBuf<uint16_t> kt;            // FP8 caches: K of the call as bf16 in pages [tile][64][d], tiles numbered as vt's (tcgen05 prefill attention)
    CUtensorMap tm_kt{};
    DevBuf<float> sk_acc, sk_ml;    // stream-K decode attention: [CTAs][2][n_rep][d] / [CTAs][2][n_rep][2] partials of shared pairs
    DevBuf<float> moe_out, route_w;
    DevBuf<int> route_sel;          // [L][rows of the call][top_k] picked experts of the last forward (fl_cache_moe_routing)
    DevBuf<float> route_margin;     // [L][rows of the call]
    int route_rows = 0;             // rows of the last Mixtral forward
    // grouped expert GEMMs (decode batches): per-expert blocks of gathered rows, their counts, and the row -> slot map
    DevBuf<uint16_t> gx_hi, gx_lo;   // [E_local * rows per expert block (16 / 32 / 64 / 128), H]
    DevBuf<int> grp_cnt, grp_pos;    // [E_local], [expert rows (rows, or rows * ep), E_local]
    // expert parallelism with data-parallel attention: dispatch / combine staging (all rows of all ranks, rank-major)
    DevBuf<uint16_t> g_xhi, g_xlo;   // [ep * rows, H] gathered block inputs
    DevBuf<float> g_route;           // [ep * rows, E]
    DevBuf<float> comb;              // [ep sources][rows, H] expert outputs returned to this rank
    // (batched-decode attention partials: sk_acc / sk_ml above)
    DevBuf<int> counters;
    // scoring calls (fl_forward_logprobs), sized on first use for lp_rows rows
    size_t lp_rows = 0;
    DevBuf<LogprobPart> lp_part;     // [rows][lm_head N tiles][4] soft-max partials of the lm_head epilogue
    DevBuf<float> lp_target_logit;   // [rows]
    DevBuf<uint32_t> lp_targets;     // [rows]
    DevBuf<uint32_t> lp_out;         // [2][rows]: log-probs (f32 bits), then arg-max ids
    PinnedBuf<uint32_t> h_lp;        // [2][rows] staging: the targets up, lp_out down
};

struct GraphKey {
    int b;
    int loop;
    bool operator<(const GraphKey& o) const { return b != o.b ? b < o.b : loop < o.loop; }
};
struct GraphEntry {
    cudaGraphExec_t exec = nullptr;
    uint64_t kernels = 0;
};

}  // namespace fl

struct fl_model {
    std::shared_ptr<fl::Weights> w;       // causal LMs
    std::shared_ptr<fl::BertModel> bert;  // BERT-family encoder (arch == FL_ARCH_BERT)
};

struct fl_cache {
    std::shared_ptr<fl::Weights> w;
    cudaStream_t stream = nullptr;
    int max_batch = 0, max_seq = 0, pages_per_seq = 0, nsplit = 1;
    int kv_len = 0;                       // host mirror of StepState.kv_base (same for every sequence; the uniform calls)
    // continuous batching (fl_forward_slots): every sequence slot has its own length; once a slot call was made the cache is
    // driven by slots until fl_cache_reset
    bool slots_used = false;
    std::vector<int> slot_len;            // host mirror of StepState.kv_base per slot
    fl::DevBuf<int> slot_tab;             // [2 * max_batch] staging of (slot, RoPE position) per batch row
    fl::PinnedBuf<int> h_slot_tab;
    // packed calls (fl_forward_packed): ids, row table, per-sequence tables and attention work lists of one call, uploaded at once
    fl::DevBuf<int> pack_tab;
    fl::PinnedBuf<int> h_pack_tab;
    std::vector<int> pack_perm;           // row of the last forward's internal row r in the caller's ids order (packed calls), else empty
    fl::DevBuf<uint32_t> sample_out;      // device-side sampling: the picked token
    fl::DevBuf<fl::StepState> state;
    fl::DevBuf<int> page_table;           // [max_batch, pages_per_seq]
    fl::KvPool pool;                      // owner of every page: refcounts, per-slot page lists, the host side of page_table
    fl::DevBuf<int2> pt_upd;              // (table index, page) of the entries a call changed, scattered into page_table
    fl::PinnedBuf<int2> h_pt_upd;
    fl::DevBuf<uint16_t> kpool, vpool;    // [L][pool pages][nkv][kKvPage][d] elements of kv_bytes bytes (bf16, or e4m3 when kv_fp8)
    size_t layer_pool_elems = 0;
    bool kv_fp8 = false;                  // FL_KV_FP8_E4M3: K/V pages hold e4m3; driven by slot and packed calls only
    int kv_bytes = 2;                     // bytes per K/V element
    CUtensorMap tm_kpool{}, tm_vpool{};   // the pools as [rows, d] matrices (stream-K decode attention); valid when kv_tmaps
    bool kv_tmaps = false;
    bool fresh_call = false;              // the forward being enqueued starts on empty sequences (every row's KV length is 0)
    fl::DevBuf<uint32_t> ids, next_ids, trace;
    fl::DevBuf<int> trace_pos;
    fl::DevBuf<float> resid, q, attn_out, act, logits, part_acc, part_ml, amax_val;
    fl::DevBuf<int> amax_idx, counters;
    fl::PinnedBuf<uint32_t> h_ids;
    fl::PinnedBuf<float> h_logits;
    size_t trace_cap = 0;
    int amax_parts = 0;
    std::map<fl::GraphKey, fl::GraphEntry> graphs;
    fl::PkPlan pk;
    fl::DenseWs dw;
    fl::DevBuf<unsigned int> gbar;
    fl::DevBuf<unsigned int> pk_pool;  // persistent decode kernel: ticket counters of the per-phase dynamic block pools
    fl::DevBuf<uint16_t> pk_xhl;    // persistent decode kernel: hi/lo bf16 hand-over of attn_out and the MLP activation
    fl::DevBuf<float> resid2;        // second residual buffer (tp > 1: the fused residual-add prologue ping-pongs)
    fl::DevBuf<float> tp_buf;        // [rows, H] partial o_proj / down_proj outputs awaiting the all-reduce (tp > 1)
    fl::DevBuf<float> tp_gather;     // [tp, max_batch, V] vocab-parallel logits gathered from all ranks
    fl::DevBuf<float> tp_local;      // [max_batch, V] this rank's logits slice
    bool poisoned = false;
};
