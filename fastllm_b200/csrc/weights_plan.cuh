// Plan step of fl_model_create for both model kinds: check the config, set the dimensions, and register every HuggingFace
// tensor the model reads in its TensorTable, laying out the weight slab as it goes.  No CUDA call: the slab is made afterwards
// by TensorTable::alloc(), so tests/tensor_table_dump.cu runs this on a machine without a GPU.
#pragma once
#include <algorithm>

#include "model.cuh"

namespace fl {

inline void plan_weights(Weights& w) {
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
    FL_CHECK(c.arch != FL_ARCH_BERT, FL_ERR_INVALID, "internal: BERT goes through bert_plan");

    // The slab in allocation order: embed, lm_head, final norm, per layer q|k|v, its bias, o, router + experts or gate|up + down,
    // the two norms; then the RoPE tables.  Each tensor is registered with the buffer it lands in.
    TensorTable& t = w.table;
    const int64_t H = w.H, I = w.I, V = w.V, d = w.d, nq = (int64_t)w.nh * d, nk = (int64_t)w.nkv * d, tp = w.tp, rk = trank;
    // this rank's head windows of the attention tensors: q rows [q0, q0 + qreal) (nq - qreal trailing local rows are zero
    // padding), k / v rows [k0, k0 + nk)
    const int64_t qreal = (int64_t)w.q_real * d, q0 = (int64_t)w.q_head0 * d, k0 = (int64_t)w.kv_head0 * d;
    const RowMap ident{0, 0, 0, 0}, ropeq{0, 1, (int32_t)d, 0}, ropek{nq, 1, (int32_t)d, 0}, vmap{nq + nk, 0, 0, 0},
                 gate{0, 2, 0, 0}, up{0, 2, 0, 1};
    // bf16 matrix: local [rows, cols] (row stride ld) = window (row0, col0) of the full [full_rows, full_cols] tensor
    auto mat = [&](const std::string& name, size_t off, int64_t rows, int64_t cols, int64_t ld, RowMap m, int64_t full_rows,
                   int64_t full_cols, int64_t row0, int64_t col0, bool required = true) {
        t.add({name, true, off, rows, cols, ld, m, full_rows, full_cols, row0, col0, false, false, required});
    };
    // f32 vector holding bf16-rounded values: local [rows] = rows [row0, row0 + rows) of the full [full_rows] tensor
    auto vec = [&](const std::string& name, size_t off, int64_t rows, RowMap m, int64_t full_rows, int64_t row0, bool ones) {
        t.add({name, false, off, rows, 1, 1, m, full_rows, 1, row0, 0, ones, true, true});
    };
    mat("model.embed_tokens.weight", t.take(w.Vfull * H * 2, w.embed), w.Vfull, H, H, ident, w.Vfull, H, 0, 0);
    // optional: without it the head is tied to the embedding (finalize)
    mat("lm_head.weight", t.take(V * H * 2, w.lm_head), V, H, H, ident, V * tp, H, rk * V, 0, false);
    vec("model.norm.weight", t.take(H * 4, w.final_norm), H, ident, H, 0, true);
    w.layers.resize(w.L);
    for (int l = 0; l < w.L; ++l) {
        LayerW& lw = w.layers[l];
        const std::string p = "model.layers." + std::to_string(l) + ".";
        const size_t o_qkv = t.take(w.nqkv * H * 2, lw.wqkv);
        mat(p + "self_attn.q_proj.weight", o_qkv, qreal, H, H, ropeq, nh_f * d, H, q0, 0);
        mat(p + "self_attn.k_proj.weight", o_qkv, nk, H, H, ropek, nkv_f * d, H, k0, 0);
        mat(p + "self_attn.v_proj.weight", o_qkv, nk, H, H, vmap, nkv_f * d, H, k0, 0);
        if (c.qkv_bias) {
            const size_t o_b = t.take(w.nqkv * 4, lw.bqkv);
            vec(p + "self_attn.q_proj.bias", o_b, qreal, ropeq, nh_f * d, q0, false);
            vec(p + "self_attn.k_proj.bias", o_b, nk, ropek, nkv_f * d, k0, false);
            vec(p + "self_attn.v_proj.bias", o_b, nk, vmap, nkv_f * d, k0, false);
        }
        mat(p + "self_attn.o_proj.weight", t.take(H * nq * 2, lw.wo), H, qreal, nq, ident, H, nh_f * d, 0, q0);
        if (moe) {
            vec(p + "block_sparse_moe.gate.weight", t.take(w.E * H * 4, lw.wgate), w.E * H, ident, w.E * H, 0, false);  // [E, H] in f32
            // a layer's w1|w3 matrices back to back, then its w2 matrices back to back: each set is also ONE stacked matrix
            // ([E_local * 2I, H] / [E_local * H, I]), the A operand of the grouped expert GEMMs.  Only this rank's experts are
            // registered: the others are ignored on upload.
            const size_t gu0 = t.take(w.E_local * 2 * I * H * 2), dn0 = t.take(w.E_local * H * I * 2);
            lw.ewgu.resize(w.E_local);
            lw.ewdown.resize(w.E_local);
            for (int e = 0; e < w.E_local; ++e) {
                const size_t o_gu = gu0 + e * 2 * I * H * 2, o_dn = dn0 + e * H * I * 2;
                t.bind(o_gu, lw.ewgu[e]);
                t.bind(o_dn, lw.ewdown[e]);
                const std::string q = p + "block_sparse_moe.experts." + std::to_string(w.rank * w.E_local + e) + ".";
                mat(q + "w1.weight", o_gu, I, H, H, gate, I, H, 0, 0);
                mat(q + "w2.weight", o_dn, H, I, I, ident, H, I, 0, 0);
                mat(q + "w3.weight", o_gu, I, H, H, up, I, H, 0, 0);
            }
        } else {
            const size_t o_gu = t.take(2 * I * H * 2, lw.wgu);   // row 2j = gate_j, row 2j + 1 = up_j
            mat(p + "mlp.gate_proj.weight", o_gu, I, H, H, gate, I * tp, H, rk * I, 0);
            mat(p + "mlp.up_proj.weight", o_gu, I, H, H, up, I * tp, H, rk * I, 0);
            mat(p + "mlp.down_proj.weight", t.take(H * I * 2, lw.wdown), H, I, I, ident, H, I * tp, 0, rk * I);
        }
        vec(p + "input_layernorm.weight", t.take(H * 4, lw.ln1), H, ident, H, 0, true);
        vec(p + "post_attention_layernorm.weight", t.take(H * 4, lw.ln2), H, ident, H, 0, true);
    }
    t.take((size_t)w.max_pos * (w.d / 2) * 4, w.rope_cos);
    t.take((size_t)w.max_pos * (w.d / 2) * 4, w.rope_sin);
    // bytes one decode step must stream: every parameter except the embedding table (SURVEY.md section 8d)
    const uint64_t mlp = moe ? (uint64_t)w.E_local * 3 * I * H : 3 * I * H;     // every local expert is streamed each step
    w.streamed_bytes = 2 * ((uint64_t)w.L * ((uint64_t)w.nqkv * H + H * nq + mlp) + V * H) +
                       4 * ((uint64_t)w.L * (2 * H + (c.qkv_bias ? w.nqkv : 0) + (moe ? (uint64_t)w.E * H : 0)) + H);
}

inline void bert_plan(BertModel& m) {
    const fl_config& c = m.cfg;
    m.H = c.hidden_size; m.I = c.intermediate_size; m.V = c.vocab_size; m.L = c.num_hidden_layers; m.nh = c.num_attention_heads;
    m.d = m.H / m.nh; m.maxpos = c.max_position_embeddings;
    FL_CHECK(m.d * m.nh == m.H, FL_ERR_INVALID, "hidden_size must be divisible by num_attention_heads");
    // head_dim: the attention kernels are built for 32 (all-MiniLM-L6-v2) and 64 (BERT-base / -large, e5, gte); the GEMMs take
    // K and N in 64-column blocks; the LayerNorm kernels hold a row in one warp and pool_l2_kernel a row in one CTA: hidden <= 1024
    FL_CHECK(m.d == 32 || m.d == 64, FL_ERR_UNSUPPORTED,
             "BERT path is built for head_dim 32 and 64 (hidden_size / num_attention_heads = " + std::to_string(m.d) + ")");
    FL_CHECK(m.H % 64 == 0 && m.I % 64 == 0, FL_ERR_UNSUPPORTED, "BERT path needs hidden_size and intermediate_size to be multiples of 64");
    FL_CHECK(m.H <= 1024, FL_ERR_UNSUPPORTED, "BERT path is built for hidden_size <= 1024");

    // The slab in allocation order: word and position embeddings, embedding LayerNorm, then per layer the four matrices, the
    // four biases and the two LayerNorms.  The reference loads BERT as f32 (embeddings.rs:298): uploads are f32 only, and
    // vectors are kept as uploaded.
    TensorTable& t = m.table;
    t.f32_only = true;
    const int64_t H = m.H, I = m.I;
    // bf16 matrix [rows, cols] landing at row row0 of its buffer
    auto mat = [&](const std::string& name, size_t off, int64_t rows, int64_t cols, int64_t row0 = 0) {
        t.add({name, true, off, rows, cols, cols, RowMap{row0, 0, 0, 0}, rows, cols, 0, 0, false, false, true});
    };
    // f32 vector [rows] landing at element row0 of its buffer; LayerNorm weights are initialised to ones
    auto vec = [&](const std::string& name, size_t off, int64_t rows, int64_t row0 = 0, bool ones = false) {
        t.add({name, false, off, rows, 1, 1, RowMap{row0, 0, 0, 0}, rows, 1, 0, 0, ones, false, true});
    };
    mat("embeddings.word_embeddings.weight", t.take(m.V * H * 2, m.wemb), m.V, H);
    mat("embeddings.position_embeddings.weight", t.take(m.maxpos * H * 2, m.pemb), m.maxpos, H);
    vec("embeddings.LayerNorm.weight", t.take(H * 4, m.lnw), H, 0, true);
    vec("embeddings.LayerNorm.bias", t.take(H * 4, m.lnb), H);
    m.layers.resize(m.L);
    for (int l = 0; l < m.L; ++l) {
        BertLayerW& w = m.layers[l];
        const std::string p = "encoder.layer." + std::to_string(l) + ".";
        const size_t o_qkv = t.take(3 * H * H * 2, w.wqkv);   // q | k | v rows
        mat(p + "attention.self.query.weight", o_qkv, H, H, 0);
        mat(p + "attention.self.key.weight", o_qkv, H, H, H);
        mat(p + "attention.self.value.weight", o_qkv, H, H, 2 * H);
        mat(p + "attention.output.dense.weight", t.take(H * H * 2, w.wo), H, H);
        mat(p + "intermediate.dense.weight", t.take(I * H * 2, w.wi), I, H);
        mat(p + "output.dense.weight", t.take(H * I * 2, w.wo2), H, I);
        const size_t o_bqkv = t.take(3 * H * 4, w.bqkv);
        vec(p + "attention.self.query.bias", o_bqkv, H, 0);
        vec(p + "attention.self.key.bias", o_bqkv, H, H);
        vec(p + "attention.self.value.bias", o_bqkv, H, 2 * H);
        vec(p + "attention.output.dense.bias", t.take(H * 4, w.bo), H);
        vec(p + "intermediate.dense.bias", t.take(I * 4, w.bi), I);
        vec(p + "output.dense.bias", t.take(H * 4, w.bo2), H);
        vec(p + "attention.output.LayerNorm.weight", t.take(H * 4, w.ln1w), H, 0, true);
        vec(p + "attention.output.LayerNorm.bias", t.take(H * 4, w.ln1b), H);
        vec(p + "output.LayerNorm.weight", t.take(H * 4, w.ln2w), H, 0, true);
        vec(p + "output.LayerNorm.bias", t.take(H * 4, w.ln2b), H);
    }
}

}  // namespace fl
