// Runs a model's plan step (no CUDA call, no GPU needed) and prints its tensor table as JSON for test_tensor_table_cpu.py.
// usage: tensor_table_dump arch hidden intermediate vocab layers heads kv_heads max_pos qkv_bias experts tp_size tp_rank
#include <cstdio>
#include <cstdlib>

#include "../fastllm_b200/csrc/model.cuh"
#include "../fastllm_b200/csrc/weights_plan.cuh"

static void dump(const fl::TensorTable& t, unsigned long long streamed_bytes) {
    std::printf("{\"size\": %zu, \"streamed_bytes\": %llu, \"slots\": [", t.size, streamed_bytes);
    for (size_t i = 0; i < t.slots.size(); ++i) {
        const fl::TensorSlot& s = t.slots[i];
        std::printf("%s\n{\"name\": \"%s\", \"mat\": %d, \"off\": %zu, \"rows\": %lld, \"cols\": %lld, \"ld\": %lld, "
                    "\"map\": [%lld, %d, %d, %d], \"full\": [%lld, %lld], \"win\": [%lld, %lld], \"ones\": %d, \"round\": %d, "
                    "\"required\": %d}",
                    i ? "," : "", s.name.c_str(), (int)s.mat, s.off, (long long)s.rows, (long long)s.cols, (long long)s.ld,
                    (long long)s.map.dst_row0, s.map.mode, s.map.head_dim, s.map.lane, (long long)s.full_rows, (long long)s.full_cols,
                    (long long)s.row0, (long long)s.col0, (int)s.ones, (int)s.round, (int)s.required);
    }
    std::printf("]}\n");
}

int main(int argc, char** argv) {
    fl_config c{};
    int32_t* fields[] = {&c.arch, &c.hidden_size, &c.intermediate_size, &c.vocab_size, &c.num_hidden_layers, &c.num_attention_heads,
                         &c.num_key_value_heads, &c.max_position_embeddings, &c.qkv_bias, &c.num_local_experts, &c.tp_size, &c.tp_rank};
    const int n = sizeof(fields) / sizeof(fields[0]);
    if (argc != n + 1) {
        std::fprintf(stderr, "usage: %s arch hidden intermediate vocab layers heads kv_heads max_pos qkv_bias experts tp_size tp_rank\n",
                     argv[0]);
        return 2;
    }
    for (int i = 0; i < n; ++i) *fields[i] = std::atoi(argv[i + 1]);
    c.num_experts_per_tok = 2;
    try {
        if (c.arch == FL_ARCH_BERT) {
            fl::BertModel m;
            m.cfg = c;
            fl::bert_plan(m);
            dump(m.table, 0);
        } else {
            fl::Weights w;
            w.cfg = c;
            fl::plan_weights(w);
            dump(w.table, w.streamed_bytes);
        }
    } catch (const fl::Error& e) {
        std::fprintf(stderr, "error %d: %s\n", e.code, e.what());
        return 1;
    }
    return 0;
}
