// Self-test of the C++ host mirror: builds a tiny synthetic Llama through the reference-shaped interface, runs
// Model::generate, prints the greedy ids as JSON.  tests/test_host_cpp_gpu.py compares them with the oracle.
// `host_selftest --sampler seed temperature vocab logits.bin` needs no GPU: it runs the mirror's LogitsProcessor over the f32 rows
// of logits.bin and prints the sampled ids (tests/test_sampling_cpu.py compares them with the oracle).
// `host_selftest manifest weights 0 --loglikelihood context... / continuation...` prints Model::loglikelihood as [sum, is_greedy].
// `host_selftest manifest weights max_tokens --batch|--packed max_batch ids / ids / ...` prints the ContinuousBatcher's / PackedBatcher's ids.
// `host_selftest manifest weights max_tokens --packed-pool max_batch pool_tokens prefix_len ids / ...`: the Mistral PackedBatcher on a KV
// pool with a shared prefix.
// Build: g++ -std=c++17 -O2 host/host_selftest.cpp -o host/_build/host_selftest -Lfastllm_b200 -lfastllm_b200 -Wl,-rpath,...
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "fastllm_host.hpp"

int main(int argc, char** argv) {
    if (argc == 6 && std::strcmp(argv[1], "--sampler") == 0) {
        try {
            const uint64_t seed = std::strtoull(argv[2], nullptr, 10);
            const double temperature = std::atof(argv[3]);
            const size_t vocab = (size_t)std::strtoull(argv[4], nullptr, 10);
            FILE* lf = std::fopen(argv[5], "rb");
            if (!lf || vocab == 0) throw std::runtime_error("cannot open logits");
            fastllm::LogitsProcessor lp(seed, temperature < 0 ? std::nullopt : std::optional<double>(temperature));
            std::vector<float> row(vocab);
            std::printf("[");
            for (int i = 0; std::fread(row.data(), 4, vocab, lf) == vocab; ++i) std::printf("%s%u", i ? "," : "", lp.sample(row.data(), vocab));
            std::printf("]\n");
            std::fclose(lf);
            return 0;
        } catch (const std::exception& e) {
            std::fprintf(stderr, "host_selftest --sampler failed: %s\n", e.what());
            return 1;
        }
    }
    // argv: weights.bin (concatenated f32 tensors in manifest order), manifest.txt (name ndim dims...), prompt ids...
    if (argc < 4) { std::fprintf(stderr, "usage: host_selftest manifest.txt weights.bin max_tokens id...\n"); return 2; }
    try {
        FILE* mf = std::fopen(argv[1], "r");
        FILE* wf = std::fopen(argv[2], "rb");
        if (!mf || !wf) throw std::runtime_error("cannot open inputs");
        fastllm::ConfigFile cfg;
        int nkv = 0, maxpos = 0;
        double theta = 0;
        if (std::fscanf(mf, "%d %d %d %d %d %d %lf %lf %d", &cfg.hidden_size, &cfg.intermediate_size, &cfg.vocab_size, &cfg.num_hidden_layers,
                        &cfg.num_attention_heads, &nkv, &cfg.rms_norm_eps, &theta, &maxpos) != 9) throw std::runtime_error("bad manifest header");
        cfg.num_key_value_heads = nkv; cfg.rope_theta = theta; cfg.max_position_embeddings = maxpos;
        std::vector<std::vector<float>> storage;
        fastllm::TensorMap tensors;
        char name[256];
        int nd;
        while (std::fscanf(mf, "%255s %d", name, &nd) == 2) {
            std::vector<int64_t> shape(nd);
            size_t n = 1;
            for (int i = 0; i < nd; ++i) { long long d; if (std::fscanf(mf, "%lld", &d) != 1) throw std::runtime_error("bad shape"); shape[i] = d; n *= (size_t)d; }
            storage.emplace_back(n);
            if (std::fread(storage.back().data(), 4, n, wf) != n) throw std::runtime_error("short weights file");
            tensors[name] = fastllm::HostTensor{FL_DTYPE_F32, shape, storage.back().data()};
        }
        const int max_tokens = std::atoi(argv[3]);
        if (argc > 4 && std::strcmp(argv[4], "--loglikelihood") == 0) {
            // host_selftest manifest weights 0 --loglikelihood context ids / continuation ids: Model::loglikelihood
            std::vector<uint32_t> parts[2];
            int k = 0;
            for (int i = 5; i < argc; ++i) {
                if (std::strcmp(argv[i], "/") == 0) k = 1;
                else parts[k].push_back((uint32_t)std::strtoul(argv[i], nullptr, 10));
            }
            auto pr = fastllm::LlamaWithConfig::initialize_model(cfg, tensors, 0);
            fastllm::Model<fastllm::LlamaWithConfig> model{std::move(pr.first), std::move(pr.second), std::nullopt};
            const auto ll = model.loglikelihood(parts[0], parts[1]);
            std::printf("[%.17g, %s]\n", ll.first, ll.second ? "true" : "false");
            return 0;
        }
        if (argc > 7 && std::strcmp(argv[4], "--packed-pool") == 0) {
            // host_selftest manifest weights max_tokens --packed-pool max_batch pool_tokens prefix_len id id / id ... : the C++ PackedBatcher
            // of the Mistral adapter on a KV pool of pool_tokens, with the first prefix_len ids of the first prompt as the shared prefix
            const int max_batch = std::atoi(argv[5]), pool_tokens = std::atoi(argv[6]), prefix_len = std::atoi(argv[7]);
            std::vector<std::vector<uint32_t>> prompts(1);
            for (int i = 8; i < argc; ++i) {
                if (std::strcmp(argv[i], "/") == 0) prompts.emplace_back();
                else prompts.back().push_back((uint32_t)std::strtoul(argv[i], nullptr, 10));
            }
            const std::vector<uint32_t> prefix(prompts[0].begin(), prompts[0].begin() + prefix_len);
            auto pr = fastllm::MistralWithConfig::initialize_model(cfg, tensors, 0);
            fastllm::PackedBatcher<fastllm::MistralWithConfig> pb(pr.first, max_batch, std::nullopt, 4096, pool_tokens);
            const auto outs = pb.generate(prompts, max_tokens, 0.0f, &prefix);
            std::fprintf(stderr, "packed forwards: %d\n", pb.forwards);
            std::printf("[");
            for (size_t r = 0; r < outs.size(); ++r) {
                std::printf("%s[", r ? "," : "");
                for (size_t i = 0; i < outs[r].size(); ++i) std::printf("%s%u", i ? "," : "", outs[r][i]);
                std::printf("]");
            }
            std::printf("]\n");
            return 0;
        }
        if (argc > 5 && (std::strcmp(argv[4], "--batch") == 0 || std::strcmp(argv[4], "--packed") == 0)) {
            // host_selftest manifest weights max_tokens --batch max_batch id id / id id id / ...: the C++ ContinuousBatcher over sequence slots
            // (--packed: the C++ PackedBatcher, prompts admitted into the decode steps' packed forwards)
            const bool packed = std::strcmp(argv[4], "--packed") == 0;
            const int max_batch = std::atoi(argv[5]);
            std::vector<std::vector<uint32_t>> prompts(1);
            for (int i = 6; i < argc; ++i) {
                if (std::strcmp(argv[i], "/") == 0) prompts.emplace_back();
                else prompts.back().push_back((uint32_t)std::strtoul(argv[i], nullptr, 10));
            }
            auto pr = fastllm::LlamaWithConfig::initialize_model(cfg, tensors, 0);
            std::vector<std::vector<uint32_t>> outs;
            if (packed) {
                fastllm::PackedBatcher<fastllm::LlamaWithConfig> pb(pr.first, max_batch, std::nullopt);
                outs = pb.generate(prompts, max_tokens);
                std::fprintf(stderr, "packed forwards: %d\n", pb.forwards);
            } else {
                fastllm::ContinuousBatcher<fastllm::LlamaWithConfig> cb(pr.first, max_batch, std::nullopt);
                outs = cb.generate(prompts, max_tokens);
                std::fprintf(stderr, "ragged steps: %d\n", cb.steps);
            }
            std::printf("[");
            for (size_t r = 0; r < outs.size(); ++r) {
                std::printf("%s[", r ? "," : "");
                for (size_t i = 0; i < outs[r].size(); ++i) std::printf("%s%u", i ? "," : "", outs[r][i]);
                std::printf("]");
            }
            std::printf("]\n");
            return 0;
        }
        std::vector<uint32_t> prompt;
        for (int i = 4; i < argc; ++i) prompt.push_back((uint32_t)std::strtoul(argv[i], nullptr, 10));
        auto pair = fastllm::LlamaWithConfig::initialize_model(cfg, tensors, 0);
        fastllm::Model<fastllm::LlamaWithConfig> model{std::move(pair.first), std::move(pair.second), std::nullopt};
        const auto ids = model.generate(prompt, max_tokens);
        std::printf("[");
        for (size_t i = 0; i < ids.size(); ++i) std::printf("%s%u", i ? "," : "", ids[i]);
        std::printf("]\n");
        // failure point parity: multi-token forward on a non-empty Llama cache must be an error, not a crash
        try {
            model.model.forward(prompt.data(), 1, (int)prompt.size(), prompt.size(), model.cache);
            std::printf("ERROR: expected failure\n");
            return 1;
        } catch (const fastllm::Error& e) { std::fprintf(stderr, "expected error: %s\n", e.what()); }
        return 0;
    } catch (const std::exception& e) {
        std::fprintf(stderr, "host_selftest failed: %s\n", e.what());
        return 1;
    }
}
