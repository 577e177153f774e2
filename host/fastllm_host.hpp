// C++ mirror of fastllm's trait-based model API over the C ABI (include/fastllm_b200.h).
//
// The reference's host side is Rust (compiled code) and there is no Rust toolchain in this image, so the compiled
// host-side mirror is C++: same type names, same argument meaning, same offset rules and the same failure points as
//   ModelInitializer / ModelArchitecture   src/models/model_initializer.rs:6-27
//   ModelCache / CommonCache               src/models/cache.rs:5-46
//   LlamaWithConfig / LlamaCache           src/models/llama.rs:52-160
//   MistralWithConfig / MistralCache       src/models/mistral.rs:16-248
//   QwenWithConfig / QwenCache             src/models/qwen.rs:12-186
//   Model<M>::generate + LogitsProcessor   src/models/mod.rs:342-464
//   EmbeddingModel / MiniLMModel           src/models/embeddings.rs:17-38, 245-447
// INTEGRATION.md shows the Rust shim (a transliteration of this file) a maintainer would add.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <map>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "../include/fastllm_b200.h"

namespace fastllm {

struct Error : std::runtime_error {   // anyhow::Error
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
inline void check(int rc) {
    if (rc != FL_OK) throw Error(rc, fl_last_error());
}

// A host tensor as handed over by load_model (providers/huggingface/huggingface.rs:85-130): name -> (dtype, shape, data)
struct HostTensor {
    fl_dtype dtype;
    std::vector<int64_t> shape;
    const void* data;
};
using TensorMap = std::map<std::string, HostTensor>;

// llama.rs:17-29 / mistral.rs:78-91 / models/config.rs:5-18
struct ConfigFile {
    int hidden_size = 0, intermediate_size = 0, vocab_size = 0, num_hidden_layers = 0, num_attention_heads = 0;
    std::optional<int> num_key_value_heads;
    double rms_norm_eps = 1e-5;
    std::optional<double> rope_theta;
    std::optional<int> max_position_embeddings;
    std::optional<int> sliding_window;
};

// ---- ModelCache (cache.rs:5-10) -------------------------------------------------------------------------------------
struct ModelCache {
    virtual ~ModelCache() = default;
    virtual void increment_offset() = 0;
    virtual void reset() = 0;
    virtual size_t get_offset() const = 0;
};
struct CommonCache : ModelCache {   // cache.rs:12-46
    size_t seqlen_offset = 0;
    void increment_offset() override { seqlen_offset += 1; }
    void reset() override { seqlen_offset = 0; }
    size_t get_offset() const override { return seqlen_offset; }
};

struct DeviceModel {   // shared device weights (fl_model*)
    fl_model* h = nullptr;
    fl_config cfg{};
    explicit DeviceModel(const fl_config& c) : cfg(c) { check(fl_model_create(&c, &h)); }
    DeviceModel(fl_model* handle, const fl_config& c) : h(handle), cfg(c) {}
    ~DeviceModel() { if (h) fl_model_destroy(h); }
    DeviceModel(const DeviceModel&) = delete;
    DeviceModel& operator=(const DeviceModel&) = delete;
};
struct DeviceCache {   // paged KV cache + stream (fl_cache*)
    fl_cache* h = nullptr;
    DeviceCache(fl_model* m, int max_batch, int max_seq) { check(fl_cache_create(m, max_batch, max_seq, &h)); }
    ~DeviceCache() { if (h) fl_cache_destroy(h); }
    DeviceCache(const DeviceCache&) = delete;
    DeviceCache& operator=(const DeviceCache&) = delete;
};

struct LlamaCache : CommonCache {     // llama.rs:61-92: owns the KV (candle `Cache`); bound lazily on first forward
    std::unique_ptr<DeviceCache> inner;
};
struct MistralCache : CommonCache {}; // mistral.rs:16-47: offset only, KV lives in the model
struct QwenCache : CommonCache {};    // qwen.rs:58-87

inline fl_config to_fl_config(fl_arch arch, const ConfigFile& cf, int default_max_pos, int sliding_window, bool qkv_bias) {
    fl_config c{};
    c.arch = arch;
    c.hidden_size = cf.hidden_size; c.intermediate_size = cf.intermediate_size; c.vocab_size = cf.vocab_size;
    c.num_hidden_layers = cf.num_hidden_layers; c.num_attention_heads = cf.num_attention_heads;
    c.num_key_value_heads = cf.num_key_value_heads.value_or(cf.num_attention_heads);
    c.max_position_embeddings = cf.max_position_embeddings.value_or(default_max_pos);
    c.sliding_window = sliding_window; c.qkv_bias = qkv_bias ? 1 : 0;
    c.norm_eps = (float)cf.rms_norm_eps; c.rope_theta = cf.rope_theta.value_or(10000.0);
    c.tp_rank = 0; c.tp_size = 1;
    return c;
}

inline std::shared_ptr<DeviceModel> upload(const fl_config& c, const TensorMap& tensors) {
    auto m = std::make_shared<DeviceModel>(c);
    for (const auto& kv : tensors)
        check(fl_model_put_tensor(m->h, kv.first.c_str(), kv.second.dtype, kv.second.shape.data(), (int)kv.second.shape.size(), kv.second.data));
    check(fl_model_finalize(m->h));
    return m;
}

// Logits of one forward: [b, V] (Llama) or [b, 1, V] (Mistral/Qwen2); the generate loop flattens row 0 either way.
struct Logits {
    std::vector<float> data;
    int batch = 0, vocab = 0;
    const float* row(int b) const { return data.data() + (size_t)b * vocab; }
};

constexpr int kKvCapacity = 4096;   // the reference grows KV by `cat`; pages are preallocated here

// ---- LlamaWithConfig (llama.rs:52-160) --------------------------------------------------------------------------------
struct LlamaWithConfig {
    using Config = ConfigFile;
    using Cache = LlamaCache;
    std::shared_ptr<DeviceModel> dev;
    static constexpr bool kPositionPerCall = false;   // the caller's position is the RoPE offset (llama.rs:147-149)
    static const char* get_family() { return "Llama"; }
    static bool supports_architecture(const std::string& a) { return a == "LlamaForCausalLM"; }
    // initialize_model(&Config, HashMap<String,Tensor>, DType, &Device) -> (Self, Cache)   llama.rs:98-123
    static std::pair<LlamaWithConfig, Cache> initialize_model(const Config& cfg, const TensorMap& tensors, int device) {
        check(fl_init(device));
        LlamaWithConfig m{upload(to_fl_config(FL_ARCH_LLAMA, cfg, 4096, 0, false), tensors)};
        return {std::move(m), Cache{}};
    }
    static Cache initialize_cache(int /*device*/) { return Cache{}; }   // llama.rs:125-145
    // forward(&self, &Tensor, pos, &mut Cache): model.forward(input, pos, &mut cache.inner)   llama.rs:147-149
    Logits forward(const uint32_t* ids, int b, int t, size_t pos, Cache& cache) const {
        if (!cache.inner) cache.inner = std::make_unique<DeviceCache>(dev->h, b, std::min(kKvCapacity, dev->cfg.max_position_embeddings));
        Logits out; out.batch = b; out.vocab = dev->cfg.vocab_size; out.data.resize((size_t)b * out.vocab);
        check(fl_forward(dev->h, cache.inner->h, ids, b, t, pos, out.data.data()));
        return out;
    }
};

// ---- MistralWithConfig / QwenWithConfig (mistral.rs:49-248, qwen.rs:12-186) -------------------------------------------
template <fl_arch ARCH, typename CacheT>
struct OffsetAdapter {
    using Config = ConfigFile;
    using Cache = CacheT;
    std::shared_ptr<DeviceModel> dev;
    mutable std::unique_ptr<DeviceCache> kv;   // candle keeps the KV inside the model (RefCell<Model>)
    static constexpr bool kPositionPerCall = true;    // RoPE offset + 1 per CALL (mistral.rs:234, qwen.rs:143)
    static std::pair<OffsetAdapter, Cache> initialize_model(const Config& cfg, const TensorMap& tensors, int device) {
        check(fl_init(device));
        // mistral.rs:139 / qwen.rs:49: sliding_window.unwrap_or(4096); bad head dims make fl_model_create fail where the reference asserts
        OffsetAdapter m{upload(to_fl_config(ARCH, cfg, 32768, cfg.sliding_window.value_or(4096), ARCH == FL_ARCH_QWEN2), tensors), nullptr};
        return {std::move(m), Cache{}};
    }
    static Cache initialize_cache(int /*device*/) { return Cache{}; }
    void clear_kv_cache() const { if (kv) check(fl_cache_reset(kv->h)); }
    // forward(&self, input, _pos, cache): clear KV at offset 0; rope offset = cache offset; offset += 1 PER CALL
    Logits forward(const uint32_t* ids, int b, int t, size_t /*_pos*/, Cache& cache) const {
        if (!kv) kv = std::make_unique<DeviceCache>(dev->h, b, std::min(kKvCapacity, dev->cfg.max_position_embeddings));
        if (cache.get_offset() == 0) clear_kv_cache();
        Logits out; out.batch = b; out.vocab = dev->cfg.vocab_size; out.data.resize((size_t)b * out.vocab);
        check(fl_forward(dev->h, kv->h, ids, b, t, cache.get_offset(), out.data.data()));
        cache.increment_offset();
        return out;
    }
    OffsetAdapter clone() const { return OffsetAdapter{dev, nullptr}; }   // shared weights, independent KV (mod.rs:155)
};
using MistralWithConfig = OffsetAdapter<FL_ARCH_MISTRAL, MistralCache>;
using QwenWithConfig = OffsetAdapter<FL_ARCH_QWEN2, QwenCache>;

// candle's LogitsProcessor as the generate loops build it (mod.rs:157-158, 373-374): LogitsProcessor::new(seed, Some(temperature),
// None).  The arithmetic (arg-max in IEEE total order with the LAST maximum winning; soft-max + WeightedIndex over
// StdRng::seed_from_u64) is the library's fl_sampler_*: host code, as in the reference.
struct LogitsProcessor {
    fl_sampler* h = nullptr;
    LogitsProcessor(uint64_t seed, std::optional<double> temperature) { check(fl_sampler_create(seed, temperature.value_or(-1.0), &h)); }
    ~LogitsProcessor() { if (h) fl_sampler_destroy(h); }
    LogitsProcessor(const LogitsProcessor&) = delete;
    LogitsProcessor& operator=(const LogitsProcessor&) = delete;
    uint32_t sample(const float* logits, size_t n) {
        uint32_t tok = 0;
        check(fl_sampler_sample(h, logits, n, &tok));
        return tok;
    }
};

// ---- Model<M>::generate (mod.rs:363-463), prompts already tokenised ----------------------------------------------------
template <typename M>
struct Model {
    M model;
    typename M::Cache cache;
    std::optional<uint32_t> eos_token_id = 2;   // tokenizer.token_to_id("</s>")
    std::vector<uint32_t> generate(const std::vector<uint32_t>& prompt, int max_tokens, float temperature = 0.0f) {
        cache = M::initialize_cache(0);                                           // mod.rs:370
        LogitsProcessor logits_processor(0, (double)temperature);                 // mod.rs:373-374
        size_t pos = 0;
        Logits logits = model.forward(prompt.data(), 1, (int)prompt.size(), pos, cache);   // mod.rs:402-405
        pos += prompt.size();
        std::vector<uint32_t> out;
        for (int i = 0; i < max_tokens; ++i) {                                    // mod.rs:411-453
            const uint32_t tok = logits_processor.sample(logits.row(0), (size_t)logits.vocab);   // logits.get(0)?.flatten_all()?
            if (eos_token_id && tok == *eos_token_id) break;                      // break BEFORE emitting
            out.push_back(tok);
            logits = model.forward(&tok, 1, 1, pos, cache);
            pos += 1;
        }
        return out;
    }
};

// ---- continuous batching above fl_forward_slots (SURVEY.md section 8f-3; the reference serialises requests at batch 1 under one
// mutex, api/chat.rs:206-208).  Transliteration of fastllm_b200/models.py ContinuousBatcher: a request is admitted into a free
// sequence slot (its prompt prefilled alone), every step advances all running requests by one token in ONE ragged forward, a
// finished request frees its slot.  Per request: its own LogitsProcessor seeded 0, EOS break before emitting, the adapter's
// position rule.
template <typename M>
struct ContinuousBatcher {
    const M& model;
    int max_batch;
    std::optional<uint32_t> eos_token_id = 2;
    DeviceCache cache;
    int steps = 0;      // ragged decode forwards issued
    ContinuousBatcher(const M& m, int max_batch_, std::optional<uint32_t> eos = 2)
        : model(m), max_batch(max_batch_), eos_token_id(eos),
          cache(m.dev->h, max_batch_, std::min(kKvCapacity, m.dev->cfg.max_position_embeddings)) {}

    std::vector<std::vector<uint32_t>> generate(const std::vector<std::vector<uint32_t>>& prompts, int max_tokens, float temperature = 0.0f) {
        struct Running { size_t req; size_t rope; std::unique_ptr<LogitsProcessor> lp; uint32_t tok; };
        std::vector<std::vector<uint32_t>> out(prompts.size());
        if (max_tokens <= 0) return out;
        std::vector<size_t> waiting;
        for (size_t i = prompts.size(); i-- > 0;) waiting.push_back(i);
        std::vector<int> free_slots;
        for (int s = max_batch; s-- > 0;) free_slots.push_back(s);
        std::map<int, Running> running;
        const int V = model.dev->cfg.vocab_size;
        std::vector<float> logits((size_t)max_batch * V);
        auto take = [&](const float* row, int slot, Running&& st) {      // sample -> EOS / budget -> keep the slot or free it
            const uint32_t tok = st.lp->sample(row, (size_t)V);
            bool done;
            if (eos_token_id && tok == *eos_token_id) {
                done = true;
            } else {
                out[st.req].push_back(tok);
                st.tok = tok;
                done = (int)out[st.req].size() >= max_tokens;
            }
            if (done) {
                running.erase(slot);
                check(fl_cache_slot_reset(cache.h, slot));
                free_slots.push_back(slot);
            } else {
                running[slot] = std::move(st);
            }
        };
        while (!waiting.empty() || !running.empty()) {
            while (!waiting.empty() && !free_slots.empty()) {             // admit: one prompt at a time, alone in its forward
                const size_t req = waiting.back(); waiting.pop_back();
                const int slot = free_slots.back(); free_slots.pop_back();
                const std::vector<uint32_t>& p = prompts[req];
                const size_t ro = 0;
                check(fl_forward_slots(model.dev->h, cache.h, &slot, p.data(), 1, (int)p.size(), &ro, logits.data()));
                Running st{req, M::kPositionPerCall ? (size_t)1 : p.size(), std::make_unique<LogitsProcessor>(0, (double)temperature), 0};
                take(logits.data(), slot, std::move(st));
            }
            if (running.empty()) continue;
            std::vector<int> slots;
            std::vector<uint32_t> ids;
            std::vector<size_t> ropes;
            for (auto& kv : running) { slots.push_back(kv.first); ids.push_back(kv.second.tok); ropes.push_back(kv.second.rope); }   // ascending slots
            check(fl_forward_slots(model.dev->h, cache.h, slots.data(), ids.data(), (int)slots.size(), 1, ropes.data(), logits.data()));
            steps += 1;
            for (size_t i = 0; i < slots.size(); ++i) {
                Running st = std::move(running[slots[i]]);
                st.rope += 1;
                take(logits.data() + i * (size_t)V, slots[i], std::move(st));
            }
        }
        return out;
    }
};

// ---- EmbeddingModel (models/embeddings.rs:17-38) / MiniLMModel (:245-447) after tokenisation -------------------------------------
struct BertConfig {   // models/embeddings.rs:46-54 (+ the vocabulary size the reference takes from the tokenizer, :301-306)
    int hidden_size = 384, num_attention_heads = 12, num_hidden_layers = 6, intermediate_size = 1536, max_position_embeddings = 512;
    double layer_norm_eps = 1e-12;
    int vocab_size = 30522;
};
struct MiniLMModel {
    std::shared_ptr<DeviceModel> dev;
    std::string id = "sentence-transformers/all-MiniLM-L6-v2";
    static const char* get_family() { return "bert"; }
    static bool supports_architecture(const std::string& a) { return a == "BertModel" || a == "RobertaModel" || a == "DebertaModel"; }
    static MiniLMModel create(const BertConfig& cfg, const TensorMap& tensors, int device) {   // MiniLMModel::new (:257-339)
        check(fl_init(device));
        fl_config c{};
        c.arch = FL_ARCH_BERT;
        c.hidden_size = cfg.hidden_size; c.intermediate_size = cfg.intermediate_size; c.vocab_size = cfg.vocab_size;
        c.num_hidden_layers = cfg.num_hidden_layers; c.num_attention_heads = cfg.num_attention_heads; c.num_key_value_heads = cfg.num_attention_heads;
        c.max_position_embeddings = cfg.max_position_embeddings; c.norm_eps = (float)cfg.layer_norm_eps; c.tp_size = 1;
        return MiniLMModel{upload(c, tensors)};
    }
    const std::string& model_id() const { return id; }
    size_t embedding_size() const { return (size_t)dev->cfg.hidden_size; }   // the reference hard-codes 384 (:453-455)
    // EmbeddingModel::embed after tokenisation: ids (and the tokenizer's attention mask, or nullptr = all ones) [b, t] -> f32 [b, hidden]
    std::vector<float> embed_ids(const uint32_t* ids, const uint32_t* mask, int b, int t) const {
        std::vector<float> out((size_t)b * dev->cfg.hidden_size);
        check(fl_embed(dev->h, ids, mask, b, t, out.data()));
        return out;
    }
    // default impl of EmbeddingModel::compute_similarity (:22-37): cosine of the two embeddings
    float compute_similarity(const std::vector<uint32_t>& a, const std::vector<uint32_t>& b) const {
        const std::vector<float> va = embed_ids(a.data(), nullptr, 1, (int)a.size()), vb = embed_ids(b.data(), nullptr, 1, (int)b.size());
        double dot = 0, na = 0, nb = 0;
        for (size_t i = 0; i < va.size(); ++i) { dot += (double)va[i] * vb[i]; na += (double)va[i] * va[i]; nb += (double)vb[i] * vb[i]; }
        return (float)(dot / (std::sqrt(na) * std::sqrt(nb)));
    }
    // `input: [String]` batching (SURVEY.md section 8f-3), exact: only sentences of EQUAL token length share a [b, t] call (the
    // reference's attention has no mask, so padding would change results); rows come back in request order
    std::vector<std::vector<float>> embed_many(const std::vector<std::vector<uint32_t>>& sentences, int max_batch = 256) const {
        std::vector<std::vector<float>> out(sentences.size());
        std::map<size_t, std::vector<size_t>> groups;
        for (size_t i = 0; i < sentences.size(); ++i) groups[sentences[i].size()].push_back(i);
        const size_t H = embedding_size();
        for (const auto& kv : groups)
            for (size_t k = 0; k < kv.second.size(); k += (size_t)max_batch) {
                const size_t n = std::min(kv.second.size() - k, (size_t)max_batch);
                std::vector<uint32_t> ids;
                for (size_t j = 0; j < n; ++j) ids.insert(ids.end(), sentences[kv.second[k + j]].begin(), sentences[kv.second[k + j]].end());
                const std::vector<float> e = embed_ids(ids.data(), nullptr, (int)n, (int)kv.first);
                for (size_t j = 0; j < n; ++j) out[kv.second[k + j]].assign(e.begin() + j * H, e.begin() + (j + 1) * H);
            }
        return out;
    }
    // `input: [String]` in ONE encoder pass (fl_embed_packed): the sentences are concatenated without padding; row i equals
    // embed_ids of sentence i alone bit for bit; rows come back in request order
    std::vector<std::vector<float>> embed_packed(const std::vector<std::vector<uint32_t>>& sentences) const {
        if (sentences.empty()) return {};
        std::vector<uint32_t> ids;
        std::vector<int32_t> lengths;
        for (const auto& s : sentences) {
            ids.insert(ids.end(), s.begin(), s.end());
            lengths.push_back((int32_t)s.size());
        }
        const size_t H = embedding_size();
        std::vector<float> e(sentences.size() * H);
        check(fl_embed_packed(dev->h, ids.data(), lengths.data(), (int)sentences.size(), e.data()));
        std::vector<std::vector<float>> out(sentences.size());
        for (size_t i = 0; i < out.size(); ++i) out[i].assign(e.begin() + i * H, e.begin() + (i + 1) * H);
        return out;
    }
};

}  // namespace fastllm
