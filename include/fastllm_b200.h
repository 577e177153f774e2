/* fastllm_b200 — C ABI of the B200-native transformer forward pass that slots in under fastllm's
 * trait-based model API (the L2->L0 boundary of SURVEY.md section 1 / section 8b).
 *
 * Every entry point is `extern "C"`, takes plain pointers/sizes, returns 0 on success and a negative
 * fl_status on failure; the message for the calling thread's last failure is fl_last_error().  Nothing
 * throws or aborts across this boundary.  The library owns all device memory (weights, paged KV cache,
 * workspaces), its own CUDA stream per cache, and the NCCL communicator.  There is no CPU fallback.
 *
 * Reference interface each group replaces (paths under /root/reference/src):
 *   fl_model_create / fl_model_put_tensor / fl_model_finalize
 *        <- ModelInitializer::initialize_model(&Config, HashMap<String,Tensor>, DType, &Device)
 *           models/model_initializer.rs:10-17; called from providers/huggingface/huggingface.rs:135;
 *           bodies models/llama.rs:98-123, models/mistral.rs:160-200, models/qwen.rs:93-117,
 *           and MiniLMModel::new models/embeddings.rs:257-339 (BERT family)
 *   fl_model_clone            <- `M: Clone` required by the streaming path, models/mod.rs:155,181,207
 *   fl_cache_create / reset   <- ModelInitializer::initialize_cache models/model_initializer.rs:19
 *                                (llama.rs:125-145, mistral.rs:202-204, qwen.rs:119-121) and
 *                                ModelCache::reset models/cache.rs:5-10; Mistral/Qwen2 `clear_kv_cache`
 *                                at offset 0 (mistral.rs:218-221, qwen.rs:138-140)
 *   fl_forward                <- ModelInitializer::forward(&self, &Tensor (u32 [b,t]), usize pos, &mut Cache)
 *                                models/model_initializer.rs:21 (llama.rs:147-149, mistral.rs:206-236,
 *                                qwen.rs:123-145); returns the last-position logits as f32 [b, V]
 *   fl_forward_greedy         <- forward + LogitsProcessor arg-max of models/mod.rs:421-428 fused on device
 *                                (ties resolve to the LAST index, as candle's max_by(total_cmp) does)
 *   fl_sampler_* / fl_forward_sample
 *                             <- candle's LogitsProcessor as the generate loops build and call it:
 *                                LogitsProcessor::new(Default::default(), Some(temperature as f64), None)
 *                                models/mod.rs:157-158,373-374 and logits_processor.sample(&last_logits)
 *                                models/mod.rs:308-310,425-428 (arg-max below 1e-7, else soft-max + WeightedIndex
 *                                over rand 0.8's StdRng seeded with seed_from_u64)
 *   fl_forward_slots          <- the same forward for a batch of requests of different lengths (no reference counterpart: requests
 *                                are serialised at batch 1, api/chat.rs:206-208; streams run side by side, models/mod.rs:151-175)
 *   fl_embed                  <- EmbeddingModel::embed models/embeddings.rs:397-447 after tokenisation:
 *                                encoder forward + mean_pooling (:346-368) + normalize_l2 (:341-344)
 *   fl_embed_packed           <- the same embed for a batch of sentences of different lengths in ONE encoder pass (no reference
 *                                counterpart: api/embeddings.rs takes one string per request); row i is what embed returns for
 *                                sentence i alone
 */
#ifndef FASTLLM_B200_H
#define FASTLLM_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define FL_EXPORT __attribute__((visibility("default")))
#else
#define FL_EXPORT
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fl_model fl_model;
typedef struct fl_cache fl_cache;
typedef struct fl_sampler fl_sampler;

typedef enum fl_status {
    FL_OK = 0,
    FL_ERR_INVALID = -1,   /* bad argument / bad config (the reference panics: mistral.rs:109-127, models/config.rs:20-54) */
    FL_ERR_CUDA = -2,      /* CUDA runtime/driver error; the handle is poisoned */
    FL_ERR_STATE = -3,     /* call out of order (e.g. forward before finalize, cache full) */
    FL_ERR_NCCL = -4,
    FL_ERR_UNSUPPORTED = -5
} fl_status;

typedef enum fl_arch {
    FL_ARCH_LLAMA = 0,     /* LlamaForCausalLM          (models/llama.rs)   */
    FL_ARCH_MISTRAL = 1,   /* MistralForCausalLM        (models/mistral.rs) */
    FL_ARCH_QWEN2 = 2,     /* Qwen2ForCausalLM, qkv bias (models/qwen.rs)    */
    FL_ARCH_MIXTRAL = 3,   /* MixtralForCausalLM top-k MoE (no reference path; candle mixtral.rs) */
    FL_ARCH_BERT = 4       /* BertModel encoder         (models/embeddings.rs) */
} fl_arch;

typedef enum fl_dtype { FL_DTYPE_F32 = 0, FL_DTYPE_BF16 = 1, FL_DTYPE_F16 = 2 } fl_dtype;

/* Mirrors the fields the reference adapters read from config.json
 * (llama.rs:17-29, mistral.rs:78-91, models/config.rs:5-18, models/embeddings.rs:46-54). */
typedef struct fl_config {
    int32_t arch;                      /* fl_arch */
    int32_t hidden_size;
    int32_t intermediate_size;
    int32_t vocab_size;
    int32_t num_hidden_layers;
    int32_t num_attention_heads;
    int32_t num_key_value_heads;       /* 0 => num_attention_heads */
    int32_t max_position_embeddings;   /* RoPE table length (causal LMs) / position table rows (BERT) */
    int32_t sliding_window;            /* Mistral/Qwen2 prefill mask: key j banned when j + sw < i; <=0 => none */
    int32_t qkv_bias;                  /* Qwen2 */
    int32_t num_local_experts;         /* Mixtral */
    int32_t num_experts_per_tok;       /* Mixtral */
    float norm_eps;                    /* rms_norm_eps, or layer_norm_eps for BERT layers (embeddings LN is 1e-12) */
    double rope_theta;
    int32_t tp_rank;                   /* tensor-parallel rank / size of THIS process (1 process per GPU) */
    int32_t tp_size;                   /* 0 or 1 => no tensor parallelism (Mixtral: the same two fields are the expert-parallel rank / size) */
    int32_t ep_dp_attention;           /* Mixtral, tp_size > 1: 1 => sequences are data-parallel (every rank is called with ITS slice of the batch,
                                          same [b, t] shape on every rank) and tokens travel to the experts and back by all-to-all;
                                          0 => every rank is called with the whole batch (attention replicated, expert outputs all-reduced) */
    int32_t reserved[5];
} fl_config;

/* ---- process / device -------------------------------------------------------------------------- */
FL_EXPORT int fl_init(int device);                               /* cudaSetDevice + one-time setup; idempotent */
FL_EXPORT const char* fl_last_error(void);                       /* thread-local, never NULL */
FL_EXPORT int fl_version(void);
FL_EXPORT int fl_device_synchronize(void);

/* ---- model (weights) --------------------------------------------------------------------------- */
FL_EXPORT int fl_model_create(const fl_config* cfg, fl_model** out);
/* Upload one tensor by its HuggingFace name (same names VarBuilder asks for).  f32/f16 inputs are rounded to
 * bf16 (round-to-nearest-even), as VarBuilder::from_tensors(.., DType::BF16, ..) does (main.rs:120).  The host
 * buffer may be freed on return.  q/k/v and gate/up are fused and row-permuted on upload (DESIGN.md). */
FL_EXPORT int fl_model_put_tensor(fl_model* m, const char* name, int dtype, const int64_t* shape, int rank, const void* host_ptr);
/* Deterministic synthetic weights generated on the device (rule: oracle/synth.py; N(0,std^2)-like -> bf16,
 * norm weights 1.0).  Used by the benchmark instead of shipping 14-93 GB of tensors. */
FL_EXPORT int fl_model_random_init(fl_model* m, uint64_t seed, float std);
FL_EXPORT int fl_model_finalize(fl_model* m);                    /* checks every tensor arrived; builds RoPE tables */
FL_EXPORT int fl_model_clone(fl_model* m, fl_model** out);       /* shares weights (ref-counted), independent otherwise */
FL_EXPORT int fl_model_destroy(fl_model* m);
FL_EXPORT int fl_model_weight_bytes(fl_model* m, uint64_t* streamed_bytes); /* bytes one decode step must stream (no embedding table) */

/* ---- KV cache ---------------------------------------------------------------------------------- */
FL_EXPORT int fl_cache_create(fl_model* m, int max_batch, int max_seq, fl_cache** out);
FL_EXPORT int fl_cache_reset(fl_cache* c);                       /* kv length := 0 for every sequence */
FL_EXPORT int fl_cache_kv_len(fl_cache* c, int* out);            /* tokens currently held (same for every sequence) */
FL_EXPORT int fl_cache_fill_synthetic(fl_cache* c, int batch, int kv_len, uint64_t seed); /* benchmark: pretend a kv_len-token prefill */
FL_EXPORT int fl_cache_destroy(fl_cache* c);

/* ---- forward (causal LMs) ---------------------------------------------------------------------- */
/* ids: host u32 [b, t] row-major.  rope_offset: RoPE position of ids[:,0] (explicit so the Mistral/Qwen2 adapter's
 * +1-per-call rule survives unchanged; the KV length is tracked inside the cache).  logits_host: f32 [b, vocab]. */
FL_EXPORT int fl_forward(fl_model* m, fl_cache* c, const uint32_t* ids, int b, int t, size_t rope_offset, float* logits_host);
/* Same forward, arg-max on device (last index wins ties); next_ids: host u32 [b]. */
FL_EXPORT int fl_forward_greedy(fl_model* m, fl_cache* c, const uint32_t* ids, int b, int t, size_t rope_offset, uint32_t* next_ids);
/* Device-resident greedy decode: `steps` single-token steps where step i feeds the arg-max of step i-1 (first step feeds
 * first_ids), RoPE position rope_offset+i.  One CUDA-graph launch per step, no host sync inside.  out_ids: host u32
 * [steps, b] or NULL.  elapsed_ms: CUDA-event time of the whole loop on the cache's stream, or NULL. */
FL_EXPORT int fl_decode_greedy_loop(fl_model* m, fl_cache* c, const uint32_t* first_ids, int b, size_t rope_offset, int steps,
                          uint32_t* out_ids, float* elapsed_ms);

/* ---- continuous batching: sequence slots with their own lengths (SURVEY.md section 8f-3) -------------------------------------
 * The reference serialises requests at batch 1 under a mutex (api/chat.rs:206-208) and runs streams concurrently at batch 1 each
 * (models/mod.rs:151-175).  A cache created with max_batch > 1 holds max_batch independent sequence SLOTS; fl_forward_slots feeds
 * t new tokens to each of n distinct slots in ONE forward -- a new request's prompt (n = 1, t = prompt length) or one decode step
 * of every running request (t = 1), whatever their lengths -- with a RoPE position per row (explicit, like fl_forward's, so the
 * Mistral/Qwen2 adapters' +1-per-call rule survives per request).  logits_host: f32 [n, vocab], row i = slot slots[i].
 * A cache is driven either by the uniform calls above or by slots; fl_cache_reset switches back. */
FL_EXPORT int fl_forward_slots(fl_model* m, fl_cache* c, const int* slots, const uint32_t* ids, int n, int t, const size_t* rope_offsets,
                               float* logits_host);
FL_EXPORT int fl_cache_slot_reset(fl_cache* c, int slot);        /* the slot's sequence is finished: length := 0 */
FL_EXPORT int fl_cache_slot_len(fl_cache* c, int slot, int* out);

/* Diagnostics (no reference counterpart): the router's decisions in the LAST forward on this cache (Mixtral only) -- experts
 * [layers][rows][num_experts_per_tok] in pick order (MixtralSparseMoeBlock's sort, models/mixtral.rs via candle-transformers) and
 * margins [layers][rows] = softmax-probability gap between the last picked expert and the best one left out; rows = batch x t of
 * that forward.  top-k routing is discontinuous: a sharded run whose hidden state differs in the last f32 bits can pick another
 * expert where the margin is ~0, so the sharded-vs-single-GPU checks (bench.py, tests/test_tp.py) compare logits only where the
 * routing agrees and require every disagreement to sit on such a near-tie. */
FL_EXPORT int fl_cache_moe_routing(fl_cache* c, int rows, int32_t* experts, float* margins);

/* ---- sampling (host arithmetic: the reference samples on the host from every forward's logits) --- */
/* LogitsProcessor::new(seed, Some(temperature), None): temperature < 1e-7 => arg-max (IEEE total order, LAST index among
 * equal maxima); otherwise softmax(logits * (1/T as f32)) with a sequential f32 denominator, then
 * WeightedIndex<f32>::sample over StdRng::seed_from_u64(seed) (ChaCha12).  The reference always passes seed 0. */
FL_EXPORT int fl_sampler_create(uint64_t seed, double temperature, fl_sampler** out);
FL_EXPORT int fl_sampler_sample(fl_sampler* s, const float* logits_host, size_t n, uint32_t* token);
/* The arg-max rule above for every row of a host f32 [rows, n] matrix (a batch of greedy requests); tokens: host u32 [rows]. */
FL_EXPORT int fl_argmax_rows(const float* logits_host, int rows, size_t n, uint32_t* tokens);
FL_EXPORT int fl_sampler_next_u32(fl_sampler* s, uint32_t* out);  /* the generator's next raw word (known-answer tests) */
FL_EXPORT int fl_sampler_destroy(fl_sampler* s);
/* fl_forward, then sample row 0 of the logits (the generate loop only looks at logits.get(0), models/mod.rs:421); one
 * vocab*4-byte read-back, no caller-side logits buffer.  next_id: host u32 [1]. */
FL_EXPORT int fl_forward_sample(fl_model* m, fl_cache* c, const uint32_t* ids, int b, int t, size_t rope_offset, fl_sampler* s,
                                uint32_t* next_id);

/* Opt-in fast path of the same call: the soft-max weights, their prefix sums and the search run ON THE DEVICE (the sampler object
 * still owns the generator and hands over its one draw per sample, so a request's random stream is unchanged); 4 bytes travel back
 * instead of vocab * 4.  Not bit-identical to the host path by construction: the prefix sums come from a block scan, so a draw
 * within ~1e-6 (relative) of a boundary between two tokens may pick the neighbour.  The parity path is fl_forward_sample. */
FL_EXPORT int fl_forward_sample_device(fl_model* m, fl_cache* c, const uint32_t* ids, int b, int t, size_t rope_offset, fl_sampler* s,
                                       uint32_t* next_id);

/* ---- embeddings (BERT family) ------------------------------------------------------------------ */
/* Supported encoder shapes: head_dim (hidden / heads) 32 or 64, hidden and intermediate multiples of 64 with hidden <= 1024
 * (all-MiniLM-L6-v2, BERT-base and BERT-large sized models such as e5 / gte), up to 512 positions; any other shape fails at
 * fl_model_create with FL_ERR_UNSUPPORTED.
 * ids/mask: host u32 [b, t]; mask may be NULL (all ones).  out: host f32 [b, hidden], mean-pooled and L2-normalised. */
FL_EXPORT int fl_embed(fl_model* m, const uint32_t* ids, const uint32_t* mask, int b, int t, float* out);
/* Sentences of different lengths in ONE encoder pass, no padding: sentence i is ids[o_i, o_i + lengths[i]) with
 * o_i = lengths[0] + ... + lengths[i-1]; every token of a sentence is pooled (the all-ones mask a lone sentence has).
 * out: host f32 [n, hidden].  Row i equals fl_embed(m, ids + o_i, NULL, 1, lengths[i], ...) bit for bit.
 * FL_ERR_INVALID for a NULL pointer, n < 1, a non-BERT model, a length < 1 or > max_position_embeddings, an id >= vocab, or a
 * total token count T with T x max(3 x hidden, intermediate) > INT32_MAX; all are rejected before any device work. */
FL_EXPORT int fl_embed_packed(fl_model* m, const uint32_t* ids, const int32_t* lengths, int n, float* out);
/* Benchmark hook: one fl_embed, then `repeats` device-resident encoder passes over the same (already uploaded) batch;
 * device_ms = CUDA-event time of those repeats on the model's stream. */
FL_EXPORT int fl_embed_timed(fl_model* m, const uint32_t* ids, const uint32_t* mask, int b, int t, float* out, int repeats, float* device_ms);

/* ---- tensor / expert parallelism (one process per GPU; the library owns the NCCL communicator) -- */
FL_EXPORT int fl_comm_unique_id(void* out_128_bytes);            /* rank 0 creates, the host side broadcasts it */
FL_EXPORT int fl_comm_init(int rank, int world, const void* unique_id_128_bytes);
/* Peer-memory exchange area of the persistent decode kernel's in-kernel all-reduce (CUDA IPC over NVLink): every rank exports
 * its buffer handle, the host side all-gathers the 64-byte handles, every rank imports all of them ([world][64] bytes). */
FL_EXPORT int fl_comm_ipc_export(void* handle_64_bytes);
FL_EXPORT int fl_comm_ipc_import(const void* handles, int world, int rank);
FL_EXPORT int fl_comm_destroy(void);

/* ---- measurement hooks (bench.py / tests) ------------------------------------------------------- */
/* Per-kernel CUDA-event profile of subsequent forwards and embeddings (eager launches without PDL, events on the launching stream). */
FL_EXPORT int fl_prof_begin(void);
/* Writes a JSON array [{"kernel": name, "launches": n, "ms": total_ms, "bytes": algorithmic_bytes}, ...]. */
FL_EXPORT int fl_prof_end(char* json_out, size_t cap);
FL_EXPORT int fl_launch_count(uint64_t* kernels_launched);       /* kernels this library launched since load */

#ifdef __cplusplus
}
#endif
#endif /* FASTLLM_B200_H */
