"""Host-side mirror of the reference's trait-based model API over the C ABI.

The reference is Rust and there is no Rust toolchain in this image, so the drop-in host side ships twice:
  * `host/fastllm_host.hpp` -- the C++ mirror (compiled, what INTEGRATION.md's Rust shim is a transliteration of);
  * this module -- the same interface in Python, used by tests/ and bench.py so the parity tests read like the
    reference's own tests (same names, same argument meaning, same offset rules, same error behaviour).

Reference interfaces mirrored (paths under /root/reference/src/models):
  ModelInitializer {initialize_model, initialize_cache, forward}     model_initializer.rs:6-22
  ModelCache {increment_offset, reset, get_offset}                   cache.rs:5-10
  LlamaWithConfig / LlamaCache                                       llama.rs:52-149
  MistralWithConfig / MistralCache                                   mistral.rs:16-236
  QwenWithConfig / QwenCache                                         qwen.rs:12-151
  Model::generate + candle LogitsProcessor (arg-max / temperature)   mod.rs:363-463
"""
from __future__ import annotations

import ctypes as C
import json
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import FastllmError, FlConfig


# --------------------------------------------------------------------------------------------------------------------
# thin RAII handles over the C ABI
# --------------------------------------------------------------------------------------------------------------------
class DeviceModel:
    """fl_model*: device weights (shared between clones)."""

    def __init__(self, cfg: FlConfig, device: int = 0, _handle=None):
        _lib.init(device)
        self.lib = _lib.load()
        self.cfg = cfg
        self.device = device
        if _handle is None:
            h = C.c_void_p()
            _lib.check(self.lib.fl_model_create(C.byref(cfg), C.byref(h)))
            self.h = h
        else:
            self.h = _handle

    def put_tensor(self, name: str, arr: np.ndarray):
        if arr.dtype == np.float32:
            dt = _lib.FL_DTYPE_F32
        elif arr.dtype == np.float16:
            dt = _lib.FL_DTYPE_F16
        elif arr.dtype == np.uint16:        # raw bf16 bit patterns
            dt = _lib.FL_DTYPE_BF16
        else:
            raise FastllmError(-1, f"unsupported dtype {arr.dtype} for {name}")
        arr = np.ascontiguousarray(arr)
        shape = (C.c_int64 * arr.ndim)(*arr.shape)
        _lib.check(self.lib.fl_model_put_tensor(self.h, name.encode(), dt, shape, arr.ndim, arr.ctypes.data_as(C.c_void_p)))

    def random_init(self, seed: int = 0, std: float = 0.02):
        _lib.check(self.lib.fl_model_random_init(self.h, seed, std))

    def finalize(self):
        _lib.check(self.lib.fl_model_finalize(self.h))

    def clone(self) -> "DeviceModel":
        h = C.c_void_p()
        _lib.check(self.lib.fl_model_clone(self.h, C.byref(h)))
        return DeviceModel(self.cfg, self.device, _handle=h)

    def streamed_bytes(self) -> int:
        n = C.c_uint64()
        _lib.check(self.lib.fl_model_weight_bytes(self.h, C.byref(n)))
        return n.value

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.fl_model_destroy(self.h)
                self.h = None
        except Exception:
            pass


class DeviceCache:
    """fl_cache*: paged KV cache + per-cache stream/workspaces."""

    def __init__(self, model: DeviceModel, max_batch: int, max_seq: int):
        self.model, self.lib = model, model.lib
        self.max_batch, self.max_seq = max_batch, max_seq
        self.vocab = model.cfg.vocab_size
        h = C.c_void_p()
        _lib.check(self.lib.fl_cache_create(model.h, max_batch, max_seq, C.byref(h)))
        self.h = h

    def reset(self):
        _lib.check(self.lib.fl_cache_reset(self.h))

    def kv_len(self) -> int:
        n = C.c_int()
        _lib.check(self.lib.fl_cache_kv_len(self.h, C.byref(n)))
        return n.value

    def fill_synthetic(self, batch: int, kv_len: int, seed: int = 3):
        _lib.check(self.lib.fl_cache_fill_synthetic(self.h, batch, kv_len, seed))

    def forward(self, ids: np.ndarray, rope_offset: int) -> np.ndarray:
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        if ids.ndim != 2:
            raise FastllmError(-1, f"input must be [batch, seq], got shape {ids.shape}")   # input.dims2()? in the reference
        b, t = ids.shape
        out = np.empty((b, self.vocab), dtype=np.float32)
        _lib.check(self.lib.fl_forward(self.model.h, self.h, ids.ctypes.data_as(C.c_void_p), b, t, rope_offset,
                                       out.ctypes.data_as(C.c_void_p)))
        return out

    def forward_greedy(self, ids: np.ndarray, rope_offset: int) -> np.ndarray:
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        b, t = ids.shape
        out = np.empty((b,), dtype=np.uint32)
        _lib.check(self.lib.fl_forward_greedy(self.model.h, self.h, ids.ctypes.data_as(C.c_void_p), b, t, rope_offset,
                                              out.ctypes.data_as(C.c_void_p)))
        return out

    def forward_sample(self, ids: np.ndarray, rope_offset: int, logits_processor: "LogitsProcessor") -> int:
        """fl_forward + LogitsProcessor::sample of row 0 in one call (one V*4-byte read-back, no logits array on this side)."""
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        if ids.ndim != 2:
            raise FastllmError(-1, f"input must be [batch, seq], got shape {ids.shape}")
        b, t = ids.shape
        tok = C.c_uint32()
        _lib.check(self.lib.fl_forward_sample(self.model.h, self.h, ids.ctypes.data_as(C.c_void_p), b, t, rope_offset,
                                              logits_processor.h, C.byref(tok)))
        return tok.value

    def forward_sample_device(self, ids: np.ndarray, rope_offset: int, logits_processor: "LogitsProcessor") -> int:
        """The opt-in fast path of forward_sample: soft-max weights, prefix sums and the search run on the device (4 bytes come
        back instead of vocab * 4); the sampler object still owns the generator.  Not bit-identical to the host path by
        construction (block scan instead of a sequential sum): see include/fastllm_b200.h."""
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        if ids.ndim != 2:
            raise FastllmError(-1, f"input must be [batch, seq], got shape {ids.shape}")
        b, t = ids.shape
        tok = C.c_uint32()
        _lib.check(self.lib.fl_forward_sample_device(self.model.h, self.h, ids.ctypes.data_as(C.c_void_p), b, t, rope_offset,
                                                     logits_processor.h, C.byref(tok)))
        return tok.value

    def forward_slots(self, slots, ids: np.ndarray, rope_offsets) -> np.ndarray:
        """Ragged forward (continuous batching): row i of ids [n, t] is fed to the sequence in cache slot slots[i] at RoPE
        position rope_offsets[i]; the slots keep their own lengths.  -> f32 [n, vocab]."""
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        if ids.ndim != 2:
            raise FastllmError(-1, f"input must be [batch, seq], got shape {ids.shape}")
        n, t = ids.shape
        sl = np.ascontiguousarray(slots, dtype=np.int32).reshape(-1)
        ro = np.ascontiguousarray(rope_offsets, dtype=np.uint64).reshape(-1)
        if sl.size != n or ro.size != n:
            raise FastllmError(-1, "slots / rope_offsets must have one entry per row of ids")
        out = np.empty((n, self.vocab), dtype=np.float32)
        _lib.check(self.lib.fl_forward_slots(self.model.h, self.h, sl.ctypes.data_as(C.c_void_p), ids.ctypes.data_as(C.c_void_p), n, t,
                                             ro.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)))
        return out

    def slot_reset(self, slot: int):
        _lib.check(self.lib.fl_cache_slot_reset(self.h, slot))

    def slot_len(self, slot: int) -> int:
        n = C.c_int()
        _lib.check(self.lib.fl_cache_slot_len(self.h, slot, C.byref(n)))
        return n.value

    def moe_routing(self, rows: int):
        """Router decisions of the last forward (Mixtral): experts [layers, rows, top_k] int32 in pick order, margins [layers, rows] f32."""
        cfg = self.model.cfg
        ex = np.empty((cfg.num_hidden_layers, rows, cfg.num_experts_per_tok), dtype=np.int32)
        mg = np.empty((cfg.num_hidden_layers, rows), dtype=np.float32)
        _lib.check(self.lib.fl_cache_moe_routing(self.h, rows, ex.ctypes.data_as(C.c_void_p), mg.ctypes.data_as(C.c_void_p)))
        return ex, mg

    def decode_greedy_loop(self, first_ids: np.ndarray, rope_offset: int, steps: int):
        first = np.ascontiguousarray(first_ids, dtype=np.uint32).reshape(-1)
        b = first.shape[0]
        out = np.empty((steps, b), dtype=np.uint32)
        ms = C.c_float()
        _lib.check(self.lib.fl_decode_greedy_loop(self.model.h, self.h, first.ctypes.data_as(C.c_void_p), b, rope_offset,
                                                  steps, out.ctypes.data_as(C.c_void_p), C.byref(ms)))
        return out, ms.value

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.fl_cache_destroy(self.h)
                self.h = None
        except Exception:
            pass


def prof_begin():
    _lib.check(_lib.load().fl_prof_begin())


def prof_end() -> list:
    buf = C.create_string_buffer(1 << 16)
    _lib.check(_lib.load().fl_prof_end(buf, len(buf)))
    return json.loads(buf.value.decode())


def launch_count() -> int:
    n = C.c_uint64()
    _lib.check(_lib.load().fl_launch_count(C.byref(n)))
    return n.value


# --------------------------------------------------------------------------------------------------------------------
# configs (what the adapters deserialize from config.json)
# --------------------------------------------------------------------------------------------------------------------
@dataclass
class ConfigFile:
    """llama.rs:17-29 / mistral.rs:78-91 / models/config.rs:5-18 (BaseModelConfig)."""
    hidden_size: int
    intermediate_size: int
    vocab_size: int
    num_hidden_layers: int
    num_attention_heads: int
    num_key_value_heads: int | None = None
    rms_norm_eps: float = 1e-5
    rope_theta: float | None = None
    max_position_embeddings: int | None = None
    sliding_window: int | None = None
    torch_dtype: str | None = None     # never consulted by the reference (huggingface.rs:132)
    tp_rank: int = 0                   # tensor parallelism (no reference counterpart): rank / size of this process
    tp_size: int = 1                   # (for Mixtral the same two fields mean expert-parallel rank / size)
    num_local_experts: int = 0         # Mixtral
    num_experts_per_tok: int = 2
    ep_dp_attention: bool = False      # Mixtral expert parallelism: sequences data-parallel, tokens all-to-all to the experts


def _fl_config(arch: str, cf: ConfigFile, default_max_pos: int, sliding_window: int, qkv_bias: bool) -> FlConfig:
    c = FlConfig()
    c.arch = _lib.FL_ARCH[arch]
    c.hidden_size, c.intermediate_size, c.vocab_size = cf.hidden_size, cf.intermediate_size, cf.vocab_size
    c.num_hidden_layers, c.num_attention_heads = cf.num_hidden_layers, cf.num_attention_heads
    c.num_key_value_heads = cf.num_key_value_heads or cf.num_attention_heads
    c.max_position_embeddings = cf.max_position_embeddings or default_max_pos
    c.sliding_window = sliding_window
    c.qkv_bias = 1 if qkv_bias else 0
    c.norm_eps = cf.rms_norm_eps
    c.rope_theta = float(cf.rope_theta if cf.rope_theta is not None else 10000.0)
    c.tp_rank, c.tp_size = cf.tp_rank, cf.tp_size
    c.num_local_experts, c.num_experts_per_tok = cf.num_local_experts, cf.num_experts_per_tok
    c.ep_dp_attention = 1 if cf.ep_dp_attention else 0
    return c


# --------------------------------------------------------------------------------------------------------------------
# ModelCache implementations
# --------------------------------------------------------------------------------------------------------------------
class _OffsetCache:
    """ModelCache (cache.rs:5-10): increment_offset / reset / get_offset."""

    def __init__(self):
        self.seqlen_offset = 0

    def increment_offset(self):
        self.seqlen_offset += 1

    def reset(self):
        self.seqlen_offset = 0

    def get_offset(self) -> int:
        return self.seqlen_offset


class LlamaCache(_OffsetCache):
    """llama.rs:61-92.  In the reference this owns candle's KV `Cache`; here it owns the device KV cache, created lazily
    on the first forward because initialize_cache(device, dtype) gets no model argument (SURVEY.md section 8b)."""

    def __init__(self):
        super().__init__()
        self.inner: DeviceCache | None = None


class MistralCache(_OffsetCache):
    """mistral.rs:16-47: only the offset; the KV lives inside the model object."""


class QwenCache(_OffsetCache):
    """qwen.rs:58-87."""


# --------------------------------------------------------------------------------------------------------------------
# ModelInitializer implementations
# --------------------------------------------------------------------------------------------------------------------
class _CausalBase:
    arch = ""
    family = ""
    architectures: tuple = ()
    KV_CAPACITY = 4096        # tokens of KV a cache can hold (the reference grows by `cat`; we preallocate pages)
    MAX_BATCH = 1

    def __init__(self, dev: DeviceModel, cfg: FlConfig):
        self.dev, self.cfg = dev, cfg

    @classmethod
    def _to_fl_config(cls, config: ConfigFile) -> FlConfig:
        raise NotImplementedError

    @classmethod
    def initialize_model(cls, config: ConfigFile, tensors: dict | None, dtype="bf16", device: int = 0, *, random_seed=None,
                         std: float = 0.02):
        """ModelInitializer::initialize_model(&Config, HashMap<String,Tensor>, DType, &Device) -> (Self, Cache).
        `tensors` maps HF names to numpy arrays (f32 / f16 / uint16 bf16 bits); they are rounded to bf16 as
        VarBuilder::from_tensors(.., BF16, ..) would (main.rs:120).  tensors=None + random_seed = synthetic weights."""
        cfg = cls._to_fl_config(config)
        dev = DeviceModel(cfg, device)
        if tensors is None:
            dev.random_init(0 if random_seed is None else random_seed, std)
        else:
            # a dict, or any iterable of (name, array) -- e.g. safetensors_io.iter_tensors(dir), which hands over views of the
            # memory-mapped checkpoint one tensor at a time (huggingface.rs:81-130 without the whole-file reads)
            for name, arr in (tensors.items() if hasattr(tensors, "items") else tensors):
                dev.put_tensor(name, np.asarray(arr))
        dev.finalize()
        self = cls(dev, cfg)
        return self, cls.initialize_cache(device, dtype)

    @classmethod
    def get_family(cls) -> str:
        return cls.family

    @classmethod
    def supports_architecture(cls, architecture: str) -> bool:
        return architecture in cls.architectures

    def _capacity(self) -> int:
        return min(self.KV_CAPACITY, self.cfg.max_position_embeddings)


class LlamaWithConfig(_CausalBase):
    """llama.rs:52-160."""
    arch, family, architectures = "llama", "Llama", ("LlamaForCausalLM",)

    @classmethod
    def _to_fl_config(cls, cf: ConfigFile) -> FlConfig:
        # llama.rs:31-50: rope_theta default 1e4, max_position_embeddings default 4096, no sliding window, no bias
        return _fl_config("llama", cf, 4096, 0, False)

    @staticmethod
    def initialize_cache(device=0, dtype="bf16") -> LlamaCache:
        return LlamaCache()

    def forward(self, input: np.ndarray, pos: int, cache: LlamaCache) -> np.ndarray:
        """llama.rs:147-149: model.forward(input, pos, &mut cache.inner) -> f32 [b, V]."""
        ids = np.asarray(input)
        if cache.inner is None:
            cache.inner = DeviceCache(self.dev, max(self.MAX_BATCH, ids.shape[0] if ids.ndim == 2 else 1), self._capacity())
        return cache.inner.forward(ids, pos)

    def clone(self) -> "LlamaWithConfig":
        return LlamaWithConfig(self.dev.clone(), self.cfg)


class MistralWithConfig(_CausalBase):
    """mistral.rs:49-248.  The KV cache lives in the model object (one per clone), as in candle's mistral::Model."""
    arch, family, architectures = "mistral", "Mistral", ("MistralForCausalLM",)
    cache_cls = MistralCache

    def __init__(self, dev: DeviceModel, cfg: FlConfig):
        super().__init__(dev, cfg)
        self._kv: DeviceCache | None = None

    @classmethod
    def _to_fl_config(cls, cf: ConfigFile) -> FlConfig:
        # mistral.rs:93-154: asserts on head dims / GQA (raised as FastllmError by fl_model_create),
        # sliding_window = Some(cfg.unwrap_or(4096)), max_position_embeddings default 32768
        return _fl_config("mistral", cf, 32768, cf.sliding_window if cf.sliding_window is not None else 4096, False)

    @classmethod
    def initialize_cache(cls, device=0, dtype="bf16"):
        return cls.cache_cls()

    def clear_kv_cache(self):
        if self._kv is not None:
            self._kv.reset()

    def forward(self, input: np.ndarray, _pos: int, cache) -> np.ndarray:
        """mistral.rs:206-236 / qwen.rs:129-145: `_pos` ignored; KV cleared when the offset is 0; RoPE offset = the
        cache's seqlen_offset, which then grows by ONE per call (not by seq_len).  Returns [b, 1, V]."""
        ids = np.asarray(input)
        if ids.ndim != 2:
            raise FastllmError(-1, f"input must be [batch, seq], got shape {ids.shape}")
        if self._kv is None or (cache.get_offset() == 0 and self._kv.max_batch < ids.shape[0]):
            self._kv = DeviceCache(self.dev, max(self.MAX_BATCH, ids.shape[0]), self._capacity())   # a wider batch starts a new KV
        if cache.get_offset() == 0:
            self.clear_kv_cache()
        out = self._kv.forward(ids, cache.get_offset())
        cache.increment_offset()
        return out[:, None, :]

    def clone(self):
        return type(self)(self.dev.clone(), self.cfg)


class QwenWithConfig(MistralWithConfig):
    """qwen.rs:12-186 (ModelForward::forward_pass + clear_cache; q/k/v bias)."""
    arch, family = "qwen2", "Qwen"
    architectures = ("Qwen2ForCausalLM", "Qwen2_5_VLForConditionalGeneration")
    cache_cls = QwenCache

    @classmethod
    def _to_fl_config(cls, cf: ConfigFile) -> FlConfig:
        # qwen.rs:30-56: sliding_window.unwrap_or(4096), max_position_embeddings default 32768, rope default 1e4
        return _fl_config("qwen2", cf, 32768, cf.sliding_window if cf.sliding_window is not None else 4096, True)

    def forward_pass(self, input, cache):
        return self.forward(input, 0, cache)

    def clear_cache(self):
        self.clear_kv_cache()


class MixtralWithConfig(MistralWithConfig):
    """MixtralForCausalLM.  The reference does NOT wire this architecture (model_registry.rs:169-182 has no matching key,
    mistral.rs:244-246 accepts only MistralForCausalLM); the adapter follows the Mistral one (same offset rule) over
    candle-transformers' mixtral model: attention as Mistral, MLP replaced by the top-k sparse-MoE block."""
    arch, family, architectures = "mixtral", "Mixtral", ("MixtralForCausalLM",)

    @classmethod
    def _to_fl_config(cls, cf: ConfigFile) -> FlConfig:
        return _fl_config("mixtral", cf, 32768, cf.sliding_window if cf.sliding_window is not None else 4096, False)


class LogitsProcessor:
    """candle's LogitsProcessor as the reference builds it: LogitsProcessor::new(Default::default(), Some(temperature as f64),
    None) (mod.rs:157-158, 373-374).  Temperature < 1e-7 => arg-max (IEEE total order, LAST index among equal maxima);
    otherwise soft-max + WeightedIndex over StdRng::seed_from_u64(seed).  The arithmetic is the library's (fl_sampler_*,
    csrc/sampler.hpp): host code, because the reference samples on the host from the logits every forward returns."""

    def __init__(self, seed: int = 0, temperature: float | None = None):
        self.lib = _lib.load()
        h = C.c_void_p()
        _lib.check(self.lib.fl_sampler_create(seed, -1.0 if temperature is None else float(temperature), C.byref(h)))
        self.h = h

    def sample(self, logits: np.ndarray) -> int:
        v = np.ascontiguousarray(logits, dtype=np.float32).reshape(-1)       # logits.to_dtype(F32)
        tok = C.c_uint32()
        _lib.check(self.lib.fl_sampler_sample(self.h, v.ctypes.data_as(C.c_void_p), v.size, C.byref(tok)))
        return tok.value

    def next_u32(self) -> int:
        w = C.c_uint32()
        _lib.check(self.lib.fl_sampler_next_u32(self.h, C.byref(w)))
        return w.value

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.fl_sampler_destroy(self.h)
                self.h = None
        except Exception:
            pass


def sample_argmax(logits: np.ndarray) -> int:
    """LogitsProcessor::sample with temperature None/<1e-7: arg-max, LAST index among equal maxima (mod.rs:425-428)."""
    global _greedy
    if _greedy is None:
        _greedy = LogitsProcessor(0, None)      # arg-max never touches the generator: one shared instance
    return _greedy.sample(logits)


_greedy = None


def sample_argmax_rows(logits: np.ndarray) -> np.ndarray:
    """sample_argmax for every row of [b, V] logits (a batch of greedy requests) in one library call -> u32 [b]."""
    v = np.ascontiguousarray(logits, dtype=np.float32)
    v = v.reshape(v.shape[0], -1)
    out = np.empty((v.shape[0],), dtype=np.uint32)
    _lib.check(_lib.load().fl_argmax_rows(v.ctypes.data_as(C.c_void_p), v.shape[0], v.shape[1], out.ctypes.data_as(C.c_void_p)))
    return out


class Model:
    """Model<M> (mod.rs:342-464) without the tokenizer: prompts are already token ids."""

    def __init__(self, model, cache, eos_token_id: int | None = 2):
        self.model, self.cache, self.eos_token_id = model, cache, eos_token_id

    def generate(self, prompt_ids, max_tokens: int, temperature: float = 0.0, return_logits: bool = False):
        self.cache = self.model.initialize_cache()                       # mod.rs:370
        # mod.rs:373-374: seed Default::default() = 0, `temperature as f64` of the API's f32 (chat.rs:24-25 defaults it to 0.0)
        logits_processor = LogitsProcessor(0, float(np.float32(temperature)))
        ids = np.asarray(prompt_ids, dtype=np.uint32).reshape(1, -1)    # mod.rs:386-394
        pos = 0
        logits = self.model.forward(ids, pos, self.cache)               # mod.rs:402-405
        pos += ids.shape[1]
        out, trace = [], []
        for _ in range(max_tokens):                                      # mod.rs:411-453
            last = np.asarray(logits)[0].reshape(-1)                     # logits.get(0)?.flatten_all()?
            if return_logits:
                trace.append(last.copy())
            tok = logits_processor.sample(last)                          # mod.rs:425-428
            if self.eos_token_id is not None and tok == self.eos_token_id:
                break                                                    # EOS: break before emitting (mod.rs:431-436)
            out.append(tok)
            logits = self.model.forward(np.array([[tok]], dtype=np.uint32), pos, self.cache)
            pos += 1
        return (out, trace) if return_logits else out

    def generate_batch(self, prompts, max_tokens: int, temperature: float = 0.0, max_batch: int = 64):
        """Request batching at the API boundary (SURVEY.md section 8f-3; the reference serialises requests at batch 1 under a
        mutex, chat.rs:206-208).  Exact by construction: only prompts of EQUAL token length share a batch, so the sequences of
        a group advance in lock-step through one [b, t] forward per step (no padding, one KV length), every sequence has its
        own LogitsProcessor seeded 0 like every request of the reference, and a sequence that hit EOS keeps its row (fed its
        last token, output ignored) until the group is done.  Same arithmetic per sequence as generate(p); the batch-b decode
        step runs on the dense path and batch-1 on the persistent path, so logits agree to the kernel tolerance (3e-3), not
        bitwise.  Returns one id list per prompt, in request order."""
        out = [None] * len(prompts)
        groups: dict = {}
        for i, p in enumerate(prompts):
            groups.setdefault(len(p), []).append(i)
        for idxs in groups.values():
            for k in range(0, len(idxs), max_batch):
                chunk = idxs[k:k + max_batch]
                for i, toks in zip(chunk, self._generate_group([prompts[i] for i in chunk], max_tokens, temperature)):
                    out[i] = toks
        return out

    def _generate_group(self, prompts, max_tokens: int, temperature: float):
        b = len(prompts)
        self.cache = self.model.initialize_cache()
        processors = [LogitsProcessor(0, float(np.float32(temperature))) for _ in range(b)]
        ids = np.asarray(prompts, dtype=np.uint32).reshape(b, -1)
        pos = 0
        logits = self.model.forward(ids, pos, self.cache)
        pos += ids.shape[1]
        outs = [[] for _ in range(b)]
        done = [False] * b
        nxt = np.ascontiguousarray(ids[:, -1:])
        for _ in range(max_tokens):
            rows = np.asarray(logits).reshape(b, -1)
            for i in range(b):
                if done[i]:
                    continue
                tok = processors[i].sample(rows[i])
                if self.eos_token_id is not None and tok == self.eos_token_id:
                    done[i] = True                                       # break before emitting, for this sequence only
                    continue
                outs[i].append(tok)
                nxt[i, 0] = tok
            if all(done):
                break
            logits = self.model.forward(nxt, pos, self.cache)
            pos += 1
        return outs


class ContinuousBatcher:
    """Continuous batching above fl_forward_slots (SURVEY.md section 8f-3).  The reference serialises chat requests at batch 1
    under one mutex (api/chat.rs:206-208); here up to `max_batch` requests of ANY lengths share the decode steps: a request is
    admitted into a free sequence slot as soon as one exists (its prompt is prefilled alone, [1, T]), every step then advances all
    running requests by one token in ONE ragged forward ([n, 1], per-slot KV lengths and RoPE positions), and a request that
    hits EOS or its token budget frees its slot for the next waiting one.  Per request the arithmetic is that of
    Model.generate: its own LogitsProcessor seeded 0 (mod.rs:373-374), EOS break before emitting (mod.rs:431-436), and the
    adapter's position rule -- Llama: the caller's position; Mistral / Qwen2: +1 per CALL (mistral.rs:234, qwen.rs:143).
    `cache` needs forward_slots(slots, ids, rope_offsets) -> [n, V], slot_reset(slot): a DeviceCache, or a stand-in in tests."""

    def __init__(self, model, max_batch: int = 8, eos_token_id: int | None = 2, cache=None):
        self.model, self.max_batch, self.eos_token_id = model, max_batch, eos_token_id
        self.position_per_call = getattr(model, "arch", "llama") != "llama"      # the Mistral/Qwen2 adapters' offset rule
        self.cache = cache if cache is not None else DeviceCache(model.dev, max_batch, model._capacity())
        self.steps = 0          # ragged decode forwards issued (tests / stats)

    def generate(self, prompts, max_tokens: int, temperature: float = 0.0):
        """-> one id list per prompt, in request order."""
        out = [[] for _ in prompts]
        waiting = list(range(len(prompts)))[::-1]
        free = list(range(self.max_batch))[::-1]
        running = {}            # slot -> [request, next RoPE position, LogitsProcessor, token to feed]
        if max_tokens <= 0:
            return out

        def take(logits_row, req, slot, state):
            """sample -> EOS / budget -> either keep the slot running or free it"""
            tok = state[2].sample(logits_row)
            if self.eos_token_id is not None and tok == self.eos_token_id:
                done = True
            else:
                out[req].append(tok)
                state[3] = tok
                done = len(out[req]) >= max_tokens
            if done:
                running.pop(slot, None)
                self.cache.slot_reset(slot)
                free.append(slot)
            else:
                running[slot] = state

        while waiting or running:
            while waiting and free:                                   # admit: one prompt at a time, alone in its forward
                req, slot = waiting.pop(), free.pop()
                ids = np.asarray(prompts[req], dtype=np.uint32).reshape(1, -1)
                logits = self.cache.forward_slots([slot], ids, [0])
                state = [req, 1 if self.position_per_call else ids.shape[1], LogitsProcessor(0, float(np.float32(temperature))), 0]
                take(np.asarray(logits)[0].reshape(-1), req, slot, state)
            if not running:
                continue
            slots = sorted(running)
            ids = np.array([[running[s][3]] for s in slots], dtype=np.uint32)
            logits = np.asarray(self.cache.forward_slots(slots, ids, [running[s][1] for s in slots]))
            self.steps += 1
            for i, s in enumerate(slots):
                st = running[s]
                st[1] += 1
                take(logits[i].reshape(-1), st[0], s, st)
        return out


# --------------------------------------------------------------------------------------------------------------------
# EmbeddingModel (models/embeddings.rs:17-38) -- BERT / MiniLM sentence encoder
# --------------------------------------------------------------------------------------------------------------------
@dataclass
class BertConfig:
    """models/embeddings.rs:46-54 (+ the vocabulary size the reference takes from the tokenizer, :301-306)."""
    hidden_size: int = 384
    num_attention_heads: int = 12
    num_hidden_layers: int = 6
    intermediate_size: int = 1536
    max_position_embeddings: int = 512
    layer_norm_eps: float = 1e-12
    vocab_size: int = 30522

    @classmethod
    def from_json(cls, path_or_dict) -> "BertConfig":
        """The seven dimensions from a HuggingFace BERT `config.json` (a path, or the parsed dict).  Every other key
        (`type_vocab_size`, `architectures`, `hidden_act`, ...) is ignored; a missing dimension raises ValueError naming it."""
        if isinstance(path_or_dict, dict):
            d = path_or_dict
        else:
            with open(path_or_dict) as f:
                d = json.load(f)
        missing = [k for k in cls.__dataclass_fields__ if k not in d]
        if missing:
            raise ValueError(f"BERT config.json lacks {', '.join(missing)}")
        return cls(int(d["hidden_size"]), int(d["num_attention_heads"]), int(d["num_hidden_layers"]), int(d["intermediate_size"]),
                   int(d["max_position_embeddings"]), float(d["layer_norm_eps"]), int(d["vocab_size"]))


class MiniLMModel:
    """MiniLMModel (models/embeddings.rs:245-447) after tokenisation: `embed_ids` takes the token ids (and the tokenizer's
    attention mask) and returns what EmbeddingModel::embed returns: the mean-pooled, L2-normalised f32 vector(s)."""
    family, architectures = "bert", ("BertModel", "RobertaModel", "DebertaModel")

    def __init__(self, config: BertConfig, tensors: dict | None, device: int = 0, model_id: str = "sentence-transformers/all-MiniLM-L6-v2",
                 random_seed=None, std: float = 0.02):
        c = FlConfig()
        c.arch = _lib.FL_ARCH["bert"]
        c.hidden_size, c.intermediate_size, c.vocab_size = config.hidden_size, config.intermediate_size, config.vocab_size
        c.num_hidden_layers, c.num_attention_heads = config.num_hidden_layers, config.num_attention_heads
        c.num_key_value_heads = config.num_attention_heads
        c.max_position_embeddings = config.max_position_embeddings
        c.norm_eps = config.layer_norm_eps
        c.rope_theta, c.tp_rank, c.tp_size = 0.0, 0, 1
        self.config, self._model_id = config, model_id
        self.dev = DeviceModel(c, device)
        if tensors is None:
            self.dev.random_init(0 if random_seed is None else random_seed, std)
        else:
            for name, arr in tensors.items():
                self.dev.put_tensor(name, np.asarray(arr, dtype=np.float32))
        self.dev.finalize()

    @classmethod
    def get_family(cls) -> str:
        return cls.family

    @classmethod
    def supports_architecture(cls, architecture: str) -> bool:
        return architecture in cls.architectures

    def model_id(self) -> str:
        return self._model_id

    def embedding_size(self) -> int:
        return self.config.hidden_size          # the reference hard-codes 384 (embeddings.rs:453-455)

    def embed_ids(self, ids: np.ndarray, mask: np.ndarray | None = None) -> np.ndarray:
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        if ids.ndim == 1:
            ids = ids[None]
        b, t = ids.shape
        out = np.empty((b, self.config.hidden_size), dtype=np.float32)
        mptr = None
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint32).reshape(b, t)
            mptr = mask.ctypes.data_as(C.c_void_p)
        _lib.check(self.dev.lib.fl_embed(self.dev.h, ids.ctypes.data_as(C.c_void_p), mptr, b, t, out.ctypes.data_as(C.c_void_p)))
        return out

    def embed_many(self, sentences, max_batch: int = 256) -> np.ndarray:
        """`input: [String]` batching (SURVEY.md section 8f-3; the reference takes one string per request, api/embeddings.rs:11-15).
        Exact by construction: the reference's attention applies NO mask (embeddings.rs:155-159) and a lone sentence has an
        all-ones mask, so padding would change results; sentences of EQUAL token length are therefore grouped into one [b, t]
        call each (no padding) and the rows scattered back in request order.  Returns f32 [len(sentences), hidden]."""
        out = np.empty((len(sentences), self.config.hidden_size), dtype=np.float32)
        groups: dict = {}
        for i, s in enumerate(sentences):
            groups.setdefault(len(s), []).append(i)
        for idxs in groups.values():
            for k in range(0, len(idxs), max_batch):
                chunk = idxs[k:k + max_batch]
                out[chunk] = self.embed_ids(np.asarray([sentences[i] for i in chunk], dtype=np.uint32))
        return out

    def embed_packed(self, sentences) -> np.ndarray:
        """`input: [String]` in ONE encoder pass (fl_embed_packed): the sentences (1-D id sequences of any lengths) are concatenated
        without padding, and row i equals embed_ids of sentence i alone bit for bit.  Returns f32 [len(sentences), hidden] in request
        order."""
        out = np.empty((len(sentences), self.config.hidden_size), dtype=np.float32)
        if not len(sentences):
            return out
        parts = [np.asarray(s, dtype=np.uint32).reshape(-1) for s in sentences]
        ids = np.ascontiguousarray(np.concatenate(parts), dtype=np.uint32)
        lengths = np.array([len(p) for p in parts], dtype=np.int32)
        _lib.check(self.dev.lib.fl_embed_packed(self.dev.h, ids.ctypes.data_as(C.c_void_p), lengths.ctypes.data_as(C.c_void_p),
                                                len(parts), out.ctypes.data_as(C.c_void_p)))
        return out

    def embed_ids_timed(self, ids: np.ndarray, repeats: int):
        """-> (embeddings, device ms for `repeats` device-resident encoder passes over the uploaded batch)."""
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        b, t = ids.shape
        out = np.empty((b, self.config.hidden_size), dtype=np.float32)
        ms = C.c_float()
        _lib.check(self.dev.lib.fl_embed_timed(self.dev.h, ids.ctypes.data_as(C.c_void_p), None, b, t, out.ctypes.data_as(C.c_void_p),
                                               repeats, C.byref(ms)))
        return out, ms.value

    def compute_similarity(self, ids1, ids2) -> float:
        """EmbeddingModel::compute_similarity default impl (embeddings.rs:22-37): cosine of the two embeddings."""
        v1, v2 = self.embed_ids(ids1)[0], self.embed_ids(ids2)[0]
        return float(np.dot(v1, v2) / (np.linalg.norm(v1) * np.linalg.norm(v2)))
