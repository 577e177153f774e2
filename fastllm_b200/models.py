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

    def load(self, tensors, random_seed=None, std: float = 0.02, dtype=None):
        """Synthetic weights (tensors=None: fl_model_random_init with random_seed, default 0) or an upload of `tensors`, then
        finalize.  `tensors` is a dict or any iterable of (name, array) -- e.g. safetensors_io.iter_tensors(dir), which hands over
        views of the memory-mapped checkpoint one tensor at a time (huggingface.rs:81-130 without the whole-file reads); `dtype`
        casts every array first."""
        if tensors is None:
            self.random_init(0 if random_seed is None else random_seed, std)
        else:
            for name, arr in (tensors.items() if hasattr(tensors, "items") else tensors):
                self.put_tensor(name, np.asarray(arr, dtype=dtype))
        self.finalize()

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
    """fl_cache*: paged KV cache + per-cache stream/workspaces.  pool_tokens=None: every slot can reach max_seq (a pool of
    max_batch * ceil(max_seq / 64) pages); otherwise the slots share a pool of pool_tokens tokens (rounded up to 64-token pages),
    taken as sequences grow.  kv_dtype="fp8_e4m3" stores K and V as FP8 e4m3 (fl_cache_create_pool_kv): half the bytes per token,
    slot and packed calls only."""

    KV_DTYPES = {"bf16": 0, "fp8_e4m3": 1}      # fl_kv_dtype

    def __init__(self, model: DeviceModel, max_batch: int, max_seq: int, pool_tokens: int | None = None, kv_dtype: str = "bf16"):
        if kv_dtype not in self.KV_DTYPES:
            raise ValueError(f"kv_dtype must be one of {sorted(self.KV_DTYPES)}, not {kv_dtype!r}")
        self.model, self.lib = model, model.lib
        self.max_batch, self.max_seq, self.kv_dtype = max_batch, max_seq, kv_dtype
        self.vocab = model.cfg.vocab_size
        h = C.c_void_p()
        if kv_dtype != "bf16":
            tokens = pool_tokens if pool_tokens is not None else max_batch * _pages(max_seq) * KV_PAGE
            _lib.check(self.lib.fl_cache_create_pool_kv(model.h, max_batch, max_seq, tokens, self.KV_DTYPES[kv_dtype], C.byref(h)))
        elif pool_tokens is None:
            _lib.check(self.lib.fl_cache_create(model.h, max_batch, max_seq, C.byref(h)))
        else:
            _lib.check(self.lib.fl_cache_create_pool(model.h, max_batch, max_seq, pool_tokens, C.byref(h)))
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

    def forward_logprobs(self, ids: np.ndarray, targets: np.ndarray, rope_offset: int):
        """fl_forward_logprobs: ONE forward over ids [b, t] that feeds the cache like forward() and scores every position against
        targets [b, t].  -> (log_softmax(logits)[target] f32 [b, t], arg-max u32 [b, t] with forward_greedy's tie rule)."""
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        if ids.ndim != 2:
            raise FastllmError(-1, f"input must be [batch, seq], got shape {ids.shape}")
        targets = np.ascontiguousarray(targets, dtype=np.uint32)
        if targets.shape != ids.shape:
            raise FastllmError(-1, f"targets must have the shape of ids {ids.shape}, got {targets.shape}")
        b, t = ids.shape
        lp = np.empty((b, t), dtype=np.float32)
        am = np.empty((b, t), dtype=np.uint32)
        _lib.check(self.lib.fl_forward_logprobs(self.model.h, self.h, ids.ctypes.data_as(C.c_void_p), targets.ctypes.data_as(C.c_void_p),
                                                b, t, rope_offset, lp.ctypes.data_as(C.c_void_p), am.ctypes.data_as(C.c_void_p)))
        return lp, am

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

    def forward_packed(self, slots, seqs, rope_offsets) -> np.ndarray:
        """Packed forward (fl_forward_packed): sequence i (a 1-D id array of any length >= 1) is fed to cache slot slots[i] at RoPE
        positions rope_offsets[i] + j, all in ONE forward -- new prompts and decode steps of running requests side by side.
        -> f32 [n, vocab], row i = the last position of sequence i."""
        parts = [np.asarray(s, dtype=np.uint32).reshape(-1) for s in seqs]
        n = len(parts)
        sl = np.ascontiguousarray(slots, dtype=np.int32).reshape(-1)
        ro = np.ascontiguousarray(rope_offsets, dtype=np.uint64).reshape(-1)
        if sl.size != n or ro.size != n:
            raise FastllmError(-1, "slots / rope_offsets must have one entry per sequence")
        ids = np.ascontiguousarray(np.concatenate(parts) if n else np.zeros(0, np.uint32), dtype=np.uint32)
        lengths = np.array([p.size for p in parts], dtype=np.int32)
        out = np.empty((n, self.vocab), dtype=np.float32)
        _lib.check(self.lib.fl_forward_packed(self.model.h, self.h, sl.ctypes.data_as(C.c_void_p), lengths.ctypes.data_as(C.c_void_p), n,
                                              ids.ctypes.data_as(C.c_void_p), ro.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)))
        return out

    def slot_reset(self, slot: int):
        _lib.check(self.lib.fl_cache_slot_reset(self.h, slot))

    def slot_len(self, slot: int) -> int:
        n = C.c_int()
        _lib.check(self.lib.fl_cache_slot_len(self.h, slot, C.byref(n)))
        return n.value

    def slot_fork(self, src: int, dst: int):
        """fl_cache_slot_fork: the empty slot dst continues from src's cached tokens (full pages shared, the partial one copied)."""
        _lib.check(self.lib.fl_cache_slot_fork(self.h, src, dst))

    def pool_pages(self):
        """-> (free pages, total pages) of the KV pool."""
        f, t = C.c_int(), C.c_int()
        _lib.check(self.lib.fl_cache_pool_pages(self.h, C.byref(f), C.byref(t)))
        return f.value, t.value

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
        self._score: DeviceCache | None = None

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
        dev.load(tensors, random_seed, std)
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

    def logprobs(self, ids: np.ndarray, targets: np.ndarray):
        """Scores ids [b, t] against targets [b, t] in one forward from an empty sequence at RoPE offset 0, for every family alike.
        -> (log-probs f32 [b, t], arg-max u32 [b, t]).  Runs on a cache of its own, reset before and after each call, so the
        generate caches (LlamaCache.inner, the Mistral/Qwen2 model-internal KV) are never touched."""
        ids = np.asarray(ids)
        b = ids.shape[0] if ids.ndim == 2 else 1
        if self._score is None or self._score.max_batch < b:
            self._score = DeviceCache(self.dev, max(self.MAX_BATCH, b), self._capacity())
        self._score.reset()
        try:
            return self._score.forward_logprobs(ids, targets, 0)
        finally:
            self._score.reset()


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

    def loglikelihood(self, context_ids, continuation_ids):
        """The `loglikelihood(context, continuation)` request of evaluation harnesses: ONE scoring call over context + continuation
        (targets = the ids shifted left by one).  -> (sum of the continuation's log-probs, whether every continuation token is the
        arg-max at its position).  Summed in f64 in position order, as host/fastllm_host.hpp does."""
        ctx = np.asarray(context_ids, dtype=np.uint32).reshape(-1)
        cont = np.asarray(continuation_ids, dtype=np.uint32).reshape(-1)
        if ctx.size == 0 or cont.size == 0:
            raise ValueError("loglikelihood needs a non-empty context and continuation")
        ids = np.concatenate([ctx, cont])
        targets = np.concatenate([ids[1:], np.zeros(1, dtype=np.uint32)])   # the last position predicts nothing asked for
        lp, am = self.model.logprobs(ids[None], targets[None])
        pos = range(ctx.size - 1, ids.size - 1)                               # position j predicts ids[j + 1]
        total = 0.0
        for j in pos:
            total += float(lp[0, j])
        return total, all(int(am[0, j]) == int(ids[j + 1]) for j in pos)

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


KV_PAGE = 64        # tokens per KV page


def _pages(tokens: int) -> int:
    return -(-tokens // KV_PAGE)


class PackedBatcher:
    """Continuous batching above fl_forward_packed: every step is ONE forward that carries the next token of every running request
    AND the prompts of newly admitted ones, so admitting a prompt neither costs a forward of its own nor stalls the running
    requests.  A waiting request is admitted into a free slot while the step's tokens (one per running request plus the prompts
    admitted so far) stay within `token_budget`; when a slot is free at least one prompt is admitted, even one longer than the
    budget.  Per request the arithmetic is that of Model.generate, as in ContinuousBatcher: its own LogitsProcessor seeded 0, EOS
    break before emitting, and the adapter's position rule (Llama: the caller's position; Mistral / Qwen2: +1 per call).
    `cache` needs forward_packed(slots, seqs, rope_offsets) -> [n, V] and slot_reset(slot) (and slot_fork(src, dst) for a shared
    prefix): a DeviceCache, or a stand-in in tests.

    pool_tokens: the slots share a KV pool of that many tokens instead of max_seq each.  A waiting request is then also admitted only
    if the pages it can ever need -- its prompt plus max_tokens, less the prefix pages it shares -- fit the pool minus the pages
    reserved for running requests (and the shared prefix), so no call can run out of pages and nothing is preempted.  Requests are
    admitted in order: one that does not fit waits for pages to free up.

    kv_dtype: element type of the cache the batcher builds ("bf16" or "fp8_e4m3"; DeviceCache)."""

    def __init__(self, model, max_batch: int = 8, eos_token_id: int | None = 2, cache=None, token_budget: int = 4096,
                 pool_tokens: int | None = None, kv_dtype: str = "bf16"):
        self.model, self.max_batch, self.eos_token_id, self.token_budget = model, max_batch, eos_token_id, token_budget
        self.position_per_call = getattr(model, "arch", "llama") != "llama"      # the Mistral/Qwen2 adapters' offset rule
        self.sliding_window = getattr(getattr(model, "cfg", None), "sliding_window", 0) if self.position_per_call else 0
        self.cache = cache if cache is not None else DeviceCache(model.dev, max_batch, model._capacity(), pool_tokens, kv_dtype)
        self.pool_pages = None if pool_tokens is None else _pages(pool_tokens)
        self.slot_pages = _pages(self.cache.max_seq) if hasattr(self.cache, "max_seq") else None   # a slot never holds more
        self.forwards = 0       # packed forwards issued (tests / stats)
        self.prefill_tokens = 0  # prompt tokens fed (tests / stats): a shared prefix counts once
        self.peak_pages = 0      # most pages reserved at once (with pool_tokens)

    def _uses_prefix(self, prompt, prefix) -> bool:
        """A request continues from the shared prefix's slot when its prompt extends the prefix and splitting the prompt there
        computes what the one-call prompt does: not on Llama (a multi-token call on a non-empty sequence is refused there), and not
        for a prompt longer than the sliding window (the window of a multi-token call applies to an empty sequence only)."""
        return (prefix is not None and self.position_per_call and len(prompt) > len(prefix) and list(prompt[:len(prefix)]) == prefix
                and not (self.sliding_window and len(prompt) > self.sliding_window))

    def generate(self, prompts, max_tokens: int, temperature: float = 0.0, shared_prefix=None):
        """-> one id list per prompt, in request order.  shared_prefix: token ids that many prompts start with; it is fed once into a
        slot held for the call, and each request that extends it starts as a fork of that slot, fed only the rest of its prompt at
        RoPE offset len(shared_prefix) (the positions of the one-call prompt).  Other requests take the normal path."""
        out = [[] for _ in prompts]
        if max_tokens <= 0:
            return out
        prompts = [[int(x) for x in np.asarray(p).reshape(-1)] for p in prompts]
        prefix = None if shared_prefix is None else [int(x) for x in np.asarray(shared_prefix).reshape(-1)]
        if not prefix or self.max_batch < 2:
            prefix = None       # nothing to share, or no slot left for requests beside the prefix's
        forked = [self._uses_prefix(p, prefix) for p in prompts]
        waiting = list(range(len(prompts)))[::-1]
        free = list(range(self.max_batch))[::-1]
        running = {}            # slot -> [request, next RoPE position, LogitsProcessor, token to feed, pages reserved]
        reserved = 0            # pages the admission rule holds for running requests and the prefix

        def need(req):
            n = _pages(len(prompts[req]) + max_tokens)
            if self.slot_pages is not None:
                n = min(n, self.slot_pages)
            return n - (len(prefix) // KV_PAGE if forked[req] else 0)

        pslot = None
        if any(forked):
            pslot = free.pop()
            reserved = _pages(len(prefix))
            self.cache.forward_packed([pslot], [prefix], [0])
            self.forwards += 1
            self.prefill_tokens += len(prefix)
        try:
            while waiting or running:
                slots = sorted(running)
                seqs = [[running[s][3]] for s in slots]
                ropes = [running[s][1] for s in slots]
                budget = self.token_budget - len(slots)
                admitted = 0
                while waiting and free:
                    req = waiting[-1]
                    seq = prompts[req][len(prefix):] if forked[req] else prompts[req]
                    if admitted and len(seq) > budget:
                        break
                    if self.pool_pages is not None and reserved + need(req) > self.pool_pages:
                        if not running and not admitted:
                            raise ValueError(f"request {req} needs {need(req)} KV pages; the pool holds {self.pool_pages - reserved}")
                        break
                    waiting.pop()
                    slot = free.pop()
                    if forked[req]:
                        self.cache.slot_fork(pslot, slot)
                    slots.append(slot)
                    seqs.append(seq)
                    ropes.append(len(prefix) if forked[req] else 0)
                    budget -= len(seq)
                    admitted += 1
                    self.prefill_tokens += len(seq)
                    pages = need(req) if self.pool_pages is not None else 0
                    reserved += pages
                    running[slot] = [req, 0, LogitsProcessor(0, float(np.float32(temperature))), 0, pages]
                self.peak_pages = max(self.peak_pages, reserved)
                logits = np.asarray(self.cache.forward_packed(slots, seqs, ropes))
                self.forwards += 1
                for i, s in enumerate(slots):
                    st = running[s]
                    # a prompt starts at 0; a decode row feeds one token.  A forked request's suffix is the rest of its prompt: the
                    # Mistral/Qwen2 rule then continues from 1, as after the one-call prompt.
                    st[1] += 1 if self.position_per_call else len(seqs[i])
                    tok = st[2].sample(logits[i].reshape(-1))
                    if self.eos_token_id is not None and tok == self.eos_token_id:
                        done = True
                    else:
                        out[st[0]].append(tok)
                        st[3] = tok
                        done = len(out[st[0]]) >= max_tokens
                    if done:
                        running.pop(s)
                        reserved -= st[4]
                        self.cache.slot_reset(s)
                        free.append(s)
        finally:
            if pslot is not None:
                self.cache.slot_reset(pslot)
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
        self.dev.load(tensors, random_seed, std, np.float32)

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
