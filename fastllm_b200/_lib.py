"""ctypes binding of the C ABI in include/fastllm_b200.h.

This is the Python twin of the cgo/FFI stub a maintainer of the reference would add (INTEGRATION.md shows the Rust
one).  There is no fallback: if libfastllm_b200.so is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libfastllm_b200.so")

FL_ARCH = {"llama": 0, "mistral": 1, "qwen2": 2, "mixtral": 3, "bert": 4}
FL_DTYPE_F32, FL_DTYPE_BF16, FL_DTYPE_F16 = 0, 1, 2


class FlConfig(C.Structure):
    _fields_ = [("arch", C.c_int32), ("hidden_size", C.c_int32), ("intermediate_size", C.c_int32),
                ("vocab_size", C.c_int32), ("num_hidden_layers", C.c_int32), ("num_attention_heads", C.c_int32),
                ("num_key_value_heads", C.c_int32), ("max_position_embeddings", C.c_int32),
                ("sliding_window", C.c_int32), ("qkv_bias", C.c_int32), ("num_local_experts", C.c_int32),
                ("num_experts_per_tok", C.c_int32), ("norm_eps", C.c_float), ("rope_theta", C.c_double),
                ("tp_rank", C.c_int32), ("tp_size", C.c_int32), ("ep_dp_attention", C.c_int32), ("reserved", C.c_int32 * 5)]


class FastllmError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"fastllm_b200 error {code}: {msg}")
        self.code = code


# every symbol include/fastllm_b200.h declares: name -> (restype, argtypes)
_VP, _I, _U64, _SZ = C.c_void_p, C.c_int, C.c_uint64, C.c_size_t
SYMBOLS = {
    "fl_init": (_I, [_I]),
    "fl_last_error": (C.c_char_p, []),
    "fl_version": (_I, []),
    "fl_device_synchronize": (_I, []),
    "fl_model_create": (_I, [C.POINTER(FlConfig), C.POINTER(_VP)]),
    "fl_model_put_tensor": (_I, [_VP, C.c_char_p, _I, C.POINTER(C.c_int64), _I, _VP]),
    "fl_model_random_init": (_I, [_VP, _U64, C.c_float]),
    "fl_model_finalize": (_I, [_VP]),
    "fl_model_clone": (_I, [_VP, C.POINTER(_VP)]),
    "fl_model_destroy": (_I, [_VP]),
    "fl_model_weight_bytes": (_I, [_VP, C.POINTER(_U64)]),
    "fl_cache_create": (_I, [_VP, _I, _I, C.POINTER(_VP)]),
    "fl_cache_create_pool": (_I, [_VP, _I, _I, _I, C.POINTER(_VP)]),
    "fl_cache_create_pool_kv": (_I, [_VP, _I, _I, _I, _I, C.POINTER(_VP)]),
    "fl_cache_pool_pages": (_I, [_VP, C.POINTER(_I), C.POINTER(_I)]),
    "fl_cache_slot_fork": (_I, [_VP, _I, _I]),
    "fl_cache_reset": (_I, [_VP]),
    "fl_cache_kv_len": (_I, [_VP, C.POINTER(_I)]),
    "fl_cache_fill_synthetic": (_I, [_VP, _I, _I, _U64]),
    "fl_cache_destroy": (_I, [_VP]),
    "fl_forward": (_I, [_VP, _VP, _VP, _I, _I, _SZ, _VP]),
    "fl_forward_greedy": (_I, [_VP, _VP, _VP, _I, _I, _SZ, _VP]),
    "fl_decode_greedy_loop": (_I, [_VP, _VP, _VP, _I, _SZ, _I, _VP, C.POINTER(C.c_float)]),
    "fl_forward_logprobs": (_I, [_VP, _VP, _VP, _VP, _I, _I, _SZ, _VP, _VP]),
    "fl_sampler_create": (_I, [_U64, C.c_double, C.POINTER(_VP)]),
    "fl_sampler_sample": (_I, [_VP, _VP, _SZ, C.POINTER(C.c_uint32)]),
    "fl_argmax_rows": (_I, [_VP, _I, _SZ, _VP]),
    "fl_sampler_next_u32": (_I, [_VP, C.POINTER(C.c_uint32)]),
    "fl_sampler_destroy": (_I, [_VP]),
    "fl_forward_sample": (_I, [_VP, _VP, _VP, _I, _I, _SZ, _VP, C.POINTER(C.c_uint32)]),
    "fl_forward_slots": (_I, [_VP, _VP, _VP, _VP, _I, _I, _VP, _VP]),
    "fl_forward_packed": (_I, [_VP, _VP, _VP, _VP, _I, _VP, _VP, _VP]),
    "fl_cache_slot_reset": (_I, [_VP, _I]),
    "fl_cache_slot_len": (_I, [_VP, _I, C.POINTER(_I)]),
    "fl_cache_moe_routing": (_I, [_VP, _I, _VP, _VP]),
    "fl_forward_sample_device": (_I, [_VP, _VP, _VP, _I, _I, _SZ, _VP, C.POINTER(C.c_uint32)]),
    "fl_embed": (_I, [_VP, _VP, _VP, _I, _I, _VP]),
    "fl_embed_packed": (_I, [_VP, _VP, _VP, _I, _VP]),
    "fl_embed_timed": (_I, [_VP, _VP, _VP, _I, _I, _VP, _I, C.POINTER(C.c_float)]),
    "fl_comm_unique_id": (_I, [_VP]),
    "fl_comm_init": (_I, [_I, _I, _VP]),
    "fl_comm_ipc_export": (_I, [_VP]),
    "fl_comm_ipc_import": (_I, [_VP, _I, _I]),
    "fl_comm_destroy": (_I, []),
    "fl_prof_begin": (_I, []),
    "fl_prof_end": (_I, [C.c_char_p, _SZ]),
    "fl_launch_count": (_I, [C.POINTER(_U64)]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library and bind every declared symbol.  Raises if the library is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FastllmError(-3, f"{LIB_PATH} is not built; run `python -c 'import __graft_entry__ as g; g.build()'` "
                                   "(there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(rc: int):
    if rc != 0:
        raise FastllmError(rc, load().fl_last_error().decode("utf-8", "replace"))


_initialised = None


def init(device: int = 0):
    global _initialised
    if _initialised != device:
        check(load().fl_init(device))
        _initialised = device
