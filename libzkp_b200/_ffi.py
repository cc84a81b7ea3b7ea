"""ctypes binding of libzkp_b200/_lib/liblzkp_b200.so — the C ABI declared in include/lzkp_b200.h.

This is the same set of symbols a Rust ``extern "C"`` crate inside libzkp would bind
(INTEGRATION.md).  There is no fallback: if the library has not been built, importing a
computing entry point raises, and every call fails with LZKP_E_NO_DEVICE without a GPU.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LZKP_B200_LIB selects another build of the same library (kernel A/B runs); there is still no fallback.
LIB_PATH = os.environ.get("LZKP_B200_LIB") or os.path.join(_HERE, "_lib", "liblzkp_b200.so")

LZKP_OK = 0
LZKP_E_INVALID = -1
LZKP_E_NO_DEVICE = -2
LZKP_E_CUDA = -3
LZKP_E_STATE = -4
LZKP_E_NOMEM = -5
LZKP_E_UNSUPPORTED = -6
LZKP_CIRCUIT_EQUALITY = 0
LZKP_CIRCUIT_MEMBERSHIP = 1
LZKP_PARTIAL_BYTES = 768


class PkOptions(C.Structure):
    _fields_ = [("window_bits", C.c_int), ("table_budget_bytes", C.c_uint64), ("max_chunk", C.c_uint32),
                ("shard_index", C.c_uint32), ("shard_count", C.c_uint32)]


# name -> (restype, argtypes); kept in one table so tests can check it against the header.
_vp, _sz, _int = C.c_void_p, C.c_size_t, C.c_int
_u32, _u64 = C.c_uint32, C.c_uint64
SIGNATURES = {
    "lzkp_init": (_int, [_vp, _int]),
    "lzkp_device_count": (_int, []),
    "lzkp_shutdown": (_int, []),
    "lzkp_last_error": (C.c_char_p, []),
    "lzkp_kernel_launches": (_u64, []),
    "lzkp_profile_enable": (_int, [_int]),
    "lzkp_profile_read": (_int, [_vp, C.POINTER(C.c_double), C.POINTER(_u64), _int]),
    "lzkp_pk_load": (_int, [_vp, _sz, _int, C.POINTER(_vp)]),
    "lzkp_pk_load_ex": (_int, [_vp, _sz, _int, C.POINTER(PkOptions), C.POINTER(_vp)]),
    "lzkp_pk_free": (None, [_vp]),
    "lzkp_pk_info": (_int, [_vp, C.POINTER(_u64)]),
    "lzkp_pk_work": (_int, [_vp, C.POINTER(_u64)]),
    "lzkp_pk_shard_info": (_int, [_vp, C.POINTER(_u32), C.POINTER(_u32), C.POINTER(_u32)]),
    "lzkp_circuit_load": (_int, [_vp, _u32, _u32, _u32] + [_vp] * 9),
    "lzkp_circuit_builtin": (_int, [_vp, _int, _u32]),
    "lzkp_builtin_circuit_csr": (_int, [_int, _u32, C.POINTER(_u64), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "lzkp_key_sizes": (_int, [_u32, _u32, _u32, C.POINTER(_sz), C.POINTER(_sz)]),
    "lzkp_setup": (_int, [_u32, _u32, _u32] + [_vp] * 9 + [_vp, _vp, _sz, _vp, _sz]),
    "lzkp_setup_builtin": (_int, [_int, _u32, _vp, _vp, _sz, _vp, _sz]),
    "lzkp_generator_mul": (_int, [_int, _vp, _sz, _vp]),
    "lzkp_prove_batch": (_int, [_vp, _sz, _vp, _vp, _vp, _vp, _vp]),
    "lzkp_prove_batch_device": (_int, [_vp, _sz, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lzkp_builtin_witness": (_int, [_int, _u32, _u64, _u64, _vp, _u32, _vp, _vp, _sz]),
    "lzkp_prove_equality_batch": (_int, [_vp, _sz, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lzkp_prove_membership_batch": (_int, [_vp, _sz, _vp, _vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lzkp_prove_equality_enveloped": (_int, [_vp, _sz, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lzkp_prove_membership_enveloped": (_int, [_vp, _sz, _vp, _vp, _vp, _u32, _vp, _vp, _vp, _u32, _vp, _vp]),
    "lzkp_prove_equality_batch_device": (_int, [_vp, _sz, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lzkp_witness_map": (_int, [_vp, _sz, _vp, _vp]),
    "lzkp_witness_map_device": (_int, [_vp, _vp, _vp, _vp]),
    "lzkp_prove_partial_device": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int]),
    "lzkp_prove_combine_device": (_int, [_vp, _vp, _int, _vp, _vp, _vp, _vp]),
    "lzkp_msm_g1": (_int, [_vp, _vp, _sz, _vp]),
    "lzkp_msm_g2": (_int, [_vp, _vp, _sz, _vp]),
    "lzkp_bases_load": (_int, [_int, _vp, _sz, _int, _int, _int, C.POINTER(_vp)]),
    "lzkp_bases_free": (None, [_vp]),
    "lzkp_msm": (_int, [_vp, _vp, _sz, _vp]),
    "lzkp_msm_device": (_int, [_vp, _vp, _sz, _vp, _vp]),
    "lzkp_ntt": (_int, [_vp, _u32, _int, _int]),
    "lzkp_ntt_device": (_int, [_vp, _vp, _u32, _int, _int, _vp]),
    "lzkp_vk_load": (_int, [_vp, _sz, C.POINTER(_vp)]),
    "lzkp_vk_free": (None, [_vp]),
    "lzkp_vk_info": (_int, [_vp, C.POINTER(_u64)]),
    "lzkp_verify_batch": (_int, [_vp, _sz, _vp, _vp, _sz, _vp]),
    "lzkp_verify_batch_device": (_int, [_vp, _sz, _vp, _vp, _sz, _vp, _vp]),
    "lzkp_commit_value_snark": (_int, [_u64, _vp]),
}

_lib = None


def lib():
    """Load the engine library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(the engine has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def last_error() -> str:
    return (lib().lzkp_last_error() or b"").decode("utf-8", "replace")


def check(rc: int) -> None:
    if rc != LZKP_OK:
        from .errors import EngineError
        raise EngineError(rc, last_error())
