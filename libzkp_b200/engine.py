"""Thin numpy-level wrappers over the C ABI (include/lzkp_b200.h).

Byte formats are ark-serialize's (SURVEY.md §8b): field elements 32 B canonical little-endian,
G1 affine 64 B, G2 affine 128 B, proofs 256 B.  Arrays are ``uint8`` with a trailing byte axis.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np

from . import _ffi
from ._ffi import check, lib

EQUALITY = _ffi.LZKP_CIRCUIT_EQUALITY
MEMBERSHIP = _ffi.LZKP_CIRCUIT_MEMBERSHIP


def _p(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _u8(a, shape_tail: int) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if a.size % shape_tail:
        raise ValueError(f"byte array size {a.size} is not a multiple of {shape_tail}")
    return a.reshape(-1, shape_tail)


def init(device=None) -> None:
    """lzkp_init: bind this process to one CUDA device (one process per GPU), or - given a sequence of device
    indices - to several: proving keys loaded afterwards are replicated on each, and one host-buffer batch call
    fans out over all of them (the reference's batch path is one process, src/advanced/batch.rs:110-140)."""
    if device is None:
        check(lib().lzkp_init(None, 0))
    else:
        devs = [int(device)] if isinstance(device, (int, np.integer)) else [int(d) for d in device]
        arr = (C.c_int * len(devs))(*devs)
        check(lib().lzkp_init(arr, len(devs)))


def device_count() -> int:
    return int(lib().lzkp_device_count())


def profile_enable(on: bool) -> None:
    check(lib().lzkp_profile_enable(int(on)))


def kernel_launches() -> int:
    return int(lib().lzkp_kernel_launches())


def commit_value_snark(value: int) -> bytes:
    """commit_value_snark (src/utils/commitment.rs:14-16): 32 B LE MiMC-5 commitment of a u64."""
    out = (C.c_uint8 * 32)()
    check(lib().lzkp_commit_value_snark(C.c_uint64(int(value) & (2**64 - 1)), out))
    return bytes(out)


def builtin_circuit_csr(kind: int, param: int):
    """Shape and CSR matrices of a builtin circuit: (m, n_inst, n_wit), [(rowptr, col, val)] * 3."""
    shape = (C.c_uint64 * 6)()
    check(lib().lzkp_builtin_circuit_csr(kind, param, shape, None, None, None))
    m, n_inst, n_wit = int(shape[0]), int(shape[1]), int(shape[2])
    mats = [(np.zeros(m + 1, np.uint32), np.zeros(int(shape[3 + k]), np.uint32),
             np.zeros((int(shape[3 + k]), 32), np.uint8)) for k in range(3)]
    rp = (C.c_void_p * 3)(*[m_[0].ctypes.data for m_ in mats])
    cl = (C.c_void_p * 3)(*[m_[1].ctypes.data for m_ in mats])
    vl = (C.c_void_p * 3)(*[m_[2].ctypes.data for m_ in mats])
    check(lib().lzkp_builtin_circuit_csr(kind, param, shape, rp, cl, vl))
    return (m, n_inst, n_wit), mats


def key_sizes(m: int, n_inst: int, n_wit: int) -> Tuple[int, int]:
    pl, vl = C.c_size_t(), C.c_size_t()
    check(lib().lzkp_key_sizes(m, n_inst, n_wit, C.byref(pl), C.byref(vl)))
    return int(pl.value), int(vl.value)


def _toxic(toxic: Sequence[int]) -> np.ndarray:
    if len(toxic) != 5:
        raise ValueError("toxic waste = (alpha, beta, gamma, delta, tau)")
    return np.frombuffer(b"".join(int(t).to_bytes(32, "little") for t in toxic), np.uint8).copy()


def setup_builtin(kind: int, param: int, toxic: Sequence[int]) -> Tuple[bytes, bytes]:
    """circuit_specific_setup for a builtin circuit on the device -> (pk_bytes, vk_bytes), ark layout."""
    (m, n_inst, n_wit), _ = builtin_circuit_csr(kind, param)
    pl, vl = key_sizes(m, n_inst, n_wit)
    pk, vk, tx = np.zeros(pl, np.uint8), np.zeros(vl, np.uint8), _toxic(toxic)
    check(lib().lzkp_setup_builtin(kind, param, _p(tx), _p(pk), pl, _p(vk), vl))
    return pk.tobytes(), vk.tobytes()


def setup(m: int, n_inst: int, n_wit: int, mats, toxic: Sequence[int]) -> Tuple[bytes, bytes]:
    pl, vl = key_sizes(m, n_inst, n_wit)
    pk, vk, tx = np.zeros(pl, np.uint8), np.zeros(vl, np.uint8), _toxic(toxic)
    flat, keep = [], []
    for rowptr, col, val in mats:
        arrs = [np.ascontiguousarray(rowptr, np.uint32), np.ascontiguousarray(col, np.uint32),
                np.ascontiguousarray(val, np.uint8)]
        keep += arrs
        flat += [_p(a) for a in arrs]
    check(lib().lzkp_setup(m, n_inst, n_wit, *flat, _p(tx), _p(pk), pl, _p(vk), vl))
    return pk.tobytes(), vk.tobytes()


def builtin_witness(kind: int, param: int, value: int, other: int = 0, set_: Optional[Sequence[int]] = None,
                    commitment: Optional[bytes] = None) -> np.ndarray:
    """Full assignment z (n_vars x 32 B canonical) of a builtin circuit (lzkp_builtin_witness, host arithmetic)."""
    (_, n_inst, n_wit), _ = (builtin_circuit_shape(kind, param), None)
    z = np.zeros((n_inst + n_wit, 32), np.uint8)
    sa = None if set_ is None else np.asarray(list(set_), np.uint64)
    cm = None if commitment is None else np.frombuffer(commitment, np.uint8).copy()
    check(lib().lzkp_builtin_witness(kind, param, int(value), int(other), _p(sa), 0 if sa is None else len(sa), _p(cm),
                                     _p(z), z.size))
    return z


def builtin_circuit_shape(kind: int, param: int) -> Tuple[int, int, int]:
    shape = (C.c_uint64 * 6)()
    check(lib().lzkp_builtin_circuit_csr(kind, param, shape, None, None, None))
    return int(shape[0]), int(shape[1]), int(shape[2])


class ProvingKey:
    """A proving key resident in HBM (lzkp_pk): the object the reference keeps in its OnceLock
    (src/backend/snark.rs:295-339), plus the circuit's R1CS matrices and NTT tables."""

    def __init__(self, pk_bytes: bytes, validate: bool = False, window_bits: int = 0,
                 table_budget_bytes: int = 0, max_chunk: int = 0, shard_index: int = 0, shard_count: int = 0):
        self._h = C.c_void_p()
        buf = np.frombuffer(pk_bytes, dtype=np.uint8)
        opt = _ffi.PkOptions(window_bits, table_budget_bytes, max_chunk, shard_index, shard_count)
        check(lib().lzkp_pk_load_ex(_p(buf), len(pk_bytes), int(validate), C.byref(opt), C.byref(self._h)))
        info = (C.c_uint64 * 8)()
        check(lib().lzkp_pk_info(self._h, info))
        (self.n_vars, self.n_inst, self.n_wit, self.n, self.window_bits, self.windows, self.table_bytes,
         self.max_chunk) = [int(x) for x in info]

    def work(self):
        """(G1 units, G2 units, G1 table rows, G2 table rows): mixed additions per proof on the batched path."""
        w = (C.c_uint64 * 4)()
        check(lib().lzkp_pk_work(self._h, w))
        return tuple(int(x) for x in w)

    def shard_info(self):
        """(first[5], count[5], map_ranks): this shard's point ranges of a, b1, l, h, b2 (large-domain keys)."""
        first, count, k = (C.c_uint32 * 5)(), (C.c_uint32 * 5)(), C.c_uint32()
        check(lib().lzkp_pk_shard_info(self._h, first, count, C.byref(k)))
        return list(first), list(count), int(k.value)

    def close(self):
        if self._h:
            lib().lzkp_pk_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    REGIONS = ("witgen", "witness_map", "digits", "msm_g1", "msm_g2", "assemble")

    def profile_read(self, reset: bool = True):
        """Accumulated device milliseconds / bracket counts per pipeline stage (lzkp_profile_read)."""
        ms, cnt = (C.c_double * 8)(), (C.c_uint64 * 8)()
        check(lib().lzkp_profile_read(self._h, ms, cnt, int(reset)))
        return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(self.REGIONS)}

    # ---- circuit binding
    def circuit_builtin(self, kind: int, param: int) -> "ProvingKey":
        check(lib().lzkp_circuit_builtin(self._h, kind, param))
        return self

    def circuit_load(self, m: int, n_inst: int, n_wit: int, mats) -> "ProvingKey":
        flat = []
        keep = []
        for rowptr, col, val in mats:
            rowptr = np.ascontiguousarray(rowptr, np.uint32)
            col = np.ascontiguousarray(col, np.uint32)
            val = np.ascontiguousarray(val, np.uint8)
            keep += [rowptr, col, val]
            flat += [_p(rowptr), _p(col), _p(val)]
        check(lib().lzkp_circuit_load(self._h, m, n_inst, n_wit, *flat))
        return self

    # ---- proving
    def prove_batch(self, z, r, s) -> Tuple[np.ndarray, np.ndarray]:
        z = _u8(z, 32 * self.n_vars)
        n = z.shape[0]
        r, s = _u8(r, 32), _u8(s, 32)
        if r.shape[0] != n or s.shape[0] != n:
            raise ValueError("r, s must hold one scalar per proof")
        proofs = np.zeros((n, 256), np.uint8)
        status = np.zeros(n, np.int32)
        check(lib().lzkp_prove_batch(self._h, n, _p(z), _p(r), _p(s), _p(proofs), _p(status)))
        return proofs, status

    def prove_batch_device(self, n: int, d_z: int, d_r: int, d_s: int, d_proofs: int, d_status: int,
                           stream: int = 0) -> None:
        """lzkp_prove_batch_device: all arguments are device pointers (ints); asynchronous on `stream`."""
        check(lib().lzkp_prove_batch_device(self._h, n, d_z, d_r, d_s, d_proofs, d_status, stream))

    # ---- single large proof split across GPUs (device pointers, asynchronous on `stream`)
    def witness_map_device(self, d_z: int, d_h: int, stream: int = 0) -> None:
        check(lib().lzkp_witness_map_device(self._h, d_z, d_h, stream))

    def prove_partial_device(self, d_z: int, d_r: int, d_s: int, d_h: int, d_partial: int, d_status: int,
                             stream: int = 0, phase: int = 3) -> None:
        check(lib().lzkp_prove_partial_device(self._h, d_z, d_r, d_s, d_h, d_partial, d_status, stream, phase))

    def prove_combine_device(self, d_partials: int, n_partials: int, d_r: int, d_s: int, d_proof: int,
                             stream: int = 0) -> None:
        check(lib().lzkp_prove_combine_device(self._h, d_partials, n_partials, d_r, d_s, d_proof, stream))

    def prove_equality_batch(self, a, b, r, s, commitments=None, out=None):
        """out = (proofs[n, 256] uint8, commitments[n, 32] uint8, status[n] int32) reuses caller-owned result buffers
        (a server proving batch after batch keeps them, e.g. pinned); by default fresh arrays are returned."""
        a = np.ascontiguousarray(a, np.uint64)
        b = np.ascontiguousarray(b, np.uint64)
        n = a.shape[0]
        r, s = _u8(r, 32), _u8(s, 32)
        cm = None if commitments is None else _u8(commitments, 32)
        if out is not None:
            proofs, cm_out, status = out
            if (proofs.shape, cm_out.shape, status.shape) != ((n, 256), (n, 32), (n,)) or proofs.dtype != np.uint8 \
                    or cm_out.dtype != np.uint8 or status.dtype != np.int32 or not (proofs.flags.c_contiguous and cm_out.flags.c_contiguous):
                raise ValueError("out buffers must be C-contiguous (n, 256) uint8, (n, 32) uint8, (n,) int32")
        else:
            proofs = np.zeros((n, 256), np.uint8)
            cm_out = np.zeros((n, 32), np.uint8)
            status = np.zeros(n, np.int32)
        check(lib().lzkp_prove_equality_batch(self._h, n, _p(a), _p(b), _p(cm), _p(r), _p(s), _p(proofs), _p(cm_out),
                                              _p(status)))
        return proofs, cm_out, status

    def prove_equality_enveloped(self, a, b, r, s):
        """n x prove_equality's final bytes (298 B envelopes built on the device) -> (envelopes[n, 298], lengths, status)."""
        a = np.ascontiguousarray(a, np.uint64)
        b = np.ascontiguousarray(b, np.uint64)
        n = a.shape[0]
        r, s = _u8(r, 32), _u8(s, 32)
        env = np.zeros((n, 298), np.uint8)
        lens = np.zeros(n, np.uint32)
        status = np.zeros(n, np.int32)
        check(lib().lzkp_prove_equality_enveloped(self._h, n, _p(a), _p(b), _p(r), _p(s), _p(env), _p(lens), _p(status)))
        return env, lens, status

    def prove_membership_enveloped(self, value, sets, set_len, r, s):
        value = np.ascontiguousarray(value, np.uint64)
        sets = np.ascontiguousarray(sets, np.uint64)
        set_len = np.ascontiguousarray(set_len, np.uint32)
        n, stride = value.shape[0], sets.shape[1]
        r, s = _u8(r, 32), _u8(s, 32)
        row = 302 + 8 * stride
        env = np.zeros((n, row), np.uint8)
        lens = np.zeros(n, np.uint32)
        status = np.zeros(n, np.int32)
        check(lib().lzkp_prove_membership_enveloped(self._h, n, _p(value), _p(sets), _p(set_len), stride, _p(r), _p(s),
                                                    _p(env), row, _p(lens), _p(status)))
        return env, lens, status

    def prove_membership_batch(self, value, sets, set_len, r, s, commitments=None):
        value = np.ascontiguousarray(value, np.uint64)
        sets = np.ascontiguousarray(sets, np.uint64)
        set_len = np.ascontiguousarray(set_len, np.uint32)
        n = value.shape[0]
        stride = sets.shape[1] if sets.ndim == 2 else 0
        r, s = _u8(r, 32), _u8(s, 32)
        cm = None if commitments is None else _u8(commitments, 32)
        proofs = np.zeros((n, 256), np.uint8)
        cm_out = np.zeros((n, 32), np.uint8)
        status = np.zeros(n, np.int32)
        check(lib().lzkp_prove_membership_batch(self._h, n, _p(value), _p(sets), _p(set_len), stride, _p(cm), _p(r),
                                                _p(s), _p(proofs), _p(cm_out), _p(status)))
        return proofs, cm_out, status

    def prove_equality_batch_device(self, n: int, d_a: int, d_b: int, d_r: int, d_s: int, d_proofs: int,
                                    d_status: int, stream: int = 0) -> None:
        """All arguments are device pointers (ints); asynchronous on `stream`."""
        check(lib().lzkp_prove_equality_batch_device(self._h, n, d_a, d_b, d_r, d_s, d_proofs, d_status, stream))

    def witness_map(self, z) -> np.ndarray:
        z = _u8(z, 32 * self.n_vars)
        n = z.shape[0]
        h = np.zeros((n, self.n, 32), np.uint8)
        check(lib().lzkp_witness_map(self._h, n, _p(z), _p(h)))
        return h


def msm_g1(bases, scalars) -> bytes:
    bases, scalars = _u8(bases, 64), _u8(scalars, 32)
    n = min(bases.shape[0], scalars.shape[0])       # msm_bigint truncates to the shorter input
    out = np.zeros(64, np.uint8)
    check(lib().lzkp_msm_g1(_p(bases), _p(scalars), n, _p(out)))
    return out.tobytes()


def msm_g2(bases, scalars) -> bytes:
    bases, scalars = _u8(bases, 128), _u8(scalars, 32)
    n = min(bases.shape[0], scalars.shape[0])
    out = np.zeros(128, np.uint8)
    check(lib().lzkp_msm_g2(_p(bases), _p(scalars), n, _p(out)))
    return out.tobytes()


def ntt(data, inverse: bool = False, coset: bool = False) -> np.ndarray:
    a = _u8(data, 32).copy()
    n = a.shape[0]
    log_n = n.bit_length() - 1
    if n == 0 or (1 << log_n) != n:
        raise ValueError("NTT size must be a power of two")
    check(lib().lzkp_ntt(_p(a), log_n, int(inverse), int(coset)))
    return a


def ntt_device(d_in: int, d_out: int, log_n: int, inverse: bool = False, coset: bool = False, stream: int = 0) -> None:
    """lzkp_ntt_device on raw device pointers (asynchronous on `stream`); d_in is clobbered above 2^11."""
    check(lib().lzkp_ntt_device(d_in, d_out, log_n, int(inverse), int(coset), stream))


class MsmBases:
    """MSM bases resident in HBM (lzkp_bases): group 1 = G1, 2 = G2."""

    def __init__(self, group: int, bases, window_bits: int = 0, resident_windows: bool = True, validate: bool = False):
        self.group = group
        self.point_bytes = 64 if group == 1 else 128
        bases = _u8(bases, self.point_bytes)
        self.n = bases.shape[0]
        self._h = C.c_void_p()
        check(lib().lzkp_bases_load(group, _p(bases), self.n, window_bits, int(resident_windows), int(validate),
                                    C.byref(self._h)))

    def msm(self, scalars) -> bytes:
        scalars = _u8(scalars, 32)
        out = np.zeros(self.point_bytes, np.uint8)
        check(lib().lzkp_msm(self._h, _p(scalars), scalars.shape[0], _p(out)))
        return out.tobytes()

    def msm_device(self, d_scalars: int, n: int, d_out: int, stream: int = 0) -> None:
        check(lib().lzkp_msm_device(self._h, d_scalars, n, d_out, stream))

    def close(self):
        if self._h:
            lib().lzkp_bases_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def generator_mul(group: int, scalars) -> np.ndarray:
    """scalars[i] * G (standard generator of G1 / G2) as ark-serialize affine bytes."""
    scalars = _u8(scalars, 32)
    out = np.zeros((scalars.shape[0], 64 if group == 1 else 128), np.uint8)
    check(lib().lzkp_generator_mul(group, _p(scalars), scalars.shape[0], _p(out)))
    return out


class VerifyingKey:
    """A verifying key resident on the device with e(alpha, beta) precomputed (lzkp_vk)."""

    def __init__(self, vk_bytes: bytes):
        self._h = C.c_void_p()
        buf = np.frombuffer(vk_bytes, dtype=np.uint8)
        check(lib().lzkp_vk_load(_p(buf), len(vk_bytes), C.byref(self._h)))
        self.n_pub = (len(vk_bytes) - 456) // 64 - 1

    def verify_batch(self, proofs, public_inputs) -> np.ndarray:
        """proofs (n, 256) bytes; public_inputs (n, n_pub, 32) canonical bytes -> bool array."""
        proofs = _u8(proofs, 256)
        n = proofs.shape[0]
        x = np.ascontiguousarray(public_inputs, np.uint8).reshape(n, -1) if n else np.zeros((0, 0), np.uint8)
        n_pub = x.shape[1] // 32 if n else self.n_pub
        ok = np.zeros(n, np.uint8)
        check(lib().lzkp_verify_batch(self._h, n, _p(proofs), _p(x) if x.size else None, n_pub, _p(ok)))
        return ok.astype(bool)

    def verify_batch_device(self, n: int, d_proofs: int, d_inputs: int, n_pub: int, d_ok: int, stream: int = 0) -> None:
        """lzkp_verify_batch_device: proofs (n x 256 B), public inputs (n x n_pub x 32 B) and ok (n bytes) are device
        pointers (ints) on the key's device; asynchronous on `stream`.  Refused on a stream that is being captured."""
        check(lib().lzkp_verify_batch_device(self._h, n, d_proofs, d_inputs, n_pub, d_ok, stream))

    def info(self):
        """(n_pub, table bytes, latency form available, combined form available) of the loaded key."""
        v = (C.c_uint64 * 4)()
        check(lib().lzkp_vk_info(self._h, v))
        return int(v[0]), int(v[1]), bool(v[2]), bool(v[3])

    def close(self):
        if self._h:
            lib().lzkp_vk_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
