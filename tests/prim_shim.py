"""Builds and drives tests/device_shim/prim_ops.h: the device build (prim_kernels.cu, nvcc for sm_100a with the library's
flags) and the host build (host_shim/prim_host.cpp, g++).  Records are rows of little-endian 32-bit words; field elements
are 8 words in Montgomery form (R = 2^256) unless an operation says otherwise.  Also converts pairing.cuh's tower
Fq12 = Fq6[w]/(w^2 - v), Fq6 = Fq2[v]/(v^3 - xi), xi = 9 + u, to the oracle's Fq[w]/(w^12 - 18 w^6 + 82) with
u = w^6 - 9."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np

from conftest import ROOT

R = 1 << 256
FAM_FR, FAM_FQ, FAM_FQ2, FAM_TOWER, FAM_PAIRING, FAM_G2 = range(6)
SHIM = os.path.join(ROOT, "tests", "device_shim")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared"]


def nvcc():
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    return cand if os.path.exists(cand) else None


def compile_device(out_dir):
    """nvcc build of the device shim (no LZKP_FQ2_INLINE: the out-of-line Fq2 product, as in the library)."""
    out = os.path.join(str(out_dir), "prim_dev.so")
    subprocess.run([nvcc()] + NVCC_FLAGS + ["-o", out, os.path.join(SHIM, "prim_kernels.cu")], check=True)
    return out


def compile_host(out_dir):
    out = os.path.join(str(out_dir), "prim_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", out,
                    os.path.join(ROOT, "tests", "host_shim", "prim_host.cpp")], check=True)
    return out


_BUILT = {}


def device(tmp_path_factory):
    """the device shim, compiled once per session (it takes about two minutes)"""
    if "device" not in _BUILT:
        _BUILT["device"] = Device(compile_device(tmp_path_factory.mktemp("prim_dev")))
    return _BUILT["device"]


def host(tmp_path_factory):
    if "host" not in _BUILT:
        _BUILT["host"] = Host(compile_host(tmp_path_factory.mktemp("prim_host")))
    return _BUILT["host"]


def words(vals, k=8):
    """ints -> (n, k) uint32 rows"""
    return np.frombuffer(b"".join(int(v).to_bytes(4 * k, "little") for v in vals), "<u4").reshape(len(vals), k).copy()


def ints(rows):
    """(n, k) uint32 rows -> ints"""
    return [int.from_bytes(r.tobytes(), "little") for r in np.ascontiguousarray(rows, "<u4")]


def records(in_words, *cols):
    """Rows of `in_words` words: column j (an (n, k) word array, or a list of ints as 8-word values) from word offset
    cols[j][0]."""
    n = None
    parts = []
    for off, c in cols:
        a = c if isinstance(c, np.ndarray) else words(c)
        n = a.shape[0]
        parts.append((off, a))
    rec = np.zeros((n, in_words), np.uint32)
    for off, a in parts:
        rec[:, off:off + a.shape[1]] = a
    return rec


class Host:
    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.lib.prim_run_host.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]

    def shape(self, fam):
        i, o = C.c_int(), C.c_int()
        assert self.lib.prim_words(fam, C.byref(i), C.byref(o)) == 0
        return i.value, o.value

    def run(self, fam, code, rec):
        iw, ow = self.shape(fam)
        rec = np.ascontiguousarray(rec, np.uint32)
        assert rec.shape[1] == iw
        out = np.zeros((rec.shape[0], ow), np.uint32)
        self.lib.prim_run_host(fam, code, rec.ctypes.data, out.ctypes.data, rec.shape[0])
        return out


class Device:
    """The launchers take device pointers (torch tensors), a count and the current stream; each returns
    cudaGetLastError()."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        vp, i = C.c_void_p, C.c_int
        self.lib.prim_launch.argtypes = [i, i, vp, vp, i, vp]
        self.lib.prim_fq_half.argtypes = [vp, vp, i, vp]
        self.lib.prim_coop_f12_mul.argtypes = [i, i, vp, vp, i, vp]
        self.lib.prim_coop_f12_map.argtypes = [i, vp, vp, i, vp]
        self.lib.prim_coop_subgroup.argtypes = [vp, vp, i, vp]
        self.lib.prim_coop_ladder.argtypes = [i, vp, vp, i, vp]

    def shape(self, fam):
        i, o = C.c_int(), C.c_int()
        assert self.lib.prim_words(fam, C.byref(i), C.byref(o)) == 0
        return i.value, o.value

    def _call(self, fn, args, rec, out_words):
        import torch
        rec = np.ascontiguousarray(rec, np.uint32)
        n = rec.shape[0]
        d_in = torch.from_numpy(rec.view(np.int32)).cuda()
        d_out = torch.zeros((n, out_words), dtype=torch.int32, device="cuda")
        err = fn(*args, d_in.data_ptr(), d_out.data_ptr(), n, torch.cuda.current_stream().cuda_stream)
        assert err == 0, f"launch error {err}"
        torch.cuda.synchronize()
        return d_out.cpu().numpy().view(np.uint32)

    def run(self, fam, code, rec):
        iw, ow = self.shape(fam)
        assert rec.shape[1] == iw
        return self._call(self.lib.prim_launch, (fam, code), rec, ow)

    def fq_half(self, rec):
        return self._call(self.lib.prim_fq_half, (), rec, 8)

    def coop_f12_mul(self, sparse, mode, rec):          # rec: a (96) | b (96) | sa (16) | sb (16) -> r (96) | so (16)
        assert rec.shape[1] == 224
        return self._call(self.lib.prim_coop_f12_mul, (int(sparse), mode), rec, 112)

    def coop_f12_map(self, k, rec):                     # 0: f12_conj, 1 / 2 / 3: f12_frob<k>
        return self._call(self.lib.prim_coop_f12_map, (k,), rec, 96)

    def coop_subgroup(self, rec):
        return self._call(self.lib.prim_coop_subgroup, (), rec, 1)[:, 0]

    def coop_ladder(self, mode, rec):                   # X | Y | ZZ | ZZZ | bx | by | add -> X | Y | ZZ | ZZZ | madd's result
        assert rec.shape[1] == 97
        return self._call(self.lib.prim_coop_ladder, (mode,), rec, 65)


# ---- Montgomery form and the tower
class Mont:
    def __init__(self, m):
        self.m, self.rinv = m, pow(R, -1, m)

    def to(self, v):
        return v * R % self.m

    def frm(self, v):
        return v * self.rinv % self.m


def tower_to_flat(po, coeffs):
    """Six Fq2 coefficients in tower order (index 3h + k: v^k of c_h), canonical (a, b) pairs -> the oracle's Fq12.
    Coefficient (a + b u) of v^k w^h adds a - 9b to flat index 2k + h and b to 2k + h + 6."""
    q = po.Q_MOD
    flat = [0] * 12
    for h in range(2):
        for k in range(3):
            a, b = coeffs[3 * h + k]
            j = 2 * k + h
            flat[j] = (flat[j] + a - 9 * b) % q
            flat[j + 6] = (flat[j + 6] + b) % q
    return flat


def flat_to_tower(po, flat):
    q = po.Q_MOD
    out = [None] * 6
    for h in range(2):
        for k in range(3):
            j = 2 * k + h
            b = flat[j + 6] % q
            out[3 * h + k] = ((flat[j] + 9 * b) % q, b)
    return out


def fq12_words(po, flat):
    """oracle Fq12 -> 96 words of Montgomery limbs"""
    mq = Mont(po.Q_MOD)
    return words([mq.to(v) for c in flat_to_tower(po, flat) for v in c]).reshape(96)


def fq12_flat(po, row):
    """96 words of Montgomery limbs -> oracle Fq12"""
    mq = Mont(po.Q_MOD)
    v = [mq.frm(x) for x in ints(np.asarray(row, np.uint32).reshape(12, 8))]
    return tower_to_flat(po, [(v[2 * i], v[2 * i + 1]) for i in range(6)])


def g1_words(po, P):
    mq = Mont(po.Q_MOD)
    return words([mq.to(P[0]), mq.to(P[1])]).reshape(16)


def g2_words(po, Q):
    mq = Mont(po.Q_MOD)
    return words([mq.to(Q[0][0]), mq.to(Q[0][1]), mq.to(Q[1][0]), mq.to(Q[1][1])]).reshape(32)


def g2_from_words(po, row):
    """32 words (affine x | y, Montgomery) -> oracle point, all zero -> None"""
    mq = Mont(po.Q_MOD)
    v = ints(np.asarray(row, np.uint32)[:32].reshape(4, 8))
    if not any(v):
        return None
    v = [mq.frm(x) for x in v]
    return ((v[0], v[1]), (v[2], v[3]))


# The final exponentiation of pairing.cuh raises to (p^12 - 1) / r times this constant (coprime to r): its pairing is
# the oracle's to this power.
def pairing_power(po):
    x = po.BN_X
    return 2 * x * (6 * x * x + 3 * x + 1)
