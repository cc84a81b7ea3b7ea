"""ark-serialize's compressed form on the device: decompression (one square root per point) gives the uncompressed bytes
of the same points, rejects what ark rejects with bytes every verifier form refuses, compressed keys load to keys that
prove byte-identically and decide identically, and proofs go prove -> compress -> decompress -> verify on one stream."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from libzkp_b200 import _ffi, engine
from libzkp_b200.errors import EngineError
from oracle import zkp_compressed as pc

pytestmark = pytest.mark.gpu
WINDOW_BITS = 10


def _forms(monkeypatch, form):
    """Environment that forces one verifier form at small sizes (as test_gpu_verify_device.py does)."""
    for k in ("LZKP_VERIFY_RLC_MIN", "LZKP_VERIFY_COOP_MAX"):
        monkeypatch.delenv(k, raising=False)
    if form == "latency":
        monkeypatch.setenv("LZKP_VERIFY_RLC_MIN", "1000000000")
        monkeypatch.setenv("LZKP_VERIFY_COOP_MAX", "100000")
    elif form == "lanes":
        monkeypatch.setenv("LZKP_VERIFY_RLC_MIN", "1000000000")
        monkeypatch.setenv("LZKP_VERIFY_COOP_MAX", "0")
    elif form == "combined":
        monkeypatch.setenv("LZKP_VERIFY_RLC_MIN", "64")


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _decompress_device(comp, stream=None):
    import torch
    n = comp.shape[0]
    d_in = _cuda(comp)
    d_out = torch.full((n, 256), 0x5A, dtype=torch.uint8, device="cuda")
    d_ok = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
    st = stream if stream is not None else torch.cuda.current_stream()
    engine.proofs_decompress_device(n, d_in.data_ptr(), d_out.data_ptr(), d_ok.data_ptr(), st.cuda_stream)
    torch.cuda.synchronize()
    return d_out.cpu().numpy(), d_ok.cpu().numpy()


@pytest.fixture(scope="module")
def eq_batch(eq_keys, po, frs):
    """130 valid equality proofs (three groups of the combined form at LZKP_VERIFY_RLC_MIN=64) and their commitments."""
    pk = engine.ProvingKey(eq_keys.pk_bytes, window_bits=WINDOW_BITS)
    try:
        pk.circuit_builtin(engine.EQUALITY, 110)
        n = 130
        rng = po.SplitMix64(5151)
        a = np.array([rng.next_u64() for _ in range(n)], np.uint64)
        proofs, cms, st = pk.prove_equality_batch(a, a, frs(5152, n), frs(5153, n))
    finally:
        pk.close()
    assert not st.any()
    return proofs, cms


def _random_points(po, frs, seed, n):
    s = frs(seed, n)
    return engine.generator_mul(1, s), engine.generator_mul(2, s)


def test_decompression_equals_uncompressed_bytes(po, frs):
    n = 300
    g1, g2 = _random_points(po, frs, 6000, n + 1)
    proofs = np.concatenate([g1[:n], g2[:n], g1[1:n + 1]], axis=1)
    inf1 = np.frombuffer(po.g1_to_bytes(None), np.uint8)
    inf2 = np.frombuffer(po.g2_to_bytes(None), np.uint8)
    proofs[5, 0:64] = inf1
    proofs[6, 64:192] = inf2
    proofs[7, 192:256] = inf1
    # both roots: the uncompressed sign bit of A / B / C takes both values among the rows
    for off in (63, 191, 255):
        assert set((proofs[:, off] >> 7).tolist()) == {0, 1}
    comp, ok = engine.proofs_compress(proofs)
    assert ok.all()
    for i in (0, 5, 6, 7, 299):
        P = po.proof_from_bytes(proofs[i].tobytes(), False)
        assert comp[i].tobytes() == pc.proof_to_bytes_compressed(P)
    out, ok = engine.proofs_decompress(comp)
    assert ok.all() and np.array_equal(out, proofs)
    out, ok = _decompress_device(comp)
    assert (ok == 1).all() and np.array_equal(out, proofs)


def _malformed_rows(po, eq_batch):
    """(row, label): one defect each on top of a valid compressed proof."""
    proofs, _ = eq_batch
    comp, ok = engine.proofs_compress(proofs[:8])
    assert ok.all()
    rows = comp.copy()
    rows[0, 0:32] = np.frombuffer(po.Q_MOD.to_bytes(32, "little"), np.uint8)            # A.x = q
    rows[1, 127] |= 0xC0                                                                # both flags on C
    x = next(x for x in range(1, 100) if pc.fq_sqrt(x ** 3 + 3) is None)
    rows[2, 0:32] = np.frombuffer(x.to_bytes(32, "little"), np.uint8)                   # x^3 + 3 a non-residue
    k = 1
    while True:                                                                          # a twist x with no root
        try:
            pc.g2_from_bytes_compressed(k.to_bytes(32, "little") + (k + 1).to_bytes(32, "little"))
        except ValueError:
            break
        k += 1
    rows[3, 32:96] = np.frombuffer(k.to_bytes(32, "little") + (k + 1).to_bytes(32, "little"), np.uint8)
    rows[4, 63] |= 0x80                                                                 # flags on B's x.c0
    return rows[:5], ["x >= q", "both flags", "G1 non-residue", "G2 no root", "flags on x.c0"]


def test_malformed_inputs_are_rejected(po, eq_batch, eq_keys):
    rows, labels = _malformed_rows(po, eq_batch)
    for r in rows:
        with pytest.raises(ValueError):
            pc.proof_from_bytes_compressed(r.tobytes())
    out, ok = engine.proofs_decompress(rows)
    assert not ok.any(), labels
    dout, dok = _decompress_device(rows)
    assert (dok == 0).all() and np.array_equal(dout, out)
    for r in out:                                                      # malformed to every reader
        with pytest.raises(ValueError):
            po.proof_from_bytes(r.tobytes(), False)
    _, cms = eq_batch
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        assert not vk.verify_batch(out, cms[:5]).any()
    finally:
        vk.close()


def _prove_eq(pk, po, frs, n=40, seed=700):
    rng = po.SplitMix64(seed)
    a = np.array([rng.next_u64() for _ in range(n)], np.uint64)
    proofs, _, st = pk.prove_equality_batch(a, a, frs(seed + 1, n), frs(seed + 2, n))
    assert not st.any()
    return proofs


def _prove_mb(pk, po, frs, n=12, seed=800):
    rng = po.SplitMix64(seed)
    sets = np.zeros((n, 64), np.uint64)
    lens = (1 + (np.arange(n) * 7) % 64).astype(np.uint32)
    for i in range(n):
        sets[i, :lens[i]] = [rng.next_u64() for _ in range(lens[i])]
    vals = sets[np.arange(n), np.arange(n) % lens]
    proofs, _, st = pk.prove_membership_batch(vals, sets, lens, frs(seed + 1, n), frs(seed + 2, n))
    assert not st.any()
    return proofs


@pytest.mark.parametrize("which,validate", [("eq", 0), ("eq", 1), ("mb", 0), ("mb", 1)])
def test_compressed_key_proves_identically(eq_keys, mb_keys, po, frs, which, validate):
    keys = eq_keys if which == "eq" else mb_keys
    kind, param, prove = (engine.EQUALITY, 110, _prove_eq) if which == "eq" else (engine.MEMBERSHIP, 64, _prove_mb)
    comp = engine.pk_compress(keys.pk_bytes)
    want_pk = engine.ProvingKey(keys.pk_bytes, validate=bool(validate), window_bits=WINDOW_BITS)
    got_pk = engine.ProvingKey(comp, validate=bool(validate), window_bits=WINDOW_BITS, compressed=True)
    try:
        assert (got_pk.n_vars, got_pk.n, got_pk.table_bytes) == (want_pk.n_vars, want_pk.n, want_pk.table_bytes)
        want_pk.circuit_builtin(kind, param)
        got_pk.circuit_builtin(kind, param)
        assert np.array_equal(prove(got_pk, po, frs), prove(want_pk, po, frs))
    finally:
        want_pk.close()
        got_pk.close()


@pytest.mark.parametrize("validate", [0, 1])
def test_compressed_key_large_mode(eq_keys, co, frs, monkeypatch, validate):
    monkeypatch.setenv("LZKP_FORCE_LARGE", "1")
    comp = engine.pk_compress(eq_keys.pk_bytes)
    want_pk = engine.ProvingKey(eq_keys.pk_bytes, validate=bool(validate))
    got_pk = engine.ProvingKey(comp, validate=bool(validate), compressed=True)
    try:
        assert got_pk.max_chunk == 1 and want_pk.max_chunk == 1                  # both in large mode
        z = np.stack([eq_keys.circuit.assign(v, v) for v in (3, 77)])
        r, s = frs(901, 2), frs(902, 2)
        for pk in (want_pk, got_pk):
            pk.circuit_builtin(engine.EQUALITY, 110)
        p_got, st_got = got_pk.prove_batch(z, r, s)
        p_want, st_want = want_pk.prove_batch(z, r, s)
        assert not st_got.any() and not st_want.any() and np.array_equal(p_got, p_want)
    finally:
        want_pk.close()
        got_pk.close()


def _twist_point_outside_subgroup(po):
    k = 3
    while True:
        b = k.to_bytes(32, "little") + bytes(32)
        try:
            Q = pc.g2_from_bytes_compressed(b)
        except ValueError:
            k += 1
            continue
        if po.G2.mul(Q, po.R_MOD) is not None:
            return Q
        k += 1


def test_compressed_vk_loads_and_decides_like_uncompressed(eq_keys, mb_keys, po, eq_batch):
    for keys in (eq_keys, mb_keys):
        a = engine.VerifyingKey(keys.vk_bytes)
        b = engine.VerifyingKey(engine.vk_compress(keys.vk_bytes), compressed=True)
        try:
            assert a.info() == b.info() and a.n_pub == b.n_pub
            if keys is eq_keys:
                proofs, cms = eq_batch
                x = cms.copy()
                x[3] = x[4]
                assert np.array_equal(a.verify_batch(proofs, x), b.verify_batch(proofs, x))
                assert not b.verify_batch(proofs, x)[3] and b.verify_batch(proofs, x).sum() == len(proofs) - 1
        finally:
            a.close()
            b.close()
    # a G2 point of the key outside the r-torsion: refused by the validating loads
    bad = np.frombuffer(pc.g2_to_bytes_compressed(_twist_point_outside_subgroup(po)), np.uint8)
    vk_c = np.frombuffer(engine.vk_compress(eq_keys.vk_bytes), np.uint8).copy()
    vk_c[160:224] = bad                                                           # delta_g2
    with pytest.raises(EngineError) as e:
        engine.VerifyingKey(vk_c.tobytes(), compressed=True)
    assert e.value.code == _ffi.LZKP_E_INVALID
    pk_c = np.frombuffer(engine.pk_compress(eq_keys.pk_bytes), np.uint8).copy()
    pk_c[160:224] = bad
    with pytest.raises(EngineError) as e:
        engine.ProvingKey(pk_c.tobytes(), validate=True, window_bits=WINDOW_BITS, compressed=True)
    assert e.value.code == _ffi.LZKP_E_INVALID
    # a point that does not decode at all: refused with or without validation
    pk_c[0:32] = np.frombuffer(po.Q_MOD.to_bytes(32, "little"), np.uint8)
    with pytest.raises(EngineError) as e:
        engine.ProvingKey(pk_c.tobytes(), window_bits=WINDOW_BITS, compressed=True)
    assert e.value.code == _ffi.LZKP_E_INVALID


def _verification_cases(po, eq_batch):
    proofs, cms = eq_batch
    comp, ok = engine.proofs_compress(proofs)
    assert ok.all()
    comp = comp.copy()
    comp[10, 31] ^= 0x80                                                          # sign of A
    comp[70, 95] ^= 0x80                                                          # sign of B
    comp[71, 127] ^= 0x80                                                         # sign of C
    comp[128, 32:96] = np.frombuffer(pc.g2_to_bytes_compressed(_twist_point_outside_subgroup(po)), np.uint8)
    comp[129, 0:32] = np.frombuffer(po.Q_MOD.to_bytes(32, "little"), np.uint8)   # does not decode
    return comp, cms


@pytest.fixture(scope="module")
def oracle_decisions(po, eq_batch, eq_keys):
    """The oracle's decode followed by its pairing verifier, for the altered rows and two untouched ones."""
    comp, cms = _verification_cases(po, eq_batch)
    vk = po.vk_from_bytes(eq_keys.vk_bytes)
    want = {}
    for i in (0, 10, 70, 71, 128, 129, 127):
        try:
            P = pc.proof_from_bytes_compressed(comp[i].tobytes())
        except ValueError:
            want[i] = False
            continue
        want[i] = po.verify(vk, [int.from_bytes(cms[i].tobytes(), "little")], P)
    return want


@pytest.mark.parametrize("form", ["latency", "lanes", "combined"])
def test_compressed_verification_equals_oracle(po, eq_batch, eq_keys, oracle_decisions, monkeypatch, form):
    import torch
    _forms(monkeypatch, form)
    comp, cms = _verification_cases(po, eq_batch)
    n = comp.shape[0]
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        d_c, d_x = _cuda(comp), _cuda(cms)
        d_p = torch.zeros((n, 256), dtype=torch.uint8, device="cuda")
        d_dok = torch.zeros(n, dtype=torch.uint8, device="cuda")
        d_ok = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            engine.proofs_decompress_device(n, d_c.data_ptr(), d_p.data_ptr(), d_dok.data_ptr(), st.cuda_stream)
            vk.verify_batch_device(n, d_p.data_ptr(), d_x.data_ptr(), 1, d_ok.data_ptr(), st.cuda_stream)
        st.synchronize()
        got = d_ok.cpu().numpy()
        dok = d_dok.cpu().numpy()
    finally:
        vk.close()
    assert set(np.unique(got)) <= {0, 1}
    assert dok.tolist() == [0 if i == 129 else 1 for i in range(n)]
    want = np.ones(n, bool)
    for i, v in oracle_decisions.items():
        want[i] = v
    assert [oracle_decisions[i] for i in (0, 127)] == [True, True]
    assert not any(oracle_decisions[i] for i in (10, 70, 71, 128, 129))
    assert np.array_equal(got.astype(bool), want), np.flatnonzero(got.astype(bool) != want)


def test_device_round_trip_on_one_stream(eq_keys, po, frs):
    import torch
    n = 96
    pk = engine.ProvingKey(eq_keys.pk_bytes, window_bits=WINDOW_BITS)
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        pk.circuit_builtin(engine.EQUALITY, 110)
        rng = po.SplitMix64(990)
        a = np.array([rng.next_u64() for _ in range(n)], np.uint64)
        r, s = frs(991, n), frs(992, n)
        _, cms, _ = pk.prove_equality_batch(a, a, r, s)
        d_a, d_r, d_s = _cuda(a), _cuda(r), _cuda(s)
        d_x = _cuda(cms)
        d_p = torch.zeros((n, 256), dtype=torch.uint8, device="cuda")
        d_st = torch.zeros(n, dtype=torch.int32, device="cuda")
        d_c = torch.zeros((n, 128), dtype=torch.uint8, device="cuda")
        d_cok = torch.zeros(n, dtype=torch.uint8, device="cuda")
        d_p2 = torch.zeros((n, 256), dtype=torch.uint8, device="cuda")
        d_dok = torch.zeros(n, dtype=torch.uint8, device="cuda")
        d_ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        st = torch.cuda.Stream()
        h = st.cuda_stream
        pk.prove_equality_batch_device(n, d_a.data_ptr(), d_a.data_ptr(), d_r.data_ptr(), d_s.data_ptr(), d_p.data_ptr(),
                                       d_st.data_ptr(), h)
        engine.proofs_compress_device(n, d_p.data_ptr(), d_c.data_ptr(), d_cok.data_ptr(), h)
        engine.proofs_decompress_device(n, d_c.data_ptr(), d_p2.data_ptr(), d_dok.data_ptr(), h)
        vk.verify_batch_device(n, d_p2.data_ptr(), d_x.data_ptr(), 1, d_ok.data_ptr(), h)
        st.synchronize()
        proofs = d_p.cpu().numpy()
        assert not d_st.cpu().numpy().any()
        assert d_cok.cpu().numpy().all() and d_dok.cpu().numpy().all() and d_ok.cpu().numpy().all()
        assert np.array_equal(d_p2.cpu().numpy(), proofs)
        comp = d_c.cpu().numpy()
        for i in range(0, n, 7):
            assert comp[i].tobytes() == pc.proof_to_bytes_compressed(po.proof_from_bytes(proofs[i].tobytes(), False))
        host_c, _ = engine.proofs_compress(proofs)
        assert np.array_equal(host_c, comp)
    finally:
        pk.close()
        vk.close()


def test_arguments():
    import torch
    buf = torch.zeros(256, dtype=torch.uint8, device="cuda")
    p = buf.data_ptr()
    for fn in (engine.proofs_compress_device, engine.proofs_decompress_device):
        for args in ((0, p, p), (p, 0, p), (p, p, 0)):
            with pytest.raises(EngineError) as e:
                fn(1, *args)
            assert e.value.code == _ffi.LZKP_E_INVALID
        host = np.zeros(256, np.uint8)
        with pytest.raises(EngineError) as e:                          # host memory is refused, not read
            fn(1, host.ctypes.data, p, p)
        assert e.value.code == _ffi.LZKP_E_INVALID
        before = engine.kernel_launches()
        fn(0, 0, 0, 0)                                                 # n == 0: nothing enqueued
        fn(0, p, p, p)
        assert engine.kernel_launches() == before
    L = _ffi.lib()
    assert L.lzkp_proofs_decompress(1, None, None, None) == _ffi.LZKP_E_INVALID
    assert L.lzkp_proofs_compress(1, None, None, None) == _ffi.LZKP_E_INVALID
    out, ok = engine.proofs_decompress(np.zeros((0, 128), np.uint8))
    assert out.shape == (0, 256) and ok.shape == (0,)


_MULTI = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from libzkp_b200 import engine
from oracle import c_oracle as co, zkp_oracle as po
engine.init([0, 1])
td = po.Trapdoor.from_seed(1)
circ = co.Circuit("equality")
pk_bytes, _ = circ.setup((td.alpha, td.beta, td.gamma, td.delta, td.tau))
n = 1100                                                  # >= 512: one block per device
rng = po.SplitMix64(31)
a = np.array([rng.next_u64() for _ in range(n)], np.uint64)
def frs(seed):
    g = po.SplitMix64(seed)
    return np.frombuffer(b"".join(g.next_fr().to_bytes(32, "little") for _ in range(n)), np.uint8).reshape(n, 32).copy()
r, s = frs(32), frs(33)
out = []
for comp in (False, True):
    key = engine.pk_compress(pk_bytes) if comp else pk_bytes
    pk = engine.ProvingKey(key, window_bits=10, compressed=comp)
    pk.circuit_builtin(engine.EQUALITY, 110)
    p, _, st = pk.prove_equality_batch(a, a, r, s)
    out.append((p, st))
    pk.close()
print(json.dumps({"identical": bool(np.array_equal(out[0][0], out[1][0])), "ok": bool(not out[0][1].any() and not out[1][1].any())}))
"""


def test_multi_gpu_compressed_key_fans_out():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two visible GPUs")
    res = subprocess.run([sys.executable, "-c", _MULTI, ROOT], capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    rep = json.loads(res.stdout.strip().splitlines()[-1])
    assert rep["identical"] and rep["ok"]
