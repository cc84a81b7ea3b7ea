"""Proof rerandomization on the device (lzkp_proofs_rerandomize, ark-groth16's rerandomize_proof): byte-equal to the
big-integer checker (oracle/zkp_rerandomize.py) on three keys, edge factors, infinity inputs and results; malformed rows
get ok 0 and 0xFF without touching their neighbours; rerandomized proofs keep every verifier form's decisions and
compose; the device form matches the host form in place, on one stream with proving, verifying and the compressed
codecs, under graph capture and on two streams at once, and checks its arguments."""
import numpy as np
import pytest

from libzkp_b200 import _ffi, engine
from libzkp_b200.errors import EngineError
from oracle import zkp_compressed as pc
from oracle import zkp_rerandomize as zr

pytestmark = pytest.mark.gpu
WINDOW_BITS = 10
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
L = zr.LAMBDA_PSI
FF = b"\xff" * 256


def _fr(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), np.uint8).reshape(-1, 32).copy()


def _ints(a):
    return [int.from_bytes(a[i].tobytes(), "little") for i in range(a.shape[0])]


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _forms(monkeypatch, form):
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


@pytest.fixture(scope="module")
def eq_proofs(eq_keys, po, frs):
    """300 valid equality proofs and their commitments."""
    pk = engine.ProvingKey(eq_keys.pk_bytes, window_bits=WINDOW_BITS)
    try:
        pk.circuit_builtin(engine.EQUALITY, 110)
        n = 300
        rng = po.SplitMix64(7070)
        a = np.array([rng.next_u64() for _ in range(n)], np.uint64)
        proofs, cms, st = pk.prove_equality_batch(a, a, frs(7071, n), frs(7072, n))
    finally:
        pk.close()
    assert not st.any()
    return proofs, cms


@pytest.fixture(scope="module")
def mb_proofs(mb_keys, po, frs, co):
    """96 valid membership-64 proofs and their public inputs (n, 129, 32)."""
    pk = engine.ProvingKey(mb_keys.pk_bytes, window_bits=8)
    try:
        pk.circuit_builtin(engine.MEMBERSHIP, 64)
        m = 96
        rng = po.SplitMix64(7170)
        sets = np.zeros((m, 64), np.uint64)
        lens = (1 + (np.arange(m) * 5) % 64).astype(np.uint32)
        for i in range(m):
            sets[i, :lens[i]] = [rng.next_u64() for _ in range(lens[i])]
        vals = sets[np.arange(m), np.arange(m) % lens]
        proofs, cms, st = pk.prove_membership_batch(vals, sets, lens, frs(7171, m), frs(7172, m))
    finally:
        pk.close()
    assert not st.any()
    xs = np.zeros((m, 129, 32), np.uint8)
    for i in range(m):
        xs[i] = co.fr_array(po.membership_public_inputs(int.from_bytes(cms[i].tobytes(), "little"),
                                                        [int(v) for v in sets[i, :lens[i]]]))
    return proofs, xs


def _big_vk_bytes(eq_keys, frs):
    """The equality key's alpha, beta, gamma, delta with 301 gamma_abc points: a key with 300 public inputs."""
    abc = engine.generator_mul(1, frs(7300, 301))
    return eq_keys.vk_bytes[:448] + (301).to_bytes(8, "little") + abc.tobytes()


def _check_rows(po, vk_bytes, proofs, r1, r2, out, ok, rows):
    delta = po.vk_from_bytes(vk_bytes).delta_g2
    a1, a2 = _ints(r1), _ints(r2)
    for i in rows:
        want = zr.rerandomize_bytes(delta, proofs[i].tobytes(), a1[i], a2[i])
        assert out[i].tobytes() == want, i
        assert bool(ok[i]) == (want != FF), i


@pytest.mark.parametrize("key", ["eq", "mb", "big"])
def test_bytes_equal_oracle(key, eq_keys, mb_keys, eq_proofs, mb_proofs, po, frs):
    if key == "eq":
        vk_bytes, proofs = eq_keys.vk_bytes, eq_proofs[0]
    elif key == "mb":
        vk_bytes, proofs = mb_keys.vk_bytes, mb_proofs[0]
    else:
        vk_bytes, proofs = _big_vk_bytes(eq_keys, frs), eq_proofs[0]
    vk = engine.VerifyingKey(vk_bytes)
    try:
        if key == "big":
            assert vk.n_pub == 300
        for n in (1, 31, 32, 33, 300, 4096):
            p = np.tile(proofs, (n // proofs.shape[0] + 1, 1))[:n]
            r1, r2 = frs(7400 + n, n), frs(7500 + n, n)
            out, ok = vk.rerandomize(p, r1, r2)
            assert ok.all(), n
            # every row up to 300; seeded rows sampled from 4096
            rows = range(n) if n <= 300 else sorted(set(np.random.default_rng(7603).integers(0, n, 48).tolist()) | {0, n - 1})
            _check_rows(po, vk_bytes, p, r1, r2, out, ok, rows)
    finally:
        vk.close()


def test_edge_factors(eq_keys, eq_proofs, po):
    edges = [1, R - 1, L - 1, L, L + 1, 2 * L, 2 * L + 1, R - L, ((R - 1) // L) * L, ((R - 1) // L) * L - 1]
    pairs = [(a, b) for a in edges for b in (1, R - 1, L, L + 1)]
    pairs += [(a, pow(a, -1, R)) for a in (2, L, R - 1, 0x1234567)]          # r1 r2 == 1
    pairs += [(k * pow(7, -1, R) % R, 7) for k in (L - 1, L, L + 1, 2 * L)]     # r1 r2 at the split's edges
    n = len(pairs)
    proofs = np.tile(eq_proofs[0][:7], (n // 7 + 1, 1))[:n].copy()
    r1, r2 = _fr([a for a, _ in pairs]), _fr([b for _, b in pairs])
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        out, ok = vk.rerandomize(proofs, r1, r2)
    finally:
        vk.close()
    assert ok.all()
    _check_rows(po, eq_keys.vk_bytes, proofs, r1, r2, out, ok, range(n))


def test_infinity_inputs_and_results(eq_keys, eq_proofs, po):
    delta = po.vk_from_bytes(eq_keys.vk_bytes).delta_g2
    A, B, C = po.proof_from_bytes(eq_proofs[0][0].tobytes())
    r1, r2 = 0x5EED1, 0xC0FFEE
    cases = [(None, B, C), (A, None, C), (A, B, None), (None, None, None),
             (A, B, po.G1.neg(po.G1.mul(A, r2))),                               # C' = C + r2 A = infinity
             (A, po.G2.neg(po.G2.mul(delta, r2)), C)]                            # B' = r1 (B + r2 delta) = infinity
    proofs = np.frombuffer(b"".join(po.proof_to_bytes(P) for P in cases), np.uint8).reshape(-1, 256).copy()
    n = len(cases)
    f1, f2 = _fr([r1] * n), _fr([r2] * n)
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        out, ok = vk.rerandomize(proofs, f1, f2)
    finally:
        vk.close()
    assert ok.all()
    _check_rows(po, eq_keys.vk_bytes, proofs, f1, f2, out, ok, range(n))
    inf1, inf2 = po.g1_to_bytes(None), po.g2_to_bytes(None)
    assert out[4, 192:].tobytes() == inf1 and out[5, 64:192].tobytes() == inf2


def _twist_point_outside_subgroup(po):
    for x in range(1, 1000):
        try:
            P = pc.g2_from_bytes_compressed(x.to_bytes(32, "little") + bytes(32))
        except ValueError:
            continue
        if P is not None and po.G2.mul(P, R) is not None:
            return P
    raise AssertionError("no twist point found")


def test_malformed_rows(eq_keys, eq_proofs, po):
    good = eq_proofs[0][0]
    bad = []

    def row(f):
        b = bytearray(good.tobytes())
        f(b)
        bad.append(bytes(b))

    q = po.Q_MOD.to_bytes(32, "little")
    row(lambda b: b.__setitem__(slice(0, 32), q))                              # A.x = q (non-canonical)
    row(lambda b: b.__setitem__(slice(128, 160), q))                           # B.y.c0 = q
    row(lambda b: b.__setitem__(31, b[31] | 0x40))                             # a flag on A.x
    row(lambda b: b.__setitem__(95, b[95] | 0x80))                             # a flag on B.x.c0
    row(lambda b: b.__setitem__(63, b[63] | 0xC0))                             # both flags on A.y
    row(lambda b: b.__setitem__(191, b[191] | 0xC0))                           # both flags on B.y
    row(lambda b: b.__setitem__(255, b[255] | 0xC0))                           # both flags on C.y
    row(lambda b: b.__setitem__(32, b[32] ^ 1))                                # A off the curve
    row(lambda b: b.__setitem__(64, b[64] ^ 1))                                # B off the twist
    row(lambda b: b.__setitem__(224, b[224] ^ 1))                              # C off the curve
    T = _twist_point_outside_subgroup(po)
    row(lambda b: b.__setitem__(slice(64, 192), po.g2_to_bytes(T)))            # B on the twist, outside the r-torsion
    Bp = po.proof_from_bytes(good.tobytes())[1]
    row(lambda b: b.__setitem__(slice(64, 192), po.g2_to_bytes(po.G2.add(Bp, T))))   # the proof's B shifted by T
    n_fmt = len(bad)
    # interleave: good, bad, good, bad, ..., then three rows with bad factors
    rows, f1, f2 = [], [], []
    for i, b in enumerate(bad):
        rows += [good.tobytes(), b]
        f1 += [3 + i, 5 + i]
        f2 += [7 + i, 11 + i]
    rows += [good.tobytes()] * 4
    f1 += [0, 9, R, 13]
    f2 += [9, 0, 9, R + 1]
    proofs = np.frombuffer(b"".join(rows), np.uint8).reshape(-1, 256).copy()
    r1 = np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in f1), np.uint8).reshape(-1, 32).copy()
    r2 = np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in f2), np.uint8).reshape(-1, 32).copy()
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        out, ok = vk.rerandomize(proofs, r1, r2)
        want_ok = [True, False] * n_fmt + [False, False, False, False]
        assert ok.tolist() == want_ok
        for i, w in enumerate(want_ok):
            if not w:
                assert out[i].tobytes() == FF, i
        _check_rows(po, eq_keys.vk_bytes, proofs, r1, r2, out, ok, range(len(rows)))
        # every verifier form rejects the 0xFF rows
        x = np.tile(eq_proofs[1][0], (len(rows), 1))
        assert not vk.verify_batch(out[~ok], x[~ok]).any()
        assert vk.verify_batch(out[ok], x[ok]).all()
    finally:
        vk.close()


@pytest.mark.parametrize("form", ["latency", "combined", "lanes"])
def test_decisions_preserved(eq_keys, mb_keys, eq_proofs, mb_proofs, frs, monkeypatch, form):
    n = 4096 if form == "combined" else 300
    proofs = np.tile(eq_proofs[0], (n // 300 + 1, 1))[:n].copy()
    cms = np.tile(eq_proofs[1], (n // 300 + 1, 1))[:n].copy()
    cms[5, 0] ^= 1                                                   # wrong commitment
    proofs[17, 192:256] = proofs[18, 192:256]                        # C of another proof: on the curve, wrong
    proofs[29, 200] ^= 4                                             # tampered C: off the curve
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    vkm = engine.VerifyingKey(mb_keys.vk_bytes)
    try:
        _forms(monkeypatch, form)
        before = vk.verify_batch(proofs, cms)
        assert before.sum() == n - 3 and not before[[5, 17, 29]].any()
        out, ok = vk.rerandomize(proofs, frs(7700, n), frs(7701, n))
        assert ok.sum() == n - 1 and not ok[29]
        assert np.array_equal(vk.verify_batch(out, cms), before)
        # every point of a rerandomized valid proof differs from the input (r1 != +-1, r2 != 0)
        for i in (0, 1, 100, n - 1):
            for lo, hi in ((0, 64), (64, 192), (192, 256)):
                assert out[i, lo:hi].tobytes() != proofs[i, lo:hi].tobytes(), (i, lo)
        mp, xs = mb_proofs
        mp = mp.copy()
        xs = xs.copy()
        xs[3, 2, 0] ^= 1                                             # one set element changed
        mp[40, 192:256] = mp[41, 192:256]
        mb_before = vkm.verify_batch(mp, xs)
        assert mb_before.sum() == mp.shape[0] - 2
        mout, mok = vkm.rerandomize(mp)
        assert mok.all()
        assert np.array_equal(vkm.verify_batch(mout, xs), mb_before)
    finally:
        vk.close()
        vkm.close()


def test_composition_on_the_device_at_65536(eq_keys, eq_proofs, frs):
    n = 65536
    proofs = np.tile(eq_proofs[0], (n // 300 + 1, 1))[:n].copy()
    r1, r2, s1, s2 = frs(7800, n), frs(7801, n), frs(7802, n), frs(7803, n)
    a1, a2, b1, b2 = _ints(r1), _ints(r2), _ints(s1), _ints(s2)
    t1 = _fr([x * y % R for x, y in zip(a1, b1)])
    t2 = _fr([(y + s * pow(x, -1, R)) % R for x, y, s in zip(a1, a2, b2)])
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        p1, ok1 = vk.rerandomize(proofs, r1, r2)
        p2, ok2 = vk.rerandomize(p1, s1, s2)
        once, ok3 = vk.rerandomize(proofs, t1, t2)
        assert ok1.all() and ok2.all() and ok3.all()
        assert np.array_equal(p2, once)
        cms = np.tile(eq_proofs[1], (n // 300 + 1, 1))[:n]
        assert vk.verify_batch(p2, cms).all()
    finally:
        vk.close()


def _device(vk, proofs, r1, r2, stream=None, in_place=False):
    import torch
    n = proofs.shape[0]
    d_p, d_r1, d_r2 = _cuda(proofs), _cuda(r1), _cuda(r2)
    d_out = d_p if in_place else torch.full((n, 256), 0x5A, dtype=torch.uint8, device="cuda")
    d_ok = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
    st = stream if stream is not None else torch.cuda.current_stream()
    vk.rerandomize_device(n, d_p.data_ptr(), d_r1.data_ptr(), d_r2.data_ptr(), d_out.data_ptr(), d_ok.data_ptr(), st.cuda_stream)
    torch.cuda.synchronize()
    return d_out.cpu().numpy(), d_ok.cpu().numpy().astype(bool)


def test_device_form_equals_host_form(eq_keys, eq_proofs, frs):
    proofs = eq_proofs[0].copy()
    proofs[7, 0] ^= 1                                                 # one malformed row
    n = proofs.shape[0]
    r1, r2 = frs(7900, n), frs(7901, n)
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        want, wok = vk.rerandomize(proofs, r1, r2)
        assert wok.sum() == n - 1
        for in_place in (False, True):
            got, gok = _device(vk, proofs, r1, r2, in_place=in_place)
            assert np.array_equal(got, want) and np.array_equal(gok, wok), in_place
        # the host form in place (proofs_out == proofs)
        buf = proofs.copy()
        ok = np.zeros(n, np.uint8)
        _ffi.check(_ffi.lib().lzkp_proofs_rerandomize(vk._h, n, engine._p(buf), engine._p(r1), engine._p(r2),
                                                      engine._p(buf), engine._p(ok)))
        assert np.array_equal(buf, want) and np.array_equal(ok.astype(bool), wok)
    finally:
        vk.close()


def test_prove_rerandomize_verify_on_one_stream(eq_keys, po, frs):
    import torch
    n = 96
    pk = engine.ProvingKey(eq_keys.pk_bytes, window_bits=WINDOW_BITS)
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        pk.circuit_builtin(engine.EQUALITY, 110)
        rng = po.SplitMix64(8000)
        a = np.array([rng.next_u64() for _ in range(n)], np.uint64)
        r, s = frs(8001, n), frs(8002, n)
        _, cms, _ = pk.prove_equality_batch(a, a, r, s)
        r1, r2 = frs(8003, n), frs(8004, n)
        d_a, d_r, d_s, d_x, d_r1, d_r2 = _cuda(a), _cuda(r), _cuda(s), _cuda(cms), _cuda(r1), _cuda(r2)
        d_p = torch.zeros((n, 256), dtype=torch.uint8, device="cuda")
        d_st = torch.zeros(n, dtype=torch.int32, device="cuda")
        d_q = torch.zeros((n, 256), dtype=torch.uint8, device="cuda")
        d_rok = torch.zeros(n, dtype=torch.uint8, device="cuda")
        d_ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        st = torch.cuda.Stream()
        h = st.cuda_stream
        pk.prove_equality_batch_device(n, d_a.data_ptr(), d_a.data_ptr(), d_r.data_ptr(), d_s.data_ptr(), d_p.data_ptr(),
                                       d_st.data_ptr(), h)
        vk.rerandomize_device(n, d_p.data_ptr(), d_r1.data_ptr(), d_r2.data_ptr(), d_q.data_ptr(), d_rok.data_ptr(), h)
        vk.verify_batch_device(n, d_q.data_ptr(), d_x.data_ptr(), 1, d_ok.data_ptr(), h)
        st.synchronize()
        assert not d_st.cpu().numpy().any() and d_rok.cpu().numpy().all() and d_ok.cpu().numpy().all()
        want, _ = vk.rerandomize(d_p.cpu().numpy(), r1, r2)
        assert np.array_equal(d_q.cpu().numpy(), want)
    finally:
        pk.close()
        vk.close()


def test_compressed_chain_matches_host_path(eq_keys, eq_proofs, frs):
    import torch
    proofs = eq_proofs[0][:64]
    n = proofs.shape[0]
    comp, cok = engine.proofs_compress(proofs)
    assert cok.all()
    r1, r2 = frs(8100, n), frs(8101, n)
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        dec, _ = engine.proofs_decompress(comp)
        rr, _ = vk.rerandomize(dec, r1, r2)
        want, _ = engine.proofs_compress(rr)
        d_c, d_r1, d_r2 = _cuda(comp), _cuda(r1), _cuda(r2)
        d_p = torch.zeros((n, 256), dtype=torch.uint8, device="cuda")
        d_c2 = torch.zeros((n, 128), dtype=torch.uint8, device="cuda")
        oks = [torch.zeros(n, dtype=torch.uint8, device="cuda") for _ in range(3)]
        torch.cuda.synchronize()
        st = torch.cuda.Stream()
        h = st.cuda_stream
        engine.proofs_decompress_device(n, d_c.data_ptr(), d_p.data_ptr(), oks[0].data_ptr(), h)
        vk.rerandomize_device(n, d_p.data_ptr(), d_r1.data_ptr(), d_r2.data_ptr(), d_p.data_ptr(), oks[1].data_ptr(), h)
        engine.proofs_compress_device(n, d_p.data_ptr(), d_c2.data_ptr(), oks[2].data_ptr(), h)
        st.synchronize()
        assert all(o.cpu().numpy().all() for o in oks)
        assert np.array_equal(d_c2.cpu().numpy(), want)
    finally:
        vk.close()


def test_graph_capture_replays(eq_keys, eq_proofs, frs):
    import torch
    proofs = eq_proofs[0][:128]
    n = proofs.shape[0]
    r1, r2 = frs(8200, n), frs(8201, n)
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        want, _ = vk.rerandomize(proofs, r1, r2)
        d_p, d_r1, d_r2 = _cuda(proofs), _cuda(r1), _cuda(r2)
        d_out = torch.zeros((n, 256), dtype=torch.uint8, device="cuda")
        d_ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            g.capture_begin()
            vk.rerandomize_device(n, d_p.data_ptr(), d_r1.data_ptr(), d_r2.data_ptr(), d_out.data_ptr(), d_ok.data_ptr(),
                                  st.cuda_stream)
            g.capture_end()
        for _ in range(2):
            d_out.zero_()
            d_ok.zero_()
            g.replay()
            torch.cuda.synchronize()
            assert np.array_equal(d_out.cpu().numpy(), want) and d_ok.cpu().numpy().all()
    finally:
        vk.close()


def test_two_streams_on_one_key(eq_keys, eq_proofs, frs):
    import torch
    proofs, cms = eq_proofs
    n = proofs.shape[0]
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        bufs = []
        for k in range(2):
            r1, r2 = frs(8300 + k, n), frs(8310 + k, n)
            want, _ = vk.rerandomize(proofs, r1, r2)
            bufs.append((want, _cuda(proofs), _cuda(r1), _cuda(r2), torch.zeros((n, 256), dtype=torch.uint8, device="cuda"),
                         torch.zeros(n, dtype=torch.uint8, device="cuda"), torch.zeros(n, dtype=torch.uint8, device="cuda")))
        d_x = _cuda(cms)
        torch.cuda.synchronize()
        streams = [torch.cuda.Stream(), torch.cuda.Stream()]
        for (want, d_p, d_r1, d_r2, d_out, d_rok, d_ok), st in zip(bufs, streams):
            vk.rerandomize_device(n, d_p.data_ptr(), d_r1.data_ptr(), d_r2.data_ptr(), d_out.data_ptr(), d_rok.data_ptr(),
                                  st.cuda_stream)
            vk.verify_batch_device(n, d_out.data_ptr(), d_x.data_ptr(), 1, d_ok.data_ptr(), st.cuda_stream)
        torch.cuda.synchronize()
        for want, _, _, _, d_out, d_rok, d_ok in bufs:
            assert np.array_equal(d_out.cpu().numpy(), want)
            assert d_rok.cpu().numpy().all() and d_ok.cpu().numpy().all()
    finally:
        vk.close()


def test_arguments(eq_keys):
    import torch
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        p = torch.zeros(512, dtype=torch.uint8, device="cuda")
        f = torch.zeros(64, dtype=torch.uint8, device="cuda")
        ok = torch.zeros(2, dtype=torch.uint8, device="cuda")
        host = np.zeros(512, np.uint8)
        P, F, O = p.data_ptr(), f.data_ptr(), ok.data_ptr()
        bad = [
            (None, F, F, P, O), (P, None, F, P, O), (P, F, None, P, O), (P, F, F, None, O), (P, F, F, P, None),
            (host.ctypes.data, F, F, P, O), (P, F, F, host.ctypes.data, O),
            (P + 8, F, F, P, O), (P, F + 4, F, P, O), (P, F, F, P + 1, O),
        ]
        for args in bad:
            with pytest.raises(EngineError) as e:
                vk.rerandomize_device(1, *args)
            assert e.value.code == _ffi.LZKP_E_INVALID, args
        launches = engine.kernel_launches()
        vk.rerandomize_device(0, 0, 0, 0, 0, 0)                       # n == 0: nothing enqueued
        assert engine.kernel_launches() == launches
        out, oks = vk.rerandomize(np.zeros((0, 256), np.uint8))
        assert out.shape == (0, 256) and oks.shape == (0,)
        if torch.cuda.device_count() > 1:
            with torch.cuda.device(1):
                other = torch.zeros(512, dtype=torch.uint8, device="cuda:1")
            with pytest.raises(EngineError) as e:
                vk.rerandomize_device(1, other.data_ptr(), F, F, P, O)
            assert e.value.code == _ffi.LZKP_E_INVALID
    finally:
        vk.close()


def test_drawn_factors_are_fresh(eq_keys, eq_proofs):
    proofs, cms = eq_proofs
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        a, oka = vk.rerandomize(proofs[:32])
        b, okb = vk.rerandomize(proofs[:32])
        assert oka.all() and okb.all()
        assert not (a == b).all(axis=1).any()
        assert vk.verify_batch(a, cms[:32]).all() and vk.verify_batch(b, cms[:32]).all()
    finally:
        vk.close()
