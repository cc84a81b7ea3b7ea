"""lzkp_verify_batch_device: verification of proofs already in device memory, asynchronous on the caller's stream.  Its
decisions are those of lzkp_verify_batch on the same bytes in every form (latency, lane per proof, combined with the
failing groups re-verified on the device), it returns before the device has run it, calls on one key from several
streams share the key's scratch safely, and bad arguments are refused without a crash."""
import numpy as np
import pytest

from libzkp_b200 import _ffi, engine
from libzkp_b200.errors import EngineError

pytestmark = pytest.mark.gpu
WINDOW_BITS = 10
# an all-valid combined-form call of a key with at most 256 inputs, at the default thresholds with n > 444: k_rlc_rho,
# the per-proof kernel, scalar sums, input shares, combined check, k_rlc_failed, then the three gated re-verifying forms
# (latency form at one and at two CTAs per SM, one proof per lane) whose CTAs all leave
COMBINED_DEVICE_LAUNCHES = 9


def _forms(monkeypatch, form):
    """Environment that forces one form at small sizes (as test_gpu_verify.py does)."""
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


class Dev:
    """A batch uploaded to the device: proofs, inputs and an ok buffer, as torch tensors."""

    def __init__(self, proofs, x):
        import torch
        self.n = len(proofs)
        self.p = torch.from_numpy(np.ascontiguousarray(proofs)).cuda()
        self.x = torch.from_numpy(np.ascontiguousarray(x).reshape(self.n, -1)).cuda()
        self.n_pub = self.x.shape[1] // 32
        self.ok = torch.full((self.n,), 7, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()

    def enqueue(self, vk, stream=None):
        import torch
        st = stream if stream is not None else torch.cuda.current_stream()
        vk.verify_batch_device(self.n, self.p.data_ptr(), self.x.data_ptr(), self.n_pub, self.ok.data_ptr(), st.cuda_stream)

    def result(self):
        import torch
        torch.cuda.synchronize()
        ok = self.ok.cpu().numpy()
        assert set(np.unique(ok)) <= {0, 1}, np.unique(ok)              # every entry written
        return ok.astype(bool)


def dev_verify(vk, proofs, x, stream=None):
    d = Dev(proofs, x)
    d.enqueue(vk, stream)
    return d.result()


@pytest.fixture(scope="module")
def eq_batch(eq_keys, po, frs):
    """4096 valid equality proofs and their commitments."""
    pk = engine.ProvingKey(eq_keys.pk_bytes, window_bits=WINDOW_BITS)
    try:
        pk.circuit_builtin(engine.EQUALITY, 110)
        n = 4096
        rng = po.SplitMix64(4242)
        a = np.array([rng.next_u64() for _ in range(n)], np.uint64)
        proofs, cms, st = pk.prove_equality_batch(a, a, frs(4243, n), frs(4244, n))
    finally:
        pk.close()
    assert not st.any()
    return proofs, cms


@pytest.fixture(scope="module")
def eq_vk(eq_keys):
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    yield vk
    vk.close()


def _g1(po, b):
    return po.g1_from_bytes(bytes(b), False)


def _g1_bytes(po, P):
    return np.frombuffer(po.g1_to_bytes(P), np.uint8)


def _fr_bytes(v):
    return np.frombuffer(int(v).to_bytes(32, "little"), np.uint8)


def test_form_boundaries(eq_batch, eq_vk, mb_keys, co, po, frs, monkeypatch):
    # 1 / 148: latency form at one CTA per SM;  149 / 444: two per SM;  445 / 4096: combined form
    _forms(monkeypatch, "default")
    proofs, cms = eq_batch
    for m in (1, 148, 149, 444, 445, 4096):
        got = dev_verify(eq_vk, proofs[:m], cms[:m])
        assert got.all(), (m, np.flatnonzero(~got)[:8])
        assert np.array_equal(got, eq_vk.verify_batch(proofs[:m], cms[:m])), m
    pkm = engine.ProvingKey(mb_keys.pk_bytes, window_bits=8)
    try:
        pkm.circuit_builtin(engine.MEMBERSHIP, 64)
        m = 445
        rng = po.SplitMix64(4300)
        sets = np.zeros((m, 64), np.uint64)
        lens = (1 + (np.arange(m) * 5) % 64).astype(np.uint32)
        for i in range(m):
            sets[i, :lens[i]] = [rng.next_u64() for _ in range(lens[i])]
        vals = sets[np.arange(m), np.arange(m) % lens]
        mp, mcm, mst = pkm.prove_membership_batch(vals, sets, lens, frs(4301, m), frs(4302, m))
    finally:
        pkm.close()
    assert not mst.any()
    xs = np.zeros((m, 129, 32), np.uint8)
    for i in range(m):
        xs[i] = co.fr_array(po.membership_public_inputs(int.from_bytes(mcm[i].tobytes(), "little"),
                                                        [int(v) for v in sets[i, :lens[i]]]))
    vkm = engine.VerifyingKey(mb_keys.vk_bytes)
    try:
        for k in (1, 445):
            got = dev_verify(vkm, mp[:k], xs[:k])
            assert got.all() and np.array_equal(got, vkm.verify_batch(mp[:k], xs[:k])), k
        xs[300, 2, 0] ^= 1                                                   # one set element changed
        want = np.ones(m, bool)
        want[300] = False
        assert np.array_equal(dev_verify(vkm, mp, xs), want)
    finally:
        vkm.close()


def _mixed_cases(proofs, cms, po):
    """(name, proofs, inputs, expected) over five groups of 64, the last one partial."""
    n = 64 * 4 + 21
    p, x = proofs[:n], cms[:n]
    bad, xb = p.copy(), x.copy()
    bad[3, 5] ^= 1                                                           # off-curve A                 (group 0)
    bad[70, 192:256] = p[71, 192:256]                                        # a valid point, wrong C      (group 1)
    xb[200] = x[201]                                                         # wrong public input          (group 3)
    bad[270, 64:192] = np.frombuffer(po.g2_to_bytes(po.G2.mul(po.G2_GEN, 5)), np.uint8)    # wrong B   (group 4)
    want = np.ones(n, bool)
    want[[3, 70, 200, 270]] = False
    malformed = p.copy()
    malformed[130:140, 0] ^= 1                                               # malformed rows only (group 2)
    wm = np.ones(n, bool)
    wm[130:140] = False
    return [("mixed", bad, xb, want), ("malformed_only", malformed, x, wm),
            ("all_false", p, np.roll(x, 1, axis=0), np.zeros(n, bool))]


@pytest.mark.parametrize("form", ["latency", "lanes", "combined"])
def test_mixed_bad_proofs_in_every_form(eq_batch, eq_vk, po, form, monkeypatch):
    _forms(monkeypatch, form)
    proofs, cms = eq_batch
    for name, p, x, want in _mixed_cases(proofs, cms, po):
        host = eq_vk.verify_batch(p, x)
        dev = dev_verify(eq_vk, p, x)
        assert np.array_equal(host, want), (name, np.flatnonzero(host != want))
        assert np.array_equal(dev, host), (name, np.flatnonzero(dev != host))


def _cancelling(proofs, cms, po):
    """Forgeries whose errors cancel in an UNWEIGHTED sum, all inside group 0."""
    n = 64 * 4 + 21
    bad, x = proofs[:n].copy(), cms[:n].copy()
    D = po.G1.mul(po.G1_GEN, 7)
    C = _g1(po, proofs[20, 192:256])
    bad[20, 192:256] = _g1_bytes(po, po.G1.add(C, D))                        # (A, B, C + D)
    bad[21] = bad[20]
    bad[21, 192:256] = _g1_bytes(po, po.G1.add(C, po.G1.neg(D)))             # (A, B, C - D), the same input
    x[21] = x[20]
    x[30] = _fr_bytes((int.from_bytes(cms[30].tobytes(), "little") + 1) % po.R_MOD)    # input raised by 1 ...
    x[31] = _fr_bytes((int.from_bytes(cms[31].tobytes(), "little") - 1) % po.R_MOD)    # ... and lowered by 1
    want = np.ones(n, bool)
    want[[20, 21, 30, 31]] = False
    return bad, x, want


@pytest.mark.parametrize("coop_max, failing_groups", [
    (None, [0]),             # F = 64: latency form, one CTA per SM
    (None, [0, 1, 3]),       # F = 192: latency form, two CTAs per SM
    ("32", [0]),             # F = 64 > coop_max: one proof per lane
    ("32", [0, 1, 2, 3, 4]),  # every group fails
])
def test_both_reverification_regimes(eq_batch, eq_vk, po, coop_max, failing_groups, monkeypatch):
    _forms(monkeypatch, "combined")
    if coop_max:
        monkeypatch.setenv("LZKP_VERIFY_COOP_MAX", coop_max)
    proofs, cms = eq_batch
    bad, x, want = _cancelling(proofs, cms, po)
    for g in failing_groups[1:]:
        k = 64 * g + 5
        x[k] = cms[k + 1]                                                    # wrong public input in group g
        want[k] = False
    host = eq_vk.verify_batch(bad, x)
    dev = dev_verify(eq_vk, bad, x)
    assert np.array_equal(host, want), np.flatnonzero(host != want)
    assert np.array_equal(dev, want), np.flatnonzero(dev != want)


def test_key_above_256_inputs(po, trapdoor, frs, monkeypatch):
    from test_gpu_verify_many_inputs import _squares_key_and_proofs
    n_in, n = 300, 150
    vk_bytes, proofs, x = _squares_key_and_proofs(po, trapdoor, frs, n_in, n, 3000)
    bad, xs = proofs.copy(), x.copy()
    xs[5, 17] = x[6, 17]                                                     # one input of another proof  (group 0)
    bad[100, 192:256] = proofs[101, 192:256]                                 # wrong C                      (group 1)
    xs[140, n_in - 1, 0] ^= 1                                                # the last input               (group 2)
    want = np.ones(n, bool)
    want[[5, 100, 140]] = False
    vk = engine.VerifyingKey(vk_bytes)
    try:
        for form, coop_max in (("latency", None), ("combined", None), ("combined", "32")):
            _forms(monkeypatch, form)
            if coop_max:
                monkeypatch.setenv("LZKP_VERIFY_COOP_MAX", coop_max)
            host = vk.verify_batch(bad, xs)
            assert np.array_equal(host, want), (form, coop_max, np.flatnonzero(host != want))
            assert np.array_equal(dev_verify(vk, bad, xs), want), (form, coop_max)
            assert dev_verify(vk, proofs, x).all(), (form, coop_max)
        # launches: the latency form runs k_vkx<false> first; the combined form lists with k_vkx<true> before its re-verification
        _forms(monkeypatch, "latency")
        d = Dev(proofs[:3], x[:3])
        before = engine.kernel_launches()
        d.enqueue(vk)
        assert engine.kernel_launches() - before == 2 and d.result().all()
        _forms(monkeypatch, "combined")
        d = Dev(proofs, x)
        before = engine.kernel_launches()
        d.enqueue(vk)
        # rho, per-proof kernel, input sums, input shares, combined check, k_rlc_failed, k_vkx<true>, two latency forms
        assert engine.kernel_launches() - before == 9 and d.result().all()
    finally:
        vk.close()


def test_prove_then_verify_without_the_host(eq_keys, eq_vk, po, frs, monkeypatch):
    import torch
    _forms(monkeypatch, "default")
    pk = engine.ProvingKey(eq_keys.pk_bytes, window_bits=WINDOW_BITS)
    try:
        pk.circuit_builtin(engine.EQUALITY, 110)
        n = 600
        rng = po.SplitMix64(4400)
        a = np.array([rng.next_u64() for _ in range(n)], np.uint64)
        b = a.copy()
        b[[7, 300, 599]] += np.uint64(1)                                     # a != b: status 1, no proof
        cms = np.stack([np.frombuffer(engine.commit_value_snark(int(v)), np.uint8) for v in a])
        d_a = torch.from_numpy(a.view(np.int64)).cuda()
        d_b = torch.from_numpy(b.view(np.int64)).cuda()
        d_r, d_s = torch.from_numpy(frs(4401, n)).cuda(), torch.from_numpy(frs(4402, n)).cuda()
        d_x = torch.from_numpy(cms).cuda()
        d_p = torch.zeros((n, 256), dtype=torch.uint8, device="cuda")
        d_st = torch.zeros(n, dtype=torch.int32, device="cuda")
        d_ok = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        s = torch.cuda.Stream()
        pk.prove_equality_batch_device(n, d_a.data_ptr(), d_b.data_ptr(), d_r.data_ptr(), d_s.data_ptr(), d_p.data_ptr(),
                                       d_st.data_ptr(), s.cuda_stream)
        eq_vk.verify_batch_device(n, d_p.data_ptr(), d_x.data_ptr(), 1, d_ok.data_ptr(), s.cuda_stream)
        s.synchronize()
        status, ok = d_st.cpu().numpy(), d_ok.cpu().numpy()
    finally:
        pk.close()
    assert np.flatnonzero(status).tolist() == [7, 300, 599]
    assert ok[status == 0].all() and set(np.unique(ok)) <= {0, 1}


def test_the_call_does_not_block(eq_batch, eq_vk, po, monkeypatch):
    import torch
    _forms(monkeypatch, "default")
    proofs, cms = eq_batch
    m = 1000
    x = cms[:m].copy()
    x[500] = cms[501]                                                        # one failing group: the device fallback runs
    want = np.ones(m, bool)
    want[500] = False
    d = Dev(proofs[:m], x)
    s = torch.cuda.Stream()
    d.enqueue(eq_vk, s)                                                      # warm-up: the key's scratch holds this size
    assert np.array_equal(d.result(), want)
    d.ok.fill_(7)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)                                       # about 0.1 s
    d.enqueue(eq_vk, s)
    assert not s.query()                                                     # returned while the sleep still runs
    s.synchronize()
    assert np.array_equal(d.result(), want)


def test_shared_scratch_across_streams_and_the_host_call(eq_batch, eq_vk, po, monkeypatch):
    import torch
    _forms(monkeypatch, "default")
    proofs, cms = eq_batch
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    jobs = []
    for k in range(4):
        m = 600 + 200 * k
        x = cms[:m].copy()
        want = np.ones(m, bool)
        for i in range(k + 1):                                               # a different failing set per call
            j = (97 * (k + 1) * (i + 1)) % m
            x[j] = cms[(j + 1) % m]
            want[j] = False
        jobs.append((Dev(proofs[:m], x), want))
    with torch.cuda.stream(streams[0]):
        torch.cuda._sleep(100_000_000)                                       # keep the first calls in flight
    for k, (d, _) in enumerate(jobs):
        d.enqueue(eq_vk, streams[k & 1])
    hx = cms[:700].copy()                                                    # a host-buffer call on the same key meanwhile
    hx[[3, 650]] = cms[[4, 651]]
    hw = np.ones(700, bool)
    hw[[3, 650]] = False
    assert np.array_equal(eq_vk.verify_batch(proofs[:700], hx), hw)
    for k, (d, want) in enumerate(jobs):
        got = d.result()
        assert np.array_equal(got, want), (k, np.flatnonzero(got != want))


def test_argument_checks(eq_batch, eq_vk, monkeypatch):
    import torch
    _forms(monkeypatch, "default")
    proofs, cms = eq_batch
    d = Dev(proofs[:8], cms[:8])
    st = torch.cuda.current_stream().cuda_stream
    host = np.zeros((8, 256), np.uint8)
    bad_calls = [
        (host.ctypes.data, d.x.data_ptr(), d.ok.data_ptr()),                 # host memory
        (d.p.data_ptr(), host.ctypes.data, d.ok.data_ptr()),
        (d.p.data_ptr(), d.x.data_ptr(), host.ctypes.data),
        (d.p.data_ptr() + 1, d.x.data_ptr(), d.ok.data_ptr()),               # not 16-byte aligned
        (d.p.data_ptr(), d.x.data_ptr() + 1, d.ok.data_ptr()),
        (None, d.x.data_ptr(), d.ok.data_ptr()),                             # null
        (d.p.data_ptr(), None, d.ok.data_ptr()),
        (d.p.data_ptr(), d.x.data_ptr(), None),
    ]
    for k, (p, x, ok) in enumerate(bad_calls):
        with pytest.raises(EngineError) as e:
            eq_vk.verify_batch_device(8, p, x, 1, ok, st)
        assert e.value.code == _ffi.LZKP_E_INVALID, k
    # the wrong number of inputs: every proof rejected
    d.ok.fill_(1)
    eq_vk.verify_batch_device(8, d.p.data_ptr(), d.x.data_ptr(), 2, d.ok.data_ptr(), st)
    assert not d.result().any()
    # n = 0: nothing launched, null buffers allowed
    before = engine.kernel_launches()
    eq_vk.verify_batch_device(0, None, None, 1, None, st)
    assert engine.kernel_launches() == before
    # a capturing stream is refused and the capture still ends cleanly
    g = torch.cuda.CUDAGraph()
    t = torch.zeros(4, device="cuda")
    torch.cuda.synchronize()
    launches = engine.kernel_launches()
    with torch.cuda.graph(g):
        t.add_(1)
        with pytest.raises(EngineError) as e:
            d.enqueue(eq_vk)
    assert e.value.code == _ffi.LZKP_E_UNSUPPORTED
    assert engine.kernel_launches() == launches
    g.replay()
    torch.cuda.synchronize()
    assert t.tolist() == [1, 1, 1, 1]
    d.enqueue(eq_vk)                                                         # the key still works
    assert d.result().all()


def test_launch_counts(eq_batch, eq_vk, monkeypatch):
    _forms(monkeypatch, "default")
    proofs, cms = eq_batch
    d = Dev(proofs[:445], cms[:445])
    d.enqueue(eq_vk)                                                         # scratch grown once
    d.result()
    before = engine.kernel_launches()
    d.enqueue(eq_vk)
    assert engine.kernel_launches() - before == COMBINED_DEVICE_LAUNCHES
    assert d.result().all()
    d = Dev(proofs[:64], cms[:64])
    before = engine.kernel_launches()
    d.enqueue(eq_vk)
    device = engine.kernel_launches() - before
    assert d.result().all()
    before = engine.kernel_launches()
    assert eq_vk.verify_batch(proofs[:64], cms[:64]).all()
    assert device == engine.kernel_launches() - before == 1
