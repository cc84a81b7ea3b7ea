"""Verification of keys with more than 256 public inputs: membership with a 1024-slot set (2049 inputs), dense custom
circuits and the 256 / 257 boundary.  Such keys get the latency form and the combined form like small keys; vk_x of each
proof comes from k_vkx, the combined form's scalar sums from k_rlc_input_sums."""
import numpy as np
import pytest

from libzkp_b200 import engine

pytestmark = pytest.mark.gpu

SLOTS = 1024
N_PUB = 1 + 2 * SLOTS
TABLE_ROW_BYTES = 32 * 255 * 64            # byte windows of one table row: 32 windows x 255 digits x affine G1


def _membership_inputs(cms, sets, lens):
    """(n, 2049, 32) canonical inputs [commitment, set[1024], is_real[1024]] (po.membership_public_inputs layout)."""
    n = len(lens)
    x = np.zeros((n, N_PUB, 32), np.uint8)
    x[:, 0] = cms
    x[:, 1:1 + SLOTS, :8] = np.ascontiguousarray(sets, "<u8").view(np.uint8).reshape(n, SLOTS, 8)
    x[:, 1 + SLOTS:, 0] = np.arange(SLOTS)[None, :] < lens[:, None]
    return x


@pytest.fixture(scope="module")
def m1024(trapdoor, frs, po, co):
    """Membership-1024 key, 4096 valid proofs over sets of lengths 1 .. 1024, and their public inputs."""
    pk_bytes, vk_bytes = engine.setup_builtin(engine.MEMBERSHIP, SLOTS, trapdoor)
    n = 4096
    rng = np.random.default_rng(1024)
    lens = (1 + (np.arange(n) * 37) % SLOTS).astype(np.uint32)
    lens[:4] = [1, SLOTS, 2, SLOTS - 1]
    sets = rng.integers(0, 2**64, size=(n, SLOTS), dtype=np.uint64)
    sets[np.arange(SLOTS)[None, :] >= lens[:, None]] = 0
    vals = sets[np.arange(n), np.arange(n) % lens]
    pk = engine.ProvingKey(pk_bytes, window_bits=8)
    try:
        pk.circuit_builtin(engine.MEMBERSHIP, SLOTS)
        proofs, cms, status = pk.prove_membership_batch(vals, sets, lens, frs(1101, n), frs(1102, n))
    finally:
        pk.close()
    assert not status.any()
    x = _membership_inputs(cms, sets, lens)
    for i in (0, 1, 777):                                                    # the layout is the oracle's
        pub = po.membership_public_inputs(int.from_bytes(cms[i].tobytes(), "little"),
                                          [int(v) for v in sets[i, :lens[i]]], slots=SLOTS)
        assert np.array_equal(x[i], co.fr_array(pub)), i
    return vk_bytes, proofs, x, sets, lens


def _three_forms(vk, proofs, x, monkeypatch):
    """Decisions of the latency form, the lane-per-proof form and the combined form (failing groups re-verified one
    proof per lane)."""
    out = {}
    monkeypatch.setenv("LZKP_VERIFY_RLC_MIN", "1000000000")
    monkeypatch.setenv("LZKP_VERIFY_COOP_MAX", "100000")
    out["latency"] = vk.verify_batch(proofs, x)
    monkeypatch.setenv("LZKP_VERIFY_COOP_MAX", "0")
    out["lanes"] = vk.verify_batch(proofs, x)
    monkeypatch.setenv("LZKP_VERIFY_RLC_MIN", "1")
    out["combined"] = vk.verify_batch(proofs, x)
    for k in ("LZKP_VERIFY_RLC_MIN", "LZKP_VERIFY_COOP_MAX"):
        monkeypatch.delenv(k)
    return out


def _g1(po, b):
    return po.g1_from_bytes(bytes(b), False)


def _g1_bytes(po, P):
    return np.frombuffer(po.g1_to_bytes(P), np.uint8)


def test_valid_proofs_verify_at_every_form_boundary(m1024, monkeypatch):
    # 1 / 64 / 148: latency form, one CTA per SM;  149 / 444: two per SM;  445 / 4096: combined form
    vk_bytes, proofs, x, _, _ = m1024
    monkeypatch.delenv("LZKP_VERIFY_RLC_MIN", raising=False)
    monkeypatch.delenv("LZKP_VERIFY_COOP_MAX", raising=False)
    vk = engine.VerifyingKey(vk_bytes)
    try:
        for m in (1, 64, 148, 149, 444, 445, 4096):
            ok = vk.verify_batch(proofs[:m], x[:m])
            assert ok.all(), (m, np.flatnonzero(~ok)[:8])
        assert vk.verify_batch(proofs[-300:], x[-300:]).all()              # sets of every length, other offsets
    finally:
        vk.close()


def test_malformed_and_forged_proofs_in_three_forms(m1024, po, monkeypatch):
    vk_bytes, proofs, x, sets, lens = m1024
    n = 128                                                                # two groups of 64; group 1 clean
    bad, xs = proofs[:n].copy(), x[:n].copy()
    bad[1, 5] ^= 1                                                         # A off the curve
    bad[2, 192:256] = proofs[3, 192:256]                                   # a valid point, wrong C
    bad[4, 64:192] = np.frombuffer(po.g2_to_bytes(po.G2.mul(po.G2_GEN, 5)), np.uint8)     # wrong B
    assert lens[5] >= 1
    xs[5, 1, 0] ^= 1                                                       # first set value changed
    assert lens[6] < SLOTS
    xs[6, 1 + SLOTS + SLOTS - 1, 0] ^= 1                                   # is_real of an empty slot set to 1
    xs[7, 0] = x[8, 0]                                                     # wrong commitment
    xs[9, 1 + 1] = 0xFF                                                    # non-canonical set value (> r)
    v = int.from_bytes(xs[10, 1].tobytes(), "little") + po.R_MOD           # the same value mod r, not canonical
    xs[10, 1] = np.frombuffer(v.to_bytes(32, "little"), np.uint8)
    want = np.ones(n, bool)
    want[[1, 2, 4, 5, 6, 7, 9, 10]] = False
    # the oracle's pairing verifier on a sample (about 10 s per proof at 2049 inputs on a CPU): A off the curve fails to
    # deserialize; the valid proof, the wrong C, the flipped is_real bit and the wrong commitment go through the pairing
    ovk = po.vk_from_bytes(vk_bytes)
    with pytest.raises(ValueError):
        po.proof_from_bytes(bad[1].tobytes())
    for k in (0, 2, 6, 7):
        o = po.verify(ovk, [int.from_bytes(xs[k, j].tobytes(), "little") for j in range(N_PUB)],
                      po.proof_from_bytes(bad[k].tobytes()))
        assert bool(o) == bool(want[k]), k
    vk = engine.VerifyingKey(vk_bytes)
    try:
        for form, got in _three_forms(vk, bad, xs, monkeypatch).items():
            assert np.array_equal(got, want), (form, np.flatnonzero(got != want))
        # the wrong number of inputs rejects every proof, as for other keys
        assert not vk.verify_batch(proofs[:8], x[:8, :N_PUB - 1]).any()
    finally:
        vk.close()


def test_cancelling_forgeries_inside_one_group(m1024, po, monkeypatch):
    # Pairs of false proofs whose errors cancel in an UNWEIGHTED sum; with random weights the group's combined check
    # fails and both proofs of every pair are rejected on re-verification.
    vk_bytes, proofs, x, sets, lens = m1024
    n = 64
    bad, xs = proofs[:n].copy(), x[:n].copy()
    D = po.G1.mul(po.G1_GEN, 7)
    C = _g1(po, proofs[20, 192:256])
    bad[20, 192:256] = _g1_bytes(po, po.G1.add(C, D))                      # (A, B, C + D)
    bad[21, :] = proofs[20]
    bad[21, 192:256] = _g1_bytes(po, po.G1.add(C, po.G1.neg(D)))           # (A, B, C - D), same inputs as proof 20
    xs[21] = x[20]
    j = 1 + 3                                                              # set slot 3 of proofs 30 and 31
    assert lens[30] > 3 and lens[31] > 3 and 0 < sets[30, 3] < 2**64 - 1 and sets[31, 3] > 0
    xs[30, j, :8] = np.frombuffer(np.uint64(int(sets[30, 3]) + 1).tobytes(), np.uint8)    # input j raised by 1 ...
    xs[31, j, :8] = np.frombuffer(np.uint64(int(sets[31, 3]) - 1).tobytes(), np.uint8)    # ... and lowered by 1
    want = np.ones(n, bool)
    want[[20, 21, 30, 31]] = False
    vk = engine.VerifyingKey(vk_bytes)
    try:
        monkeypatch.setenv("LZKP_VERIFY_RLC_MIN", "64")
        assert np.array_equal(vk.verify_batch(bad, xs), want)
    finally:
        vk.close()


def test_key_without_tables_verifies_one_proof_per_lane(m1024):
    # A key whose 1.07 GB of tables cannot be allocated still loads: a torch allocation holds all but 512 MB of the
    # device's free memory while it does.  Every call then runs k_verify4 with its own scalar multiplications.
    import torch
    vk_bytes, proofs, x, _, _ = m1024
    free, _ = torch.cuda.mem_get_info()
    hold = torch.empty(free - (512 << 20), dtype=torch.uint8, device="cuda")
    try:
        vk = engine.VerifyingKey(vk_bytes)
    finally:
        del hold
        torch.cuda.empty_cache()
    try:
        assert vk.info() == (N_PUB, 0, False, False)
        xs = x[:3].copy()
        xs[1, 1, 0] ^= 1                                                   # one set value changed
        xs[2, 2] = 0xFF                                                    # non-canonical input
        before = engine.kernel_launches()
        assert vk.verify_batch(proofs[:3], xs).tolist() == [True, False, False]
        assert engine.kernel_launches() - before == 1                      # k_verify4 alone
    finally:
        vk.close()


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    return [e.name for e in prof.events() if e.device_type.name == "CUDA"]


def test_launches_of_the_two_fast_forms(m1024, monkeypatch):
    vk_bytes, proofs, x, _, _ = m1024
    monkeypatch.delenv("LZKP_VERIFY_RLC_MIN", raising=False)
    monkeypatch.delenv("LZKP_VERIFY_COOP_MAX", raising=False)
    vk = engine.VerifyingKey(vk_bytes)
    try:
        vk.verify_batch(proofs[:1], x[:1])                                 # staging buffers grown once
        before = engine.kernel_launches()
        assert vk.verify_batch(proofs[:445], x[:445]).all()
        assert engine.kernel_launches() - before == 4                      # per-proof kernel, input sums, input shares, combined check
        before = engine.kernel_launches()
        assert vk.verify_batch(proofs[:1], x[:1]).all()
        assert engine.kernel_launches() - before == 2                      # k_vkx, then the latency form
        names = _kernel_names(lambda: vk.verify_batch(proofs[:1], x[:1]))
        assert any("k_vkx" in s for s in names) and any("k_verify_coop" in s for s in names), names
        assert not any("k_verify4" in s for s in names), names
    finally:
        vk.close()


def _squares(po, n_in, seed):
    """x_i * x_i = w_i: n_in full-width public inputs, n_in witnesses, n_in constraints."""
    cs = po.ConstraintSystem()
    rng = po.SplitMix64(seed)
    for _ in range(n_in):
        v = rng.next_fr()
        x = cs.new_input(v)
        w = cs.new_witness(v * v)
        cs.enforce(x.lc, x.lc, w.lc)
    return cs


def _csr(po, rows):
    rowptr, col, val = [0], [], []
    for row in rows:
        for v, c in row:
            col.append(c)
            val.append(np.frombuffer((v % po.R_MOD).to_bytes(32, "little"), np.uint8))
        rowptr.append(len(col))
    return (np.array(rowptr, np.uint32), np.array(col, np.uint32),
            np.stack(val) if val else np.zeros((0, 32), np.uint8))


def _squares_key_and_proofs(po, trapdoor, frs, n_in, n, seed, check_oracle=False):
    cs = _squares(po, n_in, seed)
    A, B, C = cs.matrices()
    ni, nw = cs.num_instance(), cs.num_witness()
    mats = [_csr(po, M) for M in (A, B, C)]
    pk_bytes, vk_bytes = engine.setup(len(A), ni, nw, mats, trapdoor)
    if check_oracle:
        opk = po.setup(cs, po.Trapdoor(*trapdoor))
        assert pk_bytes == po.pk_to_bytes(opk) and vk_bytes == po.vk_to_bytes(opk.vk)
    rng = po.SplitMix64(seed + 1)
    xs = [[rng.next_fr() for _ in range(n_in)] for _ in range(n)]
    z = np.stack([np.frombuffer(b"".join(v.to_bytes(32, "little") for v in [1] + xi + [a * a % po.R_MOD for a in xi]),
                                np.uint8) for xi in xs])
    pk = engine.ProvingKey(pk_bytes, window_bits=8)
    try:
        pk.circuit_load(len(A), ni, nw, mats)
        proofs, status = pk.prove_batch(z, frs(seed + 2, n), frs(seed + 3, n))
    finally:
        pk.close()
    assert not status.any()
    x = z[:, 32:32 * ni].reshape(n, n_in, 32).copy()
    return vk_bytes, proofs, x


def test_dense_custom_circuit_three_forms(po, trapdoor, frs, monkeypatch):
    n_in, n = 600, 460
    vk_bytes, proofs, x = _squares_key_and_proofs(po, trapdoor, frs, n_in, n, 600, check_oracle=True)
    vk = engine.VerifyingKey(vk_bytes)
    try:
        assert vk.info()[0] == n_in and vk.info()[2] and vk.info()[3]
        monkeypatch.delenv("LZKP_VERIFY_RLC_MIN", raising=False)
        monkeypatch.delenv("LZKP_VERIFY_COOP_MAX", raising=False)
        assert vk.verify_batch(proofs, x).all()                            # combined form
        assert vk.verify_batch(proofs[:200], x[:200]).all()                # latency form
        bad, xs = proofs.copy(), x.copy()
        xs[3, 10] = x[4, 10]                                               # one input of another proof
        xs[70, n_in - 1, 0] ^= 1                                           # the last input
        bad[130, 192:256] = proofs[131, 192:256]                           # wrong C
        bad[200, 0:64] = proofs[201, 0:64]                                 # wrong A
        want = np.ones(n, bool)
        want[[3, 70, 130, 200]] = False
        for form, got in _three_forms(vk, bad, xs, monkeypatch).items():
            assert np.array_equal(got, want), (form, np.flatnonzero(got != want))
    finally:
        vk.close()


@pytest.mark.parametrize("n_in, launches", [(256, 1), (257, 2)])
def test_boundary_keys(po, trapdoor, frs, n_in, launches, monkeypatch):
    # 256 inputs: the latency form's own scan of the tables (one launch); 257: k_vkx first
    vk_bytes, proofs, x = _squares_key_and_proofs(po, trapdoor, frs, n_in, 3, 256 + n_in)
    monkeypatch.delenv("LZKP_VERIFY_RLC_MIN", raising=False)
    monkeypatch.delenv("LZKP_VERIFY_COOP_MAX", raising=False)
    vk = engine.VerifyingKey(vk_bytes)
    try:
        assert vk.info() == (n_in, (n_in + 2) * TABLE_ROW_BYTES, True, True)
        assert vk.verify_batch(proofs, x).all()
        before = engine.kernel_launches()
        assert vk.verify_batch(proofs[:1], x[:1]).all()
        assert engine.kernel_launches() - before == launches
        xs = x.copy()
        xs[1, n_in // 2, 5] ^= 1
        assert np.array_equal(vk.verify_batch(proofs, xs), [True, False, True])
    finally:
        vk.close()


def test_info_reports_table_bytes(mb_keys, m1024):
    vk = engine.VerifyingKey(mb_keys.vk_bytes)
    try:
        assert vk.info() == (129, 131 * TABLE_ROW_BYTES, True, True)      # 68.4 MB
    finally:
        vk.close()
    vk = engine.VerifyingKey(m1024[0])
    try:
        assert vk.info() == (N_PUB, (N_PUB + 2) * TABLE_ROW_BYTES, True, True)     # 1.07 GB
    finally:
        vk.close()
