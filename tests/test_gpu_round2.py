"""GPU tests added in round 2, all through the C ABI:
  * the asynchronous device-buffer entry points against the oracle - including a batch larger than one device pass
    (fork onto the engine's two streams) and calls issued back to back from two non-blocking caller streams, which
    share the key's workspaces (ordered by the per-workspace last-use events, include/lzkp_b200.h);
  * key files: persist -> reload from {prefix}_pk.bin / _vk.bin (validated, as deserialize_uncompressed does) ->
    identical proofs (reference: src/backend/snark.rs:40-115, 122-139);
  * the 2^20-constraint proof (BASELINE.json configs[3]) byte for byte against the C oracle;
  * validation of verifying keys, set_stride handling of the membership batch;
  * ONE process driving several GPUs (src/advanced/batch.rs:110-140): needs >= 2 devices, runs in a subprocess.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import libzkp_b200 as zk
from libzkp_b200 import engine, snark

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WINDOW_BITS = int(os.environ.get("LZKP_TEST_WINDOW_BITS", "12"))


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("n,chunk", [(5, 0), (300, 0), (700, 256), (1100, 512)])
def test_equality_batch_device_api_vs_oracle(eq_keys, co, po, frs, n, chunk):
    import torch
    pk = engine.ProvingKey(eq_keys.pk_bytes, window_bits=WINDOW_BITS, max_chunk=chunk)
    pk.circuit_builtin(engine.EQUALITY, 110)
    assert chunk == 0 or n > pk.max_chunk                     # the fork branch: chunks alternate between two streams
    rng = po.SplitMix64(61)
    a = np.array([rng.next_u64() for _ in range(n)], np.uint64)
    b = a.copy()
    b[n // 2] ^= 1
    r, s = frs(62, n), frs(63, n)
    d_a, d_b = _dev(torch, a.view(np.int64)), _dev(torch, b.view(np.int64))
    d_r, d_s = _dev(torch, r), _dev(torch, s)
    d_proofs = torch.zeros((n, 256), dtype=torch.uint8, device="cuda")
    d_status = torch.full((n,), 7, dtype=torch.int32, device="cuda")
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        pk.prove_equality_batch_device(n, d_a.data_ptr(), d_b.data_ptr(), d_r.data_ptr(), d_s.data_ptr(),
                                       d_proofs.data_ptr(), d_status.data_ptr(), st.cuda_stream)
    st.synchronize()
    want, wstat = co.prove_batch(eq_keys.circuit, eq_keys.opk, a, b, None, None, r, s)
    status = d_status.cpu().numpy()
    assert np.array_equal(status != 0, wstat != 0) and status[n // 2] == 1
    got = d_proofs.cpu().numpy()
    good = status == 0
    assert np.array_equal(got[good], want[good])
    pk.close()


def test_device_api_two_caller_streams_share_one_key(eq_keys, co, po, frs):
    # Two non-blocking streams issue calls on ONE key back to back, then a host-buffer call follows without any
    # synchronisation in between: every result must be the oracle's (round 1 raced on the shared workspace here).
    import torch
    pk = engine.ProvingKey(eq_keys.pk_bytes, window_bits=WINDOW_BITS)
    pk.circuit_builtin(engine.EQUALITY, 110)
    n, rounds = 600, 3
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    jobs = []
    for k in range(2 * rounds):
        rng = po.SplitMix64(100 + k)
        a = np.array([rng.next_u64() for _ in range(n)], np.uint64)
        r, s = frs(200 + k, n), frs(300 + k, n)
        jobs.append((a, r, s, _dev(torch, a.view(np.int64)), _dev(torch, r), _dev(torch, s),
                     torch.zeros((n, 256), dtype=torch.uint8, device="cuda"), torch.zeros(n, dtype=torch.int32, device="cuda")))
    torch.cuda.synchronize()
    for k, (a, r, s, d_a, d_r, d_s, d_p, d_st) in enumerate(jobs):
        st = streams[k & 1]
        pk.prove_equality_batch_device(n, d_a.data_ptr(), d_a.data_ptr(), d_r.data_ptr(), d_s.data_ptr(), d_p.data_ptr(),
                                       d_st.data_ptr(), st.cuda_stream)
    # host-buffer call on the same key while the device calls are still in flight
    a_h = np.arange(1, 41, dtype=np.uint64)
    r_h, s_h = frs(400, 40), frs(401, 40)
    proofs_h, _, status_h = pk.prove_equality_batch(a_h, a_h, r_h, s_h)
    torch.cuda.synchronize()
    want_h, _ = co.prove_batch(eq_keys.circuit, eq_keys.opk, a_h, a_h, None, None, r_h, s_h)
    assert not status_h.any() and np.array_equal(proofs_h, want_h)
    for k, (a, r, s, *_d, d_p, d_st) in enumerate(jobs):
        assert not d_st.cpu().numpy().any()
        got = d_p.cpu().numpy()
        m = 48                                               # the oracle is slow: a sample from both ends of each batch
        idx = np.r_[0:m // 2, n - m // 2:n]
        want, _ = co.prove_batch(eq_keys.circuit, eq_keys.opk, a[idx], a[idx], None, None, r[idx], s[idx])
        assert np.array_equal(got[idx], want), f"job {k}"
    pk.close()


def test_prove_batch_device_explicit_z(eq_keys, co, frs):
    import torch
    pk = engine.ProvingKey(eq_keys.pk_bytes, window_bits=WINDOW_BITS, max_chunk=32)
    pk.circuit_builtin(engine.EQUALITY, 110)
    n = 70                                                   # three chunks of <= 32 on the two engine streams
    z = np.stack([eq_keys.circuit.assign(100 + i, 100 + i) for i in range(n)])
    r, s = frs(71, n), frs(72, n)
    d_z, d_r, d_s = _dev(torch, z), _dev(torch, r), _dev(torch, s)
    d_p = torch.zeros((n, 256), dtype=torch.uint8, device="cuda")
    d_st = torch.zeros(n, dtype=torch.int32, device="cuda")
    pk.prove_batch_device(n, d_z.data_ptr(), d_r.data_ptr(), d_s.data_ptr(), d_p.data_ptr(), d_st.data_ptr(),
                          torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    a = np.arange(100, 100 + n, dtype=np.uint64)
    want, _ = co.prove_batch(eq_keys.circuit, eq_keys.opk, a, a, None, None, r, s)
    assert not d_st.cpu().numpy().any() and np.array_equal(d_p.cpu().numpy(), want)
    pk.close()


def test_key_dir_file_round_trip(tmp_path, po, co):
    # snark.rs:40-115,122-139: first use generates the keys and persists them; a second process-lifetime loads
    # {prefix}_pk.bin / _vk.bin (validating, as deserialize_uncompressed does) and must produce identical proofs.
    snark.reset()
    snark.configure(window_bits=WINDOW_BITS)
    try:
        assert zk.set_snark_key_dir(str(tmp_path))
        rng = po.SplitMix64(9)
        p1 = zk.SnarkBackend.prove_equality_zk(5, 5, zk.snark_commit_value(5), rng=rng)
        setup1 = zk.SnarkBackend.get_universal_setup()
        pk_file, vk_file = tmp_path / "equality_mimc_pk.bin", tmp_path / "equality_mimc_vk.bin"
        assert pk_file.exists() and vk_file.exists()
        assert pk_file.stat().st_size == 140208 and vk_file.read_bytes() == setup1.vk_bytes
        pk_bytes = pk_file.read_bytes()
        snark.reset()                                        # "new process": drops the OnceLock analogue and the key dir
        snark.configure(window_bits=WINDOW_BITS)
        assert zk.set_snark_key_dir(str(tmp_path))
        rng = po.SplitMix64(9)
        p2 = zk.SnarkBackend.prove_equality_zk(5, 5, zk.snark_commit_value(5), rng=rng)
        assert p2 == p1
        assert pk_file.read_bytes() == pk_bytes              # files are read, not rewritten
        # the oracle proves the same bytes from the same file
        rng = po.SplitMix64(9)
        r, s = rng.next_fr(), rng.next_fr()
        circ = co.Circuit("equality")
        assert p1 == co.prove(circ, co.ProvingKey(pk_bytes), circ.assign(5, 5), r, s)
        vk = po.vk_from_bytes(vk_file.read_bytes())
        cm = int.from_bytes(zk.snark_commit_value(5), "little")
        assert po.verify(vk, po.equality_public_inputs(cm), po.proof_from_bytes(p1))
        # a corrupted key file is rejected at load (validation is on for files) and the failure is sticky
        snark.reset()
        snark.configure(window_bits=WINDOW_BITS)
        bad = bytearray(pk_bytes)
        bad[64 + 3 * 128 + 8 + 2 * 64 + 64 + 64 + 8 + 5 * 64] ^= 1          # x of a_query[5]: off the curve
        pk_file.write_bytes(bytes(bad))
        assert zk.set_snark_key_dir(str(tmp_path))
        assert zk.SnarkBackend.prove_equality_zk(5, 5, zk.snark_commit_value(5)) == b""      # empty Vec = failure
        with pytest.raises(RuntimeError):                    # ... which prove_equality turns into ProofGenerationFailed
            zk.prove_equality(5, 5)
    finally:
        snark.reset()
        snark.configure()


def test_vk_validation_rejects_bad_points(eq_keys):
    good = bytearray(eq_keys.vk_bytes)
    engine.VerifyingKey(bytes(good)).close()
    bad = bytearray(good)
    bad[0] ^= 1                                              # alpha_g1.x
    with pytest.raises(zk.EngineError, match="off-curve"):
        engine.VerifyingKey(bytes(bad))
    bad = bytearray(good)
    bad[64 + 128] ^= 1                                       # gamma_g2.x.c0
    with pytest.raises(zk.EngineError, match="off-curve"):
        engine.VerifyingKey(bytes(bad))
    bad = bytearray(good)
    bad[456 + 64] ^= 1                                       # gamma_abc_g1[1].x
    with pytest.raises(zk.EngineError, match="off-curve"):
        engine.VerifyingKey(bytes(bad))


def test_membership_set_stride_is_validated(mb_keys, co, frs):
    pk = engine.ProvingKey(mb_keys.pk_bytes, window_bits=8)
    pk.circuit_builtin(engine.MEMBERSHIP, 64)
    vals = np.array([3, 9], np.uint64)
    sets = np.array([[1, 2, 3, 4], [9, 9, 9, 9]], np.uint64)            # rows are 4 wide
    r, s = frs(81, 2), frs(82, 2)
    lens = np.array([3, 6], np.uint32)                                    # second row claims more entries than a row holds
    proofs, _, status = pk.prove_membership_batch(vals, sets, lens, r, s)
    assert status[0] == 0 and status[1] == 2 and not proofs[1].any()
    z = mb_keys.circuit.assign(3, set_=[1, 2, 3])
    assert proofs[0].tobytes() == co.prove(mb_keys.circuit, mb_keys.opk, z, co.fr_list(r[0])[0], co.fr_list(s[0])[0])
    with pytest.raises(zk.EngineError):                                   # set_stride == 0
        pk.prove_membership_batch(vals, np.zeros((2, 0), np.uint64), np.array([1, 1], np.uint32), r, s)
    pk.close()


def test_config4_2_20_proof_bit_exact_vs_c_oracle(co, trapdoor, frs):
    # BASELINE.json configs[3] at full size, byte for byte: the C oracle (OpenMP Pippenger + radix-2 FFT) proves
    # from the same 384 MiB key file image
    rounds = 349524
    pk_bytes, _ = engine.setup_builtin(engine.EQUALITY, rounds, trapdoor)
    pk = engine.ProvingKey(pk_bytes)
    pk.circuit_builtin(engine.EQUALITY, rounds)
    z = engine.builtin_witness(engine.EQUALITY, rounds, 6, 6)
    r, s = frs(4, 1), frs(40, 1)
    proofs, status = pk.prove_batch(z[None], r, s)
    assert not status.any()
    pk.close()
    circ = co.Circuit("equality", rounds)
    assert circ.n == 1 << 20
    want = co.prove(circ, co.ProvingKey(pk_bytes), z, co.fr_list(r)[0], co.fr_list(s)[0])
    assert proofs[0].tobytes() == want


def test_one_process_drives_every_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two visible GPUs")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "run_fanout_check.py")], capture_output=True,
                         text=True, timeout=1200)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    rep = json.loads(out.stdout.strip().splitlines()[-1])
    assert rep["devices"] >= 2 and rep["equality_bit_exact"] and rep["membership_bit_exact"] and rep["explicit_z_bit_exact"]
    assert rep["small_call_on_primary_ok"] and rep["all_devices_launched"]


def test_sharded_prover_two_ranks_over_nccl():
    # SURVEY 8e "single large proof": two real ranks, NCCL broadcast of z || r || s and all_gather of the partial sums;
    # rank 0 compares the bytes with the unsharded single-GPU proof (tools/run_sharded_proof.py)
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two visible GPUs")
    env = dict(os.environ, LZKP_FORCE_LARGE="1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29671",
                          os.path.join(ROOT, "tools", "run_sharded_proof.py"), "2730"],
                         capture_output=True, text=True, timeout=900, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    rep = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert rep["world"] == 2 and rep["matches_single_gpu"]
