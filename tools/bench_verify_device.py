"""lzkp_verify_batch_device against lzkp_verify_batch, with the proofs and public inputs already on the device.

Keys: equality (1 public input), membership-64 (129) and membership-1024 (2049), at 1, 64, 444, 445, 4096 and 16 384 proofs
(batches above 4096 repeat the 4096 proofs).  Per key and count, one JSON line with the median over --reps calls of
  host_wall_ms      verify_batch from host arrays (its copies in and out included)
  device_wall_ms    verify_batch_device on a non-blocking stream plus a synchronise of that stream
  device_kernel_ms  CUDA events recorded on that stream around the call
and the same at 4096 proofs with one forged proof (a wrong C), where a group's combined check fails and its proofs are
re-verified: from the host (verify_batch) or on the device (verify_batch_device).  The first line names the card and
its power limit.  Every line is also written to --out (default profiles/r5_verify_device.txt).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_verify_many_inputs import card, membership_batch, tile  # noqa: E402
from libzkp_b200 import engine, transforms  # noqa: E402

COUNTS = [1, 64, 444, 445, 4096, 16384]
LINES = []


def emit(**kw):
    line = json.dumps(kw)
    LINES.append(line)
    print(line, flush=True)


def equality_batch(n, seed):
    pk_bytes, vk_bytes = engine.setup_builtin(engine.EQUALITY, 110, transforms._toxic(1))
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 2**63, size=n, dtype=np.uint64)
    r = np.zeros((n, 32), np.uint8); r[:, :8] = rng.integers(1, 2**63, size=(n, 1), dtype=np.uint64).view(np.uint8)
    s = np.zeros((n, 32), np.uint8); s[:, :8] = rng.integers(1, 2**63, size=(n, 1), dtype=np.uint64).view(np.uint8)
    pk = engine.ProvingKey(pk_bytes, window_bits=10)
    pk.circuit_builtin(engine.EQUALITY, 110)
    proofs, cms, st = pk.prove_equality_batch(a, a, r, s)
    pk.close()
    assert not st.any()
    return vk_bytes, proofs, cms.reshape(n, 1, 32)


def median(ts):
    return round(float(np.median(ts)), 3)


def time_pair(vk, proofs, x, reps, want):
    """(host wall, device wall, device kernel) medians in ms; every call's decisions are checked against `want`."""
    import torch
    m = len(proofs)
    d_p = torch.from_numpy(np.ascontiguousarray(proofs)).cuda()
    d_x = torch.from_numpy(np.ascontiguousarray(x).reshape(m, -1)).cuda()
    d_ok = torch.zeros(m, dtype=torch.uint8, device="cuda")
    n_pub = d_x.shape[1] // 32
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    host, dev, kern = [], [], []
    for k in range(reps + 1):                               # the first of each is a warm-up (scratch, module load)
        t0 = time.perf_counter()
        ok = vk.verify_batch(proofs, x)
        t1 = time.perf_counter()
        assert np.array_equal(ok, want), np.flatnonzero(ok != want)[:8]
        d_ok.fill_(7)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        e0.record(s)
        vk.verify_batch_device(m, d_p.data_ptr(), d_x.data_ptr(), n_pub, d_ok.data_ptr(), s.cuda_stream)
        e1.record(s)
        s.synchronize()
        t3 = time.perf_counter()
        assert np.array_equal(d_ok.cpu().numpy().astype(bool), want)
        if k:
            host.append(1e3 * (t1 - t0))
            dev.append(1e3 * (t3 - t2))
            kern.append(e0.elapsed_time(e1))
    del d_p, d_x, d_ok
    torch.cuda.empty_cache()
    return median(host), median(dev), median(kern)


def run_key(name, vk_bytes, proofs, x, reps):
    vk = engine.VerifyingKey(vk_bytes)
    n_pub, tab, lat, comb = vk.info()
    emit(key=name, n_pub=n_pub, table_bytes=tab, latency_form=lat, combined_form=comb)
    for m in COUNTS:
        p, xx = tile(proofs, x, m)
        h, d, k = time_pair(vk, p, xx, reps, np.ones(m, bool))
        emit(key=name, proofs=m, input_bytes=int(xx.nbytes), host_wall_ms=h, device_wall_ms=d, device_kernel_ms=k)
    m = 4096
    p, xx = tile(proofs, x, m)
    p = p.copy()
    p[1000, 192:256] = p[1001, 192:256]                    # a valid curve point, the wrong C: group 15 fails
    want = np.ones(m, bool)
    want[1000] = False
    h, d, k = time_pair(vk, p, xx, reps, want)
    emit(key=name, proofs=m, forged=1, host_wall_ms=h, device_wall_ms=d, device_kernel_ms=k)
    vk.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_verify_device.txt"))
    a = ap.parse_args()
    engine.init(0)
    emit(card=card())
    n = 4096
    run_key("equality", *equality_batch(n, 21), a.reps)
    run_key("membership-64", *membership_batch(64, n, 12), a.reps)
    run_key("membership-1024", *membership_batch(1024, n, 11), a.reps)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
