"""Verification of a membership-1024 key (2049 public inputs) against membership-64 (129), in one process.

Prints one JSON line per measurement: the card and its power limit, lzkp_vk_load time and table bytes, and per proof count
the median wall time of verify_batch (host -> device copies included), the host -> device copy of the public inputs alone
(timed separately with the same pageable source) and, from one profiled call, the kernel time by kernel.
  --save DIR    keep the membership-1024 key and one proof in DIR
  --one DIR     time only that 1-proof call.  It uses nothing but VerifyingKey and verify_batch, so a copy of this script
                placed in another checkout times that checkout's build (the "before" figure of a change)
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from libzkp_b200 import engine, transforms  # noqa: E402

COUNTS = [1, 64, 148, 296, 444, 445, 1024, 4096, 16384]


def emit(**kw):
    print(json.dumps(kw), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def membership_batch(slots, n, seed):
    """n valid proofs of a `slots`-slot membership key (sets of lengths 1 .. slots) and their public inputs."""
    pk_bytes, vk_bytes = engine.setup_builtin(engine.MEMBERSHIP, slots, transforms._toxic(1))
    rng = np.random.default_rng(seed)
    lens = (1 + (np.arange(n) * 37) % slots).astype(np.uint32)
    sets = rng.integers(0, 2**64, size=(n, slots), dtype=np.uint64)
    sets[np.arange(slots)[None, :] >= lens[:, None]] = 0
    vals = sets[np.arange(n), np.arange(n) % lens]
    r = np.zeros((n, 32), np.uint8); r[:, :8] = rng.integers(1, 2**63, size=(n, 1), dtype=np.uint64).view(np.uint8)
    s = np.zeros((n, 32), np.uint8); s[:, :8] = rng.integers(1, 2**63, size=(n, 1), dtype=np.uint64).view(np.uint8)
    pk = engine.ProvingKey(pk_bytes, window_bits=8)
    pk.circuit_builtin(engine.MEMBERSHIP, slots)
    proofs, cms, st = pk.prove_membership_batch(vals, sets, lens, r, s)
    pk.close()
    assert not st.any()
    x = np.zeros((n, 1 + 2 * slots, 32), np.uint8)
    x[:, 0] = cms
    x[:, 1:1 + slots, :8] = sets.view(np.uint8).reshape(n, slots, 8)
    x[:, 1 + slots:, 0] = np.arange(slots)[None, :] < lens[:, None]
    return vk_bytes, proofs, x


def h2d_ms(x, reps=3):
    import torch
    src = torch.from_numpy(x.reshape(-1))
    dst = torch.empty(src.numel(), dtype=torch.uint8, device="cuda")
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dst.copy_(src)
        torch.cuda.synchronize()
        ts.append(1e3 * (time.perf_counter() - t0))
    del dst
    return round(float(np.median(ts)), 3)


def kernel_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    by = {}
    for e in prof.events():
        if e.device_type.name != "CUDA" or "Memcpy" in e.name or "Memset" in e.name:
            continue
        k = e.name.replace("void ", "").replace("lzkp::(anonymous namespace)::", "").split("(")[0]
        by[k] = by.get(k, 0.0) + e.device_time / 1e3
    return round(sum(by.values()), 3), {k: round(v, 3) for k, v in by.items()}


def time_call(vk, proofs, x, reps):
    ok = vk.verify_batch(proofs, x)                  # warm-up: staging buffers, module load
    assert ok.all(), np.flatnonzero(~ok)[:8]
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        vk.verify_batch(proofs, x)
        ts.append(1e3 * (time.perf_counter() - t0))
    return round(float(np.median(ts)), 3), [round(t, 3) for t in ts]


def run_key(name, vk_bytes, proofs, x, counts, reps):
    t0 = time.perf_counter()
    vk = engine.VerifyingKey(vk_bytes)
    load = 1e3 * (time.perf_counter() - t0)
    n_pub, tab, lat, comb = vk.info()
    emit(key=name, n_pub=n_pub, vk_load_ms=round(load, 1), table_bytes=tab, latency_form=lat, combined_form=comb)
    for m in counts:
        p, xx = tile(proofs, x, m)
        med, each = time_call(vk, p, xx, reps)
        ktot, kby = kernel_ms(lambda: vk.verify_batch(p, xx))
        emit(key=name, proofs=m, wall_ms=med, each=each, h2d_inputs_ms=h2d_ms(xx), input_bytes=int(xx.nbytes),
             kernel_ms=ktot, kernels=kby, verifies_per_s=round(m / med * 1e3, 1))
    return vk


def tile(proofs, x, m):
    if m <= len(proofs):
        return proofs[:m], x[:m]
    k = -(-m // len(proofs))
    return np.concatenate([proofs] * k)[:m], np.concatenate([x] * k)[:m]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--save")
    ap.add_argument("--one")
    a = ap.parse_args()
    engine.init(0)
    emit(card=card(), checkout=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    if a.one:
        d = np.load(os.path.join(a.one, "m1024.npz"))
        t0 = time.perf_counter()
        vk = engine.VerifyingKey(d["vk"].tobytes())
        load = 1e3 * (time.perf_counter() - t0)
        t0 = time.perf_counter()
        ok = vk.verify_batch(d["proofs"], d["x"])
        emit(key="membership-1024", proofs=1, vk_load_ms=round(load, 1), wall_ms=round(1e3 * (time.perf_counter() - t0), 3),
             ok=bool(ok.all()))
        return
    vk1024_bytes, p1024, x1024 = membership_batch(1024, 4096, 11)
    if a.save:
        os.makedirs(a.save, exist_ok=True)
        np.savez(os.path.join(a.save, "m1024.npz"), vk=np.frombuffer(vk1024_bytes, np.uint8), proofs=p1024[:1], x=x1024[:1])
    vk64_bytes, p64, x64 = membership_batch(64, 4096, 12)
    run_key("membership-64", vk64_bytes, p64, x64, COUNTS, a.reps).close()
    run_key("membership-1024", vk1024_bytes, p1024, x1024, COUNTS, a.reps).close()


if __name__ == "__main__":
    main()
