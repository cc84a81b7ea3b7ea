"""Proof rerandomization on one GPU: lzkp_proofs_rerandomize_device kernel time (CUDA events, median of warm calls),
lzkp_proofs_rerandomize wall time (host buffers, staging included), and lzkp_verify_batch_device on the same proofs,
for n = 1, 64, 4096, 65 536 and 2^20.  Prints and writes JSON lines (--out), the first one naming the card, its power
limit and its maximum SM clock.

Proofs are 300 equality proofs tiled to n (the kernel's work does not depend on which valid proof a row holds);
factors are seeded.  The per-proof Fq-product count is an estimate from the formulas (rerandomize.cu header)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from libzkp_b200 import engine  # noqa: E402
from oracle import c_oracle  # noqa: E402
from oracle import zkp_oracle as po  # noqa: E402

EST_FQ_PRODUCTS = 14_200        # 2.3 k subgroup + 9.0 k joint G2 ladder + 2.6 k G1 ladders + 0.3 k affine (estimated)


def frs(seed, n):
    rng = np.random.default_rng(seed)
    v = rng.integers(0, 2 ** 63, size=(n, 4), dtype=np.uint64)
    v[:, 3] &= (1 << 59) - 1                                   # < 2^251 < r
    v[:, 0] |= 1                                               # non-zero
    return v.view(np.uint8).reshape(n, 32).copy()


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return {"card": q, "torch_name": torch.cuda.get_device_name(0)}


def median_event_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,64,4096,65536,1048576")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    c_oracle.build()
    circ = c_oracle.Circuit("equality")
    td = po.Trapdoor.from_seed(1)
    pk_bytes, vk_bytes = circ.setup((td.alpha, td.beta, td.gamma, td.delta, td.tau))
    pk = engine.ProvingKey(pk_bytes, window_bits=10)
    pk.circuit_builtin(engine.EQUALITY, 110)
    a = np.arange(1, 301, dtype=np.uint64)
    base, cms, st = pk.prove_equality_batch(a, a, frs(1, 300), frs(2, 300))
    pk.close()
    assert not st.any()
    vk = engine.VerifyingKey(vk_bytes)
    s = torch.cuda.current_stream().cuda_stream
    for n in [int(x) for x in args.sizes.split(",")]:
        reps = max(args.reps, 5)
        tile = n // 300 + 1
        proofs = np.tile(base, (tile, 1))[:n]
        x = np.tile(cms, (tile, 1))[:n]
        r1, r2 = frs(10 + n, n), frs(20 + n, n)
        d_p, d_r1, d_r2 = (torch.from_numpy(v).cuda() for v in (proofs, r1, r2))
        d_x = torch.from_numpy(np.ascontiguousarray(x)).cuda()
        d_out = torch.empty((n, 256), dtype=torch.uint8, device="cuda")
        d_ok = torch.empty(n, dtype=torch.uint8, device="cuda")
        d_vok = torch.empty(n, dtype=torch.uint8, device="cuda")
        rr = lambda: vk.rerandomize_device(n, d_p.data_ptr(), d_r1.data_ptr(), d_r2.data_ptr(), d_out.data_ptr(),
                                           d_ok.data_ptr(), s)
        vf = lambda: vk.verify_batch_device(n, d_out.data_ptr(), d_x.data_ptr(), 1, d_vok.data_ptr(), s)
        rr_ms = median_event_ms(rr, reps)
        vf_ms = median_event_ms(vf, reps)
        assert d_ok.cpu().numpy().all() and d_vok.cpu().numpy().all(), n
        walls = []
        for _ in range(3 if n >= 65536 else reps):
            t0 = time.perf_counter()
            out, ok = vk.rerandomize(proofs, r1, r2)
            walls.append((time.perf_counter() - t0) * 1e3)
        assert ok.all() and np.array_equal(out, d_out.cpu().numpy()), n
        rec = {"n": n, "rerandomize_device_ms": round(rr_ms, 3), "rerandomize_host_wall_ms": round(statistics.median(walls), 3),
               "verify_batch_device_ms": round(vf_ms, 3), "rerandomize_per_s": round(n / rr_ms * 1e3),
               "verify_per_s": round(n / vf_ms * 1e3), "rerandomize_over_verify": round(rr_ms / vf_ms, 2),
               "fq_products_per_proof_estimated": EST_FQ_PRODUCTS,
               "fq_products_per_s_estimated": round(EST_FQ_PRODUCTS * n / rr_ms * 1e3), "reps": reps}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
        del d_p, d_r1, d_r2, d_x, d_out, d_ok, d_vok
        torch.cuda.empty_cache()
    vk.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
