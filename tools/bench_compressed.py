"""Compressed proofs and keys on one GPU: decompression rate of G1 and G2 points, lzkp_pk_load_compressed against
lzkp_pk_load_ex, and proofs_decompress_device + verify_batch_device against verify_batch_device alone.  Prints and
writes JSON lines (--out), the first one naming the card and its power limit.

Rates come from CUDA events around lzkp_proofs_decompress_device on batches of 2^20 proofs whose other points are the
point at infinity (which decodes without a square root), so one kernel of the three carries the time."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from libzkp_b200 import engine  # noqa: E402
from oracle import zkp_oracle as po  # noqa: E402


def frs(seed, n):
    rng = np.random.default_rng(seed)
    v = rng.integers(0, 2 ** 63, size=(n, 4), dtype=np.uint64)
    v[:, 3] &= (1 << 59) - 1                                   # < 2^251 < r
    return v.view(np.uint8).reshape(n, 32).copy()


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return {"card": q, "torch_name": torch.cuda.get_device_name(0)}


def event_ms(fn, reps):
    st = torch.cuda.current_stream()
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(reps):
        fn()
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b) / reps


def decompress_rates(n):
    g1 = torch.from_numpy(engine.generator_mul(1, frs(1, n))).cuda()
    g2 = torch.from_numpy(engine.generator_mul(2, frs(2, n))).cuda()
    inf1 = torch.from_numpy(np.frombuffer(po.g1_to_bytes(None), np.uint8).copy()).cuda()
    inf2 = torch.from_numpy(np.frombuffer(po.g2_to_bytes(None), np.uint8).copy()).cuda()
    out = {}
    for name, rows in (("g1", torch.cat([g1, inf2.expand(n, 128), g1.roll(1, 0)], 1)),
                       ("g2", torch.cat([inf1.expand(n, 64), g2, inf1.expand(n, 64)], 1))):
        rows = rows.contiguous()
        comp = torch.empty((n, 128), dtype=torch.uint8, device="cuda")
        ok = torch.empty(n, dtype=torch.uint8, device="cuda")
        s = torch.cuda.current_stream().cuda_stream
        engine.proofs_compress_device(n, rows.data_ptr(), comp.data_ptr(), ok.data_ptr(), s)
        dec = torch.empty((n, 256), dtype=torch.uint8, device="cuda")
        ms = event_ms(lambda: engine.proofs_decompress_device(n, comp.data_ptr(), dec.data_ptr(), ok.data_ptr(), s), 5)
        torch.cuda.synchronize()
        assert bool(ok.all()) and torch.equal(dec, rows)
        pts = 2 * n if name == "g1" else n
        out[name] = {"points": pts, "ms": round(ms, 3), "points_per_s": round(pts / ms * 1e3)}
    return out


def load_times(pk_bytes, reps, **kw):
    comp = engine.pk_compress(pk_bytes)
    res = {"uncompressed_bytes": len(pk_bytes), "compressed_bytes": len(comp), "ex_s": [], "compressed_s": []}
    for _ in range(reps):                                     # alternate the two loads
        for key, field, c in ((pk_bytes, "ex_s", False), (comp, "compressed_s", True)):
            torch.cuda.synchronize()
            t = time.perf_counter()
            pk = engine.ProvingKey(key, compressed=c, **kw)
            torch.cuda.synchronize()
            res[field].append(round(time.perf_counter() - t, 4))
            pk.close()
    for f in ("ex_s", "compressed_s"):
        res[f + "_median"] = float(np.median(res[f]))
    return res


def verify_times(pk_bytes, vk_bytes, sizes, reps):
    pk = engine.ProvingKey(pk_bytes, window_bits=12)
    pk.circuit_builtin(engine.EQUALITY, 110)
    n = max(sizes)
    a = np.arange(1, n + 1, dtype=np.uint64)
    proofs, cms, st = pk.prove_equality_batch(a, a, frs(3, n), frs(4, n))
    pk.close()
    assert not st.any()
    vk = engine.VerifyingKey(vk_bytes)
    d_p = torch.from_numpy(proofs).cuda()
    d_x = torch.from_numpy(cms).cuda()
    d_c = torch.empty((n, 128), dtype=torch.uint8, device="cuda")
    d_cok = torch.empty(n, dtype=torch.uint8, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    engine.proofs_compress_device(n, d_p.data_ptr(), d_c.data_ptr(), d_cok.data_ptr(), s)
    d_p2 = torch.empty((n, 256), dtype=torch.uint8, device="cuda")
    d_ok = torch.empty(n, dtype=torch.uint8, device="cuda")
    res = []
    for m in sizes:
        plain = event_ms(lambda: vk.verify_batch_device(m, d_p.data_ptr(), d_x.data_ptr(), 1, d_ok.data_ptr(), s), reps)
        assert bool(d_ok[:m].all())

        def both():
            engine.proofs_decompress_device(m, d_c.data_ptr(), d_p2.data_ptr(), d_cok.data_ptr(), s)
            vk.verify_batch_device(m, d_p2.data_ptr(), d_x.data_ptr(), 1, d_ok.data_ptr(), s)
        comp = event_ms(both, reps)
        dec = event_ms(lambda: engine.proofs_decompress_device(m, d_c.data_ptr(), d_p2.data_ptr(), d_cok.data_ptr(), s), reps)
        assert bool(d_ok[:m].all()) and bool(d_cok[:m].all())
        res.append({"proofs": m, "verify_device_ms": round(plain, 3), "decompress_then_verify_ms": round(comp, 3),
                    "decompress_ms": round(dec, 3)})
    vk.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--points", type=int, default=1 << 20)
    ap.add_argument("--skip-large", action="store_true")
    args = ap.parse_args()
    engine.init(0)
    lines = [dict(card(), what="device")]
    lines.append({"what": "decompress_rate", **decompress_rates(args.points)})
    td = po.Trapdoor.from_seed(1)
    toxic = (td.alpha, td.beta, td.gamma, td.delta, td.tau)
    pk_b, vk_b = engine.setup_builtin(engine.EQUALITY, 110, toxic)
    lines.append({"what": "pk_load_equality", **load_times(pk_b, 5, window_bits=12)})
    lines.append({"what": "verify", "rows": verify_times(pk_b, vk_b, (4096, 65536), 10)})
    if not args.skip_large:
        big, _ = engine.setup_builtin(engine.EQUALITY, 349524, toxic)
        lines.append({"what": "pk_load_2^20", **load_times(big, 3)})
    for ln in lines:
        print(json.dumps(ln), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
