#!/usr/bin/env python3
"""bench.py — batched Groth16/BN254 proving throughput on B200 (BASELINE.json configs[1]).

A "step" is one pass of the hot path over one batch: `--batch` (default 4096) equality proofs per
GPU — device witness generation, R1CS->QAP witness map (7 NTTs), the five MSMs over the HBM-resident
proving key, assembly and ark-serialize output.  One process per GPU (torchrun sets RANK /
LOCAL_RANK / WORLD_SIZE); proofs are independent, so ranks shard the batch with no collective
("weak": every rank proves its own `--batch` proofs per step).

  value   proofs/s with inputs (a, b, r, s) already resident in HBM, timed with CUDA events
  e2e     the same through the C-ABI call lzkp_prove_equality_batch with HOST buffers
          (H2D of inputs and D2H of proofs/status/commitments inside the timed region)
  roofline  the dominant kernel (G1 table MSM): algorithmic IMADs / its CUDA-event time vs the
          measured peak of the 32x32->64 multiplier on this pool's B200 (profiles/r2_imadrate.jsonl)
  cpu_baseline  the CPU restatement (oracle/, C, OpenMP) on a bounded sample of the same workload
  extra   G1 MSM points/s @2^20 and NTT elements/s @2^22 (BASELINE.json's other two metrics)

`--gpus N` (torchrun) adds, in `extra`: BASELINE.json configs[3] (one 2^20-constraint proof split over the N ranks, bytes
asserted equal to the one-GPU proof), configs[4] (65 536-proof mixed batch sharded over the ranks, gather included) and
the same 4096-per-GPU batch through ONE process driving all N GPUs (lzkp_init with N devices).

`--impl reference` times the CPU restatement of the reference's prover (oracle/: the reference is
Rust + un-vendored arkworks crates and cannot be built here, DESIGN.md "Oracle") on the same config.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # a run leaves the tree as it found it (it may be read-only)

import numpy as np  # noqa: E402

R_MOD = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
IMAD_PER_MUL = 272            # SURVEY.md §8d: 136 32x32 multiply-accumulates = 272 mad.lo/mad.hi issues
M_MADD_G1 = 10                # XYZZ mixed add: 8M + 2S
M_MADD_G2 = 28                # over Fq2: 8 * 3 + 2 * 2 base-field products
# What the kernels execute per mixed add since lazy reduction went in (field.cuh): G1 = 8 products + one a*b - c*d with
# a shared reduction (2 * 128 + 144); G2 = 8 Fq2 products of 3 * 128 + 2 * 144 and 2 Fq2 squares of 2 * 272.
# (round 2: the two squarings of a G1 mixed add are dedicated 36 + 64 + 4 limb-product squarings = 208 issues each)
IMAD_EXEC_MADD_G1 = 6 * 272 + 2 * 208 + 400
IMAD_EXEC_MADD_G2 = 8 * 672 + 2 * 544
# Peak of the 32x32->64 multiplier, in SURVEY units (mad.lo and mad.hi counted separately = 2 per IMAD.WIDE):
# tools/microbench/imadrate.cu on this pool's B200 measures 31.8 IMAD.WIDE lanes per SM per clock for EVERY form of the
# instruction a big-integer product can use (carry-in .X rows, carry-out only, IMAD.HI; vector or uniform operands),
# i.e. 9.25 T wide/s = 18.49 T IMAD/s at 148 SMs x 1965 MHz.  Round 1's 17.25 T/s "independent IMAD.WIDE" figure was an
# artefact: ptxas had strength-reduced that microbenchmark's loop-invariant products into IADD3 pairs (its SASS holds
# 9 IMAD.WIDE and 128 IADD3), so it measured the ALU pipe.  There is no 2x-faster flag-free form to move to.
IMAD_PEAK_FALLBACK = 18.49e12


class SplitMix64:
    def __init__(self, seed):
        self.s = seed & 0xFFFFFFFFFFFFFFFF

    def next_u64(self):
        self.s = (self.s + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        z = self.s
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
        return z ^ (z >> 31)

    def next_fr(self):
        while True:
            v = 0
            for i in range(4):
                v |= self.next_u64() << (64 * i)
            v &= (1 << 254) - 1
            if v < R_MOD:
                return v


def fr_bytes(seed, n):
    rng = SplitMix64(seed)
    return np.frombuffer(b"".join(rng.next_fr().to_bytes(32, "little") for _ in range(n)), np.uint8).reshape(n, 32).copy()


def u64s(seed, n):
    rng = SplitMix64(seed)
    return np.array([rng.next_u64() for _ in range(n)], np.uint64)


def imad_peak():
    p = os.path.join(ROOT, "profiles", "r2_imadrate.jsonl")
    best = 0.0
    try:
        for line in open(p):
            d = json.loads(line)
            if d.get("bench") in ("imad_wide_x_rows", "imad_wide_carry_out", "imad_hi"):
                best = max(best, 2 * d["Tops_per_s"] * 1e12)
    except OSError:
        pass
    return (best, "measured (profiles/r2_imadrate.jsonl: IMAD.WIDE.U32[.X] / IMAD.HI lanes per second x 2 mad.lo/hi "
                  "issues; the 32x32->64 multiplier runs at 31.8 lanes per SM per clock in every form)") if best \
        else (IMAD_PEAK_FALLBACK, "fallback")


def ncu_traffic(kernel_substr):
    """dram__bytes_read + dram__bytes_write per launch of a kernel, from the committed ncu --set full summary."""
    path = os.path.join(ROOT, "profiles", "r2_ncu_msm_batch.txt")
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    try:
        lines = open(path).read().splitlines()
    except OSError:
        return None
    for i, line in enumerate(lines):
        if line.startswith("==") and kernel_substr in line:
            tot = 0.0
            for l2 in lines[i + 1:i + 8]:
                parts = l2.split()
                if len(parts) >= 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tot += float(parts[1]) * unit.get(parts[2], 1.0)
            return tot or None
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.1] or [r for _, r in self.rows[-3:]]
        sm = sorted(int(float(r[0])) for r in rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        power = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(float(rows[0][1])) if rows else None,
                "power_w_max": max(power) if power else None, "samples": len(rows), "reasons": reasons}


def toxic(seed):
    rng = SplitMix64(seed)
    return [rng.next_fr() for _ in range(5)]


DUMP_BYTES = 64 << 20


def dump_outputs(path, proofs, status):
    """--dump-outputs: the proofs (n x 256 bytes) and status codes a caller of the timed path receives, as float32
    path/proofs.npy and path/status.npy (exact: bytes and small integers), plus path/rows.npy (float64), the batch rows
    written: all of them while the files fit in 64 MiB, else a fixed seeded sample.  Inputs are seeded, so two builds
    run with the same arguments can be compared file for file."""
    n = len(proofs)
    row_bytes = 4 * proofs.shape[1] + 4 + 8
    rows = np.arange(n)
    if n * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // row_bytes, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "proofs.npy"), proofs[rows].astype(np.float32))
    np.save(os.path.join(path, "status.npy"), status[rows].astype(np.float32))
    np.save(os.path.join(path, "rows.npy"), rows.astype(np.float64))


# ----------------------------------------------------------------------------- reference arm (CPU)
def host_cores():
    """Host threads this process may use.  torchrun exports OMP_NUM_THREADS=1 to every rank, which made the OpenMP
    oracle run single-threaded at N > 1 in round 1; the thread count is therefore always passed explicitly."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def run_reference(args, rank, world):
    """The reference's CPU prover path (oracle/: restatement of ark-groth16's create_proof, proof-parallel the way
    src/advanced/batch.rs:123-131 maps a batch over rayon workers) on every host core, rank 0 only."""
    if rank != 0:
        return
    from oracle import c_oracle as co
    co.build()
    circ = co.Circuit("equality")
    pk_bytes, _ = circ.setup(toxic(1))
    opk = co.ProvingKey(pk_bytes)
    cores = host_cores()
    # a step = a bounded sample of the step's batch: proofs are independent, so proofs/s over the sample is the rate of
    # the whole batch; sized for ~1 s per step (about 20 proofs/s per core)
    sample = min(args.batch, args.ref_sample or max(cores * 16, 64))
    a = u64s(3, sample)
    r, s = fr_bytes(4, sample), fr_bytes(40, sample)
    for _ in range(min(args.warmup, 2)):
        co.prove_batch(circ, opk, a[:cores], a[:cores], None, None, r[:cores], s[:cores], threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        proofs, status = co.prove_batch(circ, opk, a, a, None, None, r, s, threads=cores)
    dt = time.perf_counter() - t0
    assert not status.any()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, proofs, status)
    v = sample * args.steps / dt
    desc = (f"each step proves the first {sample} of the batch's {args.batch} independent equality proofs, "
            f"proof-parallel over {cores} OpenMP threads (explicit; OMP_NUM_THREADS is ignored)")
    print(json.dumps({
        "impl": "reference", "metric": "groth16_bn254_proofs_per_sec_batched", "value": v, "unit": "proofs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u256 (4x64-bit Montgomery limbs)",
        "data": "synthetic", "config": config_dict(args),
        "cpu_baseline": {"value": v, "unit": "proofs/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": v, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "CPU restatement (C, OpenMP) of the arkworks prover the reference calls; not arkworks itself "
                "(no Rust toolchain in this image). The reference's README quotes ~10 ms per proof per core "
                "(/root/reference/README.md:327); this port takes ~48 ms, so a real arkworks arm would be ~5x faster."}))


def config_dict(args):
    return {"workload": f"process_batch of {args.batch} prove_equality proofs per GPU (BASELINE.json configs[1]): "
                        "MiMC-5 equality circuit, m=332 constraints, domain n=512, MSM sizes 333/333/333(G2)/332/511",
            "batch_per_gpu": args.batch,
            "l2": "inputs larger than L2: every step gathers from the resident window tables "
                  "(62 GB at c=16, 116 GB at c=17) and rewrites > 126 MB of workspace"}


# ----------------------------------------------------------------------------- our arm (GPU)
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from libzkp_b200 import engine

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    engine.init(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    P = args.batch

    # proving key: device-side setup (deterministic toxic waste: synthetic benchmark key), resident tables
    t0 = time.perf_counter()
    pk_bytes, _ = engine.setup_builtin(engine.EQUALITY, 110, toxic(1))
    t_setup = time.perf_counter() - t0
    t0 = time.perf_counter()
    # c = 17 (15 windows, 116 GB of tables for this key) when the GPU has the room, else the engine's own choice
    # from its memory budget (c <= 16); --window-bits pins it
    try:
        pk = engine.ProvingKey(pk_bytes, window_bits=args.window_bits or 17, max_chunk=args.chunk)
    except Exception:                           # EngineError(LZKP_E_NOMEM): the tables do not fit beside other users
        if args.window_bits:
            raise
        pk = engine.ProvingKey(pk_bytes, window_bits=0, max_chunk=args.chunk)
    pk.circuit_builtin(engine.EQUALITY, 110)
    torch.cuda.synchronize()
    t_load = time.perf_counter() - t0

    # synthetic inputs (SURVEY.md §8d config 2): a_i = b_i = SplitMix64(seed 3), r_i, s_i seed 4
    a_h = u64s(3 + 1000 * rank, P)
    r_h, s_h = fr_bytes(4 + 1000 * rank, P), fr_bytes(40 + 1000 * rank, P)
    as_i64 = lambda x: torch.from_numpy(x.view(np.int64))
    d_a = as_i64(a_h).to(dev)
    d_r, d_s = torch.from_numpy(r_h).to(dev), torch.from_numpy(s_h).to(dev)
    d_proofs = torch.zeros((P, 256), dtype=torch.uint8, device=dev)
    d_status = torch.zeros(P, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream()

    def step():
        pk.prove_equality_batch_device(P, d_a.data_ptr(), d_a.data_ptr(), d_r.data_ptr(), d_s.data_ptr(),
                                       d_proofs.data_ptr(), d_status.data_ptr(), stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    assert int(d_status.abs().sum().item()) == 0
    engine.profile_enable(True)
    pk.profile_read(reset=True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    launches0 = engine.kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    w0 = time.time()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    w1 = time.time()
    ms = ev0.elapsed_time(ev1)
    launches = engine.kernel_launches() - launches0
    clocks = sampler.stop(w0, w1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_proofs.cpu().numpy(), d_status.cpu().numpy())
    regions = pk.profile_read(reset=True)
    engine.profile_enable(False)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * P * args.steps / (ms * 1e-3)

    # ---- end to end through the C ABI with host buffers (pinned), copies inside the timed region
    pin = lambda x: torch.from_numpy(x).pin_memory().numpy()
    a_p, r_p, s_p = as_i64(a_h).pin_memory().numpy().view(np.uint64), pin(r_h), pin(s_h)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    zp = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory().numpy()
    out_p = (zp((P, 256), torch.uint8), zp((P, 32), torch.uint8), zp((P,), torch.int32))     # caller-owned pinned result buffers
    pk.prove_equality_batch(a_p, a_p, r_p, s_p, out=out_p)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        proofs_h, cms_h, status_h = pk.prove_equality_batch(a_p, a_p, r_p, s_p, out=out_p)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    assert not status_h.any()
    assert np.array_equal(proofs_h, d_proofs.cpu().numpy()), "host-buffer and device-buffer paths disagree"
    e2e = {"value": world * P * e2e_steps / e2e_s, "unit": "proofs/s", "h2d_bytes_per_step": P * (8 + 8 + 32 + 32),
           "d2h_bytes_per_step": P * (256 + 4 + 32), "steps": e2e_steps,
           "api": "lzkp_prove_equality_batch (C ABI, pinned host buffers)"}

    # ---- N > 1: BASELINE.json configs[3] and configs[4], measured with every rank taking part, then ONE process
    # driving all N GPUs (rank 0 alone, after the other ranks have left and released their devices)
    multi = {}
    work = pk.work()
    engine_info = {"window_bits": pk.window_bits, "windows": pk.windows, "table_gb": pk.table_bytes / 1e9,
                   "setup_s": t_setup, "pk_load_s": t_load}
    if world > 1 and not args.no_extra:
        pk.close()
        torch.cuda.empty_cache()
        dist.barrier()
        # a failure in an extra must not cost the headline line: it is recorded under its key instead
        for key, fn in (("proof_2^20_sharded", bench_sharded_proof), ("mixed_batch_65536", bench_mixed_sharded),
                        ("transform_replicas", bench_replicas)):
            try:
                multi[key] = fn(torch, dist, dev, rank, world)
            except Exception as e:  # noqa: BLE001
                multi[key] = {"error": repr(e)}
            torch.cuda.empty_cache()
            dist.barrier()
    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return
    if world > 1 and not args.no_extra:
        try:
            multi["single_process_fanout"] = bench_fanout(torch, world, pk_bytes, engine_info["window_bits"], P, a_p, r_p, s_p,
                                                          proofs_h, e2e["value"], max(2, e2e_steps))
        except Exception as e:  # noqa: BLE001
            multi["single_process_fanout"] = {"error": repr(e)}

    # ---- roofline of the dominant kernel (G1 table MSM)
    peak, peak_src = imad_peak()
    # mixed additions per proof = (base, window) units the engine actually walks: identity points of the key
    # (variables absent from a matrix) are dropped at load and NOT counted as work
    g1_units, g2_units, g1_rows, g2_rows = work
    ms_g1, n_g1 = regions["msm_g1"]
    imad_per_launch = P * g1_units * M_MADD_G1 * IMAD_PER_MUL
    achieved = imad_per_launch / (ms_g1 / max(n_g1, 1) * 1e-3) if ms_g1 else 0.0
    bytes_per_launch = P * g1_units * (64 + 4)       # one 64 B table point + one int32 digit per madd
    roofline = {
        "bound": "imad", "kernel": "k_msm_batch<Fq> + k_msm_reduce<Fq> (G1 fixed-base table MSM)",
        "achieved": achieved / 1e12, "peak": peak / 1e12, "unit": "T IMAD/s", "frac": achieved / peak,
        "peak_source": peak_src, "traffic": ncu_traffic("k_msm_batch<Fp<FqParams>"),
        "traffic_note": "DRAM bytes per launch from profiles/r2_ncu_msm_batch.txt (ncu --set full of the shipped kernel: 128 "
                        "registers, 4 CTAs per SM, 5312-CTA grid); algorithmic bytes "
                        "are in hbm.algorithmic_bytes_per_launch - 64 B table entries are fetched as 128 B lines",
        "algorithmic_imad_per_launch": imad_per_launch, "avg_launch_ms": ms_g1 / max(n_g1, 1),
        "algorithmic_note": "SURVEY.md 8d unit: a mixed add = 10 Montgomery products of 272 IMAD; the kernel executes "
                            "fewer (executed.*: shared reductions), so frac is useful work over peak, executed.frac is "
                            "the pipe utilisation",
        "executed": {"imad_per_launch": P * g1_units * IMAD_EXEC_MADD_G1,
                     "frac": (P * g1_units * IMAD_EXEC_MADD_G1 / (ms_g1 / max(n_g1, 1) * 1e-3) / peak) if ms_g1 else 0.0},
        "mixed_adds_per_proof": {"g1": g1_units, "g2": g2_units, "g1_bases": g1_rows, "g2_bases": g2_rows,
                                 "note": "non-identity bases x windows; the key's identity points are not counted"},
        "share_of_step": ms_g1 / ms,
        "hbm": {"algorithmic_bytes_per_launch": bytes_per_launch,
                "achieved_gbs": bytes_per_launch / (ms_g1 / max(n_g1, 1) * 1e-3) / 1e9 if ms_g1 else 0.0,
                "peak_gbs": measured_hbm(), "note": "table gathers; the kernel is IMAD-bound, not HBM-bound"},
        "stage_ms_per_step": {k: v[0] / args.steps for k, v in regions.items()},
        "g2_msm": {"algorithmic_imad_per_launch": P * g2_units * M_MADD_G2 * IMAD_PER_MUL,
                   "achieved": (P * g2_units * M_MADD_G2 * IMAD_PER_MUL) / (regions["msm_g2"][0] / max(regions["msm_g2"][1], 1) * 1e-3) / 1e12
                   if regions["msm_g2"][0] else 0.0, "unit": "T IMAD/s",
                   "executed_frac": (P * g2_units * IMAD_EXEC_MADD_G2) / (regions["msm_g2"][0] / max(regions["msm_g2"][1], 1) * 1e-3) / peak
                   if regions["msm_g2"][0] else 0.0},
    }

    # ---- CPU baseline on a bounded sample (rank 0, N=1 only)
    cpu = None
    if world == 1 and not args.no_cpu:
        from oracle import c_oracle as co
        co.build()
        circ = co.Circuit("equality")
        opk = co.ProvingKey(pk_bytes)
        cores = host_cores()
        sample = min(P, max(cores * 16, 64))
        co.prove_batch(circ, opk, a_h[:cores], a_h[:cores], None, None, r_h[:cores], s_h[:cores], threads=cores)
        t0 = time.perf_counter()
        want, wstat = co.prove_batch(circ, opk, a_h[:sample], a_h[:sample], None, None, r_h[:sample], s_h[:sample],
                                     threads=cores)
        dt = time.perf_counter() - t0
        assert np.array_equal(want, proofs_h[:sample]), "GPU proofs differ from the CPU oracle's"
        cpu = {"value": sample / dt, "unit": "proofs/s", "cores": cores, "kind": "port",
               "sample": f"first {sample} proofs of the step's {P}, proof-parallel over {cores} OpenMP threads; "
                         "bytes compared equal to the GPU's"}

    extra = {}
    if world == 1 and not args.no_extra:
        lat = {}
        for nb in (1, 8, 64, 512):                  # BASELINE.json configs[0]: latency of small calls, host buffers
            for _ in range(3):
                pk.prove_equality_batch(a_p[:nb], a_p[:nb], r_p[:nb], s_p[:nb])
            t0 = time.perf_counter()
            for _ in range(10):
                pk.prove_equality_batch(a_p[:nb], a_p[:nb], r_p[:nb], s_p[:nb])
            lat[str(nb)] = round(1e2 * (time.perf_counter() - t0), 3)
        pk.close()                                  # free the 60 GB of tables before the other workloads load theirs
        extra = bench_transforms(engine, torch, dev, args)
        extra["latency_ms_by_batch_size"] = lat
        try:
            extra["api_process_batch"] = bench_python_api(pk_bytes, P)
        except Exception as e:  # noqa: BLE001
            extra["api_process_batch"] = {"error": repr(e)}

    out = {
        "metric": "groth16_bn254_proofs_per_sec_batched", "value": value, "unit": "proofs/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u256 (8x32-bit Montgomery limbs, integer)",
        "data": "synthetic", "config": config_dict(args), "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
        "roofline": roofline, "cpu_baseline": cpu, "extra": {**extra, **multi}, "engine": engine_info,
    }
    print(json.dumps(out))


def _np_fr(rng, n):
    """n canonical Fr scalars (below 2^252 < r), 32 B little-endian each."""
    w = rng.integers(0, 2**63, size=(n, 4), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=(n, 4), dtype=np.uint64)
    w[:, 3] &= np.uint64(0x0FFFFFFFFFFFFFFF)
    return w.view(np.uint8).reshape(n, 32).copy()


def bench_sharded_proof(torch, dist, dev, rank, world, rounds=349524, iters=5):
    """BASELINE.json configs[3]: ONE proof of the 2^20-constraint circuit split across the N ranks (point ranges of the
    five MSMs per rank, one NCCL gather of partial sums; libzkp_b200/multi.py).  ms per proof = device time, max over
    ranks; rank 0 then proves the same statement on one GPU from the unsharded key and the bytes must be identical."""
    from libzkp_b200 import engine
    from libzkp_b200.multi import ShardedProver
    pk_bytes, _ = engine.setup_builtin(engine.EQUALITY, rounds, toxic(1))       # deterministic: identical on every rank
    t0 = time.perf_counter()
    sp = ShardedProver(pk_bytes, engine.EQUALITY, rounds, rank, world, dev)
    t_load = time.perf_counter() - t0
    z = engine.builtin_witness(engine.EQUALITY, rounds, 6, 6) if rank == 0 else None
    r, s = fr_bytes(4, 1)[0].tobytes(), fr_bytes(40, 1)[0].tobytes()
    proof = sp.prove(z, r, s)
    for _ in range(2):
        sp.prove(resident=True)
    torch.cuda.synchronize()
    dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(iters):
        sp.prove(resident=True)
    ev1.record()
    torch.cuda.synchronize()
    t = torch.tensor([ev0.elapsed_time(ev1) / iters], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out = {"n_gpus": world, "constraints": 3 * rounds + 2, "domain": sp.n, "ms_per_proof": float(t.item()),
           "shard_pk_load_s": t_load, "collectives_per_proof": sp.collectives_per_proof,
           "witness_map_ranks": sp.map_ranks}
    if rank == 0:
        full = engine.ProvingKey(pk_bytes)
        full.circuit_builtin(engine.EQUALITY, rounds)
        rr, ss = np.frombuffer(r, np.uint8)[None], np.frombuffer(s, np.uint8)[None]
        want, status = full.prove_batch(z[None], rr, ss)
        d_z = torch.from_numpy(z).to(dev)
        d_rs = torch.from_numpy(np.concatenate([rr, ss])).to(dev)
        d_p, d_st = torch.zeros(256, dtype=torch.uint8, device=dev), torch.zeros(1, dtype=torch.int32, device=dev)
        st = torch.cuda.current_stream().cuda_stream
        one = lambda: full.prove_batch_device(1, d_z.data_ptr(), d_rs[0].data_ptr(), d_rs[1].data_ptr(), d_p.data_ptr(),
                                              d_st.data_ptr(), st)
        one(); one()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(iters):
            one()
        ev1.record()
        torch.cuda.synchronize()
        out["one_gpu_ms_per_proof"] = ev0.elapsed_time(ev1) / iters
        out["speedup_vs_one_gpu"] = out["one_gpu_ms_per_proof"] / out["ms_per_proof"]
        out["bytes_identical_to_one_gpu_proof"] = bool(not status.any() and want[0].tobytes() == proof)
        assert out["bytes_identical_to_one_gpu_proof"], "sharded proof differs from the single-GPU proof"
        full.close()
    sp.close()
    return out


def bench_replicas(torch, dist, dev, rank, world):
    """The stand-alone transforms do not shard (DESIGN.md section 6: replicas only): every rank runs its own 2^20 G1 MSM
    and 2^22 NTT at the same time; the aggregate is the sum, the slowest rank is reported beside it."""
    from libzkp_b200 import transforms
    peak, _ = imad_peak()
    dist.barrier()
    m = transforms.bench_msm(torch, dev, peak, 20, 1)
    dist.barrier()
    t = transforms.bench_ntt(torch, dev, peak, measured_hbm(), 22)
    v = torch.tensor([m["points_per_s"], t["elements_per_s"], -m["points_per_s"], -t["elements_per_s"]], device=dev, dtype=torch.float64)
    tot = v.clone()
    dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    mx = v.clone()
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    return {"n_gpus": world, "msm_g1_2^20_points_per_s_total": float(tot[0]), "msm_g1_2^20_points_per_s_slowest_rank": float(-mx[2]),
            "msm_g1_2^20_frac_of_imad_peak_rank0": m["imad_frac_of_measured_peak"], "msm_result_checked": m["result_equals_sum_k_s_times_G"],
            "ntt_2^22_elements_per_s_total": float(tot[1]), "ntt_2^22_elements_per_s_slowest_rank": float(-mx[3]),
            "what": "independent replicas, one per GPU, timed side by side (no collective: these transforms do not shard)"}


def bench_mixed_sharded(torch, dist, dev, rank, world, total=65536, iters=3):
    """BASELINE.json configs[4]: a 65 536-proof mixed batch (even operations equality, odd ones membership with 64
    slots) sharded proof-parallel over the N ranks, both keys resident on every GPU; host buffers in, libzkp envelopes
    out, INCLUDING the gather of all proof bytes to rank 0 (the reference hands a batch's results to one caller).
    Wall clock between barriers, max over ranks."""
    from libzkp_b200 import engine, parallel
    pk_e = engine.ProvingKey(engine.setup_builtin(engine.EQUALITY, 110, toxic(1))[0])
    pk_e.circuit_builtin(engine.EQUALITY, 110)
    pk_m = engine.ProvingKey(engine.setup_builtin(engine.MEMBERSHIP, 64, toxic(1))[0])
    pk_m.circuit_builtin(engine.MEMBERSHIP, 64)
    half = total // 2
    rng = np.random.default_rng(7)                   # same seed on every rank: every rank holds the whole batch
    a = rng.integers(0, 2**63, size=half, dtype=np.uint64)
    sets = rng.integers(0, 2**63, size=(half, 64), dtype=np.uint64)
    lens = np.full(half, 64, np.uint32)
    vals = sets[np.arange(half), np.arange(half) % 64].copy()
    r1, s1, r2, s2 = (_np_fr(rng, half) for _ in range(4))

    def once():
        return parallel.prove_mixed_enveloped_sharded(pk_e, pk_m, a, vals, sets, lens, r1, s1, r2, s2, rank, world, dev, dst=0)
    res = once()
    best = None
    for _ in range(iters):
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        res = once()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        best = float(t.item()) if best is None else min(best, float(t.item()))
    ok = True
    if rank == 0:
        env_e, len_e, st_e, env_m, len_m, st_m = res
        ok = (not st_e.any() and not st_m.any() and (len_e == 298).all() and (len_m == 302 + 8 * 64).all()
              and env_e.shape == (half, 298) and env_m.shape[0] == half)
        # spot check of the gathered bytes: rank 0 re-proves two operations of EVERY other rank's block
        for other in range(1, world):
            lo, _ = parallel.shard_range(half, other, world)
            chk, _, _ = pk_e.prove_equality_enveloped(a[lo:lo + 2], a[lo:lo + 2], r1[lo:lo + 2], s1[lo:lo + 2])
            ok = bool(ok and np.array_equal(chk, env_e[lo:lo + 2]))
    out = {"n_gpus": world, "proofs": total, "ms_per_batch": 1e3 * best, "proofs_per_s_e2e": total / best,
           "all_ok_and_gather_checked": ok, "tables_gb_per_gpu": (pk_e.table_bytes + pk_m.table_bytes) / 1e9,
           "window_bits": [pk_e.window_bits, pk_m.window_bits],
           "what": "host buffers -> envelopes gathered on rank 0 (one NCCL gather of bytes per kind), best of %d" % iters}
    assert ok, "mixed sharded batch: failed proofs or gathered bytes differ"
    pk_e.close()
    pk_m.close()
    return out


def bench_fanout(torch, world, pk_bytes, window_bits, P, a_p, r_p, s_p, proofs_block0, e2e_one_job, steps):
    """ONE process, N GPUs (the reference's batch path is one process: src/advanced/batch.rs:110-140): lzkp_init with
    all N devices replicates the key; a single lzkp_prove_equality_batch call of N x P proofs fans out, one host
    thread per device, results in disjoint slices of the caller's buffer.  Rank 0 runs this alone after the other
    ranks have exited."""
    from libzkp_b200 import engine
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < 120:                 # the other ranks' processes release their devices as they exit
        if all(torch.cuda.mem_get_info(d)[0] > 150e9 for d in range(1, world)):
            break
        time.sleep(0.5)
    engine.init(list(range(world)))
    t0 = time.perf_counter()
    pk = engine.ProvingKey(pk_bytes, window_bits=window_bits)
    pk.circuit_builtin(engine.EQUALITY, 110)
    t_load = time.perf_counter() - t0
    n = world * P
    rep = lambda x: torch.from_numpy(np.ascontiguousarray(np.concatenate([x] * world)).view(np.uint8)).pin_memory().numpy()
    a, r, s = rep(a_p).view(np.uint64), rep(r_p).reshape(n, 32), rep(s_p).reshape(n, 32)
    pinned = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory().numpy()
    out = (pinned((n, 256), torch.uint8), pinned((n, 32), torch.uint8), pinned((n,), torch.int32))    # caller-owned result buffers
    proofs, _, status = pk.prove_equality_batch(a, a, r, s, out=out)
    ok = bool(not status.any() and all(np.array_equal(proofs[g * P:(g + 1) * P], proofs_block0) for g in range(world)))
    t0 = time.perf_counter()
    for _ in range(steps):
        pk.prove_equality_batch(a, a, r, s, out=out)
    dt = (time.perf_counter() - t0) / steps
    pk.close()
    assert ok, "fan-out proofs differ from the one-GPU proofs of the same inputs"
    res = {"devices": world, "proofs_per_call": n, "ms_per_call": 1e3 * dt, "proofs_per_s_e2e": n / dt,
           "vs_n_processes_e2e": (n / dt) / e2e_one_job, "bytes_equal_one_gpu_proofs": ok, "pk_load_all_devices_s": t_load,
           "api": "one lzkp_prove_equality_batch call, host buffers, one process"}
    # BASELINE.json configs[4] the way the reference would run it: ONE process, one grouped call per circuit, every call
    # fanned out over all GPUs, envelopes written straight into the caller's buffers (no gather step at all)
    try:
        total = 65536
        half = total // 2
        pk_e = engine.ProvingKey(engine.setup_builtin(engine.EQUALITY, 110, toxic(1))[0])
        pk_e.circuit_builtin(engine.EQUALITY, 110)
        pk_m = engine.ProvingKey(engine.setup_builtin(engine.MEMBERSHIP, 64, toxic(1))[0])
        pk_m.circuit_builtin(engine.MEMBERSHIP, 64)
        rng = np.random.default_rng(7)
        av = rng.integers(0, 2**63, size=half, dtype=np.uint64)
        sets = rng.integers(0, 2**63, size=(half, 64), dtype=np.uint64)
        lens = np.full(half, 64, np.uint32)
        vals = sets[np.arange(half), np.arange(half) % 64].copy()
        r1, s1, r2, s2 = (_np_fr(rng, half) for _ in range(4))

        def once():
            ee, le, se = pk_e.prove_equality_enveloped(av, av, r1, s1)
            em, lm, sm = pk_m.prove_membership_enveloped(vals, sets, lens, r2, s2)
            return int((se != 0).sum() + (sm != 0).sum()), ee, em
        once()
        best = None
        for _ in range(3):
            t0 = time.perf_counter()
            failed, ee, em = once()
            d = time.perf_counter() - t0
            best = d if best is None else min(best, d)
        res["mixed_batch_65536_one_process"] = {"proofs": total, "ms_per_batch": 1e3 * best, "proofs_per_s_e2e": total / best,
                                                "failed": failed, "window_bits": [pk_e.window_bits, pk_m.window_bits]}
        pk_e.close()
        pk_m.close()
    except Exception as e:  # noqa: BLE001
        res["mixed_batch_65536_one_process"] = {"error": repr(e)}
    return res


def bench_python_api(pk_bytes, P):
    """The same batch through the Python mirror of the reference's API: create_proof_batch /
    batch_add_equality_proof x P / process_batch (validation, OS randomness, device call, envelopes)."""
    import libzkp_b200 as zk
    from libzkp_b200 import snark
    snark.reset()
    snark.configure(generator=lambda prefix: (pk_bytes, b""))
    vals = u64s(3, P)
    try:
        def once():
            bid = zk.create_proof_batch()
            for v in vals:
                zk.batch_add_equality_proof(bid, int(v), int(v))
            t0 = time.perf_counter()
            out = zk.process_batch(bid)
            return time.perf_counter() - t0, out
        once()
        dt, out = min((once() for _ in range(3)), key=lambda x: x[0])
        assert len(out) == P and all(len(p) == 298 for p in out)
        return {"proofs_per_s": P / dt, "ms_per_batch": 1e3 * dt, "what": "process_batch(batch of %d equality ops), "
                "Python host mirror incl. OS randomness and 298-byte envelopes" % P}
    finally:
        snark.reset()
        snark.configure()


def measured_hbm():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        return 6650.0


def bench_transforms(engine, torch, dev, args):
    """BASELINE.json's other two metrics: G1 MSM points/s @2^20, NTT elements/s @2^22 (device-resident)."""
    out = {}
    try:
        from libzkp_b200 import transforms
    except ImportError:
        return {"note": "large MSM / NTT device-resident entry points not built in this revision"}
    try:
        out.update(transforms.bench(torch, dev, imad_peak()[0], measured_hbm()))
    except Exception as e:  # noqa: BLE001
        out["error"] = repr(e)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--chunk", type=int, default=0, help="proofs per device pass (0 = engine default)")
    ap.add_argument("--window-bits", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--ref-sample", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's proofs and "
                    "status codes (rank 0's) as .npy files in DIR")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
