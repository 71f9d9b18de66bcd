#!/usr/bin/env python
"""Headline benchmark: OILMM logpdf + posterior evals/s at p=64, m=64, N=16384 (BASELINE.json
config 4), Float64, latents block-sharded over the ranks (strong scaling of one eval).

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's CPU path (oracle port) on host cores

One step = one eval = logpdf(fx, y) AND posterior(fx, y) on the same (fx, y), one shared
factorisation per latent (the reference factorises twice; SURVEY.md §8d counts it once).
Timed path (default): the wide Cholesky updates run as integer-slice products on the int8 tensor cores (--ozaki 7 --ozaki-bits 8:
library options "ozaki" / "ozaki_bits"; FP64 results to ~1e-13, checked in every line against the CPU oracle (`parity_check`) and
against the library's default all-FP64 DMMA path, which is measured in the same process (`dmma_path`); --ozaki 0 times that path).
`value`: inputs x, y already resident in HBM (device pointers through the C ABI), timed with the
CUDA events liblmm records on its own compute stream around all device work of the call.
`e2e`: the same call with pinned HOST buffers, H2D/D2H inside the timed region, wall clock between
device-synchronised points.  Prints ONE JSON line on rank 0.
`--dump-outputs DIR`: rank 0 writes what the last device-resident timed step returned as DIR/*.npy (see `dump_outputs`); the
inputs depend on the arguments only, so two builds run with the same arguments can be compared file for file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "OILMM logpdf+posterior evals/s (p=64,m=64,N=16384); % FP64 TC peak"
UNIT = "evals/s"


def workload(p, m, N, seed=0):
    """SURVEY.md §8d synthetic inputs (identical bytes for GPU and oracle)."""
    rng = np.random.default_rng(seed)
    x = np.sort(rng.uniform(0.0, N / 100.0, N))
    rngH = np.random.default_rng(seed + 1)
    U, S, _ = np.linalg.svd(rngH.uniform(0.0, 1.0, size=(p, m)), full_matrices=False)
    rngK = np.random.default_rng(seed + 2)
    inv_ls = rngK.uniform(0.5, 2.0, m)
    # y = H f + eps with f from random Fourier features of each latent's SE kernel (O(1) values)
    nfeat = 64
    H = U * np.sqrt(S)[None, :]
    F = np.empty((m, N))
    for i in range(m):
        w = rng.standard_normal(nfeat) * inv_ls[i]
        b = rng.uniform(0, 2 * np.pi, nfeat)
        a = rng.standard_normal(nfeat)
        F[i] = np.sqrt(2.0 / nfeat) * (np.cos(np.outer(x, w) + b) @ a)
    sigma2 = 0.1
    Y = H @ F + np.sqrt(sigma2) * rng.standard_normal((p, N))
    return x, np.ascontiguousarray(U), np.ascontiguousarray(S), inv_ls, Y.reshape(-1).copy(), sigma2


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def fp64_peak_tflops():
    """Roofline denominator: MEASURED_PEAKS.json carries no FP64 number, so the measured cuBLAS
    DGEMM rate on this pool's B200 (tools/microbench/fp64_peak.cu -> profiles/r01_fp64_peaks.json)
    is used; fallback = the same figure hard-coded."""
    try:
        with open(os.path.join(ROOT, "profiles", "r01_fp64_peaks.json")) as fh:
            d = json.load(fh)
        return float(d["cublas"]["dgemm_nt_8192_sustained"]), "measured cuBLAS DGEMM 8192^3 sustained (profiles/r01_fp64_peaks.json)"
    except Exception:
        return 35.9, "fallback: cuBLAS DGEMM 8192^3 measured earlier on this pool"


def ncu_traffic(p, N, mloc):
    """DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of the Cholesky launch sequence of
    one step on one rank, from the committed ncu pass over a full C4 eval
    (profiles/r02_launches_c4_summary.json, falling back to round 1's: 64 latents); per-latent work is independent, so a rank
    holding mloc latents moves mloc/64 of it.  null for any other problem size."""
    for name in ("r02_launches_c4_summary.json", "r01_launches_c4_summary.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as fh:
                d = json.load(fh)
            if p == 64 and N == 16384:
                return d["cholesky_sequence"]["dram_bytes_per_step"] * mloc / 64.0
        except Exception:
            continue
    return None


def host_cores():
    """Host threads this process may run on (the affinity mask, not the machine's CPU count)."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def blas_threads(n):
    """All host threads for OpenBLAS regardless of the environment: torch.distributed.run exports OMP_NUM_THREADS=1 to
    its workers, which would silently turn the CPU arm into a one-thread run (VERDICT r01, weak #2b)."""
    from threadpoolctl import threadpool_limits

    return threadpool_limits(limits=int(n))


def blas_description():
    from threadpoolctl import threadpool_info

    blas = [d for d in threadpool_info() if d.get("user_api") == "blas"]
    return (blas[0].get("internal_api", "?") + " " + str(blas[0].get("version", "?")) + f" threads={blas[0].get('num_threads')}") if blas else "?"


def cpu_latent_eval(x, inv_ls_i, noise_i, delta, threads, once=False):
    """Reference structure for ONE latent at FULL N (oracle port): logpdf builds the kernel matrix and factorises,
    posterior does both again (src/oilmm.jl:90 and :128).  Returns (seconds, lml term).
    once=False: both passes are executed (o.gp_logpdf + o.gp_posterior).
    once=True : every phase is executed and timed ONCE at full N and the reference's repeats of the IDENTICAL operation
    are counted by multiplicity (2 kernel-matrix builds, 2 dpotrf, 2 forward solves, 1 backward solve) -- no scaling in
    N, so no assumption about how dpotrf efficiency changes with size."""
    import scipy.linalg as sla

    from oracle import lmm_oracle as o

    f = o.GP(o.Kernel(o.SE, 1.0, float(inv_ls_i)))
    with blas_threads(threads):
        if not once:
            t0 = time.perf_counter()
            lml = o.gp_logpdf(f, x, float(noise_i), delta)
            post = o.gp_posterior(f, x, float(noise_i), delta)
            dt = time.perf_counter() - t0
            del post
            return dt, lml
        n = len(x)
        t0 = time.perf_counter()
        C = o.kernelmatrix(f.kernel, x)
        C[np.diag_indices_from(C)] += float(noise_i)
        t1 = time.perf_counter()
        L = sla.cholesky(C, lower=True, check_finite=False)
        t2 = time.perf_counter()
        del C
        z = sla.solve_triangular(L, delta, lower=True, check_finite=False)
        t3 = time.perf_counter()
        sla.solve_triangular(L, z, lower=True, trans="T", check_finite=False)
        t4 = time.perf_counter()
        lml = -0.5 * (n * o.LOG2PI + 2.0 * float(np.sum(np.log(np.diag(L)))) + float(z @ z))
        return 2 * (t1 - t0) + 2 * (t2 - t1) + 2 * (t3 - t2) + (t4 - t3), lml


def run_reference(args, cfg):
    """--impl reference: the reference's own CPU implementation of the path.  Julia cannot run in
    this image (SURVEY.md §8c), so this is the oracle port on all host cores; each step is a
    bounded sample -- one latent of m at FULL N, reference structure -- extrapolated linearly in m
    (the m latents are independent, identical-size problems the reference maps over serially, src/oilmm.jl:90)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    p, m, N = cfg["p"], cfg["m"], cfg["N"]
    cores = host_cores()
    x, U, S, inv_ls, y, s2 = workload(p, m, N)
    T = U.T / np.sqrt(S)[:, None]
    delta = T[0] @ y.reshape(p, N)
    noise0 = s2 / S[0]
    # keep the whole run within minutes whatever K and W are, ALWAYS at full N: both passes executed when W + K <= 6,
    # else each phase executed once per step and counted by its multiplicity in the reference (identical repeats)
    once = (args.warmup + args.steps) > 6
    for _ in range(min(args.warmup, 2) if once else args.warmup):  # CPU BLAS has no clock ramp to warm: 2 passes fault the pages in
        cpu_latent_eval(x, inv_ls[0], noise0, delta, cores, once)
    times = []
    for _ in range(args.steps):
        dt, _ = cpu_latent_eval(x, inv_ls[0], noise0, delta, cores, once)
        times.append(dt)
    per_eval = float(np.mean(times)) * m
    with blas_threads(cores):
        blas = blas_description()
    val = 1.0 / per_eval
    sample = (f"1 of {m} latents at full N={N} per step (2 kernel-matrix builds + 2 dpotrf + 3 triangular solves, reference structure"
              + (", each phase executed once per step and counted by its multiplicity" if once else ", every pass executed")
              + f"), x{m} extrapolated")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": per_eval * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": cfg["config"],
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "blas": blas,
                         "sample_seconds": float(np.sum(times)), "extrapolated_seconds_per_eval": per_eval},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def int8_peak_tops(sm_mhz=1965.0):
    """Dense int8 tensor peak of this pool's B200: the per-SM rate MEASURED by tools/microbench/i8_mma.cu in SM cycles (8190 MAC/clk/SM
    = the nominal 8192; profiles/r02_i8_mma*.jsonl) x 148 SMs x 2 x the SM clock sampled during the run -- 4.76 POPS at 1965 MHz (NVIDIA's
    nominal 4.5 POPS assumes a lower clock).  The wall-clock rate of the microbenchmark's own 1 ms kernels (4.09 POPS, launch included)
    is a LOWER bound and was what earlier lines of this round used.  MEASURED_PEAKS.json has no int8 entry."""
    best = 0.0
    for name in ("r02_i8_mma.jsonl", "r02_i8_mma_2cta.jsonl"):
        try:
            for ln in open(os.path.join(ROOT, "profiles", name)):
                d = json.loads(ln)
                if "rate" in d.get("test", ""):
                    best = max(best, float(d.get("mac_per_clk_per_sm", 0.0)))
        except Exception:
            pass
    if best > 0:
        return 148 * best * 2 * sm_mhz * 1e6 / 1e12, (f"measured {best:.0f} int8 MAC/clk/SM (tools/microbench/i8_mma.cu, profiles/r02_i8_mma*.jsonl) x 148 SM x 2 x "
                                                      f"{sm_mhz:.0f} MHz (median SM clock sampled during the timed region); nominal dense int8: 4500")
    return 4500.0, "nominal dense int8 (no measurement file)"


def ncu_traffic_ozaki():
    """dram bytes (read + write) of ONE launch of the int8 update from the committed ncu --set full capture (profiles/r02_ncu_ozaki.json)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_ozaki.json")))
        return d["ozaki_update_kernel"]["dram_bytes_per_launch"]
    except Exception:
        return None


DUMP_SAMPLES = 1 << 20


def seeded_sample(a, k, seed):
    """`a` itself if it has at most k entries, else k of its entries at positions drawn from a fixed seed."""
    if a.size <= k:
        return a
    return np.ravel(a)[np.random.default_rng(seed).choice(a.size, size=k, replace=False)]


def dump_outputs(path, post, lp, latents, N):
    """What a caller of the timed path receives from one step, as float64 .npy files (at most 48 MB in all):
    logpdf.npy   -- (1,) the log marginal likelihood;
    alpha.npy    -- the posterior weights alpha_i = (K_i + noise_i I)^-1 delta_i, one row per latent in `latents` (at most 2^21
                    values: a fixed, seeded sample of a larger array);
    delta.npy    -- the projected observations delta_i the posterior holds, sampled the same way;
    L_sample.npy -- (2, k) entries of the lower Cholesky factors of the first and of the last latent in `latents`, at the same
                    2^20 seeded lower-triangle positions in both (a factor has N^2 entries)."""
    os.makedirs(path, exist_ok=True)
    lat = post.f.fs
    np.save(os.path.join(path, "logpdf.npy"), np.array([lp], dtype=np.float64))
    vec = np.array([lat[i]._export()[1:] for i in latents])  # (latents, 2, N): alpha, delta
    np.save(os.path.join(path, "alpha.npy"), seeded_sample(vec[:, 0], 2 * DUMP_SAMPLES, 1))
    np.save(os.path.join(path, "delta.npy"), seeded_sample(vec[:, 1], 2 * DUMP_SAMPLES, 2))
    rng = np.random.default_rng(3)
    k = min(DUMP_SAMPLES, N * (N + 1) // 2)
    r, c = rng.integers(0, N, k), rng.integers(0, N, k)
    rows, cols = np.maximum(r, c), np.minimum(r, c)
    L_sample = np.empty((2, k))
    for j, i in enumerate((latents[0], latents[-1])):
        L_sample[j] = lat[i].C[rows, cols]
    np.save(os.path.join(path, "L_sample.npy"), L_sample)


def multi_gpu_extras(lmm, ctx, dist, torch, world, rank):
    """Driver-visible records of the two other multi-GPU paths of the north star, run by every rank AFTER the timed region
    (they are collective) and attached to rank 0's JSON line; neither touches `value`.
    (1) `ilmm_rowcyclic`: ONE large factor (general-ILMM-shaped work, N = 16384) factored by every rank on identical
        inputs, replicated vs row-cyclic partitioned over the ranks (option "partition_ilmm": trailing updates split by tile
        row, one ncclAllGather of the current block column per step); time = max over ranks, parity = logdet.
    (2) `c5_sweep`: BASELINE config 5 -- OILMM p = 256, m = 128, N = 8192, 32 lengthscale settings in one
        lmm_oilmm_logpdf_sweep call, the (sweep x latent) grid of 4096 factorizations block-sharded over the ranks."""
    from tools.chol_bench import run

    def maxed(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    out = {}
    rec = {"N": 16384, "ranks": world}
    # the partitioned schedules run the FP64 DMMA trailing update: compare like with like (int8 option off), then note what the
    # int8 update does for the unpartitioned factor on one GPU
    oz_saved = int(getattr(ctx, "_bench_ozaki", 0))
    if oz_saved:
        ctx.set_option("ozaki", oz_saved)
        ms_oz, _, ld_oz = run(ctx, 16384, 1, reps=2)
        rec["replicated_int8_update_ms"] = maxed(ms_oz)
        rec["replicated_int8_update_logdet"] = ld_oz
    ctx.set_option("ozaki", 0)
    for part, key in ((0, "replicated"), (1, "rowcyclic")):
        ctx.set_option("partition_ilmm", part)
        dist.barrier()
        ms, _, ld = run(ctx, 16384, 1, reps=2)
        rec[key + "_ms"] = maxed(ms)
        rec[key + "_logdet"] = ld
    ctx.set_option("partition_ilmm", 0)
    rec["speedup"] = rec["replicated_ms"] / rec["rowcyclic_ms"]
    rec["logdet_rel_diff"] = abs(rec["rowcyclic_logdet"] - rec["replicated_logdet"]) / abs(rec["replicated_logdet"])
    rec["tflops_rowcyclic"] = 16384 ** 3 / 3.0 / (rec["rowcyclic_ms"] * 1e-3) / 1e12
    out["ilmm_rowcyclic"] = rec
    # the same joint dimension through the public API (lmm.logpdf of a general ILMM, p = 8, m = 4, N = 4096): replicated vs row-cyclic vs
    # row-cyclic with DISTRIBUTED STORAGE (each rank assembles and keeps 1/G of the joint matrix; "partition_ilmm" = 2)
    from tools.multigpu_ilmm import ilmm_logpdf_record

    out["ilmm_distributed"] = ilmm_logpdf_record(lmm, ctx, dist, torch, 8, 4, 4096)
    ctx.set_option("ozaki", oz_saved)
    p, m, N, nsweep = 256, 128, 8192, 32
    rng = np.random.default_rng(0)
    x = np.sort(rng.uniform(0, N / 100.0, N))
    U, S, _ = np.linalg.svd(np.random.default_rng(1).uniform(0, 1, (p, m)), full_matrices=False)
    f = lmm.ILMM(lmm.independent_mogp([lmm.GP(lmm.SEKernel()) for _ in range(m)]), lmm.Orthogonal(U, S))
    y = rng.standard_normal(p * N)
    fx = f(lmm.MOInputIsotopicByOutputs(x, p), 0.1)
    scales = np.geomspace(0.25, 4.0, nsweep)
    lmm.logpdf_sweep(fx, y, scales)  # warm-up
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    vals = lmm.logpdf_sweep(fx, y, scales)
    torch.cuda.synchronize()
    sec = maxed(time.perf_counter() - t0)
    flops = m * nsweep * N ** 3 / 3.0
    out["c5_sweep"] = {"config": f"BASELINE config 5: OILMM p={p} m={m} N={N} x {nsweep} lengthscales in one call", "n_gpus": world,
                       "seconds_per_call": sec, "factorizations": m * nsweep, "tflops_total": flops / sec / 1e12,
                       "tflops_per_gpu": flops / sec / 1e12 / world, "trailing_update": (f"int8 digit planes: {oz_saved}" if oz_saved else "FP64 DMMA"),
                       "logpdf_at_scale_1": float(vals[int(np.argmin(np.abs(scales - 1.0)))]),
                       "argmax_scale": float(scales[int(np.argmax(vals))])}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--p", type=int, default=64)
    ap.add_argument("--m", type=int, default=64)
    ap.add_argument("--N", type=int, default=16384)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the untimed multi-GPU records (row-cyclic ILMM factor, config-5 sweep)")
    ap.add_argument("--ozaki", type=int, default=7, help="digit planes (6/7/8) of the integer-slice (int8 tcgen05) trailing update of the timed path; "
                                                          "0 = FP64 DMMA only (the library's own default; always measured beside it as `dmma_path`)")
    ap.add_argument("--ozaki-bits", type=int, default=8, help="bits per digit plane: 7 = radix 128 (8 planes = 55 bits), 8 = radix 256 (7 planes = 54 bits)")
    ap.add_argument("--no-dmma", action="store_true", help="skip the untimed kernel-timing pass and the DMMA comparison (for runs under ncu)")
    ap.add_argument("--streams", type=int, default=0, help="latent groups on separate CUDA streams (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/*.npy (float64, seeded samples of "
                                                          "large arrays) for output-for-output comparison of two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 implementation")
    p, m, N = args.p, args.m, args.N
    cfg = {"p": p, "m": m, "N": N,
           "config": {"workload": ("BASELINE config 4" if (p, m, N) == (64, 64, 16384) else "reduced shape (NOT the headline config)") + f": OILMM p={p} m={m} N={N} SEKernel (per-latent lengthscales), sigma2=0.1, "
                                  "logpdf+posterior per eval, one shared factorisation per latent",
                      "partition": f"latents block-sharded over {args.gpus} rank(s); one NCCL all-reduce of m+1 lml terms",
                      "l2": f"working set (packed-lower factors, {8.0 * N * (N + 1) / 2 / 1e9:.2f} GB per latent, {m} latents) >> 126 MB L2: no flush needed"}}
    if args.impl == "reference":
        return run_reference(args, cfg)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import lmm_b200 as lmm

    ctx = lmm.Context(local)
    lmm.set_default_context(ctx)
    if world > 1:
        lmm.dist.init_context_distributed(ctx)
    if args.streams > 0:
        ctx.set_option("streams", args.streams)
    ctx.set_option("ozaki", args.ozaki)
    ctx.set_option("ozaki_bits", args.ozaki_bits)
    ctx._bench_ozaki = args.ozaki

    x, U, S, inv_ls, y, s2 = workload(p, m, N)
    H = lmm.Orthogonal(U, S)
    fs = [lmm.GP(lmm.SEKernel().compose(lmm.ScaleTransform(float(s)))) for s in inv_ls]
    f = lmm.ILMM(lmm.independent_mogp(fs), H)
    # HBM-resident inputs
    xd = torch.from_numpy(x.reshape(-1, 1)).cuda()
    yd = torch.from_numpy(y).cuda()
    fx_dev = f(lmm.MOInputIsotopicByOutputs(xd, p), s2)
    # pinned host inputs
    xh = torch.from_numpy(x.reshape(-1, 1).copy()).pin_memory()
    yh = torch.from_numpy(y.copy()).pin_memory()
    fx_host = f(lmm.MOInputIsotopicByOutputs(xh.numpy().reshape(-1), p), s2)
    yh_np = yh.numpy()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(fx, yy, keep=None):
        post, lp = lmm.posterior(fx, yy, with_logpdf=True)
        tm = ctx.last_timings().copy()
        if keep is not None:  # handed to the caller, which frees it
            keep.append(post)
        else:
            post.f.fs[0]._owner.free()
        return lp, tm

    for _ in range(args.warmup):
        lp, _ = step(fx_dev, yd)
    # ---- timed: device-resident
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    l0, h0, d0 = ctx.counters()
    ev_ms, chol_ms, kmat_ms, solve_ms, proj_ms = 0.0, 0.0, 0.0, 0.0, 0.0
    kept = []  # the last step's posterior when its outputs are dumped
    t0 = time.perf_counter()
    for k in range(args.steps):
        lp, tm = step(fx_dev, yd, kept if args.dump_outputs and k == args.steps - 1 else None)
        ev_ms += tm[0]; kmat_ms += tm[1]; chol_ms += tm[2]; solve_ms += tm[3]; proj_ms += tm[4]
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop() if rank == 0 else None
    l1, h1, d1 = ctx.counters()
    if kept:
        if rank == 0:
            dump_outputs(args.dump_outputs, kept[0], lp, range(*lmm.dist.shard_range(m, world, rank)), N)
        kept[0].f.fs[0]._owner.free()
        barrier()
    # ---- timed: end to end from pinned host buffers (public API call, H2D + D2H inside)
    step(fx_host, yh_np)
    barrier()
    lh0, hh0, dh0 = ctx.counters()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        lp_host, _ = step(fx_host, yh_np)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    lh1, hh1, dh1 = ctx.counters()

    stats = torch.tensor([ev_ms, wall_ms, e2e_ms, chol_ms], dtype=torch.float64, device="cuda")
    launches = torch.tensor([float(l1 - l0)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(launches, op=dist.ReduceOp.SUM)
    ev_ms, wall_ms, e2e_ms, chol_ms_max = [float(v) for v in stats.cpu()]

    # ---- untimed checks.  Every rank: the sharded eval once more, keeping the posterior, and the sharded prediction at 256
    # test points (rank-local back-projection partial sums + ONE ncclAllReduce of 2 p N* doubles, SURVEY.md §8e collective 2).
    Ns_chk = 256
    xs_chk = np.random.default_rng(7).uniform(0.0, N / 100.0, Ns_chk)
    terms = lmm.logpdf_terms(fx_dev, yd)  # all m + 1 terms on every rank (all-reduced inside the library)
    post_s, lp_s = lmm.posterior(fx_dev, yd, with_logpdf=True)
    M_s, V_s = lmm.mean_and_var(post_s(lmm.MOInputIsotopicByOutputs(xs_chk, p), s2))
    pred_ms = float(ctx.last_timings()[5])
    post_s.f.fs[0]._owner.free()
    barrier()
    # ---- untimed: (1) the int8 trailing-update kernel on its own -- one eval on ONE stream with CUDA events around every launch of
    # it (library option "ozaki_time"); (2) the same eval on the FP64 DMMA path (option "ozaki" = 0) for the step time it would have
    # had and for the difference of the results.
    oz_kernel = None
    dmma = None
    if args.ozaki and not args.no_dmma:
        ctx.set_option("streams", 1)
        ctx.set_option("ozaki_time", 1)
        ctx.last_timings()  # drop earlier events
        _, tmk = step(fx_dev, yd)  # (step() reads the timings itself: the event sum is consumed by that read)
        ctx.set_option("ozaki_time", 0)
        ctx.set_option("streams", args.streams if args.streams > 0 else 4)
        oz_kernel = {"ms": float(tmk[7]), "tile_products": float(tmk[5])}
        ctx.set_option("ozaki", 0)
        step(fx_dev, yd)
        barrier()
        dm_ms, dm_chol = 0.0, 0.0
        nd_steps = min(2, args.steps)
        for _ in range(nd_steps):
            lp_d, tmd = step(fx_dev, yd)
            dm_ms += tmd[0]; dm_chol += tmd[2]
        post_d, lp_d = lmm.posterior(fx_dev, yd, with_logpdf=True)
        M_d, V_d = lmm.mean_and_var(post_d(lmm.MOInputIsotopicByOutputs(xs_chk, p), s2))
        post_d.f.fs[0]._owner.free()
        ctx.set_option("ozaki", args.ozaki)
        barrier()
        dstats = torch.tensor([dm_ms / nd_steps, dm_chol / nd_steps], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(dstats, op=dist.ReduceOp.MAX)
        dmma = {"ms_per_step": float(dstats[0]), "cholesky_ms": float(dstats[1]), "steps": nd_steps, "logpdf": lp_d,
                "logpdf_rel_diff": abs(lp_s - lp_d) / abs(lp_d), "mean_relnorm": float(np.linalg.norm(M_s - M_d) / np.linalg.norm(M_d)),
                "var_max_rel": float(np.max(np.abs(V_s - V_d) / np.abs(V_d)))}
    extras = None
    if world > 1 and not args.no_extras:
        try:  # untimed records: a failure there (the same on every rank: identical inputs and calls) must not cost the timed result
            extras = multi_gpu_extras(lmm, ctx, dist, torch, world, rank)
        except Exception as exc:  # noqa: BLE001
            extras = {"extras_error": f"{type(exc).__name__}: {exc}"[:500]}
            ctx.set_option("partition_ilmm", 0)
            ctx.set_option("ozaki", args.ozaki)
    barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    K = args.steps
    ms_per_step = ev_ms / K
    value = 1e3 / ms_per_step
    mloc = (m * (rank + 1)) // world - (m * rank) // world
    peak, peak_src = fp64_peak_tflops()
    chol_flops = mloc * (N ** 3) / 3.0  # algorithmic potrf flops of one launch sequence on this rank
    achieved = chol_flops / (chol_ms_max / K * 1e-3) / 1e12
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    pipe_peak = 148 * 64 * 2 * sm_mhz * 1e6 / 1e12  # 64 FP64 FMA / clk / SM (DMMA and DFMA share it: profiles/r01_fp64_mix.json)
    if args.ozaki:
        cfg["config"]["trailing_update"] = (
            f"wide left-looking updates as an integer-slice (Ozaki) product on the int8 tensor cores: {args.ozaki} digit planes of {args.ozaki_bits} bits per FP64 operand "
            f"({6 + args.ozaki_bits * (args.ozaki - 1)} bits below the row scale), "
            f"{args.ozaki * (args.ozaki + 1) // 2} tcgen05.mma kind::i8 per 128^3 tile product, exact int32 accumulation in TMEM, FP64 recombination; panels, in-block "
            "updates, triangular solves, kernel matrices in FP64 (DMMA / DFMA).  The library default is DMMA everywhere (--ozaki 0): measured beside it as dmma_path")
    dmma_roofline = {"bound": "tensor", "kernel": "batched blocked Cholesky (gemm_tile_kernel_v2 DMMA updates + TRSM-as-GEMM + potrf_tile_kernel2)",
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": ncu_traffic(p, N, mloc),
                     "peak_source": peak_src, "flops_per_rank_step": chol_flops,
                     "fp64_pipe_peak": pipe_peak, "frac_of_fp64_pipe_peak": achieved / pipe_peak,
                     "fp64_pipe_peak_source": f"148 SM x 64 FMA/clk x 2 x {sm_mhz:.0f} MHz (median SM clock sampled during the timed region)",
                     "whole_eval_tflops": (m * (N ** 3 / 3.0 + 2.0 * N * N) + 4.0 * p * m * N) / (ms_per_step * 1e-3) / 1e12 / world}
    if args.ozaki and oz_kernel and oz_kernel["ms"] > 0:
        # dominant kernel of the timed path: the int8 wide update.  Algorithmic work of its launches = tile products x S(S+1)/2 MMAs x
        # 2 * 128^3 int8 ops, over the summed CUDA-event time of exactly those launches (one stream: serial).
        i8_peak, i8_src = int8_peak_tops(sm_mhz)
        nmma = args.ozaki * (args.ozaki + 1) // 2
        ops = oz_kernel["tile_products"] * nmma * 2.0 * 128 ** 3
        a_tops = ops / (oz_kernel["ms"] * 1e-3) / 1e12
        dd = dmma["cholesky_ms"] if dmma else None
        roof = {"bound": "tensor", "kernel": f"ozaki_update_kernel<{args.ozaki}> (tcgen05.mma.cta_group::1.kind::i8, TMEM int32 accumulators, TMA bulk-copy ring)",
                "achieved": a_tops, "peak": i8_peak, "unit": "TOP/s", "frac": a_tops / i8_peak, "traffic": ncu_traffic_ozaki(),
                "peak_source": i8_src, "int8_ops_per_rank_step": ops, "kernel_ms_per_step": oz_kernel["ms"],
                "kernel_share_of_step": oz_kernel["ms"] / (ev_ms / K),
                "fp64_equivalent_tflops_of_the_kernel": oz_kernel["tile_products"] * 2.0 * 128 ** 3 / (oz_kernel["ms"] * 1e-3) / 1e12,
                "fp64_equivalent_tflops_of_the_cholesky": achieved, "fp64_pipe_peak": pipe_peak,
                "cholesky_speedup_over_dmma": (dd / (chol_ms_max / K)) if dd else None,
                "note": "the kernel time is taken on one stream in an untimed pass right after the timed region (CUDA events around each launch); "
                        "FP64-equivalent = 2 * 128^3 flop per tile product, i.e. what the DMMA path would have executed"}
    else:
        roof = dmma_roofline
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "wall_ms_per_step": wall_ms / K, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": ("f64 (wide Cholesky updates: f64 split into int8 digit planes, exact int32 accumulation)" if args.ozaki else "f64"),
        "data": "synthetic", "config": cfg["config"],
        "e2e": {"value": 1e3 / (e2e_ms / K), "unit": UNIT, "h2d_bytes_per_step": int((hh1 - hh0) / K), "d2h_bytes_per_step": int((dh1 - dh0) / K)},
        "gpu_launches": int(launches.item()),
        "clocks": clocks,
        "roofline": roof,
        "stage_ms_per_step": {"stage_in+project": proj_ms / K, "kmat": kmat_ms / K, "cholesky": chol_ms / K, "solves": solve_ms / K},
        "hbm_stage_gbs": {"kmat_written": mloc * 8.0 * N * (N + 1) / 2 / (kmat_ms / K * 1e-3) / 1e9,
                          "solves_read": 2 * mloc * 8.0 * N * (N + 1) / 2 / (solve_ms / K * 1e-3) / 1e9,
                          "note": "rank 0's stages: algorithmic bytes (8 N(N+1)/2 per latent written by the kernel-matrix build, read once by "
                                  "each of the two triangular solves) / CUDA-event stage time"},
        "prediction_check_ms": pred_ms,
        "logpdf": lp,
    }
    if dmma:
        fl = mloc * (N ** 3) / 3.0
        dmma["value"] = 1e3 / dmma["ms_per_step"]
        dmma["cholesky_tflops"] = fl / (dmma["cholesky_ms"] * 1e-3) / 1e12
        dmma["frac_of_fp64_pipe_peak"] = dmma["cholesky_tflops"] / pipe_peak
        dmma["frac_of_measured_dgemm"] = dmma["cholesky_tflops"] / peak
        dmma["what"] = ("the same eval with the library's default FP64 DMMA trailing update (option ozaki = 0), measured untimed right after the timed region; "
                        "logpdf / posterior mean / variance differences are timed path vs this path at 256 test points")
        out["dmma_path"] = dmma
    if extras:
        out.update(extras)
    if world > 1:
        dist.destroy_process_group()
        # the same eval + prediction on ONE GPU (a second, communicator-less context on rank 0's device), untimed
        ctx1 = lmm.Context(local)
        lmm.set_default_context(ctx1)
        post_u, lp_u = lmm.posterior(fx_dev, yd, with_logpdf=True)
        M_u, V_u = lmm.mean_and_var(post_u(lmm.MOInputIsotopicByOutputs(xs_chk, p), s2))
        post_u.f.fs[0]._owner.free()
        lmm.set_default_context(ctx)
        out["sharded_vs_unsharded"] = {
            "what": f"{world}-rank sharded eval (NCCL all-reduce of lml terms; prediction at {Ns_chk} points with the NCCL all-reduce of the "
                    "partial back-projections; the timed path) vs the same calls on one GPU in a fresh context with the library's defaults (FP64 DMMA everywhere)",
            "logpdf_rel": abs(lp_s - lp_u) / abs(lp_u),
            "mean_relnorm": float(np.linalg.norm(M_s - M_u) / np.linalg.norm(M_u)),
            "var_max_rel": float(np.max(np.abs(V_s - V_u) / np.abs(V_u)))}
    if not args.no_cpu_baseline:
        cores = host_cores()
        T = U.T / np.sqrt(S)[:, None]
        Y = y.reshape(p, N)
        dt, lml0 = cpu_latent_eval(x, inv_ls[0], s2 / S[0], T[0] @ Y, cores)
        if world == 1:
            with blas_threads(cores):
                blas = blas_description()
            out["cpu_baseline"] = {"value": 1.0 / (dt * m), "unit": UNIT, "cores": cores, "kind": "port", "blas": blas,
                                   "sample": f"1 of {m} latents at full N={N} (2 kernel-matrix builds + 2 dpotrf + 3 triangular solves, reference "
                                             f"structure, every pass executed: {dt:.1f} s), x{m} extrapolated"}
        _, lml_last = cpu_latent_eval(x, inv_ls[m - 1], s2 / S[m - 1], T[m - 1] @ Y, cores, once=True)
        out["parity_check"] = {"what": "lml terms of latent 0 and of the last latent at full size, GPU (sharded over n_gpus ranks) vs CPU oracle",
                               "gpu": [float(terms[0]), float(terms[m - 1])], "oracle": [float(lml0), float(lml_last)],
                               "rel_err": max(abs(float(terms[0]) - lml0) / abs(lml0), abs(float(terms[m - 1]) - lml_last) / abs(lml_last))}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
