#!/usr/bin/env python
"""bench.py -- AdaPGM iterations/s on the dense fp64 lasso (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host cores

A step is ONE AdaPGM iteration (src/AdaProx.jl:334-362: value and gradient of
the least-squares term, the stepsize rule, the prox step) on the planted lasso
of lasso/runme.jl:40-77 generated on the device.  N = 1 runs configs[3] at its
full size, 65536 x 131072 fp64 (68.7 GB, far larger than the 126 MB L2, so no
L2 flush is needed between iterations).  N > 1 row-shards the same instance
(strong scaling): each rank keeps ONE persistent launch of the single-sweep
kernel for the whole solve and all-reduces the A'r partials (n + 2 doubles)
inside its iteration loop over NVLink peer memory (--nccl: split-phase launches
around ncclAllReduce for the A/B).

The default kernel is the single-sweep fused kernel (A is read ONCE per
iteration: g = A'(Ax - b) per row block while the rows are in shared memory);
--two-pass times the two-sweep persistent kernel (A*x, then A'r) for the A/B.
`roofline.achieved` counts the bytes the kernel that ran has to move.

`value` comes from CUDA events recorded by the library on the stream its kernels
run on, around a solve of exactly K iterations with everything resident in HBM
(the solve's prologue -- one more gradient evaluation -- is inside the timed
region, so the figure is slightly pessimistic); the solve is repeated --reps
times and the median repetition is reported, all samples under `repetitions`.
`e2e` is the same solve timed from the caller's side of the C ABI with host
buffers: x0 copied in from pinned host memory, x and the per-iteration records
copied back.

Also in the default line: `time_to_tol` (the BASELINE metric's time to 1e-6),
at N > 1 a `sharded_parity` block (configs[0] row-sharded over the N ranks
against the CPU oracle, before the timed region), at N = 1 a `configs` block
(configs[0], [1], [2], [4] with their rooflines and the oracle port timed beside
them) and `cpu_baseline` (the oracle port on a planted row slab of the same
width, every host thread; measured per-step time and scale factor are separate
keys, `extrapolated` says so).

--dump-outputs DIR writes what the last timed solve returned to its caller as
DIR/<name>.npy (float64): the iterate `x` after K steps and the per-iteration
records `gamma`, `norm_res`, `objective`.  The inputs are generated from a
fixed seed, so two builds run with the same arguments can be compared output
for output.  An array that would push the total past 64 MB is replaced by a
fixed, seeded sample of its entries.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

M_FULL, N_FULL = 65536, 131072
METRIC = "AdaPGM iters/sec on 65536x131072 fp64 lasso"


def b_iter_bytes(m_loc, n, passes=2):
    """Algorithmic bytes of one AdaPGM lasso iteration.  passes = 2 is SURVEY.md section 8d's figure (A read once
    for A*x and once for A'*r, the reference's two oracle calls) plus the vector traffic; passes = 1 is what the
    single-pass fused kernel (solver_fused.cuh) has to move: A once."""
    return passes * 8 * m_loc * n + 8 * (3 * m_loc + 8 * n)


NCU_SUMMARY = {1: "r01_ncu_k_adapgm_fused.json", 2: "r01_ncu_k_primal_dual_ring.json"}


def ncu_traffic_per_eval(m, n, passes):
    """DRAM bytes (read + write) per gradient evaluation from the committed `ncu --set full` capture of the
    persistent kernel that ran, at the full size; None for other sizes or when no capture is committed."""
    p = os.path.join(ROOT, "profiles", NCU_SUMMARY.get(passes, ""))
    if (m, n) != (M_FULL, N_FULL) or not os.path.isfile(p):
        return None, None
    with open(p) as f:
        return float(json.load(f)["_derived"]["dram_bytes_per_gradient_eval"]), os.path.relpath(p, ROOT)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region: NVML polled every 5 ms from a thread (the timed region
    of a multi-GPU run lasts only tens of milliseconds), nvidia-smi at 100 ms as the fallback."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None
        self.nv, self.samples, self.stop_flag, self.t = None, [], threading.Event(), None

    def _nvml_loop(self):
        nv, hd = self.nv, self.handle
        while not self.stop_flag.is_set():
            try:
                self.samples.append((nv.nvmlDeviceGetClockInfo(hd, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetCurrentClocksEventReasons(hd)))
            except Exception:
                break
            time.sleep(0.005)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.handle = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.handle, nv.NVML_CLOCK_SM)
            self.nv = nv
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def stop(self):
        if self.nv is not None:
            self.stop_flag.set()
            self.t.join(timeout=2)
            nv = self.nv
            names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
            sm = [s[0] for s in self.samples]
            reasons = sorted(k for k, bit in names.items() if any(s[1] & bit for s in self.samples))
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_mhz, "samples": len(sm),
                    "reasons": reasons, "source": "NVML, 5 ms period"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            parts = [s.strip() for s in l.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi, 100 ms period"}


# ----------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm (oracle port; Julia is not installed) on the host cores
# ----------------------------------------------------------------------------------------------
def blas_threads_all_cores():
    """torch.distributed.run exports OMP_NUM_THREADS=1 to its workers; the CPU arm must use the cores the box has.
    Returns (threads now in use, how it was set)."""
    want = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=want)                       # process-wide from here on (OpenBLAS / OpenMP pools)
        got = max([d.get("num_threads", 1) for d in threadpool_info()] or [1])
        return int(got), f"threadpoolctl.threadpool_limits({want}) (OMP_NUM_THREADS was {os.environ.get('OMP_NUM_THREADS', 'unset')})"
    except Exception as e:                                   # pragma: no cover
        return 1, f"threadpoolctl unavailable ({e}); BLAS default"


def planted_slab(rows, n, seed=0, lam=1.0, pfactor=5):
    """The planted lasso of lasso/runme.jl:40-77 on a rows x n matrix (Fortran order like a Julia Matrix), vectorised.
    numpy's own generator: this instance only feeds the CPU timing, nothing is compared against it."""
    rng = np.random.default_rng(seed)
    p = n / pfactor
    y_star = rng.random(rows); y_star /= np.linalg.norm(y_star)                   # :48-49
    A = np.empty((rows, n), order="F")
    step = max(1, int(2 ** 27 // rows))                                          # fill ~1 GB of columns at a time
    for j0 in range(0, n, step):
        j1 = min(n, j0 + step)
        A[:, j0:j1] = rng.random((j1 - j0, rows)).T * 2.0 - 1.0                    # :50
    cty = A.T @ y_star                                                            # :52
    sgn, cabs = np.sign(cty), np.abs(cty)
    perm = np.argsort(-cabs, kind="stable")                                       # :53
    rank = np.empty(n, dtype=np.int64); rank[perm] = np.arange(1, n + 1)
    top = rank <= p
    u = rng.random(n)
    alpha = np.where(top, lam / cabs, np.where(cabs < 0.1 * lam, lam, lam * u / cabs))   # :56-68
    A *= alpha[None, :]                                                           # :69
    x_star = np.where(top, rng.random(n) / np.sqrt(p) * sgn, 0.0)                 # :71-75
    b = A @ x_star + y_star                                                       # :76
    return A, b


def cpu_reference(m, n, steps, warmup, rows_sample=None, budget_gb=None, seed=0):
    """AdaPGM (OurRule) of src/AdaProx.jl:312-364 + lasso/runme.jl:16-27 through the oracle port (numpy -> OpenBLAS dgemv on
    every host thread) on the planted instance of a row slab of the same width n.  Everything in the returned dict was
    MEASURED on the slab; `value` is the slab time scaled by m / rows (dgemv cost is linear in the rows), flagged."""
    thr, how = blas_threads_all_cores()
    from oracle import adaprox_oracle as O
    if rows_sample is None:
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = 16e9
        gb = budget_gb if budget_gb else min(16.0, 0.25 * avail / 1e9)           # 16 GB: ~25 s to build, ~0.4 s per iteration
        rows_sample = int(max(64, min(m, gb * 1e9 // (8 * n))))
    t_gen = time.perf_counter()
    A, b = planted_slab(rows_sample, n, seed)
    t_gen = time.perf_counter() - t_gen
    f, g = O.LinearLeastSquares(A, b), O.NormL1(1.0)
    v = np.ones(n) / np.sqrt(n)
    for _ in range(3):
        w = A.T @ (A @ v); lf = float(np.linalg.norm(w)); v = w / lf
    rule = O.OurRule(gamma=1.0 / lf)
    if warmup > 0:
        O.adaptive_proxgrad(np.zeros(n), f=f, g=g, rule=rule, tol=0.0, maxit=warmup)
    t0 = time.perf_counter()
    O.adaptive_proxgrad(np.zeros(n), f=f, g=g, rule=rule, tol=0.0, maxit=steps)
    dt = time.perf_counter() - t0
    ms_sample = dt / steps * 1e3
    scale = m / rows_sample
    return {
        "value": 1e3 / (ms_sample * scale), "threads": thr, "threads_how": how, "rows_sample": rows_sample,
        "ms_per_step_sample": ms_sample, "scale": scale, "extrapolated": rows_sample != m, "timed_region_s": dt, "generation_s": t_gen,
        "host_gbs": 2 * 8 * rows_sample * n / (ms_sample * 1e-3) / 1e9,
        "sample": (f"oracle port of src/AdaProx.jl:312-364 + lasso/runme.jl:16-27 (numpy -> OpenBLAS dgemv, {thr} threads): {steps} AdaPGM "
                   f"iterations MEASURED on the planted lasso of a {rows_sample} x {n} row slab ({rows_sample * n * 8 / 1e9:.2f} GB, Fortran "
                   f"order), {ms_sample:.1f} ms per iteration" + ("" if rows_sample == m else
                   f"; value = that time x m/rows = {scale:.2f} (EXTRAPOLATED to the full {m} x {n}; dgemv cost is linear in the rows)")),
    }


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    m, n = args.m, args.n
    c = cpu_reference(m, n, args.steps, args.warmup, args.cpu_rows, args.cpu_gb)
    out = {
        "impl": "reference", "metric": METRIC if (m, n) == (M_FULL, N_FULL) else f"AdaPGM iters/sec on {m}x{n} fp64 lasso",
        "value": c["value"], "unit": "it/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        # ms_per_step is what one timed step of THIS run took (the slab); steps x ms_per_step is the timed region
        "ms_per_step": c["ms_per_step_sample"], "ms_per_step_sample": c["ms_per_step_sample"], "extrapolated": c["extrapolated"],
        "ms_per_step_full_size_equivalent": c["ms_per_step_sample"] * c["scale"], "sample_rows": c["rows_sample"], "sample_scale": c["scale"],
        "timed_region_s": c["timed_region_s"], "host_gbs": c["host_gbs"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"configs[3]: dense lasso AdaPGM {m}x{n} fp64, OurRule, CPU", "m": m, "n": n},
        "cpu_baseline": {"value": c["value"], "unit": "it/s", "cores": c["threads"], "kind": "port", "sample": c["sample"],
                         "extrapolated": c["extrapolated"], "threads_how": c["threads_how"]},
        "e2e": {"value": c["value"], "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
DUMP_BUDGET_BYTES = 64_000_000


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy in float64; an array over its share of DUMP_BUDGET_BYTES is replaced by the
    entries at a fixed, seeded, sorted sample of its indices (the same sample in every run with the same sizes)."""
    os.makedirs(out_dir, exist_ok=True)
    cap = (DUMP_BUDGET_BYTES // len(arrays) - 128) // 8          # 128: the .npy header
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def dmma_peak():
    """fp64 tensor-pipe peak measured by tools/probes/fp64_peak_probe.cu on this pool's B200 (profiles/r02_fp64_peaks.jsonl)."""
    p = os.path.join(ROOT, "profiles", "r02_fp64_peaks.jsonl")
    best = None
    if os.path.isfile(p):
        for line in open(p):
            d = json.loads(line)
            if d.get("probe", "").startswith("DMMA.8x8x4"):
                best = max(best or 0.0, d["tflops"])
    return (best, "measured: profiles/r02_fp64_peaks.jsonl (DMMA.8x8x4 issue-bound probe)") if best else (40.0, "fallback: B200 datasheet fp64 40 TFLOP/s")


def sharded_parity(AdaProx, dev, dist, world, rank):
    """N > 1, before the timed region: the 400 x 1000 planted lasso of configs[0] row-sharded over the N ranks, against the CPU
    oracle on the whole problem -- through the path the timed region uses (single-sweep kernel + in-kernel all-reduce, forced on
    for this small matrix) and through the split-phase two-pass path.  Every rank solves; rank 0 reports."""
    import torch
    from oracle import adaprox_oracle as O
    m, n = 400, 1000
    P = AdaProx.synth.planted_lasso(m, n, 5, 0)
    Lf = AdaProx.synth.spectral_norm_sq(P["A"], iters=1000, tol=1e-15)
    row0, rows = AdaProx.sharding.shard_rows(m, world, rank)
    A = AdaProx.DeviceMatrix(P["A"][row0:row0 + rows], dev=dev)
    A.set_shard(m, row0)
    f = AdaProx.LinearLeastSquares(A, P["b"][row0:row0 + rows])
    out = {"instance": f"planted lasso {m}x{n} (configs[0]), rows split over {world} ranks, AdaPGM OurRule tol 1e-6"}
    logo = []
    xo, ito = O.adaptive_proxgrad(np.zeros(n), f=O.LinearLeastSquares(P["A"], P["b"]), g=O.NormL1(1.0), rule=O.OurRule(gamma=1 / Lf),
                                  tol=1e-6, maxit=10000, log=logo)
    go = np.array([r["gamma"] for r in logo[:40]])
    for tag, env in (("fused_sweep_in_kernel_allreduce", "1"), ("two_pass_split_phase_nccl", "0")):
        os.environ["ADAPROX_FUSED"] = env
        try:
            log = []
            x, it = AdaProx.adaptive_proxgrad(np.zeros(n), f=f, g=AdaProx.NormL1(1.0), rule=AdaProx.OurRule(gamma=1 / Lf), tol=1e-6, maxit=10000, log=log)
            info = AdaProx.last_solve_info()
        finally:
            os.environ.pop("ADAPROX_FUSED", None)
        xs = [torch.empty(n, dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(xs, torch.from_numpy(x).cuda())
        same = all(bool(torch.equal(xs[0], t)) for t in xs[1:])
        gd = np.array([r["gamma"] for r in log[:40]])
        k = min(len(gd), len(go))
        out[tag] = {"iterations": int(it), "oracle_iterations": int(ito), "gamma_prefix15_max_rel_diff": float(np.max(np.abs(gd[:15] / go[:15] - 1))),
                    "gamma_prefix40_max_rel_diff": float(np.max(np.abs(gd[:k] / go[:k] - 1))),
                    "final_objective_rel_diff": float(abs(log[-1]["objective"] - logo[-1]["objective"]) / abs(logo[-1]["objective"])),
                    "x_rel_diff": float(np.linalg.norm(x - xo) / np.linalg.norm(xo)), "iterates_bit_identical_across_ranks": bool(same),
                    "matrix_passes": info["matrix_passes"], "collective": info["collective"]}
    ok = all(v["gamma_prefix15_max_rel_diff"] < 1e-12 and v["final_objective_rel_diff"] < 1e-10 and v["iterates_bit_identical_across_ranks"]
             and abs(v["iterations"] - v["oracle_iterations"]) <= max(2, 0.05 * v["oracle_iterations"]) for k_, v in out.items() if isinstance(v, dict))
    out["pass"] = bool(ok)
    A.free()
    return out


def configs_block(AdaProx, peak_hbm):
    """Short device-timed runs of the other BASELINE configs on this GPU (N = 1), each with the roofline that bounds it and the
    oracle port timed on the host beside it.  Parity for these shapes lives in tests/test_gpu_full_shapes.py."""
    import scipy.sparse as sp
    from oracle import adaprox_oracle as O
    out = {}

    def cpu_time(fn, reps=1):
        t0 = time.perf_counter()
        for _ in range(reps):
            r = fn()
        return (time.perf_counter() - t0) / reps, r

    # C1 -------------------------------------------------------------------------------------------------------
    P = AdaProx.synth.planted_lasso(400, 1000, 5, 0)
    Lf = AdaProx.synth.spectral_norm_sq(P["A"], iters=1000, tol=1e-15)
    f, g = AdaProx.LinearLeastSquares(P["A"], P["b"]), AdaProx.NormL1(1.0)
    AdaProx.adaptive_proxgrad(np.zeros(1000), f=f, g=g, rule=AdaProx.OurRule(gamma=1 / Lf), tol=1e-6, maxit=200)
    x, it = AdaProx.adaptive_proxgrad(np.zeros(1000), f=f, g=g, rule=AdaProx.OurRule(gamma=1 / Lf), tol=1e-6, maxit=10000)
    info = AdaProx.last_solve_info()
    dt, (xo, ito) = cpu_time(lambda: O.adaptive_proxgrad(np.zeros(1000), f=O.LinearLeastSquares(P["A"], P["b"]), g=O.NormL1(1.0),
                                                         rule=O.OurRule(gamma=1 / Lf), tol=1e-6, maxit=10000))
    us = 1e3 * info["solve_ms"] / it
    out["c1_lasso_400x1000_adapgm"] = {
        "iterations_to_1e-6": int(it), "oracle_iterations": int(ito), "us_per_iteration": us, "iters_per_s": 1e6 / us, "time_to_tol_ms": info["solve_ms"],
        "kernel": info.get("kernel", "persistent"), "launches": info["kernel_launches"],
        "roofline": {"bound": "latency (3.2 MB matrix, L2/SMEM resident)", "achieved_l2_gbs": 2 * 8 * 400 * 1000 / (us * 1e-6) / 1e9, "frac": None},
        "cpu_port": {"us_per_iteration": 1e6 * dt / ito, "time_to_tol_ms": 1e3 * dt}}
    # the other two sizes of the reference's lasso experiment (lasso/runme.jl:191-195, pfactor 10): grid-resident kernel
    for (mm, nn) in ((500, 1000), (4000, 1000)):
        P = AdaProx.synth.planted_lasso(mm, nn, 10, 0)
        Lf = AdaProx.synth.spectral_norm_sq(P["A"], iters=300, tol=1e-13)
        f, g = AdaProx.LinearLeastSquares(P["A"], P["b"]), AdaProx.NormL1(1.0)
        AdaProx.adaptive_proxgrad(np.zeros(nn), f=f, g=g, rule=AdaProx.OurRule(gamma=1 / Lf), tol=1e-7, maxit=200)
        x, it = AdaProx.adaptive_proxgrad(np.zeros(nn), f=f, g=g, rule=AdaProx.OurRule(gamma=1 / Lf), tol=1e-7, maxit=2000)
        info = AdaProx.last_solve_info()
        Kc = 300
        dt, _ = cpu_time(lambda: O.adaptive_proxgrad(np.zeros(nn), f=O.LinearLeastSquares(P["A"], P["b"]), g=O.NormL1(1.0),
                                                     rule=O.OurRule(gamma=1 / Lf), tol=0.0, maxit=Kc))
        us = 1e3 * info["solve_ms"] / it
        out[f"lasso_{mm}x{nn}_adapgm"] = {
            "iterations": int(it), "tol": 1e-7, "maxit": 2000, "us_per_iteration": us, "iters_per_s": 1e6 / us, "time_ms": info["solve_ms"],
            "matrix_passes_code": int(info["matrix_passes"]), "launches": info["kernel_launches"], "final_norm_res": info["final_norm_res"],
            "roofline": {"bound": "latency (matrix resident in the shared memory of all SMs; two grid barriers per iteration)", "frac": None},
            "cpu_port": {"us_per_iteration": 1e6 * dt / Kc, "sample": f"{Kc} iterations, numpy/OpenBLAS dgemv"}}
        f.mat.free()
    # C2 -------------------------------------------------------------------------------------------------------
    m, n = 20242, 47236
    rp, ci, va, y = AdaProx.synth.sparse_logreg(m, n, 0)
    X = sp.csr_matrix((va, ci, rp), shape=(m, n))
    lam = 0.03 * AdaProx.synth.logreg_lambda_max(X, y)
    gam = 4 * m / (va @ va + m)
    f = AdaProx.LogisticLoss(X, y)
    K = 300
    AdaProx.adaptive_proxgrad(np.zeros(n + 1), f=f, g=AdaProx.NormL1(lam), rule=AdaProx.OurRule(gamma=gam), tol=0.0, maxit=20)
    x, it = AdaProx.adaptive_proxgrad(np.zeros(n + 1), f=f, g=AdaProx.NormL1(lam), rule=AdaProx.OurRule(gamma=gam), tol=0.0, maxit=K)
    info = AdaProx.last_solve_info()
    dt, _ = cpu_time(lambda: O.adaptive_proxgrad(np.zeros(n + 1), f=O.LogisticLoss(X, y), g=O.NormL1(lam), rule=O.OurRule(gamma=gam), tol=0.0, maxit=20))
    us = 1e3 * info["solve_ms"] / K
    nnz = len(va)
    bytes_iter = 2 * 12 * nnz + 4 * (m + 1) + 4 * (n + 1) + 8 * (4 * m + 8 * n)
    out["c2_sparse_logreg_20242x47236_adapgm"] = {
        "iterations": K, "lambda": lam, "lambda_over_lambda_max": 0.03, "nnz": nnz, "nnz_w_after_K": int(np.count_nonzero(x[:-1])),
        "us_per_iteration": us, "iters_per_s": 1e6 / us, "final_norm_res": info["final_norm_res"],
        "roofline": {"bound": "L2 sector rate of the CSR gathers (36 MB, L2-resident)", "achieved_l2_gbs": bytes_iter / (us * 1e-6) / 1e9,
                     "algorithmic_bytes_per_iteration": bytes_iter, "frac": None},
        "cpu_port": {"us_per_iteration": 1e6 * dt / 20, "sample": "20 iterations, scipy.sparse CSR"}}
    f.mat.free()
    # C3 -------------------------------------------------------------------------------------------------------
    m, d = 50000, 2000
    rng = np.random.default_rng(0)
    Xd = rng.standard_normal((m, d)) / np.sqrt(d)
    w = np.where(rng.random(d) < 0.05, 3.0 * rng.standard_normal(d), 0.0)
    yv = Xd @ w + rng.laplace(scale=0.1, size=m)
    A = np.hstack([Xd, np.ones((m, 1))])
    nA = float(np.linalg.norm(A))
    Ad = AdaProx.Counting(AdaProx.DeviceMatrix(A))
    kw = dict(f=AdaProx.Zero(), g=AdaProx.NormL1(10.0), h=AdaProx.Translate(AdaProx.NormL1(), -yv), A=Ad, eta=nA, t=1.0, tol=0.0)
    AdaProx.adaptive_linesearch_primal_dual(np.zeros(d + 1), np.zeros(m), maxit=20, **kw)
    Ad.mul_count = Ad.amul_count = 0
    K = 500
    AdaProx.adaptive_linesearch_primal_dual(np.zeros(d + 1), np.zeros(m), maxit=K, **kw)
    info = AdaProx.last_solve_info()
    passes = Ad.mul_count + Ad.amul_count
    Ao = O.Counting(A)
    dt, _ = cpu_time(lambda: O.adaptive_linesearch_primal_dual(np.zeros(d + 1), np.zeros(m), f=O.Zero(), g=O.NormL1(10.0), h=O.Translate(O.NormL1(), -yv),
                                                               A=Ao, eta=nA, t=1.0, tol=0.0, maxit=10))
    gbs = passes * 8 * m * (d + 1) / (info["solve_ms"] * 1e-3) / 1e9
    out["c3_lad_50000x2001_adapdm_plus"] = {
        "iterations": K, "us_per_iteration": 1e3 * info["solve_ms"] / K, "matrix_passes": int(passes),
        "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak_hbm, "unit": "GB/s", "frac": gbs / peak_hbm,
                     "algorithmic_bytes": "8 m (n+1) per application of A or A' (counted: mul_count + amul_count)"},
        "cpu_port": {"us_per_iteration": 1e6 * dt / 10, "sample": "10 iterations, numpy/OpenBLAS dgemv"}}
    Ad.f.free()
    # dual SVM, Gram form (dual_svm/runme.jl:47-59 with Q = Z Z' by its factor)
    s_ = np.sign(Xd @ rng.standard_normal(d)); s_[s_ == 0] = 1.0
    ysvm = np.where(rng.random(m) < 0.1, -s_, s_)
    Zm = AdaProx.DeviceMatrix(ysvm[:, None] * Xd)
    fq = AdaProx.QuadraticGram(Zm, -np.ones(m))
    Amat = AdaProx.DeviceMatrix(ysvm[None, :].copy())
    kw = dict(f=fq, g=AdaProx.IndBox(0.0, 0.1), h=AdaProx.IndZero(), A=Amat, rule=AdaProx.OurRule(t=0.1, norm_A=float(np.sqrt(m))), tol=0.0)
    AdaProx.adaptive_primal_dual(np.zeros(m), np.zeros(1), maxit=20, **kw)
    K = 500
    AdaProx.adaptive_primal_dual(np.zeros(m), np.zeros(1), maxit=K, **kw)
    info = AdaProx.last_solve_info()
    gbs = K * 2 * 8 * m * d / (info["solve_ms"] * 1e-3) / 1e9
    Zh = ysvm[:, None] * Xd

    class _GramOracle:                                   # the reference's Quadratic (dual_svm/runme.jl:19-28) with Q x = Z (Z' x)
        def eval_with_pullback(self, x):
            temp = Zh @ (Zh.T @ x)
            return 0.5 * np.dot(x, temp) - np.sum(x), (lambda: temp - 1.0)

        def __call__(self, x):
            return self.eval_with_pullback(x)[0]

    dt, _ = cpu_time(lambda: O.adaptive_primal_dual(np.zeros(m), np.zeros(1), f=_GramOracle(), g=O.IndBox(0.0, 0.1), h=O.IndZero(), A=ysvm[None, :].copy(),
                                                    rule=O.OurRule(t=0.1, norm_A=float(np.sqrt(m))), tol=0.0, maxit=10))
    out["c3_dual_svm_N50000_d2000_gram_adapdm"] = {
        "iterations": K, "us_per_iteration": 1e3 * info["solve_ms"] / K,
        "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak_hbm, "unit": "GB/s", "frac": gbs / peak_hbm,
                     "algorithmic_bytes": "2 * 8 N d per iteration (Z'x then Z u); the dense Q of the reference would be 8 N^2 = 20 GB"},
        "cpu_port": {"us_per_iteration": 1e6 * dt / 10, "sample": "10 iterations, Q x evaluated as Z (Z'x) with numpy/OpenBLAS"}}
    Zm.free(); Amat.free()
    del Xd, A, Zh
    # C5 -------------------------------------------------------------------------------------------------------
    m, n, Lc = 16384, 8192, 256
    P = AdaProx.generate_planted_lasso(m, n, pfactor=5, seed=0, power_iters=30)
    f = AdaProx.LinearLeastSquares(P["A"], P["b"])
    lam_max = float(np.max(np.abs(P["A"].T @ P["b"].download())))
    lambdas = lam_max * (1e-3) ** (np.arange(Lc) / (Lc - 1))
    ms_r = P["A"].time_path_gemm(Lc, 0, reps=5)
    ms_g = P["A"].time_path_gemm(Lc, 1, reps=5)
    K = 30
    AdaProx.adaptive_proxgrad_path(None, f=f, lambdas=lambdas, rule=AdaProx.OurRule(gamma=1 / P["Lf"]), tol=0.0, maxit=3)
    X, its, info = AdaProx.adaptive_proxgrad_path(None, f=f, lambdas=lambdas, rule=AdaProx.OurRule(gamma=1 / P["Lf"]), tol=0.0, maxit=K)
    evals = info["batched_evals"]
    flop = 4.0 * m * n * Lc
    tf = flop * evals / (info["solve_ms"] * 1e-3) / 1e12
    pk, pk_src = dmma_peak()
    out["c5_lambda_path_256x16384x8192"] = {
        "batched_iterations": K, "ms_per_batched_iteration": info["solve_ms"] / evals,
        "gemm_AX_ms": ms_r, "gemm_AtR_ms": ms_g, "gemm_AX_tflops": 2.0 * m * n * Lc / (ms_r * 1e-3) / 1e12, "gemm_AtR_tflops": 2.0 * m * n * Lc / (ms_g * 1e-3) / 1e12,
        "roofline": {"bound": "tensor (fp64 DMMA)", "achieved": tf, "peak": pk, "unit": "TFLOP/s", "frac": tf / pk, "peak_source": pk_src,
                     "algorithmic_flop_per_iteration": flop}}
    P["A"].free()
    return out


def run_b200(args):
    import torch
    import adaprox_b200 as AdaProx
    import ctypes as C
    from adaprox_b200 import _lib as L

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N > 1 with torch.distributed.run (one process per GPU)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    dev = AdaProx.Device(local)
    AdaProx.set_default_device(dev)
    if world > 1:
        AdaProx.sharding.attach_communicator(dev, dist)
        if not args.nccl:
            AdaProx.sharding.attach_p2p(dev, args.n, dist)       # all-reduce inside the sweep kernel over NVLink peer memory

    def stage(msg):
        if args.verbose:
            print(f"[bench rank {rank}] {msg}", file=sys.stderr, flush=True)

    parity = None
    if world > 1 and not args.no_parity:
        stage("sharded_parity ...")
        parity = sharded_parity(AdaProx, dev, dist, world, rank)
        stage(f"sharded_parity done: {parity.get('pass')}")

    m, n = args.m, args.n
    row0, rows = AdaProx.sharding.shard_rows(m, world, rank)
    t_gen = time.perf_counter()
    P = AdaProx.generate_planted_lasso(m, n, pfactor=5, seed=0, lam=1.0, power_iters=args.power_iters, row0=row0, rows=rows, dev=dev)
    t_gen = time.perf_counter() - t_gen
    f = AdaProx.LinearLeastSquares(P["A"], P["b"])
    g = AdaProx.NormL1(1.0)
    gamma0 = 1.0 / P["Lf"]

    # pinned host buffers for the C-ABI call
    x0_t = torch.zeros(n, dtype=torch.float64).pin_memory()
    xo_t = torch.zeros(n, dtype=torch.float64).pin_memory()
    x0 = x0_t.numpy(); xo = xo_t.numpy()

    def solve(maxit, tol, records):
        p = f._problem(n)
        p.g = g._desc()
        o = AdaProx.core._opts(tol, maxit)
        AdaProx.OurRule(gamma=gamma0)._fill(o)
        o.solver = L.S_ADAPTIVE_PROXGRAD
        o.want_objective = 1 if records else 0
        o.max_records = maxit if records else 0
        recs = (L.Record * max(maxit, 1))() if records else None
        res = L.Result()
        dev.check(dev.lib.adaprox_solve(dev.h, C.byref(p), C.byref(o), x0.ctypes.data_as(L.c_dp), None,
                                        xo.ctypes.data_as(L.c_dp), None, recs, C.byref(res)))
        return res, recs

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(v):
        if dist is None:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    W, K = max(args.warmup, 3), args.steps
    stage(f"generated in {t_gen:.1f} s; warm-up ...")
    solve(W, 0.0, False)                                       # warm-up iterations (untimed)
    stage("timed region ...")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # The timed region is one blocking solve of exactly K iterations; it is repeated `reps` times (each bracketed by a
    # barrier + synchronize on both sides, device time = max over ranks) and the MEDIAN repetition is the reported value:
    # at N = 8 one solve lasts ~50 ms, a single sample says little.
    reps = max(1, args.reps)
    samples = []
    for _ in range(reps):
        sync_all()
        t0 = time.perf_counter()
        res, recs = solve(K, 0.0, True)                        # exactly K iterations, blocking C-ABI call
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        sync_all()
        assert res.iters == K, (res.iters, K)
        samples.append((max_over_ranks(res.solve_ms), max_over_ranks(t1 - t0), int(res.kernel_launches)))
    clocks = sampler.stop() if rank == 0 else None
    order = sorted(range(reps), key=lambda i: samples[i][0])
    med = order[len(order) // 2]
    dev_ms, e2e_s, launches = samples[med]
    last = recs[K - 1]
    if args.dump_outputs and rank == 0:                        # x is replicated on every rank; xo is reused by later solves
        dump_outputs(args.dump_outputs, {"x": xo, "gamma": [r.gamma for r in recs], "norm_res": [r.norm_res for r in recs],
                                         "objective": [r.f_x + r.g_x for r in recs]})

    # per-kernel-family timing (profile breakdown; the shares the ncu launch list must agree with)
    ms_n = max_over_ranks(P["A"].time_kernel(0, reps=3))
    ms_t = max_over_ranks(P["A"].time_kernel(1, reps=3))

    extra = {}
    if args.to_tol > 0:
        sync_all()
        t0 = time.perf_counter()
        r2, _ = solve(args.tol_maxit, args.to_tol, False)
        torch.cuda.synchronize()
        tt = max_over_ranks(time.perf_counter() - t0)
        extra = {"time_to_tol": {"tol": args.to_tol, "seconds": tt, "device_seconds": max_over_ranks(r2.solve_ms) / 1e3,
                                 "iterations": int(r2.iters), "converged": bool(r2.flags & 1),
                                 "final_norm_res": r2.final_norm_res,
                                 "what": "one blocking adaprox_solve from x0 = 0 until norm_res <= tol (BASELINE.json metric: time-to-1e-6), wall clock incl. copies"}}

    if rank == 0:
        peak, peak_src = peaks()
        passes = int(res.matrix_passes)                            # 1: single-pass fused kernel, 2: A*x then A'r
        bytes_iter_rank = b_iter_bytes(rows, n, passes)
        # the timed launch(es) perform K iterations plus the solver's prologue (one more gradient evaluation, :327-332)
        bytes_launch = bytes_iter_rank * K + passes * 8 * rows * n
        achieved = bytes_launch / (dev_ms * 1e-3) / 1e9            # per-GPU GB/s actually required of HBM
        per_eval, per_eval_src = ncu_traffic_per_eval(m, n, passes) if world == 1 else (None, None)
        if world > 1 and passes == 1:
            kernel = "k_adapgm_fused in sweep-only mode (one sweep of the row shard per iteration)"
        elif world > 1:
            kernel = "k_sh_A + k_sh_C (split-phase GEMV kernels)"
        elif passes == 1:
            kernel = ("k_adapgm_fused (persistent cooperative cluster kernel: the whole solve is one launch; "
                      "A'(Ax-b) in ONE sweep over A per iteration)")
        else:
            kernel = "k_primal_dual<false> (persistent cooperative kernel: the whole solve is one launch)"
        out = {
            "metric": METRIC if (m, n) == (M_FULL, N_FULL) else f"AdaPGM iters/sec on {m}x{n} fp64 lasso",
            "value": K / (dev_ms * 1e-3), "unit": "it/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"configs[3]: dense lasso AdaPGM {m}x{n} fp64 (planted instance of lasso/runme.jl:40-77), "
                                   f"OurRule gamma0=1/Lf, row-sharded over {world} GPU(s)",
                       "m": m, "n": n, "rows_per_gpu": rows, "rule": "OurRule", "lambda": 1.0,
                       "l2": "inputs larger than L2 (matrix shard %.1f GB vs 126 MB), no flush needed" % (rows * n * 8 / 1e9),
                       "timing": f"library CUDA events on the kernels' stream around one solve of K iterations; max over ranks; median of {reps} repetitions",
                       "generation_s": round(t_gen, 2), "gamma0": gamma0},
            "repetitions": {"n": reps, "ms_per_step": [s_[0] / K for s_ in samples], "median_ms_per_step": dev_ms / K,
                            "min_ms_per_step": samples[order[0]][0] / K, "max_ms_per_step": samples[order[-1]][0] / K,
                            "spread_rel": (samples[order[-1]][0] - samples[order[0]][0]) / dev_ms},
            "achieved_hbm_gbs_per_gpu": bytes_iter_rank * K / (dev_ms * 1e-3) / 1e9,
            "matrix_passes_per_iteration": passes,
            "two_pass_equivalent_gbs_per_gpu": b_iter_bytes(rows, n, 2) * K / (dev_ms * 1e-3) / 1e9,
            "two_pass_equivalent_note": "SURVEY 8d's B_iter (A counted twice, as the reference's two oracle calls read it) x it/s; "
                                        "equals achieved_hbm_gbs_per_gpu when matrix_passes_per_iteration = 2; with the single-pass "
                                        "kernel it is a throughput equivalent, NOT a bandwidth (roofline.achieved counts A once)",
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (per_eval * (K + 1)) if per_eval else None, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": bytes_launch,
                         "launch": "one persistent launch = K iterations + prologue = K+1 gradient evaluations" if world == 1
                                   else ("K+1 gradient evaluations as 3 launches each (fused sweep + all-reduce, 2 small kernels)" if passes == 1
                                         else "K+1 gradient evaluations as 6 launches + 1 all-reduce each"),
                         "traffic_source": ("STATIC, not measured in this run: dram__bytes_read.sum + dram__bytes_write.sum per gradient evaluation "
                                            "from the committed ncu --set full capture x (K+1), " + per_eval_src) if per_eval else None,
                         "kernel": kernel, "matrix_passes": passes,
                         "algorithmic_bytes_per_iteration_per_gpu": bytes_iter_rank,
                         "gemv_n_ms": ms_n, "gemv_t_ms": ms_t,
                         "gemv_n_gbs": rows * n * 8 / (ms_n * 1e-3) / 1e9, "gemv_t_gbs": rows * n * 8 / (ms_t * 1e-3) / 1e9},
            "e2e": {"value": K / e2e_s, "unit": "it/s", "h2d_bytes_per_step": n * 8 / K,
                    "d2h_bytes_per_step": (n * 8 + K * C.sizeof(L.Record) + C.sizeof(L.Result)) / K,
                    "call": "one blocking adaprox_solve (C ABI) of K iterations: x0 from pinned host memory, x and K records copied back"},
            "gpu_launches": launches,
            "collective": {0: "none", 1: "ncclAllReduce of n+2 doubles per iteration",
                           2: "all-reduce inside the sweep kernel over NVLink peer memory (no NCCL on the data path)"}[int(res.collective)],
            "clocks": clocks,
            "final_record": {"it": int(last.it), "gamma": last.gamma, "norm_res": last.norm_res,
                             "objective": last.f_x + last.g_x, "optimum": P["optimum"]},
        }
        out.update(extra)
        if parity is not None:
            out["sharded_parity"] = parity
    P["A"].free()                                              # 68.7 GB back before the other configs allocate
    if rank == 0:
        if world == 1 and not args.no_configs:
            try:
                out["configs"] = configs_block(AdaProx, peaks()[0])
            except Exception as e:                                 # the headline line must survive a failure of the side block
                out["configs"] = {"error": repr(e)}
        if world == 1 and not args.no_cpu:
            c = cpu_reference(m, n, args.cpu_steps, 1, args.cpu_rows, args.cpu_gb)
            out["cpu_baseline"] = {"value": c["value"], "unit": "it/s", "cores": c["threads"], "kind": "port", "sample": c["sample"],
                                   "extrapolated": c["extrapolated"], "ms_per_step_sample": c["ms_per_step_sample"], "sample_rows": c["rows_sample"],
                                   "threads_how": c["threads_how"]}
        print(json.dumps(out), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--m", type=int, default=M_FULL)
    ap.add_argument("--n", type=int, default=N_FULL)
    ap.add_argument("--power-iters", type=int, default=30)
    ap.add_argument("--to-tol", type=float, default=1e-6, help="also report the time to reach norm_res <= tol (BASELINE metric; 0 = skip)")
    ap.add_argument("--tol-maxit", type=int, default=20000)
    ap.add_argument("--reps", type=int, default=5, help="repetitions of the timed K-step solve (the median is reported)")
    ap.add_argument("--verbose", action="store_true", help="progress markers on stderr")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs block (C1, C2, C3, C5 side measurements, N = 1 only)")
    ap.add_argument("--no-parity", action="store_true", help="skip the sharded_parity block (N > 1)")
    ap.add_argument("--cpu-gb", type=float, default=None, help="size of the CPU arm's row slab in GB (default: min(16, RAM/4))")
    ap.add_argument("--two-pass", action="store_true", help="A/B: force the two-pass kernel (ADAPROX_FUSED=0)")
    ap.add_argument("--nccl", action="store_true", help="A/B (N > 1): ncclAllReduce per iteration instead of the in-kernel all-reduce")
    ap.add_argument("--cpu-steps", type=int, default=20)
    ap.add_argument("--cpu-rows", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write x and the per-iteration records of the last timed solve to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the CUDA path (--impl b200)")
    if args.two_pass:
        os.environ["ADAPROX_FUSED"] = "0"
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
