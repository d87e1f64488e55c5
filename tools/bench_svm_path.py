"""Batched C path of the dual SVM (adaptive_primal_dual_path) on the dense-classification instances of config C3: dense Q at
N = 20000 and the Gram form at N = 20000 and N = 50000 (d = 2000), A = y', OurRule(t = 1, norm_A = sqrt(N)).

For L = 32, 64, 128, 256 C values: ms per batched iteration, us per C-iteration, the speed-up over the single-C
adaptive_primal_dual iteration timed in the same run, and the TFLOP/s of every contraction of the iteration (timed alone
with adaprox_time_path_gemm) against the DMMA probe peak of profiles/r02_fp64_peaks.jsonl.  Then the time to tol = 1e-5 of
a 64-value C grid against single solves of a sample of the grid, extrapolated to the whole grid.

    python tools/bench_svm_path.py [--out FILE] [--reps 3] [--iters 20]

Prints one JSON line (and writes it to FILE).  Times are device-event times of the solve loop (adaprox_result.solve_ms)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import adaprox_b200 as AdaProx  # noqa: E402

DMMA_PEAK_TFLOPS = 37.1            # mma.sync f64 m8n8k4 probe, NVIDIA B200 (profiles/r02_fp64_peaks.jsonl)


def gpu_facts():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi query failed: " + r.stderr)
    name, plim, clk = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=plim, max_sm_clock=clk)


def spread(v):
    v = np.asarray(v, dtype=float)
    return dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()))


def c_grid(L):
    return np.geomspace(1e-2, 1e1, L)


def bench_instance(form, N, d, a):
    X, y = AdaProx.synth.dense_classification(N, d, 0)
    Z = np.ascontiguousarray(y[:, None] * X)
    q = -np.ones(N)
    Zm = AdaProx.DeviceMatrix(Z)
    if form == "quadratic":
        Zt = torch.from_numpy(Z).cuda()
        Q = (Zt @ Zt.T).cpu().numpy()                              # Q = D_y X X' D_y (dual_svm/runme.jl:47-49)
        del Zt
        torch.cuda.empty_cache()
        Qm = AdaProx.DeviceMatrix(Q)
        del Q
        f = AdaProx.Quadratic(Qm, q)
    else:
        f = AdaProx.QuadraticGram(Zm, q)
    A = y[None, :]
    rule = AdaProx.OurRule(t=1, norm_A=np.sqrt(N))
    K = a.iters
    out = dict(form=form, N=N, d=d)

    # single-C baseline, tol = 0: exactly K iterations
    g = AdaProx.IndBox(0.0, 1.0)
    AdaProx.adaptive_primal_dual(np.zeros(N), np.zeros(1), f=f, g=g, h=AdaProx.IndZero(), A=A, rule=rule, tol=0.0, maxit=3)
    single = []
    for _ in range(a.reps):
        AdaProx.adaptive_primal_dual(np.zeros(N), np.zeros(1), f=f, g=g, h=AdaProx.IndZero(), A=A, rule=rule, tol=0.0, maxit=K)
        single.append(1e3 * AdaProx.last_solve_info()["solve_ms"] / K)
    out["single_us_per_iter"] = spread(single)
    s_us = out["single_us_per_iter"]["median"]

    rows = []
    for Lc in (32, 64, 128, 256):
        C_ = c_grid(Lc)
        AdaProx.adaptive_primal_dual_path(f=f, A=A, upper=C_, rule=rule, tol=0.0, maxit=3)     # warm-up at this shape
        t = []
        for _ in range(a.reps):
            _, _, its, info = AdaProx.adaptive_primal_dual_path(f=f, A=A, upper=C_, rule=rule, tol=0.0, maxit=K)
            assert np.all(its == K)
            t.append(info["solve_ms"] / info["batched_evals"])
        it_ms = float(np.median(t))
        # the contractions of one iteration, each timed alone on an Lc-column batch
        if form == "quadratic":
            con = dict(QX=(Qm.time_path_gemm(Lc, 0, reps=10), 2.0 * N * N * Lc))
        else:
            con = dict(ZtX=(Zm.time_path_gemm(Lc, 1, reps=10), 2.0 * N * d * Lc), ZU=(Zm.time_path_gemm(Lc, 0, reps=10), 2.0 * N * d * Lc))
        flops = sum(fl for _, fl in con.values())
        rows.append(dict(L=Lc, ms_per_iter=spread(t), us_per_C_iter=1e3 * it_ms / Lc, speedup_vs_single=s_us / (1e3 * it_ms / Lc),
                         path_TFLOPs=flops / (it_ms * 1e-3) / 1e12,
                         contractions={k: dict(ms=ms, TFLOPs=fl / (ms * 1e-3) / 1e12, share_of_dmma_peak=fl / (ms * 1e-3) / 1e12 / DMMA_PEAK_TFLOPS)
                                       for k, (ms, fl) in con.items()}))
    out["batched"] = rows

    # time to tol 1e-5 of a 64-value C grid against single solves of every eighth C value (extrapolated to the grid)
    Lc = 64
    C_ = c_grid(Lc)
    X_, Y_, its, info = AdaProx.adaptive_primal_dual_path(f=f, A=A, upper=C_, rule=rule, tol=1e-5, maxit=a.tol_maxit)
    path = dict(L=Lc, tol=1e-5, maxit=a.tol_maxit, solve_ms=info["solve_ms"], batched_evals=info["batched_evals"],
                converged=int((info["norm_res"] <= 1e-5).sum()), iters_median=float(np.median(its)), iters_max=int(its.max()))
    idx = np.arange(0, Lc, 8)
    sm, sit, dx = [], [], []
    for j in idx:
        xs, _, itj = AdaProx.adaptive_primal_dual(np.zeros(N), np.zeros(1), f=f, g=AdaProx.IndBox(0.0, float(C_[j])), h=AdaProx.IndZero(),
                                                  A=A, rule=rule, tol=1e-5, maxit=a.tol_maxit)
        sm.append(AdaProx.last_solve_info()["solve_ms"])
        sit.append(int(itj))
        dx.append(float(np.linalg.norm(X_[:, j] - xs) / max(np.linalg.norm(xs), 1e-300)))
    path["single_sampled"] = dict(C_index=idx.tolist(), solve_ms=sm, iters=sit, batch_iters_same_columns=[int(its[j]) for j in idx],
                                  rel_diff_x=dx)
    path["single_sum_ms_extrapolated"] = float(np.mean(sm) * Lc)
    path["speedup_vs_single_sum_extrapolated"] = path["single_sum_ms_extrapolated"] / info["solve_ms"]
    out["time_to_tol"] = path
    Zm.free()
    if form == "quadratic":
        Qm.free()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--tol-maxit", type=int, default=20000)
    ap.add_argument("--sizes", default="quadratic:20000,gram:20000,gram:50000")
    a = ap.parse_args()
    out = dict(bench="svm_c_path", d=2000, rule="OurRule(t=1, norm_A=sqrt(N))", C_grid="geomspace(1e-2, 1e1, L)", **gpu_facts(),
               dmma_peak_TFLOPs=DMMA_PEAK_TFLOPS)
    out["instances"] = [bench_instance(s.split(":")[0], int(s.split(":")[1]), 2000, a) for s in a.sizes.split(",")]
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
