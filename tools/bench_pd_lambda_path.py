"""Batched lambda path of LAD and the square-root lasso (adaptive_primal_dual_lambda_path) on the C3 instance:
synth.dense_regression(50000, 2000), A = [X 1] (50000 x 2001), h = |A x - y|_1 (LAD) or |A x - y|_2 (square-root lasso),
f = Zero, OurRule(t = 1, norm_A = |A|_2).

For LAD at L = 32, 64, 128, 256 and the square-root lasso at L = 256: the median ms per batched iteration over --reps
repetitions (with min / max), us per lambda-iteration, the speed-up over the single-lambda adaptive_primal_dual iteration
timed in the same run, and each contraction of the iteration (A X and A' Y) timed alone with adaprox_time_path_gemm, in
TFLOP/s and as a share of the DMMA probe peak of profiles/r02_fp64_peaks.jsonl.

    python tools/bench_pd_lambda_path.py [--out FILE] [--reps 5] [--iters 20]

Prints one JSON line (and writes it to FILE).  Times are device-event times of the solve loop (adaprox_result.solve_ms)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
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
    return dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()), n=int(v.size))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    X, y = AdaProx.synth.dense_regression(50000, 2000)
    A = np.ascontiguousarray(np.hstack([X, np.ones((X.shape[0], 1))]))
    del X
    m, n = A.shape
    Am = AdaProx.DeviceMatrix(A)
    nA = float(np.linalg.norm(A, 2))
    rule = AdaProx.OurRule(t=1, norm_A=nA)
    K = a.iters
    out = dict(bench="pd_lambda_path", instance="dense_regression(50000, 2000), A = [X 1]", m=m, n=n, rule="OurRule(t=1, norm_A=|A|_2)",
               iters=K, reps=a.reps, **gpu_facts(), dmma_peak_TFLOPs=DMMA_PEAK_TFLOPS)
    lam_max = float(np.max(np.abs(A.T @ np.sign(y))))
    hs = dict(lad=AdaProx.Translate(AdaProx.NormL1(), -y), sqrt_lasso=AdaProx.Translate(AdaProx.NormL2(), -y))
    rows = []
    for kind, Ls in (("lad", (32, 64, 128, 256)), ("sqrt_lasso", (256,))):
        h = hs[kind]
        # single-lambda baseline, tol = 0: exactly K iterations
        kw = dict(f=AdaProx.Zero(), g=AdaProx.NormL1(0.1 * lam_max), h=h, A=Am, rule=rule, tol=0.0)
        AdaProx.adaptive_primal_dual(np.zeros(n), np.zeros(m), maxit=3, **kw)
        single = []
        for _ in range(a.reps):
            AdaProx.adaptive_primal_dual(np.zeros(n), np.zeros(m), maxit=K, **kw)
            single.append(1e3 * AdaProx.last_solve_info()["solve_ms"] / K)
        s = spread(single)
        rows.append(dict(problem=kind, single_us_per_iter=s))
        for L in Ls:
            lams = np.geomspace(1e-3, 1.0, L) * lam_max
            pk = dict(f=AdaProx.Zero(), h=h, A=Am, lambdas=lams, rule=rule, tol=0.0)
            AdaProx.adaptive_primal_dual_lambda_path(maxit=3, **pk)                   # warm-up at this shape
            t = []
            for _ in range(a.reps):
                _, _, its, info = AdaProx.adaptive_primal_dual_lambda_path(maxit=K, **pk)
                assert np.all(its == K)
                t.append(info["solve_ms"] / info["batched_evals"])
            it_ms = float(np.median(t))
            fl = 2.0 * m * n * L
            con = dict(AX=Am.time_path_gemm(L, 0, reps=10), ATY=Am.time_path_gemm(L, 1, reps=10))
            rows.append(dict(problem=kind, L=L, ms_per_iter=spread(t), us_per_lambda_iter=1e3 * it_ms / L,
                             speedup_vs_single=s["median"] / (1e3 * it_ms / L), path_TFLOPs=2 * fl / (it_ms * 1e-3) / 1e12,
                             contractions={k: dict(ms=ms, TFLOPs=fl / (ms * 1e-3) / 1e12,
                                                   share_of_dmma_peak=fl / (ms * 1e-3) / 1e12 / DMMA_PEAK_TFLOPS)
                                           for k, ms in con.items()}))
    out["results"] = rows
    Am.free()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
