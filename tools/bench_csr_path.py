"""Batched lambda path over the C2 sparse logistic instance (20242 x 47236 CSR, 1.5 M non-zeros): per-iteration time of the
batch for L = 32, 64, 128, 256 against the single-lambda adaptive_proxgrad on the same GPU in the same run, time to tol 1e-6 of
a 256-lambda path against the (extrapolated) sum of single solves, and the byte model of one batched iteration.

    python tools/bench_csr_path.py [--out FILE] [--reps 5] [--iters 20]

Prints one JSON line (and writes it to FILE).  Times are device-event times of the solve loop (adaprox_result.solve_ms)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import scipy.sparse as sp

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import adaprox_b200 as AdaProx  # noqa: E402


def gpu_facts():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi query failed: " + r.stderr)
    name, plim, clk = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=plim, max_sm_clock=clk)


def copy_peak_tbs(nbytes=4 << 30, reps=10):
    """Device-to-device copy rate (read + write bytes over time), the attainable HBM figure the byte model is set against."""
    a = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 0.0
    for _ in range(reps):
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 2 * nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    del a, b
    torch.cuda.empty_cache()
    return best


def spread(v):
    v = np.asarray(v, dtype=float)
    return dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--tol-maxit", type=int, default=20000)
    a = ap.parse_args()
    m, n = 20242, 47236
    rp, ci, va, y = AdaProx.synth.sparse_logreg(m, n, 0)
    X = sp.csr_matrix((va, ci, rp), shape=(m, n))
    nnz = int(X.nnz)
    gam = 4 * m / (va @ va + m)
    lam_max = AdaProx.synth.logreg_lambda_max(X, y)
    f = AdaProx.LogisticLoss(X, y)
    rule = AdaProx.OurRule(gamma=gam)
    out = dict(bench="csr_lambda_path", instance=dict(m=m, n=n, nnz=nnz, loss="logistic"), **gpu_facts())
    out["copy_peak_TBps"] = copy_peak_tbs()
    K = a.iters

    # single-lambda baseline (lambda = 0.03 lambda_max, as test_c2_sparse_logreg_full_shape), tol = 0: exactly K iterations
    AdaProx.adaptive_proxgrad(np.zeros(n + 1), f=f, g=AdaProx.NormL1(0.03 * lam_max), rule=rule, tol=0.0, maxit=3)
    single = []
    for _ in range(a.reps):
        AdaProx.adaptive_proxgrad(np.zeros(n + 1), f=f, g=AdaProx.NormL1(0.03 * lam_max), rule=rule, tol=0.0, maxit=K)
        single.append(1e3 * AdaProx.last_solve_info()["solve_ms"] / K)
    out["single_us_per_iter"] = spread(single)
    s_us = out["single_us_per_iter"]["median"]

    # batched iteration time, tol = 0: every column runs K iterations
    rows = []
    for Lc in (32, 64, 128, 256):
        lambdas = lam_max * (1e-3) ** (np.arange(Lc) / (Lc - 1))
        AdaProx.adaptive_proxgrad_path(None, f=f, lambdas=lambdas, rule=rule, tol=0.0, maxit=3)          # warm-up at this shape
        t = []
        for _ in range(a.reps):
            _, its, info = AdaProx.adaptive_proxgrad_path(None, f=f, lambdas=lambdas, rule=rule, tol=0.0, maxit=K)
            assert np.all(its == K)
            t.append(1e3 * info["solve_ms"] / info["batched_evals"])
        it_us = float(np.median(t))
        # byte model of one batched iteration
        gather = 2 * 8 * Lc * nnz                                # both sweeps gather one Lc-double row per non-zero (mostly L2)
        csr = 2 * 12 * nnz                                       # column index + value of X and X'
        vec = 8 * (n + 1) * Lc * 8 + 2 * m * Lc * 8              # iterate / gradient / v reads and writes; residual block write + read
        tot = gather + csr + vec
        rows.append(dict(L=Lc, iter_us=spread(t), us_per_lambda_iter=it_us / Lc, speedup_vs_single=s_us / (it_us / Lc),
                         bytes=dict(gather=gather, csr=csr, vector=vec, total=tot),
                         achieved_TBps=tot / (it_us * 1e-6) / 1e12, share_of_copy_peak=tot / (it_us * 1e-6) / 1e12 / out["copy_peak_TBps"]))
    out["batched"] = rows
    out["byte_model_note"] = ("gather bytes are whole rows of the lambda block, served mostly from L2 (the 97 MB iterate block and the 41 MB "
                              "residual block at L = 256 sit near the 126 MB L2): achieved_TBps is a mixed L2 + HBM figure, not an HBM rate")

    # time to tol 1e-6 of a 256-lambda path (lambda_max .. 1e-3 lambda_max) against single solves
    Lc = 256
    lambdas = lam_max * (1e-3) ** (np.arange(Lc) / (Lc - 1))
    _, its, info = AdaProx.adaptive_proxgrad_path(None, f=f, lambdas=lambdas, rule=rule, tol=1e-6, maxit=a.tol_maxit)
    path = dict(L=Lc, tol=1e-6, maxit=a.tol_maxit, solve_ms=info["solve_ms"], batched_evals=info["batched_evals"],
                converged=int((its < a.tol_maxit).sum()), iters_median=float(np.median(its)), iters_max=int(its.max()))
    idx = np.linspace(0, Lc - 1, 16).round().astype(int)
    sm, sit = [], []
    for j in idx:
        _, itj = AdaProx.adaptive_proxgrad(np.zeros(n + 1), f=f, g=AdaProx.NormL1(float(lambdas[j])), rule=rule, tol=1e-6, maxit=a.tol_maxit)
        sm.append(AdaProx.last_solve_info()["solve_ms"])
        sit.append(int(itj))
    path["single_sampled"] = dict(lambda_index=idx.tolist(), solve_ms=sm, iters=sit, batch_iters_same_columns=[int(its[j]) for j in idx])
    path["single_sum_ms_extrapolated"] = float(np.mean(sm) * Lc)
    path["speedup_vs_single_sum_extrapolated"] = path["single_sum_ms_extrapolated"] / info["solve_ms"]
    out["time_to_tol"] = path
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
