"""Batched lambda path over a CSR smooth term (adaprox_solve_lambda_path with a sparse LogisticLoss or LinearLeastSquares).

Column j of the batch must be what adaptive_proxgrad returns for NormL1(lambdas[j]): the oracle runs the columns one by one
(oracle.adaptive_proxgrad_path).  Free-running stepsize sequences are bounded by the rounding drift of the algorithm
(oracle/drift.py), stopping iterations by the oracle's own sensitivity to the summation order.
"""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import adaprox_oracle as O
from oracle import drift

pytestmark = pytest.mark.gpu


def _logreg(AdaProx, m, n, seed=0, lo=40, hi=112):
    rp, ci, va, y = AdaProx.synth.sparse_logreg(m, n, seed, nnz_lo=lo, nnz_hi=hi)
    return sp.csr_matrix((va, ci, rp), shape=(m, n)), y


def _problem(AdaProx, kind, m, n, lo, hi, seed=0):
    """-> (X, v, gamma, lam_max, make_dev_f, make_oracle_f, n_unknowns): v = labels (logistic) or b (least squares)."""
    X, y = _logreg(AdaProx, m, n, seed, lo, hi)
    if kind == "logistic":
        gam = 4 * m / (X.data @ X.data + m)                      # 4 m / |[X 1]|_F^2 (SURVEY 8d)
        return X, y, gam, AdaProx.synth.logreg_lambda_max(X, y), AdaProx.LogisticLoss, O.LogisticLoss, n + 1
    rng = np.random.default_rng(seed)
    w = np.where(rng.random(n) < 0.05, rng.standard_normal(n), 0.0)
    b = X @ w + 0.1 * rng.standard_normal(m)
    gam = 1 / AdaProx.synth.spectral_norm_sq(X.toarray(), iters=500)
    return X, b, gam, float(np.max(np.abs(X.T @ b))), AdaProx.LinearLeastSquares, O.LinearLeastSquares, n


def _objective(kind, X, v, w, lam):
    if kind == "logistic":
        logits = X @ w[:-1] + w[-1]
        f = -np.mean((v - 1) * logits - np.log(1 + np.exp(-logits)))
    else:
        f = 0.5 * np.linalg.norm(X @ w - v) ** 2
    return f + lam * np.abs(w).sum()


CASES = [("logistic", 600, 900, 1, 40, 112), ("logistic", 600, 900, 33, 8, 30), ("logistic", 1500, 4000, 7, 20, 60),
         ("logistic", 1500, 4000, 130, 40, 112), ("lsq", 600, 900, 33, 40, 112), ("lsq", 1500, 4000, 7, 20, 60)]


@pytest.mark.parametrize("kind,m,n,Lc,lo,hi", CASES)
def test_csr_path_matches_per_lambda_solves(AdaProx, kind, m, n, Lc, lo, hi):
    X, v, gam, lam_max, Fd, Fo, nu = _problem(AdaProx, kind, m, n, lo, hi)
    lambdas = lam_max * (1e-2) ** (np.arange(Lc) / max(Lc - 1, 1))
    maxit, H, K = 800, 40, 25
    Xd, its, info = AdaProx.adaptive_proxgrad_path(None, f=Fd(X, v), lambdas=lambdas, rule=AdaProx.OurRule(gamma=gam), tol=1e-6,
                                                   maxit=maxit, history=H)
    Xo, itso, gh, rh, oh = O.adaptive_proxgrad_path(np.zeros((nu, Lc)), f=Fo(X, v), lambdas=lambdas, rule_of=lambda j: O.OurRule(gamma=gam),
                                                   tol=1e-6, maxit=maxit, history=H)
    assert Xd.shape == (nu, Lc) and info["batched_evals"] >= int(its.max())
    sample = sorted({0, Lc // 2, Lc - 1})
    for j in sample:
        kj = int(min(K, its[j], itso[j]))
        if kj < 3:
            continue

        def run(dtype, rng, j=j, kj=kj):
            Xr, vr = X, v
            if rng is not None:                                  # permute samples AND features: other summation orders
                pr, pc = rng.permutation(m), rng.permutation(n)
                Xr, vr = X[pr][:, pc].tocsr(), v[pr]
            log = []
            O.adaptive_proxgrad(np.zeros(nu, dtype=dtype), f=Fo(Xr.astype(dtype), vr.astype(dtype)), g=O.NormL1(float(lambdas[j])),
                                rule=O.OurRule(gamma=gam), tol=0.0, maxit=kj, log=log)
            return log

        truth = drift.collect(run, nperm=2, seed=j)
        ok, dd, allowed = drift.check_inside(info["gamma_hist"][:kj, j], truth, factor=20.0, floor=1e-12)
        assert ok, (j, float(np.max(dd / allowed)), float(dd.max()))
    live = ~np.isnan(oh[:K]) & ~np.isnan(info["obj_hist"][:K])
    assert np.allclose(info["obj_hist"][:K][live], oh[:K][live], rtol=1e-10)
    assert np.all(np.abs(its - itso) <= np.maximum(5, 0.1 * itso)), (its, itso)
    rng = np.random.default_rng(1)
    pr, pc = rng.permutation(m), rng.permutation(n)
    Xp = X[pr][:, pc].tocsr()
    for j in sample:
        _, itp = O.adaptive_proxgrad(np.zeros(nu), f=Fo(Xp, v[pr]), g=O.NormL1(float(lambdas[j])), rule=O.OurRule(gamma=gam), tol=1e-6, maxit=maxit)
        assert abs(int(its[j]) - int(itso[j])) <= max(3, 0.03 * itso[j], 2 * abs(itp - int(itso[j]))), (j, its[j], itso[j], itp)
    # columns that converged on both sides: the minimiser to O(tol), the objective to 1e-9 (columns cut off at maxit are
    # compared through their records above: their trajectories are chaotic w.r.t. rounding, SURVEY 0.7)
    conv = (its < maxit) & (itso < maxit)
    assert conv.sum() >= (1 if Lc > 1 else 0)
    fd = np.array([_objective(kind, X, v, Xd[:, j], lambdas[j]) for j in range(Lc)])
    fo = np.array([_objective(kind, X, v, Xo[:, j], lambdas[j]) for j in range(Lc)])
    if conv.any():
        scale = np.maximum(np.linalg.norm(Xo, axis=0), 1e-12)
        assert np.max((np.linalg.norm(Xd - Xo, axis=0) / scale)[conv]) < 1e-4
        assert np.max((np.abs(fd - fo) / np.abs(fo))[conv]) < 1e-9
    assert np.all(info["norm_res"][its < maxit] <= 1e-6)


@pytest.mark.parametrize("rule", ["OurRule", "FixedStepsize", "MalitskyMishchenkoRule", "OurRulePlus"])
def test_csr_path_equals_single_solves_on_device(AdaProx, rule):
    """The batched columns against adaptive_proxgrad per lambda on the same device, with per-column gamma0 and a non-zero X0."""
    m, n, Lc = 600, 900, 6
    X, y = _logreg(AdaProx, m, n, 3)
    gam = 4 * m / (X.data @ X.data + m)
    lambdas = AdaProx.synth.logreg_lambda_max(X, y) * np.linspace(0.2, 0.8, Lc)
    gam0 = gam * np.linspace(0.5, 1.0, Lc)
    X0 = 0.01 * np.random.default_rng(0).standard_normal((n + 1, Lc))
    R = getattr(AdaProx, rule)
    f = AdaProx.LogisticLoss(X, y)
    maxit = 3000
    Xd, its, info = AdaProx.adaptive_proxgrad_path(X0, f=f, lambdas=lambdas, rule=R(gamma=gam), gamma0=gam0, tol=1e-5, maxit=maxit)
    for j in range(Lc):
        xj, itj = AdaProx.adaptive_proxgrad(X0[:, j], f=f, g=AdaProx.NormL1(lambdas[j]), rule=R(gamma=gam0[j]), tol=1e-5, maxit=maxit)
        if rule == "FixedStepsize":                              # contractive: the two summation orders stay within rounding
            assert abs(int(its[j]) - itj) <= 1, (j, its[j], itj)
            assert np.linalg.norm(Xd[:, j] - xj) <= 1e-6 * max(np.linalg.norm(xj), 1e-9)
        else:                                                    # both stopped at norm_res <= 1e-5; the adaptive rules amplify rounding
            assert abs(int(its[j]) - itj) <= max(3, 0.1 * itj), (j, its[j], itj)
            assert np.linalg.norm(Xd[:, j] - xj) <= 2e-2 * max(np.linalg.norm(xj), 1e-9)
    if rule != "FixedStepsize":
        assert (its < maxit).sum() >= Lc // 2


def test_csr_path_deterministic_and_position_free(AdaProx):
    """Reruns are bit-identical; permuting the lambdas permutes the columns bit for bit; a column does not depend on the batch
    width either (L = 31, 32, 33, 65 around the 32-column padding)."""
    m, n = 600, 900
    X, y = _logreg(AdaProx, m, n, 1)
    gam = 4 * m / (X.data @ X.data + m)
    lambdas = AdaProx.synth.logreg_lambda_max(X, y) * (1e-2) ** (np.arange(65) / 64)
    f = AdaProx.LogisticLoss(X, y)
    kw = dict(f=f, rule=AdaProx.OurRule(gamma=gam), tol=1e-6, maxit=300, history=30)
    A1 = AdaProx.adaptive_proxgrad_path(None, lambdas=lambdas, **kw)
    A2 = AdaProx.adaptive_proxgrad_path(None, lambdas=lambdas, **kw)
    assert np.array_equal(A1[0], A2[0]) and np.array_equal(A1[1], A2[1])
    for key in ("gamma_hist", "res_hist", "obj_hist", "norm_res", "gamma", "f_x"):
        assert np.array_equal(A1[2][key], A2[2][key], equal_nan=True), key
    perm = np.random.default_rng(0).permutation(65)
    B = AdaProx.adaptive_proxgrad_path(None, lambdas=lambdas[perm], **kw)
    assert np.array_equal(B[0], A1[0][:, perm]) and np.array_equal(B[1], A1[1][perm])
    assert np.array_equal(B[2]["gamma_hist"], A1[2]["gamma_hist"][:, perm], equal_nan=True)
    for Lc in (31, 32, 33):
        C = AdaProx.adaptive_proxgrad_path(None, lambdas=lambdas[:Lc], **kw)
        assert np.array_equal(C[0], A1[0][:, :Lc]) and np.array_equal(C[1], A1[1][:Lc]), Lc
        assert np.array_equal(C[2]["obj_hist"], A1[2]["obj_hist"][:, :Lc], equal_nan=True), Lc


def test_csr_path_edge_cases(AdaProx):
    """L = 1, lambda = 0, maxit = 1, an empty row of X and a feature without nonzeros, columns that stop far apart (NaN in the
    history after the stop)."""
    m, n = 300, 500
    X, y = _logreg(AdaProx, m, n, 4, 10, 30)
    X = X.tolil()
    X[5, :] = 0                                                  # empty row of X
    X[:, 7] = 0                                                  # empty row of X'
    X = X.tocsr()
    X.eliminate_zeros()
    assert X.indptr[6] == X.indptr[5] and 7 not in set(X.indices)
    gam = 4 * m / (X.data @ X.data + m)
    lam_max = AdaProx.synth.logreg_lambda_max(X, y)
    b = X @ np.linspace(-1, 1, n) + 0.05
    gls = 1 / AdaProx.synth.spectral_norm_sq(X.toarray(), iters=500)
    for Fd, Fo, v, g, nu, lams in ((AdaProx.LogisticLoss, O.LogisticLoss, y, gam, n + 1, [0.0, 0.1 * lam_max, lam_max]),
                                   (AdaProx.LinearLeastSquares, O.LinearLeastSquares, b, gls, n, [0.0, 0.5, 5.0])):
        lams = np.asarray(lams)
        for maxit in (1, 40):
            Xd, its, info = AdaProx.adaptive_proxgrad_path(None, f=Fd(X, v), lambdas=lams, rule=AdaProx.OurRule(gamma=g), tol=0.0, maxit=maxit,
                                                           history=maxit)
            Xo, itso, gh, rh, oh = O.adaptive_proxgrad_path(np.zeros((nu, len(lams))), f=Fo(X, v), lambdas=lams,
                                                           rule_of=lambda j: O.OurRule(gamma=g), tol=0.0, maxit=maxit, history=maxit)
            assert its.max() == maxit and np.array_equal(its, itso)          # tol = 0 still stops a column whose residual is exactly 0
            k = min(maxit, 15)                                   # where the free-running stepsizes still agree to ~1e-12
            assert np.allclose(info["obj_hist"][:k], oh[:k], rtol=1e-10, equal_nan=True)
            assert np.allclose(info["res_hist"][:k], rh[:k], rtol=1e-9, equal_nan=True)
            assert np.all(Xd[7, :] == 0)                         # no data for feature 7: its gradient is 0, it never leaves 0
            if maxit == 1:
                assert np.allclose(Xd, Xo, rtol=1e-12, atol=1e-15)
        # L = 1
        x1, it1, _ = AdaProx.adaptive_proxgrad_path(None, f=Fd(X, v), lambdas=lams[1:2], rule=AdaProx.OurRule(gamma=g), tol=0.0, maxit=40)
        assert it1[0] == 40 and np.linalg.norm(x1[:, 0] - Xd[:, 1]) == 0.0          # a column does not depend on the batch
    # columns that stop far apart; the history is NaN after a column stopped
    lams = lam_max * np.array([1.0, 0.3, 0.03, 0.01])
    H = 400
    Xd, its, info = AdaProx.adaptive_proxgrad_path(None, f=AdaProx.LogisticLoss(X, y), lambdas=lams, rule=AdaProx.OurRule(gamma=gam), tol=1e-6,
                                                   maxit=H, history=H)
    assert its.min() < its.max() / 2, its
    for j in range(len(lams)):
        k = int(its[j])
        assert np.all(np.isfinite(info["gamma_hist"][:k, j])) and np.all(np.isnan(info["gamma_hist"][k:, j])), j
        assert np.all(np.isnan(info["obj_hist"][k:, j])) and np.all(np.isnan(info["res_hist"][k:, j])), j


def test_csr_path_errors(AdaProx):
    m, n = 200, 300
    X, y = _logreg(AdaProx, m, n, 5, 10, 30)
    gam = 4 * m / (X.data @ X.data + m)
    rule = AdaProx.OurRule(gamma=gam)
    with pytest.raises(AdaProx.AdaproxError) as e:               # dense logistic: no batched kernel
        AdaProx.adaptive_proxgrad_path(None, f=AdaProx.LogisticLoss(X.toarray(), y), lambdas=[0.1], rule=rule)
    assert e.value.code == -3
    Xs = AdaProx.DeviceMatrix(X)
    Xs.set_shard(2 * m, 0)                                       # a row shard of a larger matrix
    with pytest.raises(AdaProx.AdaproxError) as e:
        AdaProx.adaptive_proxgrad_path(None, f=AdaProx.LogisticLoss(Xs, y), lambdas=[0.1], rule=rule)
    assert e.value.code == -3
    f = AdaProx.LogisticLoss(X, y)
    with pytest.raises(AdaProx.AdaproxError) as e:
        AdaProx.adaptive_proxgrad_path(None, f=f, lambdas=[0.1, -1.0], rule=rule)
    assert e.value.code == -1
    with pytest.raises(ValueError):
        AdaProx.adaptive_proxgrad_path(np.zeros((n, 2)), f=f, lambdas=[0.1, 0.2], rule=rule)         # n + 1 rows expected
    with pytest.raises(ValueError):
        AdaProx.adaptive_proxgrad_path(None, f=f, lambdas=[0.1, 0.2], rule=rule, gamma0=[gam])


def test_csr_path_c2_full_shape(AdaProx):
    """C2 (20242 x 47236 CSR, 1.5 M non-zeros) with 64 lambdas, 30 iterations at tol = 0: eight sampled columns against the
    oracle's natural-order run inside the envelope of three permuted runs."""
    m, n, Lc, K = 20242, 47236, 64, 30
    X, y = _logreg(AdaProx, m, n, 0)
    gam = 4 * m / (X.data @ X.data + m)
    lambdas = AdaProx.synth.logreg_lambda_max(X, y) * (1e-2) ** (np.arange(Lc) / (Lc - 1))
    try:
        Xd, its, info = AdaProx.adaptive_proxgrad_path(None, f=AdaProx.LogisticLoss(X, y), lambdas=lambdas, rule=AdaProx.OurRule(gamma=gam),
                                                       tol=0.0, maxit=K, history=K)
    except AdaProx.AdaproxError as e:
        if e.code == -5:
            pytest.skip(f"device memory: {e}")
        raise
    assert np.all(its == K)
    fo = O.LogisticLoss(X, y)
    rng = np.random.default_rng(0)
    perms = []
    for _ in range(3):
        pr, pc = rng.permutation(m), rng.permutation(n)
        perms.append(O.LogisticLoss(X[pr][:, pc].tocsr(), y[pr]))
    for j in (0, 9, 18, 27, 36, 45, 54, 63):
        lam = O.NormL1(float(lambdas[j]))
        logo = []
        xo, _ = O.adaptive_proxgrad(np.zeros(n + 1), f=fo, g=lam, rule=O.OurRule(gamma=gam), tol=0.0, maxit=K, log=logo)
        gps = []
        for fp in perms:
            logp = []
            O.adaptive_proxgrad(np.zeros(n + 1), f=fp, g=lam, rule=O.OurRule(gamma=gam), tol=0.0, maxit=K, log=logp)
            gps.append([r["gamma"] for r in logp])
        go = np.array([r["gamma"] for r in logo])
        env = drift.perm_envelope(go, gps)
        gd = info["gamma_hist"][:K, j]
        assert np.all(np.abs(gd / go - 1) <= np.maximum(1e-12, 20 * env)), (j, np.abs(gd / go - 1).max(), env.max())
        assert np.allclose(info["res_hist"][:K, j], [r["norm_res"] for r in logo], rtol=1e-10), j
        assert np.allclose(info["obj_hist"][:K, j], [r["objective"] for r in logo], rtol=1e-10), j
        assert np.linalg.norm(Xd[:, j] - xo) <= 1e-9 * max(np.linalg.norm(xo), 1e-300), j
