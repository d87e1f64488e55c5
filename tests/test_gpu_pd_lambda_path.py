"""The batched lambda path of LAD and the square-root lasso (adaptive_primal_dual_lambda_path, include/adaprox.h:
adaprox_solve_pd_lambda_path).

Column j is AdaPDM / Condat-Vu on lambda_j |x|_1 + h(A x) with f = Zero and h = |. - b|_1 (LAD) or |. - b|_2 (square-root
lasso).  The checks:
  - one and two primal-dual steps of every column against the extended-precision reference (xprec_reference.PD: pd_fixed,
    pd_ourrule) under its a-priori rounding bounds, at shapes that reach both tile widths and K-split 1 and > 1 of both
    contractions A X and A' Y; the square-root lasso cases have columns whose w / sigma + shift lies inside the ball of the
    dual prox and columns where it lies outside;
  - per-lambda agreement with the single device solve: with f = Zero the stepsizes depend on the stepsize history only, so
    the gamma and sigma histories are equal bit for bit (the NaN of Malitsky-Mishchenko where dx = 0 included), and x, y lie
    inside 20 x the drift envelope of the float64 oracle under permuted summation orders;
  - frozen columns and their history, maxit = 0, bitwise determinism under reruns and permutations of the lambdas, L = 1;
  - every refusal of the entry point;
  - the C3 shape (50000 x 2001, 64 lambdas), sampled columns against the oracle.
"""
import ctypes as C

import numpy as np
import pytest

from adaprox_b200 import _lib as Lb
from oracle import adaprox_oracle as O
from test_gpu_lambda_path_reference import path_ksplit
from xprec_reference import LinMap, PD, Prox, Smooth, pd_fixed, pd_ourrule, within


# ---------------------------------------------------------------- shapes and the contractions they reach
# (m, n, L): A is m x n
SHAPES = [(2000, 50, 40), (300, 2000, 40), (200, 300, 70), (2000, 50, 100), (300, 2000, 70)]


def branches(shapes, sm):
    """-> names of the branches reached: tile width, AX = A X (tiles over m, K = n) and ATY = A' Y (tiles over n, K = m)
    with K-split 1 or > 1"""
    hit = set()
    for m, n, L in shapes:
        hit.add("tile:narrow" if L <= 64 else "tile:wide")
        hit.add("AX:" + ("1" if path_ksplit(m, n, L, sm) == 1 else ">1"))
        hit.add("ATY:" + ("1" if path_ksplit(n, m, L, sm) == 1 else ">1"))
    return hit


REQUIRED = {"tile:narrow", "tile:wide", "AX:1", "AX:>1", "ATY:1", "ATY:>1"}


def test_shapes_reach_every_contraction_branch_at_148_sms():
    assert REQUIRED <= branches(SHAPES, 148), REQUIRED - branches(SHAPES, 148)


# ---------------------------------------------------------------- instances
def instance(m, n, L, kind, seed=0):
    """A (m x n), b, lambdas over two decades below lambda_max, X0 with zeros, Y0 inside (LAD: the box) or near (l2) the
    dual ball of h"""
    rng = np.random.default_rng([m, n, L, seed])
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    b = rng.standard_normal(m)
    lam_max = np.max(np.abs(A.T @ (np.sign(b) if kind == "l1" else b / np.linalg.norm(b))))
    lams = np.geomspace(0.01, 1.0, L) * lam_max
    X0 = 0.3 * rng.standard_normal((n, L))
    X0[rng.random(X0.shape) < 0.3] = 0.0
    Y0 = rng.uniform(-1.0, 1.0, (m, L)) if kind == "l1" else 0.5 * rng.standard_normal((m, L)) / np.sqrt(m)
    return A, b, lams, X0, Y0


def dev_h(AdaProx, kind, b):
    return AdaProx.Translate(AdaProx.NormL1() if kind == "l1" else AdaProx.NormL2(), -b)


def oracle_h(kind, b):
    return O.Translate(O.NormL1() if kind == "l1" else O.NormL2(), -b)


def ourrule_gammas(nA, t, L):
    """OurRule gamma_0 with a = t gamma |A| on both sides of the switch of its min: with f = Zero the third term is
    gamma (1 - 4 a^2)^(1/4) / sqrt(2 a), below gamma sqrt(2) for a > 0.2236, and 1 / (2 Theta t |A|) wins for a > 0.2946"""
    a = np.concatenate([np.linspace(0.05, 0.2, L - L // 2), np.linspace(0.24, 0.28, L // 2)])
    return a / (t * nA)


# ---------------------------------------------------------------- (1) one and two steps against the reference
@pytest.mark.gpu
def test_shapes_reach_every_contraction_branch_on_this_device(AdaProx):
    sm = AdaProx.default_device().info()["sm_count"]
    assert REQUIRED <= branches(SHAPES, sm), REQUIRED - branches(SHAPES, sm)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["l1", "l2"])
@pytest.mark.parametrize("shape", SHAPES, ids=[f"m{s[0]}-n{s[1]}-L{s[2]}" for s in SHAPES])
def test_one_and_two_steps_match_extended_precision(AdaProx, shape, kind):
    m, n, L = shape
    A, b, lams, X0, Y0 = instance(m, n, L, kind)
    nA = float(np.linalg.norm(A, 2))
    t = 1.0
    gf = np.geomspace(1e-3, 0.5, L) / nA            # sigma = gamma: |w / sigma - b| on both sides of 1 / sigma (l2)
    go = ourrule_gammas(nA, t, L)
    fixed = AdaProx.FixedStepsize(gf[0], t)
    our = AdaProx.OurRule(gamma=go[0], t=t, norm_A=nA)
    kw = dict(f=AdaProx.Zero(), h=dev_h(AdaProx, kind, b), A=A, lambdas=lams, tol=0.0)
    x1, y0, it0, _ = AdaProx.adaptive_primal_dual_lambda_path(X0, Y0, rule=fixed, gamma0=gf, maxit=0, **kw)
    x2, y1, it1, i1 = AdaProx.adaptive_primal_dual_lambda_path(X0, Y0, rule=fixed, gamma0=gf, maxit=1, history=1, **kw)
    xo, yo, ito, io = AdaProx.adaptive_primal_dual_lambda_path(X0, Y0, rule=our, gamma0=go, maxit=1, history=1, **kw)
    assert AdaProx.last_solve_info()["matrix_passes"] == 2
    assert np.all(it0 == 0) and np.all(it1 == 1) and np.all(ito == 1)
    assert np.array_equal(y0, Y0), "maxit = 0: Y0 comes back bit for bit"
    Amap, h = LinMap(A), Prox(kind, 1.0, shift=-b)
    inside = []
    for j in range(L):
        P = PD(Smooth("zero", n=n), Prox("l1", lams[j]), h, Amap)
        R = pd_fixed(P, X0[:, j], Y0[:, j], gf[j], t)
        ok, ratio = within(x1[:, j], R["X1"], R["B1"])
        assert ok, ("maxit = 0: x_1", j, ratio)
        ok, ratio = within(x2[:, j], R["X2"], R["B2"])
        assert ok, ("maxit = 1: x_2", j, ratio)
        D = R["D"]
        ok, ratio = within(y1[:, j], D["Y1"], D["ey1"] + D["sy1"])
        assert ok, ("maxit = 1: y_1", j, ratio)
        assert i1["gamma"][j] == gf[j] and i1["sigma"][j] == R["sigma"], "FixedStepsize: gamma and sigma exact"
        assert i1["gamma_hist"][0, j] == gf[j]
        ok, ratio = within(i1["res_hist"][0, j], R["res1"], R["dres1"])
        assert ok, ("norm_res", j, ratio)
        ok, ratio = within(i1["obj_hist"][0, j], R["obj1"], R["dobj1"])
        assert ok, ("objective", j, ratio)
        if kind == "l2":
            # the block soft threshold of the dual step: |w / sigma + shift| against its radius 1 / sigma
            s = R["sigma"]
            inside.append(float(np.linalg.norm(D["W"] / s - b)) * s < 1.0)
        Ro = pd_ourrule(P, X0[:, j], Y0[:, j], go[j], t, nA)
        ok, ratio = within(io["gamma_hist"][0, j], Ro["gamma1"], Ro["dgamma1"])
        assert ok, ("OurRule gamma_1", j, ratio)
        ok, ratio = within(xo[:, j], Ro["X2"], Ro["B2"])
        assert ok, ("OurRule x_2", j, ratio)
        D = Ro["D"]
        ok, ratio = within(yo[:, j], D["Y1"], D["ey1"] + D["sy1"])
        assert ok, ("OurRule y_1", j, ratio)
    if kind == "l2":
        assert any(inside) and not all(inside), "the columns should reach both branches of the NormL2 prox"


# ---------------------------------------------------------------- (2) per-lambda agreement with the single solve
PAR_M, PAR_N, PAR_L, PAR_IT = 600, 150, 40, 100
RULES = ["our", "condat_vu", "mm"]


def parity_problem(AdaProx, kind, rule, seed=1):
    """PAR_L lambdas; the last one lies above every |A' y| over the dual ball of h, so its x stays 0 for every y"""
    A, b, lams, _, _ = instance(PAR_M, PAR_N, PAR_L, kind, seed=seed)
    col = np.abs(A).sum(axis=0) if kind == "l1" else np.linalg.norm(A, axis=0)
    lams = lams.copy()
    lams[-1] = 1.1 * np.max(col)
    nA = float(np.linalg.norm(A, 2))
    if rule == "our":
        r, mk = AdaProx.OurRule(t=1.0, norm_A=nA), (lambda M: M.OurRule(t=1.0, norm_A=nA))
    elif rule == "condat_vu":
        nF = float(np.linalg.norm(A))                 # src/AdaProx.jl:398-412 with Lf = 0: alpha = 1
        gam, sig = 1.0 / (0.0 / 2 + nF / 1.0), 0.99 / (nF * 1.0)
        t = float(np.sqrt(sig / gam))
        r, mk = AdaProx.FixedStepsize(gam, t), (lambda M: M.FixedStepsize(gam, t))
    else:
        r, mk = AdaProx.MalitskyMishchenkoRule(0.5 / nA, 0.9), (lambda M: M.MalitskyMishchenkoRule(0.5 / nA, 0.9))
    return A, b, lams, r, mk


def oracle_runs(A, b, lam, kind, mk, maxit, nperm=3, seed=0):
    """float64 oracle: natural order, then nperm runs with the rows and columns of A permuted -> [(x, y), ...]"""
    def run(Ap, bp):
        return O.adaptive_primal_dual(np.zeros(Ap.shape[1]), np.zeros(Ap.shape[0]), f=O.Zero(), g=O.NormL1(lam),
                                      h=oracle_h(kind, bp), A=Ap, rule=mk(O), tol=0.0, maxit=maxit)[:2]
    out = [run(A, b)]
    rng = np.random.default_rng(seed)
    for _ in range(nperm):
        pr, pc = rng.permutation(A.shape[0]), rng.permutation(A.shape[1])
        xp, yp = run(np.ascontiguousarray(A[pr][:, pc]), b[pr])
        x, y = np.empty_like(xp), np.empty_like(yp)
        x[pc], y[pr] = xp, yp
        out.append((x, y))
    return out


def inside_envelope(got, runs, k, factor=20.0, floor=1e-14):
    """|got - oracle| / |oracle| <= factor x the largest such distance of the permuted-order oracle runs (never tighter
    than floor: an iterate the rounding cannot touch, such as x = 0, has an envelope of 0).  Non-finite entries must be
    non-finite in both."""
    base = runs[0][k]
    if not np.all(np.isfinite(base)):
        return bool(np.array_equal(np.isfinite(got), np.isfinite(base))), 0.0
    nb = max(np.linalg.norm(base), 1e-300)
    env = max(np.linalg.norm(r[k] - base) / nb for r in runs[1:])
    d = np.linalg.norm(got - base) / nb
    return bool(np.all(np.isfinite(got)) and d <= max(floor, factor * env)), d / max(floor, factor * env)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["l1", "l2"])
@pytest.mark.parametrize("rule", RULES)
def test_every_column_matches_the_single_solve(AdaProx, kind, rule):
    A, b, lams, r, mk = parity_problem(AdaProx, kind, rule)
    h = dev_h(AdaProx, kind, b)
    X, Y, its, info = AdaProx.adaptive_primal_dual_lambda_path(f=AdaProx.Zero(), h=h, A=A, lambdas=lams, rule=r, tol=0.0,
                                                               maxit=PAR_IT, history=PAR_IT)
    assert np.all(its == PAR_IT)
    tt = r.t * r.t
    for j in range(PAR_L):
        log = []
        xs, ys, its_s = AdaProx.adaptive_primal_dual(np.zeros(PAR_N), np.zeros(PAR_M), f=AdaProx.Zero(), g=AdaProx.NormL1(lams[j]),
                                                     h=h, A=A, rule=r, tol=0.0, maxit=PAR_IT, log=log)
        s = AdaProx.last_solve_info()
        assert its_s == PAR_IT
        gam_s = np.array([rec["gamma"] for rec in log])
        sig_s = np.array([rec["sigma"] for rec in log])
        assert np.array_equal(info["gamma_hist"][:, j], gam_s, equal_nan=True), (j, info["gamma_hist"][:, j], gam_s)
        assert np.array_equal(info["gamma_hist"][:, j] * tt, sig_s, equal_nan=True), j
        assert np.array_equal(info["gamma"][j], s["final_gamma"], equal_nan=True)
        assert np.array_equal(info["sigma"][j], s["final_sigma"], equal_nan=True)
        if j == PAR_L - 1 and rule != "mm":
            assert not np.any(X[:, j]) and not np.any(xs), "lambda above lambda_max: x stays 0"
    if rule == "mm":
        # f = Zero: dx = 0 on the x = 0 column makes Malitsky-Mishchenko's L = 0 / 0 (src/AdaProx.jl:228)
        assert np.isnan(info["gamma_hist"][0, -1])
    for j in (0, PAR_L // 2, PAR_L - 2, PAR_L - 1):
        runs = oracle_runs(A, b, lams[j], kind, mk, PAR_IT)
        for k, got in ((0, X[:, j]), (1, Y[:, j])):
            ok, ratio = inside_envelope(got, runs, k)
            assert ok, (j, "xy"[k], ratio)


STOP_TOL = dict(l1=1e-2, l2=1e-4)      # LAD's residual falls slowly: about 1000 to 4000 iterations at 1e-2


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["l1", "l2"])
def test_iteration_counts_match_the_single_solve(AdaProx, kind):
    A, b, lams, r, _ = parity_problem(AdaProx, kind, "our", seed=2)
    h = dev_h(AdaProx, kind, b)
    tol, maxit = STOP_TOL[kind], 6000
    X, Y, its, info = AdaProx.adaptive_primal_dual_lambda_path(f=AdaProx.Zero(), h=h, A=A, lambdas=lams, rule=r, tol=tol,
                                                               maxit=maxit)
    assert its.max() >= 2 * its.min(), ("the lambdas should stop at very different iterations", its)
    for j in range(0, PAR_L, 3):
        xs, ys, its_s = AdaProx.adaptive_primal_dual(np.zeros(PAR_N), np.zeros(PAR_M), f=AdaProx.Zero(), g=AdaProx.NormL1(lams[j]),
                                                     h=h, A=A, rule=r, tol=tol, maxit=maxit)
        assert its[j] == its_s, (j, its[j], its_s)


# ---------------------------------------------------------------- (3) batch behaviour
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["l1", "l2"])
def test_columns_freeze_at_their_stop_and_the_history_ends_there(AdaProx, kind):
    A, b, lams, r, _ = parity_problem(AdaProx, kind, "our", seed=2)
    h = dev_h(AdaProx, kind, b)
    tol, maxit = STOP_TOL[kind], 6000
    X, Y, its, info = AdaProx.adaptive_primal_dual_lambda_path(f=AdaProx.Zero(), h=h, A=A, lambdas=lams, rule=r, tol=tol,
                                                               maxit=maxit, history=maxit)
    res = info["res_hist"]
    for j in range(PAR_L):
        k = int(its[j])
        assert 1 <= k < maxit
        first = int(np.argmax(res[:, j] <= tol)) + 1
        assert res[first - 1, j] <= tol and first == k, (j, first, k)
        assert np.all(np.isfinite(res[:k, j])) and np.all(np.isnan(res[k:, j]))
        assert np.all(np.isnan(info["gamma_hist"][k:, j])) and np.all(np.isnan(info["obj_hist"][k:, j]))
        assert np.all(np.isfinite(info["obj_hist"][:k, j]))
        assert info["gamma_hist"][k - 1, j] == info["gamma"][j] and res[k - 1, j] == info["norm_res"][j]
    # the result of a stopped column is x_k: maxit = k - 1 returns x_k too; y is the dual iterate of iteration k
    j = int(np.argmin(its))
    Xk, Yk, itk, _ = AdaProx.adaptive_primal_dual_lambda_path(f=AdaProx.Zero(), h=h, A=A, lambdas=lams, rule=r, tol=0.0,
                                                              maxit=int(its[j]) - 1)
    assert np.all(itk == its[j] - 1)
    assert np.array_equal(Xk[:, j], X[:, j])
    Xk1, Yk1, _, _ = AdaProx.adaptive_primal_dual_lambda_path(f=AdaProx.Zero(), h=h, A=A, lambdas=lams, rule=r, tol=0.0,
                                                              maxit=int(its[j]))
    assert np.array_equal(Yk1[:, j], Y[:, j])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["l1", "l2"])
def test_maxit_zero_matches_the_single_solve(AdaProx, kind):
    A, b, lams, X0, Y0 = instance(PAR_M, PAR_N, 6, kind, seed=3)
    h = dev_h(AdaProx, kind, b)
    r = AdaProx.OurRule(t=1.0, norm_A=float(np.linalg.norm(A, 2)))
    X, Y, its, _ = AdaProx.adaptive_primal_dual_lambda_path(X0, Y0, f=AdaProx.Zero(), h=h, A=A, lambdas=lams, rule=r, maxit=0)
    assert np.all(its == 0) and np.array_equal(Y, Y0)
    for j in range(6):
        xs, ys, its_s = AdaProx.adaptive_primal_dual(X0[:, j], Y0[:, j], f=AdaProx.Zero(), g=AdaProx.NormL1(lams[j]), h=h, A=A,
                                                     rule=r, maxit=0)
        assert its_s == 0 and np.array_equal(ys, Y0[:, j])
        assert np.max(np.abs(X[:, j] - xs)) <= 1e-12 * max(np.max(np.abs(xs)), 1.0), j


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["l1", "l2"])
def test_reruns_and_permutations_are_bit_identical(AdaProx, kind):
    m, n, L = 300, 2000, 70                          # both contractions K-split
    A, b, lams, X0, Y0 = instance(m, n, L, kind, seed=4)
    h = dev_h(AdaProx, kind, b)
    r = AdaProx.OurRule(t=1.0, norm_A=float(np.linalg.norm(A, 2)))
    g0 = np.linspace(0.5, 1.0, L) * r.gamma
    kw = dict(f=AdaProx.Zero(), h=h, A=A, rule=r, tol=1e-3, maxit=200, history=50)
    a = AdaProx.adaptive_primal_dual_lambda_path(X0, Y0, lambdas=lams, gamma0=g0, **kw)
    b_ = AdaProx.adaptive_primal_dual_lambda_path(X0, Y0, lambdas=lams, gamma0=g0, **kw)
    perm = np.random.default_rng(5).permutation(L)
    c = AdaProx.adaptive_primal_dual_lambda_path(X0[:, perm], Y0[:, perm], lambdas=lams[perm], gamma0=g0[perm], **kw)
    for u, v, w in zip(a[:3], b_[:3], c[:3]):
        assert np.array_equal(u, v)
        assert np.array_equal(u[..., perm], w)
    for k in ("norm_res", "gamma", "sigma", "gamma_hist", "res_hist", "obj_hist"):
        assert np.array_equal(a[3][k], b_[3][k], equal_nan=True), k
        assert np.array_equal(a[3][k][..., perm], c[3][k], equal_nan=True), k
    # L = 1: one column is the same column of the batch
    j = int(perm[0])
    d = AdaProx.adaptive_primal_dual_lambda_path(X0[:, j:j + 1], Y0[:, j:j + 1], lambdas=lams[j:j + 1], gamma0=g0[j:j + 1], **kw)
    for u, w in zip(a[:3], d[:3]):
        assert np.array_equal(u[..., j], w[..., 0])
    for k in ("norm_res", "gamma", "gamma_hist", "res_hist", "obj_hist"):
        assert np.array_equal(a[3][k][..., j], d[3][k][..., 0], equal_nan=True), k


# ---------------------------------------------------------------- (4) refusals
def raw_call(AdaProx, A, lams, edit=lambda p, o: None, L=None, b=None):
    """adaprox_solve_pd_lambda_path through the C ABI with the problem the Python entry point builds (LAD), after
    `edit(p, o)`"""
    dev = AdaProx.default_device()
    Am = A if isinstance(A, AdaProx.DeviceMatrix) else AdaProx.DeviceMatrix(A, dev=dev)
    m, n = Am.shape
    p = AdaProx.Zero()._problem(n)
    p.g = AdaProx.NormL1(1.0)._desc()
    h = AdaProx.Translate(AdaProx.NormL1(), -np.ones(m) if b is None else b)
    p.h = h._desc()
    p.A_mat, p.m_dual = Am.id, m
    o = Lb.Options()
    o.solver, o.rule, o.gamma, o.t, o.Theta, o.tol, o.maxit = Lb.S_ADAPTIVE_PRIMAL_DUAL, Lb.RULE_FIXED, 1e-3, 1.0, 1.2, 1e-6, 5
    o.eta, o.R, o.r = 1.0, 0.95, 0.5
    edit(p, o)
    lam = np.ascontiguousarray(lams, dtype=np.float64)
    Lc = len(lam) if L is None else L
    xo = np.empty((max(len(lam), 1), n))
    res = Lb.Result()
    dp = lambda a: a.ctypes.data_as(Lb.c_dp)
    rc = dev.lib.adaprox_solve_pd_lambda_path(dev.h, C.byref(p), C.byref(o), Lc, dp(lam), None, None, None, dp(xo), None, None,
                                              None, None, None, None, 0, C.byref(res))
    return rc, dev.lib.adaprox_last_error(dev.h).decode() if rc else ""


@pytest.mark.gpu
def test_refusals(AdaProx):
    m, n = 60, 8
    A, b, lams, _, _ = instance(m, n, 3, "l1", seed=6)
    assert raw_call(AdaProx, A, lams)[0] == 0
    UNSUP, INVAL = -3, -1
    import scipy.sparse as sps
    # f other than Zero
    fl = AdaProx.LinearLeastSquares(A.copy(), b)
    assert raw_call(AdaProx, A, lams, lambda p, o: (setattr(p, "f_kind", Lb.F_LEAST_SQUARES), setattr(p, "f_mat", fl.mat.id),
                                                    setattr(p, "f_vec", fl.vec.id)))[0] == UNSUP
    # A CSR or row-sharded
    assert raw_call(AdaProx, sps.csr_matrix(A), lams)[0] == UNSUP
    As = AdaProx.DeviceMatrix(np.ascontiguousarray(A[: m // 2]))
    As.set_shard(m, 0)
    rc, msg = raw_call(AdaProx, As, lams, b=-np.ones(m // 2))
    assert rc == UNSUP and "ranks" in msg, msg
    # g other than a plain NormL1
    assert raw_call(AdaProx, A, lams, lambda p, o: setattr(p, "g", AdaProx.NormL2(1.0)._desc()))[0] == UNSUP
    assert raw_call(AdaProx, A, lams, lambda p, o: setattr(p, "g", AdaProx.IndBox(0.0, 1.0)._desc()))[0] == UNSUP
    assert raw_call(AdaProx, A, lams, lambda p, o: setattr(p.g, "conjugate", 1))[0] == UNSUP
    gt = AdaProx.Translate(AdaProx.NormL1(), np.ones(n))
    assert raw_call(AdaProx, A, lams, lambda p, o: setattr(p, "g", gt._desc()))[0] == UNSUP
    # h other than an unconjugated NormL1 / NormL2
    assert raw_call(AdaProx, A, lams, lambda p, o: setattr(p, "h", AdaProx.IndZero()._desc()))[0] == UNSUP
    assert raw_call(AdaProx, A, lams, lambda p, o: setattr(p, "h", AdaProx.IndBox(-1.0, 1.0)._desc()))[0] == UNSUP
    assert raw_call(AdaProx, A, lams, lambda p, o: setattr(p.h, "conjugate", 1))[0] == UNSUP
    # another solver; AdaPDM+ in particular
    assert raw_call(AdaProx, A, lams, lambda p, o: setattr(o, "solver", Lb.S_LINESEARCH_PRIMAL_DUAL))[0] == UNSUP
    assert raw_call(AdaProx, A, lams, lambda p, o: setattr(o, "solver", Lb.S_MALITSKY_POCK))[0] == UNSUP
    # the plain forms are accepted: h without Translate, NormL2 of another weight
    assert raw_call(AdaProx, A, lams, lambda p, o: setattr(p, "h", AdaProx.NormL1(0.5)._desc()))[0] == 0
    assert raw_call(AdaProx, A, lams, lambda p, o: setattr(p, "h", AdaProx.NormL2(2.0)._desc()))[0] == 0
    # invalid lambdas, batch size, pointers
    assert raw_call(AdaProx, A, np.array([1.0, -0.5, 2.0]))[0] == INVAL
    assert raw_call(AdaProx, A, np.array([1.0, np.nan, 2.0]))[0] == INVAL
    assert raw_call(AdaProx, A, lams, L=0)[0] == INVAL
    dev = AdaProx.default_device()
    assert dev.lib.adaprox_solve_pd_lambda_path(dev.h, None, None, 3, None, None, None, None, None, None, None, None, None,
                                                None, None, 0, None) == INVAL
    # the same refusals reach Python as AdaproxError with the code
    h = dev_h(AdaProx, "l1", b)
    r = AdaProx.FixedStepsize(1e-3)
    with pytest.raises(AdaProx.AdaproxError) as e:
        AdaProx.adaptive_primal_dual_lambda_path(f=fl, h=h, A=A, lambdas=lams, rule=r)
    assert e.value.code == UNSUP
    with pytest.raises(AdaProx.AdaproxError) as e:
        AdaProx.adaptive_primal_dual_lambda_path(f=AdaProx.Zero(), h=AdaProx.IndZero(), A=A, lambdas=lams, rule=r)
    assert e.value.code == UNSUP
    with pytest.raises(AdaProx.AdaproxError) as e:
        AdaProx.adaptive_primal_dual_lambda_path(f=AdaProx.Zero(), h=h, A=A, lambdas=[1.0, -1.0], rule=r)
    assert e.value.code == INVAL
    # shapes checked in Python
    for kw in (dict(X0=np.zeros((n, 2))), dict(X0=np.zeros((n + 1, 3))), dict(Y0=np.zeros((m, 2))), dict(Y0=np.zeros(m)),
               dict(gamma0=np.ones(4)), dict(lambdas=np.ones((3, 1))), dict(lambdas=np.zeros(0))):
        args = dict(f=AdaProx.Zero(), h=h, A=A, lambdas=lams, rule=r)
        args.update(kw)
        with pytest.raises(ValueError):
            AdaProx.adaptive_primal_dual_lambda_path(**args)


# ---------------------------------------------------------------- (5) the C3 shape
@pytest.mark.gpu
def test_c3_shape_sampled_columns_inside_the_oracle_envelope(AdaProx):
    X, b = AdaProx.synth.dense_regression(50000, 2000)
    A = np.ascontiguousarray(np.hstack([X, np.ones((X.shape[0], 1))]))
    L, K = 64, 30
    lam_max = float(np.max(np.abs(A.T @ np.sign(b))))
    lams = np.geomspace(1e-3, 1.0, L) * lam_max
    nA = float(np.linalg.norm(A, 2))
    r, mk = AdaProx.OurRule(t=1.0, norm_A=nA), (lambda M: M.OurRule(t=1.0, norm_A=nA))
    Xd, Yd, its, _ = AdaProx.adaptive_primal_dual_lambda_path(f=AdaProx.Zero(), h=dev_h(AdaProx, "l1", b), A=A, lambdas=lams,
                                                              rule=r, tol=0.0, maxit=K)
    assert np.all(its == K)
    for j in np.linspace(0, L - 1, 8).astype(int):
        runs = oracle_runs(A, b, lams[j], "l1", mk, K, nperm=2, seed=int(j))
        for k, got in ((0, Xd[:, j]), (1, Yd[:, j])):
            ok, ratio = inside_envelope(got, runs, k)
            assert ok, (int(j), "xy"[k], ratio)
