"""The batched C path of the dual SVM (adaptive_primal_dual_path, include/adaprox.h: adaprox_solve_box_path).

Column j is AdaPDM / Condat-Vu on f(x) + IndBox(0, C_j)(x) + IndZero(y'x), f = Quadratic(Q, -1) with Q = Z Z' or its Gram
form QuadraticGram(Z, -1).  The checks:
  - one and two primal steps of every column against the extended-precision reference (xprec_reference.PD: pd_fixed,
    pd_ourrule) under its a-priori rounding bounds, at shapes that reach both tile widths, K-split 1 and > 1 of every
    contraction of both f forms (the U = Z'X slab sum included), N not a multiple of 16 and a ragged last column tile;
  - per-C parity with the single-C device solve and a spot check against the CPU oracle;
  - frozen columns and their history, maxit = 0, bitwise determinism under reruns and permutations of the C values;
  - every refusal of the entry point.
"""
import ctypes as C

import numpy as np
import pytest

from adaprox_b200 import _lib as Lb
from oracle import adaprox_oracle as O
from test_gpu_lambda_path_reference import path_ksplit
from xprec_reference import LinMap, PD, Prox, Smooth, pd_fixed, pd_ourrule, within


# ---------------------------------------------------------------- shapes and the contractions they reach
# (f form, N, d, L).  d is the width of Z; dense Q is Z Z'.
SHAPES = [("quadratic", 200, 24, 40), ("quadratic", 301, 24, 100), ("gram", 301, 40, 40), ("gram", 250, 300, 100)]


def branches(shapes, sm):
    """-> names of the contraction branches reached: G = Q X (dense), U = Z'X and G = Z U (Gram) with K-split 1 or > 1"""
    hit = set()
    for form, N, d, L in shapes:
        hit.add("tile:narrow" if L <= 64 else "tile:wide")
        if L % (32 if L <= 64 else 128):
            hit.add("ragged:L")
        if N % 16:
            hit.add("ragged:N")
        if form == "quadratic":
            hit.add("Q:" + ("1" if path_ksplit(N, N, L, sm) == 1 else ">1"))
        else:
            hit.add("U:" + ("1" if path_ksplit(d, N, L, sm) == 1 else ">1"))
            hit.add("ZU:" + ("1" if path_ksplit(N, d, L, sm) == 1 else ">1"))
    return hit


REQUIRED = {"tile:narrow", "tile:wide", "ragged:L", "ragged:N", "Q:1", "Q:>1", "U:1", "U:>1", "ZU:1", "ZU:>1"}


def test_shapes_reach_every_contraction_branch_at_148_sms():
    assert REQUIRED <= branches(SHAPES, 148), REQUIRED - branches(SHAPES, 148)


# ---------------------------------------------------------------- instances
def instance(N, d, L, seed=0):
    """Z = D_y X (N x d), labels y, q = -1, C values spread over two decades, X0 in and on the boxes, small Y0"""
    rng = np.random.default_rng([N, d, L, seed])
    X = rng.standard_normal((N, d)) / np.sqrt(d)
    y = np.where(rng.random(N) < 0.5, -1.0, 1.0)
    Z = y[:, None] * X
    q = -np.ones(N)
    C_ = np.geomspace(0.02, 2.0, L)
    X0 = rng.random((N, L)) * C_
    X0[rng.random(X0.shape) < 0.2] = 0.0
    Y0 = 0.1 * rng.standard_normal(L)
    return Z, y, q, C_, X0, Y0


def dev_f(AdaProx, form, Z, q):
    return AdaProx.Quadratic(Z @ Z.T, q) if form == "quadratic" else AdaProx.QuadraticGram(Z, q)


def ref_smooth(form, Z, q):
    return Smooth("quadratic", Z @ Z.T, q) if form == "quadratic" else Smooth("gram", Z, q)


def steps(Lf, nA, L):
    """FixedStepsize gamma_j in [0.5, 0.9] / (L_f + t |A|) with t = 0.7, OurRule gamma_j below 1 / (2 Theta t |A|)"""
    t = 0.7
    return t, np.linspace(0.5, 0.9, L) / (Lf + t * nA), np.linspace(0.3, 0.6, L) / (2 * 1.2 * t * nA)


# ---------------------------------------------------------------- (1) one and two steps against the reference
@pytest.mark.gpu
def test_shapes_reach_every_contraction_branch_on_this_device(AdaProx):
    sm = AdaProx.default_device().info()["sm_count"]
    assert REQUIRED <= branches(SHAPES, sm), REQUIRED - branches(SHAPES, sm)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=[f"{s[0]}-N{s[1]}-d{s[2]}-L{s[3]}" for s in SHAPES])
def test_one_and_two_steps_match_extended_precision(AdaProx, shape):
    form, N, d, L = shape
    Z, y, q, C_, X0, Y0 = instance(N, d, L)
    f = dev_f(AdaProx, form, Z, q)
    A = y[None, :]
    nA = float(np.linalg.norm(y))
    Lf = float(np.linalg.norm(Z, 2) ** 2)
    t, gf, go = steps(Lf, nA, L)
    fixed = AdaProx.FixedStepsize(gf[0], t)
    our = AdaProx.OurRule(gamma=go[0], t=t, norm_A=nA)
    kw = dict(f=f, A=A, upper=C_, tol=0.0)
    x1, y0, it0, _ = AdaProx.adaptive_primal_dual_path(X0, Y0, rule=fixed, gamma0=gf, maxit=0, **kw)
    x2, y1, it1, i1 = AdaProx.adaptive_primal_dual_path(X0, Y0, rule=fixed, gamma0=gf, maxit=1, history=1, **kw)
    xo, yo, ito, io = AdaProx.adaptive_primal_dual_path(X0, Y0, rule=our, gamma0=go, maxit=1, history=1, **kw)
    assert AdaProx.last_solve_info()["matrix_passes"] == (1 if form == "quadratic" else 2)
    assert np.all(it0 == 0) and np.all(it1 == 1) and np.all(ito == 1)
    assert np.array_equal(y0, Y0), "maxit = 0: Y0 comes back"
    sm = ref_smooth(form, Z, q)
    Amap, h = LinMap(A), Prox("indzero")
    for j in range(L):
        P = PD(sm, Prox("box", lo=0.0, hi=C_[j]), h, Amap)
        R = pd_fixed(P, X0[:, j], Y0[j:j + 1], gf[j], t)
        ok, ratio = within(x1[:, j], R["X1"], R["B1"])
        assert ok, ("maxit = 0: x_1", j, ratio)
        ok, ratio = within(x2[:, j], R["X2"], R["B2"])
        assert ok, ("maxit = 1: x_2", j, ratio)
        D = R["D"]
        ok, ratio = within(y1[j], D["Y1"], D["ey1"] + D["sy1"])
        assert ok, ("maxit = 1: y_1", j, ratio)
        assert i1["gamma"][j] == gf[j] and i1["sigma"][j] == R["sigma"], "FixedStepsize: gamma and sigma exact"
        assert i1["gamma_hist"][0, j] == gf[j]
        ok, ratio = within(i1["res_hist"][0, j], R["res1"], R["dres1"])
        assert ok, ("norm_res", j, ratio)
        if np.isfinite(R["obj1"]):
            ok, ratio = within(i1["obj_hist"][0, j], R["obj1"], R["dobj1"])
            assert ok, ("objective", j, ratio)
        else:
            assert i1["obj_hist"][0, j] == R["obj1"], ("objective", j)
        Ro = pd_ourrule(P, X0[:, j], Y0[j:j + 1], go[j], t, nA)
        ok, ratio = within(io["gamma_hist"][0, j], Ro["gamma1"], Ro["dgamma1"])
        assert ok, ("OurRule gamma_1", j, ratio)
        ok, ratio = within(xo[:, j], Ro["X2"], Ro["B2"])
        assert ok, ("OurRule x_2", j, ratio)
        D = Ro["D"]
        ok, ratio = within(yo[j], D["Y1"], D["ey1"] + D["sy1"])
        assert ok, ("OurRule y_1", j, ratio)


# ---------------------------------------------------------------- (2) per-C parity with the single solve
PAR_N, PAR_D, PAR_L = 300, 400, 6
RULES = ["our", "condat_vu", "mm"]
# per rule, C values from every coordinate at a bound (a few iterations) to an inactive upper bound (thousands)
PAR_C = dict(our=[0.05, 0.3, 1.0, 3.0, 10.0, 30.0], condat_vu=[0.01, 0.1, 1.0, 3.0, 10.0, 30.0],
             mm=[0.3, 1.0, 3.0, 10.0, 30.0, 100.0])


def parity_problem(AdaProx, form, rule):
    Z, y, q, _, _, _ = instance(PAR_N, PAR_D, PAR_L, seed=1)
    C_ = np.array(PAR_C[rule])
    f = dev_f(AdaProx, form, Z, q)
    nA = float(np.linalg.norm(y))
    Lf = float(np.linalg.norm(Z, 2) ** 2)
    if rule == "our":
        r = AdaProx.OurRule(t=1.0, norm_A=nA)
    elif rule == "condat_vu":
        gam, sig = 1.0 / (Lf / 2 + nA / (100 * nA / Lf)), 0.99 / (nA * (100 * nA / Lf))   # src/AdaProx.jl:398-412
        r = AdaProx.FixedStepsize(gam, np.sqrt(sig / gam))
    else:
        r = AdaProx.MalitskyMishchenkoRule(0.5 / (Lf + nA), 0.1)
    return Z, y, q, C_, f, r


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["quadratic", "gram"])
@pytest.mark.parametrize("rule", RULES)
def test_every_column_matches_the_single_solve(AdaProx, form, rule):
    Z, y, q, C_, f, r = parity_problem(AdaProx, form, rule)
    A = y[None, :]
    tol, maxit = 1e-7, 50_000
    H = 20
    X, Y, its, info = AdaProx.adaptive_primal_dual_path(f=f, A=A, upper=C_, rule=r, tol=tol, maxit=maxit, history=H)
    assert np.all(info["norm_res"] <= tol) and np.all(its < maxit)
    assert its.max() >= 2 * its.min(), ("the C values should stop at very different iterations", its)
    for j in range(PAR_L):
        log = []
        xs, ys, its_s = AdaProx.adaptive_primal_dual(np.zeros(PAR_N), np.zeros(1), f=f, g=AdaProx.IndBox(0.0, C_[j]),
                                                     h=AdaProx.IndZero(), A=A, rule=r, tol=tol, maxit=maxit, log=log)
        gs = AdaProx.last_solve_info()["final_gamma"]
        assert abs(int(its[j]) - its_s) <= max(3, 0.05 * its_s), (j, its[j], its_s)
        assert np.linalg.norm(X[:, j] - xs) <= 1e-6 * np.linalg.norm(xs), (j, np.linalg.norm(X[:, j] - xs) / np.linalg.norm(xs))
        assert abs(Y[j] - ys[0]) <= 1e-6 * max(abs(ys[0]), 1.0), (j, Y[j], ys[0])
        k = min(H, int(its[j]), its_s)
        gam_s = np.array([rec["gamma"] for rec in log[:k]])
        assert np.allclose(info["gamma_hist"][:k, j], gam_s, rtol=1e-9, atol=0), (j, info["gamma_hist"][:k, j], gam_s)
        if rule != "mm":
            # Malitsky-Mishchenko's gamma near the stop is min(.., 1 / (2 |dg| / |dx|)) of two differences at rounding
            # level: it depends on the summation order of the gradient (DMMA vs GEMV), while x and y do not
            assert abs(info["gamma"][j] - gs) <= 1e-6 * gs, (j, info["gamma"][j], gs)


@pytest.mark.gpu
def test_a_column_matches_the_cpu_oracle(AdaProx):
    Z, y, q, C_, f, r = parity_problem(AdaProx, "gram", "our")
    A = y[None, :]
    X, Y, its, _ = AdaProx.adaptive_primal_dual_path(f=f, A=A, upper=C_, rule=r, tol=1e-7, maxit=50_000)
    for j in (1, 4):
        xo, yo, ito = O.adaptive_primal_dual(np.zeros(PAR_N), np.zeros(1), f=O.Quadratic(Z @ Z.T, q), g=O.IndBox(0.0, C_[j]),
                                             h=O.IndZero(), A=A, rule=O.OurRule(t=1.0, norm_A=float(np.linalg.norm(y))),
                                             tol=1e-7, maxit=50_000)
        assert abs(int(its[j]) - ito) <= max(3, 0.05 * ito), (j, its[j], ito)
        assert np.linalg.norm(X[:, j] - xo) <= 1e-6 * np.linalg.norm(xo)
        assert abs(Y[j] - yo[0]) <= 1e-6 * max(abs(yo[0]), 1.0)


# ---------------------------------------------------------------- (3) frozen columns and history, (4) maxit = 0
@pytest.mark.gpu
@pytest.mark.parametrize("form", ["quadratic", "gram"])
def test_columns_freeze_at_their_stop_and_the_history_ends_there(AdaProx, form):
    Z, y, q, C_, f, r = parity_problem(AdaProx, form, "our")
    A = y[None, :]
    tol, maxit = 1e-6, 20_000
    X, Y, its, info = AdaProx.adaptive_primal_dual_path(f=f, A=A, upper=C_, rule=r, tol=tol, maxit=maxit, history=maxit)
    res = info["res_hist"]
    for j in range(PAR_L):
        k = int(its[j])
        first = int(np.argmax(res[:, j] <= tol)) + 1
        assert res[first - 1, j] <= tol and first == k, (j, first, k)
        assert np.all(np.isfinite(res[:k, j])) and np.all(np.isnan(res[k:, j]))
        assert np.all(np.isnan(info["gamma_hist"][k:, j])) and np.all(np.isnan(info["obj_hist"][k:, j]))
        assert info["gamma_hist"][k - 1, j] == info["gamma"][j] and res[k - 1, j] == info["norm_res"][j]
    # the result is the iterate at the stop: maxit = k - 1 returns x_k, which is what a column stopping at k returns
    j = int(np.argmin(its))
    Xk, _, itk, _ = AdaProx.adaptive_primal_dual_path(f=f, A=A, upper=C_, rule=r, tol=0.0, maxit=int(its[j]) - 1)
    assert np.all(itk == its[j] - 1)
    assert np.array_equal(Xk[:, j], X[:, j])


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["quadratic", "gram"])
def test_maxit_zero_matches_the_single_solve(AdaProx, form):
    Z, y, q, C_, X0, Y0 = instance(PAR_N, PAR_D, PAR_L, seed=2)
    f = dev_f(AdaProx, form, Z, q)
    A = y[None, :]
    r = AdaProx.OurRule(t=1.0, norm_A=float(np.linalg.norm(y)))
    X, Y, its, _ = AdaProx.adaptive_primal_dual_path(X0, Y0, f=f, A=A, upper=C_, rule=r, maxit=0)
    assert np.all(its == 0) and np.array_equal(Y, Y0)
    for j in range(PAR_L):
        xs, ys, its_s = AdaProx.adaptive_primal_dual(X0[:, j], Y0[j:j + 1], f=f, g=AdaProx.IndBox(0.0, C_[j]), h=AdaProx.IndZero(),
                                                     A=A, rule=r, maxit=0)
        assert its_s == 0 and ys[0] == Y0[j]
        assert np.max(np.abs(X[:, j] - xs)) <= 1e-12 * max(np.max(np.abs(xs)), 1.0), j


# ---------------------------------------------------------------- (5) determinism
@pytest.mark.gpu
@pytest.mark.parametrize("form", ["quadratic", "gram"])
def test_reruns_and_permutations_are_bit_identical(AdaProx, form):
    N, d, L = 301, 40, 70
    Z, y, q, C_, X0, Y0 = instance(N, d, L, seed=3)
    f = dev_f(AdaProx, form, Z, q)
    A = y[None, :]
    r = AdaProx.OurRule(t=1.0, norm_A=float(np.linalg.norm(y)))
    g0 = np.linspace(0.5, 1.0, L) * r.gamma
    kw = dict(f=f, A=A, rule=r, tol=1e-6, maxit=300, history=50)
    a = AdaProx.adaptive_primal_dual_path(X0, Y0, upper=C_, gamma0=g0, **kw)
    b = AdaProx.adaptive_primal_dual_path(X0, Y0, upper=C_, gamma0=g0, **kw)
    perm = np.random.default_rng(5).permutation(L)
    c = AdaProx.adaptive_primal_dual_path(X0[:, perm], Y0[perm], upper=C_[perm], gamma0=g0[perm], **kw)
    for u, v, w in zip(a[:3], b[:3], c[:3]):
        assert np.array_equal(u, v)
        assert np.array_equal(u[..., perm], w)
    for k in ("norm_res", "gamma", "sigma", "f_x", "gamma_hist", "res_hist", "obj_hist"):
        assert np.array_equal(a[3][k], b[3][k], equal_nan=True), k
        assert np.array_equal(a[3][k][..., perm], c[3][k], equal_nan=True), k


# ---------------------------------------------------------------- (6) refusals
def raw_call(AdaProx, f, A, upper, edit=lambda p, o: None, L=None):
    """adaprox_solve_box_path through the C ABI with the problem the Python entry point builds, after `edit(p, o)`"""
    dev = f._dev()
    Am = AdaProx.DeviceMatrix(A, dev=dev)
    p = f._problem(Am.shape[1])
    p.g = AdaProx.IndBox(0.0, 0.0)._desc()
    p.h = AdaProx.IndZero()._desc()
    p.A_mat, p.m_dual = Am.id, Am.shape[0]
    o = Lb.Options()
    o.solver, o.rule, o.gamma, o.t, o.Theta, o.tol, o.maxit = Lb.S_ADAPTIVE_PRIMAL_DUAL, Lb.RULE_FIXED, 1e-3, 1.0, 1.2, 1e-6, 5
    edit(p, o)
    up = np.ascontiguousarray(upper, dtype=np.float64)
    n = Am.shape[1]
    Lc = len(up) if L is None else L
    xo = np.empty((max(len(up), 1), n))
    res = Lb.Result()
    dp = lambda a: a.ctypes.data_as(Lb.c_dp)
    return dev.lib.adaprox_solve_box_path(dev.h, C.byref(p), C.byref(o), Lc, dp(up), None, None, None, dp(xo), None, None, None,
                                          None, None, None, None, 0, C.byref(res))


@pytest.mark.gpu
def test_refusals(AdaProx):
    N, d = 40, 6
    Z, y, q, C_, _, _ = instance(N, d, 3, seed=4)
    A = y[None, :]
    fq = AdaProx.Quadratic(Z @ Z.T, q)
    assert raw_call(AdaProx, fq, A, C_) == 0
    UNSUP, INVAL = -3, -1
    # f other than a dense Quadratic / QuadraticGram
    assert raw_call(AdaProx, AdaProx.LinearLeastSquares(Z.T.copy(), np.ones(d)), A, C_) == UNSUP
    import scipy.sparse as sps
    assert raw_call(AdaProx, AdaProx.Quadratic(sps.csr_matrix(Z @ Z.T), q), A, C_) == UNSUP
    # A not a dense 1 x n matrix
    assert raw_call(AdaProx, fq, np.vstack([y, y]), C_) == UNSUP
    assert raw_call(AdaProx, fq, sps.csr_matrix(A), C_) == UNSUP
    # g not a scalar IndBox, h not IndZero, another solver
    assert raw_call(AdaProx, fq, A, C_, lambda p, o: setattr(p, "g", AdaProx.NormL1(1.0)._desc())) == UNSUP
    assert raw_call(AdaProx, fq, A, C_, lambda p, o: setattr(p, "g", AdaProx.IndBox(np.zeros(N), np.ones(N))._desc())) == UNSUP
    assert raw_call(AdaProx, fq, A, C_, lambda p, o: setattr(p.g, "conjugate", 1)) == UNSUP
    assert raw_call(AdaProx, fq, A, C_, lambda p, o: setattr(p, "h", AdaProx.Zero()._desc())) == UNSUP
    assert raw_call(AdaProx, fq, A, C_, lambda p, o: setattr(p.h, "conjugate", 1)) == UNSUP
    assert raw_call(AdaProx, fq, A, C_, lambda p, o: setattr(o, "solver", 2)) == UNSUP
    # a row shard of Q
    Qs = AdaProx.DeviceMatrix(np.ascontiguousarray((Z @ Z.T)[: N // 2]))
    Qs.set_shard(N, 0)
    fs = AdaProx.Quadratic(Qs, q)
    assert raw_call(AdaProx, fs, A, C_) == UNSUP
    assert "ranks" in AdaProx.default_device().lib.adaprox_last_error(AdaProx.default_device().h).decode()
    # invalid bounds and batch size
    assert raw_call(AdaProx, fq, A, np.array([1.0, -0.5, 2.0])) == INVAL
    assert raw_call(AdaProx, fq, A, np.array([1.0, np.nan, 2.0])) == INVAL
    assert raw_call(AdaProx, fq, A, C_, lambda p, o: setattr(p.g, "lo", 1.5)) == INVAL
    assert raw_call(AdaProx, fq, A, C_, L=0) == INVAL
    # the same refusals reach Python as AdaproxError with the code
    with pytest.raises(AdaProx.AdaproxError) as e:
        AdaProx.adaptive_primal_dual_path(f=AdaProx.LinearLeastSquares(Z.T.copy(), np.ones(d)), A=A, upper=C_, rule=AdaProx.FixedStepsize(1e-3))
    assert e.value.code == UNSUP
    with pytest.raises(AdaProx.AdaproxError) as e:
        AdaProx.adaptive_primal_dual_path(f=fq, A=A, upper=[1.0, -1.0], rule=AdaProx.FixedStepsize(1e-3))
    assert e.value.code == INVAL
    # shapes checked in Python
    r = AdaProx.FixedStepsize(1e-3)
    for kw in (dict(X0=np.zeros((N, 2))), dict(X0=np.zeros((N + 1, 3))), dict(Y0=np.zeros(2)), dict(Y0=np.zeros((3, 1))),
               dict(gamma0=np.ones(4)), dict(upper=np.ones((3, 1))), dict(upper=np.zeros(0))):
        args = dict(f=fq, A=A, upper=C_, rule=r)
        args.update(kw)
        with pytest.raises(ValueError):
            AdaProx.adaptive_primal_dual_path(**args)
