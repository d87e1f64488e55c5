"""The batched lambda path (adaptive_proxgrad_path) step by step against an extended-precision reference.

One and two AdaPGM steps of the whole batch are restated in np.longdouble (64-bit mantissa) for least squares over a dense
matrix, least squares over a CSR matrix and the logistic loss over a CSR matrix (intercept last, penalised).  With
FixedStepsize and per-column gamma_j <= 1 / L_f, maxit = 0 returns x_1 = S_{gamma lambda}(x_0 - gamma grad f(x_0)) and
maxit = 1 returns x_2.  The device's X is compared against a-priori rounding bounds, not a fixed rtol (u = 2^-53; M the
matrix, m its rows, K1 its columns, s = 1 for least squares and 1 / N for the logistic loss):

    least squares   |dP| <= (K1 + 2) u (|M| |w| + |b|)                       P = M w - b
    logistic        |dP| <= 1/4 (K1 + 2) u (|M| |w_f| + |w_0|) + 4 u          P = 1 / (1 + exp(-M w_f - w_0)) - y
                    (sigma' <= 1/4 carries the logit error; exp, the division and "- y" add at most 4 u)
    gradient        |dG| <= s (|M|' |dP| + (m + 2) u |M|' |P|) + u |G|        (intercept: the column sums of |dP| and |P|)
    step            |dx_1| <= 2 [gamma |dG| + 2 u (|w| + gamma |G|) + u gamma lambda]

For least squares this is 2 [gamma (m + K1 + 4) u |M|' (|M| |w| + |b|) + 2 u (|w| + gamma |G|)] up to the threshold term.
The soft threshold is 1-Lipschitz, so the bound carries through the prox; the factor 2 also covers the reference's own
rounding (2^-64).  For two steps the bound is per column in the 2-norm: with gamma <= 1 / L_f both I - gamma grad f and the
prox are non-expansive, so |x_2 - x_2^ref| <= |dx_1| + |dx_2(x_1)|.  f(x) and the records get the same treatment (the
input error of x_1 enters the residuals linearly).  The CPU self-check below shows that these bounds reject a dropped K
slab of M' P and two swapped columns of X0, and accept a plain float64 evaluation in another summation order.

The dense shapes are chosen by a restatement of the K-split heuristic (path.inl: path_ksplit) and of the slab arithmetic
of k_path_gemm, the CSR batch widths by the column-tile choice of csr_path_launch_sweep; both tests assert which kernel
branches the set reaches on the device at hand.
"""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import adaprox_oracle as O
from oracle import drift
from xprec_reference import Term, reference, within, within_cols


# ---------------------------------------------------------------- restatement of the kernel selection
def path_ksplit(mdim, kdim, L, sm_count):
    """path.inl: path_ksplit (tile 128 x BN; slabs of at least 8 x 16 of K; only a > 8 % shorter makespan splits)."""
    bn = 32 if L <= 64 else 128
    ctas = -(-mdim // 128) * -(-L // bn)
    best, best_span = 1, float(-(-ctas // sm_count))
    for ks in range(2, 9):
        if kdim // ks < 128:
            break
        span = -(-(ctas * ks) // sm_count) / ks
        if span < 0.92 * best_span:
            best, best_span = ks, span
    return best


def k_slabs(kdim, ks, L):
    """k_path_gemm: [kbeg, kend) of each blockIdx.z; slabs are whole BK tiles (32 on the wide tile, 16 on the narrow one)."""
    if ks <= 1:
        return [(0, kdim)]
    bk = 16 if L <= 64 else 32
    per = -(-(-(-kdim // bk)) // ks)
    out = []
    for z in range(ks):
        kbeg = z * per * bk
        kend = min(kbeg + per * bk, kdim)
        out.append((min(kbeg, kend), kend))
    return out


def dense_branches(shapes, sm_count):
    """Names of the dense-path branches that (m, n, L) in `shapes` reach on a device with sm_count SMs."""
    hit = set()
    for m, n, L in shapes:
        narrow = L <= 64
        bn, bk = (32, 16) if narrow else (128, 32)
        hit.add("tile:narrow" if narrow else "tile:wide")
        kg, kr = path_ksplit(n, m, L, sm_count), path_ksplit(m, n, L, sm_count)
        hit.add("G:1" if kg == 1 else ("G:8" if kg == 8 else "G:mid"))
        hit.add("R:1" if kr == 1 else "R:>1")
        if kg > 1 and any(b == e for b, e in k_slabs(m, kg, L)):
            hit.add("G:empty_slab")
        if m % 128 or n % 128:
            hit.add("ragged:M")
        if L % bn:
            hit.add("ragged:N")
        if m % bk or n % bk:
            hit.add("ragged:K")
        if -(-L // bn) >= 3:
            hit.add("N_tiles>=3")
    return hit


DENSE_REQUIRED = {"tile:narrow", "tile:wide", "G:1", "G:mid", "G:8", "G:empty_slab", "R:1", "R:>1", "ragged:M", "ragged:N",
                  "ragged:K", "N_tiles>=3"}


def csr_nq(L):
    """path_csr.inl: csr_path_launch_sweep -> (NQ, column tiles)."""
    chunks = -(-L // 32)
    nq = 8 if chunks >= 8 else (4 if chunks >= 4 else (2 if chunks >= 2 else 1))
    return nq, -(-chunks // nq)


DENSE_SHAPES = [(1, 40, 1), (17, 33, 3), (129, 131, 2), (300, 200, 64), (300, 200, 65), (400, 1000, 7), (1040, 300, 40),
                (1040, 300, 100), (2100, 90, 1), (300, 2600, 257), (1100, 1100, 300)]
CSR_WIDTHS = [1, 32, 33, 64, 65, 96, 128, 129, 224, 225, 256, 257, 300, 520]


# ---------------------------------------------------------------- instances
def dense_instance(m, n, L, seed=0):
    rng = np.random.default_rng(seed + 7919 * m + n)
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    b = rng.standard_normal(m)
    term = Term("lsq", A, b)
    return term, _batch(term, L, rng)


def _batch(term, L, rng):
    """per-column gamma_j in [0.5, 0.999] / L_f, lambda_j spanning 0 .. lambda_max, a non-zero X0"""
    g = 1.0 / term.lipschitz()
    gam = g * np.linspace(0.5, 0.999, L)
    X0 = 0.1 * rng.standard_normal((term.n, L))
    X0[rng.random(X0.shape) < 0.2] = 0.0
    _, _, G0 = term.eval(np.zeros((term.n, 1)))
    lam = float(np.max(np.abs(G0))) * np.linspace(0.0, 1.0, L)
    return X0, gam, lam, g * 0.7123                                      # the rule's own gamma differs from every gamma0[j]


ROW_LENGTHS = [0, 1, 3, 4, 5, 31, 32, 33, 64, 65, 230]


def csr_matrix(m, nf, lengths, seed):
    """CSR with the given row lengths (cycled); feature 1 has no non-zeros, feature 0 sits in every row of >= 3 non-zeros."""
    rng = np.random.default_rng(seed)
    pool = np.array([c for c in range(nf) if c != 1])
    rows, cols = [], []
    for i in range(m):
        k = min(lengths[i % len(lengths)], pool.size - 1)
        c = rng.choice(pool[1:], size=k, replace=False) if k else np.zeros(0, dtype=int)
        if k >= 3:
            c[0] = 0
        rows += [i] * k
        cols += list(c)
    vals = rng.uniform(-1.0, 1.0, len(rows))
    X = sp.csr_matrix((vals, (rows, cols)), shape=(m, nf))
    X.sort_indices()
    return X


def csr_instance(kind, size, L, seed=0):
    m, nf, lengths = (203, 301, ROW_LENGTHS) if size == "mid" else (13, 21, [0, 1, 3, 4, 5, 18, 19])
    X = csr_matrix(m, nf, lengths, seed)
    rng = np.random.default_rng(seed + 17)
    v = rng.standard_normal(m) if kind == "lsq" else (rng.random(m) < 0.4).astype(np.float64)
    term = Term(kind, X.toarray(), v)
    return X, term, _batch(term, L, rng)


# ---------------------------------------------------------------- CPU self-checks of the comparator and of the coverage
def test_bound_rejects_a_dropped_slab_and_swapped_columns():
    """The bounds are tight enough: a reference with one K slab of M' P left out, or with two neighbouring columns of X0
    swapped, fails them; a float64 evaluation (another summation order) passes."""
    for term, (X0, gam, lam, _) in (dense_instance(400, 1000, 7), csr_instance("lsq", "mid", 9)[1:], csr_instance("logistic", "mid", 9)[1:]):
        R = reference(term, X0, gam, lam)
        # plain float64, BLAS summation order
        x1, _, _, f0, _ = term.step(X0, gam, lam)
        assert within(x1, R["X1"], R["B1"])[0]
        assert within(f0, R["f0"], R["df0"])[0]
        x2 = term.step(x1, gam, lam)[0]
        assert within_cols(x2, R["X2"], R["B2col"])[0]
        # one K slab of G = M' P missing (the slabs of a 3-way split of the m rows)
        _, P, G = term.eval(X0)
        for kbeg, kend in k_slabs(term.m, 3, X0.shape[1]):
            Gd = G.copy()
            Gd[:term.nf] -= term.M[kbeg:kend].T @ P[kbeg:kend] * term.s
            ok, ratio = within(term.step(X0, gam, lam, G=Gd)[0], R["X1"], R["B1"])
            assert not ok and ratio > 1e6, (kbeg, kend, ratio)
        # columns 2 and 3 of X0 swapped
        Xs = X0.copy()
        Xs[:, [2, 3]] = Xs[:, [3, 2]]
        ok, ratio = within(term.step(Xs, gam, lam)[0], R["X1"], R["B1"])
        assert not ok and ratio > 1e6, ratio
        ok, ratio = within_cols(term.step(term.step(Xs, gam, lam)[0], gam, lam)[0], R["X2"], R["B2col"])
        assert not ok and ratio > 1e6, ratio
        # the bound is not vacuous: far below the size of the entries it guards
        assert np.max(R["B1"]) < 1e-9 * max(np.max(np.abs(R["X1"])), 1.0)


def test_dense_shapes_cover_the_kernel_branches_at_148_sms():
    assert DENSE_REQUIRED <= dense_branches(DENSE_SHAPES, 148), DENSE_REQUIRED - dense_branches(DENSE_SHAPES, 148)
    assert path_ksplit(300, 1040, 100, 148) == 8 and k_slabs(1040, 8, 100)[7] == (1040, 1040)


def test_csr_widths_cover_every_column_tile():
    nq = {csr_nq(L) for L in CSR_WIDTHS}
    assert {q for q, _ in nq} == {1, 2, 4, 8}
    assert max(t for q, t in nq if q == 8) == 3 and any(q == 8 and t == 2 for q, t in nq)
    X = csr_matrix(203, 301, ROW_LENGTHS, 0)
    lens = np.diff(X.indptr)
    assert set(ROW_LENGTHS) <= set(lens.tolist()) and lens.max() >= 200
    cnt = np.bincount(X.indices, minlength=301)
    assert cnt[1] == 0 and cnt[0] > 64
    assert 203 % 32 and 301 % 32 and 13 < 32 and 21 < 32


# ---------------------------------------------------------------- (a) device against the reference
def _check_against_reference(AdaProx, Fd, term, X0, gam, lam, rule_gamma):
    R = reference(term, X0, gam, lam)
    rule = AdaProx.FixedStepsize(gamma=rule_gamma)
    Xd, its, info = AdaProx.adaptive_proxgrad_path(X0, f=Fd, lambdas=lam, rule=rule, gamma0=gam, tol=0.0, maxit=0)
    assert np.all(its == 0) and info["flags"] == 0 and np.all(np.isinf(info["norm_res"]))
    ok, ratio = within(Xd, R["X1"], R["B1"])
    assert ok, ("maxit = 0: x_1", ratio)
    assert np.array_equal(info["gamma"], gam)
    assert within(info["f_x"], R["f0"], R["df0"])[0], ("f(x_0)", within(info["f_x"], R["f0"], R["df0"])[1])
    Xd, its, info = AdaProx.adaptive_proxgrad_path(X0, f=Fd, lambdas=lam, rule=rule, gamma0=gam, tol=0.0, maxit=1, history=1)
    assert np.all(its == 1)
    ok, ratio = within_cols(Xd, R["X2"], R["B2col"])
    assert ok, ("maxit = 1: x_2", ratio)
    assert np.array_equal(info["gamma"], gam), "FixedStepsize: every column keeps its own gamma0"
    assert np.array_equal(info["gamma_hist"][0], gam)
    for key, ref, bnd in (("f_x", "f1", "df1"), ("obj_hist", "obj1", "dobj1"), ("res_hist", "res1", "dres1")):
        got = info[key][0] if key != "f_x" else info[key]
        ok, ratio = within(got, R[ref], R[bnd])
        assert ok, (key, ratio)


@pytest.mark.gpu
def test_dense_shapes_reach_the_kernel_branches(AdaProx):
    sm = AdaProx.default_device().info()["sm_count"]
    hit = dense_branches(DENSE_SHAPES, sm)
    assert DENSE_REQUIRED <= hit, (sm, DENSE_REQUIRED - hit)


@pytest.mark.gpu
@pytest.mark.parametrize("m,n,Lc", DENSE_SHAPES)
def test_dense_path_steps_match_extended_precision(AdaProx, m, n, Lc):
    term, (X0, gam, lam, rg) = dense_instance(m, n, Lc)
    _check_against_reference(AdaProx, AdaProx.LinearLeastSquares(term.M, term.v), term, X0, gam, lam, rg)


CSR_CASES = [(kind, "mid", L) for kind in ("lsq", "logistic") for L in CSR_WIDTHS] + \
            [(kind, "tiny", L) for kind in ("lsq", "logistic") for L in (1, 65, 257)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,size,Lc", CSR_CASES)
def test_csr_path_steps_match_extended_precision(AdaProx, kind, size, Lc):
    X, term, (X0, gam, lam, rg) = csr_instance(kind, size, Lc)
    Fd = AdaProx.LinearLeastSquares(X, term.v) if kind == "lsq" else AdaProx.LogisticLoss(X, term.v)
    _check_against_reference(AdaProx, Fd, term, X0, gam, lam, rg)


# ---------------------------------------------------------------- (b) stepsize rules x gamma0 x X0 on the dense path
@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["OurRule", "FixedStepsize", "MalitskyMishchenkoRule", "OurRulePlus"])
def test_dense_path_equals_single_solves_on_device(AdaProx, rule):
    """The batched columns against adaptive_proxgrad per lambda on the same device, with per-column gamma0 and a non-zero X0
    (the dense counterpart of test_csr_path_equals_single_solves_on_device, same tolerances)."""
    m, n, Lc = 200, 520, 6
    P = AdaProx.synth.planted_lasso(m, n, 5, 5)
    Lf = AdaProx.synth.spectral_norm_sq(P["A"], iters=500)
    lambdas = np.linspace(0.2, 2.0, Lc)
    gam0 = (1 / Lf) * np.linspace(0.5, 1.0, Lc)
    X0 = 0.01 * np.random.default_rng(0).standard_normal((n, Lc))
    R = getattr(AdaProx, rule)
    f = AdaProx.LinearLeastSquares(P["A"], P["b"])
    maxit = 20000                                                # this instance needs a few thousand iterations to reach tol = 1e-5
    Xd, its, info = AdaProx.adaptive_proxgrad_path(X0, f=f, lambdas=lambdas, rule=R(gamma=0.9 / Lf), gamma0=gam0, tol=1e-5, maxit=maxit)
    for j in range(Lc):
        xj, itj = AdaProx.adaptive_proxgrad(X0[:, j], f=f, g=AdaProx.NormL1(lambdas[j]), rule=R(gamma=gam0[j]), tol=1e-5, maxit=maxit)
        if rule == "FixedStepsize":                              # contractive: the two summation orders stay within rounding
            assert abs(int(its[j]) - itj) <= 1, (j, its[j], itj)
            assert np.linalg.norm(Xd[:, j] - xj) <= 1e-6 * max(np.linalg.norm(xj), 1e-9)
            assert info["gamma"][j] == gam0[j], (j, info["gamma"][j], gam0[j])
        else:                                                    # both stopped at norm_res <= 1e-5; the adaptive rules amplify rounding
            assert abs(int(its[j]) - itj) <= max(3, 0.1 * itj), (j, its[j], itj)
            assert np.linalg.norm(Xd[:, j] - xj) <= 2e-2 * max(np.linalg.norm(xj), 1e-9)
    if rule != "FixedStepsize":
        assert (its < maxit).sum() >= Lc // 2


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["MalitskyMishchenkoRule", "OurRulePlus"])
def test_dense_path_adaptive_rules_match_the_oracle(AdaProx, rule):
    """The other two adaptive rules against the oracle per lambda, inside the drift envelope (as the OurRule test does)."""
    m, n, Lc = 130, 300, 33
    P = AdaProx.synth.planted_lasso(m, n, 5, 2)
    Lf = AdaProx.synth.spectral_norm_sq(P["A"], iters=500)
    lambdas = float(np.max(np.abs(P["A"].T @ P["b"]))) * (1e-2) ** (np.arange(Lc) / (Lc - 1)) * 0.5
    gam0 = (1 / Lf) * np.linspace(0.6, 1.0, Lc)
    f = AdaProx.LinearLeastSquares(P["A"], P["b"])
    H, K, maxit = 60, 25, 400
    X, its, info = AdaProx.adaptive_proxgrad_path(None, f=f, lambdas=lambdas, rule=getattr(AdaProx, rule)(gamma=1 / Lf), gamma0=gam0,
                                                  tol=1e-6, maxit=maxit, history=H)
    Xo, itso, gh, rh, oh = O.adaptive_proxgrad_path(np.zeros((n, Lc)), f=O.LinearLeastSquares(P["A"], P["b"]), lambdas=lambdas,
                                                   rule_of=lambda j: getattr(O, rule)(gamma=gam0[j]), tol=1e-6, maxit=maxit, history=H)
    for j in sorted({0, Lc // 2, Lc - 1}):
        kj = int(min(K, its[j], itso[j]))
        if kj < 3:
            continue
        truth = drift.lasso_runs(P["A"], P["b"], float(lambdas[j]), lambda O_, j=j: getattr(O_, rule)(gamma=gam0[j]), kj, nperm=2, seed=j)
        ok, dd, allowed = drift.check_inside(info["gamma_hist"][:kj, j], truth, factor=20.0, floor=1e-12)
        assert ok, (j, float(np.max(dd / allowed)), float(dd.max()))
    live = ~np.isnan(oh[:K]) & ~np.isnan(info["obj_hist"][:K])
    assert np.allclose(info["obj_hist"][:K][live], oh[:K][live], rtol=1e-10)
    assert np.all(np.abs(its - itso) <= np.maximum(5, 0.1 * itso)), (its, itso)


# ---------------------------------------------------------------- (c) maxit = 0 everywhere
@pytest.mark.gpu
def test_path_engines_at_maxit_zero_match_the_oracle(AdaProx):
    """Both path engines at maxit = 0 against O.adaptive_proxgrad(maxit = 0): x_1 and its = 0."""
    term, (X0, gam, lam, rg) = dense_instance(130, 300, 5)
    X, term_c, (Xc0, gamc, lamc, rgc) = csr_instance("logistic", "mid", 5)
    for Fd, Fo, t, x0, g, l, r in ((AdaProx.LinearLeastSquares(term.M, term.v), O.LinearLeastSquares(term.M, term.v), term, X0, gam, lam, rg),
                                   (AdaProx.LogisticLoss(X, term_c.v), O.LogisticLoss(X, term_c.v), term_c, Xc0, gamc, lamc, rgc)):
        B1 = reference(t, x0, g, l)["B1"]
        Xd, its, info = AdaProx.adaptive_proxgrad_path(x0, f=Fd, lambdas=l, rule=AdaProx.OurRule(gamma=r), gamma0=g, tol=1e-6, maxit=0)
        Xo, itso, *_ = O.adaptive_proxgrad_path(x0, f=Fo, lambdas=l, rule_of=lambda j: O.OurRule(gamma=g[j]), tol=1e-6, maxit=0)
        assert np.all(its == 0) and np.all(itso == 0)
        ok, ratio = within(Xd, Xo, 2 * B1)
        assert ok, ratio


def _single_lambda_families(AdaProx):
    """(name, env, matrix_passes, device f, term): one AdaPGM kernel family each, forced with the environment switches."""
    term = dense_instance(100, 300, 1)[0]
    fd = AdaProx.LinearLeastSquares(term.M, term.v)
    X, tc, _ = csr_instance("logistic", "mid", 1)
    return [("cluster-resident", {"ADAPROX_RESIDENT": "1"}, 3, fd, term),
            ("grid-resident", {"ADAPROX_RESIDENT": "0", "ADAPROX_GRIDRES": "1"}, 4, fd, term),
            ("single-sweep", {"ADAPROX_FUSED": "1"}, 1, fd, term),
            ("two-pass grid", {"ADAPROX_RESIDENT": "0", "ADAPROX_GRIDRES": "0", "ADAPROX_FUSED": "0"}, 2, fd, term),
            ("csr", {}, None, AdaProx.LogisticLoss(X, tc.v), tc)]


@pytest.mark.gpu
def test_single_lambda_kernels_at_maxit_zero(AdaProx, monkeypatch):
    """Every single-lambda AdaPGM kernel family returns the prologue's x_1 at maxit = 0, as the reference does."""
    for name, env, passes, fd, term in _single_lambda_families(AdaProx):
        rng = np.random.default_rng(5)
        x0 = 0.1 * rng.standard_normal(term.n)
        gam = 0.9 / term.lipschitz()
        _, _, G0 = term.eval(np.zeros((term.n, 1)))
        lam = 0.3 * float(np.max(np.abs(G0)))
        R = reference(term, x0[:, None], np.array([gam]), np.array([lam]))
        with monkeypatch.context() as mp:
            for k, v in env.items():
                mp.setenv(k, v)
            x, it = AdaProx.adaptive_proxgrad(x0, f=fd, g=AdaProx.NormL1(lam), rule=AdaProx.FixedStepsize(gamma=gam), tol=0.0, maxit=0)
            info = AdaProx.last_solve_info()
        if passes is not None:
            assert info["matrix_passes"] == passes, (name, info["matrix_passes"])
        assert it == 0 and not (info["flags"] & 1), name
        ok, ratio = within(x[:, None], R["X1"], R["B1"])
        assert ok, (name, ratio)


# ---------------------------------------------------------------- (d) dense-path determinism
@pytest.mark.gpu
@pytest.mark.parametrize("m,n,Lc", [(1040, 300, 100), (2100, 90, 40)])
def test_dense_path_deterministic_and_position_free(AdaProx, m, n, Lc):
    """Reruns are bit-identical; permuting the lambdas permutes the columns bit for bit.  The shapes split G = A' R into 8 K
    slabs (the first with an empty last slab) and R = A X into several."""
    term, (X0, gam, lam, rg) = dense_instance(m, n, Lc)
    f = AdaProx.LinearLeastSquares(term.M, term.v)
    kw = dict(f=f, rule=AdaProx.OurRule(gamma=rg), tol=1e-6, maxit=200, history=30)
    A1 = AdaProx.adaptive_proxgrad_path(X0, lambdas=lam, gamma0=gam, **kw)
    A2 = AdaProx.adaptive_proxgrad_path(X0, lambdas=lam, gamma0=gam, **kw)
    assert np.array_equal(A1[0], A2[0]) and np.array_equal(A1[1], A2[1])
    for key in ("gamma_hist", "res_hist", "obj_hist", "norm_res", "gamma", "f_x"):
        assert np.array_equal(A1[2][key], A2[2][key], equal_nan=True), key
    perm = np.random.default_rng(0).permutation(Lc)
    B = AdaProx.adaptive_proxgrad_path(X0[:, perm], lambdas=lam[perm], gamma0=gam[perm], **kw)
    assert np.array_equal(B[0], A1[0][:, perm]) and np.array_equal(B[1], A1[1][perm])
    for key in ("gamma_hist", "res_hist", "obj_hist"):
        assert np.array_equal(B[2][key], A1[2][key][:, perm], equal_nan=True), key


# ---------------------------------------------------------------- (e) two devices in one process
@pytest.mark.gpu
def test_path_on_two_devices_in_one_process(AdaProx):
    """The kernels' shared-memory opt-in is per device: the same solves on Device(0) and then Device(1) give the same bits."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    term65, b65 = dense_instance(300, 200, 65)
    term7, b7 = dense_instance(400, 1000, 7)
    X, tc, bc = csr_instance("logistic", "mid", 257)
    default = AdaProx.default_device()
    devs = [AdaProx.Device(0), AdaProx.Device(1)]
    out = []
    try:
        for dev in devs:
            AdaProx.set_default_device(dev)
            got = []
            for f, (X0, gam, lam, rg) in ((AdaProx.LinearLeastSquares(term65.M, term65.v, dev=dev), b65),
                                         (AdaProx.LinearLeastSquares(term7.M, term7.v, dev=dev), b7),
                                         (AdaProx.LogisticLoss(X, tc.v, dev=dev), bc)):
                got.append(AdaProx.adaptive_proxgrad_path(X0, f=f, lambdas=lam, rule=AdaProx.OurRule(gamma=rg), gamma0=gam, tol=1e-6,
                                                          maxit=50, history=10))
            out.append(got)
    finally:
        AdaProx.set_default_device(default)
        for dev in devs:
            dev.close()
    for a, b in zip(*out):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
        for key in ("gamma_hist", "res_hist", "obj_hist"):
            assert np.array_equal(a[2][key], b[2][key], equal_nan=True), key
