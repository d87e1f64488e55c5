"""The primal-dual kernels step by step against an extended-precision reference, over every smooth term, prox object and
linear map.

    k_primal_dual<false>   adaptive_primal_dual, condat_vu, and adaptive_proxgrad on the terms the fused / resident kernels
                           do not take (A = none)                                                  matrix_passes 2 (0: f = Zero)
    k_primal_dual<true>    adaptive_linesearch_primal_dual (AdaPDM+)
    k_malitsky_pock        malitsky_pock

The reference (tests/xprec_reference.py: Smooth, Prox, LinMap, PD, pd_fixed, pd_ourrule, pd_linesearch, mp_reference) restates
one and two steps in np.longdouble and carries an a-priori bound on the device's float64 rounding.  Notation: u = 2^-53; a
vector's error is a pair (e, s), |d1| <= e componentwise plus |d2|_2 <= s.

Sums.  A sum of K products in any order (chunk partials, CTA partials, warp trees, CSR lanes) is off by at most
(K + 2) u sum |a_i b_i| (K - 1 additions, one product, and the slack of the two-level partial sums); an input error e, s adds
|A| e + (row norms) s.  So A x, A' y, F x, F' r and the Gram form's u = Z' x (n + 2) and Z u (d + 2, with u's error) all get
componentwise bounds.  Least squares and the logistic loss keep the bounds of the single-lambda test (Term.dP / Term.dG);
Quadratic: grad = Q x + q, value 0.5 sum x temp + sum x q; Cubic: |x|^2 is off by (n + 2) u |x|^2 + 2 |x| e + e^2, its square
root by that / |x| + u |x|, coef = |x| c / 2 by c / 2 times that + 2 u coef, and coef enters every gradient entry and the
value (sum x g + sum q x) / 2 - |x|^3 c / 12.  f = Zero is exact.

Prox objects.  The separable ones (Zero, IndZero, NormL1, IndBox) are 1-Lipschitz componentwise in their argument and the
soft threshold also in its threshold gamma lambda; a Translate adds u |z| on z = x + b and u |y - b| on the way out.  NormL2
(block soft threshold) is nonexpansive in the 2-norm only: its result is (0, |e_z| + s + lambda d_gamma + (n / 2 + 6) u lambda
gamma + 2 u |z|), the last terms covering the rounded |z|, the scale max(0, 1 - lambda gamma / |z|) and the product.  A
conjugate in ProximalCore's Moreau order (u = w / s, p = prox_{f / s}(u), w - s p) costs e + s e_p + 2 u (|w| + s |p|); an
uncertain step s (OurRule, AdaPDM+) adds d_s times the magnitude of d/ds prox_{s f*}(w) = prox_{s f*}(w + s b)': |b|, plus
the largest finite box bound for IndBox, and |b|_2 for NormL2.  The value of an indicator is exactly 0 or Inf and is compared
by equality; a case in which a point's distance to the box (or to 0) is within its bound is refused when it is built.

One step.  With FixedStepsize(gamma, t): rho = 1 exactly and sigma = gamma (t t) in float64, so record 1's gamma and sigma are
exact; w = y_0 + sigma (2 A x_1 - A x_0) is off by sigma (2 e_Ax1 + e_Ax0) + 4 u (|y_0| + sigma (2 |Ax_1| + |Ax_0|)); then
y_1 = prox_{sigma h*}(w), dual_res = (w - y_1) / sigma - A x_1, the primal residual (v_0 - x_1) / gamma + grad f(x_1) + A' y_0,
norm_res = sqrt(|pr|^2 + |dr|^2) (off by the norms of their errors plus (n + m + 6) u norm_res), the objective
f(x_1) + g(x_1) + h(A x_1), and x_2 = prox_{gamma g}(x_1 - gamma (grad f(x_1) + A' y_1)).  A conjugate g or h has no value on
the device: the objective is NaN.

OurRule with norm_A > 0 extends the single-lambda derivation by xi = t^2 gamma^2 |A|^2 (the device's float64 bits):
S = D + sqrt(D^2 + xi m4) has |dS| / S <= |dD| / sqrt(D^2 + xi m4), so the third term is off by |dS| / 2S + 8 u of itself;
1 / (2 Theta t |A|) is the same float64 operation on both sides.  The bound on gamma_1 is twice that of the active term, and
a case in which two terms of the min are closer than their bounds is refused.  sigma_1 = t^2 gamma_1 and rho = gamma_1 / gamma
then carry d_gamma into w, y_1 and x_2.

AdaPDM+ (first iteration): every trial's gamma_next follows the same first-order bound (eta and the second term are float64
operations the device repeats bit for bit); the test eta >= |A'y+ - A'y| / |y+ - y| is refused when eta is within twice the
first-order relative error of the ratio.  Malitsky-Pock: sigma_0 sqrt(2) and the halvings are exact float64 operations;
lhs = gamma sigma |A x - A x_prev|^2 + 2 gamma (f(x) - f(x_prev) - <grad f(x_prev), x - x_prev>): f(x) - f(x_prev) cancels,
so its bound is that of the difference (the value bounds of both points), and a trial with |lhs - 0.95 |dx|^2| within the
bound is refused.

The shapes come from tests/kernel_plan.py: the linear map A reaches every branch of plan_dense / gsum_slice of the
single-lambda set at the primal-dual grid of 2 CTAs per SM (grid:sm cannot occur with an A), including ADAPROX_GRID 7 and 149
(read at solve time, while A's plan is made at upload for the handle's grid), and CSR A with 4 and 32 lanes per row both from
the mean and forced, with an empty row and an empty column.  A CPU test asserts that the case table reaches every listed branch
and kind at 148 SMs, that every case is well posed, and that the bounds reject each of a list of dropped contributions.
"""
import functools

import numpy as np
import pytest

from kernel_plan import DENSE_REQUIRED, _csr, csr_branches, dense_branches, environ, plan_dense
from xprec_reference import LinMap, PD, Prox, Smooth, mp_reference, pd_fixed, pd_linesearch, pd_ourrule, within

THETA = 1.2


# ---------------------------------------------------------------- problem data
@functools.lru_cache(None)
def dense(m, n, seed):
    return np.random.default_rng([m, n, seed]).standard_normal((m, n)) / np.sqrt(n)


CSR_A = {
    "lpr32": functools.lru_cache(None)(lambda: _csr(300, 260, [215, 230, 240, 225, 0], 12)),   # means 182 rows / 209 cols -> forced
    "lpr32m": functools.lru_cache(None)(lambda: _csr(300, 260, [215, 230, 240, 225], 2)),      # means 227 / 262: 32 lanes both ways
    "lpr4": functools.lru_cache(None)(lambda: _csr(400, 300, [0, 1, 3, 4, 5, 2], 5)),          # 2 / 3: 4 lanes; empty rows and column 1
    "f4100": functools.lru_cache(None)(lambda: _csr(200, 4100, [0, 3, 40, 7, 300], 8)),         # the CSR f of the ADAPROX_GRID cases
    "f4099": functools.lru_cache(None)(lambda: _csr(150, 4099, [2, 30, 9, 100], 9)),
    "f259": functools.lru_cache(None)(lambda: _csr(120, 259, [0, 2, 5, 9, 14], 10)),
}


def smooth(spec, n):
    """spec -> Smooth; the primal dimension is n"""
    kind = spec[0]
    if kind == "zero":
        return Smooth("zero", n=n)
    if kind in ("lsq", "logistic") and spec[1] == "csr":
        X = CSR_A[spec[2]]()
        rng = np.random.default_rng(X.shape[0])
        v = rng.standard_normal(X.shape[0]) if kind == "lsq" else (rng.random(X.shape[0]) < 0.4).astype(np.float64)
        return Smooth(kind, X.toarray(), v)
    if kind in ("lsq", "logistic"):
        m = spec[1]
        M = dense(m, n - (kind == "logistic"), 1)
        rng = np.random.default_rng([m, n, 2])
        v = rng.standard_normal(m) if kind == "lsq" else (rng.random(m) < 0.4).astype(np.float64)
        return Smooth(kind, M, v)
    rng = np.random.default_rng([n, 3])
    q = 0.3 * rng.standard_normal(n)
    if kind == "gram":
        return Smooth("gram", dense(n, spec[1], 4), q)
    B = dense(n, n, 5)
    Q = B @ B.T / 2 + 0.1 * np.eye(n)
    return Smooth(kind, Q, q, c=0.7 if kind == "cubic" else 0.0)


def lipschitz(f, x0):
    if f.kind == "zero":
        return 1.0
    if f.kind in ("lsq", "logistic"):
        return f.term.lipschitz()
    if f.kind == "gram":
        return np.linalg.norm(f.M, 2) ** 2
    L = np.linalg.norm(f.M, 2)
    return L + (f.c * np.linalg.norm(x0) if f.kind == "cubic" else 0.0)


def prox(spec, n, seed, data=None):
    rng = np.random.default_rng([n, seed, 6])
    b = 0.1 * rng.standard_normal(n)
    if spec == "l1":
        return Prox("l1", 0.05)
    if spec == "l2":
        return Prox("l2", 0.2)
    if spec == "zero":
        return Prox("zero")
    if spec == "indzero":
        return Prox("indzero")
    if spec == "box":
        return Prox("box", lo=-0.05, hi=0.07)
    if spec == "boxvec":
        lo = np.where(rng.random(n) < 0.3, -np.inf, -0.05 * rng.random(n))
        hi = np.where(rng.random(n) < 0.3, np.inf, 0.05 * rng.random(n))
        return Prox("box", lo=lo, hi=hi)
    if spec == "tl1":
        return Prox("l1", 0.05, shift=b)
    if spec == "tl2":
        return Prox("l2", 0.2, shift=b)
    if spec == "tl1neg":                            # h = |. - b|_1 (least absolute deviation)
        return Prox("l1", 1.0, shift=-data)
    if spec == "tl2neg":                            # h = |. - b|_2 (square-root lasso)
        return Prox("l2", 1.0, shift=-data)
    if spec == "hbox":
        return Prox("box", lo=-0.6, hi=0.6)
    if spec in ("cl1", "cl2", "cbox"):
        base = prox({"cl1": "l1", "cl2": "l2", "cbox": "box"}[spec], n, seed)
        base.conj = True
        return base
    raise ValueError(spec)


# ---------------------------------------------------------------- the case table
# A: ("dense", m, n, ADAPROX_GRID) / ("csr", name, ADAPROX_CSR_LPR) / None; f: smooth spec; g, h: prox specs
PD_CASES = [
    dict(name="svm300", A=("dense", 1, 300, None), f=("quadratic",), g="box", h="indzero"),
    dict(name="svm50000", A=("dense", 1, 50000, None), f=("gram", 16), g="boxvec", h="indzero"),
    dict(name="lad8190", A=("dense", 8190, 14, None), f=("zero",), g="l1", h="tl1neg"),
    dict(name="sqrtlasso3chunk", A=("dense", 40, 5000, None), f=("lsq", 30), g="l2", h="tl2neg"),
    dict(name="rowA_fmulti", A=("dense", 1, 4500, None), f=("logistic", 60), g="tl1", h="hbox"),
    dict(name="flocal_Amulti", A=("dense", 30, 2049, None), f=("logistic", 50), g="cl1", h="zero"),
    dict(name="grid7", A=("dense", 700, 4100, 7), f=("lsq", "csr", "f4100"), g="cbox", h="cl1"),
    dict(name="grid149", A=("dense", 700, 4100, 149), f=("logistic", "csr", "f4099"), g="cl2", h="cl2"),
    dict(name="rb16", A=("dense", 75777, 5, None), f=("cubic",), g="boxvec", h="tl1neg"),
    dict(name="rb32", A=("dense", 151553, 6, None), f=("quadratic",), g="tl2", h="tl2neg"),
    dict(name="rb64", A=("dense", 303105, 3, None), f=("zero",), g="l1", h="tl1neg"),
    dict(name="csr32mean", A=("csr", "lpr32m", None), f=("lsq", 20), g="l1", h="tl1neg"),
    dict(name="csr4mean", A=("csr", "lpr4", None), f=("quadratic",), g="box", h="tl2neg"),
    dict(name="csr4forced", A=("csr", "lpr32", 4), f=("logistic", "csr", "f259"), g="tl1", h="indzero"),
    dict(name="csr32forced", A=("csr", "lpr4", 32), f=("zero",), g="l2", h="hbox"),
]
# AdaPGM (A = none) on the terms the single-lambda file does not reach: k_primal_dual<false>, matrix_passes 2
PG_CASES = [
    dict(name="logistic_1chunk", A=None, n=301, f=("logistic", 60), g="l1"),
    dict(name="logistic_3chunks", A=None, n=4501, f=("logistic", 50), g="l1"),
    dict(name="quadratic", A=None, n=200, f=("quadratic",), g="l1"),
    dict(name="gram_1chunk", A=None, n=300, f=("gram", 100), g="boxvec"),
    dict(name="gram_3chunks", A=None, n=200, f=("gram", 4500), g="l1"),
    dict(name="cubic", A=None, n=150, f=("cubic",), g="tl1"),
    dict(name="lsq_l2", A=None, n=700, f=("lsq", 90), g="l2"),
    dict(name="lsq_conj", A=None, n=500, f=("lsq", 80), g="cl1"),
]
PDPLUS_CASES = ["svm300", "lad8190", "csr32mean"]
MP_CASES = ["svm300", "lad8190", "csr4mean"]
CV_CASE = "sqrtlasso3chunk"
BY_NAME = {c["name"]: c for c in PD_CASES}


def a_matrix(spec):
    if spec[0] == "dense":
        return dense(spec[1], spec[2], 7)
    return CSR_A[spec[1]]()


def a_dense(spec):
    A = a_matrix(spec)
    return A if spec[0] == "dense" else A.toarray()


@functools.lru_cache(None)
def build(name):
    """-> (PD problem, x_0, y_0, data vector b of h or None)"""
    c = BY_NAME.get(name) or next(p for p in PG_CASES if p["name"] == name)
    if c["A"] is None:
        n = c["n"]
        A = None
    else:
        A = LinMap(a_dense(c["A"]))
        n = A.n
    rng = np.random.default_rng([len(name), n, 8])
    f = smooth(c["f"], n)
    assert f.n == n, (name, f.n, n)
    g = prox(c["g"], n, 1)
    x0 = 0.1 * rng.standard_normal(n)
    if A is None:
        return PD(f, g), x0, None, None
    data = A.A @ (0.1 * rng.standard_normal(n)) + 0.05 * rng.standard_normal(A.m)
    h = prox(c["h"], A.m, 2, data)
    y0 = 0.1 * rng.standard_normal(A.m)
    return PD(f, g, h, A), x0, y0, data


def params(name):
    """FixedStepsize (gamma, t), OurRule's starting gamma (A: kappa / (2 Theta t |A|); none: 3 / L_f) and t"""
    P, x0, _, _ = build(name)
    Lf = lipschitz(P.f, x0)
    if P.A is None:
        return dict(gam=0.8 / Lf, t=1.0, gam_our=3.0 / Lf, t_our=1.0, normA=0.0)
    nA = P.A.norm2
    t = 0.7
    return dict(gam=0.7 / (Lf + t * nA), t=t, gam_our=0.6 / (2 * THETA * t * nA), t_our=t, normA=nA)


@functools.lru_cache(None)
def pd_refs(name):
    P, x0, y0, _ = build(name)
    p = params(name)
    return pd_fixed(P, x0, y0, p["gam"], p["t"]), pd_ourrule(P, x0, y0, p["gam_our"], p["t_our"], p["normA"])


def pdplus_params(name):
    P = build(name)[0]
    eta = 0.2 * P.A.norm2
    return dict(eta=eta, gam=0.9 / (2 * THETA * 1.0 * eta), t=1.0)


@functools.lru_cache(None)
def pdplus_ref(name):
    P, x0, y0, _ = build(name)
    p = pdplus_params(name)
    return pd_linesearch(P, x0, y0, p["gam"], p["eta"], p["t"])


def mp_params(name):
    P, x0, _, _ = build(name)
    t = 0.8
    return dict(sigma=4.0 / (t * (P.A.norm2 + np.sqrt(lipschitz(P.f, x0)))), t=t)


@functools.lru_cache(None)
def mp_ref(name):
    P, x0, y0, _ = build(name)
    p = mp_params(name)
    return mp_reference(P, x0, y0, p["sigma"], p["t"])


def cv_params(name):
    """condat_vu's parameter selection (src/AdaProx.jl:398-412) in float64, as the Python entry point forms it"""
    P, x0, _, _ = build(name)
    f64 = np.float64
    Lf, nA = f64(lipschitz(P.f, x0)), f64(np.linalg.norm(P.A.A))
    alpha = f64(1) if nA > f64(5) * Lf else f64(100) * nA / Lf
    gam = f64(1) / (Lf / 2 + nA / alpha)
    sig = f64(0.99) / (nA * alpha)
    return dict(Lf=float(Lf), normA=float(nA), gam=float(gam), t=float(np.sqrt(sig / gam)))


@functools.lru_cache(None)
def cv_ref(name):
    P, x0, y0, _ = build(name)
    p = cv_params(name)
    return pd_fixed(P, x0, y0, p["gam"], p["t"])


# ---------------------------------------------------------------- coverage of the table
def _a_dense_shapes():
    return [(c["A"][1], c["A"][2], c["A"][3]) for c in PD_CASES if c["A"][0] == "dense"]


def coverage(sm):
    hit = dense_branches(_a_dense_shapes(), sm, has_A=True)
    csr_cases = [(c["A"][1], "lsq", c["A"][2]) for c in PD_CASES if c["A"][0] == "csr"]
    hit |= {"csrA:" + k for k in csr_branches(csr_cases, CSR_A) if k.startswith(("Xw:4:", "Xw:32:", "Xtr:4:", "Xtr:32:"))}
    for name, _, _ in csr_cases:
        X = CSR_A[name]()
        if np.any(np.diff(X.indptr) == 0):
            hit.add("csrA:empty_row")
        if np.any(np.bincount(X.indices, minlength=X.shape[1]) == 0):
            hit.add("csrA:empty_column")
    grid = 2 * sm
    for c in PD_CASES + PG_CASES:
        f = c["f"]
        tag = f[0] + (":csr" if len(f) > 1 and f[1] == "csr" else "")
        n = c["A"][2] if c["A"] and c["A"][0] == "dense" else (build(c["name"])[0].f.n)
        if f[0] in ("lsq", "logistic") and f[1] != "csr":
            nf = n - (f[0] == "logistic")
            nch = plan_dense(f[1], nf, grid)[0]
            if f[0] == "logistic":
                tag += ":1chunk" if nch == 1 else (":multichunk" if nch >= 3 and nf % 2048 else ":2chunks")
            if c["A"] and c["A"][0] == "dense":
                na = plan_dense(c["A"][1], c["A"][2], grid)
                if nch == 1 and na[0] > 1:
                    hit.add("two:F1chunk_Amulti")
                if nch > 1 and c["A"][1] == 1:
                    hit.add("two:Fmulti_Arow")
        if f[0] == "gram":
            tag += ":>2048" if f[1] > 2048 else ":1chunk"
        hit.add("f:" + tag)
        hit.add("g:" + c["g"])
        if c["A"]:
            hit.add("h:" + c["h"])
    return hit


PD_REQUIRED = ((DENSE_REQUIRED - {"grid:sm"}) |
               {f"csrA:{d}:{k}:{h}" for d in ("Xw", "Xtr") for k in (4, 32) for h in ("mean", "forced")} |
               {"csrA:empty_row", "csrA:empty_column", "two:F1chunk_Amulti", "two:Fmulti_Arow"} |
               {"f:" + k for k in ("lsq", "lsq:csr", "logistic:1chunk", "logistic:multichunk", "logistic:csr", "quadratic",
                                   "gram:1chunk", "gram:>2048", "cubic", "zero")} |
               {"g:" + k for k in ("l1", "box", "boxvec", "l2", "tl1", "tl2", "cl1", "cl2", "cbox")} |
               {"h:" + k for k in ("indzero", "zero", "tl1neg", "tl2neg", "hbox", "cl1", "cl2")})


def test_case_table_covers_every_branch_at_148_sms():
    hit = coverage(148)
    assert PD_REQUIRED <= hit, sorted(PD_REQUIRED - hit)


def test_every_case_is_well_posed():
    """Builds every reference: no refusal (the min of OurRule and AdaPDM+, the linesearch / backtracking tests and every
    indicator value are decided by their bounds), AdaPDM+ rejects at least once, Malitsky-Pock halves at least once."""
    for c in PD_CASES + PG_CASES:
        R, O = pd_refs(c["name"])
        assert np.all(np.isfinite(R["B2"])) and np.isfinite(O["dgamma1"]), c["name"]
    for name in PDPLUS_CASES:
        assert pdplus_ref(name)["trials"] >= 2, name
    for name in MP_CASES:
        assert mp_ref(name)["trials"] >= 2, name
    cv_ref(CV_CASE)


# ---------------------------------------------------------------- CPU self-check of the comparator
def test_bounds_reject_dropped_contributions_and_accept_another_order():
    """Each fault below makes the device-side quantity fail its bound by a large ratio; the same quantity in float64 in another
    summation order passes; the bounds are far below the entries they guard."""
    f64 = np.float64

    def rejected(got, ref, bound):
        ok, ratio = within(got, ref, bound)
        assert not ok and ratio > 1e6, ratio

    def accepted(got, ref, bound):
        ok, ratio = within(got, ref, bound)
        assert ok, ratio

    # A x and A' y of a 3-chunk A
    P, x0, y0, _ = build("sqrtlasso3chunk")
    R = pd_refs("sqrtlasso3chunk")[0]
    S, D = R["S"], R["D"]
    A = P.A.A
    x1 = np.asarray(S["X1"], dtype=f64)
    perm = np.random.default_rng(0).permutation(A.shape[1])
    accepted(A[:, perm] @ x1[perm], S["AX1"], S["eAX1"])
    assert np.max(S["eAX1"]) < 1e-9 * np.max(np.abs(np.asarray(S["AX1"], dtype=f64)))
    rejected(A @ x1 - A[:, 2048:4096] @ x1[2048:4096], S["AX1"], S["eAX1"])          # one 2048-column chunk of A x
    y1 = np.asarray(D["Y1"], dtype=f64)
    accepted(A[::-1].T @ y1[::-1], D["ATY1"], D["eATY1"])
    rejected(A.T @ y1 - A[17] * y1[17], D["ATY1"], D["eATY1"])                        # one row of A' y
    # w without the -rho A x_prev term
    sig = R["sigma"]
    AX0, AX1 = A @ x0, A[:, perm] @ x1[perm]
    accepted(y0 + sig * (2 * AX1 - AX0), D["W"], D["eW"])
    rejected(y0 + sig * (2 * AX1), D["W"], D["eW"])
    # one CSR non-zero of A
    P, x0, y0, _ = build("csr4mean")
    S = pd_refs("csr4mean")[0]["S"]
    X = CSR_A["lpr4"]()
    i = int(np.argmax(np.diff(X.indptr)))
    k = X.indptr[i + 1] - 1
    ax = X @ x0
    accepted(ax, S["AX0"], S["eAX0"])
    ax[i] -= X.data[k] * x0[X.indices[k]]
    rejected(ax, S["AX0"], S["eAX0"])
    # one CTA slice of u = Z' x (Gram form, d > 2048)
    P, x0, _, _ = build("gram_3chunks")
    S = pd_refs("gram_3chunks")[0]["S"]
    Z, q = P.f.M, P.f.q
    accepted(Z @ (Z.T @ x0) + q, S["G0"], S["eG0"])
    u = Z.T @ x0
    u[2048:2048 + 15] = Z[:100].T[2048:2048 + 15] @ x0[:100]                           # rows 100.. of that slice left out
    rejected(Z @ u + q, S["G0"], S["eG0"])
    # Translate shift with the wrong sign
    P, x0, _, _ = build("cubic")
    R = pd_refs("cubic")[0]
    S = R["S"]
    gp = P.g
    v0 = np.asarray(S["V0"], dtype=f64)
    z = v0 + gp.b
    good = np.sign(z) * np.maximum(np.abs(z) - R["S"]["gam"] * gp.lam, 0) - gp.b
    accepted(good, S["X1"], R["B1"])
    z = v0 - gp.b
    rejected(np.sign(z) * np.maximum(np.abs(z) - R["S"]["gam"] * gp.lam, 0) + gp.b, S["X1"], R["B1"])
    # the cubic coefficient from |x|^2 instead of |x|
    Q, q, c = P.f.M, P.f.q, P.f.c
    accepted(Q @ x0 + q + np.linalg.norm(x0) * c / 2 * x0, S["G0"], S["eG0"])
    rejected(Q @ x0 + q + (x0 @ x0) * c / 2 * x0, S["G0"], S["eG0"])
    # the logistic intercept left out of a dense multi-chunk gradient
    P, x0, _, _ = build("logistic_3chunks")
    S = pd_refs("logistic_3chunks")[0]["S"]
    t = P.f.term
    z = t.M @ x0[:-1] + x0[-1]
    r = 1 / (1 + np.exp(-z)) - t.v
    G = np.append(t.M.T @ r / t.m, r.sum() / t.m)
    accepted(G, S["G0"], S["eG0"])
    assert np.max(S["eG0"]) < 1e-9 * np.max(np.abs(G))
    z = t.M @ x0[:-1]
    r = 1 / (1 + np.exp(-z)) - t.v
    rejected(np.append(t.M.T @ r / t.m, r.sum() / t.m), S["G0"], S["eG0"])


# ---------------------------------------------------------------- device objects
def dev_smooth(AdaProx, P, spec):
    f = P.f
    if f.kind == "zero":
        return AdaProx.Zero()
    if f.kind in ("lsq", "logistic"):
        M = CSR_A[spec[2]]() if spec[1] == "csr" else f.term.M
        return (AdaProx.LinearLeastSquares if f.kind == "lsq" else AdaProx.LogisticLoss)(M, f.term.v)
    if f.kind == "gram":
        return AdaProx.QuadraticGram(f.M, f.q)
    if f.kind == "cubic":
        return AdaProx.Cubic(f.M, f.q, f.c)
    return AdaProx.Quadratic(f.M, f.q)


def dev_prox(AdaProx, p):
    base = {"zero": AdaProx.Zero, "indzero": AdaProx.IndZero, "l1": lambda: AdaProx.NormL1(p.lam),
            "l2": lambda: AdaProx.NormL2(p.lam), "box": lambda: AdaProx.IndBox(p.lo, p.hi)}[p.kind]()
    if p.b is not None:
        base = AdaProx.Translate(base, p.b)
    return AdaProx.convex_conjugate(base) if p.conj else base


class Device:
    """the device objects of one case (A uploaded with the case's ADAPROX_CSR_LPR / ADAPROX_GEMV)"""

    def __init__(self, AdaProx, name):
        c = BY_NAME.get(name) or next(p for p in PG_CASES if p["name"] == name)
        P, self.x0, self.y0, _ = build(name)
        self.env = {}
        if c["A"] is not None and c["A"][0] == "dense" and c["A"][3]:
            self.env["ADAPROX_GRID"] = c["A"][3]
        up = {"ADAPROX_CSR_LPR": c["A"][2] or 0} if c["A"] is not None and c["A"][0] == "csr" else {}
        with environ(up):
            self.f = dev_smooth(AdaProx, P, c["f"])
            self.A = AdaProx.DeviceMatrix(a_matrix(c["A"])) if c["A"] is not None else None
        self.g = dev_prox(AdaProx, P.g)
        self.h = dev_prox(AdaProx, P.h) if P.h is not None else None
        self.passes = 0 if P.f.kind == "zero" else 2

    def free(self):
        for m in (getattr(self.f, "mat", None), self.A):
            if m is not None:
                m.free()


def _check_record(rec, R, key_res="res1", key_obj="obj1"):
    ok, ratio = within(rec["norm_res"], R[key_res], R["dres1"])
    assert ok, ("norm_res", ratio, rec["norm_res"], R[key_res])
    obj = R[key_obj]
    if np.isfinite(obj):
        ok, ratio = within(rec["objective"], obj, R["dobj1"])
        assert ok, ("objective", ratio, rec["objective"], obj)
    else:
        assert np.array_equal(rec["objective"], obj, equal_nan=True), ("objective", rec["objective"], obj)


def _pd_solves(AdaProx, d, solve, R, O, y_is_pd):
    """maxit = 0, maxit = 1 (FixedStepsize) and one OurRule step through `solve(rule, maxit, log)`"""
    x, y, it = solve(None, 0, None)
    i0 = AdaProx.last_solve_info()
    log = []
    x2, y1, it2 = solve(None, 1, log)
    i1 = AdaProx.last_solve_info()
    logo = []
    xo, yo, ito = solve("our", 1, logo)
    i2 = AdaProx.last_solve_info()
    assert [i["matrix_passes"] for i in (i0, i1, i2)] == [d.passes] * 3, "kernel selection"
    assert it == 0 and it2 == 1 and ito == 1
    ok, ratio = within(x, R["X1"], R["B1"])
    assert ok, ("maxit = 0: x_1", ratio)
    ok, ratio = within(x2, R["X2"], R["B2"])
    assert ok, ("maxit = 1: x_2", ratio)
    if y_is_pd:
        assert np.array_equal(y, d.y0), "maxit = 0: y_0 comes back"
        D = R["D"]
        ok, ratio = within(y1, D["Y1"], D["ey1"] + D["sy1"])
        assert ok, ("maxit = 1: y_1", ratio)
    assert log[0]["gamma"] == R["S"]["gam"] and log[0]["sigma"] == R["sigma"], "FixedStepsize: gamma and sigma exact"
    _check_record(log[0], R)
    ok, ratio = within(logo[0]["gamma"], O["gamma1"], O["dgamma1"])
    assert ok, ("OurRule gamma_1", ratio, logo[0]["gamma"], O["gamma1"])
    ok, ratio = within(xo, O["X2"], O["B2"])
    assert ok, ("OurRule x_2", ratio)
    if y_is_pd:
        D = O["D"]
        ok, ratio = within(yo, D["Y1"], D["ey1"] + D["sy1"])
        assert ok, ("OurRule y_1", ratio)


def _device_sm(AdaProx):
    return AdaProx.default_device().info()["sm_count"]


@pytest.mark.gpu
def test_case_table_reaches_every_branch_on_this_device(AdaProx):
    hit = coverage(_device_sm(AdaProx))
    assert PD_REQUIRED <= hit, sorted(PD_REQUIRED - hit)


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in PD_CASES])
def test_adaptive_primal_dual_matches_extended_precision(AdaProx, name):
    R, O = pd_refs(name)
    p = params(name)
    d = Device(AdaProx, name)

    def solve(rule, maxit, log):
        r = AdaProx.OurRule(gamma=p["gam_our"], t=p["t_our"], norm_A=p["normA"]) if rule else AdaProx.FixedStepsize(p["gam"], p["t"])
        return AdaProx.adaptive_primal_dual(d.x0, d.y0, f=d.f, g=d.g, h=d.h, A=d.A, rule=r, tol=0.0, maxit=maxit, log=log)

    try:
        with environ(d.env):
            _pd_solves(AdaProx, d, solve, R, O, True)
    finally:
        d.free()


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in PG_CASES])
def test_adaptive_proxgrad_general_kernel_matches_extended_precision(AdaProx, name):
    R, O = pd_refs(name)
    p = params(name)
    d = Device(AdaProx, name)

    def solve(rule, maxit, log):
        r = AdaProx.OurRule(gamma=p["gam_our"]) if rule else AdaProx.FixedStepsize(p["gam"])
        x, it = AdaProx.adaptive_proxgrad(d.x0, f=d.f, g=d.g, rule=r, tol=0.0, maxit=maxit, log=log)
        return x, None, it

    try:
        _pd_solves(AdaProx, d, solve, R, O, False)
    finally:
        d.free()


@pytest.mark.gpu
def test_condat_vu_matches_extended_precision(AdaProx):
    R = cv_ref(CV_CASE)
    p = cv_params(CV_CASE)
    d = Device(AdaProx, CV_CASE)
    try:
        log = []
        x2, y1, it = AdaProx.condat_vu(d.x0, d.y0, f=d.f, g=d.g, h=d.h, A=d.A, Lf=p["Lf"], norm_A=p["normA"], tol=0.0, maxit=1, log=log)
        assert AdaProx.last_solve_info()["matrix_passes"] == d.passes and it == 1
    finally:
        d.free()
    assert log[0]["gamma"] == R["S"]["gam"] and log[0]["sigma"] == R["sigma"]
    ok, ratio = within(x2, R["X2"], R["B2"])
    assert ok, ("x_2", ratio)
    ok, ratio = within(y1, R["D"]["Y1"], R["D"]["ey1"] + R["D"]["sy1"])
    assert ok, ("y_1", ratio)
    _check_record(log[0], R)


@pytest.mark.gpu
@pytest.mark.parametrize("name", PDPLUS_CASES)
def test_adapdm_plus_linesearch_matches_extended_precision(AdaProx, name):
    R = pdplus_ref(name)
    p = pdplus_params(name)
    d = Device(AdaProx, name)
    try:
        with environ(d.env):
            x, y, it = AdaProx.adaptive_linesearch_primal_dual(d.x0, d.y0, f=d.f, g=d.g, h=d.h, A=d.A, gamma=p["gam"], eta=p["eta"],
                                                              t=p["t"], tol=0.0, maxit=0)
            i0 = AdaProx.last_solve_info()
            log = []
            A = AdaProx.Counting(d.A)                  # counts accumulate over the calls of one wrapper: a fresh one
            x2, y1, it1 = AdaProx.adaptive_linesearch_primal_dual(d.x0, d.y0, f=d.f, g=d.g, h=d.h, A=A, gamma=p["gam"],
                                                                  eta=p["eta"], t=p["t"], tol=0.0, maxit=1, log=log)
            i1 = AdaProx.last_solve_info()
    finally:
        d.free()
    assert i0["matrix_passes"] == i1["matrix_passes"] == d.passes
    assert it == 0 and it1 == 1
    ok, ratio = within(x, R["S"]["X1"], R["S"]["e1"] + R["S"]["s1"])
    assert ok, ("maxit = 0: x_1", ratio)
    assert np.array_equal(y, d.y0)
    assert log[0]["At_evals"] == 1 + R["trials"], ("linesearch trials", log[0]["At_evals"] - 1, R["trials"], R["tests"])
    ok, ratio = within(log[0]["gamma"], R["gamma1"], R["dgamma1"])
    assert ok, ("gamma_1", ratio, log[0]["gamma"], R["gamma1"])
    D = R["D"]
    ok, ratio = within(y1, D["Y1"], D["ey1"] + D["sy1"])
    assert ok, ("y_1", ratio)
    ok, ratio = within(x2, R["X2"], R["B2"])                    # x_2 carries A' y_1
    assert ok, ("x_2", ratio)


@pytest.mark.gpu
@pytest.mark.parametrize("name", MP_CASES)
def test_malitsky_pock_backtracking_matches_extended_precision(AdaProx, name):
    R = mp_ref(name)
    p = mp_params(name)
    d = Device(AdaProx, name)
    try:
        x, y, it = AdaProx.malitsky_pock(d.x0, d.y0, f=d.f, g=d.g, h=d.h, A=d.A, sigma=p["sigma"], t=p["t"], tol=0.0, maxit=0)
        i0 = AdaProx.last_solve_info()
        log = []
        g = AdaProx.Counting(d.g)                      # counts accumulate over the calls of one wrapper: a fresh one
        x1, y1, it1 = AdaProx.malitsky_pock(d.x0, d.y0, f=d.f, g=g, h=d.h, A=d.A, sigma=p["sigma"], t=p["t"], tol=0.0, maxit=1, log=log)
        i1 = AdaProx.last_solve_info()
    finally:
        d.free()
    assert i0["matrix_passes"] == i1["matrix_passes"] == d.passes
    assert it == 0 and np.array_equal(x, d.x0) and np.array_equal(y, d.y0), "maxit = 0: x_0 and y_0 come back"
    assert it1 == 1
    assert log[0]["sigma"] == R["sigma"] and log[0]["gamma"] == R["gamma"], "sigma_0 sqrt(2) and the halvings are exact"
    assert log[0]["prox_g_evals"] == R["trials"], ("backtracking trials", log[0]["prox_g_evals"], R["trials"], R["tests"])
    ok, ratio = within(x1, R["X1"], R["B1"])
    assert ok, ("x_1", ratio)
    ok, ratio = within(y1, R["Y1"], R["BY1"])
    assert ok, ("y_1", ratio)
    _check_record(log[0], R)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["g=NormL2", "g conjugate", "h conjugate"])
def test_malitsky_pock_refuses_what_it_has_no_kernel_for(AdaProx, which):
    P, x0, y0, _ = build("lad8190")
    d = Device(AdaProx, "lad8190")
    g, h = d.g, d.h
    if which == "g=NormL2":
        g = AdaProx.NormL2(0.2)
    elif which == "g conjugate":
        g = AdaProx.convex_conjugate(AdaProx.NormL1(0.05))
    else:
        h = AdaProx.convex_conjugate(AdaProx.NormL1(1.0))
    try:
        with pytest.raises(AdaProx.AdaproxError) as e:
            AdaProx.malitsky_pock(x0, y0, f=d.f, g=g, h=h, A=d.A, sigma=1.0, tol=0.0, maxit=1)
    finally:
        d.free()
    assert e.value.code == -3


# ---------------------------------------------------------------- bit-identical reruns at the largest case of each kernel
@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["adapdm", "adapdm+", "mp"])
def test_reruns_are_bit_identical(AdaProx, kernel):
    name = {"adapdm": "rb64", "adapdm+": "lad8190", "mp": "lad8190"}[kernel]
    d = Device(AdaProx, name)
    runs = []
    try:
        for _ in range(2):
            log = []
            if kernel == "adapdm":
                p = params(name)
                x, y, it = AdaProx.adaptive_primal_dual(d.x0, d.y0, f=d.f, g=d.g, h=d.h, A=d.A, tol=0.0, maxit=12, log=log,
                                                        rule=AdaProx.OurRule(gamma=p["gam_our"], t=p["t_our"], norm_A=p["normA"]))
            elif kernel == "adapdm+":
                p = pdplus_params(name)
                x, y, it = AdaProx.adaptive_linesearch_primal_dual(d.x0, d.y0, f=d.f, g=d.g, h=d.h, A=d.A, gamma=p["gam"],
                                                                  eta=p["eta"], tol=0.0, maxit=12, log=log)
            else:
                p = mp_params(name)
                x, y, it = AdaProx.malitsky_pock(d.x0, d.y0, f=d.f, g=d.g, h=d.h, A=d.A, sigma=p["sigma"], t=p["t"], tol=0.0,
                                                 maxit=12, log=log)
            runs.append((x, y, it, np.array([(r["gamma"], r["sigma"], r["norm_res"], r["objective"]) for r in log]),
                         AdaProx.last_solve_info()))
    finally:
        d.free()
    (xa, ya, ia, la, fa), (xb, yb, ib, lb, fb) = runs
    assert fa["matrix_passes"] == fb["matrix_passes"] == d.passes
    assert ia == ib == 12 and la.shape == (12, 4)
    assert np.array_equal(xa, xb) and np.array_equal(ya, yb) and np.array_equal(la, lb, equal_nan=True)
    assert np.all(np.isfinite(xa)) and np.all(np.isfinite(ya))
