"""The single-lambda AdaPGM kernels (adaptive_proxgrad) step by step against an extended-precision reference.

Every kernel family that runs adaptive_proxgrad on a least-squares or logistic term is forced in turn and compared with the
np.longdouble restatement of tests/xprec_reference.py (the L = 1 column of the batched-path check, whose bounds are derived
in test_gpu_lambda_path_reference.py):

    k_adapgm_fused          single sweep, clusters of C = ceil(ld / 8192) CTAs        ADAPROX_FUSED=1         matrix_passes 1
    k_primal_dual<false>    two-pass grid kernel, dense (ring and ldg) and CSR        ADAPROX_FUSED=0 ...     matrix_passes 2
    k_adapgm_resident       matrix in the shared memory of one 16-CTA cluster          ADAPROX_RESIDENT=1      matrix_passes 3
    k_adapgm_gridres<0>     matrix in the shared memory of one CTA per SM             ADAPROX_GRIDRES=1       matrix_passes 4

With FixedStepsize(gamma), gamma in [0.5, 0.999] / L_f and g = NormL1(lambda), maxit = 0 must return x_1 inside the
componentwise bound B1, and maxit = 1 must return x_2 inside the per-column 2-norm bound, with record 1's gamma equal to gamma
and its norm_res / objective inside dres1 / dobj1.  lambda = 0 makes x_1 - x_0 = -gamma grad f(x_0): the gradient itself is
compared.

One adaptive step (OurRule, t = 1, norm_A = 0, delta = 0, started at gamma = 3 / L_f so that its third term is the active
one) is checked with a first-order bound.  With dx = x_1 - x_0, dg = grad f(x_1) - grad f(x_0) and

    a = |dg|^2,   b = <dg, dx>,   c = |dx|^2,   C = a / b,   L = b / c,   D = gamma L (gamma C - 1),
    gamma_1 = min(gamma sqrt(2), gamma / sqrt(2 (D + |D|)))      (= gamma sqrt(2) when D <= 0)

the device's dx and dg differ from the reference's componentwise by at most e_x = B1 + u |dx| and
e_g = dG(x_0) + dG(x_1) + u |dg| (dG: the gradient bounds of the reference; the one at x_1 carries x_1's error B1).  Hence

    e_a = sum(2 |dg| e_g + e_g^2) + (n + 2) u a
    e_b = sum(|dg| e_x + |dx| e_g + e_g e_x) + (n + 2) u sum(|dg| |dx|)
    e_c = sum(2 |dx| e_x + e_x^2) + (n + 2) u c

and, to first order, |dD| / D <= e_b / b + e_c / c + (gamma C (e_a / a + e_b / b + 2 u) + u) / |gamma C - 1| + 4 u,
so the third term is off by at most (|dD| / 2 D + 8 u) of itself; gamma sqrt(2) by 4 u of itself.  The bound on gamma_1 is
twice that of the active term (the factor covers the neglected second-order terms); a case in which the two terms are closer
than their bounds would leave the choice of the minimum open and is refused as ill-posed.  Then x_2 = S_{gamma_1 lambda}(x_1 -
gamma_1 grad f(x_1)) is bounded componentwise (no contraction is assumed: gamma_1 > 1 / L_f here):

    |dx_2| <= 2 [B1 + gamma_1 dG(x_1) + |d gamma_1| |grad f(x_1)| + 2 u (|x_1| + gamma_1 |grad f(x_1)|) + (u gamma_1 + |d gamma_1|) lambda]

The shapes come from a restatement of the work split of each kernel (api.cu: fused_cluster_size, fused_plan, plan_dense,
solver_grid, gridres_eligible; gemv.cuh: csr_lanes_per_row, gsum_slice; solver_fused.cuh: fused_pass, fused_gradient_slice);
the parts the primal-dual reference test shares live in tests/kernel_plan.py.
A CPU test asserts that the shape set reaches every branch at 148 SMs, a GPU test at the device's SM count.  The CPU self-check
shows that the bounds reject a result with one 2048-column chunk of A x, one row of A' r, one 8192-column CTA slice or one CSR
non-zero left out, and accept a float64 evaluation in another summation order.
"""
import functools

import numpy as np
import pytest

from kernel_plan import DENSE_REQUIRED, _csr, cdiv, csr_branches, dense_branches, environ, r16
from xprec_reference import LD, U, Term, reference, within, within_cols

B200_SMEM_OPTIN = 232448          # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200 (227 KB)
KFCOLS, KFMAXC = 8192, 16


# ---------------------------------------------------------------- restatement of the kernel selection
def fused_cluster_size(n):
    """api.cu: fused_cluster_size -- CTAs of 8192 columns over the padded row (ld = n rounded up to 16)."""
    return cdiv(r16(n), KFCOLS)


def fused_clusters_at_least(C, sm):
    """A lower bound on the clusters of C CTAs (one CTA per SM, 192 KB of shared memory each) that fit the device: at least
    half of its SMs take part for every cluster size up to 16 (B200: 148 one-CTA clusters, 7 of 16 CTAs)."""
    return max(1, sm // (2 * C))


def fused_chunk_rows(m, Q, chunk):
    """api.cu: fused_plan -> (chunk_rows, nchunks) for Q resident clusters and ADAPROX_FUSED_CHUNK = chunk (None: unset)."""
    kper = 8 if m // max(Q, 1) >= 4096 else 4
    pw = max(16, cdiv(m, Q * kper))
    if chunk is not None:
        pw = int(chunk)
    return pw, cdiv(m, pw)


def fused_branches(cases, sm):
    hit = set()
    for m, n, chunk, helpers in cases:
        C = fused_cluster_size(n)
        Qmin = fused_clusters_at_least(C, sm)
        if chunk is None:                           # the default chunk is 16 rows whenever m <= 64 Q: known from the lower bound
            assert cdiv(m, 4 * Qmin) <= 16 and m // Qmin < 4096, (m, n)
        pw, nch = fused_chunk_rows(m, Qmin, chunk)
        hit.add(f"C:{C}")
        last = r16(n) - KFCOLS * (C - 1)
        hit |= {"last:16"} if last == 16 else ({"last:8192"} if last == KFCOLS else set())
        if n % 16:
            hit.add("n%16")
        hit.add("chunk:default" if chunk is None else ("chunk:>=m" if int(chunk) >= m else f"chunk:{chunk}"))
        rows = {min(pw, m), m - (nch - 1) * pw}     # rows of a full chunk and of the last one
        if min(pw, m) < 3:
            hit.add("rows<3")
        elif min(pw, m) < 8:
            hit.add("rows<8")
        if any(r > 32 and r % 32 for r in rows):
            hit.add("b_reload")
        hit.add("chunks>8" if nch > 8 else ("chunks<8" if nch < 8 else "chunks=8"))
        if m < Qmin:
            hit.add("rows<clusters")
        if helpers and C == KFMAXC:
            hit.add("helpers")
    return hit


FUSED_REQUIRED = {f"C:{c}" for c in range(1, 17)} | {"last:16", "last:8192", "n%16", "chunk:1", "chunk:5", "chunk:default",
                                                      "chunk:>=m", "rows<3", "rows<8", "b_reload", "chunks>8", "chunks<8",
                                                      "rows<clusters", "helpers"}


def gridres_x_in_smem(m, n, sm, optin=B200_SMEM_OPTIN):
    """api.cu: gridres_eligible -> True / False (x in shared / global memory); None: not eligible."""
    ld = r16(n)
    rows_cap = cdiv(m, sm)
    need = lambda xs: 8 * (rows_cap * ld + 2 * rows_cap + 16 + 16 * 8 + 16 + (ld if xs else 0))
    if ld > 1024 or cdiv(n, sm) > 16 or need(False) + 1024 > optin:
        return None
    return need(True) + 1024 <= optin


def resident_fits(m, n, optin=B200_SMEM_OPTIN):
    """api.cu: resident_eligible"""
    ld = r16(n)
    rows_cap = cdiv(m, 16)
    return ld <= 1024 and 8 * (rows_cap * ld + 2 * ld + 2 * rows_cap + 16 + 32) + 1024 <= optin


CSR_REQUIRED = ({f"{d}:{k}:{h}" for d in ("Xw", "Xtr") for k in (4, 8, 16, 32) for h in ("mean", "forced")} |
                {f"rows:{k}" for k in (4, 8, 16, 32)} | {"kind:lsq", "kind:logistic", "empty_feature", "rows<group"})


# ---------------------------------------------------------------- the shape sets
# fused: (m, n, ADAPROX_FUSED_CHUNK, helpers); n = 8192 (C - 1) + w
FUSED_CASES = [(3, 16, None, False), (70, 8192, "5", False), (45, 8192 + 16, "64", False), (100, 2 * 8192 + 4001, None, False),
               (37, 3 * 8192 + 8192, "1", False), (40, 4 * 8192 + 5, None, False), (33, 5 * 8192 + 8000, "5", False),
               (50, 6 * 8192 + 16, None, False), (20, 7 * 8192 + 8192, "100", False), (24, 8 * 8192 + 3333, "1", False),
               (30, 9 * 8192 + 17, None, False), (20, 10 * 8192 + 8191, "5", False), (16, 11 * 8192 + 16, None, False),
               (12, 12 * 8192 + 2048, "2", False), (12, 13 * 8192 + 8192, None, False), (10, 14 * 8192 + 1234, "1", False),
               (40, 15 * 8192 + 16, None, False), (40, 16 * 8192, "4", True)]
# two-pass dense: (m, n, ADAPROX_GRID)
DENSE_CASES = [(5, 40, None), (1000, 1000, None), (1003, 5000, None), (700, 4100, 7), (700, 4100, 149), (300, 8000, None),
               (75777, 16, None), (151553, 16, None), (303105, 8, None), (2, 6000, None)]
RESIDENT_CASES = [(400, 1000), (100, 300), (7, 1), (5, 1024), (33, 517), (416, 1024)]
GRIDRES_CASES = [(500, 1000), (4000, 1000), (120, 40), (1, 1024), (3000, 517), (4100, 1024), (4144, 1000)]


MIXED_LENGTHS = [0, 1, 3, 7, 15, 31, 4, 16, 17, 8, 32, 33, 64, 65, 128, 129, 2100]
CSR_MATRICES = {
    "mixed": functools.lru_cache(None)(lambda: _csr(340, 2500, MIXED_LENGTHS, 1)),           # every LPR's edge lengths, one > 2000
    "lpr32": functools.lru_cache(None)(lambda: _csr(300, 260, [215, 230, 240, 225], 2)),    # means 227 / 262: 32 lanes both ways
    "lpr16": functools.lru_cache(None)(lambda: _csr(200, 150, [40, 60, 80, 2, 118], 3)),    # 60 / 80: 16 lanes
    "lpr8": functools.lru_cache(None)(lambda: _csr(200, 200, [10, 18, 26, 0, 30], 4)),      # 16 / 16: 8 lanes
    "lpr4": functools.lru_cache(None)(lambda: _csr(400, 300, [0, 1, 3, 4, 5, 2], 5)),       # 2 / 3: 4 lanes
    "tiny": functools.lru_cache(None)(lambda: _csr(5, 40, [0, 1, 3, 7, 2], 6)),             # fewer rows than one row group
}
CSR_CASES = ([(name, kind, None) for name in CSR_MATRICES for kind in ("lsq", "logistic")] +
             [("mixed", kind, lpr) for lpr in (4, 8, 16, 32) for kind in ("lsq", "logistic")] +
             [("tiny", "lsq", 32), ("lpr4", "logistic", 32)])


def _assert_reaches_everything(sm):
    for hit, req in ((fused_branches(FUSED_CASES, sm), FUSED_REQUIRED), (dense_branches(DENSE_CASES, sm), DENSE_REQUIRED),
                     (csr_branches(CSR_CASES, CSR_MATRICES), CSR_REQUIRED)):
        assert req <= hit, (sm, sorted(req - hit))
    xs = {gridres_x_in_smem(m, n, sm) for m, n in GRIDRES_CASES}
    assert xs == {True, False}, (sm, xs)
    assert all(resident_fits(m, n) for m, n in RESIDENT_CASES)


def test_shape_sets_cover_every_branch_at_148_sms():
    _assert_reaches_everything(148)
    assert fused_cluster_size(16 * 8192) == 16 and fused_cluster_size(16 * 8192 + 1) == 17


# ---------------------------------------------------------------- instances
LAM_FRACTIONS = (0.0, 0.9, 0.3, 0.97, 0.0, 0.5)     # lambda / lambda_max, cycled through a family (the first case: lambda = 0)


def _instance(term, k, seed):
    """x_0 (about 20 % exact zeros), FixedStepsize gamma in [0.5, 0.999] / L_f, lambda, OurRule's starting gamma = 3 / L_f"""
    rng = np.random.default_rng(seed)
    Lf = term.lipschitz()
    x0 = 0.1 * rng.standard_normal(term.n)
    x0[rng.random(term.n) < 0.2] = 0.0
    _, _, G0 = term.eval(np.zeros((term.n, 1)))
    lam = LAM_FRACTIONS[k % len(LAM_FRACTIONS)] * float(np.max(np.abs(G0)))
    return x0, float(rng.uniform(0.5, 0.999)) / Lf, lam, 3.0 / Lf


@functools.lru_cache(None)
def dense_term(m, n):
    rng = np.random.default_rng(31 * m + n)
    return Term("lsq", rng.standard_normal((m, n)) / np.sqrt(n), rng.standard_normal(m))


@functools.lru_cache(None)
def csr_term(name, kind):
    X = CSR_MATRICES[name]()
    rng = np.random.default_rng(len(name) * 7 + (kind == "logistic"))
    v = rng.standard_normal(X.shape[0]) if kind == "lsq" else (rng.random(X.shape[0]) < 0.4).astype(np.float64)
    return Term(kind, X.toarray(), v)


# ---------------------------------------------------------------- the adaptive step in extended precision and its bound
def ourrule_step(term, R, col, gam, lam):
    """OurRule's gamma_1 and x_2 after the step x_0 -> x_1 of column `col` of `R` (reference() with gamma as its gamma),
    with the first-order bounds of the module docstring."""
    f = lambda a: np.asarray(a, dtype=np.float64)
    X0, X1, G0, G1 = (R["ld"][k][:, col] for k in ("X0", "X1", "G0", "G1"))
    dx, dg = X1 - X0, G1 - G0
    a, b, c = np.sum(dg * dg), np.sum(dg * dx), np.sum(dx * dx)
    g = LD(gam)
    D = g * (b / c) * (g * (a / b) - 1)
    t1 = g * np.sqrt(LD(2))
    t3 = g / np.sqrt(2 * (D + abs(D))) if D > 0 else LD(np.inf)
    g1 = min(t1, t3)
    X2 = X1 - g1 * G1
    X2 = np.sign(X2) * np.maximum(np.abs(X2) - g1 * LD(lam), 0)
    # first-order bound on gamma_1
    dxa, dga, B1 = np.abs(f(dx)), np.abs(f(dg)), R["B1"][:, col]
    ex = B1 + U * dxa
    eg = R["dG0"][:, col] + R["dG1"][:, col] + U * dga
    n = term.n
    a, b, c = float(a), float(b), float(c)
    ea = np.sum(2 * dga * eg + eg * eg) + (n + 2) * U * a
    eb = np.sum(dga * ex + dxa * eg + eg * ex) + (n + 2) * U * np.sum(dga * dxa)
    ec = np.sum(2 * dxa * ex + ex * ex) + (n + 2) * U * c
    gC = gam * a / b
    rD = eb / b + ec / c + (gC * (ea / a + eb / b + 2 * U) + U) / abs(gC - 1) + 4 * U
    e3 = 2 * (0.5 * rD + 8 * U) * float(t3) if np.isfinite(float(t3)) else np.inf
    e1 = 2 * 4 * U * float(t1)
    assert abs(float(t1) - float(t3)) > e1 + e3, ("the active term of OurRule is not decided by the bound", float(t1), float(t3))
    dgam = e3 if t3 < t1 else e1
    G1a = np.abs(f(G1))
    eV = B1 + float(g1) * R["dG1"][:, col] + dgam * G1a + 2 * U * (np.abs(f(X1)) + float(g1) * G1a)
    return dict(gamma1=float(g1), dgamma1=dgam, X2=f(X2), B2=2 * (eV + (U * float(g1) + dgam) * lam), third=bool(t3 < t1))


def full_reference(term, x0, gam, lam, gam_our):
    """column 0: FixedStepsize(gam); column 1: OurRule started at gam_our"""
    R = reference(term, np.column_stack([x0, x0]), np.array([gam, gam_our]), np.array([lam, lam]))
    R["our"] = ourrule_step(term, R, 1, gam_our, lam)
    return R


# ---------------------------------------------------------------- CPU self-checks of the comparator and of the coverage
def test_bounds_reject_dropped_contributions_and_accept_another_order():
    """A result with one 2048-column chunk of A x, one row of A' r, one 8192-column CTA slice of A x or one CSR row's last
    non-zero left out fails the bounds; a plain float64 evaluation (BLAS summation order) passes them; the bounds are far
    below the entries they guard.  The same for OurRule's gamma_1 and x_2."""
    rng = np.random.default_rng(11)
    m, n = 40, 9000                                  # 5 column chunks of 2048, 2 CTA slices of 8192
    term = Term("lsq", rng.standard_normal((m, n)) / np.sqrt(n), rng.standard_normal(m))
    Xc = _csr(60, 300, [0, 1, 3, 7, 40], 9)
    cterm = Term("lsq", Xc.toarray(), rng.standard_normal(60))
    lterm = Term("logistic", Xc.toarray(), (rng.random(60) < 0.4).astype(np.float64))

    def x1_with(t, x0, gam, P):                      # x_1 from a residual P (lambda = 0 below)
        G = t.M.T @ P * t.s
        if t.kind == "logistic":
            G = np.append(G, P.sum() * t.s)
        return x0 - gam * G

    for t in (term, cterm, lterm):
        x0, gam, _, gam_our = _instance(t, 0, 3)
        lam = 0.0
        R = full_reference(t, x0, gam, lam, gam_our)
        x1, _, _, f0, P = t.step(x0[:, None], np.array([gam]), np.array([lam]))
        assert within(x1, R["X1"][:, :1], R["B1"][:, :1])[0]
        assert within(f0, R["f0"][:1], R["df0"][:1])[0]
        assert within_cols(t.step(x1, np.array([gam]), np.array([lam]))[0], R["X2"][:, :1], R["B2col"][:1])[0]
        assert np.max(R["B1"]) < 1e-9 * max(np.max(np.abs(R["X1"])), 1.0)
        # OurRule in float64
        xo1, _, G0 = t.step(x0[:, None], np.array([gam_our]), np.array([lam]))[:3]
        G1 = t.eval(xo1)[2]
        dx, dg = (xo1 - x0[:, None])[:, 0], (G1 - G0)[:, 0]
        a, b, c = dg @ dg, dg @ dx, dx @ dx
        D = gam_our * (b / c) * (gam_our * (a / b) - 1)
        g1 = min(gam_our * np.sqrt(2), gam_our / np.sqrt(2 * (D + abs(D))) if D > 0 else np.inf)
        O = R["our"]
        assert O["third"] and abs(g1 - O["gamma1"]) <= O["dgamma1"] < 1e-7 * g1, (g1, O["gamma1"], O["dgamma1"])
        assert within(xo1[:, 0] - g1 * G1[:, 0], O["X2"], O["B2"])[0]
        assert not within(xo1[:, 0] - g1 * (1 + 1e-6) * G1[:, 0], O["X2"], O["B2"])[0]

    def rejected(t, x0, gam, R, P):
        ok, ratio = within(x1_with(t, x0, gam, P), R["X1"][:, 0], R["B1"][:, 0])
        assert not ok and ratio > 1e6, ratio

    x0, gam, _, gam_our = _instance(term, 0, 3)
    R = full_reference(term, x0, gam, 0.0, gam_our)
    P = term.M @ x0 - term.v
    rejected(term, x0, gam, R, P - term.M[:, 2048:4096] @ x0[2048:4096])            # one column chunk of A x
    rejected(term, x0, gam, R, P - term.M[:, 8192:] @ x0[8192:])                    # the second CTA slice of A x
    Pd = P.copy()
    Pd[17] = 0.0                                                                    # one row of A' r
    rejected(term, x0, gam, R, Pd)
    for t in (cterm, lterm):
        x0, gam, _, gam_our = _instance(t, 0, 3)
        R = full_reference(t, x0, gam, 0.0, gam_our)
        i = 4                                                                       # a row of 40 non-zeros
        k = Xc.indptr[i + 1] - 1
        z = t.M @ x0[:t.nf] + (x0[-1] if t.kind == "logistic" else 0.0)
        z[i] -= Xc.data[k] * x0[Xc.indices[k]]
        P = z - t.v if t.kind == "lsq" else 1 / (1 + np.exp(-z)) - t.v
        rejected(t, x0, gam, R, P)


# ---------------------------------------------------------------- device against the reference
def _check(AdaProx, fd, term, k, seed, env, passes):
    x0, gam, lam, gam_our = _instance(term, k, seed)
    R = full_reference(term, x0, gam, lam, gam_our)
    g = AdaProx.NormL1(lam)
    with environ(env):
        x, it = AdaProx.adaptive_proxgrad(x0, f=fd, g=g, rule=AdaProx.FixedStepsize(gam), tol=0.0, maxit=0)
        info0 = AdaProx.last_solve_info()
        log = []
        x2, it2 = AdaProx.adaptive_proxgrad(x0, f=fd, g=g, rule=AdaProx.FixedStepsize(gam), tol=0.0, maxit=1, log=log)
        info1 = AdaProx.last_solve_info()
        logo = []
        xo, ito = AdaProx.adaptive_proxgrad(x0, f=fd, g=g, rule=AdaProx.OurRule(gamma=gam_our), tol=0.0, maxit=1, log=logo)
        info2 = AdaProx.last_solve_info()
    assert [i["matrix_passes"] for i in (info0, info1, info2)] == [passes] * 3, "kernel selection"
    assert it == 0 and it2 == 1 and ito == 1
    ok, ratio = within(x, R["X1"][:, 0], R["B1"][:, 0])
    assert ok, ("maxit = 0: x_1", ratio)
    ok, ratio = within_cols(x2[:, None], R["X2"][:, :1], R["B2col"][:1])
    assert ok, ("maxit = 1: x_2", ratio)
    assert len(log) == 1 and log[0]["gamma"] == gam, "FixedStepsize: record 1 carries gamma itself"
    for key, ref, bnd in (("norm_res", "res1", "dres1"), ("objective", "obj1", "dobj1")):
        ok, ratio = within(log[0][key], R[ref][0], R[bnd][0])
        assert ok, (key, ratio)
    O = R["our"]
    ok, ratio = within(logo[0]["gamma"], O["gamma1"], O["dgamma1"])
    assert ok, ("OurRule gamma_1", ratio, logo[0]["gamma"], O["gamma1"])
    ok, ratio = within(xo, O["X2"], O["B2"])
    assert ok, ("OurRule x_2", ratio)


def _device_sm(AdaProx):
    return AdaProx.default_device().info()["sm_count"]


@pytest.mark.gpu
def test_shape_sets_reach_every_branch_on_this_device(AdaProx):
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    if optin != B200_SMEM_OPTIN:
        pytest.skip(f"the grid-resident sizes are restated for B200's {B200_SMEM_OPTIN} B of opt-in shared memory, not {optin}")
    _assert_reaches_everything(_device_sm(AdaProx))


def _fused_env(chunk, helpers):
    env = {"ADAPROX_FUSED": "1"}
    if chunk is not None:
        env["ADAPROX_FUSED_CHUNK"] = chunk
    if helpers:
        env.update(ADAPROX_HELPERS="2", ADAPROX_HELPER_HOLD="0", ADAPROX_HELPER_ROWS="3")
    return env


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(len(FUSED_CASES)))
def test_fused_sweep_matches_extended_precision(AdaProx, k):
    m, n, chunk, helpers = FUSED_CASES[k]
    term = dense_term(m, n)
    fd = AdaProx.LinearLeastSquares(term.M, term.v)
    try:
        _check(AdaProx, fd, term, k, k, _fused_env(chunk, helpers), 1)
    finally:
        fd.mat.free()


TWO_PASS = {"ADAPROX_FUSED": "0", "ADAPROX_RESIDENT": "0", "ADAPROX_GRIDRES": "0"}


@pytest.mark.gpu
@pytest.mark.parametrize("gemv", ["ring", "ldg"])
@pytest.mark.parametrize("k", range(len(DENSE_CASES)))
def test_two_pass_dense_matches_extended_precision(AdaProx, k, gemv):
    m, n, env_grid = DENSE_CASES[k]
    term = dense_term(m, n)
    env = dict(TWO_PASS, ADAPROX_GEMV=gemv)          # read at upload (plan_dense)
    if env_grid:
        env["ADAPROX_GRID"] = env_grid
    with environ(env):
        fd = AdaProx.LinearLeastSquares(term.M, term.v)
    try:
        _check(AdaProx, fd, term, k, 100 + k, env, 2)
    finally:
        fd.mat.free()


def _csr_device(AdaProx, name, kind, lpr):
    X = CSR_MATRICES[name]()
    term = csr_term(name, kind)
    with environ({"ADAPROX_CSR_LPR": lpr or 0}):      # read at upload; 0 = from the mean row length
        fd = AdaProx.LinearLeastSquares(X, term.v) if kind == "lsq" else AdaProx.LogisticLoss(X, term.v)
    return fd, term


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(len(CSR_CASES)))
def test_two_pass_csr_matches_extended_precision(AdaProx, k):
    fd, term = _csr_device(AdaProx, *CSR_CASES[k])
    try:
        _check(AdaProx, fd, term, k, 200 + k, TWO_PASS, 2)
    finally:
        fd.mat.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(len(RESIDENT_CASES)))
def test_cluster_resident_matches_extended_precision(AdaProx, k):
    term = dense_term(*RESIDENT_CASES[k])
    fd = AdaProx.LinearLeastSquares(term.M, term.v)
    try:
        _check(AdaProx, fd, term, k, 300 + k, {"ADAPROX_FUSED": "0", "ADAPROX_RESIDENT": "1"}, 3)
    finally:
        fd.mat.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(len(GRIDRES_CASES)))
def test_grid_resident_matches_extended_precision(AdaProx, k):
    term = dense_term(*GRIDRES_CASES[k])
    fd = AdaProx.LinearLeastSquares(term.M, term.v)
    try:
        _check(AdaProx, fd, term, k, 400 + k, {"ADAPROX_FUSED": "0", "ADAPROX_RESIDENT": "0", "ADAPROX_GRIDRES": "1"}, 4)
    finally:
        fd.mat.free()


# ---------------------------------------------------------------- bit-identical reruns at the largest shape of each family
def _largest(cases, key):
    return max(cases, key=key)


RERUNS = {
    "fused": (lambda: FUSED_CASES[-1][:2], _fused_env("4", True), 1, None),
    "two-pass ring": (lambda: (303105, 8), dict(TWO_PASS, ADAPROX_GEMV="ring"), 2, None),
    "two-pass ldg": (lambda: (1003, 5000), dict(TWO_PASS, ADAPROX_GEMV="ldg"), 2, None),
    "csr": (None, dict(TWO_PASS, ADAPROX_CSR_LPR="32"), 2, ("mixed", "logistic", 32)),
    "resident": (lambda: (416, 1024), {"ADAPROX_FUSED": "0", "ADAPROX_RESIDENT": "1"}, 3, None),
    "grid-resident": (lambda: (4144, 1000), {"ADAPROX_FUSED": "0", "ADAPROX_RESIDENT": "0", "ADAPROX_GRIDRES": "1"}, 4, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(RERUNS))
def test_reruns_are_bit_identical(AdaProx, family):
    shape, env, passes, csr = RERUNS[family]
    if csr:
        fd, term = _csr_device(AdaProx, *csr)
    else:
        term = dense_term(*shape())
        with environ(env):
            fd = AdaProx.LinearLeastSquares(term.M, term.v)
    x0, _, lam, gam_our = _instance(term, 2, 7)
    runs = []
    try:
        with environ(env):
            for _ in range(2):
                log = []
                x, it = AdaProx.adaptive_proxgrad(x0, f=fd, g=AdaProx.NormL1(lam), rule=AdaProx.OurRule(gamma=gam_our), tol=0.0, maxit=12, log=log)
                runs.append((x, it, np.array([(r["gamma"], r["norm_res"], r["objective"]) for r in log]), AdaProx.last_solve_info()))
    finally:
        fd.mat.free()
    (xa, ia, la, fa), (xb, ib, lb, fb) = runs
    assert fa["matrix_passes"] == fb["matrix_passes"] == passes
    if family == "fused":
        assert fa["kernel_launches"] == fb["kernel_launches"] == 2, "the helper CTAs were launched"
    # (12 iterations: the 8-column instance reaches an exact fixed point near iteration 29, where OurRule's 0 / 0 turns x into
    # NaN exactly as the reference does)
    assert ia == ib == 12 and np.array_equal(xa, xb, equal_nan=True) and np.array_equal(la, lb, equal_nan=True)
    assert np.all(np.isfinite(xa)) and la.shape == (12, 3)
