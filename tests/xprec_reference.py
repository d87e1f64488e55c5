"""One and two AdaPGM steps in np.longdouble (64-bit mantissa) and a-priori bounds on the rounding error of a float64 device.

Shared by the batched-path and the single-lambda reference tests; the derivation of the bounds is in the module docstring of
test_gpu_lambda_path_reference.py.  A single solve is the L = 1 column of the same machinery.
"""
import numpy as np

LD = np.longdouble
U = 2.0 ** -53


class Term:
    """f over the matrix M (dense float64 array, m x nf): kind "lsq" (v = b) or "logistic" (v = labels, intercept last)."""

    def __init__(self, kind, M, v):
        self.kind, self.M, self.v = kind, np.asarray(M, dtype=np.float64), np.asarray(v, dtype=np.float64)
        self.m, self.nf = self.M.shape
        self.n = self.nf + (kind == "logistic")
        self.s = 1.0 / self.m if kind == "logistic" else 1.0
        self.Ma = np.abs(self.M)
        self.M_ld, self.v_ld = self.M.astype(LD), self.v.astype(LD)

    def lipschitz(self):
        Mx = np.hstack([self.M, np.ones((self.m, 1))]) if self.kind == "logistic" else self.M
        s2 = np.linalg.norm(Mx, 2) ** 2
        return s2 / (4 * self.m) if self.kind == "logistic" else s2

    def eval(self, W):
        """-> (f [L], P [m, L], G [n, L]) in the dtype of W."""
        M, v = (self.M_ld, self.v_ld) if W.dtype == LD else (self.M, self.v)
        if self.kind == "lsq":
            P = M @ W - v[:, None]
            return 0.5 * np.sum(P * P, axis=0), P, M.T @ P
        logits = M @ W[:-1] + W[-1]
        u = 1 + np.exp(-logits)
        P = 1 / u - v[:, None]
        G = np.empty_like(W)
        G[:-1] = (M.T @ P) / self.m
        G[-1] = P.sum(axis=0) / self.m
        return -np.sum((v[:, None] - 1) * logits - np.log(u), axis=0) / self.m, P, G

    def step(self, W, gam, lam, G=None):
        """-> (x+, v, G, f, P): v = W - gam G, x+ = S_{gam lam}(v)."""
        f, P, G0 = self.eval(W)
        G = G0 if G is None else G
        V = W - gam * G
        return np.sign(V) * np.maximum(np.abs(V) - gam * lam, 0), V, G, f, P

    def dP(self, Wa, dW):
        """bound on the device error of P at |w| <= Wa with an input error <= dW"""
        K1 = self.nf
        if self.kind == "lsq":
            return (K1 + 2) * U * (self.Ma @ Wa + np.abs(self.v)[:, None]) + self.Ma @ dW
        dlog = (K1 + 2) * U * (self.Ma @ Wa[:-1] + Wa[-1]) + self.Ma @ dW[:-1] + dW[-1]
        return 0.25 * dlog + 4 * U

    def dG(self, Wa, dW, Pa, Ga):
        """bound on the device error of the gradient at |w| <= Wa with an input error <= dW"""
        dP = self.dP(Wa, dW)
        dG = np.empty_like(Wa)
        dG[:self.nf] = self.s * (self.Ma.T @ dP + (self.m + 2) * U * (self.Ma.T @ Pa)) + U * Ga[:self.nf]
        if self.kind == "logistic":
            dG[-1] = self.s * (dP.sum(axis=0) + (self.m + 2) * U * Pa.sum(axis=0)) + U * Ga[-1]
        return dG

    def step_bound(self, Wa, dW, Pa, Ga, gam, lam):
        """componentwise bound on |x+_device - x+_ref| and on |v_device - v_ref|"""
        dG = self.dG(Wa, dW, Pa, Ga)
        dV = gam * dG + dW + 2 * U * (Wa + gam * Ga)
        return 2 * (dV + U * gam * lam), 2 * dV, dG

    def value_bound(self, W, Wa, dW):
        """bound on |f_device(w_device) - f_ref(w)| per column"""
        W = W.astype(np.float64)
        if self.kind == "lsq":
            r = np.abs(self.M @ W - self.v[:, None])
            dr = self.dP(Wa, dW)
            return 2 * (np.sum(r * dr + 0.5 * dr * dr, axis=0) + (self.m + 2) * U * 0.5 * np.sum(r * r, axis=0))
        logits = self.M @ W[:-1] + W[-1]
        lu = np.log1p(np.exp(-logits))
        dlog = (self.nf + 2) * U * (self.Ma @ Wa[:-1] + Wa[-1]) + self.Ma @ dW[:-1] + dW[-1]
        term = np.abs((self.v[:, None] - 1) * logits) + lu
        per = (np.abs(self.v[:, None] - 1) + 1) * dlog + 4 * U * (1 + np.abs(logits) + lu)
        return 2 * (np.sum(per, axis=0) + (self.m + 2) * U * np.sum(term, axis=0)) / self.m


def reference(term, X0, gam, lam):
    """Extended-precision x_1, x_2 and the bounds of the device's maxit = 0 / maxit = 1 outputs."""
    W0 = X0.astype(LD)
    g_ld, l_ld = gam.astype(LD), lam.astype(LD)
    X1, V0, G0, f0, P0 = term.step(W0, g_ld, l_ld)
    X2, V1, G1, f1, P1 = term.step(X1, g_ld, l_ld)
    f = lambda a: np.asarray(a, dtype=np.float64)
    zero = np.zeros_like(X0)
    B1, BV0, dG0 = term.step_bound(np.abs(X0), zero, np.abs(f(P0)), np.abs(f(G0)), gam, lam)
    X1a = np.abs(f(X1)) + B1
    B2 = term.step_bound(X1a, zero, np.abs(f(P1)), np.abs(f(G1)), gam, lam)[0]      # the local error of step 2 ...
    dG1 = term.step_bound(X1a, B1, np.abs(f(P1)), np.abs(f(G1)), gam, lam)[2]       # ... and grad f(x_1) with x_1's error
    # record of iteration 1: norm of (v_0 - x_1) / gamma + grad f(x_1), and f(x_1) + lambda |x_1|_1
    pr = f((V0 - X1) / g_ld + G1)
    dpr = (BV0 + B1) / gam + 2 * U * (np.abs(f(V0 - X1)) / gam + np.abs(pr)) + dG1
    res = np.linalg.norm(pr, axis=0)
    dres = 2 * (np.linalg.norm(dpr, axis=0) + (term.n + 2) * U * res)
    df1 = term.value_bound(f(X1), X1a, B1)
    l1 = np.abs(f(X1)).sum(axis=0)
    return dict(X1=f(X1), X2=f(X2), B1=B1, B2col=np.linalg.norm(B1, axis=0) + np.linalg.norm(B2, axis=0),
                f0=f(f0), df0=term.value_bound(X0, np.abs(X0), zero), f1=f(f1), df1=df1,
                res1=res, dres1=dres, obj1=f(f1) + lam * l1, dobj1=df1 + lam * (B1.sum(axis=0) + (term.n + 2) * U * l1),
                ld=dict(X0=W0, X1=X1, G0=G0, G1=G1), dG0=dG0, dG1=dG1)


def within(got, ref, bound):
    """-> (ok, worst ratio |got - ref| / bound)"""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    err = np.abs(got - ref)
    ratio = np.max(err / np.maximum(bound, 1e-300)) if err.size else 0.0
    return bool(np.all(np.isfinite(got)) and np.all(err <= bound)), float(ratio)


def within_cols(got, ref, bound_col):
    err = np.linalg.norm(np.asarray(got, dtype=np.float64) - ref, axis=0)
    return bool(np.all(np.isfinite(got)) and np.all(err <= bound_col)), float(np.max(err / np.maximum(bound_col, 1e-300)))


# ================================================================ the primal-dual extension
# Errors are carried as a pair (e, s): the device's vector differs from the reference's by d1 + d2 with |d1| <= e componentwise
# and |d2|_2 <= s.  Separable maps keep the pair apart; a matrix turns s into a componentwise bound through its row norms;
# the block soft threshold (NormL2) is nonexpansive in the 2-norm only, so its result goes into s.  A componentwise check
# against e + s is then rigorous (|d2_i| <= |d2|_2).  The derivation of every bound is in the module docstring of
# tests/test_gpu_primal_dual_reference.py.

def _a(x):
    return np.abs(np.asarray(x, dtype=np.float64))


def _nrm(x):
    return float(np.linalg.norm(np.asarray(x, dtype=np.float64)))


class Smooth:
    """The smooth term f of a single solve: "lsq" / "logistic" (dense or CSR, through Term), "quadratic" (Q, q), "gram"
    (QuadraticGram: Q = Z Z', Z n x d), "cubic" (Q, q, c) or "zero"."""

    def __init__(self, kind, M=None, v=None, c=0.0, n=None):
        self.kind = kind
        if kind in ("lsq", "logistic"):
            self.term = Term(kind, M, v)
            self.n = self.term.n
        elif kind == "zero":
            self.n = int(n)
        else:
            self.M, self.q, self.c = np.asarray(M, dtype=np.float64), np.asarray(v, dtype=np.float64), float(c)
            self.Ma, self.M_ld, self.q_ld = np.abs(self.M), self.M.astype(LD), self.q.astype(LD)
            self.n = self.M.shape[0]

    def value_grad(self, x):
        """-> (f(x), grad f(x)) in long double"""
        x = np.asarray(x, dtype=LD)
        if self.kind in ("lsq", "logistic"):
            f, _, G = self.term.eval(x[:, None])
            return f[0], G[:, 0]
        if self.kind == "zero":
            return LD(0), np.zeros(self.n, dtype=LD)
        if self.kind == "gram":
            temp = self.M_ld @ (self.M_ld.T @ x)
        else:
            temp = self.M_ld @ x
        if self.kind == "cubic":
            g = temp + self.q_ld + (np.sqrt(np.sum(x * x)) * LD(self.c) / 2) * x
            return (np.sum(x * g) + np.sum(self.q_ld * x)) / 2 - np.sqrt(np.sum(x * x)) ** 3 * LD(self.c) / 12, g
        return np.sum(x * temp) / 2 + np.sum(x * self.q_ld), temp + self.q_ld

    def _temp_err(self, xa, ex):
        """bound on the device error of Q x (Z (Z' x) for the Gram form) and a bound on |Q x|"""
        n = self.n
        if self.kind == "gram":
            d = self.M.shape[1]
            ua = self.Ma.T @ xa
            eu = (n + 2) * U * ua + self.Ma.T @ ex                     # u = Z' x: sums over the n rows, any order
            return (d + 2) * U * (self.Ma @ (ua + eu)) + self.Ma @ eu, self.Ma @ (ua + eu)
        return (n + 2) * U * (self.Ma @ xa) + self.Ma @ ex, self.Ma @ xa

    def _cubic_coef(self, x, xa, ex):
        nx = float(np.sqrt(np.sum(_a(x) ** 2)))
        exx = (self.n + 2) * U * np.sum(xa * xa) + np.sum(2 * xa * ex + ex * ex)
        enx = exx / nx + U * (nx + exx / nx)
        return nx, nx * abs(self.c) / 2, abs(self.c) / 2 * enx + 2 * U * nx * abs(self.c) / 2, enx

    def grad_err(self, x, ex):
        """componentwise bound on |grad f_device(x^) - grad f(x)| for |x^ - x| <= ex"""
        ex = np.asarray(ex, dtype=np.float64) * np.ones(self.n)
        xa = _a(x) + ex
        if self.kind == "zero":
            return np.zeros(self.n)
        if self.kind in ("lsq", "logistic"):
            t = self.term
            _, P, G = t.eval(np.asarray(x, dtype=LD)[:, None])
            return t.dG(xa[:, None], ex[:, None], _a(P), _a(G))[:, 0]
        et, ta = self._temp_err(xa, ex)
        if self.kind == "cubic":
            _, coef, ecoef, _ = self._cubic_coef(x, xa, ex)
            return et + ecoef * xa + coef * ex + 3 * U * (ta + _a(self.q) + coef * xa)
        return et + U * (ta + _a(self.q))

    def value_err(self, x, ex):
        """bound on |f_device(x^) - f(x)| for |x^ - x| <= ex"""
        ex = np.asarray(ex, dtype=np.float64) * np.ones(self.n)
        xa = _a(x) + ex
        n = self.n
        if self.kind == "zero":
            return 0.0
        if self.kind in ("lsq", "logistic"):
            return float(self.term.value_bound(np.asarray(x, dtype=np.float64)[:, None], xa[:, None], ex[:, None])[0])
        et, ta = self._temp_err(xa, ex)
        qa = _a(self.q)
        if self.kind == "cubic":
            nx, coef, ecoef, enx = self._cubic_coef(x, xa, ex)
            ga = ta + qa + coef * xa
            eg = et + ecoef * xa + coef * ex + 3 * U * ga
            s0 = np.sum(xa * eg + ga * ex) + (n + 2) * U * np.sum(xa * ga)
            s1 = np.sum(qa * ex) + (n + 2) * U * np.sum(qa * xa)
            cub = abs(self.c) / 12 * (3 * (nx + enx) ** 2 * enx + 6 * U * nx ** 3)
            return 0.5 * (s0 + s1) + cub + 2 * U * (0.5 * np.sum(xa * (ga + qa)) + abs(self.c) * nx ** 3 / 12)
        s0 = np.sum(xa * et + ta * ex) + (n + 2) * U * np.sum(xa * ta)
        s1 = np.sum(qa * ex) + (n + 2) * U * np.sum(qa * xa)
        return 0.5 * s0 + s1 + 2 * U * (0.5 * np.sum(xa * ta) + np.sum(xa * qa))


class Prox:
    """A prox object: kind "zero" / "indzero" / "l1" / "l2" / "box" (scalar or per-coordinate lo / hi, +-inf allowed), an
    optional Translate shift b (x -> f(x + b)), and conj = the ConvexConjugate of it (prox through Moreau in ProximalCore's
    order u = w / s, p = prox_{f / s}(u), w - s p)."""

    def __init__(self, kind, lam=1.0, lo=0.0, hi=0.0, shift=None, conj=False):
        self.kind, self.lam, self.conj = kind, float(lam), bool(conj)
        self.lo, self.hi = lo, hi
        self.b = None if shift is None else np.asarray(shift, dtype=np.float64)

    def flipped(self):
        """the object whose prox the dual step takes: h* for a plain h, the base function for an h given as a conjugate"""
        return Prox(self.kind, self.lam, self.lo, self.hi, self.b, not self.conj)

    def _b(self, n):
        return np.zeros(n, dtype=LD) if self.b is None else self.b.astype(LD)

    def _base(self, z, tau):
        if self.kind == "zero":
            return z.copy()
        if self.kind == "indzero":
            return np.zeros_like(z)
        if self.kind == "l1":
            gl = LD(tau) * LD(self.lam)
            return np.sign(z) * np.maximum(np.abs(z) - gl, 0)
        if self.kind == "l2":
            nz = np.sqrt(np.sum(z * z))
            return max(LD(0), 1 - LD(self.lam) * LD(tau) / nz) * z
        return np.minimum(np.maximum(z, np.asarray(self.lo, dtype=LD)), np.asarray(self.hi, dtype=LD))

    def _plain(self, v, tau):
        b = self._b(v.size)
        return self._base(v + b, tau) - b

    def prox(self, v, step):
        v = np.asarray(v, dtype=LD)
        if not self.conj:
            return self._plain(v, step)
        if self.b is None and self.kind == "zero":
            return np.zeros_like(v)
        if self.b is None and self.kind == "indzero":
            return v.copy()
        s = LD(step)
        return v - s * self._plain(v / s, 1 / s)

    def _plain_err(self, v, ev, sv, tau, dtau):
        n = v.size
        ba = np.zeros(n) if self.b is None else np.abs(self.b)
        za = _a(v) + ev + sv + ba
        ez = ev + U * za
        if self.kind == "indzero":
            ey, sy = np.zeros(n), 0.0
        elif self.kind in ("zero", "box"):
            ey, sy = ez, sv
        elif self.kind == "l1":
            ey, sy = ez + self.lam * dtau + 2 * U * (za + tau * self.lam), sv
        else:
            ey, sy = np.zeros(n), _nrm(ez) + sv + self.lam * dtau + self.lam * tau * (n / 2 + 6) * U + 2 * U * _nrm(za)
        return ey + U * (za + ba), sy

    def prox_err(self, v, ev, sv, step, dstep=0.0):
        """(e, s) bound on the device's prox_{step f}(v^) - prox_{step f}(v) for v^ = v + (ev, sv) and |step^ - step| <= dstep"""
        v = np.asarray(v, dtype=LD)
        ev = np.asarray(ev, dtype=np.float64) * np.ones(v.size)
        if not self.conj:
            return self._plain_err(v, ev, sv, step, dstep)
        if self.b is None and self.kind == "zero":
            return np.zeros(v.size), 0.0
        if self.b is None and self.kind == "indzero":
            return ev, sv
        s = float(step)
        ua = _a(v) / s
        ep, sp = self._plain_err(v / LD(s), ev / s + U * ua, sv / s, 1 / s, 2 * U / s)
        pa = _a(self._plain(v / LD(s), 1 / LD(s))) + ep + sp
        e, so = ev + s * ep + 2 * U * (_a(v) + s * pa), sv + s * sp
        if dstep:                                   # d/ds prox_{s f*}(w) = b (+ the finite box bounds) in magnitude
            ba = np.zeros(v.size) if self.b is None else np.abs(self.b)
            if self.kind == "l2":
                so += dstep * _nrm(ba)
            else:
                box = 0.0
                if self.kind == "box":
                    fin = lambda t: np.where(np.isfinite(t), np.abs(t), 0.0)
                    box = np.maximum(fin(np.asarray(self.lo, dtype=np.float64)), fin(np.asarray(self.hi, dtype=np.float64)))
                e = e + dstep * (ba + box)
        return e, so

    def value(self, x):
        """f(x) in long double (a conjugate has no value on the device: NaN)"""
        if self.conj:
            return LD(np.nan)
        x = np.asarray(x, dtype=LD)
        z = x + self._b(x.size)
        if self.kind == "zero":
            return LD(0)
        if self.kind == "l1":
            return LD(self.lam) * np.sum(np.abs(z))
        if self.kind == "l2":
            return LD(self.lam) * np.sqrt(np.sum(z * z))
        if self.kind == "indzero":
            return LD(0) if not np.any(z) else LD(np.inf)
        ok = (z >= np.asarray(self.lo, dtype=LD)) & (z <= np.asarray(self.hi, dtype=LD))
        return LD(0) if np.all(ok) else LD(np.inf)

    def value_err(self, x, ex, sx, own_output=False):
        """bound on |f_device(x^) - f(x)|.  An indicator's value is exactly 0 or Inf: the bound is 0, and a point whose distance
        to the set is not decided by the bound is refused (AssertionError).  own_output: x is this object's own prox output
        (an unshifted box or IndZero then holds its point exactly)."""
        x = np.asarray(x, dtype=LD)
        n = x.size
        ex = np.asarray(ex, dtype=np.float64) * np.ones(n)
        if self.conj or self.kind == "zero":
            return 0.0
        ba = np.zeros(n) if self.b is None else np.abs(self.b)
        za = _a(x + self._b(n))
        ez = ex + sx + U * (_a(x) + ba)
        if self.kind == "l1":
            return self.lam * (np.sum(ex + U * (_a(x) + ba)) + np.sqrt(n) * sx + (n + 2) * U * np.sum(za)) + U * float(self.value(x))
        if self.kind == "l2":
            return self.lam * (_nrm(ex + U * (_a(x) + ba)) + sx + (n / 2 + 3) * U * _nrm(za)) + U * float(self.value(x))
        if own_output and self.b is None:
            return 0.0
        z = np.asarray(x + self._b(n), dtype=np.float64)
        if self.kind == "indzero":
            assert np.any(np.abs(z) > ez) or (not np.any(z) and not np.any(ez)), "IndZero: the zero test is not decided by the bound"
            return 0.0
        dist = np.minimum(z - np.asarray(self.lo, dtype=np.float64), np.asarray(self.hi, dtype=np.float64) - z)
        assert np.any(dist < -ez) or np.all(dist > ez), "IndBox: a boundary lies inside the bound"
        return 0.0


class LinMap:
    """The linear map A (dense float64 array; a CSR A is passed densified: zeros add nothing to a bound)."""

    def __init__(self, A):
        self.A = np.asarray(A, dtype=np.float64)
        self.m, self.n = self.A.shape
        self.Aa, self.A_ld = np.abs(self.A), self.A.astype(LD)
        self.rown, self.coln = np.linalg.norm(self.A, axis=1), np.linalg.norm(self.A, axis=0)
        self.norm2 = float(np.linalg.norm(self.A, 2))

    def mv(self, x):
        return self.A_ld @ np.asarray(x, dtype=LD)

    def tmv(self, y):
        return self.A_ld.T @ np.asarray(y, dtype=LD)

    def mv_err(self, x, ex, sx):
        xa = _a(x) + ex + sx
        return (self.n + 2) * U * (self.Aa @ xa) + self.Aa @ ex + self.rown * sx

    def tmv_err(self, y, ey, sy):
        ya = _a(y) + ey + sy
        return (self.m + 2) * U * (self.Aa.T @ ya) + self.Aa.T @ ey + self.coln * sy


def rel_err_D(dx, dg, ex, eg, gam):
    """OurRule's D = gamma L (gamma C - 1) from dx, dg (long double) and their componentwise errors -> (D, |dD| bound) (the
    first-order derivation of tests/test_gpu_single_lambda_reference.py)"""
    a, b, c = np.sum(dg * dg), np.sum(dg * dx), np.sum(dx * dx)
    g = LD(gam)
    if a == 0:                                        # f = Zero: C = L = 0 exactly (0 / 0 -> NaN -> 0), D = 0
        return LD(0), 0.0
    D = g * (b / c) * (g * (a / b) - 1)
    dxa, dga = _a(dx), _a(dg)
    n = dx.size
    a, b, c = float(a), float(b), float(c)
    ea = np.sum(2 * dga * eg + eg * eg) + (n + 2) * U * a
    eb = np.sum(dga * ex + dxa * eg + eg * ex) + (n + 2) * U * np.sum(dga * dxa)
    ec = np.sum(2 * dxa * ex + ex * ex) + (n + 2) * U * c
    gC = gam * a / b
    rD = eb / b + ec / c + (gC * (ea / a + eb / b + 2 * U) + U) / abs(gC - 1) + 4 * U
    return D, abs(float(D)) * rD


def third_term(gam, D, eD, K, m4=1.0):
    """gamma sqrt(m4) / sqrt(2 (D + sqrt(D^2 + K))) and twice its first-order bound: S = D + sqrt(D^2 + K) has
    |dS| / S <= |dD| / sqrt(D^2 + K) (+ rounding)."""
    S = D + np.sqrt(D * D + LD(K))
    if not S > 0:
        return LD(np.inf), 0.0
    t3 = LD(gam) * np.sqrt(LD(m4)) / np.sqrt(2 * S)
    rS = eD / float(np.sqrt(D * D + LD(K))) + 6 * U
    return t3, 2 * (0.5 * rS + 8 * U) * float(t3)


def decided_min(terms):
    """terms: [(value, bound)] -> (min, its bound); refuses a case in which two terms are closer than their bounds"""
    for i in range(len(terms)):
        for j in range(i + 1, len(terms)):
            (vi, ei), (vj, ej) = terms[i], terms[j]
            if np.isfinite(float(vi)) and np.isfinite(float(vj)):
                assert abs(float(vi) - float(vj)) > ei + ej, ("the minimum is not decided by the bounds", float(vi), float(vj))
    k = min(range(len(terms)), key=lambda i: float(terms[i][0]))
    return terms[k]


class PD:
    """One primal-dual problem f(x) + g(x) + h(A x); A = None: AdaPGM (h unused)."""

    def __init__(self, f, g, h=None, A=None):
        self.f, self.g, self.h, self.A = f, g, h, A
        self.hs = h.flipped() if h is not None else None

    def prologue(self, x0, y0, gam):
        """x_1 = prox_{gam g}(x_0 - gam (grad f(x_0) + A' y_0)) and everything the first iteration needs"""
        f, A = self.f, self.A
        S = dict(X0=np.asarray(x0, dtype=LD), gam=gam)
        S["f0"], S["G0"] = f.value_grad(S["X0"])
        S["eG0"] = f.grad_err(S["X0"], 0.0)
        n = f.n
        if A is not None:
            S["Y0"] = np.asarray(y0, dtype=LD)
            S["AX0"], S["eAX0"] = A.mv(S["X0"]), A.mv_err(S["X0"], np.zeros(n), 0.0)
            S["ATY0"], S["eATY0"] = A.tmv(S["Y0"]), A.tmv_err(S["Y0"], np.zeros(A.m), 0.0)
        else:
            S["ATY0"], S["eATY0"] = np.zeros(n, dtype=LD), np.zeros(n)
        S["V0"] = S["X0"] - LD(gam) * (S["G0"] + S["ATY0"])
        S["eV0"] = gam * (S["eG0"] + S["eATY0"]) + 3 * U * (_a(x0) + gam * (_a(S["G0"]) + _a(S["ATY0"])))
        S["X1"] = self.g.prox(S["V0"], gam)
        S["e1"], S["s1"] = self.g.prox_err(S["V0"], S["eV0"], 0.0, gam)
        S["f1"], S["G1"] = f.value_grad(S["X1"])
        x1e = S["e1"] + S["s1"]
        S["eG1"] = f.grad_err(S["X1"], x1e)
        S["df1"] = f.value_err(S["X1"], x1e)
        if A is not None:
            S["AX1"], S["eAX1"] = A.mv(S["X1"]), A.mv_err(S["X1"], S["e1"], S["s1"])
        return S

    def dual(self, S, gam1, dgam1, sig, dsig):
        """w = y_0 + sig ((1 + rho) A x_1 - rho A x_0), y_1 = prox_{sig h*}(w), A' y_1, with rho = gam1 / gam"""
        A, gam = self.A, S["gam"]
        rho = LD(gam1) / LD(gam)
        drho = dgam1 / gam + U * float(rho)
        s = LD(sig)
        comb = (1 + rho) * S["AX1"] - rho * S["AX0"]
        W = S["Y0"] + s * comb
        r = float(rho)
        eW = (sig * ((1 + r) * S["eAX1"] + r * S["eAX0"]) + dsig * _a(comb) + drho * sig * (_a(S["AX1"]) + _a(S["AX0"])) +
              4 * U * (_a(S["Y0"]) + sig * ((1 + r) * _a(S["AX1"]) + r * _a(S["AX0"]))))
        Y1 = self.hs.prox(W, sig)
        ey, sy = self.hs.prox_err(W, eW, 0.0, sig, dsig)
        return dict(W=W, eW=eW, Y1=Y1, ey1=ey, sy1=sy, ATY1=A.tmv(Y1), eATY1=A.tmv_err(Y1, ey, sy))

    def record(self, S, D, gam0, sig):
        """record 1: norm_res (primal residual with gam0, dual residual with sig) and the objective f(x_1) + g(x_1) + h(A x_1)"""
        n = self.f.n
        PR = (S["V0"] - S["X1"]) / LD(gam0) + S["G1"] + S["ATY0"]
        ePR = ((S["eV0"] + S["e1"]) / gam0 + S["eG1"] + S["eATY0"] +
               3 * U * (_a(S["V0"] - S["X1"]) / gam0 + _a(S["G1"]) + _a(S["ATY0"])))
        dpr = _nrm(ePR) + S["s1"] / gam0
        sq = np.sum(PR * PR)
        ddr, m = 0.0, 0
        if D is not None:
            DR = (D["W"] - D["Y1"]) / LD(sig) - S["AX1"]
            eDR = (D["eW"] + D["ey1"]) / sig + S["eAX1"] + 3 * U * (_a(D["W"] - D["Y1"]) / sig + _a(S["AX1"]))
            ddr = _nrm(eDR) + D["sy1"] / sig
            sq = sq + np.sum(DR * DR)
            m = self.A.m
        res = float(np.sqrt(sq))
        dres = dpr + ddr + (n + m + 6) * U * res
        obj = S["f1"] + self.g.value(S["X1"])
        dobj = S["df1"] + self.g.value_err(S["X1"], S["e1"], S["s1"], own_output=True)
        if self.A is not None:
            obj = obj + (self.h.value(S["AX1"]) if not self.h.conj else LD(np.nan))
            dobj += self.h.value_err(S["AX1"], S["eAX1"], 0.0)
        objf = float(obj)
        return dict(res1=res, dres1=dres, obj1=objf, dobj1=dobj + (2 * U * abs(objf) if np.isfinite(objf) else 0.0))

    def primal(self, S, D, gam1, dgam1):
        """x_2 = prox_{gam1 g}(x_1 - gam1 (grad f(x_1) + A' y_1))"""
        ATY1, eATY1 = (D["ATY1"], D["eATY1"]) if D is not None else (S["ATY0"], S["eATY0"])
        gsum = S["G1"] + ATY1
        V1 = S["X1"] - LD(gam1) * gsum
        eV1 = (S["e1"] + gam1 * (S["eG1"] + eATY1) + dgam1 * _a(gsum) +
               3 * U * (_a(S["X1"]) + gam1 * (_a(S["G1"]) + _a(ATY1))))
        X2 = self.g.prox(V1, gam1)
        e2, s2 = self.g.prox_err(V1, eV1, S["s1"], gam1, dgam1)
        return X2, e2 + s2

    def ourrule(self, S, t, norm_A, Theta=1.2):
        """gamma_1 of OurRule (delta = 0) after the prologue with gamma = S["gam"], and its first-order bound"""
        gam = S["gam"]
        dx, dg = S["X1"] - S["X0"], S["G1"] - S["G0"]
        ex = S["e1"] + S["s1"] + U * _a(dx)
        eg = S["eG0"] + S["eG1"] + U * _a(dg)
        D, eD = rel_err_D(dx, dg, ex, eg, gam)
        f64 = np.float64
        xi = (f64(t) * f64(t)) * (f64(gam) * f64(gam)) * (f64(norm_A) * f64(norm_A))      # the device's own float64 bits
        m4 = f64(1.0) - f64(4.0) * xi * (f64(1.0) * f64(1.0))
        t1 = LD(gam) * np.sqrt(LD(2))
        terms = [(t1, 8 * U * float(t1)), third_term(gam, D, eD, LD(xi) * LD(m4), m4)]
        if norm_A > 0:
            terms.append((LD(f64(1.0) / (f64(2.0) * f64(Theta) * f64(t) * f64(norm_A))), 0.0))
        return decided_min(terms)


def pd_fixed(P, x0, y0, gam, t):
    """maxit = 0 / maxit = 1 of adaptive_primal_dual with FixedStepsize(gam, t): rho = 1 exactly, sigma = gam (t t) in float64"""
    S = P.prologue(x0, y0, gam)
    sig = float(np.float64(gam) * (np.float64(t) * np.float64(t)))
    D = P.dual(S, gam, 0.0, sig, 0.0) if P.A is not None else None
    X2, B2 = P.primal(S, D, gam, 0.0)
    R = dict(S=S, D=D, X1=S["X1"], B1=S["e1"] + S["s1"], X2=X2, B2=B2, sigma=sig)
    R.update(P.record(S, D, gam, sig))
    return R


def pd_ourrule(P, x0, y0, gam, t, norm_A):
    """one OurRule step: gamma_1 (first-order bound), then y_1 and x_2"""
    S = P.prologue(x0, y0, gam)
    g1, dg1 = P.ourrule(S, t, norm_A)
    g1f = float(g1)
    tt = float(t) * float(t)
    sig, dsig = g1f * tt, dg1 * tt + U * g1f * tt
    D = P.dual(S, g1f, dg1, sig, dsig) if P.A is not None else None
    X2, B2 = P.primal(S, D, g1f, dg1)
    return dict(S=S, D=D, gamma1=g1f, dgamma1=dg1, X2=X2, B2=B2)


def pd_linesearch(P, x0, y0, gam, eta, t, delta=1e-8, Theta=1.2, r=2.0, R=0.95):
    """the first iteration of AdaPDM+ (k_primal_dual<true>): the trials of the linesearch, gamma_1, y_1, A' y_1 and x_2.
    eta and the second term of the min are float64 operations the device repeats bit for bit; a trial whose test
    eta >= |A'y+ - A'y| / |y+ - y| is not decided by the bound is refused."""
    f64 = np.float64
    S = P.prologue(x0, y0, gam)
    dx, dg = S["X1"] - S["X0"], S["G1"] - S["G0"]
    D_, eD = rel_err_D(dx, dg, S["e1"] + S["s1"] + U * _a(dx), S["eG0"] + S["eG1"] + U * _a(dg), gam)
    d1 = f64(1.0) + f64(delta)
    xib = (f64(t) * f64(t)) * (f64(gam) * f64(gam)) * (f64(eta) * f64(eta)) * (d1 * d1)
    m4 = f64(1.0) - f64(4.0) * xib
    eta = f64(R) * f64(eta)
    n, m = P.f.n, P.A.m
    trials = []
    while True:
        t1 = LD(gam) * np.sqrt(LD(2))
        K = LD(m4) * LD((f64(t) * eta * f64(gam)) ** 2)
        S3 = D_ + np.sqrt(D_ * D_ + K)
        t3 = LD(gam) * np.sqrt(LD(m4) / (2 * LD(d1) * S3))
        rS = eD / float(np.sqrt(D_ * D_ + K)) + 6 * U
        terms = [(t1, 8 * U * float(t1)), (LD(f64(1.0) / (f64(2.0) * f64(Theta) * f64(t) * eta)), 0.0),
                 (t3, 2 * (0.5 * rS + 8 * U) * float(t3))]
        gn, dgn = decided_min(terms)
        gnf = float(gn)
        tt = float(t) * float(t)
        sig, dsig = gnf * tt, dgn * tt + U * gnf * tt
        Dd = P.dual(S, gnf, dgn, sig, dsig)
        dAty = Dd["ATY1"] - S["ATY0"]
        dy = Dd["Y1"] - S["Y0"]
        nA, ny = _nrm(dAty), _nrm(dy)
        eA = _nrm(Dd["eATY1"] + S["eATY0"] + U * _a(dAty)) + (n + 4) * U * nA
        ey = _nrm(Dd["ey1"] + U * _a(dy)) + Dd["sy1"] + (m + 4) * U * ny
        ratio = nA / ny
        dratio = 2 * ratio * (eA / nA + ey / ny + 4 * U)
        assert abs(float(eta) - ratio) > dratio, ("the linesearch test is not decided by the bound", float(eta), ratio, dratio)
        trials.append((float(eta), ratio, dratio))
        if eta >= ratio:
            break
        eta = eta * f64(r)
    X2, B2 = P.primal(S, Dd, gnf, dgn)
    return dict(S=S, D=Dd, trials=len(trials), tests=trials, gamma1=gnf, dgamma1=dgn, sigma1=sig, X2=X2, B2=B2)


def mp_reference(P, x0, y0, sigma0, t):
    """the first iteration of malitsky_pock: y_1, the backtracking (sigma, gamma and the trial count exact: float64 halvings),
    x_1 and record 1.  f(x) - f(x_prev) cancels: its bound is that of the difference, and a trial whose test
    lhs > 0.95 |x - x_prev|^2 is not decided by the bound is refused."""
    f64 = np.float64
    f, g, A = P.f, P.g, P.A
    n, m = f.n, A.m
    S = dict(X0=np.asarray(x0, dtype=LD), Y0=np.asarray(y0, dtype=LD))
    S["f0"], S["G0"] = f.value_grad(S["X0"])
    eG0, df0 = f.grad_err(S["X0"], 0.0), f.value_err(S["X0"], 0.0)
    AX0, eAX0 = A.mv(S["X0"]), A.mv_err(S["X0"], np.zeros(n), 0.0)
    ATY0, eATY0 = A.tmv(S["Y0"]), A.tmv_err(S["Y0"], np.zeros(m), 0.0)
    s0 = f64(sigma0)
    W = S["Y0"] + LD(s0) * AX0
    eW = float(s0) * eAX0 + 2 * U * (_a(S["Y0"]) + float(s0) * _a(AX0))
    Y1 = P.hs.prox(W, float(s0))
    ey, sy = P.hs.prox_err(W, eW, 0.0, float(s0))
    ATY1, eATY1 = A.tmv(Y1), A.tmv_err(Y1, ey, sy)
    sigma = s0 * np.sqrt(f64(2.0))
    tests = []
    while True:
        th = sigma / s0
        gam = f64(t) * f64(t) * sigma
        gf, thf = float(gam), float(th)
        bar = (1 + LD(th)) * ATY1 - LD(th) * ATY0
        ebar = (1 + thf) * eATY1 + thf * eATY0 + 3 * U * ((1 + thf) * _a(ATY1) + thf * _a(ATY0))
        V = S["X0"] - LD(gam) * (bar + S["G0"])
        eV = gf * (ebar + eG0) + 3 * U * (_a(S["X0"]) + gf * (_a(bar) + _a(S["G0"])))
        X = g.prox(V, gf)
        ex, sx = g.prox_err(V, eV, 0.0, gf)
        xe = ex + sx
        d = X - S["X0"]
        nd = _nrm(d)
        edd = _nrm(xe + U * _a(d))
        e_dd = 2 * nd * edd + edd ** 2 + (n + 2) * U * nd ** 2
        AX, eAX = A.mv(X), A.mv_err(X, ex, sx)
        dA = AX - AX0
        na = _nrm(dA)
        eda = _nrm(eAX + eAX0 + U * _a(dA))
        e_aa = 2 * na * eda + eda ** 2 + (m + 2) * U * na ** 2
        fX, _ = f.value_grad(X)
        gd = np.sum(S["G0"] * d)
        e_gd = float(np.sum(eG0 * (_a(d) + xe) + _a(S["G0"]) * (xe + U * _a(d)))) + (n + 2) * U * float(np.sum(_a(S["G0"] * d)))
        e_f = f.value_err(X, xe) + df0 + U * (abs(float(fX)) + abs(float(S["f0"])))
        lhs = LD(gam) * LD(sigma) * np.sum(dA * dA) + 2 * LD(gam) * (fX - S["f0"] - gd)
        rhs = LD(0.95) * np.sum(d * d)
        inner = abs(float(fX - S["f0"])) + abs(float(gd))
        e_lhs = gf * float(sigma) * e_aa + 2 * gf * (e_f + e_gd) + 6 * U * (gf * float(sigma) * na ** 2 + 2 * gf * inner)
        e_rhs = 0.95 * e_dd + 2 * U * float(rhs)
        tests.append((float(lhs), float(rhs), e_lhs + e_rhs))
        assert abs(float(lhs - rhs)) > e_lhs + e_rhs, ("the backtracking test is not decided by the bound", float(lhs), float(rhs))
        if not lhs > rhs:
            break
        sigma = sigma / f64(2.0)
    fX, G = f.value_grad(X)
    eG = f.grad_err(X, xe)
    PR = (V - X) / LD(gam) + G + ATY1
    ePR = (eV + ex) / gf + eG + eATY1 + 3 * U * (_a(V - X) / gf + _a(G) + _a(ATY1))
    DR = (W - Y1) / LD(s0) - AX
    eDR = (eW + ey) / float(s0) + eAX + 3 * U * (_a(W - Y1) / float(s0) + _a(AX))
    res = float(np.sqrt(np.sum(PR * PR) + np.sum(DR * DR)))
    dres = _nrm(ePR) + sx / gf + _nrm(eDR) + sy / float(s0) + (n + m + 6) * U * res
    obj = fX + g.value(X) + P.h.value(AX)
    dobj = f.value_err(X, xe) + g.value_err(X, ex, sx, own_output=True) + P.h.value_err(AX, eAX, 0.0)
    objf = float(obj)
    return dict(sigma=float(sigma), gamma=float(gam), trials=len(tests), tests=tests, X1=X, B1=xe, Y1=Y1, BY1=ey + sy,
                res1=res, dres1=dres, obj1=objf, dobj1=dobj + (2 * U * abs(objf) if np.isfinite(objf) else 0.0))
