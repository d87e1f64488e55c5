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

    def step_bound(self, Wa, dW, Pa, Ga, gam, lam):
        """componentwise bound on |x+_device - x+_ref| and on |v_device - v_ref|"""
        dP = self.dP(Wa, dW)
        dG = np.empty_like(Wa)
        dG[:self.nf] = self.s * (self.Ma.T @ dP + (self.m + 2) * U * (self.Ma.T @ Pa)) + U * Ga[:self.nf]
        if self.kind == "logistic":
            dG[-1] = self.s * (dP.sum(axis=0) + (self.m + 2) * U * Pa.sum(axis=0)) + U * Ga[-1]
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
