"""Host-side mirror of the reference's operator / solver interface.

Same entry points, keyword names, defaults and error behaviour as
``AdaProx`` (src/AdaProx.jl) and the oracle structs of the experiment scripts;
the arithmetic happens in libadaprox_cuda.so.  Julia reaches the same C ABI
with ``ccall`` (julia/AdaProxCUDA.jl, INTEGRATION.md); this module is the
stand-in that can run in this image, so the parity tests read like the
reference's own tests.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _lib as L

F64 = np.float64


def _dp(a):
    return a.ctypes.data_as(L.c_dp)


def _vec(a, n=None):
    a = np.ascontiguousarray(a, dtype=F64).ravel()
    if n is not None and a.shape[0] != n:
        raise ValueError(f"expected a vector of length {n}, got {a.shape[0]}")
    return a


# --------------------------------------------------------------------------
# device handle
# --------------------------------------------------------------------------

class Device:
    """One adaprox_handle bound to one CUDA device."""

    def __init__(self, device=None):
        self.lib = L.load()
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        h = C.c_void_p()
        rc = self.lib.adaprox_create(C.byref(h), int(device))
        if rc != 0:
            raise L.AdaproxError(rc, "adaprox_create failed (no usable CUDA device? there is no CPU fallback)")
        self.h = h
        self.device = int(device)
        self.launches = 0

    def check(self, rc):
        if rc != 0:
            raise L.AdaproxError(rc, self.lib.adaprox_last_error(self.h).decode())

    def info(self):
        sm, ma, mi, fr = C.c_int(), C.c_int(), C.c_int(), C.c_int64()
        self.check(self.lib.adaprox_device_info(self.h, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(fr)))
        return dict(sm_count=sm.value, cc=(ma.value, mi.value), free_bytes=fr.value)

    # -- communicator (row-sharded multi-GPU) --
    def comm_unique_id(self):
        buf = C.create_string_buffer(128)
        rc = self.lib.adaprox_comm_unique_id(buf)
        if rc != 0:
            raise L.AdaproxError(rc, "adaprox_comm_unique_id failed (libnccl not loadable?)")
        return buf.raw

    def comm_init(self, nranks, rank, unique_id: bytes):
        buf = C.create_string_buffer(unique_id, 128)
        self.check(self.lib.adaprox_comm_init(self.h, int(nranks), int(rank), buf))

    def p2p_export(self, n_max) -> bytes:
        """allocate this rank's peer-visible exchange block (vectors up to n_max) and return its 64-byte CUDA IPC handle"""
        buf = C.create_string_buffer(64)
        self.check(self.lib.adaprox_p2p_export(self.h, int(n_max), buf))
        return buf.raw

    def p2p_attach(self, nranks, rank, handles: bytes):
        buf = C.create_string_buffer(handles, 64 * int(nranks))
        self.check(self.lib.adaprox_p2p_attach(self.h, int(nranks), int(rank), buf))

    def p2p_reset(self):
        """After a sharded solve failed with ADAPROX_ERR_COMM: clear this rank's exchange flags (every rank, then a host barrier)."""
        self.check(self.lib.adaprox_p2p_reset(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.lib.adaprox_destroy(self.h)
            self.h = None


_default = None


def default_device():
    global _default
    if _default is None:
        _default = Device()
    return _default


def set_default_device(dev):
    global _default
    _default = dev


class DeviceVector:
    def __init__(self, v=None, dev=None, _id=None, _len=None):
        self.dev = dev or default_device()
        if _id is not None:
            self.id, self.len = _id, _len
            return
        v = _vec(v)
        out = L.c_id()
        self.dev.check(self.dev.lib.adaprox_vector_upload(self.dev.h, _dp(v), v.shape[0], C.byref(out)))
        self.id, self.len = out.value, v.shape[0]

    def download(self):
        out = np.empty(self.len, dtype=F64)
        self.dev.check(self.dev.lib.adaprox_vector_download(self.dev.h, self.id, _dp(out), self.len))
        return out


class DeviceMatrix:
    """A matrix resident in HBM.  Accepts numpy arrays (Fortran order = Julia's
    layout, or C order) and scipy.sparse matrices (converted to CSR)."""

    def __init__(self, A=None, dev=None, _id=None, _shape=None):
        self.dev = dev or default_device()
        lib, h = self.dev.lib, self.dev.h
        if _id is not None:
            self.id, self.shape = _id, _shape
            return
        out = L.c_id()
        if hasattr(A, "tocsr"):
            S = A.tocsr()
            S.sort_indices()
            rp = np.ascontiguousarray(S.indptr, dtype=np.int64)
            ci = np.ascontiguousarray(S.indices, dtype=np.int32)
            va = np.ascontiguousarray(S.data, dtype=F64)
            self.dev.check(lib.adaprox_matrix_upload_csr(h, S.shape[0], S.shape[1], va.shape[0],
                                                         rp.ctypes.data_as(C.POINTER(C.c_int64)),
                                                         ci.ctypes.data_as(C.POINTER(C.c_int32)), _dp(va), C.byref(out)))
            self.shape = tuple(S.shape)
        else:
            A = np.asarray(A, dtype=F64)
            if A.ndim != 2:
                raise ValueError("a matrix is required")
            m, n = A.shape
            if A.flags.f_contiguous and not A.flags.c_contiguous:
                self.dev.check(lib.adaprox_matrix_upload_colmajor(h, _dp(A), m, n, m, C.byref(out)))
            else:
                A = np.ascontiguousarray(A)
                self.dev.check(lib.adaprox_matrix_upload_rowmajor(h, _dp(A), m, n, n, C.byref(out)))
            self.shape = (m, n)
        self.id = out.value

    def set_shard(self, m_global, row0):
        self.dev.check(self.dev.lib.adaprox_matrix_set_shard(self.dev.h, self.id, int(m_global), int(row0)))

    def free(self):
        if self.id:
            self.dev.lib.adaprox_matrix_free(self.dev.h, self.id)
            self.id = 0

    # `A * x`, `A' * y`
    def __matmul__(self, x):
        x = _vec(x, self.shape[1])
        out = np.empty(self.shape[0], dtype=F64)
        self.dev.check(self.dev.lib.adaprox_mul(self.dev.h, self.id, _dp(x), _dp(out)))
        return out

    @property
    def T(self):
        return _Adjoint(self)

    def time_path_gemm(self, L_cols, which, reps=5):
        """mean device ms of one DMMA contraction of the lambda-path solver (0: R = A X - b, 1: G = A' R) on L_cols columns"""
        ms = C.c_double()
        self.dev.check(self.dev.lib.adaprox_time_path_gemm(self.dev.h, self.id, int(L_cols), int(which), int(reps), C.byref(ms)))
        return ms.value

    def time_kernel(self, which, reps=5):
        ms = C.c_double()
        self.dev.check(self.dev.lib.adaprox_time_kernel(self.dev.h, self.id, int(which), int(reps), C.byref(ms)))
        return ms.value


class _Adjoint:
    def __init__(self, M):
        self.M = M

    def __matmul__(self, y):
        M = self.M
        y = _vec(y, M.shape[0])
        out = np.empty(M.shape[1], dtype=F64)
        M.dev.check(M.dev.lib.adaprox_amul(M.dev.h, M.id, _dp(y), _dp(out)))
        return out


def _as_matrix(A, dev=None):
    return A if isinstance(A, DeviceMatrix) else DeviceMatrix(A, dev=dev)


def _as_vector(v, dev=None):
    return v if isinstance(v, DeviceVector) else DeviceVector(v, dev=dev)


# --------------------------------------------------------------------------
# Counting (src/counting.jl)
# --------------------------------------------------------------------------

_counting_enabled = True


def is_counting_enabled():
    return _counting_enabled


class without_counting:
    def __enter__(self):
        global _counting_enabled
        _counting_enabled = False

    def __exit__(self, *exc):
        global _counting_enabled
        _counting_enabled = True
        return False


class Counting:
    """src/counting.jl:16-33."""

    def __init__(self, f):
        self.f = f
        self.eval_count = 0
        self.grad_count = 0
        self.prox_count = 0
        self.mul_count = 0
        self.amul_count = 0

    def __call__(self, *args):
        return self.f(*args)

    def __matmul__(self, x):
        if is_counting_enabled():
            self.mul_count += 1
        return self.f @ x

    @property
    def T(self):
        return _AdjointCounting(self)


class _AdjointCounting:
    def __init__(self, op):
        self.op = op

    def __matmul__(self, x):
        if is_counting_enabled():
            self.op.amul_count += 1
        return self.op.f.T @ x


def _unwrap(o):
    return (o.f, True) if isinstance(o, Counting) else (o, False)


def _cnt(c, name):
    return getattr(c, name) if isinstance(c, Counting) else None


def grad_count(c):
    return _cnt(c, "grad_count")


def prox_count(c):
    return _cnt(c, "prox_count")


def mul_count(c):
    return _cnt(c, "mul_count")


def amul_count(c):
    return _cnt(c, "amul_count")


def eval_count(c):
    return _cnt(c, "eval_count")


# --------------------------------------------------------------------------
# smooth terms (the experiment scripts' oracle structs, same field names)
# --------------------------------------------------------------------------

class _Smooth:
    kind = None
    mat = None
    vec = None
    c = 0.0
    ipar = 0
    n = None

    def _problem(self, n):
        p = L.Problem()
        p.f_kind = self.kind
        p.f_ipar = int(self.ipar)
        p.f_mat = self.mat.id if self.mat is not None else 0
        p.f_vec = self.vec.id if self.vec is not None else 0
        p.f_c = float(self.c)
        p.n = int(n)
        return p

    def _dev(self):
        return self.mat.dev if self.mat is not None else default_device()

    def eval_with_pullback(self, x):
        """AdaProx.eval_with_pullback (src/AdaProx.jl:11): the value costs one
        matrix pass; calling the pullback costs the transposed pass."""
        x = _vec(x, self.n)
        dev = self._dev()
        p = self._problem(x.shape[0])
        fx = C.c_double()
        dev.check(dev.lib.adaprox_eval_f(dev.h, C.byref(p), _dp(x), C.byref(fx), None))

        def pullback():
            g = np.empty_like(x)
            dev.check(dev.lib.adaprox_eval_f(dev.h, C.byref(p), _dp(x), C.byref(fx), _dp(g)))
            return g

        return F64(fx.value), pullback

    def __call__(self, x):
        return self.eval_with_pullback(x)[0]


class LinearLeastSquares(_Smooth):
    """experiments/lasso/runme.jl:16-27."""
    kind = L.F_LEAST_SQUARES

    def __init__(self, A, b, dev=None):
        self.A = A
        self.b = b
        self.mat = _as_matrix(A, dev)
        self.vec = _as_vector(b, self.mat.dev)
        self.n = self.mat.shape[1]


class LogisticLoss(_Smooth):
    """experiments/sparse_logreg/runme.jl:18-39 (w[end] is the intercept)."""
    kind = L.F_LOGISTIC

    def __init__(self, X, y, dev=None):
        self.X = X
        self.y = y
        self.mat = _as_matrix(X, dev)
        self.vec = _as_vector(y, self.mat.dev)
        self.n = self.mat.shape[1] + 1


class Quadratic(_Smooth):
    """experiments/dual_svm/runme.jl:19-28 (Q symmetric)."""
    kind = L.F_QUADRATIC

    def __init__(self, Q, q, dev=None):
        self.Q = Q
        self.q = q
        self.mat = _as_matrix(Q, dev)
        self.vec = _as_vector(q, self.mat.dev)
        self.n = self.mat.shape[1]


class QuadraticGram(_Smooth):
    """`Quadratic(Z * Z', q)` of experiments/dual_svm/runme.jl:19-28 given by its factor: the script builds
    `Q = Dy * X * X' * Dy` (:47-49), i.e. Z = Dy * X (N x d).  `Q * x` is evaluated as `Z * (Z' * x)`: two sweeps over Z
    (16 N d bytes) instead of one over the N x N matrix (8 N^2 bytes); same value up to rounding.  A row shard of Z
    (`set_shard`) needs `n` = the global number of rows."""
    kind = L.F_QUADRATIC_GRAM

    def __init__(self, Z, q, dev=None):
        self.Z = Z
        self.q = q
        self.mat = _as_matrix(Z, dev)
        self.vec = _as_vector(q, self.mat.dev)
        self.n = self.vec.len


class Cubic(_Smooth):
    """experiments/cubic_sparse_logreg/runme.jl:20-32."""
    kind = L.F_CUBIC

    def __init__(self, Q, q, c, dev=None):
        self.Q = Q
        self.q = q
        self.c = float(c)
        self.mat = _as_matrix(Q, dev)
        self.vec = _as_vector(q, self.mat.dev)
        self.n = self.mat.shape[1]


def logistic_loss_grad_Hessian(X, y, w, dev=None):
    """experiments/cubic_sparse_logreg/runme.jl:34-45: ``H, g`` of the logistic loss at ``w`` (intercept last), the setup
    of the Cubic oracle ``Cubic(H, g, lam)`` (:66-67).  X: dense / scipy.sparse / DeviceMatrix with n columns; H is
    (n+1) x (n+1), g has n+1 entries.  Computed on the device (csrc/hessian.inl)."""
    mat = _as_matrix(X, dev)
    vec = _as_vector(y, mat.dev)
    n1 = mat.shape[1] + 1
    w = _vec(w, n1)
    H = np.empty((n1, n1), dtype=F64)
    g = np.empty(n1, dtype=F64)
    mat.dev.check(mat.dev.lib.adaprox_logistic_grad_hessian(mat.dev.h, mat.id, vec.id, _dp(w), _dp(H), _dp(g)))
    mat.dev.launches += 2
    return H, g


class WorstQuadratic(_Smooth):
    """experiments/nesterov_worst_case/runme.jl:14-40."""
    kind = L.F_WORST_QUADRATIC

    def __init__(self, k, L_):
        self.k = int(k)
        self.L = float(L_)
        self.ipar = self.k
        self.c = self.L


class Simple2DObjective(_Smooth):
    """test/runtests.jl:6-13."""
    kind = L.F_SIMPLE2D
    n = 2


# --------------------------------------------------------------------------
# nonsmooth terms (ProximalCore / ProximalOperators objects)
# --------------------------------------------------------------------------

class _ProxObj:
    kind = L.P_ZERO
    lam = 1.0
    lo = 0.0
    hi = 0.0
    lo_vec = None
    hi_vec = None
    shift = None
    conjugate = 0

    def _desc(self):
        p = L.Prox()
        p.kind = self.kind
        p.conjugate = int(self.conjugate)
        p.lam = float(self.lam)
        p.lo, p.hi = float(self.lo), float(self.hi)
        p.lo_vec = self.lo_vec.id if self.lo_vec is not None else 0
        p.hi_vec = self.hi_vec.id if self.hi_vec is not None else 0
        p.shift = self.shift.id if self.shift is not None else 0
        return p


class Zero(_ProxObj, _Smooth):
    """ProximalCore.Zero; also the zero smooth term of the LAD / square-root
    lasso scripts (least_absolute_deviation/runme.jl:18-21)."""
    kind = L.P_ZERO

    def __call__(self, x):
        return F64(0.0)

    def eval_with_pullback(self, x):
        x = np.asarray(x, dtype=F64)
        return F64(0.0), (lambda: np.zeros_like(x))

    def _problem(self, n):
        p = L.Problem()
        p.f_kind = L.F_ZERO
        p.n = int(n)
        return p


class IndZero(_ProxObj):
    kind = L.P_IND_ZERO

    def __call__(self, x):
        return F64(0.0) if not np.any(x) else F64(np.inf)


class NormL1(_ProxObj):
    kind = L.P_NORM_L1

    def __init__(self, lam=1.0):
        self.lam = float(lam)

    def __call__(self, x):
        return F64(self.lam) * F64(np.sum(np.abs(x)))


class NormL2(_ProxObj):
    kind = L.P_NORM_L2

    def __init__(self, lam=1.0):
        self.lam = float(lam)

    def __call__(self, x):
        return F64(self.lam) * F64(np.sqrt(np.dot(x, x)))


class IndBox(_ProxObj):
    kind = L.P_IND_BOX

    def __init__(self, lo, hi, dev=None):
        self._lo, self._hi = lo, hi
        if np.isscalar(lo) and np.isscalar(hi):
            self.lo, self.hi = float(lo), float(hi)
        else:
            n = max(np.size(lo), np.size(hi))
            self.lo_vec = DeviceVector(np.broadcast_to(np.asarray(lo, dtype=F64), (n,)), dev=dev)
            self.hi_vec = DeviceVector(np.broadcast_to(np.asarray(hi, dtype=F64), (n,)), dev=dev)

    def __call__(self, x):
        return F64(0.0) if np.all((x >= self._lo) & (x <= self._hi)) else F64(np.inf)


def Simple2DBox():
    """test/runtests.jl:15-23: clamp x[1] to +-2.9, leave x[2] alone."""
    return IndBox(np.array([-2.9, -np.inf]), np.array([2.9, np.inf]))


class Translate(_ProxObj):
    """ProximalOperators.Translate(f, b): x -> f(x + b)."""

    def __init__(self, f, b, dev=None):
        if isinstance(f, Translate) or f.conjugate:
            raise L.AdaproxError(-3, "nested Translate / Translate of a conjugate has no device kernel")
        self.f = f
        self.b = np.asarray(b, dtype=F64)
        self.kind, self.lam, self.lo, self.hi = f.kind, f.lam, f.lo, f.hi
        self.lo_vec, self.hi_vec = f.lo_vec, f.hi_vec
        self.shift = DeviceVector(self.b, dev=dev)

    def __call__(self, x):
        return self.f(x + self.b)


class _Conjugate(_ProxObj):
    def __init__(self, f):
        self.f = f
        self.kind, self.lam, self.lo, self.hi = f.kind, f.lam, f.lo, f.hi
        self.lo_vec, self.hi_vec, self.shift = f.lo_vec, f.hi_vec, f.shift
        self.conjugate = 1


def convex_conjugate(h):
    """ProximalCore.convex_conjugate."""
    hh, _ = _unwrap(h)
    if type(hh) is Zero:
        return IndZero()
    if type(hh) is IndZero:
        return Zero()
    return _Conjugate(hh)


def prox(g, x, gamma=1.0, dev=None):
    """ProximalCore.prox(f, x, gamma) -> (y, f(y))."""
    gg, counted = _unwrap(g)
    if counted and is_counting_enabled():
        g.prox_count += 1
    x = _vec(x)
    dev = dev or default_device()
    d = gg._desc()
    y = np.empty_like(x)
    gy = C.c_double()
    dev.check(dev.lib.adaprox_prox_eval(dev.h, C.byref(d), _dp(x), x.shape[0], float(gamma), _dp(y), C.byref(gy)))
    return y, F64(gy.value)


def eval_with_pullback(f, x):
    """AdaProx.eval_with_pullback with the Counting wrapper of src/counting.jl:36-51."""
    ff, counted = _unwrap(f)
    if not hasattr(ff, "eval_with_pullback"):
        raise L.AdaproxError(-3, f"eval_with_pullback not defined for type {type(ff).__name__}")
    if counted and is_counting_enabled():
        f.eval_count += 1
    f_x, pb = ff.eval_with_pullback(x)
    if not counted:
        return f_x, pb

    def counting_pullback():
        if is_counting_enabled():
            f.grad_count += 1
        return pb()

    return f_x, counting_pullback


def eval_with_gradient(f, x):
    f_x, pb = eval_with_pullback(f, x)
    return f_x, pb()


# --------------------------------------------------------------------------
# stepsize rules (src/AdaProx.jl:208-308)
# --------------------------------------------------------------------------

class FixedStepsize:
    kind = L.RULE_FIXED

    def __init__(self, gamma, t=1.0):
        self.gamma, self.t = float(gamma), float(t)

    def _fill(self, o):
        o.rule, o.gamma, o.t = self.kind, self.gamma, self.t


class MalitskyMishchenkoRule:
    kind = L.RULE_MM

    def __init__(self, gamma, t=1.0):
        self.gamma, self.t = float(gamma), float(t)

    def _fill(self, o):
        o.rule, o.gamma, o.t = self.kind, self.gamma, self.t


class OurRule:
    kind = L.RULE_OUR

    def __init__(self, gamma=0, t=1, norm_A=0, delta=0, Theta=1.2):
        if gamma > 0:                                             # :241-247
            _gamma = float(gamma)
        elif norm_A > 0:
            _gamma = 1 / (2 * Theta * t * norm_A)
        else:
            raise ValueError("you must provide gamma > 0 if norm_A = 0")
        self.gamma, self.t, self.norm_A, self.delta, self.Theta = _gamma, float(t), float(norm_A), float(delta), float(Theta)

    def _fill(self, o):
        o.rule, o.gamma, o.t, o.norm_A, o.delta, o.Theta = self.kind, self.gamma, self.t, self.norm_A, self.delta, self.Theta


class OurRulePlus:
    kind = L.RULE_OUR_PLUS

    def __init__(self, gamma=0, nu=1, xi=1, r=0.5):
        if not gamma > 0:
            raise ValueError("you must provide gamma > 0")
        self.gamma, self.nu, self.xi, self.r = float(gamma), float(nu), float(xi), float(r)

    def _fill(self, o):
        o.rule, o.gamma, o.xi, o.nu, o.r, o.t = self.kind, self.gamma, self.xi, self.nu, self.r, 1.0


def stepsize(rule, state=None, dgg=None, dgx=None, dxx=None):
    """``stepsize(rule)`` / ``stepsize(rule, state, ...)`` from the three
    reductions |dgrad|^2, <dgrad, dx>, |dx|^2 (what the kernels fuse)."""
    o = L.Options()
    rule._fill(o)
    if state is None:
        g = rule.gamma
        if isinstance(rule, FixedStepsize):
            return (g, g * rule.t ** 2), None
        if isinstance(rule, MalitskyMishchenkoRule):
            return (g, g * rule.t ** 2), (g, np.inf)
        if isinstance(rule, OurRule):
            return (g, g * rule.t ** 2), (g, g)
        return (g, g), (g, g)
    lib = L.load()
    gam, sig, s1 = C.c_double(), C.c_double(), C.c_double()
    lib.adaprox_stepsize(C.byref(o), float(state[0]), float(state[1]), float(dgg), float(dgx), float(dxx),
                         C.byref(gam), C.byref(sig), C.byref(s1))
    return (gam.value, sig.value), (gam.value, s1.value)


# --------------------------------------------------------------------------
# solver entry points (src/AdaProx.jl), same keywords and defaults
# --------------------------------------------------------------------------

_REC_KEYS = ("it", "gamma", "sigma", "norm_res")


def _solve(solver, x0, y0, *, f, g, h=None, A=None, opts, name, log, pd):
    ff, cf = _unwrap(f)
    gg, cg_ = _unwrap(g)
    hh, ch = _unwrap(h) if h is not None else (None, False)
    AA, cA = _unwrap(A) if A is not None else (None, False)
    x0 = _vec(x0)
    n = x0.shape[0]
    if not isinstance(ff, _Smooth):
        raise L.AdaproxError(-3, f"eval_with_pullback not defined for type {type(ff).__name__} (no CPU fallback)")
    if getattr(ff, "n", None) is not None and ff.n != n:
        raise ValueError(f"x has length {n} but f expects {ff.n}")
    dev = ff._dev()
    p = ff._problem(n)
    p.g = gg._desc()
    if pd:
        Amat = _as_matrix(AA, dev)
        p.A_mat = Amat.id
        p.m_dual = Amat.shape[0]
        p.h = hh._desc()
        y0 = _vec(y0, Amat.shape[0])
    elif solver == L.S_AGRAAL:
        y0 = _vec(y0, n)
    opts.solver = solver
    maxit = int(opts.maxit)
    want_log = log is not None
    opts.want_objective = 1 if want_log else 0
    opts.max_records = maxit if want_log else 0
    opts.counting_f, opts.counting_g, opts.counting_h, opts.counting_A = int(cf), int(cg_), int(ch), int(cA)
    recs = (L.Record * max(maxit, 1))() if want_log else None
    res = L.Result()
    x_out = np.empty(n, dtype=F64)
    y_out = np.empty(max(p.m_dual, 1), dtype=F64) if pd else None
    dev.check(dev.lib.adaprox_solve(dev.h, C.byref(p), C.byref(opts), _dp(x0), _dp(y0) if y0 is not None else None,
                                    _dp(x_out), _dp(y_out) if y_out is not None else None, recs, C.byref(res)))
    dev.launches += res.kernel_launches
    # Counting wrappers accumulate across calls like the Julia objects do
    if cf:
        f.eval_count += res.f_evals
        f.grad_count += res.grad_f_evals
    if cg_:
        g.prox_count += res.prox_g_evals
    if ch:
        h.prox_count += res.prox_h_evals
    if cA:
        A.mul_count += res.A_evals
        A.amul_count += res.At_evals
    if want_log:
        base = dict(f=(f.eval_count - res.f_evals) if cf else 0, gr=(f.grad_count - res.grad_f_evals) if cf else 0,
                    pg=(g.prox_count - res.prox_g_evals) if cg_ else 0, ph=(h.prox_count - res.prox_h_evals) if ch else 0,
                    mu=(A.mul_count - res.A_evals) if cA else 0, am=(A.amul_count - res.At_evals) if cA else 0)
        for k in range(res.n_records):
            r = recs[k]
            d = dict(method=name, it=int(r.it), gamma=F64(r.gamma))
            if pd or solver == L.S_ADAPTIVE_PROXGRAD:
                d["sigma"] = F64(r.sigma)
            d["norm_res"] = F64(r.norm_res)
            d["objective"] = F64(r.f_x) + F64(r.g_x) + F64(r.h_Ax)
            d["grad_f_evals"] = base["gr"] + r.grad_f_evals if cf else None
            d["prox_g_evals"] = base["pg"] + r.prox_g_evals if cg_ else None
            if pd or solver == L.S_ADAPTIVE_PROXGRAD:
                d["prox_h_evals"] = base["ph"] + r.prox_h_evals if ch else None
                d["A_evals"] = base["mu"] + r.A_evals if cA else None
                d["At_evals"] = base["am"] + r.At_evals if cA else None
            d["f_evals"] = base["f"] + r.f_evals if cf else None
            log.append(d)
    info = dict(flags=int(res.flags), solve_ms=res.solve_ms, kernel_launches=int(res.kernel_launches), matrix_passes=int(res.matrix_passes), collective=int(res.collective),
                final_gamma=res.final_gamma, final_sigma=res.final_sigma, final_norm_res=res.final_norm_res)
    return x_out, (y_out[: p.m_dual] if pd else None), int(res.iters), info


_last_info = {}


def last_solve_info():
    """Device-side facts about the most recent solve (flags, device ms, launches)."""
    return dict(_last_info)


def _opts(tol, maxit):
    o = L.Options()
    o.tol, o.maxit = float(tol), int(maxit)
    o.t, o.Theta, o.xi, o.nu, o.r, o.R, o.shrink, o.phi, o.gamma_max, o.theta = 1.0, 1.2, 1.0, 1.0, 0.5, 0.95, 0.5, 1.5, 1e6, -1.0
    return o


def adaptive_primal_dual(x, y, *, f, g, h, A, rule, tol=1e-5, maxit=10_000, name="AdaPDM", log=None):
    """src/AdaProx.jl:312-364."""
    o = _opts(tol, maxit)
    rule._fill(o)
    xo, yo, it, info = _solve(L.S_ADAPTIVE_PRIMAL_DUAL, x, y, f=f, g=g, h=h, A=A, opts=o, name=name, log=log, pd=True)
    _last_info.update(info)
    return xo, yo, it


def condat_vu(x, y, *, f, g, h, A, Lf, gamma=None, sigma=None, norm_A=None, tol=1e-5, maxit=10_000,
              name="Condat-Vu", log=None):
    """src/AdaProx.jl:367-416 (parameter selection :398-412, then the generic loop)."""
    if gamma is None and sigma is None:
        Lf = F64(Lf)
        par, par2 = F64(5), F64(100)
        if norm_A is None:
            raise L.AdaproxError(-3, "norm(A) of a device matrix: pass norm_A (Frobenius) explicitly")
        norm_A = F64(norm_A)
        with np.errstate(divide="ignore", invalid="ignore"):
            alpha = F64(1) if norm_A > par * Lf else par2 * norm_A / Lf
            gamma = F64(1) / (Lf / 2 + norm_A / alpha)
            sigma = F64(0.99) / (norm_A * alpha)
    assert gamma is not None and sigma is not None
    rule = FixedStepsize(gamma, np.sqrt(F64(sigma) / F64(gamma)))
    return adaptive_primal_dual(x, y, f=f, g=g, h=h, A=A, rule=rule, tol=tol, maxit=maxit, name=name, log=log)


def adaptive_proxgrad(x, *, f, g, rule, tol=1e-5, maxit=100_000, name="AdaPGM", log=None):
    """src/AdaProx.jl:418-421."""
    o = _opts(tol, maxit)
    rule._fill(o)
    xo, _, it, info = _solve(L.S_ADAPTIVE_PROXGRAD, x, None, f=f, g=g, opts=o, name=name, log=log, pd=False)
    _last_info.update(info)
    return xo, it


def adaptive_proxgrad_path(X0=None, *, f, lambdas, rule, gamma0=None, tol=1e-5, maxit=100_000, history=0):
    """Batched multi-lambda path (BASELINE config 5; include/adaprox.h: adaprox_solve_lambda_path): column j of the
    result is what ``adaptive_proxgrad(X0[:, j], f=f, g=NormL1(lambdas[j]), rule=rule_j, tol=tol, maxit=maxit)`` returns,
    where rule_j is ``rule`` with ``gamma = gamma0[j]`` when ``gamma0`` is given (with ``FixedStepsize`` every step of column j
    uses ``gamma0[j]``; ``maxit = 0`` returns the first prox step with ``its = 0``).  ``f`` is a ``LinearLeastSquares`` over
    a dense or scipy sparse matrix, or a ``LogisticLoss`` over a scipy sparse matrix; for the logistic loss n is
    features + 1 (``LogisticLoss.n``, intercept last, penalised by the l1 term like every other entry).  Returns
    ``(X, its, info)`` with X of shape (n, L), ``its`` the per-column iteration counts and ``info`` holding per-column
    ``norm_res``, ``gamma``, ``f_x`` and, with ``history = H > 0``, the arrays ``gamma_hist``, ``res_hist``, ``obj_hist``
    of shape (min(H, maxit), L) (NaN after a column stopped)."""
    ff, _ = _unwrap(f)
    if not isinstance(ff, (LinearLeastSquares, LogisticLoss)):
        raise L.AdaproxError(-3, "adaptive_proxgrad_path: f must be a LinearLeastSquares or LogisticLoss term (no CPU fallback)")
    lam = np.ascontiguousarray(np.asarray(lambdas, dtype=F64).ravel())
    Lc = lam.shape[0]
    n = ff.n if getattr(ff, "n", None) is not None else ff.A.shape[1]
    dev = ff._dev()
    p = ff._problem(n)
    p.g = NormL1(1.0)._desc()
    o = _opts(tol, maxit)
    rule._fill(o)
    o.solver = L.S_ADAPTIVE_PROXGRAD
    x0T = None
    if X0 is not None:
        X0 = np.asarray(X0, dtype=F64)
        if X0.shape != (n, Lc):
            raise ValueError(f"X0 has shape {X0.shape}, expected {(n, Lc)}")
        x0T = np.ascontiguousarray(X0.T)
    g0 = None
    if gamma0 is not None:
        g0 = np.ascontiguousarray(np.asarray(gamma0, dtype=F64).ravel())
        if g0.shape[0] != Lc:
            raise ValueError("gamma0 must have one entry per lambda")
    xoT = np.empty((Lc, n), dtype=F64)
    its = np.zeros(Lc, dtype=np.int64)
    nres, gout, fout = np.empty(Lc, dtype=F64), np.empty(Lc, dtype=F64), np.empty(Lc, dtype=F64)
    H = int(min(history, maxit)) if history else 0
    hist = np.empty((3, max(H, 1), Lc), dtype=F64) if H > 0 else None
    res = L.Result()
    dev.check(dev.lib.adaprox_solve_lambda_path(dev.h, C.byref(p), C.byref(o), Lc, _dp(lam), _dp(g0) if g0 is not None else None,
                                                _dp(x0T) if x0T is not None else None, _dp(xoT),
                                                its.ctypes.data_as(C.POINTER(C.c_int64)), _dp(nres), _dp(gout), _dp(fout),
                                                _dp(hist) if hist is not None else None, H, C.byref(res)))
    dev.launches += res.kernel_launches
    info = dict(norm_res=nres, gamma=gout, f_x=fout, flags=int(res.flags), solve_ms=res.solve_ms, kernel_launches=int(res.kernel_launches),
                batched_evals=int(res.f_evals), iters_max=int(res.iters))
    if hist is not None:
        info.update(gamma_hist=hist[0], res_hist=hist[1], obj_hist=hist[2])
    _last_info.update(dict(flags=info["flags"], solve_ms=res.solve_ms, kernel_launches=int(res.kernel_launches), matrix_passes=2))
    return np.ascontiguousarray(xoT.T), its, info


def adaptive_primal_dual_path(X0=None, Y0=None, *, f, A, upper, rule, lower=0.0, gamma0=None, tol=1e-5, maxit=10_000, history=0):
    """Batched C path of the dual SVM (dual_svm/runme.jl:47-59; include/adaprox.h: adaprox_solve_box_path): column j of
    the result is what ``adaptive_primal_dual(X0[:, j], [Y0[j]], f=f, g=IndBox(lower, upper[j]), h=IndZero(), A=A,
    rule=rule_j, tol=tol, maxit=maxit)`` returns, where rule_j is ``rule`` with ``gamma = gamma0[j]`` when ``gamma0`` is given
    (condat_vu's parameters arrive as a ``FixedStepsize``).  ``f`` is a ``Quadratic`` or a ``QuadraticGram`` over a dense
    matrix, ``A`` the 1 x n label row.  X0 (n, L) and Y0 (L,) default to zeros.  Returns ``(X, Y, its, info)`` with X of
    shape (n, L), Y the L dual scalars, ``its`` the per-column iteration counts and ``info`` holding per-column
    ``norm_res``, ``gamma``, ``sigma``, ``f_x`` and, with ``history = H > 0``, the arrays ``gamma_hist``, ``res_hist``,
    ``obj_hist`` (objective f + g + h(A x)) of shape (min(H, maxit), L) (NaN after a column stopped)."""
    ff, _ = _unwrap(f)
    AA, _ = _unwrap(A)
    if not isinstance(ff, _Smooth):
        raise L.AdaproxError(-3, f"eval_with_pullback not defined for type {type(ff).__name__} (no CPU fallback)")
    dev = ff._dev()
    Amat = _as_matrix(AA, dev)
    n = Amat.shape[1]
    up = np.ascontiguousarray(np.asarray(upper, dtype=F64).ravel())
    Lc = up.shape[0]
    if np.ndim(upper) != 1 or Lc < 1:
        raise ValueError("upper must be a non-empty vector of box bounds")
    p = ff._problem(n)
    p.g = IndBox(float(lower), float(lower))._desc()
    p.h = IndZero()._desc()
    p.A_mat, p.m_dual = Amat.id, Amat.shape[0]
    o = _opts(tol, maxit)
    rule._fill(o)
    o.solver = L.S_ADAPTIVE_PRIMAL_DUAL
    x0T = y0 = g0 = None
    if X0 is not None:
        X0 = np.asarray(X0, dtype=F64)
        if X0.shape != (n, Lc):
            raise ValueError(f"X0 has shape {X0.shape}, expected {(n, Lc)}")
        x0T = np.ascontiguousarray(X0.T)
    if Y0 is not None:
        y0 = np.ascontiguousarray(np.asarray(Y0, dtype=F64))
        if y0.shape != (Lc,):
            raise ValueError(f"Y0 has shape {y0.shape}, expected {(Lc,)}")
    if gamma0 is not None:
        g0 = np.ascontiguousarray(np.asarray(gamma0, dtype=F64))
        if g0.shape != (Lc,):
            raise ValueError("gamma0 must have one entry per C value")
    xoT = np.empty((Lc, n), dtype=F64)
    yo = np.empty(Lc, dtype=F64)
    its = np.zeros(Lc, dtype=np.int64)
    nres, gout, sout, fout = (np.empty(Lc, dtype=F64) for _ in range(4))
    H = int(min(history, maxit)) if history else 0
    hist = np.empty((3, max(H, 1), Lc), dtype=F64) if H > 0 else None
    res = L.Result()
    opt = lambda a: _dp(a) if a is not None else None
    dev.check(dev.lib.adaprox_solve_box_path(dev.h, C.byref(p), C.byref(o), Lc, _dp(up), opt(g0), opt(x0T), opt(y0), _dp(xoT), _dp(yo),
                                             its.ctypes.data_as(C.POINTER(C.c_int64)), _dp(nres), _dp(gout), _dp(sout), _dp(fout),
                                             opt(hist), H, C.byref(res)))
    dev.launches += res.kernel_launches
    info = dict(norm_res=nres, gamma=gout, sigma=sout, f_x=fout, flags=int(res.flags), solve_ms=res.solve_ms,
                kernel_launches=int(res.kernel_launches), batched_evals=int(res.f_evals), iters_max=int(res.iters))
    if hist is not None:
        info.update(gamma_hist=hist[0], res_hist=hist[1], obj_hist=hist[2])
    _last_info.update(dict(flags=info["flags"], solve_ms=res.solve_ms, kernel_launches=int(res.kernel_launches),
                           matrix_passes=int(res.matrix_passes)))
    return np.ascontiguousarray(xoT.T), yo, its, info


def adaptive_primal_dual_lambda_path(X0=None, Y0=None, *, f, h, A, lambdas, rule, gamma0=None, tol=1e-5, maxit=10_000, history=0):
    """Batched lambda path of LAD and the square-root lasso (least_absolute_deviation/runme.jl, square_root_lasso/runme.jl;
    include/adaprox.h: adaprox_solve_pd_lambda_path): column j of the result is what ``adaptive_primal_dual(X0[:, j],
    Y0[:, j], f=f, g=NormL1(lambdas[j]), h=h, A=A, rule=rule_j, tol=tol, maxit=maxit)`` returns, where rule_j is ``rule``
    with ``gamma = gamma0[j]`` when ``gamma0`` is given (condat_vu's parameters arrive as a ``FixedStepsize``).  ``f`` is
    ``Zero()``, ``h`` a ``NormL1`` / ``NormL2`` of any weight, optionally ``Translate``'d, and ``A`` a dense m x n matrix.
    X0 (n, L) and Y0 (m, L) default to zeros.  Returns ``(X, Y, its, info)`` with X of shape (n, L), Y of shape (m, L),
    ``its`` the per-column iteration counts and ``info`` holding per-column ``norm_res``, ``gamma``, ``sigma`` and, with
    ``history = H > 0``, the arrays ``gamma_hist``, ``res_hist``, ``obj_hist`` (objective g + h(A x)) of shape
    (min(H, maxit), L) (NaN after a column stopped)."""
    ff, _ = _unwrap(f)
    hh, _ = _unwrap(h)
    AA, _ = _unwrap(A)
    if not isinstance(ff, _Smooth):
        raise L.AdaproxError(-3, f"eval_with_pullback not defined for type {type(ff).__name__} (no CPU fallback)")
    dev = ff._dev()
    Amat = _as_matrix(AA, dev)
    m, n = Amat.shape
    if np.ndim(lambdas) != 1 or np.size(lambdas) < 1:
        raise ValueError("lambdas must be a non-empty vector")
    lam = np.ascontiguousarray(np.asarray(lambdas, dtype=F64))
    Lc = lam.shape[0]
    p = ff._problem(n)
    p.g = NormL1(1.0)._desc()
    p.h = hh._desc()
    p.A_mat, p.m_dual = Amat.id, m
    o = _opts(tol, maxit)
    rule._fill(o)
    o.solver = L.S_ADAPTIVE_PRIMAL_DUAL
    x0T = y0T = g0 = None
    if X0 is not None:
        X0 = np.asarray(X0, dtype=F64)
        if X0.shape != (n, Lc):
            raise ValueError(f"X0 has shape {X0.shape}, expected {(n, Lc)}")
        x0T = np.ascontiguousarray(X0.T)
    if Y0 is not None:
        Y0 = np.asarray(Y0, dtype=F64)
        if Y0.shape != (m, Lc):
            raise ValueError(f"Y0 has shape {Y0.shape}, expected {(m, Lc)}")
        y0T = np.ascontiguousarray(Y0.T)
    if gamma0 is not None:
        g0 = np.ascontiguousarray(np.asarray(gamma0, dtype=F64))
        if g0.shape != (Lc,):
            raise ValueError("gamma0 must have one entry per lambda")
    xoT = np.empty((Lc, n), dtype=F64)
    yoT = np.empty((Lc, m), dtype=F64)
    its = np.zeros(Lc, dtype=np.int64)
    nres, gout, sout = (np.empty(Lc, dtype=F64) for _ in range(3))
    H = int(min(history, maxit)) if history else 0
    hist = np.empty((3, max(H, 1), Lc), dtype=F64) if H > 0 else None
    res = L.Result()
    opt = lambda a: _dp(a) if a is not None else None
    dev.check(dev.lib.adaprox_solve_pd_lambda_path(dev.h, C.byref(p), C.byref(o), Lc, _dp(lam), opt(g0), opt(x0T), opt(y0T), _dp(xoT),
                                                   _dp(yoT), its.ctypes.data_as(C.POINTER(C.c_int64)), _dp(nres), _dp(gout), _dp(sout),
                                                   opt(hist), H, C.byref(res)))
    dev.launches += res.kernel_launches
    info = dict(norm_res=nres, gamma=gout, sigma=sout, flags=int(res.flags), solve_ms=res.solve_ms,
                kernel_launches=int(res.kernel_launches), batched_evals=int(res.f_evals), iters_max=int(res.iters))
    if hist is not None:
        info.update(gamma_hist=hist[0], res_hist=hist[1], obj_hist=hist[2])
    _last_info.update(dict(flags=info["flags"], solve_ms=res.solve_ms, kernel_launches=int(res.kernel_launches),
                           matrix_passes=int(res.matrix_passes)))
    return np.ascontiguousarray(xoT.T), np.ascontiguousarray(yoT.T), its, info


def auto_adaptive_proxgrad(x, *, f, g, gamma=None, tol=1e-5, maxit=100_000, name="AutoAdaPGM", log=None):
    """src/AdaProx.jl:423-455: two gradient evaluations and one (or two) prox steps estimate the initial stepsize, then
    AdaPGM with OurRule from the ORIGINAL point.  Every oracle call below is a device call (eval_with_gradient / prox
    through the C ABI); the loop itself is the persistent kernel.  ``gamma = nothing`` cannot run in the reference
    (:431 calls ``prox`` without ``g`` -> MethodError) and raises here as well."""
    x = _vec(x)
    _, grad_x = eval_with_gradient(f, x)
    if np.sqrt(np.dot(grad_x, grad_x)) <= tol:                       # :426-428
        return x, 0
    if gamma is None:
        raise TypeError("auto_adaptive_proxgrad: the reference's `gamma = nothing` branch calls prox(x, gamma) without g (src/AdaProx.jl:431): MethodError")
    assert gamma > 0                                                  # :437
    gamma = F64(gamma)
    with np.errstate(divide="ignore", invalid="ignore"):
        x_prev, grad_x_prev, gamma_prev = x, grad_x, gamma            # :439
        x, _ = prox(g, x - gamma * grad_x, gamma)                     # :440
        _, grad_x = eval_with_gradient(f, x)
        dx = x - x_prev
        L_ = np.dot(grad_x - grad_x_prev, dx) / np.sqrt(np.dot(dx, dx)) ** 2
        gamma = np.sqrt(F64(2)) * gamma if L_ == 0 else F64(1) / L_   # :443
        if gamma_prev / gamma > 1e5:                                  # :445-450
            x, _ = prox(g, x_prev - gamma * grad_x_prev, gamma)
            _, grad_x = eval_with_gradient(f, x)
            dx = x - x_prev
            L_ = np.dot(grad_x - grad_x_prev, dx) / np.sqrt(np.dot(dx, dx)) ** 2
            gamma = np.sqrt(F64(2)) * gamma if L_ == 0 else F64(1) / L_
    rule = OurRule(gamma=float(gamma), t=1, norm_A=0, delta=0, Theta=1.2)      # :452
    return adaptive_proxgrad(x_prev, f=f, g=g, rule=rule, tol=tol, maxit=maxit, name=name, log=log)


def fixed_proxgrad(x, *, f, g, gamma, tol=1e-5, maxit=100_000, name="Fixed stepsize PGM", log=None):
    """src/AdaProx.jl:457-459."""
    return adaptive_proxgrad(x, f=f, g=g, rule=FixedStepsize(gamma, 1.0), tol=tol, maxit=maxit, name=name, log=log)


def adaptive_linesearch_primal_dual(x, y, *, f, g, h, A, gamma=None, eta=1.0, t=1.0, delta=1e-8, Theta=1.2,
                                    r=2, R=0.95, tol=1e-5, maxit=10_000, name="AdaPDM+", log=None):
    """src/AdaProx.jl:463-550."""
    assert eta > 0, "eta must be positive"
    assert Theta > (delta + 1), "must be Theta > (delta + 1)"
    if gamma is None:
        gamma = 1 / (2 * Theta * t * eta)
    assert gamma <= 1 / (2 * Theta * t * eta), "gamma is too large"
    o = _opts(tol, maxit)
    o.gamma, o.eta, o.t, o.delta, o.Theta, o.r, o.R = float(gamma), float(eta), float(t), float(delta), float(Theta), float(r), float(R)
    xo, yo, it, info = _solve(L.S_LINESEARCH_PRIMAL_DUAL, x, y, f=f, g=g, h=h, A=A, opts=o, name=name, log=log, pd=True)
    _last_info.update(info)
    return xo, yo, it


def malitsky_pock(x, y, *, f, g, h, A, sigma, t=1.0, tol=1e-5, maxit=10_000, name="MP-ls", log=None):
    """src/AdaProx.jl:581-629."""
    o = _opts(tol, maxit)
    o.sigma, o.t = float(sigma), float(t)
    xo, yo, it, info = _solve(L.S_MALITSKY_POCK, x, y, f=f, g=g, h=h, A=A, opts=o, name=name, log=log, pd=True)
    _last_info.update(info)
    return xo, yo, it


def backtracking_proxgrad(x0, *, f, g, gamma0, xi=1.0, shrink=0.5, tol=1e-5, maxit=100_000,
                          name="Backtracking PG", log=None):
    """src/AdaProx.jl:50-64."""
    o = _opts(tol, maxit)
    o.gamma, o.xi, o.shrink = float(gamma0), float(xi), float(shrink)
    xo, _, it, info = _solve(L.S_BACKTRACKING_PROXGRAD, x0, None, f=f, g=g, opts=o, name=name, log=log, pd=False)
    _last_info.update(info)
    return xo, it


def backtracking_nesterov(x0, *, f, g, gamma0, shrink=0.5, tol=1e-5, maxit=100_000,
                          name="Backtracking Nesterov", log=None):
    """src/AdaProx.jl:66-84."""
    o = _opts(tol, maxit)
    o.gamma, o.shrink = float(gamma0), float(shrink)
    xo, _, it, info = _solve(L.S_BACKTRACKING_NESTEROV, x0, None, f=f, g=g, opts=o, name=name, log=log, pd=False)
    _last_info.update(info)
    return xo, it


def fixed_nesterov(x0, *, f, g, Lf=None, muf=0, mug=0, gamma=None, theta=None, tol=1e-5, maxit=100_000,
                   name="Fixed Nesterov", log=None):
    """src/AdaProx.jl:91-142."""
    assert (gamma is None) != (Lf is None)
    if gamma is None:
        gamma = 1 / Lf
    mu = muf + mug
    q = gamma * mu / (1 + gamma * mug)
    assert q < 1
    if theta is None:
        theta = 1 / np.sqrt(q) if q > 0 else 0
    with np.errstate(divide="ignore"):
        assert 0 <= theta <= 1 / np.sqrt(F64(q))
    o = _opts(tol, maxit)
    o.gamma, o.muf, o.mug, o.theta = float(gamma), float(muf), float(mug), float(theta)
    xo, _, it, info = _solve(L.S_FIXED_NESTEROV, x0, None, f=f, g=g, opts=o, name=name, log=log, pd=False)
    _last_info.update(info)
    return xo, it


def agraal(x1, *, f, g, x0=None, gamma0=None, gamma_max=1e6, phi=1.5, tol=1e-5, maxit=100_000, name="aGRAAL",
           log=None, rng=None):
    """src/AdaProx.jl:150-192."""
    x1 = _vec(x1)
    if x0 is None:
        rng = np.random.default_rng(0) if rng is None else rng
        x0 = x1 + rng.standard_normal(x1.shape)
    o = _opts(tol, maxit)
    o.gamma = float(gamma0) if gamma0 is not None else 0.0
    o.gamma_max, o.phi = float(gamma_max), float(phi)
    xo, _, it, info = _solve(L.S_AGRAAL, x1, x0, f=f, g=g, opts=o, name=name, log=log, pd=False)
    _last_info.update(info)
    return xo, it


# --------------------------------------------------------------------------
# device-side problem generation (config C4: the matrix never exists on the host)
# --------------------------------------------------------------------------

def generate_planted_lasso(m, n, pfactor=5, seed=0, lam=1.0, rho=1.0, power_iters=30, row0=0, rows=None, dev=None):
    """lasso/runme.jl:40-77 on the device for the row shard [row0, row0+rows)."""
    dev = dev or default_device()
    rows = m - row0 if rows is None else rows
    A_id, b_id = L.c_id(), L.c_id()
    x_star = np.empty(n, dtype=F64)
    opt, Lf = C.c_double(), C.c_double()
    dev.check(dev.lib.adaprox_generate_planted_lasso(dev.h, m, n, row0, rows, float(pfactor), int(seed), float(lam),
                                                     float(rho), int(power_iters), C.byref(A_id), C.byref(b_id),
                                                     _dp(x_star), C.byref(opt), C.byref(Lf)))
    A = DeviceMatrix(dev=dev, _id=A_id.value, _shape=(rows, n))
    b = DeviceVector(dev=dev, _id=b_id.value, _len=rows)
    return dict(A=A, b=b, x_star=x_star, optimum=opt.value, Lf=Lf.value, lam=float(lam))
