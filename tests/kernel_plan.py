"""A pure-Python restatement of the kernel selection arithmetic that the extended-precision tests build their shape sets from.

api.cu: plan_dense (work split of a dense matrix, made at upload for the handle's grid of 2 CTAs per SM) and solver_grid (the
grid a solve launches); gemv.cuh: csr_lanes_per_row and the gsum_slice predicate.  `dense_branches` / `csr_branches` name the
branches of the two-pass matrix sweeps a set of shapes reaches, so that a test can assert that none is left out.
"""
import contextlib
import os

import numpy as np
import scipy.sparse as sp

KCHUNK = 2048
SMALL_BYTES = 8 << 20             # api.cu: kSmallProblemBytes


def r16(n):
    return -(-n // 16) * 16


def cdiv(a, b):
    return -(-a // b)


def plan_dense(m, n, grid):
    """api.cu: plan_dense at upload, for the handle's grid (2 CTAs per SM) -> (nchunks, rb, nrb)."""
    nch = cdiv(n, KCHUNK)
    rb = 64
    while rb > 8 and nch * cdiv(m, rb) < 16 * grid:
        rb //= 2
    return nch, rb, cdiv(m, rb)


def solver_grid(m, n, sm, grid, env_grid=None, has_A=False):
    """api.cu: solver_grid (ADAPROX_GRID = env_grid).  Without a linear map, a dense least-squares term of fewer than 8 MB runs
    on one CTA per SM; the primal-dual loops (an A is given) always keep the handle's grid of 2 CTAs per SM."""
    if env_grid:
        return min(env_grid, grid)
    if has_A:
        return grid
    return min(grid, sm) if m * r16(n) * 8 < SMALL_BYTES else grid


def dense_branches(shapes, sm, has_A=False):
    """Branches of gemv_n_dense / gemv_t_dense / gsum_slice that the (m, n, ADAPROX_GRID) shapes reach on `sm` SMs.  With
    has_A the shapes are those of the linear map of a primal-dual solve (solver_grid never picks one CTA per SM)."""
    grid = 2 * sm
    hit = set()
    for m, n, env_grid in shapes:
        nch, rb, nrb = plan_dense(m, n, grid)
        G = solver_grid(m, n, sm, grid, env_grid, has_A)
        Uu = nch * nrb
        hit.add(f"rb:{rb}")
        hit.add("grid:env" if env_grid else ("grid:sm" if G == min(grid, sm) and G < grid else "grid:2sm"))
        if env_grid and Uu % G:
            hit.add("grid:env_nondiv")
        if nch == 1:
            hit.add("chunks:1")                      # phases.cuh: f_rows_local
        elif nch <= 4 and r16(n) % KCHUNK:
            hit.add("chunks:2-4_ragged")
        bounds = [(Uu * b // G, Uu * (b + 1) // G) for b in range(G)]
        if any(u0 == u1 for u0, u1 in bounds):
            hit.add("idle_cta")
        if any(u0 < u1 and u0 % nrb and (u1 - 1) // nrb > u0 // nrb for u0, u1 in bounds):
            hit.add("slab_mid_chunk_crossing")
        hit.add("gsum:warp" if (G > 16 * nch and nrb > 16) else "gsum:thread")    # gemv.cuh: gsum_slice
        if m % 4:
            hit.add("m%4")                           # gemv_t_dense: row remainder
    return hit


DENSE_REQUIRED = {"rb:8", "rb:16", "rb:32", "rb:64", "grid:sm", "grid:2sm", "grid:env", "grid:env_nondiv", "chunks:1",
                  "chunks:2-4_ragged", "idle_cta", "slab_mid_chunk_crossing", "gsum:warp", "gsum:thread", "m%4"}


def csr_lanes_per_row(nnz, nrows):
    """gemv.cuh: csr_lanes_per_row"""
    avg = nnz // max(nrows, 1)
    return 32 if avg > 192 else (16 if avg > 24 else (8 if avg > 12 else 4))


def csr_branches(cases, matrices):
    """cases: (matrix name, f kind, ADAPROX_CSR_LPR or None); matrices: name -> callable returning the scipy CSR matrix."""
    hit = set()
    for name, kind, lpr in cases:
        X = matrices[name]()
        m, nf = X.shape
        how = "forced" if lpr else "mean"
        ln = lpr or csr_lanes_per_row(X.nnz, m)
        lt = lpr or csr_lanes_per_row(X.nnz, nf)
        hit |= {f"Xw:{ln}:{how}", f"Xtr:{lt}:{how}", f"kind:{kind}"}
        lens = set(np.diff(X.indptr).tolist())
        if {0, 1, ln - 1, 4 * ln, 4 * ln + 1} <= lens and max(lens) > 2000:
            hit.add(f"rows:{ln}")
        if np.any(np.bincount(X.indices, minlength=nf) == 0):
            hit.add("empty_feature")
        if m < 32 // ln:
            hit.add("rows<group")
    return hit


def _csr(m, nf, lengths, seed, empty=(1,)):
    """CSR with the given row lengths (cycled, capped at the usable features); the features in `empty` have no non-zeros."""
    rng = np.random.default_rng(seed)
    pool = np.array([c for c in range(nf) if c not in empty])
    indptr, cols = [0], []
    for i in range(m):
        k = min(lengths[i % len(lengths)], pool.size)
        cols.append(np.sort(rng.choice(pool, size=k, replace=False)) if k else np.zeros(0, dtype=np.int64))
        indptr.append(indptr[-1] + k)
    ind = np.concatenate(cols).astype(np.int32)
    return sp.csr_matrix((rng.uniform(-1.0, 1.0, ind.size), ind, np.array(indptr)), shape=(m, nf))


@contextlib.contextmanager
def environ(env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
