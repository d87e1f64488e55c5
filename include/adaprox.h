/*
 * adaprox.h -- C ABI of libadaprox_cuda.so (sm_100a).
 *
 * The library replaces the iteration hot path of AdaProx.jl (reference paths
 * below are relative to the reference repository root): the concrete smooth
 * oracles, the prox operators, the stepsize rules and the loop bodies of the
 * solver entry points run as hand-written fp64 CUDA kernels; the Julia (or
 * Python) front end keeps the reference's entry points and keyword API and
 * reaches this file through `ccall` / ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; every function returns an adaprox_status
 *     (0 = ok, < 0 = error; adaprox_last_error() has the text); nothing throws.
 *   - `double*` arguments are HOST pointers unless the name ends in `_dev`.
 *   - the library owns all device memory; matrices and long-lived vectors are
 *     uploaded (or generated) once and referenced by integer ids.
 *   - one in-flight call per handle; a handle is bound to one CUDA device.
 *   - dense matrices are accepted column-major (Julia) or row-major (C) and are
 *     repacked once into the device layout (row-major, rows padded to 128 B).
 */
#ifndef ADAPROX_H
#define ADAPROX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct adaprox_ctx* adaprox_handle;
typedef int64_t adaprox_id;            /* matrix / vector id; 0 = none */

typedef enum {
  ADAPROX_OK = 0,
  ADAPROX_ERR_INVALID = -1,            /* bad argument (the reference @assert / error()) */
  ADAPROX_ERR_CUDA = -2,
  ADAPROX_ERR_UNSUPPORTED = -3,        /* combination without a device kernel: no CPU fallback */
  ADAPROX_ERR_COMM = -4,
  ADAPROX_ERR_NOMEM = -5
} adaprox_status;

/* result.flags bits */
#define ADAPROX_FLAG_CONVERGED      1u  /* norm_res <= tol                       */
#define ADAPROX_FLAG_STEP_TOO_SMALL 2u  /* src/AdaProx.jl:40-42,566-568 @error   */
#define ADAPROX_FLAG_NONFINITE      4u  /* NaN/Inf stepsize or residual observed */
#define ADAPROX_FLAG_LS_CAP         8u  /* a linesearch hit its trial cap        */
#define ADAPROX_FLAG_COMM          16u  /* a peer rank did not show up in an in-kernel exchange; the call returns ADAPROX_ERR_COMM */

/* ---- smooth term f: the experiment scripts' oracle structs ----------------- */
typedef enum {
  ADAPROX_F_ZERO = 0,           /* least_absolute_deviation/runme.jl:18-21            */
  ADAPROX_F_LEAST_SQUARES = 1,  /* lasso/runme.jl:16-27: mat=A, vec=b                  */
  ADAPROX_F_LOGISTIC = 2,       /* sparse_logreg/runme.jl:18-39: mat=X, vec=y, w[end] intercept */
  ADAPROX_F_QUADRATIC = 3,      /* dual_svm/runme.jl:19-28: mat=Q (symmetric), vec=q   */
  ADAPROX_F_CUBIC = 4,          /* cubic_sparse_logreg/runme.jl:20-32: mat=Q, vec=q, c */
  ADAPROX_F_WORST_QUADRATIC = 5,/* nesterov_worst_case/runme.jl:14-40: k=ipar, L=c     */
  ADAPROX_F_SIMPLE2D = 6,       /* test/runtests.jl:6-13                               */
  ADAPROX_F_QUADRATIC_GRAM = 7  /* Quadratic with Q = Z*Z' given by its factor: mat=Z (n x d), vec=q.  dual_svm/runme.jl:47-49
                                   builds Q = Dy*X*X'*Dy, i.e. Z = Dy*X; Q*x is evaluated as Z*(Z'*x), 16*n*d bytes
                                   instead of 8*n^2 (same value up to rounding, not bitwise)                  */
} adaprox_f_kind;

/* ---- nonsmooth terms g, h: ProximalCore / ProximalOperators objects -------- */
typedef enum {
  ADAPROX_P_ZERO = 0,           /* ProximalCore.Zero                                   */
  ADAPROX_P_IND_ZERO = 1,       /* ProximalCore.IndZero                                */
  ADAPROX_P_NORM_L1 = 2,        /* NormL1(lambda)                                      */
  ADAPROX_P_NORM_L2 = 3,        /* NormL2(lambda)                                      */
  ADAPROX_P_IND_BOX = 4         /* IndBox(lo, hi), scalar bounds or per-coordinate vectors */
} adaprox_prox_kind;

typedef struct {
  int32_t kind;                 /* adaprox_prox_kind                                    */
  int32_t conjugate;            /* 1: use convex_conjugate(.) (Moreau, src/AdaProx.jl:325) */
  double lambda;                /* NormL1 / NormL2 weight                               */
  double lo, hi;                /* IndBox scalar bounds (used when lo_vec/hi_vec are 0) */
  adaprox_id lo_vec, hi_vec;    /* IndBox per-coordinate bounds                         */
  adaprox_id shift;             /* Translate(f, shift): x -> f(x + shift); 0 = none     */
} adaprox_prox;

typedef struct {
  int32_t f_kind;               /* adaprox_f_kind                                       */
  int32_t f_ipar;               /* WORST_QUADRATIC: k                                   */
  adaprox_id f_mat;             /* A / X / Q                                            */
  adaprox_id f_vec;             /* b / y / q                                            */
  double f_c;                   /* CUBIC: c ; WORST_QUADRATIC: L                        */
  adaprox_prox g;
  adaprox_prox h;               /* ignored by the proximal-gradient solvers             */
  adaprox_id A_mat;             /* linear map of the primal-dual solvers; 0 = `A = 0`   */
  int64_t n;                    /* primal dimension (length of x)                       */
  int64_t m_dual;               /* dual dimension (length of y); 0 for proximal gradient */
} adaprox_problem;

/* ---- solvers (src/AdaProx.jl entry points) --------------------------------- */
typedef enum {
  ADAPROX_S_ADAPTIVE_PRIMAL_DUAL = 0,   /* :312-364  AdaPDM (also condat_vu :367-416 via RULE_FIXED) */
  ADAPROX_S_ADAPTIVE_PROXGRAD = 1,      /* :418-421  AdaPGM ; fixed_proxgrad :457-459 via RULE_FIXED  */
  ADAPROX_S_LINESEARCH_PRIMAL_DUAL = 2, /* :463-550  AdaPDM+                                          */
  ADAPROX_S_BACKTRACKING_PROXGRAD = 3,  /* :50-64                                                     */
  ADAPROX_S_BACKTRACKING_NESTEROV = 4,  /* :66-84                                                     */
  ADAPROX_S_FIXED_NESTEROV = 5,         /* :91-142                                                    */
  ADAPROX_S_MALITSKY_POCK = 6,          /* :581-629                                                   */
  ADAPROX_S_AGRAAL = 7                  /* :150-192                                                   */
} adaprox_solver;

typedef enum {
  ADAPROX_RULE_FIXED = 0,       /* FixedStepsize            :208-215 */
  ADAPROX_RULE_MM = 1,          /* MalitskyMishchenkoRule   :217-230 */
  ADAPROX_RULE_OUR = 2,         /* OurRule                  :232-273 */
  ADAPROX_RULE_OUR_PLUS = 3     /* OurRulePlus              :277-308 */
} adaprox_rule_kind;

typedef struct {
  int32_t solver;               /* adaprox_solver                                        */
  int32_t rule;                 /* adaprox_rule_kind (solvers 0, 1)                      */
  double gamma;                 /* rule.gamma (already resolved by the front end, :241-247);
                                   gamma0 of the backtracking solvers; gamma of fixed_nesterov / AdaPDM+ */
  double t;                     /* rule.t ; AdaPDM+ t ; malitsky_pock t                  */
  double norm_A;                /* OurRule.norm_A                                        */
  double delta;                 /* OurRule.delta ; AdaPDM+ delta                         */
  double Theta;                 /* OurRule.Theta ; AdaPDM+ Theta                         */
  double xi;                    /* OurRulePlus.xi ; backtracking_proxgrad xi             */
  double nu;                    /* OurRulePlus.nu                                        */
  double r;                     /* OurRulePlus.r ; AdaPDM+ r                             */
  double R;                     /* AdaPDM+ R                                             */
  double eta;                   /* AdaPDM+ eta                                           */
  double shrink;                /* backtracking shrink                                   */
  double sigma;                 /* malitsky_pock sigma                                   */
  double muf, mug, theta;       /* fixed_nesterov (theta < 0: derive it, :111-117)       */
  double gamma_max, phi;        /* agraal                                                */
  double tol;
  int64_t maxit;
  int32_t want_objective;       /* 1: records carry f_x, g(x), h(A x) (a logger is attached, :350-352) */
  int32_t counting_f, counting_g, counting_h, counting_A;   /* which objects are wrapped in Counting */
  int64_t max_records;          /* capacity of the caller's record buffer                */
} adaprox_options;

/* one per iteration: the `@logmsg Record` payload (src/AdaProx.jl:351) */
typedef struct {
  int64_t it;
  double gamma, sigma, norm_res;
  double f_x, g_x, h_Ax;        /* objective = f_x + g_x + h_Ax (NaN when !want_objective) */
  int64_t f_evals, grad_f_evals, prox_g_evals, prox_h_evals, A_evals, At_evals;
} adaprox_record;

typedef struct {
  int64_t iters;                /* the reference's returned `it` / `numit`               */
  uint32_t flags;
  int32_t reserved;
  int64_t f_evals, grad_f_evals, prox_g_evals, prox_h_evals, A_evals, At_evals;  /* src/counting.jl */
  int64_t n_records;
  double final_gamma, final_sigma, final_norm_res;
  double solve_ms;              /* device time of the solve (CUDA events)                */
  int64_t kernel_launches;      /* library kernels launched by this call                 */
  int64_t matrix_passes;        /* sweeps over the matrix of f per gradient evaluation: 1 = single-pass
                                   fused A'(Ax-b) kernel, 2 = A*x then A'*r; 0 = f has no matrix;
                                   3 = the matrix is resident in the shared memory of one cluster for the
                                   whole solve (small dense least squares): HBM is read once per SOLVE;
                                   4 = the same with the rows spread over the shared memory of all SMs    */
  int64_t collective;           /* row-sharded solves: 1 = ncclAllReduce per iteration, 2 = all-reduce inside the sweep
                                   kernel over NVLink peer memory; 0 = single GPU                       */
} adaprox_result;

/* ---- life cycle ------------------------------------------------------------- */
int adaprox_version(void);
int adaprox_create(adaprox_handle* out, int device);
int adaprox_destroy(adaprox_handle h);
const char* adaprox_last_error(adaprox_handle h);
int adaprox_device_info(adaprox_handle h, int* sm_count, int* cc_major, int* cc_minor, int64_t* free_bytes);

/* ---- device-resident data --------------------------------------------------- */
/* `f.A` / `A`: Julia Matrix{Float64} (column-major, leading dimension lda). */
int adaprox_matrix_upload_colmajor(adaprox_handle h, const double* A, int64_t m, int64_t n, int64_t lda, adaprox_id* out);
/* numpy C-order / any row-major source. */
int adaprox_matrix_upload_rowmajor(adaprox_handle h, const double* A, int64_t m, int64_t n, int64_t lda, adaprox_id* out);
/* SparseMatrixCSC is converted to CSR by the front end; 0-based indices. The
 * library also builds the CSR of the transpose so `X' * v` needs no atomics. */
int adaprox_matrix_upload_csr(adaprox_handle h, int64_t m, int64_t n, int64_t nnz, const int64_t* rowptr,
                              const int32_t* colind, const double* vals, adaprox_id* out);
int adaprox_matrix_free(adaprox_handle h, adaprox_id mat);
int adaprox_matrix_shape(adaprox_handle h, adaprox_id mat, int64_t* m, int64_t* n, int64_t* nnz);
int adaprox_vector_upload(adaprox_handle h, const double* v, int64_t len, adaprox_id* out);
int adaprox_vector_download(adaprox_handle h, adaprox_id vec, double* out, int64_t len);
int adaprox_vector_free(adaprox_handle h, adaprox_id vec);

/* Planted lasso of lasso/runme.jl:40-77, generated on the device for the row
 * shard [row0, row0+rows) of the m x n instance (counter-based RNG, identical
 * bits on every rank and in the host generator).  Outputs: the matrix id, the
 * id of b (shard rows), x_star (host, n), the optimum value and
 * Lf = opnorm(A)^2 by `power_iters` power iterations (global when a
 * communicator is attached). */
int adaprox_generate_planted_lasso(adaprox_handle h, int64_t m, int64_t n, int64_t row0, int64_t rows,
                                   double pfactor, uint64_t seed, double lam, double rho, int32_t power_iters,
                                   adaprox_id* A_out, adaprox_id* b_out, double* x_star, double* optimum, double* Lf);

/* ---- the operator protocol, one call each (used by Counting-compatible front
 *      ends and by the parity tests) ------------------------------------------- */
/* `A * x` and `A' * y`  (src/AdaProx.jl:327,329). */
int adaprox_mul(adaprox_handle h, adaprox_id mat, const double* x, double* out);
int adaprox_amul(adaprox_handle h, adaprox_id mat, const double* y, double* out);
/* eval_with_pullback + pb()  (src/AdaProx.jl:11-16): f(x) and, if grad != NULL, the gradient. */
int adaprox_eval_f(adaprox_handle h, const adaprox_problem* p, const double* x, double* f_x, double* grad);
/* ProximalCore.prox(g, x, gamma) -> (y, g(y)).  For a conjugate (g->conjugate = 1) y is the Moreau prox of g*; *g_y is
 * then g(y_f) of the BASE function at its inner prox point, not the conjugate's value (no solver uses it: `y, _ = prox(...)`). */
int adaprox_prox_eval(adaprox_handle h, const adaprox_prox* g, const double* x, int64_t len, double gamma,
                      double* y, double* g_y);
/* stepsize(rule, state, x1, grad1, x0, grad0)  (src/AdaProx.jl:226,258,299) from the three
 * reductions the kernels fuse: dgg = |dgrad|^2, dgx = <dgrad, dx>, dxx = |dx|^2. */
int adaprox_stepsize(const adaprox_options* o, double gamma1, double gamma0_or_rho, double dgg, double dgx,
                     double dxx, double* gamma, double* sigma, double* state1);

/* logistic_loss_grad_Hessian(X, y, w) of experiments/cubic_sparse_logreg/runme.jl:34-45 -- the setup that turns a
 * logistic-regression data set into the Cubic oracle's (Q, q): H_out = [X'RX  X'sb; (X'sb)'  sum(sb)] ((n+1)^2 doubles,
 * symmetric), g_out = the logistic gradient at w (n+1).  X dense or CSR (n features), y the 0/1 labels, w of length n+1. */
int adaprox_logistic_grad_hessian(adaprox_handle h, adaprox_id X_mat, adaprox_id y_vec, const double* w,
                                  double* H_out, double* g_out);

/* ---- solvers ---------------------------------------------------------------- */
/* x0 (n), y0 (m_dual, may be NULL for proximal gradient) are read; x_out, y_out
 * (may be NULL) and `records` (max_records entries, may be NULL) are written. */
int adaprox_solve(adaprox_handle h, const adaprox_problem* p, const adaprox_options* o, const double* x0,
                  const double* y0, double* x_out, double* y_out, adaprox_record* records, adaprox_result* res);

/* ---- batched multi-lambda path (BASELINE config 5) ----------------------------- */
/* AdaPGM (src/AdaProx.jl:418-421 -> :312-364 with A = 0, h = Zero) on the L problems
 *     min_x f(x) + lambdas[j] |x|_1 ,  j = 0 .. L-1
 * that share the smooth term f of `p` (p->g is ignored).  f is
 *   - least squares 1/2 |A x - b|^2 (lasso/runme.jl:16-27) over a dense or a CSR matrix, or
 *   - the logistic loss of sparse_logreg/runme.jl:18-39 over a CSR matrix (n = features + 1, intercept last and
 *     penalised by the l1 term like every other entry).
 * Dense logistic, a row-sharded matrix and other f kinds return ADAPROX_ERR_UNSUPPORTED.  The reference has no batched
 * entry point: running adaptive_proxgrad once per lambda is the behaviour this call reproduces column by column -- every
 * column has its own stepsize state, residual and stopping iteration and is frozen when it converges (its result is the
 * iterate the single-lambda call returns).  The L iterates advance together: for a dense matrix A*X and A'*R are fp64
 * tensor-core contractions (mma.sync DMMA) instead of 2 L matrix-vector products; for a CSR matrix both sweeps gather whole
 * lambda-contiguous rows of the iterate / residual block, so every gathered 32-byte sector is used.
 *   gamma0  : L initial stepsizes, or NULL to use o->gamma for every column; with FixedStepsize column j keeps
 *             gamma0[j] for every step.  maxit = 0 returns x_1 = prox(x_0 - gamma_0 grad f(x_0)) with iters 0, as
 *             adaptive_proxgrad does
 *   x0T     : [L][n] (column j contiguous), or NULL for zeros
 *   x_outT  : [L][n];  iters / norm_res / gamma_out / f_out : [L] (each may be NULL)
 *   hist    : optional 3 * hist_rows * L doubles: gamma, norm_res, objective per (iteration - 1, column); NaN where a
 *             column had already stopped.  res->iters = largest per-column iteration count. */
int adaprox_solve_lambda_path(adaprox_handle h, const adaprox_problem* p, const adaprox_options* o, int64_t L,
                              const double* lambdas, const double* gamma0, const double* x0T, double* x_outT,
                              int64_t* iters, double* norm_res, double* gamma_out, double* f_out,
                              double* hist, int64_t hist_rows, adaprox_result* res);
/* which: 0 = R = A X - b (K = n), 1 = G = A' R (K = m); mean device ms per launch over `reps` launches on an L-column
 * batch of zeros (measurement hook of tools/bench_configs.py) */
int adaprox_time_path_gemm(adaprox_handle h, adaprox_id mat, int64_t L, int which, int reps, double* ms_per_launch);

/* ---- row-sharded multi-GPU (one process per GPU) ---------------------------- */
/* NCCL bootstrap: rank 0 calls unique_id, the host side broadcasts the 128
 * bytes, every rank calls comm_init.  After that, solves on matrices flagged as
 * row shards all-reduce the A'r partials and the stepsize scalars once per
 * iteration. */
int adaprox_comm_unique_id(void* id128);
int adaprox_comm_init(adaprox_handle h, int nranks, int rank, const void* id128);
int adaprox_comm_info(adaprox_handle h, int* nranks, int* rank);
/* Optional: in-kernel all-reduce over NVLink peer memory for row-sharded dense least squares (replaces the NCCL call
 * of every iteration).  After comm_init every rank calls p2p_export (allocates its exchange block for vectors of up to
 * n_max entries and returns a 64-byte CUDA IPC handle), the host side all-gathers the handles (rank order), every rank
 * calls p2p_attach.  All ranks must then issue the same sharded solves in the same order. */
int adaprox_p2p_export(adaprox_handle h, int64_t n_max, void* ipc_handle64);
int adaprox_p2p_attach(adaprox_handle h, int nranks, int rank, const void* ipc_handles);
/* After a sharded solve returned ADAPROX_ERR_COMM (a peer did not arrive within 5 s): clears this rank's exchange flags,
 * counters and error flag.  Every rank calls it, then the host side synchronises the ranks (no kernel of the failed solve
 * may still be running anywhere) before the next sharded solve. */
int adaprox_p2p_reset(adaprox_handle h);
/* mark a matrix as the local row block [row0, row0+rows) of an m_global-row matrix */
int adaprox_matrix_set_shard(adaprox_handle h, adaprox_id mat, int64_t m_global, int64_t row0);

/* ---- measurement hooks (bench.py) ------------------------------------------- */
/* Launch `reps` back-to-back passes of one kernel family on the handle's stream
 * and return the mean device time per pass in ms (CUDA events on that stream).
 * which: 0 = gemv_n (A*x partials + finalize), 1 = gemv_t (A'r partials + finalize). */
int adaprox_time_kernel(adaprox_handle h, adaprox_id mat, int which, int reps, double* ms_per_pass);

#ifdef __cplusplus
}
#endif
#endif /* ADAPROX_H */
