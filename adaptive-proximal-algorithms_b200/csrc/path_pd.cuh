// path_pd.cuh -- the batched C path of the dual SVM (dual_svm/runme.jl:47-59): AdaPDM / Condat-Vu on the L problems
//     min_x f(x) + IndBox(lower, upper_j)(x) + IndZero(a' x),   j = 0 .. L-1,
// that share the smooth term f = Quadratic(Q, q) or QuadraticGram(Z, q) and the one-row linear map A = a' (a = labels).
// The L iterates are the columns of X; the gradients G = Q X + q 1' (dense Q: one contraction) or G = Z (Z' X) + q 1'
// (Gram form: two) run on the DMMA engine of path_gemm.cuh unchanged.  The dual variable of a column is one scalar, A x
// is one dot product and A' y is y a, so everything else of an iteration -- stepsize rule, dual step, primal step,
// records -- is one CTA per column (k_path_pd_step).
//
// Layout: columns contiguous, XT / GT / VT [L][ldN] and UT [L][ldd], zero padded, as in the dense lambda path.
#pragma once
#include "path_gemm.cuh"

namespace adaprox {

// UT[j][c] = sum over z of slabs[z][j][c], slab order (deterministic): the K slabs of U = Z' X.  Grid (c blocks, L).
__global__ void __launch_bounds__(256) k_path_slab_sum(const double* slabs, int ks, int64_t stride, int64_t d, int64_t ldd,
                                                       double* UT) {
  const int64_t j = blockIdx.y;
  for (int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x; c < d; c += (int64_t)gridDim.x * 256) {
    double s = 0.0;
    for (int z = 0; z < ks; ++z) s += slabs[(int64_t)z * stride + j * ldd + c];
    UT[j * ldd + c] = s;
  }
}

struct PdPathCol {         // per-column solver state
  double gamma, sigma, s0, s1, norm_res, f_x;
  double upper;            // the column's box bound C_j
  double y;                // dual scalar
  double ax_prev;          // A x of the previous iterate
  long long it_done;       // iteration at which the column stopped
  unsigned flags;
  int done;                // 1: stopped (frozen)
};

struct PdPathStepArgs {
  int64_t n, ldx, L;
  DOpts O;
  double lower;
  const double* a;         // the row of A (n)
  const double* q;         // linear term of f (n)
  double* XT[3];           // iterate ring [L][ldx]
  const double* GT[2];     // gradient ring, G = grad f(X)
  double* VT;              // v = x - gamma (g + A'y)
  double* XoutT;           // result columns
  PdPathCol* col;
  double* gamma_hist; double* res_hist; double* obj_hist;   // optional [max_records][L]
  long long it;            // iteration being finished (0 = prologue)
  int* n_active;           // columns still running after this step (device counter)
};

// One iteration of k_primal_dual<false> (solver_pd.cuh P4-P7) for one column: A = a' (one row), h = IndZero,
// g = IndBox(lower, upper_j).  it = 0 is the prologue x_1 = prox(x_0 - gamma_0 (grad f(x_0) + A' y_0)) (:327-332).
__global__ void __launch_bounds__(kPT, 2) k_path_pd_step(PdPathStepArgs a) {
  constexpr int K = 8;
  __shared__ double s_scr[kPT / 32 * K];
  __shared__ double s_bc[K];
  const int64_t j = blockIdx.x;
  const long long it = a.it;
  PdPathCol st = a.col[j];
  if (st.done) return;                                                 // frozen: result and history stay as they are
  const double* x = a.XT[it % 3] + j * a.ldx;
  const double* x_prev = a.XT[(it + 2) % 3] + j * a.ldx;
  double* xn = a.XT[(it + 1) % 3] + j * a.ldx;
  const double* grad = a.GT[it & 1] + j * a.ldx;
  const double* grad_prev = a.GT[(it + 1) & 1] + j * a.ldx;
  double* v = a.VT + j * a.ldx;
  const double lo = a.lower, hi = st.upper;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  // A x, the two value sums x'G and x'q, box violations of x (g(x) of the record); it > 0: |primal_res|^2 (:338, with the
  // old gamma and A'y_it = y a), |dgrad|^2, <dgrad, dx>, |dx|^2
  double gamma = st.gamma, sigma = st.sigma, s0 = st.s0, s1 = st.s1;
  {
    double acc[K] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    const double yd = st.y;
    for (int64_t q = threadIdx.x; q < a.n; q += kPT) {
      const double xj = x[q], gj = grad[q], aj = __ldg(a.a + q);
      acc[0] = fma(aj, xj, acc[0]);
      acc[1] = fma(xj, gj, acc[1]);
      acc[2] = fma(xj, __ldg(a.q + q), acc[2]);
      acc[3] += (xj < lo || xj > hi) ? 1.0 : 0.0;
      if (it > 0) {
        const double pr = (v[q] - xj) / gamma + gj + aj * yd;
        const double dg = gj - grad_prev[q], dx = xj - x_prev[q];
        acc[4] = fma(pr, pr, acc[4]);
        acc[5] = fma(dg, dg, acc[5]);
        acc[6] = fma(dg, dx, acc[6]);
        acc[7] = fma(dx, dx, acc[7]);
      }
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const double s = warp_sum(acc[k]);
      if (lane == 0) s_scr[warp * K + k] = s;
    }
    __syncthreads();
    if (threadIdx.x < K) {
      double s = 0.0;
#pragma unroll
      for (int w = 0; w < kPT / 32; ++w) s += s_scr[w * K + threadIdx.x];
      s_bc[threadIdx.x] = s;
    }
    __syncthreads();
  }
  const double ax = s_bc[0];
  const double f_x = 0.5 * (s_bc[1] + s_bc[2]);                        // x'(Q x + q) / 2 + q'x / 2 = f_value (phases.cuh)
  double y = st.y, norm_res = st.norm_res;
  unsigned flags = st.flags;
  bool stop = false;
  if (it > 0) {
    DOpts Oc = a.O;
    if (Oc.rule == ADAPROX_RULE_FIXED) Oc.gamma = gamma;                 // the column's own fixed stepsize (gamma0)
    const double gamma_old = gamma;                                      // :340
    rule_step(Oc, s_bc[5], s_bc[6], s_bc[7], gamma, sigma, s0, s1);      // :341
    const double rho = gamma / gamma_old;                                // :342
    const double w = y + sigma * ((1.0 + rho) * ax - rho * st.ax_prev);  // :344
    const double y_new = w;                                              // :345  prox of sigma h* = Zero: the identity
    const double dr = (w - y_new) / sigma - ax;                          // :347
    norm_res = sqrt(norm_sq_jl(s_bc[4]) + norm_sq_jl(dr * dr));          // :348
    if (!(gamma == gamma) || !(norm_res == norm_res) || isinf(gamma)) flags |= ADAPROX_FLAG_NONFINITE;
    y = y_new;
    if (norm_res <= a.O.tol) stop = true;                                // :354
    if (a.gamma_hist != nullptr && it <= a.O.max_records && threadIdx.x == 0) {   // :350-352
      a.gamma_hist[(it - 1) * a.L + j] = gamma;
      a.res_hist[(it - 1) * a.L + j] = norm_res;
      a.obj_hist[(it - 1) * a.L + j] = f_x + prox_value_finish(ADAPROX_P_IND_BOX, 0.0, s_bc[3]) +
                                       prox_value_finish(ADAPROX_P_IND_ZERO, 0.0, ax != 0.0 ? 1.0 : 0.0);
    }
  }
  const bool last = !stop && it >= a.O.maxit;
  if (stop) {
    // converged: the result is x_it and the y that was just formed (:353-355)
    for (int64_t q = threadIdx.x; q < a.n; q += kPT) a.XoutT[j * a.ldx + q] = x[q];
  } else {
    // v = x - gamma (grad + A'y), x+ = prox_{gamma g}(v) (:359-361); after the last iteration x+ is the result (:361-363)
    for (int64_t q = threadIdx.x; q < a.n; q += kPT) {
      const double vj = x[q] - gamma * (grad[q] + __ldg(a.a + q) * y);
      v[q] = vj;
      const double xj = vj < lo ? lo : (vj > hi ? hi : vj);
      xn[q] = xj;
      if (last) a.XoutT[j * a.ldx + q] = xj;
    }
  }
  if (threadIdx.x == 0) {
    st.gamma = gamma; st.sigma = sigma; st.s0 = s0; st.s1 = s1; st.norm_res = norm_res; st.f_x = f_x;
    st.y = y; st.ax_prev = ax;
    if (stop || last) {
      st.done = 1; st.it_done = it;
      st.flags = flags | (stop ? ADAPROX_FLAG_CONVERGED : 0u);
    } else {
      st.flags = flags;
      atomicAdd(a.n_active, 1);
    }
    a.col[j] = st;
  }
}

}  // namespace adaprox
