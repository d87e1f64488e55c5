// path_lin.cuh -- the batched lambda path of the primal-dual experiments least_absolute_deviation/runme.jl and
// square_root_lasso/runme.jl: AdaPDM / Condat-Vu on the L problems
//     min_x lambda_j |x|_1 + h(A x),   j = 0 .. L-1,
// with f = Zero, h = NormL1 or NormL2 (optionally Translate'd: h = |. - b|) and one dense m x n matrix A.  The L iterates
// are the columns of X, the L dual vectors the columns of Y, so the two matrix products of an iteration are the DMMA
// contractions of path_gemm.cuh, unchanged:  AX = A X (mode 1, b = 0) and ATY = A' Y (mode 2, its K slabs kept apart).
// Everything else is one CTA per column: k_path_lin_dual (stepsize, dual step, residual, record, stop) between the two
// contractions and k_path_lin_primal (v, soft threshold) after the second.
//
// Layout: columns contiguous, XT [L][ldx], AXT / YT [L][ldr], zero padded (the tile loads read the padding), as in the
// dense lambda path.  f = Zero makes grad f = 0, so the rule's |dgrad|^2 and <dgrad, dx> are exactly 0 and no gradient is
// stored; the primal kernel forms the next iteration's |primal_res|^2 and |dx|^2 in its own pass, from the same operands
// k_primal_dual<false> reads in P4 (v, x+, the gamma that formed v, A'y).
#pragma once
#include "path_gemm.cuh"

namespace adaprox {

struct LinPathCol {        // per-column solver state
  double gamma, sigma, s0, s1, norm_res;
  double lambda;           // weight of g = NormL1
  double pr2, dx2, l1;     // |primal_res|^2, |x - x_prev|^2 and |x|_1 of the current iterate (from the primal kernel)
  long long it_done;       // iteration at which the column stopped
  unsigned flags;
  int done;                // 1: stopped (frozen)
};

struct LinPathArgs {
  int64_t n, m, ldx, ldr, L;
  DOpts O;
  DProx g, h;              // g = NormL1 (its weight is the column's lambda), h = NormL1 / NormL2 on the m rows
  double* XT[2];           // iterate ring [L][ldx]
  const double* AXT[2];    // A x of the iterate ring [L][ldr]
  double* YT;              // dual iterates [L][ldr], updated in place
  const double* ATY;       // A'y: ksplit slabs [ksplit][L][ldx], summed in slab order
  int ksplit; int64_t gstride;
  double* XoutT;           // result columns [L][ldx]
  LinPathCol* col;
  double* gamma_hist; double* res_hist; double* obj_hist;   // optional [max_records][L]
  long long it;            // iteration (0 = prologue)
  int* n_active;           // columns still running after this iteration (device counter)
};

// sums K per-thread values over the CTA in a fixed order (warp butterflies, then warps in order); every thread gets them
template <int K>
__device__ __forceinline__ void lin_block_sum(double (&v)[K], double* s_scr) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const double s = warp_sum(v[k]);
    if (lane == 0) s_scr[warp * K + k] = s;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kPT / 32; ++w) s += s_scr[w * K + k];
    v[k] = s;
  }
  __syncthreads();
}

// P5-P6 of k_primal_dual<false> (src/AdaProx.jl:340-356) for one column, it >= 1: rule step, the dual step
// y+ = prox_{sigma h*}(w) over the m rows (in place), |dual_res|^2, norm_res, the record, the convergence test.
__global__ void __launch_bounds__(kPT, 2) k_path_lin_dual(LinPathArgs a) {
  __shared__ double s_scr[kPT / 32 * 2];
  const int64_t j = blockIdx.x;
  const long long it = a.it;
  LinPathCol st = a.col[j];
  if (st.done) return;                                                 // frozen: result and history stay as they are
  const double* ax = a.AXT[it & 1] + j * a.ldr;
  const double* ax_prev = a.AXT[(it + 1) & 1] + j * a.ldr;
  double* y = a.YT + j * a.ldr;

  double gamma = st.gamma, sigma = st.sigma, s0 = st.s0, s1 = st.s1;
  DOpts Oc = a.O;
  if (Oc.rule == ADAPROX_RULE_FIXED) Oc.gamma = gamma;                   // the column's own fixed stepsize (gamma0)
  const double gamma_old = gamma;                                        // :340
  rule_step(Oc, 0.0, 0.0, st.dx2, gamma, sigma, s0, s1);                 // :341 (grad f = 0)
  const double rho = gamma / gamma_old;                                  // :342
  // NormL2: |w / sigma + shift|^2 over the whole column before any y is written (dual_rows' l2sum)
  double l2scale = 0.0;
  if (a.h.kind == ADAPROX_P_NORM_L2) {
    double acc[1] = {0.0};
#pragma unroll 4
    for (int64_t i = threadIdx.x; i < a.m; i += kPT) {
      const double wi = y[i] + sigma * ((1.0 + rho) * ax[i] - rho * ax_prev[i]);   // :344
      const double z = prox_l2_arg(a.h, wi / sigma, i);
      acc[0] = fma(z, z, acc[0]);
    }
    lin_block_sum<1>(acc, s_scr);
    l2scale = prox_l2_scale(a.h.lambda, 1.0 / sigma, acc[0]);
  }
  const bool rec = a.gamma_hist != nullptr && it <= a.O.max_records;
  double acc[2] = {0.0, 0.0};                                            // |dual_res|^2, h(A x) sum
#pragma unroll 4
  for (int64_t i = threadIdx.x; i < a.m; i += kPT) {
    const double axi = ax[i];
    const double wi = y[i] + sigma * ((1.0 + rho) * axi - rho * ax_prev[i]);       // :344
    const double yi = prox_conj_elem(a.h, wi, sigma, i, l2scale);                  // :345
    y[i] = yi;
    const double dr = (wi - yi) / sigma - axi;                                     // :347
    acc[0] = fma(dr, dr, acc[0]);
    if (rec) acc[1] += prox_value_elem(a.h, axi, i);
  }
  lin_block_sum<2>(acc, s_scr);
  const double norm_res = sqrt(norm_sq_jl(st.pr2) + norm_sq_jl(acc[0]));          // :348
  if (threadIdx.x != 0) return;
  unsigned flags = st.flags;
  if (!(gamma == gamma) || !(norm_res == norm_res) || isinf(gamma)) flags |= ADAPROX_FLAG_NONFINITE;
  if (rec) {                                                                       // :350-352
    a.gamma_hist[(it - 1) * a.L + j] = gamma;
    a.res_hist[(it - 1) * a.L + j] = norm_res;
    a.obj_hist[(it - 1) * a.L + j] = prox_value_finish(ADAPROX_P_NORM_L1, st.lambda, st.l1) +
                                     prox_value_finish(a.h.kind, a.h.lambda, acc[1]);
  }
  st.gamma = gamma; st.sigma = sigma; st.s0 = s0; st.s1 = s1; st.norm_res = norm_res;
  if (norm_res <= a.O.tol) {                                                       // :354: the result is x_it and this y
    st.done = 1; st.it_done = it; flags |= ADAPROX_FLAG_CONVERGED;
  }
  st.flags = flags;
  a.col[j] = st;
}

// P7 of k_primal_dual<false> (:359-361) for one column: A'y from its K slabs (slab order), v = x - gamma A'y,
// x+ = prox_{gamma lambda_j |.|_1}(v), and in the same pass the next iteration's |primal_res|^2 = |(v - x+) / gamma + A'y|^2
// (:338), |x+ - x|^2 and, for its record, |x+|_1.  it = 0 is the prologue x_1 = prox(x_0 - gamma_0 A'y_0) (:330-332).  A column
// that converged in this iteration copies x_it out; after iteration maxit x+ is the result (:361-363).
__global__ void __launch_bounds__(kPT, 2) k_path_lin_primal(LinPathArgs a) {
  __shared__ double s_scr[kPT / 32 * 3];
  const int64_t j = blockIdx.x;
  const long long it = a.it;
  LinPathCol st = a.col[j];
  if (st.done && st.it_done < it) return;                              // frozen earlier
  const double* x = a.XT[it & 1] + j * a.ldx;
  double* xout = a.XoutT + j * a.ldx;
  if (st.done) {
    for (int64_t q = threadIdx.x; q < a.n; q += kPT) xout[q] = x[q];
    return;
  }
  double* xn = a.XT[(it + 1) & 1] + j * a.ldx;
  const double* aty = a.ATY + j * a.ldx;
  const bool last = it >= a.O.maxit;
  const bool rec = a.gamma_hist != nullptr && it + 1 <= a.O.max_records;
  DProx g = a.g;
  g.lambda = st.lambda;
  const double gamma = st.gamma;
  double acc[3] = {0.0, 0.0, 0.0};
  for (int64_t q = threadIdx.x; q < a.n; q += kPT) {
    double s = 0.0;
    for (int z = 0; z < a.ksplit; ++z) s += aty[(int64_t)z * a.gstride + q];
    const double xj = x[q];
    const double vj = xj - gamma * s;                                  // :359 (grad f = 0)
    const double xp = prox_elem(g, vj, gamma, q, 0.0);                 // :361
    xn[q] = xp;
    if (last) xout[q] = xp;
    const double pr = (vj - xp) / gamma + s;                           // :338 of the next iteration
    const double dx = xp - xj;
    acc[0] = fma(pr, pr, acc[0]);
    acc[1] = fma(dx, dx, acc[1]);
    if (rec) acc[2] += prox_value_elem(g, xp, q);
  }
  lin_block_sum<3>(acc, s_scr);
  if (threadIdx.x != 0) return;
  st.pr2 = acc[0]; st.dx2 = acc[1]; st.l1 = acc[2];
  if (last) {
    st.done = 1; st.it_done = it;
  } else {
    atomicAdd(a.n_active, 1);
  }
  a.col[j] = st;
}

}  // namespace adaprox
