// path_csr.cuh -- the batched multi-lambda path for a CSR smooth term: AdaPGM on the L problems
//     min_x f(x) + lambda_j |x|_1 ,  j = 0 .. L-1,
// that share f = least squares 1/2 |X x - b|^2 (lasso/runme.jl:16-27) or the logistic loss of sparse_logreg/runme.jl:18-39
// (intercept last, penalised by NormL1 like every other entry).  Host side: path_csr.inl.
//
// Layout: every block is lambda-CONTIGUOUS, [rows][ldL] with ldL = L rounded up to 32 (iterate ring, gradient ring, v, the
// result block, the residual block P).  Both matrix passes are then "CSR row x row-major dense block":
//   X W  : CSR(X)  row i gathers rows W[colind] -> P[i][.]  = 1/u - y (logistic) or r = X w - b (least squares)
//   X' P : CSR(X') row j gathers rows P[colind] -> G[j][.]  (/ N for logistic)
// Each gathered row is ldL contiguous doubles, so the 32-byte sectors of the single-lambda gather (one double per sector,
// gemv.cuh spmv_rows_t) are fully used.
//
// Work split: one warp per CSR row, lane l owns columns l, l + 32, ... of a column tile of 32 NQ columns; every lane adds
// the row's nonzeros sequentially in CSR order (no atomics, no cross-lane reduction).  A CTA owns kCPRows consecutive rows
// (a partition that does not depend on L) and writes one partial per (CTA, quantity, column); k_csr_path_finish adds the
// partials in CTA order.  So every sum of column j is formed in an order that depends on neither L nor j: reruns are
// bit-identical and permuting the lambdas permutes the columns bit for bit.
// Padding columns (L <= c < ldL) are never stepped, never counted and never written out; their P and G entries are 0.
#pragma once
#include "path_gemm.cuh"

namespace adaprox {

constexpr int kCPWarps = 8, kCPThreads = kCPWarps * 32;
constexpr int kCPRowsPerWarp = 4;
constexpr int kCPRows = kCPWarps * kCPRowsPerWarp;   // CSR rows per CTA of a sweep
constexpr int kCPU = 4;                              // nonzeros of a row whose gathers are issued together
constexpr int kCPFinWarps = 16;                      // warps of k_csr_path_finish (they split the partials of a column)
constexpr int kCPFwdK = 2, kCPBwdK = 5;              // partial sums per column written by each sweep

enum { CP_STEP = 0, CP_CONV = 1, CP_MAXIT = 2, CP_FROZEN = 3 };

struct CsrColStep {        // what k_csr_path_finish decided for a column, read by k_csr_path_prox and the next X' P sweep
  double gamma, gl;        // stepsize of v = x - gamma g, threshold gamma * lambda
  int mode, pad;           // CP_*
};

struct CsrPathArgs {
  int f_kind;
  int64_t m, n, nfeat;     // rows of X, unknowns, columns of X (n - 1 for logistic: the intercept is row n - 1 of the blocks)
  int64_t L, ldL;
  double N;                // logistic: number of samples
  const int64_t* rowptr; const int* colind; const double* vals;          // CSR(X)
  const int64_t* t_rowptr; const int* t_colind; const double* t_vals;    // CSR(X')
  const double* yb;        // b (least squares) / labels y (logistic), [m]
  double* X[3];            // iterate ring [n][ldL]
  double* G[2];            // gradient ring
  double* V;               // v = x - gamma g
  double* Xout;            // result columns
  double* P;               // residual block [m][ldL]
  double* fpart; int64_t fblocks;   // [fblocks][kCPFwdK][ldL]: value sum, logistic intercept sum
  double* tpart; int64_t tblocks;   // [tblocks][kCPBwdK][ldL]: |primal_res|^2, |dg|^2, <dg,dx>, |dx|^2, |x|_1
  PathCol* col;
  CsrColStep* step;
  DOpts O;
  double* gamma_hist; double* res_hist; double* obj_hist;   // optional [max_records][L]
  long long it;            // iteration being evaluated / finished (0 = prologue)
  int want_l1;             // this iteration is recorded: the X' P sweep also sums |x|
  int* n_active;           // columns still running after this iteration (device counter)
};

// MODE 0: X W (rows of X, gathers the iterate block), MODE 1: X' P (rows of X', gathers the residual block).
// NQ = 32-column chunks per lane of a column tile (blockIdx.y); dynamic shared memory: kCPWarps * K * 32 NQ doubles.
template <int MODE, int NQ>
__device__ __forceinline__ void csr_path_sweep(const CsrPathArgs& a) {
  constexpr int K = (MODE == 0) ? kCPFwdK : kCPBwdK;
  constexpr int CT = 32 * NQ;
  extern __shared__ double s_acc[];                  // [warp][K][CT]: per-warp running sums of the row epilogues
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool logistic = a.f_kind == ADAPROX_F_LOGISTIC;
  const long long it = a.it;
  const int64_t ldL = a.ldL;
  const int64_t nrows = (MODE == 0) ? a.m : a.nfeat;
  const int64_t* __restrict__ rp = (MODE == 0) ? a.rowptr : a.t_rowptr;
  const int* __restrict__ ci = (MODE == 0) ? a.colind : a.t_colind;
  const double* __restrict__ va = (MODE == 0) ? a.vals : a.t_vals;
  const double* __restrict__ src = (MODE == 0) ? a.X[it % 3] : a.P;
  const int64_t tile0 = (int64_t)blockIdx.y * CT;
  const int nqv = (int)min((int64_t)NQ, (ldL - tile0) / 32);   // chunks of this tile inside the block (ldL is a multiple of 32)
  const int64_t c0 = tile0 + lane;
  double* sw = s_acc + warp * K * CT;
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int q = 0; q < NQ; ++q) sw[k * CT + lane + 32 * q] = 0.0;
  const bool partials = (MODE == 0) || it > 0;
  double cst[NQ];                                    // MODE 0: intercept of the column (logistic); MODE 1: old gamma of the column
#pragma unroll
  for (int q = 0; q < NQ; ++q) {
    const int64_t c = c0 + 32 * q;
    cst[q] = 0.0;
    if (q < nqv && c < a.L) {
      if (MODE == 0 && logistic) cst[q] = src[(a.n - 1) * ldL + c];
      if (MODE == 1 && it > 0) cst[q] = a.step[c].gamma;
    }
  }
  const double* xc = a.X[it % 3];
  const double* xp = a.X[(it + 2) % 3];
  const double* gp = a.G[(it + 1) & 1];
  double* gout = a.G[it & 1];

  const int64_t rbeg = (int64_t)blockIdx.x * kCPRows + warp * kCPRowsPerWarp;
  for (int rr = 0; rr < kCPRowsPerWarp; ++rr) {
    const int64_t row = rbeg + rr;
    if (row >= nrows) break;                         // warp-uniform
    double acc[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) acc[q] = 0.0;
    const int64_t k0 = rp[row], k1 = rp[row + 1];
    for (int64_t kb = k0; kb < k1; kb += 32) {
      const int cnt = (int)min((int64_t)32, k1 - kb);
      int cl = 0;
      double vl = 0.0;
      if (lane < cnt) { cl = ci[kb + lane]; vl = va[kb + lane]; }   // 32 nonzeros per coalesced load, then broadcast
      for (int u0 = 0; u0 < cnt; u0 += kCPU) {
        int cc[kCPU];
        double vv[kCPU], g[kCPU][NQ];
#pragma unroll
        for (int u = 0; u < kCPU; ++u) {
          cc[u] = __shfl_sync(0xffffffffu, cl, u0 + u);
          vv[u] = __shfl_sync(0xffffffffu, vl, u0 + u);
        }
#pragma unroll
        for (int u = 0; u < kCPU; ++u)
#pragma unroll
          for (int q = 0; q < NQ; ++q)
            g[u][q] = (u0 + u < cnt && q < nqv) ? __ldg(src + (int64_t)cc[u] * ldL + c0 + 32 * q) : 0.0;
#pragma unroll
        for (int u = 0; u < kCPU; ++u)
          if (u0 + u < cnt)                          // warp-uniform: the sum runs over the row's nonzeros in CSR order
#pragma unroll
            for (int q = 0; q < NQ; ++q) acc[q] = fma(vv[u], g[u][q], acc[q]);
      }
    }
    // row epilogue
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      if (q >= nqv) break;
      const int64_t c = c0 + 32 * q;
      const int s = lane + 32 * q;
      const int64_t e = row * ldL + c;
      if (MODE == 0) {
        double pv = 0.0;
        if (c < a.L) {
          const double yi = a.yb[row];
          if (logistic) {                            // sparse_logreg/runme.jl:24-36, as f_phase_B
            const double logits = acc[q] + cst[q];
            const double u = 1.0 + exp(-logits);
            const double ri = 1.0 / u - yi;          // probs - y
            pv = ri;
            sw[s] += (yi - 1.0) * logits - log(u);
            sw[CT + s] += ri;
          } else {                                   // lasso/runme.jl:22
            const double res = acc[q] - yi;
            pv = res;
            sw[s] = fma(res, res, sw[s]);
          }
        }
        a.P[e] = pv;
      } else {
        double gj = 0.0;
        if (c < a.L) {
          gj = logistic ? acc[q] / a.N : acc[q];     // grad_slice: X' r / N
          if (it > 0) {
            const double xj = xc[e];
            const double pr = (a.V[e] - xj) / cst[q] + gj;                   // src/AdaProx.jl:338 (old gamma)
            const double dg = gj - gp[e], dx = xj - xp[e];
            sw[s] = fma(pr, pr, sw[s]);
            sw[CT + s] = fma(dg, dg, sw[CT + s]);
            sw[2 * CT + s] = fma(dg, dx, sw[2 * CT + s]);
            sw[3 * CT + s] = fma(dx, dx, sw[3 * CT + s]);
            if (a.want_l1) sw[4 * CT + s] += fabs(xj);
          }
        }
        gout[e] = gj;
      }
    }
  }
  __syncthreads();
  if (!partials) return;
  // this CTA's partials: the warps' sums added in warp order (= row order)
  double* part = (MODE == 0) ? a.fpart : a.tpart;
  for (int t = threadIdx.x; t < nqv * 32; t += kCPThreads) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      double v = 0.0;
#pragma unroll
      for (int w = 0; w < kCPWarps; ++w) v += s_acc[(w * K + k) * CT + t];
      part[((int64_t)blockIdx.x * K + k) * ldL + tile0 + t] = v;
    }
  }
}

template <int NQ>
__global__ void __launch_bounds__(kCPThreads) k_csr_path_xw(CsrPathArgs a) { csr_path_sweep<0, NQ>(a); }
template <int NQ>
__global__ void __launch_bounds__(kCPThreads) k_csr_path_xtp(CsrPathArgs a) { csr_path_sweep<1, NQ>(a); }

// sum of p[b * stride] over b = b0, b0 + step, ... < count, added in that order; eight loads in flight
__device__ __forceinline__ double cp_strided_sum(const double* p, int64_t count, int64_t stride, int64_t b0, int64_t step) {
  double s = 0.0;
  for (int64_t b = b0; b < count; b += 8 * step) {
    double v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = (b + u * step < count) ? p[(b + u * step) * stride] : 0.0;
#pragma unroll
    for (int u = 0; u < 8; ++u) if (b + u * step < count) s += v[u];
  }
  return s;
}

// Per-column finish of an iteration (src/AdaProx.jl:334-362 with A = 0, h = Zero; the CSR form of k_path_step): one CTA per
// 32 columns, lane = column.  Warp w adds the partials of CTAs w, w + 16, ... in order, then warp 0 adds the 16 warp sums in
// order; the logistic intercept (row n - 1, not part of X' P) is added last, as it is the last entry of the single-lambda sums.
__global__ void __launch_bounds__(kCPFinWarps * 32) k_csr_path_finish(CsrPathArgs a) {
  constexpr int NS = kCPFwdK + kCPBwdK;
  __shared__ double s_w[kCPFinWarps][NS][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t c = (int64_t)blockIdx.x * 32 + lane;
  const long long it = a.it;
  const int64_t ldL = a.ldL;
#pragma unroll
  for (int k = 0; k < kCPFwdK; ++k) s_w[warp][k][lane] = cp_strided_sum(a.fpart + k * ldL + c, a.fblocks, kCPFwdK * ldL, warp, kCPFinWarps);
  const int kb = it == 0 ? 0 : (a.want_l1 ? kCPBwdK : kCPBwdK - 1);       // the X' P partials exist from iteration 1 on
  for (int k = 0; k < kCPBwdK; ++k)
    s_w[warp][kCPFwdK + k][lane] = k < kb ? cp_strided_sum(a.tpart + k * ldL + c, a.tblocks, kCPBwdK * ldL, warp, kCPFinWarps) : 0.0;
  __syncthreads();
  if (warp != 0) return;
  double tot[NS];
#pragma unroll
  for (int k = 0; k < NS; ++k) {
    double s = 0.0;
    for (int w = 0; w < kCPFinWarps; ++w) s += s_w[w][k][lane];
    tot[k] = s;
  }
  const bool live = c < a.L;
  bool stepping = false;
  if (live) {
    const bool logistic = a.f_kind == ADAPROX_F_LOGISTIC;
    PathCol st = a.col[c];
    const bool frozen = st.it_done != 0;
    const double f_x = logistic ? -(tot[0] / a.N) : 0.5 * norm_sq_jl(tot[0]);    // f_value
    const int64_t ie = (a.n - 1) * ldL + c;          // logistic: intercept entry
    const double* x = a.X[it % 3];
    double g_end = 0.0;
    if (logistic) {
      g_end = tot[1] / a.N;                          // grad_slice: mean(1/u - y)
      a.G[it & 1][ie] = g_end;
    }
    double gamma = st.gamma, sigma = st.sigma, s0 = st.s0, s1 = st.s1;
    double norm_res = st.norm_res;
    bool stop = false;
    if (it > 0 && !frozen) {
      double spr = tot[2], sgg = tot[3], sgx = tot[4], sxx = tot[5];
      if (logistic) {
        const double xj = x[ie];
        const double pr = (a.V[ie] - xj) / gamma + g_end;
        const double dg = g_end - a.G[(it + 1) & 1][ie], dx = xj - a.X[(it + 2) % 3][ie];
        spr = fma(pr, pr, spr); sgg = fma(dg, dg, sgg); sgx = fma(dg, dx, sgx); sxx = fma(dx, dx, sxx);
      }
      DOpts Oc = a.O;
      if (Oc.rule == ADAPROX_RULE_FIXED) Oc.gamma = gamma;                      // the column's own fixed stepsize (gamma0)
      const double gamma_prev = gamma;
      rule_step(Oc, sgg, sgx, sxx, gamma, sigma, s0, s1);                      // :341
      norm_res = sqrt(norm_sq_jl(spr) + adapgm_dual_res_sq(gamma, gamma_prev, sigma));   // :348
      if (norm_res <= a.O.tol) stop = true;                                     // :354
    }
    if (a.want_l1 && !frozen) {                      // record of iteration `it`: gamma, norm_res, f(x) + lambda |x|_1
      double l1 = tot[6];
      if (logistic) l1 += fabs(x[ie]);
      a.gamma_hist[(it - 1) * a.L + c] = gamma;
      a.res_hist[(it - 1) * a.L + c] = norm_res;
      a.obj_hist[(it - 1) * a.L + c] = f_x + st.lambda * l1;
    }
    CsrColStep cs{};
    if (frozen) {
      cs.gamma = st.gamma; cs.mode = CP_FROZEN;
    } else {
      st.gamma = gamma; st.sigma = sigma; st.s0 = s0; st.s1 = s1; st.norm_res = norm_res; st.f_x = f_x;
      cs.gamma = gamma; cs.gl = gamma * st.lambda;
      if (stop || it >= a.O.maxit) {
        // converged: the result is x_it (:355); maxit: the reference returns x after the last prox (:361-363), which at
        // maxit = 0 is the prologue's x_1 (:330-332)
        st.it_done = it; st.flags = stop ? ADAPROX_FLAG_CONVERGED : 0u;
        cs.mode = stop ? CP_CONV : CP_MAXIT;
      } else {
        cs.mode = CP_STEP;
        stepping = true;
      }
      a.col[c] = st;
    }
    a.step[c] = cs;
  }
  const unsigned run = __ballot_sync(0xffffffffu, stepping);
  if (lane == 0 && run) atomicAdd(a.n_active, __popc(run));
}

// v = x - gamma g ; x+ = prox_{gamma lambda |.|_1}(v) over the block (:359-361), or the column's stop / frozen action.
// Thread (tx, ty): column blockIdx.x * 32 + tx, rows blockIdx.y * 8 + ty, + 8 gridDim.y, ...
__global__ void __launch_bounds__(256) k_csr_path_prox(CsrPathArgs a) {
  const int64_t c = (int64_t)blockIdx.x * 32 + threadIdx.x;
  if (c >= a.L) return;                              // padding columns stay 0
  const CsrColStep cs = a.step[c];
  const long long it = a.it;
  const double* x = a.X[it % 3];
  const double* g = a.G[it & 1];
  double* xn = a.X[(it + 1) % 3];
  const int64_t ldL = a.ldL;
  for (int64_t row = (int64_t)blockIdx.y * 8 + threadIdx.y; row < a.n; row += (int64_t)gridDim.y * 8) {
    const int64_t e = row * ldL + c;
    const double xj = x[e];
    if (cs.mode == CP_STEP) {
      const double vj = xj - cs.gamma * g[e];
      a.V[e] = vj;
      xn[e] = vj + (vj <= -cs.gl ? cs.gl : (vj >= cs.gl ? -cs.gl : -vj));
    } else {
      if (cs.mode == CP_CONV) {
        a.Xout[e] = xj;
      } else if (cs.mode == CP_MAXIT) {
        const double vj = xj - cs.gamma * g[e];
        a.Xout[e] = vj + (vj <= -cs.gl ? cs.gl : (vj >= cs.gl ? -cs.gl : -vj));
      }
      xn[e] = xj;                                    // a stopped column is copied through the ring
    }
  }
}

}  // namespace adaprox
