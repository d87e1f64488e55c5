// path_gemm.cuh -- the batched multi-lambda lasso path (BASELINE config 5): AdaPGM on L problems
//     min_x 1/2 |A x - b|^2 + lambda_j |x|_1,   j = 0 .. L-1,
// that share A and b.  The L iterates are the columns of X, so the two oracle calls of the loop
// (lasso/runme.jl:22-23) become dense fp64 contractions
//     R = A X - b 1'   (m x L, K = n)        G = A' R   (n x L, K = m)
// with ~L/4 flop per byte of A: compute bound, the one place of this library where tensor cores apply.
// fp64 has no tcgen05 kind; the fp64 tensor-core path of sm_100a is mma.sync (SASS: DMMA).
//
// Layout: every column of X, R, G is CONTIGUOUS (XT[L][ldx], RT[L][ldr], GT[L][ldx]; ld = length rounded up
// to 16 doubles, zero padded), which is the natural layout for the per-column vector work and makes both mma
// operands of R = A X k-contiguous.
//
// Tile engine: 128 x 128 output tile per CTA, 16 warps as 4 x 4, 32 x 32 per warp = 4 x 4 DMMA m8n8k4 tiles
// (32 accumulator doubles per thread); BK = 16 per stage, 4-stage cp.async (LDGSTS) ring.  Shared-memory rows are
// padded by 4 doubles (row stride = 32 bytes mod 128), so the fragment loads -- lane l reads element
// [8 r + l / 4][k + l % 4] -- are bank-conflict free.
//   mode 1 (R = A X - b):  M index = row i of A, N index = column j; A-operand A[i][k], B-operand XT[j][k].
//   mode 2 (G = A' R):     M index = column c of A, N index = column j; A-operand A[i][c] staged [k][m], B-operand RT[j][i]
//                          (A is row-major, so c is the contiguous index of the A tile).
#pragma once
#include "phases.cuh"

namespace adaprox {

constexpr int kGT = 512;                 // threads per CTA of the GEMM kernels
#ifndef ADAPROX_GEMM_BK
#define ADAPROX_GEMM_BK 32
#endif
// BK doubles of K per stage and CTA barrier.  Wide tile (NT = 4): 32 with a 3-stage ring (216 KB) instead of 16 with 4 stages
// (160 KB) halves the barriers + ring refills per contraction: 16384 x 8192 x 256 A X 2.37 -> 2.24 ms, A'R 2.29 -> 2.20 ms
// (profiles/r02_notes.md; -DADAPROX_GEMM_BK=16 restores the round-1 shape).  The narrow tile (NT = 1) keeps 16 x 4 stages:
// with 32 it lost 12 % on A X (its CTAs are short, the deeper ring matters more than the barrier count).
constexpr int kGBM = 128;
constexpr int kGBKWide = ADAPROX_GEMM_BK, kGBKNarrow = 16;
constexpr int kGPadM = kGBM + 4;         // 132 doubles: row stride of the [k][m] tile of mode 2 (32 B mod 128)
// NT = 8-column DMMA tiles per warp along N: NT = 4 -> 128 x 128 CTA tile, NT = 1 -> 128 x 32 (narrow batches:
// the lambdas of one rank when the path is split over 8 GPUs)
template <int NT> struct GemmCfg {
  static constexpr int BN = 32 * NT;
  static constexpr int BK = (NT == 4) ? kGBKWide : kGBKNarrow;
  static constexpr int Stages = (BK >= 32) ? 3 : 4;
  static constexpr int PadK = BK + 4;                                    // row stride of the k-contiguous tiles (32 B mod 128: conflict-free LDS.64)
  static constexpr int ChunksK = BK / 2;                                 // 16-byte chunks per k-contiguous tile row
  static constexpr int ATile = (kGBM * PadK > BK * kGPadM) ? kGBM * PadK : BK * kGPadM;   // doubles
  static constexpr int BTile = BN * PadK;
  static constexpr int Stage = ATile + BTile;
  static constexpr int SmemBytes = Stages * Stage * 8;                   // NT = 4: 221 184 B
};
constexpr int kGBK = 16;                 // granularity of the K slabs (both tile shapes are multiples of it)

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, int src_bytes) {
  // 16-byte global -> shared copy; bytes beyond src_bytes (0 or 16) are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

struct PathGemmArgs {
  const double* A; int64_t m, n, lda;       // row-major m x n
  const double* b;                          // [m]
  int64_t L;
  const double* XT; int64_t ldx;            // [L][ldx]   (mode 1: B operand)
  double* RT; int64_t ldr;                  // [L][ldr]   (mode 1: output, mode 2: A operand)
  double* GT;                               // [L][ldx]   (mode 2: output)
  double* fpart;                            // [m tiles][L]  per-tile sums of r^2 (mode 1), reduced in tile order later
  int ksplit;                               // mode 2: K = m is cut into ksplit slabs (blockIdx.z); slab z writes GT + z * gstride
  int64_t gstride;                          //         (the slabs are summed in slab order by k_path_step: deterministic)
  int ksplit1;                              // mode 1: K = n cut into ksplit1 slabs; slab z writes the RAW partial product to
  int64_t rstride;                          //         RT + z * rstride; k_path_rfix sums the slabs in order, subtracts b, forms fpart
};

// MODE 1: RT[j][i] = sum_k A[i][k] XT[j][k] - b[i]  (+ fpart): M index = row i of A, N index = column j, K = n.
//         A-operand A[i][k] and B-operand XT[j][k] are both k-contiguous.
// MODE 2: GT[j][c] = sum_i A[i][c] RT[j][i]: M index = column c of A, N index = column j, K = m.
//         A-operand A[i][c] is staged [k][m] (A is row-major, so c is the contiguous index), B-operand RT[j][i] is
//         k-contiguous.  In both modes the batch is the N dimension, so a narrow batch only needs a narrow N tile.
template <int MODE, int NT>
__global__ void __launch_bounds__(kGT, 1) k_path_gemm(PathGemmArgs g) {
  constexpr int kGBN = GemmCfg<NT>::BN, kGStage = GemmCfg<NT>::Stage, kGBK = GemmCfg<NT>::BK, kGStages = GemmCfg<NT>::Stages;
  constexpr int kGPadK = GemmCfg<NT>::PadK, kGChunksK = GemmCfg<NT>::ChunksK;
  extern __shared__ __align__(16) double gsm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp >> 2, wn = warp & 3;
  const int64_t Mdim = (MODE == 1) ? g.m : g.n;
  const int64_t Ndim = g.L;
  const int64_t Kdim = (MODE == 1) ? g.n : g.m;
  const int64_t m0 = (int64_t)blockIdx.x * kGBM, n0 = (int64_t)blockIdx.y * kGBN;
  const double* Bop = (MODE == 1) ? g.XT : g.RT;         // rows = column j, k contiguous
  const int64_t ldb = (MODE == 1) ? g.ldx : g.ldr;
  const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(gsm);
  // k range of this CTA (mode 2 may split K over blockIdx.z; slabs are multiples of BK)
  int64_t kbeg = 0, kend = Kdim;
  const int ksp = (MODE == 2) ? g.ksplit : g.ksplit1;
  if (ksp > 1) {
    const int64_t tiles = (Kdim + kGBK - 1) / kGBK;
    const int64_t per = (tiles + ksp - 1) / ksp;
    kbeg = (int64_t)blockIdx.z * per * kGBK;
    kend = kbeg + per * kGBK;
    if (kend > Kdim) kend = Kdim;
    if (kbeg > kend) kbeg = kend;
  }

  auto load_stage = [&](int stage, int64_t k0) {
    const uint32_t sa = smem0 + (uint32_t)(stage * kGStage) * 8;
    const uint32_t sb = sa + GemmCfg<NT>::ATile * 8;
    if (MODE == 1) {
      // A tile: 128 rows i x BK doubles (k contiguous) = 128 x BK/2 chunks of 16 B
#pragma unroll
      for (int q = 0; q < (kGBM * kGBK / 2) / kGT; ++q) {
        const int ch = tid + q * kGT;
        const int r = ch / kGChunksK, kc = (ch % kGChunksK) * 2;
        const int64_t row = m0 + r, k = k0 + kc;
        const bool ok = (row < Mdim) && (k + 2 <= g.lda) && (k < kend);   // the zero padding up to lda may be read
        const double* src = g.A + (ok ? row * g.lda + k : 0);
        cp_async16(sa + (uint32_t)(r * kGPadK + kc) * 8, src, ok ? 16 : 0);
      }
    } else {
      // A tile: BK rows (k = row i of A) x 128 columns c (c contiguous) = BK x 64 chunks
#pragma unroll
      for (int q = 0; q < (kGBK * kGBM / 2) / kGT; ++q) {
        const int ch = tid + q * kGT;
        const int r = ch >> 6, cc = (ch & 63) * 2;
        const int64_t krow = k0 + r, col = m0 + cc;
        const bool ok = (krow < kend) && (col + 2 <= g.lda);
        const double* src = g.A + (ok ? krow * g.lda + col : 0);
        cp_async16(sa + (uint32_t)(r * kGPadM + cc) * 8, src, ok ? 16 : 0);
      }
    }
    // B tile: BN rows (columns j of the batch) x BK doubles, k contiguous
#pragma unroll
    for (int q = 0; q < (kGBN * kGBK / 2 + kGT - 1) / kGT; ++q) {
      const int ch = tid + q * kGT;
      if (ch >= kGBN * kGBK / 2) break;
      const int r = ch / kGChunksK, kc = (ch % kGChunksK) * 2;
      const int64_t col = n0 + r, k = k0 + kc;
      const bool ok = (col < Ndim) && (k + 2 <= ldb) && (k < kend);   // slabs end on even k (multiples of BK, or the padded end)
      const double* src = Bop + (ok ? col * ldb + k : 0);
      cp_async16(sb + (uint32_t)(r * kGPadK + kc) * 8, src, ok ? 16 : 0);
    }
  };

  double acc[4][NT][2];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < NT; ++c) acc[r][c][0] = acc[r][c][1] = 0.0;

  const int64_t nk = (kend - kbeg + kGBK - 1) / kGBK;
#pragma unroll
  for (int s = 0; s < kGStages - 1; ++s) {
    if (s < nk) load_stage(s, kbeg + (int64_t)s * kGBK);
    cp_async_commit();
  }
  const int lr = lane >> 2, lk = lane & 3;
  for (int64_t kt = 0; kt < nk; ++kt) {
    cp_async_wait<kGStages - 2>();
    __syncthreads();                                    // stage kt landed for every thread; stage kt-1 is free
    {
      const int64_t kn = kt + kGStages - 1;
      if (kn < nk) load_stage((int)(kn % kGStages), kbeg + kn * kGBK);
      cp_async_commit();
    }
    const double* sa = gsm + (size_t)(kt % kGStages) * kGStage;
    const double* sb = sa + GemmCfg<NT>::ATile;
#pragma unroll
    for (int kk = 0; kk < kGBK; kk += 4) {
      double a[4], b[NT];
      if (MODE == 1) {
#pragma unroll
        for (int r = 0; r < 4; ++r) a[r] = sa[(wm * 32 + r * 8 + lr) * kGPadK + kk + lk];
      } else {
#pragma unroll
        for (int r = 0; r < 4; ++r) a[r] = sa[(kk + lk) * kGPadM + wm * 32 + r * 8 + lr];
      }
#pragma unroll
      for (int c = 0; c < NT; ++c) b[c] = sb[(wn * 8 * NT + c * 8 + lr) * kGPadK + kk + lk];
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < NT; ++c) dmma_m8n8k4(acc[r][c][0], acc[r][c][1], a[r], b[c]);
    }
  }
  cp_async_wait<0>();

  // epilogue.  Accumulator fragment: row = lane / 4 (M index within the 8 x 8 tile), cols = 2 (lane % 4) + {0, 1}.
  if (MODE == 1 && g.ksplit1 > 1) {
    double* out = g.RT + (int64_t)blockIdx.z * g.rstride;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int64_t i = m0 + wm * 32 + r * 8 + lr;
#pragma unroll
      for (int c = 0; c < NT; ++c)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int64_t j = n0 + wn * 8 * NT + c * 8 + 2 * lk + e;
          if (i < g.m && j < g.L) out[j * g.ldr + i] = acc[r][c][e];
        }
    }
  } else if (MODE == 1) {
    __shared__ double s_f[4][kGBN];                     // [wm][column within the CTA tile]
    double fs[NT][2];
#pragma unroll
    for (int c = 0; c < NT; ++c) fs[c][0] = fs[c][1] = 0.0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int64_t i = m0 + wm * 32 + r * 8 + lr;
      const double bi = (i < g.m) ? __ldg(g.b + i) : 0.0;
#pragma unroll
      for (int c = 0; c < NT; ++c)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int64_t j = n0 + wn * 8 * NT + c * 8 + 2 * lk + e;
          if (i < g.m && j < g.L) {
            const double rv = acc[r][c][e] - bi;        // lasso/runme.jl:22
            g.RT[j * g.ldr + i] = rv;
            fs[c][e] = fma(rv, rv, fs[c][e]);
          }
        }
    }
    // sum over the 8 row-lanes (lane / 4) with a fixed xor tree, then over the 4 warps along M in fixed order
#pragma unroll
    for (int c = 0; c < NT; ++c)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        double v = fs[c][e];
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        v += __shfl_xor_sync(0xffffffffu, v, 8);
        v += __shfl_xor_sync(0xffffffffu, v, 16);
        if (lr == 0) s_f[wm][wn * 8 * NT + c * 8 + 2 * lk + e] = v;
      }
    __syncthreads();
    if (tid < kGBN) {
      const int64_t j = n0 + tid;
      if (j < g.L) g.fpart[(int64_t)blockIdx.x * g.L + j] = ((s_f[0][tid] + s_f[1][tid]) + s_f[2][tid]) + s_f[3][tid];
    }
  } else {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int64_t col = m0 + wm * 32 + r * 8 + lr;                     // column c of A = row of the accumulator tile
#pragma unroll
      for (int c = 0; c < NT; ++c)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int64_t j = n0 + wn * 8 * NT + c * 8 + 2 * lk + e;
          if (col < g.n && j < g.L) g.GT[(int64_t)blockIdx.z * g.gstride + j * g.ldx + col] = acc[r][c][e];   // lasso/runme.jl:23
        }
    }
  }
}

// R = sum of the K slabs of A X (slab order) - b, and the per-(row chunk, column) sums of r^2.  One CTA per (1024-row chunk,
// column); fpart[chunk][j] is reduced over the chunks in order by k_path_step.
constexpr int kRFixRows = 1024;
__global__ void __launch_bounds__(256, 4) k_path_rfix(PathGemmArgs g, const double* slabs) {
  __shared__ double s_w[8];
  const int64_t j = blockIdx.y, i0 = (int64_t)blockIdx.x * kRFixRows;
  double fs = 0.0;
  for (int64_t i = i0 + threadIdx.x; i < i0 + kRFixRows && i < g.m; i += 256) {
    double s = 0.0;
    for (int z = 0; z < g.ksplit1; ++z) s += slabs[(int64_t)z * g.rstride + j * g.ldr + i];
    const double rv = s - __ldg(g.b + i);                  // lasso/runme.jl:22
    g.RT[j * g.ldr + i] = rv;
    fs = fma(rv, rv, fs);
  }
  fs = warp_sum(fs);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = fs;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += s_w[w];
    g.fpart[(int64_t)blockIdx.x * g.L + j] = s;
  }
}

// ---------------------------------------------------------------------------
// per-column step of the loop (src/AdaProx.jl:334-362 with A = 0, h = Zero): one CTA per column
// ---------------------------------------------------------------------------
struct PathCol {           // per-column solver state
  double gamma, sigma, s0, s1, norm_res, f_x, lambda;
  long long it_done;       // iteration at which the column stopped (0 = still running)
  unsigned flags;
  int pad;
};

struct PathStepArgs {
  int64_t n, ldx, L, mtiles;
  DOpts O;
  double* XT[3];           // iterate ring [L][ldx]
  double* GT[2];           // gradient ring
  const double* Gslab;     // mode-2 K slabs [ksplit][L][ldx] (ksplit > 1), summed in slab order into GT[it & 1]
  int ksplit; int64_t gstride;
  double* VT;              // v = x - gamma g
  double* XoutT;           // result columns (frozen at convergence)
  const double* fpart;     // [mtiles][L]
  PathCol* col;
  double* gamma_hist; double* res_hist; double* obj_hist;   // optional [max_records][L]
  long long it;            // iteration being finished (0 = prologue)
  int* n_active;           // columns still running after this step (device counter)
};

constexpr int kPT = 256;

__global__ void __launch_bounds__(kPT, 2) k_path_step(PathStepArgs a) {
  __shared__ double s_scr[kPT / 32 * 4 + 8];
  __shared__ double s_bc[4];
  const int64_t j = blockIdx.x;
  const long long it = a.it;
  PathCol st = a.col[j];
  const double* x = a.XT[it % 3] + j * a.ldx;
  const double* x_prev = a.XT[(it + 2) % 3] + j * a.ldx;
  double* xn = a.XT[(it + 1) % 3] + j * a.ldx;
  if (a.ksplit > 1) {
    double* gw = a.GT[it & 1] + j * a.ldx;
    for (int64_t q = threadIdx.x; q < a.n; q += kPT) {
      double s = 0.0;
      for (int z = 0; z < a.ksplit; ++z) s += a.Gslab[(int64_t)z * a.gstride + j * a.ldx + q];
      gw[q] = s;
    }
    __syncthreads();
  }
  const double* grad = a.GT[it & 1] + j * a.ldx;
  const double* grad_prev = a.GT[(it + 1) & 1] + j * a.ldx;
  double* v = a.VT + j * a.ldx;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool frozen = st.it_done != 0;

  // value of f (fixed order over the row tiles)
  double f_x;
  {
    double s = 0.0;
    for (int64_t t = 0; t < a.mtiles; ++t) s += a.fpart[t * a.L + j];
    f_x = 0.5 * norm_sq_jl(s);
  }
  double gamma = st.gamma, sigma = st.sigma, s0 = st.s0, s1 = st.s1;
  bool stop = false;
  double norm_res = st.norm_res;
  if (it > 0 && !frozen) {
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int64_t q = threadIdx.x; q < a.n; q += kPT) {
      const double xj = x[q], gj = grad[q];
      const double pr = (v[q] - xj) / gamma + gj;                       // :338 (old gamma)
      const double dg = gj - grad_prev[q], dx = xj - x_prev[q];
      acc[0] = fma(pr, pr, acc[0]);
      acc[1] = fma(dg, dg, acc[1]);
      acc[2] = fma(dg, dx, acc[2]);
      acc[3] = fma(dx, dx, acc[3]);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const double s = warp_sum(acc[k]);
      if (lane == 0) s_scr[warp * 4 + k] = s;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
      double s = 0.0;
#pragma unroll
      for (int w = 0; w < kPT / 32; ++w) s += s_scr[w * 4 + threadIdx.x];
      s_bc[threadIdx.x] = s;
    }
    __syncthreads();
    DOpts Oc = a.O;
    if (Oc.rule == ADAPROX_RULE_FIXED) Oc.gamma = gamma;                 // the column's own fixed stepsize (gamma0)
    const double gamma_prev = gamma;
    rule_step(Oc, s_bc[1], s_bc[2], s_bc[3], gamma, sigma, s0, s1);       // :341
    norm_res = sqrt(norm_sq_jl(s_bc[0]) + adapgm_dual_res_sq(gamma, gamma_prev, sigma));   // :348 (dual part: 0, or NaN -- phases.cuh)
    if (norm_res <= a.O.tol) stop = true;                                // :354
  }
  // objective of the record: f(x) + lambda |x|_1
  const bool want_hist = a.gamma_hist != nullptr && it >= 1 && it <= a.O.max_records && !frozen;
  if (want_hist) {
    double l1 = 0.0;
    for (int64_t q = threadIdx.x; q < a.n; q += kPT) l1 += fabs(x[q]);
    l1 = warp_sum(l1);
    __syncthreads();
    if (lane == 0) s_scr[warp] = l1;
    __syncthreads();
    if (threadIdx.x == 0) {
      double s = 0.0;
      for (int w = 0; w < kPT / 32; ++w) s += s_scr[w];
      a.gamma_hist[(it - 1) * a.L + j] = gamma;
      a.res_hist[(it - 1) * a.L + j] = norm_res;
      a.obj_hist[(it - 1) * a.L + j] = f_x + st.lambda * s;
    }
  }
  if (frozen) return;
  if (stop || it >= a.O.maxit) {
    // converged: the result is x_it (:355); maxit: the reference returns x after the last prox (:361-363), which at
    // maxit = 0 is the prologue's x_1 = prox(x_0 - gamma_0 grad f(x_0)) (:330-332)
    const bool conv = stop;
    if (conv) {
      for (int64_t q = threadIdx.x; q < a.n; q += kPT) a.XoutT[j * a.ldx + q] = x[q];
    } else {
      for (int64_t q = threadIdx.x; q < a.n; q += kPT) {
        const double vj = x[q] - gamma * grad[q];
        const double gl = gamma * st.lambda;
        a.XoutT[j * a.ldx + q] = vj + (vj <= -gl ? gl : (vj >= gl ? -gl : -vj));
      }
    }
    if (threadIdx.x == 0) {
      st.gamma = gamma; st.sigma = sigma; st.s0 = s0; st.s1 = s1; st.norm_res = norm_res; st.f_x = f_x;
      st.it_done = it; st.flags = conv ? ADAPROX_FLAG_CONVERGED : 0u;
      a.col[j] = st;
    }
    // keep the ring defined for the (ignored) later iterations of this column
    for (int64_t q = threadIdx.x; q < a.n; q += kPT) xn[q] = x[q];
    return;
  }
  // v = x - gamma grad ; x+ = prox_{gamma lambda |.|_1}(v)   (:359-361; NormL1 in ProximalOperators' form, Appendix A)
  const double gl = gamma * st.lambda;
  for (int64_t q = threadIdx.x; q < a.n; q += kPT) {
    const double vj = x[q] - gamma * grad[q];
    v[q] = vj;
    xn[q] = vj + (vj <= -gl ? gl : (vj >= gl ? -gl : -vj));
  }
  if (threadIdx.x == 0) {
    st.gamma = gamma; st.sigma = sigma; st.s0 = s0; st.s1 = s1; st.norm_res = norm_res; st.f_x = f_x;
    a.col[j] = st;
    atomicAdd(a.n_active, 1);
  }
}

}  // namespace adaprox
