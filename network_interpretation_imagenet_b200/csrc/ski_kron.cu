// ski_kron.cu — the SKI pixel GP of ski.cu on large inducing grids (grid_size 300: G = 90 000), without any G x G matrix.
//
// Same model as ski.cu / oracle/ski.py: K = os * K1 (x) K1 on the gs x gs grid, W the folded Keys cubic interpolation,
// A = W^T W, b = W^T (y - c), B = s2 I + S^T A S for a square root K = S S^T.  Here S = M_R (x) M_C with gs x gs factors
// chosen on the host (package ski.py): M = os^(1/4) Q Lambda^(1/2) V per axis, K1 = Q Lambda Q^T, and V the eigenvectors
// of Lambda^(1/2) Q^T A_axis Q Lambda^(1/2), so that the diagonal s2 + coef * theta_R[i] theta_C[j] is exactly S^T A S + s2 I
// when the training pixels form a lattice and is the preconditioner otherwise.  The parts of order G and above live here:
//   kron apply     Y = (M_R (x) M_C) X or its transpose for r right-hand sides: two fp64 tensor-core GEMMs (mma.sync
//                  m8n8k4, as gp.cu's dgemm_sub_kernel) whose epilogues write each gs x gs block transposed
//   band A         A in band form [G][7][7] (points couple grid nodes at most 3 apart per axis) and b, summed without
//                  floating-point atomics: points are bucketed by stencil anchor with a counting sort made stable by
//                  sorting each bucket, then one thread per (grid node, offset) sums its pairs in bucket order
//   band SpMV      Y = A X over r right-hand sides
//   block PCG      per-column alpha / beta from fixed-order block reductions, the diagonal preconditioner fused into the
//                  vector updates, no host synchronisation except a status read every `check_every` iterations
//   variance       rank-one right-hand sides (M_R^T w0) (x) (M_C^T w1) built in place, var = s2 rhs^T x per query
// Every reduction has a fixed order, so two runs on the same inputs are bitwise equal whatever the stream.
#include "common.cuh"

namespace nib {
namespace {

// Keys cubic convolution kernel, a = -0.5 (as ski.cu)
__device__ __forceinline__ double keys(double s) {
  s = fabs(s);
  if (s <= 1.0) return (1.5 * s - 2.5) * s * s + 1.0;
  if (s < 2.0) return ((-0.5 * s + 2.5) * s - 4.0) * s + 2.0;
  return 0.0;
}

// 1-D stencil of coordinate x folded onto 4 consecutive grid nodes ap..ap+3 (0 <= ap <= gs-4).  ski.cu clamps each stencil
// index to [0, gs-1] separately; pixel 0 sits less than one spacing inside the grid, so its stencil reaches node -1 and
// ski.cu's W adds that weight to node 0.  Folding the clamped weights keeps the same W while every point's stencil is a
// whole 4 x 4 block, which is what the band form needs.
__device__ __forceinline__ int stencil1d(double x, double g0, double h, int gs, double (&w)[4]) {
  const double u = (x - g0) / h;
  const int a = (int)floor(u) - 1;
  const int ap = min(max(a, 0), gs - 4);
#pragma unroll
  for (int k = 0; k < 4; ++k) w[k] = 0.0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int slot = min(max(a + k, 0), gs - 1) - ap;
    const double v = keys(u - (double)(a + k));
#pragma unroll
    for (int m = 0; m < 4; ++m) w[m] += (m == slot) ? v : 0.0;    // keeps w in registers
  }
  return ap;
}

// ---- deterministic band accumulation of A and b -----------------------------------------------------------------------
__global__ void __launch_bounds__(256)
band_key_kernel(const double* __restrict__ X, int n, double g0, double h, int gs, int* __restrict__ key,
                int* __restrict__ count) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  double w[4];
  const int k = stencil1d(X[2 * p], g0, h, gs, w) * gs + stencil1d(X[2 * p + 1], g0, h, gs, w);
  key[p] = k;
  atomicAdd(count + k, 1);        // integer: the total does not depend on the order
}

// exclusive scan of count[G] into start[G + 1]: one block, each thread a contiguous slice
__global__ void __launch_bounds__(1024)
band_scan_kernel(const int* __restrict__ count, int G, int* __restrict__ start) {
  __shared__ int part[1024];
  const int t = threadIdx.x;
  const int per = (G + 1023) / 1024;
  const int lo = min(t * per, G), hi = min(lo + per, G);
  int s = 0;
  for (int i = lo; i < hi; ++i) s += count[i];
  part[t] = s;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {            // Hillis-Steele inclusive scan of the slice sums
    const int v = t >= o ? part[t - o] : 0;
    __syncthreads();
    part[t] += v;
    __syncthreads();
  }
  int run = t ? part[t - 1] : 0;
  for (int i = lo; i < hi; ++i) { start[i] = run; run += count[i]; }
  if (t == 1023) start[G] = part[1023];
}

__global__ void __launch_bounds__(256)
band_place_kernel(const int* __restrict__ key, int n, const int* __restrict__ start, int* __restrict__ cursor,
                  int* __restrict__ perm) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const int k = key[p];
  perm[start[k] + atomicAdd(cursor + k, 1)] = p;
}

// The placement order within a bucket depends on scheduling; sorting each bucket by point index makes the sort stable.
// Buckets hold the points of one grid cell (about h^2 pixels, times any duplicates), so insertion sort suffices.
__global__ void __launch_bounds__(256)
band_bucket_sort_kernel(const int* __restrict__ start, int G, int* __restrict__ perm) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= G) return;
  const int lo = start[c], hi = start[c + 1];
  for (int i = lo + 1; i < hi; ++i) {
    const int v = perm[i];
    int j = i - 1;
    while (j >= lo && perm[j] > v) { perm[j + 1] = perm[j]; --j; }
    perm[j + 1] = v;
  }
}

// sorted position i: the folded weights of its point (w0[4], w1[4]) and y - c
__global__ void __launch_bounds__(256)
band_gather_kernel(const double* __restrict__ X, const double* __restrict__ y, const int* __restrict__ perm, int n,
                   double g0, double h, int gs, double cmean, double* __restrict__ pw, double* __restrict__ py) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int p = perm[i];
  double w0[4], w1[4];
  stencil1d(X[2 * p], g0, h, gs, w0);
  stencil1d(X[2 * p + 1], g0, h, gs, w1);
#pragma unroll
  for (int k = 0; k < 4; ++k) { pw[(size_t)i * 8 + k] = w0[k]; pw[(size_t)i * 8 + 4 + k] = w1[k]; }
  py[i] = y[p] - cmean;
}

// thread (g, o): o < 49 -> A[g][o] = sum_p w_p(g) w_p(g + off(o)), off(o) = (o / 7 - 3, o % 7 - 3); o == 49 -> b[g].
// Anchor cells in row-major order, points in bucket order: a fixed summation order.
__global__ void __launch_bounds__(250)
band_sum_kernel(const int* __restrict__ start, const double* __restrict__ pw, const double* __restrict__ py, int gs,
                double* __restrict__ A, double* __restrict__ b) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long G = (long long)gs * gs;
  if (t >= G * 50) return;
  const int g = (int)(t / 50), o = (int)(t - (long long)g * 50);
  const int g0 = g / gs, g1 = g - g0 * gs;
  const bool is_b = (o == 49);
  const int d0 = is_b ? 0 : o / 7 - 3, d1 = is_b ? 0 : o % 7 - 3;
  const int h0 = g0 + d0, h1 = g1 + d1;
  double acc = 0.0;
  if (h0 >= 0 && h0 < gs && h1 >= 0 && h1 < gs) {
    const int a0lo = max(max(g0, h0) - 3, 0), a0hi = min(min(g0, h0), gs - 4);
    const int a1lo = max(max(g1, h1) - 3, 0), a1hi = min(min(g1, h1), gs - 4);
    for (int a0 = a0lo; a0 <= a0hi; ++a0)
      for (int a1 = a1lo; a1 <= a1hi; ++a1) {
        const int c = a0 * gs + a1;
        for (int i = start[c]; i < start[c + 1]; ++i) {
          const double* w = pw + (size_t)i * 8;
          const double wg = w[g0 - a0] * w[4 + g1 - a1];
          acc = fma(wg, is_b ? py[i] : w[h0 - a0] * w[4 + h1 - a1], acc);
        }
      }
  }
  if (is_b) b[g] = acc;
  else A[(size_t)g * 49 + o] = acc;
}

// ---- band SpMV: Y[c] = A X[c] for r columns of G ----------------------------------------------------------------------
static constexpr int SPMV_COLS = 8;   // columns per thread: the 49 band entries of a node are loaded once for these
__global__ void __launch_bounds__(256)
band_spmv_kernel(const double* __restrict__ A, int gs, const double* __restrict__ X, double* __restrict__ Y, int r,
                 const int* __restrict__ skip) {
  const int G = gs * gs;
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const int g0 = g / gs, g1 = g - g0 * gs;
  double a[49];
#pragma unroll
  for (int o = 0; o < 49; ++o) a[o] = A[(size_t)g * 49 + o];
  const int c_end = min(r, (int)(blockIdx.y + 1) * SPMV_COLS);
  for (int c = blockIdx.y * SPMV_COLS; c < c_end; ++c) {
    if (skip && skip[c]) continue;
    const double* x = X + (size_t)c * G;
    double acc = 0.0;
#pragma unroll
    for (int d0 = -3; d0 <= 3; ++d0) {
      const int h0 = g0 + d0;
      if (h0 < 0 || h0 >= gs) continue;
#pragma unroll
      for (int d1 = -3; d1 <= 3; ++d1) {
        const int h1 = g1 + d1;
        if (h1 < 0 || h1 >= gs) continue;
        acc = fma(a[(d0 + 3) * 7 + d1 + 3], x[h0 * gs + h1], acc);
      }
    }
    Y[(size_t)c * G + g] = acc;
  }
}

// ---- Kronecker factor GEMM with a transposing epilogue ----------------------------------------------------------------
// In: r blocks of gs x gs, row-major, stacked as one (r*gs) x gs matrix.  For block c and row i:
//     Out[c][j][i] = sum_k In[c][i][k] * F(k, j)  (+ add_coef * Add[c][j][i]),   F(k, j) = trans ? Fm[k][j] : Fm[j][k]
// Two such passes apply a whole Kronecker factor: (M_R (x) M_C) X = M_R X M_C^T is the pass with M_C then the pass with
// M_R (trans = 0); the transpose uses trans = 1.  64 x 64 output tile per block, 16-deep K chunks in two shared-memory
// stages, 4 warps of 32 x 32 each on mma.sync.m8n8k4.f64; the next chunk's global loads are issued before the current
// chunk's MMAs.  skip[c] != 0 marks a column whose result is not needed: a tile whose rows all belong to such columns
// returns at once (converged PCG columns).
static constexpr int KT = 64, KK = 16, KP = KT + 4;   // KP: smem pitch = 8 words mod 32 -> conflict-free fragment loads

__device__ __forceinline__ void dmma(double (&d)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(d[0]), "+d"(d[1]) : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(128)
kron_pass_kernel(const double* __restrict__ In, int r, int gs, const double* __restrict__ Fm, int trans,
                 double* __restrict__ Out, const double* __restrict__ Add, double add_coef, const int* __restrict__ skip) {
  const int M = r * gs;
  const int i0 = blockIdx.x * KT, j0 = blockIdx.y * KT;
  if (skip) {
    const int c_lo = i0 / gs, c_hi = min(i0 + KT - 1, M - 1) / gs;
    bool all = true;
    for (int c = c_lo; c <= c_hi; ++c) all = all && skip[c] != 0;
    if (all) return;
  }
  __shared__ __align__(16) double As[2][KK][KP];
  __shared__ __align__(16) double Bs[2][KK][KP];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 1, wn = warp & 1;
  const int fr = lane >> 2, fk = lane & 3;
  double acc[4][4][2];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
  // loaders: 64 x 16 of In (k fastest: 16 threads per row, 8 rows per pass) and 16 x 64 of F (unit stride along k for
  // trans = 0, along j for trans = 1)
  const int a_k = tid & 15, a_i = tid >> 4;
  const int b_k = trans ? (tid >> 6) : (tid & 15);
  const int b_j = trans ? (tid & 63) : (tid >> 4);
  double av[8], bv[8];
  auto load_chunk = [&](int k0) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int i = i0 + a_i + 8 * e, k = k0 + a_k;
      av[e] = (i < M && k < gs) ? In[(long long)i * gs + k] : 0.0;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = k0 + b_k + (trans ? 2 * e : 0), j = j0 + b_j + (trans ? 0 : 8 * e);
      bv[e] = (j < gs && k < gs) ? (trans ? Fm[k * gs + j] : Fm[j * gs + k]) : 0.0;
    }
  };
  auto park = [&](int st) {
#pragma unroll
    for (int e = 0; e < 8; ++e) As[st][a_k][a_i + 8 * e] = av[e];
#pragma unroll
    for (int e = 0; e < 8; ++e) Bs[st][b_k + (trans ? 2 * e : 0)][b_j + (trans ? 0 : 8 * e)] = bv[e];
  };
  load_chunk(0);
  park(0);
  __syncthreads();
  int cur = 0;
  for (int k0 = 0; k0 < gs; k0 += KK) {
    const bool more = k0 + KK < gs;
    if (more) load_chunk(k0 + KK);
#pragma unroll
    for (int t = 0; t < KK; t += 4) {
      double a[4], b[4];
#pragma unroll
      for (int mt = 0; mt < 4; ++mt) a[mt] = As[cur][t + fk][wm * 32 + mt * 8 + fr];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) b[nt] = Bs[cur][t + fk][wn * 32 + nt * 8 + fr];
#pragma unroll
      for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) dmma(acc[mt][nt], a[mt], b[nt]);
    }
    if (more) park(cur ^ 1);
    __syncthreads();
    cur ^= 1;
  }
  // transposed epilogue: lanes fr = 0..7 of a fragment hold consecutive rows i, i.e. consecutive addresses of Out
#pragma unroll
  for (int mt = 0; mt < 4; ++mt) {
    const int row = i0 + wm * 32 + mt * 8 + fr;
    if (row >= M) continue;
    const int c = row / gs, i = row - c * gs;
    const long long base = (long long)c * gs * gs + i;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int j = j0 + wn * 32 + nt * 8 + 2 * fk + e;
        if (j >= gs) continue;
        const long long at = base + (long long)j * gs;
        Out[at] = Add ? fma(add_coef, Add[at], acc[mt][nt][e]) : acc[mt][nt][e];
      }
  }
}

// ---- block PCG ----------------------------------------------------------------------------------------------------------
// State of column c (doubles, then ints, in the caller's workspace): bnorm, rz (= r^T D^-1 r), relres; done, iters.
struct PcgState {
  double *bnorm, *rz, *relres;
  int *done, *iters;
};

static constexpr int RT = 256;   // threads of the per-column kernels

// fixed-order block sum of two values (thread-strided partial sums, xor butterfly per warp, warps summed in order)
__device__ __forceinline__ void block_sum2(double& a, double& b) {
  __shared__ double sh[2][RT / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  __syncthreads();                 // the previous call's readers are done with sh
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = a; sh[1][threadIdx.x >> 5] = b; }
  __syncthreads();
  a = 0.0;
  b = 0.0;
#pragma unroll
  for (int w = 0; w < RT / 32; ++w) { a += sh[0][w]; b += sh[1][w]; }
}

__device__ __forceinline__ double dinv_at(int g, int gs, const double* thR, const double* thC, double coef, double s2) {
  const int i = g / gs;
  return 1.0 / fma(coef * thR[i], thC[g - i * gs], s2);
}

// x = 0, r = rhs, p = D^-1 r
__global__ void __launch_bounds__(RT)
pcg_init_kernel(const double* __restrict__ rhs, int G, int gs, const double* __restrict__ thR,
                const double* __restrict__ thC, double coef, double s2, double* __restrict__ x, double* __restrict__ rr,
                double* __restrict__ p, PcgState s) {
  const int c = blockIdx.x;
  const size_t off = (size_t)c * G;
  double nb = 0.0, rz = 0.0;
  for (int g = threadIdx.x; g < G; g += RT) {
    const double v = rhs[off + g], d = dinv_at(g, gs, thR, thC, coef, s2);
    x[off + g] = 0.0;
    rr[off + g] = v;
    p[off + g] = d * v;
    nb = fma(v, v, nb);
    rz = fma(v, d * v, rz);
  }
  block_sum2(nb, rz);
  if (threadIdx.x == 0) {
    s.bnorm[c] = sqrt(nb);
    s.rz[c] = rz;
    s.relres[c] = nb > 0.0 ? 1.0 : 0.0;
    s.done[c] = nb > 0.0 ? 0 : 1;     // a zero right-hand side has the solution x = 0
    s.iters[c] = 0;
  }
}

// one PCG step of column c, given q = B p:  alpha = rz / p^T q;  x += alpha p;  r -= alpha q;  z = D^-1 r;
// beta = r^T z / rz;  p = z + beta p.  Converged columns (relative residual <= tol) stop and are marked done.
__global__ void __launch_bounds__(RT)
pcg_step_kernel(int G, int gs, const double* __restrict__ thR, const double* __restrict__ thC, double coef, double s2,
                double tol, double* __restrict__ x, double* __restrict__ rr, double* __restrict__ p,
                const double* __restrict__ q, PcgState s) {
  const int c = blockIdx.x;
  if (s.done[c]) return;
  const size_t off = (size_t)c * G;
  double pq = 0.0, unused = 0.0;
  for (int g = threadIdx.x; g < G; g += RT) pq = fma(p[off + g], q[off + g], pq);
  block_sum2(pq, unused);
  const double alpha = s.rz[c] / pq;
  double r2 = 0.0, rz = 0.0;
  for (int g = threadIdx.x; g < G; g += RT) {
    const double pv = p[off + g];
    x[off + g] = fma(alpha, pv, x[off + g]);
    const double rv = fma(-alpha, q[off + g], rr[off + g]);
    rr[off + g] = rv;
    r2 = fma(rv, rv, r2);
    rz = fma(rv, dinv_at(g, gs, thR, thC, coef, s2) * rv, rz);
  }
  block_sum2(r2, rz);
  const double relres = sqrt(r2) / s.bnorm[c];
  const bool conv = relres <= tol;
  if (!conv) {
    const double beta = rz / s.rz[c];
    for (int g = threadIdx.x; g < G; g += RT)
      p[off + g] = fma(beta, p[off + g], dinv_at(g, gs, thR, thC, coef, s2) * rr[off + g]);
  }
  __syncthreads();                   // every thread has read s.rz[c] before it changes
  if (threadIdx.x == 0) {
    s.rz[c] = rz;
    s.relres[c] = relres;
    s.iters[c] += 1;
    s.done[c] = conv ? 1 : 0;
  }
}

// status[0] = columns still running, status[1] = largest relative residual, status[2] = most iterations of a column
__global__ void __launch_bounds__(RT)
pcg_status_kernel(int r, PcgState s, double* __restrict__ status) {
  double active = 0.0, worst = 0.0, its = 0.0;
  for (int c = threadIdx.x; c < r; c += RT) {
    active += s.done[c] ? 0.0 : 1.0;
    worst = fmax(worst, s.relres[c]);
    its = fmax(its, (double)s.iters[c]);
  }
  __shared__ double sh[3][RT];
  sh[0][threadIdx.x] = active;
  sh[1][threadIdx.x] = worst;
  sh[2][threadIdx.x] = its;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int t = 1; t < RT; ++t) {
      active += sh[0][t];
      worst = fmax(worst, sh[1][t]);
      its = fmax(its, sh[2][t]);
    }
    status[0] = active;
    status[1] = worst;
    status[2] = its;
  }
}

// ---- variance -----------------------------------------------------------------------------------------------------------
// rhs[q] = (M_R^T w0) (x) (M_C^T w1), w0 / w1 the folded 1-D stencils of query q: one block per query
__global__ void __launch_bounds__(RT)
var_rhs_kernel(const double* __restrict__ Xq, double g0, double h, int gs, const double* __restrict__ MR,
               const double* __restrict__ MC, double* __restrict__ rhs) {
  extern __shared__ double uv[];        // [2][gs]
  const int q = blockIdx.x;
  double w0[4], w1[4];
  const int a0 = stencil1d(Xq[2 * q], g0, h, gs, w0);
  const int a1 = stencil1d(Xq[2 * q + 1], g0, h, gs, w1);
  for (int j = threadIdx.x; j < gs; j += RT) {
    double u = 0.0, v = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      u = fma(w0[k], MR[(a0 + k) * gs + j], u);
      v = fma(w1[k], MC[(a1 + k) * gs + j], v);
    }
    uv[j] = u;
    uv[gs + j] = v;
  }
  __syncthreads();
  const int G = gs * gs;
  double* out = rhs + (size_t)q * G;
  for (int g = threadIdx.x; g < G; g += RT) {
    const int i = g / gs;
    out[g] = uv[i] * uv[gs + g - i * gs];
  }
}

// var[q] = s2 * rhs[q]^T x[q] (+ s2)
__global__ void __launch_bounds__(RT)
var_reduce_kernel(const double* __restrict__ rhs, const double* __restrict__ x, int G, double s2, int add_noise,
                  double* __restrict__ var) {
  const int q = blockIdx.x;
  const size_t off = (size_t)q * G;
  double a = 0.0, unused = 0.0;
  for (int g = threadIdx.x; g < G; g += RT) a = fma(rhs[off + g], x[off + g], a);
  block_sum2(a, unused);
  if (threadIdx.x == 0) var[q] = s2 * a + (add_noise ? s2 : 0.0);
}

int kron_apply(const double* X, double* Y, int r, int gs, const double* MR, const double* MC, int trans, double* work,
               const double* add, double add_coef, const int* skip, cudaStream_t st) {
  dim3 grid(ceil_div(r * gs, KT), ceil_div(gs, KT));
  kron_pass_kernel<<<grid, 128, 0, st>>>(X, r, gs, MC, trans, work, nullptr, 0.0, skip);
  NIB_LAUNCH_CHECK();
  kron_pass_kernel<<<grid, 128, 0, st>>>(work, r, gs, MR, trans, Y, add, add_coef, skip);
  NIB_LAUNCH_CHECK();
  return NIB_OK;
}

int band_spmv(const double* A, int gs, const double* X, double* Y, int r, const int* skip, cudaStream_t st) {
  dim3 grid(ceil_div(gs * gs, 256), ceil_div(r, SPMV_COLS));
  band_spmv_kernel<<<grid, 256, 0, st>>>(A, gs, X, Y, r, skip);
  NIB_LAUNCH_CHECK();
  return NIB_OK;
}

}  // namespace
}  // namespace nib

extern "C" {

// gs <= 46340 keeps G = gs^2 in int, r * gs < 2^31 - 64 the GEMM rows; r <= 65535 keeps the SpMV grid in range
#define NIB_KRON_SHAPE_OK(r, gs) \
  ((gs) >= 1 && (gs) <= 46340 && (r) >= 1 && (r) <= 65535 && (long long)(r) * (gs) < (1LL << 31) - 64)

int nib_ski_kron_apply(const double* d_X, double* d_Y, int r, int grid_size, const double* d_MR, const double* d_MC,
                       int trans, double* d_work, void* stream) {
  NIB_DEVICE_OR_FAIL();
  using namespace nib;
  NIB_REQUIRE(d_X && d_Y && d_MR && d_MC && d_work && NIB_KRON_SHAPE_OK(r, grid_size) && (trans == 0 || trans == 1),
              "nib_ski_kron_apply: bad arguments");
  return kron_apply(d_X, d_Y, r, grid_size, d_MR, d_MC, trans, d_work, nullptr, 0.0, nullptr, (cudaStream_t)stream);
}

int nib_ski_band_accumulate(const double* d_X, const double* d_y, int n, double grid0, double spacing, int grid_size,
                            double const_mean, double* d_A, double* d_b, void* d_work, void* stream) {
  NIB_DEVICE_OR_FAIL();
  using namespace nib;
  NIB_REQUIRE(d_X && d_y && d_A && d_b && d_work && n > 0 && grid_size >= 4 && grid_size <= 46340 && spacing > 0.0,
              "nib_ski_band_accumulate: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int G = grid_size * grid_size;
  // workspace: ints key[n], perm[n], count[G], start[G + 1], cursor[G]; then (8-byte aligned) doubles pw[8n], py[n]
  int* key = static_cast<int*>(d_work);
  int* perm = key + n;
  int* count = perm + n;
  int* start = count + G;
  int* cursor = start + G + 1;
  const size_t ints = (size_t)2 * n + 3 * (size_t)G + 1;
  double* pw = static_cast<double*>(d_work) + (ints + 1) / 2;
  double* py = pw + (size_t)8 * n;
  NIB_CUDA(cudaMemsetAsync(count, 0, sizeof(int) * G, st));
  NIB_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int) * G, st));
  band_key_kernel<<<ceil_div(n, 256), 256, 0, st>>>(d_X, n, grid0, spacing, grid_size, key, count);
  NIB_LAUNCH_CHECK();
  band_scan_kernel<<<1, 1024, 0, st>>>(count, G, start);
  NIB_LAUNCH_CHECK();
  band_place_kernel<<<ceil_div(n, 256), 256, 0, st>>>(key, n, start, cursor, perm);
  NIB_LAUNCH_CHECK();
  band_bucket_sort_kernel<<<ceil_div(G, 256), 256, 0, st>>>(start, G, perm);
  NIB_LAUNCH_CHECK();
  band_gather_kernel<<<ceil_div(n, 256), 256, 0, st>>>(d_X, d_y, perm, n, grid0, spacing, grid_size, const_mean, pw, py);
  NIB_LAUNCH_CHECK();
  band_sum_kernel<<<(unsigned)ceil_div_ll((long long)G * 50, 250), 250, 0, st>>>(start, pw, py, grid_size, d_A, d_b);
  NIB_LAUNCH_CHECK();
  return NIB_OK;
}


int nib_ski_band_spmv(const double* d_A, int grid_size, const double* d_X, double* d_Y, int r, void* stream) {
  NIB_DEVICE_OR_FAIL();
  using namespace nib;
  NIB_REQUIRE(d_A && d_X && d_Y && NIB_KRON_SHAPE_OK(r, grid_size), "nib_ski_band_spmv: bad arguments");
  return band_spmv(d_A, grid_size, d_X, d_Y, r, nullptr, (cudaStream_t)stream);
}

int nib_ski_kron_pcg(const double* d_A, int grid_size, const double* d_MR, const double* d_MC, const double* d_thetaR,
                     const double* d_thetaC, double coef, double noise, const double* d_rhs, double* d_x, int r,
                     double tol, int max_iter, int check_every, double* d_work, int* h_iters, double* h_relres,
                     void* stream) {
  NIB_DEVICE_OR_FAIL();
  using namespace nib;
  NIB_REQUIRE(d_A && d_MR && d_MC && d_thetaR && d_thetaC && d_rhs && d_x && d_work && h_iters && h_relres &&
                  NIB_KRON_SHAPE_OK(r, grid_size) && noise > 0.0 && coef >= 0.0 && tol >= 0.0 && max_iter >= 1 &&
                  check_every >= 1,
              "nib_ski_kron_pcg: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int gs = grid_size;
  const size_t rG = (size_t)r * gs * gs;
  double* rr = d_work;
  double* p = rr + rG;
  double* q = p + rG;
  double* t1 = q + rG;
  double* t2 = t1 + rG;
  PcgState s;
  s.bnorm = t2 + rG;
  s.rz = s.bnorm + r;
  s.relres = s.rz + r;
  double* status = s.relres + r;           // 4 doubles
  s.done = reinterpret_cast<int*>(status + 4);
  s.iters = s.done + r;
  pcg_init_kernel<<<r, RT, 0, st>>>(d_rhs, gs * gs, gs, d_thetaR, d_thetaC, coef, noise, d_x, rr, p, s);
  NIB_LAUNCH_CHECK();
  double hs[3] = {0.0, 0.0, 0.0};
  for (int it = 1; it <= max_iter; ++it) {
    // q = s2 p + S^T A S p, skipping converged columns
    int rc = kron_apply(p, t1, r, gs, d_MR, d_MC, 0, t2, nullptr, 0.0, s.done, st);
    if (rc != NIB_OK) return rc;
    rc = band_spmv(d_A, gs, t1, t2, r, s.done, st);
    if (rc != NIB_OK) return rc;
    rc = kron_apply(t2, q, r, gs, d_MR, d_MC, 1, t1, p, noise, s.done, st);
    if (rc != NIB_OK) return rc;
    pcg_step_kernel<<<r, RT, 0, st>>>(gs * gs, gs, d_thetaR, d_thetaC, coef, noise, tol, d_x, rr, p, q, s);
    NIB_LAUNCH_CHECK();
    if (it % check_every == 0 || it == max_iter) {
      pcg_status_kernel<<<1, RT, 0, st>>>(r, s, status);
      NIB_LAUNCH_CHECK();
      NIB_CUDA(cudaMemcpyAsync(hs, status, sizeof(hs), cudaMemcpyDeviceToHost, st));
      NIB_CUDA(cudaStreamSynchronize(st));
      if (hs[0] == 0.0) break;
    }
  }
  *h_iters = (int)hs[2];
  *h_relres = hs[1];
  return NIB_OK;
}


int nib_ski_kron_var_rhs(const double* d_Xq, int m, double grid0, double spacing, int grid_size, const double* d_MR,
                         const double* d_MC, double* d_rhs, void* stream) {
  NIB_DEVICE_OR_FAIL();
  using namespace nib;
  NIB_REQUIRE(d_Xq && d_MR && d_MC && d_rhs && m >= 1 && grid_size >= 4 && grid_size <= 3072 && spacing > 0.0,
              "nib_ski_kron_var_rhs: bad arguments");
  var_rhs_kernel<<<m, RT, 2 * grid_size * sizeof(double), (cudaStream_t)stream>>>(d_Xq, grid0, spacing, grid_size, d_MR,
                                                                                  d_MC, d_rhs);
  NIB_LAUNCH_CHECK();
  return NIB_OK;
}

int nib_ski_kron_var_reduce(const double* d_rhs, const double* d_x, int m, int grid_size, double noise, int add_noise,
                            double* d_var, void* stream) {
  NIB_DEVICE_OR_FAIL();
  using namespace nib;
  NIB_REQUIRE(d_rhs && d_x && d_var && m >= 1 && grid_size >= 1 && grid_size <= 46340,
              "nib_ski_kron_var_reduce: bad arguments");
  var_reduce_kernel<<<m, RT, 0, (cudaStream_t)stream>>>(d_rhs, d_x, grid_size * grid_size, noise, add_noise, d_var);
  NIB_LAUNCH_CHECK();
  return NIB_OK;
}

}  // extern "C"
