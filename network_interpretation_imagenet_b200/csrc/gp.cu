// gp.cu — stage 3: exact Gaussian-process surrogate over binary masks + Expected Improvement, fp64.
//
// Arithmetic restated from scikit-learn 1.9.0 `GaussianProcessRegressor` as configured at
// BayesianOptimization.py:154-159 (RBF kernel, alpha=1e-5, normalize_y=True):
//   fit      sklearn/gaussian_process/_gpr.py:233-368   (Gram, +alpha*I, cholesky, cho_solve)
//   predict  _gpr.py:446-496                             (K* alpha; V = L^-1 K*^T; 1 - sum V^2, clip)
//   LML/grad _gpr.py:588-655
//   RBF      sklearn/gaussian_process/kernels.py:1561-1569 (exp(-0.5 * sqeuclidean(X / l)))
// and the acquisition from BayesianOptimization.py:37-54.
//
// For binary X, sqeuclidean(z_i, z_j) = popcount(z_i xor z_j), so the Gram matrix is a (S+1)-entry
// LUT over Hamming distances: integer ALU + an n^2*8-byte HBM write.  Cholesky/TRSM are blocked
// (NB = 64) around one fp64 SIMT GEMM kernel (128x128 tiles, 8x8 register micro-tiles).
#include "common.cuh"
#include <math.h>

namespace nib {

static constexpr int NB = 64;

// ---- Gram ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gram_binary_kernel(const uint64_t* __restrict__ Za, int na, const uint64_t* __restrict__ Zb, int nb, int words,
                   double inv_l2_half /* 0.5 / l^2 */, double jitter, int same, double* __restrict__ K, int ldk) {
  extern __shared__ double lut[];  // [64*words + 1]
  const int nl = 64 * words + 1;
  for (int h = threadIdx.x + threadIdx.y * blockDim.x; h < nl; h += blockDim.x * blockDim.y)
    lut[h] = exp(-(double)h * inv_l2_half);
  __syncthreads();
  const int j = blockIdx.x * 32 + threadIdx.x;
  const int i0 = blockIdx.y * 32;
  if (j >= nb) return;
  if (words == 1) {
    const uint64_t zj = Zb[j];
    for (int ii = threadIdx.y; ii < 32; ii += blockDim.y) {
      const int i = i0 + ii;
      if (i >= na) break;
      const int h = __popcll(Za[i] ^ zj);
      double v = lut[h];
      if (same && i == j) v += jitter;
      K[(size_t)i * ldk + j] = v;
    }
  } else {
    for (int ii = threadIdx.y; ii < 32; ii += blockDim.y) {
      const int i = i0 + ii;
      if (i >= na) break;
      int h = 0;
      for (int w = 0; w < words; ++w) h += __popcll(Za[(size_t)i * words + w] ^ Zb[(size_t)j * words + w]);
      double v = lut[h];
      if (same && i == j) v += jitter;
      K[(size_t)i * ldk + j] = v;
    }
  }
}

__global__ void __launch_bounds__(256)
gram_rbf_kernel(const double* __restrict__ Xa, int na, const double* __restrict__ Xb, int nb, int d, double inv_l,
                double jitter, int same, double* __restrict__ K, int ldk) {
  const int j = blockIdx.x * 32 + threadIdx.x;
  const int i0 = blockIdx.y * 32;
  if (j >= nb) return;
  for (int ii = threadIdx.y; ii < 32; ii += blockDim.y) {
    const int i = i0 + ii;
    if (i >= na) break;
    double s = 0.0;
    for (int k = 0; k < d; ++k) {
      // kernels.py:1566: dists on X / length_scale
      const double diff = Xa[(size_t)i * d + k] * inv_l - Xb[(size_t)j * d + k] * inv_l;
      s += diff * diff;
    }
    double v = exp(-0.5 * s);
    if (same && i == j) v = 1.0 + jitter;  // np.fill_diagonal(K, 1) then K[diag] += alpha
    K[(size_t)i * ldk + j] = v;
  }
}

// ---- generic fp64 GEMM update:  C[i][j] -= sum_t A(i,t) * B(t,j) ------------------------------
// A(i,t) = A[i*sai + t*sat], B(t,j) = B[t*sbt + j*sbj], C row-major ldc.  lower_only skips tiles
// strictly above the diagonal (SYRK trailing update of the Cholesky).
struct DgemmArgs {
  const double* A; long long sai, sat;
  const double* B; long long sbt, sbj;
  double* C; long long ldc;
  int M, N, K;
  int lower_only;
};

// 128 x 128 output tile per block, 16-deep K chunks, 8 warps (2 x 4) each accumulating a 64 x 32 sub-tile with the fp64
// tensor-core instruction mma.sync.m8n8k4 (32 MMA tiles, 64 accumulator doubles per thread): per 4-deep K step a warp
// issues 12 shared-memory fragment loads for 32 MMAs.  B200's fp64 rate sits behind the tensor pipe: the CUDA-core DFMA
// version of this kernel measured 9 TFLOP/s (profiles/README.md).  The next chunk's global loads are issued into
// registers before the current chunk's MMAs, so DRAM / L2 latency is covered by arithmetic instead of by occupancy.
static constexpr int GT = 128, GK = 16, GS = GT + 4;   // GS: smem row pitch, = 8 words mod 32 -> conflict-free fragments

__device__ __forceinline__ void dmma_m8n8k4(double (&d)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(d[0]), "+d"(d[1]) : "d"(a), "d"(b));
}

// GTM = 128: one block per SM (64 accumulator doubles per thread).  GTM = 64: two blocks per SM, so one block's K loop
// overlaps the other's C read-modify-write — with one block per SM every tile paid ~25 us of exposed epilogue/prologue
// (rate model t = a + b*K fitted to 8.2 / 17 / 25.7 TFLOP/s at K = 64 / 256 / 4096), because the blocks of a wave
// finish together and all fetch their 128 KB of C at the same moment.
template <int GTM>
__global__ void __launch_bounds__(256, GTM == 64 ? 2 : 1)
dgemm_sub_kernel(DgemmArgs g) {
  constexpr int MT = GTM / 16;          // 8-row MMA tiles per warp (warp tile = GTM/2 x 32)
  constexpr int AE = GTM * GK / 256;    // A elements per thread per chunk
  constexpr int ASP = GTM + 4;          // A pitch: = 8 words mod 32 for both tile heights
  const int bi = blockIdx.y, bj = blockIdx.x;
  if (g.lower_only && bj * GT > bi * GTM + GTM - 1) return;
  // two smem stages (dynamic: 51 / 66 KB): global loads of chunk c+1 are issued before the MMAs of chunk c and parked
  // after them, one __syncthreads per chunk
  extern __shared__ __align__(16) double dg_smem[];
  double (*As)[GK][ASP] = reinterpret_cast<double (*)[GK][ASP]>(dg_smem);
  double (*Bs)[GK][GS] = reinterpret_cast<double (*)[GK][GS]>(dg_smem + 2 * GK * ASP);
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 2, wn = warp & 3;          // warp tile: rows wm*GTM/2.., cols wn*32..
  const int fr = lane >> 2, fk = lane & 3;          // fragment coordinates (groupID, threadID_in_group)
  const int i0 = bi * GTM, j0 = bj * GT;
  double acc[MT][4][2];
#pragma unroll
  for (int a = 0; a < MT; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;

  // loader mapping: GTM x 16 elements of A and 128 x 16 of B per chunk; the fastest-varying thread index runs along the
  // unit-stride direction of the operand so a warp reads whole 128 B lines.  Element pointers and row/column validity
  // are fixed per thread; a chunk only adds k0 * stride (the per-element 64-bit index arithmetic of the first version
  // cost as many instructions as the MMAs themselves).
  const bool a_t_fast = (g.sat == 1);
  const bool b_j_fast = (g.sbj == 1);
  double av[AE], bv[8];
  // element e of a thread = element 0 shifted by e * (di rows, dt depth) — 256 threads tile the chunk in whole rows /
  // columns — so one base pointer and one 64-bit step per operand describe all of them
  constexpr int A_DI_T = 16, A_DT_I = 256 / GTM;    // a_t_fast: +16 rows per e;  otherwise: +256/GTM depth per e
  const int a_i0 = a_t_fast ? (tid >> 4) : (tid & (GTM - 1));
  const int a_t0 = a_t_fast ? (tid & (GK - 1)) : (tid / GTM);
  const int a_di = a_t_fast ? A_DI_T : 0, a_dt = a_t_fast ? 0 : A_DT_I;
  const int b_j0 = b_j_fast ? (tid & (GT - 1)) : (tid >> 4);
  const int b_t0 = b_j_fast ? (tid >> 7) : (tid & (GK - 1));
  const int b_dj = b_j_fast ? 0 : 16, b_dt = b_j_fast ? 2 : 0;
  const double* ap0 = g.A + (long long)(i0 + a_i0) * g.sai + (long long)a_t0 * g.sat;
  const long long astep = (long long)a_di * g.sai + (long long)a_dt * g.sat;
  const double* bp0 = g.B + (long long)b_t0 * g.sbt + (long long)(j0 + b_j0) * g.sbj;
  const long long bstep = (long long)b_dt * g.sbt + (long long)b_dj * g.sbj;
  auto load_chunk = [&](int k0) {
    const double* pa = ap0 + (long long)k0 * g.sat;
    const double* pb = bp0 + (long long)k0 * g.sbt;
#pragma unroll
    for (int e = 0; e < AE; ++e)
      av[e] = (i0 + a_i0 + e * a_di < g.M && k0 + a_t0 + e * a_dt < g.K) ? pa[e * astep] : 0.0;
#pragma unroll
    for (int e = 0; e < 8; ++e)
      bv[e] = (j0 + b_j0 + e * b_dj < g.N && k0 + b_t0 + e * b_dt < g.K) ? pb[e * bstep] : 0.0;
  };
  auto park = [&](int st) {
#pragma unroll
    for (int e = 0; e < AE; ++e) As[st][a_t0 + e * a_dt][a_i0 + e * a_di] = av[e];
#pragma unroll
    for (int e = 0; e < 8; ++e) Bs[st][b_t0 + e * b_dt][b_j0 + e * b_dj] = bv[e];
  };
  load_chunk(0);
  park(0);
  __syncthreads();
  int cur = 0;
  for (int k0 = 0; k0 < g.K; k0 += GK) {
    const bool more = k0 + GK < g.K;
    if (more) load_chunk(k0 + GK);
#pragma unroll
    for (int t = 0; t < GK; t += 4) {
      double a[MT], b[4];
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) a[mt] = As[cur][t + fk][wm * (GTM / 2) + mt * 8 + fr];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) b[nt] = Bs[cur][t + fk][wn * 32 + nt * 8 + fr];
#pragma unroll
      for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) dmma_m8n8k4(acc[mt][nt], a[mt], b[nt]);
    }
    if (more) park(cur ^ 1);     // the stage read two iterations ago: everyone passed the barrier that followed it
    __syncthreads();
    cur ^= 1;
  }
  // C -= acc.  Each thread owns column pairs (2fk, 2fk+1): one 16-byte access per pair, so the four lanes of a fragment
  // row cover a whole 64 B (two full sectors) — 8-byte accesses wrote every sector in four partial pieces and the
  // read-modify-write of C ran at ~1 TB/s.  Loads are gathered in batches before any store of the batch (a store may
  // alias the next load as far as the compiler knows, which would serialise the L2 round trips).  Row offsets are
  // 64-bit like the operand pointers': C may span more than 2^31 elements.
  const bool vec_ok = ((g.ldc & 1) == 0) && ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0);
#pragma unroll
  for (int mb = 0; mb < MT; mb += 2) {
    double2 cv[2][4];
#pragma unroll
    for (int m2 = 0; m2 < 2; ++m2) {
      const int i = i0 + wm * (GTM / 2) + (mb + m2) * 8 + fr;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const int j = j0 + wn * 32 + nt * 8 + 2 * fk;
        const bool ok0 = i < g.M && j < g.N && !(g.lower_only && j > i);
        const bool ok1 = i < g.M && j + 1 < g.N && !(g.lower_only && j + 1 > i);
        if (vec_ok && ok0 && ok1) cv[m2][nt] = *reinterpret_cast<const double2*>(g.C + (long long)i * g.ldc + j);
        else {
          cv[m2][nt].x = ok0 ? g.C[(long long)i * g.ldc + j] : 0.0;
          cv[m2][nt].y = ok1 ? g.C[(long long)i * g.ldc + j + 1] : 0.0;
        }
      }
    }
#pragma unroll
    for (int m2 = 0; m2 < 2; ++m2) {
      const int i = i0 + wm * (GTM / 2) + (mb + m2) * 8 + fr;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const int j = j0 + wn * 32 + nt * 8 + 2 * fk;
        const bool ok0 = i < g.M && j < g.N && !(g.lower_only && j > i);
        const bool ok1 = i < g.M && j + 1 < g.N && !(g.lower_only && j + 1 > i);
        const double2 o = make_double2(cv[m2][nt].x - acc[mb + m2][nt][0], cv[m2][nt].y - acc[mb + m2][nt][1]);
        if (vec_ok && ok0 && ok1) *reinterpret_cast<double2*>(g.C + (long long)i * g.ldc + j) = o;
        else {
          if (ok0) g.C[(long long)i * g.ldc + j] = o.x;
          if (ok1) g.C[(long long)i * g.ldc + j + 1] = o.y;
        }
      }
    }
  }
}

static constexpr size_t dgemm_smem(int gtm) { return (size_t)2 * GK * ((gtm + 4) + GS) * sizeof(double); }
static int dgemm_sub(const DgemmArgs& g, cudaStream_t st) {
  if (g.M <= 0 || g.N <= 0 || g.K <= 0) return NIB_OK;
  static const int tile_m = [] { const char* e = getenv("NIB_GP_TILE_M"); return e && atoi(e) == 128 ? 128 : 64; }();
  static bool attr = false;
  if (!attr) {
    NIB_CUDA(cudaFuncSetAttribute(dgemm_sub_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dgemm_smem(128)));
    NIB_CUDA(cudaFuncSetAttribute(dgemm_sub_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dgemm_smem(64)));
    attr = true;
  }
  dim3 grid(ceil_div(g.N, GT), ceil_div(g.M, tile_m));
  if (tile_m == 128) dgemm_sub_kernel<128><<<grid, 256, dgemm_smem(128), st>>>(g);
  else dgemm_sub_kernel<64><<<grid, 256, dgemm_smem(64), st>>>(g);
  NIB_LAUNCH_CHECK();
  return NIB_OK;
}

// ---- inverses of the 64 x 64 diagonal blocks -----------------------------------------------------
// Every latency-bound triangular step (panel solve below a diagonal block, diagonal solve of a TRSM step, single-vector
// solves) becomes a 64-deep matrix product once inv(Lkk) is known, and the rest of the solve is GEMM.  A dependent fp64
// operation costs ~48 cycles here (measured: 64 elimination steps of ~25 dependent operations took 41.6 us), so the
// inverse is built by block doubling with all 256 threads instead of 64 independent forward substitutions (27 us):
// 4 x 4 diagonal blocks directly, then inv([[A,0],[B,C]]) = [[Ai,0],[-Ci*B*Ai,Ci]] for block sizes 4, 8, 16, 32 —
// about 80 dependent operations in total.  Ls: the factor block (identity padded), Xs: the inverse (zeros above the
// diagonal), both 64 x 65 in shared memory; called by all 256 threads.
__device__ __forceinline__ void trtri64_coop(const double (*Ls)[NB + 1], double (*Xs)[NB + 1], const double* rdiag) {
  // rdiag[r] = 1 / Ls[r][r] (shared memory).  Every loop below has a uniform trip count — the zeros above the diagonal of
  // Xs stand in for the triangular bounds — so a thread's elements advance together as independent FMA chains.
  const int tid = threadIdx.x;
  for (int idx = tid; idx < NB * NB; idx += 256) Xs[idx >> 6][idx & 63] = 0.0;
  __syncthreads();
  if (tid < NB) {   // 4 x 4 diagonal blocks: thread = (block, column)
    const int b0 = tid & ~3, c = tid & 3;
    double x[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      double sacc = (r == c) ? 1.0 : 0.0;
#pragma unroll
      for (int t = 0; t < r; ++t) sacc = fma(-Ls[b0 + r][b0 + t], x[t], sacc);
      x[r] = (r >= c) ? sacc * rdiag[b0 + r] : 0.0;
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) Xs[b0 + r][b0 + c] = x[r];
  }
  __syncthreads();
#pragma unroll
  for (int lv = 0; lv < 4; ++lv) {
    const int sz = 4 << lv;                     // 4, 8, 16, 32 (compile-time after unrolling)
    const int per = sz * sz;                    // elements of one off-diagonal block
    const int total = (NB / (2 * sz)) * per;    // 32 * sz
    constexpr int EMAX = 4;
    const int ne = (total + 255) / 256;         // elements per thread: 1, 1, 2, 4
    int ri[EMAX], cj[EMAX], bs[EMAX];
    double tv[EMAX];
#pragma unroll
    for (int e = 0; e < EMAX; ++e) {
      const int idx = tid + e * 256;
      const int pr = idx / per, w = idx - pr * per;
      ri[e] = w / sz; cj[e] = w - ri[e] * sz; bs[e] = 2 * sz * pr;
    }
    // T = B * Ai, parked where the result block will live
#pragma unroll
    for (int e = 0; e < EMAX; ++e) {
      if (e < ne && tid + e * 256 < total) {
        double a0 = 0.0, a1 = 0.0;
#pragma unroll 4
        for (int t = 0; t < sz; t += 2) {
          a0 = fma(Ls[bs[e] + sz + ri[e]][bs[e] + t], Xs[bs[e] + t][bs[e] + cj[e]], a0);
          a1 = fma(Ls[bs[e] + sz + ri[e]][bs[e] + t + 1], Xs[bs[e] + t + 1][bs[e] + cj[e]], a1);
        }
        tv[e] = a0 + a1;
      }
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < EMAX; ++e)
      if (e < ne && tid + e * 256 < total) Xs[bs[e] + sz + ri[e]][bs[e] + cj[e]] = tv[e];
    __syncthreads();
    // O = -Ci * T
#pragma unroll
    for (int e = 0; e < EMAX; ++e) {
      if (e < ne && tid + e * 256 < total) {
        double a0 = 0.0, a1 = 0.0;
#pragma unroll 4
        for (int t = 0; t < sz; t += 2) {
          a0 = fma(Xs[bs[e] + sz + ri[e]][bs[e] + sz + t], Xs[bs[e] + sz + t][bs[e] + cj[e]], a0);
          a1 = fma(Xs[bs[e] + sz + ri[e]][bs[e] + sz + t + 1], Xs[bs[e] + sz + t + 1][bs[e] + cj[e]], a1);
        }
        tv[e] = -(a0 + a1);
      }
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < EMAX; ++e)
      if (e < ne && tid + e * 256 < total) Xs[bs[e] + sz + ri[e]][bs[e] + cj[e]] = tv[e];
    __syncthreads();
  }
}

static constexpr size_t TRTRI_SMEM = (size_t)2 * NB * (NB + 1) * sizeof(double);   // Ls + Xs, dynamic (66.5 KB)

// all diagonal blocks of a finished factor at once (TRSM entry points are stateless: they rebuild the inverses)
__global__ void __launch_bounds__(256)
trtri64_batched_kernel(const double* __restrict__ Lm, int ldl, int n, double* __restrict__ dinv) {
  extern __shared__ __align__(16) double tt_smem[];
  double (*Ls)[NB + 1] = reinterpret_cast<double (*)[NB + 1]>(tt_smem);
  double (*Xs)[NB + 1] = reinterpret_cast<double (*)[NB + 1]>(tt_smem + NB * (NB + 1));
  const int k0 = blockIdx.x * NB;
  const int nb = min(NB, n - k0);
  double lv[16];
#pragma unroll
  for (int e = 0; e < 16; ++e) {
    const int idx = threadIdx.x + e * 256, i = idx >> 6, j = idx & 63;
    lv[e] = (i < nb && j <= i) ? Lm[(size_t)(k0 + i) * ldl + k0 + j] : ((i == j) ? 1.0 : 0.0);
  }
#pragma unroll
  for (int e = 0; e < 16; ++e) {
    const int idx = threadIdx.x + e * 256;
    Ls[idx >> 6][idx & 63] = lv[e];
  }
  __shared__ double rdiag[NB];
  __syncthreads();
  if (threadIdx.x < NB) rdiag[threadIdx.x] = 1.0 / Ls[threadIdx.x][threadIdx.x];
  __syncthreads();
  trtri64_coop(Ls, Xs, rdiag);
  double* out = dinv + (size_t)blockIdx.x * NB * NB;
  for (int idx = threadIdx.x; idx < NB * NB; idx += 256) out[idx] = Xs[idx >> 6][idx & 63];
}

// out = P * Q on one 64 x 64 tile with a 64-deep product, in place on the matrix operand:
//   mode 0  rows [k0, k0+nb) of M  <-  D * rows          (forward TRSM step; tile = 64 columns from 64 * blockIdx.x)
//   mode 1  rows [k0, k0+nb) of M  <-  D^T * rows        (backward TRSM step)
//   mode 2  M[r0 + rows, k0 : k0+nb)  <-  rows * D^T     (panel below a Cholesky diagonal block; tile = 64 rows)
// D = inverse of the diagonal block.  256 threads, 4 x 4 outputs each; the in-place operand is staged whole before any
// store.  66 KB of dynamic shared memory.
static constexpr int AP = NB + 2;   // Q pitch: keeps 16-byte alignment for the paired loads
__global__ void __launch_bounds__(256)
apply_dinv_kernel(const double* __restrict__ D, double* __restrict__ Mx, long long ld, int k0, int nb, int r0, int count,
                  int mode, const int* __restrict__ info) {
  extern __shared__ __align__(16) double ap_smem[];
  double (*Ps)[NB + 1] = reinterpret_cast<double (*)[NB + 1]>(ap_smem);
  double (*Qs)[AP] = reinterpret_cast<double (*)[AP]>(ap_smem + NB * (NB + 1));   // 4160 doubles: 16-byte aligned
  if (info != nullptr && *info != 0) return;
  const int tid = threadIdx.x;
  const int o0 = blockIdx.x * NB;                 // first column (modes 0/1) or first row offset (mode 2) of this tile
  // both 64 x 64 operands are fetched into registers first (32 independent loads in flight per thread), then parked:
  // a load -> store loop pays one DRAM/L2 round trip per iteration
  double mv[16], dv[16];
#pragma unroll
  for (int e = 0; e < 16; ++e) {
    const int idx = tid + e * 256;
    const int a = idx >> 6, b = idx & 63;          // b runs along the unit-stride direction of both sources
    dv[e] = D[a * NB + b];
    if (mode == 2) mv[e] = (o0 + a < count && b < nb) ? Mx[(size_t)(r0 + o0 + a) * ld + k0 + b] : 0.0;
    else mv[e] = (a < nb && o0 + b < count) ? Mx[(size_t)(k0 + a) * ld + o0 + b] : 0.0;
  }
#pragma unroll
  for (int e = 0; e < 16; ++e) {
    const int idx = tid + e * 256;
    const int a = idx >> 6, b = idx & 63;
    if (mode == 2) {
      Ps[a][b] = mv[e];          // P[i][t] = rows
      Qs[b][a] = dv[e];          // Q[t][j] = D[j][t]
    } else {
      Qs[a][b] = mv[e];          // Q[t][j] = rows
      if (mode == 0) Ps[a][b] = dv[e]; else Ps[b][a] = dv[e];   // P = D or D^T
    }
  }
  __syncthreads();
  const int ty = tid >> 4, tx = tid & 15;
  double acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
#pragma unroll 8
  for (int t = 0; t < NB; ++t) {
    double pv[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) pv[a] = Ps[4 * ty + a][t];
    const double2 q01 = *reinterpret_cast<const double2*>(&Qs[t][4 * tx]);
    const double2 q23 = *reinterpret_cast<const double2*>(&Qs[t][4 * tx + 2]);
    const double qv[4] = {q01.x, q01.y, q23.x, q23.y};
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[a][b] = fma(pv[a], qv[b], acc[a][b]);
  }
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int i = 4 * ty + a, j = 4 * tx + b;
      if (mode == 2) {
        if (o0 + i < count && j < nb) Mx[(size_t)(r0 + o0 + i) * ld + k0 + j] = acc[a][b];
      } else {
        if (i < nb && o0 + j < count) Mx[(size_t)(k0 + i) * ld + o0 + j] = acc[a][b];
      }
    }
}
static constexpr size_t AP_SMEM = (size_t)(NB * (NB + 1) + 2 + NB * AP) * sizeof(double);

static int apply_dinv(const double* D, double* Mx, long long ld, int k0, int nb, int r0, int count, int mode,
                      const int* info, cudaStream_t st) {
  static bool attr = false;
  if (!attr) {
    NIB_CUDA(cudaFuncSetAttribute(apply_dinv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AP_SMEM));
    attr = true;
  }
  if (count <= 0 || nb <= 0) return NIB_OK;
  apply_dinv_kernel<<<ceil_div(count, NB), 256, AP_SMEM, st>>>(D, Mx, ld, k0, nb, r0, count, mode, info);
  NIB_LAUNCH_CHECK();
  return NIB_OK;
}

__global__ void potrf_diag_kernel(double* __restrict__ A, int ld, int k0, int nb, int* __restrict__ info, double* __restrict__ dinv);
static int trtri_attrs() {
  static bool done = false;
  if (!done) {
    NIB_CUDA(cudaFuncSetAttribute(trtri64_batched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TRTRI_SMEM));
    NIB_CUDA(cudaFuncSetAttribute(potrf_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TRTRI_SMEM));
    done = true;
  }
  return NIB_OK;
}

// scratch for the diagonal-block inverses of the factor currently being built / solved with (per stream, common.cuh)
static int get_dinv(int n, cudaStream_t st, double** dinv) {
  const size_t need = (size_t)ceil_div(n, NB) * NB * NB * sizeof(double);
  return stream_scratch(SCRATCH_GP_DINV, st, need, (size_t)256 * NB * NB * sizeof(double), reinterpret_cast<void**>(dinv));
}
static inline int split64(int w) { return ((w / 2 + NB - 1) / NB) * NB; }   // NB <= split < w for w > NB

// ---- Cholesky --------------------------------------------------------------------------------
// Factor the nb x nb (<= 64) diagonal block at (k0,k0).  The block lives in registers: thread (br, bc) of a 16 x 16
// grid owns the 4 x 4 sub-block (rows 4br.., cols 4bc..); each of the 64 elimination steps publishes one column
// through a double-buffered 64-entry smem vector, so a step costs one __syncthreads and 16 predicated FMAs per thread
// (right-looking, the update order of LAPACK dpotf2 that scipy.linalg.cholesky ends in, _gpr.py:352).
__global__ void __launch_bounds__(256)
potrf_diag_kernel(double* __restrict__ A, int ld, int k0, int nb, int* __restrict__ info, double* __restrict__ dinv) {
  __shared__ __align__(16) double colbuf[2][NB];
  __shared__ double rdiag[NB];
  extern __shared__ __align__(16) double pd_smem[];   // the factored block and its inverse (dinv != null), TRTRI_SMEM bytes
  double (*Lsh)[NB + 1] = reinterpret_cast<double (*)[NB + 1]>(pd_smem);
  double (*Xsh)[NB + 1] = reinterpret_cast<double (*)[NB + 1]>(pd_smem + NB * (NB + 1));
  const int tid = threadIdx.x;
  const int br = tid >> 4, bc = tid & 15;
  double r[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int i = 4 * br + a, j = 4 * bc + b;
      r[a][b] = (i < nb && j <= i) ? A[(size_t)(k0 + i) * ld + k0 + j] : ((i == j) ? 1.0 : 0.0);   // identity padding
    }
  // The pivot loop is bound by the number of instructions each warp issues per pivot (two warps per scheduler, every
  // instruction waiting on the one before): with the update predicated per element it was ~240 instructions and 1400
  // cycles per pivot.  Here the 16 FMAs are unconditional — the scaled column is zeroed for the columns that are
  // already final, and the strictly upper part of the block carries values nothing reads — and the column index is a
  // compile-time constant (j = 4 jb + cj, cj unrolled).
  for (int jb = 0; jb < NB / 4; ++jb) {
#pragma unroll
    for (int cj = 0; cj < 4; ++cj) {
      const int j = 4 * jb + cj;
      double* col = colbuf[cj & 1];
      if (bc == jb) {
        *reinterpret_cast<double2*>(col + 4 * br) = make_double2(r[0][cj], r[1][cj]);
        *reinterpret_cast<double2*>(col + 4 * br + 2) = make_double2(r[2][cj], r[3][cj]);
      }
      __syncthreads();
      const double d = col[j];
      if (!(d > 0.0)) {  // also catches NaN; uniform across the block
        if (tid == 0 && *info == 0) *info = k0 + j + 1;
        return;
      }
      // one reciprocal square root instead of a square root followed by a division (CUDA's double rsqrt: 1 ulp)
      const double inv = rsqrt(d);
      if (tid == 0) rdiag[j] = inv;     // = 1 / L[j][j], reused by the inverse
      const double2 c01 = *reinterpret_cast<const double2*>(col + 4 * br);
      const double2 c23 = *reinterpret_cast<const double2*>(col + 4 * br + 2);
      const double2 k01 = *reinterpret_cast<const double2*>(col + 4 * bc);
      const double2 k23 = *reinterpret_cast<const double2*>(col + 4 * bc + 2);
      const double lr[4] = {c01.x * inv, c01.y * inv, c23.x * inv, c23.y * inv};
      double lc[4] = {k01.x * inv, k01.y * inv, k23.x * inv, k23.y * inv};
      if (bc < jb) { lc[0] = 0.0; lc[1] = 0.0; lc[2] = 0.0; lc[3] = 0.0; }
      if (bc == jb) {
#pragma unroll
        for (int b = 0; b <= cj; ++b) lc[b] = 0.0;
      }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) r[a][b] = fma(-lr[a], lc[b], r[a][b]);
      if (bc == jb) {
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          const int i = 4 * br + a;
          if (i > j) r[a][cj] = lr[a];
          if (i == j) r[a][cj] = d * inv;
        }
      }
    }
  }
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int i = 4 * br + a, j = 4 * bc + b;
      if (i < nb && j <= i) A[(size_t)(k0 + i) * ld + k0 + j] = r[a][b];
      if (dinv != nullptr) Lsh[i][j] = (j <= i) ? r[a][b] : 0.0;   // identity padding beyond nb comes out of the elimination itself
    }
  if (dinv == nullptr) return;
  __syncthreads();
  trtri64_coop(Lsh, Xsh, rdiag);
  for (int idx = tid; idx < NB * NB; idx += 256) dinv[idx] = Xsh[idx >> 6][idx & 63];
}

// rows below the diagonal block: solve X * Lkk^T = A[i, k0:k0+nb], one row per thread; four interleaved partial sums
// keep four independent FMA chains in flight (the single-chain version is bound by the fp64 FMA latency)
__global__ void __launch_bounds__(128)
trsm_panel_kernel(double* __restrict__ A, int ld, int k0, int nb, int n, const int* __restrict__ info) {
  __shared__ double L[NB][NB + 1];
  if (*info != 0) return;
  for (int idx = threadIdx.x; idx < NB * NB; idx += blockDim.x) {
    int i = idx / NB, j = idx - i * NB;
    L[i][j] = (i < nb && j <= i) ? A[(size_t)(k0 + i) * ld + k0 + j] : ((i == j) ? 1.0 : 0.0);
  }
  __syncthreads();
  const int i = k0 + nb + blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double x[NB];
  double* row = A + (size_t)i * ld + k0;
#pragma unroll
  for (int j = 0; j < NB; ++j) x[j] = (j < nb) ? row[j] : 0.0;
#pragma unroll
  for (int j = 0; j < NB; ++j) {
    double s0 = x[j], s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
    for (int t = 0; t + 3 < j; t += 4) {
      s0 = fma(-x[t], L[j][t], s0);
      s1 = fma(-x[t + 1], L[j][t + 1], s1);
      s2 = fma(-x[t + 2], L[j][t + 2], s2);
      s3 = fma(-x[t + 3], L[j][t + 3], s3);
    }
#pragma unroll
    for (int t = j & ~3; t < j; ++t) s0 = fma(-x[t], L[j][t], s0);
    x[j] = ((s0 + s1) + (s2 + s3)) / L[j][j];
  }
#pragma unroll
  for (int j = 0; j < NB; ++j)
    if (j < nb) row[j] = x[j];
}

// ---- triangular solves on many right-hand sides ----------------------------------------------
// forward:  rows [k0,k0+nb) of B <- Lkk^{-1} * rows;  one column per thread
__global__ void __launch_bounds__(128)
trsm_diag_fwd_kernel(const double* __restrict__ Lm, int ldl, double* __restrict__ B, int ldb, int nrhs, int k0, int nb) {
  __shared__ double L[NB][NB + 1];
  for (int idx = threadIdx.x; idx < nb * nb; idx += blockDim.x) {
    int i = idx / nb, j = idx - i * nb;
    L[i][j] = (j <= i) ? Lm[(size_t)(k0 + i) * ldl + k0 + j] : 0.0;
  }
  __syncthreads();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nrhs) return;
  double x[NB];
#pragma unroll
  for (int r = 0; r < NB; ++r) {
    if (r < nb) {
      double s0 = B[(size_t)(k0 + r) * ldb + c], s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
      for (int t = 0; t + 3 < r; t += 4) {
        s0 = fma(-L[r][t], x[t], s0);
        s1 = fma(-L[r][t + 1], x[t + 1], s1);
        s2 = fma(-L[r][t + 2], x[t + 2], s2);
        s3 = fma(-L[r][t + 3], x[t + 3], s3);
      }
#pragma unroll
      for (int t = r & ~3; t < r; ++t) s0 = fma(-L[r][t], x[t], s0);
      x[r] = ((s0 + s1) + (s2 + s3)) / L[r][r];
      B[(size_t)(k0 + r) * ldb + c] = x[r];
    }
  }
}
// backward: rows [k0,k0+nb) of B <- Lkk^{-T} * rows
__global__ void __launch_bounds__(128)
trsm_diag_bwd_kernel(const double* __restrict__ Lm, int ldl, double* __restrict__ B, int ldb, int nrhs, int k0, int nb) {
  __shared__ double L[NB][NB + 1];
  for (int idx = threadIdx.x; idx < nb * nb; idx += blockDim.x) {
    int i = idx / nb, j = idx - i * nb;
    L[i][j] = (j <= i) ? Lm[(size_t)(k0 + i) * ldl + k0 + j] : 0.0;
  }
  __syncthreads();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nrhs) return;
  double x[NB];
#pragma unroll
  for (int rr = 0; rr < NB; ++rr) {
    const int r = NB - 1 - rr;
    if (r < nb) {
      double sacc = B[(size_t)(k0 + r) * ldb + c];
#pragma unroll
      for (int t = r + 1; t < NB; ++t)
        if (t < nb) sacc = fma(-L[t][r], x[t], sacc);
      x[r] = sacc / L[r][r];
      B[(size_t)(k0 + r) * ldb + c] = x[r];
    }
  }
}

// ---- single right-hand side (alpha = K^-1 y, _gpr.py:363-367) ----------------------------------
// One launch per 64-row block of L.  Every thread block re-solves the 64 x 64 diagonal system in its first warp (64
// shuffle-broadcast steps, cheaper than a grid-wide dependency) and then applies the block column / block row of L to
// its own slice of the remaining vector: a streaming GEMV, L is read exactly once per solve.
__device__ __forceinline__ void trsv_diag_warp(const double (*Ls)[NB + 1], double* xs, int nb, bool transposed) {
  // warp 0: lane owns entries lane and lane + 32 of the block's right-hand side (already in xs)
  const int lane = threadIdx.x;
  double b0 = xs[lane], b1 = xs[lane + 32];
  if (!transposed) {
    for (int j = 0; j < NB; ++j) {
      const double bj = __shfl_sync(0xffffffffu, j < 32 ? b0 : b1, j & 31);
      const double xj = bj / Ls[j][j];
      if (lane == (j & 31)) { if (j < 32) b0 = xj; else b1 = xj; }
      if (lane > j) b0 = fma(-Ls[lane][j], xj, b0);
      if (lane + 32 > j) b1 = fma(-Ls[lane + 32][j], xj, b1);
    }
  } else {
    for (int j = NB - 1; j >= 0; --j) {
      const double bj = __shfl_sync(0xffffffffu, j < 32 ? b0 : b1, j & 31);
      const double xj = bj / Ls[j][j];
      if (lane == (j & 31)) { if (j < 32) b0 = xj; else b1 = xj; }
      if (lane < j) b0 = fma(-Ls[j][lane], xj, b0);
      if (lane + 32 < j) b1 = fma(-Ls[j][lane + 32], xj, b1);
    }
  }
  (void)nb;
  xs[lane] = b0;
  xs[lane + 32] = b1;
}

__global__ void __launch_bounds__(256)
trsv_step_kernel(const double* __restrict__ Lm, int ldl, double* __restrict__ b, double* __restrict__ x, int n, int k0,
                 int nb, int trans, const double* __restrict__ dinv) {
  __shared__ double Ls[NB][NB + 1];
  __shared__ double xs[NB];
  __shared__ double bs[NB];
  const int tid = threadIdx.x;
  if (dinv != nullptr) {
    // diagonal system through the block inverse: a 64 x 64 product (4 threads per row, 16-deep chains) instead of 64
    // dependent divide / broadcast steps in one warp (~20 us of the 23 us this kernel used to take)
    const double* D = dinv + (size_t)(k0 / NB) * NB * NB;
    double dv[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) dv[e] = D[tid + e * 256];
    if (tid < NB) bs[tid] = tid < nb ? b[k0 + tid] : 0.0;
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      const int idx = tid + e * 256, a = idx >> 6, c = idx & 63;
      if (trans) Ls[c][a] = dv[e]; else Ls[a][c] = dv[e];     // Ls = D or D^T
    }
    __syncthreads();
    const int row = tid >> 2, q = tid & 3;
    double acc = 0.0;
#pragma unroll
    for (int t = 0; t < 16; ++t) acc = fma(Ls[row][q * 16 + t], bs[q * 16 + t], acc);
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    if (q == 0) xs[row] = acc;
  } else {
    for (int idx = tid; idx < NB * NB; idx += 256) {
      const int i = idx / NB, j = idx - i * NB;
      Ls[i][j] = (i < nb && j <= i) ? Lm[(size_t)(k0 + i) * ldl + k0 + j] : ((i == j) ? 1.0 : 0.0);
    }
    if (tid < NB) xs[tid] = tid < nb ? b[k0 + tid] : 0.0;
    __syncthreads();
    if (tid < 32) trsv_diag_warp(Ls, xs, nb, trans != 0);
  }
  __syncthreads();
  // the solved entries go to a separate vector: blocks of this launch that start late must still read the unsolved b
  if (blockIdx.x == 0 && tid < nb) x[k0 + tid] = xs[tid];
  if (!trans) {
    // rows below the block: b[i] -= L[i][k0 .. k0+nb) . x   (one warp per row, lanes along the 64 columns)
    const int warp = tid >> 5, lane = tid & 31;
    for (int i = k0 + nb + blockIdx.x * 8 + warp; i < n; i += gridDim.x * 8) {
      const double* row = Lm + (size_t)i * ldl + k0;
      double acc = row[lane] * xs[lane];
      if (lane + 32 < nb) acc = fma(row[lane + 32], xs[lane + 32], acc);
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) b[i] -= acc;
    }
  } else {
    // columns left of the block: b[j] -= sum_t L[k0+t][j] * x[t]   (one thread per column, coalesced along j)
    for (int j = blockIdx.x * 256 + tid; j < k0; j += gridDim.x * 256) {
      double acc = 0.0;
      for (int t = 0; t < nb; ++t) acc = fma(Lm[(size_t)(k0 + t) * ldl + j], xs[t], acc);
      b[j] -= acc;
    }
  }
}

// Wavefront form of the same solve: ONE launch, one thread block per 64-row block of L.  Block i accumulates
// L[i][k] x_k (L^T: L[k][i]^T x_k) for its dependencies k in the order they finish, then multiplies by the inverse
// diagonal block and publishes x_i.  There is no flag: the solved vector goes to a scratch copy that starts out as a
// sentinel bit pattern (all ones, a NaN no computation produces: NaN results are canonicalised before the store), and
// warp 0 of every waiting block polls the 64 values it needs until none is the sentinel — data and "ready" arrive in the
// same L2 round trip.  The L tile of the next dependency is already in registers when x_k arrives, so a chain step is
// one L2 round trip, two 4-deep FMA chains and two block barriers instead of a kernel launch (128 launches of ~10 us
// at n = 8192 before; 0.77 / 0.49 ms per solve with an acquire flag + fence per step).
// Forward progress: block i only waits on blocks the hardware dispatched before it (blockIdx order follows the dependency
// order in both directions), so the lowest unfinished block is always resident; the spin is bounded and traps.
static constexpr unsigned long long TRSV_SENTINEL = 0xFFFFFFFFFFFFFFFFull;

__device__ __forceinline__ void wave_fetch(const double* xw, int k, int n, double* dst) {
  // warp 0: lane owns entries lane and lane + 32 of block k
  const int lane = threadIdx.x;
  const int r0 = k * NB + lane, r1 = r0 + 32;
  const volatile unsigned long long* p = reinterpret_cast<const volatile unsigned long long*>(xw);
  unsigned long long v0 = 0ull, v1 = 0ull;
  unsigned spins = 0;
  for (;;) {
    v0 = r0 < n ? p[r0] : 0ull;
    v1 = r1 < n ? p[r1] : 0ull;
    if (__all_sync(0xffffffffu, v0 != TRSV_SENTINEL && v1 != TRSV_SENTINEL)) break;
    if (++spins > 256u) __nanosleep(20);
    if (spins > (1u << 26)) __trap();
  }
  dst[lane] = __longlong_as_double((long long)v0);
  dst[lane + 32] = __longlong_as_double((long long)v1);
}

__global__ void __launch_bounds__(256)
trsv_wave_kernel(const double* __restrict__ Lm, int ldl, double* __restrict__ b, int n, int trans,
                 const double* __restrict__ dinv, double* xw) {
  __shared__ double Ds[NB][NB + 1];
  __shared__ double part[4][NB];
  __shared__ double bs[NB];
  __shared__ double xs[2][NB];
  const int tid = threadIdx.x;
  const int nblk = (n + NB - 1) / NB;
  const int blk = trans ? nblk - 1 - (int)blockIdx.x : (int)blockIdx.x;
  const int k0 = blk * NB;
  const int nb = min(NB, n - k0);
  {
    const double* D = dinv + (size_t)blk * NB * NB;
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      const int idx = tid + e * 256, a = idx >> 6, c = idx & 63;
      const double v = D[idx];
      if (trans) Ds[c][a] = v; else Ds[a][c] = v;              // Ds = inv(Lkk) or its transpose
    }
  }
  const int ndeps = (int)blockIdx.x;
  double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
  double l[16];
  if (!trans) {
    // thread (row, q): 16 consecutive columns of row k0+row in block column k
    const int row = tid >> 2, q = tid & 3;
    const bool live = row < nb;
    const double* base = Lm + (size_t)(k0 + (live ? row : 0)) * ldl + q * 16;
    if (ndeps > 0) {
#pragma unroll
      for (int t = 0; t < 16; ++t) l[t] = live ? __ldg(base + t) : 0.0;
    }
    for (int k = 0; k < ndeps; ++k) {
      if (tid < 32) wave_fetch(xw, k, n, xs[k & 1]);
      __syncthreads();
      const double* xv = xs[k & 1] + q * 16;
#pragma unroll
      for (int t = 0; t < 16; t += 4) {
        acc0 = fma(l[t], xv[t], acc0);
        acc1 = fma(l[t + 1], xv[t + 1], acc1);
        acc2 = fma(l[t + 2], xv[t + 2], acc2);
        acc3 = fma(l[t + 3], xv[t + 3], acc3);
      }
      if (k + 1 < ndeps) {
        const double* nx = base + (size_t)(k + 1) * NB;
#pragma unroll
        for (int t = 0; t < 16; ++t) l[t] = live ? __ldg(nx + t) : 0.0;
      }
    }
    double acc = (acc0 + acc1) + (acc2 + acc3);
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    if (q == 0) bs[row] = live ? b[k0 + row] - acc : 0.0;
  } else {
    // thread (c, tq): column k0+c of rows k*NB + tq*16 .. +16 (coalesced along c)
    const int c = tid & 63, tq = tid >> 6;
    const bool live = c < nb;
    const double* base = Lm + k0 + (live ? c : 0);
    auto load_tile = [&](int k) {
#pragma unroll
      for (int t = 0; t < 16; ++t) {
        const int r = k * NB + tq * 16 + t;
        l[t] = (live && r < n) ? __ldg(base + (size_t)r * ldl) : 0.0;
      }
    };
    if (ndeps > 0) load_tile(nblk - 1);
    for (int s = 0; s < ndeps; ++s) {
      const int k = nblk - 1 - s;
      if (tid < 32) wave_fetch(xw, k, n, xs[s & 1]);
      __syncthreads();
      const double* xv = xs[s & 1] + tq * 16;
#pragma unroll
      for (int t = 0; t < 16; t += 4) {
        acc0 = fma(l[t], xv[t], acc0);
        acc1 = fma(l[t + 1], xv[t + 1], acc1);
        acc2 = fma(l[t + 2], xv[t + 2], acc2);
        acc3 = fma(l[t + 3], xv[t + 3], acc3);
      }
      if (s + 1 < ndeps) load_tile(k - 1);
    }
    part[tq][c] = (acc0 + acc1) + (acc2 + acc3);
    __syncthreads();
    if (tid < NB) bs[tid] = tid < nb ? b[k0 + tid] - ((part[0][tid] + part[1][tid]) + (part[2][tid] + part[3][tid])) : 0.0;
  }
  __syncthreads();
  {
    const int row = tid >> 2, q = tid & 3;
    double x0 = 0.0, x1 = 0.0, x2 = 0.0, x3 = 0.0;
#pragma unroll
    for (int t = 0; t < 16; t += 4) {
      x0 = fma(Ds[row][q * 16 + t], bs[q * 16 + t], x0);
      x1 = fma(Ds[row][q * 16 + t + 1], bs[q * 16 + t + 1], x1);
      x2 = fma(Ds[row][q * 16 + t + 2], bs[q * 16 + t + 2], x2);
      x3 = fma(Ds[row][q * 16 + t + 3], bs[q * 16 + t + 3], x3);
    }
    double x = (x0 + x1) + (x2 + x3);
    x += __shfl_xor_sync(0xffffffffu, x, 1);
    x += __shfl_xor_sync(0xffffffffu, x, 2);
    if (q == 0 && row < nb) {
      if (x != x) x = __longlong_as_double(0x7ff8000000000000ll);   // never the sentinel
      __stcg(xw + k0 + row, x);
      b[k0 + row] = x;
    }
  }
}

static bool trsv_wave_on() {
  static const bool v = getenv("NIB_GP_TRSV_STEPS") == nullptr;   // A/B switch: the one-launch-per-block form
  return v;
}

static int trsv_impl(const double* L, int n, int ldl, double* b, int trans, const double* dinv, cudaStream_t st) {
  const int nblk = ceil_div(n, NB);
  if (dinv != nullptr && trsv_wave_on()) {
    double* xw = nullptr;
    int rcf = stream_scratch(SCRATCH_GP_TRSV, st, (size_t)n * sizeof(double), 16384 * sizeof(double), reinterpret_cast<void**>(&xw));
    if (rcf != NIB_OK) return rcf;
    NIB_CUDA(cudaMemsetAsync(xw, 0xFF, (size_t)n * sizeof(double), st));
    trsv_wave_kernel<<<nblk, 256, 0, st>>>(L, ldl, b, n, trans, dinv, xw);
    NIB_LAUNCH_CHECK();
    return NIB_OK;
  }
  double* g_trsv_x = nullptr;
  int rcs = stream_scratch(SCRATCH_GP_TRSV, st, (size_t)n * sizeof(double), 16384 * sizeof(double), reinterpret_cast<void**>(&g_trsv_x));
  if (rcs != NIB_OK) return rcs;
  for (int s = 0; s < nblk; ++s) {
    const int blk = trans ? nblk - 1 - s : s;
    const int k0 = blk * NB;
    const int nb = min(NB, n - k0);
    const int work = trans ? ceil_div(k0, 256) : ceil_div(n - (k0 + nb), 8);
    int grid = work < 1 ? 1 : work;
    if (grid > 4 * num_sms()) grid = 4 * num_sms();
    trsv_step_kernel<<<grid, 256, 0, st>>>(L, ldl, b, g_trsv_x, n, k0, nb, trans, dinv);
    NIB_LAUNCH_CHECK();
  }
  NIB_CUDA(cudaMemcpyAsync(b, g_trsv_x, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, st));
  return NIB_OK;
}

// Two-level blocking: 64-wide steps (diagonal solves, one column per thread) inside 256-wide super-blocks.  Inside a
// super-block the rank-64 updates only touch the super-block's own rows; everything outside gets ONE rank-256 update
// per super-block.  The trailing GEMM is read-modify-write on its output: at K = 64 it measured 8-9 TFLOP/s (the tile's
// C round trip dominates), at K = 256 17 TFLOP/s, at large K 25.7 of the 37 TFLOP/s DMMA peak (tools/gp_profile.py).
static constexpr int NBO = 256;
static const int NBC = [] { const char* e = getenv("NIB_GP_NBC"); const int v = e ? atoi(e) : 512; return v >= 64 && v % 64 == 0 ? v : 512; }();   // Cholesky super-block width (measured at n = 8192: 128 -> 21.1, 256 -> 20.7, 512 -> 20.4 ms fit)

static int trsm_impl_v1(const double* L, int n, int ldl, double* B, int nrhs, int ldb, int trans, cudaStream_t st) {
  if (n <= 0 || nrhs <= 0) return NIB_OK;
  if (nrhs == 1 && ldb == 1) return trsv_impl(L, n, ldl, B, trans, nullptr, st);
  const int cb = ceil_div(nrhs, 128);
  DgemmArgs g;
  g.lower_only = 0;
  g.N = nrhs;
  g.ldc = ldb;
  g.sbt = ldb; g.sbj = 1;
  if (!trans) {
    for (int K0 = 0; K0 < n; K0 += NBO) {
      const int W = min(NBO, n - K0);
      for (int k0 = K0; k0 < K0 + W; k0 += NB) {
        const int nb = min(NB, K0 + W - k0);
        trsm_diag_fwd_kernel<<<cb, 128, 0, st>>>(L, ldl, B, ldb, nrhs, k0, nb);
        NIB_LAUNCH_CHECK();
        const int rest = K0 + W - (k0 + nb);   // remaining rows of this super-block
        if (rest > 0) {
          g.A = L + (size_t)(k0 + nb) * ldl + k0; g.sai = ldl; g.sat = 1;   // L[i][k0+t]
          g.B = B + (size_t)k0 * ldb;                                        // X[t][j]
          g.C = B + (size_t)(k0 + nb) * ldb;
          g.M = rest; g.K = nb;
          int rc = dgemm_sub(g, st);
          if (rc != NIB_OK) return rc;
        }
      }
      const int below = n - (K0 + W);
      if (below > 0) {
        g.A = L + (size_t)(K0 + W) * ldl + K0; g.sai = ldl; g.sat = 1;
        g.B = B + (size_t)K0 * ldb;
        g.C = B + (size_t)(K0 + W) * ldb;
        g.M = below; g.K = W;
        int rc = dgemm_sub(g, st);
        if (rc != NIB_OK) return rc;
      }
    }
  } else {
    const int nsb = ceil_div(n, NBO);
    for (int sb = nsb - 1; sb >= 0; --sb) {
      const int K0 = sb * NBO;
      const int W = min(NBO, n - K0);
      const int nblk = ceil_div(W, NB);
      for (int b = nblk - 1; b >= 0; --b) {
        const int k0 = K0 + b * NB;
        const int nb = min(NB, K0 + W - k0);
        trsm_diag_bwd_kernel<<<cb, 128, 0, st>>>(L, ldl, B, ldb, nrhs, k0, nb);
        NIB_LAUNCH_CHECK();
        const int rest = k0 - K0;   // rows of this super-block above the block just solved
        if (rest > 0) {
          g.A = L + (size_t)k0 * ldl + K0; g.sai = 1; g.sat = ldl;          // A(i,t) = L[k0+t][K0+i]
          g.B = B + (size_t)k0 * ldb;
          g.C = B + (size_t)K0 * ldb;
          g.M = rest; g.K = nb;
          int rc = dgemm_sub(g, st);
          if (rc != NIB_OK) return rc;
        }
      }
      if (K0 > 0) {
        g.A = L + (size_t)K0 * ldl; g.sai = 1; g.sat = ldl;                 // A(i,t) = L[K0+t][i]
        g.B = B + (size_t)K0 * ldb;
        g.C = B;
        g.M = K0; g.K = W;
        int rc = dgemm_sub(g, st);
        if (rc != NIB_OK) return rc;
      }
    }
  }
  return NIB_OK;
}


// Recursive TRSM on the block inverses: solve rows [r0, r0+nr) given everything before (forward) / after (backward) has
// been eliminated.  A leaf is one 64-deep product with inv(Lkk); every off-diagonal elimination is a GEMM whose depth is
// half the current range — half of all flops run at depth n/2, a quarter at n/4, ... (the DMMA GEMM measured
// 8 / 17 / 25.7 TFLOP/s at depth 64 / 256 / 4096), against depth 64 and 256 in the two-level blocked version.
static int trsm_rec(const double* L, int ldl, double* B, int nrhs, int ldb, int r0, int nr, int trans, const double* dinv,
                    cudaStream_t st) {
  if (nr <= NB)
    return apply_dinv(dinv + (size_t)(r0 / NB) * NB * NB, B, ldb, r0, nr, 0, nrhs, trans ? 1 : 0, nullptr, st);
  const int h = split64(nr);
  DgemmArgs g;
  g.lower_only = 0;
  g.N = nrhs;
  g.ldc = ldb;
  g.sbt = ldb; g.sbj = 1;
  int rc;
  if (!trans) {
    if ((rc = trsm_rec(L, ldl, B, nrhs, ldb, r0, h, trans, dinv, st)) != NIB_OK) return rc;
    g.A = L + (size_t)(r0 + h) * ldl + r0; g.sai = ldl; g.sat = 1;      // L[r0+h+i][r0+t]
    g.B = B + (size_t)r0 * ldb;
    g.C = B + (size_t)(r0 + h) * ldb;
    g.M = nr - h; g.K = h;
    if ((rc = dgemm_sub(g, st)) != NIB_OK) return rc;
    return trsm_rec(L, ldl, B, nrhs, ldb, r0 + h, nr - h, trans, dinv, st);
  }
  if ((rc = trsm_rec(L, ldl, B, nrhs, ldb, r0 + h, nr - h, trans, dinv, st)) != NIB_OK) return rc;
  g.A = L + (size_t)(r0 + h) * ldl + r0; g.sai = 1; g.sat = ldl;        // A(i,t) = L[r0+h+t][r0+i]
  g.B = B + (size_t)(r0 + h) * ldb;
  g.C = B + (size_t)r0 * ldb;
  g.M = h; g.K = nr - h;
  if ((rc = dgemm_sub(g, st)) != NIB_OK) return rc;
  return trsm_rec(L, ldl, B, nrhs, ldb, r0, h, trans, dinv, st);
}

static bool gp_v1() {
  static const bool v = getenv("NIB_GP_V1") != nullptr;   // the two-level blocked solves of the first version (A/B timing)
  return v;
}

static int trsm_impl(const double* L, int n, int ldl, double* B, int nrhs, int ldb, int trans, cudaStream_t st) {
  if (n <= 0 || nrhs <= 0) return NIB_OK;
  if (gp_v1()) return trsm_impl_v1(L, n, ldl, B, nrhs, ldb, trans, st);
  double* dinv = nullptr;
  int rc = get_dinv(n, st, &dinv);
  if (rc != NIB_OK) return rc;
  if ((rc = trtri_attrs()) != NIB_OK) return rc;
  trtri64_batched_kernel<<<ceil_div(n, NB), 256, TRTRI_SMEM, st>>>(L, ldl, n, dinv);
  NIB_LAUNCH_CHECK();
  if (nrhs == 1 && ldb == 1) return trsv_impl(L, n, ldl, B, trans, dinv, st);
  return trsm_rec(L, ldl, B, nrhs, ldb, 0, n, trans, dinv, st);
}


// Recursive Cholesky: factor the leading half, solve the off-diagonal block against it (recursively: 64-wide leaves are
// one product with inv(Lkk)^T, the rest is GEMM), subtract its Gram from the trailing half, recurse.  Same flops as the
// right-looking sweep, but the symmetric updates run at depth w/2 instead of 64 / 256.
static int rtrsm_rec(double* Kx, int ld, int c0, int w, int r0, int nr, const double* dinv, const int* info, cudaStream_t st) {
  if (w <= NB) return apply_dinv(dinv + (size_t)(c0 / NB) * NB * NB, Kx, ld, c0, w, r0, nr, 2, info, st);
  const int wa = split64(w);
  int rc;
  if ((rc = rtrsm_rec(Kx, ld, c0, wa, r0, nr, dinv, info, st)) != NIB_OK) return rc;
  DgemmArgs g;
  g.A = Kx + (size_t)r0 * ld + c0; g.sai = ld; g.sat = 1;                  // X1[i][t]
  g.B = Kx + (size_t)(c0 + wa) * ld + c0; g.sbt = 1; g.sbj = ld;           // B(t,j) = L[c0+wa+j][c0+t]
  g.C = Kx + (size_t)r0 * ld + c0 + wa; g.ldc = ld;
  g.M = nr; g.N = w - wa; g.K = wa; g.lower_only = 0;
  if ((rc = dgemm_sub(g, st)) != NIB_OK) return rc;
  return rtrsm_rec(Kx, ld, c0 + wa, w - wa, r0, nr, dinv, info, st);
}

static int chol_rec(double* Kx, int ld, int k0, int w, double* dinv, int* info, cudaStream_t st) {
  if (w <= NB) {
    potrf_diag_kernel<<<1, 256, TRTRI_SMEM, st>>>(Kx, ld, k0, w, info, dinv + (size_t)(k0 / NB) * NB * NB);
    NIB_LAUNCH_CHECK();
    return NIB_OK;
  }
  const int wa = split64(w), wb = w - wa;
  int rc;
  if ((rc = chol_rec(Kx, ld, k0, wa, dinv, info, st)) != NIB_OK) return rc;
  if ((rc = rtrsm_rec(Kx, ld, k0, wa, k0 + wa, wb, dinv, info, st)) != NIB_OK) return rc;
  DgemmArgs g;
  const double* X = Kx + (size_t)(k0 + wa) * ld + k0;
  g.A = X; g.sai = ld; g.sat = 1;
  g.B = X; g.sbt = 1; g.sbj = ld;
  g.C = Kx + (size_t)(k0 + wa) * ld + (k0 + wa); g.ldc = ld;
  g.M = wb; g.N = wb; g.K = wa; g.lower_only = 1;
  if ((rc = dgemm_sub(g, st)) != NIB_OK) return rc;
  return chol_rec(Kx, ld, k0 + wa, wb, dinv, info, st);
}

// Right-looking Cholesky with one step of lookahead.  The diagonal-block factorisation (+ inverse) is a one-block kernel
// of ~44 us whose 64 pivots form an unavoidable dependent chain; 128 of them were 5.7 of the 16.4 ms of an n = 8192
// factorisation.  Each update (rank 64 inside a super-block, rank NBC behind it) is therefore split in three: the next
// diagonal block first, then — while a second stream already factors that block — the column block below it and the
// rest.  The main stream only waits for the factorisation when it needs the inverse for the next panel product.
static cudaStream_t g_chol_side = nullptr;
static cudaEvent_t g_chol_ev_diag = nullptr, g_chol_ev_potrf = nullptr;

static int syrk_part(double* Kx, int ld, int r0, int M, int cc0, int N, int c0, int Kd, int lower_only, cudaStream_t st) {
  if (M <= 0 || N <= 0 || Kd <= 0) return NIB_OK;
  DgemmArgs g;
  g.A = Kx + (size_t)r0 * ld + c0; g.sai = ld; g.sat = 1;        // X[r0 + i][c0 + t]
  g.B = Kx + (size_t)cc0 * ld + c0; g.sbt = 1; g.sbj = ld;       // B(t, j) = X[cc0 + j][c0 + t]
  g.C = Kx + (size_t)r0 * ld + cc0; g.ldc = ld;
  g.M = M; g.N = N; g.K = Kd; g.lower_only = lower_only;
  return dgemm_sub(g, st);
}

static int chol_lookahead(double* Kx, int n, int ld, int* info, double* g_dinv, cudaStream_t st) {
  if (!g_chol_side) {
    NIB_CUDA(cudaStreamCreateWithFlags(&g_chol_side, cudaStreamNonBlocking));
    NIB_CUDA(cudaEventCreateWithFlags(&g_chol_ev_diag, cudaEventDisableTiming));
    NIB_CUDA(cudaEventCreateWithFlags(&g_chol_ev_potrf, cudaEventDisableTiming));
  }
  cudaStream_t s2 = g_chol_side;
  int rc;
  auto potrf_side = [&](int k0, int nb) -> int {
    // everything the main stream has queued so far (the update of this diagonal block) precedes the factorisation
    NIB_CUDA(cudaEventRecord(g_chol_ev_diag, st));
    NIB_CUDA(cudaStreamWaitEvent(s2, g_chol_ev_diag, 0));
    potrf_diag_kernel<<<1, 256, TRTRI_SMEM, s2>>>(Kx, ld, k0, nb, info, g_dinv + (size_t)(k0 / NB) * NB * NB);
    NIB_LAUNCH_CHECK();
    NIB_CUDA(cudaEventRecord(g_chol_ev_potrf, s2));
    return NIB_OK;
  };
  if ((rc = potrf_side(0, min(NB, n))) != NIB_OK) return rc;
  for (int K0 = 0; K0 < n; K0 += NBC) {
    const int W = min(NBC, n - K0);
    for (int k0 = K0; k0 < K0 + W; k0 += NB) {
      const int nb = min(NB, K0 + W - k0);
      NIB_CUDA(cudaStreamWaitEvent(st, g_chol_ev_potrf, 0));      // block (k0, k0) is factored and inverted
      const int t0 = k0 + nb, below = n - t0;
      if (below <= 0) continue;
      if ((rc = apply_dinv(g_dinv + (size_t)(k0 / NB) * NB * NB, Kx, ld, k0, nb, t0, below, 2, info, st)) != NIB_OK) return rc;
      const bool in_block = t0 < K0 + W;
      const int c0 = in_block ? k0 : K0, Kd = in_block ? nb : W;   // the panel whose outer product is subtracted
      const int cend = in_block ? K0 + W : n;                      // ... from the columns [t0, cend)
      const int nbn = min(NB, (in_block ? K0 + W : n) - t0);       // the next diagonal block
      if ((rc = syrk_part(Kx, ld, t0, nbn, t0, nbn, c0, Kd, 1, st)) != NIB_OK) return rc;
      if ((rc = potrf_side(t0, nbn)) != NIB_OK) return rc;
      if ((rc = syrk_part(Kx, ld, t0 + nbn, n - (t0 + nbn), t0, nbn, c0, Kd, 0, st)) != NIB_OK) return rc;
      if ((rc = syrk_part(Kx, ld, t0 + nbn, n - (t0 + nbn), t0 + nbn, cend - (t0 + nbn), c0, Kd, 1, st)) != NIB_OK) return rc;
    }
  }
  NIB_CUDA(cudaStreamWaitEvent(st, g_chol_ev_potrf, 0));
  return NIB_OK;
}

// ---- posterior pieces ------------------------------------------------------------------------
__global__ void transpose_kernel(const double* __restrict__ in, int rows, int cols, int ldi, double* __restrict__ out,
                                 int ldo) {
  __shared__ double tile[32][33];
  int x = blockIdx.x * 32 + threadIdx.x, y0 = blockIdx.y * 32;
  for (int yy = threadIdx.y; yy < 32; yy += blockDim.y) {
    int y = y0 + yy;
    if (x < cols && y < rows) tile[yy][threadIdx.x] = in[(size_t)y * ldi + x];
  }
  __syncthreads();
  int ox = blockIdx.y * 32 + threadIdx.x, oy0 = blockIdx.x * 32;
  for (int yy = threadIdx.y; yy < 32; yy += blockDim.y) {
    int oy = oy0 + yy;
    if (ox < rows && oy < cols) out[(size_t)oy * ldo + ox] = tile[threadIdx.x][yy];
  }
}

__global__ void __launch_bounds__(256)
gemv_mean_kernel(const double* __restrict__ Ks, int m, int n, int ldks, const double* __restrict__ alpha, double y_mean,
                 double y_std, double* __restrict__ mu) {
  const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);   // one warp per query
  const int lane = threadIdx.x & 31;
  if (q >= m) return;
  double acc = 0.0;
  for (int i = lane; i < n; i += 32) acc = fma(Ks[(size_t)q * ldks + i], alpha[i], acc);
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) mu[q] = y_std * acc + y_mean;
}

// ---- column reductions over V [n][m] (row-major): one pass over HBM, rows split into slices so the grid fills the GPU --
// mode 0: partial[s][j] = sum_t x[t] * V[t][j];  mode 1: partial[s][j] = sum_t V[t][j]^2   (t in slice s)
static constexpr int CR_ROWS = 64;   // rows per slice
__global__ void __launch_bounds__(256)
colreduce_partial_kernel(const double* __restrict__ V, long long ldv, int n, int m, const double* __restrict__ x, int mode,
                         double* __restrict__ partial) {
  const int j = blockIdx.x * 256 + threadIdx.x;
  const int t0 = blockIdx.y * CR_ROWS, t1 = min(n, t0 + CR_ROWS);
  if (j >= m) return;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  int t = t0;
  for (; t + 3 < t1; t += 4) {
    const double v0 = V[(size_t)t * ldv + j], v1 = V[(size_t)(t + 1) * ldv + j];
    const double v2 = V[(size_t)(t + 2) * ldv + j], v3 = V[(size_t)(t + 3) * ldv + j];
    if (mode == 0) { a0 = fma(x[t], v0, a0); a1 = fma(x[t + 1], v1, a1); a2 = fma(x[t + 2], v2, a2); a3 = fma(x[t + 3], v3, a3); }
    else { a0 = fma(v0, v0, a0); a1 = fma(v1, v1, a1); a2 = fma(v2, v2, a2); a3 = fma(v3, v3, a3); }
  }
  for (; t < t1; ++t) {
    const double v0 = V[(size_t)t * ldv + j];
    a0 = (mode == 0) ? fma(x[t], v0, a0) : fma(v0, v0, a0);
  }
  partial[(size_t)blockIdx.y * m + j] = (a0 + a1) + (a2 + a3);
}
// out[j] = sum_s partial[s][j] (fixed order: deterministic); var/sd epilogue of _gpr.py:485-496 when var_mode
__global__ void __launch_bounds__(256)
colreduce_final_kernel(const double* __restrict__ partial, int slices, int m, double* __restrict__ out, int var_mode,
                       double prior_var, double y_std, double* __restrict__ sd) {
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= m) return;
  double acc = 0.0;
  for (int sidx = 0; sidx < slices; ++sidx) acc += partial[(size_t)sidx * m + j];
  if (var_mode) {
    double r = prior_var - acc;
    if (r < 0.0) r = 0.0;
    r = r * y_std * y_std;
    if (out) out[j] = r;
    if (sd) sd[j] = sqrt(r);
  } else {
    out[j] = acc;
  }
}
static int colreduce(const double* V, long long ldv, int n, int m, const double* x, int mode, double* out, int var_mode,
                     double prior_var, double y_std, double* sd, cudaStream_t st) {
  const int slices = ceil_div(n, CR_ROWS);
  const size_t need = (size_t)slices * m;
  double* g_cr = nullptr;
  int rcs = stream_scratch(SCRATCH_GP_COLREDUCE, st, need * sizeof(double), ((size_t)1 << 21) * sizeof(double), reinterpret_cast<void**>(&g_cr));
  if (rcs != NIB_OK) return rcs;
  dim3 grid(ceil_div(m, 256), slices);
  colreduce_partial_kernel<<<grid, 256, 0, st>>>(V, ldv, n, m, x, mode, g_cr);
  NIB_LAUNCH_CHECK();
  colreduce_final_kernel<<<ceil_div(m, 256), 256, 0, st>>>(g_cr, slices, m, out, var_mode, prior_var, y_std, sd);
  NIB_LAUNCH_CHECK();
  return NIB_OK;
}

// rank-one extension of the posterior workspace (ActiveMaskGP.append): v = (ks - dot) / d becomes row n of V, ssq += v^2
__global__ void __launch_bounds__(256)
append_row_kernel(const double* __restrict__ ks, const double* __restrict__ dot, double d, double* __restrict__ vrow,
                  double* __restrict__ ssq, int m) {
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= m) return;
  const double v = (ks[j] - dot[j]) / d;
  vrow[j] = v;
  ssq[j] = fma(v, v, ssq[j]);
}

// ---- LML -------------------------------------------------------------------------------------
__global__ void lml_kernel(const double* __restrict__ L, int n, int ldl, const double* __restrict__ y,
                           const double* __restrict__ alpha, double* __restrict__ out) {
  __shared__ double s1[32], s2[32];
  double a = 0.0, b = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    a = fma(y[i], alpha[i], a);
    b += log(L[(size_t)i * ldl + i]);
  }
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  if ((threadIdx.x & 31) == 0) { s1[threadIdx.x >> 5] = a; s2[threadIdx.x >> 5] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ta = 0, tb = 0;
    for (int i = 0; i < (blockDim.x >> 5); ++i) { ta += s1[i]; tb += s2[i]; }
    out[0] = -0.5 * ta - tb - 0.5 * (double)n * 1.8378770664093453;  // log(2*pi)
  }
}

__global__ void __launch_bounds__(256)
lml_grad_kernel(const double* __restrict__ K0, const double* __restrict__ Kinv, const double* __restrict__ alpha,
                const uint64_t* __restrict__ Z, int words, int n, int ld, double* __restrict__ partial) {
  // partial[block] = sum over this block's rows of (alpha_i alpha_j - Kinv_ij) * K0_ij * hamming_ij
  const int i = blockIdx.x;
  double acc = 0.0;
  const double ai = alpha[i];
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    int h = 0;
    for (int w = 0; w < words; ++w) h += __popcll(Z[(size_t)i * words + w] ^ Z[(size_t)j * words + w]);
    acc = fma((ai * alpha[j] - Kinv[(size_t)i * ld + j]) * K0[(size_t)i * ld + j], (double)h, acc);
  }
  __shared__ double s[32];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int k = 0; k < (blockDim.x >> 5); ++k) t += s[k];
    partial[i] = t;
  }
}
__global__ void __launch_bounds__(256)
lml_grad_rbf_kernel(const double* __restrict__ K0, const double* __restrict__ Kinv, const double* __restrict__ alpha,
                    const double* __restrict__ X, int d, int n, int ld, double inv_l, double* __restrict__ partial) {
  const int i = blockIdx.x;
  double acc = 0.0;
  const double ai = alpha[i];
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    double s2 = 0.0;
    for (int k = 0; k < d; ++k) {
      const double diff = X[(size_t)i * d + k] * inv_l - X[(size_t)j * d + k] * inv_l;
      s2 += diff * diff;
    }
    acc = fma((ai * alpha[j] - Kinv[(size_t)i * ld + j]) * K0[(size_t)i * ld + j], s2, acc);
  }
  __shared__ double s[32];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int k = 0; k < (blockDim.x >> 5); ++k) t += s[k];
    partial[i] = t;
  }
}
__global__ void sum_kernel(const double* __restrict__ v, int n, double* __restrict__ out) {
  __shared__ double s[32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += v[i];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int k = 0; k < (blockDim.x >> 5); ++k) t += s[k];
    out[0] = t;
  }
}

// ---- Expected improvement ----------------------------------------------------------------------
// shared by ei_kernel and the Kriging-believer selection so that both produce the same bits
__device__ __forceinline__ double ei_value(double mu, double s, double best, double sf) {
  const double d = sf * (mu - best);
  const double Z = d / s;  // sigma == 0 -> inf/NaN, as the reference (np.errstate(divide='ignore'))
  const double Phi = 0.5 * erfc(-Z * 0.70710678118654752440);
  const double phi = exp(-0.5 * Z * Z) * 0.39894228040143267794;
  return d * Phi + s * phi;
}
__global__ void ei_kernel(const double* __restrict__ mu, const double* __restrict__ sigma, int m, double best, double sf,
                          double* __restrict__ ei) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= m) return;
  ei[q] = ei_value(mu[q], sigma[q], best, sf);
}
__global__ void argmax_kernel(const double* __restrict__ v, int m, long long* __restrict__ out) {
  __shared__ double sv[32];
  __shared__ long long si[32];
  double best = -INFINITY;
  long long bi = -1;
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    const double x = v[i];
    if (x == x && (bi < 0 || x > best)) { best = x; bi = i; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, best, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (oi >= 0 && (bi < 0 || ov > best || (ov == best && oi < bi))) { best = ov; bi = oi; }
  }
  if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = best; si[threadIdx.x >> 5] = bi; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < (blockDim.x >> 5); ++k) {
      if (si[k] >= 0 && (bi < 0 || sv[k] > best || (sv[k] == best && si[k] < bi))) { best = sv[k]; bi = si[k]; }
    }
    out[0] = bi;
  }
}

// ---- Kriging-believer batch selection (nib_gp_kb_select) ---------------------------------------------------------------
// Greedy q-pick acquisition on the resident rank-one state of ActiveMaskGP.  The fantasy observation at a pick equals its
// posterior mean, which leaves every other mean unchanged, so a pick only shrinks variances: one new row of V per pick.
// Per pick two launches, with the pick index passed through device memory so the host never waits inside a batch:
//   kb_colreduce_kernel  dot[x] = sum_t V[t][x] * l_t over row slices, l = V[:, j] (= the new row of L, written too)
//   kb_finalize_kernel   fixed-order slice sum, V[n+k][x] = (k(x, z_j) - dot[x]) / d, ssq update, sigma, EI, block
//                        arg-max; the last block to finish (atomic counter, no spinning) publishes the next pick.
// No floating-point atomics: picks and V are bitwise reproducible.
static constexpr int KB_THREADS = 256, KB_COLS = 2, KB_TILE = KB_THREADS * KB_COLS, KB_UNROLL = 8;

struct KbCtrl {
  long long pick;       // index of the pick whose row is being added; -1 once selection has stopped
  double d;             // its new diagonal entry of L
  double best;          // incumbent after the picks so far (Kriging believer: the picked means count as observed)
  unsigned int done;    // finalize blocks finished (reset by the last one)
};

struct KbArgs {
  double* L; int ldl; double* V; long long ldv; double* ssq; unsigned char* alive;
  const uint64_t* cand; int m; int words; uint64_t* X; int n;
  const double* mu; double var_scale; double alpha; double inv_l2_half; double sf; double best0;
  long long* picks; double* ei; int* status;
  KbCtrl* ctrl; const double* partial; double* bval; long long* bidx;
};

// (v, i) beats (bv, bi): larger non-NaN value, lower index on ties (argmax_kernel's rule); a total order, so any
// reduction tree gives the same winner
__device__ __forceinline__ void kb_better(double& bv, long long& bi, double v, long long i) {
  if (i >= 0 && (bi < 0 || v > bv || (v == bv && i < bi))) { bv = v; bi = i; }
}
__device__ __forceinline__ void kb_block_argmax(double& bv, long long& bi, double* sv, long long* si) {
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
    kb_better(bv, bi, ov, oi);
  }
  if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = bv; si[threadIdx.x >> 5] = bi; }
  __syncthreads();
  if (threadIdx.x == 0)
    for (int w = 1; w < KB_THREADS / 32; ++w) kb_better(bv, bi, sv[w], si[w]);
}

// partial[s][x] = sum_{t in slice s} V[t][x] * V[t][j]   (t < nk).  Each thread owns KB_COLS columns 256 apart and keeps
// KB_UNROLL * KB_COLS independent loads in flight; l is staged through shared memory 256 rows at a time.
__global__ void __launch_bounds__(KB_THREADS)
kb_colreduce_kernel(const double* __restrict__ V, long long ldv, int nk, int m, int rows, double* __restrict__ Lrow,
                    const KbCtrl* __restrict__ ctrl, double* __restrict__ partial) {
  const long long j = ctrl->pick;
  if (j < 0) return;
  __shared__ double ls[KB_THREADS];
  const int t0 = blockIdx.y * rows, t1 = min(nk, t0 + rows);
  const int x0 = blockIdx.x * KB_TILE + threadIdx.x;
  double acc[KB_COLS];
#pragma unroll
  for (int c = 0; c < KB_COLS; ++c) acc[c] = 0.0;
  for (int c0 = t0; c0 < t1; c0 += KB_THREADS) {
    const int cn = min(KB_THREADS, t1 - c0);
    __syncthreads();
    if (threadIdx.x < cn) {
      const double l = V[(size_t)(c0 + threadIdx.x) * ldv + j];
      ls[threadIdx.x] = l;
      if (blockIdx.x == 0) Lrow[c0 + threadIdx.x] = l;
    }
    __syncthreads();
    for (int u0 = 0; u0 < cn; u0 += KB_UNROLL) {
      double v[KB_UNROLL][KB_COLS];
#pragma unroll
      for (int u = 0; u < KB_UNROLL; ++u)
#pragma unroll
        for (int c = 0; c < KB_COLS; ++c) {
          const int x = x0 + c * KB_THREADS;
          v[u][c] = (u0 + u < cn && x < m) ? __ldcs(V + (size_t)(c0 + u0 + u) * ldv + x) : 0.0;
        }
#pragma unroll
      for (int u = 0; u < KB_UNROLL; ++u) {
        const double l = u0 + u < cn ? ls[u0 + u] : 0.0;
#pragma unroll
        for (int c = 0; c < KB_COLS; ++c) acc[c] = fma(v[u][c], l, acc[c]);
      }
    }
  }
#pragma unroll
  for (int c = 0; c < KB_COLS; ++c) {
    const int x = x0 + c * KB_THREADS;
    if (x < m) partial[(size_t)blockIdx.y * m + x] = acc[c];
  }
}

// kpub: index of the pick this launch publishes (q: none).  add_row: first append row n + kpub - 1 for the current pick
// from the `slices` partial sums.  Dynamic shared memory: the (64 * words + 1)-entry Hamming LUT of gram_binary_kernel.
__global__ void __launch_bounds__(KB_THREADS)
kb_finalize_kernel(KbArgs a, int kpub, int q, int add_row, int slices) {
  extern __shared__ double lut[];
  __shared__ double sv[KB_THREADS / 32];
  __shared__ long long si[KB_THREADS / 32];
  __shared__ int last;
  KbCtrl* c = a.ctrl;
  const long long jc = add_row ? c->pick : 0;
  if (jc < 0) return;
  const int x = blockIdx.x * KB_THREADS + threadIdx.x;
  double s2 = x < a.m ? a.ssq[x] : 0.0;
  if (add_row) {
    const int nl = 64 * a.words + 1;
    for (int h = threadIdx.x; h < nl; h += KB_THREADS) lut[h] = exp(-(double)h * a.inv_l2_half);
    __syncthreads();
    if (x < a.m) {
      double dot = 0.0;
      for (int s = 0; s < slices; ++s) dot += a.partial[(size_t)s * a.m + x];
      int h = 0;
      for (int w = 0; w < a.words; ++w) h += __popcll(a.cand[(size_t)x * a.words + w] ^ a.cand[(size_t)jc * a.words + w]);
      const double v = (lut[h] - dot) / c->d;
      a.V[(size_t)(a.n + kpub - 1) * a.ldv + x] = v;
      s2 = fma(v, v, s2);
      a.ssq[x] = s2;
      __threadfence();   // the last block reads ssq[j] of the new pick
    }
  }
  if (kpub >= q) return;
  const double best = add_row ? c->best : a.best0;
  double bv = NAN;
  long long bi = -1;
  if (x < a.m && a.alive[x]) {
    double r = 1.0 - s2;   // ActiveMaskGP.posterior(): var = clamp(1 - ssq, 0) * ystd^2, sd = sqrt(var)
    if (r < 0.0) r = 0.0;
    const double e = ei_value(a.mu[x], sqrt(r * a.var_scale), best, a.sf);
    if (e == e) { bv = e; bi = x; }
  }
  kb_block_argmax(bv, bi, sv, si);
  if (threadIdx.x == 0) {
    a.bval[blockIdx.x] = bv;
    a.bidx[blockIdx.x] = bi;
    __threadfence();
    last = atomicAdd(&c->done, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  bv = NAN;
  bi = -1;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += KB_THREADS) kb_better(bv, bi, __ldcg(a.bval + b), __ldcg(a.bidx + b));
  __syncthreads();
  kb_block_argmax(bv, bi, sv, si);
  if (threadIdx.x != 0) return;
  c->done = 0;
  if (bi < 0) { c->pick = -1; return; }                       // no candidate with a defined EI left
  const double d2 = 1.0 + a.alpha - __ldcg(a.ssq + bi);
  if (!(d2 > 0.0)) { *a.status = kpub + 1; c->pick = -1; return; }
  const double d = sqrt(d2);
  const int row = a.n + kpub;
  a.picks[kpub] = bi;
  a.ei[kpub] = bv;
  c->pick = bi;
  c->d = d;
  const double mj = a.mu[bi];
  c->best = a.sf > 0.0 ? (mj > best ? mj : best) : (mj < best ? mj : best);
  a.alive[bi] = 0;
  a.L[(size_t)row * a.ldl + row] = d;
  for (int w = 0; w < a.words; ++w) a.X[(size_t)row * a.words + w] = a.cand[(size_t)bi * a.words + w];
}

// rows per colreduce slice for nk rows: enough slices that the grid covers every SM about four times, at least 64 rows each
static void kb_slices(int nk, int m, int* slices, int* rows) {
  const int tiles = ceil_div(m, KB_TILE);
  const int s = max(1, min(ceil_div(nk, 64), ceil_div(4 * num_sms(), tiles)));
  *rows = ceil_div(nk, s);
  *slices = ceil_div(nk, *rows);
}

// small device scratch for scalar reductions (per stream, common.cuh)
static int get_scratch(size_t doubles, cudaStream_t st, double** out) {
  return stream_scratch(SCRATCH_GP_SCALARS, st, doubles * sizeof(double), 16384 * sizeof(double), reinterpret_cast<void**>(out));
}

}  // namespace nib

using namespace nib;

extern "C" {

int nib_gp_gram_binary(const uint64_t* d_Za, int na, const uint64_t* d_Zb, int nb, int words, double length_scale,
                       double jitter, double* d_K, int ldk, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_Za && d_Zb && d_K, "nib_gp_gram_binary: null pointer");
  NIB_REQUIRE(na > 0 && nb > 0 && words > 0 && words <= 64 && ldk >= nb, "nib_gp_gram_binary: bad shape");
  NIB_REQUIRE(length_scale > 0.0, "nib_gp_gram_binary: length_scale must be > 0");
  dim3 grid(ceil_div(nb, 32), ceil_div(na, 32)), block(32, 8);
  const size_t smem = sizeof(double) * (64 * words + 1);
  gram_binary_kernel<<<grid, block, smem, (cudaStream_t)stream>>>(d_Za, na, d_Zb, nb, words,
                                                                  0.5 / (length_scale * length_scale), jitter,
                                                                  d_Za == d_Zb ? 1 : 0, d_K, ldk);
  NIB_LAUNCH_CHECK();
  return NIB_OK;
}

int nib_gp_gram_rbf(const double* d_Xa, int na, const double* d_Xb, int nb, int d, double length_scale, double jitter,
                    int same, double* d_K, int ldk, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_Xa && d_Xb && d_K, "nib_gp_gram_rbf: null pointer");
  NIB_REQUIRE(na > 0 && nb > 0 && d > 0 && ldk >= nb && length_scale > 0.0, "nib_gp_gram_rbf: bad shape");
  dim3 grid(ceil_div(nb, 32), ceil_div(na, 32)), block(32, 8);
  gram_rbf_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(d_Xa, na, d_Xb, nb, d, 1.0 / length_scale, jitter, same,
                                                            d_K, ldk);
  NIB_LAUNCH_CHECK();
  return NIB_OK;
}

int nib_gp_cholesky(double* d_K, int n, int ldk, int* d_info, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_K && d_info && n > 0 && ldk >= n, "nib_gp_cholesky: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  NIB_CUDA(cudaMemsetAsync(d_info, 0, sizeof(int), st));
  if (!gp_v1()) {
    double* g_dinv = nullptr;
    int rc = get_dinv(n, st, &g_dinv);
    if (rc != NIB_OK) return rc;
    if ((rc = trtri_attrs()) != NIB_OK) return rc;
    static const bool rec = getenv("NIB_GP_CHOL_REC") != nullptr;   // fully recursive variant: measured slower (its
    if (rec) return chol_rec(d_K, ldk, 0, n, g_dinv, d_info, st);   // small symmetric updates leave most SMs idle)
    // measured at n = 8192: 19.8 ms fit with the lookahead, 19.1 without — the update GEMMs hold every SM's registers
    // (two 256-thread blocks of 128 registers), so the one-block factorisation on the side stream only gets an SM when
    // a GEMM wave drains, and three GEMM launches per step instead of one cost more than that wins.  Opt-in.
    static const bool la = getenv("NIB_GP_LOOKAHEAD") != nullptr;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    if (la && cap == cudaStreamCaptureStatusNone) return chol_lookahead(d_K, n, ldk, d_info, g_dinv, st);
    // Right-looking, two-level: 64-wide steps inside NBC-wide super-blocks.  Each step factors the diagonal block AND
    // inverts it (potrf_diag_kernel), turns the panel solve for every row below into one 64-deep product with that
    // inverse (apply_dinv_kernel) and updates the rest of the super-block's columns (rank 64); everything to the right of
    // the super-block gets one rank-NBC update.
    for (int K0 = 0; K0 < n; K0 += NBC) {
      const int W = min(NBC, n - K0);
      for (int k0 = K0; k0 < K0 + W; k0 += NB) {
        const int nb = min(NB, K0 + W - k0);
        double* dk = g_dinv + (size_t)(k0 / NB) * NB * NB;
        potrf_diag_kernel<<<1, 256, TRTRI_SMEM, st>>>(d_K, ldk, k0, nb, d_info, dk);
        NIB_LAUNCH_CHECK();
        const int below = n - (k0 + nb);
        if (below > 0 && (rc = apply_dinv(dk, d_K, ldk, k0, nb, k0 + nb, below, 2, d_info, st)) != NIB_OK) return rc;
        const int cols = K0 + W - (k0 + nb);
        if (below > 0 && cols > 0) {
          DgemmArgs g;
          const double* X = d_K + (size_t)(k0 + nb) * ldk + k0;
          g.A = X; g.sai = ldk; g.sat = 1;
          g.B = X; g.sbt = 1; g.sbj = ldk;
          g.C = d_K + (size_t)(k0 + nb) * ldk + (k0 + nb); g.ldc = ldk;
          g.M = below; g.N = cols; g.K = nb; g.lower_only = 1;
          if ((rc = dgemm_sub(g, st)) != NIB_OK) return rc;
        }
      }
      const int below = n - (K0 + W);
      if (below > 0) {
        DgemmArgs g;
        const double* X = d_K + (size_t)(K0 + W) * ldk + K0;
        g.A = X; g.sai = ldk; g.sat = 1;
        g.B = X; g.sbt = 1; g.sbj = ldk;
        g.C = d_K + (size_t)(K0 + W) * ldk + (K0 + W); g.ldc = ldk;
        g.M = below; g.N = below; g.K = W; g.lower_only = 1;
        if ((rc = dgemm_sub(g, st)) != NIB_OK) return rc;
      }
    }
    return NIB_OK;
  }
  // right-looking, two-level: 64-wide panels inside 256-wide super-blocks (see trsm_impl for why)
  for (int K0 = 0; K0 < n; K0 += NBO) {
    const int W = min(NBO, n - K0);
    for (int k0 = K0; k0 < K0 + W; k0 += NB) {
      const int nb = min(NB, K0 + W - k0);
      potrf_diag_kernel<<<1, 256, 0, st>>>(d_K, ldk, k0, nb, d_info, nullptr);
      NIB_LAUNCH_CHECK();
      const int below = n - (k0 + nb);
      if (below > 0) {
        trsm_panel_kernel<<<ceil_div(below, 128), 128, 0, st>>>(d_K, ldk, k0, nb, n, d_info);
        NIB_LAUNCH_CHECK();
      }
      const int cols = K0 + W - (k0 + nb);   // columns of this super-block still to be factored
      if (below > 0 && cols > 0) {
        DgemmArgs g;
        const double* X = d_K + (size_t)(k0 + nb) * ldk + k0;
        g.A = X; g.sai = ldk; g.sat = 1;      // X[i][t]
        g.B = X; g.sbt = 1; g.sbj = ldk;      // B(t,j) = X[j][t]
        g.C = d_K + (size_t)(k0 + nb) * ldk + (k0 + nb); g.ldc = ldk;
        g.M = below; g.N = cols; g.K = nb; g.lower_only = 1;
        int rc = dgemm_sub(g, st);
        if (rc != NIB_OK) return rc;
      }
    }
    const int below = n - (K0 + W);
    if (below > 0) {
      DgemmArgs g;
      const double* X = d_K + (size_t)(K0 + W) * ldk + K0;
      g.A = X; g.sai = ldk; g.sat = 1;
      g.B = X; g.sbt = 1; g.sbj = ldk;
      g.C = d_K + (size_t)(K0 + W) * ldk + (K0 + W); g.ldc = ldk;
      g.M = below; g.N = below; g.K = W; g.lower_only = 1;
      int rc = dgemm_sub(g, st);
      if (rc != NIB_OK) return rc;
    }
  }
  return NIB_OK;
}

// Diagnostic hook (tools/gp_profile.py): C[M,N] -= A[M,K] * B[K,N], all row-major, through the same fp64 tensor-core
// GEMM the Cholesky / TRSM trailing updates use.
int nib_gp_dgemm_sub(const double* d_A, const double* d_B, double* d_C, int M, int N, int K, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_A && d_B && d_C && M > 0 && N > 0 && K > 0, "nib_gp_dgemm_sub: bad arguments");
  DgemmArgs g;
  g.A = d_A; g.sai = K; g.sat = 1;
  g.B = d_B; g.sbt = N; g.sbj = 1;
  g.C = d_C; g.ldc = N;
  g.M = M; g.N = N; g.K = K; g.lower_only = 0;
  return dgemm_sub(g, (cudaStream_t)stream);
}

int nib_gp_trsm(const double* d_L, int n, int ldl, double* d_B, int nrhs, int ldb, int trans, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_L && d_B && n > 0 && nrhs > 0 && ldl >= n && ldb >= nrhs, "nib_gp_trsm: bad arguments");
  return trsm_impl(d_L, n, ldl, d_B, nrhs, ldb, trans, (cudaStream_t)stream);
}

int nib_gp_posterior(const double* d_L, int n, int ldl, const double* d_alpha, const double* d_Ks, int m, int ldks,
                     double y_mean, double y_std, double prior_var, double* d_work, double* d_mu, double* d_var,
                     double* d_std, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_L && d_alpha && d_Ks && n > 0 && m > 0 && ldl >= n && ldks >= n, "nib_gp_posterior: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (d_mu) {
    gemv_mean_kernel<<<ceil_div(m, 8), 256, 0, st>>>(d_Ks, m, n, ldks, d_alpha, y_mean, y_std, d_mu);
    NIB_LAUNCH_CHECK();
  }
  if (d_var || d_std) {
    NIB_REQUIRE(d_work != nullptr, "nib_gp_posterior: variance needs d_work (m*n doubles)");
    dim3 grid(ceil_div(n, 32), ceil_div(m, 32)), block(32, 8);
    transpose_kernel<<<grid, block, 0, st>>>(d_Ks, m, n, ldks, d_work, m);  // work = Ks^T  [n][m]
    NIB_LAUNCH_CHECK();
    int rc = trsm_impl(d_L, n, ldl, d_work, m, m, 0, st);
    if (rc != NIB_OK) return rc;
    if ((rc = colreduce(d_work, m, n, m, nullptr, 1, d_var, 1, prior_var, y_std, d_std, st)) != NIB_OK) return rc;
  }
  return NIB_OK;
}

int nib_gp_gemv_t(const double* d_V, int n, int m, int ldv, const double* d_x, double* d_out, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_V && d_x && d_out && n > 0 && m > 0 && ldv >= m, "nib_gp_gemv_t: bad arguments");
  return colreduce(d_V, ldv, n, m, d_x, 0, d_out, 0, 0.0, 1.0, nullptr, (cudaStream_t)stream);
}

int nib_gp_colsumsq(const double* d_V, int n, int m, int ldv, double* d_out, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_V && d_out && n > 0 && m > 0 && ldv >= m, "nib_gp_colsumsq: bad arguments");
  return colreduce(d_V, ldv, n, m, nullptr, 1, d_out, 0, 0.0, 1.0, nullptr, (cudaStream_t)stream);
}

int nib_gp_append_row(const double* d_ks, const double* d_dot, double d, double* d_vrow, double* d_ssq, int m,
                      void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_ks && d_dot && d_vrow && d_ssq && m > 0 && d > 0.0, "nib_gp_append_row: bad arguments");
  append_row_kernel<<<ceil_div(m, 256), 256, 0, (cudaStream_t)stream>>>(d_ks, d_dot, d, d_vrow, d_ssq, m);
  NIB_LAUNCH_CHECK();
  return NIB_OK;
}

int nib_gp_kb_select(double* d_L, int ldl, double* d_V, int ldv, double* d_ssq, unsigned char* d_alive,
                     const uint64_t* d_cand, int m, int words, uint64_t* d_X, int n, int q, const double* d_mu,
                     double y_std, double best, int greater_is_better, double length_scale, double alpha,
                     long long* d_picks, double* d_ei, int* d_status, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_L && d_V && d_ssq && d_alive && d_cand && d_X && d_mu && d_picks && d_ei && d_status,
              "nib_gp_kb_select: null pointer");
  NIB_REQUIRE(n > 0 && q > 0 && m > 0 && words > 0 && words <= 64 && ldl >= n + q && ldv >= m,
              "nib_gp_kb_select: bad shape");
  NIB_REQUIRE(length_scale > 0.0 && alpha >= 0.0 && y_std > 0.0, "nib_gp_kb_select: bad hyper-parameters");
  cudaStream_t st = (cudaStream_t)stream;
  const int nblk = ceil_div(m, KB_THREADS);
  // ceil(nk / ceil(nk / s)) is not monotone in nk (m = 1792 on 148 SMs: 148 slices for nk = 9458 .. 9472, 146 at
  // nk = 9473), so the partials buffer is sized for the largest count any pick of this batch launches
  int max_slices = 0, rows = 0;
  for (int k = 0; k < q; ++k) {
    int slices = 0;
    kb_slices(n + k, m, &slices, &rows);
    max_slices = max(max_slices, slices);
  }
  // scratch: control block | per-block arg-max values | indices | colreduce partial sums [slices][m]
  const size_t head = 64, bytes = head + (size_t)nblk * 16 + (size_t)max_slices * m * sizeof(double);
  unsigned char* scratch = nullptr;
  int rc = stream_scratch(SCRATCH_GP_KB, st, bytes, bytes, reinterpret_cast<void**>(&scratch));
  if (rc != NIB_OK) return rc;
  KbArgs a;
  a.L = d_L; a.ldl = ldl; a.V = d_V; a.ldv = ldv; a.ssq = d_ssq; a.alive = d_alive;
  a.cand = d_cand; a.m = m; a.words = words; a.X = d_X; a.n = n;
  a.mu = d_mu; a.var_scale = y_std * y_std; a.alpha = alpha; a.inv_l2_half = 0.5 / (length_scale * length_scale);
  a.sf = greater_is_better ? 1.0 : -1.0; a.best0 = best;
  a.picks = d_picks; a.ei = d_ei; a.status = d_status;
  a.ctrl = reinterpret_cast<KbCtrl*>(scratch);
  a.bval = reinterpret_cast<double*>(scratch + head);
  a.bidx = reinterpret_cast<long long*>(scratch + head + (size_t)nblk * 8);
  double* partial = reinterpret_cast<double*>(scratch + head + (size_t)nblk * 16);
  a.partial = partial;
  NIB_CUDA(cudaMemsetAsync(scratch, 0, head, st));
  NIB_CUDA(cudaMemsetAsync(d_picks, 0xff, (size_t)q * sizeof(long long), st));   // -1: not picked
  NIB_CUDA(cudaMemsetAsync(d_status, 0, sizeof(int), st));
  const size_t lut = sizeof(double) * (64 * words + 1);
  kb_finalize_kernel<<<nblk, KB_THREADS, 0, st>>>(a, 0, q, 0, 0);   // pick 0 from the current state
  NIB_LAUNCH_CHECK();
  for (int k = 0; k < q; ++k) {
    int slices = 0;
    kb_slices(n + k, m, &slices, &rows);
    dim3 grid(ceil_div(m, KB_TILE), slices);
    kb_colreduce_kernel<<<grid, KB_THREADS, 0, st>>>(d_V, ldv, n + k, m, rows, d_L + (size_t)(n + k) * ldl, a.ctrl,
                                                     partial);
    NIB_LAUNCH_CHECK();
    kb_finalize_kernel<<<nblk, KB_THREADS, lut, st>>>(a, k + 1, q, 1, slices);   // row n + k, then pick k + 1
    NIB_LAUNCH_CHECK();
  }
  return NIB_OK;
}

int nib_gp_lml(const double* d_L, int n, int ldl, const double* d_y, const double* d_alpha, double* h_lml,
               void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_L && d_y && d_alpha && h_lml && n > 0, "nib_gp_lml: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  double* g_scratch = nullptr;
  int rc = get_scratch(16, st, &g_scratch);
  if (rc != NIB_OK) return rc;
  lml_kernel<<<1, 1024, 0, st>>>(d_L, n, ldl, d_y, d_alpha, g_scratch);
  NIB_LAUNCH_CHECK();
  NIB_CUDA(cudaMemcpyAsync(h_lml, g_scratch, sizeof(double), cudaMemcpyDeviceToHost, st));
  NIB_CUDA(cudaStreamSynchronize(st));
  return NIB_OK;
}

int nib_gp_lml_grad(const double* d_K0, const double* d_Kinv, const double* d_alpha, const uint64_t* d_Z, int words,
                    int n, int ld, double length_scale, double* h_grad, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_K0 && d_Kinv && d_alpha && d_Z && h_grad && n > 0 && ld >= n, "nib_gp_lml_grad: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  double* g_scratch = nullptr;
  int rc = get_scratch((size_t)n + 16, st, &g_scratch);
  if (rc != NIB_OK) return rc;
  lml_grad_kernel<<<n, 256, 0, st>>>(d_K0, d_Kinv, d_alpha, d_Z, words, n, ld, g_scratch + 16);
  NIB_LAUNCH_CHECK();
  sum_kernel<<<1, 1024, 0, st>>>(g_scratch + 16, n, g_scratch);
  NIB_LAUNCH_CHECK();
  double t = 0.0;
  NIB_CUDA(cudaMemcpyAsync(&t, g_scratch, sizeof(double), cudaMemcpyDeviceToHost, st));
  NIB_CUDA(cudaStreamSynchronize(st));
  // dK/dtheta = K0 .* D2 / l^2 ;  grad = 0.5 * sum((alpha alpha^T - K^-1) .* dK/dtheta)
  *h_grad = 0.5 * t / (length_scale * length_scale);
  return NIB_OK;
}

int nib_gp_lml_grad_rbf(const double* d_K0, const double* d_Kinv, const double* d_alpha, const double* d_X, int d,
                        int n, int ld, double length_scale, double* h_grad, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_K0 && d_Kinv && d_alpha && d_X && h_grad && n > 0 && d > 0 && ld >= n, "nib_gp_lml_grad_rbf: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  double* g_scratch = nullptr;
  int rc = get_scratch((size_t)n + 16, st, &g_scratch);
  if (rc != NIB_OK) return rc;
  lml_grad_rbf_kernel<<<n, 256, 0, st>>>(d_K0, d_Kinv, d_alpha, d_X, d, n, ld, 1.0 / length_scale, g_scratch + 16);
  NIB_LAUNCH_CHECK();
  sum_kernel<<<1, 1024, 0, st>>>(g_scratch + 16, n, g_scratch);
  NIB_LAUNCH_CHECK();
  double t = 0.0;
  NIB_CUDA(cudaMemcpyAsync(&t, g_scratch, sizeof(double), cudaMemcpyDeviceToHost, st));
  NIB_CUDA(cudaStreamSynchronize(st));
  *h_grad = 0.5 * t;  // D2 here is already sqeuclidean(X / l): dK/dtheta = K0 .* D2
  return NIB_OK;
}

int nib_gp_ei(const double* d_mu, const double* d_sigma, int m, double best, int greater_is_better, double* d_ei,
              long long* d_argmax, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(d_mu && d_sigma && d_ei && m > 0, "nib_gp_ei: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  ei_kernel<<<ceil_div(m, 256), 256, 0, st>>>(d_mu, d_sigma, m, best, greater_is_better ? 1.0 : -1.0, d_ei);
  NIB_LAUNCH_CHECK();
  if (d_argmax) {
    argmax_kernel<<<1, 1024, 0, st>>>(d_ei, m, d_argmax);
    NIB_LAUNCH_CHECK();
  }
  return NIB_OK;
}

}  // extern "C"
