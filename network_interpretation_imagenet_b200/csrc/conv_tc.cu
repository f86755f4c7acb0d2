// conv_tc.cu — stage 2 hot kernel: implicit-GEMM convolution on the 5th-gen tensor cores.
//
//   out[m, co] = act( sum_k A[m, k] * Wt[co, k] + bias[co] + residual[m, co] ),  bf16 x bf16 -> fp32
//
// with m = (n, p, q) flattened output pixels, k = (r, s, c).  A is never materialised:
//   * 1x1 stride-1 convs read the NHWC activation matrix [N*H*W, C] with a tiled TMA map;
//   * every other geometry (3x3, strided) uses a TMA *im2col* map: the copy engine walks 128
//     consecutive output pixels (w fastest, then h, then n) of the padded bounding box and
//     fetches 64 channels of filter tap (r, s) for each, zero-filling the padding.
// Both land as a 128 x 64 bf16, 128B-swizzled, K-major tile = one tcgen05.mma operand.
// Weights are KRSC ([Cout][R*S*Cin], BN folded) and arrive through a second tiled map.
// Round 2 added three ways of NOT fetching one box per tap (the L2 -> SM port, ~43 B/clk/SM, was the bound of the
// layers concerned), all in conv_tc3_kernel and selected by TcKernelParams::a_mode:
//   * TC_A_HALO: 3x3 stride-1 pad-1 convs with 64 -> 64, 64 -> 32 or 128 -> 32 channels read ONE resident input patch per
//     tile (whole image rows in the raster of the padded width); tap (dy, dx) is the same swizzled operand started
//     (dy * Wp + dx) rows further on (descriptor base offset 0: the swizzle phase is address-based);
//   * TC_A_RAW: the 7x7 stride-2 stem reads the raw padded input rows through an UNSWIZZLED descriptor whose rows
//     overlap (row pitch 16 B = the stride-2 window over 8-byte pixels); a 3x3 stride-1 first conv on 16-byte pixels
//     (VGG's conv1_1) reads its three rows the same way (row pitch 16 B = one pixel);
//   * pre-activation 1x1 convs (DenseNet): four extra warps apply relu(x * scale + shift) to every A tile in shared
//     memory between its TMA completion and the MMA, instead of a separate pack pass.
//
// Three kernels live in this file: conv_tc_kernel (one CTA per tile, described next; serves Cout = 32 tiles and the
// fp32-output GEMM self-test), conv_tc3_kernel (the default: persistent CTA pairs with tcgen05 cta_group::2) and
// conv_fused_ca_kernel (a 1x1 expansion + the next 1x1 reduction in one launch).  DESIGN.md section 4 has the
// measurements that led from one to the next (an intermediate one-CTA persistent generation was removed in round 2).
//
// conv_tc_kernel: CTA = 192 threads, warp-specialised:  warp 0 lane 0 = TMA producer, warp 1 lane 0 = MMA issuer
// (warp 1 also owns the TMEM allocation), warps 2..5 = epilogue (TMEM -> registers -> bias /
// residual / ReLU -> bf16 -> global).  The accumulator (128 lanes x BLOCK_N fp32 columns) lives
// in TMEM; smem holds a STAGES-deep ring of (A, B) tiles guarded by full/empty mbarriers.
// Two CTAs are co-resident per SM (<= 113 KB smem, <= 256 TMEM columns each) so one CTA's
// epilogue overlaps the other's main loop.
//
// This replaces the cuDNN calls behind `model(masked_img_tensor)`
// (generate_gp_training_data_imagenet.py:246, bayesian_active_learning_imagenet.py:192).
#include "common.cuh"
#include "layers.cuh"
#include <cuda.h>
#include <string.h>
#include <stdlib.h>
#include <memory>

namespace nib {

static constexpr int TC_BLOCK_M = 128;
static constexpr int TC_BLOCK_K = 64;   // 64 bf16 = 128 B = one swizzle row
static constexpr int TC_UMMA_K = 16;
static constexpr int TC_THREADS = 192;

// How the A operand (the activations) reaches shared memory: TcKernelParams::a_mode.
enum TcAMode : int {
  TC_A_DENSE = 0,    // tiled 2D map over the NHWC activation matrix (1x1 stride-1 convs, the GEMM self-test)
  TC_A_IM2COL = 1,   // TMA im2col 4D map, one box per filter tap
  TC_A_STEM8 = 2,    // stem rows: overlapping-window 4D tiled map over 8-channel pixels, one filter row per K block
  TC_A_STEM4 = 3,    // stem row PAIRS over 4-channel pixels (CTA-pair kernel only)
  TC_A_HALO = 4,     // one resident input patch per tile (3x3 stride 1)
  TC_A_RAW = 5,      // raw padded input rows through an unswizzled descriptor with overlapping rows
};

struct TcKernelParams {
  const float* bias;
  const __nv_bfloat16* res;
  void* out;
  int M;            // valid output rows
  int Cout;
  int out_cstride, out_coff;
  int res_cstride, res_coff;
  int relu;
  int out_f32;      // 1: store fp32 (GEMM self-test), 0: bf16
  int num_k_blocks;
  int cblocks;      // Cin / 64
  int S;            // filter width (tap -> (r, s))
  int a_mode;       // TcAMode
  int tile_rows;    // valid output rows per M tile (128; Q for the stem mode: one output row per tile)
  int a_bytes;      // bytes the A load delivers per stage (tile_rows * 128)
  int P, Q, stride, pad;
  int in_coff;
  int n_tiles;      // ceil(Cout / BLOCK_N)
  int m_tiles;      // ceil(M / tile_rows)
  unsigned int* err_flag;
  unsigned long long* dbg;   // NIB_TC_DBG=1: per-CTA role timers (cycles), 16 slots per CTA; null in production
  // split-bf16 mode of the pair kernel (NIB_PREC_SPLIT): activations are [hi | lo] channel halves, the K loop walks
  // hi, lo, hi of every tap against weights [Wh | Wh | Wl]; the epilogue emits both halves of the fp32 result
  int a_wrap;                // 64-channel blocks after which the A channel index wraps back to the hi half (2 * Cin / 64)
  int lo_off_out;            // channel offset of the lo half in the output tensor
  int lo_off_res;            // ... and in the residual tensor
  const int* dyn_n;          // split mode: optional device-side live image count (the tie policy's re-score batch); tiles
                             // beyond live * P * Q rows are not computed
  // TC_A_HALO (3x3 stride-1 pad-1, 64 -> 64 channels): an M tile is halo_r whole image rows in the raster of the PADDED
  // width halo_wp = Q + 2; the (halo_r + 2) x halo_wp input patch is loaded once and all nine taps read it at shifted
  // start addresses
  int halo_wp, halo_r, halo_tpi;   // padded width, image rows per tile, tiles per image
  int halo_cb, halo_n;             // 64-channel blocks of Cin (1 | 2: one 32 KB patch block each) and the MMA's N (64 | 32:
                                   // DenseNet's 128 -> 32 growth convs; the weights stay resident either way, 36 KB per CTA)
  // pre-activation (DenseNet BN-ReLU-conv 1x1): y = relu(x * xf_scale[c] + xf_shift[c]) applied to the A tile in shared
  // memory by four extra warps per CTA between the TMA load and the MMA (arrays zero-padded to the 64-channel K block:
  // channels past Cin become exact zeros whatever the concat buffer holds there)
  const float* xf_scale;
  const float* xf_shift;
  int halo_swap;                   // TC_A_RAW diagnostics: swap the LBO / SBO roles of the unswizzled descriptor
  // TC_A_RAW (raw input rows): filter rows per tile (7: the 7x7/2 stem, 3: a 3x3/1 first conv) and column tiles per
  // output row (1 unless the row is wider than the 128-row M tile).  Pair tile mp holds output rows 2 (mp / col_tiles) and
  // 2 (mp / col_tiles) + 1 (one per CTA) in the SAME column tile mp % col_tiles, so both CTAs' A operands start at the same
  // shared-memory offset: the leader's descriptor addresses both.
  int raw_rows, col_tiles;
};

// ---- PTX wrappers -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done != 0;
}
// Bounded wait: a descriptor bug must fail the launch, not hang the GPU box.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, unsigned int* err_flag, int code) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {  // ~2 s at 1.9 GHz
      if (err_flag) atomicExch(err_flag, (unsigned)code);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_im2col_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c, int w,
                                                   int h, int n, uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w),
      "h"(off_h)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// L2 prefetch of a tile the kernel will TMA-load a little later (the fused kernel's next residual chunk)
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* tm, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];"
               ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128B-swizzled smem tile (rows of 128 B, 8-row groups 1024 B apart).
// cute::UMMA::SmemDescriptor (cute/arch/mma_sm100_desc.hpp): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout_type [61,64) with SWIZZLE_128B = 2.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;            // LBO (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;  // SBO
  d |= (uint64_t)1 << 46;            // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;            // SWIZZLE_128B
  return d;
}

// K-major, unswizzled: core matrices of 8 rows x 16 B (128 contiguous bytes); lbo = distance between core matrices along K,
// sbo = between 8-row groups.  With lbo = 16 and sbo = 128 row r starts 16 r bytes into the buffer and its K run simply
// continues: overlapping rows, which is exactly a stride-2 window over 8-byte pixels (the stem, TC_A_RAW).
__device__ __forceinline__ uint64_t make_smem_desc_nosw(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

// K-major, 64B-swizzled smem tile: rows of 64 B (32 bf16 of K), 8-row groups 512 B apart (cute LayoutType SWIZZLE_64B = 4)
__device__ __forceinline__ uint64_t make_smem_desc_sw64(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;
  return d;
}

template <int BLOCK_N>
__host__ __device__ constexpr uint32_t make_idesc_bf16() {
  // cute::UMMA::InstrDescriptor: c_format F32=1 @4, a_format BF16=1 @7, b_format BF16=1 @10,
  // a_major/b_major K=0 @15/@16, N>>3 @17, M>>4 @24
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(TC_BLOCK_M >> 4) << 24);
}

template <int BLOCK_N, int STAGES>
struct TcSmem {
  static constexpr int A_BYTES = TC_BLOCK_M * TC_BLOCK_K * 2;  // 16 KB
  static constexpr int B_BYTES = BLOCK_N * TC_BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BAR_OFFSET = STAGES * STAGE_BYTES;
  static constexpr int TOTAL = BAR_OFFSET + (2 * STAGES + 1) * 8 + 16 + 1024 /*alignment slack*/;
};

template <int BLOCK_N, int STAGES>
__global__ void __launch_bounds__(TC_THREADS)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const TcKernelParams p) {
  using SM = TcSmem<BLOCK_N, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + SM::BAR_OFFSET;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * STAGES);
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 1);
  uint32_t* tmem_slot_ptr =
      reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n_tile = blockIdx.x % p.n_tiles;
  const int m_tile = blockIdx.x / p.n_tiles;
  const int m0 = m_tile * p.tile_rows;
  const int n0 = n_tile * BLOCK_N;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                 "r"((uint32_t)(BLOCK_N < 32 ? 32 : BLOCK_N))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer =====
      int w0 = 0, h0 = 0, img = 0;
      if (p.a_mode == TC_A_IM2COL) {
        const int pq = p.P * p.Q;
        img = m0 / pq;
        const int rem = m0 - img * pq;
        const int pp = rem / p.Q, qq = rem - pp * p.Q;
        w0 = qq * p.stride - p.pad;
        h0 = pp * p.stride - p.pad;
      } else if (p.a_mode == TC_A_STEM8) {   // one output row (img, pp) per tile; input rows pp*stride + r of the haloed image
        img = m_tile / p.P;
        h0 = (m_tile - img * p.P) * p.stride;
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < p.num_k_blocks; ++kb) {
        mbar_wait(empty_bar(stage), phase ^ 1u, p.err_flag, 1);
        const uint32_t a_dst = smem_base + stage * SM::STAGE_BYTES;
        const uint32_t b_dst = a_dst + SM::A_BYTES;
        mbar_arrive_expect_tx(full_bar(stage), (uint32_t)(p.a_bytes + SM::B_BYTES));
        const int tap = kb / p.cblocks;
        const int c0 = (kb - tap * p.cblocks) * TC_BLOCK_K + p.in_coff;
        if (p.a_mode == TC_A_IM2COL) {
          const int r = tap / p.S, s = tap - r * p.S;
          tma_load_im2col_4d(a_dst, &tmA, full_bar(stage), c0, w0, h0, img, (uint16_t)s, (uint16_t)r);
        } else if (p.a_mode == TC_A_STEM8) {
          tma_load_4d(a_dst, &tmA, full_bar(stage), 0, 0, h0 + kb, img);   // k-block kb = filter row r
        } else {
          tma_load_2d(a_dst, &tmA, full_bar(stage), c0, m0);
        }
        tma_load_2d(b_dst, &tmB, full_bar(stage), kb * TC_BLOCK_K, n0);
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer =====
      constexpr uint32_t idesc = make_idesc_bf16<BLOCK_N>();
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < p.num_k_blocks; ++kb) {
        mbar_wait(full_bar(stage), phase, p.err_flag, 2);
        tc_fence_after();
        const uint32_t a_addr = smem_base + stage * SM::STAGE_BYTES;
        const uint32_t b_addr = a_addr + SM::A_BYTES;
        const uint64_t adesc = make_smem_desc_sw128(a_addr);
        const uint64_t bdesc = make_smem_desc_sw128(b_addr);
#pragma unroll
        for (int k = 0; k < TC_BLOCK_K / TC_UMMA_K; ++k) {
          // advance 16 bf16 = 32 B along K inside the swizzle row: +2 in the (addr >> 4) field
          umma_bf16(tmem_base, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0);
        }
        umma_commit(empty_bar(stage));  // frees the smem slot when these MMAs retire
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
      umma_commit(tmem_full_bar);  // accumulator complete
    }
  } else {
    // ===== epilogue: warps 2..5, TMEM lane quarter = warp % 4 =====
    const int quarter = warp & 3;
    mbar_wait(tmem_full_bar, 0, p.err_flag, 3);
    tc_fence_after();
    const int lrow = quarter * 32 + lane;
    const int row = m0 + lrow;
    const bool row_ok = row < p.M && lrow < p.tile_rows;
#pragma unroll 1
    for (int cc = 0; cc < BLOCK_N; cc += 32) {
      uint32_t v[32];
      __syncwarp();  // .sync.aligned TMEM loads need the full warp converged
      tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)cc, v);
      tmem_ld_wait();
      const int col0 = n0 + cc;
      if (row_ok && col0 < p.Cout) {
      float f[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
      if (p.bias != nullptr) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + j));
          f[j] += b.x; f[j + 1] += b.y; f[j + 2] += b.z; f[j + 3] += b.w;
        }
      }
      if (p.res != nullptr) {
        const __nv_bfloat16* rp = p.res + (size_t)row * p.res_cstride + p.res_coff + col0;
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          const uint4 raw = *reinterpret_cast<const uint4*>(rp + j);
          const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float2 r2 = __bfloat1622float2(h2[t]);
            f[j + 2 * t] += r2.x;
            f[j + 2 * t + 1] += r2.y;
          }
        }
      }
      if (p.relu) {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
      }
      if (p.out_f32) {
        float* op = reinterpret_cast<float*>(p.out) + (size_t)row * p.out_cstride + p.out_coff + col0;
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<float4*>(op + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
      } else {
        __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + (size_t)row * p.out_cstride + p.out_coff + col0;
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          uint4 o;
          __nv_bfloat162 h;
          h = __floats2bfloat162_rn(f[j], f[j + 1]);     o.x = *reinterpret_cast<uint32_t*>(&h);
          h = __floats2bfloat162_rn(f[j + 2], f[j + 3]); o.y = *reinterpret_cast<uint32_t*>(&h);
          h = __floats2bfloat162_rn(f[j + 4], f[j + 5]); o.z = *reinterpret_cast<uint32_t*>(&h);
          h = __floats2bfloat162_rn(f[j + 6], f[j + 7]); o.w = *reinterpret_cast<uint32_t*>(&h);
          *reinterpret_cast<uint4*>(op + j) = o;
        }
      }
      }  // row_ok
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"((uint32_t)(BLOCK_N < 32 ? 32 : BLOCK_N))
                 : "memory");
  }
}


__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tm, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_v4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// =====================================================================================================
// CTA-pair kernel (tcgen05 cta_group::2).  Two CTAs of a (2,1,1) cluster sit on the two SMs of a TPC and
// compute one 256 x BLOCK_N output tile together: each CTA loads its own 128 activation rows and HALF of the
// weight tile (BLOCK_N/2 rows); the leader CTA issues one M=256 MMA per K step that reads A and B from both
// CTAs' shared memory and writes rows 0..127 of the accumulator into its own TMEM and rows 128..255 into the
// peer's.  Per output element this halves the weight traffic L2 -> SM, which is what bounded the one-CTA persistent kernel
// (profiles/README.md: 694 MB of smem fill per 3x3 256->256 launch = 11.7 TB/s, the measured L2 ceiling).
//   * smem ring per CTA: STAGES x (16 KB A + BLOCK_N/2 x 128 B of B); both CTAs' TMA loads complete on the
//     LEADER's full barrier, one tcgen05.commit.multicast frees the slot in both CTAs;
//   * TMEM: 2 accumulator buffers of BLOCK_N columns per CTA (all 512 columns at BLOCK_N = 256);
//   * epilogue: 8 warps (2 warpgroups, each owns half of the tile's columns) in each CTA drain their own
//     TMEM lanes; the residual box is TMA-loaded into the SAME smem box the result is staged in (add in
//     place), so a 128 x 256 tile with residual still leaves room for a 5-deep ring;
//   * the tile order keeps the CTA pairs that share activation rows adjacent in time (n fastest).
static constexpr int TC3_THREADS = 64 + 256;
static constexpr int TC3_XF_WARPS = 4;                         // pre-activation mode: warps 10..13 transform the A tiles
static constexpr int TC3_THREADS_XF = TC3_THREADS + 32 * TC3_XF_WARPS;

// BRES: the layer's whole weight matrix (Cout == BLOCK_N, <= 9 K blocks: the 64-channel layers and the stem) is loaded
// once per CTA and stays resident; the ring then carries activation tiles only, which halves the TMA instructions
// the producer has to issue per K block (the issue rate, not the bytes, bounds these layers).
static constexpr int TC3_BRES_KBLOCKS = 9;
template <int BLOCK_N, int STAGES, bool HAS_RES, bool BRES = false, bool SPLIT = false>
struct Tc3Smem {
  static constexpr int A_BYTES = TC_BLOCK_M * TC_BLOCK_K * 2;
  static constexpr int BH_BYTES = (BLOCK_N / 2) * TC_BLOCK_K * 2;   // this CTA's half of the weight tile
  static constexpr int STAGE_BYTES = A_BYTES + (BRES ? 0 : BH_BYTES);
  static constexpr int BRES_BYTES = BRES ? TC3_BRES_KBLOCKS * BH_BYTES : 0;
  static constexpr int NBOX = BLOCK_N / 64;                          // 64-channel output boxes per tile
  static constexpr bool SPLIT_COLS = NBOX >= 2;                      // warpgroup g drains columns [g*BLOCK_N/2, ...) of every
                                                                     // tile; BLOCK_N = 64: warpgroup g drains the tiles in TMEM buffer g
  static constexpr int CW = SPLIT_COLS ? BLOCK_N / 2 : 64;           // columns one warpgroup drains per tile
  static constexpr int UNITS = CW / 64;                              // 64-channel boxes per warpgroup per tile
  static constexpr int BOX_BYTES = TC_BLOCK_M * 128;
  static constexpr int RSETS = HAS_RES ? (BLOCK_N == 256 ? 1 : 2) : 1;
  static constexpr int RBOX = SPLIT ? 2 * NBOX : NBOX;               // boxes of one residual set (split mode: hi boxes, then lo boxes)
  static constexpr int NBUF = HAS_RES ? RSETS * RBOX : 2;            // residual/output boxes, or 8 x 4 KB per-warp staging
  static constexpr int BRES_OFFSET = STAGES * STAGE_BYTES;
  static constexpr int BOX_OFFSET = BRES_OFFSET + BRES_BYTES;
  static constexpr int BIAS_OFFSET = BOX_OFFSET + NBUF * BOX_BYTES;   // [warpgroup][2][CW] floats: the tile's folded-BN bias
  static constexpr int BAR_OFFSET = BIAS_OFFSET + 2 * 2 * CW * 4;
  static constexpr int NUM_BARS = 2 * STAGES + 4 + 2 * NBUF + 1 + 2 * STAGES;   // + A-landed (local) and A-transformed
                                                                                 // (leader) per stage: pre-activation mode
  static constexpr int EMPTY_ARRIVALS = SPLIT_COLS ? 16 : 8;         // epilogue warps (both CTAs) that drain one accumulator
  // dynamic smem is the only shared allocation of the kernel, so it starts 1024-aligned in the CTA window; the kernel
  // checks that (the 128B swizzle needs it) instead of spending 1 KB of slack on it
  static constexpr int TOTAL = BAR_OFFSET + NUM_BARS * 8 + 16;
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives (once the MMAs issued so far have retired) on the barrier at this smem offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma2_commit_both(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}
// pair loads: data lands in this CTA's smem, the transaction bytes are counted on the leader CTA's barrier
__device__ __forceinline__ void tma2_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma2_load_4d(uint32_t dst, const CUtensorMap* tm, uint32_t leader_bar, int c0, int c1,
                                             int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma2_load_5d(uint32_t dst, const CUtensorMap* tm, uint32_t leader_bar, int c0, int c1,
                                             int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma2_load_im2col_4d(uint32_t dst, const CUtensorMap* tm, uint32_t leader_bar, int c,
                                                    int w, int h, int n, uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.im2col.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(leader_bar), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w),
      "h"(off_h)
      : "memory");
}
__device__ __forceinline__ bool elect_one() {   // true in exactly one lane of the (converged) warp
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ void tmem_ld_32x32b_x64(uint32_t taddr, uint32_t (&v)[64]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, "
      "%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, "
      "%48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]),
        "=r"(v[32]), "=r"(v[33]), "=r"(v[34]), "=r"(v[35]), "=r"(v[36]), "=r"(v[37]), "=r"(v[38]), "=r"(v[39]),
        "=r"(v[40]), "=r"(v[41]), "=r"(v[42]), "=r"(v[43]), "=r"(v[44]), "=r"(v[45]), "=r"(v[46]), "=r"(v[47]),
        "=r"(v[48]), "=r"(v[49]), "=r"(v[50]), "=r"(v[51]), "=r"(v[52]), "=r"(v[53]), "=r"(v[54]), "=r"(v[55]),
        "=r"(v[56]), "=r"(v[57]), "=r"(v[58]), "=r"(v[59]), "=r"(v[60]), "=r"(v[61]), "=r"(v[62]), "=r"(v[63])
      : "r"(taddr)
      : "memory");
}
// packed epilogue math: two fp32 lanes per instruction (FADD2), one convert per bf16 pair, ReLU on the packed pair
__device__ __forceinline__ uint64_t pack_f32x2(uint32_t lo, uint32_t hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}
__device__ __forceinline__ uint64_t add_f32x2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint32_t cvt_bf16x2(uint64_t a) {   // {lo, hi} fp32 -> bf16x2 (lo in the low half), RN
  uint32_t lo, hi, r;
  asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(a));
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(__uint_as_float(hi)), "f"(__uint_as_float(lo)));
  return r;
}
__device__ __forceinline__ uint32_t max_bf16x2(uint32_t a, uint32_t b) {   // NaN-propagating, like torch.relu
  uint32_t r;
  asm("max.NaN.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}

template <int BLOCK_N>
__host__ __device__ constexpr uint32_t make_idesc_bf16_pair() {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
}

template <int BLOCK_N, int STAGES, bool HAS_RES, bool BRES, bool SPLIT = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC3_THREADS_XF, 1)
conv_tc3_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmOut, const __grid_constant__ CUtensorMap tmOutTail,
                const __grid_constant__ CUtensorMap tmRes, const TcKernelParams p) {
  using SM = Tc3Smem<BLOCK_N, STAGES, HAS_RES, BRES, SPLIT>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = smem_u32(smem_raw);
  if ((smem_base & 1023u) != 0) {
    if (threadIdx.x == 0 && p.err_flag) atomicExch(p.err_flag, 9u);
    __trap();
  }
  const uint32_t bar_base = smem_base + SM::BAR_OFFSET;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };                         // used in the leader CTA
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tmem_full_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + b); };
  auto tmem_empty_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + 2 + b); }; // used in the leader CTA
  auto res_full_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + 4 + b); };
  auto box_free_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + 4 + SM::NBUF + b); };
  const uint32_t bres_full_bar = bar_base + 8u * (2 * STAGES + 4 + 2 * SM::NBUF);   // used in the leader CTA
  auto afull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + 5 + 2 * SM::NBUF + s); };            // this CTA's A tile landed
  auto xf_bar = [&](int s) { return bar_base + 8u * (3 * STAGES + 5 + 2 * SM::NBUF + s); };               // leader: both transformed
  const bool xform = !BRES && !SPLIT && p.xf_scale != nullptr;
  const uint32_t tmem_slot = bar_base + 8u * SM::NUM_BARS;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
  auto box_addr = [&](int buf) { return smem_base + SM::BOX_OFFSET + (uint32_t)buf * SM::BOX_BYTES; };

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1;
  const int npairs = gridDim.x >> 1;
  int m_tiles_live = p.m_tiles;
  if (SPLIT && p.dyn_n != nullptr) {   // written many launches ago (score.cu tie_compact_kernel): safe before griddepcontrol.wait
    const long long live = (long long)max(*p.dyn_n, 0) * p.P * p.Q;
    const int t = (int)((live + p.tile_rows - 1) / p.tile_rows);
    if (t < m_tiles_live) m_tiles_live = t;
  }
  const int m_pairs = (m_tiles_live + 1) >> 1;
  const int total_tiles = m_pairs * p.n_tiles;
  constexpr uint32_t TMEM_COLS = 2 * BLOCK_N;
  // role timers (debug builds of a launch only: p.dbg != null)
  const bool dbg_on = p.dbg != nullptr;
  long long t_acc[4] = {0, 0, 0, 0};
  long long t_loop0 = 0;
  if (dbg_on && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    p.dbg[(size_t)blockIdx.x * 16 + 12] = gt;
    p.dbg[(size_t)blockIdx.x * 16 + 14] = (unsigned long long)clock64();
  }
#define TC3_TIMED(slot, stmt)                                      \
  do {                                                             \
    if (dbg_on) { const long long _t = clock64(); stmt; t_acc[slot] += clock64() - _t; } \
    else { stmt; }                                                 \
  } while (0)

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    prefetch_tmap(&tmOut);
    if (HAS_RES) prefetch_tmap(&tmRes);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tmem_full_bar(b), 1);
      mbar_init(tmem_empty_bar(b), SM::EMPTY_ARRIVALS);   // the epilogue warps of both CTAs that drain one accumulator
    }
    for (int b = 0; b < SM::NBUF; ++b) {
      mbar_init(res_full_bar(b), 1);
      mbar_init(box_free_bar(b), 4);   // the four warps that store a box hand it back
    }
    mbar_init(bres_full_bar, 1);
    for (int s2 = 0; s2 < STAGES; ++s2) {
      mbar_init(afull_bar(s2), 1);
      mbar_init(xf_bar(s2), 2 * TC3_XF_WARPS);   // the transform warps of both CTAs
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  if (p.a_mode == TC_A_RAW && p.stride == 1) {
    // 3x3 raw rows: the last output pixel's zero-weight filler tap reads the 16 bytes just past the third row, which no
    // TMA load ever writes.  Zero the ring once so that 0 * (whatever the SM held before) cannot inject a NaN.
    for (uint32_t off = 16u * threadIdx.x; off < (uint32_t)(STAGES * SM::STAGE_BYTES); off += 16u * blockDim.x)
      sts_v4(smem_base + off, make_uint4(0u, 0u, 0u, 0u));
    fence_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // the peer's barriers exist before anything arrives on them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor prefetch, cluster
  // handshake) ran while the previous layer's kernel was still draining; from here on we touch its output.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  // The producer and MMA roles run their loops with the whole warp converged and elect one lane only around the
  // asynchronous instructions themselves: loop state stays in uniform registers, so each TMA / MMA issue is a handful of
  // instructions (a role nested inside `if (lane == 0)` makes the compiler wrap every UTMALDG / UTCHMMA in an
  // ELECT + R2UR.BROADCAST waterfall, ~100 cycles per issue, which was the actual ceiling of the 64-channel layers).
  if (warp == 0) {
    // ===== TMA producer (both CTAs) =====
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    const uint32_t lbar0 = mapa_shared(full_bar(0), 0);   // leader CTA's full barriers
    const uint32_t tx_bytes = (uint32_t)(2 * ((xform ? 0 : p.a_bytes) + (BRES ? 0 : SM::BH_BYTES)));
    const int b_row0 = (int)rank * ((BRES && p.a_mode == TC_A_HALO ? p.halo_n : BLOCK_N) / 2);
    // residual boxes of the previous tile still to be requested: they are issued opportunistically while this
    // tile's operands stream (a box frees up when the epilogue's store of the tile before has drained), so a
    // busy epilogue never stalls the operand ring
    int pend_b = SM::RBOX, pend_set = 0, pend_m0 = 0, pend_n0 = 0;
    uint32_t pend_par = 0;
    auto issue_pending = [&](bool block) {
      while (pend_b < SM::RBOX) {
        const int buf = pend_set * SM::RBOX + pend_b;
        if (block) {
          TC3_TIMED(1, mbar_wait(box_free_bar(buf), pend_par ^ 1u, p.err_flag, 4));
        } else {
          const int ready = __shfl_sync(0xffffffffu, (int)mbar_try_wait(box_free_bar(buf), pend_par ^ 1u), 0);
          if (!ready) return;
        }
        if (elect_one()) {
          mbar_arrive_expect_tx(res_full_bar(buf), (uint32_t)SM::BOX_BYTES);
          const int rc = SPLIT ? p.res_coff + pend_n0 + 64 * (pend_b % SM::NBOX) + (pend_b >= SM::NBOX ? p.lo_off_res : 0)
                               : p.res_coff + pend_n0 + 64 * pend_b;
          tma_load_2d(box_addr(buf), &tmRes, res_full_bar(buf), rc, pend_m0);
        }
        __syncwarp();
        ++pend_b;
      }
    };
    if (dbg_on) t_loop0 = clock64();
    if (BRES) {   // both CTAs fetch their half of every K block of the weights once
      if (elect_one()) {
        const uint32_t lb = mapa_shared(bres_full_bar, 0);
        const uint32_t bhb = p.a_mode == TC_A_HALO ? (uint32_t)(p.halo_n * 64) : (uint32_t)SM::BH_BYTES;   // halo_n / 2 rows x 128 B
        if (rank == 0) mbar_arrive_expect_tx(bres_full_bar, (uint32_t)(2 * p.num_k_blocks) * bhb);
        for (int kb = 0; kb < p.num_k_blocks; ++kb) {
          const uint32_t dst = smem_base + SM::BRES_OFFSET + kb * bhb;
          if (p.a_mode == TC_A_STEM4 || p.a_mode == TC_A_RAW) {   // 64B-swizzled: the K block is two 32-element atoms
            tma2_load_2d(dst, &tmB, lb, kb * TC_BLOCK_K, b_row0);
            tma2_load_2d(dst + SM::BH_BYTES / 2, &tmB, lb, kb * TC_BLOCK_K + 32, b_row0);
          } else {
            tma2_load_2d(dst, &tmB, lb, kb * TC_BLOCK_K, b_row0);
          }
        }
      }
      __syncwarp();
    }
    for (int tile = pair; tile < total_tiles; tile += npairs, ++it) {
      const int n_tile = tile % p.n_tiles;
      const int mp = tile / p.n_tiles;
      // raw rows: m_tile is the output row (image-major); the tile covers column tile mp % col_tiles of it
      const int m_tile = p.a_mode == TC_A_RAW ? (mp / p.col_tiles) * 2 + (int)rank : mp * 2 + (int)rank;
      const int m0 = p.a_mode == TC_A_RAW ? (m_tile * p.col_tiles + mp % p.col_tiles) * p.tile_rows : m_tile * p.tile_rows;
      const int n0 = n_tile * BLOCK_N;
      int w0 = 0, h0 = 0, img = 0;
      if (p.a_mode == TC_A_IM2COL) {
        const int pq = p.P * p.Q;
        img = m0 / pq;
        const int rem = m0 - img * pq;
        const int pp = rem / p.Q, qq = rem - pp * p.Q;
        w0 = qq * p.stride - p.pad;
        h0 = pp * p.stride - p.pad;
      } else if (p.a_mode >= TC_A_STEM8) {
        img = m_tile / p.P;
        h0 = (m_tile - img * p.P) * p.stride;
      }
      if (BRES && !HAS_RES && p.a_mode == TC_A_HALO) {
        // halo patch: ONE 4D tiled load per tile (rows y0-1 .. y0+halo_r, columns -1 .. Q; out-of-range coordinates are
        // zero-filled = the convolution's padding) into one of four 32 KB buffers (ring stages 0, 2, 4, 6)
        // (two 32 KB blocks per buffer and two buffers when Cin = 128)
        const int npb = 4 / p.halo_cb, pbuf = it % npb;
        const int st4 = 2 * p.halo_cb * pbuf;
        TC3_TIMED(0, mbar_wait(empty_bar(st4), (uint32_t)(((it / npb) & 1) ^ 1), p.err_flag, 1));
        if (elect_one()) {
          const int im = m_tile / p.halo_tpi;
          const int y0 = (m_tile - im * p.halo_tpi) * p.halo_r;
          if (rank == 0) mbar_arrive_expect_tx(full_bar(st4), (uint32_t)(2 * p.halo_cb * p.a_bytes));
          for (int c = 0; c < p.halo_cb; ++c)
            tma2_load_4d(smem_base + (st4 + 2 * c) * SM::STAGE_BYTES, &tmA, lbar0 + 8u * st4, p.in_coff + 64 * c, -1, y0 - 1, im);
        }
        __syncwarp();
        continue;
      }
      if (BRES && !HAS_RES && p.a_mode == TC_A_RAW) {
        // the padded input rows under one output row (7 for the stem, 3 for a 3x3 conv), raw, one ring stage per tile
        TC3_TIMED(0, mbar_wait(empty_bar(stage), phase ^ 1u, p.err_flag, 1));
        if (elect_one()) {
          if (rank == 0) mbar_arrive_expect_tx(full_bar(stage), (uint32_t)(2 * p.a_bytes));
          tma2_load_4d(smem_base + stage * SM::STAGE_BYTES, &tmA, lbar0 + 8u * stage, 0, 0, h0, img);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        continue;
      }
      int kb = 0, cb = 0, tap_s = 0, tap_r = 0;   // k-block -> (filter row, column, 64-channel block)
      for (int kk = 0; kk < p.num_k_blocks; ++kk) {
        if (HAS_RES) issue_pending(false);
        TC3_TIMED(0, mbar_wait(empty_bar(stage), phase ^ 1u, p.err_flag, 1));
        if (elect_one()) {
          const uint32_t a_dst = smem_base + stage * SM::STAGE_BYTES;
          const uint32_t lbar = lbar0 + 8u * stage;
          if (rank == 0) mbar_arrive_expect_tx(full_bar(stage), tx_bytes);
          const int ca = SPLIT ? (cb >= p.a_wrap ? cb - p.a_wrap : cb) : cb;   // split mode: hi, lo, hi again
          const int c0 = ca * TC_BLOCK_K + p.in_coff;
          if (p.a_mode == TC_A_IM2COL) {
            tma2_load_im2col_4d(a_dst, &tmA, lbar, c0, w0, h0, img, (uint16_t)tap_s, (uint16_t)tap_r);
          } else if (p.a_mode == TC_A_STEM8) {
            tma2_load_4d(a_dst, &tmA, lbar, 0, 0, h0 + kb, img);
          } else if (p.a_mode == TC_A_STEM4) {
            // K block kb = filter rows 2kb, 2kb+1: two 64B-swizzled K atoms of [Q rows x 32 elements]
            tma2_load_4d(a_dst, &tmA, lbar, 0, 0, h0 + 2 * kb, img);
            tma2_load_4d(a_dst + SM::A_BYTES / 2, &tmA, lbar, 0, 0, h0 + 2 * kb + 1, img);
          } else if (xform) {
            // pre-activation: this CTA's A tile completes on its OWN barrier (its transform warps cannot wait on the leader's)
            mbar_arrive_expect_tx(afull_bar(stage), (uint32_t)p.a_bytes);
            tma_load_2d(a_dst, &tmA, afull_bar(stage), c0, m0);
          } else {
            tma2_load_2d(a_dst, &tmA, lbar, c0, m0);
          }
          if (!BRES) tma2_load_2d(a_dst + SM::A_BYTES, &tmB, lbar, kb * TC_BLOCK_K, n0 + b_row0);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        ++kb;
        if (++cb == p.cblocks) { cb = 0; if (++tap_s == p.S) { tap_s = 0; ++tap_r; } }
      }
      if (HAS_RES) {
        issue_pending(true);   // the tile before this one: its boxes were freed at least one whole tile ago
        pend_b = 0;
        pend_set = it % SM::RSETS;
        pend_par = (uint32_t)((it / SM::RSETS) & 1);
        pend_m0 = m0;
        pend_n0 = n0;
      }
    }
    if (HAS_RES) issue_pending(true);
    if (dbg_on && lane == 0) {
      unsigned long long* d = p.dbg + (size_t)blockIdx.x * 16;
      d[0] = (unsigned long long)t_acc[0]; d[1] = (unsigned long long)t_acc[1];
      d[8] = (unsigned long long)(clock64() - t_loop0);
    }
  } else if (warp == 1) {
    if (rank == 0) {
      // ===== MMA issuer (leader CTA only) =====
      constexpr uint32_t idesc = make_idesc_bf16_pair<BLOCK_N>();
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      if (dbg_on) t_loop0 = clock64();
      if (BRES) mbar_wait(bres_full_bar, 0, p.err_flag, 7);
      for (int tile = pair; tile < total_tiles; tile += npairs, ++it) {
        const int ab = it & 1;
        TC3_TIMED(1, mbar_wait(tmem_empty_bar(ab), (uint32_t)(((it >> 1) & 1) ^ 1), p.err_flag, 5));
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(ab * BLOCK_N);
        if (BRES && !HAS_RES && p.a_mode == TC_A_HALO) {
          // nine taps out of one resident patch: tap (dy, dx) is the same 128-row operand started (dy * Wp + dx) pixels
          // = that many 128 B swizzle rows further on.  The tensor core derives the swizzle phase from the absolute
          // shared-memory address, like the copy engine that wrote the patch, so a start that is not a multiple of 8 rows
          // needs nothing else: the descriptor's base-offset field stays 0 (measured: setting it to (address >> 7) & 7
          // breaks parity, profiles/r02_pytest_halo_base_offset.log)
          const int npb = 4 / p.halo_cb, pbuf = it % npb;
          const int st4 = 2 * p.halo_cb * pbuf;
          TC3_TIMED(0, mbar_wait(full_bar(st4), (uint32_t)((it / npb) & 1), p.err_flag, 2));
          tc_fence_after();
          if (elect_one()) {
            const uint32_t patch = smem_base + st4 * SM::STAGE_BYTES;
            const uint32_t bhb = (uint32_t)(p.halo_n * 64);
            const uint32_t idesc_h = p.halo_n == 32 ? make_idesc_bf16_pair<32>() : idesc;
#pragma unroll 1
            for (int kb = 0; kb < 9 * p.halo_cb; ++kb) {      // K order of the KRSC weights: tap major, channel block minor
              const int tap = p.halo_cb == 2 ? (kb >> 1) : kb, c = p.halo_cb == 2 ? (kb & 1) : 0;
              const int dy = tap / 3, dx = tap - 3 * dy;
              const uint32_t a_addr = patch + (uint32_t)(2 * c) * SM::STAGE_BYTES + (uint32_t)(dy * p.halo_wp + dx) * 128u;
              const uint64_t adesc = make_smem_desc_sw128(a_addr);
              const uint64_t bdesc = make_smem_desc_sw128(smem_base + SM::BRES_OFFSET + (uint32_t)kb * bhb);
#pragma unroll
              for (int k = 0; k < TC_BLOCK_K / TC_UMMA_K; ++k)
                umma2_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc_h, (kb | k) != 0);
            }
            umma2_commit_both(empty_bar(st4));
            umma2_commit_both(tmem_full_bar(ab));
          }
          __syncwarp();
          continue;
        }
        if (BRES && !HAS_RES && p.a_mode == TC_A_RAW) {
          // stem on raw input rows: output pixel q of filter row r reads 32 elements (8 taps x 4 channels) starting at
          // pixel 2q of input row 2p + r, i.e. 16 q bytes into that row - an unswizzled K-major operand whose rows
          // OVERLAP (row pitch 16 B, K chunk pitch 16 B).  Each input byte crosses L2 -> SM once per output row instead
          // of once per tap: 12.9 KB per tile instead of 56 KB of 64-byte rows.
          // The 3x3 stride-1 form is the same operand over 16-byte pixels: 3 taps x 8 channels + one filler tap per filter
          // row, row pitch 16 B = one pixel; column tile c starts 16 (c * tile_rows) bytes into the rows (both CTAs of the
          // pair are in the same column tile).
          TC3_TIMED(0, mbar_wait(full_bar(stage), phase, p.err_flag, 2));
          tc_fence_after();
          if (elect_one()) {
            const int q0 = ((tile / p.n_tiles) % p.col_tiles) * p.tile_rows;
            const uint32_t a_addr = smem_base + stage * SM::STAGE_BYTES + 16u * (uint32_t)q0;
            const uint32_t lbo = p.halo_swap ? 128u : 16u, sbo = p.halo_swap ? 16u : 128u;
#pragma unroll 1
            for (int r = 0; r < p.raw_rows; ++r) {
              const uint32_t b_addr = smem_base + SM::BRES_OFFSET + (r >> 1) * SM::BH_BYTES + (r & 1) * (SM::BH_BYTES / 2);
#pragma unroll
              for (int ks = 0; ks < 2; ++ks) {
                const uint64_t adesc = make_smem_desc_nosw(a_addr + (uint32_t)(r * p.halo_wp) + ks * 32, lbo, sbo);
                const uint64_t bdesc = make_smem_desc_sw64(b_addr + ks * 32);
                umma2_bf16(d_tmem, adesc, bdesc, idesc, (r | ks) != 0);
              }
            }
            umma2_commit_both(empty_bar(stage));
            umma2_commit_both(tmem_full_bar(ab));
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          continue;
        }
        for (int kk = 0; kk < p.num_k_blocks; ++kk) {
          const int kb = kk;
          TC3_TIMED(0, mbar_wait(full_bar(stage), phase, p.err_flag, 2));
          if (xform) TC3_TIMED(0, mbar_wait(xf_bar(stage), phase, p.err_flag, 8));
          tc_fence_after();
          if (elect_one()) {
            const uint32_t a_addr = smem_base + stage * SM::STAGE_BYTES;
            const uint32_t b_addr = BRES ? smem_base + SM::BRES_OFFSET + kb * SM::BH_BYTES : a_addr + SM::A_BYTES;
            if (BRES && p.a_mode == TC_A_STEM4) {
              // 64B-swizzled operands: K atom a (32 elements) at +a * half the tile, 16-element step inside it = +32 B
#pragma unroll
              for (int k = 0; k < TC_BLOCK_K / TC_UMMA_K; ++k) {
                const uint64_t adesc = make_smem_desc_sw64(a_addr + (k >> 1) * (SM::A_BYTES / 2) + (k & 1) * 32);
                const uint64_t bdesc = make_smem_desc_sw64(b_addr + (k >> 1) * (SM::BH_BYTES / 2) + (k & 1) * 32);
                umma2_bf16(d_tmem, adesc, bdesc, idesc, (kk | k) != 0);
              }
            } else {
              const uint64_t adesc = make_smem_desc_sw128(a_addr);
              const uint64_t bdesc = make_smem_desc_sw128(b_addr);
#pragma unroll
              for (int k = 0; k < TC_BLOCK_K / TC_UMMA_K; ++k)
                umma2_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kk | k) != 0);
            }
            umma2_commit_both(empty_bar(stage));
            if (kk == p.num_k_blocks - 1) umma2_commit_both(tmem_full_bar(ab));
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
      if (dbg_on && lane == 0) {
        unsigned long long* d = p.dbg + (size_t)blockIdx.x * 16;
        d[2] = (unsigned long long)t_acc[0]; d[3] = (unsigned long long)t_acc[1];
        d[9] = (unsigned long long)(clock64() - t_loop0);
      }
    }
  } else if (warp >= 2 + 8) {
    // ===== pre-activation transform (launched only when p.xf_scale is set): relu(x * scale + shift) in place on every A
    // tile, between its TMA completion and the MMA.  Thread t owns the 16-byte chunk of logical channels 8 (t % 8) .. +7 in
    // rows t / 8 + 16 i: its eight scales and shifts live in registers for the whole K block, a warp touches 512
    // contiguous bytes per access (conflict-free), and the arithmetic is the pack kernel's (fmaf, fmaxf, round to nearest).
    if (xform) {
      const int t = (int)threadIdx.x - 32 * (2 + 8);
      const int cl = t & 7, rb = t >> 3;
      const uint32_t lead_xf0 = mapa_shared(xf_bar(0), 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = pair; tile < total_tiles; tile += npairs) {
        for (int kk = 0; kk < p.num_k_blocks; ++kk) {
          const float4 s0 = __ldg(reinterpret_cast<const float4*>(p.xf_scale + kk * TC_BLOCK_K + 8 * cl));
          const float4 s1 = __ldg(reinterpret_cast<const float4*>(p.xf_scale + kk * TC_BLOCK_K + 8 * cl + 4));
          const float4 h0 = __ldg(reinterpret_cast<const float4*>(p.xf_shift + kk * TC_BLOCK_K + 8 * cl));
          const float4 h1 = __ldg(reinterpret_cast<const float4*>(p.xf_shift + kk * TC_BLOCK_K + 8 * cl + 4));
          mbar_wait(afull_bar(stage), phase, p.err_flag, 9);
          const uint32_t a_addr = smem_base + stage * SM::STAGE_BYTES;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = rb + 16 * i;
            const uint32_t addr = a_addr + (uint32_t)r * 128u + ((uint32_t)(cl ^ (r & 7)) << 4);
            const uint4 raw = lds_v4(addr);
            const __nv_bfloat162* v = reinterpret_cast<const __nv_bfloat162*>(&raw);
            const float2 a = __bfloat1622float2(v[0]), b = __bfloat1622float2(v[1]), c = __bfloat1622float2(v[2]), d = __bfloat1622float2(v[3]);
            uint4 o;
            __nv_bfloat162 q;
            q = __floats2bfloat162_rn(fmaxf(fmaf(a.x, s0.x, h0.x), 0.f), fmaxf(fmaf(a.y, s0.y, h0.y), 0.f)); o.x = *reinterpret_cast<uint32_t*>(&q);
            q = __floats2bfloat162_rn(fmaxf(fmaf(b.x, s0.z, h0.z), 0.f), fmaxf(fmaf(b.y, s0.w, h0.w), 0.f)); o.y = *reinterpret_cast<uint32_t*>(&q);
            q = __floats2bfloat162_rn(fmaxf(fmaf(c.x, s1.x, h1.x), 0.f), fmaxf(fmaf(c.y, s1.y, h1.y), 0.f)); o.z = *reinterpret_cast<uint32_t*>(&q);
            q = __floats2bfloat162_rn(fmaxf(fmaf(d.x, s1.z, h1.z), 0.f), fmaxf(fmaf(d.y, s1.w, h1.w), 0.f)); o.w = *reinterpret_cast<uint32_t*>(&q);
            sts_v4(addr, o);
          }
          fence_async_smem();     // generic-proxy writes -> visible to tcgen05.mma (async proxy)
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(lead_xf0 + 8u * stage);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else {
    // ===== epilogue: 8 warps per CTA, every warp an independent pipeline =====
    // A warp drains its 32 TMEM lanes (= 32 output rows) of the columns its warpgroup owns, 64 channels at a time:
    // tcgen05.ld -> bias / residual / ReLU (packed) -> swizzled 4 KB smem slab -> its own 32-row TMA store.  No
    // warp waits for another one except for the once-per-tile bias hand-over inside its warpgroup.
    const int ew = warp - 2;
    const int g = ew >> 2;
    const int quarter = warp & 3;                          // TMEM lane quarter this warp may read
    const uint32_t sw = (uint32_t)(lane & 7);
    const int wt = (int)threadIdx.x - 64 - g * 128;        // 0..127 inside the warpgroup
    const uint32_t lead_empty0 = mapa_shared(tmem_empty_bar(0), 0);
    const uint32_t lead_empty1 = mapa_shared(tmem_empty_bar(1), 0);
    const bool has_bias = p.bias != nullptr;
    const uint32_t relu_floor = p.relu ? 0u : 0xFF80FF80u; // max.bf16x2 against (0,0) or (-inf,-inf)
    const int colbase = SM::SPLIT_COLS ? g * SM::CW : 0;   // first tile column of this warpgroup
    const uint32_t bias_wg = smem_base + SM::BIAS_OFFSET + (uint32_t)(g * 2 * SM::CW * 4);
    const int rows_here = p.tile_rows - quarter * 32;      // valid rows of this warp's slab (stem tiles have 112 rows)
    const int step = SM::SPLIT_COLS ? npairs : 2 * npairs;
    int it = SM::SPLIT_COLS ? 0 : g;
    int lt = 0;
    int tile = SM::SPLIT_COLS ? pair : pair + g * npairs;
    // With ~225 KB of the SM carved out as shared memory there is no L1 to speak of: the tile's bias slice is fetched
    // one tile ahead into a register, parked in smem and read back as broadcast LDS.128.
    // halo mode: TMEM lane i is raster position i of the padded-width tile; its dense output row (junk columns dropped)
    const bool halo = BRES && !HAS_RES && !SPLIT && p.a_mode == TC_A_HALO;
    bool halo_valid = false;
    uint32_t halo_base = 0, halo_sw = 0;
    if (halo) {
      const int i = quarter * 32 + lane;
      const int y = i / p.halo_wp, x = i - y * p.halo_wp;
      halo_valid = y < p.halo_r && x < p.Q;
      const int ip = y * p.Q + x;
      if (p.halo_n == 32) {   // 32 channels = 64 B rows under the 64B swizzle (16-byte chunk ^= address bits 7..8)
        halo_base = box_addr(g) + (uint32_t)ip * 64u;
        halo_sw = (uint32_t)((ip >> 1) & 3);
      } else {
        halo_base = box_addr(g) + (uint32_t)ip * 128u;
        halo_sw = (uint32_t)(ip & 7);
      }
    }
    float bias_pre = 0.f;
    const int bias_cols = (BRES && p.a_mode == TC_A_HALO) ? p.halo_n : SM::CW;   // the resident-patch mode may have only 32 outputs
    if (has_bias && wt < bias_cols && tile < total_tiles) bias_pre = __ldg(p.bias + (tile % p.n_tiles) * BLOCK_N + colbase + wt);
    if (dbg_on) t_loop0 = clock64();
    for (; tile < total_tiles; tile += step, it += (SM::SPLIT_COLS ? 1 : 2), ++lt) {
      const int n_tile = tile % p.n_tiles;
      const int mp = tile / p.n_tiles;
      const int m_tile = p.a_mode == TC_A_RAW ? (mp / p.col_tiles) * 2 + (int)rank : mp * 2 + (int)rank;
      const int m0 = p.a_mode == TC_A_RAW ? (m_tile * p.col_tiles + mp % p.col_tiles) * p.tile_rows : m_tile * p.tile_rows;
      const int n0 = n_tile * BLOCK_N;
      const int ab = it & 1;
      TC3_TIMED(0, mbar_wait(tmem_full_bar(ab), (uint32_t)((it >> 1) & 1), p.err_flag, 3));
      tc_fence_after();
      const uint32_t bias_s = bias_wg + (uint32_t)((lt & 1) * SM::CW * 4);
      if (has_bias) {
        if (wt < SM::CW) asm volatile("st.shared.f32 [%0], %1;" ::"r"(bias_s + 4u * wt), "f"(bias_pre) : "memory");
        TC3_TIMED(3, named_bar_sync(1 + g, 128));
        const int nt = tile + step;
        if (wt < bias_cols && nt < total_tiles) bias_pre = __ldg(p.bias + (nt % p.n_tiles) * BLOCK_N + colbase + wt);
      }
      const int set = it % SM::RSETS;
      const uint32_t rpar = (uint32_t)((it / SM::RSETS) & 1);
#pragma unroll 1
      for (int u = 0; u < SM::UNITS; ++u) {
        const int b = SM::SPLIT_COLS ? g * SM::UNITS + u : 0;                   // output box (64 channels) of the tile
        const int buf = set * SM::RBOX + b;                                    // residual/output box (HAS_RES)
        const uint32_t slab = HAS_RES ? box_addr(buf) + (uint32_t)(quarter * 4096)
                                      : smem_base + SM::BOX_OFFSET + (uint32_t)(ew * 4096);
        const uint32_t obase = slab + (uint32_t)lane * 128u;
        if (HAS_RES) TC3_TIMED(1, mbar_wait(res_full_bar(buf), rpar, p.err_flag, 6));
        if (HAS_RES && SPLIT) TC3_TIMED(1, mbar_wait(res_full_bar(buf + SM::NBOX), rpar, p.err_flag, 6));
        uint32_t v[64];
        __syncwarp();
        tmem_ld_32x32b_x64(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(ab * BLOCK_N + b * 64), v);
        tmem_ld_wait();
        if (u == SM::UNITS - 1) {    // this warp has read its whole share of the accumulator
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(ab ? lead_empty1 : lead_empty0);
        }
        if constexpr (SPLIT) {
          // fp32 result -> (hi, lo) bf16 halves.  hi goes to the hi box / the private slab, lo to the lo box / the same slab
          // once the hi store has read it; the residual is the sum of its own two halves, added in fp32.
          const int buf_lo = buf + SM::NBOX;
          const uint32_t slab_lo = HAS_RES ? box_addr(buf_lo) + (uint32_t)(quarter * 4096) : slab;
          const uint32_t obase_lo = slab_lo + (uint32_t)lane * 128u;
          const uint32_t bsrc = bias_s + (uint32_t)(u * 64 * 4);
          uint32_t lo[32];
          if (!HAS_RES) {
            if (lane == 0) bulk_wait_read<0>();
            __syncwarp();
          }
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            float x[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) x[j] = __uint_as_float(v[c * 8 + j]);
            if (has_bias) {
              const uint4 b0 = lds_v4(bsrc + (uint32_t)(c * 32)), b1 = lds_v4(bsrc + (uint32_t)(c * 32 + 16));
              x[0] += __uint_as_float(b0.x); x[1] += __uint_as_float(b0.y); x[2] += __uint_as_float(b0.z); x[3] += __uint_as_float(b0.w);
              x[4] += __uint_as_float(b1.x); x[5] += __uint_as_float(b1.y); x[6] += __uint_as_float(b1.z); x[7] += __uint_as_float(b1.w);
            }
            const uint32_t swz = (((uint32_t)c) ^ sw) << 4;
            if (HAS_RES) {
              const uint4 rh = lds_v4(obase + swz), rl = lds_v4(obase_lo + swz);
              const uint32_t h4[4] = {rh.x, rh.y, rh.z, rh.w}, l4[4] = {rl.x, rl.y, rl.z, rl.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                x[2 * j] += __uint_as_float(h4[j] << 16) + __uint_as_float(l4[j] << 16);
                x[2 * j + 1] += __uint_as_float(h4[j] & 0xFFFF0000u) + __uint_as_float(l4[j] & 0xFFFF0000u);
              }
            }
            if (p.relu) {
#pragma unroll
              for (int j = 0; j < 8; ++j) x[j] = fmaxf(x[j], 0.f);
            }
            uint32_t h[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(h[j]) : "f"(x[2 * j + 1]), "f"(x[2 * j]));
              const float r0 = x[2 * j] - __uint_as_float(h[j] << 16), r1 = x[2 * j + 1] - __uint_as_float(h[j] & 0xFFFF0000u);
              asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo[c * 4 + j]) : "f"(r1), "f"(r0));
            }
            sts_v4(obase + swz, make_uint4(h[0], h[1], h[2], h[3]));
          }
          fence_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tmOut, slab, p.out_coff + n0 + b * 64, m0 + quarter * 32);
            bulk_commit();
            if (!HAS_RES) bulk_wait_read<0>();     // the slab is about to be overwritten with the lo half
          }
          __syncwarp();
#pragma unroll
          for (int c = 0; c < 8; ++c)
            sts_v4(obase_lo + ((((uint32_t)c) ^ sw) << 4), make_uint4(lo[c * 4], lo[c * 4 + 1], lo[c * 4 + 2], lo[c * 4 + 3]));
          fence_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tmOut, slab_lo, p.out_coff + p.lo_off_out + n0 + b * 64, m0 + quarter * 32);
            bulk_commit();
            if (HAS_RES) {
              bulk_wait_read<0>();
              mbar_arrive(box_free_bar(buf));
              mbar_arrive(box_free_bar(buf_lo));
            }
          }
          continue;
        }
        uint32_t o[32];
        const uint32_t bsrc = bias_s + (uint32_t)(u * 64 * 4);
#pragma unroll
        for (int c = 0; c < 8; ++c) {          // 8 chunks of 8 channels (16 B of bf16)
          uint64_t a0 = pack_f32x2(v[c * 8 + 0], v[c * 8 + 1]), a1 = pack_f32x2(v[c * 8 + 2], v[c * 8 + 3]);
          uint64_t a2 = pack_f32x2(v[c * 8 + 4], v[c * 8 + 5]), a3 = pack_f32x2(v[c * 8 + 6], v[c * 8 + 7]);
          if (has_bias) {
            const uint4 b0 = lds_v4(bsrc + (uint32_t)(c * 32)), b1 = lds_v4(bsrc + (uint32_t)(c * 32 + 16));
            a0 = add_f32x2(a0, pack_f32x2(b0.x, b0.y)); a1 = add_f32x2(a1, pack_f32x2(b0.z, b0.w));
            a2 = add_f32x2(a2, pack_f32x2(b1.x, b1.y)); a3 = add_f32x2(a3, pack_f32x2(b1.z, b1.w));
          }
          if (HAS_RES) {
            const uint4 r = lds_v4(obase + ((((uint32_t)c) ^ sw) << 4));   // 8 bf16 residual values of this row
            a0 = add_f32x2(a0, pack_f32x2(r.x << 16, r.x & 0xFFFF0000u)); a1 = add_f32x2(a1, pack_f32x2(r.y << 16, r.y & 0xFFFF0000u));
            a2 = add_f32x2(a2, pack_f32x2(r.z << 16, r.z & 0xFFFF0000u)); a3 = add_f32x2(a3, pack_f32x2(r.w << 16, r.w & 0xFFFF0000u));
          }
          o[c * 4 + 0] = max_bf16x2(cvt_bf16x2(a0), relu_floor); o[c * 4 + 1] = max_bf16x2(cvt_bf16x2(a1), relu_floor);
          o[c * 4 + 2] = max_bf16x2(cvt_bf16x2(a2), relu_floor); o[c * 4 + 3] = max_bf16x2(cvt_bf16x2(a3), relu_floor);
        }
        if (halo) {
          // the warpgroup's four slabs are one 128-row staging box: rows land compacted at their dense index and ONE
          // store of tile_rows rows leaves per tile (issued by the warpgroup's first lane, which also owns the drain)
          if (quarter == 0 && lane == 0) TC3_TIMED(2, bulk_wait_read<0>());
          TC3_TIMED(3, named_bar_sync(1 + g, 128));
          if (halo_valid) {
#pragma unroll
            for (int c = 0; c < 8; ++c)
              if (c < 4 || p.halo_n == 64)
                sts_v4(halo_base + ((((uint32_t)c) ^ halo_sw) << 4), make_uint4(o[c * 4], o[c * 4 + 1], o[c * 4 + 2], o[c * 4 + 3]));
          }
          fence_async_smem();
          TC3_TIMED(3, named_bar_sync(1 + g, 128));
          if (quarter == 0 && lane == 0) {
            tma_store_2d(&tmOutTail, box_addr(g), p.out_coff + n0, m0);
            bulk_commit();
          }
          continue;
        }
        if (!HAS_RES) {              // private slab: the previous store of this warp must have read it
          if (lane == 0) TC3_TIMED(2, bulk_wait_read<0>());
          __syncwarp();
        }
#pragma unroll
        for (int c = 0; c < 8; ++c)
          sts_v4(obase + ((((uint32_t)c) ^ sw) << 4), make_uint4(o[c * 4], o[c * 4 + 1], o[c * 4 + 2], o[c * 4 + 3]));
        fence_async_smem();   // generic-proxy smem writes -> visible to the TMA (async proxy)
        __syncwarp();
        if (lane == 0) {
          if (rows_here >= 32) tma_store_2d(&tmOut, slab, p.out_coff + n0 + b * 64, m0 + quarter * 32);
          else if (rows_here > 0) tma_store_2d(&tmOutTail, slab, p.out_coff + n0 + b * 64, m0 + quarter * 32);
          bulk_commit();
          if (HAS_RES) {
            // hand boxes back to the producer as soon as the store engine has read them
            if (u > 0) {
              TC3_TIMED(2, bulk_wait_read<1>());
              mbar_arrive(box_free_bar(buf - 1));
            }
            if (u == SM::UNITS - 1) {
              TC3_TIMED(2, bulk_wait_read<0>());
              mbar_arrive(box_free_bar(buf));
            }
          }
        }
      }
    }
    if (lane == 0) bulk_wait_read<0>();
    if (dbg_on && warp == 2 && lane == 0) {
      unsigned long long* d = p.dbg + (size_t)blockIdx.x * 16;
      d[4] = (unsigned long long)t_acc[0]; d[5] = (unsigned long long)t_acc[1];
      d[6] = (unsigned long long)t_acc[2]; d[7] = (unsigned long long)t_acc[3];
      d[10] = (unsigned long long)(clock64() - t_loop0);
      d[11] = (unsigned long long)lt;
    }
    tc_fence_before();
  }
#undef TC3_TIMED
  __syncthreads();
  cluster_sync_all();   // no CTA of the pair retires (or frees TMEM) while the other may still touch it
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
  if (dbg_on && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    p.dbg[(size_t)blockIdx.x * 16 + 13] = gt;
    p.dbg[(size_t)blockIdx.x * 16 + 15] = (unsigned long long)clock64();
  }
}


// =====================================================================================================
// Fused pair of 1x1 convolutions: a bottleneck's expansion c (K1 -> N1, + residual, ReLU) and the NEXT bottleneck's
// reduction a (N1 -> N2, ReLU), one kernel.  Run separately, the N1-channel tensor y is written by c and read back by a
// (103 MB per launch at micro-batch 256 in layer 3, the largest single stream of bytes in the network); here each
// 128-column chunk of y is converted to bf16 in shared memory once, TMA-stored to global (the next block's residual
// still needs it) AND consumed in place as the A operand of the second GEMM — the epilogue's swizzled 128 x 64 boxes are
// exactly a K-major SWIZZLE_128B UMMA operand.
//
//   per CTA pair and 256-row tile:   for chunk j of N1/128:
//     MMA1(j):  acc1[j&1] (128 TMEM columns, double buffered) = h[256 x K1] * Wc[chunk j]^T        (ring 1: A1 + B1)
//     EPI1(j):  + bias + residual (TMA-loaded into the staging set, added in place) -> ReLU -> bf16 staging set j&1
//               -> TMA store of y;  signals y_ready
//     MMA2(j):  acc2 (N2 columns) += y_chunk[256 x 128] * Wa[:, chunk j]^T                         (ring 2: B2)
//   EPI2: acc2 + bias -> ReLU -> bf16 -> (the warpgroup's own staging set) -> TMA store.
// TMEM: 2 x 128 + N2 <= 512 columns.  Warp roles as in conv_tc3_kernel; warpgroup g of the epilogue owns the chunks of
// parity g, TMEM buffer g and staging set g, and half of the N2 output columns.
struct TcFusedParams {
  const float* bias1;
  const float* bias2;
  const __nv_bfloat16* res;   // residual [M][N1], compact
  int M, m_tiles;
  int kb1;      // K1 / 64
  int nch;      // N1 / 128 (even)
  int n1;
  int relu1, relu2;
  unsigned int* err_flag;
  unsigned long long* dbg;   // NIB_TC_DBG=1: per-CTA wait timers (cycles), 32 slots per CTA; null in production
};

template <int N2>
struct TcFusedSmem {
  static constexpr int S1 = 4, S2 = 4;                               // one chunk of B1, two chunks of B2
  static constexpr int A1_BYTES = TC_BLOCK_M * TC_BLOCK_K * 2;       // 16 KB per K block
  static constexpr int A1_KB = 4;                                    // K1 <= 256: the tile's whole A operand stays resident
  static constexpr int B1_BYTES = 64 * TC_BLOCK_K * 2;               // this CTA's 64 of the chunk's 128 weight rows
  static constexpr int B2_BYTES = (N2 / 2) * TC_BLOCK_K * 2;         // this CTA's half of Wa's rows, one K block
  static constexpr int BOX_BYTES = TC_BLOCK_M * 128;                 // 128 rows x 64 channels bf16
  static constexpr int R1_OFFSET = A1_KB * A1_BYTES;                 // ring 1: B1 only
  static constexpr int R2_OFFSET = R1_OFFSET + S1 * B1_BYTES;
  static constexpr int STG_OFFSET = R2_OFFSET + S2 * B2_BYTES;       // [set 2][box 2] x 16 KB
  static constexpr int BIAS1_OFFSET = STG_OFFSET + 4 * BOX_BYTES;    // [warpgroup][128] floats: the current chunk's bias
  static constexpr int BIAS2_OFFSET = BIAS1_OFFSET + 2 * 128 * 4;
  static constexpr int BAR_OFFSET = BIAS2_OFFSET + N2 * 4;
  static constexpr int NUM_BARS = 2 * S1 + 2 * S2 + 14;
  static constexpr int TOTAL = BAR_OFFSET + NUM_BARS * 8 + 16;
  static constexpr int EP2_WARPS = N2 / 16;                          // epilogue warps per CTA that drain acc2 (4 per 64 columns)
};

// 2 control warps + 16 epilogue warps: the kernel is bound by its epilogue (80 warp-boxes of ~2.6 kcycles per 128-row tile),
// whose cost is latency, not issue slots, so the fix is more warps in flight; 32-column TMEM loads keep them under the
// 113 registers a 576-thread block may use.
static constexpr int TCF_THREADS = 64 + 512;
template <int N2>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TCF_THREADS, 1)
conv_fused_ca_kernel(const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmB1,
                     const __grid_constant__ CUtensorMap tmRes, const __grid_constant__ CUtensorMap tmY,
                     const __grid_constant__ CUtensorMap tmB2, const __grid_constant__ CUtensorMap tmOut2,
                     const TcFusedParams p) {
  using SM = TcFusedSmem<N2>;
  constexpr int S1 = SM::S1, S2 = SM::S2;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = smem_u32(smem_raw);
  if ((smem_base & 1023u) != 0) {
    if (threadIdx.x == 0 && p.err_flag) atomicExch(p.err_flag, 9u);
    __trap();
  }
  const uint32_t bar_base = smem_base + SM::BAR_OFFSET;
  auto full1 = [&](int s) { return bar_base + 8u * s; };                       // leader
  auto empty1 = [&](int s) { return bar_base + 8u * (S1 + s); };
  auto full2 = [&](int s) { return bar_base + 8u * (2 * S1 + s); };            // leader
  auto empty2 = [&](int s) { return bar_base + 8u * (2 * S1 + S2 + s); };
  const uint32_t bar2 = bar_base + 8u * (2 * S1 + 2 * S2);
  auto acc1_full = [&](int b) { return bar2 + 8u * b; };
  auto acc1_empty = [&](int b) { return bar2 + 8u * (2 + b); };                // leader
  auto res_full = [&](int b) { return bar2 + 8u * (4 + b); };
  auto y_ready = [&](int b) { return bar2 + 8u * (6 + b); };                   // leader
  auto stage_free = [&](int b) { return bar2 + 8u * (8 + b); };
  const uint32_t acc2_full = bar2 + 8u * 10;
  const uint32_t acc2_empty = bar2 + 8u * 11;                                  // leader
  const uint32_t a1_full = bar2 + 8u * 12;                                     // leader
  const uint32_t a1_empty = bar2 + 8u * 13;
  const uint32_t tmem_slot = bar_base + 8u * SM::NUM_BARS;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_base));
  auto stg = [&](int set, int box) { return smem_base + SM::STG_OFFSET + (uint32_t)(set * 2 + box) * SM::BOX_BYTES; };
  float* bias1_s = reinterpret_cast<float*>(smem_raw + SM::BIAS1_OFFSET);
  float* bias2_s = reinterpret_cast<float*>(smem_raw + SM::BIAS2_OFFSET);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1;
  const int npairs = gridDim.x >> 1;
  const int m_pairs = (p.m_tiles + 1) >> 1;
  constexpr uint32_t TMEM_COLS = 512;
  constexpr uint32_t ACC2_COL = 256;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA1); prefetch_tmap(&tmB1); prefetch_tmap(&tmRes);
    prefetch_tmap(&tmY); prefetch_tmap(&tmB2); prefetch_tmap(&tmOut2);
    for (int s = 0; s < S1; ++s) { mbar_init(full1(s), 1); mbar_init(empty1(s), 1); }
    for (int s = 0; s < S2; ++s) { mbar_init(full2(s), 1); mbar_init(empty2(s), 1); }
    for (int b = 0; b < 2; ++b) {
      mbar_init(acc1_full(b), 1);
      mbar_init(acc1_empty(b), 16);    // 8 warps (both boxes of the chunk) in each CTA
      mbar_init(res_full(b), 1);
      mbar_init(y_ready(b), 16);
      mbar_init(stage_free(b), 9);     // MMA2 commit + the 8 warps whose stores read the set
    }
    mbar_init(acc2_full, 1);
    mbar_init(acc2_empty, 2 * SM::EP2_WARPS);
    mbar_init(a1_full, 1);
    mbar_init(a1_empty, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  // biases are weights: safe to read before the previous layer has finished
  for (int i = threadIdx.x; i < N2; i += blockDim.x) bias2_s[i] = p.bias2 ? p.bias2[i] : 0.f;
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  const bool dbg_on = p.dbg != nullptr;
  long long t_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const long long t_role0 = clock64();
#define FT(slot, stmt)                                                                      \
  do {                                                                                      \
    if (dbg_on) { const long long _t = clock64(); stmt; t_acc[slot] += clock64() - _t; }    \
    else { stmt; }                                                                          \
  } while (0)
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp == 0) {
    // ===== TMA producer (both CTAs) =====
    int s1 = 0, s2 = 0;
    uint32_t ph1 = 0, ph2 = 0;
    const uint32_t lfull1 = mapa_shared(full1(0), 0), lfull2 = mapa_shared(full2(0), 0);
    const uint32_t la1_full = mapa_shared(a1_full, 0);
    int it = 0;
    for (int tile = pair; tile < m_pairs; tile += npairs, ++it) {
      const int m0 = (tile * 2 + (int)rank) * TC_BLOCK_M;
      // the tile's A operand (128 rows x K1) is loaded once and reused by every chunk: re-streaming it per chunk made A
      // 40 % of all bytes the SM had to receive, and the kernel is bound by exactly that
      FT(0, mbar_wait(a1_empty, ((uint32_t)it & 1u) ^ 1u, p.err_flag, 32));
      if (elect_one()) {
        if (rank == 0) mbar_arrive_expect_tx(a1_full, (uint32_t)(2 * p.kb1 * SM::A1_BYTES));
        for (int kb = 0; kb < p.kb1; ++kb)
          tma2_load_2d(smem_base + (uint32_t)kb * SM::A1_BYTES, &tmA1, la1_full, kb * TC_BLOCK_K, m0);
      }
      __syncwarp();
      // issue order = consumption order of the MMA warp: MMA1(0), MMA1(1), MMA2(0), MMA1(2), MMA2(1), ...  (with B2 of chunk
      // j ahead of B1 of chunk j+1 the producer sat in the ring-2 wait while MMA1 starved: 60 % of the kernel time)
      auto issue_b1 = [&](int j) {
        for (int kb = 0; kb < p.kb1; ++kb) {
          FT(1, mbar_wait(empty1(s1), ph1 ^ 1u, p.err_flag, 22));
          if (elect_one()) {
            if (rank == 0) mbar_arrive_expect_tx(full1(s1), (uint32_t)(2 * SM::B1_BYTES));
            tma2_load_2d(smem_base + SM::R1_OFFSET + (uint32_t)s1 * SM::B1_BYTES, &tmB1, lfull1 + 8u * s1, kb * TC_BLOCK_K,
                         j * 128 + (int)rank * 64);
          }
          __syncwarp();
          if (++s1 == S1) { s1 = 0; ph1 ^= 1u; }
        }
      };
      auto issue_b2 = [&](int j) {
        for (int kk = 0; kk < 2; ++kk) {
          FT(2, mbar_wait(empty2(s2), ph2 ^ 1u, p.err_flag, 23));
          if (elect_one()) {
            const uint32_t dst = smem_base + SM::R2_OFFSET + (uint32_t)s2 * SM::B2_BYTES;
            if (rank == 0) mbar_arrive_expect_tx(full2(s2), (uint32_t)(2 * SM::B2_BYTES));
            tma2_load_2d(dst, &tmB2, lfull2 + 8u * s2, j * 128 + kk * TC_BLOCK_K, (int)rank * (N2 / 2));
          }
          __syncwarp();
          if (++s2 == S2) { s2 = 0; ph2 ^= 1u; }
        }
      };
      issue_b1(0);
      for (int j = 0; j < p.nch; ++j) {
        if (j + 1 < p.nch) issue_b1(j + 1);
        issue_b2(j);
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      // ===== MMA issuer (leader CTA only) =====
      constexpr uint32_t idesc1 = make_idesc_bf16_pair<128>();
      constexpr uint32_t idesc2 = make_idesc_bf16_pair<N2>();
      int s1 = 0, s2 = 0;
      uint32_t ph1 = 0, ph2 = 0;
      int it = 0;
      for (int tile = pair; tile < m_pairs; tile += npairs, ++it) {
        for (int j = 0; j <= p.nch; ++j) {
          if (j < p.nch) {
            const int b = j & 1;
            const uint32_t use = (uint32_t)((it * p.nch + j) >> 1);
            FT(0, mbar_wait(acc1_empty(b), (use & 1u) ^ 1u, p.err_flag, 24));
            if (j == 0) FT(1, mbar_wait(a1_full, (uint32_t)it & 1u, p.err_flag, 33));
            tc_fence_after();
            const uint32_t d1 = tmem_base + (uint32_t)(b * 128);
            for (int kb = 0; kb < p.kb1; ++kb) {
              FT(2, mbar_wait(full1(s1), ph1, p.err_flag, 25));
              tc_fence_after();
              if (elect_one()) {
                const uint64_t adesc = make_smem_desc_sw128(smem_base + (uint32_t)kb * SM::A1_BYTES);
                const uint64_t bdesc = make_smem_desc_sw128(smem_base + SM::R1_OFFSET + (uint32_t)s1 * SM::B1_BYTES);
#pragma unroll
                for (int k = 0; k < TC_BLOCK_K / TC_UMMA_K; ++k)
                  umma2_bf16(d1, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc1, (kb | k) != 0);
                umma2_commit_both(empty1(s1));
                if (kb == p.kb1 - 1) {
                  umma2_commit_both(acc1_full(b));
                  if (j == p.nch - 1) umma2_commit_both(a1_empty);     // the next tile's A may land
                }
              }
              __syncwarp();
              if (++s1 == S1) { s1 = 0; ph1 ^= 1u; }
            }
          }
          if (j >= 1) {
            const int jj = j - 1, b = jj & 1;
            const uint32_t use = (uint32_t)((it * p.nch + jj) >> 1);
            FT(3, mbar_wait(y_ready(b), use & 1u, p.err_flag, 26));
            if (jj == 0) FT(4, mbar_wait(acc2_empty, ((uint32_t)it & 1u) ^ 1u, p.err_flag, 27));
            tc_fence_after();
            const uint32_t d2 = tmem_base + ACC2_COL;
            for (int kk = 0; kk < 2; ++kk) {
              FT(5, mbar_wait(full2(s2), ph2, p.err_flag, 28));
              tc_fence_after();
              if (elect_one()) {
                const uint64_t adesc = make_smem_desc_sw128(stg(b, kk));
                const uint64_t bdesc = make_smem_desc_sw128(smem_base + SM::R2_OFFSET + (uint32_t)s2 * SM::B2_BYTES);
#pragma unroll
                for (int k = 0; k < TC_BLOCK_K / TC_UMMA_K; ++k)
                  umma2_bf16(d2, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc2, (jj | kk | k) != 0);
                umma2_commit_both(empty2(s2));
                if (kk == 1) {
                  umma2_commit_both(stage_free(b));
                  if (jj == p.nch - 1) umma2_commit_both(acc2_full);
                }
              }
              __syncwarp();
              if (++s2 == S2) { s2 = 0; ph2 ^= 1u; }
            }
          }
        }
      }
    }
  } else {
    // ===== epilogue: 4 warpgroups.  Warpgroup G owns box h = G >> 1 (64 of the chunk's 128 columns) of the chunks of
    // parity g = G & 1 (TMEM buffer g, staging set g), and 64 of the N2 output columns. =====
    const int ew = warp - 2;
    const int G = ew >> 2;
    const int g = G & 1, h = G >> 1;
    const int quarter = warp & 3;
    const uint32_t sw = (uint32_t)(lane & 7);
    const uint32_t lead_acc1_empty = mapa_shared(acc1_empty(g), 0);
    const uint32_t lead_y_ready = mapa_shared(y_ready(g), 0);
    const uint32_t lead_acc2_empty = mapa_shared(acc2_empty, 0);
    const uint32_t relu1_floor = p.relu1 ? 0u : 0xFF80FF80u;
    const uint32_t relu2_floor = p.relu2 ? 0u : 0xFF80FF80u;
    const bool ep2 = G * 64 < N2;                        // this warpgroup drains columns [G*64, G*64+64) of acc2
    const uint32_t lane_taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const uint32_t slab = stg(g, h) + (uint32_t)(quarter * 4096);
    const uint32_t obase = slab + (uint32_t)lane * 128u;
    // one lane per parity fetches the set's residual chunk the moment the set is free again (its eight warps' stores have
    // read it and MMA2 has consumed it); the residual is added in place in the staging set
    auto fetch_residual = [&](uint32_t use_next, int j_next, int m0_next) {
      if (h == 0 && quarter == 0 && lane == 0) {
        FT(0, mbar_wait(stage_free(g), (use_next & 1u) ^ 1u, p.err_flag, 21));
        mbar_arrive_expect_tx(res_full(g), (uint32_t)(2 * SM::BOX_BYTES));
        tma_load_2d(stg(g, 0), &tmRes, res_full(g), j_next * 128, m0_next);
        tma_load_2d(stg(g, 1), &tmRes, res_full(g), j_next * 128 + 64, m0_next);
        if (j_next + 2 < p.nch) {   // the chunk after that one: have it in L2 by the time its load is issued
          tma_prefetch_2d(&tmRes, (j_next + 2) * 128, m0_next);
          tma_prefetch_2d(&tmRes, (j_next + 2) * 128 + 64, m0_next);
        }
      }
      __syncwarp();
    };
    const int wt = h * 128 + ((int)threadIdx.x - 64 - G * 128);    // 0..255 inside the parity group
    float* bias1_wg = bias1_s + g * 128;
    // 32 accumulator columns -> bias (+ residual, in place) -> ReLU -> bf16 -> the slab's 16-byte chunks cbase..cbase+3
    auto drain32 = [&](uint32_t taddr, const float* bsrc, int cbase, bool with_res, uint32_t floor_) {
      uint32_t v[32];
      tmem_ld_32x32b_x32(taddr, v);
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint64_t a0 = pack_f32x2(v[c * 8 + 0], v[c * 8 + 1]), a1 = pack_f32x2(v[c * 8 + 2], v[c * 8 + 3]);
        uint64_t a2 = pack_f32x2(v[c * 8 + 4], v[c * 8 + 5]), a3 = pack_f32x2(v[c * 8 + 6], v[c * 8 + 7]);
        const float4 b0 = *reinterpret_cast<const float4*>(bsrc + c * 8), b1 = *reinterpret_cast<const float4*>(bsrc + c * 8 + 4);
        a0 = add_f32x2(a0, pack_f32x2(__float_as_uint(b0.x), __float_as_uint(b0.y)));
        a1 = add_f32x2(a1, pack_f32x2(__float_as_uint(b0.z), __float_as_uint(b0.w)));
        a2 = add_f32x2(a2, pack_f32x2(__float_as_uint(b1.x), __float_as_uint(b1.y)));
        a3 = add_f32x2(a3, pack_f32x2(__float_as_uint(b1.z), __float_as_uint(b1.w)));
        const uint32_t addr = obase + ((((uint32_t)(cbase + c)) ^ sw) << 4);
        if (with_res) {
          const uint4 r = lds_v4(addr);                                  // 8 bf16 residual values of this row
          a0 = add_f32x2(a0, pack_f32x2(r.x << 16, r.x & 0xFFFF0000u)); a1 = add_f32x2(a1, pack_f32x2(r.y << 16, r.y & 0xFFFF0000u));
          a2 = add_f32x2(a2, pack_f32x2(r.z << 16, r.z & 0xFFFF0000u)); a3 = add_f32x2(a3, pack_f32x2(r.w << 16, r.w & 0xFFFF0000u));
        }
        sts_v4(addr, make_uint4(max_bf16x2(cvt_bf16x2(a0), floor_), max_bf16x2(cvt_bf16x2(a1), floor_),
                                max_bf16x2(cvt_bf16x2(a2), floor_), max_bf16x2(cvt_bf16x2(a3), floor_)));
      }
    };
    if (pair < m_pairs) fetch_residual(0u, g, (pair * 2 + (int)rank) * TC_BLOCK_M);
    float bias_next = (wt < 128 && p.bias1) ? __ldg(p.bias1 + g * 128 + wt) : 0.f;
    int it = 0;
    for (int tile = pair; tile < m_pairs; tile += npairs, ++it) {
      const int m0 = (tile * 2 + (int)rank) * TC_BLOCK_M;
      const bool more_tiles = tile + npairs < m_pairs;
      const int m0_next = ((tile + npairs) * 2 + (int)rank) * TC_BLOCK_M;
      for (int j = g; j < p.nch; j += 2) {
        const uint32_t use = (uint32_t)((it * p.nch + j) >> 1);
        // this chunk's 128 bias values into the parity group's window (256 threads; the barrier pair orders the write
        // against the previous chunk's readers and publishes it)
        const float bias_reg = bias_next;
        named_bar_sync(1 + g, 256);
        if (wt < 128) bias1_wg[wt] = bias_reg;
        named_bar_sync(1 + g, 256);
        {   // the NEXT chunk's bias is fetched now: a load issued at the top of its own chunk sat on the critical path
          const int jn = (j + 2 < p.nch) ? j + 2 : g;
          bias_next = (wt < 128 && p.bias1) ? __ldg(p.bias1 + jn * 128 + wt) : 0.f;
        }
        FT(1, mbar_wait(res_full(g), use & 1u, p.err_flag, 29));
        FT(2, mbar_wait(acc1_full(g), use & 1u, p.err_flag, 30));
        tc_fence_after();
        __syncwarp();
        FT(6, drain32(lane_taddr + (uint32_t)(g * 128 + h * 64), bias1_wg + h * 64, 0, true, relu1_floor));
        FT(6, drain32(lane_taddr + (uint32_t)(g * 128 + h * 64 + 32), bias1_wg + h * 64 + 32, 4, true, relu1_floor));
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(lead_acc1_empty);
        FT(4, fence_async_smem());   // generic-proxy writes -> visible to the TMA store and to tcgen05.mma (async proxy)
        __syncwarp();
        if (lane == 0) {
          // Signal first, store second, and a plain (CTA-scope release) remote arrive: `arrive.release.cluster` issued
          // behind the bulk store cost ~3 kcycles per chunk and was the largest single item of the epilogue's time
          // (118 -> 110 kcycles per launch by reordering, -> 94 with the plain arrive).  What orders the box against
          // MMA2 is the fence.proxy.async above — the tensor core of THIS SM reads this CTA's box through the async
          // proxy — followed in program order by the arrive; conv_tc3's cross-CTA handshakes use the same arrive.
          FT(5, mbar_arrive_remote(lead_y_ready));
          tma_store_2d(&tmY, slab, j * 128 + h * 64, m0 + quarter * 32);
          bulk_commit();
        }
        const bool defer = ep2 && (j + 2 >= p.nch);            // the slab is reused by EPI2 before the set goes back
        if (!defer) {
          if (lane == 0) {
            bulk_wait_read<0>();
            mbar_arrive(stage_free(g));
          }
          __syncwarp();
          if (j + 2 < p.nch) fetch_residual(use + 1u, j + 2, m0);
          else if (more_tiles) fetch_residual(use + 1u, g, m0_next);
        }
      }
      if (ep2) {
        FT(3, mbar_wait(acc2_full, (uint32_t)it & 1u, p.err_flag, 31));
        tc_fence_after();
        if (lane == 0) bulk_wait_read<0>();     // the y store of this warp's last chunk has read the slab
        __syncwarp();
        const int col2 = G * 64;
        drain32(lane_taddr + ACC2_COL + (uint32_t)col2, bias2_s + col2, 0, false, relu2_floor);
        drain32(lane_taddr + ACC2_COL + (uint32_t)(col2 + 32), bias2_s + col2 + 32, 4, false, relu2_floor);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(lead_acc2_empty);
        fence_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tmOut2, slab, col2, m0 + quarter * 32);
          bulk_commit();
          bulk_wait_read<0>();
          mbar_arrive(stage_free(g));
        }
        __syncwarp();
      }
      // a warpgroup that took part in EPI2 handed its slab back only now: its parity's residual lane queues the next
      // tile's first chunk here (the others did so from inside the chunk loop)
      if (ep2 && more_tiles) fetch_residual((uint32_t)((it * p.nch + (p.nch - 2 + g)) >> 1) + 1u, g, m0_next);
    }
    if (lane == 0) bulk_wait_read<0>();
    tc_fence_before();
  }
#undef FT
  if (dbg_on && lane == 0 && (warp == 0 || warp == 1 || warp == 4 || warp == 8)) {
    // slots: producer 0-7, MMA 8-15, epilogue warpgroup 0 (its residual-issuing warp) 16-23, warpgroup 1 24-31;
    // entry 7 of each = the role's whole time
    const int role = warp == 0 ? 0 : warp == 1 ? 1 : warp == 4 ? 2 : 3;
    unsigned long long* d = p.dbg + (size_t)blockIdx.x * 32 + role * 8;
    for (int i = 0; i < 7; ++i) d[i] = (unsigned long long)t_acc[i];
    d[7] = (unsigned long long)(clock64() - t_role0);
  }
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ---- host side ----------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*PFN_encodeIm2col)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                     const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                     CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled g_encodeTiled = nullptr;
static PFN_encodeIm2col g_encodeIm2col = nullptr;
static unsigned int* g_err_flag = nullptr;

// driver entry points for the tensor maps and the kernels' shared error flag
static int init_tc() {
  if (!g_encodeTiled || !g_encodeIm2col) {
    cudaDriverEntryPointQueryResult q;
    void* fn = nullptr;
    NIB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || !fn) { set_error("cuTensorMapEncodeTiled not available"); return NIB_ECUDA; }
    g_encodeTiled = (PFN_encodeTiled)fn;
    fn = nullptr;
    NIB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || !fn) { set_error("cuTensorMapEncodeIm2col not available"); return NIB_ECUDA; }
    g_encodeIm2col = (PFN_encodeIm2col)fn;
  }
  if (!g_err_flag) {
    NIB_CUDA(cudaMalloc(&g_err_flag, sizeof(unsigned int)));
    NIB_CUDA(cudaMemset(g_err_flag, 0, sizeof(unsigned int)));
  }
  return NIB_OK;
}

typedef int (*TcLauncher)(const TcConvPlan* plan, const TcKernelParams& kp, cudaStream_t st);

struct TcConvPlan {
  CUtensorMap tmA, tmB, tmOut, tmRes;
  CUtensorMap tmBh;   // pair kernel: weight map with a BLOCK_N/2-row box (each CTA of the pair loads half of the tile)
  CUtensorMap tmOut32, tmOutTail;   // pair kernel: per-warp 32-row output boxes (+ the short last box of a 112-row stem tile)
  int v3;             // 1: the CTA-pair kernel serves this layer; 0: the one-CTA kernel (Cout = 32, NIB_TC_V1)
  int split;          // split-bf16 tensors: K = 3 x Cin per tap, both halves of the result are stored
  int block_n;
  TcKernelParams kp;  // every launch parameter except the batch-dependent M, m_tiles and dyn_n (tc_conv_launch)
  TcLauncher launch;  // the kernel instance (pick_instance)
};

static int encode_tiled_bf16(CUtensorMap* tm, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                             const cuuint32_t* box, CUtensorMapSwizzle swizzle) {
  const cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = g_encodeTiled(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(ptr), dims, strides, box, es,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): rank %d dims=(%llu,%llu,...) box=(%u,%u,...) swizzle %d ptr=%p", (int)r,
              rank, (unsigned long long)dims[0], (unsigned long long)dims[1], box[0], box[1], (int)swizzle, ptr);
    return NIB_ECUDA;
  }
  return NIB_OK;
}

static int encode_2d_bf16(CUtensorMap* tm, const void* ptr, uint64_t inner, uint64_t outer, uint64_t row_bytes,
                          uint32_t box_inner, uint32_t box_outer, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  const cuuint64_t dims[2] = {inner, outer};
  const cuuint64_t strides[1] = {row_bytes};
  const cuuint32_t box[2] = {box_inner, box_outer};
  return encode_tiled_bf16(tm, ptr, 2, dims, strides, box, swizzle);
}

// dims {inner, ..., outer}; strides in bytes of dims 1..3
static int encode_4d_bf16(CUtensorMap* tm, const void* ptr, const cuuint64_t (&dims)[4], const cuuint64_t (&strides)[3],
                          const cuuint32_t (&box)[4], CUtensorMapSwizzle swizzle) {
  return encode_tiled_bf16(tm, ptr, 4, dims, strides, box, swizzle);
}

RawRowLayout tc_raw_row_layout(int R, int S, int stride, int pad, int Cin, int in_cstride, int in_halo) {
  if (R == 7 && S == 7 && stride == 2 && pad == 3 && in_halo == 3) {
    if (in_cstride == 8 && Cin <= 8) return {7, 8, 8};   // stem on 8-channel pixels: a K block is one filter row
    if (in_cstride == 4 && Cin <= 4) return {8, 8, 4};   // on 4-channel pixels: two filter rows per K block, row 7 zero
  }
  if (R == 3 && S == 3 && stride == 1 && pad == 1 && in_halo == 1 && in_cstride == 8 && Cin <= 8)
    return {4, 4, 8};                                   // 3x3 first conv: a 32-element K atom per filter row, row 3 zero
  return {0, 0, 0};
}

static RawRowLayout raw_row_layout(const ConvParams& p) {
  return tc_raw_row_layout(p.R, p.S, p.stride, p.pad, p.Cin, p.in_cstride, p.in_halo);
}

// 7x7 stride-2 pad-3 stem on a haloed, 8-channel-padded NHWC input (torchvision conv1): for filter row r the 7 taps x 8
// channels of output pixel q are 56 contiguous elements starting at pixel 2q of input row 2p+r, so a tiled map whose
// pixel dimension advances 2 pixels (32 B) per index delivers a [Q x 64] K-major tile per filter row (8 zero-weight
// filler elements).  K = 7 x 64.
static bool tc_conv_is_stem(const ConvParams& p) {
  return raw_row_layout(p).rows == 7 && p.in_coff == 0 && p.Cout % 32 == 0 && p.Q <= TC_BLOCK_M && p.out_halo == 0 &&
         p.out_cstride % 8 == 0 && p.out_coff % 8 == 0 && p.pre_scale == nullptr && p.res == nullptr &&
         p.w_alt != nullptr && (p.Win + 2 * p.in_halo) >= 2 * (p.Q - 1) + 8;
}

// Same stem on 4-channel-padded pixels (8 B): a K block is TWO filter rows x (7 taps + 1 filler) x 4 channels.  Each
// filter row is its own 64B-swizzled K atom [Q pixels x 32 elements] (a 64 B inner box under the 128 B swizzle gets
// padded to 128 B rows by the copy engine, measured with tools/stem_diag.py, hence SWIZZLE_64B + matching UMMA
// descriptors).  K = 4 x 64 instead of 7 x 64: 43 % fewer activation bytes through the TMA and 43 % fewer MMAs.
// CTA-pair kernel with resident weights only.
static bool tc_conv_is_stem4(const ConvParams& p) {
  return raw_row_layout(p).rows == 8 && p.in_coff == 0 && p.Cout % 64 == 0 && p.Q <= TC_BLOCK_M && p.out_halo == 0 &&
         p.out_cstride % 8 == 0 && p.out_coff % 8 == 0 && p.pre_scale == nullptr && p.res == nullptr &&
         p.w_alt != nullptr && (p.Win + 2 * p.in_halo) % 2 == 0 && (p.Win + 2 * p.in_halo) >= 2 * (p.Q - 1) + 8 &&
         (p.Hin + 2 * p.in_halo) >= 2 * (p.P - 1) + 8;
}

// Raw-row TMA box of a padded row of row_el elements: {inner, row_el / inner} with a legal inner extent (a multiple of 8
// elements = 16 B, at most 256, dividing the row, at most 256 chunks); 0 if there is none.
static int raw_row_inner(int row_el) {
  for (int c = 256; c >= 8; c -= 8)
    if (row_el % c == 0 && row_el / c <= 256) return c;
  return 0;
}

// 3x3 raw rows: column tiles per output row.  One tile when the row fits the 128-row M tile; otherwise the smallest
// split into equal tiles of at most 128 columns, provided a tile keeps at least half of the MMA's rows busy.  0: no split.
static int raw3x3_col_tiles(int Q) {
  if (Q <= TC_BLOCK_M) return 1;
  for (int t = 2; Q / t >= TC_BLOCK_M / 2; ++t)
    if (Q % t == 0 && Q / t <= TC_BLOCK_M) return t;
  return 0;
}

// 3x3 stride-1 pad-1 first conv (VGG conv1_1) on 8-channel-padded pixels (16 B) inside a 1-pixel zero halo, TC_A_RAW:
// output pixel q of filter row r reads 3 taps x 8 channels starting at pixel q of padded row p + r, so each filter row is
// one 32-element K atom (3 taps + a zero-weight filler tap) of the overlapping-row operand the stem uses; K = 3 x 32, six
// MMAs per tile.  Weights [Cout][4][32] (row 3 zero), resident; Cout 64 or 128 (the resident-weight pair kernel holds one
// N tile).  The three rows of one image row (plus the filler's 16 B) must fit one 16 KB ring stage.
static bool tc_conv_is_raw3x3(const ConvParams& p) {
  static const bool off = getenv("NIB_TC_NO_HALO") != nullptr;
  if (off || p.split) return false;
  if (raw_row_layout(p).rows != 4 || p.in_coff != 0) return false;
  if (!(p.Cout == 64 || p.Cout == 128) || p.out_halo != 0 || p.out_cstride % 8 != 0 || p.out_coff % 8 != 0) return false;
  if (p.pre_scale != nullptr || p.res != nullptr || p.w_alt == nullptr || p.P != p.Hin || p.Q != p.Win) return false;
  const int t = raw3x3_col_tiles(p.Q);
  if (t == 0) return false;
  const int Wp = p.Win + 2, row_bytes = Wp * 16;
  if (3 * row_bytes + 16 > TC_BLOCK_M * TC_BLOCK_K * 2) return false;
  // the last MMA row of the last column tile reads 2 rows + 127 pixels + 64 B past the tile's first pixel
  if (2 * row_bytes + 16 * (p.Q - p.Q / t + TC_BLOCK_M - 1) + 64 > TC_BLOCK_M * TC_BLOCK_K * 2) return false;
  return raw_row_inner(Wp * 8) > 0;
}

// 3x3 stride-1 pad-1 convolution, 64 -> 64 channels, on the CTA-pair kernel with resident weights: the im2col path reads
// every input pixel nine times from L2 (16 KB per K block per SM against a ~43 B/clk/SM L2 port: 385 cycles per K block
// for 128 cycles of MMA), this one loads each tile's input patch once.  Whole image rows per tile, in the raster of the
// padded width; the junk columns cost 2 / (W + 2) of the MMA work.
// image rows per tile: the most that fit 128 raster positions of the padded width AND divide the image height (a tile never
// spans two images: the patch is one box of one image)
static int halo_rows_per_tile(int H, int Wp) {
  for (int r = TC_BLOCK_M / Wp; r >= 1; --r)
    if (H % r == 0) return r;
  return 0;
}
static bool tc_conv_is_halo3x3(const ConvParams& p) {
  static const bool off = getenv("NIB_TC_NO_HALO") != nullptr;
  if (off || p.split) return false;
  if (!(p.R == 3 && p.S == 3 && p.stride == 1 && p.pad == 1)) return false;
  // resident weights: 9 x (Cin / 64) K blocks of Cout / 2 rows must fit the 36 KB the 64-channel instance reserves
  if (!((p.Cin == 64 && (p.Cout == 64 || p.Cout == 32)) || (p.Cin == 128 && p.Cout == 32))) return false;
  if (p.res != nullptr || p.pre_scale != nullptr || p.in_halo != 0 || p.out_halo != 0) return false;
  if (p.in_cstride % 8 != 0 || p.in_coff % 8 != 0 || p.out_cstride % 8 != 0 || p.out_coff % 8 != 0) return false;
  if (p.P != p.Hin || p.Q != p.Win) return false;
  const int Wp = p.Win + 2;
  if (Wp > 63) return false;                    // the last tap's 128 rows must stay inside the 32 KB patch buffer
  const int R = halo_rows_per_tile(p.Hin, Wp);
  return R >= 1 && R * Wp >= 56;                // 7x7 images (one per tile, 63 of 128 rows real) still beat nine im2col boxes
}

bool tc_conv_supported(const ConvParams& p) {
  if (p.split) {
    // hi / lo halves must be adjacent (the K loop wraps from the lo blocks back to the hi blocks), 64-channel granularity
    if (p.Cin % TC_BLOCK_K != 0 || p.Cout % 64 != 0 || p.in_coff != 0 || p.out_coff != 0 || p.in_lo_off != p.Cin) return false;
    if (p.in_cstride != 2 * p.Cin || p.out_cstride < p.out_lo_off + p.Cout || p.out_lo_off % 64 != 0) return false;
    if (p.in_halo != 0 || p.out_halo != 0 || p.pre_scale != nullptr || p.R != p.S || p.pad > 127 || p.R > 16) return false;
    if (p.res != nullptr && (p.res_C != p.Cout || p.res_coff != 0 || p.res_lo_off % 64 != 0 || p.res_cstride < p.res_lo_off + p.Cout))
      return false;
    return true;
  }
  if (tc_conv_is_stem(p) || tc_conv_is_stem4(p) || tc_conv_is_raw3x3(p)) return true;
  if (p.Cin % TC_BLOCK_K != 0) return false;
  if (p.in_cstride % 8 != 0 || p.in_coff % 8 != 0) return false;   // 16 B TMA alignment
  if (p.Cout % 32 != 0) return false;
  if (p.out_cstride % 8 != 0 || p.out_coff % 8 != 0) return false;
  if (p.in_halo != 0 || p.out_halo != 0) return false;
  // pre-activation: only as the in-kernel transform of a 1x1 conv's A tiles on the pair kernel (scale / shift arrays
  // zero-padded to the K block by the caller, net.cu), never on the im2col / one-CTA paths
  if (p.pre_scale != nullptr && !(p.pre_padded && p.R == 1 && p.S == 1 && p.stride == 1 && p.pad == 0 && p.Cout % 64 == 0 &&
                                  p.res == nullptr))
    return false;
  if (p.res != nullptr && (p.res_C != p.Cout || p.res_cstride % 8 != 0 || p.res_coff % 8 != 0)) return false;
  if (p.R != p.S) return false;
  if (p.pad > 127 || p.R > 16) return false;
  return true;
}

// Widest tile the layer allows: 128 x 256 per CTA (256 x 256 per pair) - L2 -> SM fill is the limiter, and the pair
// kernel halves the weight bytes per output element.  Cout = 32 (DenseNet growth) stays on the one-CTA kernel.
static int pick_block_n(int Cout) {
  if (Cout % 256 == 0) return 256;
  if (Cout % 128 == 0) return 128;
  if (Cout % 64 == 0) return 64;
  return 32;
}

// the CTA-pair kernel's output, residual and half-width weight maps; leaves v3 = 0 (one-CTA kernel) where it does not apply
static int finish_plan(TcConvPlan* plan, const ConvParams& p, int max_batch, const void* w_ptr, int K) {
  plan->v3 = 0;
  static const bool v1_only = getenv("NIB_TC_V1") != nullptr;   // debugging aid: everything on the one-CTA kernel
  if (v1_only) return NIB_OK;
  const bool bn_ok = plan->block_n == 64 || plan->block_n == 128 || plan->block_n == 256;
  if (!bn_ok || p.Cout % plan->block_n != 0) return NIB_OK;
  const uint64_t rows = (uint64_t)max_batch * p.P * p.Q;
  const int tile_rows = plan->kp.tile_rows;
  int rc = encode_2d_bf16(&plan->tmOut, p.out, (uint64_t)p.out_cstride, rows, (uint64_t)p.out_cstride * 2, 64,
                          (uint32_t)tile_rows);
  if (rc != NIB_OK) return rc;
  if (p.res != nullptr) {
    rc = encode_2d_bf16(&plan->tmRes, p.res, (uint64_t)p.res_cstride, rows, (uint64_t)p.res_cstride * 2, 64, TC_BLOCK_M);
    if (rc != NIB_OK) return rc;
  } else {
    plan->tmRes = plan->tmOut;
  }
  rc = encode_2d_bf16(&plan->tmBh, w_ptr, (uint64_t)K, (uint64_t)p.Cout, (uint64_t)K * 2, TC_BLOCK_K,
                      (uint32_t)(plan->block_n / 2));
  if (rc != NIB_OK) return rc;
  rc = encode_2d_bf16(&plan->tmOut32, p.out, (uint64_t)p.out_cstride, rows, (uint64_t)p.out_cstride * 2, 64, 32);
  if (rc != NIB_OK) return rc;
  const int tail = tile_rows % 32;
  rc = encode_2d_bf16(&plan->tmOutTail, p.out, (uint64_t)p.out_cstride, rows, (uint64_t)p.out_cstride * 2, 64,
                      (uint32_t)(tail ? tail : 32));
  if (rc != NIB_OK) return rc;
  plan->v3 = 1;
  return NIB_OK;
}

// resident raw-row weights [Cout][K] as 64B-swizzled K atoms of 32 elements, BLOCK_N/2 rows per CTA, for both kernels
// (replaces finish_plan's map)
static int encode_raw_row_weights(TcConvPlan* plan, const ConvParams& p, int K) {
  int rc = encode_2d_bf16(&plan->tmBh, p.w_alt, (uint64_t)K, (uint64_t)p.Cout, (uint64_t)K * 2, 32,
                          (uint32_t)(plan->block_n / 2), CU_TENSOR_MAP_SWIZZLE_64B);
  plan->tmB = plan->tmBh;
  return rc;
}

// The A operand's tensor map and the mode's tile geometry (kp.a_mode, cblocks, num_k_blocks, tile_rows, a_bytes and the
// resident-patch / raw-row fields), then the weight and output maps.
static int build_maps(TcConvPlan* plan, const ConvParams& p, int max_batch) {
  TcKernelParams& kp = plan->kp;
  int rc;
  if (tc_conv_is_stem4(p)) {
    const int K = raw_row_layout(p).k();
    kp.a_mode = TC_A_STEM4;
    kp.cblocks = 1;
    kp.num_k_blocks = K / TC_BLOCK_K;
    kp.tile_rows = p.Q;
    kp.a_bytes = kp.tile_rows * TC_BLOCK_K * 2;
    const int Hp = p.Hin + 6, Wp = p.Win + 6;
    // raw-row mode: the padded row (Wp pixels x 4 channels) as inner x outer with a TMA-legal inner extent
    int inner = 0;
    {
      static const bool off = getenv("NIB_TC_NO_HALO") != nullptr;
      if (!off && 6 * Wp * 8 + 16 * 127 + 64 <= 16384) inner = raw_row_inner(Wp * 4);
    }
    if (inner > 0) {
      kp.a_mode = TC_A_RAW;
      kp.raw_rows = 7;
      kp.col_tiles = 1;
      kp.halo_wp = Wp * 8;
      kp.a_bytes = kp.raw_rows * kp.halo_wp;
      rc = encode_4d_bf16(&plan->tmA, p.in, {(cuuint64_t)inner, (cuuint64_t)(Wp * 4 / inner), (cuuint64_t)Hp, (cuuint64_t)max_batch},
                          {(cuuint64_t)inner * 2, (cuuint64_t)Wp * 8, (cuuint64_t)Hp * Wp * 8},
                          {(cuuint32_t)inner, (cuuint32_t)(Wp * 4 / inner), 7, 1}, CU_TENSOR_MAP_SWIZZLE_NONE);
    } else {
      // one filter row of one output row: {window element (8 pixels x 4 ch), output pixel q (+2 pixels), input row, image}
      rc = encode_4d_bf16(&plan->tmA, p.in, {32, (cuuint64_t)p.Q, (cuuint64_t)Hp, (cuuint64_t)max_batch},
                          {16, (cuuint64_t)Wp * 8, (cuuint64_t)Hp * Wp * 8}, {32, (cuuint32_t)p.Q, 1, 1},
                          CU_TENSOR_MAP_SWIZZLE_64B);
    }
    if (rc != NIB_OK) return rc;
    if ((rc = finish_plan(plan, p, max_batch, p.w_alt, K)) != NIB_OK) return rc;
    return encode_raw_row_weights(plan, p, K);
  }
  if (tc_conv_is_raw3x3(p)) {
    const int K = raw_row_layout(p).k();
    const int Hp = p.Hin + 2, Wp = p.Win + 2, row_el = Wp * 8, inner = raw_row_inner(row_el);
    kp.a_mode = TC_A_RAW;
    kp.raw_rows = 3;
    kp.col_tiles = raw3x3_col_tiles(p.Q);
    kp.cblocks = 1;
    kp.num_k_blocks = K / TC_BLOCK_K;       // resident weights: filter rows (0, 1) and (2, zero row)
    kp.tile_rows = p.Q / kp.col_tiles;
    kp.halo_wp = Wp * 16;
    kp.a_bytes = kp.raw_rows * kp.halo_wp;
    // three padded rows of one image as {inner, chunk, row, image}
    rc = encode_4d_bf16(&plan->tmA, p.in, {(cuuint64_t)inner, (cuuint64_t)(row_el / inner), (cuuint64_t)Hp, (cuuint64_t)max_batch},
                        {(cuuint64_t)inner * 2, (cuuint64_t)Wp * 16, (cuuint64_t)Hp * Wp * 16},
                        {(cuuint32_t)inner, (cuuint32_t)(row_el / inner), 3, 1}, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc != NIB_OK) return rc;
    if ((rc = finish_plan(plan, p, max_batch, p.w_alt, K)) != NIB_OK) return rc;
    return encode_raw_row_weights(plan, p, K);
  }
  if (tc_conv_is_stem(p)) {
    const int K = raw_row_layout(p).k();
    kp.a_mode = TC_A_STEM8;
    kp.cblocks = 1;
    kp.num_k_blocks = K / TC_BLOCK_K;
    kp.tile_rows = p.Q;
    kp.a_bytes = kp.tile_rows * TC_BLOCK_K * 2;
    rc = encode_2d_bf16(&plan->tmB, p.w_alt, (uint64_t)K, (uint64_t)p.Cout, (uint64_t)K * 2, TC_BLOCK_K, plan->block_n);
    if (rc != NIB_OK) return rc;
    const int Hp = p.Hin + 6, Wp = p.Win + 6;
    // {window element, output pixel q (+2 pixels), input row, image}
    rc = encode_4d_bf16(&plan->tmA, p.in, {64, (cuuint64_t)p.Q, (cuuint64_t)Hp, (cuuint64_t)max_batch},
                        {32, (cuuint64_t)Wp * 16, (cuuint64_t)Hp * Wp * 16}, {64, (cuuint32_t)p.Q, 1, 1},
                        CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc != NIB_OK) return rc;
    return finish_plan(plan, p, max_batch, p.w_alt, K);
  }
  if (tc_conv_is_halo3x3(p)) {
    const int Wp = p.Win + 2, R = halo_rows_per_tile(p.Hin, Wp);
    kp.a_mode = TC_A_HALO;
    kp.cblocks = p.Cin / 64;
    kp.num_k_blocks = 9 * kp.cblocks;
    kp.tile_rows = R * p.Win;
    kp.halo_wp = Wp; kp.halo_r = R; kp.halo_tpi = p.Hin / R;
    kp.halo_cb = kp.cblocks; kp.halo_n = p.Cout;
    kp.a_bytes = (R + 2) * Wp * 128;
    plan->block_n = 64;                               // the kernel instance; the MMA's N is halo_n
    const int Kh = 9 * p.Cin;
    rc = encode_2d_bf16(&plan->tmB, p.w, (uint64_t)Kh, (uint64_t)p.Cout, (uint64_t)Kh * 2, TC_BLOCK_K, (uint32_t)p.Cout);
    if (rc != NIB_OK) return rc;
    // the dense NHWC input as {channel, column, row, image}; the box is the whole patch of one tile
    rc = encode_4d_bf16(&plan->tmA, p.in, {(cuuint64_t)p.in_cstride, (cuuint64_t)p.Win, (cuuint64_t)p.Hin, (cuuint64_t)max_batch},
                        {(cuuint64_t)p.in_cstride * 2, (cuuint64_t)p.Win * p.in_cstride * 2,
                         (cuuint64_t)p.Hin * p.Win * p.in_cstride * 2},
                        {64, (cuuint32_t)Wp, (cuuint32_t)(R + 2), 1}, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc != NIB_OK) return rc;
    // each CTA of the pair holds Cout / 2 weight rows per K block; the kernel's "tail" slot carries the whole-tile output
    // box (Cout channels: 64 B rows under the 64B swizzle when Cout = 32); the other output / residual maps are unused
    rc = encode_2d_bf16(&plan->tmBh, p.w, (uint64_t)Kh, (uint64_t)p.Cout, (uint64_t)Kh * 2, TC_BLOCK_K, (uint32_t)(p.Cout / 2));
    if (rc != NIB_OK) return rc;
    rc = encode_2d_bf16(&plan->tmOutTail, p.out, (uint64_t)p.out_cstride, (uint64_t)max_batch * p.P * p.Q,
                        (uint64_t)p.out_cstride * 2, (uint32_t)p.Cout, (uint32_t)kp.tile_rows,
                        p.Cout == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc != NIB_OK) return rc;
    plan->tmOut = plan->tmOut32 = plan->tmRes = plan->tmOutTail;
    plan->v3 = 1;
    return NIB_OK;
  }
  kp.cblocks = (p.split ? 3 : 1) * p.Cin / TC_BLOCK_K;
  kp.num_k_blocks = p.R * p.S * kp.cblocks;
  kp.a_mode = (p.R == 1 && p.S == 1 && p.stride == 1 && p.pad == 0) ? TC_A_DENSE : TC_A_IM2COL;
  kp.a_bytes = kp.tile_rows * TC_BLOCK_K * 2;
  const int K = p.R * p.S * p.Cin * (p.split ? 3 : 1);
  // B: weights [Cout][K]
  rc = encode_2d_bf16(&plan->tmB, p.w, (uint64_t)K, (uint64_t)p.Cout, (uint64_t)K * 2, TC_BLOCK_K, plan->block_n);
  if (rc != NIB_OK) return rc;
  if (kp.a_mode == TC_A_DENSE) {
    const uint64_t rows = (uint64_t)max_batch * p.Hin * p.Win;
    rc = encode_2d_bf16(&plan->tmA, p.in, (uint64_t)p.in_cstride, rows, (uint64_t)p.in_cstride * 2, TC_BLOCK_K,
                        TC_BLOCK_M);
    if (rc != NIB_OK) return rc;
  } else {
    cuuint64_t dims[4] = {(cuuint64_t)p.in_cstride, (cuuint64_t)p.Win, (cuuint64_t)p.Hin, (cuuint64_t)max_batch};
    cuuint64_t strides[3] = {(cuuint64_t)p.in_cstride * 2, (cuuint64_t)p.Win * p.in_cstride * 2,
                             (cuuint64_t)p.Hin * p.Win * p.in_cstride * 2};
    int lower[2] = {-p.pad, -p.pad};
    int upper[2] = {p.pad - (p.S - 1), p.pad - (p.R - 1)};
    cuuint32_t es[4] = {1, (cuuint32_t)p.stride, (cuuint32_t)p.stride, 1};
    CUresult r = g_encodeIm2col(&plan->tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(p.in), dims,
                                strides, lower, upper, TC_BLOCK_K, TC_BLOCK_M, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("cuTensorMapEncodeIm2col failed (%d): C=%d W=%d H=%d N=%d R=%d stride=%d pad=%d", (int)r,
                p.in_cstride, p.Win, p.Hin, max_batch, p.R, p.stride, p.pad);
      return NIB_ECUDA;
    }
    // Driver quirk mirrored from CUTLASS (cute/atom/copy_traits_sm90_im2col.hpp): for tensors smaller
    // than 128 KiB, drivers <= 13.1 set a descriptor bit that must be cleared.
    int drv = 0;
    cudaDriverGetVersion(&drv);
    const uint64_t bytes = (uint64_t)max_batch * p.Hin * p.Win * p.in_cstride * 2;
    if (drv <= 13010 && bytes < 131072) reinterpret_cast<uint64_t*>(&plan->tmA)[1] &= ~(1ull << 21);
  }
  return finish_plan(plan, p, max_batch, p.w, K);
}

template <int BLOCK_N, int STAGES>
static int launch_tc(const TcConvPlan* plan, const TcKernelParams& kp, cudaStream_t st) {
  using SM = TcSmem<BLOCK_N, STAGES>;
  static bool attr_set = false;
  if (!attr_set) {
    NIB_CUDA(cudaFuncSetAttribute(conv_tc_kernel<BLOCK_N, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  SM::TOTAL));
    attr_set = true;
  }
  conv_tc_kernel<BLOCK_N, STAGES><<<kp.m_tiles * kp.n_tiles, TC_THREADS, SM::TOTAL, st>>>(plan->tmA, plan->tmB, kp);
  NIB_LAUNCH_CHECK();
  return NIB_OK;
}

template <int BLOCK_N, int STAGES, bool HAS_RES, bool BRES = false, bool SPLIT = false>
static int launch_tc3(const TcConvPlan* plan, const TcKernelParams& kp, cudaStream_t st) {
  using SM = Tc3Smem<BLOCK_N, STAGES, HAS_RES, BRES, SPLIT>;
  static_assert(SM::TOTAL <= 232448, "exceeds the 227 KB per-CTA shared memory limit");
  static bool attr_set = false;
  if (!attr_set) {
    NIB_CUDA(cudaFuncSetAttribute(conv_tc3_kernel<BLOCK_N, STAGES, HAS_RES, BRES, SPLIT>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, SM::TOTAL));
    attr_set = true;
  }
  const int pair_tiles = ((kp.m_tiles + 1) / 2) * kp.n_tiles;
  const int max_pairs = num_sms() / 2;
  const int pairs = pair_tiles < max_pairs ? pair_tiles : max_pairs;
  // launched with programmatic stream serialization: the CTAs become resident (and run their prologue) as the SMs of
  // the previous kernel free up, then block in griddepcontrol.wait until that kernel has completed
  static const bool pdl = getenv("NIB_TC_NO_PDL") == nullptr;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(st, &cap);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3((!BRES && !SPLIT && kp.xf_scale != nullptr) ? TC3_THREADS_XF : TC3_THREADS);
  cfg.dynamicSmemBytes = SM::TOTAL;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl && cap == cudaStreamCaptureStatusNone && kp.dbg == nullptr) ? 1 : 0;
  NIB_CUDA(cudaLaunchKernelEx(&cfg, conv_tc3_kernel<BLOCK_N, STAGES, HAS_RES, BRES, SPLIT>, plan->tmA, plan->tmBh, plan->tmOut32,
                              plan->tmOutTail, plan->tmRes, kp));
  return NIB_OK;
}

// The kernel instance of a plan whose kp is filled in.  CTA-pair stage counts fill the 227 KB of each SM (ring +
// output / residual boxes).  Only the streamed-weight CTA-pair instances have the transform warps a pre-activated conv
// needs; a plan that would land elsewhere is refused here rather than run without its BN-ReLU.
static int pick_instance(TcConvPlan* plan) {
  const TcKernelParams& kp = plan->kp;
  const bool res = kp.res != nullptr;
  bool xf_role = false;
  TcLauncher L = nullptr;
  if (plan->split) {
    // split-bf16 tensors: twice the residual / staging boxes, so shallower operand rings where a residual is added
    if (!plan->v3) { set_error("tc_conv_plan_create: split mode needs the CTA-pair kernel"); return NIB_EINVAL; }
    if (plan->block_n == 256) L = res ? &launch_tc3<256, 3, true, false, true> : &launch_tc3<256, 6, false, false, true>;
    else if (plan->block_n == 128) L = res ? &launch_tc3<128, 4, true, false, true> : &launch_tc3<128, 8, false, false, true>;
    else L = res ? &launch_tc3<64, 8, true, false, true> : &launch_tc3<64, 9, false, false, true>;
  } else if (plan->v3 && !kp.out_f32) {
    xf_role = true;
    if (kp.a_mode == TC_A_HALO) {                                   // resident patch + resident weights
      L = &launch_tc3<64, 9, false, true>;
      xf_role = false;
    } else if (kp.a_mode == TC_A_RAW && plan->block_n == 128) {     // raw rows, 128 outputs
      L = &launch_tc3<128, 6, false, true>;
      xf_role = false;
    } else if (plan->block_n == 256) {
      L = res ? &launch_tc3<256, 5, true> : &launch_tc3<256, 6, false>;
    } else if (plan->block_n == 128) {
      L = res ? &launch_tc3<128, 6, true> : &launch_tc3<128, 8, false>;
    } else if (!res && kp.n_tiles == 1 && kp.num_k_blocks <= TC3_BRES_KBLOCKS && kp.xf_scale == nullptr) {
      // resident weights: stem, 56x56 64-channel layers.  Not for a pre-activated conv (DenseNet-BC with
      // bn_size * growth == 64): it stays on the streamed instance, which has the transform warps
      L = &launch_tc3<64, 9, false, true>;
      xf_role = false;
    } else {
      L = res ? &launch_tc3<64, 9, true> : &launch_tc3<64, 9, false>;
    }
  } else {
    if (kp.a_mode > TC_A_STEM8) {   // the one-CTA kernel has no row-pair, resident-patch or raw-row operand
      set_error("tc_conv_plan_create: A-operand mode %d needs the CTA-pair kernel", kp.a_mode);
      return NIB_EINVAL;
    }
    switch (plan->block_n) {
      case 32:  L = &launch_tc<32, 4>; break;
      case 64:  L = &launch_tc<64, 4>; break;
      case 128: L = &launch_tc<128, 3>; break;
      default:  L = &launch_tc<256, 4>; break;
    }
  }
  if (kp.xf_scale != nullptr && !xf_role) {
    set_error("tc_conv_plan_create: no kernel instance with the BN-ReLU transform warps serves this pre-activation conv "
              "(Cout=%d, block_n=%d, CTA pair %d)", kp.Cout, plan->block_n, plan->v3);
    return NIB_EINVAL;
  }
  plan->launch = L;
  return NIB_OK;
}

int tc_conv_plan_create(const ConvParams& p, int max_batch, TcConvPlan** out) {
  int rc = init_tc();
  if (rc != NIB_OK) return rc;
  std::unique_ptr<TcConvPlan> plan(new TcConvPlan());
  TcKernelParams& kp = plan->kp;
  plan->split = p.split;
  plan->block_n = pick_block_n(p.Cout);
  kp.tile_rows = TC_BLOCK_M;
  if ((rc = build_maps(plan.get(), p, max_batch)) != NIB_OK) return rc;
  kp.bias = p.bias;
  kp.res = reinterpret_cast<const __nv_bfloat16*>(p.res);
  kp.out = p.out;
  kp.Cout = p.Cout;
  kp.out_cstride = p.out_cstride;
  kp.out_coff = p.out_coff;
  kp.res_cstride = p.res_cstride;
  kp.res_coff = p.res_coff;
  kp.relu = p.relu;
  kp.S = p.S;
  kp.P = p.P;
  kp.Q = p.Q;
  kp.stride = p.stride;
  kp.pad = p.pad;
  kp.in_coff = p.in_coff;
  kp.n_tiles = kp.a_mode == TC_A_HALO ? 1 : ceil_div(p.Cout, plan->block_n);
  kp.err_flag = g_err_flag;
  kp.a_wrap = plan->split ? 2 * p.Cin / TC_BLOCK_K : kp.cblocks;
  kp.lo_off_out = p.out_lo_off;
  kp.lo_off_res = p.res_lo_off;
  kp.xf_scale = p.pre_scale;
  kp.xf_shift = p.pre_shift;
  static const bool swap = getenv("NIB_TC_STEM_SWAP") != nullptr;
  kp.halo_swap = kp.a_mode == TC_A_RAW && swap ? 1 : 0;
  if ((rc = pick_instance(plan.get())) != NIB_OK) return rc;
  *out = plan.release();
  return NIB_OK;
}

void tc_conv_plan_destroy(TcConvPlan* plan) { delete plan; }
int tc_conv_plan_block_n(const TcConvPlan* plan) { return plan->block_n; }

// ---- fused expansion + next reduction (conv_fused_ca_kernel) ------------------------------------------------
struct TcFusedPlan {
  CUtensorMap tmA1, tmB1, tmRes, tmY, tmB2, tmOut2;
  int n2;
  unsigned int* err_flag;
};

static bool compact_1x1(const ConvParams& p) {
  return p.R == 1 && p.S == 1 && p.stride == 1 && p.pad == 0 && p.in_cstride == p.Cin && p.in_coff == 0 &&
         p.out_cstride == p.Cout && p.out_coff == 0 && p.in_halo == 0 && p.out_halo == 0 && p.pre_scale == nullptr;
}

// c: 1x1 K1 -> N1 with a full-width residual; a: 1x1 N1 -> N2 reading exactly c's output.  NIB_TC_FUSE=0 disables.
bool tc_fuse_supported(const ConvParams& c, const ConvParams& a) {
  const char* e = getenv("NIB_TC_FUSE");
  if (e != nullptr && atoi(e) == 0) return false;
  static const bool v1_only = getenv("NIB_TC_V1") != nullptr;
  if (v1_only) return false;
  if (c.split || a.split) return false;   // the fused kernel's staging box is a plain bf16 operand
  if (!compact_1x1(c) || !compact_1x1(a)) return false;
  if (c.res == nullptr || c.res_C != c.Cout || c.res_cstride != c.Cout || c.res_coff != 0) return false;
  if (c.Cin % TC_BLOCK_K != 0 || c.Cin > 256 || c.Cout % 256 != 0 || c.Cout > 1024) return false;
  if (a.in != c.out || a.Cin != c.Cout || a.res != nullptr) return false;
  if (a.Cout != 64 && a.Cout != 128 && a.Cout != 256) return false;
  if (a.P != c.P || a.Q != c.Q || a.M != c.M) return false;
  // Buffer aliasing.  classifier.py's LIFO buffer pool usually hands the reduction's output the very buffer the expansion
  // reads its A operand from (a.out == c.in).  The kernel tolerates exactly that case: a CTA pair loads the whole A tile
  // of its 256 rows before the tile's last MMA1, Out2 of those rows is data-dependent on all of it, and no other pair
  // touches these rows - provided both tensors have the same row pitch, so "these rows" are the same bytes.  Every other
  // overlap (y or Out2 over the residual, y over A) would be a write-after-read race between pairs: not fused.
  if (a.out == c.in && (a.Cout != c.Cin || a.out_cstride != c.in_cstride || a.out_coff != c.in_coff)) return false;
  if (a.out == c.res || c.out == c.res || c.out == c.in) return false;
  return true;
}

int tc_fused_plan_create(const ConvParams& c, const ConvParams& a, int max_batch, TcFusedPlan** out) {
  int rc = init_tc();
  if (rc != NIB_OK) return rc;
  std::unique_ptr<TcFusedPlan> plan(new TcFusedPlan());
  plan->err_flag = g_err_flag;
  plan->n2 = a.Cout;
  const uint64_t rows = (uint64_t)max_batch * c.P * c.Q;
  const uint64_t K1 = (uint64_t)c.Cin, N1 = (uint64_t)c.Cout, N2 = (uint64_t)a.Cout;
  rc = encode_2d_bf16(&plan->tmA1, c.in, K1, rows, K1 * 2, TC_BLOCK_K, TC_BLOCK_M);
  if (rc == NIB_OK) rc = encode_2d_bf16(&plan->tmB1, c.w, K1, N1, K1 * 2, TC_BLOCK_K, 64);
  if (rc == NIB_OK) rc = encode_2d_bf16(&plan->tmRes, c.res, N1, rows, N1 * 2, 64, TC_BLOCK_M);
  if (rc == NIB_OK) rc = encode_2d_bf16(&plan->tmY, c.out, N1, rows, N1 * 2, 64, 32);
  if (rc == NIB_OK) rc = encode_2d_bf16(&plan->tmB2, a.w, N1, N2, N1 * 2, TC_BLOCK_K, (uint32_t)(N2 / 2));
  if (rc == NIB_OK) rc = encode_2d_bf16(&plan->tmOut2, a.out, N2, rows, N2 * 2, 64, 32);
  if (rc != NIB_OK) return rc;
  *out = plan.release();
  return NIB_OK;
}

void tc_fused_plan_destroy(TcFusedPlan* plan) { delete plan; }

template <int N2>
static int launch_fused(const TcFusedPlan* plan, const TcFusedParams& kp, cudaStream_t st) {
  using SM = TcFusedSmem<N2>;
  static_assert(SM::TOTAL <= 232448, "exceeds the 227 KB per-CTA shared memory limit");
  static bool attr_set = false;
  if (!attr_set) {
    NIB_CUDA(cudaFuncSetAttribute(conv_fused_ca_kernel<N2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::TOTAL));
    attr_set = true;
  }
  const int m_pairs = (kp.m_tiles + 1) / 2;
  const int max_pairs = num_sms() / 2;
  const int pairs = m_pairs < max_pairs ? m_pairs : max_pairs;
  static const bool pdl = getenv("NIB_TC_NO_PDL") == nullptr;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(st, &cap);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(TCF_THREADS);
  cfg.dynamicSmemBytes = SM::TOTAL;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl && cap == cudaStreamCaptureStatusNone) ? 1 : 0;
  NIB_CUDA(cudaLaunchKernelEx(&cfg, conv_fused_ca_kernel<N2>, plan->tmA1, plan->tmB1, plan->tmRes, plan->tmY, plan->tmB2,
                              plan->tmOut2, kp));
  return NIB_OK;
}

int tc_fused_launch(const TcFusedPlan* plan, const ConvParams& c, const ConvParams& a, cudaStream_t st) {
  TcFusedParams kp;
  memset(&kp, 0, sizeof(kp));
  kp.bias1 = c.bias;
  kp.bias2 = a.bias;
  kp.res = reinterpret_cast<const __nv_bfloat16*>(c.res);
  kp.M = c.M;
  kp.m_tiles = ceil_div(c.M, TC_BLOCK_M);
  kp.kb1 = c.Cin / TC_BLOCK_K;
  kp.nch = c.Cout / 128;
  kp.n1 = c.Cout;
  kp.relu1 = c.relu;
  kp.relu2 = a.relu;
  kp.err_flag = plan->err_flag;
  static const bool dbg = getenv("NIB_TC_DBG") != nullptr;
  if (dbg) {
    const int nblk = num_sms();
    unsigned long long* d = nullptr;
    NIB_CUDA(cudaMalloc(&d, (size_t)nblk * 32 * 8));
    NIB_CUDA(cudaMemsetAsync(d, 0, (size_t)nblk * 32 * 8, st));
    kp.dbg = d;
    int rc = plan->n2 == 64 ? launch_fused<64>(plan, kp, st) : plan->n2 == 128 ? launch_fused<128>(plan, kp, st)
                                                                                : launch_fused<256>(plan, kp, st);
    if (rc != NIB_OK) return rc;
    NIB_CUDA(cudaStreamSynchronize(st));
    unsigned long long* h = (unsigned long long*)malloc((size_t)nblk * 32 * 8);
    NIB_CUDA(cudaMemcpy(h, d, (size_t)nblk * 32 * 8, cudaMemcpyDeviceToHost));
    cudaFree(d);
    double avg[32] = {0};
    int n = 0;
    for (int b = 0; b < nblk; b += 2) {   // leader CTAs
      for (int i = 0; i < 32; ++i) avg[i] += (double)h[(size_t)b * 32 + i];
      ++n;
    }
    fprintf(stderr, "[fused K1=%d N1=%d N2=%d M=%d] leader-CTA averages (kcycles)\n", c.Cin, c.Cout, a.Cout, c.M);
    const char* names[4] = {"producer: a1_empty empty1 empty2 - - - - | total", "mma: acc1_empty a1_full full1 y_ready acc2_empty full2 - | total",
                            "epi wg0: stage_free res_full acc1_full acc2_full fence_async arrive_cluster drain | total", "epi wg1: stage_free res_full acc1_full acc2_full fence_async arrive_cluster drain | total"};
    for (int r = 0; r < 4; ++r) {
      fprintf(stderr, "  %s\n   ", names[r]);
      for (int i = 0; i < 8; ++i) fprintf(stderr, " %9.1f", avg[r * 8 + i] / n / 1e3);
      fprintf(stderr, "\n");
    }
    free(h);
    return NIB_OK;
  }
  switch (plan->n2) {
    case 64: return launch_fused<64>(plan, kp, st);
    case 128: return launch_fused<128>(plan, kp, st);
    case 256: return launch_fused<256>(plan, kp, st);
  }
  set_error("tc_fused_launch: unsupported N2=%d", plan->n2);
  return NIB_EINVAL;
}
// NIB_TC_DBG=1: run the launch with the role timers on, synchronise and print where each warp role of the CTA-pair
// kernel spent its time (average over CTAs, microseconds at the SM clock).  Diagnostic only.
static int tc_launch_debug(const TcConvPlan* plan, TcKernelParams kp, const ConvParams& p, cudaStream_t st) {
  static unsigned long long* d_dbg = nullptr;
  const int nslots = 160 * 16;
  if (!d_dbg) NIB_CUDA(cudaMalloc(&d_dbg, nslots * sizeof(unsigned long long)));
  NIB_CUDA(cudaMemsetAsync(d_dbg, 0, nslots * sizeof(unsigned long long), st));
  kp.dbg = d_dbg;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  cudaEventRecord(e0, st);
  int rc = plan->launch(plan, kp, st);
  cudaEventRecord(e1, st);
  if (rc != NIB_OK) return rc;
  NIB_CUDA(cudaStreamSynchronize(st));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  static unsigned long long h[160 * 16];
  NIB_CUDA(cudaMemcpy(h, d_dbg, sizeof(h), cudaMemcpyDeviceToHost));
  int clk_khz = 1965000;
  cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, 0);
  const double us = 1e3 / (double)clk_khz;   // cycles -> us
  double a[16] = {0};
  int nc = 0;
  unsigned long long g0 = ~0ull, g1 = 0, g0max = 0, g1min = ~0ull;
  double mhz = 0, loop_max = 0;
  for (int c = 0; c < 148; ++c) {
    if (h[c * 16 + 8] == 0) continue;
    ++nc;
    for (int j = 0; j < 12; ++j) a[j] += (double)h[c * 16 + j];
    const unsigned long long e = h[c * 16 + 12], x = h[c * 16 + 13];
    if (e < g0) g0 = e;
    if (e > g0max) g0max = e;
    if (x > g1) g1 = x;
    if (x < g1min) g1min = x;
    if (x > e) mhz += (double)(h[c * 16 + 15] - h[c * 16 + 14]) / (double)(x - e) * 1e3;
    if ((double)h[c * 16 + 10] > loop_max) loop_max = (double)h[c * 16 + 10];
  }
  fprintf(stderr, "[tc3t] in-kernel span %.1f us (first entry -> last exit), entry skew %.1f us, exit skew %.1f us, SM clock %.0f MHz, "
          "max epi loop %.1f us\n", (g1 - g0) / 1e3, (g0max - g0) / 1e3, (g1 - g1min) / 1e3, mhz / (nc ? nc : 1), loop_max * us);
  if (nc == 0) nc = 1;
  for (int j = 0; j < 16; ++j) a[j] = a[j] / nc * us;
  // leader-only slots (MMA) are averaged over all CTAs: scale back
  fprintf(stderr,
          "[tc3] %dx%d %d->%d k%d s%d res%d bn%d M=%d tiles/cta=%.1f  %.1f us | prod: loop %.1f wait_empty %.1f wait_box %.1f"
          " | mma(x2): loop %.1f wait_full %.1f wait_tmem %.1f | epi: loop %.1f wait_tmem_full %.1f wait_res %.1f"
          " store_drain %.1f bar %.1f\n",
          p.P, p.Q, p.Cin, p.Cout, p.R, p.stride, p.res != nullptr, plan->block_n, p.M, a[11], ms * 1e3, a[8], a[0], a[1],
          2 * a[9], 2 * a[2], 2 * a[3], a[10], a[4], a[5], a[6], a[7]);
  return NIB_OK;
}

int tc_conv_launch(const TcConvPlan* plan, const ConvParams& p, cudaStream_t st) {
  TcKernelParams kp = plan->kp;
  kp.M = p.M;
  // raw rows: pair tiles = output-row pairs x column tiles (an odd last row pairs with a row past the batch, as any odd
  // tile count)
  kp.m_tiles = kp.a_mode == TC_A_RAW ? (p.M / p.Q + 1) / 2 * 2 * kp.col_tiles : ceil_div(p.M, kp.tile_rows);
  kp.dyn_n = plan->split ? p.dyn_n : nullptr;
  static const bool dbg = getenv("NIB_TC_DBG") != nullptr;
  if (dbg && plan->v3) return tc_launch_debug(plan, kp, p, st);
  return plan->launch(plan, kp, st);
}

}  // namespace nib

// Standalone GEMM hook: C[M,N] (fp32) = A[M,K] (bf16) * B[N,K]^T (bf16).  Exercises exactly the
// descriptors, swizzle and pipeline of the convolution kernel (tiled A map).
extern "C" int nib_tc_gemm_bf16(const void* d_A, const void* d_B, float* d_C, int M, int N, int K, void* stream) {
  NIB_DEVICE_OR_FAIL();
  using namespace nib;
  NIB_REQUIRE(d_A && d_B && d_C, "nib_tc_gemm_bf16: null pointer");
  NIB_REQUIRE(M > 0 && N > 0 && K > 0 && K % 64 == 0 && N % 32 == 0, "nib_tc_gemm_bf16: need K%%64==0, N%%32==0");
  int rc = init_tc();
  if (rc != NIB_OK) return rc;
  TcConvPlan plan = {};
  plan.block_n = pick_block_n(N);
  TcKernelParams& kp = plan.kp;
  kp.a_mode = TC_A_DENSE;
  kp.cblocks = K / TC_BLOCK_K;
  kp.num_k_blocks = kp.cblocks;
  kp.out = d_C;
  kp.M = M;
  kp.Cout = N;
  kp.out_cstride = N;
  kp.out_f32 = 1;
  kp.S = 1;
  kp.n_tiles = ceil_div(N, plan.block_n);
  kp.tile_rows = TC_BLOCK_M;
  kp.a_bytes = TC_BLOCK_M * TC_BLOCK_K * 2;
  kp.m_tiles = ceil_div(M, TC_BLOCK_M);
  kp.err_flag = g_err_flag;
  rc = encode_2d_bf16(&plan.tmB, d_B, (uint64_t)K, (uint64_t)N, (uint64_t)K * 2, TC_BLOCK_K, plan.block_n);
  if (rc != NIB_OK) return rc;
  rc = encode_2d_bf16(&plan.tmA, d_A, (uint64_t)K, (uint64_t)M, (uint64_t)K * 2, TC_BLOCK_K, TC_BLOCK_M);
  if (rc != NIB_OK) return rc;
  if ((rc = pick_instance(&plan)) != NIB_OK) return rc;
  return plan.launch(&plan, kp, (cudaStream_t)stream);
}
