// layers.cuh — parameter blocks and launchers shared by the network executor (net.cu).
#pragma once
#include "common.cuh"

namespace nib {

struct ConvParams {
  const void* in;       // NHWC activations (T)
  const void* w;        // KRSC weights (T)
  const void* w_alt;    // raw-row modes only (tc_raw_row_layout): bf16 [Cout][rows][taps][ch], or null
  const float* bias;    // [Cout] fp32 or null
  const void* res;      // residual NHWC (T) or null
  void* out;
  const float* pre_scale;  // [Cin] or null (DenseNet pre-activation BN+ReLU on the input)
  const float* pre_shift;
  int pre_padded;          // 1: both arrays are zero-padded to a multiple of 64 channels and Cin counts the padded channels
                           // (the pair kernel's in-kernel transform, conv_tc.cu); the weights carry the same zero padding
  int M;                // N * P * Q output pixels
  int Hin, Win, Cin, in_cstride, in_coff, in_halo;
  int P, Q, Cout, out_cstride, out_coff, out_halo;
  int res_cstride, res_coff, res_C;
  int R, S, stride, pad;
  int relu;
  const int* dyn_n;     // optional device int: live image count (<= M / (P*Q)); rows of the images beyond it are skipped
                        // by the CUDA-core kernels (the fp32 tie re-score runs on a device-side count, score.cu)
  // split-bf16 tensors (NIB_PREC_SPLIT, conv_tc.cu): Cin / Cout / res_C stay LOGICAL channel counts, the *_cstride values
  // are the physical ones (2 x logical), `w` is the [Cout][R*S][3*Cin] arrangement [Wh | Wh | Wl]; the lo half of each
  // tensor starts *_lo_off channels after its hi half
  int split;
  int in_lo_off, out_lo_off, res_lo_off;
};

struct PoolParams {
  const void* in;
  void* out;
  const float* pre_scale;
  const float* pre_shift;
  int kind, N, Hin, Win, C, in_cstride, in_coff;
  int P, Q, out_cstride, out_coff;
  int k, stride, pad;
  const int* dyn_n;     // as ConvParams::dyn_n
};

int launch_conv_simt(const ConvParams& p, bool bf16, cudaStream_t st);
// split-bf16 tensor-core conv on fp32 activations (conv_x3.cu); w_hi / w_lo: bf16 KRSC halves of the fp32 weights
bool conv_x3_supported(const ConvParams& p);
int launch_conv_x3(const ConvParams& p, const void* w_hi, const void* w_lo, cudaStream_t st);
int launch_pool(const PoolParams& p, bool bf16, cudaStream_t st);
bool fc_x2_supported(int Cin, int feat_stride);
int launch_fc_x2(const void* feat, int feat_stride, const void* w_hi, const void* w_lo, const float* b, int N, int Cin,
                 int Cout, float* logits, const int* dyn_n, cudaStream_t st);
int launch_fc(const void* feat, int feat_stride, bool bf16, const float* w, const float* b, int N, int Cin,
              int Cout, float* logits, const int* dyn_n, cudaStream_t st);
int launch_bnrelu_pack(const void* x, int in_cstride, int in_coff, int Cin, int Cpad, const float* scale,
                       const float* shift, void* y, long long M, cudaStream_t st);
int launch_nchw_to_nhwc(const float* x, int N, int C, int H, int W, void* out, int cs, int halo, bool bf16,
                        cudaStream_t st);
int launch_nhwc_to_nchw(const void* in, int N, int C, int H, int W, int cs, int halo, bool bf16, float* out,
                        cudaStream_t st);
// fp32 [M][C] <-> split bf16 [M][hi(C) | lo(C)], x = hi + lo with hi = bf16(x), lo = bf16(x - hi)   (NIB_PREC_SPLIT)
int launch_split_convert(const void* in, void* out, long long M, int C, bool to_split, const int* dyn_n, int rows_per_image,
                         cudaStream_t st);
// dyn_n: optional device-side live mask count (<= a->N); masks beyond it are not synthesised
int mask_synth_impl(const nib_mask_args* a, cudaStream_t st, bool skip_halo, const int* dyn_n = nullptr);

// ---- tcgen05 implicit-GEMM convolution (conv_tc.cu) ---------------------------------------------
struct TcConvPlan;  // opaque: tensor maps + tile configuration for one conv layer

// Weights of the tcgen05 modes that read raw input rows (the 7x7 stride-2 stem, a 3x3 stride-1 first conv): bf16
// [Cout][rows][taps][ch], zero past the filter's R x S x Cin, uploaded as ConvParams::w_alt.  rows == 0: no such mode.
struct RawRowLayout {
  int rows, taps, ch;
  int k() const { return rows * taps * ch; }
};
RawRowLayout tc_raw_row_layout(int R, int S, int stride, int pad, int Cin, int in_cstride, int in_halo);

// true when the layer geometry is covered by the tcgen05 kernel
bool tc_conv_supported(const ConvParams& p);
// builds tensor maps for the given buffers (max_batch images); returns NIB_OK or error
int tc_conv_plan_create(const ConvParams& p, int max_batch, TcConvPlan** out);
void tc_conv_plan_destroy(TcConvPlan* plan);
int tc_conv_plan_block_n(const TcConvPlan* plan);
// launch for a batch with M = N*P*Q valid rows (p.M)
int tc_conv_launch(const TcConvPlan* plan, const ConvParams& p, cudaStream_t st);

// a bottleneck's 1x1 expansion (+ residual, ReLU) fused with the next bottleneck's 1x1 reduction (conv_fused_ca_kernel)
struct TcFusedPlan;
bool tc_fuse_supported(const ConvParams& c, const ConvParams& a);
int tc_fused_plan_create(const ConvParams& c, const ConvParams& a, int max_batch, TcFusedPlan** out);
void tc_fused_plan_destroy(TcFusedPlan* plan);
int tc_fused_launch(const TcFusedPlan* plan, const ConvParams& c, const ConvParams& a, cudaStream_t st);

}  // namespace nib
