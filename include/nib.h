/*
 * nib.h — C ABI of libnib.so, the B200 (sm_100a) engine for the perturbation-interpretation
 * hot path of LiliMeng/network_interpretation_imagenet:
 *
 *     mask synthesis  ->  classifier scoring  ->  Gaussian-process surrogate + acquisition
 *
 * The reference has no FFI of its own (it is flat Python, SURVEY.md §8b); every entry point
 * below names the reference call site (file:line under the reference tree) whose arithmetic
 * it replaces.  INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 (NIB_OK) or a negative NIB_E* code; nib_last_error() gives the
 *     text of the most recent failure on the calling thread.
 *   - pointers named d_* are DEVICE pointers owned by the caller (torch tensors in practice);
 *     pointers named h_* are HOST pointers, read during the call only.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *     NIB_ENODEVICE.
 *   - handles are not thread-safe; one handle per rank/process.
 */
#ifndef NIB_H_
#define NIB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NIB_ABI_VERSION 4   /* 2: + tie policy, device-side batch size, NCCL score all-gather, threshold/bbox helpers
                               3: + Kronecker-structured SKI (nib_ski_kron_*, nib_ski_band_*)
                               4: + Kriging-believer batch acquisition (nib_gp_kb_select) */

enum nib_status {
  NIB_OK = 0,
  NIB_EINVAL = -1,      /* bad argument (shape, alignment, enum)            */
  NIB_ECUDA = -2,       /* a CUDA runtime/driver call failed                */
  NIB_ENODEVICE = -3,   /* no CUDA device / not an sm_100 part              */
  NIB_ENOMEM = -4,      /* device allocation failed                         */
  NIB_ESTATE = -5,      /* handle used in the wrong state                   */
  NIB_ENUMERIC = -6     /* numerical failure (Cholesky pivot <= 0)          */
};

int nib_abi_version(void);
const char* nib_last_error(void);
/* device_count<0 on error; sets *sm_major/*sm_minor/*num_sms of device `dev` when non-NULL */
int nib_device_info(int dev, int* sm_major, int* sm_minor, int* num_sms);

/* ------------------------------------------------------------------------------------------
 * Stage 1 — mask synthesis
 * ---------------------------------------------------------------------------------------- */

/* How a selection bit-vector z in {0,1}^S turns a label map into a classifier input. */
enum nib_mask_mode {
  /* generate_gp_training_data_imagenet.py:234-240, bayesian_active_learning_imagenet.py:182-187
   * mask[p] = z[label[p]] (uint8 0/1);  out = x * (float)mask   — signed zeros preserved. */
  NIB_MASK_KEEP_MUL = 0,
  /* generate_gp_training_data_mnist.py:218-242, generate_gp_training_data_cifar.py:310-321
   * mask[p] = z[label[p]] ? 0 : 255;  m = org*mask; m -= min(m); m /= max(m); m *= 255;
   * out = m * float32(1/255)  (utils.py:92-94) — all fp32, this operation order. */
  NIB_MASK_REMOVE_MINMAX = 1
};

enum nib_dtype { NIB_F32 = 0, NIB_BF16 = 1 };

/* Output placement.  NCHW: out[n][c][h][w] (the reference's layout, C channels exactly).
 * NHWC: out[n][h+pad_h][w+pad_w][c], row pitch (W+2*pad_w)*c_stride, channels c>=C and the
 * pad_h/pad_w halo are written as +0 (the conv path wants a zero halo and padded channels). */
enum nib_layout { NIB_NCHW = 0, NIB_NHWC = 1 };

typedef struct nib_mask_args {
  const float* d_img;        /* [C,H,W] fp32: normalised image (KEEP_MUL) or the [0,255]-rescaled
                                image `org_img` (REMOVE_MINMAX, mnist :169-177)                    */
  const void* d_labels;      /* [H,W] superpixel labels 0..S-1, uint8 (label_bytes=1) or uint16   */
  int label_bytes;
  const uint64_t* d_sel;     /* [N, sel_words] selection bit-vectors, bit s of word s/64 = z[s]   */
  int sel_words;
  int N, C, H, W, S;
  int mode;                  /* nib_mask_mode */
  const float* d_seg_minmax; /* [S,2] per-segment (min,max) of d_img over all channels; required
                                for REMOVE_MINMAX (see nib_segment_minmax), ignored otherwise     */
  void* d_out;
  int out_dtype;             /* nib_dtype */
  int layout;                /* nib_layout */
  int c_stride;              /* NHWC only: channels per pixel in memory (>= C)                    */
  int pad_h, pad_w;          /* NHWC only: zero halo                                              */
  uint8_t* d_pixel_mask;     /* optional [N,H,W] uint8 pixel masks exactly as the reference holds
                                them (0/1 KEEP_MUL, 0/255 REMOVE_MINMAX) — the PNG payload of
                                imagenet :260/:265; NULL to skip                                   */
} nib_mask_args;

/* Per-segment (min,max) of a [C,H,W] fp32 image over all channels -> d_seg_minmax[S][2].
 * Replaces the two global reductions of mnist :228-231 / cifar :318-319 for every mask at once. */
int nib_segment_minmax(const float* d_img, const void* d_labels, int label_bytes,
                       int C, int H, int W, int S, float* d_seg_minmax, void* stream);

int nib_mask_synth(const nib_mask_args* args, void* stream);

/* Display images of the PNG side channel (./mask_on_img/..., bayesian_active_learning_imagenet.py:199-216,
 * generate_gp_training_data_mnist.py:225-236,:263-269): d_out [N][H][W][C] uint8 =
 *   KEEP_MUL       uint8 truncation of (x*mask - min) / max * 255 per mask (fp32, the reference's operation order)
 *   REMOVE_MINMAX  the [0,255] float image `pic`, rounded to nearest as cv2.imwrite does
 * args->d_seg_minmax is required in both modes; d_out / out_dtype / layout / c_stride / pad_* of args are ignored. */
int nib_mask_display_u8(const nib_mask_args* args, uint8_t* d_out, void* stream);

/* In-place per-image min-max rescale to [0,255] and the truncated uint8 HWC view (a1):
 * mnist :169-177, cifar :275-283, imagenet :171-178.   d_org [C,H,W] fp32 (overwritten),
 * d_u8 [H,W,C] uint8 (may be NULL). */
int nib_prep_minmax_u8(float* d_org, int C, int H, int W, uint8_t* d_u8, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stage 2 — classifier forward (models/resnet.py, models/densenet.py, mnist :86-105,
 * torchvision resnet101/densenet121 via imagenet :579) and scoring
 * ---------------------------------------------------------------------------------------- */

typedef struct nib_net nib_net;

enum nib_precision {
  NIB_PREC_FP32 = 0,  /* fp32 activations/weights, SIMT kernels: the 1e-4 parity mode         */
  NIB_PREC_BF16 = 1,  /* bf16 activations/weights, fp32 accumulate, tcgen05 implicit GEMM     */
  NIB_PREC_X3 = 2,    /* fp32 activations; convs with Cin % 16 == 0 multiply split-bf16 operands
                         (hi*hi + lo*hi + hi*lo) on the tensor cores with fp32 accumulate, ~1e-5 of
                         the fp32 mode at several times its rate: the tie policy's re-score net  */
  NIB_PREC_SPLIT = 3  /* the same split arithmetic on the tcgen05 pair kernel: body tensors hold each value as
                         two bf16 halves in the channel dimension ([hi(C) | lo(C)]), weights are
                         [Wh | Wh | Wl] along K, the epilogue stores both halves of the fp32 result.
                         Buffers are split by default; stems / pooled features live in fp32 buffers
                         (nib_net_add_buffer_f32) joined to the body by nib_net_add_convert.  Convs on
                         split tensors need Cin % 64 == 0 and Cout % 64 == 0 (ResNet bottleneck / basic
                         blocks); others: NIB_PREC_X3                                             */
};

/* A network is a flat list of ops over numbered activation buffers (NHWC, per-image geometry
 * H x W x C).  The host mirror (network_interpretation_imagenet_b200/classifier.py) walks the
 * reference's nn.Module and emits this list with BatchNorm folded. */
int nib_net_create(int precision, int max_batch, nib_net** out);
int nib_net_destroy(nib_net* net);

/* returns buffer id >= 0.  pad = zero halo kept around H and W (0 for all but the stem input) */
int nib_net_add_buffer(nib_net* net, int H, int W, int C, int pad);

/* NIB_PREC_X3 / NIB_PREC_SPLIT / NIB_PREC_FP32 networks: an fp32 buffer whatever the network's default kind. */
int nib_net_add_buffer_f32(nib_net* net, int H, int W, int C, int pad);
/* NIB_PREC_SPLIT networks: out <- in across the fp32 / split boundary (same H, W, C; one side fp32, the other split). */
int nib_net_add_convert(nib_net* net, int in_buf, int out_buf);

enum nib_conv_flags {
  NIB_CONV_RELU = 1,         /* ReLU after bias (+residual)                                    */
  NIB_CONV_PRE_BNRELU = 2    /* DenseNet pre-activation: x <- relu(x*pre_scale+pre_shift) on the
                                conv INPUT, per input channel (models/densenet.py:16-27)         */
};

typedef struct nib_conv_desc {
  int in_buf, in_coff, Cin;       /* input = channels [in_coff, in_coff+Cin) of in_buf           */
  int out_buf, out_coff, Cout;    /* output written to channels [out_coff, out_coff+Cout)        */
  int res_buf, res_coff, res_C;   /* residual added to output channels [0,res_C); res_buf=-1:none
                                     (res_C < Cout = DownsampleB zero-channel concat,
                                     models/resnet.py:67-76)                                      */
  int R, S, stride, pad;
  int flags;
} nib_conv_desc;

/* h_weight [Cout][Cin][R][S] fp32 (torch layout), already BN-folded; h_bias [Cout] fp32 or NULL;
 * h_pre_scale/h_pre_shift [Cin] fp32 when NIB_CONV_PRE_BNRELU. */
int nib_net_add_conv(nib_net* net, const nib_conv_desc* d, const float* h_weight,
                     const float* h_bias, const float* h_pre_scale, const float* h_pre_shift);

enum nib_pool_kind { NIB_POOL_MAX = 0, NIB_POOL_AVG = 1 };
/* window k x k, given stride/pad; avg divides by k*k (count_include_pad, as nn.AvgPool2d).
 * out channels [out_coff, out_coff+C) of out_buf.  Optional per-channel affine+ReLU applied to
 * the input first (DenseNet transition/norm5: BN-ReLU before the pool commutes only for AVG
 * when done first, so it is applied to each element before pooling). */
int nib_net_add_pool(nib_net* net, int kind, int in_buf, int in_coff, int C, int out_buf,
                     int out_coff, int k, int stride, int pad,
                     const float* h_pre_scale, const float* h_pre_shift);

/* logits[n][k] = sum_c W[k][c] * feat[n][c] + b[k]; feat = buffer with H=W=1. fp32 math always. */
int nib_net_add_fc(nib_net* net, int in_buf, int Cin, int Cout, const float* h_weight,
                   const float* h_bias);

int nib_net_set_input(nib_net* net, int buf);
int nib_net_finalize(nib_net* net);

/* Input layouts accepted by nib_net_forward */
enum nib_input_layout {
  NIB_IN_NCHW_F32 = 0,   /* the reference's tensor: N x C x H x W fp32 (imagenet :245-246)        */
  NIB_IN_NATIVE = 1      /* already in the input buffer's own layout/dtype (written by
                            nib_mask_synth with NHWC + the buffer's c_stride/pad)                 */
};

/* logits: d_logits [N, num_classes] fp32.  N <= max_batch. */
int nib_net_forward(nib_net* net, const void* d_x, int x_layout, int N, float* d_logits,
                    void* stream);

/* Fused stages 1+2: masks are synthesised straight into the network's input buffer
 * (args->d_out/out_dtype/layout/c_stride/pad_* are ignored and taken from the network). */
int nib_net_forward_masked(nib_net* net, const nib_mask_args* args, float* d_logits, void* stream);

/* Device address + geometry of an activation buffer (MNIST returns x0,x1,x2 besides the logits,
 * mnist :97-105).  *dtype is nib_dtype.  Layout NHWC, c_stride = C of the buffer. */
int nib_net_buffer_info(nib_net* net, int buf, void** d_ptr, int* H, int* W, int* C, int* pad,
                        int* dtype);
/* NHWC (buffer dtype) -> NCHW fp32 copy of channels [0,C) for N images. */
int nib_net_read_buffer_nchw(nib_net* net, int buf, int N, float* d_out, void* stream);

/* Counters for bench.py: kernels launched by this handle since creation, and how many of those
 * were tcgen05 implicit-GEMM launches. */
int nib_net_launch_counts(nib_net* net, long long* total, long long* tcgen05);
/* force (1) / forbid (0) the tcgen05 path for eligible convs of a bf16 net (default 1). */
int nib_net_set_tensor_core(nib_net* net, int enable);
/* 1 = replay forward through a CUDA graph per batch size (default 0) */
int nib_net_set_graph(nib_net* net, int enable);

/* Per-op device timing of one forward (CUDA events on `stream` around every launch; the input buffer must
 * already hold N images, e.g. from a previous nib_net_forward_masked).  Arrays are host, length >= cap;
 * *num_ops receives the op count.  h_kind: 0 SIMT conv, 1 tcgen05 conv, 2 pool, 3 fc, 4 tcgen05 conv that ran inside the
 * previous op's fused launch (no launch of its own).
 * h_flops: 2*M*K*Cout for convs / fc (the algorithmic FLOPs SURVEY.md §8d counts), 0 for pools.
 * h_geom (optional, 8 ints per op): Hout, Wout, Cin, Cout, R, stride, has_residual, block_n. */
int nib_net_profile(nib_net* net, int N, float* h_ms, int* h_kind, double* h_flops, int* h_geom,
                    int cap, int* num_ops, void* stream);

/* Scoring: top-1 index (first maximum, as torch .max(1)), softmax probability of `target`,
 * max softmax probability, and correct = (top1 == target).
 * imagenet :248,:257 ; bayesian_active_learning_imagenet.py:196-198 ; mnist :249-259.
 * d_margin: (top1 logit - runner-up logit) / max|logit| per row — the tie detector of the bf16 path: rows whose
 * relative margin is inside the bf16 logit tolerance are re-scored in fp32 by the host mirror so that top-1 is
 * identical to the reference's on every mask.  Any output pointer may be NULL. */
int nib_score(const float* d_logits, int N, int K, int target, int32_t* d_top1,
              float* d_target_prob, float* d_max_prob, uint8_t* d_correct, float* d_margin,
              void* stream);

/* nib_score plus d_table [N][2] fp32 = (target_prob, (float)top1) per row: the layout of the score all-gather's send
 * buffer (class ids < 2^24 are exact in fp32), written by the same kernel so no packing pass sits between scoring and
 * the collective.  Any output pointer may be NULL. */
int nib_score_table(const float* d_logits, int N, int K, int target, int32_t* d_top1,
                    float* d_target_prob, float* d_max_prob, uint8_t* d_correct, float* d_margin,
                    float* d_table, void* stream);

/* Tie policy of the bf16 path, entirely on the stream (no host synchronisation).  The reference compares the arg-max
 * of fp32 logits with the target (imagenet :248-257); bf16 logits are within a stated tolerance of those, so rows whose
 * top-2 margin is inside the band are re-scored by an fp32 copy of the classifier:
 *   nib_tie_compact  d_idx[cap] <- ascending row indices with d_margin[r] < threshold (first `cap` of them; unused
 *                    slots -1), d_sel_out[cap][words] <- their selection words (unused slots 0), *d_count <- how many
 *                    rows qualified in total (> cap means overflow: the rows beyond the buffer keep their bf16 score);
 *                    d_totals (optional, int64[2]) accumulates (qualified, did-not-fit) over calls
 *   nib_net_set_dynamic_batch + nib_net_forward_masked(N = cap) on the fp32 network: only *d_count images are computed
 *   nib_tie_scatter  refined results of slot s < min(*d_count, cap) overwrite row d_idx[s] of the score arrays / table */
int nib_tie_compact(const float* d_margin, int N, float threshold, const uint64_t* d_sel, int words, int cap,
                    int32_t* d_idx, uint64_t* d_sel_out, int32_t* d_count, long long* d_totals, void* stream);
int nib_tie_scatter(const int32_t* d_idx, const int32_t* d_count, int cap, const int32_t* r_top1,
                    const float* r_target_prob, const float* r_max_prob, const uint8_t* r_correct,
                    int32_t* d_top1, float* d_target_prob, float* d_max_prob, uint8_t* d_correct,
                    float* d_table, void* stream);
/* fp32 (CUDA-core) networks only: the kernels of every following forward read the live image count from *d_count
 * (clamped to the N passed to the call) and skip the rest of the batch; NULL restores host-side N. */
int nib_net_set_dynamic_batch(nib_net* net, const int32_t* d_count);

/* ------------------------------------------------------------------------------------------
 * Multi-GPU: the path's only exchange step.  Rank r of W scores masks [r*per, (r+1)*per) (contiguous shards of the
 * global, seed-generated selection table) and every rank receives the whole (target_prob, top1) table — the GP rank fits
 * on all of it.  The reference declares --world-size / --dist-backend (generate_gp_training_data_imagenet.py:72-77) and
 * stops at `args.distributed = args.world_size > 1` (:572).  NCCL is bound at run time (dlopen; PyTorch's copy is reused
 * when loaded).  Bootstrap: rank 0 calls nib_comm_unique_id, the 128 bytes travel by any side channel
 * (torch.distributed broadcast in the host mirror), every rank calls nib_comm_init.
 * ---------------------------------------------------------------------------------------- */
typedef struct nib_comm nib_comm;
int nib_comm_unique_id(void* h_id128);
int nib_comm_init(const void* h_id128, int rank, int world, nib_comm** out);
int nib_comm_destroy(nib_comm* comm);
/* d_local [rows_per_rank][2] fp32 (nib_score_table's d_table) -> d_table [world*rows_per_rank][2], rank-major */
int nib_allgather_scores(nib_comm* comm, const float* d_local, int rows_per_rank, float* d_table, void* stream);

/* Standalone tcgen05 GEMM self-test hook: C[M,N] = A[M,K] * B[N,K]^T (bf16 in, fp32 out).
 * Used by tests to validate descriptors independent of the network executor. */
int nib_tc_gemm_bf16(const void* d_A, const void* d_B, float* d_C, int M, int N, int K,
                     void* stream);

/* ------------------------------------------------------------------------------------------
 * Stage 3 — Gaussian-process surrogate over binary masks + Expected Improvement
 * sklearn GaussianProcessRegressor(kernel=RBF(), alpha=1e-5, normalize_y=True) as configured at
 * BayesianOptimization.py:154-159, arithmetic of sklearn/gaussian_process/_gpr.py (1.9.0).
 * All matrices fp64, column-major is never used: K and L are row-major [n][ld].
 * ---------------------------------------------------------------------------------------- */

/* K[i][j] = exp(-0.5 * hamming(z_i, z_j) / l^2) (+ jitter on the diagonal when Zb==Za).
 * For binary X the sklearn RBF (kernels.py:1561-1569) reduces to this LUT over popcounts.
 * Za [na,words], Zb [nb,words]; d_K [na][ldk].  d_H (optional, int32 [na][ldk]) receives the
 * Hamming distances (needed for the LML gradient). */
int nib_gp_gram_binary(const uint64_t* d_Za, int na, const uint64_t* d_Zb, int nb, int words,
                       double length_scale, double jitter, double* d_K, int ldk, void* stream);

/* Real-valued RBF Gram: K[i][j] = exp(-0.5*||xa_i - xb_j||^2 / l^2) (+jitter if same & i==j).
 * Xa [na,d], Xb [nb,d] fp64 row-major.  The reference's actual 1-D firstIndex GP
 * (BayesianOptimization.py:137-166) uses this with d=1. */
int nib_gp_gram_rbf(const double* d_Xa, int na, const double* d_Xb, int nb, int d,
                    double length_scale, double jitter, int same, double* d_K, int ldk,
                    void* stream);

/* In-place lower Cholesky K = L L^T of the leading n x n block (upper triangle left untouched).
 * d_info (device int) receives 0 or the 1-based index of the first non-positive pivot
 * (_gpr.py:352). */
int nib_gp_cholesky(double* d_K, int n, int ldk, int* d_info, void* stream);

/* Diagnostic hook: C[M,N] -= A[M,K] * B[K,N] (row-major fp64) through the GEMM the blocked Cholesky / TRSM trailing
 * updates use (gp.cu dgemm_sub_kernel).  No reference counterpart; used by tools/gp_profile.py to measure the kernel
 * against the fp64 peak. */
int nib_gp_dgemm_sub(const double* d_A, const double* d_B, double* d_C, int M, int N, int K, void* stream);

/* Triangular solves with the lower factor L ([n][ldl]) on B ([n][ldb], nrhs columns), in place.
 * trans=0: B <- L^{-1} B ;  trans=1: B <- L^{-T} B.   (cho_solve = trans 0 then trans 1) */
int nib_gp_trsm(const double* d_L, int n, int ldl, double* d_B, int nrhs, int ldb, int trans,
                void* stream);

/* Posterior for m queries given Ks = k(Xq, Xtrain) [m][ldks] (row q = query q):
 *   mu[q]  = y_std * (Ks[q] . alpha) + y_mean
 *   var[q] = y_std^2 * max(0, prior_var - || L^{-1} Ks[q]^T ||^2)          (_gpr.py:446-496)
 * d_work: m*n doubles scratch ([n][m] row-major V).  d_std optional (sqrt(var)). */
int nib_gp_posterior(const double* d_L, int n, int ldl, const double* d_alpha,
                     const double* d_Ks, int m, int ldks, double y_mean, double y_std,
                     double prior_var, double* d_work, double* d_mu, double* d_var,
                     double* d_std, void* stream);

/* log marginal likelihood and d/d(log l) at the current factor (_gpr.py:588-655):
 *   lml = -0.5 y^T alpha - sum log L_ii - n/2 log 2pi
 *   grad = 0.5 * tr((alpha alpha^T - K^{-1}) dK/dtheta),  dK/dtheta = K_noisefree .* D2 / l^2
 * d_K0: noise-free Gram [n][ld]; d_Kinv: K^{-1} [n][ld]; squared distances are recomputed on the fly
 * from the inputs (popcounts of d_Z for binary masks).  Results to host doubles (synchronises). */
int nib_gp_lml(const double* d_L, int n, int ldl, const double* d_y, const double* d_alpha,
               double* h_lml, void* stream);
int nib_gp_lml_grad(const double* d_K0, const double* d_Kinv, const double* d_alpha,
                    const uint64_t* d_Z, int words, int n, int ld, double length_scale,
                    double* h_grad, void* stream);
/* same for real-valued inputs X [n,d] (the reference's 1-D firstIndex GP) */
int nib_gp_lml_grad_rbf(const double* d_K0, const double* d_Kinv, const double* d_alpha,
                        const double* d_X, int d, int n, int ld, double length_scale,
                        double* h_grad, void* stream);

/* Rank-one maintenance of the posterior workspace, for acquisition loops that add ONE training mask per round
 * (bayesian_active_learning_imagenet.py / BayesianOptimization.py:140-185 refit the GP from scratch every round).
 * With V = L^-1 K*^T [n x m] resident, appending a point needs l = L^-1 k (nib_gp_trsm, one vector), d = sqrt(k_nn +
 * alpha - l.l), the new row of V: (k*_new - l^T V) / d, and sum-of-squares += row^2 — O(n^2 + m n) instead of O(n^3 + m n^2).
 *   nib_gp_gemv_t      d_out[j] = sum_t d_x[t] * d_V[t*ldv + j]            (t < n, j < m)
 *   nib_gp_colsumsq    d_out[j] = sum_t d_V[t*ldv + j]^2
 *   nib_gp_append_row  v = (d_ks - d_dot) / d;  d_vrow = v;  d_ssq += v^2    (all length m) */
int nib_gp_gemv_t(const double* d_V, int n, int m, int ldv, const double* d_x, double* d_out, void* stream);
int nib_gp_colsumsq(const double* d_V, int n, int m, int ldv, double* d_out, void* stream);
int nib_gp_append_row(const double* d_ks, const double* d_dot, double d, double* d_vrow, double* d_ssq, int m,
                      void* stream);

/* Batch acquisition on the same resident state: q picks by greedy Kriging believer, all on the device.  The fantasy
 * observation at a pick is its posterior mean, which leaves every other mean unchanged, so with the mean d_mu [m] fixed
 * (computed once at the current y-normalisation) each pick only adds one row to L and V.  For k = 0 .. q-1:
 *   sigma_x = y_std * sqrt(max(0, 1 - ssq_x)), NaN where !alive_x;   EI_x as nib_gp_ei with incumbent b
 *   j = arg-max of the non-NaN EI (lowest index on ties); none -> stop (d_picks[k..q) stay -1)
 *   l = V[0:n+k, j] (= L^-1 k(X, z_j));  d^2 = 1 + alpha - ssq_j;  d^2 <= 0 -> *d_status = k + 1, stop
 *   L[n+k, 0:n+k] = l;  L[n+k, n+k] = d;  X[n+k] = cand[j];  V[n+k][x] = (k(x, z_j) - sum_t V[t][x] l_t) / d;
 *   ssq += V[n+k]^2;  alive_j = 0;  b = max(b, mu_j) (min when !greater_is_better);  d_picks[k] = j;  d_ei[k] = EI_j
 * d_L [>= n+q][ldl] with n rows filled, d_V [>= n+q][ldv] with n rows filled, d_ssq / d_alive (bytes) [m],
 * d_cand [m][words] and d_X [>= n+q][words] selection bits, kernel exp(-popcount(a ^ b) * 0.5 / length_scale^2) as
 * nib_gp_gram_binary.  One pass over V per pick and no host synchronisation inside the batch; d_picks [q] (int64),
 * d_ei [q] and d_status (int) are the only outputs the caller has to read.  Deterministic (no floating-point atomics).
 * The observed values then enter u = L^-1 y, w = L^-1 1 through rows n .. n+q-1 of L (ActiveMaskGP.set_batch_values). */
int nib_gp_kb_select(double* d_L, int ldl, double* d_V, int ldv, double* d_ssq, unsigned char* d_alive,
                     const uint64_t* d_cand, int m, int words, uint64_t* d_X, int n, int q, const double* d_mu,
                     double y_std, double best, int greater_is_better, double length_scale, double alpha,
                     long long* d_picks, double* d_ei, int* d_status, void* stream);

/* Expected improvement, BayesianOptimization.py:37-54 (returns +EI; the reference returns -EI):
 *   s = greater_is_better ? 1 : -1;  Z = s*(mu-best)/sigma;  EI = s*(mu-best)*Phi(Z)+sigma*phi(Z)
 * sigma == 0 yields NaN exactly as the reference (its `== 0.0` line :52 is a no-op comparison).
 * d_argmax (optional, device int64) = index of the largest non-NaN EI (first on ties). */
int nib_gp_ei(const double* d_mu, const double* d_sigma, int m, double best,
              int greater_is_better, double* d_ei, long long* d_argmax, void* stream);

/* ------------------------------------------------------------------------------------------
 * "Next" row 1 — heat map H = sum_i y_i * mask_i  (gp_regression.py:82-94,
 * gp_superpixel_data_imagenet.py:322-323): per-segment weighted counts scattered to pixels.
 * d_heat [H*W] fp32;  weights d_y [N] fp32;  keep-mode selection bits.
 * ---------------------------------------------------------------------------------------- */
int nib_heatmap(const void* d_labels, int label_bytes, int H, int W, int S,
                const uint64_t* d_sel, int sel_words, const float* d_y, int N, float* d_heat,
                void* stream);

/* The heat map is constant on superpixels when its masks are superpixel masks of one label map: d_wseg[s] = sum of d_y[i]
 * over the masks that select segment s (double, exact for integer labels), d_cover[s] (optional) = how many do.  The
 * threshold search of generate_gp_training_data_imagenet.py:334-488 works on these S numbers instead of n x n pixels. */
int nib_segment_weights(const uint64_t* d_sel, int sel_words, const float* d_y, int N, int S, double* d_wseg,
                        int32_t* d_cover, void* stream);

/* Localisation tail of the heat map (generate_gp_training_data_imagenet.py:519-525, bayesian_active_learning_imagenet.py
 * :349-377, utils.py:96-109):
 *   nib_heat_normalize_u8  gray = uint8((H - min(H)) / max(H - min(H)) * 255), float64 arithmetic in numpy's operation
 *                          order, truncation; d_minmax (optional, double[2]) receives (min, max) of the heat map
 *   nib_threshold_bbox     cv2.threshold(gray, t, 255, THRESH_BINARY) + findContours(RETR_EXTERNAL) + the boundingRect of
 *                          largest w*h (OpenCV's order on ties): d_box int32[6] = {x, y, w, h, #components, #pixels > t},
 *                          zeros when no pixel exceeds t.  H*W <= 65535. */
int nib_heat_normalize_u8(const float* d_heat, int P, uint8_t* d_gray, double* d_minmax, void* stream);
int nib_threshold_bbox(const uint8_t* d_gray, int H, int W, int threshold, int32_t* d_box, void* stream);

/* ------------------------------------------------------------------------------------------
 * Pixel-coordinate GP regression on an inducing grid (KISS-GP / SKI) and its training heat map.
 * Replaces gp_regression.py:63-104 (heat map from the ./masks PNGs), :160-176 (GPRegressionModel:
 * ExactGP + GridInterpolationKernel(RBF, grid_size=30) + outputscale) and :244-261 (posterior over
 * all n x n pixels).  gpytorch is absent and unpinned (pre-0.1 API): parity unpinned; arithmetic
 * restated from the published SKI construction, see csrc/ski.cu.  The dense G x G algebra
 * (G = grid_size^2) uses nib_gp_gram_rbf / nib_gp_dgemm_sub / nib_gp_cholesky / nib_gp_trsm.
 *   nib_heatmap_pixels  d_heat[p] += sum_i d_y[i] * [d_masks[i*P + p] == on_value]   (u8 masks)
 *   nib_ski_accumulate  A += W^T W [G,G], b += W^T (y - const_mean) [G] over n points d_X [n,2]
 *                       (cubic-convolution weights on the grid grid0 + k*spacing, k < grid_size)
 *   nib_ski_predict     mean[q] = const_mean + w_q^T mean_u;  var[q] = noise*|Gm w_q|^2 (+ noise)
 * ---------------------------------------------------------------------------------------- */
int nib_heatmap_pixels(const uint8_t* d_masks, const float* d_y, int N, int P, int on_value,
                       float* d_heat, void* stream);
int nib_ski_accumulate(const double* d_X, const double* d_y, int n, double grid0, double spacing,
                       int grid_size, double const_mean, double* d_A, double* d_b, void* stream);
int nib_ski_predict(const double* d_Xq, int m, double grid0, double spacing, int grid_size,
                    double const_mean, const double* d_mean_u, const double* d_Gm, double noise,
                    int add_noise, double* d_mean, double* d_var, void* stream);

/* The same SKI model on grids too large for dense G x G factors (grid_size 300: G = 90 000), csrc/ski_kron.cu.
 * K = os K1 (x) K1 has the square root S = M_R (x) M_C with gs x gs factors built on the host (ski.py), and
 *   mean_U = S B^-1 S^T b,   var(x*) = noise (S^T w*)^T B^-1 (S^T w*) (+ noise),   B = noise I + S^T A S,
 * solved by preconditioned CG with the diagonal D = noise + coef * thetaR[i] * thetaC[j] (exact for a lattice of pixels).
 * Vectors over the grid are G = gs^2 doubles, row-major (index i0 * gs + i1); r right-hand sides are r such vectors
 * back to back.  r <= 65535, grid_size <= 46340.
 *   nib_ski_kron_apply        Y[:, c] = (M_R (x) M_C) X[:, c] (trans 0) or (M_R (x) M_C)^T X[:, c] (trans 1), i.e.
 *                             M_R X_c M_C^T / M_R^T X_c M_C per gs x gs block; d_MR, d_MC [gs][gs]; d_work r*G doubles
 *   nib_ski_band_accumulate   A = W^T W in band form d_A [G][7][7] (A[g][(d0+3)*7 + d1+3] couples g with g + (d0, d1),
 *                             zero where that leaves the grid) and d_b = W^T (y - const_mean) [G], without floating-point
 *                             atomics (bitwise reproducible).  d_work: 4 * (2n + 3G + 2) + 72 n bytes
 *   nib_ski_band_spmv         Y[:, c] = A X[:, c] for the band A above
 *   nib_ski_kron_pcg          solves B x = rhs for r columns (d_rhs, d_x [r][G]) to relative residual <= tol per column;
 *                             d_thetaR, d_thetaC [gs]; d_work 8 * (5 r G + 5 r + 4) bytes.  The host reads the state every
 *                             check_every iterations; on return *h_iters = most iterations taken by a column and
 *                             *h_relres = largest relative residual reached (> tol: not converged within max_iter)
 *   nib_ski_kron_var_rhs      d_rhs[q] = (M_R^T w0_q) (x) (M_C^T w1_q) for m queries d_Xq [m, 2] (grid_size <= 3072)
 *   nib_ski_kron_var_reduce   d_var[q] = noise * d_rhs[q] . d_x[q] (+ noise when add_noise) */
int nib_ski_kron_apply(const double* d_X, double* d_Y, int r, int grid_size, const double* d_MR, const double* d_MC,
                       int trans, double* d_work, void* stream);
int nib_ski_band_accumulate(const double* d_X, const double* d_y, int n, double grid0, double spacing, int grid_size,
                            double const_mean, double* d_A, double* d_b, void* d_work, void* stream);
int nib_ski_band_spmv(const double* d_A, int grid_size, const double* d_X, double* d_Y, int r, void* stream);
int nib_ski_kron_pcg(const double* d_A, int grid_size, const double* d_MR, const double* d_MC, const double* d_thetaR,
                     const double* d_thetaC, double coef, double noise, const double* d_rhs, double* d_x, int r,
                     double tol, int max_iter, int check_every, double* d_work, int* h_iters, double* h_relres,
                     void* stream);
int nib_ski_kron_var_rhs(const double* d_Xq, int m, double grid0, double spacing, int grid_size, const double* d_MR,
                         const double* d_MC, double* d_rhs, void* stream);
int nib_ski_kron_var_reduce(const double* d_rhs, const double* d_x, int m, int grid_size, double noise, int add_noise,
                            double* d_var, void* stream);

/* ------------------------------------------------------------------------------------------
 * Variational GP classification on the inducing grid: the O(n) part of one optimiser step of
 * gp_classification.py:160-217 (`-mll(model(train_x), train_y)` + backward) and its prediction loop :241-253
 * (`likelihood(model(test_x)).mean()`).  gpytorch (GridInducingVariationalGP, BernoulliLikelihood, pre-0.1 API) is absent
 * and unpinned -> parity unpinned; the model is restated in csrc/ski.cu: u ~ N(0, K_UU) on the grid, q(u) = N(m, S),
 * f(x) = c + w(x)^T u, p(y | f) = Phi(y f), expectations by 20-point Gauss-Hermite quadrature.
 *   nib_vgp_loglik_grad  *d_ell = sum_i E_q[log Phi(y_i f_i)], d_grad_m [G] and d_grad_S [G,G] its gradients w.r.t. the
 *                        variational mean / covariance, d_grad_c (optional) w.r.t. the constant mean; outputs are zeroed
 *                        by the call.  d_S is the dense symmetric covariance [G,G].
 *   nib_vgp_predict      d_prob[q] = Phi(mu_q / sqrt(1 + s2_q)); latent moments to d_mu / d_var (any may be NULL)
 * ---------------------------------------------------------------------------------------- */
int nib_vgp_loglik_grad(const double* d_X, const double* d_y, int n, double grid0, double spacing, int grid_size,
                        double const_mean, const double* d_m, const double* d_S, double* d_ell, double* d_grad_m,
                        double* d_grad_S, double* d_grad_c, void* stream);
int nib_vgp_predict(const double* d_Xq, int m, double grid0, double spacing, int grid_size, double const_mean,
                    const double* d_m, const double* d_S, double* d_prob, double* d_mu, double* d_var, void* stream);

/* ------------------------------------------------------------------------------------------
 * Superpixel label map (SURVEY.md §8 a2) — HOST function, HOST pointers, no device needed.
 * Replaces `felzenszwalb(img_as_float(img), scale=100, sigma=0.5, min_size=50)`
 * (generate_gp_training_data_imagenet.py:183, generate_gp_training_data_mnist.py:187,
 * generate_gp_training_data_cifar.py:293, bayesian_active_learning_imagenet.py:150,:263,:463):
 * scikit-image's graph-based segmentation (Gaussian blur, 8-connected colour-distance edges,
 * sorted-edge union-find with threshold scale/|C|, min_size clean-up), labels 0..S-1 numbered in
 * raster order of first appearance.  h_image [H,W,C] float64 in [0,1]; h_labels [H,W] int32.
 * ---------------------------------------------------------------------------------------- */
int nib_felzenszwalb(const double* h_image, int H, int W, int C, double scale, double sigma,
                     int min_size, int32_t* h_labels, int* num_segments);

#ifdef __cplusplus
}
#endif
#endif /* NIB_H_ */
