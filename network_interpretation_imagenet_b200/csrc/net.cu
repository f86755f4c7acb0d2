// net.cu — classifier executor: a flat op list over NHWC activation buffers (include/nib.h §Stage 2).
//
// The host mirror (classifier.py) walks the reference's nn.Module (models/resnet.py:79-146,
// models/densenet.py:44-99, generate_gp_training_data_mnist.py:86-105, torchvision resnet101 /
// densenet121 as loaded at generate_gp_training_data_imagenet.py:579), folds eval-mode BatchNorm
// into conv weights/bias and emits the ops.  This file owns device weights (packed KRSC), the
// activation buffers sized for max_batch, per-layer tcgen05 plans, and the launch sequence.
#include "common.cuh"
#include "layers.cuh"
#include <vector>
#include <map>
#include <string.h>

using namespace nib;

// longest reduction (R * S * Cin) an fp32-grade net puts on split-bf16 tensor-core products; classifier.py mirrors it
static constexpr size_t NIB_X3_MAX_K = 16384;

enum BufKind { BUF_F32 = 0, BUF_BF16 = 1, BUF_SPLIT = 2 };   // BUF_SPLIT: bf16 [hi(C) | lo(C)] per pixel, x = hi + lo

struct NetBuffer {
  int H, W, C, pad;      // C = logical channels
  int kind;              // BufKind
  void* ptr;
  size_t elems_per_image;   // physical elements (2 * C per pixel for BUF_SPLIT)
  int phys_c() const { return kind == BUF_SPLIT ? 2 * C : C; }
  size_t esize() const { return kind == BUF_F32 ? 4 : 2; }
};

enum OpKind { OP_CONV, OP_POOL, OP_FC, OP_CONVERT };   // OP_CONVERT: fp32 <-> split

// How a conv runs, resolved once by nib_net_finalize.
enum ConvPath {
  PATH_TC,           // tcgen05 plan on the conv's own operands
  PATH_TC_XFORM,     // tcgen05 on the raw channel slice, BN-ReLU applied to the A tiles by the pair kernel's transform warps
  PATH_TC_PACK,      // relu(bn(x)) packed into pack_scratch by a separate pass, then tcgen05 on it
  PATH_FUSED_HEAD,   // a 1x1 expansion that also computes the next op (the following bottleneck's 1x1 reduction)
  PATH_FUSED_TAIL,   // computed by the previous op's fused launch
  PATH_X3,           // split-bf16 tensor-core products on fp32 activations (conv_x3.cu)
  PATH_SIMT,         // CUDA cores
};

static bool on_tcgen05(ConvPath p) { return p != PATH_X3 && p != PATH_SIMT; }

struct NetOp {
  OpKind kind;
  nib_conv_desc cd;
  void* d_w;          // conv: KRSC in net dtype; fc: fp32 [Cout][Cin]
  void* d_w_alt;      // bf16 nets, raw-row tcgen05 modes: the weights in tc_raw_row_layout
  float* d_bias;
  float* d_pre_scale;
  float* d_pre_shift;
  void* d_w_pack;     // pre-activation convs in bf16 nets: KRSC weights with Cin zero-padded to a multiple of 64
  int pack_cin;       // that padded Cin (0: no packed tensor-core path for this op)
  float* d_pre_scale_pad;   // scale / shift zero-padded to pack_cin (the pair kernel's in-kernel transform)
  float* d_pre_shift_pad;
  void* d_w_hi;       // NIB_PREC_X3 convs and bf16 nets' fc: bf16 split of the fp32 weights, w = hi + lo (conv_x3.cu)
  void* d_w_lo;
  ConvPath path;        // with the tensor cores on
  ConvPath cuda_path;   // after nib_net_set_tensor_core(0): PATH_X3 or PATH_SIMT
  TcConvPlan* plan;
  TcFusedPlan* fplan;   // PATH_FUSED_HEAD
  // pool
  int pool_kind, k, stride, pad, C, in_buf, in_coff, out_buf, out_coff;
  // fc
  int fc_in, fc_cin, fc_cout;
};

struct nib_net {
  int precision;
  int max_batch;
  bool bf16;
  bool x3;                    // fp32 activations, split-bf16 tensor-core products for the convs that qualify
  bool split;                 // NIB_PREC_SPLIT: body tensors are BUF_SPLIT, convs run on the tcgen05 pair kernel in split mode
  std::vector<NetBuffer> bufs;
  std::vector<NetOp> ops;
  std::vector<void*> allocs;  // every device allocation (upload), freed by nib_net_destroy
  void* pack_scratch;        // [max_batch * H * W][pack_cin] bf16: relu(bn(x)) of the conv being run (largest such layer)
  size_t pack_scratch_bytes;
  int input_buf;
  bool finalized;
  int num_classes;
  bool use_tc;
  bool use_graph;
  const int* dyn_n;           // device-side live batch size for the CUDA-core kernels (fp32 nets), or null
  long long launches, tc_launches;
  // CUDA graphs of the op list, one per batch size: the graph reads the net's own input buffer and writes the net's own
  // logits buffer (staging the caller's input and copying the logits out happen outside it), so caller pointers are not
  // part of the key and the cache is bounded by the number of distinct batch sizes (at most kMaxGraphs, then flushed).
  static constexpr size_t kMaxGraphs = 8;
  struct GraphVal { cudaGraphExec_t exec; long long launches, tc_launches; };
  std::map<int, GraphVal> graphs;
  float* graph_logits;
};

// Every device allocation of the net: bytes + 256 B of slack (TMA boxes never read past the tensor-map extent, but SIMT
// vector loads on the last element may touch up to 16 B beyond it), copied from h or zeroed when h is null.  Recorded
// before anything else can fail, so nib_net_destroy frees it even when the op or buffer it was for is never added.
static int upload(nib_net* net, const void* h, size_t bytes, void** d) {
  NIB_CUDA(cudaMalloc(d, bytes + 256));
  net->allocs.push_back(*d);
  if (h) NIB_CUDA(cudaMemcpy(*d, h, bytes, cudaMemcpyHostToDevice));
  else NIB_CUDA(cudaMemset(*d, 0, bytes + 256));
  return NIB_OK;
}

static int upload_floats(nib_net* net, const float* h, size_t n, float** d) {
  *d = nullptr;
  if (!h || n == 0) return NIB_OK;
  void* p = nullptr;
  int rc = upload(net, h, n * sizeof(float), &p);
  *d = (float*)p;
  return rc;
}

static inline uint16_t f32_to_bf16_rn(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);  // NaN
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

// w = hi + lo with hi = bf16(w), lo = bf16(w - hi)
static inline void bf16_hi_lo(float w, uint16_t* hi, uint16_t* lo) {
  *hi = f32_to_bf16_rn(w);
  const uint32_t u = (uint32_t)*hi << 16;
  float hf;
  memcpy(&hf, &u, 4);
  *lo = f32_to_bf16_rn(w - hf);
}

static std::vector<uint16_t> to_bf16(const std::vector<float>& v) {
  std::vector<uint16_t> out(v.size());
  for (size_t i = 0; i < v.size(); ++i) out[i] = f32_to_bf16_rn(v[i]);
  return out;
}

// [Cout][Cin][R][S] -> [Cout][Rp][Sp][Cp], zero past the filter's R x S x Cin: KRSC (Rp, Sp, Cp = R, S, Cin), KRSC with
// Cin padded to the K block, and the raw-row layouts of conv_tc.cu
static std::vector<float> to_krsc(const float* w, const nib_conv_desc& d, int Rp, int Sp, int Cp) {
  std::vector<float> out((size_t)d.Cout * Rp * Sp * Cp, 0.f);
  for (int co = 0; co < d.Cout; ++co)
    for (int c = 0; c < d.Cin; ++c)
      for (int r = 0; r < d.R; ++r)
        for (int s = 0; s < d.S; ++s)
          out[(((size_t)co * Rp + r) * Sp + s) * Cp + c] = w[(((size_t)co * d.Cin + c) * d.R + r) * d.S + s];
  return out;
}

extern "C" {

int nib_net_create(int precision, int max_batch, nib_net** out) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(out != nullptr, "nib_net_create: null out");
  NIB_REQUIRE(precision == NIB_PREC_FP32 || precision == NIB_PREC_BF16 || precision == NIB_PREC_X3 || precision == NIB_PREC_SPLIT,
              "nib_net_create: bad precision %d", precision);
  NIB_REQUIRE(max_batch > 0, "nib_net_create: max_batch must be > 0");
  nib_net* n = new nib_net();
  n->precision = precision;
  n->bf16 = precision == NIB_PREC_BF16;
  n->x3 = precision == NIB_PREC_X3;
  n->split = precision == NIB_PREC_SPLIT;
  n->max_batch = max_batch;
  n->input_buf = -1;
  n->pack_scratch = nullptr;
  n->pack_scratch_bytes = 0;
  n->finalized = false;
  n->num_classes = 0;
  n->use_tc = true;
  n->use_graph = false;
  n->dyn_n = nullptr;
  n->graph_logits = nullptr;
  n->launches = n->tc_launches = 0;
  *out = n;
  return NIB_OK;
}

int nib_net_destroy(nib_net* net) {
  if (!net) return NIB_OK;
  for (auto& g : net->graphs) cudaGraphExecDestroy(g.second.exec);
  for (void* p : net->allocs) cudaFree(p);
  for (auto& o : net->ops) {
    if (o.plan) tc_conv_plan_destroy(o.plan);
    if (o.fplan) tc_fused_plan_destroy(o.fplan);
  }
  delete net;
  return NIB_OK;
}

static int add_buffer_kind(nib_net* net, int H, int W, int C, int pad, int kind) {
  NIB_REQUIRE(net && !net->finalized, "nib_net_add_buffer: bad handle/state");
  NIB_REQUIRE(H > 0 && W > 0 && C > 0 && pad >= 0, "nib_net_add_buffer: bad geometry");
  NetBuffer b;
  b.H = H; b.W = W; b.C = C; b.pad = pad;
  b.kind = kind;
  b.elems_per_image = (size_t)(H + 2 * pad) * (W + 2 * pad) * b.phys_c();
  int rc = upload(net, nullptr, b.elems_per_image * net->max_batch * b.esize(), &b.ptr);
  if (rc != NIB_OK) return rc;
  net->bufs.push_back(b);
  return (int)net->bufs.size() - 1;
}

int nib_net_add_buffer(nib_net* net, int H, int W, int C, int pad) {
  NIB_REQUIRE(net != nullptr, "nib_net_add_buffer: null handle");
  return add_buffer_kind(net, H, W, C, pad, net->bf16 ? BUF_BF16 : net->split ? BUF_SPLIT : BUF_F32);
}

int nib_net_add_buffer_f32(nib_net* net, int H, int W, int C, int pad) {
  NIB_REQUIRE(net != nullptr, "nib_net_add_buffer_f32: null handle");
  NIB_REQUIRE(!net->bf16, "nib_net_add_buffer_f32: bf16 networks have bf16 buffers only");
  return add_buffer_kind(net, H, W, C, pad, BUF_F32);
}

int nib_net_add_convert(nib_net* net, int in_buf, int out_buf) {
  NIB_REQUIRE(net && !net->finalized && net->split, "nib_net_add_convert: needs an unfinalized NIB_PREC_SPLIT network");
  const int nb = (int)net->bufs.size();
  NIB_REQUIRE(in_buf >= 0 && in_buf < nb && out_buf >= 0 && out_buf < nb, "nib_net_add_convert: bad buffer id");
  const NetBuffer& bi = net->bufs[in_buf];
  const NetBuffer& bo = net->bufs[out_buf];
  NIB_REQUIRE(bi.H == bo.H && bi.W == bo.W && bi.C == bo.C && bi.pad == 0 && bo.pad == 0, "nib_net_add_convert: geometry mismatch");
  NIB_REQUIRE((bi.kind == BUF_F32 && bo.kind == BUF_SPLIT) || (bi.kind == BUF_SPLIT && bo.kind == BUF_F32),
              "nib_net_add_convert: one side must be fp32, the other split");
  NetOp op = {};
  op.kind = OP_CONVERT;
  op.in_buf = in_buf;
  op.out_buf = out_buf;
  net->ops.push_back(op);
  return NIB_OK;
}

int nib_net_add_conv(nib_net* net, const nib_conv_desc* d, const float* h_weight, const float* h_bias,
                     const float* h_pre_scale, const float* h_pre_shift) {
  NIB_REQUIRE(net && !net->finalized && d && h_weight, "nib_net_add_conv: bad handle/state/args");
  const int nb = (int)net->bufs.size();
  NIB_REQUIRE(d->in_buf >= 0 && d->in_buf < nb && d->out_buf >= 0 && d->out_buf < nb, "nib_net_add_conv: bad buffer id");
  NIB_REQUIRE(d->res_buf < nb, "nib_net_add_conv: bad residual buffer id");
  const NetBuffer& bi = net->bufs[d->in_buf];
  const NetBuffer& bo = net->bufs[d->out_buf];
  NIB_REQUIRE(d->in_coff >= 0 && d->in_coff + d->Cin <= bi.C, "nib_net_add_conv: input channel slice out of range");
  NIB_REQUIRE(d->out_coff >= 0 && d->out_coff + d->Cout <= bo.C, "nib_net_add_conv: output channel slice out of range");
  NIB_REQUIRE(d->R > 0 && d->S > 0 && d->stride > 0 && d->pad >= 0, "nib_net_add_conv: bad filter geometry");
  const int P = (bi.H + 2 * d->pad - d->R) / d->stride + 1;
  const int Q = (bi.W + 2 * d->pad - d->S) / d->stride + 1;
  NIB_REQUIRE(P == bo.H && Q == bo.W, "nib_net_add_conv: output buffer is %dx%d but conv produces %dx%d", bo.H, bo.W, P, Q);
  NIB_REQUIRE(bo.pad == 0, "nib_net_add_conv: output buffers with halo are not supported");
  if (d->res_buf >= 0) {
    const NetBuffer& br = net->bufs[d->res_buf];
    NIB_REQUIRE(br.H == bo.H && br.W == bo.W && br.pad == 0, "nib_net_add_conv: residual geometry mismatch");
    NIB_REQUIRE(d->res_C > 0 && d->res_C <= d->Cout && d->res_coff + d->res_C <= br.C, "nib_net_add_conv: residual channels out of range");
  }
  if (d->flags & NIB_CONV_PRE_BNRELU) NIB_REQUIRE(h_pre_scale && h_pre_shift, "nib_net_add_conv: PRE_BNRELU needs scale/shift");

  NetOp op = {};
  op.kind = OP_CONV;
  op.cd = *d;
  NIB_REQUIRE(bi.kind == bo.kind, "nib_net_add_conv: input and output buffers must have the same kind (use nib_net_add_convert)");
  if (d->res_buf >= 0) NIB_REQUIRE(net->bufs[d->res_buf].kind == bo.kind, "nib_net_add_conv: residual buffer kind mismatch");
  const size_t K = (size_t)d->R * d->S * d->Cin;
  const std::vector<float> krsc = to_krsc(h_weight, *d, d->R, d->S, d->Cin);
  const size_t nel = krsc.size();
  int rc;
  if (bi.kind == BUF_SPLIT) {
    // [Cout][tap][Wh(Cin) | Wh(Cin) | Wl(Cin)]: against activations walked as hi, lo, hi (conv_tc.cu split mode)
    std::vector<uint16_t> hb(nel * 3);
    for (size_t i = 0; i < nel; ++i) {
      uint16_t hi, lo;
      bf16_hi_lo(krsc[i], &hi, &lo);
      const size_t base = i / d->Cin * 3 * d->Cin, c = i % d->Cin;
      hb[base + c] = hi;
      hb[base + d->Cin + c] = hi;
      hb[base + 2 * (size_t)d->Cin + c] = lo;
    }
    rc = upload(net, hb.data(), hb.size() * 2, &op.d_w);
  } else if (net->bf16) {
    rc = upload(net, to_bf16(krsc).data(), nel * 2, &op.d_w);
  } else {
    rc = upload(net, krsc.data(), nel * 4, &op.d_w);
    // Not for reductions longer than NIB_X3_MAX_K: the tensor cores' fp32 accumulation drifts with K (VGG's fc6,
    // K = 25088, measured 1.6e-4 .. 1.9e-4 of the logits' scale against 1e-4 for fp32 grade), so those run on the CUDA cores
    if (rc == NIB_OK && net->x3 && d->Cin % 16 == 0 && K <= NIB_X3_MAX_K) {
      std::vector<uint16_t> hi(nel), lo(nel);
      for (size_t i = 0; i < nel; ++i) bf16_hi_lo(krsc[i], &hi[i], &lo[i]);
      rc = upload(net, hi.data(), nel * 2, &op.d_w_hi);
      if (rc == NIB_OK) rc = upload(net, lo.data(), nel * 2, &op.d_w_lo);
    }
  }
  if (rc != NIB_OK) return rc;
  const RawRowLayout raw = tc_raw_row_layout(d->R, d->S, d->stride, d->pad, d->Cin, bi.phys_c(), bi.pad);
  if (net->bf16 && raw.rows > 0) {
    rc = upload(net, to_bf16(to_krsc(h_weight, *d, raw.rows, raw.taps, raw.ch)).data(), (size_t)d->Cout * raw.k() * 2,
                &op.d_w_alt);
    if (rc != NIB_OK) return rc;
  }
  // BN-ReLU-conv (DenseNet) on the tensor-core path: the conv reads relu(bn(x)) from a packed scratch tensor whose
  // channel count is rounded up to the 64-channel K block, so the weights get the same zero padding along Cin.
  if (net->bf16 && (d->flags & NIB_CONV_PRE_BNRELU) && d->Cin % 8 == 0 && d->in_coff % 8 == 0 && bi.C % 8 == 0 &&
      bi.pad == 0 && d->Cout % 32 == 0) {
    const int cpad = (d->Cin + 63) / 64 * 64;
    rc = upload(net, to_bf16(to_krsc(h_weight, *d, d->R, d->S, cpad)).data(), (size_t)d->Cout * d->R * d->S * cpad * 2,
                &op.d_w_pack);
    if (rc != NIB_OK) return rc;
    op.pack_cin = cpad;
  }
  rc = upload_floats(net, h_bias, d->Cout, &op.d_bias);
  if (rc != NIB_OK) return rc;
  if (d->flags & NIB_CONV_PRE_BNRELU) {
    rc = upload_floats(net, h_pre_scale, d->Cin, &op.d_pre_scale);
    if (rc != NIB_OK) return rc;
    rc = upload_floats(net, h_pre_shift, d->Cin, &op.d_pre_shift);
    if (rc != NIB_OK) return rc;
    if (op.pack_cin) {
      std::vector<float> sp(op.pack_cin, 0.f), hp(op.pack_cin, 0.f);
      for (int c = 0; c < d->Cin; ++c) { sp[c] = h_pre_scale[c]; hp[c] = h_pre_shift[c]; }
      if ((rc = upload_floats(net, sp.data(), sp.size(), &op.d_pre_scale_pad)) != NIB_OK) return rc;
      if ((rc = upload_floats(net, hp.data(), hp.size(), &op.d_pre_shift_pad)) != NIB_OK) return rc;
    }
  }
  net->ops.push_back(op);
  return NIB_OK;
}

int nib_net_add_pool(nib_net* net, int kind, int in_buf, int in_coff, int C, int out_buf, int out_coff, int k,
                     int stride, int pad, const float* h_pre_scale, const float* h_pre_shift) {
  NIB_REQUIRE(net && !net->finalized, "nib_net_add_pool: bad handle/state");
  const int nb = (int)net->bufs.size();
  NIB_REQUIRE(in_buf >= 0 && in_buf < nb && out_buf >= 0 && out_buf < nb, "nib_net_add_pool: bad buffer id");
  NIB_REQUIRE(kind == NIB_POOL_MAX || kind == NIB_POOL_AVG, "nib_net_add_pool: bad kind");
  const NetBuffer& bi = net->bufs[in_buf];
  const NetBuffer& bo = net->bufs[out_buf];
  NIB_REQUIRE(bi.pad == 0 && bo.pad == 0, "nib_net_add_pool: halo buffers unsupported");
  NIB_REQUIRE(bi.kind == bo.kind && bi.kind != BUF_SPLIT, "nib_net_add_pool: pooling runs on fp32 or bf16 buffers (convert split tensors first)");
  NIB_REQUIRE(in_coff + C <= bi.C && out_coff + C <= bo.C, "nib_net_add_pool: channel slice out of range");
  const int P = (bi.H + 2 * pad - k) / stride + 1, Q = (bi.W + 2 * pad - k) / stride + 1;
  NIB_REQUIRE(P == bo.H && Q == bo.W, "nib_net_add_pool: output buffer is %dx%d but pool produces %dx%d", bo.H, bo.W, P, Q);
  NetOp op = {};
  op.kind = OP_POOL;
  op.pool_kind = kind; op.k = k; op.stride = stride; op.pad = pad; op.C = C;
  op.in_buf = in_buf; op.in_coff = in_coff; op.out_buf = out_buf; op.out_coff = out_coff;
  int rc = upload_floats(net, h_pre_scale, C, &op.d_pre_scale);
  if (rc != NIB_OK) return rc;
  rc = upload_floats(net, h_pre_shift, C, &op.d_pre_shift);
  if (rc != NIB_OK) return rc;
  net->ops.push_back(op);
  return NIB_OK;
}

int nib_net_add_fc(nib_net* net, int in_buf, int Cin, int Cout, const float* h_weight, const float* h_bias) {
  NIB_REQUIRE(net && !net->finalized && h_weight, "nib_net_add_fc: bad handle/state/args");
  NIB_REQUIRE(in_buf >= 0 && in_buf < (int)net->bufs.size(), "nib_net_add_fc: bad buffer id");
  const NetBuffer& bi = net->bufs[in_buf];
  NIB_REQUIRE(bi.H == 1 && bi.W == 1 && bi.C >= Cin, "nib_net_add_fc: input must be a 1x1xC feature buffer");
  NIB_REQUIRE(bi.kind != BUF_SPLIT, "nib_net_add_fc: the feature buffer must be fp32 or bf16");
  NetOp op = {};
  op.kind = OP_FC;
  op.fc_in = in_buf; op.fc_cin = Cin; op.fc_cout = Cout;
  float* w = nullptr;
  int rc = upload_floats(net, h_weight, (size_t)Cin * Cout, &w);
  if (rc != NIB_OK) return rc;
  op.d_w = w;
  rc = upload_floats(net, h_bias, Cout, &op.d_bias);
  if (rc != NIB_OK) return rc;
  if (bi.kind == BUF_BF16 && fc_x2_supported(Cin, bi.C)) {   // bf16 features: tensor-core fc on W = hi + lo (conv_x3.cu)
    const size_t nel = (size_t)Cin * Cout;
    std::vector<uint16_t> hi(nel), lo(nel);
    for (size_t i = 0; i < nel; ++i) bf16_hi_lo(h_weight[i], &hi[i], &lo[i]);
    rc = upload(net, hi.data(), nel * 2, &op.d_w_hi);
    if (rc == NIB_OK) rc = upload(net, lo.data(), nel * 2, &op.d_w_lo);
    if (rc != NIB_OK) return rc;
  }
  net->ops.push_back(op);
  net->num_classes = Cout;
  return NIB_OK;
}

int nib_net_set_input(nib_net* net, int buf) {
  NIB_REQUIRE(net && buf >= 0 && buf < (int)net->bufs.size(), "nib_net_set_input: bad buffer id");
  net->input_buf = buf;
  return NIB_OK;
}

// The conv's kernel parameters for N images on the given path
static void fill_conv_params(const nib_net* net, const NetOp& op, ConvPath path, int N, ConvParams* p) {
  const nib_conv_desc& d = op.cd;
  const NetBuffer& bi = net->bufs[d.in_buf];
  const NetBuffer& bo = net->bufs[d.out_buf];
  memset(p, 0, sizeof(*p));
  p->in = bi.ptr;
  p->w = op.d_w;
  p->w_alt = op.d_w_alt;
  p->bias = op.d_bias;
  p->out = bo.ptr;
  p->pre_scale = op.d_pre_scale;
  p->pre_shift = op.d_pre_shift;
  p->Hin = bi.H; p->Win = bi.W; p->Cin = d.Cin; p->in_cstride = bi.phys_c(); p->in_coff = d.in_coff; p->in_halo = bi.pad;
  p->P = bo.H; p->Q = bo.W; p->Cout = d.Cout; p->out_cstride = bo.phys_c(); p->out_coff = d.out_coff; p->out_halo = bo.pad;
  p->split = bi.kind == BUF_SPLIT ? 1 : 0;
  p->in_lo_off = bi.C;
  p->out_lo_off = bo.C;
  p->M = N * bo.H * bo.W;
  if (d.res_buf >= 0) {
    const NetBuffer& br = net->bufs[d.res_buf];
    p->res = br.ptr;
    p->res_cstride = br.phys_c(); p->res_coff = d.res_coff; p->res_C = d.res_C;
    p->res_lo_off = br.C;
  }
  p->R = d.R; p->S = d.S; p->stride = d.stride; p->pad = d.pad;
  p->relu = (d.flags & NIB_CONV_RELU) ? 1 : 0;
  p->dyn_n = net->dyn_n;
  if (path == PATH_TC_XFORM) {
    // the raw channel slice: padded channel count, padded weights, padded scale / shift (channels past Cin come out as
    // exact zeros)
    p->w = op.d_w_pack;
    p->pre_scale = op.d_pre_scale_pad;
    p->pre_shift = op.d_pre_shift_pad;
    p->pre_padded = 1;
    p->Cin = op.pack_cin;
  } else if (path == PATH_TC_PACK) {
    // the packed relu(bn(x)) scratch tensor instead of the raw channel slice
    p->in = net->pack_scratch;
    p->w = op.d_w_pack;
    p->pre_scale = nullptr;
    p->pre_shift = nullptr;
    p->Cin = op.pack_cin;
    p->in_cstride = op.pack_cin;
    p->in_coff = 0;
  }
}

// The conv's paths, in order of preference.  Only tc_conv_supported is consulted: the plans are built afterwards.
static int resolve_paths(const nib_net* net, NetOp& op) {
  static const bool no_xform = getenv("NIB_TC_NO_XFORM") != nullptr;   // A/B: the separate pack pass
  ConvParams p, pt;
  fill_conv_params(net, op, PATH_TC, net->max_batch, &p);
  op.cuda_path = net->x3 && op.d_w_hi && conv_x3_supported(p) ? PATH_X3 : PATH_SIMT;
  op.path = op.cuda_path;
  if (p.split) {
    NIB_REQUIRE(tc_conv_supported(p), "nib_net_finalize: a conv on split tensors needs Cin %% 64 == 0, Cout %% 64 == 0, whole-buffer channel ranges (Cin=%d Cout=%d)", p.Cin, p.Cout);
    op.path = PATH_TC;
  } else if (net->bf16 && op.pack_cin) {
    fill_conv_params(net, op, PATH_TC_XFORM, net->max_batch, &pt);
    if (!no_xform && tc_conv_supported(pt)) {
      op.path = PATH_TC_XFORM;
    } else {
      fill_conv_params(net, op, PATH_TC_PACK, net->max_batch, &pt);
      if (tc_conv_supported(pt)) op.path = PATH_TC_PACK;
    }
  } else if (net->bf16 && tc_conv_supported(p)) {
    op.path = PATH_TC;
  }
  return NIB_OK;
}

int nib_net_finalize(nib_net* net) {
  NIB_REQUIRE(net && !net->finalized, "nib_net_finalize: bad handle/state");
  NIB_REQUIRE(net->input_buf >= 0, "nib_net_finalize: input buffer not set");
  NIB_REQUIRE(!net->ops.empty() && net->ops.back().kind == OP_FC, "nib_net_finalize: the last op must be the fc layer");
  int rc;
  for (auto& op : net->ops) {
    if (op.kind != OP_CONV) continue;
    if ((rc = resolve_paths(net, op)) != NIB_OK) return rc;
    if (op.path == PATH_TC_PACK) {
      const NetBuffer& bi = net->bufs[op.cd.in_buf];
      const size_t need = (size_t)net->max_batch * bi.H * bi.W * op.pack_cin * 2;
      if (need > net->pack_scratch_bytes) net->pack_scratch_bytes = need;
    }
  }
  // one scratch tensor serves every packed pre-activation conv (ops run one at a time on the stream); the plans of those
  // convs read it, so it exists before they are built
  if (net->pack_scratch_bytes && (rc = upload(net, nullptr, net->pack_scratch_bytes, &net->pack_scratch)) != NIB_OK) return rc;
  for (auto& op : net->ops) {
    if (op.kind != OP_CONV || !on_tcgen05(op.path)) continue;
    ConvParams p;
    fill_conv_params(net, op, op.path, net->max_batch, &p);
    rc = tc_conv_plan_create(p, net->max_batch, &op.plan);
    if (rc != NIB_OK) {
      if (op.path != PATH_TC || op.d_w_alt == nullptr) return rc;
      op.path = op.cuda_path;   // the raw-row modes are optional: the CUDA-core kernel covers the conv
    }
  }
  for (size_t i = 0; i + 1 < net->ops.size(); ++i) {
    NetOp& c = net->ops[i];
    NetOp& a = net->ops[i + 1];
    if (c.kind != OP_CONV || a.kind != OP_CONV || c.path != PATH_TC || a.path != PATH_TC) continue;
    ConvParams pc, pa;
    fill_conv_params(net, c, PATH_TC, net->max_batch, &pc);
    fill_conv_params(net, a, PATH_TC, net->max_batch, &pa);
    if (!tc_fuse_supported(pc, pa)) continue;
    if ((rc = tc_fused_plan_create(pc, pa, net->max_batch, &c.fplan)) != NIB_OK) return rc;
    c.path = PATH_FUSED_HEAD;
    a.path = PATH_FUSED_TAIL;
  }
  net->finalized = true;
  return NIB_OK;
}

static int run_conv(nib_net* net, size_t i, int N, cudaStream_t st) {
  const NetOp& op = net->ops[i];
  const ConvPath path = net->use_tc ? op.path : op.cuda_path;
  if (path == PATH_FUSED_TAIL) return NIB_OK;
  ConvParams p;
  fill_conv_params(net, op, path, N, &p);
  int rc = NIB_OK;
  switch (path) {
    case PATH_FUSED_HEAD: {
      ConvParams pa;
      fill_conv_params(net, net->ops[i + 1], PATH_FUSED_TAIL, N, &pa);
      rc = tc_fused_launch(op.fplan, p, pa, st);
      break;
    }
    case PATH_TC_PACK: {
      const NetBuffer& bi = net->bufs[op.cd.in_buf];
      rc = launch_bnrelu_pack(bi.ptr, bi.C, op.cd.in_coff, op.cd.Cin, op.pack_cin, op.d_pre_scale, op.d_pre_shift,
                              net->pack_scratch, (long long)N * bi.H * bi.W, st);
      net->launches++;
      if (rc != NIB_OK) return rc;
      rc = tc_conv_launch(op.plan, p, st);
      break;
    }
    case PATH_TC:
    case PATH_TC_XFORM:
      rc = tc_conv_launch(op.plan, p, st);
      break;
    case PATH_X3:
      rc = launch_conv_x3(p, op.d_w_hi, op.d_w_lo, st);
      break;
    default:
      rc = launch_conv_simt(p, net->bf16, st);
      break;
  }
  if (on_tcgen05(path)) net->tc_launches++;
  net->launches++;
  return rc;
}

// ops [begin, end) on N images
static int run_ops(nib_net* net, size_t begin, size_t end, int N, float* d_logits, cudaStream_t st) {
  for (size_t i = begin; i < end; ++i) {
    const NetOp& op = net->ops[i];
    int rc = NIB_OK;
    switch (op.kind) {
      case OP_CONV:
        rc = run_conv(net, i, N, st);
        break;
      case OP_CONVERT: {
        const NetBuffer& bi = net->bufs[op.in_buf];
        const NetBuffer& bo = net->bufs[op.out_buf];
        rc = launch_split_convert(bi.ptr, bo.ptr, (long long)N * bi.H * bi.W, bi.C, bi.kind == BUF_F32, net->dyn_n, bi.H * bi.W, st);
        net->launches++;
        break;
      }
      case OP_POOL: {
        const NetBuffer& bi = net->bufs[op.in_buf];
        const NetBuffer& bo = net->bufs[op.out_buf];
        PoolParams p;
        memset(&p, 0, sizeof(p));
        p.in = bi.ptr; p.out = bo.ptr;
        p.pre_scale = op.d_pre_scale; p.pre_shift = op.d_pre_shift;
        p.kind = op.pool_kind; p.N = N; p.Hin = bi.H; p.Win = bi.W; p.C = op.C;
        p.in_cstride = bi.C; p.in_coff = op.in_coff;
        p.P = bo.H; p.Q = bo.W; p.out_cstride = bo.C; p.out_coff = op.out_coff;
        p.k = op.k; p.stride = op.stride; p.pad = op.pad;
        p.dyn_n = net->dyn_n;
        rc = launch_pool(p, bi.kind == BUF_BF16, st);
        net->launches++;
        break;
      }
      case OP_FC: {
        const NetBuffer& bi = net->bufs[op.fc_in];
        static const bool fc_simt = getenv("NIB_FC_SIMT") != nullptr;   // A/B: the CUDA-core SGEMM
        rc = (op.d_w_hi && !fc_simt)
                 ? launch_fc_x2(bi.ptr, bi.C, op.d_w_hi, op.d_w_lo, op.d_bias, N, op.fc_cin, op.fc_cout, d_logits, net->dyn_n, st)
                 : launch_fc(bi.ptr, bi.C, bi.kind == BUF_BF16, (const float*)op.d_w, op.d_bias, N, op.fc_cin, op.fc_cout,
                             d_logits, net->dyn_n, st);
        net->launches++;
        break;
      }
    }
    if (rc != NIB_OK) return rc;
  }
  return NIB_OK;
}

static int stage_input(nib_net* net, const void* d_x, int x_layout, int N, cudaStream_t st) {
  const NetBuffer& bi = net->bufs[net->input_buf];
  NIB_REQUIRE(bi.kind != BUF_SPLIT, "nib_net_forward: the input buffer of a split network must be fp32 (nib_net_add_buffer_f32)");
  if (x_layout == NIB_IN_NCHW_F32) {
    // the reference hands an N x C x H x W fp32 tensor (imagenet :245); channels beyond the model's
    // real C are zero padding for the tensor-core path.
    int C = bi.C;
    // real channel count = Cin of the first conv reading this buffer
    for (auto& op : net->ops)
      if (op.kind == OP_CONV && op.cd.in_buf == net->input_buf) { C = op.cd.Cin; break; }
    int rc = launch_nchw_to_nhwc((const float*)d_x, N, C, bi.H, bi.W, bi.ptr, bi.C, bi.pad, net->bf16, st);
    net->launches++;
    return rc;
  }
  if (d_x != bi.ptr)
    NIB_CUDA(cudaMemcpyAsync(bi.ptr, d_x, bi.elems_per_image * N * bi.esize(), cudaMemcpyDeviceToDevice, st));
  return NIB_OK;
}

int nib_net_forward(nib_net* net, const void* d_x, int x_layout, int N, float* d_logits, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(net && net->finalized, "nib_net_forward: network not finalized");
  NIB_REQUIRE(d_x && d_logits, "nib_net_forward: null pointer");
  NIB_REQUIRE(N > 0 && N <= net->max_batch, "nib_net_forward: N=%d outside (0, max_batch=%d]", N, net->max_batch);
  NIB_REQUIRE(x_layout == NIB_IN_NCHW_F32 || x_layout == NIB_IN_NATIVE, "nib_net_forward: bad x_layout");
  cudaStream_t st = (cudaStream_t)stream;
  if (!net->use_graph) {
    int rc = stage_input(net, d_x, x_layout, N, st);
    if (rc != NIB_OK) return rc;
    return run_ops(net, 0, net->ops.size(), N, d_logits, st);
  }
  int rc = stage_input(net, d_x, x_layout, N, st);
  if (rc != NIB_OK) return rc;
  if (!net->graph_logits) {
    void* p = nullptr;
    rc = upload(net, nullptr, sizeof(float) * (size_t)net->max_batch * (net->num_classes > 0 ? net->num_classes : 1), &p);
    if (rc != NIB_OK) return rc;
    net->graph_logits = (float*)p;
  }
  auto it = net->graphs.find(N);
  if (it == net->graphs.end()) {
    if (net->graphs.size() >= nib_net::kMaxGraphs) {
      for (auto& g : net->graphs) cudaGraphExecDestroy(g.second.exec);
      net->graphs.clear();
    }
    cudaStream_t cap;
    NIB_CUDA(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
    const long long l0 = net->launches, t0 = net->tc_launches;
    NIB_CUDA(cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal));
    rc = run_ops(net, 0, net->ops.size(), N, net->graph_logits, cap);
    cudaGraph_t graph = nullptr;
    cudaError_t ce = cudaStreamEndCapture(cap, &graph);
    if (rc != NIB_OK || ce != cudaSuccess) {
      if (graph) cudaGraphDestroy(graph);
      cudaStreamDestroy(cap);
      if (rc == NIB_OK) { set_error("cudaStreamEndCapture: %s", cudaGetErrorString(ce)); rc = NIB_ECUDA; }
      return rc;
    }
    nib_net::GraphVal val;
    val.launches = net->launches - l0;
    val.tc_launches = net->tc_launches - t0;
    net->launches = l0;
    net->tc_launches = t0;
    NIB_CUDA(cudaGraphInstantiate(&val.exec, graph, 0));
    cudaGraphDestroy(graph);
    cudaStreamDestroy(cap);
    it = net->graphs.insert({N, val}).first;
  }
  NIB_CUDA(cudaGraphLaunch(it->second.exec, st));
  NIB_CUDA(cudaMemcpyAsync(d_logits, net->graph_logits, sizeof(float) * (size_t)N * net->num_classes, cudaMemcpyDeviceToDevice, st));
  net->launches += it->second.launches;
  net->tc_launches += it->second.tc_launches;
  return NIB_OK;
}

int nib_net_profile(nib_net* net, int N, float* h_ms, int* h_kind, double* h_flops, int* h_geom, int cap,
                    int* num_ops, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(net && net->finalized && h_ms && h_kind && h_flops && num_ops, "nib_net_profile: bad arguments");
  NIB_REQUIRE(N > 0 && N <= net->max_batch, "nib_net_profile: bad N");
  const int nops = (int)net->ops.size();
  NIB_REQUIRE(cap >= nops, "nib_net_profile: cap=%d < %d ops", cap, nops);
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<cudaEvent_t> ev(nops + 1);
  for (auto& e : ev) NIB_CUDA(cudaEventCreate(&e));
  float* d_logits = nullptr;
  NIB_CUDA(cudaMalloc(&d_logits, sizeof(float) * (size_t)N * (net->num_classes > 0 ? net->num_classes : 1)));
  int rc = NIB_OK;
  for (int i = 0; i < nops && rc == NIB_OK; ++i) {
    cudaEventRecord(ev[i], st);
    rc = run_ops(net, i, i + 1, N, d_logits, st);
  }
  cudaEventRecord(ev[nops], st);
  cudaError_t ce = cudaStreamSynchronize(st);
  if (rc == NIB_OK && ce != cudaSuccess) { set_error("nib_net_profile: %s", cudaGetErrorString(ce)); rc = NIB_ECUDA; }
  for (int i = 0; i < nops && rc == NIB_OK; ++i) {
    cudaEventElapsedTime(&h_ms[i], ev[i], ev[i + 1]);
    const NetOp& op = net->ops[i];
    if (op.kind == OP_CONV) {
      const NetBuffer& bo = net->bufs[op.cd.out_buf];
      const ConvPath path = net->use_tc ? op.path : op.cuda_path;
      // 4: a tcgen05 conv computed by the PREVIOUS op's fused launch (its own slot only holds event overhead)
      h_kind[i] = path == PATH_FUSED_TAIL ? 4 : on_tcgen05(path) ? 1 : 0;
      h_flops[i] = 2.0 * N * bo.H * bo.W * (double)op.cd.R * op.cd.S * op.cd.Cin * op.cd.Cout;
      if (h_geom) {
        int* g = h_geom + 8 * i;
        g[0] = bo.H; g[1] = bo.W; g[2] = op.cd.Cin; g[3] = op.cd.Cout; g[4] = op.cd.R; g[5] = op.cd.stride;
        g[6] = op.cd.res_buf >= 0; g[7] = op.plan ? tc_conv_plan_block_n(op.plan) : 0;
      }
    } else if (op.kind == OP_POOL || op.kind == OP_CONVERT) {
      h_kind[i] = 2;
      h_flops[i] = 0.0;
      if (h_geom) {
        const NetBuffer& bo = net->bufs[op.out_buf];
        int* g = h_geom + 8 * i;
        g[0] = bo.H; g[1] = bo.W; g[2] = bo.C; g[3] = bo.C; g[4] = op.kind == OP_POOL ? op.k : 0; g[5] = op.kind == OP_POOL ? op.stride : 1; g[6] = 0; g[7] = 0;
      }
    } else {
      h_kind[i] = 3;
      h_flops[i] = 2.0 * N * (double)op.fc_cin * op.fc_cout;
      if (h_geom) {
        int* g = h_geom + 8 * i;
        g[0] = 1; g[1] = 1; g[2] = op.fc_cin; g[3] = op.fc_cout; g[4] = 1; g[5] = 1; g[6] = 0; g[7] = 0;
      }
    }
  }
  *num_ops = nops;
  for (auto& e : ev) cudaEventDestroy(e);
  cudaFree(d_logits);
  return rc;
}

int nib_net_forward_masked(nib_net* net, const nib_mask_args* args, float* d_logits, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(net && net->finalized && args, "nib_net_forward_masked: bad handle/args");
  NIB_REQUIRE(args->N > 0 && args->N <= net->max_batch, "nib_net_forward_masked: N=%d outside (0, max_batch=%d]",
              args->N, net->max_batch);
  const NetBuffer& bi = net->bufs[net->input_buf];
  NIB_REQUIRE(args->H == bi.H && args->W == bi.W && args->C <= bi.C, "nib_net_forward_masked: image %dx%dx%d does not match the network input %dx%dx%d",
              args->C, args->H, args->W, bi.C, bi.H, bi.W);
  nib_mask_args a = *args;
  a.d_out = bi.ptr;
  a.out_dtype = net->bf16 ? NIB_BF16 : NIB_F32;
  a.layout = NIB_NHWC;
  a.c_stride = bi.C;
  a.pad_h = a.pad_w = bi.pad;
  // the input buffer's halo ring was zeroed by nib_net_add_buffer and no op writes it: skip the per-forward re-zeroing
  int rc = mask_synth_impl(&a, (cudaStream_t)stream, true, net->dyn_n);
  net->launches += 1;
  if (rc != NIB_OK) return rc;
  return nib_net_forward(net, bi.ptr, NIB_IN_NATIVE, args->N, d_logits, stream);
}

int nib_net_buffer_info(nib_net* net, int buf, void** d_ptr, int* H, int* W, int* C, int* pad, int* dtype) {
  NIB_REQUIRE(net && buf >= 0 && buf < (int)net->bufs.size(), "nib_net_buffer_info: bad buffer id");
  const NetBuffer& b = net->bufs[buf];
  if (d_ptr) *d_ptr = b.ptr;
  if (H) *H = b.H;
  if (W) *W = b.W;
  if (C) *C = b.C;
  if (pad) *pad = b.pad;
  if (dtype) *dtype = b.kind == BUF_F32 ? NIB_F32 : b.kind == BUF_BF16 ? NIB_BF16 : 2 /* split: bf16 [hi | lo] */;
  return NIB_OK;
}

int nib_net_read_buffer_nchw(nib_net* net, int buf, int N, float* d_out, void* stream) {
  NIB_DEVICE_OR_FAIL();
  NIB_REQUIRE(net && buf >= 0 && buf < (int)net->bufs.size() && d_out, "nib_net_read_buffer_nchw: bad arguments");
  NIB_REQUIRE(N > 0 && N <= net->max_batch, "nib_net_read_buffer_nchw: bad N");
  const NetBuffer& b = net->bufs[buf];
  NIB_REQUIRE(b.kind != BUF_SPLIT, "nib_net_read_buffer_nchw: convert a split buffer to fp32 first (nib_net_add_convert)");
  return launch_nhwc_to_nchw(b.ptr, N, b.C, b.H, b.W, b.C, b.pad, b.kind == BUF_BF16, d_out, (cudaStream_t)stream);
}

int nib_net_launch_counts(nib_net* net, long long* total, long long* tcgen05) {
  NIB_REQUIRE(net != nullptr, "nib_net_launch_counts: null handle");
  if (total) *total = net->launches;
  if (tcgen05) *tcgen05 = net->tc_launches;
  return NIB_OK;
}

int nib_net_set_tensor_core(nib_net* net, int enable) {
  NIB_REQUIRE(net != nullptr, "nib_net_set_tensor_core: null handle");
  NIB_REQUIRE(enable || !net->split, "nib_net_set_tensor_core: split-bf16 tensors exist only on the tensor path");
  net->use_tc = enable != 0;
  for (auto& g : net->graphs) cudaGraphExecDestroy(g.second.exec);
  net->graphs.clear();
  return NIB_OK;
}

int nib_net_set_dynamic_batch(nib_net* net, const int32_t* d_count) {
  NIB_REQUIRE(net != nullptr, "nib_net_set_dynamic_batch: null handle");
  NIB_REQUIRE(d_count == nullptr || !net->bf16, "nib_net_set_dynamic_batch: only fp32 / x3 networks honour a device-side batch size");
  net->dyn_n = d_count;
  for (auto& g : net->graphs) cudaGraphExecDestroy(g.second.exec);
  net->graphs.clear();
  return NIB_OK;
}

int nib_net_set_graph(nib_net* net, int enable) {
  NIB_REQUIRE(net != nullptr, "nib_net_set_graph: null handle");
  net->use_graph = enable != 0;
  return NIB_OK;
}

}  // extern "C"
