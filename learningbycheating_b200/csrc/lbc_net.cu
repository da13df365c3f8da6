// lbc_net.cu -- graph executor: builds the layer plan of ImagePolicyModelSS('resnet34') /
// BirdViewPolicyModelSS('resnet18') and runs forward / backward over NHWC activations in HBM.
// Reference call stack being replaced: SURVEY.md 3.3 (image.py:64-89, resnet.py:148-159,38-54).
#include "lbc_net.h"

#include <algorithm>
#include <type_traits>

#include "lbc_fast.h"
#include "lbc_head.h"

namespace lbc {

namespace ref {
struct k_nhwc_to_nchw;
template <class T>
void nhwc_to_nchw_f32(lbc_stream_t s, const T* x, float* out, int N, int H, int W, int C) {
  int64_t n = (int64_t)N * C * H * W;
  par_for<k_nhwc_to_nchw>(s, n, [=] LBC_LAMBDA(int64_t i) {
    int w = (int)(i % W);
    int64_t t = i / W;
    int h = (int)(t % H);
    t /= H;
    int c = (int)(t % C);
    int b = (int)(t / C);
    out[i] = ldf(x, (((int64_t)b * H + h) * W + w) * C + c);
  });
}
}  // namespace ref

#ifndef LBC_HOST_EMU
void NetBase::infer_drop_graphs() {
  for (InferGraph& g : infer_graphs)
    if (g.exec) cudaGraphExecDestroy((cudaGraphExec_t)g.exec);
  infer_graphs.clear();
  packs_current = false;
}
void NetBase::infer_release() {
  infer_drop_graphs();
  for (void* p : {(void*)inf_img, (void*)inf_speed, (void*)inf_onehot, (void*)inf_pred, (void*)inf_preds, (void*)inf_img_u8})
    if (p) cudaFree(p);
  inf_img = inf_speed = inf_onehot = inf_pred = inf_preds = nullptr;
  inf_img_u8 = nullptr;
  if (infer_ev_in) cudaEventDestroy((cudaEvent_t)infer_ev_in);
  if (infer_ev_out) cudaEventDestroy((cudaEvent_t)infer_ev_out);
  if (infer_stream) cudaStreamDestroy((cudaStream_t)infer_stream);
  infer_ev_in = infer_ev_out = infer_stream = nullptr;
}
void NetBase::infer(const float* image, const uint8_t* image_u8, int layout, const float* speed, const float* onehot, int B,
                    bool weights_changed, float* out_pred, float* out_preds, lbc_stream_t s) {
  LBC_CHECK((image != nullptr) != (image_u8 != nullptr), "lbc_net_infer: exactly one of image / image_u8");
  LBC_CHECK(speed && onehot, "lbc_net_infer: null input");
  LBC_CHECK(B >= 1 && B <= max_batch, "lbc_net_infer: batch " + std::to_string(B) + " outside [1, max_batch]");
  LBC_CHECK(P && BUF, "lbc_net_infer: parameters not bound");
  const int64_t img_n = (int64_t)max_batch * in_ch * in_h * in_w;
  if (!infer_stream) {
    cudaStream_t st;
    cudaEvent_t e0, e1;
    LBC_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    LBC_CUDA(cudaEventCreateWithFlags(&e0, cudaEventDisableTiming));
    LBC_CUDA(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
    infer_stream = st;
    infer_ev_in = e0;
    infer_ev_out = e1;
    LBC_CUDA(cudaMalloc((void**)&inf_speed, sizeof(float) * max_batch));
    LBC_CUDA(cudaMalloc((void**)&inf_onehot, sizeof(float) * max_batch * 4));
    LBC_CUDA(cudaMalloc((void**)&inf_pred, sizeof(float) * max_batch * 10));
    LBC_CUDA(cudaMalloc((void**)&inf_preds, sizeof(float) * max_batch * 40));
  }
  if (image && !inf_img) LBC_CUDA(cudaMalloc((void**)&inf_img, sizeof(float) * img_n));
  if (image_u8 && !inf_img_u8) LBC_CUDA(cudaMalloc((void**)&inf_img_u8, (size_t)img_n));
  cudaStream_t is = (cudaStream_t)infer_stream;
  lbc_stream_t ls = (lbc_stream_t)infer_stream;
  // join the caller's stream, stage the inputs at fixed addresses
  LBC_CUDA(cudaEventRecord((cudaEvent_t)infer_ev_in, (cudaStream_t)s));
  LBC_CUDA(cudaStreamWaitEvent(is, (cudaEvent_t)infer_ev_in, 0));
  const int64_t n_img = (int64_t)B * in_ch * in_h * in_w;
  if (image) dev_copy(inf_img, image, sizeof(float) * n_img, ls);
  if (image_u8) dev_copy(inf_img_u8, image_u8, (size_t)n_img, ls);
  dev_copy(inf_speed, speed, sizeof(float) * B, ls);
  dev_copy(inf_onehot, onehot, sizeof(float) * B * 4, ls);
  if (weights_changed || !packs_current) {
    repack(ls);
    packs_current = true;
  }
  const int kind_in = image ? 0 : 1;
  const int variant = (fast::enabled() ? 1 : 0) | (fast::pair_mode() << 1);
  InferGraph* g = nullptr;
  for (InferGraph& c : infer_graphs)
    if (c.B == B && c.kind == kind_in && c.layout == layout && c.variant == variant) g = &c;
  auto run = [&] {
    const bool keep = packs_current;
    skip_pack = true;
    try {
      if (image)
        forward(inf_img, inf_speed, inf_onehot, B, false, inf_pred, inf_preds, ls);
      else
        forward_u8(inf_img_u8, layout, inf_speed, inf_onehot, B, false, inf_pred, inf_preds, ls);
    } catch (...) {
      skip_pack = false;
      throw;
    }
    skip_pack = false;
    packs_current = keep;
  };
  if (!g || infer_no_graph) {
    const bool prof = g_prof_on;
    g_prof_on = false;   // (event brackets cannot be captured)
    try {
      run();   // eager: this call's result, and every one-time attribute / occupancy query / lazy allocation of the path
    } catch (...) {
      g_prof_on = prof;
      throw;
    }
    if (!infer_no_graph) {
      // capture the same call sequence; a path that cannot be captured keeps running eagerly (results are the eager run's)
      cudaGraphExec_t exec = nullptr;
      bool ok = cudaStreamBeginCapture(is, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
      if (ok) {
        try {
          run();
        } catch (...) {
          ok = false;
        }
        cudaGraph_t graph = nullptr;
        if (cudaStreamEndCapture(is, &graph) != cudaSuccess || !graph) ok = false;
        if (ok && cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) ok = false;
        if (graph) cudaGraphDestroy(graph);
      }
      if (ok && exec) {
        InferGraph ng;
        ng.B = B;
        ng.kind = kind_in;
        ng.layout = layout;
        ng.variant = variant;
        ng.exec = exec;
        infer_graphs.push_back(ng);
      } else {
        cudaGetLastError();
        infer_no_graph = true;
      }
    }
    g_prof_on = prof;
  } else {
    LBC_CUDA(cudaGraphLaunch((cudaGraphExec_t)g->exec, is));
    ++infer_replays;
  }
  if (out_preds) dev_copy(out_preds, inf_preds, sizeof(float) * B * 40, ls);
  if (out_pred) dev_copy(out_pred, inf_pred, sizeof(float) * B * 10, ls);
  LBC_CUDA(cudaEventRecord((cudaEvent_t)infer_ev_out, is));
  LBC_CUDA(cudaStreamWaitEvent((cudaStream_t)s, (cudaEvent_t)infer_ev_out, 0));
}
#else
void NetBase::infer_drop_graphs() {}
void NetBase::infer_release() {}
void NetBase::infer(const float* image, const uint8_t* image_u8, int layout, const float* speed, const float* onehot, int B,
                    bool, float* out_pred, float* out_preds, lbc_stream_t s) {
  LBC_CHECK((image != nullptr) != (image_u8 != nullptr), "lbc_net_infer: exactly one of image / image_u8");
  if (image)
    forward(image, speed, onehot, B, false, out_pred, out_preds, s);
  else
    forward_u8(image_u8, layout, speed, onehot, B, false, out_pred, out_preds, s);
}
#endif

void NetBase::enable_grad_events(bool on) {
#ifndef LBC_HOST_EMU
  for (GradBucket& b : buckets) {
    if (on && !b.event) {
      cudaEvent_t e;
      LBC_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      b.event = e;
    }
  }
#endif
  grad_events = on;
}
void NetBase::stream_wait_bucket(int bucket, lbc_stream_t s) {
  LBC_CHECK(bucket >= 0 && bucket < (int)buckets.size(), "gradient bucket index out of range");
  LBC_CHECK(grad_events, "gradient events are not enabled (lbc_net_enable_grad_events)");
#ifndef LBC_HOST_EMU
  LBC_CUDA(cudaStreamWaitEvent(s, (cudaEvent_t)buckets[bucket].event, 0));
#else
  (void)s;
#endif
}

static const float kBnEps = 1e-5f;
static const float kBnMomentum = 0.1f;

template <class T>
class Net : public NetBase {
 public:
  struct Block {
    ConvL c1, c2, cd;
    BNL b1, b2, bd;
    bool ds = false;
    int Cin, Cout, Hin, Win, Hout, Wout;
    T *r1 = nullptr, *a1 = nullptr, *r2 = nullptr, *rd = nullptr, *idn = nullptr, *out = nullptr;
    bool obits_ok = false;
    uint8_t* obits = nullptr;   // bf16 path: (out > 0) as one bit per element, written by bn2's apply kernel; the three
                                // backward consumers of that mask read 1/16 of the bytes of `out`
    const T* xin = nullptr;
    std::string name;
  };
  std::vector<void*> allocs;
  ConvL stem;
  BNL stem_bn;
  int stem_oh, stem_ow, pool_h, pool_w;
  T *x0 = nullptr, *r_stem = nullptr, *a_stem = nullptr, *pool = nullptr;
  uint8_t* pool_idx = nullptr;
  // bf16 fast path of the stem: im2col columns [B,OH,OW,Kp] + a 1x1 "conv" descriptor over them
  T* stem_col = nullptr;
  ConvL stem_gemm;
  float* stem_dw_col = nullptr;
  bool stem_fast_used = false;
  // C_in <= 4: zero-padded NHWC4 bf16 image + overlapping-window TMA instead of the column tensor
  T* stem_x4 = nullptr;
  T* stem_w224 = nullptr;
  bool stem_direct_used = false;
  int stem_layout = 0;   // fast::stem_ch code of stem_x4 / stem_w224 (4, 8, 16)
  std::vector<Block> blocks;
  int trunk_h, trunk_w;
  BNL dbn[3];
  ConvL dcv[3];
  T *dec_in[3], *dec_bn[3], *dec_out[3];
  BNL hbn[4];
  int64_t hw_off[4], hb_off[4];
  float *logits = nullptr, *dlogits = nullptr, *rowmax = nullptr, *rowsum = nullptr, *preds = nullptr;
  float *onehot_saved = nullptr, *speed_saved = nullptr;
  double* headS = nullptr;
  T* g[4];
  // ---- backward overlap (bf16 throughput mode): the weight gradients leave the dependency chain of backward() -- nothing
  // but the optimizer reads them -- so they run on a second, low-priority stream while the chain (BatchNorm backward ->
  // data gradient -> BatchNorm backward ...) runs on a high-priority one.  The HBM-bound BatchNorm / elementwise kernels of
  // the chain then share the SMs with tensor-bound weight-gradient GEMMs, and weight-gradient CTAs fill the partial last
  // wave of the persistent data-gradient GEMMs.  d(r2) / d(r1) / d(rd), the gradients a weight-gradient GEMM reads, rotate
  // through kRing extra buffers so that the chain does not have to wait for the side stream before it moves on; every
  // buffer carries the event of its last side-stream reader, waited for before the chain overwrites it (wr()).
  static constexpr int kRing = 8;   // allocated; ring_n of them rotate (LBC_RING)
  int ring_n = 4;
  T* gring[kRing] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  bool ovl_capable = false;   // ring buffers + streams exist
  bool ovl = false;           // the running backward() uses them
  int ring_next = 0;
#ifndef LBC_HOST_EMU
  cudaStream_t side_stream = nullptr, chain_stream = nullptr;
  cudaEvent_t ev_ready = nullptr, ev_join = nullptr, ev_in = nullptr, ev_out = nullptr;
  cudaEvent_t gdone[4 + kRing] = {};
#endif
  bool gpending[4 + kRing] = {};
  int gindex(const T* p) const {
    for (int i = 0; i < 4; ++i)
      if (p == g[i]) return i;
    for (int i = 0; i < kRing; ++i)
      if (p == gring[i]) return 4 + i;
    return -1;
  }
  // the chain is about to overwrite gradient buffer p: wait for its last side-stream reader
  T* wr(T* p, lbc_stream_t s) {
#ifndef LBC_HOST_EMU
    if (ovl) {
      const int i = gindex(p);
      if (i >= 0 && gpending[i]) {
        LBC_CUDA(cudaStreamWaitEvent(s, gdone[i], 0));
        gpending[i] = false;
      }
    }
#else
    (void)s;
#endif
    return p;
  }
  // next buffer for a gradient that a side-stream weight gradient will read (serial mode: the caller's fallback)
  T* ring(T* fallback, lbc_stream_t s) {
    if (!ovl) return fallback;
    T* p = gring[ring_next];
    ring_next = (ring_next + 1) % ring_n;
    return wr(p, s);
  }
  // everything enqueued on the chain so far is what the next side-stream weight gradient depends on
  void mark_ready(lbc_stream_t s) {
#ifndef LBC_HOST_EMU
    if (ovl) LBC_CUDA(cudaEventRecord(ev_ready, s));
#else
    (void)s;
#endif
  }
  // weight gradient of conv c: on the side stream after the last mark_ready() (overlap mode) or in line on s
  void wgrad_side(const ConvL& c, const T* x, const T* dy, int B, lbc_stream_t s, bool x_is_grad, const T* gbuf) {
#ifndef LBC_HOST_EMU
    if (ovl) {
      LBC_CUDA(cudaStreamWaitEvent(side_stream, ev_ready, 0));
      conv_backward_weight(c, x, dy, B, side_stream, x_is_grad);
      const int i = gindex(gbuf);
      LBC_CHECK(i >= 0, "wgrad_side: operand is not a gradient buffer");
      LBC_CUDA(cudaEventRecord(gdone[i], side_stream));
      gpending[i] = true;
      return;
    }
#else
    (void)gbuf;
#endif
    conv_backward_weight(c, x, dy, B, s, x_is_grad);
  }
  // all side-stream work enqueued so far completes before anything enqueued on s from here on
  void join_side(lbc_stream_t s) {
#ifndef LBC_HOST_EMU
    if (!ovl) return;
    LBC_CUDA(cudaEventRecord(ev_join, side_stream));
    LBC_CUDA(cudaStreamWaitEvent(s, ev_join, 0));
    for (bool& b : gpending) b = false;
#else
    (void)s;
#endif
  }
  float* ws_f = nullptr;
  int64_t ws_f_n = 0;
  double* ws_d = nullptr;
  float* bn_sums = nullptr;  // 2*C floats scratch of the fast BN kernels
  float* negshift_all = nullptr;  // [n_buffers] (indexed like the running_mean entries)
  std::vector<ref::PackEntry> pack_host;
  ref::PackEntry* pack_dev = nullptr;
  std::vector<BNL*> conv_bns;     // BNs fed directly by a trunk convolution
  float* head_fold = nullptr;  // folded BN+1x1 map A[20][64], b'[20]; coef c0/c1 [128]
  bool stem_pool_fused = false;
  // PREC_F32TC (T = float): convolutions on the tensor cores with split-precision operands
  bool mask_bits_valid = false;   // the last bn_forward call wrote its mask bits (fast bf16 path)
  bool tc = false;
  fast::TcWork tcw;
  bool stem_tc_used = false;
  size_t total_bytes = 0;
  int cur_B = 0;
  bool cur_train = false;
  bool normalize = false;

  template <class U>
  U* alloc(int64_t n) {
    size_t bytes = (size_t)n * sizeof(U);
    void* p = dev_alloc(bytes);
    allocs.push_back(p);
    total_bytes += bytes;
    return (U*)p;
  }
  ~Net() override {
    for (void* p : allocs) dev_free(p);
#ifndef LBC_HOST_EMU
    for (GradBucket& b : buckets)
      if (b.event) cudaEventDestroy((cudaEvent_t)b.event);
    if (side_stream) {
      cudaStreamSynchronize(side_stream);
      cudaStreamDestroy(side_stream);
    }
    if (chain_stream) {
      cudaStreamSynchronize(chain_stream);
      cudaStreamDestroy(chain_stream);
    }
    for (cudaEvent_t e : {ev_ready, ev_join, ev_in, ev_out})
      if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : gdone)
      if (e) cudaEventDestroy(e);
#endif
  }
  void mark_bucket(int k, lbc_stream_t s) {   // bucket k's gradients are all enqueued on s
#ifndef LBC_HOST_EMU
    if (grad_events && buckets[k].event) {
      join_side(s);   // (overlap mode) the bucket's weight gradients run on the side stream
      LBC_CUDA(cudaEventRecord((cudaEvent_t)buckets[k].event, s));
    }
#else
    (void)k;
    (void)s;
#endif
  }
  size_t workspace_bytes() const override { return total_bytes; }

  // ------------------------------------------------------------------ parameter table
  int64_t add_param(const std::string& name, std::vector<int> shape, bool on_path = true) {
    ParamInfo pi;
    pi.name = name;
    pi.ndim = (int)shape.size();
    pi.numel = 1;
    for (int i = 0; i < 4; ++i) pi.shape[i] = i < pi.ndim ? shape[i] : 1;
    for (int d : shape) pi.numel *= d;
    pi.offset = n_params;
    pi.on_path = on_path;
    n_params += pi.numel;
    params.push_back(pi);
    return pi.offset;
  }
  void add_bn(const std::string& prefix, int C, BNL& bn) {
    bn.C = C;
    bn.g_off = add_param(prefix + ".weight", {C});
    bn.b_off = add_param(prefix + ".bias", {C});
    for (int i = 0; i < 2; ++i) {
      BufferInfo bi;
      bi.name = prefix + (i == 0 ? ".running_mean" : ".running_var");
      bi.numel = C;
      bi.offset = n_buffers;
      n_buffers += C;
      buffers.push_back(bi);
      (i == 0 ? bn.rm_off : bn.rv_off) = bi.offset;
    }
    bn.mean = alloc<float>(C);
    bn.var = alloc<float>(C);
    bn.rstd = alloc<float>(C);
  }
  void add_conv(const std::string& name, int Ci, int Co, int K, int stride, int pad, int H, int W, ConvL& c) {
    c.Ci = Ci;
    c.Co = Co;
    c.K = K;
    c.stride = stride;
    c.pad = pad;
    c.H = H;
    c.W = W;
    c.OH = (H + 2 * pad - K) / stride + 1;
    c.OW = (W + 2 * pad - K) / stride + 1;
    c.w_off = add_param(name + ".weight", {Co, Ci, K, K});
    c.wp = alloc<T>((int64_t)Co * K * K * Ci);
    c.wpt = alloc<T>((int64_t)Co * K * K * Ci);
    if (tc) {   // [hi | lo] fp16 planes: 2 x 2 bytes per element
      c.wp16 = alloc<float>((int64_t)Co * K * K * Ci);
      c.wpt16 = alloc<float>((int64_t)Co * K * K * Ci);
    }
  }
  // nn.ConvTranspose2d(Cin, Cout, 3, 2, 1, 1): as the input-gradient of a 3x3/s2/p1 conv whose
  // conv-role Co = deconv Cin, Ci = deconv Cout; conv-role input is the (2h x 2w) deconv output.
  void add_deconv(const std::string& name, int Cin, int Cout, int h, int w, ConvL& c) {
    c.deconv = true;
    c.Ci = Cout;
    c.Co = Cin;
    c.K = 3;
    c.stride = 2;
    c.pad = 1;
    c.H = 2 * h;
    c.W = 2 * w;
    c.OH = h;
    c.OW = w;
    c.w_off = add_param(name + ".weight", {Cin, Cout, 3, 3});
    c.b_off = add_param(name + ".bias", {Cout});
    c.wp = alloc<T>((int64_t)Cin * 9 * Cout);
    c.wpt = alloc<T>((int64_t)Cin * 9 * Cout);
    if (tc) {
      c.wp16 = alloc<float>((int64_t)Cin * 9 * Cout);
      c.wpt16 = alloc<float>((int64_t)Cin * 9 * Cout);
    }
  }

  Net(NetKind k, Precision p, int maxB) {
    kind = k;
    prec = p;
    max_batch = maxB;
    tc = (p == PREC_F32TC);
    LBC_CHECK(!tc || (std::is_same<T, float>::value), "PREC_F32TC runs on fp32 storage");
    std::vector<int> layers;
    if (k == NET_IMAGE_RESNET34) {
      in_ch = 3;
      in_h = 160;
      in_w = 384;
      layers = {3, 4, 6, 3};
      normalize = true;
    } else {
      in_ch = 7;
      in_h = 192;
      in_w = 192;
      layers = {2, 2, 2, 2};
      normalize = false;
    }
    const int64_t B = maxB;
    // ---- stem (resnet.py:102-106)
    add_conv("conv.conv1", in_ch, 64, 7, 2, 3, in_h, in_w, stem);
    add_bn("conv.bn1", 64, stem_bn);
    stem_oh = stem.OH;
    stem_ow = stem.OW;
    pool_h = (stem_oh + 2 - 3) / 2 + 1;
    pool_w = (stem_ow + 2 - 3) / 2 + 1;
    x0 = alloc<T>(B * in_h * in_w * in_ch);
    r_stem = alloc<T>(B * stem_oh * stem_ow * 64);
    a_stem = alloc<T>(B * stem_oh * stem_ow * 64);
    pool = alloc<T>(B * pool_h * pool_w * 64);
    pool_idx = alloc<uint8_t>(B * pool_h * pool_w * 64);
    if (std::is_same<T, bf16>::value || tc) {
      int Kp = ((49 * in_ch + 63) / 64) * 64;
      stem_gemm.Ci = Kp;
      stem_gemm.Co = 64;
      stem_gemm.K = 1;
      stem_gemm.stride = 1;
      stem_gemm.pad = 0;
      stem_gemm.H = stem_gemm.OH = stem_oh;
      stem_gemm.W = stem_gemm.OW = stem_ow;
      stem_gemm.wp = alloc<T>(64 * Kp);
      stem_dw_col = alloc<float>(64 * Kp);
      if (tc) {
        stem_gemm.wp16 = alloc<float>(64 * Kp);
      } else if (fast::stem_ch(in_ch)) {   // zero-padded NHWC4 / NHWC8 image + overlapping-window TMA: no column tensor
        stem_layout = fast::stem_ch(in_ch, in_w, normalize);
        stem_x4 = alloc<T>(B * (in_h + 6) * (in_w + 8) * fast::stem_x_ch(stem_layout));
        stem_w224 = alloc<T>(fast::stem_w_elems(stem_layout));
      } else {
        stem_col = alloc<T>(B * stem_oh * stem_ow * Kp);
      }
    }
    // ---- BasicBlocks (resnet.py:25-54,132-146)
    int C = 64, H = pool_h, W = pool_w;
    const T* prev = pool;
    for (int li = 0; li < 4; ++li) {
      int planes = 64 << li;
      for (int bi = 0; bi < layers[li]; ++bi) {
        blocks.emplace_back();
        Block& b = blocks.back();
        b.name = "conv.layer" + std::to_string(li + 1) + "." + std::to_string(bi);
        int stride = (li > 0 && bi == 0) ? 2 : 1;
        b.Cin = C;
        b.Cout = planes;
        b.Hin = H;
        b.Win = W;
        add_conv(b.name + ".conv1", C, planes, 3, stride, 1, H, W, b.c1);
        add_bn(b.name + ".bn1", planes, b.b1);
        b.Hout = b.c1.OH;
        b.Wout = b.c1.OW;
        add_conv(b.name + ".conv2", planes, planes, 3, 1, 1, b.Hout, b.Wout, b.c2);
        add_bn(b.name + ".bn2", planes, b.b2);
        b.ds = (stride != 1 || C != planes);
        if (b.ds) {
          add_conv(b.name + ".downsample.0", C, planes, 1, stride, 0, H, W, b.cd);
          add_bn(b.name + ".downsample.1", planes, b.bd);
          if ((std::is_same<T, bf16>::value || tc) && stride == 2) {
            b.c1.wcomb = alloc<T>((int64_t)C * 2 * planes);
            if (tc) b.c1.wcomb16 = alloc<float>((int64_t)C * 2 * planes);
          }
        }
        int64_t ne = B * b.Hout * b.Wout * planes;
        b.r1 = alloc<T>(ne);
        b.a1 = alloc<T>(ne);
        b.r2 = alloc<T>(ne);
        b.out = alloc<T>(ne);
        if (std::is_same<T, bf16>::value) b.obits = alloc<uint8_t>(ne / 8);
        if (b.ds) {
          b.rd = alloc<T>(ne);
          b.idn = alloc<T>(ne);
        }
        b.xin = prev;
        prev = b.out;
        C = planes;
        H = b.Hout;
        W = b.Wout;
      }
    }
    trunk_h = H;
    trunk_w = W;
    // conv.fc exists in the state_dict but is never executed (resnet.py:112,148-159)
    add_param("conv.fc.weight", {1000, 512}, false);
    add_param("conv.fc.bias", {1000}, false);
    // ---- decoder (image.py:37-47 / birdview.py:34-44)
    int dc_in[3] = {640, 256, 128}, dc_out[3] = {256, 128, 64};
    int h = H, w = W;
    for (int i = 0; i < 3; ++i) {
      add_bn("deconv." + std::to_string(3 * i), dc_in[i], dbn[i]);
      add_deconv("deconv." + std::to_string(3 * i + 1), dc_in[i], dc_out[i], h, w, dcv[i]);
      dec_bn[i] = alloc<T>(B * h * w * dc_in[i]);
      dec_in[i] = i == 0 ? alloc<T>(B * h * w * dc_in[0]) : dec_out[i - 1];
      h *= 2;
      w *= 2;
      dec_out[i] = alloc<T>(B * h * w * dc_out[i]);
    }
    head_h = h;
    head_w = w;
    // ---- heads (image.py:54-60)
    for (int k2 = 0; k2 < 4; ++k2) {
      std::string p2 = "location_pred." + std::to_string(k2);
      add_bn(p2 + ".0", 64, hbn[k2]);
      hw_off[k2] = add_param(p2 + ".1.weight", {5, 64, 1, 1});
      hb_off[k2] = add_param(p2 + ".1.bias", {5});
    }
    int HW = head_h * head_w;
    logits = alloc<float>(B * 20 * HW);
    dlogits = alloc<float>(B * 20 * HW);
    rowmax = alloc<float>(B * 20);
    rowsum = alloc<float>(B * 20);
    preds = alloc<float>(B * 40);
    onehot_saved = alloc<float>(B * 4);
    speed_saved = alloc<float>(B);
    headS = alloc<double>(20 * 65);
    // ---- scratch
    int64_t gmax = B * stem_oh * stem_ow * 64;
    for (int i = 0; i < 4; ++i) g[i] = alloc<T>(gmax);
#ifndef LBC_HOST_EMU
    if (std::is_same<T, bf16>::value && !tc) {
      // ring buffers hold block-level gradients only (largest: layer 1 = the pooled stem output's shape)
      {
        const char* e = getenv("LBC_RING");
        const int r = e ? atoi(e) : 4;
        ring_n = r < 2 ? 2 : (r > kRing ? kRing : r);
      }
      for (int i = 0; i < ring_n; ++i) gring[i] = alloc<T>(B * pool_h * pool_w * 64);
      int lo = 0, hi = 0;
      LBC_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));   // lo = least priority (0), hi = greatest (negative)
      LBC_CUDA(cudaStreamCreateWithPriority(&side_stream, cudaStreamNonBlocking, lo));
      LBC_CUDA(cudaStreamCreateWithPriority(&chain_stream, cudaStreamNonBlocking, hi));
      for (cudaEvent_t* e : {&ev_ready, &ev_join, &ev_in, &ev_out}) LBC_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
      for (cudaEvent_t& e : gdone) LBC_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      ovl_capable = true;
    }
#endif
    ws_f_n = 4 << 20;
    ws_f = alloc<float>(ws_f_n);
    int64_t wd = (1 << 20);
    if (B * 20 * 65 + 4096 > wd) wd = B * 20 * 65 + 4096;
    ws_d = alloc<double>(wd);
    bn_sums = alloc<float>(2 * 1024);
    if (tc) {
      // operand-split scratch: a16 holds the largest conv operand (or the split stem column tensor), b16 the second
      // operand of a weight gradient / the downsample gradient of a fused block-entry data gradient
      tcw.b_bytes = gmax * 4;
      tcw.a_bytes = std::max<int64_t>(gmax * 4, B * stem_oh * stem_ow * (int64_t)stem_gemm.Ci * 2 * 2);
      tcw.a16 = alloc<uint8_t>(tcw.a_bytes);
      tcw.b16 = alloc<uint8_t>(tcw.b_bytes);
    }
    if (std::is_same<T, bf16>::value) {
      negshift_all = alloc<float>(n_buffers);
      dev_memset(negshift_all, 0, sizeof(float) * n_buffers, (lbc_stream_t)0);
      stem_bn.negshift = negshift_all + stem_bn.rm_off;
      for (Block& b : blocks) {
        b.b1.negshift = negshift_all + b.b1.rm_off;
        b.b2.negshift = negshift_all + b.b2.rm_off;
        if (b.ds) b.bd.negshift = negshift_all + b.bd.rm_off;
      }
    }
    // weight-pack table (one launch per forward)
    auto add_pack = [&](const ConvL& c, bool with_t) {
      ref::PackEntry e;
      e.src_off = c.w_off;
      e.src2_off = 0;
      e.dst = c.wp;
      e.type = 0;
      e.Co = c.Co;
      e.Ci = c.Ci;
      e.K = c.K;
      e.aux = 0;
      e.n = (int64_t)c.Co * c.K * c.K * c.Ci;
      pack_host.push_back(e);
      if (with_t) {
        e.dst = c.wpt;
        e.type = 1;
        pack_host.push_back(e);
      }
    };
    const bool is_bf16 = std::is_same<T, bf16>::value || tc;   // (tc: the transposed / combined packs are needed too)
    add_pack(stem, false);
    for (Block& b : blocks) {
      add_pack(b.c1, is_bf16);
      add_pack(b.c2, is_bf16);
      if (b.ds) add_pack(b.cd, is_bf16);
      if (b.c1.wcomb) {
        ref::PackEntry e;
        e.src_off = b.c1.w_off;
        e.src2_off = b.cd.w_off;
        e.dst = b.c1.wcomb;
        e.type = 2;
        e.Co = b.c1.Co;
        e.Ci = b.c1.Ci;
        e.K = 3;
        e.aux = 0;
        e.n = (int64_t)b.c1.Ci * 2 * b.c1.Co;
        pack_host.push_back(e);
      }
    }
    for (int i = 0; i < 3; ++i) add_pack(dcv[i], is_bf16);
    if (is_bf16) {
      ref::PackEntry e;
      e.src_off = stem.w_off;
      e.src2_off = 0;
      e.dst = stem_gemm.wp;
      e.type = 3;
      e.Co = 64;
      e.Ci = in_ch;
      e.K = 7;
      e.aux = stem_gemm.Ci;
      e.n = (int64_t)64 * stem_gemm.Ci;
      pack_host.push_back(e);
    }
    pack_dev = alloc<ref::PackEntry>((int64_t)pack_host.size());
#ifdef LBC_HOST_EMU
    memcpy(pack_dev, pack_host.data(), sizeof(ref::PackEntry) * pack_host.size());
#else
    LBC_CUDA(cudaMemcpy(pack_dev, pack_host.data(), sizeof(ref::PackEntry) * pack_host.size(), cudaMemcpyHostToDevice));
#endif
    head_fold = alloc<float>(1300 + 128 + 28);
    // gradient buckets (ranges of the flat array in state_dict order: stem, layer1..4, [conv.fc: never trained], decoder, heads)
    {
      auto off_of = [&](const std::string& prefix) {
        for (const ParamInfo& pi : params)
          if (pi.name.compare(0, prefix.size(), prefix) == 0) return pi.offset;
        return n_params;
      };
      const int64_t o_l2 = off_of("conv.layer2."), o_l3 = off_of("conv.layer3."), o_l4 = off_of("conv.layer4."),
                    o_fc = off_of("conv.fc."), o_dec = off_of("deconv.");
      buckets.resize(5);
      buckets[0].offset = o_dec;
      buckets[0].numel = n_params - o_dec;
      buckets[1].offset = o_l4;
      buckets[1].numel = o_fc - o_l4;
      buckets[2].offset = o_l3;
      buckets[2].numel = o_l4 - o_l3;
      buckets[3].offset = o_l2;
      buckets[3].numel = o_l3 - o_l2;
      buckets[4].offset = 0;
      buckets[4].numel = o_l2;
    }
  }

  // ------------------------------------------------------------------ op wrappers (fast-path hooks)
  void repack(lbc_stream_t s) override { pack_weights(s); }
  void pack_weights(lbc_stream_t s) {
    ProfScope ps("pack", s, 0, 0);
    if (fast::enabled())   // pair walk: coalesced stores, no div/mod per element (271 -> ~170 us per forward at measured B = 256)
      ref::pack_all_pairs<T>(s, P, pack_dev, (int)pack_host.size());
    else
      ref::pack_all<T>(s, P, pack_dev, (int)pack_host.size());
    if (tc) {
      bool ok = true;
      auto split = [&](const void* src, void* dst, int64_t rows, int C, int fmt) {
        if (src && dst) ok = ok && fast::tc_split((const float*)src, dst, rows, C, fmt, fast::kTcWeightScale, s);
      };
      // the pack a layer's FORWARD uses is split into fp16 planes, the packs of its backward GEMMs into bf16 planes
      // (trunk conv: forward = wp, data gradient = wpt / wcomb; ConvTranspose2d: forward = wpt, backward-data = wp)
      auto split_conv = [&](const ConvL& c) {
        split(c.wp, c.wp16, (int64_t)c.Co * c.K * c.K, c.Ci, c.deconv ? fast::TC_BF16 : fast::TC_F16);
        split(c.wpt, c.wpt16, (int64_t)c.Ci * c.K * c.K, c.Co, c.deconv ? fast::TC_F16 : fast::TC_BF16);
        split(c.wcomb, c.wcomb16, (int64_t)c.Ci * 2, c.Co, fast::TC_BF16);
      };
      for (Block& b : blocks) {
        split_conv(b.c1);
        split_conv(b.c2);
        if (b.ds) split_conv(b.cd);
      }
      for (int i = 0; i < 3; ++i) split_conv(dcv[i]);
      split(stem_gemm.wp, stem_gemm.wp16, 64, stem_gemm.Ci, fast::TC_F16);
      LBC_CHECK(ok, "PREC_F32TC: weight split failed (fast kernels disabled or host-emulation build)");
    }
  }
  static double conv_flops(const ConvL& c, int B) {
    return 2.0 * B * c.OH * c.OW * (double)c.Co * c.K * c.K * c.Ci;
  }
  // returns true when the per-channel centring shift `negshift` was added to the stored output (fast path only)
  // stat_rows != null: ask the fast kernel to also emit the BatchNorm statistics partials of its output
  // (*stat_rows = number of partial rows, 0 when not emitted)
  bool conv_forward(const ConvL& c, const T* x, T* y, int B, lbc_stream_t s, const float* negshift = nullptr,
                    int* stat_rows = nullptr, bool x_is_grad = false) {
    ProfScope ps("conv_fwd", s, conv_flops(c, B), 0);
    if (stat_rows) *stat_rows = 0;
    float* part = (stat_rows && cur_train && (int64_t)c.Co * 2 * ((int64_t)B * c.OH * c.OW / 128 + 64) <= fast::stat_partial_capacity())
                      ? fast::stat_partial_buffer()
                      : nullptr;
    int rows = 0;
    if (tc) {
      LBC_CHECK(fast::conv_fwd_tc(c, (const float*)x, nullptr, (float*)y, B, nullptr, false, x_is_grad ? fast::TC_BF16 : fast::TC_F16,
                                  tcw, s),
                "PREC_F32TC: tensor-core convolution unavailable for this layer");
      return false;
    }
    if (fast::conv_fwd<T>(c, x, y, B, s, negshift, part, &rows)) {
      if (stat_rows && part) *stat_rows = rows;
      return negshift != nullptr;
    }
    ref::conv_fwd<T>(s, x, (const T*)c.wp, nullptr, false, y, B, c.H, c.W, c.Ci, c.Co, c.K, c.stride, c.pad, c.OH,
                     c.OW);
    return false;
  }
  void conv_backward_data(const ConvL& c, const T* dy, T* dx, int B, bool accumulate, lbc_stream_t s) {
    ProfScope ps("conv_dgrad", s, conv_flops(c, B), 0);
    if (tc && !accumulate && c.K != 1) {
      LBC_CHECK(fast::conv_dgrad_tc(c, (const float*)dy, nullptr, (float*)dx, B, nullptr, false, fast::TC_BF16, tcw, s),
                "PREC_F32TC: tensor-core data gradient unavailable for this layer");
      return;
    }
    if (!accumulate && fast::conv_dgrad<T>(c, dy, dx, B, nullptr, false, s)) return;
    ref::conv_dgrad<T>(s, dy, (const T*)c.wp, dx, B, c.H, c.W, c.Ci, c.Co, c.K, c.stride, c.pad, c.OH, c.OW, nullptr,
                       false, accumulate);
  }
  // x_is_grad: the conv-role x is a gradient and dy an activation (weight gradient of a ConvTranspose2d)
  void conv_backward_weight(const ConvL& c, const T* x, const T* dy, int B, lbc_stream_t s, bool x_is_grad = false) {
    ProfScope ps("conv_wgrad", s, conv_flops(c, B), 0);
    if (tc) {
      (void)x_is_grad;   // either way one operand is a gradient: bf16 planes for both
      LBC_CHECK(fast::conv_wgrad_tc(c, (const float*)x, nullptr, (const float*)dy, G + c.w_off, B, fast::TC_BF16, fast::TC_BF16, tcw,
                                    s),
                "PREC_F32TC: tensor-core weight gradient unavailable for this layer");
      return;
    }
    if (fast::conv_wgrad<T>(c, x, dy, G + c.w_off, B, s)) return;
    ref::conv_wgrad<T>(s, x, dy, G + c.w_off, B, c.H, c.W, c.Ci, c.Co, c.K, c.stride, c.pad, c.OH, c.OW, ws_f, ws_f_n);
  }
  void bn_forward(BNL& bn, const T* x, int64_t M, const T* residual, bool relu, T* y, bool train, lbc_stream_t s,
                  bool shifted = false, int conv_stat_rows = 0, uint8_t* maskbits = nullptr) {
    // algorithmic bytes: stats read (train) + apply read (+residual) + write
    ProfScope ps("bn_fwd", s, 0, (double)M * bn.C * sizeof(T) * ((train && conv_stat_rows == 0 ? 1 : 0) + 2 + (residual ? 1 : 0)));
    if (fast::Fast<T>::bn_fwd(x, M, bn.C, P + bn.g_off, P + bn.b_off, kBnEps, kBnMomentum, BUF + bn.rm_off, BUF + bn.rv_off,
                              bn.mean, bn.rstd, residual, relu, train, y, bn_sums, shifted ? bn.negshift : nullptr, s,
                              conv_stat_rows, maskbits)) {
      mask_bits_valid = maskbits != nullptr;
      return;
    }
    mask_bits_valid = false;
    LBC_CHECK(conv_stat_rows == 0, "BatchNorm fast path unavailable after a statistics-emitting convolution");
    LBC_CHECK(!shifted, "BatchNorm fast path unavailable after a shifted convolution");
    if (train) {
      ref::bn_stats<T>(s, x, M, bn.C, bn.mean, bn.var, ws_d);
      ref::bn_finalize(s, bn.mean, bn.var, bn.C, M, kBnEps, kBnMomentum, bn.rstd, BUF + bn.rm_off, BUF + bn.rv_off);
    } else {
      ref::bn_eval_stats(s, BUF + bn.rm_off, BUF + bn.rv_off, bn.C, kBnEps, bn.mean, bn.rstd);
    }
    ref::bn_apply<T>(s, x, bn.mean, bn.rstd, P + bn.g_off, P + bn.b_off, residual, relu, y, M, bn.C);
  }
  // dy_m = dy * (mask_act > 0) when mask_act != null (the ReLU that follows the BN, nn.ReLU(True) backward).
  // Correctness-first path: masks dy in place first; fast path: the mask is fused into both passes, dy untouched.
  // own_relu: mask_act is relu(bn(x)) of this very BatchNorm (no residual): the fast kernels then recompute the mask
  // from x instead of reading the activation (2 of the 7 tensor passes disappear).
  // pre_rows > 0: the reduce pass already ran inside add_masked_reduce (its partial rows are in the shared scratch)
  void bn_backward(BNL& bn, T* dy, const T* mask_act, const T* x, T* dx, int64_t M, lbc_stream_t s, bool own_relu = false,
                   const uint8_t* mask_bits = nullptr, int pre_rows = 0) {
    // algorithmic bytes: reduce pass reads dy,(mask),x ; apply pass reads dy,(mask),x writes dx (mask as bits: 1/16 pass each)
    const double passes = pre_rows > 0 ? 3 + 0.0625 : 5 + (mask_act && !own_relu ? (mask_bits ? 0.125 : 2) : 0);
    ProfScope ps("bn_bwd", s, 0, (double)M * bn.C * sizeof(T) * passes);
    if (fast::Fast<T>::bn_bwd(dy, mask_act, x, bn.mean, bn.rstd, P + bn.g_off, G + bn.g_off, G + bn.b_off, dx, M, bn.C,
                              bn_sums, s, own_relu ? P + bn.b_off : nullptr, mask_bits, pre_rows))
      return;
    LBC_CHECK(pre_rows == 0, "BatchNorm backward fast path unavailable after a fused residual-add + reduce");
    if (mask_act) ref::relu_mask_inplace<T>(s, dy, mask_act, M * bn.C);
    ref::bn_bwd<T>(s, dy, x, bn.mean, bn.rstd, P + bn.g_off, G + bn.g_off, G + bn.b_off, dx, M, bn.C, ws_d);
  }
  void relu_mask(T* g, const T* act, int64_t n, lbc_stream_t s) {
    ProfScope ps("elementwise", s, 0, (double)n * sizeof(T) * 3);
    if (fast::Fast<T>::ew(g, nullptr, act, n, 2, s)) return;
    ref::relu_mask_inplace<T>(s, g, act, n);
  }
  void add_masked(T* dst, const T* g, const T* act, int64_t n, lbc_stream_t s, const uint8_t* mask_bits = nullptr) {
    ProfScope ps("elementwise", s, 0, (double)n * sizeof(T) * (mask_bits ? 3.0625 : 4));
    if (fast::Fast<T>::ew(dst, g, act, n, 1, s, mask_bits)) return;
    ref::add_masked_inplace<T>(s, dst, g, act, n);
  }
  // dst += g * mask (the residual branch of the block just differentiated) fused with the reduce pass of the BatchNorm
  // that consumes dst next (the previous block's bn2, mask = that block's output bits); returns its partial rows or 0
  int add_masked_reduce(T* dst, const T* g, const uint8_t* g_bits, BNL& next_bn, const T* next_x, const uint8_t* next_bits,
                        int64_t M, lbc_stream_t s) {
    if (!g_bits || !next_bits) return 0;
    static const bool on = [] {
      const char* e = getenv("LBC_RESID_FUSE");   // 0: separate ew_kernel + reduce launches (A/B)
      return e ? atoi(e) != 0 : true;
    }();
    if (!on) return 0;
    int rows = 0;
    // algorithmic bytes: dst read + written, g read, x read, two bit masks
    ProfScope ps("elementwise", s, 0, (double)M * next_bn.C * sizeof(T) * 4.125);
    if (!fast::Fast<T>::resid_bn_reduce(dst, g, g_bits, next_x, next_bn.mean, next_bn.rstd, next_bits, M, next_bn.C, &rows, s))
      return 0;
    return rows;
  }
  HeadCtx hc;
  HeadCtx& head_ctx() {   // (parameter / buffer pointers follow the currently bound flat arrays)
    hc.H = head_h;
    hc.W = head_w;
    hc.logits = logits;
    hc.dlogits = dlogits;
    hc.rowmax = rowmax;
    hc.rowsum = rowsum;
    hc.preds = preds;
    hc.S = headS;
    hc.fold = head_fold;
    hc.bn_sums = bn_sums;
    hc.ws_d = ws_d;
    hc.var0 = hbn[0].var;
    for (int k = 0; k < 4; ++k) {
      hc.gamma[k] = P + hbn[k].g_off;
      hc.beta[k] = P + hbn[k].b_off;
      hc.w[k] = P + hw_off[k];
      hc.bias[k] = P + hb_off[k];
      hc.mean[k] = hbn[k].mean;
      hc.rstd[k] = hbn[k].rstd;
      hc.rm[k] = BUF + hbn[k].rm_off;
      hc.rv[k] = BUF + hbn[k].rv_off;
    }
    return hc;
  }

  // ------------------------------------------------------------------ forward
  void forward(const float* image, const float* speed, const float* onehot, int B, bool train, float* out_pred,
               float* out_preds, lbc_stream_t s) override {
    LBC_CHECK(P && BUF, "lbc_net_forward: parameters not bound");
    LBC_CHECK(B >= 1 && B <= max_batch, "lbc_net_forward: batch " + std::to_string(B) + " outside [1, max_batch]");
    LBC_CHECK(!train || B * head_h * head_w > 1, "train-mode BatchNorm needs more than one value per channel");
    cur_B = B;
    cur_train = train;
    // the weight operands of the residual blocks / decoder are packed on the side stream while the stem runs (the stem has its
    // own small pack): 0.15 ms of gather traffic next to 0.65 ms of TMA- and HBM-bound stem kernels
    bool pack_on_side = false;
    if (!skip_pack) {
#ifndef LBC_HOST_EMU
      static const bool side_ok = [] {
        const char* e = getenv("LBC_PACK_SIDE");   // 0: pack on the caller's stream (A/B)
        return e ? atoi(e) != 0 : true;
      }();
      pack_on_side = side_ok && ovl_capable && g_wgrad_overlap > 0 && !g_prof_on && std::is_same<T, bf16>::value && stem_x4 &&
                     fast::enabled();
      if (pack_on_side) {
        LBC_CUDA(cudaEventRecord(ev_ready, s));                  // after the optimizer step that wrote the parameters
        LBC_CUDA(cudaStreamWaitEvent(side_stream, ev_ready, 0));
        pack_weights(side_stream);
        LBC_CUDA(cudaEventRecord(ev_join, side_stream));
      } else
#endif
        pack_weights(s);
      packs_current = false;   // (whoever updates the parameters next does not tell the engine)
    }
    dev_copy(onehot_saved, onehot, sizeof(float) * B * 4, s);
    dev_copy(speed_saved, speed, sizeof(float) * B, s);
    if (!train && negshift_all && fast::enabled()) ref::negate_into(s, BUF, negshift_all, n_buffers);  // centre on running_mean
    // stem
    stem_fast_used = false;
    stem_direct_used = false;
    int stem_stat_rows = 0;
    if (std::is_same<T, bf16>::value && stem_x4 && fast::enabled()) {
      ProfScope ps("conv_fwd", s, conv_flops(stem, B), 0);
      // statistics partials from the epilogue only while they fit the shared scratch (one 128-float row per 128-pixel
      // tile); larger batches fall back to the separate statistics pass (bn_stats_bf16 below)
      const bool part_fits = ((int64_t)B * stem_oh * stem_ow / 128 + 64) * 128 <= fast::stat_partial_capacity();
      float* part = (train && part_fits) ? fast::stat_partial_buffer() : nullptr;
      bool ok = (u8_image ? fast::stem_pad4_u8_bf16(u8_image, u8_layout, (bf16*)stem_x4, B, in_ch, in_h, in_w, normalize, s)
                          : fast::stem_pad4_bf16(image, (bf16*)stem_x4, B, in_ch, in_h, in_w, normalize, s)) &&
                fast::stem_pack_w224_bf16(P + stem.w_off, (bf16*)stem_w224, in_ch, s, stem_layout) &&
                fast::stem_conv_bf16((const bf16*)stem_x4, (const bf16*)stem_w224, (bf16*)r_stem, B, in_h, in_w, stem_oh,
                                     stem_ow, stem_bn.negshift, part, &stem_stat_rows, s, stem_layout);
      LBC_CHECK(ok, "stem direct (overlapping-window TMA) path failed");
      stem_fast_used = stem_direct_used = true;
      if (!part) stem_stat_rows = 0;
    } else if (std::is_same<T, bf16>::value && stem_col) {
      ProfScope ps("conv_fwd", s, conv_flops(stem, B), 0);
      if (fast::stem_im2col_bf16(image, (bf16*)stem_col, B, in_ch, in_h, in_w, stem_oh, stem_ow, stem_gemm.Ci, normalize, s))
        stem_fast_used = fast::conv_fwd<T>(stem_gemm, stem_col, r_stem, B, s, stem_bn.negshift);
    }
    stem_tc_used = false;
    if (!stem_fast_used) {
      ref::input_to_nhwc<T>(s, image, x0, B, in_ch, in_h, in_w, in_ch, normalize, 0.485f, 0.456f, 0.406f, 0.229f,
                            0.224f, 0.225f);
      if (tc) {   // split fp16 column tensor -> the generic tensor-core GEMM as a 1x1 convolution over [B,OH,OW,2*Kp]
        ProfScope ps("conv_fwd", s, conv_flops(stem, B), 0);
        bool ok = fast::tc_stem_im2col((const float*)x0, tcw.a16, B, in_ch, in_h, in_w, stem_oh, stem_ow, stem_gemm.Ci, fast::TC_F16, s) &&
                  fast::conv_fwd_tc(stem_gemm, nullptr, tcw.a16, (float*)r_stem, B, nullptr, false, fast::TC_F16, tcw, s);
        LBC_CHECK(ok, "PREC_F32TC: tensor-core stem unavailable");
        stem_tc_used = true;
      } else {
        conv_forward(stem, x0, r_stem, B, s);
      }
    }
    stem_pool_fused = false;
    {
      const int64_t Ms = (int64_t)B * stem_oh * stem_ow;
      if (std::is_same<T, bf16>::value && fast::enabled()) {
        // statistics -> (mean, rstd, running buffers) -> fused BN+ReLU+MaxPool; the activation is never written
        ProfScope ps("bn_fwd", s, 0, (double)Ms * 64 * sizeof(T) * 2.25);
        bool ok = true;
        if (train) {
          ok = stem_stat_rows > 0 ? fast::col_finalize_bf16(fast::stat_partial_buffer(), stem_stat_rows, 128, bn_sums, s)
                                  : fast::bn_stats_bf16((const bf16*)r_stem, Ms, 64, bn_sums, s);
          if (ok) {
            ref::bn_finalize_sums(s, bn_sums, 64, Ms, kBnEps, kBnMomentum, stem_bn.mean, stem_bn.rstd, BUF + stem_bn.rm_off,
                                  BUF + stem_bn.rv_off, stem_fast_used ? stem_bn.negshift : nullptr);
          }
        } else {
          ref::bn_eval_stats(s, BUF + stem_bn.rm_off, BUF + stem_bn.rv_off, 64, kBnEps, stem_bn.mean, stem_bn.rstd,
                             stem_fast_used ? stem_bn.negshift : nullptr);
        }
        if (ok)
          stem_pool_fused = fast::Fast<T>::pool_fwd(r_stem, stem_bn.mean, stem_bn.rstd, P + stem_bn.g_off, P + stem_bn.b_off,
                                                    pool, pool_idx, B, stem_oh, stem_ow, 64, pool_h, pool_w, s);
        LBC_CHECK(ok && stem_pool_fused, "stem BN+ReLU+MaxPool fast path failed");
      }
      if (!stem_pool_fused) {
        bn_forward(stem_bn, r_stem, Ms, nullptr, true, a_stem, train, s);
        ProfScope ps("pool", s, 0, (double)Ms * 64 * sizeof(T) * 1.25);
        ref::maxpool_fwd<T>(s, a_stem, pool, pool_idx, B, stem_oh, stem_ow, 64, pool_h, pool_w);
      }
    }
#ifndef LBC_HOST_EMU
    if (pack_on_side) LBC_CUDA(cudaStreamWaitEvent(s, ev_join, 0));
#else
    (void)pack_on_side;
#endif
    // residual blocks
    for (Block& b : blocks) {
      int64_t M = (int64_t)B * b.Hout * b.Wout;
      // each conv's statistics partials live in ONE shared scratch: finalise (inside bn_forward) before the next conv
      int sr = 0;
      bool sh1 = conv_forward(b.c1, b.xin, b.r1, B, s, b.b1.negshift, &sr);
      bn_forward(b.b1, b.r1, M, nullptr, true, b.a1, train, s, sh1, sr);
      const T* identity = b.xin;
      if (b.ds) {
        bool shd = conv_forward(b.cd, b.xin, b.rd, B, s, b.bd.negshift, &sr);
        bn_forward(b.bd, b.rd, M, nullptr, false, b.idn, train, s, shd, sr);
        identity = b.idn;
      }
      bool sh2 = conv_forward(b.c2, b.a1, b.r2, B, s, b.b2.negshift, &sr);
      bn_forward(b.b2, b.r2, M, identity, true, b.out, train, s, sh2, sr, train ? b.obits : nullptr);
      b.obits_ok = mask_bits_valid;
    }
    // late fusion of speed (image.py:77-79)
    const T* trunk = blocks.back().out;
    int hw = trunk_h * trunk_w;
    if (!fast::copy_channels<T>(dec_in[0], trunk, (int64_t)B * hw, 640, 512, speed, hw, s))
      ref::concat_speed<T>(s, trunk, speed, dec_in[0], B, hw, 512, 128);
    // decoder: BN -> deconv(+bias) -> ReLU
    int h = trunk_h, w = trunk_w;
    for (int i = 0; i < 3; ++i) {
      bn_forward(dbn[i], dec_in[i], (int64_t)B * h * w, nullptr, false, dec_bn[i], train, s);
      const ConvL& c = dcv[i];
      ProfScope ps("conv_dgrad", s, conv_flops(c, B), 0);
      if (tc)
        LBC_CHECK(fast::conv_dgrad_tc(c, (const float*)dec_bn[i], nullptr, (float*)dec_out[i], B, P + c.b_off, true, fast::TC_F16,
                                      tcw, s),
                  "PREC_F32TC: tensor-core ConvTranspose2d unavailable");
      else if (!fast::conv_dgrad<T>(c, dec_bn[i], dec_out[i], B, P + c.b_off, true, s))
        ref::conv_dgrad<T>(s, dec_bn[i], (const T*)c.wp, dec_out[i], B, c.H, c.W, c.Ci, c.Co, c.K, c.stride, c.pad, c.OH,
                           c.OW, P + c.b_off, true, false);
      h *= 2;
      w *= 2;
    }
    // heads
    const T* hfeat = dec_out[2];
    {
      const int64_t M = (int64_t)B * head_h * head_w;
      ProfScope ps_head("head", s, 0, (double)M * 64 * sizeof(T) * 2 + (double)M * 20 * 4 * 2);
      head_forward<T>(head_ctx(), hfeat, B, train, kBnEps, kBnMomentum, s);
    }
    if (out_preds) dev_copy(out_preds, preds, sizeof(float) * B * 40, s);
    if (out_pred) ref::head_select(s, preds, onehot_saved, out_pred, B);
  }

  float* img_f32 = nullptr;
  int64_t img_f32_n = 0;
  const uint8_t* u8_image = nullptr;   // set only while forward_u8 drives forward() through the direct stem
  int u8_layout = 0;
  void forward_u8(const uint8_t* image, int layout, const float* speed, const float* onehot, int B, bool train,
                  float* out_pred, float* out_preds, lbc_stream_t s) override {
    LBC_CHECK(layout == 0 || layout == 1, "lbc_net_forward_u8: layout must be 0 (NCHW) or 1 (NHWC)");
    LBC_CHECK(B >= 1 && B <= max_batch, "lbc_net_forward_u8: batch outside [1, max_batch]");
    if (std::is_same<T, bf16>::value && stem_x4 && fast::enabled()) {
      // direct stem: the padded NHWC4 bf16 operand is written straight from the uint8 frames (no fp32 image)
      u8_image = image;
      u8_layout = layout;
      try {
        forward(nullptr, speed, onehot, B, train, out_pred, out_preds, s);
      } catch (...) {
        u8_image = nullptr;
        throw;
      }
      u8_image = nullptr;
      return;
    }
    const int64_t need = (int64_t)max_batch * in_ch * in_h * in_w;
    if (!img_f32) {
      img_f32 = alloc<float>(need);
      img_f32_n = need;
    }
    ref::u8_to_f32_nchw(s, image, img_f32, B, in_ch, in_h, in_w, layout);
    forward(img_f32, speed, onehot, B, train, out_pred, out_preds, s);
  }

  // ------------------------------------------------------------------ backward
  void backward(const float* d_pred, const float* d_preds, lbc_stream_t s_in) override {
    LBC_CHECK(G, "lbc_net_backward: gradient buffer not bound");
    LBC_CHECK(cur_B > 0 && cur_train, "lbc_net_backward: no train-mode forward to differentiate");
    LBC_CHECK(d_pred || d_preds, "lbc_net_backward: no upstream gradient");
    packs_current = false;
    const int B = cur_B;
    const int HW = head_h * head_w;
    lbc_stream_t s = s_in;
    // overlap mode (see the members above): LBC_WGRAD_OVERLAP=0 keeps every kernel on the caller's stream; the per-category
    // profiler brackets launches of ONE stream with events, so it also runs the serial schedule
    const int ovl_mode = g_wgrad_overlap;   // 0: serial, 1: side stream, 2: + high-priority chain (lbc_set_schedule / LBC_WGRAD_OVERLAP)
    ovl = ovl_capable && ovl_mode > 0 && !g_prof_on;
    ring_next = 0;
#ifndef LBC_HOST_EMU
    if (ovl) {
      for (bool& b : gpending) b = false;
      if (ovl_mode >= 2) {
        LBC_CUDA(cudaEventRecord(ev_in, s_in));
        LBC_CUDA(cudaStreamWaitEvent(chain_stream, ev_in, 0));
        s = chain_stream;
      }
    }
#endif
    T* gcur = g[0];
    T* tA = g[1];
    T* tB = g[2];
    T* gnext = g[3];
    // heads
    const T* hfeat = dec_out[2];
    ref::HeadGrads hg;
    for (int k = 0; k < 4; ++k) {
      hg.dgamma[k] = G + hbn[k].g_off;
      hg.dbeta[k] = G + hbn[k].b_off;
      hg.dw[k] = G + hw_off[k];
      hg.dbias[k] = G + hb_off[k];
    }
    {
      ProfScope ps_head("head", s, 0, (double)B * HW * 64 * sizeof(T) * 3 + (double)B * HW * 20 * 4 * 3);
      head_backward<T>(head_ctx(), hfeat, onehot_saved, d_pred, d_preds, hg, gcur, B, s);
    }
    const bool head_mask_fused = hc.mask_fused;
    // decoder, last stage first
    for (int i = 2; i >= 0; --i) {
      const ConvL& c = dcv[i];
      int64_t Mout = (int64_t)B * c.H * c.W;   // deconv output pixels
      int64_t Min = (int64_t)B * c.OH * c.OW;  // deconv input pixels
      if (!(i == 2 && head_mask_fused)) relu_mask(gcur, dec_out[i], Mout * c.Ci, s);
      if (!fast::Fast<T>::colsum(gcur, Mout, c.Ci, G + c.b_off, bn_sums, s))
        ref::colsum<T>(s, gcur, Mout, c.Ci, G + c.b_off, ws_d);
      mark_ready(s);
      conv_forward(c, gcur, wr(tA, s), B, s, nullptr, nullptr, true);
      wgrad_side(c, gcur, dec_bn[i], B, s, true, gcur);  // conv-role x = d(out), dy = deconv input
      bn_backward(dbn[i], tA, nullptr, dec_in[i], wr(gnext, s), Min, s);
      std::swap(gcur, gnext);
    }
    mark_bucket(0, s);
    // drop the 128 speed channels (no gradient path to a parameter through them)
    if (!fast::copy_channels<T>(wr(gnext, s), gcur, (int64_t)B * trunk_h * trunk_w, 512, 640, nullptr, 1, s))
      ref::slice_channels<T>(s, gcur, gnext, (int64_t)B * trunk_h * trunk_w, 640, 512);
    std::swap(gcur, gnext);
    // residual blocks in reverse
    int pending_rows = 0;   // partial rows of the NEXT bn2 backward, when its reduce pass was fused into the residual add
    for (int bi = (int)blocks.size() - 1; bi >= 0; --bi) {
      Block& b = blocks[bi];
      int64_t M = (int64_t)B * b.Hout * b.Wout;
      int64_t ne = M * b.Cout;
      // gcur = d(out); the block-final ReLU mask (out > 0) is applied inside every consumer of gcur
      const uint8_t* ob = b.obits_ok ? b.obits : nullptr;
      T* d_r2 = ring(tA, s);
      bn_backward(b.b2, gcur, b.out, b.r2, d_r2, M, s, false, ob, pending_rows);
      pending_rows = 0;
      mark_ready(s);
      conv_backward_data(b.c2, d_r2, wr(tB, s), B, false, s);   // tB = d a1 (before the ReLU mask a1 > 0)
      wgrad_side(b.c2, b.a1, d_r2, B, s, false, d_r2);
      T* d_r1 = ring(tA, s);
      bn_backward(b.b1, tB, b.a1, b.r1, d_r1, M, s, true);   // mask a1 > 0 recomputed from r1
      mark_ready(s);
      if (b.ds) {
        T* d_rd = ring(tB, s);   // (serial mode: d a1 is dead by now)
        bn_backward(b.bd, gcur, b.out, b.rd, d_rd, M, s, false, ob);
        wgrad_side(b.c1, b.xin, d_r1, B, s, false, d_r1);
        mark_ready(s);
        bool fused = false;
        {
          ProfScope ps("conv_dgrad", s, conv_flops(b.c1, B) + conv_flops(b.cd, B), 0);
          if (tc)
            fused = fast::conv_dgrad_tc(b.c1, (const float*)d_r1, (const float*)d_rd, (float*)gnext, B, nullptr, false, fast::TC_BF16,
                                        tcw, s);
          else
            fused = fast::conv_dgrad_ds<T>(b.c1, d_r1, d_rd, wr(gnext, s), B, s);   // gnext = dgrad(conv1) + dgrad(downsample)
        }
        if (!fused) {
          conv_backward_data(b.c1, d_r1, wr(gnext, s), B, false, s);
          conv_backward_data(b.cd, d_rd, gnext, B, true, s);
        }
        wgrad_side(b.cd, b.xin, d_rd, B, s, false, d_rd);
      } else {
        conv_backward_data(b.c1, d_r1, wr(gnext, s), B, false, s);  // gnext = d xin (main path)
        wgrad_side(b.c1, b.xin, d_r1, B, s, false, d_r1);
        // + the residual branch; when the block before this one has the same shape, its bn2 reduce pass rides along
        if (bi > 0 && blocks[bi - 1].obits_ok && blocks[bi - 1].Cout == b.Cout && blocks[bi - 1].Hout == b.Hout &&
            blocks[bi - 1].Wout == b.Wout)
          pending_rows = add_masked_reduce(gnext, gcur, ob, blocks[bi - 1].b2, blocks[bi - 1].r2, blocks[bi - 1].obits, M, s);
        if (pending_rows == 0) add_masked(gnext, gcur, b.out, ne, s, ob);
      }
      std::swap(gcur, gnext);
      // a stage is complete when its entry block (the one with the downsample branch) has been differentiated
      if (b.ds && b.Cout == 512) mark_bucket(1, s);
      if (b.ds && b.Cout == 256) mark_bucket(2, s);
      if (b.ds && b.Cout == 128) mark_bucket(3, s);
    }
    // stem: maxpool -> relu -> bn -> conv1 weight gradient (no input gradient)
    int64_t Ms = (int64_t)B * stem_oh * stem_ow;
    if (stem_pool_fused) {
      ProfScope ps("pool", s, 0, (double)Ms * 64 * sizeof(T) * 2.5);
      bool ok = fast::Fast<T>::pool_bwd(gcur, pool_idx, r_stem, stem_bn.mean, stem_bn.rstd, P + stem_bn.g_off,
                                        P + stem_bn.b_off, wr(tA, s), B, stem_oh, stem_ow, 64, pool_h, pool_w, s);
      LBC_CHECK(ok, "stem MaxPool/ReLU backward fast path failed");
      bn_backward(stem_bn, tA, nullptr, r_stem, wr(tB, s), Ms, s);
    } else {
      {
        ProfScope ps("pool", s, 0, (double)Ms * 64 * sizeof(T) * 1.25);
        ref::maxpool_bwd<T>(s, gcur, pool_idx, wr(tA, s), B, stem_oh, stem_ow, 64, pool_h, pool_w);
      }
      bn_backward(stem_bn, tA, a_stem, r_stem, wr(tB, s), Ms, s);
    }
    bool stem_wgrad_done = false;
    if (stem_direct_used) {
      ProfScope ps("conv_wgrad", s, conv_flops(stem, B), 0);
      stem_wgrad_done = fast::stem_wgrad_bf16((const bf16*)stem_x4, (const bf16*)tB, G + stem.w_off, B, in_ch, in_h, in_w,
                                              stem_oh, stem_ow, s, stem_layout);
      LBC_CHECK(stem_wgrad_done, "stem direct weight gradient failed");
    } else if (stem_fast_used) {
      ProfScope ps("conv_wgrad", s, conv_flops(stem, B), 0);
      if (fast::conv_wgrad<T>(stem_gemm, stem_col, tB, stem_dw_col, B, s))
        stem_wgrad_done = fast::stem_unpack_wgrad(stem_dw_col, G + stem.w_off, in_ch, stem_gemm.Ci, s);
    }
    if (!stem_wgrad_done && stem_tc_used) {
      ProfScope ps("conv_wgrad", s, conv_flops(stem, B), 0);
      bool ok = fast::tc_stem_im2col((const float*)x0, tcw.a16, B, in_ch, in_h, in_w, stem_oh, stem_ow, stem_gemm.Ci, fast::TC_BF16, s) &&
                fast::conv_wgrad_tc(stem_gemm, nullptr, tcw.a16, (const float*)tB, stem_dw_col, B, fast::TC_BF16, fast::TC_BF16, tcw,
                                    s) &&
                fast::stem_unpack_wgrad(stem_dw_col, G + stem.w_off, in_ch, stem_gemm.Ci, s);
      LBC_CHECK(ok, "PREC_F32TC: tensor-core stem weight gradient unavailable");
      stem_wgrad_done = true;
    }
    if (!stem_wgrad_done) {
      LBC_CHECK(!stem_fast_used, "stem weight gradient: fast path failed after a fast forward");
      conv_backward_weight(stem, x0, tB, B, s);
    }
    // (the stem's weight gradient is the last kernel of the chain: nothing left to overlap it with)
    join_side(s);
    mark_bucket(4, s);
#ifndef LBC_HOST_EMU
    if (s != s_in) {
      LBC_CUDA(cudaEventRecord(ev_out, s));
      LBC_CUDA(cudaStreamWaitEvent(s_in, ev_out, 0));
    }
#endif
    ovl = false;
  }

  // ------------------------------------------------------------------ taps
  int64_t read_tap(const char* name_c, float* out, int64_t cap, lbc_stream_t s) override {
    std::string name(name_c);
    const int B = cur_B;
    LBC_CHECK(B > 0, "read_tap before forward");
    auto emit = [&](const T* x, int H, int W, int C) -> int64_t {
      int64_t n = (int64_t)B * H * W * C;
      LBC_CHECK(n <= cap, "read_tap: output buffer too small");
      ref::nhwc_to_nchw_f32<T>(s, x, out, B, H, W, C);
      return n;
    };
    if (name == "stem.raw") return emit(r_stem, stem_oh, stem_ow, 64);
    if (name == "stem.pool") return emit(pool, pool_h, pool_w, 64);
    for (Block& b : blocks)
      if (name == b.name) return emit(b.out, b.Hout, b.Wout, b.Cout);
    for (int i = 0; i < 3; ++i)
      if (name == "deconv." + std::to_string(3 * i + 1)) return emit(dec_out[i], dcv[i].H, dcv[i].W, dcv[i].Ci);
    if (name == "logits") {
      int64_t n = (int64_t)B * 20 * head_h * head_w;
      LBC_CHECK(n <= cap, "read_tap: output buffer too small");
      dev_copy(out, logits, sizeof(float) * n, s);
      return n;
    }
    throw Error("read_tap: unknown tap '" + name + "'");
  }
};

std::unique_ptr<NetBase> make_net(NetKind kind, Precision prec, int max_batch) {
  LBC_CHECK(kind == NET_IMAGE_RESNET34 || kind == NET_BIRDVIEW_RESNET18, "unknown net kind");
  LBC_CHECK(max_batch >= 1, "max_batch must be >= 1");
  if (prec == PREC_F32 || prec == PREC_F32TC) return std::unique_ptr<NetBase>(new Net<float>(kind, prec, max_batch));
  if (prec == PREC_BF16) return std::unique_ptr<NetBase>(new Net<bf16>(kind, prec, max_batch));
  throw Error("unknown precision");
}

}  // namespace lbc
