// lbc_capi.cu -- extern "C" surface declared in include/lbc_b200.h.
#include <mutex>

#include "../../include/lbc_b200.h"
#include "lbc_fast.h"
#include "lbc_head.h"
#include "lbc_net.h"
#include "lbc_ref_ops.h"

using namespace lbc;

struct lbc_net {
  std::unique_ptr<NetBase> impl;
  int device = -1;   // CUDA device the engine (workspace, streams, events) lives on
};
// The library's scratch buffers (statistics partials, split-K partials), kernel attributes and occupancy figures are
// process-wide and belong to the device of the FIRST engine: one process drives one GPU (torchrun's model).  A second engine
// on another device, or a call with another device current, is an error here rather than a corrupted buffer later.
static int g_engine_device = -1;
static void check_device(const lbc_net* net, const char* what) {
#ifndef LBC_HOST_EMU
  int dev = -1;
  cudaGetDevice(&dev);
  if (dev != net->device)
    throw Error(std::string(what) + ": CUDA device " + std::to_string(dev) + " is current, the engine lives on device " +
                std::to_string(net->device) + " (torch.cuda.set_device before calling; one process per GPU)");
#else
  (void)net;
  (void)what;
#endif
}

static thread_local std::string g_err;

template <class F>
static int guarded(F f) {
  try {
    f();
    return 0;
  } catch (const std::exception& e) {
    g_err = e.what();
    return 1;
  } catch (...) {
    g_err = "unknown error";
    return 2;
  }
}

static inline lbc_stream_t S(void* s) { return (lbc_stream_t)s; }

static void require_device() {
#ifndef LBC_HOST_EMU
  static std::once_flag once;
  static std::string err;
  std::call_once(once, [] {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
      err = std::string("liblbc_b200 needs a CUDA device (sm_100a); cudaGetDeviceCount: ") +
            (e == cudaSuccess ? "0 devices" : cudaGetErrorString(e));
      return;
    }
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceProp p;
    cudaGetDeviceProperties(&p, dev);
    if (p.major != 10) err = "liblbc_b200 is built for sm_100a only; found sm_" + std::to_string(p.major * 10 + p.minor);
  });
  if (!err.empty()) throw Error(err);
#endif
}

// ------------------------------------------------------------------ single-op entry points
namespace {
struct Tmp {
  std::vector<void*> v;
  template <class U>
  U* get(int64_t n) {
    void* p = dev_alloc(sizeof(U) * (size_t)n);
    v.push_back(p);
    return (U*)p;
  }
  ~Tmp() {
    for (void* p : v) dev_free(p);
  }
};
void sync_stream(lbc_stream_t s) {
#ifndef LBC_HOST_EMU
  LBC_CUDA(cudaStreamSynchronize(s));
#else
  (void)s;
#endif
}
// operand-split scratch of the fp32tc single-op calls
fast::TcWork make_tcwork(Tmp& t, int64_t a_bytes, int64_t b_bytes) {
  fast::TcWork w;
  w.a_bytes = a_bytes;
  w.b_bytes = b_bytes;
  w.a16 = t.get<uint8_t>(a_bytes);
  w.b16 = t.get<uint8_t>(b_bytes);
  return w;
}
ConvL make_conv(int H, int W, int Ci, int Co, int K, int stride, int pad) {
  ConvL c;
  c.Ci = Ci;
  c.Co = Co;
  c.K = K;
  c.stride = stride;
  c.pad = pad;
  c.H = H;
  c.W = W;
  c.OH = (H + 2 * pad - K) / stride + 1;
  c.OW = (W + 2 * pad - K) / stride + 1;
  return c;
}
}  // namespace

extern "C" {

const char* lbc_last_error(void) { return g_err.c_str(); }

int lbc_device_kind(void) {
#ifdef LBC_HOST_EMU
  return 0;
#else
  return 1;
#endif
}
const char* lbc_build_info(void) {
#ifdef LBC_HOST_EMU
  return "lbc host-emulation build (tests only)";
#else
  return "lbc_b200 CUDA build, sm_100a, " __DATE__ " " __TIME__;
#endif
}
int lbc_set_fast_kernels(int enabled) {
  fast::set_enabled((enabled & 1) != 0);
  fast::set_c64_variant((enabled & 2) == 0);   // bit 1 set: keep the generic tap-per-box kernel for 64->64 3x3 convs
  // variant switches (absent bits keep the LBC_PAIR default): 4 / 8 = CTA-pair (cta_group::2) conv GEMMs on / off,
  // 16 / 32 = row-of-taps weight-gradient kernel on / off
  int m = fast::pair_mode();
  if (enabled & 4) m |= 1;
  if (enabled & 8) m &= ~1;
  if (enabled & 16) m |= 2;
  if (enabled & 32) m &= ~2;
  if (enabled & 64) m |= 4;     // 64 / 128 = CTA-pair variant of the row-of-taps weight gradient on / off
  if (enabled & 128) m &= ~4;
  if (enabled & 256) m |= 8;    // 256 / 512 = space-to-depth layout of the RGB stem operand on / off
  if (enabled & 512) m &= ~8;
  if (enabled & 1024) m |= 16;    // 1024 / 2048 = shared-row CTA-pair kernel for the 3x3/s1 convolutions with 128-wide N tiles on / off
  if (enabled & 2048) m &= ~16;
  if (enabled & 4096) m |= 32;    // 4096 / 8192 = ... also for the layers whose channel count is a multiple of 256
  if (enabled & 8192) m &= ~32;
  if (enabled & 16384) m |= 64;    // 16384 / 32768 = all-nine-taps weight gradient of the 64 -> 64 3x3 convolutions on / off
  if (enabled & 32768) m &= ~64;
  if (enabled & 65536) m |= 128;    // 65536 / 131072 = 64-channel 3x3/s1 convolutions on the shared-row CTA-pair kernel (64-wide N tiles) on / off
  if (enabled & 131072) m &= ~128;
  fast::set_pair_mode(m);
  return 0;
}
int lbc_set_schedule(int wgrad_overlap, int pdl) {
  if (wgrad_overlap >= 0) g_wgrad_overlap = wgrad_overlap > 2 ? 2 : wgrad_overlap;
#ifndef LBC_HOST_EMU
  if (pdl >= 0) g_pdl = pdl ? 1 : 0;
#else
  (void)pdl;
#endif
  return 0;
}
int lbc_stem_layout(int C, int W, int normalize) { return fast::stem_ch(C, W, normalize != 0); }

long long lbc_kernel_launch_count(void) { return g_launches; }
int lbc_prof_enable(int on) {
  g_prof_on = on != 0;
  return 0;
}
int lbc_prof_reset(void) {
#ifndef LBC_HOST_EMU
  cudaDeviceSynchronize();
  for (auto& e : g_prof) {
    cudaEventDestroy(e.e0);
    cudaEventDestroy(e.e1);
  }
#endif
  g_prof.clear();
  return 0;
}
int lbc_prof_get(const char* category, double* total_ms, long long* count, double* flops, double* bytes) {
  return guarded([&] {
    double ms = 0, fl = 0, by = 0;
    long long n = 0;
#ifndef LBC_HOST_EMU
    LBC_CUDA(cudaDeviceSynchronize());
#endif
    for (auto& e : g_prof) {
      if (e.cat != category) continue;
#ifndef LBC_HOST_EMU
      float t = 0.f;
      LBC_CUDA(cudaEventElapsedTime(&t, e.e0, e.e1));
      ms += t;
#endif
      fl += e.flops;
      by += e.bytes;
      ++n;
    }
    *total_ms = ms;
    *count = n;
    *flops = fl;
    *bytes = by;
  });
}

int lbc_net_create(int kind, int precision, int max_batch, lbc_net_t** out) {
  return guarded([&] {
    require_device();
    LBC_CHECK(out, "null out pointer");
    lbc_net* n = new lbc_net;
#ifndef LBC_HOST_EMU
    cudaGetDevice(&n->device);
    if (g_engine_device < 0) g_engine_device = n->device;
    if (n->device != g_engine_device) {
      const int d = n->device;
      delete n;
      throw Error("lbc_net_create: this process already runs engines on CUDA device " + std::to_string(g_engine_device) +
                  "; device " + std::to_string(d) + " needs its own process (the library's scratch buffers are per process)");
    }
#endif
    try {
      n->impl = make_net((NetKind)kind, (Precision)precision, max_batch);
    } catch (...) {
      delete n;
      throw;
    }
    *out = n;
  });
}
void lbc_net_destroy(lbc_net_t* net) { delete net; }
int lbc_net_num_params(const lbc_net_t* net) { return (int)net->impl->params.size(); }
int lbc_net_param_info(const lbc_net_t* net, int i, const char** name, int* ndim, int shape[4], int64_t* numel,
                       int64_t* offset, int* on_path) {
  return guarded([&] {
    LBC_CHECK(i >= 0 && i < (int)net->impl->params.size(), "param index out of range");
    const ParamInfo& p = net->impl->params[i];
    *name = p.name.c_str();
    *ndim = p.ndim;
    for (int d = 0; d < 4; ++d) shape[d] = p.shape[d];
    *numel = p.numel;
    *offset = p.offset;
    *on_path = p.on_path ? 1 : 0;
  });
}
int lbc_net_num_buffers(const lbc_net_t* net) { return (int)net->impl->buffers.size(); }
int lbc_net_buffer_info(const lbc_net_t* net, int i, const char** name, int64_t* numel, int64_t* offset) {
  return guarded([&] {
    LBC_CHECK(i >= 0 && i < (int)net->impl->buffers.size(), "buffer index out of range");
    const BufferInfo& b = net->impl->buffers[i];
    *name = b.name.c_str();
    *numel = b.numel;
    *offset = b.offset;
  });
}
int64_t lbc_net_total_params(const lbc_net_t* net) { return net->impl->n_params; }
int64_t lbc_net_total_buffers(const lbc_net_t* net) { return net->impl->n_buffers; }
int64_t lbc_net_workspace_bytes(const lbc_net_t* net) { return (int64_t)net->impl->workspace_bytes(); }
int lbc_net_bind(lbc_net_t* net, float* params, float* grads, float* buffers) {
  return guarded([&] {
    LBC_CHECK(params && buffers, "lbc_net_bind: null params/buffers");
    net->impl->bind(params, grads, buffers);
  });
}
int lbc_net_forward(lbc_net_t* net, const float* image, const float* speed, const float* command_onehot, int B,
                    int train, float* out_pred, float* out_preds, void* stream) {
  return guarded([&] {
    check_device(net, "lbc_net_forward");
    LBC_CHECK(image && speed && command_onehot, "lbc_net_forward: null input");
    net->impl->forward(image, speed, command_onehot, B, train != 0, out_pred, out_preds, S(stream));
  });
}
int lbc_net_forward_u8(lbc_net_t* net, const uint8_t* image_u8, int layout, const float* speed,
                       const float* command_onehot, int B, int train, float* out_pred, float* out_preds, void* stream) {
  return guarded([&] {
    check_device(net, "lbc_net_forward_u8");
    LBC_CHECK(image_u8 && speed && command_onehot, "lbc_net_forward_u8: null input");
    net->impl->forward_u8(image_u8, layout, speed, command_onehot, B, train != 0, out_pred, out_preds, S(stream));
  });
}
int lbc_net_infer(lbc_net_t* net, const float* image, const uint8_t* image_u8, int layout, const float* speed,
                  const float* command_onehot, int B, int weights_changed, float* out_pred, float* out_preds, void* stream) {
  return guarded([&] {
    check_device(net, "lbc_net_infer");
    net->impl->infer(image, image_u8, layout, speed, command_onehot, B, weights_changed != 0, out_pred, out_preds, S(stream));
  });
}
int lbc_net_infer_replays(const lbc_net_t* net) { return net->impl->infer_replays; }
int lbc_net_backward(lbc_net_t* net, const float* d_pred, const float* d_preds, void* stream) {
  return guarded([&] {
    check_device(net, "lbc_net_backward");
    net->impl->backward(d_pred, d_preds, S(stream));
  });
}
int lbc_net_num_grad_buckets(const lbc_net_t* net) { return (int)net->impl->buckets.size(); }
int lbc_net_grad_bucket(const lbc_net_t* net, int bucket, int64_t* offset, int64_t* numel) {
  return guarded([&] {
    LBC_CHECK(bucket >= 0 && bucket < (int)net->impl->buckets.size(), "gradient bucket index out of range");
    *offset = net->impl->buckets[bucket].offset;
    *numel = net->impl->buckets[bucket].numel;
  });
}
int lbc_net_enable_grad_events(lbc_net_t* net, int on) {
  return guarded([&] { net->impl->enable_grad_events(on != 0); });
}
int lbc_net_stream_wait_grads(lbc_net_t* net, int bucket, void* stream) {
  return guarded([&] { net->impl->stream_wait_bucket(bucket, S(stream)); });
}
int64_t lbc_net_read_tap(lbc_net_t* net, const char* name, float* out, int64_t capacity, void* stream) {
  int64_t n = -1;
  int rc = guarded([&] {
    check_device(net, "lbc_net_read_tap");
    n = net->impl->read_tap(name, out, capacity, S(stream));
  });
  return rc == 0 ? n : -1;
}

int lbc_phase0_target(const float* teacher_pred, float* target_px, int64_t count, float w, float h, float fov_deg,
                      float world_y, float fixed_offset, void* stream) {
  return guarded([&] {
    require_device();
    ref::phase0_target(S(stream), teacher_pred, target_px, count, w, h, fov_deg, world_y, fixed_offset);
  });
}
int lbc_l1_loss(const float* a, const float* b, int N, int D, float sa, float ta, float sbx, float sby, float tb,
                const float* gout, float* loss_b, float* da, void* stream) {
  return guarded([&] {
    require_device();
    ref::l1_loss(S(stream), a, b, N, D, sa, ta, sbx, sby, tb, gout, loss_b, da);
  });
}
int lbc_phase1_convert_fwd(const float* p, float* out, int64_t count, float w, float h, float fov_deg,
                           float world_y, float fixed_offset, void* stream) {
  return guarded([&] {
    require_device();
    ref::phase1_convert_fwd(S(stream), p, out, count, w, h, fov_deg, world_y, fixed_offset);
  });
}
int lbc_phase1_convert_bwd(const float* p, const float* dout, float* dp, int64_t count, float w, float h,
                           float fov_deg, float world_y, float fixed_offset, void* stream) {
  return guarded([&] {
    require_device();
    ref::phase1_convert_bwd(S(stream), p, dout, dp, count, w, h, fov_deg, world_y, fixed_offset);
  });
}
int lbc_phase2_weight(const float* learner_map, const float* teacher_map, float* weight, int N, void* stream) {
  return guarded([&] {
    require_device();
    ref::phase2_weight(S(stream), learner_map, teacher_map, weight, N);
  });
}
int lbc_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                  float beta1, float beta2, float eps, int step, float grad_scale, void* stream) {
  return guarded([&] {
    require_device();
    LBC_CHECK(step >= 1, "adam step counter starts at 1");
    ref::adam(S(stream), params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step, grad_scale);
  });
}

// ------------------------------------------------------------------ launch trace
int lbc_trace_enable(int on) {
  if (on) trace_reset();
  g_trace_on = on != 0;
  return 0;
}
int lbc_trace_dump(char* buf, int cap) {
  std::string t = trace_dump();
  if (buf && cap > 0) {
    int n = (int)t.size() < cap - 1 ? (int)t.size() : cap - 1;
    memcpy(buf, t.data(), n);
    buf[n] = 0;
  }
  return (int)t.size();
}

// ------------------------------------------------------------------ single-op entry points
// precision LBC_PREC_F32: correctness-first fp32 kernels.  LBC_PREC_BF16: the operands are rounded to bf16 storage and go
// through the kernels the bf16 training step runs (tcgen05 GEMMs, fused BN / pool / head kernels); results come back as
// fp32.  The tests compare with torch on the same rounded operands and read lbc_trace_dump to see which kernel ran.

int lbc_op_conv_fwd(const float* x, const float* w_ref, float* y, int N, int H, int W, int Ci, int Co, int K,
                    int stride, int pad, int precision, const float* bias_co, float* stats_out, void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    ConvL c = make_conv(H, W, Ci, Co, K, stride, pad);
    Tmp t;
    int64_t nx = (int64_t)N * H * W * Ci, ny = (int64_t)N * c.OH * c.OW * Co, nw = (int64_t)Co * K * K * Ci;
    if (precision == PREC_F32) {
      LBC_CHECK(!stats_out, "lbc_op_conv_fwd: epilogue statistics exist on the bf16 path only");
      float* wp = t.get<float>(nw);
      ref::pack_weight<float>(s, w_ref, wp, Co, Ci, K);
      ref::conv_fwd<float>(s, x, wp, bias_co, false, y, N, H, W, Ci, Co, K, stride, pad, c.OH, c.OW);
    } else if (precision == PREC_F32TC) {
      LBC_CHECK(!stats_out, "lbc_op_conv_fwd: epilogue statistics exist on the bf16 path only");
      float *wp = t.get<float>(nw), *w16 = t.get<float>(nw);
      ref::pack_weight<float>(s, w_ref, wp, Co, Ci, K);
      LBC_CHECK(fast::tc_split(wp, w16, (int64_t)Co * K * K, Ci, fast::TC_F16, fast::kTcWeightScale, s), "tc_split unavailable");
      c.wp16 = w16;
      fast::TcWork tw = make_tcwork(t, nx * 4, 16);
      LBC_CHECK(fast::conv_fwd_tc(c, x, nullptr, y, N, bias_co, false, fast::TC_F16, tw, s), "conv_fwd_tc declined the shape");
    } else {
      bf16 *xb = t.get<bf16>(nx), *wb = t.get<bf16>(nw), *yb = t.get<bf16>(ny);
      ref::cast<float, bf16>(s, x, xb, nx);
      ref::pack_weight<bf16>(s, w_ref, wb, Co, Ci, K);
      c.wp = wb;
      int rows = 0;
      float* part = stats_out ? fast::stat_partial_buffer() : nullptr;
      if (fast::conv_fwd<bf16>(c, xb, yb, N, s, bias_co, part, &rows)) {
        if (stats_out) {
          LBC_CHECK(part && rows > 0, "lbc_op_conv_fwd: the fast kernel emitted no statistics partials");
          LBC_CHECK(fast::col_finalize_bf16(part, rows, 2 * Co, stats_out, s), "col_finalize failed");
        }
      } else {
        LBC_CHECK(!stats_out, "lbc_op_conv_fwd: statistics requested but the fast kernel did not run");
        ref::conv_fwd<bf16>(s, xb, wb, bias_co, false, yb, N, H, W, Ci, Co, K, stride, pad, c.OH, c.OW);
      }
      ref::cast<bf16, float>(s, yb, y, ny);
    }
    sync_stream(s);
  });
}
// bias_ci / relu: the epilogue of nn.ConvTranspose2d(..)+bias -> ReLU (image.py:39-46), which is this data gradient
int lbc_op_conv_dgrad(const float* dy, const float* w_ref, float* dx, int N, int H, int W, int Ci, int Co, int K,
                      int stride, int pad, int precision, const float* bias_ci, int relu, void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    ConvL c = make_conv(H, W, Ci, Co, K, stride, pad);
    Tmp t;
    int64_t nx = (int64_t)N * H * W * Ci, ny = (int64_t)N * c.OH * c.OW * Co, nw = (int64_t)Co * K * K * Ci;
    if (precision == PREC_F32) {
      float* wp = t.get<float>(nw);
      ref::pack_weight<float>(s, w_ref, wp, Co, Ci, K);
      ref::conv_dgrad<float>(s, dy, wp, dx, N, H, W, Ci, Co, K, stride, pad, c.OH, c.OW, bias_ci, relu != 0, false);
    } else if (precision == PREC_F32TC) {
      // relu != 0 marks the ConvTranspose2d forward (dy is an activation: fp16 planes); otherwise dy is a gradient (bf16 planes)
      const int fmt = relu ? fast::TC_F16 : fast::TC_BF16;
      float *wt = t.get<float>(nw), *w16 = t.get<float>(nw);
      ref::pack_weight_t<float>(s, w_ref, wt, Co, Ci, K);
      LBC_CHECK(fast::tc_split(wt, w16, (int64_t)Ci * K * K, Co, fmt, fast::kTcWeightScale, s), "tc_split unavailable");
      c.wpt16 = w16;
      fast::TcWork tw = make_tcwork(t, ny * 4, 16);
      LBC_CHECK(fast::conv_dgrad_tc(c, dy, nullptr, dx, N, bias_ci, relu != 0, fmt, tw, s), "conv_dgrad_tc declined the shape");
    } else {
      bf16 *xb = t.get<bf16>(nx), *wb = t.get<bf16>(nw), *yb = t.get<bf16>(ny);
      bf16* wtb = t.get<bf16>(nw);
      ref::cast<float, bf16>(s, dy, yb, ny);
      ref::pack_weight<bf16>(s, w_ref, wb, Co, Ci, K);
      ref::pack_weight_t<bf16>(s, w_ref, wtb, Co, Ci, K);
      c.wp = wb;
      c.wpt = wtb;
      if (!fast::conv_dgrad<bf16>(c, yb, xb, N, bias_ci, relu != 0, s))
        ref::conv_dgrad<bf16>(s, yb, wb, xb, N, H, W, Ci, Co, K, stride, pad, c.OH, c.OW, bias_ci, relu != 0, false);
      ref::cast<bf16, float>(s, xb, dx, nx);
    }
    sync_stream(s);
  });
}
// gradient wrt the input of a stage-entry block: dgrad(3x3/s2 conv1)(dy1) + dgrad(1x1/s2 downsample)(dy_ds) (resnet.py:48-52)
int lbc_op_block_dgrad_ds(const float* dy1, const float* dy_ds, const float* w1_ref, const float* wd_ref, float* dx, int N,
                          int H, int W, int Ci, int Co, int precision, void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    ConvL c1 = make_conv(H, W, Ci, Co, 3, 2, 1), cd = make_conv(H, W, Ci, Co, 1, 2, 0);
    Tmp t;
    int64_t nx = (int64_t)N * H * W * Ci, ny = (int64_t)N * c1.OH * c1.OW * Co;
    if (precision == PREC_F32) {
      float *w1 = t.get<float>((int64_t)Co * 9 * Ci), *wd = t.get<float>((int64_t)Co * Ci);
      ref::pack_weight<float>(s, w1_ref, w1, Co, Ci, 3);
      ref::pack_weight<float>(s, wd_ref, wd, Co, Ci, 1);
      ref::conv_dgrad<float>(s, dy1, w1, dx, N, H, W, Ci, Co, 3, 2, 1, c1.OH, c1.OW, nullptr, false, false);
      ref::conv_dgrad<float>(s, dy_ds, wd, dx, N, H, W, Ci, Co, 1, 2, 0, cd.OH, cd.OW, nullptr, false, true);
    } else if (precision == PREC_F32TC) {
      const int64_t nw = (int64_t)Co * 9 * Ci, nc = (int64_t)Ci * 2 * Co;
      float *w1t = t.get<float>(nw), *w1t16 = t.get<float>(nw), *wc = t.get<float>(nc), *wc16 = t.get<float>(nc);
      ref::pack_weight_t<float>(s, w1_ref, w1t, Co, Ci, 3);
      ref::pack_weight_comb<float>(s, w1_ref, wd_ref, wc, Co, Ci);
      LBC_CHECK(fast::tc_split(w1t, w1t16, (int64_t)Ci * 9, Co, fast::TC_BF16, fast::kTcWeightScale, s) &&
                    fast::tc_split(wc, wc16, (int64_t)Ci * 2, Co, fast::TC_BF16, fast::kTcWeightScale, s),
                "tc_split unavailable");
      c1.wpt16 = w1t16;
      c1.wcomb16 = wc16;
      fast::TcWork tw = make_tcwork(t, ny * 4, ny * 4);
      LBC_CHECK(fast::conv_dgrad_tc(c1, dy1, dy_ds, dx, N, nullptr, false, fast::TC_BF16, tw, s), "conv_dgrad_tc (fused) declined the shape");
    } else {
      bf16 *d1 = t.get<bf16>(ny), *d2 = t.get<bf16>(ny), *xb = t.get<bf16>(nx);
      bf16 *w1 = t.get<bf16>((int64_t)Co * 9 * Ci), *w1t = t.get<bf16>((int64_t)Co * 9 * Ci), *wd = t.get<bf16>((int64_t)Co * Ci);
      bf16* wcomb = t.get<bf16>((int64_t)Ci * 2 * Co);
      ref::cast<float, bf16>(s, dy1, d1, ny);
      ref::cast<float, bf16>(s, dy_ds, d2, ny);
      ref::pack_weight<bf16>(s, w1_ref, w1, Co, Ci, 3);
      ref::pack_weight_t<bf16>(s, w1_ref, w1t, Co, Ci, 3);
      ref::pack_weight<bf16>(s, wd_ref, wd, Co, Ci, 1);
      ref::pack_weight_comb<bf16>(s, w1_ref, wd_ref, wcomb, Co, Ci);
      c1.wp = w1;
      c1.wpt = w1t;
      c1.wcomb = wcomb;
      if (!fast::conv_dgrad_ds<bf16>(c1, d1, d2, xb, N, s)) {
        ref::conv_dgrad<bf16>(s, d1, w1, xb, N, H, W, Ci, Co, 3, 2, 1, c1.OH, c1.OW, nullptr, false, false);
        ref::conv_dgrad<bf16>(s, d2, wd, xb, N, H, W, Ci, Co, 1, 2, 0, cd.OH, cd.OW, nullptr, false, true);
      }
      ref::cast<bf16, float>(s, xb, dx, nx);
    }
    sync_stream(s);
  });
}
int lbc_op_conv_wgrad(const float* x, const float* dy, float* dw_ref, int N, int H, int W, int Ci, int Co, int K,
                      int stride, int pad, int precision, void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    ConvL c = make_conv(H, W, Ci, Co, K, stride, pad);
    Tmp t;
    int64_t nx = (int64_t)N * H * W * Ci, ny = (int64_t)N * c.OH * c.OW * Co;
    int64_t wsn = 4 << 20;
    float* ws = t.get<float>(wsn);
    if (precision == PREC_F32) {
      ref::conv_wgrad<float>(s, x, dy, dw_ref, N, H, W, Ci, Co, K, stride, pad, c.OH, c.OW, ws, wsn);
    } else if (precision == PREC_F32TC) {
      fast::TcWork tw = make_tcwork(t, nx * 4, ny * 4);
      LBC_CHECK(fast::conv_wgrad_tc(c, x, nullptr, dy, dw_ref, N, fast::TC_BF16, fast::TC_BF16, tw, s),
                "conv_wgrad_tc declined the shape");
    } else {
      bf16 *xb = t.get<bf16>(nx), *yb = t.get<bf16>(ny);
      ref::cast<float, bf16>(s, x, xb, nx);
      ref::cast<float, bf16>(s, dy, yb, ny);
      if (!fast::conv_wgrad<bf16>(c, xb, yb, dw_ref, N, s))
        ref::conv_wgrad<bf16>(s, xb, yb, dw_ref, N, H, W, Ci, Co, K, stride, pad, c.OH, c.OW, ws, wsn);
    }
    sync_stream(s);
  });
}
// nn.BatchNorm2d in train mode (+ residual, + ReLU) over [M][C].  running_mean / running_var (optional) are updated in
// place; negshift (bf16 path, optional): x holds (true x + negshift[c]) -- the centring shift of DESIGN.md -- and is
// replaced by -(batch mean of the true x).
int lbc_op_bn_train(const float* x, const float* gamma, const float* beta, const float* residual, int relu,
                    float* y, float* mean, float* var, int64_t M, int C, int precision, float* running_mean,
                    float* running_var, float* negshift, uint8_t* mask_bits_out, void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    Tmp t;
    float* rstd = t.get<float>(C);
    if (precision == PREC_F32) {
      LBC_CHECK(!negshift && !mask_bits_out, "lbc_op_bn_train: centring shift / mask bits exist on the bf16 path only");
      double* ws = t.get<double>(1 << 20);
      ref::bn_stats<float>(s, x, M, C, mean, var, ws);
      ref::bn_finalize(s, mean, var, C, M, 1e-5f, 0.1f, rstd, running_mean, running_var);
      ref::bn_apply<float>(s, x, mean, rstd, gamma, beta, residual, relu != 0, y, M, C);
    } else {
      const int64_t n = M * C;
      bf16 *xb = t.get<bf16>(n), *yb = t.get<bf16>(n), *rb = residual ? t.get<bf16>(n) : nullptr;
      float *sums = t.get<float>(2 * C), *rm = running_mean ? running_mean : t.get<float>(C),
            *rv = running_var ? running_var : t.get<float>(C);
      if (!running_mean) dev_memset(rm, 0, sizeof(float) * C, s);
      if (!running_var) dev_memset(rv, 0, sizeof(float) * C, s);
      ref::cast<float, bf16>(s, x, xb, n);
      if (residual) ref::cast<float, bf16>(s, residual, rb, n);
      if (!fast::Fast<bf16>::bn_fwd(xb, M, C, gamma, beta, 1e-5f, 0.1f, rm, rv, mean, rstd, rb, relu != 0, true, yb, sums,
                                    negshift, s, 0, mask_bits_out)) {
        LBC_CHECK(!negshift && !mask_bits_out, "lbc_op_bn_train: centring shift / mask bits requested but the fast kernels did not run");
        double* ws = t.get<double>(1 << 20);
        ref::bn_stats<bf16>(s, xb, M, C, mean, var, ws);
        ref::bn_finalize(s, mean, var, C, M, 1e-5f, 0.1f, rstd, rm, rv);
        ref::bn_apply<bf16>(s, xb, mean, rstd, gamma, beta, rb, relu != 0, yb, M, C);
      } else {
        ref::rstd_to_var(s, rstd, var, C, 1e-5f);
      }
      ref::cast<bf16, float>(s, yb, y, n);
    }
    sync_stream(s);
  });
}
// BatchNorm backward with batch statistics recomputed from x.  mask_act (optional, [M][C]): dy is first masked with
// (mask_act > 0) -- the in-place ReLU that follows the BN; own_relu != 0: that activation is relu(bn(x)) of this very BN
// (beta required), which the fast kernels recompute from x instead of reading mask_act.
int lbc_op_bn_bwd(const float* dy, const float* x, const float* gamma, float* dgamma, float* dbeta, float* dx,
                  int64_t M, int C, int precision, const float* mask_act, const float* beta, int own_relu, int use_mask_bits,
                  void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    Tmp t;
    double* ws = t.get<double>(1 << 20);
    float *mean = t.get<float>(C), *var = t.get<float>(C), *rstd = t.get<float>(C);
    const int64_t n = M * C;
    LBC_CHECK(!own_relu || (mask_act && beta), "lbc_op_bn_bwd: own_relu needs mask_act and beta");
    if (precision == PREC_F32) {
      float* dym = t.get<float>(n);
      dev_copy(dym, dy, sizeof(float) * n, s);
      if (mask_act) ref::relu_mask_inplace<float>(s, dym, mask_act, n);
      ref::bn_stats<float>(s, x, M, C, mean, var, ws);
      ref::bn_finalize(s, mean, var, C, M, 1e-5f, 0.1f, rstd, nullptr, nullptr);
      ref::bn_bwd<float>(s, dym, x, mean, rstd, gamma, dgamma, dbeta, dx, M, C, ws);
    } else {
      bf16 *xb = t.get<bf16>(n), *dyb = t.get<bf16>(n), *dxb = t.get<bf16>(n), *mb = mask_act ? t.get<bf16>(n) : nullptr;
      float* sums = t.get<float>(2 * C);
      ref::cast<float, bf16>(s, x, xb, n);
      ref::cast<float, bf16>(s, dy, dyb, n);
      if (mask_act) ref::cast<float, bf16>(s, mask_act, mb, n);
      uint8_t* bits = nullptr;
      if (use_mask_bits && mask_act && !own_relu) {   // the mask as the bits bn_apply_kernel writes for the block-final ReLU
        bits = t.get<uint8_t>(n / 8);
        ref::pack_mask_bits<bf16>(s, mb, bits, n / 8);
      }
      ref::bn_stats<bf16>(s, xb, M, C, mean, var, ws);
      ref::bn_finalize(s, mean, var, C, M, 1e-5f, 0.1f, rstd, nullptr, nullptr);
      if (!fast::Fast<bf16>::bn_bwd(dyb, mb, xb, mean, rstd, gamma, dgamma, dbeta, dxb, M, C, sums, s, own_relu ? beta : nullptr,
                                    bits)) {
        if (mb) ref::relu_mask_inplace<bf16>(s, dyb, mb, n);
        ref::bn_bwd<bf16>(s, dyb, xb, mean, rstd, gamma, dgamma, dbeta, dxb, M, C, ws);
      }
      ref::cast<bf16, float>(s, dxb, dx, n);
    }
    sync_stream(s);
  });
}
// The residual blocks' d(out) chain in one op (resnet.py:41-53 backward): dst += src * (act > 0), then the BatchNorm backward
// of  dst * (act_prev > 0)  with respect to x (batch statistics of x).  bf16 path: the add and the reduce pass are ONE kernel
// (bn_bwd_reduce_kernel<resid>), both masks travel as bits, then col_finalize + bn_bwd_apply_kernel.
int lbc_op_resid_bn_bwd(float* dst, const float* src, const float* act, const float* x, const float* act_prev,
                        const float* gamma, float* dgamma, float* dbeta, float* dx, int64_t M, int C, int precision,
                        void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    Tmp t;
    double* ws = t.get<double>(1 << 20);
    float *mean = t.get<float>(C), *var = t.get<float>(C), *rstd = t.get<float>(C);
    const int64_t n = M * C;
    if (precision == PREC_F32) {
      ref::add_masked_inplace<float>(s, dst, src, act, n);
      float* dym = t.get<float>(n);
      dev_copy(dym, dst, sizeof(float) * n, s);
      ref::relu_mask_inplace<float>(s, dym, act_prev, n);
      ref::bn_stats<float>(s, x, M, C, mean, var, ws);
      ref::bn_finalize(s, mean, var, C, M, 1e-5f, 0.1f, rstd, nullptr, nullptr);
      ref::bn_bwd<float>(s, dym, x, mean, rstd, gamma, dgamma, dbeta, dx, M, C, ws);
    } else {
      bf16 *d = t.get<bf16>(n), *sr = t.get<bf16>(n), *a = t.get<bf16>(n), *ap = t.get<bf16>(n), *xb = t.get<bf16>(n),
           *dxb = t.get<bf16>(n);
      float* sums = t.get<float>(2 * C);
      uint8_t *bits = t.get<uint8_t>(n / 8), *pbits = t.get<uint8_t>(n / 8);
      ref::cast<float, bf16>(s, dst, d, n);
      ref::cast<float, bf16>(s, src, sr, n);
      ref::cast<float, bf16>(s, act, a, n);
      ref::cast<float, bf16>(s, act_prev, ap, n);
      ref::cast<float, bf16>(s, x, xb, n);
      ref::pack_mask_bits<bf16>(s, a, bits, n / 8);
      ref::pack_mask_bits<bf16>(s, ap, pbits, n / 8);
      ref::bn_stats<bf16>(s, xb, M, C, mean, var, ws);
      ref::bn_finalize(s, mean, var, C, M, 1e-5f, 0.1f, rstd, nullptr, nullptr);
      int rows = 0;
      if (fast::Fast<bf16>::resid_bn_reduce(d, sr, bits, xb, mean, rstd, pbits, M, C, &rows, s)) {
        LBC_CHECK(fast::Fast<bf16>::bn_bwd(d, ap, xb, mean, rstd, gamma, dgamma, dbeta, dxb, M, C, sums, s, nullptr, pbits, rows),
                  "lbc_op_resid_bn_bwd: BatchNorm backward fast path unavailable");
      } else {
        ref::add_masked_inplace<bf16>(s, d, sr, a, n);
        bf16* dm = t.get<bf16>(n);
        dev_copy(dm, d, sizeof(bf16) * n, s);
        ref::relu_mask_inplace<bf16>(s, dm, ap, n);
        ref::bn_bwd<bf16>(s, dm, xb, mean, rstd, gamma, dgamma, dbeta, dxb, M, C, ws);
      }
      ref::cast<bf16, float>(s, d, dst, n);
      ref::cast<bf16, float>(s, dxb, dx, n);
    }
    sync_stream(s);
  });
}
// masked adds of the residual backward: mode 0 dst += src; 1 dst += src*(act>0); 2 dst *= (act>0)
int lbc_op_ew(float* dst, const float* src, const float* act, int64_t n, int mode, int precision, int use_mask_bits,
              void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    Tmp t;
    LBC_CHECK(mode >= 0 && mode <= 2, "lbc_op_ew: mode 0..2");
    if (precision == PREC_F32) {
      if (mode == 0) ref::add_inplace<float>(s, dst, src, n);
      else if (mode == 1) ref::add_masked_inplace<float>(s, dst, src, act, n);
      else ref::relu_mask_inplace<float>(s, dst, act, n);
    } else {
      bf16 *d = t.get<bf16>(n), *sr = src ? t.get<bf16>(n) : nullptr, *a = act ? t.get<bf16>(n) : nullptr;
      ref::cast<float, bf16>(s, dst, d, n);
      if (src) ref::cast<float, bf16>(s, src, sr, n);
      if (act) ref::cast<float, bf16>(s, act, a, n);
      uint8_t* bits = nullptr;
      if (use_mask_bits && act && mode != 0) {
        bits = t.get<uint8_t>(n / 8);
        ref::pack_mask_bits<bf16>(s, a, bits, n / 8);
      }
      if (!fast::Fast<bf16>::ew(d, sr, a, n, mode, s, bits)) {
        if (mode == 0) ref::add_inplace<bf16>(s, d, sr, n);
        else if (mode == 1) ref::add_masked_inplace<bf16>(s, d, sr, a, n);
        else ref::relu_mask_inplace<bf16>(s, d, a, n);
      }
      ref::cast<bf16, float>(s, d, dst, n);
    }
    sync_stream(s);
  });
}
int lbc_op_copy_channels(const float* src, float* dst, int64_t M, int Cd, int Cs, const float* fill, int rows_per_fill,
                         int precision, void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    LBC_CHECK(Cd <= Cs || (fill && rows_per_fill >= 1), "lbc_op_copy_channels: Cd > Cs needs a fill vector");
    LBC_CHECK(Cd <= Cs || (Cs == 512 && Cd == 640), "lbc_op_copy_channels: widening is the 512 + 128 speed fusion");
    Tmp t;
    if (precision == PREC_F32) {
      if (Cd > Cs)
        ref::concat_speed<float>(s, src, fill, dst, (int)(M / rows_per_fill), rows_per_fill, Cs, Cd - Cs);
      else
        ref::slice_channels<float>(s, src, dst, M, Cs, Cd);
    } else {
      bf16 *sb = t.get<bf16>(M * Cs), *db = t.get<bf16>(M * Cd);
      ref::cast<float, bf16>(s, src, sb, M * Cs);
      if (!fast::copy_channels<bf16>(db, sb, M, Cd, Cs, fill, rows_per_fill, s)) {
        if (Cd > Cs)
          ref::concat_speed<bf16>(s, sb, fill, db, (int)(M / rows_per_fill), rows_per_fill, Cs, Cd - Cs);
        else
          ref::slice_channels<bf16>(s, sb, db, M, Cs, Cd);
      }
      ref::cast<bf16, float>(s, db, dst, M * Cd);
    }
    sync_stream(s);
  });
}
int lbc_op_maxpool(const float* x, float* y, const float* dy, float* dx, int N, int H, int W, int C, void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    int OH = (H + 2 - 3) / 2 + 1, OW = (W + 2 - 3) / 2 + 1;
    Tmp t;
    uint8_t* idx = t.get<uint8_t>((int64_t)N * OH * OW * C);
    ref::maxpool_fwd<float>(s, x, y, idx, N, H, W, C, OH, OW);
    if (dy && dx) ref::maxpool_bwd<float>(s, dy, idx, dx, N, H, W, C, OH, OW);
    sync_stream(s);
  });
}
// stem tail: y = maxpool3x3/s2/p1(relu(bn(x))) with GIVEN statistics, and (dy, dx != null) its backward: dx = the
// gradient wrt the BatchNorm output, i.e. maxpool backward times the ReLU mask (resnet.py:150-152)
int lbc_op_bn_relu_maxpool(const float* x, const float* mean, const float* rstd, const float* gamma, const float* beta,
                           float* y, const float* dy, float* dx, int N, int H, int W, int C, int precision, void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    int OH = (H + 2 - 3) / 2 + 1, OW = (W + 2 - 3) / 2 + 1;
    Tmp t;
    const int64_t nx = (int64_t)N * H * W * C, ny = (int64_t)N * OH * OW * C;
    uint8_t* idx = t.get<uint8_t>(ny);
    if (precision == PREC_F32) {
      float* a = t.get<float>(nx);
      ref::bn_apply<float>(s, x, mean, rstd, gamma, beta, nullptr, true, a, (int64_t)N * H * W, C);
      ref::maxpool_fwd<float>(s, a, y, idx, N, H, W, C, OH, OW);
      if (dy && dx) {
        ref::maxpool_bwd<float>(s, dy, idx, dx, N, H, W, C, OH, OW);
        ref::relu_mask_inplace<float>(s, dx, a, nx);
      }
    } else {
      bf16 *xb = t.get<bf16>(nx), *yb = t.get<bf16>(ny), *dyb = t.get<bf16>(ny), *dxb = t.get<bf16>(nx);
      ref::cast<float, bf16>(s, x, xb, nx);
      const bool fwd = fast::Fast<bf16>::pool_fwd(xb, mean, rstd, gamma, beta, yb, idx, N, H, W, C, OH, OW, s);
      bf16* a = nullptr;
      if (!fwd) {
        a = t.get<bf16>(nx);
        ref::bn_apply<bf16>(s, xb, mean, rstd, gamma, beta, nullptr, true, a, (int64_t)N * H * W, C);
        ref::maxpool_fwd<bf16>(s, a, yb, idx, N, H, W, C, OH, OW);
      }
      ref::cast<bf16, float>(s, yb, y, ny);
      if (dy && dx) {
        ref::cast<float, bf16>(s, dy, dyb, ny);
        if (!(fwd && fast::Fast<bf16>::pool_bwd(dyb, idx, xb, mean, rstd, gamma, beta, dxb, N, H, W, C, OH, OW, s))) {
          if (!a) {
            a = t.get<bf16>(nx);
            ref::bn_apply<bf16>(s, xb, mean, rstd, gamma, beta, nullptr, true, a, (int64_t)N * H * W, C);
          }
          ref::maxpool_bwd<bf16>(s, dyb, idx, dxb, N, H, W, C, OH, OW);
          ref::relu_mask_inplace<bf16>(s, dxb, a, nx);
        }
        ref::cast<bf16, float>(s, dxb, dx, nx);
      }
    }
    sync_stream(s);
  });
}
// Whole stem tail, train mode: y = maxpool3x3/s2/p1(relu(batchnorm(x))) with batch statistics, and its backward from
// dy [N][OH][OW][C]: dgamma, dbeta, dx [N][H][W][C] (resnet.py:149-152).  bf16 path: the fused BN+ReLU+MaxPool forward, the
// 2x2-block pool-backward kernel (with the ReLU mask recomputed from x) and the BatchNorm backward kernels, as the step runs them.
int lbc_op_stem_tail(const float* x, const float* gamma, const float* beta, float* y, const float* dy, float* dgamma,
                     float* dbeta, float* dx, int N, int H, int W, int C, int precision, void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    int OH = (H + 2 - 3) / 2 + 1, OW = (W + 2 - 3) / 2 + 1;
    Tmp t;
    const int64_t M = (int64_t)N * H * W, nx = M * C, ny = (int64_t)N * OH * OW * C;
    uint8_t* idx = t.get<uint8_t>(ny);
    double* ws = t.get<double>(1 << 20);
    float *mean = t.get<float>(C), *var = t.get<float>(C), *rstd = t.get<float>(C);
    if (precision == PREC_F32) {
      float *a = t.get<float>(nx), *g = t.get<float>(nx);
      ref::bn_stats<float>(s, x, M, C, mean, var, ws);
      ref::bn_finalize(s, mean, var, C, M, 1e-5f, 0.1f, rstd, nullptr, nullptr);
      ref::bn_apply<float>(s, x, mean, rstd, gamma, beta, nullptr, true, a, M, C);
      ref::maxpool_fwd<float>(s, a, y, idx, N, H, W, C, OH, OW);
      ref::maxpool_bwd<float>(s, dy, idx, g, N, H, W, C, OH, OW);
      ref::relu_mask_inplace<float>(s, g, a, nx);
      ref::bn_bwd<float>(s, g, x, mean, rstd, gamma, dgamma, dbeta, dx, M, C, ws);
    } else {
      bf16 *xb = t.get<bf16>(nx), *yb = t.get<bf16>(ny), *dyb = t.get<bf16>(ny), *dxb = t.get<bf16>(nx);
      float* sums = t.get<float>(2 * C);
      ref::cast<float, bf16>(s, x, xb, nx);
      ref::cast<float, bf16>(s, dy, dyb, ny);
      ref::bn_stats<bf16>(s, xb, M, C, mean, var, ws);
      ref::bn_finalize(s, mean, var, C, M, 1e-5f, 0.1f, rstd, nullptr, nullptr);
      bf16* gb = t.get<bf16>(nx);   // gradient of the BN output = pool backward x ReLU mask
      bool ok = fast::Fast<bf16>::pool_fwd(xb, mean, rstd, gamma, beta, yb, idx, N, H, W, C, OH, OW, s) &&
                fast::Fast<bf16>::pool_bwd(dyb, idx, xb, mean, rstd, gamma, beta, gb, N, H, W, C, OH, OW, s) &&
                fast::Fast<bf16>::bn_bwd(gb, nullptr, xb, mean, rstd, gamma, dgamma, dbeta, dxb, M, C, sums, s);
      if (!ok) {
        bf16 *a = t.get<bf16>(nx), *g = t.get<bf16>(nx);
        ref::bn_apply<bf16>(s, xb, mean, rstd, gamma, beta, nullptr, true, a, M, C);
        ref::maxpool_fwd<bf16>(s, a, yb, idx, N, H, W, C, OH, OW);
        ref::maxpool_bwd<bf16>(s, dyb, idx, g, N, H, W, C, OH, OW);
        ref::relu_mask_inplace<bf16>(s, g, a, nx);
        ref::bn_bwd<bf16>(s, g, xb, mean, rstd, gamma, dgamma, dbeta, dxb, M, C, ws);
      }
      ref::cast<bf16, float>(s, yb, y, ny);
      ref::cast<bf16, float>(s, dxb, dx, nx);
    }
    sync_stream(s);
  });
}
int lbc_op_spatial_softmax(const float* logits, float* out_xy, int rows, int H, int W, int precision, void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    LBC_CHECK(rows % 20 == 0, "rows must be a multiple of 20 (4 heads x 5 steps)");
    Tmp t;
    float *rmax = t.get<float>(rows), *rsum = t.get<float>(rows);
    if (!(precision == PREC_BF16 && fast::head_softmax_f32(logits, rmax, rsum, out_xy, rows / 20, H, W, s)))
      ref::head_softmax(s, logits, rmax, rsum, out_xy, rows / 20, H, W);
    sync_stream(s);
  });
}
// The four waypoint heads (image.py:54-60,82-84) over h [N][H*W][64] (post-ReLU decoder output), train-mode BN.
// gamma/beta [4][64], w [4][5][64], bias [4][5]; running_mean / running_var [4][64] updated in place (may be null).
// Forward: logits_out [N][20][H*W] (may be null), preds_out [N][4][5][2].  Backward when d_pred or d_preds is given
// (onehot [N][4] needed with d_pred): dgamma/dbeta/dw/dbias in the parameter layouts, dh [N][H*W][64];
// *dh_masked = 1 when dh already carries the (h > 0) mask of the decoder's last ReLU (fused fast path).
int lbc_op_head(const float* h, const float* gamma, const float* beta, const float* w, const float* bias, int N, int H, int W,
                float* running_mean, float* running_var, float* logits_out, float* preds_out, const float* onehot,
                const float* d_pred, const float* d_preds, float* dgamma, float* dbeta, float* dw, float* dbias, float* dh,
                int* dh_masked, int precision, void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    Tmp t;
    const int HW = H * W;
    const int64_t M = (int64_t)N * HW;
    HeadCtx hc;
    hc.H = H;
    hc.W = W;
    hc.logits = t.get<float>(M * 20);
    hc.dlogits = t.get<float>(M * 20);
    hc.rowmax = t.get<float>(N * 20);
    hc.rowsum = t.get<float>(N * 20);
    hc.preds = t.get<float>(N * 40);
    hc.S = t.get<double>(20 * 65);
    hc.fold = t.get<float>(1300 + 128 + 28);
    hc.bn_sums = t.get<float>(2 * 1024);
    int64_t wd = (1 << 20);
    if ((int64_t)N * 20 * 65 + 4096 > wd) wd = (int64_t)N * 20 * 65 + 4096;
    hc.ws_d = t.get<double>(wd);
    hc.var0 = t.get<float>(64);
    float *rm = running_mean ? running_mean : t.get<float>(4 * 64), *rv = running_var ? running_var : t.get<float>(4 * 64);
    if (!running_mean) dev_memset(rm, 0, sizeof(float) * 256, s);
    if (!running_var) dev_memset(rv, 0, sizeof(float) * 256, s);
    for (int k = 0; k < 4; ++k) {
      hc.gamma[k] = gamma + k * 64;
      hc.beta[k] = beta + k * 64;
      hc.w[k] = w + k * 320;
      hc.bias[k] = bias + k * 5;
      hc.mean[k] = t.get<float>(64);
      hc.rstd[k] = t.get<float>(64);
      hc.rm[k] = rm + k * 64;
      hc.rv[k] = rv + k * 64;
    }
    const bool bwd = d_pred || d_preds;
    ref::HeadGrads hg;
    if (bwd) {
      LBC_CHECK(dgamma && dbeta && dw && dbias && dh, "lbc_op_head: backward outputs missing");
      LBC_CHECK(!d_pred || onehot, "lbc_op_head: d_pred needs the command one-hot");
      for (int k = 0; k < 4; ++k) {
        hg.dgamma[k] = dgamma + k * 64;
        hg.dbeta[k] = dbeta + k * 64;
        hg.dw[k] = dw + k * 320;
        hg.dbias[k] = dbias + k * 5;
      }
    }
    if (precision == PREC_F32) {
      head_forward<float>(hc, h, N, true, 1e-5f, 0.1f, s);
      if (bwd) head_backward<float>(hc, h, onehot, d_pred, d_preds, hg, dh, N, s);
    } else {
      bf16 *hb = t.get<bf16>(M * 64), *dhb = t.get<bf16>(M * 64);
      ref::cast<float, bf16>(s, h, hb, M * 64);
      head_forward<bf16>(hc, hb, N, true, 1e-5f, 0.1f, s);
      if (bwd) {
        head_backward<bf16>(hc, hb, onehot, d_pred, d_preds, hg, dhb, N, s);
        ref::cast<bf16, float>(s, dhb, dh, M * 64);
      }
    }
    if (dh_masked) *dh_masked = hc.mask_fused ? 1 : 0;
    if (logits_out) dev_copy(logits_out, hc.logits, sizeof(float) * M * 20, s);
    if (preds_out) dev_copy(preds_out, hc.preds, sizeof(float) * N * 40, s);
    sync_stream(s);
  });
}
// Stem 7x7/s2 convolution straight from the frames (resnet.py:102,148; normalisation common.py:101-109 fused when
// `normalize`): img fp32 [N][C][H][W] or (img_u8 != null) uint8 frames in layout 0 = [N][C][H][W] / 1 = [N][H][W][C] with
// torchvision ToTensor's /255 applied on the device.  w_ref [64][C][7][7].  Outputs (each may be null): x4_out = the
// zero-padded NHWC4 operand [N][H+6][W+8][4] (C <= 4, bf16 path only), y [N][OH][OW][64], stats_out [128] = per-channel
// sum | sum of squares of the stored y (bf16 path), and with dy [N][OH][OW][64]: dw [64][C][7][7].
int lbc_op_stem(const float* img, const uint8_t* img_u8, int layout, const float* w_ref, int normalize, int N, int C, int H,
                int W, float* x4_out, float* y, float* stats_out, const float* dy, float* dw, int precision, void* stream) {
  return guarded([&] {
    require_device();
    lbc_stream_t s = S(stream);
    Tmp t;
    LBC_CHECK(img || img_u8, "lbc_op_stem: no input");
    ConvL c = make_conv(H, W, C, 64, 7, 2, 3);
    const int OH = c.OH, OW = c.OW;
    const int64_t nimg = (int64_t)N * C * H * W, ny = (int64_t)N * OH * OW * 64;
    const float* imgf = img;
    if (!img) {   // the float frames the two-step path would see
      float* f = t.get<float>(nimg);
      ref::u8_to_f32_nchw(s, img_u8, f, N, C, H, W, layout);
      imgf = f;
    }
    if (precision == PREC_F32) {
      LBC_CHECK(!x4_out && !stats_out, "lbc_op_stem: x4_out / stats_out exist on the bf16 path only");
      float *x0 = t.get<float>((int64_t)N * H * W * C), *wp = t.get<float>((int64_t)64 * 49 * C);
      ref::input_to_nhwc<float>(s, imgf, x0, N, C, H, W, C, normalize != 0, 0.485f, 0.456f, 0.406f, 0.229f, 0.224f, 0.225f);
      ref::pack_weight<float>(s, w_ref, wp, 64, C, 7);
      if (y) ref::conv_fwd<float>(s, x0, wp, nullptr, false, y, N, H, W, C, 64, 7, 2, 3, OH, OW);
      if (dy && dw) {
        int64_t wsn = 4 << 20;
        float* ws = t.get<float>(wsn);
        ref::conv_wgrad<float>(s, x0, dy, dw, N, H, W, C, 64, 7, 2, 3, OH, OW, ws, wsn);
      }
    } else if (precision == PREC_F32TC) {
      LBC_CHECK(!x4_out && !stats_out, "lbc_op_stem: x4_out / stats_out exist on the bf16 path only");
      const int Kp = ((49 * C + 63) / 64) * 64;
      const int64_t npix = (int64_t)N * OH * OW;
      float *x0 = t.get<float>((int64_t)N * H * W * C), *wp = t.get<float>((int64_t)64 * Kp), *wp16 = t.get<float>((int64_t)64 * Kp);
      ref::input_to_nhwc<float>(s, imgf, x0, N, C, H, W, C, normalize != 0, 0.485f, 0.456f, 0.406f, 0.229f, 0.224f, 0.225f);
      ConvL g = make_conv(OH, OW, Kp, 64, 1, 1, 0);
      ref::pack_stem_weight(s, w_ref, wp, C, Kp);
      LBC_CHECK(fast::tc_split(wp, wp16, 64, Kp, fast::TC_F16, fast::kTcWeightScale, s), "tc_split unavailable");
      g.wp16 = wp16;
      fast::TcWork tw = make_tcwork(t, npix * Kp * 4, npix * 64 * 4);
      if (y) {
        LBC_CHECK(fast::tc_stem_im2col(x0, tw.a16, N, C, H, W, OH, OW, Kp, fast::TC_F16, s), "tc_stem_im2col unavailable");
        LBC_CHECK(fast::conv_fwd_tc(g, nullptr, tw.a16, y, N, nullptr, false, fast::TC_F16, tw, s), "stem GEMM (tc) declined the shape");
      }
      if (dy && dw) {
        int64_t wsn = 4 << 20;
        float *ws = t.get<float>(wsn), *dwc = t.get<float>((int64_t)64 * Kp);
        LBC_CHECK(fast::tc_stem_im2col(x0, tw.a16, N, C, H, W, OH, OW, Kp, fast::TC_BF16, s), "tc_stem_im2col unavailable");
        LBC_CHECK(fast::conv_wgrad_tc(g, nullptr, tw.a16, dy, dwc, N, fast::TC_BF16, fast::TC_BF16, tw, s),
                  "stem weight gradient (tc) declined the shape");
        LBC_CHECK(fast::stem_unpack_wgrad(dwc, dw, C, Kp, s), "stem_unpack_wgrad failed");
      }
    } else if (fast::stem_ch(C) && !(C > 4 && normalize)) {
      const int CH = fast::stem_ch(C, W, normalize != 0), XC = fast::stem_x_ch(CH);
      bf16 *x4 = t.get<bf16>((int64_t)N * (H + 6) * (W + 8) * XC), *w224 = t.get<bf16>(fast::stem_w_elems(CH)), *yb = t.get<bf16>(ny);
      bool ok = img_u8 && !img ? fast::stem_pad4_u8_bf16(img_u8, layout, x4, N, C, H, W, normalize != 0, s)
                               : fast::stem_pad4_bf16(imgf, x4, N, C, H, W, normalize != 0, s);
      LBC_CHECK(ok, "lbc_op_stem: stem_pad4 unavailable (fast kernels disabled or host-emulation build)");
      if (x4_out) ref::cast<bf16, float>(s, x4, x4_out, (int64_t)N * (H + 6) * (W + 8) * XC);
      LBC_CHECK(fast::stem_pack_w224_bf16(w_ref, w224, C, s, CH), "stem_pack_w224 failed");
      if (y) {
        int rows = 0;
        float* part = stats_out ? fast::stat_partial_buffer() : nullptr;
        LBC_CHECK(fast::stem_conv_bf16(x4, w224, yb, N, H, W, OH, OW, nullptr, part, &rows, s, CH), "stem_conv_bf16 declined the shape");
        if (stats_out) LBC_CHECK(part && fast::col_finalize_bf16(part, rows, 128, stats_out, s), "col_finalize failed");
        ref::cast<bf16, float>(s, yb, y, ny);
      }
      if (dy && dw) {
        bf16* dyb = t.get<bf16>(ny);
        ref::cast<float, bf16>(s, dy, dyb, ny);
        LBC_CHECK(fast::stem_wgrad_bf16(x4, dyb, dw, N, C, H, W, OH, OW, s, CH), "stem_wgrad_bf16 declined the shape");
      }
    } else {   // C > 8: explicit bf16 column tensor + the generic GEMM kernels as a 1x1 convolution
      LBC_CHECK(!x4_out && !stats_out, "lbc_op_stem: x4_out / stats_out need C <= 8");
      const int Kp = ((49 * C + 63) / 64) * 64;
      bf16 *col = t.get<bf16>((int64_t)N * OH * OW * Kp), *wp = t.get<bf16>((int64_t)64 * Kp), *yb = t.get<bf16>(ny);
      ConvL g = make_conv(OH, OW, Kp, 64, 1, 1, 0);
      g.wp = wp;
      LBC_CHECK(fast::stem_im2col_bf16(imgf, col, N, C, H, W, OH, OW, Kp, normalize != 0, s), "stem_im2col unavailable");
      LBC_CHECK(fast::stem_pack_weight_bf16(w_ref, wp, C, Kp, s), "stem_pack_weight failed");
      if (y) {
        LBC_CHECK(fast::conv_fwd<bf16>(g, col, yb, N, s), "stem GEMM declined the shape");
        ref::cast<bf16, float>(s, yb, y, ny);
      }
      if (dy && dw) {
        bf16* dyb = t.get<bf16>(ny);
        int64_t wsn = 4 << 20;
        float *ws = t.get<float>(wsn), *dwc = t.get<float>((int64_t)64 * Kp);
        ref::cast<float, bf16>(s, dy, dyb, ny);
        LBC_CHECK(fast::conv_wgrad<bf16>(g, col, dyb, dwc, N, s), "stem weight-gradient GEMM declined the shape");
        LBC_CHECK(fast::stem_unpack_wgrad(dwc, dw, C, Kp, s), "stem_unpack_wgrad failed");
      }
    }
    sync_stream(s);
  });
}

}  // extern "C"
