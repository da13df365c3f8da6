// lbc_fast.h -- hooks from the graph executor into the sm_100a fast kernels (tcgen05 implicit-GEMM
// convolutions, fused BN / head kernels).  Each hook returns false when it does not handle the
// call (shape / dtype not covered, or host-emulation build) and the executor then runs the
// correctness-first kernel of lbc_ref_ops.h instead.
#pragma once
#include "lbc_common.h"
#include "lbc_net.h"
#include "lbc_ref_ops.h"

namespace lbc {
namespace fast {

// global switch (tests flip it to compare fast kernels against the correctness-first ones)
bool enabled();
void set_enabled(bool on);

// stat_partial != null: the epilogue also writes per-tile column sums / sums of squares of the stored output
// ([*stat_rows][2*Co] floats) so that the BatchNorm statistics pass over the tensor disappears.
bool conv_fwd_bf16(const ConvL& c, const bf16* x, bf16* y, int B, const float* bias_co, lbc_stream_t s,
                   float* stat_partial = nullptr, int* stat_rows = nullptr);
void set_pair_mode(int mode);     // bit 0: CTA-pair (cta_group::2) implicit-GEMM kernels for the >= 128-wide N tiles
int pair_mode();
void set_c64_variant(bool on);   // resident-weight / shared-row variant of the 3x3 64->64 convolution (tests toggle it)
float* stat_partial_buffer();      // shared scratch of the statistics partials (single stream); null if the allocation failed
int64_t stat_partial_capacity();   // its size in floats
bool col_finalize_bf16(const float* partial, int rows, int C2, float* sums, lbc_stream_t s);
// train-mode BatchNorm statistics from partial rows ([rows][2C]: sum | sum of squares; null = the shared partial buffer) in
// one launch: mean / rstd, running buffers, centring shift and the (scale | shift) pair scsh[2C] for bn_apply_bf16
bool bn_finalize_bf16(const float* partial, int rows, int C, int64_t M, const float* gamma, const float* beta, float eps,
                      float momentum, float* running_mean, float* running_var, float* saved_mean, float* saved_rstd,
                      float* negshift, float* scsh, float* sums, lbc_stream_t s);
bool bn_stats_partials_bf16(const bf16* x, int64_t M, int C, int* rows, lbc_stream_t s);

template <class T>
inline bool conv_fwd(const ConvL& c, const T* x, T* y, int B, lbc_stream_t s, const float* bias_co = nullptr,
                     float* stat_partial = nullptr, int* stat_rows = nullptr) {
  (void)c; (void)x; (void)y; (void)B; (void)s; (void)bias_co; (void)stat_partial; (void)stat_rows;
  return false;
}
template <>
inline bool conv_fwd<bf16>(const ConvL& c, const bf16* x, bf16* y, int B, lbc_stream_t s, const float* bias_co,
                           float* stat_partial, int* stat_rows) {
  if (!enabled()) return false;
  return conv_fwd_bf16(c, x, y, B, bias_co, s, stat_partial, stat_rows);
}

bool conv_dgrad_bf16(const ConvL& c, const bf16* dy, bf16* dx, int B, const float* bias_ci, bool relu, lbc_stream_t s);

template <class T>
inline bool conv_dgrad(const ConvL& c, const T* dy, T* dx, int B, const float* bias_ci, bool relu, lbc_stream_t s) {
  (void)c; (void)dy; (void)dx; (void)B; (void)bias_ci; (void)relu; (void)s;
  return false;
}
template <>
inline bool conv_dgrad<bf16>(const ConvL& c, const bf16* dy, bf16* dx, int B, const float* bias_ci, bool relu,
                             lbc_stream_t s) {
  if (!enabled()) return false;
  return conv_dgrad_bf16(c, dy, dx, B, bias_ci, relu, s);
}

bool conv_dgrad_ds_bf16(const ConvL& c1, const bf16* dy1, const bf16* dy_ds, bf16* dx, int B, lbc_stream_t s);
template <class T>
inline bool conv_dgrad_ds(const ConvL&, const T*, const T*, T*, int, lbc_stream_t) {
  return false;
}
template <>
inline bool conv_dgrad_ds<bf16>(const ConvL& c1, const bf16* dy1, const bf16* dy_ds, bf16* dx, int B, lbc_stream_t s) {
  if (!enabled()) return false;
  return conv_dgrad_ds_bf16(c1, dy1, dy_ds, dx, B, s);
}
bool conv_wgrad_bf16(const ConvL& c, const bf16* x, const bf16* dy, float* dw_ref, int B, lbc_stream_t s);
template <class T>
inline bool conv_wgrad(const ConvL&, const T*, const T*, float*, int, lbc_stream_t) {
  return false;
}
template <>
inline bool conv_wgrad<bf16>(const ConvL& c, const bf16* x, const bf16* dy, float* dw_ref, int B, lbc_stream_t s) {
  if (!enabled()) return false;
  return conv_wgrad_bf16(c, x, dy, dw_ref, B, s);
}

// ---- fp32tc: parity-grade tensor-core convolutions over fp32 NHWC tensors (lbc_fast_conv.cu) --------------------
// Every operand is split into two 16-bit planes, x ~ hi + lo, stored [rows][hi C | lo C]; the GEMM K loop accumulates
// hi*hi + hi*lo + lo*hi in the fp32 TMEM accumulator and the epilogue stores fp32.  Formats: TC_F16 (11-bit significands:
// hi + lo carries 22 bits; for the FORWARD pass, whose activations and weights fp16's range covers -- weights are pre-scaled
// by kTcWeightScale, undone in the epilogue) and TC_BF16 (fp32's exponent range, 16 bits: every GEMM of the BACKWARD pass,
// where one operand is a gradient).  Both operands of a GEMM use the same format (a tcgen05.mma restriction).
enum { TC_F16 = 0, TC_BF16 = 1 };
constexpr float kTcWeightScale = 64.0f;
struct TcWork {       // two operand-split scratch buffers owned by the caller
  void* a16 = nullptr;
  void* b16 = nullptr;
  int64_t a_bytes = 0, b_bytes = 0;
};
bool tc_split(const float* src, void* dst16, int64_t rows, int C, int fmt, float scale, lbc_stream_t s);
// x [B,H,W,Ci] fp32 -> y [B,OH,OW,Co] fp32 (c.wp16, split in x_fmt); x_fmt: TC_F16 for an activation, TC_BF16 when x is a
// gradient (the decoder's backward-data runs through the conv-role forward).  x16 != null: x is already split.
bool conv_fwd_tc(const ConvL& c, const float* x, const void* x16, float* y, int B, const float* bias_co, bool relu, int x_fmt,
                 const TcWork& w, lbc_stream_t s);
// dy [B,OH,OW,Co] -> dx [B,H,W,Ci] (+bias, ReLU) (c.wpt16, split in dy_fmt); dy_ds != null: + the fused 1x1/s2 downsample
// gradient (c.wcomb16)
bool conv_dgrad_tc(const ConvL& c, const float* dy, const float* dy_ds, float* dx, int B, const float* bias_ci, bool relu,
                   int dy_fmt, const TcWork& w, lbc_stream_t s);
// dw_ref [Co][Ci][K][K] = sum_pixels dy x;  x16 != null: x already split (stem column tensor, in w.a16)
bool conv_wgrad_tc(const ConvL& c, const float* x, const void* x16, const float* dy, float* dw_ref, int B, int x_fmt, int dy_fmt,
                   const TcWork& w, lbc_stream_t s);
// stem: x0 [B,H,W,C] fp32 NHWC -> split column tensor [B*OH*OW][hi Kp | lo Kp] (k = (kh*7+kw)*C + c, zero padded)
bool tc_stem_im2col(const float* x0, void* col16, int B, int C, int H, int W, int OH, int OW, int Kp, int fmt, lbc_stream_t s);

// ---- HBM-bound bf16 kernels (lbc_fast_elem.cu) -------------------------------------------------------------
bool bn_stats_bf16(const bf16* x, int64_t M, int C, float* sums, lbc_stream_t s);
bool bn_apply_bf16(const bf16* x, const float* scsh, int64_t M, int C, const float* gamma, const float* beta, float eps,
                   float momentum, float* running_mean, float* running_var, float* saved_mean, float* saved_rstd,
                   const bf16* residual, bool relu, bool train, bf16* y, float* negshift, lbc_stream_t s,
                   uint8_t* maskbits = nullptr);   // maskbits [M][C/8]: also emit (y > 0) as one bit per element
// beta_own: mask_act is relu(this BN's output) -> recomputed from x.  mask_bits: the (act > 0) mask as the bits bn_apply_bf16
// wrote (16x fewer bytes than reading the activation; mask_act is then only a flag)
bool bn_bwd_bf16(const bf16* dy, const bf16* mask_act, const bf16* x, const float* mean, const float* rstd,
                 const float* gamma, float* dgamma, float* dbeta, bf16* dx, int64_t M, int C, float* sums, lbc_stream_t s,
                 const float* beta_own = nullptr, const uint8_t* mask_bits = nullptr, int pre_rows = 0);
bool resid_bn_reduce_bf16(bf16* dst, const bf16* src, const uint8_t* src_bits, const bf16* x, const float* mean, const float* rstd,
                          const uint8_t* mask_bits, int64_t M, int C, int* rows, lbc_stream_t s);
bool ew_bf16(bf16* dst, const bf16* src, const bf16* act, int64_t n, int mode, lbc_stream_t s, const uint8_t* mask_bits = nullptr);
// dst [M][Cd] = src [M][0:min(Cs, Cd)], channels beyond Cs = fill[m / rows_per_fill] (speed fusion forward / its slice backward)
bool copy_channels_bf16(bf16* dst, const bf16* src, int64_t M, int Cd, int Cs, const float* fill, int rows_per_fill, lbc_stream_t s);
template <class T>
inline bool copy_channels(T*, const T*, int64_t, int, int, const float*, int, lbc_stream_t) {
  return false;
}
template <>
inline bool copy_channels<bf16>(bf16* dst, const bf16* src, int64_t M, int Cd, int Cs, const float* fill, int rows_per_fill,
                                lbc_stream_t s) {
  if (!enabled()) return false;
  return copy_channels_bf16(dst, src, M, Cd, Cs, fill, rows_per_fill, s);
}
bool bn_relu_maxpool_bf16(const bf16* x, const float* mean, const float* rstd, const float* gamma, const float* beta,
                          bf16* y, uint8_t* idx, int N, int H, int W, int C, int OH, int OW, lbc_stream_t s);
bool maxpool_relu_bwd_bf16(const bf16* dy, const uint8_t* idx, const bf16* x, const float* mean, const float* rstd,
                           const float* gamma, const float* beta, bf16* dx, int N, int H, int W, int C, int OH, int OW,
                           lbc_stream_t s);

// generic-T front ends: only T = bf16 has fast kernels
template <class T> struct Fast {
  static bool bn_fwd(const T*, int64_t, int, const float*, const float*, float, float, float*, float*, float*, float*,
                     const T*, bool, bool, T*, float*, float*, lbc_stream_t, int = 0, uint8_t* = nullptr) { return false; }
  static bool bn_bwd(const T*, const T*, const T*, const float*, const float*, const float*, float*, float*, T*, int64_t, int,
                     float*, lbc_stream_t, const float* = nullptr, const uint8_t* = nullptr, int = 0) { return false; }
  static bool resid_bn_reduce(T*, const T*, const uint8_t*, const T*, const float*, const float*, const uint8_t*, int64_t, int,
                              int*, lbc_stream_t) { return false; }
  static bool ew(T*, const T*, const T*, int64_t, int, lbc_stream_t, const uint8_t* = nullptr) { return false; }
  static bool colsum(const T*, int64_t, int, float*, float*, lbc_stream_t) { return false; }
  static bool pool_fwd(const T*, const float*, const float*, const float*, const float*, T*, uint8_t*, int, int, int, int, int,
                       int, lbc_stream_t) { return false; }
  static bool pool_bwd(const T*, const uint8_t*, const T*, const float*, const float*, const float*, const float*, T*, int, int,
                       int, int, int, int, lbc_stream_t) { return false; }
};
template <> struct Fast<bf16> {
  // train: (statistics pass) + finalize + apply; eval: apply with the running statistics.  sums: >= 2C floats scratch
  // (receives the scale | shift pair of the finalize kernel)
  static bool bn_fwd(const bf16* x, int64_t M, int C, const float* gamma, const float* beta, float eps, float momentum,
                     float* rm, float* rv, float* saved_mean, float* saved_rstd, const bf16* res, bool relu, bool train,
                     bf16* y, float* sums, float* negshift, lbc_stream_t s, int conv_stat_rows = 0, uint8_t* maskbits = nullptr) {
    if (!enabled()) return false;
    if (train) {
      // partial rows: written by the producing conv's epilogue (conv_stat_rows > 0), else by a statistics pass over x;
      // then ONE launch: column sums + mean / rstd + running buffers + centring shift + (scale | shift)
      int rows = conv_stat_rows;
      if (rows <= 0 && !bn_stats_partials_bf16(x, M, C, &rows, s)) return false;
      if (!bn_finalize_bf16(nullptr, rows, C, M, gamma, beta, eps, momentum, rm, rv, saved_mean, saved_rstd, negshift, sums,
                            nullptr, s))
        return false;
    }
    return bn_apply_bf16(x, sums, M, C, gamma, beta, eps, momentum, rm, rv, saved_mean, saved_rstd, res, relu, train, y,
                         negshift, s, maskbits);
  }
  static bool bn_bwd(const bf16* dy, const bf16* mask, const bf16* x, const float* mean, const float* rstd, const float* gamma,
                     float* dgamma, float* dbeta, bf16* dx, int64_t M, int C, float* sums, lbc_stream_t s,
                     const float* beta_own = nullptr, const uint8_t* mask_bits = nullptr, int pre_rows = 0) {
    if (!enabled()) return false;
    return bn_bwd_bf16(dy, mask, x, mean, rstd, gamma, dgamma, dbeta, dx, M, C, sums, s, beta_own, mask_bits, pre_rows);
  }
  static bool resid_bn_reduce(bf16* dst, const bf16* src, const uint8_t* src_bits, const bf16* x, const float* mean,
                              const float* rstd, const uint8_t* mask_bits, int64_t M, int C, int* rows, lbc_stream_t s) {
    if (!enabled()) return false;
    return resid_bn_reduce_bf16(dst, src, src_bits, x, mean, rstd, mask_bits, M, C, rows, s);
  }
  static bool ew(bf16* dst, const bf16* src, const bf16* act, int64_t n, int mode, lbc_stream_t s, const uint8_t* mask_bits = nullptr) {
    if (!enabled()) return false;
    return ew_bf16(dst, src, act, n, mode, s, mask_bits);
  }
  // column sums (deconv bias gradient) = first half of the BN statistics kernel's output
  static bool colsum(const bf16* x, int64_t M, int C, float* out_via_sums, float* sums, lbc_stream_t s) {
    if (!enabled()) return false;
    if (!bn_stats_bf16(x, M, C, sums, s)) return false;
    dev_copy(out_via_sums, sums, sizeof(float) * C, s);
    return true;
  }
  static bool pool_fwd(const bf16* x, const float* mean, const float* rstd, const float* gamma, const float* beta, bf16* y,
                       uint8_t* idx, int N, int H, int W, int C, int OH, int OW, lbc_stream_t s) {
    if (!enabled()) return false;
    return bn_relu_maxpool_bf16(x, mean, rstd, gamma, beta, y, idx, N, H, W, C, OH, OW, s);
  }
  static bool pool_bwd(const bf16* dy, const uint8_t* idx, const bf16* x, const float* mean, const float* rstd,
                       const float* gamma, const float* beta, bf16* dx, int N, int H, int W, int C, int OH, int OW,
                       lbc_stream_t s) {
    if (!enabled()) return false;
    return maxpool_relu_bwd_bf16(dy, idx, x, mean, rstd, gamma, beta, dx, N, H, W, C, OH, OW, s);
  }
};

// ---- fused waypoint heads (lbc_fast_head.cu); fold: >=1300 floats, coef: >=128 floats, S: [20][65] doubles
bool head_forward_bf16(const bf16* h, ref::HeadParams hp, float* fold, float* logits, float* rowmax, float* rowsum,
                       float* preds, int N, int H, int W, lbc_stream_t s);
bool head_softmax_f32(const float* logits, float* rowmax, float* rowsum, float* preds, int N, int H, int W, lbc_stream_t s);
bool head_dlogits_f32(const float* logits, const float* rowmax, const float* rowsum, const float* preds, const float* onehot,
                      const float* d_pred, const float* d_preds, float* dlogits, int N, int H, int W, lbc_stream_t s);
bool head_backward_s_bf16(const float* dlogits, const bf16* h, const float* mean, const float* rstd, double* S, int N, int HW,
                          lbc_stream_t s);
bool head_backward_dh_bf16(const float* dlogits, const bf16* h, ref::HeadParams hp, ref::HeadGrads hg, const float* fold,
                           float* coef, bf16* dh, int N, int HW, lbc_stream_t s);

// ---- stem (7x7/s2, C_in = 3 or 7): explicit im2col (fused NCHW fp32 -> bf16 + RGB normalisation) feeding the
// same tcgen05 GEMM kernels as a 1x1 convolution over the [B,OH,OW,Kp] column tensor (Kp = 49*C padded to 64).
bool stem_im2col_bf16(const float* img, bf16* col, int B, int C, int H, int W, int OH, int OW, int Kp, bool normalize,
                      lbc_stream_t s);
bool stem_pack_weight_bf16(const float* w_ref, bf16* wp, int C, int Kp, lbc_stream_t s);      // [64][C][7][7] -> [64][Kp]
bool stem_unpack_wgrad(const float* dw_col, float* dw_ref, int C, int Kp, lbc_stream_t s);    // [64][Kp] -> [64][C][7][7]

// ---- stem without a column tensor: zero-padded NHWC bf16 image [B][H+6][W+8][CH] + overlapping-window TMA (lbc_fast_conv.cu).
// Layout code CH = stem_ch(C_in, W, normalize):
//   4  C_in <= 4 (camera): [B][H+6][W+8][4], one kernel row of one output pixel = 8 px x 4 ch = 64 contiguous bytes, 7 rows
//   8  C_in <= 8 (the teacher's 7-channel bird's-eye view): [B][H+6][W+8][8], 128-byte window rows, 7 rows
//   16 C_in <= 4, space-to-depth: [B][(H+6)/2][(W+8)/2][2 row parity][2 column parity][4] -- the SAME padded pixels with every
//      2x2 block contiguous, so the 7x7/s2 convolution is a 4x4/s1 one over 16 channels: 4 window rows of 4 x 16 = 64
//      elements = 128 bytes per output pixel instead of 7 rows of 64 bytes (the kernels are bound by TMA row requests)
bool stem_s2d();   // LBC_STEM_S2D (default on)
inline int stem_ch(int C, int W = 0, bool normalize = false) {
  if (C <= 4) return (stem_s2d() && W > 0 && W % 4 == 0 && (C == 3 || !normalize)) ? 16 : 4;
  return C <= 8 ? 8 : 0;
}
inline int stem_x_ch(int CH) { return CH == 16 ? 4 : CH; }                            // channels of the padded image
inline int stem_w_elems(int CH) { return CH == 16 ? 64 * 4 * 64 : 64 * 7 * 8 * CH; }  // packed weights
bool stem_pad4_bf16(const float* img, bf16* x4, int B, int C, int H, int W, bool normalize, lbc_stream_t s);
bool stem_pad4_u8_bf16(const uint8_t* img, int layout, bf16* x4, int B, int C, int H, int W, bool normalize, lbc_stream_t s);
// [64][C][7][7] -> [64][7][8 px][CH ch]  (CH = 16: [64][4 row pairs][4 column pairs][2][2][4])
bool stem_pack_w224_bf16(const float* w_ref, bf16* w224, int C, lbc_stream_t s, int CH = 0);
bool stem_conv_bf16(const bf16* x4, const bf16* w224, bf16* raw, int B, int H, int W, int OH, int OW, const float* bias,
                    float* stat_partial, int* stat_rows, lbc_stream_t s, int CH = 4);
bool stem_wgrad_bf16(const bf16* x4, const bf16* dy, float* dw_ref, int B, int C, int H, int W, int OH, int OW, lbc_stream_t s,
                     int CH = 4);

}  // namespace fast
}  // namespace lbc
