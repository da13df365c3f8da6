// lbc_fast_elem.cu -- HBM-bound kernels of the bf16 path: train-mode BatchNorm (statistics, apply with fused
// residual / ReLU, backward with the ReLU mask fused), MaxPool, masked adds.  NHWC bf16, one thread owns 8
// consecutive channels (one 16-byte vector) of a fixed channel group and strides over rows, so per-channel
// parameters live in registers and every global access is a coalesced 128-bit transaction; several independent
// loads are kept in flight per thread.  Reductions: per-thread fp32 partials -> shared memory -> one fp32 atomic
// per channel per block.  Reference ops: nn.BatchNorm2d in train mode + nn.ReLU(inplace) + residual add
// (resnet.py:31-53, image.py:38-46) and their autograd backward (SURVEY.md 9.1 closed forms).
#include "lbc_fast.h"

#ifndef LBC_HOST_EMU
#include <cuda_bf16.h>
#endif

namespace lbc {
namespace fast {

#ifndef LBC_HOST_EMU

__device__ __forceinline__ void unpack8(const uint4& v, float* f) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  uint4 v;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return v;
}
// bit j = (bf16 element j of v > 0)
__device__ __forceinline__ uint8_t positive_bits(const uint4& v) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  uint32_t b = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t lo = w[i] & 0xffffu, hi = w[i] >> 16;
    b |= (uint32_t)((lo & 0x7fffu) != 0 && !(lo & 0x8000u)) << (2 * i);
    b |= (uint32_t)((hi & 0x7fffu) != 0 && !(hi & 0x8000u)) << (2 * i + 1);
  }
  return (uint8_t)b;
}
__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

static int sm_count2() {
  static int n = [] {
    int dev = 0, v = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v > 0 ? v : 148;
  }();
  return n;
}
struct RowGeom {
  int tpr, rpi, threads, grid;
};
static RowGeom row_geom(int64_t M, int C, int blocks_per_sm) {
  RowGeom g;
  g.tpr = C / 8;
  g.rpi = 256 / g.tpr;
  if (g.rpi < 1) g.rpi = 1;
  g.threads = g.rpi * g.tpr;
  int64_t need = (M + g.rpi - 1) / g.rpi;
  int64_t cap = (int64_t)sm_count2() * blocks_per_sm;
  g.grid = (int)(need < cap ? need : cap);
  if (g.grid < 1) g.grid = 1;
  return g;
}

// ------------------------------------------------------------------------------------------- BN statistics
// partial[blockIdx][0..C) = sum_rows x ; partial[blockIdx][C..2C) = sum_rows x^2 over this block's rows.
// No atomics: same-address fp32 atomics from ~1000 blocks serialise in L2 (~95 us per launch measured); the
// partials are reduced by col_finalize kernels -> deterministic results.
__global__ void __launch_bounds__(256, 6) bn_stats_kernel(const uint4* __restrict__ x, int64_t M, int tpr, int rpi, float* partial,
                                                       int C) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ float red[];  // [threads][16]
  const int t = threadIdx.x;
  const int cg = t % tpr, r = t / tpr;
  float s[8], q[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
  const int64_t stride = (int64_t)gridDim.x * rpi;
  int64_t row = (int64_t)blockIdx.x * rpi + r;
  for (; row + 3 * stride < M; row += 4 * stride) {
    uint4 v0 = ldg_stream(x + row * tpr + cg);
    uint4 v1 = ldg_stream(x + (row + stride) * tpr + cg);
    uint4 v2 = ldg_stream(x + (row + 2 * stride) * tpr + cg);
    uint4 v3 = ldg_stream(x + (row + 3 * stride) * tpr + cg);
    float f[8];
    unpack8(v0, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] += f[j]; q[j] += f[j] * f[j]; }
    unpack8(v1, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] += f[j]; q[j] += f[j] * f[j]; }
    unpack8(v2, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] += f[j]; q[j] += f[j] * f[j]; }
    unpack8(v3, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] += f[j]; q[j] += f[j] * f[j]; }
  }
  for (; row < M; row += stride) {
    float f[8];
    unpack8(ldg_stream(x + row * tpr + cg), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] += f[j]; q[j] += f[j] * f[j]; }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    red[t * 16 + j] = s[j];
    red[t * 16 + 8 + j] = q[j];
  }
  __syncthreads();
  if (t < tpr) {
    for (int rr = 1; rr < rpi; ++rr) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s[j] += red[(rr * tpr + t) * 16 + j];
        q[j] += red[(rr * tpr + t) * 16 + 8 + j];
      }
    }
    float* dst = partial + (int64_t)blockIdx.x * 2 * C;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      dst[t * 8 + j] = s[j];
      dst[C + t * 8 + j] = q[j];
    }
  }
}
// out[blockIdx.y][col] = sum_p partial[p][col] for col < 2C.  32 columns x 32 partial-lanes per block (1024 threads); when
// there are many partial rows (conv-epilogue statistics: one row per 128-pixel tile) the rows are split over blockIdx.y
// into (<= 32) rows of block sums that sum_slices_kernel then adds in a fixed order (fp32 atomics would add them in the
// order the blocks finish, and the statistics would change in the last bits from run to run).
__global__ void __launch_bounds__(1024) col_finalize_kernel(const float* __restrict__ partial, int P, int C2, float* out,
                                                            int rows_per_block) {
  pdl_wait();
  pdl_trigger();
  const int col = blockIdx.x * 32 + (threadIdx.x & 31);
  const int pl = threadIdx.x >> 5;
  __shared__ float red[32][33];
  const int p0 = blockIdx.y * rows_per_block;
  int p1 = p0 + rows_per_block;
  if (p1 > P) p1 = P;
  float a = 0.f;
  if (col < C2)
    for (int p = p0 + pl; p < p1; p += 32) a += partial[(int64_t)p * C2 + col];
  red[pl][threadIdx.x & 31] = a;
  __syncthreads();
  if (pl == 0 && col < C2) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) t += red[i][threadIdx.x & 31];
    out[(int64_t)blockIdx.y * C2 + col] = t;
  }
}
constexpr int64_t kPartialFloats = (int64_t)4096 * 2 * 2560;
static float* partial_buffer() {
  static float* p = [] {
    void* q = nullptr;
    if (cudaMalloc(&q, sizeof(float) * (size_t)kPartialFloats) != cudaSuccess) {
      cudaGetLastError();
      q = nullptr;   // callers treat a null scratch as "fast path unavailable" and report it
    }
    return (float*)q;
  }();
  return p;
}
int64_t stat_partial_capacity() { return kPartialFloats; }
static float* block_sums_buffer() {   // [32][2C] rows of col_finalize block sums (C2 <= 2 x 2560, as the partial rows)
  static float* p = [] {
    void* q = nullptr;
    if (cudaMalloc(&q, sizeof(float) * 32 * 2 * 2560) != cudaSuccess) {
      cudaGetLastError();
      q = nullptr;
    }
    return (float*)q;
  }();
  return p;
}
static void col_finalize(const float* partial, int P, int C2, float* sums, lbc_stream_t s) {
  int rb = P / 512;          // >= 512 rows per block (16 per thread) before splitting
  if (rb > 32) rb = 32;
  if (rb < 1) rb = 1;
  const int rows_per_block = (P + rb - 1) / rb;
  rb = (P + rows_per_block - 1) / rows_per_block;
  float* out = sums;
  if (rb > 1) {
    out = block_sums_buffer();
    LBC_CHECK(out != nullptr && C2 <= 2 * 2560, "col_finalize: no block-sum scratch for this shape");
  }
  { auto k_ = col_finalize_kernel; LBC_LAUNCH(k_, dim3(dim3((C2 + 31) / 32, rb)), dim3(1024), 0, s, partial, P, C2, out, rows_per_block); }
  if (rb > 1) {
    LBC_LAUNCHED("col_finalize_kernel");
    auto k_ = sum_slices_kernel<float>;
    LBC_LAUNCH(k_, dim3((C2 + 255) / 256), dim3(256), 0, s, (const float*)out, sums, (int64_t)C2, rb);
    LBC_LAUNCHED("sum_slices_kernel");
    return;
  }
  LBC_LAUNCHED("col_finalize_kernel");
}

// Train-mode BatchNorm statistics in ONE small launch: column sums of the partial rows (sum | sum of squares per channel),
// then, in the same threads, everything that depends on them -- batch mean / rstd (double), the running-buffer update
// (momentum, unbiased variance), the centring-shift update, and the affine pair (scale, shift) the apply kernel needs.
// Round 1 left the finalisation to the PROLOGUE of bn_apply_kernel: every one of its 303 K threads redid the double-
// precision mean / variance / rsqrt for its eight channels, a ~13 us floor per launch that dominated the layer-3/4
// tensors (20 us per launch for 31 MB).  One block per 32 channels, 1024 threads = 32 channels x 32 row lanes.
struct BnFinalizeArgs {
  const float* partial;   // [P][2C]
  int P, C;
  double inv_m, unbias;   // 1 / M and M / (M - 1)
  const float* gamma;
  const float* beta;
  float eps, momentum;
  float* running_mean;
  float* running_var;
  float* saved_mean;
  float* saved_rstd;
  float* negshift;        // may be null
  float* scsh;            // out: [2C] = scale | shift
  float* sums;            // out (optional): [2C] raw column sums
};
__global__ void __launch_bounds__(1024) bn_finalize_kernel(const BnFinalizeArgs a) {
  pdl_wait();
  pdl_trigger();
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int pl = threadIdx.x >> 5;
  __shared__ float red0[32][33], red1[32][33];
  float s0 = 0.f, s1 = 0.f;
  // per-channel inputs of the finalisation, loaded together with the partial rows: behind the stores below the compiler
  // cannot hoist them (possible aliasing), and five dependent L2 round trips cost 2 us per launch (bn_fwd 1.74 -> 1.64 ms)
  float in_gamma = 0.f, in_beta = 0.f, in_rm = 0.f, in_rv = 0.f, in_ns = 0.f;
  if (pl == 0 && c < a.C) {
    in_gamma = a.gamma[c];
    in_beta = a.beta[c];
    in_rm = a.running_mean[c];
    in_rv = a.running_var[c];
    in_ns = a.negshift ? a.negshift[c] : 0.f;
  }
  if (c < a.C) {
    // up to 16 rows x 2 columns in flight per thread: the loop is pure L2 latency (1920 partial rows after a layer-2 conv)
    const float* p0 = a.partial + c;
    const int64_t rs = (int64_t)2 * a.C;
    for (int p = pl; p < a.P; p += 32 * 16) {
      float v0[16], v1[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const int pr = p + 32 * u;
        const bool ok = pr < a.P;
        v0[u] = ok ? __ldcg(p0 + (int64_t)pr * rs) : 0.f;
        v1[u] = ok ? __ldcg(p0 + (int64_t)pr * rs + a.C) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        s0 += v0[u];
        s1 += v1[u];
      }
    }
  }
  red0[pl][threadIdx.x & 31] = s0;
  red1[pl][threadIdx.x & 31] = s1;
  __syncthreads();
  if (pl == 0 && c < a.C) {
    float t0 = 0.f, t1 = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      t0 += red0[i][threadIdx.x & 31];
      t1 += red1[i][threadIdx.x & 31];
    }
    if (a.sums) {
      a.sums[c] = t0;
      a.sums[a.C + c] = t1;
    }
    // double only where it matters (sum / M and the E[x^2] - mean^2 cancellation), with multiplications by host-computed
    // reciprocals; 1/sqrt = float rsqrt + one Newton step in double (the software double division / square root sequences
    // made this kernel 3 us slower than the plain column sum it replaced)
    const double m = (double)t0 * a.inv_m;
    double var = (double)t1 * a.inv_m - m * m;
    if (var < 0.0) var = 0.0;
    const double v = var + (double)a.eps;
    double r = (double)rsqrtf((float)v);
    r = r * (1.5 - 0.5 * v * r * r);
    const float mean = (float)m;
    const float rstd = (float)r;
    a.saved_mean[c] = mean;
    a.saved_rstd[c] = rstd;
    const float true_mean = a.negshift ? (float)(m - (double)in_ns) : mean;
    if (a.negshift) a.negshift[c] = -true_mean;   // centring estimate for the next forward pass
    a.running_mean[c] = (1.f - a.momentum) * in_rm + a.momentum * true_mean;
    const double unb = var * a.unbias;
    a.running_var[c] = (1.f - a.momentum) * in_rv + a.momentum * (float)unb;
    const float sc = in_gamma * rstd;
    a.scsh[c] = sc;
    a.scsh[a.C + c] = in_beta - mean * sc;
  }
}
// sums (optional) / scsh: [2C] each.  partial = null: the shared partial buffer (conv epilogue / bn_stats rows)
bool bn_finalize_bf16(const float* partial, int rows, int C, int64_t M, const float* gamma, const float* beta, float eps,
                      float momentum, float* running_mean, float* running_var, float* saved_mean, float* saved_rstd,
                      float* negshift, float* scsh, float* sums, lbc_stream_t s) {
  if (!partial) partial = partial_buffer();
  if (!partial || rows <= 0 || (int64_t)rows * 2 * C > kPartialFloats) return false;
  BnFinalizeArgs a;
  a.partial = partial;
  a.P = rows;
  a.C = C;
  a.inv_m = 1.0 / (double)M;
  a.unbias = (double)M / (double)(M > 1 ? M - 1 : 1);
  a.gamma = gamma;
  a.beta = beta;
  a.eps = eps;
  a.momentum = momentum;
  a.running_mean = running_mean;
  a.running_var = running_var;
  a.saved_mean = saved_mean;
  a.saved_rstd = saved_rstd;
  a.negshift = negshift;
  a.scsh = scsh;
  a.sums = sums;
  { auto k_ = bn_finalize_kernel; LBC_LAUNCH(k_, dim3((C + 31) / 32), dim3(1024), 0, s, a); }
  LBC_LAUNCHED("bn_finalize_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}
// bn_stats_kernel without the column pass: leaves *rows partial rows in the shared partial buffer
bool bn_stats_partials_bf16(const bf16* x, int64_t M, int C, int* rows, lbc_stream_t s) {
  if (C % 8 || C > 2560) return false;
  RowGeom g = row_geom(M, C, 6);
  float* part = partial_buffer();
  if (!part) return false;
  { auto k_ = bn_stats_kernel; LBC_LAUNCH(k_, dim3(g.grid), dim3(g.threads), g.threads * 16 * sizeof(float), s, (const uint4*)x, M, g.tpr, g.rpi, part, C); }
  LBC_LAUNCHED("bn_stats_kernel");
  LBC_CUDA(cudaGetLastError());
  *rows = g.grid;
  return true;
}

float* stat_partial_buffer() { return partial_buffer(); }
bool col_finalize_bf16(const float* partial, int rows, int C2, float* sums, lbc_stream_t s) {
  if (!partial || (int64_t)rows * C2 > kPartialFloats) return false;
  col_finalize(partial, rows, C2, sums, s);
  LBC_CUDA(cudaGetLastError());
  return true;
}

bool bn_stats_bf16(const bf16* x, int64_t M, int C, float* sums, lbc_stream_t s) {
  if (C % 8 || C > 2560) return false;
  RowGeom g = row_geom(M, C, 6);
  float* part = partial_buffer();
  if (!part) return false;
  { auto k_ = bn_stats_kernel; LBC_LAUNCH(k_, dim3(g.grid), dim3(g.threads), g.threads * 16 * sizeof(float), s, (const uint4*)x, M, g.tpr, g.rpi, part, C); }
  LBC_LAUNCHED("bn_stats_kernel");
  col_finalize(part, g.grid, 2 * C, sums, s);
  LBC_CUDA(cudaGetLastError());
  return true;
}

// ------------------------------------------------------------------------------------------- BN apply
struct BnApplyArgs {
  const uint4* x;
  const uint4* res;
  uint4* y;
  const float* scsh;   // train: [2C] scale | shift from bn_finalize_kernel
  const float* gamma;
  const float* beta;
  float* running_mean;
  float* running_var;
  float* saved_mean;
  float* saved_rstd;
  float* negshift;     // x holds (conv output + negshift[c]); null = no centring shift
  uint8_t* maskbits;   // optional [M][C/8]: bit j of byte (row, channel group) = (stored output channel 8g+j > 0)
  int64_t M;
  int C, tpr, rpi;
  float eps, momentum;
  int relu, train;
};
__global__ void __launch_bounds__(256, 4) bn_apply_kernel(const BnApplyArgs a) {
  pdl_wait();
  pdl_trigger();
  const int t = threadIdx.x;
  const int cg = t % a.tpr, r = t / a.tpr;
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = cg * 8 + j;
    if (a.train) {   // statistics, running buffers, (scale, shift): bn_finalize_kernel
      sc[j] = a.scsh[c];
      sh[j] = a.scsh[a.C + c];
    } else {
      const float mean = a.running_mean[c] + (a.negshift ? a.negshift[c] : 0.f);
      const float rstd = 1.0f / sqrtf(a.running_var[c] + a.eps);
      if (blockIdx.x == 0 && r == 0) {
        a.saved_mean[c] = mean;
        a.saved_rstd[c] = rstd;
      }
      sc[j] = a.gamma[c] * rstd;
      sh[j] = a.beta[c] - mean * sc[j];
    }
  }
  const int64_t stride = (int64_t)gridDim.x * a.rpi;
  for (int64_t row = (int64_t)blockIdx.x * a.rpi + r; row < a.M; row += 2 * stride) {
    const int64_t i0 = row * a.tpr + cg;
    const int64_t row1 = row + stride;
    const bool has1 = row1 < a.M;
    const int64_t i1 = row1 * a.tpr + cg;
    uint4 v0 = ldg_stream(a.x + i0);
    uint4 v1 = has1 ? ldg_stream(a.x + i1) : v0;
    uint4 r0, r1;
    if (a.res) {
      r0 = ldg_stream(a.res + i0);
      r1 = has1 ? ldg_stream(a.res + i1) : r0;
    }
    float f[8], g[8];
    unpack8(v0, f);
    if (a.res) unpack8(r0, g);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = f[j] * sc[j] + sh[j];
      if (a.res) v += g[j];
      if (a.relu) v = fmaxf(v, 0.f);
      f[j] = v;
    }
    const uint4 o0 = pack8(f);
    a.y[i0] = o0;
    if (a.maskbits) a.maskbits[i0] = positive_bits(o0);
    if (has1) {
      unpack8(v1, f);
      if (a.res) unpack8(r1, g);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float v = f[j] * sc[j] + sh[j];
        if (a.res) v += g[j];
        if (a.relu) v = fmaxf(v, 0.f);
        f[j] = v;
      }
      const uint4 o1 = pack8(f);
      a.y[i1] = o1;
      if (a.maskbits) a.maskbits[i1] = positive_bits(o1);
    }
  }
}

bool bn_apply_bf16(const bf16* x, const float* scsh, int64_t M, int C, const float* gamma, const float* beta, float eps,
                   float momentum, float* running_mean, float* running_var, float* saved_mean, float* saved_rstd,
                   const bf16* residual, bool relu, bool train, bf16* y, float* negshift, lbc_stream_t s, uint8_t* maskbits) {
  if (C % 8 || C > 2560) return false;
  RowGeom g = row_geom(M, C, 8);
  BnApplyArgs a;
  a.negshift = negshift;
  a.maskbits = maskbits;
  a.x = (const uint4*)x;
  a.res = (const uint4*)residual;
  a.y = (uint4*)y;
  a.scsh = scsh;
  a.gamma = gamma;
  a.beta = beta;
  a.running_mean = running_mean;
  a.running_var = running_var;
  a.saved_mean = saved_mean;
  a.saved_rstd = saved_rstd;
  a.M = M;
  a.C = C;
  a.tpr = g.tpr;
  a.rpi = g.rpi;
  a.eps = eps;
  a.momentum = momentum;
  a.relu = relu ? 1 : 0;
  a.train = train ? 1 : 0;
  { auto k_ = bn_apply_kernel; LBC_LAUNCH(k_, dim3(g.grid), dim3(g.threads), 0, s, a); }
  LBC_LAUNCHED("bn_apply_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}

// ------------------------------------------------------------------------------------------- BN backward
// pass 1: sums[0..C) += sum dy_m ; sums[C..2C) += sum dy_m * xhat,  dy_m = dy * (act > 0) when act != null
// (mbits != null: the mask comes as one byte per (row, 8 channels) written by bn_apply_kernel instead of the activation)
// RESID (the residual blocks' d(out) chain): dy is produced HERE, dy = dy + (rbits ? rsrc : 0) -- the masked residual add of
// the block that was just differentiated -- stored back (bf16) and reduced as the upstream gradient of the previous block's
// bn2 in the same pass: the separate ew_kernel launch and the reduce kernel's read of dy disappear (8.25 instead of 10.25
// bytes per element for the pair).
template <bool OWN, bool RESID = false>
__global__ void __launch_bounds__(256, OWN ? 3 : 4) bn_bwd_reduce_kernel(const uint4* dy, const uint4* __restrict__ act,
                                                            const uint4* __restrict__ x, const float* __restrict__ mean,
                                                            const float* __restrict__ rstd, int64_t M, int tpr, int rpi,
                                                            float* partial, int C, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta_own,
                                                            const uint8_t* __restrict__ mbits,
                                                            const uint4* __restrict__ rsrc = nullptr,
                                                            const uint8_t* __restrict__ rbits = nullptr, uint4* dy_out = nullptr) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ float red[];
  const int t = threadIdx.x;
  const int cg = t % tpr, r = t / tpr;
  float mu[8], s0[8], s1[8], sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    mu[j] = mean[cg * 8 + j];
    s0[j] = s1[j] = 0.f;
    // beta_own != null: the mask is the ReLU of THIS BatchNorm's own output, act > 0 <=> x*sc + sh > 0 with the very
    // expressions of bn_apply_kernel -- recomputed from x (already being read) instead of reading the activation
    sc[j] = OWN ? gamma[cg * 8 + j] * rstd[cg * 8 + j] : 0.f;
    sh[j] = OWN ? beta_own[cg * 8 + j] - mu[j] * sc[j] : 0.f;
  }
  const int64_t stride = (int64_t)gridDim.x * rpi;
#pragma unroll(OWN ? 4 : 2)
  for (int64_t row = (int64_t)blockIdx.x * rpi + r; row < M; row += stride) {
    const int64_t i0 = row * tpr + cg;
    uint4 d0 = ldg_stream(dy + i0);
    const uint4 x0 = ldg_stream(x + i0);
    if (RESID) {
      const uint4 r0 = ldg_stream(rsrc + i0);
      const uint32_t rb = __ldg(rbits + i0);
      float fs[8], fr[8];
      unpack8(d0, fs);
      unpack8(r0, fr);
#pragma unroll
      for (int j = 0; j < 8; ++j) fs[j] += ((rb >> j) & 1u) ? fr[j] : 0.f;
      d0 = pack8(fs);                               // the stored (rounded) sum is what every later consumer reads
      dy_out[i0] = d0;
    }
    uint4 a0 = d0;
    uint32_t mb = 0xffu;
    if (!OWN && mbits) mb = __ldg(mbits + i0);
    else if (!OWN && act) a0 = ldg_stream(act + i0);
    float fd[8], fx[8], fa[8];
    unpack8(d0, fd);
    unpack8(x0, fx);
    unpack8(a0, fa);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (OWN) fa[j] = fx[j] * sc[j] + sh[j];
      float g = ((OWN || act) && !(fa[j] > 0.f)) ? 0.f : fd[j];
      if (!OWN && !((mb >> j) & 1u)) g = 0.f;
      s0[j] += g;
      s1[j] += g * (fx[j] - mu[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    s1[j] *= rstd[cg * 8 + j];   // sum g*xhat = rstd * sum g*(x-mu)   (scaled in the register too: row group 0 adds its own
    red[t * 16 + j] = s0[j];     //  s1 below -- round 1 scaled only the shared-memory copy, so the block's first row group
    red[t * 16 + 8 + j] = s1[j]; //  entered dgamma without rstd; found by tests/test_kernels.py::test_bn_backward_kernels_gpu)
  }
  __syncthreads();
  if (t < tpr) {
    for (int rr = 1; rr < rpi; ++rr) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s0[j] += red[(rr * tpr + t) * 16 + j];
        s1[j] += red[(rr * tpr + t) * 16 + 8 + j];
      }
    }
    float* dst = partial + (int64_t)blockIdx.x * 2 * C;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      dst[t * 8 + j] = s0[j];
      dst[C + t * 8 + j] = s1[j];
    }
  }
}
// pass 2: dx = gamma*rstd*(dy_m - dbeta/M - xhat*dgamma/M); block 0 also publishes dgamma / dbeta
template <bool OWN>
__global__ void __launch_bounds__(256, 4) bn_bwd_apply_kernel(const uint4* __restrict__ dy, const uint4* __restrict__ act,
                                                           const uint4* __restrict__ x, const float* __restrict__ mean,
                                                           const float* __restrict__ rstd, const float* __restrict__ gamma,
                                                           const float* __restrict__ sums, float* dgamma, float* dbeta,
                                                           uint4* __restrict__ dx, int64_t M, int tpr, int rpi, int C,
                                                           const float* __restrict__ beta_own,
                                                           const uint8_t* __restrict__ mbits) {
  pdl_wait();
  pdl_trigger();
  const int t = threadIdx.x;
  const int cg = t % tpr, r = t / tpr;
  // dx = k0*(g - db/M - xhat*dg/M) = k0*g + kb*x + ka,  kb = -k0*rstd*dg/M,  ka = -k0*db/M - kb*mean
  float k0[8], kb[8], ka[8], sh[8];
  const float invM = 1.0f / (float)M;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = cg * 8 + j;
    const float mu = mean[c], rs = rstd[c];
    const float db = sums[c], dg = sums[C + c];
    if (blockIdx.x == 0 && r == 0) {
      dbeta[c] = db;
      dgamma[c] = dg;
    }
    k0[j] = gamma[c] * rs;            // == sc of bn_apply_kernel
    sh[j] = OWN ? beta_own[c] - mu * k0[j] : 0.f;
    kb[j] = -k0[j] * rs * dg * invM;
    ka[j] = -k0[j] * db * invM - kb[j] * mu;
  }
  if (!dx) return;
  const int64_t stride = (int64_t)gridDim.x * rpi;
#pragma unroll 2
  for (int64_t row = (int64_t)blockIdx.x * rpi + r; row < M; row += stride) {
    const int64_t i0 = row * tpr + cg;
    const uint4 d0 = ldg_stream(dy + i0), x0 = ldg_stream(x + i0);
    uint4 a0 = d0;
    uint32_t mb = 0xffu;
    if (!OWN && mbits) mb = __ldg(mbits + i0);
    else if (!OWN && act) a0 = ldg_stream(act + i0);
    float fd[8], fx[8], fa[8], o[8];
    unpack8(d0, fd);
    unpack8(x0, fx);
    unpack8(a0, fa);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (OWN) fa[j] = fx[j] * k0[j] + sh[j];
      float g = ((OWN || act) && !(fa[j] > 0.f)) ? 0.f : fd[j];
      if (!OWN && !((mb >> j) & 1u)) g = 0.f;
      o[j] = fmaf(k0[j], g, fmaf(kb[j], fx[j], ka[j]));
    }
    dx[i0] = pack8(o);
  }
}

bool bn_bwd_bf16(const bf16* dy, const bf16* mask_act, const bf16* x, const float* mean, const float* rstd,
                 const float* gamma, float* dgamma, float* dbeta, bf16* dx, int64_t M, int C, float* sums, lbc_stream_t s,
                 const float* beta_own, const uint8_t* mask_bits, int pre_rows) {
  if (C % 8 || C > 2560) return false;
  static const bool recompute = [] {
    const char* e = getenv("LBC_BN_MASK_RECOMPUTE");
    return e ? atoi(e) != 0 : true;
  }();
  if (!recompute || !mask_act) beta_own = nullptr;
  if (beta_own) mask_bits = nullptr;
  RowGeom g = row_geom(M, C, 4);
  float* part = partial_buffer();
  if (!part) return false;
  if (beta_own) {
    RowGeom g3 = row_geom(M, C, 3);
    { auto k_ = bn_bwd_reduce_kernel<true>; LBC_LAUNCH(k_, dim3(g3.grid), dim3(g3.threads), g3.threads * 16 * sizeof(float), s,  (const uint4*)dy, (const uint4*)mask_act, (const uint4*)x, mean, rstd, M, g3.tpr, g3.rpi, part, C, gamma, beta_own, nullptr, nullptr, nullptr, nullptr); }
    LBC_LAUNCHED("bn_bwd_reduce_kernel<own>");
    col_finalize(part, g3.grid, 2 * C, sums, s);
    { auto k_ = bn_bwd_apply_kernel<true>; LBC_LAUNCH(k_, dim3(g.grid), dim3(g.threads), 0, s, (const uint4*)dy, (const uint4*)mask_act, (const uint4*)x, mean, rstd, gamma, sums, dgamma, dbeta, (uint4*)dx, M, g.tpr, g.rpi, C, beta_own, nullptr); }
    LBC_LAUNCHED("bn_bwd_apply_kernel<own>");
    LBC_CUDA(cudaGetLastError());
    return true;
  }
  if (mask_bits) mask_act = nullptr;   // the bits replace the activation read
  if (pre_rows > 0) {
    // the partial rows are already in the shared scratch: resid_bn_reduce_bf16 reduced while it produced dy
    col_finalize(part, pre_rows, 2 * C, sums, s);
  } else {
    { auto k_ = bn_bwd_reduce_kernel<false>; LBC_LAUNCH(k_, dim3(g.grid), dim3(g.threads), g.threads * 16 * sizeof(float), s,  (const uint4*)dy, (const uint4*)mask_act, (const uint4*)x, mean, rstd, M, g.tpr, g.rpi, part, C, gamma, beta_own, mask_bits, nullptr, nullptr, nullptr); }
    LBC_LAUNCHED("bn_bwd_reduce_kernel");
    col_finalize(part, g.grid, 2 * C, sums, s);
  }
  { auto k_ = bn_bwd_apply_kernel<false>; LBC_LAUNCH(k_, dim3(g.grid), dim3(g.threads), 0, s, (const uint4*)dy, (const uint4*)mask_act, (const uint4*)x, mean, rstd, gamma, sums, dgamma, dbeta, (uint4*)dx, M, g.tpr, g.rpi, C, beta_own, mask_bits); }
  LBC_LAUNCHED("bn_bwd_apply_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}

// ------------------------------------------------------------------------------------------- elementwise
// mode 0: dst = dst + src ; mode 1: dst = dst + src*(act>0) ; mode 2: dst = dst*(act>0) (src ignored)
// (mbits != null: the mask is one byte per 8 elements, as written by bn_apply_kernel, instead of the activation)
__global__ void __launch_bounds__(256) ew_kernel(uint4* __restrict__ dst, const uint4* __restrict__ src,
                                                 const uint4* __restrict__ act, int64_t n, int mode,
                                                 const uint8_t* __restrict__ mbits) {
  pdl_wait();
  pdl_trigger();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float a[8], b[8], m[8];
    unpack8(dst[i], a);
    if (mode != 2) unpack8(ldg_stream(src + i), b);
    if (mbits) {
      const uint32_t mb = __ldg(mbits + i);
#pragma unroll
      for (int j = 0; j < 8; ++j) m[j] = ((mb >> j) & 1u) ? 1.f : 0.f;
    } else if (mode != 0) {
      unpack8(ldg_stream(act + i), m);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (mode == 0) a[j] += b[j];
      else if (mode == 1) a[j] += (m[j] > 0.f) ? b[j] : 0.f;
      else a[j] = (m[j] > 0.f) ? a[j] : 0.f;
    }
    dst[i] = pack8(a);
  }
}
bool ew_bf16(bf16* dst, const bf16* src, const bf16* act, int64_t n, int mode, lbc_stream_t s, const uint8_t* mask_bits) {
  if (n % 8) return false;
  if (mode == 0) mask_bits = nullptr;
  int64_t nv = n / 8;
  int64_t blocks = (nv + 255) / 256;
  int64_t cap = (int64_t)sm_count2() * 16;
  if (blocks > cap) blocks = cap;
  { auto k_ = ew_kernel; LBC_LAUNCH(k_, dim3((unsigned)blocks), dim3(256), 0, s, (uint4*)dst, (const uint4*)src, (const uint4*)act, nv, mode, mask_bits); }
  LBC_LAUNCHED("ew_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}

// dst[m, 0:Cd] = src[m, 0:min(Cs, Cd)], channels beyond Cs filled with fill[m / rows_per_fill] (bf16-rounded): the late
// fusion of the speed (image.py:77-79: 512 trunk channels + 128 copies of the speed) and, with Cd < Cs, the slice that drops
// those channels again in backward.  One 16-byte vector per thread (the one-element-per-thread par_for versions took 42 and
// 34 us for 20 MB).
__global__ void __launch_bounds__(256) copy_channels_kernel(uint4* __restrict__ dst, const uint4* __restrict__ src, int64_t M,
                                                            int cd8, int cs8, const float* __restrict__ fill, int rows_per_fill) {
  pdl_wait();
  pdl_trigger();
  const int64_t n = M * cd8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i / cd8;
    const int j = (int)(i - m * cd8);
    if (j < cs8) {
      dst[i] = ldg_stream(src + m * cs8 + j);
    } else {
      float f[8];
      const float v = __ldg(fill + m / rows_per_fill);
#pragma unroll
      for (int k = 0; k < 8; ++k) f[k] = v;
      dst[i] = pack8(f);
    }
  }
}
bool copy_channels_bf16(bf16* dst, const bf16* src, int64_t M, int Cd, int Cs, const float* fill, int rows_per_fill, lbc_stream_t s) {
  if ((Cd % 8) || (Cs % 8) || (Cd > Cs && !fill) || rows_per_fill < 1) return false;
  const int64_t n = M * (Cd / 8);
  int64_t blocks = (n + 255) / 256;
  const int64_t cap = (int64_t)sm_count2() * 16;
  if (blocks > cap) blocks = cap;
  { auto k_ = copy_channels_kernel; LBC_LAUNCH(k_, dim3((unsigned)blocks), dim3(256), 0, s, (uint4*)dst, (const uint4*)src, M, Cd / 8, Cs / 8, fill, rows_per_fill); }
  LBC_LAUNCHED("copy_channels_kernel");
  return true;
}

// ------------------------------------------------------------------------------------------- stem BN+ReLU+MaxPool
// pool[n,oh,ow,:] = max over the 3x3/s2/p1 window of relu(bn(x)); idx = kh*3+kw of the first maximum.
// (resnet.py:150-152).  One thread per (output position, 8 channels); the BN+ReLU activation is never written.
// Both pooling kernels are instruction-bound, not HBM-bound, so: index arithmetic in IdxT (32-bit whenever the element
// count allows), and the per-channel constants hoisted out of the grid-stride loop (the stride is a multiple of tpr,
// so a thread keeps its channel group).
template <typename IdxT>
__global__ void __launch_bounds__(256) bn_relu_maxpool_kernel(const uint4* __restrict__ x, const float* __restrict__ mean,
                                                              const float* __restrict__ rstd, const float* __restrict__ gamma,
                                                              const float* __restrict__ beta, uint4* __restrict__ y,
                                                              uint2* __restrict__ idx, int N, int H, int W, int tpr, int OH,
                                                              int OW) {
  pdl_wait();
  pdl_trigger();
  const IdxT total = (IdxT)N * OH * OW * tpr;
  const IdxT stride = (IdxT)gridDim.x * blockDim.x;   // multiple of tpr (tpr divides 256)
  IdxT i = (IdxT)blockIdx.x * blockDim.x + threadIdx.x;
  const int cg = (int)(i % (IdxT)tpr);
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = cg * 8 + j;
    sc[j] = gamma[c] * rstd[c];
    sh[j] = beta[c] - mean[c] * sc[j];
  }
  for (; i < total; i += stride) {
    IdxT p = i / (IdxT)tpr;
    const int ow = (int)(p % (IdxT)OW);
    p /= (IdxT)OW;
    const int oh = (int)(p % (IdxT)OH);
    const int b = (int)(p / (IdxT)OH);
    float best[8];
    int bi[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      best[j] = -INFINITY;
      bi[j] = 0;
    }
    const uint4* xb = x + (int64_t)b * H * W * tpr + cg;
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const int ih = oh * 2 - 1 + kh;
      if (ih < 0 || ih >= H) continue;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int iw = ow * 2 - 1 + kw;
        if (iw < 0 || iw >= W) continue;
        float f[8];
        unpack8(__ldg(xb + (ih * W + iw) * tpr), f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float v = fmaxf(f[j] * sc[j] + sh[j], 0.f);
          // compare on the bf16-rounded activation, exactly what a materialised a_stem would hold
          v = __bfloat162float(__float2bfloat16_rn(v));
          if (v > best[j]) {
            best[j] = v;
            bi[j] = kh * 3 + kw;
          }
        }
      }
    }
    y[i] = pack8(best);
    uint2 id;
    id.x = (uint32_t)bi[0] | ((uint32_t)bi[1] << 8) | ((uint32_t)bi[2] << 16) | ((uint32_t)bi[3] << 24);
    id.y = (uint32_t)bi[4] | ((uint32_t)bi[5] << 8) | ((uint32_t)bi[6] << 16) | ((uint32_t)bi[7] << 24);
    idx[i] = id;
  }
}
bool bn_relu_maxpool_bf16(const bf16* x, const float* mean, const float* rstd, const float* gamma, const float* beta,
                          bf16* y, uint8_t* idx, int N, int H, int W, int C, int OH, int OW, lbc_stream_t s) {
  if (C % 8 || 256 % (C / 8)) return false;
  // (a variant computing 2x2 output blocks from the shared 5x5 patch -- 25 instead of 36 loads + transforms -- measured
  // 0.05 ms per step SLOWER on the same box, 14.498 vs 14.450 ms: more registers, fewer threads; not kept)
  int64_t total = (int64_t)N * OH * OW * (C / 8);
  int64_t blocks = (total + 255) / 256;
  int64_t cap = (int64_t)sm_count2() * 16;
  if (blocks > cap) blocks = cap;
  if ((int64_t)N * H * W * (C / 8) < (int64_t)1 << 31)
    { auto k_ = bn_relu_maxpool_kernel<uint32_t>; LBC_LAUNCH(k_, dim3((unsigned)blocks), dim3(256), 0, s, (const uint4*)x, mean, rstd, gamma, beta, (uint4*)y, (uint2*)idx, N, H, W, C / 8, OH, OW); }
  else
    { auto k_ = bn_relu_maxpool_kernel<int64_t>; LBC_LAUNCH(k_, dim3((unsigned)blocks), dim3(256), 0, s, (const uint4*)x, mean, rstd, gamma, beta, (uint4*)y, (uint2*)idx, N, H, W, C / 8, OH, OW); }
  LBC_LAUNCHED("bn_relu_maxpool_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}
// d(bn-relu output)[n,h,w,:] = sum over the <=4 pooling windows that selected (h,w), times the ReLU mask recomputed
// from the raw conv output; written as the upstream gradient of the stem BatchNorm.
// One thread owns a 2x2 block of input pixels (x 8 channels): the four pixels are touched by exactly the four windows
// (ph|ph+1, pw|pw+1), with FIXED tap codes per (pixel, window) -- so every thread runs the same nine compare-adds and loads
// each window once.  (Round 1's one-pixel-per-thread kernel looked at up to nine (kh, kw) candidates per pixel with
// parity-dependent branches that diverged inside every warp: 518 us for 1.19 GB at B = 256.)
// (A variant that fused the stem BatchNorm backward on top -- recomputing this gradient in the reduce and in the apply pass
// instead of storing it, 1.9 GB instead of 3.7 GB of traffic at B = 256 -- measured the SAME step time on the same box,
// 14.451 vs 14.450 ms: these kernels are bound by instruction issue, not by HBM; not kept.)
template <typename IdxT>
__global__ void __launch_bounds__(256) maxpool_relu_bwd_kernel(const uint4* __restrict__ dy, const uint2* __restrict__ idx,
                                                               const uint4* __restrict__ x, const float* __restrict__ mean,
                                                               const float* __restrict__ rstd, const float* __restrict__ gamma,
                                                               const float* __restrict__ beta, uint4* __restrict__ dx, int N,
                                                               int H, int W, int tpr, int OH, int OW) {
  pdl_wait();
  pdl_trigger();
  const int H2 = H >> 1, W2 = W >> 1;
  const IdxT total = (IdxT)N * H2 * W2 * tpr;
  const IdxT stride = (IdxT)gridDim.x * blockDim.x;   // multiple of tpr
  IdxT i = (IdxT)blockIdx.x * blockDim.x + threadIdx.x;
  const int cg = (int)(i % (IdxT)tpr);
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = cg * 8 + j;
    sc[j] = gamma[c] * rstd[c];
    sh[j] = beta[c] - mean[c] * sc[j];
  }
  for (; i < total; i += stride) {
    IdxT p = i / (IdxT)tpr;
    const int pw = (int)(p % (IdxT)W2);
    p /= (IdxT)W2;
    const int ph = (int)(p % (IdxT)H2);
    const int b = (int)(p / (IdxT)H2);
    float acc[2][2][8];
#pragma unroll
    for (int a2 = 0; a2 < 2; ++a2)
#pragma unroll
      for (int b2 = 0; b2 < 2; ++b2)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[a2][b2][j] = 0.f;
    const int64_t ob = (int64_t)b * OH * OW * tpr + cg;
#pragma unroll
    for (int wy = 0; wy < 2; ++wy) {
      const int oh = ph + wy;
      if (oh >= OH) continue;
#pragma unroll
      for (int wx = 0; wx < 2; ++wx) {
        const int ow = pw + wx;
        if (ow >= OW) continue;
        const int64_t o = ob + ((int64_t)oh * OW + ow) * tpr;
        const uint2 id = __ldg(idx + o);
        float g[8];
        unpack8(__ldg(dy + o), g);
        // window (ph+wy, pw+wx) covers pixel (a2, b2) of this block with tap kh = 1 + a2 - 2*wy, kw = 1 + b2 - 2*wx
#pragma unroll
        for (int a2 = wy; a2 < 2; ++a2)
#pragma unroll
          for (int b2 = wx; b2 < 2; ++b2) {
            const uint32_t want = (uint32_t)((1 + a2 - 2 * wy) * 3 + (1 + b2 - 2 * wx));
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const uint32_t sel = ((j < 4 ? id.x : id.y) >> ((j & 3) * 8)) & 0xffu;
              if (sel == want) acc[a2][b2][j] += g[j];
            }
          }
      }
    }
#pragma unroll
    for (int a2 = 0; a2 < 2; ++a2)
#pragma unroll
      for (int b2 = 0; b2 < 2; ++b2) {
        const int64_t e = (((int64_t)b * H + (2 * ph + a2)) * W + (2 * pw + b2)) * tpr + cg;
        float f[8];
        unpack8(ldg_stream(x + e), f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float v = f[j] * sc[j] + sh[j];
          if (!(v > 0.f)) acc[a2][b2][j] = 0.f;
        }
        dx[e] = pack8(acc[a2][b2]);
      }
  }
}
bool maxpool_relu_bwd_bf16(const bf16* dy, const uint8_t* idx, const bf16* x, const float* mean, const float* rstd,
                           const float* gamma, const float* beta, bf16* dx, int N, int H, int W, int C, int OH, int OW,
                           lbc_stream_t s) {
  if (C % 8 || 256 % (C / 8) || (H & 1) || (W & 1)) return false;
  int64_t total = (int64_t)N * (H / 2) * (W / 2) * (C / 8);
  int64_t blocks = (total + 255) / 256;
  int64_t cap = (int64_t)sm_count2() * 16;
  if (blocks > cap) blocks = cap;
  if ((int64_t)N * H * W * (C / 8) < (int64_t)1 << 31)
    { auto k_ = maxpool_relu_bwd_kernel<uint32_t>; LBC_LAUNCH(k_, dim3((unsigned)blocks), dim3(256), 0, s, (const uint4*)dy, (const uint2*)idx, (const uint4*)x, mean, rstd, gamma, beta, (uint4*)dx, N, H, W, C / 8, OH, OW); }
  else
    { auto k_ = maxpool_relu_bwd_kernel<int64_t>; LBC_LAUNCH(k_, dim3((unsigned)blocks), dim3(256), 0, s, (const uint4*)dy, (const uint2*)idx, (const uint4*)x, mean, rstd, gamma, beta, (uint4*)dx, N, H, W, C / 8, OH, OW); }
  LBC_LAUNCHED("maxpool_relu_bwd_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}

// dst += src * bits(src_bits)  (the masked residual add) AND the reduce pass of the BatchNorm that consumes dst next:
// partial rows of [sum g | sum g*xhat], g = dst * bits(mask_bits), left in the shared scratch for bn_bwd_bf16(..., pre_rows)
bool resid_bn_reduce_bf16(bf16* dst, const bf16* src, const uint8_t* src_bits, const bf16* x, const float* mean, const float* rstd,
                          const uint8_t* mask_bits, int64_t M, int C, int* rows, lbc_stream_t s) {
  if (C % 8 || C > 2560 || !src_bits || !mask_bits) return false;
  RowGeom g = row_geom(M, C, 4);
  float* part = partial_buffer();
  if (!part) return false;
  { auto k_ = bn_bwd_reduce_kernel<false, true>; LBC_LAUNCH(k_, dim3(g.grid), dim3(g.threads), g.threads * 16 * sizeof(float), s,  (const uint4*)dst, nullptr, (const uint4*)x, mean, rstd, M, g.tpr, g.rpi, part, C, nullptr, nullptr, mask_bits, (const uint4*)src, src_bits, (uint4*)dst); }
  LBC_LAUNCHED("bn_bwd_reduce_kernel<resid>");
  LBC_CUDA(cudaGetLastError());
  *rows = g.grid;
  return true;
}

#else  // LBC_HOST_EMU
bool bn_stats_bf16(const bf16*, int64_t, int, float*, lbc_stream_t) { return false; }
bool bn_apply_bf16(const bf16*, const float*, int64_t, int, const float*, const float*, float, float, float*, float*, float*,
                   float*, const bf16*, bool, bool, bf16*, float*, lbc_stream_t, uint8_t*) { return false; }
bool bn_bwd_bf16(const bf16*, const bf16*, const bf16*, const float*, const float*, const float*, float*, float*, bf16*,
                 int64_t, int, float*, lbc_stream_t, const float*, const uint8_t*, int) { return false; }
bool resid_bn_reduce_bf16(bf16*, const bf16*, const uint8_t*, const bf16*, const float*, const float*, const uint8_t*, int64_t, int,
                          int*, lbc_stream_t) { return false; }
bool ew_bf16(bf16*, const bf16*, const bf16*, int64_t, int, lbc_stream_t, const uint8_t*) { return false; }
bool copy_channels_bf16(bf16*, const bf16*, int64_t, int, int, const float*, int, lbc_stream_t) { return false; }
float* stat_partial_buffer() { return nullptr; }
int64_t stat_partial_capacity() { return 0; }
bool bn_finalize_bf16(const float*, int, int, int64_t, const float*, const float*, float, float, float*, float*, float*, float*,
                      float*, float*, float*, lbc_stream_t) { return false; }
bool bn_stats_partials_bf16(const bf16*, int64_t, int, int*, lbc_stream_t) { return false; }
bool col_finalize_bf16(const float*, int, int, float*, lbc_stream_t) { return false; }
bool bn_relu_maxpool_bf16(const bf16*, const float*, const float*, const float*, const float*, bf16*, uint8_t*, int, int, int,
                          int, int, int, lbc_stream_t) { return false; }
bool maxpool_relu_bwd_bf16(const bf16*, const uint8_t*, const bf16*, const float*, const float*, const float*, const float*,
                           bf16*, int, int, int, int, int, int, lbc_stream_t) { return false; }

#endif

}  // namespace fast
}  // namespace lbc
