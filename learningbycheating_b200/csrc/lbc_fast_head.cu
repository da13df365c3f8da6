// lbc_fast_head.cu -- fused waypoint heads of the bf16 path (image.py:54-60,82-84; common.py:136-152):
// 4 x [BatchNorm2d(64) -> Conv2d(64,5,1)+bias -> SpatialSoftmax] over the SAME decoder output h.
// The four BNs share batch statistics, so BN and the 1x1 convs fold into one 64->20 affine map per pixel:
//   logit[kj] = sum_c A[kj][c] * h[c] + b'[kj],  A = W_k[j,c]*gamma_kc*rstd_c,  b' = bias + sum_c W (beta - gamma*mean*rstd)
// forward = 1 pass over h; backward = 1 pass for the 20x64 moment matrix S and 1 pass producing d(h) with the decoder's
// final ReLU mask fused in (SURVEY.md 9.1 closed forms).
#include "lbc_fast.h"

#ifndef LBC_HOST_EMU
#include <cuda_bf16.h>
#endif

namespace lbc {
namespace fast {

#ifndef LBC_HOST_EMU
struct k_head_fold;
struct k_head_coef;

__device__ __forceinline__ void unpack8h(const uint4& v, float* f) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
static int sm_count3() {
  static int n = [] {
    int dev = 0, v = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v > 0 ? v : 148;
  }();
  return n;
}

// fold[0..1280) = A[kj][c]; fold[1280..1300) = b'[kj]
bool head_fold(ref::HeadParams hp, float* fold, lbc_stream_t s) {
  par_for<k_head_fold>(s, 20, [=] __device__(int64_t kj) {
    int k = (int)kj / 5, j = (int)kj % 5;
    float b = hp.bias[k][j];
    for (int c = 0; c < 64; ++c) {
      float w = hp.w[k][j * 64 + c];
      float sc = hp.gamma[k][c] * hp.rstd[k][c];
      fold[kj * 64 + c] = w * sc;
      b += w * (hp.beta[k][c] - hp.mean[k][c] * sc);
    }
    fold[1280 + kj] = b;
  });
  return true;
}

// ---- warp-level tensor-core building blocks (mma.sync m16n8k16 bf16 -> fp32) of the three head GEMMs ----
// The head products are tiny (K = 64 or 20, N = 20 or 64) and sit between a 126 MB activation read and a 78 MB logits
// read/write: they only have to keep up with HBM.  The CUDA-core versions (four pixels per thread, coefficients from shared
// memory) were bound by neither -- 92 / 177 / 156 us for kernels whose traffic is worth 31 / 31 / 51 us.  Here one warp
// owns 32 pixels, the 64-channel rows are staged with cp.async into a 128-byte-swizzled tile (ldmatrix reads it without bank
// conflicts) and fp32 operands (folded weights, dlogits) enter as bf16 hi + lo pairs (two or three MMAs per product, ~2^-17
// relative), so the results stay at fp32 level while the FMAs move to the tensor pipe.
__device__ __forceinline__ void mma_16816(float* d, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4(uint32_t* r, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t* r, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// bf16 hi / lo split of an fp32 pair (low half = first element, as the MMA fragments want)
__device__ __forceinline__ void split2(float x, float y, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 hx = __float2bfloat16_rn(x), hy = __float2bfloat16_rn(y);
  const __nv_bfloat16 lx = __float2bfloat16_rn(x - __bfloat162float(hx)), ly = __float2bfloat16_rn(y - __bfloat162float(hy));
  hi = (uint32_t)__bfloat16_as_ushort(hx) | ((uint32_t)__bfloat16_as_ushort(hy) << 16);
  lo = (uint32_t)__bfloat16_as_ushort(lx) | ((uint32_t)__bfloat16_as_ushort(ly) << 16);
}
// stage the [128 pixels][64 channels] bf16 tile of image n starting at pixel p0 (np valid pixels, the rest zero-filled):
// 16-byte chunk c of row r lands at chunk (c ^ (r & 7)) -- the 128-byte swizzle
__device__ __forceinline__ void stage_h(uint8_t* tile, const bf16* h, int64_t pix0, int np) {
  const uint8_t* src = reinterpret_cast<const uint8_t*>(h) + pix0 * 128;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int i = threadIdx.x + 128 * j;
    const int r = i >> 3, c = i & 7;
    const uint32_t dst = smem_addr(tile + r * 128 + ((c ^ (r & 7)) << 4));
    const int bytes = r < np ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src + (r < np ? (int64_t)r * 128 + c * 16 : 0)),
                 "r"(bytes)
                 : "memory");
  }
}
__device__ __forceinline__ void stage_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void stage_tile(uint8_t* tile, const bf16* h, int64_t pix0, int np) {
  stage_h(tile, h, pix0, np);
  stage_commit();
}
// the 20 dlogits rows of the same 128 pixels ([20][PAD] floats, PAD chosen by the reader against bank conflicts): rows of
// 512 contiguous bytes in global memory (HW % 4 == 0), pixels >= np zero-filled
template <int PAD>
__device__ __forceinline__ void stage_dl(float* dst, const float* dl, int HW, int np) {
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    const int i = threadIdx.x + 128 * j;
    const int kj = i >> 5, px = (i & 31) * 4;
    const int bytes = px < np ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_addr(dst + kj * PAD + px)),
                 "l"(dl + (int64_t)kj * HW + (px < np ? px : 0)), "r"(bytes)
                 : "memory");
  }
}
__device__ __forceinline__ void stage_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void stage_wait_1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

// logits[n][kj][p] = b'[kj] + sum_c A[kj][c] h[n,p,c]:  D[32 px per warp][24] = H[32][64] x (A_hi + A_lo)^T
__global__ void __launch_bounds__(128) head_logits_mma_kernel(const bf16* __restrict__ h, const float* __restrict__ fold,
                                                               float* __restrict__ logits, int N, int HW) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ __align__(1024) uint8_t hs_smem[];
  uint8_t* tile[2] = {hs_smem, hs_smem + 16384};
  float(*out)[132] = reinterpret_cast<float(*)[132]>(hs_smem + 32768);   // [20][128 px (+4)]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  uint32_t bh[4][3][2], bl[4][3][2];
  float bias[3][2];
#pragma unroll
  for (int nt = 0; nt < 3; ++nt) {
    const int kj = nt * 8 + g;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks)
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int c = ks * 16 + half * 8 + 2 * t;
        const float w0 = kj < 20 ? __ldg(fold + kj * 64 + c) : 0.f, w1 = kj < 20 ? __ldg(fold + kj * 64 + c + 1) : 0.f;
        split2(w0, w1, bh[ks][nt][half], bl[ks][nt][half]);
      }
    bias[nt][0] = nt * 8 + 2 * t < 20 ? __ldg(fold + 1280 + nt * 8 + 2 * t) : 0.f;
    bias[nt][1] = nt * 8 + 2 * t + 1 < 20 ? __ldg(fold + 1280 + nt * 8 + 2 * t + 1) : 0.f;
  }
  const int tiles_per_img = (HW + 127) / 128;
  const int ntiles = N * tiles_per_img;
  int tl = blockIdx.x, buf = 0;
  if (tl < ntiles) {
    const int n = tl / tiles_per_img, p0 = (tl - n * tiles_per_img) * 128;
    stage_tile(tile[0], h, (int64_t)n * HW + p0, min(128, HW - p0));
  }
  for (; tl < ntiles; tl += gridDim.x, buf ^= 1) {
    const int n = tl / tiles_per_img, p0 = (tl - n * tiles_per_img) * 128;
    const int np = min(128, HW - p0);
    const int nx = tl + gridDim.x;
    if (nx < ntiles) {
      const int n2 = nx / tiles_per_img, q0 = (nx - n2 * tiles_per_img) * 128;
      stage_tile(tile[buf ^ 1], h, (int64_t)n2 * HW + q0, min(128, HW - q0));
      stage_wait_1();
    } else {
      stage_wait_all();
    }
    __syncthreads();   // tile[buf] complete; every thread is past the previous tile's store loop (out is free)
    const uint32_t tb = smem_addr(tile[buf]);
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      float acc[3][4];
#pragma unroll
      for (int nt = 0; nt < 3; ++nt) {
        acc[nt][0] = acc[nt][2] = bias[nt][0];
        acc[nt][1] = acc[nt][3] = bias[nt][1];
      }
      const int r = warp * 32 + mt * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;   // ldmatrix row of this lane
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        uint32_t a[4];
        const int chunk = ks * 2 + (lane >> 4);
        ldsm_x4(a, tb + r * 128 + ((chunk ^ (r & 7)) << 4));
#pragma unroll
        for (int nt = 0; nt < 3; ++nt) {
          mma_16816(acc[nt], a, bl[ks][nt][0], bl[ks][nt][1]);
          mma_16816(acc[nt], a, bh[ks][nt][0], bh[ks][nt][1]);
        }
      }
      const int px = warp * 32 + mt * 16 + g;
#pragma unroll
      for (int nt = 0; nt < 3; ++nt) {
        const int kj = nt * 8 + 2 * t;
        if (kj < 20) {
          out[kj][px] = acc[nt][0];
          out[kj + 1][px] = acc[nt][1];
          out[kj][px + 8] = acc[nt][2];
          out[kj + 1][px + 8] = acc[nt][3];
        }
      }
    }
    __syncthreads();
    if ((int)threadIdx.x < np) {
      float* dst = logits + ((int64_t)n * 20) * HW + p0 + threadIdx.x;
#pragma unroll
      for (int kj = 0; kj < 20; ++kj) dst[(int64_t)kj * HW] = out[kj][threadIdx.x];
    }
  }
}

// one block per (n, kj) row; HW <= 128*32
__global__ void __launch_bounds__(128) head_softmax_kernel(const float* __restrict__ logits, float* __restrict__ rowmax,
                                                           float* __restrict__ rowsum, float* __restrict__ preds, int H, int W) {
  pdl_wait();
  pdl_trigger();
  const int HW = H * W;
  const float* l = logits + (int64_t)blockIdx.x * HW;
  float v[32];
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    int p = i * 128 + threadIdx.x;
    v[i] = p < HW ? l[p] : -INFINITY;
    m = fmaxf(m, v[i]);
  }
  __shared__ float red[4][4];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[0][threadIdx.x >> 5] = m;
  __syncthreads();
  m = fmaxf(fmaxf(red[0][0], red[0][1]), fmaxf(red[0][2], red[0][3]));
  __syncthreads();
  float se = 0.f, sx = 0.f, sy = 0.f;
  const float kx = W > 1 ? 2.0f / (float)(W - 1) : 0.f, ky = H > 1 ? 2.0f / (float)(H - 1) : 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    int p = i * 128 + threadIdx.x;
    if (p < HW) {
      float e = __expf(v[i] - m);
      int hh = p / W, ww = p - hh * W;
      se += e;
      sx += e * (-1.f + kx * (float)ww);
      sy += e * (-1.f + ky * (float)hh);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    se += __shfl_xor_sync(0xffffffffu, se, o);
    sx += __shfl_xor_sync(0xffffffffu, sx, o);
    sy += __shfl_xor_sync(0xffffffffu, sy, o);
  }
  if ((threadIdx.x & 31) == 0) {
    red[1][threadIdx.x >> 5] = se;
    red[2][threadIdx.x >> 5] = sx;
    red[3][threadIdx.x >> 5] = sy;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    se = red[1][0] + red[1][1] + red[1][2] + red[1][3];
    sx = red[2][0] + red[2][1] + red[2][2] + red[2][3];
    sy = red[3][0] + red[3][1] + red[3][2] + red[3][3];
    rowmax[blockIdx.x] = m;
    rowsum[blockIdx.x] = se;
    preds[blockIdx.x * 2] = sx / se;
    preds[blockIdx.x * 2 + 1] = sy / se;
  }
}

// SpatialSoftmax alone (common.py:136-152) over [N*20] rows of H*W logits
bool head_softmax_f32(const float* logits, float* rowmax, float* rowsum, float* preds, int N, int H, int W, lbc_stream_t s) {
  if (!enabled() || H * W > 4096) return false;
  { auto k_ = head_softmax_kernel; LBC_LAUNCH(k_, dim3(N * 20), dim3(128), 0, s, logits, rowmax, rowsum, preds, H, W); }
  LBC_LAUNCHED("head_softmax_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}
bool head_forward_bf16(const bf16* h, ref::HeadParams hp, float* fold, float* logits, float* rowmax, float* rowsum,
                       float* preds, int N, int H, int W, lbc_stream_t s) {
  if (!enabled()) return false;
  const int HW = H * W;
  if (HW > 4096) return false;
  head_fold(hp, fold, s);
  {
    constexpr int SMEM = 32768 + 20 * 132 * 4;
    static bool configured = false;
    if (!configured) {
      LBC_CUDA(cudaFuncSetAttribute(head_logits_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
      configured = true;
    }
    const int ntiles = N * ((HW + 127) / 128);
    int grid = sm_count3() * 4;
    if (grid > ntiles) grid = ntiles;
    { auto k_ = head_logits_mma_kernel; LBC_LAUNCH(k_, dim3(grid), dim3(128), SMEM, s, h, fold, logits, N, HW); }
    LBC_LAUNCHED("head_logits_mma_kernel");
  }
  { auto k_ = head_softmax_kernel; LBC_LAUNCH(k_, dim3(N * 20), dim3(128), 0, s, logits, rowmax, rowsum, preds, H, W); }
  LBC_LAUNCHED("head_softmax_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}

// coef[0..64) = c0, coef[64..128) = c1 :  dh = A^T dl - c0 - hhat*c1
bool head_coef(ref::HeadParams hp, ref::HeadGrads hg, float* coef, float invM, lbc_stream_t s) {
  par_for<k_head_coef>(s, 64, [=] __device__(int64_t c) {
    float a = 0.f, b = 0.f;
    for (int k = 0; k < 4; ++k) {
      a += hp.gamma[k][c] * hg.dbeta[k][c];
      b += hp.gamma[k][c] * hg.dgamma[k][c];
    }
    coef[c] = hp.rstd[0][c] * a * invM;
    coef[64 + c] = hp.rstd[0][c] * b * invM;
  });
  return true;
}
// d(pre-ReLU deconv output)[pix][c] = (h>0) * (sum_kj A[kj][c] dl[kj] - c0[c] - hhat[c]*c1[c]):
// D[32 px per warp][64] = dl^T[32][20 -> 32] x A[32][64] with hi / lo pairs on both sides (3 MMAs per product); the epilogue
// reads h from the staged tile and writes the bf16 result over it in place, the tile then leaves with 16-byte stores.
__global__ void __launch_bounds__(128) head_dh_mma_kernel(const float* __restrict__ dlogits, const bf16* __restrict__ h,
                                                          const float* __restrict__ fold, const float* __restrict__ coef,
                                                          const float* __restrict__ mean, const float* __restrict__ rstd,
                                                          bf16* __restrict__ dh, int N, int HW) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ __align__(1024) uint8_t hs_smem[];
  uint8_t* tile[2] = {hs_smem, hs_smem + 16384};
  float* cf = reinterpret_cast<float*>(hs_smem + 32768);   // c0 | c1 | mean | rstd
  constexpr int DPAD = 132;                                 // A fragments read dls[kj = 2t (+1)][px = g]: banks 8t + g (+4)
  float* dls[2] = {reinterpret_cast<float*>(hs_smem + 33792), reinterpret_cast<float*>(hs_smem + 33792 + 20 * DPAD * 4)};
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  if (threadIdx.x < 64) {
    cf[threadIdx.x] = coef[threadIdx.x];
    cf[64 + threadIdx.x] = coef[64 + threadIdx.x];
    cf[128 + threadIdx.x] = mean[threadIdx.x];
    cf[192 + threadIdx.x] = rstd[threadIdx.x];
  }
  uint32_t bh[2][8][2], bl[2][8][2];   // B[k = kj][n = c] = A[kj][c]
#pragma unroll
  for (int ks = 0; ks < 2; ++ks)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int kj = ks * 16 + half * 8 + 2 * t, c = nt * 8 + g;
        const float w0 = kj < 20 ? __ldg(fold + kj * 64 + c) : 0.f, w1 = kj + 1 < 20 ? __ldg(fold + (kj + 1) * 64 + c) : 0.f;
        split2(w0, w1, bh[ks][nt][half], bl[ks][nt][half]);
      }
  const int tiles_per_img = (HW + 127) / 128;
  const int ntiles = N * tiles_per_img;
  int tl = blockIdx.x, buf = 0;
  if (tl < ntiles) {
    const int n = tl / tiles_per_img, p0 = (tl - n * tiles_per_img) * 128;
    stage_h(tile[0], h, (int64_t)n * HW + p0, min(128, HW - p0));
    stage_dl<DPAD>(dls[0], dlogits + ((int64_t)n * 20) * HW + p0, HW, min(128, HW - p0));
    stage_commit();
  }
  for (; tl < ntiles; tl += gridDim.x, buf ^= 1) {
    const int n = tl / tiles_per_img, p0 = (tl - n * tiles_per_img) * 128;
    const int np = min(128, HW - p0);
    const int nx = tl + gridDim.x;
    if (nx < ntiles) {
      const int n2 = nx / tiles_per_img, q0 = (nx - n2 * tiles_per_img) * 128;
      stage_h(tile[buf ^ 1], h, (int64_t)n2 * HW + q0, min(128, HW - q0));   // (free: barrier at the end of the last tile)
      stage_dl<DPAD>(dls[buf ^ 1], dlogits + ((int64_t)n2 * 20) * HW + q0, HW, min(128, HW - q0));
      stage_commit();
      stage_wait_1();
    } else {
      stage_wait_all();
    }
    __syncthreads();
    // this warp's dlogits fragments, hi / lo pairs
    uint32_t ah[2][2][4], al[2][2][4];
    const float* dl = dls[buf];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int px = warp * 32 + mt * 16 + g + (q & 1) * 8;
          const int kj = ks * 16 + (q >> 1) * 8 + 2 * t;
          const float v0 = kj < 20 ? dl[kj * DPAD + px] : 0.f;
          const float v1 = kj + 1 < 20 ? dl[(kj + 1) * DPAD + px] : 0.f;
          split2(v0, v1, ah[mt][ks][q], al[mt][ks][q]);
        }
    uint8_t* tb = tile[buf];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
          mma_16816(acc, al[mt][ks], bh[ks][nt][0], bh[ks][nt][1]);
          mma_16816(acc, ah[mt][ks], bl[ks][nt][0], bl[ks][nt][1]);
          mma_16816(acc, ah[mt][ks], bh[ks][nt][0], bh[ks][nt][1]);
        }
        const int c = nt * 8 + 2 * t;
        const float c00 = cf[c], c01 = cf[c + 1], c10 = cf[64 + c], c11 = cf[64 + c + 1];
        const float m0 = cf[128 + c], m1 = cf[128 + c + 1], r0 = cf[192 + c], r1 = cf[192 + c + 1];
#pragma unroll
        for (int hrow = 0; hrow < 2; ++hrow) {
          const int row = warp * 32 + mt * 16 + g + hrow * 8;
          uint32_t* hp = reinterpret_cast<uint32_t*>(tb + row * 128 + ((nt ^ (row & 7)) << 4) + t * 4);
          const uint32_t hw = *hp;
          const float f0 = __uint_as_float(hw << 16), f1 = __uint_as_float(hw & 0xffff0000u);
          const float o0 = f0 > 0.f ? acc[hrow * 2] - c00 - (f0 - m0) * r0 * c10 : 0.f;
          const float o1 = f1 > 0.f ? acc[hrow * 2 + 1] - c01 - (f1 - m1) * r1 * c11 : 0.f;
          __nv_bfloat162 o = __floats2bfloat162_rn(o0, o1);
          *hp = *reinterpret_cast<uint32_t*>(&o);
        }
      }
    }
    __syncthreads();
    uint4* dst = reinterpret_cast<uint4*>(dh) + ((int64_t)n * HW + p0) * 8;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int i = threadIdx.x + 128 * j;
      const int r = i >> 3, c = i & 7;
      if (r < np) dst[i] = *reinterpret_cast<const uint4*>(tb + r * 128 + ((c ^ (r & 7)) << 4));
    }
    __syncthreads();   // the tile has left: the next iteration's cp.async may refill this buffer
  }
}

// dlogit = softmax * ((x - Ex) gx + (y - Ey) gy), g = d_preds + onehot * d_pred (SURVEY 9.1): one block per (n, kj) row, the
// row constants read once, coalesced 4-byte traffic.  (The one-thread-per-element version recomputed the row constants and
// the grid coordinates with integer divisions per element: 167 us for a 157 MB read + write at B = 256.)
__global__ void __launch_bounds__(128) head_dlogits_kernel(const float* __restrict__ logits, const float* __restrict__ rowmax,
                                                           const float* __restrict__ rowsum, const float* __restrict__ preds,
                                                           const float* __restrict__ onehot, const float* __restrict__ d_pred,
                                                           const float* __restrict__ d_preds, float* __restrict__ dlogits, int H,
                                                           int W) {
  pdl_wait();
  pdl_trigger();
  const int HW = H * W;
  const int r = blockIdx.x;
  const int kj = r % 20, b = r / 20;
  const int k = kj / 5, j = kj % 5;
  float gx = 0.f, gy = 0.f;
  if (d_preds) {
    gx += d_preds[r * 2];
    gy += d_preds[r * 2 + 1];
  }
  if (d_pred) {
    const float oh = onehot[b * 4 + k];
    gx += oh * d_pred[(b * 5 + j) * 2];
    gy += oh * d_pred[(b * 5 + j) * 2 + 1];
  }
  const float m = rowmax[r], inv = 1.0f / rowsum[r], ex = preds[r * 2], ey = preds[r * 2 + 1];
  const float kx = W > 1 ? 2.0f / (float)(W - 1) : 0.f, ky = H > 1 ? 2.0f / (float)(H - 1) : 0.f;
  const float* l = logits + (int64_t)r * HW;
  float* d = dlogits + (int64_t)r * HW;
  for (int p = threadIdx.x; p < HW; p += 128) {
    const int hh = p / W, ww = p - hh * W;
    const float wgt = __expf(l[p] - m) * inv;
    d[p] = wgt * ((-1.f + kx * (float)ww - ex) * gx + (-1.f + ky * (float)hh - ey) * gy);
  }
}
bool head_dlogits_f32(const float* logits, const float* rowmax, const float* rowsum, const float* preds, const float* onehot,
                      const float* d_pred, const float* d_preds, float* dlogits, int N, int H, int W, lbc_stream_t s) {
  if (!enabled()) return false;
  { auto k_ = head_dlogits_kernel; LBC_LAUNCH(k_, dim3(N * 20), dim3(128), 0, s, logits, rowmax, rowsum, preds, onehot, d_pred, d_preds, dlogits, H, W); }
  LBC_LAUNCHED("head_dlogits_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}

// S[block][kj][c] = sum_pix dl[n,kj,pix]*hhat[n,pix,c] (c<64), S[block][kj][64] = sum dl over the block's tiles:
// D[20 -> 32][64 (+8: a tile of ones gives sum dl)] += dl[32][128 px] x H[128 px][64], K = pixels; warp w owns pixels
// [32w, 32w+32) of every tile (K split over the warps), dl enters as hi + lo bf16 pairs, H as stored.  The accumulators
// (raw moments sum dl*h) live across the block's tiles; at the end  S = rstd*(raw - mean * sum dl)  per block, as doubles
// that sum_slices_kernel adds in block order.
__global__ void __launch_bounds__(128) head_s_mma_kernel(const float* __restrict__ dlogits, const bf16* __restrict__ h,
                                                         const float* __restrict__ mean, const float* __restrict__ rstd,
                                                         double* S, int N, int HW) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ __align__(1024) uint8_t hs_smem[];
  uint8_t* tile[2] = {hs_smem, hs_smem + 16384};
  constexpr int DPAD = 136;   // A fragments read 8 bytes at dls[kj = g][px = 2t]: banks 8g + 2t over a half warp
  float* dls[2] = {reinterpret_cast<float*>(hs_smem + 32768), reinterpret_cast<float*>(hs_smem + 32768 + 20 * DPAD * 4)};
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  float acc[2][9][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 9; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;
  const int tiles_per_img = (HW + 127) / 128;
  const int ntiles = N * tiles_per_img;
  int tl = blockIdx.x, buf = 0;
  if (tl < ntiles) {
    const int n = tl / tiles_per_img, p0 = (tl - n * tiles_per_img) * 128;
    stage_h(tile[0], h, (int64_t)n * HW + p0, min(128, HW - p0));
    stage_dl<DPAD>(dls[0], dlogits + ((int64_t)n * 20) * HW + p0, HW, min(128, HW - p0));
    stage_commit();
  }
  for (; tl < ntiles; tl += gridDim.x, buf ^= 1) {
    const int nx = tl + gridDim.x;
    __syncthreads();   // every warp is done with the previous tile (its buffers are refilled now)
    if (nx < ntiles) {
      const int n2 = nx / tiles_per_img, q0 = (nx - n2 * tiles_per_img) * 128;
      stage_h(tile[buf ^ 1], h, (int64_t)n2 * HW + q0, min(128, HW - q0));
      stage_dl<DPAD>(dls[buf ^ 1], dlogits + ((int64_t)n2 * 20) * HW + q0, HW, min(128, HW - q0));
      stage_commit();
      stage_wait_1();
    } else {
      stage_wait_all();
    }
    __syncthreads();
    // A fragments: dl[kj = 16 mt + g (+8)][px = 32 w + 16 ks + 2t (+8), +1], hi / lo pairs
    uint32_t ah[2][2][4], al[2][2][4];
    const float* dl = dls[buf];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int kj = mt * 16 + g + (q & 1) * 8;
          const int px = warp * 32 + ks * 16 + (q >> 1) * 8 + 2 * t;
          float2 v = make_float2(0.f, 0.f);
          if (kj < 20) v = *reinterpret_cast<const float2*>(dl + kj * DPAD + px);
          split2(v.x, v.y, ah[mt][ks][q], al[mt][ks][q]);
        }
    const uint32_t tb = smem_addr(tile[buf]);
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      // B fragments: H[k = px][n = c], transposed 8x8 loads; lane -> (matrix j = lane / 8: k half j & 1, channel half j >> 1)
      const int krow = warp * 32 + ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
#pragma unroll
      for (int np2 = 0; np2 < 4; ++np2) {   // channel tiles 2 np2, 2 np2 + 1
        uint32_t b[4];
        const int chunk = np2 * 2 + (lane >> 4);
        ldsm_x4_trans(b, tb + krow * 128 + ((chunk ^ (krow & 7)) << 4));
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          mma_16816(acc[mt][2 * np2], al[mt][ks], b[0], b[1]);
          mma_16816(acc[mt][2 * np2], ah[mt][ks], b[0], b[1]);
          mma_16816(acc[mt][2 * np2 + 1], al[mt][ks], b[2], b[3]);
          mma_16816(acc[mt][2 * np2 + 1], ah[mt][ks], b[2], b[3]);
        }
      }
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {   // ones: sum over pixels of dl
        mma_16816(acc[mt][8], al[mt][ks], 0x3F803F80u, 0x3F803F80u);
        mma_16816(acc[mt][8], ah[mt][ks], 0x3F803F80u, 0x3F803F80u);
      }
    }
  }
  stage_wait_all();
  __syncthreads();
  // combine the four warps (K split) and publish: part[w][kj 0..19][c 0..64]
  float(*part)[20][65] = reinterpret_cast<float(*)[20][65]>(hs_smem);   // 4 x 20 x 65 floats = 20.8 KB
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 9; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int kj = mt * 16 + g + (e >> 1) * 8, c = nt * 8 + 2 * t + (e & 1);
        if (kj < 20 && c < 65) part[warp][kj][c] = acc[mt][nt][e];
      }
  __syncthreads();
  for (int i = threadIdx.x; i < 20 * 65; i += 128) {
    const int kj = i / 65, c = i - kj * 65;
    const float raw = (part[0][kj][c] + part[1][kj][c]) + (part[2][kj][c] + part[3][kj][c]);
    float v = raw;
    if (c < 64) {
      const float s0 = (part[0][kj][64] + part[1][kj][64]) + (part[2][kj][64] + part[3][kj][64]);
      v = (raw - mean[c] * s0) * rstd[c];
    }
    S[(int64_t)blockIdx.x * 20 * 65 + kj * 65 + c] = (double)v;
  }
}

// S: [20][65] doubles (the blocks' partials added in block order).  Produces S, then the caller computes parameter grads (ref::head_param_grads),
// then head_backward_dh_bf16 writes the masked d(h).
bool head_backward_s_bf16(const float* dlogits, const bf16* h, const float* mean, const float* rstd, double* S, int N, int HW,
                          lbc_stream_t s) {
  if (!enabled()) return false;
  if (HW & 3) return false;   // (16-byte dlogits staging)
  int grid = sm_count3() * 2;
  int ntiles = N * ((HW + 127) / 128);
  if (grid > ntiles) grid = ntiles;
  static double* part = nullptr;   // [grid][20][65] block partials (main stream only)
  static int part_blocks = 0;
  if (grid > part_blocks) {
    if (part) {
      cudaDeviceSynchronize();
      cudaFree(part);
    }
    part = nullptr;
    part_blocks = 0;
    if (cudaMalloc(&part, sizeof(double) * 20 * 65 * (size_t)grid) != cudaSuccess) {
      cudaGetLastError();
      part = nullptr;
      return false;
    }
    part_blocks = grid;
  }
  constexpr int SMEM = 32768 + 2 * 20 * 136 * 4;
  static bool configured = false;
  if (!configured) {
    LBC_CUDA(cudaFuncSetAttribute(head_s_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    configured = true;
  }
  { auto k_ = head_s_mma_kernel; LBC_LAUNCH(k_, dim3(grid), dim3(128), SMEM, s, dlogits, h, mean, rstd, part, N, HW); }
  LBC_LAUNCHED("head_s_mma_kernel");
  { auto k_ = sum_slices_kernel<double>; LBC_LAUNCH(k_, dim3((20 * 65 + 255) / 256), dim3(256), 0, s, (const double*)part, S, (int64_t)20 * 65, grid); }
  LBC_LAUNCHED("sum_slices_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}
bool head_backward_dh_bf16(const float* dlogits, const bf16* h, ref::HeadParams hp, ref::HeadGrads hg, const float* fold,
                           float* coef, bf16* dh, int N, int HW, lbc_stream_t s) {
  if (!enabled()) return false;
  const int64_t npix = (int64_t)N * HW;
  head_coef(hp, hg, coef, 1.0f / (float)npix, s);
  const int ntiles = N * ((HW + 127) / 128);
  int grid = sm_count3() * 4;
  if (grid > ntiles) grid = ntiles;
  constexpr int SMEM = 32768 + 1024 + 2 * 20 * 132 * 4;
  static bool configured = false;
  if (!configured) {
    LBC_CUDA(cudaFuncSetAttribute(head_dh_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    configured = true;
  }
  { auto k_ = head_dh_mma_kernel; LBC_LAUNCH(k_, dim3(grid), dim3(128), SMEM, s, dlogits, h, fold, coef, hp.mean[0], hp.rstd[0], dh, N, HW); }
  LBC_LAUNCHED("head_dh_mma_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}

#else
bool head_softmax_f32(const float*, float*, float*, float*, int, int, int, lbc_stream_t) { return false; }
bool head_forward_bf16(const bf16*, ref::HeadParams, float*, float*, float*, float*, float*, int, int, int, lbc_stream_t) {
  return false;
}
bool head_backward_s_bf16(const float*, const bf16*, const float*, const float*, double*, int, int, lbc_stream_t) { return false; }
bool head_dlogits_f32(const float*, const float*, const float*, const float*, const float*, const float*, const float*, float*, int,
                      int, int, lbc_stream_t) { return false; }
bool head_backward_dh_bf16(const float*, const bf16*, ref::HeadParams, ref::HeadGrads, const float*, float*, bf16*, int, int,
                           lbc_stream_t) { return false; }
#endif

}  // namespace fast
}  // namespace lbc
