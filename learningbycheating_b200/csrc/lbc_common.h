// lbc_common.h -- shared plumbing for the LBC image-agent training engine (sm_100a).
//
// Two build modes:
//   * product: nvcc -gencode arch=compute_100a,code=sm_100a  -> liblbc_b200.so (CUDA only,
//     no CPU path; every entry point works on device pointers).
//   * LBC_HOST_EMU: g++ -x c++ of the SAME sources, kernels of the correctness-first path run
//     as plain loops over host pointers.  Test infrastructure for `pytest -m "not gpu"` (host
//     logic: graph executor, buffer plan, parameter table).  Never loaded by the package.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#ifdef LBC_HOST_EMU
#define LBC_HD
#define LBC_DEV
#define LBC_LAMBDA
typedef void* lbc_stream_t;
#else
#include <cuda_runtime.h>
#define LBC_HD __host__ __device__
#define LBC_DEV __device__
#define LBC_LAMBDA __device__   /* extended lambdas of par_for: device-only closures */
typedef cudaStream_t lbc_stream_t;
#endif

namespace lbc {

// ------------------------------------------------------------------ errors
struct Error : std::runtime_error {
  explicit Error(const std::string& s) : std::runtime_error(s) {}
};
#define LBC_CHECK(cond, msg)                                                            \
  do {                                                                                  \
    if (!(cond)) throw ::lbc::Error(std::string(__FILE__) + ":" + std::to_string(__LINE__) + \
                                    ": " + (msg));                                      \
  } while (0)

#ifndef LBC_HOST_EMU
#define LBC_CUDA(call)                                                                  \
  do {                                                                                  \
    cudaError_t e_ = (call);                                                            \
    if (e_ != cudaSuccess)                                                              \
      throw ::lbc::Error(std::string(__FILE__) + ":" + std::to_string(__LINE__) + ": " + \
                         #call + " -> " + cudaGetErrorString(e_));                      \
  } while (0)
#endif

// ------------------------------------------------------------------ bf16 storage type
// Bit-compatible with __nv_bfloat16; own struct so the same code compiles for the host emu.
struct bf16 {
  uint16_t v;
};
LBC_HD inline float bf16_to_float(bf16 h) {
  uint32_t u = ((uint32_t)h.v) << 16;
  float f;
#if defined(__CUDA_ARCH__)
  f = __uint_as_float(u);
#else
  memcpy(&f, &u, 4);
#endif
  return f;
}
LBC_HD inline bf16 float_to_bf16(float f) {
  uint32_t u;
#if defined(__CUDA_ARCH__)
  u = __float_as_uint(f);
#else
  memcpy(&u, &f, 4);
#endif
  bf16 h;
  if ((u & 0x7fffffffu) > 0x7f800000u) {  // NaN
    h.v = 0x7fff;
    return h;
  }
  u += 0x7fffu + ((u >> 16) & 1u);  // round to nearest even
  h.v = (uint16_t)(u >> 16);
  return h;
}

template <class T>
LBC_HD inline float ldf(const T* p, int64_t i);
template <>
LBC_HD inline float ldf<float>(const float* p, int64_t i) {
  return p[i];
}
template <>
LBC_HD inline float ldf<bf16>(const bf16* p, int64_t i) {
  return bf16_to_float(p[i]);
}
template <class T>
LBC_HD inline void stf(T* p, int64_t i, float v);
template <>
LBC_HD inline void stf<float>(float* p, int64_t i, float v) {
  p[i] = v;
}
template <>
LBC_HD inline void stf<bf16>(bf16* p, int64_t i, float v) {
  p[i] = float_to_bf16(v);
}

// ------------------------------------------------------------------ device memory
inline void* dev_alloc(size_t bytes) {
  if (bytes == 0) bytes = 16;
#ifdef LBC_HOST_EMU
  void* p = nullptr;
  if (posix_memalign(&p, 256, bytes) != 0) throw Error("host-emu alloc failed");
  return p;
#else
  void* p = nullptr;
  LBC_CUDA(cudaMalloc(&p, bytes));
  return p;
#endif
}
inline void dev_free(void* p) {
  if (!p) return;
#ifdef LBC_HOST_EMU
  free(p);
#else
  cudaFree(p);
#endif
}
inline void dev_memset(void* p, int v, size_t bytes, lbc_stream_t s) {
#ifdef LBC_HOST_EMU
  (void)s;
  memset(p, v, bytes);
#else
  LBC_CUDA(cudaMemsetAsync(p, v, bytes, s));
#endif
}
inline void dev_copy(void* dst, const void* src, size_t bytes, lbc_stream_t s) {
#ifdef LBC_HOST_EMU
  (void)s;
  memcpy(dst, src, bytes);
#else
  LBC_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s));
#endif
}

// ------------------------------------------------------------------ launch counter + per-category profiler
// g_launches counts every kernel the library launches (bench.py reports it as gpu_launches).
extern long long g_launches;
// launch trace (tests): when on, every launch also records its kernel-family name, so a parity test can assert WHICH
// kernel produced the result (a silent fast -> correctness-first fallback would otherwise pass).  lbc_trace_* in the C ABI.
extern bool g_trace_on;
void trace_note(const char* name);
void trace_reset();
std::string trace_dump();   // "name\tcount\n" per kernel family
template <class Tag>
inline const char* tag_name() {   // "... [with Tag = lbc::ref::k_conv_fwd]": works for the incomplete tag types
  return __PRETTY_FUNCTION__;
}
#define LBC_LAUNCHED(name)                              \
  do {                                                  \
    ++::lbc::g_launches;                                \
    if (::lbc::g_trace_on) ::lbc::trace_note(name);     \
  } while (0)
struct ProfEntry {
  std::string cat;
  double flops, bytes;
#ifndef LBC_HOST_EMU
  cudaEvent_t e0, e1;
#endif
};
extern bool g_prof_on;
extern std::vector<ProfEntry> g_prof;
// RAII: brackets the launches of one op with CUDA events on the launching stream when profiling is on.
struct ProfScope {
  bool on;
  lbc_stream_t s;
  size_t idx;
  ProfScope(const char* cat, lbc_stream_t stream, double flops, double bytes) : on(g_prof_on), s(stream), idx(0) {
    if (!on) return;
    ProfEntry e;
    e.cat = cat;
    e.flops = flops;
    e.bytes = bytes;
#ifndef LBC_HOST_EMU
    cudaEventCreate(&e.e0);
    cudaEventCreate(&e.e1);
    cudaEventRecord(e.e0, s);
#endif
    idx = g_prof.size();
    g_prof.push_back(e);
  }
  ~ProfScope() {
#ifndef LBC_HOST_EMU
    if (on) cudaEventRecord(g_prof[idx].e1, s);
#endif
  }
};

// ------------------------------------------------------------------ launches (programmatic dependent launch)
// Every kernel of the library starts with pdl_wait(); pdl_trigger(); (after smem-only setup, before its first global access)
// and is launched through LBC_LAUNCH.  With g_pdl on (LBC_PDL, lbc_set_pdl) the launch carries
// cudaLaunchAttributeProgrammaticStreamSerialization: the grid may be scheduled while its predecessor in the stream still
// runs (its CTAs take SMs as the predecessor's retire and sit in griddepcontrol.wait until the predecessor has completed
// and flushed), so the launch latency and the prologue (barrier init, TMEM allocation) of ~450 dependent launches per step
// leave the critical path.  The trigger comes right after the wait, so at most two consecutive grids overlap.  Without the
// attribute griddepcontrol.wait returns at once.
extern int g_wgrad_overlap;   // schedule of backward() in the bf16 mode (lbc_net.cu), lbc_set_schedule
#ifndef LBC_HOST_EMU
extern int g_pdl;
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// dst[i] = src[i] + src[n + i] + ... + src[(slices - 1) * n + i], added in that order: the reduction of per-split (or
// per-block) partials that keeps a split computation bitwise reproducible from run to run, where atomics into one
// buffer would add the partials in whatever order the blocks finish
template <typename T>
__global__ void sum_slices_kernel(const T* __restrict__ src, T* __restrict__ dst, int64_t n, int slices) {
  pdl_wait();
  pdl_trigger();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  T a = src[i];
  for (int s = 1; s < slices; ++s) a += src[(int64_t)s * n + i];
  dst[i] = a;
}
struct LaunchCfg {
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[2];
  LaunchCfg(dim3 grid, dim3 block, size_t smem, cudaStream_t s, int cluster_x = 1) {
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    int n = 0;
    if (cluster_x > 1) {
      attr[n].id = cudaLaunchAttributeClusterDimension;
      attr[n].val.clusterDim.x = (unsigned)cluster_x;
      attr[n].val.clusterDim.y = 1;
      attr[n].val.clusterDim.z = 1;
      ++n;
    }
    if (g_pdl) {
      attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      attr[n].val.programmaticStreamSerializationAllowed = 1;
      ++n;
    }
    cfg.attrs = attr;
    cfg.numAttrs = (unsigned)n;
  }
};
// kern: a kernel function pointer (name a template instantiation through `auto k = kernel<...>;` first)
#define LBC_LAUNCH(kern, grid, block, smem, stream, ...)                                  \
  do {                                                                                    \
    ::lbc::LaunchCfg lc_(grid, block, smem, stream);                                      \
    LBC_CUDA(cudaLaunchKernelEx(&lc_.cfg, kern, __VA_ARGS__));                            \
  } while (0)
#define LBC_LAUNCH_CLUSTER(kern, cluster_x, grid, block, smem, stream, ...)               \
  do {                                                                                    \
    ::lbc::LaunchCfg lc_(grid, block, smem, stream, cluster_x);                           \
    LBC_CUDA(cudaLaunchKernelEx(&lc_.cfg, kern, __VA_ARGS__));                            \
  } while (0)
#endif

// ------------------------------------------------------------------ par_for
// The correctness-first kernels are "independent thread" kernels: one logical thread per
// output element, no shared memory, no atomics -> bitwise deterministic, and the same body
// runs under the host emulation.  Tag names the kernel in ncu launch lists.
#ifdef LBC_HOST_EMU
template <class Tag, class F>
inline void par_for(lbc_stream_t, int64_t n, F f) {
  LBC_LAUNCHED(tag_name<Tag>());
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < n; ++i) f(i);
}
#else
template <class Tag, class F>
__global__ void __launch_bounds__(256) par_for_kernel(int64_t n, F f) {
  pdl_wait();
  pdl_trigger();
  // grid-stride walk; with the default (uncapped) grid the stride covers the whole range: exactly one iteration per thread
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
#pragma unroll 1   // no trip-count arithmetic in front of the (normally single) iteration
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) f(i);
}
template <class Tag, class F>
inline void par_for(lbc_stream_t s, int64_t n, F f) {
  if (n <= 0) return;
  const int bs = 256;
  int64_t nb = (n + bs - 1) / bs;
  LBC_CHECK(nb < (1ll << 31), "par_for grid too large");
  auto kern = par_for_kernel<Tag, F>;
  LBC_LAUNCH(kern, dim3((unsigned)nb), dim3(bs), 0, s, n, f);
  LBC_LAUNCHED(tag_name<Tag>());
}
#endif

inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

}  // namespace lbc
