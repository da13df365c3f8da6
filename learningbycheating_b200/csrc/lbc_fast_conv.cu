// lbc_fast_conv.cu -- im2col-free implicit-GEMM convolutions on the sm_100a tensor cores.
//
//   D[128 output positions x BN channels] (fp32, TMEM) += A[128 x 64] (bf16, smem) * B[BN x 64]^T (bf16, smem)
//
// * A tile = a 4-D TMA box {64 ch, TW, TH, TN} of the NHWC activation at the tap's spatial offset: the
//   hardware zero-fills out-of-bounds coordinates, which IS the convolution padding (and the batch tail).
//   The box lands in shared memory as 128 rows x 128 B with the 128-byte swizzle == the UMMA K-major
//   SWIZZLE_128B canonical layout, so no im2col buffer ever exists.
// * Stride-2 convolutions read the four (row, column) parity sub-views of the input (tensor maps with doubled
//   strides), so every TMA load is unit-stride; the data gradient of a stride-2 convolution (== the forward of
//   nn.ConvTranspose2d(3,2,1,1), image.py:39-46) is four such GEMMs writing the four parity sub-views of dx.
// * One persistent CTA per SM, warp-specialised: warp 0 = TMA producer, warp 1 = tcgen05.mma issuer (one
//   elected lane) + TMEM owner, warps 2-5 = epilogue (tcgen05.ld -> bias/ReLU -> bf16 -> swizzled smem -> TMA
//   store).  smem ring of STAGES {A,B} tiles, two TMEM accumulators so the epilogue of tile i overlaps the MMAs
//   of tile i+1.
//
// Reference ops replaced: every nn.Conv2d of resnet.BasicBlock (resnet.py:15-22,38-54), its input gradient, and
// the decoder's ConvTranspose2d (image.py:39-46).
#ifndef LBC_HOST_EMU
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#endif

#include <map>
#include <mutex>
#include <tuple>

#include "lbc_fast.h"

namespace lbc {
namespace fast {

#ifndef LBC_HOST_EMU

// ------------------------------------------------------------------------------------------- tensor maps
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled encode_fn() {
  static PFN_encodeTiled fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !p) throw Error("cuTensorMapEncodeTiled unavailable");
    return (PFN_encodeTiled)p;
  }();
  return fn;
}

// 16-bit (bf16 / fp16: same tensor-map type for our purposes, TMA only moves the bits) or fp32 tensor [N][H][W][C] with
// arbitrary (16 B aligned) strides; box {128 B of channels, bw, bh, bn}, 128 B swizzle, zero OOB fill
static CUtensorMap make_map_4d(const void* base, int C, int W, int H, int N, int64_t sW, int64_t sH, int64_t sN, int bw,
                               int bh, int bn, bool f32 = false) {
  typedef std::tuple<const void*, int, int, int, int, int64_t, int64_t, int64_t, int, int, int, bool> Key;
  static std::map<Key, CUtensorMap> cache;
  static std::mutex mu;
  Key key(base, C, W, H, N, sW, sH, sN, bw, bh, bn, f32);
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(key);
  if (it != cache.end()) return it->second;
  CUtensorMap m;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)sW, (cuuint64_t)sH, (cuuint64_t)sN};
  cuuint32_t box[4] = {f32 ? 32u : 64u, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bn};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = encode_fn()(&m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4,
                           const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LBC_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(4d) failed: " + std::to_string((int)r));
  cache[key] = m;
  return m;
}
// bf16 matrix [rows][K] (K contiguous); box {64, brows}
static CUtensorMap make_map_2d(const void* base, int64_t K, int64_t rows, int brows) {
  typedef std::tuple<const void*, int64_t, int64_t, int> Key;
  static std::map<Key, CUtensorMap> cache;
  static std::mutex mu;
  Key key(base, K, rows, brows);
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(key);
  if (it != cache.end()) return it->second;
  CUtensorMap m;
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)(K * 2)};
  cuuint32_t box[2] = {64, (cuuint32_t)brows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LBC_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(2d) failed: " + std::to_string((int)r));
  cache[key] = m;
  return m;
}

// ------------------------------------------------------------------------------------------- device helpers
struct ConvGemmParams {
  int TW, TH, TN;                   // output-position tile = TN*TH*TW = 128
  int tiles_w, tiles_h, tiles_n;    // tiles per dimension
  int n_tiles_n;                    // N (channel) tiles
  int num_taps, k_chunks;           // K loop = num_taps * k_chunks iterations of 64
  int tap_dh[9], tap_dw[9], tap_map[9], tap_koff[9];
  const float* bias;                // per output channel or null
  int relu;
  // optional BatchNorm statistics of the stored (bf16-rounded) output: partial[m_tile][2*stat_C] (sum | sum of squares)
  float* stat_partial;
  int stat_C;
  int valid_n;                      // batch size (rows of images >= valid_n are the zero-filled tail)
  // split-precision mode (fp32tc): both operands are stored as two 16-bit planes [hi | lo] along K (A: channels
  // [0,a_plane) hi, [a_plane,2*a_plane) lo; B: every tap slab [hi b_plane | lo b_plane]); the K loop runs the three
  // products hi*lo + lo*hi + hi*hi into the same fp32 accumulator.  fmt: UMMA 16-bit operand format (0 = fp16, 1 = bf16).
  int split, a_plane, b_plane;
  uint32_t fmt_a, fmt_b;
  float out_scale;                  // accumulator scale applied in the epilogue (undoes the power-of-two operand scaling)
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// bounded wait: a protocol bug traps (launch error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t addr = smem_u32(bar);
  long long t0 = 0;
  for (uint32_t spin = 0;; ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return;
    if (spin == 64) t0 = clock64();
    if (spin > 64 && (spin & 1023) == 0 && clock64() - t0 > 4000000000ll) {
      printf("lbc conv_gemm: mbarrier wait timed out (block %d thread %d parity %u)\n", blockIdx.x, threadIdx.x, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* m, void* dst, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* m, void* dst, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)m), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"((uint64_t)m),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// UMMA shared-memory descriptor, K-major, SWIZZLE_128B: rows of 128 B, 8-row atoms 1024 B apart
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);  // start address
  d |= (uint64_t)1 << 16;                       // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;             // stride byte offset
  d |= (uint64_t)1 << 46;                       // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                       // SWIZZLE_128B
  return d;
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,"
      "%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- CTA-pair (cta_group::2) helpers: two CTAs of one TPC form a cluster and issue ONE 256-row MMA; each CTA stages
// its own 128 rows of A and HALF of the B tile, so the L2->SM operand traffic per flop drops by a third (BN = 256).
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same smem offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // (default .release.cta form, as in the multicast pipelines of CUTLASS: the TMEM reads are ordered by tcgen05.wait::ld +
  // tcgen05.fence::before_thread_sync, no global-memory fence is needed per tile)
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA loads of a CTA pair: data lands in the executing CTA's smem, the transaction bytes are signalled on the
// LEADER CTA's mbarrier (bar_cluster = mapa(full[stage], 0))
__device__ __forceinline__ void tma_load_4d_pair(const CUtensorMap* m, void* dst, uint32_t bar_cluster, int c0, int c1, int c2,
                                                 int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)m), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap* m, void* dst, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)m), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
// completion of all MMAs issued so far -> one arrival on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}

constexpr int A_BYTES = 128 * 128;  // 128 positions x 64 bf16

template <int BN, int STAGES, bool PAIR = false, bool OUT_F32 = false>
struct SmemPlan {
  static constexpr int B_BYTES = PAIR ? BN * 64 : BN * 128;   // CTA pair: each CTA stages BN/2 rows of B
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  // epilogue staging: the whole 128 x BN bf16 tile in OUT_PASSES column passes.  Two passes of 128 columns would buy the
  // pair kernel (BN = 256) a fifth operand stage; measured on the B200 that is no faster (52.3 vs 51.5 us per launch),
  // so the tile is staged in one pass.  fp32 output: two passes of BN/2 columns through the same staging bytes.
  static constexpr int OUT_PASSES = OUT_F32 ? 2 : 1;
  static constexpr int OUT_BYTES = (BN / 64) * A_BYTES;
  static constexpr int BAR_OFF = STAGES * STAGE_BYTES + OUT_BYTES;
  static constexpr int RED_OFF = BAR_OFF + 256;       // 128 x 4 floats: column-statistics scratch
  static constexpr int CSTAT_OFF = RED_OFF + 2048;    // [2][Co <= 512] floats: this CTA's running column sums / sums of squares
  static constexpr int TOTAL = CSTAT_OFF + 4096 + 1024;  // barriers + scratch + alignment slack
};

// ------------------------------------------------------------------------------------------- the kernel
// PAIR = true: launched as clusters of two CTAs (one TPC).  The pair computes a 256-position x BN tile with ONE
// tcgen05.mma.cta_group::2 stream issued by the leader (cluster rank 0): every CTA stages its own 128 positions of A
// and BN/2 rows of B (its TMA loads signal the LEADER's full barrier), the leader's commits are multicast to the
// empty / accumulator-full barriers of both CTAs, both epilogues arrive on the leader's accumulator-empty barrier.
// Each CTA's 128 x BN slice of the accumulator lives in its own TMEM, so the epilogue is unchanged.
template <int BN, int STAGES, bool PAIR, bool OUT_F32>
__global__ void __launch_bounds__(192, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap mA0, const __grid_constant__ CUtensorMap mA1,
                 const __grid_constant__ CUtensorMap mA2, const __grid_constant__ CUtensorMap mA3,
                 const __grid_constant__ CUtensorMap mB, const __grid_constant__ CUtensorMap mO, const ConvGemmParams p) {
  typedef SmemPlan<BN, STAGES, PAIR, OUT_F32> SP;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* out_stage = smem + STAGES * SP::STAGE_BYTES;
  uint64_t* full = (uint64_t*)(smem + SP::BAR_OFF);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = (uint32_t*)(tempty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr uint32_t TMEM_COLS = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], PAIR ? 256 : 128);   // pair: the epilogue threads of both CTAs arrive on the leader's
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if constexpr (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if constexpr (PAIR)
    cluster_sync_all();   // barrier inits of BOTH CTAs visible before any remote arrive / multicast commit
  else
    __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // everything above touched shared / tensor memory only
  pdl_trigger();

  const int tiles_m = p.tiles_w * p.tiles_h * p.tiles_n;
  const int nterm = p.split ? 3 : 1;
  const int k_iters = p.num_taps * nterm * p.k_chunks;
  // tile walk.  single CTA: tile = blockIdx.x + i*gridDim.x over tiles_m*n_tiles_n (m_tile = tile / n_tiles_n).
  // pair: the same walk over ceil(tiles_m/2)*n_tiles_n PAIR tiles by pair index; this CTA owns m_tile = 2*(..)+rank,
  // which for an odd tiles_m can be one past the end: its coordinates are past the batch, so TMA zero-fills the
  // loads and clips the store, and only the statistics row has to be skipped.
  const uint32_t crank = PAIR ? cluster_ctarank() : 0u;
  const int walk0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int walk_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int num_tiles = (PAIR ? (tiles_m + 1) / 2 : tiles_m) * p.n_tiles_n;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = walk0; tile < num_tiles; tile += walk_step) {
        const int n_tile = tile % p.n_tiles_n;
        const int m_tile = PAIR ? 2 * (tile / p.n_tiles_n) + (int)crank : tile / p.n_tiles_n;
        const int w0 = (m_tile % p.tiles_w) * p.TW;
        const int h0 = ((m_tile / p.tiles_w) % p.tiles_h) * p.TH;
        const int n0 = (m_tile / (p.tiles_w * p.tiles_h)) * p.TN;
        // split mode: the two cross terms (hi*lo, lo*hi) go first, the hi*hi term last.  The tensor core adds into the
        // fp32 accumulator with truncation (measured: bias ~ -5e-7 of the accumulator per ~100 accumulation steps), so
        // only the K/16 steps of the hi*hi term should run against a full-size accumulator.
        for (int term = 0; term < nterm; ++term) {
          const int ac0 = (p.split && term == 1) ? p.a_plane : 0;   // term 0: A hi x B lo, 1: A lo x B hi, 2: A hi x B hi
          const int bplane = (p.split && term == 0) ? p.b_plane : 0;
          for (int tap = 0; tap < p.num_taps; ++tap) {
            const int mid = p.tap_map[tap];
            const CUtensorMap* ma = mid == 0 ? &mA0 : (mid == 1 ? &mA1 : (mid == 2 ? &mA2 : &mA3));
            const int dh = p.tap_dh[tap], dw = p.tap_dw[tap];
            const int bc0 = p.tap_koff[tap] + bplane;
            for (int kc = 0; kc < p.k_chunks; ++kc) {
              mbar_wait(&empty[stage], phase ^ 1);
              uint8_t* sa = smem + stage * SP::STAGE_BYTES;
              if constexpr (PAIR) {
                // the leader's barrier collects the bytes of both CTAs (the peer's may land before this expect_tx:
                // the tx-count goes transiently negative inside the phase, which mbarrier allows)
                if (crank == 0) mbar_expect_tx(&full[stage], 2 * SP::STAGE_BYTES);
                const uint32_t lead_full = mapa_u32(smem_u32(&full[stage]), 0);
                tma_load_4d_pair(ma, sa, lead_full, ac0 + kc * 64, w0 + dw, h0 + dh, n0);
                tma_load_2d_pair(&mB, sa + A_BYTES, lead_full, bc0 + kc * 64, n_tile * BN + (int)crank * (BN / 2));
              } else {
                mbar_expect_tx(&full[stage], SP::STAGE_BYTES);
                tma_load_4d(ma, sa, &full[stage], ac0 + kc * 64, w0 + dw, h0 + dh, n0);
                tma_load_2d(&mB, sa + A_BYTES, &full[stage], bc0 + kc * 64, n_tile * BN);
              }
              if (++stage == STAGES) {
                stage = 0;
                phase ^= 1;
              }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (pair: the leader CTA only) =====================
    // instruction descriptor: D=f32, A/B = bf16 (format 1) or fp16 (0), both K-major, N=BN, M=128 (pair: M=256 over the two CTAs)
    const uint32_t idesc = (1u << 4) | (p.fmt_a << 7) | (p.fmt_b << 10) | ((uint32_t)(BN >> 3) << 17) |
                           ((uint32_t)((PAIR ? 256 : 128) >> 4) << 24);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = walk0; tile < num_tiles && crank == 0; tile += walk_step, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tempty[acc], acc_phase ^ 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t tmem_d = tmem_base + acc * BN;
      for (int k = 0; k < k_iters; ++k) {
        mbar_wait(&full[stage], phase);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + stage * SP::STAGE_BYTES);
          const uint64_t ad = umma_desc_k_sw128(sa);
          const uint64_t bd = umma_desc_k_sw128(sa + A_BYTES);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {  // 4 x (K=16) per 64-wide chunk: advance 32 B inside the swizzle atom
            if constexpr (PAIR)
              umma_bf16_pair(tmem_d, ad + (uint64_t)(kk * 2), bd + (uint64_t)(kk * 2), idesc, (k | kk) != 0);
            else
              umma_bf16(tmem_d, ad + (uint64_t)(kk * 2), bd + (uint64_t)(kk * 2), idesc, (k | kk) != 0);
          }
          if constexpr (PAIR) {
            umma_commit_pair(&empty[stage]);                    // frees the slot in both CTAs
            if (k == k_iters - 1) umma_commit_pair(&tfull[acc]);  // both epilogues
          } else {
            umma_commit(&empty[stage]);                    // frees the smem slot when these MMAs retire
            if (k == k_iters - 1) umma_commit(&tfull[acc]);  // accumulator complete -> epilogue
          }
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else {
    // ===================== epilogue (warps 2..5 -> TMEM lane quarters 2,3,0,1) =====================
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const bool issuer = (threadIdx.x == 64);
    // BatchNorm statistics: ONE partial row per CTA (the column sums of all its tiles, accumulated in shared memory in the
    // fixed order of the tile walk), so the finalize kernel reads gridDim.x rows instead of one per 128-position tile
    float* cstat = reinterpret_cast<float*>(smem + SP::CSTAT_OFF);
    if (!OUT_F32 && p.stat_partial) {
      for (int i = threadIdx.x - 64; i < 2 * p.stat_C; i += 128) cstat[i] = 0.f;
      asm volatile("bar.sync 1, 128;" ::: "memory");
    }
    int it = 0;
    for (int tile = walk0; tile < num_tiles; tile += walk_step, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int n_tile = tile % p.n_tiles_n;
      const int m_tile = PAIR ? 2 * (tile / p.n_tiles_n) + (int)crank : tile / p.n_tiles_n;
      const int w0 = (m_tile % p.tiles_w) * p.TW;
      const int h0 = ((m_tile / p.tiles_w) % p.tiles_h) * p.TH;
      const int n0 = (m_tile / (p.tiles_w * p.tiles_h)) * p.TN;
      mbar_wait(&tfull[acc], acc_phase);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN;
      constexpr int PASSES = SP::OUT_PASSES;
      constexpr int CW = BN / PASSES;   // columns staged per pass
#pragma unroll 1
      for (int hp = 0; hp < PASSES; ++hp) {
        if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // staging buffer free again
        asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll 1
        for (int cl = 0; cl < CW / 32; ++cl) {
          const int ch = hp * (CW / 32) + cl;
          uint32_t r[32];
          tmem_ld32(taddr + ch * 32, r);
          const int col0 = n_tile * BN + ch * 32;
          if constexpr (OUT_F32) {
            // fp32 output: 32 columns = one 128-byte row of a {32 ch, TW, TH, TN} fp32 store box
            uint8_t* rowp = out_stage + cl * A_BYTES + row * 128;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float v[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                float a = __uint_as_float(r[j * 4 + e]) * p.out_scale;
                if (p.bias) a += __ldg(p.bias + col0 + j * 4 + e);
                if (p.relu) a = fmaxf(a, 0.f);
                v[e] = a;
              }
              *reinterpret_cast<float4*>(rowp + ((j ^ (row & 7)) << 4)) = make_float4(v[0], v[1], v[2], v[3]);
            }
            continue;
          }
          uint8_t* rowp = out_stage + (cl >> 1) * A_BYTES + row * 128;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint32_t pk[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float a = __uint_as_float(r[j * 8 + e * 2]);
              float b = __uint_as_float(r[j * 8 + e * 2 + 1]);
              if (p.bias) {
                a += __ldg(p.bias + col0 + j * 8 + e * 2);
                b += __ldg(p.bias + col0 + j * 8 + e * 2 + 1);
              }
              if (p.relu) {
                a = fmaxf(a, 0.f);
                b = fmaxf(b, 0.f);
              }
              __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
              pk[e] = *reinterpret_cast<uint32_t*>(&h);
            }
            const int chunk16 = (cl & 1) * 4 + j;  // 16-byte chunk index inside the 128-byte row
            *reinterpret_cast<uint4*>(rowp + ((chunk16 ^ (row & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          }
        }
        if (hp == PASSES - 1) {
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          if constexpr (PAIR)
            mbar_arrive_cluster(mapa_u32(smem_u32(&tempty[acc]), 0));  // on the leader's barrier (256 arrivals per phase)
          else
            mbar_arrive(&tempty[acc]);  // accumulator drained: the MMA warp may reuse it
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (issuer) {
          constexpr int BOXC = OUT_F32 ? 32 : 64;   // channels per 128-byte store box
#pragma unroll
          for (int b = 0; b < CW / BOXC; ++b)
            tma_store_4d(&mO, out_stage + b * A_BYTES, n_tile * BN + hp * CW + b * BOXC, w0, h0, n0);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        if (!OUT_F32 && p.stat_partial && m_tile < tiles_m) {
          // per-channel sum / sum of squares of this pass's bf16 outputs, read back from the staging tile
          constexpr int PAIRS = CW / 2, TPP = 128 / PAIRS, RPT = 128 / TPP;
          float* red = reinterpret_cast<float*>(smem + SP::RED_OFF);
          const int e = threadIdx.x - 64;
          const int pair = e % PAIRS, sub = e / PAIRS;
          const int col = 2 * pair;
          const uint8_t* boxp = out_stage + (col >> 6) * A_BYTES + ((col & 7) >> 1) * 4;
          const int chunk = (col & 63) >> 3;
          int nvalid = p.valid_n - n0;
          nvalid = nvalid < 0 ? 0 : (nvalid > p.TN ? p.TN : nvalid);
          const int valid_rows = nvalid * p.TH * p.TW;
          float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
          for (int r = sub * RPT; r < (sub + 1) * RPT && r < valid_rows; ++r) {
            const uint32_t w = *reinterpret_cast<const uint32_t*>(boxp + r * 128 + ((chunk ^ (r & 7)) << 4));
            const float a = __uint_as_float(w << 16), b = __uint_as_float(w & 0xffff0000u);
            s0 += a;
            s1 += b;
            q0 += a * a;
            q1 += b * b;
          }
          if (TPP > 1) {
            red[e * 4 + 0] = s0;
            red[e * 4 + 1] = s1;
            red[e * 4 + 2] = q0;
            red[e * 4 + 3] = q1;
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (sub == 0) {
#pragma unroll
              for (int t2 = 1; t2 < TPP; ++t2) {
                s0 += red[(t2 * PAIRS + pair) * 4 + 0];
                s1 += red[(t2 * PAIRS + pair) * 4 + 1];
                q0 += red[(t2 * PAIRS + pair) * 4 + 2];
                q1 += red[(t2 * PAIRS + pair) * 4 + 3];
              }
            }
          }
          if (sub == 0) {   // (the same thread owns a column pair in every tile: no race on cstat)
            float* dst = cstat + n_tile * BN + hp * CW + col;
            dst[0] += s0;
            dst[1] += s1;
            dst[p.stat_C] += q0;
            dst[p.stat_C + 1] += q1;
          }
        }
      }
    }
    if (!OUT_F32 && p.stat_partial) {
      asm volatile("bar.sync 1, 128;" ::: "memory");
      float* dst = p.stat_partial + (int64_t)blockIdx.x * 2 * p.stat_C;
      for (int i = threadIdx.x - 64; i < 2 * p.stat_C; i += 128) dst[i] = cstat[i];
    }
    if (issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if constexpr (PAIR) {
    __syncwarp();
    cluster_sync_all();   // the peer's smem / TMEM are operands of the leader's MMAs until both CTAs are done
    if (warp == 1)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  } else {
    __syncthreads();
    if (warp == 1) {
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
  }
}

// ------------------------------------------------------------------------------------------- 3x3/s1, 64 output channels
// Layer-1-type convolutions (N = 64) are bound by L2->SM operand traffic, not by the tensor pipe: with one TMA box per
// tap every input pixel crosses the L2->SM link 9 times and the 72 KB of weights once per tile.  This variant
//   * keeps ALL weights resident in shared memory for the life of the persistent CTA, and
//   * loads ONE activation box per kernel ROW ({64 ch, 8+2 columns, TH, TN} = 160 rows of 128 B) and feeds the three
//     kw taps from it by starting the UMMA descriptor 0/1/2 rows (128 B) into the box: with an 8-pixel-wide tile each
//     8-row core-matrix group is one image row, so consecutive groups are exactly 10 rows = 1280 B apart (the
//     descriptor's stride-byte-offset) and the 128-byte swizzle, being a function of the shared-memory address, stays
//     consistent between the TMA write and the shifted MMA read.
// => 3 x 20 KB per tile instead of 9 x 16 KB + 72 KB.
struct ConvKwParams {
  int TH, TN, tiles_w, tiles_h, tiles_n;
  int k_chunks;
  int row_dh[3];        // spatial row offset of kernel-row group g
  int shift[3][3];      // row shift (0..2) into the 10-wide box for tap j of group g
  int koff[3][3];       // K offset of that tap in the packed weight matrix
  const float* bias;
  int relu;
  float* stat_partial;
  int stat_C;
  int valid_n;
};
constexpr int AKW_BYTES = 160 * 128;

template <int STAGES>
struct SmemPlanKw {
  static constexpr int BN = 64;
  static constexpr int BRES_BYTES = 9 * BN * 128;   // one 64-channel K chunk of all nine taps
  static constexpr int OUT_OFF = STAGES * AKW_BYTES + BRES_BYTES;
  static constexpr int BAR_OFF = OUT_OFF + A_BYTES;
  static constexpr int RED_OFF = BAR_OFF + 256;
  static constexpr int TOTAL = RED_OFF + 2048 + 256 + 1024;   // 128 x 4 floats reduction scratch + 64 bias floats + alignment slack
};

__device__ __forceinline__ uint64_t umma_desc_k_sw128_sbo(uint32_t smem_addr, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// ---- BatchNorm statistics of the N = 64 kernels (conv3x3_c64_kernel, stem_conv_kernel) ----
// Epilogue thread e (0..127) owns the column pair 2*(e % 32) and the 32 staged rows [32*(e/32), 32*(e/32)+32): after a
// tile's bf16 outputs sit in the staging buffer it reads its 32 x 4 bytes back and adds them to FOUR registers that live
// across all tiles of the persistent CTA.  Round 1 reduced and wrote one partial row per TILE (a shared-memory exchange,
// a named barrier and a global store per tile, 7680 / 30720 partial rows per launch for col_finalize to sum): the forward
// launches of the layer-1 kernel took 132 us against 82 us for the same GEMM without statistics.  Now: one partial row per
// CTA, written once at the end.
struct ColStat {
  float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
};
__device__ __forceinline__ void colstat_accumulate(ColStat& cs, const uint8_t* out_stage, int e, int valid_rows) {
  const int pair = e & 31, sub = e >> 5;
  const int col = 2 * pair;
  const uint8_t* boxp = out_stage + ((col & 7) >> 1) * 4;
  const int chunk = col >> 3;
  const int r0 = sub * 32;
  if (valid_rows >= r0 + 32) {   // whole strip valid (every tile but the batch tail): 32 independent loads
    uint32_t w[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const int r = r0 + i;
      w[i] = *reinterpret_cast<const uint32_t*>(boxp + r * 128 + ((chunk ^ (r & 7)) << 4));
    }
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const float a = __uint_as_float(w[i] << 16), b = __uint_as_float(w[i] & 0xffff0000u);
      cs.s0 += a;
      cs.s1 += b;
      cs.q0 += a * a;
      cs.q1 += b * b;
    }
  } else {
    for (int r = r0; r < r0 + 32 && r < valid_rows; ++r) {
      const uint32_t w = *reinterpret_cast<const uint32_t*>(boxp + r * 128 + ((chunk ^ (r & 7)) << 4));
      const float a = __uint_as_float(w << 16), b = __uint_as_float(w & 0xffff0000u);
      cs.s0 += a;
      cs.s1 += b;
      cs.q0 += a * a;
      cs.q1 += b * b;
    }
  }
}
// end of the CTA: combine the four row strips of every column pair and write this CTA's partial row [2*64]
__device__ __forceinline__ void colstat_flush(const ColStat& cs, float* red, int e, float* dst_row) {
  red[e * 4 + 0] = cs.s0;
  red[e * 4 + 1] = cs.s1;
  red[e * 4 + 2] = cs.q0;
  red[e * 4 + 3] = cs.q1;
  asm volatile("bar.sync 1, 128;" ::: "memory");
  if (e < 32) {
    float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll
    for (int t2 = 0; t2 < 4; ++t2) {
      s0 += red[(t2 * 32 + e) * 4 + 0];
      s1 += red[(t2 * 32 + e) * 4 + 1];
      q0 += red[(t2 * 32 + e) * 4 + 2];
      q1 += red[(t2 * 32 + e) * 4 + 3];
    }
    dst_row[2 * e] = s0;
    dst_row[2 * e + 1] = s1;
    dst_row[64 + 2 * e] = q0;
    dst_row[64 + 2 * e + 1] = q1;
  }
}

template <int STAGES>
__global__ void __launch_bounds__(192, 1)
conv3x3_c64_kernel(const __grid_constant__ CUtensorMap mA, const __grid_constant__ CUtensorMap mB,
                   const __grid_constant__ CUtensorMap mO, const ConvKwParams p) {
  typedef SmemPlanKw<STAGES> SP;
  constexpr int BN = 64;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* bres = smem + STAGES * AKW_BYTES;
  uint8_t* out_stage = smem + SP::OUT_OFF;
  uint64_t* full = (uint64_t*)(smem + SP::BAR_OFF);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* bfull = tempty + 2;
  uint32_t* tmem_slot = (uint32_t*)(bfull + 1);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr uint32_t TMEM_COLS = 128;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 128);
    }
    mbar_init(bfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // everything above touched shared / tensor memory only
  pdl_trigger();
  const int num_tiles = p.tiles_w * p.tiles_h * p.tiles_n;

  if (warp == 0) {
    if (elect_one()) {
      // resident weights: nine [64 x 64] tiles (k_chunks == 1)
      mbar_expect_tx(bfull, SP::BRES_BYTES);
      for (int g = 0; g < 3; ++g)
        for (int j = 0; j < 3; ++j) tma_load_2d(&mB, bres + (g * 3 + j) * (BN * 128), bfull, p.koff[g][j], 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int w0 = (tile % p.tiles_w) * 8;
        const int h0 = ((tile / p.tiles_w) % p.tiles_h) * p.TH;
        const int n0 = (tile / (p.tiles_w * p.tiles_h)) * p.TN;
        for (int g = 0; g < 3; ++g) {
          mbar_wait(&empty[stage], phase ^ 1);
          mbar_expect_tx(&full[stage], AKW_BYTES);
          tma_load_4d(&mA, smem + stage * AKW_BYTES, &full[stage], 0, w0 - 1, h0 + p.row_dh[g], n0);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    mbar_wait(bfull, 0);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tempty[acc], acc_phase ^ 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t tmem_d = tmem_base + acc * BN;
      for (int g = 0; g < 3; ++g) {
        mbar_wait(&full[stage], phase);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + stage * AKW_BYTES);
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            const uint64_t ad = umma_desc_k_sw128_sbo(sa + p.shift[g][j] * 128, 1280);
            const uint64_t bd = umma_desc_k_sw128(smem_u32(bres + (g * 3 + j) * (BN * 128)));
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              umma_bf16(tmem_d, ad + (uint64_t)(kk * 2), bd + (uint64_t)(kk * 2), idesc, (g | j | kk) != 0);
          }
          umma_commit(&empty[stage]);
          if (g == 2) umma_commit(&tfull[acc]);
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else {
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const bool issuer = (threadIdx.x == 64);
    const int e = threadIdx.x - 64;
    float* red = reinterpret_cast<float*>(smem + SP::RED_OFF);
    float* bias_s = red + 512;   // 64 per-channel constants (zeros without a bias): broadcast LDS.128 instead of 64 LDG per tile
    if (e < 64) bias_s[e] = p.bias ? __ldg(p.bias + e) : 0.f;
    asm volatile("bar.sync 1, 128;" ::: "memory");
    ColStat cs;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int w0 = (tile % p.tiles_w) * 8;
      const int h0 = ((tile / p.tiles_w) % p.tiles_h) * p.TH;
      const int n0 = (tile / (p.tiles_w * p.tiles_h)) * p.TN;
      mbar_wait(&tfull[acc], acc_phase);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN;
#pragma unroll 1
      for (int ch = 0; ch < BN / 32; ++ch) {
        uint32_t r[32];
        tmem_ld32(taddr + ch * 32, r);
        uint8_t* rowp = out_stage + row * 128;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 b0 = *reinterpret_cast<const float4*>(bias_s + ch * 32 + j * 8);
          const float4 b1 = *reinterpret_cast<const float4*>(bias_s + ch * 32 + j * 8 + 4);
          const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
          uint32_t pk[4];
#pragma unroll
          for (int e2 = 0; e2 < 4; ++e2) {
            float a = __uint_as_float(r[j * 8 + e2 * 2]) + bb[e2 * 2];
            float b = __uint_as_float(r[j * 8 + e2 * 2 + 1]) + bb[e2 * 2 + 1];
            if (p.relu) {
              a = fmaxf(a, 0.f);
              b = fmaxf(b, 0.f);
            }
            __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
            pk[e2] = *reinterpret_cast<uint32_t*>(&h);
          }
          const int chunk16 = (ch & 1) * 4 + j;
          *reinterpret_cast<uint4*>(rowp + ((chunk16 ^ (row & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      mbar_arrive(&tempty[acc]);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (issuer) {
        tma_store_4d(&mO, out_stage, 0, w0, h0, n0);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
      if (p.stat_partial) {
        int nvalid = p.valid_n - n0;
        nvalid = nvalid < 0 ? 0 : (nvalid > p.TN ? p.TN : nvalid);
        colstat_accumulate(cs, out_stage, e, nvalid * p.TH * 8);
      }
    }
    if (p.stat_partial) colstat_flush(cs, red, e, p.stat_partial + (int64_t)blockIdx.x * 2 * p.stat_C);
    if (issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------- 3x3/s1, shared activation rows, CTA pair
// The 128-channel layers (N tile = 128) need 24 KB of operands per 256 tensor cycles with one TMA box per tap -- 96 B/clk
// against the ~68 B/clk an SM ingests (measured: layer-2 GEMMs at 48 % tensor-pipe, 66 us for the 72.5 GFLOP the 256-wide
// layers do in 52).  This variant is conv_gemm_kernel<.., PAIR> with conv3x3_c64_kernel's operand scheme: ONE activation box
// per kernel ROW and 64-channel chunk ({64 ch, 8+2 columns, TH, TN} = 160 rows of 128 B) feeds the three kw taps through
// UMMA descriptors started 0/1/2 rows into it (8-pixel-wide tiles: one 8-row core-matrix group per image row, groups
// 1280 B apart), so a stage is 20 KB of A + 3 x 8 KB of B for 3 x 256 tensor cycles = 57 B/clk.
// Epilogue: per-channel constants from shared memory (broadcast LDS.128); BatchNorm statistics in 16 registers per thread
// (one 16-byte chunk of 8 channels x 16 rows of the staged bf16 tile per thread and tile), combined once per CTA.
struct ConvRowParams {
  int TH, TN, tiles_w, tiles_h, tiles_n;   // 128-position tile = TN x TH x 8
  int n_tiles_n, k_chunks;                 // N tiles of BN output channels; 64-channel K chunks
  int row_dh[3];                           // spatial row offset of kernel-row group g
  int shift[3][3];                         // row shift (0..2) into the 10-wide box for tap j of group g
  int koff[3][3];                          // K offset of that tap's chunk 0 in the packed weight matrix
  const float* bias;
  int relu;
  float* stat_partial;
  int stat_C;
  int valid_n;
};
template <int BN, int STAGES>
struct SmemPlanRow {
  static constexpr int B_TAP = (BN / 2) * 128;                 // this CTA's half of one tap's weight tile
  static constexpr int STAGE_BYTES = AKW_BYTES + 3 * B_TAP;    // 20 KB + 3 x 8 KB
  static constexpr int OUT_OFF = STAGES * STAGE_BYTES;
  static constexpr int OUT_BYTES = (BN / 64) * A_BYTES;
  static constexpr int BAR_OFF = OUT_OFF + OUT_BYTES;
  static constexpr int BIAS_OFF = BAR_OFF + 256;               // BN floats
  static constexpr int RED_OFF = BIAS_OFF + BN * 4;            // 128 threads x 16 floats
  static constexpr int CSTAT_OFF = RED_OFF + 128 * 16 * 4;     // [2][Co <= 512] floats
  static constexpr int TOTAL = CSTAT_OFF + 4096 + 1024;
};

template <int BN, int STAGES>
__global__ void __launch_bounds__(192, 1)
conv_row_kernel(const __grid_constant__ CUtensorMap mA, const __grid_constant__ CUtensorMap mB,
                const __grid_constant__ CUtensorMap mO, const ConvRowParams p) {
  static_assert(BN == 128 || BN == 64, "N tile of the shared-row kernel");
  // statistics mapping: CH 16-byte chunks (8 channels) per staged row, RG groups of RPG rows; thread e -> chunk e % CH, group e / CH
  constexpr int CH = BN / 8, RG = 128 / CH, RPG = 128 / RG;
  typedef SmemPlanRow<BN, STAGES> SP;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* out_stage = smem + SP::OUT_OFF;
  uint64_t* full = (uint64_t*)(smem + SP::BAR_OFF);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = (uint32_t*)(tempty + 2);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr uint32_t TMEM_COLS = 2 * BN;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 256);   // the epilogue threads of both CTAs arrive on the leader's
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  cluster_sync_all();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // everything above touched shared / tensor memory only
  pdl_trigger();

  const int tiles_m = p.tiles_w * p.tiles_h * p.tiles_n;
  const int k_iters = 3 * p.k_chunks;
  const uint32_t crank = cluster_ctarank();
  const int walk0 = (int)(blockIdx.x >> 1);
  const int walk_step = (int)(gridDim.x >> 1);
  const int num_tiles = ((tiles_m + 1) / 2) * p.n_tiles_n;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = walk0; tile < num_tiles; tile += walk_step) {
        const int n_tile = tile % p.n_tiles_n;
        const int m_tile = 2 * (tile / p.n_tiles_n) + (int)crank;   // (odd tiles_m: one past the end = past the batch, zero-filled)
        const int w0 = (m_tile % p.tiles_w) * 8;
        const int h0 = ((m_tile / p.tiles_w) % p.tiles_h) * p.TH;
        const int n0 = (m_tile / (p.tiles_w * p.tiles_h)) * p.TN;
        for (int kc = 0; kc < p.k_chunks; ++kc) {
          for (int g = 0; g < 3; ++g) {
            mbar_wait(&empty[stage], phase ^ 1);
            uint8_t* sa = smem + stage * SP::STAGE_BYTES;
            if (crank == 0) mbar_expect_tx(&full[stage], 2 * SP::STAGE_BYTES);
            const uint32_t lead_full = mapa_u32(smem_u32(&full[stage]), 0);
            tma_load_4d_pair(&mA, sa, lead_full, kc * 64, w0 - 1, h0 + p.row_dh[g], n0);
#pragma unroll
            for (int j = 0; j < 3; ++j)
              tma_load_2d_pair(&mB, sa + AKW_BYTES + j * SP::B_TAP, lead_full, p.koff[g][j] + kc * 64,
                               n_tile * BN + (int)crank * (BN / 2));
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = walk0; tile < num_tiles && crank == 0; tile += walk_step, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tempty[acc], acc_phase ^ 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t tmem_d = tmem_base + acc * BN;
      int g = 0;
      for (int k = 0; k < k_iters; ++k) {
        mbar_wait(&full[stage], phase);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + stage * SP::STAGE_BYTES);
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            const uint64_t ad = umma_desc_k_sw128_sbo(sa + p.shift[g][j] * 128, 1280);
            const uint64_t bd = umma_desc_k_sw128(sa + AKW_BYTES + j * SP::B_TAP);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              umma_bf16_pair(tmem_d, ad + (uint64_t)(kk * 2), bd + (uint64_t)(kk * 2), idesc, (k | j | kk) != 0);
          }
          umma_commit_pair(&empty[stage]);
          if (k == k_iters - 1) umma_commit_pair(&tfull[acc]);
        }
        __syncwarp();
        if (++g == 3) g = 0;
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else {
    // ===================== epilogue (warps 2..5 -> TMEM lane quarters 2,3,0,1) =====================
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const bool issuer = (threadIdx.x == 64);
    const int e = threadIdx.x - 64;
    float* bias_s = reinterpret_cast<float*>(smem + SP::BIAS_OFF);
    float* red = reinterpret_cast<float*>(smem + SP::RED_OFF);
    float* cstat = reinterpret_cast<float*>(smem + SP::CSTAT_OFF);
    const bool stats = p.stat_partial != nullptr;
    if (stats)
      for (int i = e; i < 2 * p.stat_C; i += 128) cstat[i] = 0.f;
    // statistics: thread e owns the 16-byte chunk (8 channels) `cidx` of the RPG staged rows [RPG*rg, RPG*rg + RPG)
    const int cidx = e % CH, rg = e / CH;
    float as[8], aq[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) as[i] = aq[i] = 0.f;
    int cur_nt = -1;
    // fixed-order combination of the eight row groups of every channel, added to this CTA's running row
    auto flush = [&](int nt) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        red[e * 16 + i] = as[i];
        red[e * 16 + 8 + i] = aq[i];
        as[i] = aq[i] = 0.f;
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (e < BN) {   // column e: the RG row groups in order
        float s = 0.f, q2 = 0.f;
#pragma unroll
        for (int r2 = 0; r2 < RG; ++r2) {
          s += red[(r2 * CH + (e >> 3)) * 16 + (e & 7)];
          q2 += red[(r2 * CH + (e >> 3)) * 16 + 8 + (e & 7)];
        }
        cstat[nt * BN + e] += s;
        cstat[p.stat_C + nt * BN + e] += q2;
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
    };
    int it = 0;
    for (int tile = walk0; tile < num_tiles; tile += walk_step, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int n_tile = tile % p.n_tiles_n;
      const int m_tile = 2 * (tile / p.n_tiles_n) + (int)crank;
      const int w0 = (m_tile % p.tiles_w) * 8;
      const int h0 = ((m_tile / p.tiles_w) % p.tiles_h) * p.TH;
      const int n0 = (m_tile / (p.tiles_w * p.tiles_h)) * p.TN;
      if (n_tile != cur_nt) {   // (uniform over the CTA)
        if (stats && cur_nt >= 0) flush(cur_nt);
        asm volatile("bar.sync 1, 128;" ::: "memory");   // the previous tile's reads of bias_s are done
        if (e < BN) bias_s[e] = p.bias ? __ldg(p.bias + n_tile * BN + e) : 0.f;
        cur_nt = n_tile;
      }
      mbar_wait(&tfull[acc], acc_phase);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // staging buffer free again
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN;
#pragma unroll 1
      for (int ch = 0; ch < BN / 32; ++ch) {
        uint32_t r[32];
        tmem_ld32(taddr + ch * 32, r);
        uint8_t* rowp = out_stage + (ch >> 1) * A_BYTES + row * 128;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 b0 = *reinterpret_cast<const float4*>(bias_s + ch * 32 + j * 8);
          const float4 b1 = *reinterpret_cast<const float4*>(bias_s + ch * 32 + j * 8 + 4);
          const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
          uint32_t pk[4];
#pragma unroll
          for (int e2 = 0; e2 < 4; ++e2) {
            float a = __uint_as_float(r[j * 8 + e2 * 2]) + bb[e2 * 2];
            float b = __uint_as_float(r[j * 8 + e2 * 2 + 1]) + bb[e2 * 2 + 1];
            if (p.relu) {
              a = fmaxf(a, 0.f);
              b = fmaxf(b, 0.f);
            }
            __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
            pk[e2] = *reinterpret_cast<uint32_t*>(&h);
          }
          const int chunk16 = (ch & 1) * 4 + j;
          *reinterpret_cast<uint4*>(rowp + ((chunk16 ^ (row & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      mbar_arrive_cluster(mapa_u32(smem_u32(&tempty[acc]), 0));   // on the leader's barrier (256 arrivals per phase)
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (issuer) {
#pragma unroll
        for (int b = 0; b < BN / 64; ++b) tma_store_4d(&mO, out_stage + b * A_BYTES, n_tile * BN + b * 64, w0, h0, n0);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
      if (stats && m_tile < tiles_m) {
        int nvalid = p.valid_n - n0;
        nvalid = nvalid < 0 ? 0 : (nvalid > p.TN ? p.TN : nvalid);
        const int valid_rows = nvalid * p.TH * 8;
        const uint8_t* boxp = out_stage + (cidx >> 3) * A_BYTES;
        const int chunk = cidx & 7;
        if (valid_rows >= rg * RPG + RPG) {
          uint4 w[RPG];
#pragma unroll
          for (int i = 0; i < RPG; ++i) {
            const int r2 = rg * RPG + i;
            w[i] = *reinterpret_cast<const uint4*>(boxp + r2 * 128 + ((chunk ^ (r2 & 7)) << 4));
          }
#pragma unroll
          for (int i = 0; i < RPG; ++i) {
            const uint32_t ww[4] = {w[i].x, w[i].y, w[i].z, w[i].w};
#pragma unroll
            for (int t2 = 0; t2 < 4; ++t2) {
              const float a = __uint_as_float(ww[t2] << 16), b = __uint_as_float(ww[t2] & 0xffff0000u);
              as[2 * t2] += a;
              as[2 * t2 + 1] += b;
              aq[2 * t2] += a * a;
              aq[2 * t2 + 1] += b * b;
            }
          }
        } else {
          for (int r2 = rg * RPG; r2 < rg * RPG + RPG && r2 < valid_rows; ++r2) {
            const uint4 w = *reinterpret_cast<const uint4*>(boxp + r2 * 128 + ((chunk ^ (r2 & 7)) << 4));
            const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int t2 = 0; t2 < 4; ++t2) {
              const float a = __uint_as_float(ww[t2] << 16), b = __uint_as_float(ww[t2] & 0xffff0000u);
              as[2 * t2] += a;
              as[2 * t2 + 1] += b;
              aq[2 * t2] += a * a;
              aq[2 * t2 + 1] += b * b;
            }
          }
        }
      }
    }
    if (stats) {
      if (cur_nt >= 0) flush(cur_nt);
      asm volatile("bar.sync 1, 128;" ::: "memory");
      float* dst = p.stat_partial + (int64_t)blockIdx.x * 2 * p.stat_C;
      for (int i = e; i < 2 * p.stat_C; i += 128) dst[i] = cstat[i];
    }
    if (issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncwarp();
  cluster_sync_all();   // the peer's smem / TMEM are operands of the leader's MMAs until both CTAs are done
  if (warp == 1)
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
}

__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes);

// ------------------------------------------------------------------------------------------- stem 7x7/s2 (C_in <= 4)
// The stem as an implicit GEMM straight from a zero-padded NHWC4 bf16 copy of the image ([B][H+6][W+8][4]):
// for output pixel (oh, ow) and kernel row kh, the 8 pixels x 4 channels = 32 bf16 = 64 contiguous bytes starting at
// padded pixel (2*oh + kh, 2*ow) are exactly that tap row of the im2col matrix (first pixel and 4th channel carry zero
// weights).  A tensor map whose W-stride is 16 B (overlapping 64-byte windows; accepted by cuTensorMapEncodeTiled and
// verified on the B200) therefore lets TMA build the A operand with NO column tensor: 7 boxes {32, TW, TH, TN} per tile,
// K = 7 x 32.  64-byte rows -> SWIZZLE_64B operands (8-row groups 512 B apart).  Weights (28 KB) stay resident.
struct StemParams {
  int TW, TH, TN, tiles_w, tiles_h, tiles_n;
  const float* bias;
  float* stat_partial;
  int stat_C;
  int valid_n;
};
// CH = layout code of the padded image (lbc_fast.h: stem_ch): 4 = camera RGB, 8 = the 7-channel bird's-eye view -- one kernel
// row of one output pixel is 8 px x CH ch = 64 or 128 contiguous bytes (SWIZZLE_64B / SWIZZLE_128B operands), 7 rows;
// 16 = RGB space-to-depth -- one kernel ROW PAIR is 4 blocks x 16 = 64 elements = 128 bytes, 4 rows (K = 256 instead of 224,
// but 4 x 128 TMA row requests per tile instead of 7 x 128: these kernels are bound by TMA rows, not by the tensor pipe)
template <int CH>
struct StemGeom {
  static constexpr int ROWB = CH == 4 ? 64 : 128;  // bytes of one window row
  static constexpr int A_BYTES_ = 128 * ROWB;      // one A box: 128 output pixels
  static constexpr int KROW = ROWB / 2;            // K elements per window row
  static constexpr int NROWS = CH == 16 ? 4 : 7;   // window rows per output pixel
};
constexpr int ASTEM_BYTES = 128 * 64;

template <int STAGES, int CH = 4>
struct SmemPlanStem {
  static constexpr int BRES_BYTES = StemGeom<CH>::NROWS * 64 * StemGeom<CH>::ROWB;
  static constexpr int OUT_OFF = STAGES * StemGeom<CH>::A_BYTES_ + BRES_BYTES;
  static constexpr int BAR_OFF = OUT_OFF + A_BYTES;
  static constexpr int RED_OFF = BAR_OFF + 256;
  static constexpr int TOTAL = RED_OFF + 2048 + 256 + 1024;
};
__device__ __forceinline__ uint64_t umma_desc_k_sw64(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512 >> 4) << 32;   // 8 rows x 64 B
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;            // SWIZZLE_64B
  return d;
}

template <int STAGES, int CH>
__global__ void __launch_bounds__(192, CH == 8 ? 1 : 2)
stem_conv_kernel(const __grid_constant__ CUtensorMap mX0, const __grid_constant__ CUtensorMap mX1,
                 const __grid_constant__ CUtensorMap mB, const __grid_constant__ CUtensorMap mO, const StemParams p) {
  typedef SmemPlanStem<STAGES, CH> SP;
  constexpr int ASTEM_BYTES = StemGeom<CH>::A_BYTES_;   // (shadows the 4-channel constant)
  constexpr int WROW_BYTES = 64 * StemGeom<CH>::ROWB;   // weights of one kernel row: 64 output channels
  constexpr int NROWS = StemGeom<CH>::NROWS;
  constexpr int BN = 64;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* bres = smem + STAGES * ASTEM_BYTES;
  uint8_t* out_stage = smem + SP::OUT_OFF;
  uint64_t* full = (uint64_t*)(smem + SP::BAR_OFF);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* bfull = tempty + 2;
  uint32_t* tmem_slot = (uint32_t*)(bfull + 1);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr uint32_t TMEM_COLS = 128;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 128);
    }
    mbar_init(bfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // everything above touched shared / tensor memory only
  pdl_trigger();
  const int num_tiles = p.tiles_w * p.tiles_h * p.tiles_n;

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(bfull, SP::BRES_BYTES);
      for (int kh = 0; kh < NROWS; ++kh) tma_load_2d(&mB, bres + kh * WROW_BYTES, bfull, kh * StemGeom<CH>::KROW, 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int w0 = (tile % p.tiles_w) * p.TW;
        const int h0 = ((tile / p.tiles_w) % p.tiles_h) * p.TH;
        const int n0 = (tile / (p.tiles_w * p.tiles_h)) * p.TN;
        for (int kh = 0; kh < NROWS; ++kh) {
          mbar_wait(&empty[stage], phase ^ 1);
          mbar_expect_tx(&full[stage], ASTEM_BYTES);
          if (CH == 16)   // space-to-depth: row pair kh of the window = block row h0 + kh
            tma_load_4d(&mX0, smem + stage * ASTEM_BYTES, &full[stage], 0, w0, h0 + kh, n0);
          else            // even / odd padded rows through their own maps
            tma_load_4d((kh & 1) ? &mX1 : &mX0, smem + stage * ASTEM_BYTES, &full[stage], 0, w0, h0 + (kh >> 1), n0);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    mbar_wait(bfull, 0);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tempty[acc], acc_phase ^ 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t tmem_d = tmem_base + acc * BN;
      for (int kh = 0; kh < NROWS; ++kh) {
        mbar_wait(&full[stage], phase);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (elect_one()) {
          const uint32_t aaddr = smem_u32(smem + stage * ASTEM_BYTES), baddr = smem_u32(bres + kh * WROW_BYTES);
          const uint64_t ad = CH == 4 ? umma_desc_k_sw64(aaddr) : umma_desc_k_sw128(aaddr);
          const uint64_t bd = CH == 4 ? umma_desc_k_sw64(baddr) : umma_desc_k_sw128(baddr);
#pragma unroll
          for (int kk = 0; kk < StemGeom<CH>::KROW / 16; ++kk)
            umma_bf16(tmem_d, ad + (uint64_t)(kk * 2), bd + (uint64_t)(kk * 2), idesc, (kh | kk) != 0);
          umma_commit(&empty[stage]);
          if (kh == NROWS - 1) umma_commit(&tfull[acc]);
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else {
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const bool issuer = (threadIdx.x == 64);
    const int e = threadIdx.x - 64;
    float* red = reinterpret_cast<float*>(smem + SP::RED_OFF);
    float* bias_s = red + 512;
    if (e < 64) bias_s[e] = p.bias ? __ldg(p.bias + e) : 0.f;
    asm volatile("bar.sync 1, 128;" ::: "memory");
    ColStat cs;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int w0 = (tile % p.tiles_w) * p.TW;
      const int h0 = ((tile / p.tiles_w) % p.tiles_h) * p.TH;
      const int n0 = (tile / (p.tiles_w * p.tiles_h)) * p.TN;
      mbar_wait(&tfull[acc], acc_phase);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN;
#pragma unroll 1
      for (int ch = 0; ch < BN / 32; ++ch) {
        uint32_t r[32];
        tmem_ld32(taddr + ch * 32, r);
        uint8_t* rowp = out_stage + row * 128;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 b0 = *reinterpret_cast<const float4*>(bias_s + ch * 32 + j * 8);
          const float4 b1 = *reinterpret_cast<const float4*>(bias_s + ch * 32 + j * 8 + 4);
          const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
          uint32_t pk[4];
#pragma unroll
          for (int e2 = 0; e2 < 4; ++e2) {
            const float a = __uint_as_float(r[j * 8 + e2 * 2]) + bb[e2 * 2];
            const float b = __uint_as_float(r[j * 8 + e2 * 2 + 1]) + bb[e2 * 2 + 1];
            __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
            pk[e2] = *reinterpret_cast<uint32_t*>(&h);
          }
          const int chunk16 = (ch & 1) * 4 + j;
          *reinterpret_cast<uint4*>(rowp + ((chunk16 ^ (row & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      mbar_arrive(&tempty[acc]);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (issuer) {
        tma_store_4d(&mO, out_stage, 0, w0, h0, n0);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
      if (p.stat_partial) {
        int nvalid = p.valid_n - n0;
        nvalid = nvalid < 0 ? 0 : (nvalid > p.TN ? p.TN : nvalid);
        colstat_accumulate(cs, out_stage, e, nvalid * p.TH * p.TW);
      }
    }
    if (p.stat_partial) colstat_flush(cs, red, e, p.stat_partial + (int64_t)blockIdx.x * 2 * p.stat_C);
    if (issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// Stem weight gradient from the same padded image: D[(kh, e)][co] = sum_pixels x4win[pix, kh][e] * dy[pix][co];
// M tile = 4 kernel rows x 32 window elements (two M tiles cover kh 0..7, row 7 unused), N = 64, K = pixels.
// A: four {32, TW, TH, TN} boxes (MN-major, SWIZZLE_64B, blocks 8 KB apart); B: one dy box (MN-major, SWIZZLE_128B).
struct StemWgradParams {
  int TW, TH, TN, tiles_w, tiles_h, tiles_n;
  int k_tiles, k_per_split, splits;
  int C;           // real input channels (<= 4)
  float* dw_ref;   // [splits][64][C][7][7] fp32 partials: every element stored once per split (summed in split order)
};
__device__ __forceinline__ uint64_t umma_desc_mn_sw64(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;   // distance between 32-element MN blocks
  d |= (uint64_t)(512 >> 4) << 32;                    // 8 K rows x 64 B
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;
  return d;
}
template <int STAGES, int CH>
__global__ void __launch_bounds__(192, 1)
stem_wgrad_kernel(const __grid_constant__ CUtensorMap mDY, const __grid_constant__ CUtensorMap mX0,
                  const __grid_constant__ CUtensorMap mX1, const StemWgradParams p) {
  constexpr int ASTEM_BYTES = StemGeom<CH>::A_BYTES_;
  constexpr int KROW = StemGeom<CH>::KROW;         // window elements of one kernel row = M rows it contributes
  constexpr int NROWS = StemGeom<CH>::NROWS;
  constexpr int RPT = 128 / KROW;                  // kernel rows per 128-row M tile (4 or 2)
  constexpr int A_ST = RPT * ASTEM_BYTES, STAGE_BYTES = A_ST + A_BYTES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(smem + STAGES * STAGE_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint32_t* tmem_slot = (uint32_t*)(tfull + 1);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr uint32_t TMEM_COLS = 64;
  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(tfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // everything above touched shared / tensor memory only
  pdl_trigger();
  constexpr int MT = (NROWS + RPT - 1) / RPT;   // M tiles covering the window rows (7 rows: row 7 does not exist)
  const int mt = blockIdx.x % MT;          // kernel rows RPT*mt .. RPT*mt+RPT-1
  const int split = blockIdx.x / MT;
  const int kt0 = split * p.k_per_split;
  int kt1 = kt0 + p.k_per_split;
  if (kt1 > p.k_tiles) kt1 = p.k_tiles;
  const int n_k = kt1 - kt0;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kt = kt0; kt < kt1; ++kt) {
        const int w0 = (kt % p.tiles_w) * p.TW;
        const int h0 = ((kt / p.tiles_w) % p.tiles_h) * p.TH;
        const int n0 = (kt / (p.tiles_w * p.tiles_h)) * p.TN;
        mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* sa = smem + stage * STAGE_BYTES;
        mbar_expect_tx(&full[stage], STAGE_BYTES);
#pragma unroll
        for (int j = 0; j < RPT; ++j) {
          int kh = mt * RPT + j;
          if (kh > NROWS - 1) kh = NROWS - 1;   // row 7 does not exist: load a valid duplicate, its output rows are skipped
          if (CH == 16)
            tma_load_4d(&mX0, sa + j * ASTEM_BYTES, &full[stage], 0, w0, h0 + kh, n0);
          else
            tma_load_4d((kh & 1) ? &mX1 : &mX0, sa + j * ASTEM_BYTES, &full[stage], 0, w0, h0 + (kh >> 1), n0);
        }
        tma_load_4d(&mDY, sa + A_ST, &full[stage], 0, w0, h0, n0);
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(64 >> 3) << 17) |
                           ((uint32_t)(128 >> 4) << 24);
    int stage = 0;
    uint32_t phase = 0;
    for (int k = 0; k < n_k; ++k) {
      mbar_wait(&full[stage], phase);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (elect_one()) {
        const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
        const uint64_t ad = CH == 4 ? umma_desc_mn_sw64(sa, ASTEM_BYTES) : umma_desc_mn_sw128(sa, ASTEM_BYTES);
        const uint64_t bd = umma_desc_mn_sw128(sa + A_ST, A_BYTES);
        constexpr int A_STEP = 16 * StemGeom<CH>::ROWB;   // 16 pixels per MMA: two 8-row groups of the A rows (64 / 128 B each)
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)   // B: two 8-row groups of 128-byte rows = 2048 B
          umma_bf16(tmem_base, ad + (uint64_t)(kk * (A_STEP >> 4)), bd + (uint64_t)(kk * (2048 >> 4)), idesc, (k | kk) != 0);
        umma_commit(&empty[stage]);
        if (k == n_k - 1) umma_commit(tfull);
      }
      __syncwarp();
      if (++stage == STAGES) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (n_k > 0) {
    const int q = warp & 3;
    const int m = q * 32 + lane;
    const int wr = mt * RPT + m / KROW;   // window row
    const int e = m % KROW;
    // CH = 16: e = [column pair 4][row parity][column parity][4 ch] of row pair wr
    const int kh = CH == 16 ? 2 * wr + ((e >> 3) & 1) : wr;
    const int kwp = CH == 16 ? 2 * (e >> 4) + ((e >> 2) & 1) : e / CH;
    const int c = CH == 16 ? (e & 3) : e % CH;
    mbar_wait(tfull, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
    for (int ch = 0; ch < 2; ++ch) {
      uint32_t r[32];
      tmem_ld32(taddr + ch * 32, r);
      if (kh < 7 && kwp >= 1 && c < p.C) {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int co = ch * 32 + j;
          p.dw_ref[(int64_t)split * 64 * p.C * 49 + (((int64_t)co * p.C + c) * 7 + kh) * 7 + (kwp - 1)] = __uint_as_float(r[j]);
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------- host side
static int sm_count() {
  static int n = [] {
    int dev = 0, v = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v > 0 ? v : 148;
  }();
  return n;
}

static int pow2_divisor(int x, int cap) {
  int p = 1;
  while (p * 2 <= cap && x % (p * 2) == 0) p *= 2;
  return p;
}
// 128-position tile {TW, TH, TN} for an (OH x OW) output plane; false when the plane has no power-of-two factors
static bool tile_geometry(int OH, int OW, int B, ConvGemmParams& p) {
  int TW = pow2_divisor(OW, 32);
  int TH = pow2_divisor(OH, 128 / TW);
  int TN = 128 / (TW * TH);
  p.TW = TW;
  p.TH = TH;
  p.TN = TN;
  p.tiles_w = OW / TW;
  p.tiles_h = OH / TH;
  p.tiles_n = (B + TN - 1) / TN;
  return TN <= 256;
}

template <int BN, int STAGES, bool OUT_F32 = false>
static int launch_gemm(const CUtensorMap* mA, const CUtensorMap& mB, const CUtensorMap& mO, const ConvGemmParams& p,
                        lbc_stream_t s) {
  typedef SmemPlan<BN, STAGES, false, OUT_F32> SP;
  static bool configured = false;
  if (!configured) {
    LBC_CUDA(cudaFuncSetAttribute(conv_gemm_kernel<BN, STAGES, false, OUT_F32>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  SP::TOTAL));
    configured = true;
  }
  int tiles = p.tiles_w * p.tiles_h * p.tiles_n * p.n_tiles_n;
  int grid = tiles < sm_count() ? tiles : sm_count();
  { auto k_ = conv_gemm_kernel<BN, STAGES, false, OUT_F32>; LBC_LAUNCH(k_, dim3(grid), dim3(192), SP::TOTAL, s, mA[0], mA[1], mA[2], mA[3], mB, mO, p); }
  if (OUT_F32)
    LBC_LAUNCHED((BN == 64 ? "conv_gemm_kernel<64,f32>" : BN == 128 ? "conv_gemm_kernel<128,f32>" : "conv_gemm_kernel<256,f32>"));
  else
    LBC_LAUNCHED((BN == 64 ? "conv_gemm_kernel<64>" : BN == 128 ? "conv_gemm_kernel<128>" : "conv_gemm_kernel<256>"));
  LBC_CUDA(cudaGetLastError());
  return grid;
}
// CTA-pair variant: clusters of 2 (one TPC), persistent over ceil(tiles_m/2) * n_tiles_n pair tiles
template <int BN, int STAGES, bool OUT_F32 = false>
static int launch_gemm_pair(const CUtensorMap* mA, const CUtensorMap& mBhalf, const CUtensorMap& mO, const ConvGemmParams& p,
                             lbc_stream_t s) {
  typedef SmemPlan<BN, STAGES, true, OUT_F32> SP;
  static_assert(SP::TOTAL <= 232448, "smem plan of the CTA-pair kernel exceeds 227 KB");
  auto kern = conv_gemm_kernel<BN, STAGES, true, OUT_F32>;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.blockDim = dim3(192, 1, 1);
  cfg.dynamicSmemBytes = SP::TOTAL;
  cfg.stream = (cudaStream_t)s;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  static int max_clusters = 0;
  if (max_clusters == 0) {
    LBC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SP::TOTAL));
    cfg.gridDim = dim3((unsigned)(sm_count() / 2 * 2), 1, 1);
    int n = 0;
    // co-resident clusters (a GPC with an unpaired SM cannot host one): a persistent grid must not exceed it
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n <= 0) {
      cudaGetLastError();
      n = sm_count() / 2;
    }
    max_clusters = n < sm_count() / 2 ? n : sm_count() / 2;
  }
  const int tiles_m = p.tiles_w * p.tiles_h * p.tiles_n;
  const int pair_tiles = ((tiles_m + 1) / 2) * p.n_tiles_n;
  const int clusters = pair_tiles < max_clusters ? pair_tiles : max_clusters;
  LBC_LAUNCH_CLUSTER(kern, 2, dim3((unsigned)(2 * clusters)), dim3(192), SP::TOTAL, (cudaStream_t)s, mA[0], mA[1], mA[2], mA[3], mBhalf,
                     mO, p);
  if (OUT_F32)
    LBC_LAUNCHED((BN == 128 ? "conv_gemm_kernel<128,pair,f32>" : "conv_gemm_kernel<256,pair,f32>"));
  else
    LBC_LAUNCHED((BN == 128 ? "conv_gemm_kernel<128,pair>" : "conv_gemm_kernel<256,pair>"));
  LBC_CUDA(cudaGetLastError());
  return 2 * clusters;
}
// kernel variants (LBC_PAIR overrides; tests toggle them through lbc_set_fast_kernels):
//   bit 0: CTA-pair (cta_group::2) kernels for the BN >= 128 conv GEMMs   bit 1: row-of-taps weight gradient
//   bit 2: CTA-pair variant of the row-of-taps weight gradient (Co % 256 == 0)
//   bit 3: space-to-depth operand layout of the RGB stem (lbc_fast.h: stem_ch)
//   bit 6: all-nine-taps weight gradient of the 64 -> 64 3x3 convolutions (try_wgrad9; same-box A/B 12.54 -> 12.30 ms per step,
//   conv_wgrad 2.96 -> 2.86 ms; 30 consecutive bench runs + memcheck clean, tools/gpu_r2_z2.sh)
//   bit 4 / 5: shared-row CTA-pair kernel for the 3x3/s1 convolutions of the 128-channel / 256-channel layers (try_conv_row;
//   same-box A/B at B = 256: 13.79 -> 13.56 -> 13.36 ms per step, profiles/r2_ab_rowk_schedule.md)
// Bits 0-2 validated on the B200 (parity tests green, 16.61 -> 15.87 ms per step at B = 256), hence on by default.
static int g_pair_mode = [] {
  const char* e = getenv("LBC_PAIR");
  return e ? atoi(e) : 127;
}();
void set_pair_mode(int mode) { g_pair_mode = mode; }
int pair_mode() { return g_pair_mode; }
bool stem_s2d() { return (g_pair_mode & 8) != 0; }

// Operand / output format of one implicit GEMM.  Default = the bf16 training step.  fp32tc (parity-grade tensor-core
// mode): operands are [hi | lo] 16-bit planes of fp32 tensors (3 MMAs per K block), the output is stored as fp32.
struct GemmMode {
  bool split = false;
  bool out_f32 = false;
  uint32_t fmt_a = 1, fmt_b = 1;   // UMMA operand formats: 1 = bf16, 0 = fp16
  float out_scale = 1.0f;
};
static void apply_mode(ConvGemmParams& p, const GemmMode& m, int a_plane, int b_plane) {
  p.split = m.split ? 1 : 0;
  p.a_plane = a_plane;
  p.b_plane = b_plane;
  p.fmt_a = m.fmt_a;
  p.fmt_b = m.fmt_b;
  p.out_scale = m.out_scale;
}
// mB: weights [rows][K]; the box height is chosen here (BN rows, or BN/2 for the CTA-pair kernels)
// returns the number of CTAs launched (= rows of statistics partials, when asked for)
static int dispatch_gemm(int BN, const CUtensorMap* mA, const void* wbase, int64_t wK, int64_t wrows, const CUtensorMap& mO,
                          const ConvGemmParams& p, lbc_stream_t s, bool out_f32 = false) {
  const bool pair = (g_pair_mode & 1) && BN >= 128;
  if (pair) {
    CUtensorMap mB = make_map_2d(wbase, wK, wrows, BN / 2);
    if (out_f32) return BN == 128 ? launch_gemm_pair<128, 7, true>(mA, mB, mO, p, s) : launch_gemm_pair<256, 4, true>(mA, mB, mO, p, s);
    return BN == 128 ? launch_gemm_pair<128, 7>(mA, mB, mO, p, s) : launch_gemm_pair<256, 4>(mA, mB, mO, p, s);
  }
  CUtensorMap mB = make_map_2d(wbase, wK, wrows, BN);
  if (out_f32)
    return BN == 64    ? launch_gemm<64, 6, true>(mA, mB, mO, p, s)
           : BN == 128 ? launch_gemm<128, 5, true>(mA, mB, mO, p, s)
                       : launch_gemm<256, 3, true>(mA, mB, mO, p, s);
  return BN == 64 ? launch_gemm<64, 6>(mA, mB, mO, p, s) : BN == 128 ? launch_gemm<128, 5>(mA, mB, mO, p, s) : launch_gemm<256, 3>(mA, mB, mO, p, s);
}
// N tile: 256 where it divides, unless the 128-wide tiling fills the persistent grid's rounds clearly better
// (static round-robin over 148 CTAs: 480 tiles = 3.24 rounds -> 81 %, 960 tiles = 6.49 -> 93 %).
static int pick_bn(int C, int tiles_m = 0) {
  if (C == 64) return 64;
  if (C % 256 != 0) return 128;
  static int policy = [] {
    const char* e = getenv("LBC_BN_POLICY");
    return e ? atoi(e) : 0;   // measured: 256-wide tiles win despite the round quantisation (18.14 vs 18.44 ms/step)
  }();
  if (policy == 0 || tiles_m <= 0) return 256;
  auto eff = [&](int bn) {
    int tiles = tiles_m * (C / bn);
    int rounds = (tiles + sm_count() - 1) / sm_count();
    return (double)tiles / ((double)rounds * sm_count());
  };
  return eff(128) > eff(256) + 0.08 ? 128 : 256;
}

static bool supported(const ConvL& c) {
  if (c.Ci % 64 || c.Co % 64) return false;
  if (!((c.K == 3 && c.pad == 1) || (c.K == 1 && c.pad == 0))) return false;
  if (c.stride == 2) return (c.H % 2 == 0) && (c.W % 2 == 0) && c.OH * 2 == c.H && c.OW * 2 == c.W;
  return c.stride == 1 && c.OH == c.H && c.OW == c.W;
}


// 3x3 / stride 1 / 64 -> 64 channels (forward: mirrored=false, taps (kh-1, kw-1); data gradient: mirrored=true)
static bool g_c64_variant = true;
void set_c64_variant(bool on) { g_c64_variant = on; }
static bool try_conv3x3_c64(const bf16* in, const void* wpack, bf16* out, int B, int H, int W, bool mirrored,
                            const float* bias, bool relu, float* stat_partial, int* stat_rows, lbc_stream_t s) {
  if (!g_c64_variant || (W % 8) != 0) return false;
  if ((g_pair_mode & 129) == 129) return false;   // bit 7 (+ CTA pairs): the shared-row CTA-pair kernel with 64-wide N tiles takes it
  ConvKwParams p;
  memset(&p, 0, sizeof(p));
  int TH = pow2_divisor(H, 16);
  int TN = 16 / TH;
  p.TH = TH;
  p.TN = TN;
  p.tiles_w = W / 8;
  p.tiles_h = H / TH;
  p.tiles_n = (B + TN - 1) / TN;
  p.k_chunks = 1;
  for (int g = 0; g < 3; ++g) {
    // group g covers spatial row offset dh = g - 1; forward: kh = g, data gradient: kh = 2 - g
    p.row_dh[g] = g - 1;
    const int kh = mirrored ? 2 - g : g;
    for (int j = 0; j < 3; ++j) {
      // box column 0 is w0-1, so tap with column offset dw reads rows shifted by dw + 1
      const int kw = j;
      const int dw = mirrored ? 1 - kw : kw - 1;
      p.shift[g][j] = dw + 1;
      p.koff[g][j] = (kh * 3 + kw) * 64;
    }
  }
  p.bias = bias;
  p.relu = relu ? 1 : 0;
  p.stat_partial = stat_partial;
  p.stat_C = 64;
  p.valid_n = B;
  const int tiles_total = p.tiles_w * p.tiles_h * p.tiles_n;
  if (stat_rows) *stat_rows = tiles_total < sm_count() ? tiles_total : sm_count();   // one partial row per persistent CTA
  const int64_t eb = 2;
  CUtensorMap mA = make_map_4d(in, 64, W, H, B, 64 * eb, (int64_t)W * 64 * eb, (int64_t)H * W * 64 * eb, 10, TH, TN);
  CUtensorMap mB = make_map_2d(wpack, (int64_t)9 * 64, 64, 64);
  CUtensorMap mO = make_map_4d(out, 64, W, H, B, 64 * eb, (int64_t)W * 64 * eb, (int64_t)H * W * 64 * eb, 8, TH, TN);
  typedef SmemPlanKw<5> SP;
  static bool configured = false;
  if (!configured) {
    LBC_CUDA(cudaFuncSetAttribute(conv3x3_c64_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, SP::TOTAL));
    configured = true;
  }
  int tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  int grid = tiles < sm_count() ? tiles : sm_count();
  { auto k_ = conv3x3_c64_kernel<5>; LBC_LAUNCH(k_, dim3(grid), dim3(192), SP::TOTAL, s, mA, mB, mO, p); }
  LBC_LAUNCHED("conv3x3_c64_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}


// 3x3 / stride 1 / pad 1 with 128-wide N tiles on the shared-row CTA-pair kernel (forward: mirrored = false; data gradient:
// mirrored = true with the transposed pack).  in [B,H,W,Cin], wpack [Cout][9][Cin], out [B,H,W,Cout]; returns the number of
// CTAs launched (= rows of statistics partials) or 0 when the layer does not fit the kernel.
//   g_pair_mode bit 4: layers with Cout % 256 != 0 (layer 2, the teacher's layer 2)   bit 5: also Cout % 256 == 0 (layer 3)
//   bit 7: the 64-channel layers (layer 1) on the same kernel with 64-wide N tiles instead of conv3x3_c64_kernel
template <int BN, int STAGES>
static int try_conv_row_t(const bf16* in, const void* wpack, bf16* out, int B, int H, int W, int Cin, int Cout, bool mirrored,
                          const float* bias, bool relu, float* stat_partial, lbc_stream_t s) {
  if (!(g_pair_mode & 1)) return 0;
  if (!(g_pair_mode & (BN == 64 ? 128 : (Cout % 256 == 0 ? 32 : 16)))) return 0;
  if ((W % 8) || (Cin % 64) || (Cout % BN) || Cout > 512) return 0;
  ConvRowParams p;
  memset(&p, 0, sizeof(p));
  const int TH = pow2_divisor(H, 16);
  const int TN = 16 / TH;
  p.TH = TH;
  p.TN = TN;
  p.tiles_w = W / 8;
  p.tiles_h = H / TH;
  p.tiles_n = (B + TN - 1) / TN;
  p.n_tiles_n = Cout / BN;
  p.k_chunks = Cin / 64;
  for (int g = 0; g < 3; ++g) {
    p.row_dh[g] = g - 1;                       // group g covers spatial row offset g - 1
    const int kh = mirrored ? 2 - g : g;
    for (int j = 0; j < 3; ++j) {
      const int dw = mirrored ? 1 - j : j - 1;   // column offset of tap kw = j; box column 0 is w0 - 1
      p.shift[g][j] = dw + 1;
      p.koff[g][j] = (kh * 3 + j) * Cin;
    }
  }
  p.bias = bias;
  p.relu = relu ? 1 : 0;
  p.stat_partial = stat_partial;
  p.stat_C = Cout;
  p.valid_n = B;
  const int64_t eb = 2;
  CUtensorMap mA = make_map_4d(in, Cin, W, H, B, Cin * eb, (int64_t)W * Cin * eb, (int64_t)H * W * Cin * eb, 10, TH, TN);
  CUtensorMap mB = make_map_2d(wpack, (int64_t)9 * Cin, Cout, BN / 2);
  CUtensorMap mO = make_map_4d(out, Cout, W, H, B, Cout * eb, (int64_t)W * Cout * eb, (int64_t)H * W * Cout * eb, 8, TH, TN);
  typedef SmemPlanRow<BN, STAGES> SP;
  static_assert(SP::TOTAL <= 232448, "smem plan of the shared-row kernel exceeds 227 KB");
  auto kern = conv_row_kernel<BN, STAGES>;
  static int max_clusters = 0;
  if (max_clusters == 0) {
    LBC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SP::TOTAL));
    LaunchCfg q(dim3((unsigned)(sm_count() / 2 * 2)), dim3(192), SP::TOTAL, (cudaStream_t)s, 2);
    q.cfg.numAttrs = 1;   // (the cluster attribute only)
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &q.cfg) != cudaSuccess || n <= 0) {
      cudaGetLastError();
      n = sm_count() / 2;
    }
    max_clusters = n < sm_count() / 2 ? n : sm_count() / 2;
  }
  const int tiles_m = p.tiles_w * p.tiles_h * p.tiles_n;
  const int pair_tiles = ((tiles_m + 1) / 2) * p.n_tiles_n;
  const int clusters = pair_tiles < max_clusters ? pair_tiles : max_clusters;
  LBC_LAUNCH_CLUSTER(kern, 2, dim3((unsigned)(2 * clusters)), dim3(192), SP::TOTAL, (cudaStream_t)s, mA, mB, mO, p);
  LBC_LAUNCHED(BN == 64 ? "conv_row_kernel<64>" : "conv_row_kernel<128>");
  return 2 * clusters;
}
static int try_conv_row(const bf16* in, const void* wpack, bf16* out, int B, int H, int W, int Cin, int Cout, bool mirrored,
                        const float* bias, bool relu, float* stat_partial, lbc_stream_t s) {
  if (Cout == 64) return try_conv_row_t<64, 6>(in, wpack, out, B, H, W, Cin, Cout, mirrored, bias, relu, stat_partial, s);
  return try_conv_row_t<128, 4>(in, wpack, out, B, H, W, Cin, Cout, mirrored, bias, relu, stat_partial, s);
}

// ---- stem host side: x4 = zero-padded NHWC bf16 image [B][H+6][W+8][CH], CH = 4 (C_in <= 4) or 8 (C_in <= 8) ----
static CUtensorMap make_map_stem(const void* base, int OW, int rows2, int B, int64_t pitch_bytes, int64_t img_bytes, int bw,
                                 int bh, int bn, int CH) {
  CUtensorMap m;
  // W stride = one output pixel = 2 input pixels: overlapping 8-pixel windows (accepted by cuTensorMapEncodeTiled, verified)
  // CH = 16 (space-to-depth): window = 4 blocks of 16, W stride = one block (32 B), H stride = one block row (pitch_bytes)
  const int kel = CH == 16 ? 64 : 8 * CH;
  const int64_t wstride = CH == 16 ? 32 : 2 * CH * 2, hstride = CH == 16 ? pitch_bytes : 2 * pitch_bytes;
  cuuint64_t dims[4] = {(cuuint64_t)kel, (cuuint64_t)OW, (cuuint64_t)rows2, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)wstride, (cuuint64_t)hstride, (cuuint64_t)img_bytes};
  cuuint32_t box[4] = {(cuuint32_t)kel, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bn};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CH == 4 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LBC_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(stem window map) failed: " + std::to_string((int)r));
  return m;
}
static CUtensorMap make_map_stem_w(const void* base, int64_t rows, int brows, int CH) {   // weights [64][window rows x KROW]
  CUtensorMap m;
  const int krow = CH == 16 ? 64 : 8 * CH;
  const int64_t K = (CH == 16 ? 4 : 7) * krow;
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)(K * 2)};
  cuuint32_t box[2] = {(cuuint32_t)krow, (cuuint32_t)brows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CH == 4 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LBC_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(stem weights) failed: " + std::to_string((int)r));
  return m;
}
static bool stem_geometry(int OH, int OW, int B, int& TW, int& TH, int& TN) {
  TW = pow2_divisor(OW, 32);
  TH = pow2_divisor(OH, 128 / TW);
  TN = 128 / (TW * TH);
  return (OW % TW) == 0 && (OH % TH) == 0 && TN <= 256;
}
template <int CH, int STAGES, int PER_SM>
static int launch_stem_conv(const CUtensorMap& mX0, const CUtensorMap& mX1, const CUtensorMap& mB, const CUtensorMap& mO,
                            const StemParams& p, lbc_stream_t s) {
  typedef SmemPlanStem<STAGES, CH> SP;
  static_assert(PER_SM * SP::TOTAL <= 232448 - PER_SM * 1024, "stem smem plan exceeds 227 KB per SM");
  static bool configured = false;
  if (!configured) {
    LBC_CUDA(cudaFuncSetAttribute(stem_conv_kernel<STAGES, CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, SP::TOTAL));
    configured = true;
  }
  int tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  int grid = tiles < PER_SM * sm_count() ? tiles : PER_SM * sm_count();
  { auto k_ = stem_conv_kernel<STAGES, CH>; LBC_LAUNCH(k_, dim3(grid), dim3(192), SP::TOTAL, s, mX0, mX1, mB, mO, p); }
  LBC_LAUNCHED(CH == 4 ? "stem_conv_kernel" : CH == 8 ? "stem_conv_kernel<8ch>" : "stem_conv_kernel<s2d>");
  LBC_CUDA(cudaGetLastError());
  return grid;
}
// raw[B,OH,OW,64] = conv7x7/s2(x4) (+ negshift), optional BN statistics partials; x4 / w224 in the CH-channel layouts
bool stem_conv_bf16(const bf16* x4, const bf16* w224, bf16* raw, int B, int H, int W, int OH, int OW, const float* bias,
                    float* stat_partial, int* stat_rows, lbc_stream_t s, int CH) {
  if ((H % 2) || (W % 2) || OH * 2 != H || OW * 2 != W || (CH != 4 && CH != 8 && CH != 16)) return false;
  StemParams p;
  memset(&p, 0, sizeof(p));
  if (!stem_geometry(OH, OW, B, p.TW, p.TH, p.TN)) return false;
  p.tiles_w = OW / p.TW;
  p.tiles_h = OH / p.TH;
  p.tiles_n = (B + p.TN - 1) / p.TN;
  p.bias = bias;
  p.stat_partial = stat_partial;
  p.stat_C = 64;
  p.valid_n = B;
  // bytes of one padded row (CH = 16: of one row of 2x2 blocks) and of one image
  const int64_t pitch = CH == 16 ? (int64_t)(W + 8) * 16 : (int64_t)(W + 8) * CH * 2;
  const int64_t img = (int64_t)(W + 8) * (H + 6) * stem_x_ch(CH) * 2;
  CUtensorMap mX0 = make_map_stem(x4, OW, (H + 6) / 2, B, pitch, img, p.TW, p.TH, p.TN, CH);
  CUtensorMap mX1 = make_map_stem((const uint8_t*)x4 + pitch, OW, (H + 6) / 2, B, pitch, img, p.TW, p.TH, p.TN, CH);
  CUtensorMap mB = make_map_stem_w(w224, 64, 64, CH);
  const int64_t eb = 2;
  CUtensorMap mO = make_map_4d(raw, 64, OW, OH, B, 64 * eb, (int64_t)OW * 64 * eb, (int64_t)OH * OW * 64 * eb, p.TW, p.TH, p.TN);
  static const int s2d_cfg = [] {
    const char* e = getenv("LBC_STEM_S2D_CFG");   // 1: 3 stages, 2 CTAs per SM; 0: 5 stages, 1 CTA per SM
    return e ? atoi(e) : 1;
  }();
  int ctas;
  if (CH == 4)
    ctas = launch_stem_conv<4, 7, 2>(mX0, mX1, mB, mO, p, s);
  else if (CH == 8)
    ctas = launch_stem_conv<8, 5, 1>(mX0, mX1, mB, mO, p, s);
  else if (s2d_cfg)
    ctas = launch_stem_conv<16, 3, 2>(mX0, mX1, mB, mO, p, s);
  else
    ctas = launch_stem_conv<16, 5, 1>(mX0, mX1, mB, mO, p, s);
  if (stat_rows) *stat_rows = ctas;   // one partial row per CTA
  return true;
}
template <int CH>
static void launch_stem_wgrad(const CUtensorMap& mDY, const CUtensorMap& mX0, const CUtensorMap& mX1, const StemWgradParams& p,
                              lbc_stream_t s) {
  constexpr int STAGES = 4;
  constexpr int RPT = 128 / StemGeom<CH>::KROW;
  constexpr int MT = (StemGeom<CH>::NROWS + RPT - 1) / RPT;   // M tiles: 2 (CH = 4, 16) or 4 (CH = 8)
  const int smem = STAGES * (RPT * StemGeom<CH>::A_BYTES_ + A_BYTES) + 256 + 1024;
  static bool configured = false;
  if (!configured) {
    LBC_CUDA(cudaFuncSetAttribute(stem_wgrad_kernel<STAGES, CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  { auto k_ = stem_wgrad_kernel<STAGES, CH>; LBC_LAUNCH(k_, dim3(MT * p.splits), dim3(192), smem, s, mDY, mX0, mX1, p); }
  LBC_LAUNCHED(CH == 4 ? "stem_wgrad_kernel" : CH == 8 ? "stem_wgrad_kernel<8ch>" : "stem_wgrad_kernel<s2d>");
  LBC_CUDA(cudaGetLastError());
}
template <int Slot>
static float* wgrad_partials(int64_t floats);
// dw_ref[64][C][7][7] = sum_pixels dy x window(x4), the K splits' partial sums added in split order
bool stem_wgrad_bf16(const bf16* x4, const bf16* dy, float* dw_ref, int B, int C, int H, int W, int OH, int OW, lbc_stream_t s,
                     int CH) {
  if ((H % 2) || (W % 2) || OH * 2 != H || OW * 2 != W || C > stem_x_ch(CH) || (CH != 4 && CH != 8 && CH != 16)) return false;
  StemWgradParams p;
  memset(&p, 0, sizeof(p));
  if (!stem_geometry(OH, OW, B, p.TW, p.TH, p.TN)) return false;
  p.tiles_w = OW / p.TW;
  p.tiles_h = OH / p.TH;
  p.tiles_n = (B + p.TN - 1) / p.TN;
  p.k_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  int splits = sm_count() / (CH == 8 ? 4 : 2);   // M tiles per split: 2 (CH = 4, 16) or 4 (CH = 8)
  if (splits > p.k_tiles / 4) splits = p.k_tiles / 4 > 0 ? p.k_tiles / 4 : 1;
  p.k_per_split = (p.k_tiles + splits - 1) / splits;
  p.splits = (p.k_tiles + p.k_per_split - 1) / p.k_per_split;
  p.C = C;
  const int64_t slice = (int64_t)64 * C * 49;
  p.dw_ref = wgrad_partials<2>((int64_t)p.splits * slice);
  if (!p.dw_ref) return false;
  const int64_t pitch = CH == 16 ? (int64_t)(W + 8) * 16 : (int64_t)(W + 8) * CH * 2;
  const int64_t img = (int64_t)(W + 8) * (H + 6) * stem_x_ch(CH) * 2;
  CUtensorMap mX0 = make_map_stem(x4, OW, (H + 6) / 2, B, pitch, img, p.TW, p.TH, p.TN, CH);
  CUtensorMap mX1 = make_map_stem((const uint8_t*)x4 + pitch, OW, (H + 6) / 2, B, pitch, img, p.TW, p.TH, p.TN, CH);
  const int64_t eb = 2;
  CUtensorMap mDY = make_map_4d(dy, 64, OW, OH, B, 64 * eb, (int64_t)OW * 64 * eb, (int64_t)OH * OW * 64 * eb, p.TW, p.TH, p.TN);
  if (CH == 4)
    launch_stem_wgrad<4>(mDY, mX0, mX1, p, s);
  else if (CH == 8)
    launch_stem_wgrad<8>(mDY, mX0, mX1, p, s);
  else
    launch_stem_wgrad<16>(mDY, mX0, mX1, p, s);
  { auto k_ = sum_slices_kernel<float>; LBC_LAUNCH(k_, dim3((unsigned)((slice + 255) / 256)), dim3(256), 0, s, (const float*)p.dw_ref, dw_ref, slice, p.splits); }
  LBC_LAUNCHED("sum_slices_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}

// y = conv(x, w):  x [B,H,W,Ci], packed weights [Co][K*K][Ci], y [B,OH,OW,Co]
// (split mode: x [B,H,W,2Ci] = hi | lo planes, weights [Co][K*K][2Ci] = per tap hi | lo, y fp32)
static bool conv_fwd_impl(const ConvL& c, const void* x, const void* wpack, void* y, int B, const float* bias_co, bool relu,
                          lbc_stream_t s, float* stat_partial, int* stat_rows, const GemmMode& m) {
  if (!supported(c)) return false;
  if (!m.split && !m.out_f32 && c.K == 3 && c.stride == 1 && c.Ci == 64 && c.Co == 64 && !relu &&
      try_conv3x3_c64((const bf16*)x, wpack, (bf16*)y, B, c.H, c.W, false, bias_co, false, stat_partial, stat_rows, s))
    return true;
  if (!m.split && !m.out_f32 && c.K == 3 && c.stride == 1 && c.pad == 1) {
    float* part = c.Co > 512 ? nullptr : stat_partial;
    const int ctas = try_conv_row((const bf16*)x, wpack, (bf16*)y, B, c.H, c.W, c.Ci, c.Co, false, bias_co, relu, part, s);
    if (ctas > 0) {
      if (stat_rows) *stat_rows = part ? ctas : 0;
      return true;
    }
  }
  ConvGemmParams p;
  memset(&p, 0, sizeof(p));
  if (!tile_geometry(c.OH, c.OW, B, p)) return false;
  const int BN = pick_bn(c.Co, p.tiles_w * p.tiles_h * p.tiles_n);
  const int CA = m.split ? 2 * c.Ci : c.Ci;   // channels of the stored x tensor / of one tap slab of the weights
  p.n_tiles_n = c.Co / BN;
  p.num_taps = c.K * c.K;
  p.k_chunks = c.Ci / 64;
  p.bias = bias_co;   // per-output-channel constant added before the rounding (centring shift, see lbc_net.cu)
  p.relu = relu ? 1 : 0;
  p.stat_partial = (m.out_f32 || c.Co > 512) ? nullptr : stat_partial;   // (the per-CTA accumulator holds 2 x 512 floats)
  p.stat_C = c.Co;
  p.valid_n = B;
  apply_mode(p, m, c.Ci, c.Ci);
  CUtensorMap mA[4];
  const int64_t eb = 2;
  const bf16* xb = (const bf16*)x;
  if (c.stride == 1) {
    mA[0] = make_map_4d(xb, CA, c.W, c.H, B, CA * eb, (int64_t)c.W * CA * eb, (int64_t)c.H * c.W * CA * eb, p.TW, p.TH, p.TN);
    mA[1] = mA[2] = mA[3] = mA[0];
    for (int kh = 0; kh < c.K; ++kh)
      for (int kw = 0; kw < c.K; ++kw) {
        int t = kh * c.K + kw;
        p.tap_dh[t] = kh - c.pad;
        p.tap_dw[t] = kw - c.pad;
        p.tap_map[t] = 0;
        p.tap_koff[t] = t * CA;
      }
  } else {
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b)
        mA[a * 2 + b] = make_map_4d(xb + ((int64_t)a * c.W + b) * CA, CA, c.W / 2, c.H / 2, B, 2 * CA * eb,
                                    2 * (int64_t)c.W * CA * eb, (int64_t)c.H * c.W * CA * eb, p.TW, p.TH, p.TN);
    for (int kh = 0; kh < c.K; ++kh)
      for (int kw = 0; kw < c.K; ++kw) {
        int t = kh * c.K + kw;
        int th = kh - c.pad, tw = kw - c.pad;  // input row = 2*oh + th
        int a = ((th % 2) + 2) % 2, b = ((tw % 2) + 2) % 2;
        p.tap_dh[t] = (th - a) / 2;
        p.tap_dw[t] = (tw - b) / 2;
        p.tap_map[t] = a * 2 + b;
        p.tap_koff[t] = t * CA;
      }
  }
  const int64_t eo = m.out_f32 ? 4 : 2;
  CUtensorMap mO = make_map_4d(y, c.Co, c.OW, c.OH, B, c.Co * eo, (int64_t)c.OW * c.Co * eo, (int64_t)c.OH * c.OW * c.Co * eo,
                               p.TW, p.TH, p.TN, m.out_f32);
  const int ctas = dispatch_gemm(BN, mA, wpack, (int64_t)c.K * c.K * CA, c.Co, mO, p, s, m.out_f32);
  if (stat_rows) *stat_rows = p.stat_partial ? ctas : 0;   // one row of statistics partials per persistent CTA
  return true;
}
bool conv_fwd_bf16(const ConvL& c, const bf16* x, bf16* y, int B, const float* bias_co, lbc_stream_t s,
                   float* stat_partial, int* stat_rows) {
  return conv_fwd_impl(c, x, c.wp, y, B, bias_co, false, s, stat_partial, stat_rows, GemmMode());
}

// dx = conv_dgrad(dy, w):  dy [B,OH,OW,Co], transposed pack wt [Ci][K*K][Co], dx [B,H,W,Ci] (+bias[ci]) (relu)
// stride 1: one GEMM with mirrored taps; stride 2: one GEMM per output parity (also ConvTranspose2d forward).
// (split mode: dy [B,OH,OW,2Co] hi | lo, wt [Ci][K*K][2Co] per tap hi | lo, wcomb [Ci][2][2Co], dx fp32)
static bool conv_dgrad_impl(const ConvL& c, const void* dy, const void* wt, const void* wcomb, void* dx, int B,
                            const float* bias_ci, bool relu, const void* dy_ds, lbc_stream_t s, const GemmMode& m);
bool conv_dgrad_bf16(const ConvL& c, const bf16* dy, bf16* dx, int B, const float* bias_ci, bool relu, lbc_stream_t s) {
  return conv_dgrad_impl(c, dy, c.wpt, c.wcomb, dx, B, bias_ci, relu, nullptr, s, GemmMode());
}
// gradient wrt the input of a residual block's entry: dgrad(3x3/s2 conv1)(dy1) + dgrad(1x1/s2 downsample)(dy_ds).
// The 1x1/s2 gradient only touches the (even,even) parity, where it is one more K-slab of the same GEMM
// (A = dy_ds, B = the [Ci][Co] downsample weights stored behind conv1's centre tap in c1.wcomb).
bool conv_dgrad_ds_bf16(const ConvL& c1, const bf16* dy1, const bf16* dy_ds, bf16* dx, int B, lbc_stream_t s) {
  if (!c1.wcomb || c1.stride != 2 || c1.K != 3) return false;
  return conv_dgrad_impl(c1, dy1, c1.wpt, c1.wcomb, dx, B, nullptr, false, dy_ds, s, GemmMode());
}
static bool conv_dgrad_impl(const ConvL& c, const void* dy_v, const void* wt, const void* wcomb, void* dx_v, int B,
                            const float* bias_ci, bool relu, const void* dy_ds_v, lbc_stream_t s, const GemmMode& m) {
  if (!supported(c) || !wt) return false;
  if (c.K == 1) return false;  // 1x1/s2 downsample gradient scatters into one parity only: handled by the caller
  const bf16* dy = (const bf16*)dy_v;
  const bf16* dy_ds = (const bf16*)dy_ds_v;
  const int64_t eb = 2;
  const int64_t eo = m.out_f32 ? 4 : 2;
  uint8_t* dx = (uint8_t*)dx_v;
  const int CA = m.split ? 2 * c.Co : c.Co;   // channels of the stored dy tensor / of one tap slab of wt
  ConvGemmParams g0;
  memset(&g0, 0, sizeof(g0));
  if (!tile_geometry(c.stride == 1 ? c.H : c.OH, c.stride == 1 ? c.W : c.OW, B, g0)) return false;
  const int BN = pick_bn(c.Ci, g0.tiles_w * g0.tiles_h * g0.tiles_n);
  const int64_t wtK = (int64_t)c.K * c.K * CA;
  if (c.stride == 1) {
    if (!m.split && !m.out_f32 && c.K == 3 && c.Ci == 64 && c.Co == 64 && !dy_ds &&
        try_conv3x3_c64(dy, wt, (bf16*)dx_v, B, c.H, c.W, true, bias_ci, relu, nullptr, nullptr, s))
      return true;
    if (!m.split && !m.out_f32 && c.K == 3 && c.pad == 1 && !dy_ds &&
        try_conv_row(dy, wt, (bf16*)dx_v, B, c.H, c.W, c.Co, c.Ci, true, bias_ci, relu, nullptr, s) > 0)
      return true;
    ConvGemmParams p;
    memset(&p, 0, sizeof(p));
    if (!tile_geometry(c.H, c.W, B, p)) return false;
    p.n_tiles_n = c.Ci / BN;
    p.num_taps = c.K * c.K;
    p.k_chunks = c.Co / 64;
    p.bias = bias_ci;
    p.relu = relu ? 1 : 0;
    apply_mode(p, m, c.Co, c.Co);
    CUtensorMap mA[4];
    mA[0] = make_map_4d(dy, CA, c.OW, c.OH, B, CA * eb, (int64_t)c.OW * CA * eb, (int64_t)c.OH * c.OW * CA * eb, p.TW, p.TH, p.TN);
    mA[1] = mA[2] = mA[3] = mA[0];
    for (int kh = 0; kh < c.K; ++kh)
      for (int kw = 0; kw < c.K; ++kw) {
        int t = kh * c.K + kw;
        p.tap_dh[t] = c.pad - kh;
        p.tap_dw[t] = c.pad - kw;
        p.tap_map[t] = 0;
        p.tap_koff[t] = t * CA;
      }
    CUtensorMap mO = make_map_4d(dx, c.Ci, c.W, c.H, B, c.Ci * eo, (int64_t)c.W * c.Ci * eo, (int64_t)c.H * c.W * c.Ci * eo,
                                 p.TW, p.TH, p.TN, m.out_f32);
    dispatch_gemm(BN, mA, wt, wtK, c.Ci, mO, p, s, m.out_f32);
    return true;
  }
  // stride 2: dx[n, 2i+a, 2j+b, :] = sum over taps kh with (a + pad - kh) even: dy[n, i + (a+pad-kh)/2, ...]
  ConvGemmParams base;
  memset(&base, 0, sizeof(base));
  if (!tile_geometry(c.OH, c.OW, B, base)) return false;
  base.n_tiles_n = c.Ci / BN;
  base.k_chunks = c.Co / 64;
  base.bias = bias_ci;
  base.relu = relu ? 1 : 0;
  apply_mode(base, m, c.Co, c.Co);
  CUtensorMap mA[4];
  mA[0] = make_map_4d(dy, CA, c.OW, c.OH, B, CA * eb, (int64_t)c.OW * CA * eb, (int64_t)c.OH * c.OW * CA * eb, base.TW, base.TH,
                      base.TN);
  mA[1] = mA[2] = mA[3] = mA[0];
  if (dy_ds)
    mA[1] = make_map_4d(dy_ds, CA, c.OW, c.OH, B, CA * eb, (int64_t)c.OW * CA * eb, (int64_t)c.OH * c.OW * CA * eb, base.TW,
                        base.TH, base.TN);
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b) {
      ConvGemmParams p = base;
      int nt = 0;
      if (dy_ds && a == 0 && b == 0) {
        // centre tap of the 3x3 (kh=kw=1 -> dh=dw=0) + the downsample slab
        p.tap_dh[0] = p.tap_dw[0] = 0;
        p.tap_map[0] = 0;
        p.tap_koff[0] = 0;
        p.tap_dh[1] = p.tap_dw[1] = 0;
        p.tap_map[1] = 1;
        p.tap_koff[1] = CA;
        p.num_taps = 2;
        CUtensorMap mO = make_map_4d(dx, c.Ci, c.W / 2, c.H / 2, B, 2 * c.Ci * eo, 2 * (int64_t)c.W * c.Ci * eo,
                                     (int64_t)c.H * c.W * c.Ci * eo, p.TW, p.TH, p.TN, m.out_f32);
        dispatch_gemm(BN, mA, wcomb, (int64_t)2 * CA, c.Ci, mO, p, s, m.out_f32);
        continue;
      }
      for (int kh = 0; kh < c.K; ++kh) {
        if ((a + c.pad - kh) % 2 != 0) continue;
        for (int kw = 0; kw < c.K; ++kw) {
          if ((b + c.pad - kw) % 2 != 0) continue;
          p.tap_dh[nt] = (a + c.pad - kh) / 2;
          p.tap_dw[nt] = (b + c.pad - kw) / 2;
          p.tap_map[nt] = 0;
          p.tap_koff[nt] = (kh * c.K + kw) * CA;
          ++nt;
        }
      }
      p.num_taps = nt;
      CUtensorMap mO = make_map_4d(dx + ((int64_t)a * c.W + b) * c.Ci * eo, c.Ci, c.W / 2, c.H / 2, B, 2 * c.Ci * eo,
                                   2 * (int64_t)c.W * c.Ci * eo, (int64_t)c.H * c.W * c.Ci * eo, p.TW, p.TH, p.TN, m.out_f32);
      dispatch_gemm(BN, mA, wt, wtK, c.Ci, mO, p, s, m.out_f32);
    }
  return true;
}


// =============================================================================================================
// Weight gradient:  dW[co][tap][ci] = sum_{n,oh,ow} dy[n,oh,ow,co] * x[n, oh*s-p+kh, ow*s-p+kw, ci]
//
//   D[128 co x BNW ci] (fp32, TMEM) += A[128 co x 128 pixels] * B[BNW ci x 128 pixels]^T, both operands "MN-major":
//   a TMA box {64 ch, TW, TH, TN} lands as [128 pixels][64 ch] rows of 128 B (128 B swizzle) = the UMMA MN-major
//   SWIZZLE_128B canonical layout with K = pixels (8-row groups 1024 B apart, 64-channel blocks LBO apart).
//   One CTA per (co tile, tap, ci tile, K split); each split stores its partials into its own packed [Co][tap][Ci] slice,
//   and a tiny kernel adds the slices in split order while permuting into the reference's [Co][Ci][kh][kw] .grad.
// =============================================================================================================
struct WgradParams {
  int TW, TH, TN, tiles_w, tiles_h, tiles_n;
  int k_tiles, k_per_split, splits;
  int co_tiles, ci_tiles, num_taps;
  int tap_dh[9], tap_dw[9], tap_map[9];
  int Co, Ci;
  float* out;  // [splits][Co][num_taps][Ci] fp32 partials, every element stored once per split
  // swap mode (Co == 64): M = two (tap, 64-channel ci chunk) combos of x, N = the 64 output channels of dy, so the
  // 128-row MMA is full instead of half zero padding
  int swap, num_combos, chunks_per_tap;
  // split-precision mode: dy = [hi | lo] planes of dy_plane channels, x = [hi | lo] planes of x_plane channels; the K
  // (pixel) loop runs 3 x k_tiles_real tiles: (dy hi, x lo), (dy lo, x hi), (dy hi, x hi).  k_tiles = 3 * k_tiles_real.
  int split, k_tiles_real, dy_plane, x_plane;
  uint32_t fmt_dy, fmt_x;   // UMMA formats (0 = fp16, 1 = bf16)
};

__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;  // distance between 64-element MN blocks
  d |= (uint64_t)(1024 >> 4) << 32;                  // distance between 8-row K groups
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

template <int BNW, int STAGES>
struct WgradSmem {
  static constexpr int A_ST = 2 * A_BYTES;            // 128 co = 2 boxes
  static constexpr int B_ST = (BNW / 64) * A_BYTES;   // BNW ci
  static constexpr int STAGE_BYTES = A_ST + B_ST;
  static constexpr int BAR_OFF = STAGES * STAGE_BYTES;
  static constexpr int TOTAL = BAR_OFF + 256 + 1024;
};

template <int BNW, int STAGES>
__global__ void __launch_bounds__(192, 1)
wgrad_gemm_kernel(const __grid_constant__ CUtensorMap mDY, const __grid_constant__ CUtensorMap mX0,
                  const __grid_constant__ CUtensorMap mX1, const __grid_constant__ CUtensorMap mX2,
                  const __grid_constant__ CUtensorMap mX3, const WgradParams p) {
  typedef WgradSmem<BNW, STAGES> SP;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(smem + SP::BAR_OFF);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint32_t* tmem_slot = (uint32_t*)(tfull + 1);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr uint32_t TMEM_COLS = BNW <= 32 ? 32 : (BNW <= 64 ? 64 : (BNW <= 128 ? 128 : 256));

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(tfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // everything above touched shared / tensor memory only
  pdl_trigger();

  // decode this CTA's work: (split, co_tile, tap, ci_tile)   [swap mode: (split, combo pair)]
  int id = blockIdx.x;
  int ci_tile, tap, co_tile, split, combo0 = 0, combo1 = 0;
  if (p.swap) {
    const int pairs = (p.num_combos + 1) / 2;
    const int pair = id % pairs;
    split = id / pairs;
    combo0 = pair * 2;
    combo1 = combo0 + 1 < p.num_combos ? combo0 + 1 : combo0;   // odd tail: duplicate (rows 64..127 are then ignored)
    ci_tile = 0;
    tap = 0;
    co_tile = 0;
  } else {
    ci_tile = id % p.ci_tiles;
    id /= p.ci_tiles;
    tap = id % p.num_taps;
    id /= p.num_taps;
    co_tile = id % p.co_tiles;
    split = id / p.co_tiles;
  }
  const int kt0 = split * p.k_per_split;
  int kt1 = kt0 + p.k_per_split;
  if (kt1 > p.k_tiles) kt1 = p.k_tiles;
  const int n_k = kt1 - kt0;

  if (warp == 0) {
    if (elect_one()) {
      const int tapA = p.swap ? combo0 / p.chunks_per_tap : tap;
      const int tapB = p.swap ? combo1 / p.chunks_per_tap : tap;
      const int midA = p.tap_map[tapA], midB = p.tap_map[tapB];
      const CUtensorMap* mx = midA == 0 ? &mX0 : (midA == 1 ? &mX1 : (midA == 2 ? &mX2 : &mX3));
      const CUtensorMap* mx2 = midB == 0 ? &mX0 : (midB == 1 ? &mX1 : (midB == 2 ? &mX2 : &mX3));
      const int dh = p.tap_dh[tapA], dw = p.tap_dw[tapA];
      const int dh2 = p.tap_dh[tapB], dw2 = p.tap_dw[tapB];
      const int cA = p.swap ? (combo0 % p.chunks_per_tap) * 64 : 0, cB = p.swap ? (combo1 % p.chunks_per_tap) * 64 : 0;
      int stage = 0;
      uint32_t phase = 0;
      for (int kt2 = kt0; kt2 < kt1; ++kt2) {
        const int term = p.split ? kt2 / p.k_tiles_real : 0;
        const int kt = kt2 - term * p.k_tiles_real;
        const int dyo = (p.split && term == 1) ? p.dy_plane : 0;   // term 0: dy hi x x lo, 1: dy lo x x hi, 2: hi x hi (last:
        const int xo = (p.split && term == 0) ? p.x_plane : 0;     //  see the note on accumulator truncation in conv_gemm_kernel)
        const int w0 = (kt % p.tiles_w) * p.TW;
        const int h0 = ((kt / p.tiles_w) % p.tiles_h) * p.TH;
        const int n0 = (kt / (p.tiles_w * p.tiles_h)) * p.TN;
        mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* sa = smem + stage * SP::STAGE_BYTES;
        mbar_expect_tx(&full[stage], SP::STAGE_BYTES);
        if (p.swap) {   // A = two x boxes (M = 2 x 64 input channels), B = dy (N = 64 output channels); BNW == 64
          tma_load_4d(mx, sa, &full[stage], cA + xo, w0 + dw, h0 + dh, n0);
          tma_load_4d(mx2, sa + A_BYTES, &full[stage], cB + xo, w0 + dw2, h0 + dh2, n0);
          tma_load_4d(&mDY, sa + SP::A_ST, &full[stage], dyo, w0, h0, n0);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
          continue;
        }
        tma_load_4d(&mDY, sa, &full[stage], co_tile * 128 + dyo, w0, h0, n0);
        tma_load_4d(&mDY, sa + A_BYTES, &full[stage], co_tile * 128 + 64 + dyo, w0, h0, n0);  // OOB -> zeros when Co == 64
#pragma unroll
        for (int b = 0; b < BNW / 64; ++b)
          tma_load_4d(mx, sa + SP::A_ST + b * A_BYTES, &full[stage], ci_tile * BNW + b * 64 + xo, w0 + dw, h0 + dh, n0);
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // D=f32, A / B = bf16 or fp16, both MN-major (bits 15,16), N=BNW, M=128   (swap mode: A = x, B = dy)
    const uint32_t fa = p.swap ? p.fmt_x : p.fmt_dy, fb = p.swap ? p.fmt_dy : p.fmt_x;
    const uint32_t idesc = (1u << 4) | (fa << 7) | (fb << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(BNW >> 3) << 17) |
                           ((uint32_t)(128 >> 4) << 24);
    int stage = 0;
    uint32_t phase = 0;
    for (int k = 0; k < n_k; ++k) {
      mbar_wait(&full[stage], phase);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (elect_one()) {
        const uint32_t sa = smem_u32(smem + stage * SP::STAGE_BYTES);
        const uint64_t ad = umma_desc_mn_sw128(sa, A_BYTES);
        const uint64_t bd = umma_desc_mn_sw128(sa + SP::A_ST, A_BYTES);
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)  // 8 x (K=16 pixels): advance two 8-row groups = 2048 B
          umma_bf16(tmem_base, ad + (uint64_t)(kk * (2048 >> 4)), bd + (uint64_t)(kk * (2048 >> 4)), idesc, (k | kk) != 0);
        umma_commit(&empty[stage]);
        if (k == n_k - 1) umma_commit(tfull);
      }
      __syncwarp();
      if (++stage == STAGES) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (n_k > 0) {
    const int q = warp & 3;
    const int co = co_tile * 128 + q * 32 + lane;
    mbar_wait(tfull, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
    float* out = p.out + (int64_t)split * p.Co * p.num_taps * p.Ci;
#pragma unroll 1
    for (int ch = 0; ch < BNW / 32; ++ch) {
      uint32_t r[32];
      tmem_ld32(taddr + ch * 32, r);
      if (p.swap) {
        const int m = q * 32 + lane;
        const int which = m >> 6;
        const int combo = which ? combo1 : combo0;
        if (which == 0 || combo1 != combo0) {
          const int tp = combo / p.chunks_per_tap;
          const int ci = (combo % p.chunks_per_tap) * 64 + (m & 63);
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int con = ch * 32 + j;   // output channel
            out[((int64_t)con * p.num_taps + tp) * p.Ci + ci] = __uint_as_float(r[j]);
          }
        }
      } else if (co < p.Co) {
        float* dst = out + ((int64_t)co * p.num_taps + tap) * p.Ci + ci_tile * BNW + ch * 32;
#pragma unroll
        for (int j = 0; j < 32; ++j) dst[j] = __uint_as_float(r[j]);
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------- 3x3/s1 weight gradient, 64 -> 64 channels
// Layer 1 (and the teacher's): dW[co][tap][ci] for Co = Ci = 64.  wgrad_gemm_kernel's swap mode gives every CTA one PAIR of
// taps and streams 48 KB of operands per 384 MMA cycles -- 125 B/clk against the ~68 B/clk an SM ingests, so it runs at 36-39 %
// tensor pipe (87 us for 72.5 GFLOP).  Here ONE CTA owns all nine taps for its share of the pixels:
//   * per K step of 128 output pixels (8 columns x TH rows x TN images) it loads the dy tile (16 KB) and ONE x box with a
//     halo, {64 ch, 8+2, TH+2, TN} (25 KB): 41 KB for all nine taps = 24 B/clk;
//   * x is the MN-major A operand (a pixel is one 128-byte row of 64 channels).  Tap (dh, dw) is the same box read from row
//     (dh+1)*10 + (dw+1) on, with 8-pixel K groups 1280 B apart (one image row of the tile); an MMA covers 16 pixels = two
//     image rows of one image, so every MMA gets its own start address and the image boundary never falls inside one;
//   * M = 128 = TWO taps x 64 input channels: the second 64-row block of the A descriptor starts LBO bytes after the first,
//     and LBO is simply the address distance of the two taps in the box (128 B for (dw, dw+1), 1024 B for tap 2 -> tap 3);
//     five tap pairs (the ninth tap is paired with a dummy whose rows are dropped) -> five TMEM accumulators of 64 columns.
// Split-K: one CTA per SM, partials [split][Co][9][Ci] with plain stores, summed by wgrad3_reduce_kernel.
struct Wgrad9Params {
  int TH, TN, tiles_w, tiles_h, tiles_n;
  int k_tiles, k_per_split;
  float* out;   // [splits][64][9][64] fp32 partials
};
template <int STAGES>
struct Wgrad9Smem {
  static constexpr int DY_BYTES = A_BYTES;          // 128 pixels x 64 co
  static constexpr int X_BYTES = 26 * 1024;         // {64, 10, TH+2, TN}: <= 200 rows of 128 B (+ slack for the dummy tap)
  static constexpr int STAGE_BYTES = DY_BYTES + X_BYTES;
  static constexpr int BAR_OFF = STAGES * STAGE_BYTES;
  static constexpr int TOTAL = BAR_OFF + 256 + 1024;
};
__device__ __forceinline__ uint64_t umma_desc_mn_sw128_sbo(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;  // distance between 64-element MN blocks
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;  // distance between 8-row K groups
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
template <int STAGES>
__global__ void __launch_bounds__(192, 1)
wgrad9_c64_kernel(const __grid_constant__ CUtensorMap mDY, const __grid_constant__ CUtensorMap mX, const Wgrad9Params p) {
  typedef Wgrad9Smem<STAGES> SP;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(smem + SP::BAR_OFF);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint32_t* tmem_slot = (uint32_t*)(tfull + 1);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr uint32_t TMEM_COLS = 512;   // five accumulators of 64 columns

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(tfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // everything above touched shared / tensor memory only
  pdl_trigger();

  const int split = blockIdx.x;
  const int kt0 = split * p.k_per_split;
  int kt1 = kt0 + p.k_per_split;
  if (kt1 > p.k_tiles) kt1 = p.k_tiles;
  const int n_k = kt1 > kt0 ? kt1 - kt0 : 0;
  const uint32_t x_bytes = (uint32_t)(10 * (p.TH + 2) * p.TN * 128);

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kt = kt0; kt < kt1; ++kt) {
        const int w0 = (kt % p.tiles_w) * 8;
        const int h0 = ((kt / p.tiles_w) % p.tiles_h) * p.TH;
        const int n0 = (kt / (p.tiles_w * p.tiles_h)) * p.TN;
        mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* sa = smem + stage * SP::STAGE_BYTES;
        mbar_expect_tx(&full[stage], SP::DY_BYTES + x_bytes);
        tma_load_4d(&mDY, sa, &full[stage], 0, w0, h0, n0);
        tma_load_4d(&mX, sa + SP::DY_BYTES, &full[stage], 0, w0 - 1, h0 - 1, n0);
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // D = f32, A (x) and B (dy) bf16, both MN-major (bits 15, 16), N = 64, M = 128
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(64 >> 3) << 17) |
                           ((uint32_t)(128 >> 4) << 24);
    // the issuing thread is the bottleneck of a 40-MMA stage unless its per-MMA work is a couple of integer adds: the box
    // offsets of the eight 16-pixel K steps and the five constant descriptor halves are computed once
    const int half_th = p.TH >> 1;
    uint32_t xoff[8];
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
      const int ni = kk / half_th, rp = kk - ni * half_th;
      xoff[kk] = (uint32_t)((ni * (p.TH + 2) + 2 * rp) * 10 * 128);   // box row of (image row 2*rp - 1, column w0 - 1), in bytes
    }
    const uint64_t a_hi128 = umma_desc_mn_sw128_sbo(0, 128, 1280), a_hi1024 = umma_desc_mn_sw128_sbo(0, 1024, 1280);
    const uint64_t b_hi = umma_desc_mn_sw128_sbo(0, A_BYTES, 1024);
    int stage = 0;
    uint32_t phase = 0;
    for (int k = 0; k < n_k; ++k) {
      mbar_wait(&full[stage], phase);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (elect_one()) {
        const uint32_t sdy = smem_u32(smem + stage * SP::STAGE_BYTES);
        const uint32_t sx = sdy + SP::DY_BYTES;
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {   // 16 pixels = two image rows (2 * rp, 2 * rp + 1) of image ni of the tile
          const uint64_t bd = b_hi | (uint64_t)(((sdy + kk * 2048) & 0x3FFFF) >> 4);
          const uint32_t xa = sx + xoff[kk];
#pragma unroll
          for (int a = 0; a < 5; ++a) {
            constexpr int kTapOff[5] = {(0 * 10 + 0) * 128, (0 * 10 + 2) * 128, (1 * 10 + 1) * 128, (2 * 10 + 0) * 128, (2 * 10 + 2) * 128};
            // taps (2a, 2a + 1); the ninth tap is paired with a dummy; tap 2 -> tap 3 is one box row minus two columns away
            const uint64_t ad = (a == 1 ? a_hi1024 : a_hi128) | (uint64_t)(((xa + kTapOff[a]) & 0x3FFFF) >> 4);
            umma_bf16(tmem_base + a * 64, ad, bd, idesc, (k | kk) != 0);
          }
        }
        umma_commit(&empty[stage]);
        if (k == n_k - 1) umma_commit(tfull);
      }
      __syncwarp();
      if (++stage == STAGES) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else {
    const int q = warp & 3;
    const int m = q * 32 + lane;      // accumulator row: (tap of the pair, input channel)
    const int which = m >> 6, ci = m & 63;
    float* dst0 = p.out + (int64_t)split * 64 * 9 * 64;
    if (n_k > 0) {
      mbar_wait(tfull, 0);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
    for (int a = 0; a < 5; ++a) {
      const int tap = 2 * a + which;
#pragma unroll 1
      for (int ch = 0; ch < 2; ++ch) {
        uint32_t r[32];
        if (n_k > 0) {
          tmem_ld32(taddr + a * 64 + ch * 32, r);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) r[j] = 0u;
        }
        if (tap < 9) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int co = ch * 32 + j;
            dst0[((int64_t)co * 9 + tap) * 64 + ci] = __uint_as_float(r[j]);
          }
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------- 3x3 weight gradient, row of taps
// The one-tap kernel above moves 64 KB of operands into the SM per 4.2 MFLOP (64 FLOP/B).  Measured on the B200 one SM
// ingests ~65-70 B/clk from L2 (wgrad_gemm_kernel<128,3>: 64 KB per ~950 clk), so that kernel runs at half the
// tensor rate.  Here one CTA owns the THREE taps of a kernel row for a (128 co x 128 ci) tile: per 64-pixel K step
// it loads the dy tile once (16 KB) and three shifted x tiles (48 KB) and issues three MMA groups into three TMEM
// accumulators (384 columns) -> 98 FLOP/B.  PAIR: two CTAs (co tiles 2c, 2c+1) share the x tiles through one
// 256-row cta_group::2 MMA, each staging its dy tile and HALF of every x tile (40 KB per step, 157 FLOP/B).
// Split-K partials are written with plain stores to partial[split][Co][9][Ci] and summed by wgrad3_reduce_kernel
// (fp32 atomics from 49 splits cost more than the whole K loop).
struct Wgrad3Params {
  int TW, TH, TN, tiles_w, tiles_h, tiles_n;   // 64-pixel K tile = TN*TH*TW
  int k_tiles, k_per_split, splits;
  int co_tiles, ci_tiles;
  int tap_dh[9], tap_dw[9], tap_map[9];
  int Co, Ci;
  float* out;  // [splits][Co][9][Ci] fp32 partials
  int split, k_tiles_real, dy_plane, x_plane;   // split-precision mode, as in WgradParams
  uint32_t fmt_dy, fmt_x;
};
constexpr int W3_BOX = 64 * 128;   // 64 pixels x 64 channels bf16

template <int STAGES, bool PAIR>
struct Wgrad3Smem {
  static constexpr int A_ST = 2 * W3_BOX;                    // dy: 128 co = 2 boxes
  static constexpr int B_TAP = (PAIR ? 1 : 2) * W3_BOX;      // x per tap: 128 ci (pair: this CTA's 64)
  static constexpr int B_ST = 3 * B_TAP;
  static constexpr int STAGE_BYTES = A_ST + B_ST;            // 64 KB (pair: 40 KB)
  static constexpr int BAR_OFF = STAGES * STAGE_BYTES;
  static constexpr int TOTAL = BAR_OFF + 256 + 1024;
};

template <int STAGES, bool PAIR>
__global__ void __launch_bounds__(192, 1)
wgrad3_gemm_kernel(const __grid_constant__ CUtensorMap mDY, const __grid_constant__ CUtensorMap mX0,
                   const __grid_constant__ CUtensorMap mX1, const __grid_constant__ CUtensorMap mX2,
                   const __grid_constant__ CUtensorMap mX3, const Wgrad3Params p) {
  typedef Wgrad3Smem<STAGES, PAIR> SP;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(smem + SP::BAR_OFF);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint32_t* tmem_slot = (uint32_t*)(tfull + 1);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr uint32_t TMEM_COLS = 512;   // 3 accumulators x 128 columns

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(tfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if constexpr (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if constexpr (PAIR)
    cluster_sync_all();
  else
    __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // everything above touched shared / tensor memory only
  pdl_trigger();

  // this CTA's work: (split, co tile [pair: co-tile pair + rank], kernel row, ci_tile)
  const uint32_t crank = PAIR ? cluster_ctarank() : 0u;
  int id = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int ci_tile = id % p.ci_tiles;
  id /= p.ci_tiles;
  const int krow = id % 3;
  id /= 3;
  const int co_groups = PAIR ? p.co_tiles / 2 : p.co_tiles;
  const int co_tile = PAIR ? 2 * (id % co_groups) + (int)crank : id % co_groups;
  const int split = id / co_groups;
  const int kt0 = split * p.k_per_split;
  int kt1 = kt0 + p.k_per_split;
  if (kt1 > p.k_tiles) kt1 = p.k_tiles;
  const int n_k = kt1 - kt0;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kt2 = kt0; kt2 < kt1; ++kt2) {
        const int term = p.split ? kt2 / p.k_tiles_real : 0;
        const int kt = kt2 - term * p.k_tiles_real;
        const int dyo = (p.split && term == 1) ? p.dy_plane : 0;   // term 0: dy hi x x lo, 1: dy lo x x hi, 2: hi x hi (last:
        const int xo = (p.split && term == 0) ? p.x_plane : 0;     //  see the note on accumulator truncation in conv_gemm_kernel)
        const int w0 = (kt % p.tiles_w) * p.TW;
        const int h0 = ((kt / p.tiles_w) % p.tiles_h) * p.TH;
        const int n0 = (kt / (p.tiles_w * p.tiles_h)) * p.TN;
        mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* sa = smem + stage * SP::STAGE_BYTES;
        if constexpr (PAIR) {
          if (crank == 0) mbar_expect_tx(&full[stage], 2 * SP::STAGE_BYTES);
          const uint32_t lead_full = mapa_u32(smem_u32(&full[stage]), 0);
          tma_load_4d_pair(&mDY, sa, lead_full, co_tile * 128 + dyo, w0, h0, n0);
          tma_load_4d_pair(&mDY, sa + W3_BOX, lead_full, co_tile * 128 + 64 + dyo, w0, h0, n0);
#pragma unroll
          for (int t = 0; t < 3; ++t) {
            const int tap = krow * 3 + t;
            const int mid = p.tap_map[tap];
            const CUtensorMap* mx = mid == 0 ? &mX0 : (mid == 1 ? &mX1 : (mid == 2 ? &mX2 : &mX3));
            tma_load_4d_pair(mx, sa + SP::A_ST + t * SP::B_TAP, lead_full, ci_tile * 128 + (int)crank * 64 + xo, w0 + p.tap_dw[tap],
                             h0 + p.tap_dh[tap], n0);
          }
        } else {
          mbar_expect_tx(&full[stage], SP::STAGE_BYTES);
          tma_load_4d(&mDY, sa, &full[stage], co_tile * 128 + dyo, w0, h0, n0);
          tma_load_4d(&mDY, sa + W3_BOX, &full[stage], co_tile * 128 + 64 + dyo, w0, h0, n0);
#pragma unroll
          for (int t = 0; t < 3; ++t) {
            const int tap = krow * 3 + t;
            const int mid = p.tap_map[tap];
            const CUtensorMap* mx = mid == 0 ? &mX0 : (mid == 1 ? &mX1 : (mid == 2 ? &mX2 : &mX3));
            uint8_t* sb = sa + SP::A_ST + t * SP::B_TAP;
            tma_load_4d(mx, sb, &full[stage], ci_tile * 128 + xo, w0 + p.tap_dw[tap], h0 + p.tap_dh[tap], n0);
            tma_load_4d(mx, sb + W3_BOX, &full[stage], ci_tile * 128 + 64 + xo, w0 + p.tap_dw[tap], h0 + p.tap_dh[tap], n0);
          }
        }
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // D=f32, A = dy, B = x (bf16 or fp16), both MN-major (bits 15,16), N=128, M=128 (pair: 256 over the two CTAs)
    const uint32_t idesc = (1u << 4) | (p.fmt_dy << 7) | (p.fmt_x << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(128 >> 3) << 17) |
                           ((uint32_t)((PAIR ? 256 : 128) >> 4) << 24);
    int stage = 0;
    uint32_t phase = 0;
    for (int k = 0; k < n_k && crank == 0; ++k) {
      mbar_wait(&full[stage], phase);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (elect_one()) {
        const uint32_t sa = smem_u32(smem + stage * SP::STAGE_BYTES);
        const uint64_t ad = umma_desc_mn_sw128(sa, W3_BOX);
#pragma unroll
        for (int t = 0; t < 3; ++t) {
          const uint64_t bd = umma_desc_mn_sw128(sa + SP::A_ST + t * SP::B_TAP, W3_BOX);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {  // 4 x (K=16 pixels): advance two 8-row groups = 2048 B
            if constexpr (PAIR)
              umma_bf16_pair(tmem_base + t * 128, ad + (uint64_t)(kk * (2048 >> 4)), bd + (uint64_t)(kk * (2048 >> 4)), idesc,
                             (k | kk) != 0);
            else
              umma_bf16(tmem_base + t * 128, ad + (uint64_t)(kk * (2048 >> 4)), bd + (uint64_t)(kk * (2048 >> 4)), idesc,
                        (k | kk) != 0);
          }
        }
        if constexpr (PAIR) {
          umma_commit_pair(&empty[stage]);
          if (k == n_k - 1) umma_commit_pair(tfull);
        } else {
          umma_commit(&empty[stage]);
          if (k == n_k - 1) umma_commit(tfull);
        }
      }
      __syncwarp();
      if (++stage == STAGES) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (n_k > 0) {
    const int q = warp & 3;
    const int co = co_tile * 128 + q * 32 + lane;
    mbar_wait(tfull, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
    for (int t = 0; t < 3; ++t) {
#pragma unroll 1
      for (int ch = 0; ch < 4; ++ch) {
        uint32_t r[32];
        tmem_ld32(taddr + t * 128 + ch * 32, r);
        if (co < p.Co) {
          float4* dst = reinterpret_cast<float4*>(p.out + (((int64_t)split * p.Co + co) * 9 + krow * 3 + t) * p.Ci +
                                                  ci_tile * 128 + ch * 32);
#pragma unroll
          for (int j = 0; j < 8; ++j)
            dst[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                                 __uint_as_float(r[4 * j + 3]));
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if constexpr (PAIR) {
    __syncwarp();
    cluster_sync_all();
    if (warp == 1)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  } else {
    __syncthreads();
    if (warp == 1) {
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
  }
}
// dst[co][ci][t] (reference layout) = sum_split partial[split][co][t][ci].
// One block per (co, 64 ci): 144 threads = (tap, 4 ci) float4 lanes.  Round 1's kernels kept one 4-byte load in flight per
// thread and ran at 0.9 TB/s (30 us for 28 MB of L2-resident partials, 0.83 ms per step); here every thread keeps eight
// independent 16-byte loads in flight over the splits, sums them in a fixed order (deterministic), and the 576 results go
// through a shared-memory transpose so that the reference layout is written as one contiguous 2304-byte run.
// (second session: the splits are dealt to kRedGroups groups of 144 threads -- group g sums splits g, g + G, ... -- and the
//  group sums are combined in a fixed order through shared memory: with one group the 148-split reduction behind the nine-tap
//  kernel took 42 us on 64 blocks, pure L2 latency)
constexpr int kRedGroups = 4;
__global__ void __launch_bounds__(144 * kRedGroups) wgrad3_reduce_kernel(const float4* __restrict__ part, float* __restrict__ dst,
                                                                          int Co, int Ci, int splits) {
  pdl_wait();
  pdl_trigger();
  __shared__ __align__(16) float tile[64 * 9];
  __shared__ float4 gsum[kRedGroups - 1][144];
  const int cblocks = Ci / 64;
  const int co = blockIdx.x / cblocks, ci0 = (blockIdx.x % cblocks) * 64;
  const int grp = threadIdx.x / 144, l = threadIdx.x % 144;
  const int t = l / 16, c4 = l % 16;   // 9 taps x 16 float4
  const int64_t n4 = (int64_t)Co * 9 * Ci / 4;
  const float4* src = part + (((int64_t)co * 9 + t) * Ci + ci0) / 4 + c4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int sp = grp;
  for (; sp + 7 * kRedGroups < splits; sp += 8 * kRedGroups) {
    float4 v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __ldcg(src + (int64_t)(sp + j * kRedGroups) * n4);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      acc.x += v[j].x;
      acc.y += v[j].y;
      acc.z += v[j].z;
      acc.w += v[j].w;
    }
  }
  for (; sp < splits; sp += kRedGroups) {
    const float4 v = __ldcg(src + (int64_t)sp * n4);
    acc.x += v.x;
    acc.y += v.y;
    acc.z += v.z;
    acc.w += v.w;
  }
  if (grp > 0) gsum[grp - 1][l] = acc;
  __syncthreads();
  if (grp == 0) {
#pragma unroll
    for (int g = 0; g < kRedGroups - 1; ++g) {
      const float4 v = gsum[g][l];
      acc.x += v.x;
      acc.y += v.y;
      acc.z += v.z;
      acc.w += v.w;
    }
    tile[(c4 * 4 + 0) * 9 + t] = acc.x;
    tile[(c4 * 4 + 1) * 9 + t] = acc.y;
    tile[(c4 * 4 + 2) * 9 + t] = acc.z;
    tile[(c4 * 4 + 3) * 9 + t] = acc.w;
  }
  __syncthreads();
  if (threadIdx.x < 144) {
    float4* out = reinterpret_cast<float4*>(dst + ((int64_t)co * Ci + ci0) * 9);
    out[threadIdx.x] = *reinterpret_cast<const float4*>(&tile[threadIdx.x * 4]);
  }
}

// packed fp32 [splits][Co][taps][Ci] -> reference layout [Co][Ci][K][K], the splits added in order
__global__ void wgrad_unpack_kernel(const float* __restrict__ src, float* __restrict__ dst, int Co, int Ci, int KK,
                                    int splits) {
  pdl_wait();
  pdl_trigger();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t n = (int64_t)Co * Ci * KK;
  if (i >= n) return;
  int t = (int)(i % KK);
  int64_t r = i / KK;
  int ci = (int)(r % Ci);
  int co = (int)(r / Ci);
  const float* sp = src + ((int64_t)co * KK + t) * Ci + ci;
  float a = sp[0];
  for (int k = 1; k < splits; ++k) a += sp[(int64_t)k * n];
  dst[i] = a;
}

template <int BNW, int STAGES>
static void launch_wgrad(const CUtensorMap& mDY, const CUtensorMap* mX, const WgradParams& p, lbc_stream_t s) {
  typedef WgradSmem<BNW, STAGES> SP;
  static bool configured = false;
  if (!configured) {
    LBC_CUDA(cudaFuncSetAttribute(wgrad_gemm_kernel<BNW, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, SP::TOTAL));
    configured = true;
  }
  int grid = p.swap ? p.splits * ((p.num_combos + 1) / 2) : p.splits * p.co_tiles * p.num_taps * p.ci_tiles;
  { auto k_ = wgrad_gemm_kernel<BNW, STAGES>; LBC_LAUNCH(k_, dim3(grid), dim3(192), SP::TOTAL, s, mDY, mX[0], mX[1], mX[2], mX[3], p); }
  LBC_LAUNCHED((BNW == 64 ? "wgrad_gemm_kernel<64>" : "wgrad_gemm_kernel<128>"));
  LBC_CUDA(cudaGetLastError());
}

// bit 1 of the pair/variant mode (LBC_PAIR / lbc_set_fast_kernels bit 4): row-of-taps weight-gradient kernel
// (bit 2: its CTA-pair variant where Co % 256 == 0)
// split-K partial scratch, grown on demand; one buffer per kind of split computation, each used from one stream at a time
// (Slot 0: row-of-taps weight gradient [splits][Co][9][Ci], 1: wgrad_gemm [splits][Co][taps][Ci], 2: stem [splits][64][C][49])
template <int Slot>
static float* wgrad_partials(int64_t floats) {
  static float* buf = nullptr;
  static int64_t cap = 0;
  if (floats > cap) {
    if (buf) {
      cudaDeviceSynchronize();
      cudaFree(buf);
    }
    void* q = nullptr;
    if (cudaMalloc(&q, sizeof(float) * (size_t)floats) != cudaSuccess) {
      cudaGetLastError();
      buf = nullptr;
      cap = 0;
      return nullptr;
    }
    buf = (float*)q;
    cap = floats;
  }
  return buf;
}
template <int STAGES, bool PAIR>
static void launch_wgrad3(const CUtensorMap& mDY, const CUtensorMap* mX, const Wgrad3Params& p, int grid, lbc_stream_t s) {
  typedef Wgrad3Smem<STAGES, PAIR> SP;
  static_assert(SP::TOTAL <= 232448, "wgrad3 smem plan exceeds 227 KB");
  auto kern = wgrad3_gemm_kernel<STAGES, PAIR>;
  static bool configured = false;
  if (!configured) {
    LBC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SP::TOTAL));
    configured = true;
  }
  if (!PAIR) {
    { auto k_ = kern; LBC_LAUNCH(k_, dim3(grid), dim3(192), SP::TOTAL, s, mDY, mX[0], mX[1], mX[2], mX[3], p); }
  } else {
    LBC_LAUNCH_CLUSTER(kern, 2, dim3((unsigned)grid), dim3(192), SP::TOTAL, (cudaStream_t)s, mDY, mX[0], mX[1], mX[2], mX[3], p);
  }
  LBC_LAUNCHED((PAIR ? "wgrad3_gemm_kernel<pair>" : "wgrad3_gemm_kernel"));
}
static int wgrad3_pair_slots() {
  static int slots = [] {
    typedef Wgrad3Smem<5, true> SP;
    auto kern = wgrad3_gemm_kernel<5, true>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SP::TOTAL);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)(sm_count() / 2 * 2), 1, 1);
    cfg.blockDim = dim3(192, 1, 1);
    cfg.dynamicSmemBytes = SP::TOTAL;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n <= 0) {
      cudaGetLastError();
      n = sm_count() / 2;
    }
    if (n > sm_count() / 2) n = sm_count() / 2;
    return 2 * n;
  }();
  return slots;
}
// 3x3 / stride 1 / 64 -> 64 channels: all nine taps per CTA (wgrad9_c64_kernel); g_pair_mode bit 6
static bool try_wgrad9(const ConvL& c, const bf16* x, const bf16* dy, float* dw_ref, int B, lbc_stream_t s, const GemmMode& m) {
  if (!(g_pair_mode & 64) || m.split) return false;
  if (c.K != 3 || c.stride != 1 || c.pad != 1 || c.Ci != 64 || c.Co != 64 || (c.W % 8)) return false;
  Wgrad9Params p;
  memset(&p, 0, sizeof(p));
  p.TH = pow2_divisor(c.H, 16);
  if (p.TH < 2) return false;
  p.TN = 16 / p.TH;
  p.tiles_w = c.W / 8;
  p.tiles_h = c.H / p.TH;
  p.tiles_n = (B + p.TN - 1) / p.TN;
  p.k_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  int splits = p.k_tiles < sm_count() ? p.k_tiles : sm_count();
  p.k_per_split = (p.k_tiles + splits - 1) / splits;
  splits = (p.k_tiles + p.k_per_split - 1) / p.k_per_split;
  const int64_t wsize = (int64_t)64 * 9 * 64;
  p.out = wgrad_partials<0>((int64_t)splits * wsize);
  if (!p.out) return false;
  const int64_t eb = 2;
  CUtensorMap mDY = make_map_4d(dy, 64, c.W, c.H, B, 64 * eb, (int64_t)c.W * 64 * eb, (int64_t)c.H * c.W * 64 * eb, 8, p.TH, p.TN);
  CUtensorMap mX = make_map_4d(x, 64, c.W, c.H, B, 64 * eb, (int64_t)c.W * 64 * eb, (int64_t)c.H * c.W * 64 * eb, 10, p.TH + 2, p.TN);
  typedef Wgrad9Smem<4> SP;
  static_assert(SP::TOTAL <= 232448, "wgrad9 smem plan exceeds 227 KB");
  auto kern = wgrad9_c64_kernel<4>;
  static bool configured = false;
  if (!configured) {
    LBC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SP::TOTAL));
    configured = true;
  }
  LBC_LAUNCH(kern, dim3((unsigned)splits), dim3(192), SP::TOTAL, s, mDY, mX, p);
  LBC_LAUNCHED("wgrad9_c64_kernel");
  { auto k_ = wgrad3_reduce_kernel; LBC_LAUNCH(k_, dim3(64u), dim3(144 * kRedGroups), 0, s, (const float4*)p.out, dw_ref, 64, 64, splits); }
  LBC_LAUNCHED("wgrad3_reduce_kernel");
  return true;
}
static bool try_wgrad3(const ConvL& c, const bf16* x, const bf16* dy, float* dw_ref, int B, lbc_stream_t s,
                       const GemmMode& m) {
  if (!(g_pair_mode & 2)) return false;
  const int CX = m.split ? 2 * c.Ci : c.Ci, CY = m.split ? 2 * c.Co : c.Co;   // channels of the stored x / dy tensors
  const bool pair = (g_pair_mode & 4) && (c.Co % 256 == 0);
  if (c.K != 3 || c.pad != 1 || (c.Co % 128) || (c.Ci % 128)) return false;
  Wgrad3Params p;
  memset(&p, 0, sizeof(p));
  // 64-pixel K tile {TW, TH, TN}
  p.TW = pow2_divisor(c.OW, 32);
  p.TH = pow2_divisor(c.OH, 64 / p.TW);
  p.TN = 64 / (p.TW * p.TH);
  if (p.TN > 256) return false;
  p.tiles_w = c.OW / p.TW;
  p.tiles_h = c.OH / p.TH;
  p.tiles_n = (B + p.TN - 1) / p.TN;
  p.k_tiles_real = p.tiles_w * p.tiles_h * p.tiles_n;
  p.k_tiles = (m.split ? 3 : 1) * p.k_tiles_real;
  p.split = m.split ? 1 : 0;
  p.dy_plane = c.Co;
  p.x_plane = c.Ci;
  p.fmt_dy = m.fmt_a;
  p.fmt_x = m.fmt_b;
  p.co_tiles = c.Co / 128;
  p.ci_tiles = c.Ci / 128;
  p.Co = c.Co;
  p.Ci = c.Ci;
  const int out_tiles = p.co_tiles * p.ci_tiles * 3;
  const int slots = pair ? wgrad3_pair_slots() : sm_count();   // CTAs resident at once (one per SM; clusters may fit fewer)
  int best_splits = 1;
  double best_cost = 1e30;
  const int max_splits = p.k_tiles / 8 > 0 ? p.k_tiles / 8 : 1;
  for (int sp = 1; sp <= max_splits && sp <= 148; ++sp) {
    int kps = (p.k_tiles + sp - 1) / sp;
    int real = (p.k_tiles + kps - 1) / kps;
    int ctas = real * out_tiles;
    int waves = (ctas + slots - 1) / slots;
    double cost = (double)waves * (kps + 6);   // k iterations per CTA + prologue / epilogue
    if (cost < best_cost) {
      best_cost = cost;
      best_splits = sp;
    }
  }
  p.k_per_split = (p.k_tiles + best_splits - 1) / best_splits;
  p.splits = (p.k_tiles + p.k_per_split - 1) / p.k_per_split;
  const int64_t eb = 2;
  CUtensorMap mDY = make_map_4d(dy, CY, c.OW, c.OH, B, CY * eb, (int64_t)c.OW * CY * eb, (int64_t)c.OH * c.OW * CY * eb, p.TW,
                                p.TH, p.TN);
  CUtensorMap mX[4];
  if (c.stride == 1) {
    mX[0] = make_map_4d(x, CX, c.W, c.H, B, CX * eb, (int64_t)c.W * CX * eb, (int64_t)c.H * c.W * CX * eb, p.TW, p.TH, p.TN);
    mX[1] = mX[2] = mX[3] = mX[0];
    for (int t = 0; t < 9; ++t) {
      p.tap_dh[t] = t / 3 - c.pad;
      p.tap_dw[t] = t % 3 - c.pad;
      p.tap_map[t] = 0;
    }
  } else {
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b)
        mX[a * 2 + b] = make_map_4d(x + ((int64_t)a * c.W + b) * CX, CX, c.W / 2, c.H / 2, B, 2 * CX * eb,
                                    2 * (int64_t)c.W * CX * eb, (int64_t)c.H * c.W * CX * eb, p.TW, p.TH, p.TN);
    for (int t = 0; t < 9; ++t) {
      int th = t / 3 - c.pad, tw = t % 3 - c.pad;
      int a = ((th % 2) + 2) % 2, b = ((tw % 2) + 2) % 2;
      p.tap_dh[t] = (th - a) / 2;
      p.tap_dw[t] = (tw - b) / 2;
      p.tap_map[t] = a * 2 + b;
    }
  }
  const int64_t wsize = (int64_t)c.Co * 9 * c.Ci;
  p.out = wgrad_partials<0>((int64_t)p.splits * wsize);
  if (!p.out) return false;
  const int grid = p.splits * out_tiles;   // pair: consecutive blocks (2c, 2c+1) form the cluster of co tiles (2c', 2c'+1)
  if (pair)
    launch_wgrad3<5, true>(mDY, mX, p, grid, s);
  else
    launch_wgrad3<3, false>(mDY, mX, p, grid, s);
  { auto k_ = wgrad3_reduce_kernel; LBC_LAUNCH(k_, dim3((unsigned)(c.Co * (c.Ci / 64))), dim3(144 * kRedGroups), 0, s, (const float4*)p.out, dw_ref, c.Co, c.Ci, p.splits); }
  LBC_LAUNCHED("wgrad3_reduce_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}

// x [B,H,W,Ci], dy [B,OH,OW,Co] -> dw_ref fp32 [Co][Ci][K][K]
// (split mode: x [B,H,W,2Ci], dy [B,OH,OW,2Co] as hi | lo planes; fmt_a = format of dy, fmt_b = format of x)
static bool conv_wgrad_impl(const ConvL& c, const bf16* x, const bf16* dy, float* dw_ref, int B, lbc_stream_t s,
                            const GemmMode& m) {
  if (!supported(c)) return false;
  if (m.split && c.Co != 64 && (c.Co % 128)) return false;   // the 128-row dy tile must not run into the lo plane
  const int KK = c.K * c.K;
  const int64_t wsize = (int64_t)c.Co * KK * c.Ci;
  if (try_wgrad9(c, x, dy, dw_ref, B, s, m)) return true;
  if (try_wgrad3(c, x, dy, dw_ref, B, s, m)) return true;
  const int CX = m.split ? 2 * c.Ci : c.Ci, CY = m.split ? 2 * c.Co : c.Co;
  WgradParams p;
  memset(&p, 0, sizeof(p));
  ConvGemmParams g;
  if (!tile_geometry(c.OH, c.OW, B, g)) return false;
  p.TW = g.TW;
  p.TH = g.TH;
  p.TN = g.TN;
  p.tiles_w = g.tiles_w;
  p.tiles_h = g.tiles_h;
  p.tiles_n = g.tiles_n;
  p.k_tiles_real = g.tiles_w * g.tiles_h * g.tiles_n;
  p.k_tiles = (m.split ? 3 : 1) * p.k_tiles_real;
  p.split = m.split ? 1 : 0;
  p.dy_plane = c.Co;
  p.x_plane = c.Ci;
  p.fmt_dy = m.fmt_a;
  p.fmt_x = m.fmt_b;
  p.swap = (c.Co == 64) ? 1 : 0;
  const int BNW = p.swap ? 64 : ((c.Ci % 128 == 0) ? 128 : 64);
  p.co_tiles = (c.Co + 127) / 128;
  p.ci_tiles = c.Ci / BNW;
  p.num_taps = KK;
  p.Co = c.Co;
  p.Ci = c.Ci;
  p.chunks_per_tap = c.Ci / 64;
  p.num_combos = KK * p.chunks_per_tap;
  const int out_tiles = p.swap ? (p.num_combos + 1) / 2 : p.co_tiles * p.ci_tiles * KK;
  // one CTA per SM (shared memory), so the grid runs in waves of sm_count(): pick the K split that fills whole waves
  // (a 297-CTA grid on 148 SMs is THREE waves, the last one with a single CTA).
  int best_splits = 1;
  double best_cost = 1e30;
  const int max_splits = p.k_tiles / 4 > 0 ? p.k_tiles / 4 : 1;
  for (int sp = 1; sp <= max_splits && sp <= 64; ++sp) {
    int kps = (p.k_tiles + sp - 1) / sp;
    int real = (p.k_tiles + kps - 1) / kps;
    int ctas = real * out_tiles;
    int waves = (ctas + sm_count() - 1) / sm_count();
    double cost = (double)waves * (kps + 6);   // time ~ waves x (k iterations per CTA + fixed prologue/epilogue)
    if (cost < best_cost) {
      best_cost = cost;
      best_splits = sp;
    }
  }
  p.k_per_split = (p.k_tiles + best_splits - 1) / best_splits;
  p.splits = (p.k_tiles + p.k_per_split - 1) / p.k_per_split;
  const int64_t eb = 2;
  CUtensorMap mDY = make_map_4d(dy, CY, c.OW, c.OH, B, CY * eb, (int64_t)c.OW * CY * eb, (int64_t)c.OH * c.OW * CY * eb, p.TW,
                                p.TH, p.TN);
  CUtensorMap mX[4];
  if (c.stride == 1) {
    mX[0] = make_map_4d(x, CX, c.W, c.H, B, CX * eb, (int64_t)c.W * CX * eb, (int64_t)c.H * c.W * CX * eb, p.TW, p.TH, p.TN);
    mX[1] = mX[2] = mX[3] = mX[0];
    for (int kh = 0; kh < c.K; ++kh)
      for (int kw = 0; kw < c.K; ++kw) {
        int t = kh * c.K + kw;
        p.tap_dh[t] = kh - c.pad;
        p.tap_dw[t] = kw - c.pad;
        p.tap_map[t] = 0;
      }
  } else {
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b)
        mX[a * 2 + b] = make_map_4d(x + ((int64_t)a * c.W + b) * CX, CX, c.W / 2, c.H / 2, B, 2 * CX * eb,
                                    2 * (int64_t)c.W * CX * eb, (int64_t)c.H * c.W * CX * eb, p.TW, p.TH, p.TN);
    for (int kh = 0; kh < c.K; ++kh)
      for (int kw = 0; kw < c.K; ++kw) {
        int t = kh * c.K + kw;
        int th = kh - c.pad, tw = kw - c.pad;
        int a = ((th % 2) + 2) % 2, b = ((tw % 2) + 2) % 2;
        p.tap_dh[t] = (th - a) / 2;
        p.tap_dw[t] = (tw - b) / 2;
        p.tap_map[t] = a * 2 + b;
      }
  }
  p.out = wgrad_partials<1>((int64_t)p.splits * wsize);
  if (!p.out) return false;
  if (BNW == 128)
    launch_wgrad<128, 3>(mDY, mX, p, s);
  else
    launch_wgrad<64, 4>(mDY, mX, p, s);
  int64_t n = wsize;
  { auto k_ = wgrad_unpack_kernel; LBC_LAUNCH(k_, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, s, (const float*)p.out, dw_ref, c.Co, c.Ci, KK, p.splits); }
  LBC_LAUNCHED("wgrad_unpack_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}
bool conv_wgrad_bf16(const ConvL& c, const bf16* x, const bf16* dy, float* dw_ref, int B, lbc_stream_t s) {
  return conv_wgrad_impl(c, x, dy, dw_ref, B, s, GemmMode());
}

// =============================================================================================================
// fp32tc: split-precision front ends
// =============================================================================================================
template <bool F16>
__global__ void __launch_bounds__(256) split16_kernel(const float4* __restrict__ src, uint4* __restrict__ dst, int64_t rows,
                                                      int C8, float scale) {
  pdl_wait();
  pdl_trigger();
  const int64_t n = rows * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / C8;
    const int g = (int)(i - row * C8);
    const float4 a = __ldg(src + i * 2), b = __ldg(src + i * 2 + 1);
    const float v[8] = {a.x * scale, a.y * scale, a.z * scale, a.w * scale, b.x * scale, b.y * scale, b.z * scale, b.w * scale};
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (F16) {
        const float c0 = fminf(fmaxf(v[2 * j], -65504.f), 65504.f), c1 = fminf(fmaxf(v[2 * j + 1], -65504.f), 65504.f);
        const __half h0 = __float2half_rn(c0), h1 = __float2half_rn(c1);
        const __half l0 = __float2half_rn(c0 - __half2float(h0)), l1 = __float2half_rn(c1 - __half2float(h1));
        hi[j] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
        lo[j] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
      } else {
        const __nv_bfloat16 h0 = __float2bfloat16_rn(v[2 * j]), h1 = __float2bfloat16_rn(v[2 * j + 1]);
        const __nv_bfloat16 l0 = __float2bfloat16_rn(v[2 * j] - __bfloat162float(h0));
        const __nv_bfloat16 l1 = __float2bfloat16_rn(v[2 * j + 1] - __bfloat162float(h1));
        hi[j] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
        lo[j] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
      }
    }
    dst[row * 2 * C8 + g] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    dst[row * 2 * C8 + C8 + g] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}
bool tc_split(const float* src, void* dst16, int64_t rows, int C, int fmt, float scale, lbc_stream_t s) {
  if (C % 8) return false;
  const int64_t n = rows * (C / 8);
  if (n <= 0) return true;
  int64_t blocks = (n + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  if (fmt == TC_F16)
    { auto k_ = split16_kernel<true>; LBC_LAUNCH(k_, dim3((unsigned)blocks), dim3(256), 0, s, (const float4*)src, (uint4*)dst16, rows, C / 8, scale); }
  else
    { auto k_ = split16_kernel<false>; LBC_LAUNCH(k_, dim3((unsigned)blocks), dim3(256), 0, s, (const float4*)src, (uint4*)dst16, rows, C / 8, scale); }
  LBC_LAUNCHED(fmt == TC_F16 ? "split16_kernel<f16>" : "split16_kernel<bf16>");
  LBC_CUDA(cudaGetLastError());
  return true;
}
// one thread per (pixel, k): the 7x7/s2 window element k = (kh*7 + kw)*C + c of the NHWC fp32 image, split into hi | lo planes
template <bool F16>
__global__ void __launch_bounds__(256) tc_stem_im2col_kernel(const float* __restrict__ x0, uint16_t* __restrict__ col, int64_t npix,
                                                             int C, int H, int W, int OH, int OW, int Kp) {
  pdl_wait();
  pdl_trigger();
  const int64_t n = npix * Kp;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pix = i / Kp;
    const int k = (int)(i - pix * Kp);
    float v = 0.f;
    if (k < 49 * C) {
      const int tap = k / C, c = k - tap * C;
      const int kh = tap / 7, kw = tap - kh * 7;
      const int ow = (int)(pix % OW);
      const int64_t t = pix / OW;
      const int oh = (int)(t % OH);
      const int64_t b = t / OH;
      const int ih = oh * 2 - 3 + kh, iw = ow * 2 - 3 + kw;
      if (ih >= 0 && ih < H && iw >= 0 && iw < W) v = __ldg(x0 + ((b * H + ih) * W + iw) * C + c);
    }
    uint16_t hi, lo;
    if (F16) {
      const float cv = fminf(fmaxf(v, -65504.f), 65504.f);
      const __half h = __float2half_rn(cv);
      hi = __half_as_ushort(h);
      lo = __half_as_ushort(__float2half_rn(cv - __half2float(h)));
    } else {
      const __nv_bfloat16 h = __float2bfloat16_rn(v);
      hi = __bfloat16_as_ushort(h);
      lo = __bfloat16_as_ushort(__float2bfloat16_rn(v - __bfloat162float(h)));
    }
    col[pix * 2 * Kp + k] = hi;
    col[pix * 2 * Kp + Kp + k] = lo;
  }
}
bool tc_stem_im2col(const float* x0, void* col16, int B, int C, int H, int W, int OH, int OW, int Kp, int fmt, lbc_stream_t s) {
  const int64_t npix = (int64_t)B * OH * OW;
  int64_t blocks = (npix * Kp + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 32;
  if (blocks > cap) blocks = cap;
  if (fmt == TC_F16)
    { auto k_ = tc_stem_im2col_kernel<true>; LBC_LAUNCH(k_, dim3((unsigned)blocks), dim3(256), 0, s, x0, (uint16_t*)col16, npix, C, H, W, OH, OW, Kp); }
  else
    { auto k_ = tc_stem_im2col_kernel<false>; LBC_LAUNCH(k_, dim3((unsigned)blocks), dim3(256), 0, s, x0, (uint16_t*)col16, npix, C, H, W, OH, OW, Kp); }
  LBC_LAUNCHED("tc_stem_im2col_kernel");
  LBC_CUDA(cudaGetLastError());
  return true;
}
static GemmMode tc_mode(int fmt_a, int fmt_b, float out_scale) {
  GemmMode m;
  m.split = true;
  m.out_f32 = true;
  m.fmt_a = (uint32_t)fmt_a;
  m.fmt_b = (uint32_t)fmt_b;
  m.out_scale = out_scale;
  return m;
}
bool conv_fwd_tc(const ConvL& c, const float* x, const void* x16, float* y, int B, const float* bias_co, bool relu, int x_fmt,
                 const TcWork& w, lbc_stream_t s) {
  if (!enabled() || !supported(c) || !c.wp16) return false;
  if (!x16) {
    const int64_t rows = (int64_t)B * c.H * c.W;
    if (rows * c.Ci * 4 > w.a_bytes) return false;
    if (!tc_split(x, w.a16, rows, c.Ci, x_fmt, 1.0f, s)) return false;
    x16 = w.a16;
  }
  // (tcgen05.mma kind::f16 takes ONE 16-bit format per instruction: fp16 x bf16 traps as an illegal instruction on the B200,
  // so c.wp16 must have been split in x_fmt)
  return conv_fwd_impl(c, x16, c.wp16, y, B, bias_co, relu, s, nullptr, nullptr, tc_mode(x_fmt, x_fmt, 1.0f / kTcWeightScale));
}
bool conv_dgrad_tc(const ConvL& c, const float* dy, const float* dy_ds, float* dx, int B, const float* bias_ci, bool relu,
                   int dy_fmt, const TcWork& w, lbc_stream_t s) {
  if (!enabled() || !supported(c) || !c.wpt16 || c.K == 1) return false;
  if (dy_ds && (!c.wcomb16 || c.stride != 2 || c.K != 3)) return false;
  const int64_t rows = (int64_t)B * c.OH * c.OW;
  if (rows * c.Co * 4 > w.a_bytes || (dy_ds && rows * c.Co * 4 > w.b_bytes)) return false;
  if (!tc_split(dy, w.a16, rows, c.Co, dy_fmt, 1.0f, s)) return false;
  if (dy_ds && !tc_split(dy_ds, w.b16, rows, c.Co, dy_fmt, 1.0f, s)) return false;
  return conv_dgrad_impl(c, w.a16, c.wpt16, c.wcomb16, dx, B, bias_ci, relu, dy_ds ? w.b16 : nullptr, s,
                         tc_mode(dy_fmt, dy_fmt, 1.0f / kTcWeightScale));   // c.wpt16 / c.wcomb16 split in dy_fmt
}
bool conv_wgrad_tc(const ConvL& c, const float* x, const void* x16, const float* dy, float* dw_ref, int B, int x_fmt, int dy_fmt,
                   const TcWork& w, lbc_stream_t s) {
  if (!enabled() || !supported(c) || x_fmt != dy_fmt) return false;   // one operand format per MMA
  const int64_t rx = (int64_t)B * c.H * c.W, ry = (int64_t)B * c.OH * c.OW;
  if (ry * c.Co * 4 > w.b_bytes) return false;
  if (!x16) {
    if (rx * c.Ci * 4 > w.a_bytes) return false;
    if (!tc_split(x, w.a16, rx, c.Ci, x_fmt, 1.0f, s)) return false;
    x16 = w.a16;
  }
  if (!tc_split(dy, w.b16, ry, c.Co, dy_fmt, 1.0f, s)) return false;
  return conv_wgrad_impl(c, (const bf16*)x16, (const bf16*)w.b16, dw_ref, B, s, tc_mode(dy_fmt, x_fmt, 1.0f));
}

#else   // LBC_HOST_EMU: no tensor cores on the host; the executor runs the correctness-first kernels
bool conv_fwd_bf16(const ConvL&, const bf16*, bf16*, int, const float*, lbc_stream_t, float*, int*) { return false; }
bool conv_dgrad_bf16(const ConvL&, const bf16*, bf16*, int, const float*, bool, lbc_stream_t) { return false; }
bool conv_wgrad_bf16(const ConvL&, const bf16*, const bf16*, float*, int, lbc_stream_t) { return false; }
bool conv_dgrad_ds_bf16(const ConvL&, const bf16*, const bf16*, bf16*, int, lbc_stream_t) { return false; }
void set_c64_variant(bool) {}
void set_pair_mode(int) {}
int pair_mode() { return 0; }
bool stem_s2d() { return false; }
bool stem_conv_bf16(const bf16*, const bf16*, bf16*, int, int, int, int, int, const float*, float*, int*, lbc_stream_t, int) { return false; }
bool stem_wgrad_bf16(const bf16*, const bf16*, float*, int, int, int, int, int, int, lbc_stream_t, int) { return false; }
bool tc_split(const float*, void*, int64_t, int, int, float, lbc_stream_t) { return false; }
bool conv_fwd_tc(const ConvL&, const float*, const void*, float*, int, const float*, bool, int, const TcWork&, lbc_stream_t) { return false; }
bool conv_dgrad_tc(const ConvL&, const float*, const float*, float*, int, const float*, bool, int, const TcWork&, lbc_stream_t) { return false; }
bool conv_wgrad_tc(const ConvL&, const float*, const void*, const float*, float*, int, int, int, const TcWork&, lbc_stream_t) { return false; }
bool tc_stem_im2col(const float*, void*, int, int, int, int, int, int, int, int, lbc_stream_t) { return false; }
#endif

}  // namespace fast
}  // namespace lbc
