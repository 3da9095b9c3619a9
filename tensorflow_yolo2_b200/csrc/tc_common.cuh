// tc_common.cuh -- PTX wrappers (mbarrier, TMA, tcgen05) and host-side tensor-map plumbing shared by the
// tensor-core kernels (conv_tcgen05.cu: forward / dgrad, conv_wgrad_tcgen05.cu: weight gradient).
#pragma once
#include <cuda.h>
#include <type_traits>
#include <mutex>
#include <cstring>
#include <cstdlib>

#include "common.cuh"

namespace y2 {

// q = n / d for 0 <= n < 2^31 with host-computed (mul, shr); d == 1 encoded as mul == 0
__device__ __forceinline__ uint32_t fdiv(uint32_t n, uint32_t mul, uint32_t shr) {
  return mul ? (__umulhi(n, mul) >> shr) : n;
}

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
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
// identity the compiler cannot see through: keeps a loop-invariant value in a register instead of re-deriving it
// (S2R / constant-bank loads / address arithmetic) inside a latency-bound single-warp loop
__device__ __forceinline__ uint32_t opaque(uint32_t x) {
  asm volatile("mov.b32 %0, %0;" : "+r"(x));
  return x;
}
// wait on a barrier given by its 32-bit shared address (hot loops keep the addresses in registers: converting a
// generic pointer costs an S2R + two integer ops every time, and the single-warp roles are latency-bound)
__device__ __forceinline__ void mbar_wait_a(uint32_t addr, uint32_t parity) {
  uint32_t ok = 0;
  long long t0 = 0;
  uint32_t spins = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (ok) break;
    if ((++spins & 0xfff) == 0) {
      long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 6000000000ll) {   // ~3 s at 2 GHz: a protocol bug, not a slow tile
        printf("y2 conv_tc: mbarrier timeout block %d thread %d\n", blockIdx.x, threadIdx.x);
        __trap();
      }
    }
  }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) { mbar_wait_a(smem_u32(bar), parity); }
__device__ __forceinline__ void mbar_expect_tx_a(uint32_t addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_im2col_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c, int w, int h,
                                                   int n, uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h)
      : "memory");
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void umma_commit_a(uint32_t addr) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(addr) : "memory");
}
// ---- CTA pairs (tcgen05 cta_group::2): one MMA spans two SMs, each CTA feeds its own 128 rows of A and HALF of B ----
// shared::cluster addresses carry the CTA rank in bit 24; clearing it addresses the same offset in the pair's leader
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;
constexpr uint64_t TMA_CACHE_HINT_DEFAULT = 0x1000000000000000ull;
// TMA loads whose completion may be signalled on the LEADER's mbarrier (bar = leader-mapped address)
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "l"(TMA_CACHE_HINT_DEFAULT)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_2sm(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], %7;" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(TMA_CACHE_HINT_DEFAULT)
      : "memory");
}
__device__ __forceinline__ void tma_load_im2col_4d_2sm(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c, int w, int h,
                                                       int n, uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.im2col.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8}, %9;" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h),
      "l"(TMA_CACHE_HINT_DEFAULT)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// arrive (once the pair's MMAs issued so far have retired) on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_2sm_mc(uint32_t addr, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(addr),
               "h"(mask)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA store of a 4-D box from shared memory (bulk async-group completion); OOB parts of the box are clipped
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* tm, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tm)),
               "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
// [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [49,52) base_offset | [61,64) layout
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t addr, uint32_t lbo, uint32_t sbo, uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3fff);
  d |= (uint64_t)((lbo >> 4) & 0x3fff) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3fff) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(layout_type & 7) << 61;
  return d;
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*PFN_encodeIm2col)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                     const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                     CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
extern PFN_encodeTiled g_encodeTiled;
extern PFN_encodeIm2col g_encodeIm2col;
int num_sms();                    // SM count of the CURRENT device (cached per device ordinal)
#define g_num_sms (::y2::num_sms())
extern int g_driver_version;

int load_driver_entry_points();   // defined in conv_tcgen05.cu

// Tensor maps shared by the tensor-core kernels (defined in conv_tcgen05.cu).  Each returns Y2_OK, or sets the error
// "<who>: tensor map <name> encode failed" and returns Y2_ERR_DRIVER.
// bf16 NHWC [N][H][W][C] read in im2col mode for a ksize x ksize SAME window: `pixels` rows of `chans` channels per load
int tmap_im2col_nhwc(CUtensorMap* tm, const void* x, int N, int H, int W, int C, int ksize, int chans, int pixels,
                     CUtensorMapSwizzle sw, const char* who, const char* name);
// NHWC [N][H][W][C] of bf16 or float32 whose pixels are `ld` elements apart, read or written in [c, w, h, n] boxes
int tmap_nhwc_box(CUtensorMap* tm, const void* base, CUtensorMapDataType dt, int N, int H, int W, int C, int ld,
                  const cuuint32_t box[4], CUtensorMapSwizzle sw, CUtensorMapL2promotion l2, const char* who, const char* name);
// bf16 K-major rows [rows][K] (packed weights, row-major gradients), read in [box_k, box_rows] boxes
int tmap_kmajor(CUtensorMap* tm, const void* base, int K, long long rows, int box_k, int box_rows, CUtensorMapSwizzle sw,
                CUtensorMapL2promotion l2, const char* who, const char* name);

// Launch with a cluster dimension and, unless Y2_NO_PDL is set, programmatic dependent launch (fill_launch_attrs)
template <typename... KArgs, typename... Args>
static int launch_cluster(void (*kernel)(KArgs...), int grid, int threads, size_t smem, unsigned cluster, cudaStream_t st,
                          const Args&... args) {
  Y2_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  cfg.attrs = attr;
  cfg.numAttrs = fill_launch_attrs(attr, cluster);
  Y2_CUDA(cudaLaunchKernelEx(&cfg, kernel, args...));
  Y2_LAUNCHED();
  return Y2_OK;
}

// One y2_conv_fwd_bf16 call, parsed and checked before any kernel path sees it.  The paths (stream-K, input-stationary,
// generic) only decide whether they can run it.
struct ConvCall {
  const void* x;
  const void* w_packed;
  const float* scale;
  const float* shift;
  void* y;
  float alpha;
  int flags;
  int N, H, W, Cin, Cout, ksize, pad, taps;
  long long M;                      // N * H * W output rows before pooling
  bool split_in, split_out, out_f32, pool, leaky;   // split_out: OUT_SPLIT without OUT_F32
  int ldy, lo_off;                  // resolved: ldy >= Cout; with split_out lo_off >= Cout and ldy >= lo_off + Cout, else 0
  int a_cin;                        // channels per pixel of x: 2 Cin ([hi | lo]) with IN_SPLIT, else y2_conv_cin_padded(Cin)
  int b_cin;                        // K extent per tap of w_packed: 3 Cin ([w_hi | w_hi | w_lo]) with IN_SPLIT, else a_cin
};

static inline CUtensorMapSwizzle swizzle_for(int row_bytes) {
  return row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                                          : CU_TENSOR_MAP_SWIZZLE_NONE;
}

static inline void fastdiv_init(uint32_t d, uint32_t* mul, uint32_t* shr) {
  if (d <= 1) { *mul = 0; *shr = 0; return; }
  uint32_t l = 0;
  while ((1u << l) < d) ++l;                       // ceil(log2 d)
  uint32_t p = 31 + l;
  *mul = (uint32_t)(((1ull << p) + d - 1) / d);
  *shr = p - 32;
}

static inline int ilog2(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}

}  // namespace y2
