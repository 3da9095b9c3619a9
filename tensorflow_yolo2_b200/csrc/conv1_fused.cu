// conv1_fused.cu -- a10 + a1 + a2 + a3 for the FIRST Darknet19 layer in one kernel:
//
//   uint8 BGR image  --(x/255*2-1, pascal_voc.py:62-64)-->  3x3 conv 3->32 (darknet.py:20-21,150)
//   --> BN scale/shift (scale folded into the weights, shift added in the epilogue; darknet.py:42-44)
//   --> 2x2 max-pool (darknet.py:24-25,151) --> leaky (darknet.py:45)  --> bf16 [N, H/2, W/2, 32]
//
// (max-pool and leaky commute because leaky is monotonic; the shift commutes with max; the scale does not when it is
// negative, which is why it lives in the weights.)
//
// The generic implicit-GEMM kernel spends ~1000 clk per 128-pixel tile on this layer, almost all of it epilogue
// instructions (affine + leaky + cross-lane pooling on every conv pixel) and 16-byte-per-pixel operand traffic
// (the input padded 3 -> 8 channels).  Here instead:
//
//   * the input is read as raw uint8 (3 B/pixel): ONE TMA box (34 rows x 80 B, uint8 tensor map over the image,
//     16-byte aligned start) per tile into a raw smem ring; converter warps turn it into bf16 (one FFMA per
//     byte, bit-identical to the preprocessing kernel after the bf16 rounding) and lay it out as a [34 rows][18 px][4 ch] patch --
//     the padded bf16 input never exists in HBM.  (34 separate 80-byte cp.async.bulk row copies per tile were
//     measured at ~100 clk each in the TMA unit: 3500 clk per tile.)
//   * GEMM rows are POOLED pixels (tile = 8 x 16 pooled = 16 x 32 conv pixels) and GEMM columns are
//     (window position, channel) = 4 x 32 = 128: each pooled pixel multiplies its 4x4 input footprint
//     (K = 16 px x 4 ch = 64) with a [128 x 64] matrix that holds the 3x3 filter at the four window shifts.  A
//     footprint row is 32 contiguous bytes of the patch, so one tcgen05.mma (K = 16) per footprint row: 4 MMAs
//     per tile, operands addressed with (start, LBO = 16 B, SBO = 2 patch rows) descriptor arithmetic only;
//   * the 2x2 max-pool is then a max over four column groups of the thread's OWN TMEM lane: no shuffles, every
//     epilogue lane produces one output pixel (64 contiguous bytes).
//
// Warp roles (960 threads): 0-15 epilogue (four groups of four, one per TMEM buffer), 16-23 converters (each warp
// converts whole tiles into its own patch stage, so eight conversions are in flight), 24-25 TMA producers, 26-29 MMA
// issuers (one per TMEM buffer).  Every role is latency-bound per tile (a satisfied mbarrier try_wait alone costs ~90 clk
// and a tile is only 256 clk of tensor work), so each role is replicated until its per-tile latency / replicas < ~300 clk.
// Persistent grid, static round-robin over tiles; tile coordinates by magic-number division (a runtime integer
// division costs ~150 clk of dependent latency per role per tile -- measured, it dominated the first version).
#include "tc_common.cuh"

namespace y2 {

constexpr int C1_COUT = 32;
constexpr int C1_TW = 8, C1_TH = 16;                    // pooled pixels per tile
constexpr int C1_PROWS = 2 * C1_TH + 2;                 // 34 patch rows
constexpr int C1_PCOLS = 2 * C1_TW + 2;                 // 18 patch pixels per row
constexpr int C1_PITCH = C1_PCOLS * 8;                  // 144 B (4 bf16 channels per pixel)
constexpr int C1_A_STAGE = 5120;                        // >= 34 * 144 = 4896
constexpr int C1_CVT_WARPS = 8;                         // each converter warp owns whole tiles (tile it -> warp it % 8)
constexpr int C1_A_STAGES = C1_CVT_WARPS;               // ... and its own patch stage
constexpr int C1_RAW_ROW = 80;                          // TMA box row: starts 16-byte aligned, 13 B before the patch
constexpr int C1_RAW_LEAD = 13;                         // 3*(2*pw0 - 1) = 48*tw - 3  ->  box starts at 48*tw - 16
constexpr int C1_RAW_BYTES = C1_PROWS * C1_RAW_ROW;     // 2720 B delivered per tile
constexpr int C1_RAW_STAGE = 2816;                      // ring slot (128-byte aligned)
constexpr int C1_RAW_STAGES = 16;
constexpr int C1_B_BYTES = 4 * 2 * 128 * 16;            // [ty][k-group][n = 128][8] bf16 = 16 KB
constexpr int C1_NBUF = 4;                              // TMEM accumulator ring: 4 x 128 columns
constexpr int C1_EPI_GROUPS = 4;                        // epilogue groups of 4 warps (one warp per TMEM lane quarter);
                                                        // group e owns TMEM buffer e
constexpr int C1_EPI_WARPS = 4 * C1_EPI_GROUPS;
constexpr int C1_PROD_WARPS = 2, C1_MMA_WARPS = 4;      // single-thread roles are latency-bound (a satisfied mbarrier
                                                        // try_wait costs ~90 clk): several of each, on alternate tiles
constexpr int C1_WARP_PRODUCER = C1_EPI_WARPS + C1_CVT_WARPS;
constexpr int C1_WARP_MMA = C1_WARP_PRODUCER + C1_PROD_WARPS;
constexpr int C1_THREADS = (C1_WARP_MMA + C1_MMA_WARPS) * 32;
static_assert(C1_MMA_WARPS == C1_NBUF && C1_EPI_GROUPS == C1_NBUF, "MMA warp m / epilogue group m own TMEM buffer m");
// Ownership rule: successive phases of one mbarrier are always waited on by the SAME warp(s).  A waiter that may run two
// phases ahead of a barrier mistakes the older completed phase of equal parity for its own (3 epilogue groups over 4
// buffers dead-locked exactly this way at 146 tiles per CTA while passing every small test).
static_assert(C1_A_STAGES % C1_MMA_WARPS == 0 && C1_RAW_STAGES % C1_CVT_WARPS == 0 && C1_RAW_STAGES % C1_PROD_WARPS == 0,
              "stage -> warp ownership must be static");
// Output staging for the TMA-store epilogue: one buffer per epilogue group, 128 pooled pixels x 64 B (bf16) / 128 B ([hi | lo]);
// a group owns every fourth tile, so its previous box store has long been read out of smem when it writes the next one.
constexpr int C1_STG = 128 * 64;
constexpr size_t C1_SMEM = 1024 + C1_B_BYTES + C1_A_STAGES * C1_A_STAGE + C1_RAW_STAGES * C1_RAW_STAGE + C1_EPI_GROUPS * C1_STG + 1024;
// bf16x3 variant (SPLIT): the patch holds the raw bytes as EXACT bf16 integers (v0, v1, v2) plus a "ones" channel that is
// 1 inside the image and 0 in the SAME-padding halo; the preprocessing x = v*2/255 - 1 is folded into the weights
// (w*2/255 on the colour channels, -sum_c w on the ones channel), which are kept as a hi + lo bf16 pair.  So A is exact,
// B carries 16 mantissa bits, and a tile costs 8 MMAs (4 footprint rows x {hi, lo}) into the same accumulator.  The output
// row is [hi(32) | lo(32)] (Y2_CONV_OUT_SPLIT layout).
constexpr size_t C1_SMEM_SPLIT = C1_SMEM + C1_B_BYTES + C1_EPI_GROUPS * C1_STG;

struct Conv1Args {
  const uint4* w_packed;
  const float* shift;
  __nv_bfloat16* y;
  int N, H, W;
  int tiles_w, tiles_per_img, total_tiles;
  uint32_t fd_img_mul, fd_img_shr, fd_w_mul, fd_w_shr;   // magic-number division by tiles_per_img / tiles_w
  float alpha;
};

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}

// packed float32 pairs (sm_100 FADD2 / FMUL2: one issue slot for two lanes of arithmetic; IEEE results identical to the scalar ops)
__device__ __forceinline__ void c1_add2(float& a0, float& a1, float b0, float b1) {
  asm("{ .reg .b64 ra, rb, rc;\n mov.b64 ra, {%0, %1};\n mov.b64 rb, {%2, %3};\n add.rn.f32x2 rc, ra, rb;\n mov.b64 {%0, %1}, rc; }"
      : "+f"(a0), "+f"(a1)
      : "f"(b0), "f"(b1));
}
__device__ __forceinline__ void c1_mul2(float& d0, float& d1, float a0, float a1, float b) {
  asm("{ .reg .b64 ra, rb, rc;\n mov.b64 ra, {%2, %3};\n mov.b64 rb, {%4, %4};\n mul.rn.f32x2 rc, ra, rb;\n mov.b64 {%0, %1}, rc; }"
      : "=f"(d0), "=f"(d1)
      : "f"(a0), "f"(a1), "f"(b));
}

struct C1Tile {
  int n, ph0, pw0;
};
__device__ __forceinline__ C1Tile c1_tile(const Conv1Args& a, int tile) {
  C1Tile t;
  t.n = (int)fdiv((uint32_t)tile, a.fd_img_mul, a.fd_img_shr);
  const int rem = tile - t.n * a.tiles_per_img;
  const int th = (int)fdiv((uint32_t)rem, a.fd_w_mul, a.fd_w_shr);
  t.ph0 = th * C1_TH;
  t.pw0 = (rem - th * a.tiles_w) * C1_TW;
  return t;
}

template <bool SPLIT>
__global__ void __launch_bounds__(C1_THREADS, 1)
conv1_u8_pool_kernel(const __grid_constant__ CUtensorMap tmImg, const __grid_constant__ CUtensorMap tmY, const Conv1Args a) {
  constexpr int B_BYTES = SPLIT ? 2 * C1_B_BYTES : C1_B_BYTES;
  pdl_launch_dependents();   // persistent grid: layer 2 (launched with programmatic serialization) may take SMs as my CTAs retire
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t raw_full[C1_RAW_STAGES], raw_empty[C1_RAW_STAGES];
  __shared__ __align__(8) uint64_t a_full[C1_A_STAGES], a_empty[C1_A_STAGES];
  __shared__ __align__(8) uint64_t tmem_full[C1_NBUF], tmem_empty[C1_NBUF];
  __shared__ uint32_t s_tmem_base;
  __shared__ __align__(16) float s_shift[C1_COUT];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t sm0 = (smem_u32(smem) + 1023u) & ~1023u;
  const uint32_t sB = sm0;
  const uint32_t sA = sB + B_BYTES;
  const uint32_t sRaw = sA + C1_A_STAGES * C1_A_STAGE;
  constexpr uint32_t STG_BYTES = SPLIT ? 2 * C1_STG : C1_STG, STG_ROW = SPLIT ? 128 : 64;
  const uint32_t sStg = (sRaw + C1_RAW_STAGES * C1_RAW_STAGE + 1023u) & ~1023u;      // swizzle atoms: 1024-byte aligned
  uint8_t* const gen0 = smem + (sm0 - smem_u32(smem));              // generic pointer to the aligned base

  // ---- one-time setup ----
  if (threadIdx.x < C1_COUT) s_shift[threadIdx.x] = a.shift ? __ldg(a.shift + threadIdx.x) : 0.0f;
  for (int i = threadIdx.x; i < B_BYTES / 16; i += C1_THREADS)
    reinterpret_cast<uint4*>(gen0)[i] = __ldg(a.w_packed + i);
  fence_proxy_async_smem();                                         // B is read by the tensor core (async proxy)
  if (warp == C1_WARP_PRODUCER && lane == 0) {
    for (int s = 0; s < C1_RAW_STAGES; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], 1); }
    for (int s = 0; s < C1_A_STAGES; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
    for (int b = 0; b < C1_NBUF; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], 4); }
    fence_barrier_init();
  }
  if (warp == C1_WARP_MMA) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem_base)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;
  const int first = blockIdx.x, step = gridDim.x;

  if (warp >= C1_WARP_PRODUCER && warp < C1_WARP_MMA) {
    // =========================== raw uint8 patch: one TMA box per tile ===========================
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmImg)) : "memory");
      for (int it = warp - C1_WARP_PRODUCER;; it += C1_PROD_WARPS) {
        const int tile = first + it * step;
        if (tile >= a.total_tiles) break;
        const int rs = it % C1_RAW_STAGES;
        const C1Tile t = c1_tile(a, tile);
        mbar_wait(&raw_empty[rs], ((uint32_t)(it / C1_RAW_STAGES) & 1u) ^ 1u);
        mbar_expect_tx(&raw_full[rs], C1_RAW_BYTES);
        // bytes [6*pw0 - 16, +80) of rows 2ph0-1 .. 2ph0+32 (the TMA wants a 16-byte aligned start: an unaligned
        // byte coordinate raises "illegal instruction"); out-of-image bytes arrive as 0 and are masked below
        tma_load_3d(sRaw + rs * C1_RAW_STAGE, &tmImg, smem_u32(&raw_full[rs]), 6 * t.pw0 - 16, 2 * t.ph0 - 1, t.n);
      }
    }
  } else if (warp >= C1_EPI_WARPS && warp < C1_WARP_PRODUCER) {
    // =========================== converters: raw uint8 -> bf16 patch, one warp per tile ===========================
    const int cw = warp - C1_EPI_WARPS;                     // my patch stage
    const uint32_t dstA = sA + cw * C1_A_STAGE;
    for (int it = cw;; it += C1_CVT_WARPS) {
      const int tile = first + it * step;
      if (tile >= a.total_tiles) break;
      const int rs = it % C1_RAW_STAGES;
      const C1Tile t = c1_tile(a, tile);
      mbar_wait(&raw_full[rs], (uint32_t)(it / C1_RAW_STAGES) & 1u);
      mbar_wait(&a_empty[cw], ((uint32_t)(it / C1_A_STAGES) & 1u) ^ 1u);
      const uint8_t* raw = gen0 + (sRaw - sm0) + rs * C1_RAW_STAGE;
      const int row0 = 2 * t.ph0 - 1, col0 = 2 * t.pw0 - 1;
      // One patch ROW per lane: the 80 raw bytes arrive in five conflict-free 16-byte loads (rows are 80 B apart), the 54
      // image bytes sit at COMPILE-TIME positions (lead of 13 bytes), so every byte is one PRMT into the mantissa of 2^23,
      // one FADD (exact) and -- bf16 mode -- one FFMA: all independent, no byte loads, no I2F.  The per-task version (two
      // pixels per lane and iteration: 6 byte loads -> I2F -> FFMA -> pack -> store, a serial chain) took ~5 500 clk per
      // tile and warp; with four converter warps the kernel was conversion-bound at 120 us (r2n ablation).
      // rows 0..31: one per lane (static byte positions); rows 32..33: their 18 two-pixel units go to lanes 0..17 with
      // byte loads (a second full row pass would issue 235 instructions for two active lanes)
      static_assert(C1_PROWS == 34 && C1_PCOLS == 18, "converter passes are laid out for a 34 x 18 patch");
#pragma unroll 1
      for (int pass = 0; pass < 2; ++pass) {
        if (pass == 1 && lane >= 2 * (C1_PCOLS / 2)) break;
        const int pr = pass == 0 ? lane : 32 + lane / (C1_PCOLS / 2);
        const int jt = pass == 0 ? 0 : lane % (C1_PCOLS / 2);
        uint32_t w[20];
        if (pass == 0) {
#pragma unroll
          for (int i = 0; i < 5; ++i) {
            const uint4 q = *reinterpret_cast<const uint4*>(raw + pr * C1_RAW_ROW + 16 * i);
            w[4 * i] = q.x; w[4 * i + 1] = q.y; w[4 * i + 2] = q.z; w[4 * i + 3] = q.w;
          }
        } else {
          const uint8_t* pb = raw + pr * C1_RAW_ROW + C1_RAW_LEAD + 6 * jt;    // place the unit's 6 bytes where unit 0 is read from
          w[3] = (uint32_t)pb[0] << 8 | (uint32_t)pb[1] << 16 | (uint32_t)pb[2] << 24;
          w[4] = (uint32_t)pb[3] | (uint32_t)pb[4] << 8 | (uint32_t)pb[5] << 16;
        }
        const bool rok = (unsigned)(row0 + pr) < (unsigned)a.H;
#pragma unroll
        for (int j = 0; j < C1_PCOLS / 2; ++j) {
          if (pass == 1 && j > 0) break;
          const int jj = pass == 0 ? j : jt;                           // which unit of the row this is
          const int ca = col0 + 2 * jj;
          const bool va = rok && ca >= 0, vb = rok && ca + 1 < a.W;
          float f[6];
#pragma unroll
          for (int k = 0; k < 6; ++k) {
            const int bi = C1_RAW_LEAD + 6 * j + k;                  // compile-time after unrolling
            f[k] = __uint_as_float(__byte_perm(w[bi >> 2], 0x4B000000u, 0x7650u | (uint32_t)(bi & 3))) - 8388608.0f;
          }
          uint32_t w0 = 0, w1 = 0, w2 = 0, w3 = 0;
          if constexpr (SPLIT) {
            // exact integers (8 significant bits fit bf16); channel 3 = 1.0 inside the image
            if (va) {
              w0 = __byte_perm(__float_as_uint(f[0]), __float_as_uint(f[1]), 0x7632);
              w1 = (__float_as_uint(f[2]) >> 16) | 0x3f800000u;
            }
            if (vb) {
              w2 = __byte_perm(__float_as_uint(f[3]), __float_as_uint(f[4]), 0x7632);
              w3 = (__float_as_uint(f[5]) >> 16) | 0x3f800000u;
            }
          } else {
            // bf16_rn(fma(v, 2/255, -1)) == bf16_rn((v/255)*2 - 1) for all 256 byte values (tests/test_abi_cpu.py)
            const float kk = 2.0f / 255.0f;
            if (va) {
              const __nv_bfloat162 h0 = __floats2bfloat162_rn(fmaf(f[0], kk, -1.0f), fmaf(f[1], kk, -1.0f));
              const __nv_bfloat162 h1 = __floats2bfloat162_rn(fmaf(f[2], kk, -1.0f), 0.0f);        // channel 3 is zero padding
              w0 = *reinterpret_cast<const uint32_t*>(&h0);
              w1 = *reinterpret_cast<const uint32_t*>(&h1);
            }
            if (vb) {
              const __nv_bfloat162 h2 = __floats2bfloat162_rn(fmaf(f[3], kk, -1.0f), fmaf(f[4], kk, -1.0f));
              const __nv_bfloat162 h3 = __floats2bfloat162_rn(fmaf(f[5], kk, -1.0f), 0.0f);
              w2 = *reinterpret_cast<const uint32_t*>(&h2);
              w3 = *reinterpret_cast<const uint32_t*>(&h3);
            }
          }
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dstA + pr * C1_PITCH + jj * 16), "r"(w0), "r"(w1), "r"(w2),
                       "r"(w3)
                       : "memory");
        }
      }
      fence_proxy_async_smem();                       // patch is consumed by tcgen05.mma (async proxy)
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&a_full[cw]);
        mbar_arrive(&raw_empty[rs]);
      }
    }
  } else if (warp >= C1_WARP_MMA) {
    // =========================== MMA issuers: warp m takes tiles it = m, m + 4, ... (TMEM buffer m) ===========================
    const int mw = warp - C1_WARP_MMA;
    uint32_t is_leader;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(is_leader));
    // D = f32, A = B = bf16, both K-major, N = 128, M = 128
    constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    // A: row r = (g, i) of footprint row ty lives at patch + (2g + ty) * PITCH + i * 16, 32 contiguous bytes
    const uint64_t adesc0 = make_smem_desc(sA, 16u, 2u * C1_PITCH, 0u);
    const uint64_t bdesc0 = make_smem_desc(sB, 2048u, 128u, 0u);
    const uint32_t tmem_d = tmem_base + (uint32_t)(mw * 128);
    uint32_t use = 0;                                   // how many times this warp's TMEM buffer has been filled
    for (int it = mw;; it += C1_MMA_WARPS, ++use) {
      const int tile = first + it * step;
      if (tile >= a.total_tiles) break;
      const int as = it % C1_A_STAGES;
      mbar_wait(&a_full[as], (uint32_t)(it / C1_A_STAGES) & 1u);
      mbar_wait(&tmem_empty[mw], (use & 1u) ^ 1u);
      tc_fence_after();
      if (is_leader) {
        const uint64_t ad = adesc0 + (uint32_t)((as * C1_A_STAGE) >> 4);
#pragma unroll
        for (int ty = 0; ty < 4; ++ty)
          umma_bf16(tmem_d, ad + (uint32_t)((ty * C1_PITCH) >> 4), bdesc0 + (uint32_t)((ty * 4096) >> 4), idesc, ty > 0);
        if constexpr (SPLIT) {
#pragma unroll
          for (int ty = 0; ty < 4; ++ty)          // the lo halves of the weights, same patch rows
            umma_bf16(tmem_d, ad + (uint32_t)((ty * C1_PITCH) >> 4), bdesc0 + (uint32_t)((C1_B_BYTES + ty * 4096) >> 4), idesc, 1u);
        }
        umma_commit(&a_empty[as]);
        umma_commit(&tmem_full[mw]);
      }
      __syncwarp();
    }
  } else {
    // =========================== epilogue: pool over the 4 column groups, +shift, leaky, store ===========================
    const int q = warp & 3, eg = warp >> 2;
    const int r = q * 32 + lane;
    const float alpha = a.alpha;
    const bool st_leader = q == 0 && lane == 0;
    // my row of the staging box (pooled pixel (ph0 + (r >> 3), pw0 + (r & 7)), STG_ROW bytes); 16-byte unit u sits at u ^ swz
    // (SWIZZLE_64B / _128B)
    const uint32_t stg_row = sStg + (uint32_t)eg * STG_BYTES + (uint32_t)r * STG_ROW;
    const uint32_t swz = SPLIT ? (uint32_t)(r & 7) : (uint32_t)((r >> 1) & 3);
    for (int it = eg;; it += C1_EPI_GROUPS) {
      const int tile = first + it * step;
      if (tile >= a.total_tiles) break;
      const int buf = it % C1_NBUF;
      const C1Tile t = c1_tile(a, tile);
      mbar_wait(&tmem_full[buf], (uint32_t)(it / C1_NBUF) & 1u);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * 128);
      if (st_leader) bulk_wait_group_read<0>();          // my group's previous box store has read the staging buffer
      asm volatile("bar.sync %0, 128;" ::"r"(1 + eg) : "memory");
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {                  // 8 output channels at a time
        uint32_t v0[8], v1[8], v2[8], v3[8];
        tmem_ld8(taddr + 0 * 32 + ch * 8, v0);
        tmem_ld8(taddr + 1 * 32 + ch * 8, v1);
        tmem_ld8(taddr + 2 * 32 + ch * 8, v2);
        tmem_ld8(taddr + 3 * 32 + ch * 8, v3);
        tmem_ld_wait();
        if (ch == 3) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty[buf]);
        }
        const float4 sa = *reinterpret_cast<const float4*>(&s_shift[ch * 8]);
        const float4 sb = *reinterpret_cast<const float4*>(&s_shift[ch * 8 + 4]);
        const float shv[8] = {sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z, sb.w};
        float f[8];
#pragma unroll
        for (int e = 0; e < 8; e += 2) {
          float m0 = fmaxf(fmaxf(__uint_as_float(v0[e]), __uint_as_float(v1[e])),
                           fmaxf(__uint_as_float(v2[e]), __uint_as_float(v3[e])));
          float m1 = fmaxf(fmaxf(__uint_as_float(v0[e + 1]), __uint_as_float(v1[e + 1])),
                           fmaxf(__uint_as_float(v2[e + 1]), __uint_as_float(v3[e + 1])));
          float t0, t1;
          c1_add2(m0, m1, shv[e], shv[e + 1]);            // m += shift      (two channels per instruction)
          c1_mul2(t0, t1, m0, m1, alpha);                 // alpha * m
          f[e] = fmaxf(m0, t0);
          f[e + 1] = fmaxf(m1, t1);
        }
        uint32_t o[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * e], f[2 * e + 1]);
          o[e] = *reinterpret_cast<uint32_t*>(&h);
        }
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg_row + (((uint32_t)ch ^ swz) << 4)), "r"(o[0]), "r"(o[1]),
                     "r"(o[2]), "r"(o[3])
                     : "memory");
        if constexpr (SPLIT) {
          uint32_t l[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 hf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&o[e]));
            __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * e] - hf.x, f[2 * e + 1] - hf.y);
            l[e] = *reinterpret_cast<uint32_t*>(&h);
          }
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg_row + (((uint32_t)(4 + ch) ^ swz) << 4)), "r"(l[0]),
                       "r"(l[1]), "r"(l[2]), "r"(l[3])
                       : "memory");     // lo half: channels 32..63 of the row
        }
      }
      fence_proxy_async_smem();
      asm volatile("bar.sync %0, 128;" ::"r"(1 + eg) : "memory");
      if (st_leader) {
        tma_store_4d(&tmY, sStg + (uint32_t)eg * STG_BYTES, 0, t.pw0, t.ph0, t.n);
        bulk_commit_group();
      }
      __syncwarp();
    }
    if (st_leader) bulk_wait_group_read<0>();             // smem must outlive the last box store's read
  }

  tc_fence_before();
  __syncthreads();
  if (warp == C1_WARP_MMA) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// B operand: [ty 4][k-group 2][n = window*32 + ch][8 = (tx_local 2) x (c 4)] bf16
//   value = scale[ch] * w[ty-dy][tx-dx][c][ch] where the tap exists, else 0;  window = dy*2 + dx, tx = kg*2 + tx_local
__global__ void pack_conv1_u8_kernel(const float* __restrict__ w, const float* __restrict__ scale,
                                     __nv_bfloat16* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 4 * 2 * 128 * 8) return;
  const int e = idx & 7, n = (idx >> 3) & 127, kg = (idx >> 10) & 1, ty = idx >> 11;
  const int c = e & 3, tx = kg * 2 + (e >> 2);
  const int win = n >> 5, ch = n & 31, dy = win >> 1, dx = win & 1;
  const int kh = ty - dy, kw = tx - dx;
  float v = 0.0f;
  if (c < 3 && kh >= 0 && kh < 3 && kw >= 0 && kw < 3) {
    v = w[((kh * 3 + kw) * 3 + c) * C1_COUT + ch];
    if (scale) v *= scale[ch];
  }
  out[idx] = __float2bfloat16_rn(v);
}

// bf16x3 variant: same index space twice (hi at [0, 8192), lo at [8192, 16384)); value = scale[ch] * 2/255 * w on the three
// colour channels and -scale[ch] * sum_c w on the "ones" channel (the -1 of x = v*2/255 - 1, absent in the zero-padded halo)
__global__ void pack_conv1_u8_split_kernel(const float* __restrict__ w, const float* __restrict__ scale,
                                           __nv_bfloat16* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 4 * 2 * 128 * 8) return;
  const int e = idx & 7, n = (idx >> 3) & 127, kg = (idx >> 10) & 1, ty = idx >> 11;
  const int c = e & 3, tx = kg * 2 + (e >> 2);
  const int win = n >> 5, ch = n & 31, dy = win >> 1, dx = win & 1;
  const int kh = ty - dy, kw = tx - dx;
  double v = 0.0;
  if (kh >= 0 && kh < 3 && kw >= 0 && kw < 3) {
    const float* wt = w + ((kh * 3 + kw) * 3) * C1_COUT + ch;
    const double sc = scale ? (double)scale[ch] : 1.0;
    if (c < 3) v = sc * (double)wt[c * C1_COUT] * (2.0 / 255.0);
    else v = -sc * ((double)wt[0] + (double)wt[C1_COUT] + (double)wt[2 * C1_COUT]);
  }
  const __nv_bfloat16 hi = __float2bfloat16_rn((float)v);
  out[idx] = hi;
  out[4 * 2 * 128 * 8 + idx] = __float2bfloat16_rn((float)(v - (double)__bfloat162float(hi)));
}

}  // namespace y2

using namespace y2;

extern "C" size_t y2_conv1_u8_packed_weight_elems(void) { return 4 * 2 * 128 * 8; }

extern "C" int y2_pack_weights_conv1_u8_split(const float* w_hwio, const float* scale, void* w_packed, y2_stream_t stream) {
  Y2_ARG(w_hwio && w_packed);
  pack_conv1_u8_split_kernel<<<(4 * 2 * 128 * 8 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w_hwio, scale,
                                                                                               (__nv_bfloat16*)w_packed);
  Y2_LAUNCHED();
  return Y2_OK;
}

extern "C" int y2_pack_weights_conv1_u8(const float* w_hwio, const float* scale, void* w_packed, y2_stream_t stream) {
  Y2_ARG(w_hwio && w_packed);
  pack_conv1_u8_kernel<<<(4 * 2 * 128 * 8 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w_hwio, scale,
                                                                                         (__nv_bfloat16*)w_packed);
  Y2_LAUNCHED();
  return Y2_OK;
}

static int conv1_u8_pool_launch(const uint8_t* img, const void* w_packed, const float* shift, void* y, int N, int H,
                                int W, float alpha, bool split, y2_stream_t stream) {
  Y2_ARG(img && w_packed && y && N > 0 && H > 0 && W > 0);
  if (H % (2 * C1_TH) != 0 || W % (2 * C1_TW) != 0) {
    set_error("y2_conv1_u8_pool_fwd: H must be a multiple of %d and W of %d (got %dx%d)", 2 * C1_TH, 2 * C1_TW, H, W);
    return Y2_ERR_UNSUPPORTED;
  }
  Y2_ARG((reinterpret_cast<uintptr_t>(img) & 15) == 0 && (reinterpret_cast<uintptr_t>(w_packed) & 15) == 0 &&
         (reinterpret_cast<uintptr_t>(y) & 15) == 0);
  int rc = load_driver_entry_points();
  if (rc != Y2_OK) return rc;
  Conv1Args a;
  a.w_packed = reinterpret_cast<const uint4*>(w_packed);
  a.shift = shift;
  a.y = reinterpret_cast<__nv_bfloat16*>(y);
  a.N = N; a.H = H; a.W = W;
  a.tiles_w = W / (2 * C1_TW);
  a.tiles_per_img = a.tiles_w * (H / (2 * C1_TH));
  fastdiv_init((uint32_t)a.tiles_per_img, &a.fd_img_mul, &a.fd_img_shr);
  fastdiv_init((uint32_t)a.tiles_w, &a.fd_w_mul, &a.fd_w_shr);
  const long long total = (long long)N * a.tiles_per_img;
  Y2_ARG(total < (1ll << 31) - 1024);
  a.total_tiles = (int)total;
  a.alpha = alpha;
  CUtensorMap tmImg, tmY;
  {
    // pooled output [N, H/2, W/2, 32 | 64] bf16: boxes of one tile (8 x 16 pooled pixels, the whole row), swizzled rows
    const int cw = split ? 2 * C1_COUT : C1_COUT;
    const cuuint32_t box[4] = {(cuuint32_t)cw, (cuuint32_t)C1_TW, (cuuint32_t)C1_TH, 1};
    rc = tmap_nhwc_box(&tmY, y, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, N, H / 2, W / 2, cw, cw, box,
                       split ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                       "y2_conv1_u8_pool_fwd", "output");
    if (rc != Y2_OK) return rc;
  }
  {
    cuuint64_t dims[3] = {(cuuint64_t)W * 3, (cuuint64_t)H, (cuuint64_t)N};
    cuuint64_t strides[2] = {(cuuint64_t)W * 3, (cuuint64_t)H * W * 3};
    cuuint32_t box[3] = {(cuuint32_t)C1_RAW_ROW, (cuuint32_t)C1_PROWS, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = g_encodeTiled(&tmImg, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(img), dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("y2_conv1_u8_pool_fwd: tensor map encode failed (CUresult %d)", (int)r);
      return Y2_ERR_DRIVER;
    }
  }
  const int grid = (int)(total < g_num_sms ? total : g_num_sms);
  if (split) {
    Y2_CUDA(cudaFuncSetAttribute(conv1_u8_pool_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C1_SMEM_SPLIT));
    conv1_u8_pool_kernel<true><<<grid, C1_THREADS, C1_SMEM_SPLIT, (cudaStream_t)stream>>>(tmImg, tmY, a);
  } else {
    Y2_CUDA(cudaFuncSetAttribute(conv1_u8_pool_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C1_SMEM));
    conv1_u8_pool_kernel<false><<<grid, C1_THREADS, C1_SMEM, (cudaStream_t)stream>>>(tmImg, tmY, a);
  }
  Y2_LAUNCHED();
  return Y2_OK;
}

extern "C" int y2_conv1_u8_pool_fwd(const uint8_t* img, const void* w_packed, const float* shift, void* y, int N, int H,
                                    int W, float alpha, y2_stream_t stream) {
  return conv1_u8_pool_launch(img, w_packed, shift, y, N, H, W, alpha, false, stream);
}

extern "C" int y2_conv1_u8_pool_fwd_split(const uint8_t* img, const void* w_packed, const float* shift, void* y, int N, int H,
                                          int W, float alpha, y2_stream_t stream) {
  return conv1_u8_pool_launch(img, w_packed, shift, y, N, H, W, alpha, true, stream);
}
