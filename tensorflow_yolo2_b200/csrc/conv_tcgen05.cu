// conv_tcgen05.cu -- a1+a2+a3: convolution as an implicit GEMM on the sm_100a tensor cores.
//
// Replaces, per layer, the reference's tf.nn.conv2d (yolo2_nets/darknet.py:20-21) + bias (:35) +
// tf.layers.batch_normalization (:42-44, folded to per-channel scale/shift) + leaky (:45) +
// tf.nn.max_pool 2x2 (:24-25) with ONE kernel:
//
//   D[M = pixels, N = Cout] = A[M, K = taps*Cin] * B[N, K]^T      bf16 x bf16 -> fp32 in TMEM
//
//   warp 0      TMA producer.  A tile (128 pixels x KCHUNK channels of one filter tap) straight from
//               the NHWC activation tensor: either im2col-mode TMA (128 consecutive output pixels,
//               halo/padding zero-filled by the TMA unit) or tiled-mode TMA (an NB x TH x TW pixel
//               box, used by the pooled layers so that every 2x2 window sits inside one tile).
//               B tile (BLOCK_N filters x KCHUNK) from the packed K-major weights.  Both land in
//               128B/64B-swizzled (or, for the Cin=3->8 first layer, un-swizzled) K-major smem.
//   warp 1      allocates TMEM, then one lane issues tcgen05.mma (M=128, N=BLOCK_N, K=16) per
//               16-channel slice and commits to the stage's "empty" barrier; the accumulator is
//               double-buffered in TMEM so the epilogue of tile i overlaps the MMAs of tile i+1.
//   warps 2..5  epilogue: tcgen05.ld 32 columns at a time, v = acc*scale[c]+shift[c], leaky,
//               optional 2x2 max-pool across lanes (warp shuffles; the tiled box guarantees the
//               window partners are lanes r^1 and r^TW), convert, 16-byte global stores.
//   Persistent grid (<= #SMs CTAs), static round-robin over (m_tile, n_tile) with n fastest so
//   CTAs running concurrently share the same A rows in L2.
//
// Every mbarrier wait has a clock-based timeout that traps instead of hanging the GPU.
#include "tc_common.cuh"

namespace y2 {

constexpr int TILE_M = 128;

struct ConvArgs {
  const float* scale;
  const float* shift;
  void* y;
  long long M;            // N*H*W
  int N, H, W, Cout;
  int ldy;
  int flags;
  float alpha;
  int ksize, pad;
  int cin_p;              // padded input channels
  int kchunk;             // channels per smem row (8 / 32 / 64)
  int row_bytes;          // kchunk * 2
  int kblocks;            // pipeline stages per tile: taps * cin_p/kchunk   (first layer: 1)
  int cchunks;            // cin_p / kchunk
  int ksteps;             // MMAs per stage (K=16 each)
  int a_mode;             // 0 im2col, 1 tiled box, 2 halo patch (8x16 px tile, vertical tap reuse in smem)
  int tw_log2, th_log2, nb_log2;
  int tiles_w, tiles_h, tiles_nb;
  int m_tiles, n_tiles;
  int stages;
  uint32_t a_stage_bytes, b_stage_bytes;
  uint32_t a_sbo, a_lbo, b_sbo, b_lbo, layout_type, kstep_bytes;   // UMMA smem-descriptor fields (bytes)
  int first_layer;        // Cin_p == 8 special case (all taps in one stage, no swizzle)
  int b_stationary;       // whole B operand resident in smem for the CTA's lifetime (n_tiles == 1, small B)
  uint32_t b_total_bytes;
  int sps;                // (tap, channel-chunk) sub-blocks per pipeline stage
  int tma_store;          // mode 2, un-pooled bf16 output: rows leave through swizzled smem and TMA box stores
  uint32_t stg_offset;    // byte offset of the store staging area (4 groups x 2 x 8 KB) from the aligned smem base
  int cta2;               // mode 2, stationary B: CTA pair, tcgen05 cta_group::2 MMAs (M = 256, each CTA holds half of the filters)
  int kw_merge;           // mode 2: the three horizontally shifted patches share one stage (stationary B, one chunk)
  int stages_per_tile;    // kblocks / sps
  uint32_t a_sub_bytes, b_sub_bytes;
  uint32_t tx_bytes;      // A bytes the TMA reports per stage
  // magic-number division (single-thread roles must not spend their time in integer division)
  uint32_t fd_ntiles_mul, fd_ntiles_shr;
  uint32_t fd_w_mul, fd_w_shr;            // a_mode 0: W         a_mode 1: tiles_w
  uint32_t fd_h_mul, fd_h_shr;            // a_mode 0: H         a_mode 1: tiles_h
  uint32_t fd_cch_mul, fd_cch_shr;        // cchunks
  // "bf16x3" (Y2_CONV_IN_SPLIT / OUT_SPLIT, include/yolo2_b200.h): the A tensor holds [hi | lo] (a_wrap = its number of
  // channel chunks); the K loop walks cchunks = 3/2 * a_wrap chunks per tap [hi | lo | hi] against B's [w_hi | w_hi | w_lo]
  int a_wrap;             // channel chunks of the A tensor (== cchunks unless split)
  int split_out;          // bf16 output as hi at column c, lo at column lo_off + c
  int lo_off;
};


// ------------------------------------------------------------------------------------------
// tile -> coordinates
// ------------------------------------------------------------------------------------------
struct TileCoord {
  int n_tile;
  int n0, h0, w0;        // first pixel of the tile (im2col: flattened start; tiled: box origin)
  long long m0;          // im2col: first flattened pixel index
};

// `unit` = scheduling unit (CS == 1: tile index; CTA pair, CS == 2: index of two consecutive M tiles), `crank` = CTA rank
template <int CS>
__device__ __forceinline__ TileCoord decode_tile(const ConvArgs& a, int unit, uint32_t crank) {
  TileCoord t;
  const uint32_t mg = fdiv((uint32_t)unit, a.fd_ntiles_mul, a.fd_ntiles_shr);
  t.n_tile = unit - (int)mg * a.n_tiles;
  const uint32_t mt = mg * (uint32_t)CS + crank;             // may be >= m_tiles for the last group: all rows masked
  if (a.a_mode == 0) {
    t.m0 = (long long)mt * TILE_M;                       // < 2^31 (checked on the host)
    const uint32_t m = t.m0 < a.M ? (uint32_t)t.m0 : 0u; // the empty half of a last pair loads valid pixels; its rows are masked
    const uint32_t row = fdiv(m, a.fd_w_mul, a.fd_w_shr);         // n*H + h
    t.w0 = (int)(m - row * (uint32_t)a.W);
    const uint32_t img = fdiv(row, a.fd_h_mul, a.fd_h_shr);
    t.h0 = (int)(row - img * (uint32_t)a.H);
    t.n0 = (int)img;
  } else {
    const uint32_t q = fdiv(mt, a.fd_w_mul, a.fd_w_shr);          // / tiles_w
    const uint32_t tw_i = mt - q * (uint32_t)a.tiles_w;
    const uint32_t tn_i = fdiv(q, a.fd_h_mul, a.fd_h_shr);        // / tiles_h
    const uint32_t th_i = q - tn_i * (uint32_t)a.tiles_h;
    t.w0 = (int)(tw_i << a.tw_log2);
    t.h0 = (int)(th_i << a.th_log2);
    t.n0 = (int)(tn_i << a.nb_log2);
    t.m0 = 0;
  }
  return t;
}

// ------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------
// Warp roles.  Epilogue = EPI_GROUPS groups of 4 warps (one warp per TMEM lane quarter, so the warp id modulo 4
// must equal the quarter: epilogue warps come first).  The accumulator is multi-buffered in TMEM (NBUF tiles);
// TP groups work on DIFFERENT tiles at the same time and CP groups split the columns of one tile
// (EPI_GROUPS = TP * CP).  The SM's warp arbiter favours the highest warp id (B300_MICROARCH.md): the two
// roles that feed the tensor pipe (TMA producer, MMA issuer) get the top ids so the epilogue cannot starve them.
constexpr int EPI_GROUPS = 4;
constexpr int EPI_WARPS = 4 * EPI_GROUPS;
constexpr int TC_THREADS = 64 + EPI_WARPS * 32;
constexpr int WARP_PRODUCER = EPI_WARPS;
constexpr int WARP_MMA = EPI_WARPS + 1;
constexpr int MAX_STAGES = 12;
constexpr int MAX_UNITS = 448;                     // (tap, channel-chunk) units per tile: 9 * 1280/64 = 180 (passthrough concat);
                                                   // bf16x3: 9 * 3 * 1024/64 = 432

// per-unit constants, computed once per CTA so that the single-thread roles do no index arithmetic
struct __align__(8) UnitDesc {
  uint16_t a_c0;   // channel coordinate of the A load
  uint8_t kw;      // filter tap column
  uint8_t pad_;
  uint16_t kh;     // filter tap row (mode 2: index of the kh=0 sub-block in the stationary B)
  uint16_t b_k;    // K coordinate of the B load (mode 2: for kh = 0; + 3*cin_p per kh)
};

template <int CW>
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, uint32_t* v) {
  if constexpr (CW == 32) {
    tmem_ld32(taddr, v);
  } else {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
  }
}

// bf16x3 output: 8 floats -> 8 bf16 hi (16 B) + 8 bf16 lo = bf16(v - hi) (16 B)
__device__ __forceinline__ void split8_bf16(const float* f, uint4& hi, uint4& lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const __nv_bfloat162 h2 = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    const float2 hf = __bfloat1622float2(h2);
    const __nv_bfloat162 l2 = __floats2bfloat162_rn(f[2 * i] - hf.x, f[2 * i + 1] - hf.y);
    h[i] = *reinterpret_cast<const uint32_t*>(&h2);
    l[i] = *reinterpret_cast<const uint32_t*>(&l2);
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// One chunk of CW accumulator columns of one row: affine, leaky, (pool), convert, store.
template <int CW>
__device__ __forceinline__ void epilogue_chunk(const ConvArgs& a, const uint32_t* v, const float* s_scale,
                                               const float* s_shift, int cc, int c0, bool valid, long long orow,
                                               bool pool, bool leaky_on, bool out_f32) {
  float f[CW];
#pragma unroll
  for (int i = 0; i < CW; i += 4) {
    const float4 sc = *reinterpret_cast<const float4*>(&s_scale[cc + i]);   // smem broadcast
    const float4 sh = *reinterpret_cast<const float4*>(&s_shift[cc + i]);
    f[i + 0] = fmaf(__uint_as_float(v[i + 0]), sc.x, sh.x);
    f[i + 1] = fmaf(__uint_as_float(v[i + 1]), sc.y, sh.y);
    f[i + 2] = fmaf(__uint_as_float(v[i + 2]), sc.z, sh.z);
    f[i + 3] = fmaf(__uint_as_float(v[i + 3]), sc.w, sh.w);
  }
  if (leaky_on) {
#pragma unroll
    for (int i = 0; i < CW; ++i) f[i] = fmaxf(f[i], a.alpha * f[i]);
  }
  const int ncols = min(CW, a.ldy - c0);    // columns of this chunk that exist in the output row
  if (out_f32) {
    if (pool) {
#pragma unroll
      for (int i = 0; i < CW; ++i) {
        f[i] = fmaxf(f[i], __shfl_xor_sync(0xffffffffu, f[i], 1));
        f[i] = fmaxf(f[i], __shfl_xor_sync(0xffffffffu, f[i], 1 << a.tw_log2));
      }
    }
    if (valid) {
      float* dst = reinterpret_cast<float*>(a.y) + (size_t)orow * a.ldy + c0;
      if (ncols == CW && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
#pragma unroll
        for (int i = 0; i < CW; i += 4)
          *reinterpret_cast<float4*>(dst + i) = make_float4(f[i], f[i + 1], f[i + 2], f[i + 3]);
      } else {
#pragma unroll
        for (int i = 0; i < CW; ++i)
          if (i < ncols) dst[i] = f[i];
      }
    }
  } else if (a.split_out) {
    // bf16x3: pool on the float32 values, then split into hi / lo halves of the output row
    if (pool) {
#pragma unroll
      for (int i = 0; i < CW; ++i) {
        f[i] = fmaxf(f[i], __shfl_xor_sync(0xffffffffu, f[i], 1));
        f[i] = fmaxf(f[i], __shfl_xor_sync(0xffffffffu, f[i], 1 << a.tw_log2));
      }
    }
    if (valid) {
      __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(a.y) + (size_t)orow * a.ldy + c0;
      const int nc = min(CW, a.Cout - c0);        // (columns past Cout belong to the lo half / do not exist)
      if (nc == CW && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) && (a.lo_off & 7) == 0) {
#pragma unroll
        for (int i = 0; i < CW / 8; ++i) {
          uint4 hi, lo;
          split8_bf16(f + 8 * i, hi, lo);
          reinterpret_cast<uint4*>(dst)[i] = hi;
          reinterpret_cast<uint4*>(dst + a.lo_off)[i] = lo;
        }
      } else {
#pragma unroll
        for (int i = 0; i < CW; ++i)
          if (i < nc) {
            const __nv_bfloat16 h = __float2bfloat16_rn(f[i]);
            dst[i] = h;
            dst[a.lo_off + i] = __float2bfloat16_rn(f[i] - __bfloat162float(h));
          }
      }
    }
  } else {
    // pack to bf16x2 first: rounding is monotonic, so max(round(a),round(b)) == round(max(a,b))
    // and the 2x2 max-pool can run on packed pairs with half the shuffles
    uint32_t pk[CW / 2];
#pragma unroll
    for (int i = 0; i < CW / 2; ++i) {
      __nv_bfloat162 h2 = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
      pk[i] = *reinterpret_cast<uint32_t*>(&h2);
    }
    if (pool) {
#pragma unroll
      for (int i = 0; i < CW / 2; ++i) {
        uint32_t o = __shfl_xor_sync(0xffffffffu, pk[i], 1);
        __nv_bfloat162 m = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&pk[i]), *reinterpret_cast<__nv_bfloat162*>(&o));
        pk[i] = *reinterpret_cast<uint32_t*>(&m);
        o = __shfl_xor_sync(0xffffffffu, pk[i], 1 << a.tw_log2);
        m = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&pk[i]), *reinterpret_cast<__nv_bfloat162*>(&o));
        pk[i] = *reinterpret_cast<uint32_t*>(&m);
      }
    }
    if (valid) {
      __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(a.y) + (size_t)orow * a.ldy + c0;
      if (ncols == CW && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
#pragma unroll
        for (int i = 0; i < CW / 8; ++i)
          reinterpret_cast<uint4*>(dst)[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
      } else {
#pragma unroll
        for (int i = 0; i < CW; ++i)
          if (i < ncols)
            reinterpret_cast<uint16_t*>(dst)[i] = (uint16_t)((i & 1) ? (pk[i >> 1] >> 16) : (pk[i >> 1] & 0xffffu));
      }
    }
  }
}

// Pooled bf16 epilogue, 32 accumulator columns of one row per lane -> 8 output columns of one POOLED pixel per lane.
//   max-pool commutes with any increasing map, and x -> leaky(s*x + b) is increasing in sign(s)*x.  So the 2x2 max runs
//   first, on the raw accumulators with the sign of the channel's scale folded in, and the affine + leaky + convert run
//   on the pooled quarter only.  The pooling itself is a recursive halving instead of a butterfly: in each of the two
//   exchange steps a lane hands half of its columns to the partner and keeps the max over the other half, so that the
//   four lanes of a window end up with DIFFERENT 8-column slices of the result (16 B each, 64 contiguous bytes per
//   window) and every lane does useful work in the affine / store phase.  ~2x fewer instructions than
//   affine+leaky on all four pixels followed by a butterfly max -- the layers with few input channels (Cin = 32)
//   are bound by exactly these epilogue instructions (63 M warp instructions for layer 2 in the profile).
__device__ __forceinline__ void epilogue_chunk_pooled_bf16(const ConvArgs& a, const uint32_t* v, const float* s_scale,
                                                           const float* s_shift, int cc, int c0, bool valid_px, long long orow,
                                                           bool leaky_on, int lane) {
  float t[32];
#pragma unroll
  for (int i = 0; i < 32; i += 4) {
    const uint4 sb = *reinterpret_cast<const uint4*>(&s_scale[cc + i]);     // smem broadcast
    t[i + 0] = __uint_as_float(v[i + 0] ^ (sb.x & 0x80000000u));
    t[i + 1] = __uint_as_float(v[i + 1] ^ (sb.y & 0x80000000u));
    t[i + 2] = __uint_as_float(v[i + 2] ^ (sb.z & 0x80000000u));
    t[i + 3] = __uint_as_float(v[i + 3] ^ (sb.w & 0x80000000u));
  }
  const bool up1 = (lane & 1) != 0;                       // horizontal partner: lane ^ 1 (tile width >= 2)
  float m16[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const float send = up1 ? t[i] : t[16 + i];
    const float recv = __shfl_xor_sync(0xffffffffu, send, 1);
    m16[i] = fmaxf(up1 ? t[16 + i] : t[i], recv);
  }
  const bool up2 = ((lane >> a.tw_log2) & 1) != 0;        // vertical partner: lane ^ TW
  float m8[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float send = up2 ? m16[i] : m16[8 + i];
    const float recv = __shfl_xor_sync(0xffffffffu, send, 1 << a.tw_log2);
    m8[i] = fmaxf(up2 ? m16[8 + i] : m16[i], recv);
  }
  const int cb = (up1 ? 16 : 0) + (up2 ? 8 : 0);          // my 8 columns of the chunk
  const float4 sa = *reinterpret_cast<const float4*>(&s_scale[cc + cb]), sb4 = *reinterpret_cast<const float4*>(&s_scale[cc + cb + 4]);
  const float4 ha = *reinterpret_cast<const float4*>(&s_shift[cc + cb]), hb4 = *reinterpret_cast<const float4*>(&s_shift[cc + cb + 4]);
  const float sc[8] = {sa.x, sa.y, sa.z, sa.w, sb4.x, sb4.y, sb4.z, sb4.w};
  const float sh[8] = {ha.x, ha.y, ha.z, ha.w, hb4.x, hb4.y, hb4.z, hb4.w};
  float f[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    f[i] = fmaf(m8[i], fabsf(sc[i]), sh[i]);
    if (leaky_on) f[i] = fmaxf(f[i], a.alpha * f[i]);
  }
  if (valid_px && a.split_out) {
    uint4 hi, lo;
    split8_bf16(f, hi, lo);
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(a.y) + (size_t)orow * a.ldy + c0 + cb;
    *reinterpret_cast<uint4*>(dst) = hi;
    *reinterpret_cast<uint4*>(dst + a.lo_off) = lo;
  } else if (valid_px) {
    __nv_bfloat162 h0 = __floats2bfloat162_rn(f[0], f[1]), h1 = __floats2bfloat162_rn(f[2], f[3]);
    __nv_bfloat162 h2 = __floats2bfloat162_rn(f[4], f[5]), h3 = __floats2bfloat162_rn(f[6], f[7]);
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(a.y) + (size_t)orow * a.ldy + c0 + cb;
    *reinterpret_cast<uint4*>(dst) = make_uint4(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1),
                                                *reinterpret_cast<uint32_t*>(&h2), *reinterpret_cast<uint32_t*>(&h3));
  }
}

// KIND: 0 = first layer (Cin 3 -> 8, un-swizzled 16-byte rows), 1 = 64-byte rows (Cin 32), 2 = 128-byte rows
// CTA2: CTA-pair variant (tcgen05 cta_group::2).  A template parameter, not a run-time flag: a kernel that merely CONTAINS
// cta_group::2 instructions can only be launched with an even cluster size (launch error "cluster misconfiguration").
// TMAST: TMA-store epilogue (un-pooled bf16 rows through swizzled smem) -- a separate instantiation, so that its registers do
// not weigh on the other epilogues (as a run-time branch it pushed them from 24 to 100 bytes of spills under the 96-register cap).
template <int BLOCK_N, int A_MODE, int KIND, bool CTA2 = false, bool TMAST = false>
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmY, const ConvArgs a) {
  constexpr bool FIRST = KIND == 0;
  constexpr uint32_t ROW_BYTES = KIND == 0 ? 16u : (KIND == 1 ? 64u : 128u);
  extern __shared__ __align__(1024) uint8_t smem[];
  constexpr int NBUF = BLOCK_N >= 256 ? 2 : 4;                     // accumulator tiles resident in TMEM
  constexpr int TP = NBUF < EPI_GROUPS ? NBUF : EPI_GROUPS;        // epilogue groups on different tiles
  constexpr int CP = EPI_GROUPS / TP;                              // epilogue groups sharing one tile (column split)
  static_assert(TP * CP == EPI_GROUPS && NBUF % TP == 0, "epilogue group layout");
  constexpr uint32_t TMEM_COLS = (NBUF * BLOCK_N <= 32) ? 32 : (NBUF * BLOCK_N <= 64) ? 64 : (NBUF * BLOCK_N <= 128) ? 128
                                 : (NBUF * BLOCK_N <= 256) ? 256 : 512;
  static_assert(NBUF * BLOCK_N <= 512, "TMEM has 512 columns");
  __shared__ __align__(8) uint64_t full_bar[MAX_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[MAX_STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar[NBUF];
  __shared__ __align__(8) uint64_t tmem_empty_bar[NBUF];
  __shared__ __align__(8) uint64_t bfull_bar;
  __shared__ uint32_t s_tmem_base;
  __shared__ __align__(16) float s_scale[TP][BLOCK_N];
  __shared__ __align__(16) float s_shift[TP][BLOCK_N];
  __shared__ UnitDesc s_units[FIRST ? 1 : MAX_UNITS];

  pdl_launch_dependents();                              // persistent grid: the next kernel may take SMs as my CTAs retire
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // dynamic smem, 1024-byte aligned (swizzle-128B atoms): [stationary B (optional)] [stage 0: A | B] [stage 1] ...
  const uint32_t smem_b_stat = (smem_u32(smem) + 1023u) & ~1023u;
  const uint32_t smem_base = smem_b_stat + (a.b_stationary ? ((a.b_total_bytes + 1023u) & ~1023u) : 0u);
  const uint32_t stage_bytes = a.a_stage_bytes + (a.b_stationary ? 0u : a.b_stage_bytes);
  const uint32_t tx_bytes = a.tx_bytes + (a.b_stationary ? 0u : a.b_stage_bytes);
  // Work distribution.  Single CTA: CTA b takes tiles b, b+grid, ...  CTA pair on one M = 256 MMA (see
  // conv_streamk2_kernel for the why: the 64 B/clk smem operand path): the pair takes two consecutive M tiles x one N tile.
  // Each CTA keeps its own 128-pixel tile and HALF of the filters; the leader (rank 0) issues, both run producer + epilogue.
  constexpr bool cta2 = CTA2;
  constexpr int CS = CTA2 ? 2 : 1;                      // CTAs per cluster
  static_assert(!CTA2 || !FIRST, "no CTA-pair variant of the first-layer paths");
  const uint32_t crank = CTA2 ? cluster_ctarank() : 0u;
  const int sched_first = (int)(blockIdx.x / CS);
  const int sched_step = (int)(gridDim.x / CS);
  const int m_groups = (a.m_tiles + CS - 1) / CS;
  const int total_tiles = m_groups * a.n_tiles;        // scheduling units (per cluster)

  if (warp == WARP_PRODUCER) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
      for (int s = 0; s < a.stages; ++s) {
        mbar_init(&full_bar[s], 1);
        mbar_init(&empty_bar[s], 1);                    // (pair: one multicast commit releases both CTAs' copies)
      }
      for (int b = 0; b < NBUF; ++b) {
        mbar_init(&tmem_full_bar[b], 1);
        mbar_init(&tmem_empty_bar[b], 4 * CP * (cta2 ? 2 : 1));   // the warps of the CP groups that drain this buffer (pair: of both CTAs)
      }
      mbar_init(&bfull_bar, 1);
      fence_barrier_init();
    }
    if constexpr (!FIRST) {
      // unit table (one-time integer division)
      const int units = (A_MODE == 2) ? a.cchunks * 3 : a.kblocks;
      for (int u = lane; u < units; u += 32) {
        UnitDesc d;
        d.pad_ = 0;
        if (A_MODE == 2) {
          const int cc = u / 3, kw = u - cc * 3;
          const int ca = cc < a.a_wrap ? cc : cc - a.a_wrap;          // bf16x3: the third K block re-reads the hi channels
          d.a_c0 = (uint16_t)(ca * a.kchunk); d.kw = (uint8_t)kw; d.kh = (uint16_t)(kw * a.cchunks + cc);
          d.b_k = (uint16_t)(kw * a.cin_p + cc * a.kchunk);
        } else {
          const int tap = u / a.cchunks, cc = u - tap * a.cchunks;
          const int ca = cc < a.a_wrap ? cc : cc - a.a_wrap;
          const int kh = tap / a.ksize;
          d.a_c0 = (uint16_t)(ca * a.kchunk); d.kh = (uint16_t)kh; d.kw = (uint8_t)(tap - kh * a.ksize);
          d.b_k = (uint16_t)(tap * a.cin_p + cc * a.kchunk);
        }
        s_units[u] = d;
      }
    }
  }
  if (warp == WARP_MMA) {
    if constexpr (cta2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem_base)),
                   "r"(TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem_base)),
                   "r"(TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CTA2) cluster_sync_all();               // partner's barriers are initialised before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;
  pdl_wait();                                           // everything above overlapped the previous kernel's tail

  if (warp == WARP_PRODUCER) {
    // =========================== TMA producer ===========================
    // The whole warp runs the loop; lane 0 owns the barrier handshake and the stage's TMA loads are issued
    // by different lanes in the same instruction slot.
    uint32_t phase = 0;
    const int sps = a.sps;
    if (a.b_stationary) {
      // weights of this layer fit in smem: fetch them once per CTA instead of once per tile
      // pair: both CTAs' halves are counted on the LEADER's barrier (the issuer needs both resident)
      if (lane == 0 && (!cta2 || crank == 0)) mbar_expect_tx(&bfull_bar, cta2 ? 2u * a.b_total_bytes : a.b_total_bytes);
      __syncwarp();
      const uint32_t bar = cta2 ? (smem_u32(&bfull_bar) & PEER_BIT_MASK) : smem_u32(&bfull_bar);
      if constexpr (FIRST) {
        if (lane == 0) tma_load_3d(smem_b_stat, &tmB, bar, 0, 0, 0);
      } else {
        // stationary order = packed K order: index = tap * cchunks + cc
        for (int sub = lane; sub < a.kblocks; sub += 32) {
          const int tap = sub / a.cchunks, cc = sub - tap * a.cchunks;
          if constexpr (cta2) tma_load_2d_2sm(smem_b_stat + sub * a.b_sub_bytes, &tmB, bar, tap * a.cin_p + cc * a.kchunk, (int)crank * (BLOCK_N / 2));
          else tma_load_2d(smem_b_stat + sub * a.b_sub_bytes, &tmB, bar, tap * a.cin_p + cc * a.kchunk, 0);
        }
      }
      __syncwarp();
    }
    const uint32_t full0 = opaque(smem_u32(&full_bar[0])), empty0 = opaque(smem_u32(&empty_bar[0]));
    const uint32_t nstages = opaque((uint32_t)a.stages);
    const int spt = (int)opaque((uint32_t)a.stages_per_tile);
    uint32_t ustage = 0, soffb = 0;                      // stage index and its byte offset
    for (int tile = sched_first; tile < total_tiles; tile += sched_step) {
      const TileCoord t = decode_tile<CS>(a, tile, crank);
      const int nrow0 = t.n_tile * BLOCK_N;
      for (int st = 0; st < spt; ++st) {
        const uint32_t bar = cta2 ? ((full0 + 8u * ustage) & PEER_BIT_MASK) : full0 + 8u * ustage;   // pair: the leader's barrier
        if (lane == 0) {
          mbar_wait_a(empty0 + 8u * ustage, phase ^ 1u);
          if (!cta2) mbar_expect_tx_a(bar, tx_bytes);
          else if (crank == 0) mbar_expect_tx_a(bar, 2u * tx_bytes);      // both CTAs' patches
        }
        __syncwarp();
        const uint32_t sA = smem_base + soffb;
        const uint32_t sB = sA + a.a_stage_bytes;
        if constexpr (FIRST && A_MODE == 2) {
          // halo patch: ONE 18-row x 10-pixel x 16-byte load serves all 9 taps (shifted UMMA descriptors)
          if (lane == 0) tma_load_3d(sA, &tmA, bar, (t.w0 - 1) * 8, t.h0 - 1, t.n0);
          else if (lane == 1 && !a.b_stationary) tma_load_3d(sB, &tmB, bar, 0, nrow0, 0);
        } else if constexpr (FIRST) {
          // 10 k-groups of 8 padded channels: taps 0..7, a group that meets zero weights, tap 8
          if (lane < 10) {
            const int tap = lane < 8 ? lane : (lane == 8 ? 0 : 8);
            const int kh = (tap * 11) >> 5, kw = tap - kh * 3;
            if constexpr (A_MODE == 0)
              tma_load_im2col_4d(sA + lane * (TILE_M * 16), &tmA, bar, 0, t.w0 - a.pad, t.h0 - a.pad, t.n0, (uint16_t)kw,
                                 (uint16_t)kh);
            else   // tiled box over the merged (W*8 channels) inner dimension: 256-byte TMA rows
              tma_load_3d(sA + lane * (TILE_M * 16), &tmA, bar, (t.w0 + kw - a.pad) * 8, t.h0 + kh - a.pad, t.n0);
          } else if (lane == 10 && !a.b_stationary) {
            tma_load_3d(sB, &tmB, bar, 0, nrow0, 0);
          }
        } else if constexpr (A_MODE == 2) {
          if (a.kw_merge) {
            // the three horizontally shifted (16+2)-row patches of channel chunk `st`, one lane each
            if (lane < 3) {
              const int c0 = (int)s_units[st * 3].a_c0;
              if constexpr (cta2) tma_load_4d_2sm(sA + (uint32_t)lane * a.a_sub_bytes, &tmA, bar, c0, t.w0 + lane - 1, t.h0 - 1, t.n0);
              else tma_load_4d(sA + (uint32_t)lane * a.a_sub_bytes, &tmA, bar, c0, t.w0 + lane - 1, t.h0 - 1, t.n0);
            }
          } else {
            // one horizontally shifted (16+2)-row patch serves the three taps kh = 0..2 of this kw
            const UnitDesc d = s_units[st];
            if (lane == 0) {
              if constexpr (cta2) tma_load_4d_2sm(sA, &tmA, bar, d.a_c0, t.w0 + d.kw - 1, t.h0 - 1, t.n0);
              else tma_load_4d(sA, &tmA, bar, d.a_c0, t.w0 + d.kw - 1, t.h0 - 1, t.n0);
            } else if (lane < 4 && !a.b_stationary) {
              const int kh = lane - 1;
              if constexpr (cta2)      // pair, streamed filters: my half of the rows of tap (kh, kw), counted on the leader's barrier
                tma_load_2d_2sm(sB + kh * a.b_sub_bytes, &tmB, bar, d.b_k + kh * 3 * a.cin_p, nrow0 + (int)crank * (BLOCK_N / 2));
              else
                tma_load_2d(sB + kh * a.b_sub_bytes, &tmB, bar, d.b_k + kh * 3 * a.cin_p, nrow0);
            }
          }
        } else {
          if (lane == 0) {
            for (int j = 0; j < sps; ++j) {
              const UnitDesc d = s_units[st * sps + j];
              if constexpr (cta2) {
                // pair: my own pixels and my half of the filter rows, both counted on the leader's barrier
                if constexpr (A_MODE == 0)
                  tma_load_im2col_4d_2sm(sA + j * a.a_sub_bytes, &tmA, bar, d.a_c0, t.w0 - a.pad, t.h0 - a.pad, t.n0,
                                         (uint16_t)d.kw, (uint16_t)d.kh);
                else
                  tma_load_4d_2sm(sA + j * a.a_sub_bytes, &tmA, bar, d.a_c0, t.w0 + d.kw - a.pad, t.h0 + d.kh - a.pad, t.n0);
                if (!a.b_stationary) tma_load_2d_2sm(sB + j * a.b_sub_bytes, &tmB, bar, d.b_k, nrow0 + (int)crank * (BLOCK_N / 2));
                continue;
              }
              if constexpr (A_MODE == 0)
                tma_load_im2col_4d(sA + j * a.a_sub_bytes, &tmA, bar, d.a_c0, t.w0 - a.pad, t.h0 - a.pad, t.n0,
                                   (uint16_t)d.kw, (uint16_t)d.kh);
              else
                tma_load_4d(sA + j * a.a_sub_bytes, &tmA, bar, d.a_c0, t.w0 + d.kw - a.pad, t.h0 + d.kh - a.pad, t.n0);
              if (!a.b_stationary) tma_load_2d(sB + j * a.b_sub_bytes, &tmB, bar, d.b_k, nrow0);
            }
          }
        }
        __syncwarp();
        ++ustage;
        soffb += stage_bytes;
        if (ustage == nstages) { ustage = 0; soffb = 0; phase ^= 1u; }
      }
    }
  } else if (warp == WARP_MMA) {
    // =========================== MMA issuer ===========================
    // The whole warp walks the loop with warp-uniform values (so descriptors live in uniform registers and
    // an MMA costs a handful of instructions); one elected lane issues tcgen05.mma / tcgen05.commit.
    // This warp is the critical path of every layer whose stages hold few MMAs (profile of layer 2: ~140 dependent
    // instructions = ~800 clk per stage against 192 clk of tensor work), so the loop carries everything as running
    // 32-bit values -- barrier addresses, stage offsets, the stationary-B cursor -- instead of recomputing them from
    // pointers, selects and the unit table each stage.
    uint32_t is_leader;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(is_leader));
    // instruction descriptor (cute::UMMA::InstrDescriptor): D=f32, A=B=bf16, K-major both, N, M=128
    constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
    constexpr int KSTEPS = FIRST ? 5 : ROW_BYTES / 32;                       // K = 16 per MMA
    // descriptors differ only in the 14-bit start-address field: build once, then add (bytes >> 4)
    const uint64_t adesc0 = make_smem_desc(smem_base, a.a_lbo, a.a_sbo, a.layout_type);
    const uint64_t bdesc0 = make_smem_desc(a.b_stationary ? smem_b_stat : smem_base + a.a_stage_bytes, a.b_lbo, a.b_sbo,
                                           a.layout_type);
    // pair: only the leader CTA issues (M = 256 MMAs that read both CTAs' smem and write both CTAs' TMEM); the follower's
    // MMA warp owns nothing but its TMEM allocation
    const bool issuer = !cta2 || crank == 0;
    constexpr uint32_t idesc2 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
    if (a.b_stationary && issuer) {
      mbar_wait(&bfull_bar, 0);
      tc_fence_after();
    }
    constexpr uint32_t a_kstep = FIRST ? (32u * TILE_M) >> 4 : 2u;             // 32 bytes of K per MMA
    constexpr uint32_t b_kstep = FIRST ? (32u * BLOCK_N) >> 4 : 2u;
    const uint32_t a_sub16 = a.a_sub_bytes >> 4, b_sub16 = a.b_sub_bytes >> 4;
    const uint32_t stage16 = stage_bytes >> 4;
    constexpr uint32_t khshift16 = FIRST ? 0u : (8u * ROW_BYTES) >> 4;          // mode 2: one patch row = one swizzle atom
    const int subs = FIRST ? 1 : a.sps;
    const bool bstat = a.b_stationary != 0;
    const uint32_t full0 = opaque(smem_u32(&full_bar[0])), empty0 = opaque(smem_u32(&empty_bar[0]));
    const uint32_t tfull0 = opaque(smem_u32(&tmem_full_bar[0])), tempty0 = opaque(smem_u32(&tmem_empty_bar[0]));
    const uint32_t nstages = opaque((uint32_t)a.stages);
    const int spt = (int)opaque((uint32_t)a.stages_per_tile);
    // B descriptor offset: streamed B lives in the stage (stage * stage16); stationary B is addressed by a cursor
    // that runs through the resident filter bank once per tile (modes 0/1) or by the unit's tap index (mode 2)
    const uint32_t b_stage_inc = bstat ? 0u : stage16;
    const uint32_t b_cursor_inc = bstat ? (uint32_t)subs * b_sub16 : 0u;
    const uint32_t b_unit_mul = bstat ? b_sub16 : 0u;                                   // mode 2
    const uint32_t b_kh_mul = bstat ? (uint32_t)(3 * a.cchunks) * b_sub16 : b_sub16;    // mode 2
    const uint32_t b_tap16 = (uint32_t)a.cchunks * b_sub16;                             // mode 2, kw-merged: one tap's chunks
    uint32_t stage = 0, phase = 0, soff = 0, bsoff = 0;
    uint32_t it = 0;
    for (int tile = sched_first; tile < (issuer ? total_tiles : 0); tile += sched_step, ++it) {
      const uint32_t buf = it % NBUF;
      mbar_wait_a(tempty0 + 8u * buf, ((it / NBUF) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + buf * (uint32_t)BLOCK_N;
      uint32_t accum = 0;
      uint32_t bcur = 0;
      for (int st = 0; st < spt; ++st) {
        uint32_t bidx0 = 0;
        if constexpr (A_MODE == 2 && !FIRST) {
          if (!a.kw_merge) bidx0 = (uint32_t)s_units[st].kh;   // mode 2: kh field carries the stationary B index of kh = 0
        }
        // descriptors of this stage are ready before the barrier is: after the wait only the MMAs issue
        const uint64_t ad_s = adesc0 + soff;
        const uint64_t bd_s = bdesc0 + bsoff + ((A_MODE == 2 && !FIRST) ? bidx0 * b_unit_mul : bcur);
        const uint32_t empty_addr = empty0 + 8u * stage;
        mbar_wait_a(full0 + 8u * stage, phase);
        tc_fence_after();
        if constexpr (FIRST && A_MODE == 2) {
          // patch [18][10 px][8 ch]: pixel = 16 B, 8 consecutive pixels = one un-swizzled core matrix.
          // MMA p multiplies k-groups (2p, 2p+1): A start = first tap's pixel shift, LBO = distance to the
          // second tap, SBO = one patch row (10 px).  k-groups are taps 0..7, a zero-weight group, tap 8;
          // the zero-weight group re-reads tap 7's (finite) pixels so that 0 * x stays 0.
          const uint32_t sA = smem_base + stage * stage_bytes;
          if (is_leader) {
#pragma unroll
            for (int pr = 0; pr < 5; ++pr) {
              const int t0 = pr < 4 ? 2 * pr : 7, t1 = pr < 4 ? 2 * pr + 1 : 8;
              const int o0 = ((t0 / 3) * 10 + (t0 % 3)) * 16, o1 = ((t1 / 3) * 10 + (t1 % 3)) * 16;
              const uint64_t ad = make_smem_desc(sA + o0, (uint32_t)(o1 - o0), 160u, 0u);
              const uint64_t bd = bdesc0 + bsoff + (uint32_t)pr * b_kstep;
              umma_bf16(tmem_d, ad, bd, idesc, accum);
              accum = 1;
            }
          }
        } else if constexpr (A_MODE == 2) {
          // one body for both MMA flavours (the branch on the flavour stays outside the unrolled loops)
          auto issue = [&](auto two_tag) {
            constexpr bool TWO = decltype(two_tag)::value;
            auto mma = [&](uint64_t ad, uint64_t bd) {
              if constexpr (TWO) umma_bf16_2sm(tmem_d, ad, bd, idesc2, accum);
              else umma_bf16(tmem_d, ad, bd, idesc, accum);
              accum = 1;
            };
            if (a.kw_merge) {
              // all three horizontally shifted patches of channel chunk `st` in one stage, stationary B indexed by
              // (tap = kh * 3 + kw, chunk): 9 * KSTEPS MMAs behind a single barrier round trip
#pragma unroll
              for (int kw = 0; kw < 3; ++kw) {
#pragma unroll
                for (int kh = 0; kh < 3; ++kh) {
                  const uint64_t ad = ad_s + (uint32_t)kw * a_sub16 + (uint32_t)kh * khshift16;
                  const uint64_t bd = bd_s + (uint32_t)(kh * 3 + kw) * b_tap16 + (uint32_t)st * b_sub16;     // (bd_s == bdesc0: stationary, bidx0 = 0)
#pragma unroll
                  for (int ks = 0; ks < KSTEPS; ++ks) mma(ad + (uint32_t)ks * a_kstep, bd + (uint32_t)ks * b_kstep);
                }
              }
            } else {
#pragma unroll
              for (int kh = 0; kh < 3; ++kh) {
                const uint64_t ad = ad_s + (uint32_t)kh * khshift16;           // rows of tap (kh,kw) = patch rows + kh
                const uint64_t bd = bd_s + (uint32_t)kh * b_kh_mul;
#pragma unroll
                for (int ks = 0; ks < KSTEPS; ++ks) mma(ad + (uint32_t)ks * a_kstep, bd + (uint32_t)ks * b_kstep);
              }
            }
          };
          if (is_leader) {
            issue(std::integral_constant<bool, cta2>{});
          }
        } else {
          if (is_leader) {
            uint64_t ad = ad_s;
            uint64_t bd = bd_s;
#pragma unroll 1
            for (int j = 0; j < subs; ++j) {
#pragma unroll
              for (int ks = 0; ks < KSTEPS; ++ks) {
                if constexpr (cta2) umma_bf16_2sm(tmem_d, ad + (uint32_t)ks * a_kstep, bd + (uint32_t)ks * b_kstep, idesc2, accum);
                else umma_bf16(tmem_d, ad + (uint32_t)ks * a_kstep, bd + (uint32_t)ks * b_kstep, idesc, accum);
                accum = 1;
              }
              ad += a_sub16;
              bd += b_sub16;
            }
          }
          bcur += b_cursor_inc;
        }
        if (is_leader) {
          if constexpr (cta2) umma_commit_2sm_mc(empty_addr, (uint16_t)3);    // the pair's MMAs retired: both CTAs' copies of the stage are free
          else umma_commit_a(empty_addr);                           // frees the smem stage when these MMAs retire
        }
        __syncwarp();
        ++stage;
        soff += stage16;
        bsoff += b_stage_inc;
        if (stage == nstages) { stage = 0; phase ^= 1u; soff = 0; bsoff = 0; }
      }
      if (is_leader) {                                               // accumulator complete -> epilogue (pair: of both CTAs)
        if constexpr (cta2) umma_commit_2sm_mc(tfull0 + 8u * buf, (uint16_t)3);
        else umma_commit_a(tfull0 + 8u * buf);
      }
      __syncwarp();
    }
  } else {
    // =========================== epilogue ===========================
    const int q = warp & 3;                         // TMEM lane quarter this warp may access (hardware: warp id % 4)
    const int gi = warp >> 2;                       // epilogue group
    const int tp = gi % TP, cp = gi / TP;           // which tiles / which column share
    const int r = q * 32 + lane;                    // accumulator row = pixel slot within the tile
    const int et = cp * 128 + r;                    // thread index within the CP groups that share a tile
    const bool pool = (a.flags & Y2_CONV_POOL2) != 0;
    const bool leaky_on = (a.flags & Y2_CONV_LEAKY) != 0;
    const bool out_f32 = (a.flags & Y2_CONV_OUT_F32) != 0;
    float* const my_scale = s_scale[tp];
    float* const my_shift = s_shift[tp];
    // tile-independent part of the row -> pixel mapping
    const int r_tw = r & ((1 << a.tw_log2) - 1);
    const int r_th = (r >> a.tw_log2) & ((1 << a.th_log2) - 1);
    const int r_nb = r >> (a.tw_log2 + a.th_log2);
    const bool r_even = ((r_tw | r_th) & 1) == 0;
    const int Ho = pool ? a.H >> 1 : a.H, Wo = pool ? a.W >> 1 : a.W;
    int staged_ntile = -1;
    // TMA-store epilogue (mode 2, un-pooled bf16): the group's 128 rows x 32 channels of a chunk are staged in 64B-swizzled
    // smem and leave as ONE box store.  The direct path issues four 16-byte stores per lane, each touching 32 different
    // lines: ncu (layer 3 vs the pooled layer 5, identical MMA work) showed the LSU/MIO pipe congested by them -- LDS of
    // scale/shift stalling (short scoreboard), the MMA warp's own LDS delayed, tensor pipe 48 % vs 71 %.
    constexpr bool tma_store = TMAST;
    static_assert(!TMAST || A_MODE == 2, "TMA-store epilogue: halo-patch mode only");
    const uint32_t stg_group = smem_b_stat + a.stg_offset + (uint32_t)gi * 16384u;   // two 8 KB buffers per group
    uint32_t nstore = 0;
    for (int it = tp;; it += TP) {
      const int tile = sched_first + it * sched_step;
      if (tile >= total_tiles) break;
      const int buf = it % NBUF;
      const TileCoord t = decode_tile<CS>(a, tile, crank);
      const int nbase = t.n_tile * BLOCK_N;
      // ---- per-channel scale/shift of this n-tile -> smem (once per change of n-tile, per tile-parallel set) ----
      if (t.n_tile != staged_ntile) {
        asm volatile("bar.sync %0, %1;" ::"r"(1 + tp), "n"(128 * CP) : "memory");   // old values no longer in use
        for (int c = et; c < BLOCK_N; c += 128 * CP) {
          const int col = nbase + c;
          float sc = 1.0f, sh = 0.0f;
          if (col < a.Cout) {
            if (a.scale) sc = __ldg(a.scale + col);
            if (a.shift) sh = __ldg(a.shift + col);
          }
          my_scale[c] = sc;
          my_shift[c] = sh;
        }
        asm volatile("bar.sync %0, %1;" ::"r"(1 + tp), "n"(128 * CP) : "memory");
        staged_ntile = t.n_tile;
      }
      // ---- where does my row go? ----
      bool valid, valid_px = false;
      long long orow;     // output pixel row index
      if constexpr (A_MODE == 0) {
        const long long m = t.m0 + r;
        valid = m < a.M;
        orow = m;
      } else {
        const int n = t.n0 + r_nb, h = t.h0 + r_th, w = t.w0 + r_tw;
        valid_px = n < a.N && h < a.H && w < a.W;
        valid = valid_px && (!pool || r_even);
        orow = (long long)((n * Ho + (pool ? h >> 1 : h)) * Wo + (pool ? w >> 1 : w));   // < 2^31 (host-checked)
      }
      mbar_wait(&tmem_full_bar[buf], ((uint32_t)it / NBUF) & 1u);
      tc_fence_after();
      const uint32_t taddr0 = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BLOCK_N);
#pragma unroll 1
      for (int cc = cp * 32; cc < BLOCK_N; cc += 32 * CP) {
        uint32_t v[32];
        tmem_ld_cols<32>(taddr0 + (uint32_t)cc, v);
        tmem_ld_wait();
        if (cc + 32 * CP >= BLOCK_N) {
          // my last chunk is in registers: hand the accumulator buffer back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if constexpr (cta2) mbar_arrive_cluster(smem_u32(&tmem_empty_bar[buf]) & PEER_BIT_MASK);   // the leader's barrier counts both CTAs
            else mbar_arrive(&tmem_empty_bar[buf]);
          }
        }
        const int c0 = nbase + cc;
        if constexpr (tma_store) {
         if (out_f32) {
          // float32 rows (the training forward pass: conv + bias): the 32-column chunk leaves as TWO boxes of 16 columns -- 64 bytes
          // per row, the staging geometry of the bf16 case.  The direct path issues eight 16-byte stores per lane and chunk, each
          // instruction touching 32 different lines.
#pragma unroll
          for (int part = 0; part < 2; ++part) {
            const uint32_t stg = stg_group + (nstore & 1u) * 8192u;
            if (r == 0) bulk_wait_group_read<1>();
            asm volatile("bar.sync %0, 128;" ::"r"(8 + gi) : "memory");
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int i = 16 * part + 4 * j;
              const float4 sc = *reinterpret_cast<const float4*>(&my_scale[cc + i]);
              const float4 sh = *reinterpret_cast<const float4*>(&my_shift[cc + i]);
              float f0 = fmaf(__uint_as_float(v[i + 0]), sc.x, sh.x), f1 = fmaf(__uint_as_float(v[i + 1]), sc.y, sh.y);
              float f2 = fmaf(__uint_as_float(v[i + 2]), sc.z, sh.z), f3 = fmaf(__uint_as_float(v[i + 3]), sc.w, sh.w);
              if (leaky_on) {
                f0 = fmaxf(f0, a.alpha * f0); f1 = fmaxf(f1, a.alpha * f1);
                f2 = fmaxf(f2, a.alpha * f2); f3 = fmaxf(f3, a.alpha * f3);
              }
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg + (uint32_t)r * 64u + (uint32_t)((j ^ ((r >> 1) & 3)) << 4)),
                           "r"(__float_as_uint(f0)), "r"(__float_as_uint(f1)), "r"(__float_as_uint(f2)), "r"(__float_as_uint(f3))
                           : "memory");
            }
            fence_proxy_async_smem();
            asm volatile("bar.sync %0, 128;" ::"r"(8 + gi) : "memory");
            if (r == 0) {
              tma_store_4d(&tmY, stg, c0 + 16 * part, t.w0, t.h0, t.n0);
              bulk_commit_group();
            }
            ++nstore;
          }
         } else {
          // bf16 rows (not bf16x3: the hi / lo halves as two boxes per chunk were measured slower, see DESIGN.md)
          const uint32_t stg = stg_group + (nstore & 1u) * 8192u;
          if (r == 0) bulk_wait_group_read<1>();               // the store that last used this buffer has read it
          asm volatile("bar.sync %0, 128;" ::"r"(8 + gi) : "memory");
          // row r = h * 8 + w of the box, 64 B per row; 16-byte unit j (8 channels) at j ^ ((r >> 1) & 3)  (SWIZZLE_64B);
          // one unit at a time: affine + leaky + pack + store, so that only the 32 accumulators stay live
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float f[8];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int i = 8 * j + 4 * h;
              const float4 sc = *reinterpret_cast<const float4*>(&my_scale[cc + i]);
              const float4 sh = *reinterpret_cast<const float4*>(&my_shift[cc + i]);
              float f0 = fmaf(__uint_as_float(v[i + 0]), sc.x, sh.x), f1 = fmaf(__uint_as_float(v[i + 1]), sc.y, sh.y);
              float f2 = fmaf(__uint_as_float(v[i + 2]), sc.z, sh.z), f3 = fmaf(__uint_as_float(v[i + 3]), sc.w, sh.w);
              if (leaky_on) {
                f0 = fmaxf(f0, a.alpha * f0); f1 = fmaxf(f1, a.alpha * f1);
                f2 = fmaxf(f2, a.alpha * f2); f3 = fmaxf(f3, a.alpha * f3);
              }
              f[4 * h] = f0; f[4 * h + 1] = f1; f[4 * h + 2] = f2; f[4 * h + 3] = f3;
            }
            const __nv_bfloat162 h0 = __floats2bfloat162_rn(f[0], f[1]), h1 = __floats2bfloat162_rn(f[2], f[3]);
            const __nv_bfloat162 h2 = __floats2bfloat162_rn(f[4], f[5]), h3 = __floats2bfloat162_rn(f[6], f[7]);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg + (uint32_t)r * 64u + (uint32_t)((j ^ ((r >> 1) & 3)) << 4)),
                         "r"(*reinterpret_cast<const uint32_t*>(&h0)), "r"(*reinterpret_cast<const uint32_t*>(&h1)),
                         "r"(*reinterpret_cast<const uint32_t*>(&h2)), "r"(*reinterpret_cast<const uint32_t*>(&h3))
                         : "memory");
          }
          fence_proxy_async_smem();
          asm volatile("bar.sync %0, 128;" ::"r"(8 + gi) : "memory");
          if (r == 0) {
            tma_store_4d(&tmY, stg, c0, t.w0, t.h0, t.n0);     // rows / pixels outside the tensor are clipped by the TMA unit
            bulk_commit_group();
          }
          ++nstore;
         }
        } else if (A_MODE != 0 && pool && !out_f32 && c0 + 32 <= a.Cout && (a.ldy & 7) == 0 && (a.lo_off & 7) == 0) {
          epilogue_chunk_pooled_bf16(a, v, my_scale, my_shift, cc, c0, valid_px, orow, leaky_on, lane);
        } else if (c0 < (a.split_out ? a.Cout : a.ldy)) {
          epilogue_chunk<32>(a, v, my_scale, my_shift, cc, c0, valid, orow, pool, leaky_on, out_f32);
        }
        __syncwarp();                               // reconverge before the next .sync.aligned TMEM load
      }
    }
    if constexpr (tma_store) {
      if (r == 0) bulk_wait_group_read<0>();             // smem must outlive the last box stores' reads
    }
  }

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  if constexpr (CTA2) cluster_sync_all();               // nobody exits while a partner may still write/signal here
  if (warp == WARP_MMA) {
    __syncwarp();
    tc_fence_after();
    if constexpr (cta2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------
// Input-stationary 3x3 convolution for the 64-filter layers on large maps (Darknet19 layers 2 and 4), CTA pairs.
//
// Why.  At N = 64 a pair MMA fetches (4096 + 16 * 64) B of operands for 32 clk of arithmetic: 80 clk at the ~64 B/clk of
// the smem operand path, i.e. the tensor pipe cannot exceed 40 % however the loop is written (section 4.1 of DESIGN.md;
// measured 43 %).  The A slice (128 pixels x 16 channels) is what is expensive, and the tap loop re-reads it nine times.
// Here the three HORIZONTAL taps become column blocks of ONE MMA: D[p, (kw, co)] = sum_{kh, c} A[p + kh rows, c] *
// W[kh][kw][c][co] with N = 3 * 64 = 192, so an A slice is read once per filter ROW: (4096 + 16 * 192) / 64 = 112 clk for
// 96 clk of arithmetic (86 %).  The horizontal shift moves to the accumulator: out[h, w] = D[(h, w - 1), kw = 0] +
// D[(h, w), kw = 1] + D[(h, w + 1), kw = 2] -- two warp shuffles per output value in the epilogue, which is why the tile is
// 8 rows x 16 pixels (a 16-lane half warp per row): lane L of a row produces output column L from D rows L, L + 1, L + 2,
// columns 14 and 15 of every tile are halo (tiles advance by 14 pixels: 87.5 % of the MMA rows are outputs).
//   smem   [resident filters: (kh, chunk) sub-blocks of 96 rows x KCHUNK -- this CTA's half of the 192 (kw, co) rows]
//          [ring of (8 + 2) x 16 pixel patches, one per channel chunk]; the vertical taps are descriptor shifts by one patch
//          row (two swizzle atoms), as in the halo-patch mode of conv_tc_kernel
//   TMEM   two accumulators of 192 columns; roles, barriers and the epilogue math (scale/shift, leaky, pool, bf16 / bf16x3 /
//          float32 stores) are those of conv_tc_kernel.
// ------------------------------------------------------------------------------------------
constexpr int IS_N = 192, IS_COUT = 64, IS_OUT_W = 14, IS_TW = 16, IS_TH = 8, IS_PROWS = IS_TH + 2;

template <int KIND>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
conv_is_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmY,
               const ConvArgs a) {
  constexpr uint32_t ROW_BYTES = KIND == 1 ? 64u : 128u;
  constexpr int KSTEPS = ROW_BYTES / 32;
  constexpr int NBUF = 2;
  constexpr uint32_t A_STAGE = IS_PROWS * IS_TW * ROW_BYTES;           // 160 patch pixels
  constexpr uint32_t B_SUB = (IS_N / 2) * ROW_BYTES;                   // 96 (kw, co) rows of one (kh, chunk) sub-block
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], tmem_full_bar[NBUF], tmem_empty_bar[NBUF], bfull_bar;
  __shared__ uint32_t s_tmem_base;
  __shared__ __align__(16) float s_scale[IS_COUT], s_shift[IS_COUT];

  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // resident filters (b_stationary): [all (kh, chunk) sub-blocks][ring of patches]; streamed (bf16x3 at 128 channels: the bank
  // does not fit): every ring stage is [patch | the chunk's three kh sub-blocks]
  const bool bstat = a.b_stationary != 0;
  const uint32_t smem_b = (smem_u32(smem) + 1023u) & ~1023u;
  const uint32_t smem_a = smem_b + (bstat ? ((a.b_total_bytes + 1023u) & ~1023u) : 0u);
  const uint32_t stage_bytes = A_STAGE + (bstat ? 0u : 3u * B_SUB);
  const uint32_t crank = cluster_ctarank();
  const int pair = (int)(blockIdx.x >> 1), npairs = (int)(gridDim.x >> 1);
  const int nsub = 3 * a.cchunks;                                      // (kh, chunk) sub-blocks

  if (warp == WARP_PRODUCER && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
    for (int s = 0; s < a.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int b = 0; b < NBUF; ++b) { mbar_init(&tmem_full_bar[b], 1); mbar_init(&tmem_empty_bar[b], 16); }   // 2 groups x 4 warps x 2 CTAs
    mbar_init(&bfull_bar, 1);
    fence_barrier_init();
  }
  if (warp == WARP_MMA) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem_base)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;
  pdl_wait();
  if (threadIdx.x < IS_COUT) {
    s_scale[threadIdx.x] = a.scale ? __ldg(a.scale + threadIdx.x) : 1.0f;
    s_shift[threadIdx.x] = a.shift ? __ldg(a.shift + threadIdx.x) : 0.0f;
  }
  __syncthreads();
  // pair p takes super tiles p, p + npairs, ...: two consecutive tiles (rank 0 / 1); tile -> (n, th, tw)
  const int m_groups = (a.m_tiles + 1) / 2;
  auto tile_of = [&](int sg, int& n, int& h0, int& w0) {
    uint32_t mt = (uint32_t)sg * 2u + crank;
    if ((int)mt >= a.m_tiles) mt = (uint32_t)a.m_tiles - 1u;            // odd tile count: the partner repeats the last tile (same values stored twice)
    const uint32_t q = fdiv(mt, a.fd_w_mul, a.fd_w_shr);                // / tiles_w
    const uint32_t twi = mt - q * (uint32_t)a.tiles_w;
    const uint32_t ni = fdiv(q, a.fd_h_mul, a.fd_h_shr);                // / tiles_h
    const uint32_t thi = q - ni * (uint32_t)a.tiles_h;
    n = (int)ni; h0 = (int)thi * IS_TH; w0 = (int)twi * IS_OUT_W;
  };

  if (warp == WARP_PRODUCER) {
    // ---- resident filters: this CTA's 96 of the 192 (kw, co) rows of every (kh, chunk) sub-block, three 32-row pieces each ----
    if (bstat && lane == 0 && crank == 0) mbar_expect_tx(&bfull_bar, 2u * a.b_total_bytes);
    __syncwarp();
    const uint32_t bbar = smem_u32(&bfull_bar) & PEER_BIT_MASK;
    for (int i = lane; i < (bstat ? nsub * 3 : 0); i += 32) {
      const int sub = i / 3, piece = i - sub * 3;
      const int kh = sub / a.cchunks, cc = sub - kh * a.cchunks;
      const int nrow = (int)crank * (IS_N / 2) + piece * 32;           // row of the (kw, co) stack
      const int kw = nrow >> 6, co0 = nrow & 63;
      tma_load_2d_2sm(smem_b + (uint32_t)sub * B_SUB + (uint32_t)piece * 32u * ROW_BYTES, &tmB, bbar,
                      (kh * 3 + kw) * a.cin_p + cc * a.kchunk, co0);
    }
    __syncwarp();
    {
      // lane 0: the patch (and the barrier handshake); streamed filters: lanes 1..9 fetch the chunk's 3 kh x 3 row pieces
      uint32_t stage = 0, phase = 0;
      for (int sg = pair; sg < m_groups; sg += npairs) {
        int n, h0, w0;
        tile_of(sg, n, h0, w0);
        for (int cc = 0; cc < a.cchunks; ++cc) {
          if (lane == 0) {
            mbar_wait(&empty_bar[stage], phase ^ 1u);
            if (crank == 0) mbar_expect_tx(&full_bar[stage], 2u * stage_bytes);
          }
          __syncwarp();
          const uint32_t fbar = smem_u32(&full_bar[stage]) & PEER_BIT_MASK;
          const uint32_t sA = smem_a + stage * stage_bytes;
          if (lane == 0) {
            const int ca = cc < a.a_wrap ? cc : cc - a.a_wrap;            // bf16x3: the third K block re-reads the hi channels
            tma_load_4d_2sm(sA, &tmA, fbar, ca * a.kchunk, w0 - 1, h0 - 1, n);
          } else if (!bstat && lane < 10) {
            const int kh = (lane - 1) / 3, piece = (lane - 1) - kh * 3;
            const int nrow = (int)crank * (IS_N / 2) + piece * 32;
            const int kw = nrow >> 6, co0 = nrow & 63;
            tma_load_2d_2sm(sA + A_STAGE + (uint32_t)kh * B_SUB + (uint32_t)piece * 32u * ROW_BYTES, &tmB, fbar,
                            (kh * 3 + kw) * a.cin_p + cc * a.kchunk, co0);
          }
          __syncwarp();
          if (++stage == (uint32_t)a.stages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == WARP_MMA) {
    if (crank == 0) {
      uint32_t is_leader;
      asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(is_leader));
      // D = f32, A = B = bf16, K-major both, N = 192, M = 256 (the pair)
      constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(IS_N >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      constexpr uint32_t layout = KIND == 1 ? 4u : 2u;
      const uint64_t adesc0 = make_smem_desc(smem_a, 16u, 8u * ROW_BYTES, layout);
      const uint64_t bdesc0 = make_smem_desc(bstat ? smem_b : smem_a + A_STAGE, 16u, 8u * ROW_BYTES, layout);
      constexpr uint32_t KH16 = (IS_TW * ROW_BYTES) >> 4;              // one patch row = two swizzle atoms
      if (bstat) {
        mbar_wait(&bfull_bar, 0);
        tc_fence_after();
      }
      uint32_t stage = 0, phase = 0, it = 0;
      for (int sg = pair; sg < m_groups; sg += npairs, ++it) {
        const uint32_t buf = it & 1u;
        mbar_wait(&tmem_empty_bar[buf], ((it >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + buf * (uint32_t)IS_N;
        uint32_t accum = 0;
        for (int cc = 0; cc < a.cchunks; ++cc) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          if (is_leader) {
            const uint64_t ad = adesc0 + (uint32_t)((stage * stage_bytes) >> 4);
#pragma unroll
            for (int kh = 0; kh < 3; ++kh) {
              const uint64_t bd = bdesc0 + (bstat ? (uint32_t)(((uint32_t)(kh * a.cchunks + cc) * B_SUB) >> 4)
                                                  : (uint32_t)((stage * stage_bytes + (uint32_t)kh * B_SUB) >> 4));
#pragma unroll
              for (int ks = 0; ks < KSTEPS; ++ks) {
                umma_bf16_2sm(tmem_d, ad + (uint32_t)kh * KH16 + (uint32_t)(ks * 2), bd + (uint32_t)(ks * 2), idesc, accum);
                accum = 1;
              }
            }
            umma_commit_2sm_mc(smem_u32(&empty_bar[stage]), (uint16_t)3);
          }
          __syncwarp();
          if (++stage == (uint32_t)a.stages) { stage = 0; phase ^= 1u; }
        }
        if (is_leader) umma_commit_2sm_mc(smem_u32(&tmem_full_bar[buf]), (uint16_t)3);
        __syncwarp();
      }
    }
  } else {
    // ---- epilogue: group gi -> tiles of parity tp, output channels [cp * 32, cp * 32 + 32) ----
    const int q = warp & 3, gi = warp >> 2;
    const int tp = gi & 1, cp = gi >> 1;
    const int r = q * 32 + lane;
    const int r_tw = r & (IS_TW - 1), r_th = r >> 4;
    const bool pool = (a.flags & Y2_CONV_POOL2) != 0;
    const bool leaky_on = (a.flags & Y2_CONV_LEAKY) != 0;
    const bool out_f32 = (a.flags & Y2_CONV_OUT_F32) != 0;
    const int Ho = pool ? a.H >> 1 : a.H, Wo = pool ? a.W >> 1 : a.W;
    const int cc0 = cp * 32;
    // TMA-store epilogue (un-pooled outputs): the group's 8 x 14 output pixels x 32 channels are staged as 64-byte rows in
    // 64B-swizzled smem (box row = h * 14 + w) and leave as one box store -- float32 rows as two boxes of 16 channels, bf16x3 as
    // a hi and a lo box; one 8 KB buffer per group (a group stores once per two tiles).
    const bool tma_st = a.tma_store != 0 && !pool;
    const uint32_t stg = smem_a + (uint32_t)a.stages * stage_bytes + (uint32_t)gi * 8192u;
    const int brow = r_th * IS_OUT_W + r_tw;
    const uint32_t stg_row = stg + (uint32_t)brow * 64u;
    const uint32_t swz = (uint32_t)((brow >> 1) & 3);
    int it = tp;
    for (int sg = pair + tp * npairs; sg < m_groups; sg += 2 * npairs, it += 2) {
      int n, h0, w0;
      tile_of(sg, n, h0, w0);
      const int h = h0 + r_th, w = w0 + r_tw;
      const bool valid_px = r_tw < IS_OUT_W && h < a.H && w < a.W;
      const bool valid = valid_px && (!pool || (((r_tw | r_th) & 1) == 0));
      const long long orow = (long long)((n * Ho + (pool ? h >> 1 : h)) * Wo + (pool ? w >> 1 : w));
      const uint32_t buf = (uint32_t)tp;
      mbar_wait(&tmem_full_bar[buf], ((uint32_t)it >> 1) & 1u);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * (uint32_t)IS_N + (uint32_t)cc0;
      uint32_t sum[32];
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        uint32_t v0[16], v1[16], v2[16];
        tmem_ld_cols<16>(taddr + (uint32_t)(hf * 16), v0);
        tmem_ld_cols<16>(taddr + (uint32_t)(IS_COUT + hf * 16), v1);
        tmem_ld_cols<16>(taddr + (uint32_t)(2 * IS_COUT + hf * 16), v2);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float c1 = __shfl_down_sync(0xffffffffu, __uint_as_float(v1[i]), 1);
          const float c2 = __shfl_down_sync(0xffffffffu, __uint_as_float(v2[i]), 2);
          sum[hf * 16 + i] = __float_as_uint((__uint_as_float(v0[i]) + c1) + c2);      // taps kw = 0, 1, 2 in order
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(smem_u32(&tmem_empty_bar[buf]) & PEER_BIT_MASK);
      if (tma_st) {
        const int nparts = (out_f32 || a.split_out) ? 2 : 1;
#pragma unroll
        for (int part = 0; part < 2; ++part) {
          if (part >= nparts) break;
          if (r == 0) bulk_wait_group_read<0>();              // the group's previous box store has read the buffer
          asm volatile("bar.sync %0, 128;" ::"r"(8 + gi) : "memory");
          if (r_tw < IS_OUT_W) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 pk;
              if (out_f32) {
                float f[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const int i = 16 * part + 4 * j + e;
                  f[e] = fmaf(__uint_as_float(sum[i]), s_scale[cc0 + i], s_shift[cc0 + i]);
                  if (leaky_on) f[e] = fmaxf(f[e], a.alpha * f[e]);
                }
                pk = make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3]));
              } else {
                float f[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  const int i = 8 * j + e;
                  f[e] = fmaf(__uint_as_float(sum[i]), s_scale[cc0 + i], s_shift[cc0 + i]);
                  if (leaky_on) f[e] = fmaxf(f[e], a.alpha * f[e]);
                }
                uint4 hi, lo;
                split8_bf16(f, hi, lo);
                pk = part ? lo : hi;
              }
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg_row + (((uint32_t)j ^ swz) << 4)), "r"(pk.x), "r"(pk.y),
                           "r"(pk.z), "r"(pk.w)
                           : "memory");
            }
          }
          fence_proxy_async_smem();
          asm volatile("bar.sync %0, 128;" ::"r"(8 + gi) : "memory");
          if (r == 0) {
            tma_store_4d(&tmY, stg, cc0 + (out_f32 ? 16 * part : part * a.lo_off), w0, h0, n);   // clipped at the image border
            bulk_commit_group();
          }
        }
      } else if (pool && !out_f32 && (a.ldy & 7) == 0 && (a.lo_off & 7) == 0)
        epilogue_chunk_pooled_bf16(a, sum, s_scale, s_shift, cc0, cc0, valid_px, orow, leaky_on, lane);
      else
        epilogue_chunk<32>(a, sum, s_scale, s_shift, cc0, cc0, valid, orow, pool, leaky_on, out_f32);
      __syncwarp();
    }
    if (tma_st && r == 0) bulk_wait_group_read<0>();      // smem must outlive the last box store's read
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == WARP_MMA) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ------------------------------------------------------------------------------------------
// host side: tensor maps (driver entry points fetched at run time -> no libcuda link dependency)
// ------------------------------------------------------------------------------------------
PFN_encodeTiled g_encodeTiled = nullptr;
PFN_encodeIm2col g_encodeIm2col = nullptr;
int num_sms() {
  static int cache[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (!cache[dev]) {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    cache[dev] = n > 0 ? n : 148;
  }
  return cache[dev];
}
int g_driver_version = 0;
static std::mutex g_mu;

int load_driver_entry_points() {
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_encodeTiled && g_encodeIm2col) return Y2_OK;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || !fn) {
    set_error("cuTensorMapEncodeTiled not available: %s", cudaGetErrorString(e));
    return Y2_ERR_DRIVER;
  }
  g_encodeTiled = (PFN_encodeTiled)fn;
  fn = nullptr;
  e = cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || !fn) {
    set_error("cuTensorMapEncodeIm2col not available: %s", cudaGetErrorString(e));
    return Y2_ERR_DRIVER;
  }
  g_encodeIm2col = (PFN_encodeIm2col)fn;
  cudaDriverGetVersion(&g_driver_version);
  return Y2_OK;
}

static int tmap_result(CUresult r, const char* who, const char* name) {
  if (r == CUDA_SUCCESS) return Y2_OK;
  set_error("%s: tensor map %s encode failed (CUresult %d)", who, name, (int)r);
  return Y2_ERR_DRIVER;
}

int tmap_im2col_nhwc(CUtensorMap* tm, const void* x, int N, int H, int W, int C, int ksize, int chans, int pixels,
                     CUtensorMapSwizzle sw, const char* who, const char* name) {
  const int pad = ksize / 2;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  int lower[2] = {-pad, -pad};
  int upper[2] = {pad - (ksize - 1), pad - (ksize - 1)};
  CUresult r = g_encodeIm2col(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x), dims, strides, lower, upper,
                              (cuuint32_t)chans, (cuuint32_t)pixels, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  // same small-tensor fix-up CUTLASS applies (cute/atom/copy_traits_sm90_im2col.hpp) for drivers <= 13.1
  if (r == CUDA_SUCCESS && g_driver_version <= 13010 && (size_t)N * H * W * C * 2 < 131072)
    reinterpret_cast<uint64_t*>(tm)[1] &= ~(1ull << 21);
  return tmap_result(r, who, name);
}

int tmap_nhwc_box(CUtensorMap* tm, const void* base, CUtensorMapDataType dt, int N, int H, int W, int C, int ld,
                  const cuuint32_t box[4], CUtensorMapSwizzle sw, CUtensorMapL2promotion l2, const char* who, const char* name) {
  const cuuint64_t es = dt == CU_TENSOR_MAP_DATA_TYPE_FLOAT32 ? 4 : 2;          // float32 or bf16
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)ld * es, (cuuint64_t)W * ld * es, (cuuint64_t)H * W * ld * es};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encodeTiled(tm, dt, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, l2,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return tmap_result(r, who, name);
}

int tmap_kmajor(CUtensorMap* tm, const void* base, int K, long long rows, int box_k, int box_rows, CUtensorMapSwizzle sw,
                CUtensorMapL2promotion l2, const char* who, const char* name) {
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_k, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encodeTiled(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, sw, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return tmap_result(r, who, name);
}


// choose the pixel box (NB x TH x TW = 128, powers of two) with the least padding waste
static void choose_box(int N, int H, int W, bool pool, int* tw, int* th, int* nb) {
  double best = 1e30;
  int btw = 16, bth = 8, bnb = 1;
  for (int TW = (pool ? 2 : 1); TW <= (pool ? 16 : 128); TW <<= 1)
    for (int TH = (pool ? 2 : 1); TH * TW <= 128; TH <<= 1) {
      int NB = 128 / (TW * TH);
      double cover = (double)((W + TW - 1) / TW * TW) * ((H + TH - 1) / TH * TH) * ((N + NB - 1) / NB * NB);
      double waste = cover / ((double)W * H * N);
      // prefer wide boxes (longer contiguous runs for the TMA) when the waste ties
      double score = waste - 1e-6 * TW;
      if (score < best) { best = score; btw = TW; bth = TH; bnb = NB; }
    }
  *tw = btw; *th = bth; *nb = bnb;
}

template <int BLOCK_N, int A_MODE, int KIND, bool CTA2 = false, bool TMAST = false>
static int launch_conv3(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmY, const ConvArgs& a, size_t smem, cudaStream_t st) {
  constexpr int CS = CTA2 ? 2 : 1;
  long long units = (long long)((a.m_tiles + CS - 1) / CS) * a.n_tiles;
  long long want = units * CS;
  int grid = (int)(want < g_num_sms ? want : g_num_sms);
  grid -= grid % CS;
  return launch_cluster(conv_tc_kernel<BLOCK_N, A_MODE, KIND, CTA2, TMAST>, grid, TC_THREADS, smem, (unsigned)CS, st, tmA, tmB, tmY, a);
}

template <int BLOCK_N, int KIND>
static int launch_conv2(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmY, const ConvArgs& a, size_t smem, cudaStream_t st) {
  if constexpr (KIND == 2 && BLOCK_N >= 128) {
    if (a.cta2 && a.a_mode == 0) return launch_conv3<BLOCK_N, 0, KIND, true>(tmA, tmB, tmY, a, smem, st);
    if (a.cta2 && a.a_mode == 1) return launch_conv3<BLOCK_N, 1, KIND, true>(tmA, tmB, tmY, a, smem, st);
  }
  switch (a.a_mode) {
    case 0: return launch_conv3<BLOCK_N, 0, KIND>(tmA, tmB, tmY, a, smem, st);
    case 1: return launch_conv3<BLOCK_N, 1, KIND>(tmA, tmB, tmY, a, smem, st);
    default:
      if constexpr (KIND == 0) {
        if (a.tma_store) return launch_conv3<BLOCK_N, 2, KIND, false, true>(tmA, tmB, tmY, a, smem, st);
      }
      if constexpr (KIND != 0 && BLOCK_N <= 128) {
        if constexpr ((KIND == 2 && BLOCK_N == 128) || (KIND == 1 && BLOCK_N == 64)) {
          if (a.cta2 && a.tma_store) return launch_conv3<BLOCK_N, 2, KIND, true, true>(tmA, tmB, tmY, a, smem, st);
        }
        if (a.cta2) return launch_conv3<BLOCK_N, 2, KIND, true>(tmA, tmB, tmY, a, smem, st);
      }
      return launch_conv3<BLOCK_N, 2, KIND>(tmA, tmB, tmY, a, smem, st);
  }
}

static int launch_conv(int block_n, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmY, const ConvArgs& a,
                       size_t smem, cudaStream_t st) {
  if (a.first_layer) return launch_conv2<32, 0>(tmA, tmB, tmY, a, smem, st);
  if (a.row_bytes == 64) {
    switch (block_n) {
      case 64: return launch_conv2<64, 1>(tmA, tmB, tmY, a, smem, st);
      case 128: return launch_conv2<128, 1>(tmA, tmB, tmY, a, smem, st);
      default: return launch_conv2<256, 1>(tmA, tmB, tmY, a, smem, st);
    }
  }
  switch (block_n) {
    case 64: return launch_conv2<64, 2>(tmA, tmB, tmY, a, smem, st);
    case 128: return launch_conv2<128, 2>(tmA, tmB, tmY, a, smem, st);
    default: return launch_conv2<256, 2>(tmA, tmB, tmY, a, smem, st);
  }
}

int conv_streamk_try(const ConvCall& c, cudaStream_t st, int* handled);   // conv_streamk_tcgen05.cu

// The input-stationary kernel (conv_is_kernel): 3x3, Cout == 64, maps >= 64 x 64, filters resident.  *handled = 1 when issued.
static int conv_is_try(const ConvCall& c, cudaStream_t st, int* handled) {
  *handled = 0;
  if (env().conv_no_is || c.ksize != 3 || c.Cout != IS_COUT || c.H < 64 || c.W < 64 || c.Cin % 32 != 0 || g_num_sms < 2) return Y2_OK;
  // Short K (layer 2: 32 channels) is epilogue-bound, and this kernel's epilogue is the heavier one (three accumulator
  // blocks + two shuffles per value): measured 149 vs 115 us there, against 88 vs 114 us on layer 4 (128 channels).
  if (c.b_cin < 96 && !env().conv_force_is) return Y2_OK;
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.scale = c.scale; a.shift = c.shift; a.y = c.y;
  a.N = c.N; a.H = c.H; a.W = c.W; a.Cout = c.Cout;
  a.M = c.M;
  a.split_out = c.split_out ? 1 : 0;
  a.lo_off = c.lo_off;
  a.ldy = c.ldy;
  a.flags = c.flags; a.alpha = c.alpha; a.ksize = 3; a.pad = 1;
  a.cin_p = c.b_cin;
  a.kchunk = (c.Cin % 64 == 0) ? 64 : 32;
  a.row_bytes = a.kchunk * 2;
  a.cchunks = a.cin_p / a.kchunk;
  a.a_wrap = c.a_cin / a.kchunk;
  a.kblocks = 9 * a.cchunks;
  a.tw_log2 = 4; a.th_log2 = 3; a.nb_log2 = 0;
  a.tiles_w = (c.W + IS_OUT_W - 1) / IS_OUT_W; a.tiles_h = (c.H + IS_TH - 1) / IS_TH; a.tiles_nb = c.N;
  const long long tiles = (long long)a.tiles_w * a.tiles_h * c.N;
  if (tiles < 2 || tiles >= (1ll << 30) || a.M >= (1ll << 31)) return Y2_OK;
  a.m_tiles = (int)tiles; a.n_tiles = 1;
  a.a_stage_bytes = (uint32_t)(IS_PROWS * IS_TW * a.row_bytes);
  a.b_sub_bytes = (uint32_t)((IS_N / 2) * a.row_bytes);
  a.b_total_bytes = (uint32_t)(3 * a.cchunks) * a.b_sub_bytes;
  const size_t SMEM_BUDGET = 218 * 1024;
  size_t b_region = ((size_t)a.b_total_bytes + 1023) & ~(size_t)1023;
  a.b_stationary = b_region + 3 * (size_t)a.a_stage_bytes <= SMEM_BUDGET ? 1 : 0;
  size_t stage_bytes = a.a_stage_bytes;
  if (!a.b_stationary) {                                 // the bank does not fit (bf16x3, 128 channels): stream the chunk's three kh sub-blocks
    b_region = 0;
    stage_bytes += 3 * (size_t)a.b_sub_bytes;
  }
  // un-pooled outputs leave through 32 KB of staging + TMA box stores when at least three ring stages remain next to it
  const size_t IS_STG = 4 * 8192;
  a.tma_store = 0;
  if (!c.pool && a.ldy % 8 == 0 && (reinterpret_cast<uintptr_t>(c.y) & 15) == 0 &&
      (!c.split_out || a.lo_off % 8 == 0) && (SMEM_BUDGET - b_region - IS_STG) / stage_bytes >= 3)
    a.tma_store = 1;
  const size_t stg_bytes = a.tma_store ? IS_STG : 0;
  int stages = (int)((SMEM_BUDGET - b_region - stg_bytes) / stage_bytes);
  if (stages < 3) return Y2_OK;
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  a.stages = stages;
  fastdiv_init((uint32_t)a.tiles_w, &a.fd_w_mul, &a.fd_w_shr);
  fastdiv_init((uint32_t)a.tiles_h, &a.fd_h_mul, &a.fd_h_shr);
  const size_t smem = b_region + (size_t)stages * stage_bytes + stg_bytes + 1024;
  static const char* const who = "y2_conv_fwd_bf16 (input-stationary)";
  const CUtensorMapSwizzle sw = swizzle_for(a.row_bytes);
  CUtensorMap tmA, tmB, tmY;
  const cuuint32_t box_a[4] = {(cuuint32_t)a.kchunk, (cuuint32_t)IS_TW, (cuuint32_t)IS_PROWS, 1};
  int rc = tmap_nhwc_box(&tmA, c.x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, c.N, c.H, c.W, c.a_cin, c.a_cin, box_a, sw,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, who, "A");
  if (rc == Y2_OK)
    rc = tmap_kmajor(&tmB, c.w_packed, 9 * a.cin_p, IS_COUT, a.kchunk, 32, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, who, "B");
  if (rc != Y2_OK) return rc;
  memset(&tmY, 0, sizeof(tmY));
  if (a.tma_store) {
    const cuuint32_t box_y[4] = {c.out_f32 ? 16u : 32u, (cuuint32_t)IS_OUT_W, (cuuint32_t)IS_TH, 1};
    rc = tmap_nhwc_box(&tmY, c.y, c.out_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, c.N, c.H, c.W,
                       c.split_out ? a.lo_off + c.Cout : c.Cout, a.ldy, box_y, CU_TENSOR_MAP_SWIZZLE_64B,
                       CU_TENSOR_MAP_L2_PROMOTION_NONE, who, "Y");
    if (rc != Y2_OK) return rc;
  }
  const int groups = (a.m_tiles + 1) / 2;
  const int npairs = groups < g_num_sms / 2 ? groups : g_num_sms / 2;
  rc = launch_cluster(a.row_bytes == 64 ? conv_is_kernel<1> : conv_is_kernel<2>, 2 * npairs, TC_THREADS, smem, 2u, st, tmA, tmB, tmY, a);
  *handled = rc == Y2_OK;
  return rc;
}

// conv_tc_kernel: every call the other two paths decline
static int conv_generic(const ConvCall& c, cudaStream_t st) {
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.scale = c.scale;
  a.shift = c.shift;
  a.y = c.y;
  a.N = c.N; a.H = c.H; a.W = c.W; a.Cout = c.Cout;
  a.M = c.M;
  a.split_out = c.split_out ? 1 : 0;
  a.lo_off = c.lo_off;
  a.ldy = c.ldy;
  a.flags = c.flags;
  a.alpha = c.alpha;
  a.ksize = c.ksize;
  a.pad = c.pad;
  a.cin_p = c.b_cin;
  const int cout_p = (c.Cout + 15) / 16 * 16;
  a.first_layer = a.cin_p == 8;
  if (a.first_layer) {
    a.kchunk = 8; a.row_bytes = 16; a.kblocks = 1; a.cchunks = 1; a.ksteps = 5;
    a.layout_type = 0;                    // no swizzle: core matrices of 8 rows x 16 B
    a.kstep_bytes = 2 * 16;               // x rows -> two 16-byte K groups per MMA (scaled by rows in-kernel)
  } else if (c.Cin % 64 == 0) {
    a.kchunk = 64; a.row_bytes = 128; a.layout_type = 2; a.ksteps = 4; a.kstep_bytes = 32;
    a.cchunks = a.cin_p / 64; a.kblocks = c.taps * a.cchunks;
  } else {                                // Cin % 32 == 0 (checked with the call)
    a.kchunk = 32; a.row_bytes = 64; a.layout_type = 4; a.ksteps = 2; a.kstep_bytes = 32;
    a.cchunks = a.cin_p / 32; a.kblocks = c.taps * a.cchunks;
  }
  a.a_wrap = a.first_layer ? 1 : c.a_cin / a.kchunk;
  a.a_mode = c.pool ? 1 : 0;
  if (env().conv_force_tiled) a.a_mode = 1;
  // halo-patch mode for 3x3 layers on large maps: an 8 x 16 pixel tile whose (16+2)-row neighbourhood is
  // loaded once per horizontal tap (first layer: once in total) instead of once per tap
  if (c.ksize == 3 && c.H >= 64 && c.W >= 64) a.a_mode = 2;
  int TW = 1, TH = 1, NB = 128;
  if (a.a_mode == 2) {
    TW = 8; TH = 16; NB = 1;
    a.tw_log2 = 3; a.th_log2 = 4; a.nb_log2 = 0;
    a.tiles_w = (c.W + TW - 1) / TW; a.tiles_h = (c.H + TH - 1) / TH; a.tiles_nb = c.N;
    a.m_tiles = a.tiles_w * a.tiles_h * a.tiles_nb;
  } else if (a.a_mode == 1) {
    choose_box(c.N, c.H, c.W, c.pool, &TW, &TH, &NB);
    a.tw_log2 = ilog2(TW); a.th_log2 = ilog2(TH); a.nb_log2 = ilog2(NB);
    a.tiles_w = (c.W + TW - 1) / TW; a.tiles_h = (c.H + TH - 1) / TH; a.tiles_nb = (c.N + NB - 1) / NB;
    a.m_tiles = a.tiles_w * a.tiles_h * a.tiles_nb;
  } else {
    a.m_tiles = (int)((a.M + TILE_M - 1) / TILE_M);
  }
  // N tile: the kernel is L2-bandwidth bound at 128x128 tiles (64 flop per L2 byte), so take 256 columns
  // when that does not cost more in wave quantisation than it saves in operand traffic.
  int block_n = cout_p >= 128 ? 128 : 64;          // (narrower outputs: B rows beyond Cout_p are TMA zero fill)
  if (a.first_layer) block_n = 32;
  if (cout_p >= 256 && !a.first_layer) {
    auto cost = [&](int bn) {
      long long tiles = (long long)a.m_tiles * ((cout_p + bn - 1) / bn);
      long long rounds = (tiles + g_num_sms - 1) / g_num_sms;
      return rounds * (16 + bn / 8);
    };
    if (cost(256) <= cost(128)) block_n = 256;
  }
  // halo-patch mode keeps three taps of B per stage: 256-wide tiles would leave room for a single stage
  if (a.a_mode == 2 && block_n == 256) block_n = 128;
  a.n_tiles = (cout_p + block_n - 1) / block_n;
  if (a.first_layer) {
    a.a_stage_bytes = 10 * TILE_M * 16;
    a.b_stage_bytes = 10 * block_n * 16;
    a.a_sbo = 128; a.a_lbo = TILE_M * 16;
    a.b_sbo = 128; a.b_lbo = block_n * 16;
  } else {
    a.a_stage_bytes = TILE_M * a.row_bytes;
    a.b_stage_bytes = block_n * a.row_bytes;
    a.a_sbo = 8 * a.row_bytes; a.b_sbo = 8 * a.row_bytes;
    a.a_lbo = 16; a.b_lbo = 16;           // ignored for swizzled K-major layouts (CUTLASS writes 1)
  }
  // several (tap, chunk) sub-blocks per stage when they are small (Cin = 32: 12 KB), so that the barrier
  // round trip is amortised over more MMAs
  a.sps = 1;
  if (!a.first_layer && a.a_mode != 2 && a.row_bytes == 64 && a.kblocks % 3 == 0) a.sps = 3;
  a.a_sub_bytes = a.a_stage_bytes;
  a.b_sub_bytes = a.b_stage_bytes;
  if (a.a_mode == 2) {
    if (a.first_layer) {
      a.a_stage_bytes = 3072;                            // 18 x 10 px x 16 B = 2880, padded
      a.a_sub_bytes = 2880;                              // bytes the TMA actually delivers
      a.stages_per_tile = 1;
    } else {
      a.a_stage_bytes = 18 * 8 * a.row_bytes;            // one horizontally shifted patch
      a.a_sub_bytes = a.a_stage_bytes;
      a.b_stage_bytes = 3 * a.b_sub_bytes;               // the three taps (kh = 0..2) of this kw
      a.stages_per_tile = a.cchunks * 3;
    }
  } else {
    if (!a.first_layer) {
      a.a_stage_bytes *= a.sps;
      a.b_stage_bytes *= a.sps;
    }
    a.stages_per_tile = a.kblocks / a.sps;
  }
  Y2_ARG(a.M + TILE_M < (1ll << 31));
  Y2_ARG(a.kblocks <= MAX_UNITS);
  fastdiv_init((uint32_t)a.n_tiles, &a.fd_ntiles_mul, &a.fd_ntiles_shr);
  fastdiv_init((uint32_t)(a.a_mode == 0 ? c.W : a.tiles_w), &a.fd_w_mul, &a.fd_w_shr);
  fastdiv_init((uint32_t)(a.a_mode == 0 ? c.H : a.tiles_h), &a.fd_h_mul, &a.fd_h_shr);
  // bytes per pipeline stage that the TMA unit will report on the stage's mbarrier
  a.tx_bytes = (a.a_mode == 2 && a.first_layer ? a.a_sub_bytes : a.a_stage_bytes);
  fastdiv_init((uint32_t)a.cchunks, &a.fd_cch_mul, &a.fd_cch_shr);
  const size_t SMEM_BUDGET = 218 * 1024;           // dynamic smem for operands (static smem + slack stay below 227 KB)
  // CTA pair on cta_group::2 MMAs for the halo-patch layers with a single N tile (layers 2-5): a single-CTA MMA fetches
  // (4096 + 32 N) bytes of operands at ~64 B/clk -- 96 / 128 clk at N = 64 / 128 for 32 / 64 clk of arithmetic; in a
  // pair each SM fetches its own A rows and HALF of the filters (80 / 96 clk).  Each CTA keeps half of the resident bank.
  a.cta2 = 0;
  bool cta2_streamed = false;
  if (a.a_mode == 2 && !a.first_layer && a.n_tiles == 1 && a.m_tiles >= 2 && block_n >= 64 && block_n <= 128 &&
      ((block_n / 2) * a.row_bytes) % 1024 == 0 && !env().conv_no_cta2) {
    const uint32_t half = (uint32_t)(block_n / 2) * a.row_bytes;
    if ((size_t)a.kblocks * half + 4 * (size_t)a.a_stage_bytes <= SMEM_BUDGET) {
      a.cta2 = 1;
      a.b_sub_bytes = half;
      a.b_stage_bytes = 3 * half;
    } else {
      // the bank does not fit (bf16x3: three times the K extent): still a pair, each CTA STREAMING its half of the three
      // taps' filter rows next to its patch -- (4096 + 16 N) / 64 clk per MMA instead of the single CTA's (4096 + 32 N) / 64
      a.cta2 = 1;
      cta2_streamed = true;
      a.b_sub_bytes = half;
      a.b_stage_bytes = 3 * half;
    }
  }
  // ... and for the im2col / tiled-box modes with 128-byte rows and >= 128-wide tiles (pooled 52x52 / 26x26 layers, the
  // 1x1 layers): the filter tile is streamed, each CTA fetching its half of the rows per stage
  if (a.a_mode != 2 && !a.first_layer && a.row_bytes == 128 && block_n >= 128 && a.m_tiles >= 2 && !env().conv_no_cta2) {
    a.cta2 = 1;
    a.b_sub_bytes = (uint32_t)(block_n / 2) * a.row_bytes;
    a.b_stage_bytes = (uint32_t)a.sps * a.b_sub_bytes;
  }
  // B-stationary: with a single N tile and a small filter bank, every tile of the CTA needs the same B
  a.b_total_bytes = a.first_layer ? a.b_sub_bytes : (uint32_t)a.kblocks * a.b_sub_bytes;
  a.b_stationary = (a.n_tiles == 1 && a.b_total_bytes + 4 * (size_t)a.a_stage_bytes <= SMEM_BUDGET && !cta2_streamed) ? 1 : 0;
  // halo-patch mode with a resident filter bank and a single channel chunk (layer 2: Cin = 32): the three
  // horizontally shifted patches share ONE stage, so the MMA warp issues all 9 taps behind one barrier round trip.
  // With one patch per stage that warp's ~800 clk of per-stage bookkeeping hid 192 clk of tensor work (ncu, r1c).
  if (a.a_mode == 2 && !a.first_layer && a.b_stationary && (a.cchunks == 1 || c.split_in) &&
      a.b_total_bytes + 3 * (size_t)(3 * a.a_sub_bytes) <= SMEM_BUDGET) {
    a.kw_merge = 1;                                      // (several chunks -- the bf16x3 K extent -- : one merged stage per chunk)
    a.a_stage_bytes = 3 * a.a_sub_bytes;
    a.stages_per_tile = a.cchunks;
    a.tx_bytes = a.a_stage_bytes;
  }
  if (a.cta2 && a.a_mode == 2 && !a.b_stationary && !cta2_streamed) {
    set_error("y2_conv_fwd_bf16: internal: halo-patch CTA-pair mode without a resident filter bank");
    return Y2_ERR_UNSUPPORTED;
  }
  // stages: B-stage must stay 1024-byte aligned for the 128B swizzle atoms
  uint32_t stage_bytes = a.a_stage_bytes + (a.b_stationary ? 0u : a.b_stage_bytes);
  Y2_ARG(a.first_layer || (a.a_stage_bytes % 1024 == 0 && a.b_stage_bytes % 1024 == 0));
  const size_t b_region = a.b_stationary ? (((size_t)a.b_total_bytes + 1023) & ~(size_t)1023) : 0;
  // TMA-store epilogue for the un-pooled 128-channel bf16 output of the halo-patch pair kernel (layer 3): 4 groups x 2 x 8 KB
  // of staging.  (Measured: layer 3 108 -> 93 us; the 64-channel layer 4 got slower -- two chunks per tile do not amortise
  // the per-chunk group barriers and the ring loses four stages -- so it keeps the direct stores.)
  // (bf16x3: the hi / lo halves as two boxes per chunk were measured: the 64 KB of staging leaves 3 instead of 5 operand
  // stages next to the streamed filters and layer 3 got SLOWER, 308 -> 325 us -- it keeps the direct stores.)
  const size_t STG_BYTES = 4 * 2 * 8192;
  a.tma_store = 0;
  {
    const bool common = a.a_mode == 2 && !c.pool && c.Cout % 32 == 0 && a.ldy % 8 == 0 && (reinterpret_cast<uintptr_t>(c.y) & 15) == 0 &&
                        b_region + 3 * (size_t)stage_bytes + STG_BYTES <= SMEM_BUDGET;
    // bf16 rows: the 128-channel pair kernel (layer 3); float32 rows (training forward): also the first layer and the 64-channel
    // pair kernel (layer 2), whose 16-byte per-lane stores cost far more than the bf16 ones
    const bool shape_bf16 = !a.first_layer && block_n == 128 && a.row_bytes == 128 && a.cta2;
    const bool shape_f32 = shape_bf16 || (a.first_layer && block_n == 32 && c.Cout == 32) ||
                           (!a.first_layer && block_n == 64 && a.row_bytes == 64 && a.cta2 && c.Cout == 64);
    // (64 columns on 128-byte operand rows -- layer 4 without the input-stationary kernel: 131 -> 141 us, not enabled)
    if (common && !c.out_f32 && shape_bf16 && !c.split_out) a.tma_store = 1;
    if (common && c.out_f32 && shape_f32 && !env().conv_no_tma_store_f32) a.tma_store = 1;
  }
  const size_t stg_bytes = a.tma_store ? STG_BYTES : 0;
  int stages = (int)((SMEM_BUDGET - b_region - stg_bytes) / stage_bytes);
  if (stages > 12) stages = 12;
  if (stages < 2) {
    set_error("y2_conv_fwd_bf16: tile configuration needs %u B per stage; fewer than 2 stages fit", stage_bytes);
    return Y2_ERR_UNSUPPORTED;
  }
  a.stages = stages;
  a.stg_offset = (uint32_t)(b_region + (size_t)stages * stage_bytes);
  size_t smem = b_region + (size_t)stages * stage_bytes + stg_bytes + 1024;

  // ---- tensor maps ----
  static const char* const who = "y2_conv_fwd_bf16";
  CUtensorMap tmA, tmB, tmY;
  const CUtensorMapSwizzle sw = swizzle_for(a.row_bytes);
  int rc;
  if (a.a_mode == 0) {
    rc = tmap_im2col_nhwc(&tmA, c.x, c.N, c.H, c.W, c.a_cin, c.ksize, a.kchunk, TILE_M, sw, who, "A");
  } else if (a.first_layer) {
    // Cin_p == 8: pixels are 16 B, so (channel, w) is one contiguous dimension of W*8 elements.  The halo patch is
    // (8+2) px x 8 ch = 80 contiguous elements per row, 18 rows; a tiled [TW*8, TH, NB] box moves 256-byte rows instead
    // of 16-byte ones (16x fewer TMA requests), and its left/right halo is still zero-filled because the shift is a
    // multiple of one pixel.
    cuuint64_t dims3[3] = {(cuuint64_t)c.W * 8, (cuuint64_t)c.H, (cuuint64_t)c.N};
    cuuint64_t strides3[2] = {(cuuint64_t)c.W * 16, (cuuint64_t)c.H * c.W * 16};
    cuuint32_t box3[3] = {80, 18, 1};
    if (a.a_mode == 1) { box3[0] = (cuuint32_t)TW * 8; box3[1] = (cuuint32_t)TH; box3[2] = (cuuint32_t)NB; }
    cuuint32_t estr[3] = {1, 1, 1};
    rc = tmap_result(g_encodeTiled(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(c.x), dims3, strides3, box3, estr,
                                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE),
                     who, "A");
  } else {
    // halo patch (a_mode 2) or tiled box (a_mode 1)
    const cuuint32_t box[4] = {(cuuint32_t)a.kchunk, a.a_mode == 2 ? 8u : (cuuint32_t)TW, a.a_mode == 2 ? 18u : (cuuint32_t)TH,
                               a.a_mode == 2 ? 1u : (cuuint32_t)NB};
    rc = tmap_nhwc_box(&tmA, c.x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, c.N, c.H, c.W, c.a_cin, c.a_cin, box, sw,
                       CU_TENSOR_MAP_L2_PROMOTION_L2_128B, who, "A");
  }
  if (rc != Y2_OK) return rc;
  if (a.first_layer) {
    // packed as [kgroup=10][Cout_p][8]
    cuuint64_t dims[3] = {8, (cuuint64_t)cout_p, 10};
    cuuint64_t strides[2] = {16, (cuuint64_t)cout_p * 16};
    cuuint32_t box[3] = {8, (cuuint32_t)block_n, 10};
    cuuint32_t estr[3] = {1, 1, 1};
    rc = tmap_result(g_encodeTiled(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(c.w_packed), dims, strides, box,
                                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE),
                     who, "B");
  } else {
    // per-CTA slice of the B tile
    rc = tmap_kmajor(&tmB, c.w_packed, c.taps * a.cin_p, cout_p, a.kchunk, a.cta2 ? block_n / 2 : block_n, sw,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, who, "B");
  }
  if (rc != Y2_OK) return rc;
  memset(&tmY, 0, sizeof(tmY));
  if (a.tma_store) {
    // output [N, H, W, Cout] with row stride ldy: boxes of 32 channels x the 8 x 16 pixel tile, 64-byte swizzled rows
    // (float32 rows: boxes of 16 channels -- the same 64 bytes per row)
    const cuuint32_t box[4] = {c.out_f32 ? 16u : 32u, 8, 16, 1};
    rc = tmap_nhwc_box(&tmY, c.y, c.out_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, c.N, c.H, c.W,
                       c.Cout, a.ldy, box, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE, who, "Y");
    if (rc != Y2_OK) return rc;
  }
  return launch_conv(block_n, tmA, tmB, tmY, a, smem, st);
}

}  // namespace y2

using namespace y2;

extern "C" int y2_conv_fwd_bf16(const y2_conv_params* p, y2_stream_t stream) {
  Y2_ARG(p != nullptr);
  Y2_ARG(p->x && p->w_packed && p->y);
  ConvCall c;
  c.x = p->x; c.w_packed = p->w_packed; c.scale = p->scale; c.shift = p->shift; c.y = p->y;
  c.alpha = p->alpha;
  c.flags = p->flags;
  c.N = p->N; c.H = p->H; c.W = p->W; c.Cin = p->Cin; c.Cout = p->Cout; c.ksize = p->ksize;
  c.pad = c.ksize / 2;
  c.taps = c.ksize * c.ksize;
  c.M = (long long)c.N * c.H * c.W;
  c.split_in = (p->flags & Y2_CONV_IN_SPLIT) != 0;
  c.out_f32 = (p->flags & Y2_CONV_OUT_F32) != 0;
  c.split_out = (p->flags & Y2_CONV_OUT_SPLIT) != 0 && !c.out_f32;
  c.pool = (p->flags & Y2_CONV_POOL2) != 0;
  c.leaky = (p->flags & Y2_CONV_LEAKY) != 0;
  Y2_ARG(c.split_out || p->lo_off == 0);
  if (c.split_in) Y2_ARG(c.Cin % 32 == 0);
  Y2_ARG(c.N > 0 && c.H > 0 && c.W > 0 && c.Cin > 0 && c.Cout > 0 && (c.ksize == 1 || c.ksize == 3));
  if (c.pool) Y2_ARG(c.H % 2 == 0 && c.W % 2 == 0);
  c.lo_off = c.split_out ? (p->lo_off > 0 ? p->lo_off : c.Cout) : 0;
  c.ldy = p->ldy > 0 ? p->ldy : (c.split_out ? 2 * c.Cout : c.Cout);
  Y2_ARG(c.ldy >= c.Cout);
  if (c.split_out) {
    Y2_ARG(c.lo_off >= c.Cout);
    Y2_ARG(c.ldy >= c.lo_off + c.Cout);
  }
  c.a_cin = c.split_in ? 2 * c.Cin : y2_conv_cin_padded(c.Cin);
  c.b_cin = c.split_in ? 3 * c.Cin : c.a_cin;
  if (c.b_cin == 8) Y2_ARG(c.ksize == 3);         // the first layer (3 channels padded to 8)
  if (c.b_cin != 8 && c.Cin % 32 != 0) {
    set_error("y2_conv_fwd_bf16: Cin=%d unsupported (need 3, or a multiple of 32)", c.Cin);
    return Y2_ERR_UNSUPPORTED;
  }
  int rc = load_driver_entry_points();
  if (rc != Y2_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  int handled = 0;
  // float32 pre-BN rows of a deep 3x3 layer on a small map: 256x256 stream-K tiles (conv_streamk_tcgen05.cu)
  rc = conv_streamk_try(c, st, &handled);
  if (rc != Y2_OK || handled) return rc;
  rc = conv_is_try(c, st, &handled);
  if (rc != Y2_OK || handled) return rc;
  return conv_generic(c, st);
}
