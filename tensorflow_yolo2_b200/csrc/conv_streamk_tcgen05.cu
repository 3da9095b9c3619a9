// conv_streamk_tcgen05.cu -- a1 + a2 (scale/shift, leaky) for the deep 3x3 layers on the small maps (26x26 and below):
// the same implicit GEMM as conv_tcgen05.cu with 256 x 256 tiles, each computed by a CTA PAIR (tcgen05 cta_group::2),
// and a stream-K work split over the pairs.
//
// Why 256 x 256.  conv_tc_kernel on these layers is bound by the operand bytes the L2 can deliver into the SMs --
// measured 5 700 B/clk for the whole chip (l1tex__m_xbar2l1tex_read_bytes of L19: 2.41 GB in 215 us), not by the tensor
// pipe (46 % busy).  A 128 x 256 tile needs 48 KB per 64-deep K step = 85 flop per delivered byte; a 256 x 256 tile
// needs 64 KB for twice the flops = 128 flop/B, i.e. 1.5x fewer bytes for the same layer.
//
// Why a CTA pair.  With cta_group::1 every MMA fetches its whole A (128 x 16) and B (N x 16) slice from the issuing SM's
// shared memory, and that operand path moves ~64 B/clk: 12 KB = 192 clk for a 128 x 256 x 16 MMA whose arithmetic takes
// 128 clk.  ncu on the single-CTA kernels (profiles/r1c): 101 / 146 / 192 clk per MMA at N = 64 / 128 / 256, i.e.
// (4096 + 32 N) / 64 -- the tensor pipe tops out at 67 % however the loop is written.  A pair computes one 256 x 256 tile
// with M = 256 MMAs: each SM supplies its own 128 rows of A and HALF of the B rows (8 KB per MMA = the 128 clk of
// arithmetic) and accumulates its 128 rows in its own TMEM.
//   * both CTAs run a TMA producer (own A half, own B half) that signals the LEADER's full barrier (cta_group::2 loads,
//     leader-mapped barrier address); the leader alone expects the 64 KB of both;
//   * the leader's MMA warp issues tcgen05.mma.cta_group::2 and commits with a multicast arrive to the empty / tmem_full
//     barriers of both CTAs; the follower's MMA warp only allocates / frees TMEM;
//   * each CTA's 8 epilogue warps drain their own 128 x 256 accumulator and arrive on the leader's tmem_empty.
// The accumulator is 256 of the 512 TMEM columns, so segments alternate between two buffers and the epilogue of one
// segment overlaps the MMAs of the next.
//
// Stream-K.  256 x 256 tiles leave only 172 tiles for 74 pairs, so instead of whole tiles each pair takes an equal,
// contiguous range of (tile, K-step) units: a pair's range is the TAIL of one tile (its first segment), whole tiles, and
// the HEAD of the next tile (its last segment).  Every range is at least one tile long, so a tile is shared by at most two
// pairs, c (head, done LAST in c's range) and c + 1 (tail, done FIRST in c + 1's range).  Per CTA (same rank: same rows):
//   tail  -> the float32 partial goes to workspace slot blockIdx.x, then flag[blockIdx.x] is released;
//   head  -> the CTA waits for flag[blockIdx.x + 2] (in practice set ~150 k clk earlier), adds the partial to its own
//            accumulator and runs the full epilogue (scale/shift, leaky, float32 or bf16 store) -- the owner
//            finalises, so the fused epilogue survives the K split, there are no atomics and no zero-fill, and the
//            result is bit-reproducible (fixed order: head + tail).
// No circular wait: a tail segment depends on nothing, and all CTAs are co-resident (grid <= #SMs, 1 CTA/SM).
//
// Scope: ksize 1 or 3, stride 1, SAME; Cin % 64 == 0; Cout % 256 == 0; no fused pool; maps smaller than 64x64;
// >= 18 K steps (bf16x3: 6); at least two SMs.  Needs the workspace registered with y2_conv_set_workspace
// (y2_conv_workspace_bytes() bytes, one per stream); without it, or for any other layer, y2_conv_fwd_bf16 stays on
// conv_tc_kernel.  Env Y2_CONV_NO_STREAMK=1 disables the path.
#include "tc_common.cuh"

namespace y2 {

constexpr int SK_THREADS = 64 + 8 * 32;        // warps 0-7 epilogue (2 per TMEM lane quarter), 8 TMA, 9 MMA
constexpr int SK_MAX_UNITS = 1024;             // K steps per tile (bf16x3, 3x3, 1280 channels: 9 * 60 = 540)

struct SkArgs {
  const float* scale;
  const float* shift;
  void* y;
  float* ws_partial;                // [grid][128][256] float32 partial accumulators (slot = the tail CTA)
  int* ws_flags;                    // [grid + 2], all zero between launches (a head resets the flag it consumed)
  float alpha;
  int leaky, out_f32;
  long long M;
  int H, W, ldy, pad;
  int cin_p, cchunks, ksteps;       // K steps per tile = taps * cchunks   (cin_p: K extent per tap of the B operand)
  int split_out, lo_off;            // bf16x3 output: hi at column c, lo at column lo_off + c
  uint32_t fd_cc_mul, fd_cc_shr;    // division by cchunks
  int n_tiles, tiles;
  long long units;                  // tiles * ksteps
  uint32_t fd_nt_mul, fd_nt_shr, fd_w_mul, fd_w_shr, fd_h_mul, fd_h_shr, fd_ks_mul, fd_ks_shr;
};

constexpr uint32_t SK_STG_WARP = 32 * 128;     // per-warp store staging: 32 rows x 32 floats (or bf16), 128B-swizzled

// K step -> (filter tap, A channel coordinate, B K coordinate).  bf16x3 (X3): the hi chunks; the stage adds their lo partners.
__device__ __forceinline__ void sk_unit(const SkArgs& a, int k, int& tap, int& a_c0, int& b_k) {
  tap = (int)fdiv((uint32_t)k, a.fd_cc_mul, a.fd_cc_shr);
  const int j = k - tap * a.cchunks;
  a_c0 = j * 64;
  b_k = tap * a.cin_p + j * 64;
}

// 32 rows x 32 bf16 columns of one warp (lane = row, pk = its 16 packed pairs) -> global rows, through the warp's swizzled
// staging tile so that one store instruction covers whole 64-byte row segments
__device__ __forceinline__ void sk_store_rows_bf16(uint32_t stg, int lane, const uint32_t* pk, __nv_bfloat16* dst, long long grow0,
                                                   long long M, int ldy) {
  // 64-byte rows, 4 units, unit j of row r at (j ^ ((r >> 1) & 3))
#pragma unroll
  for (int j = 0; j < 4; ++j)
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4)),
                 "r"(pk[4 * j]), "r"(pk[4 * j + 1]), "r"(pk[4 * j + 2]), "r"(pk[4 * j + 3])
                 : "memory");
  __syncwarp();
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int r = t * 8 + (lane >> 2), j = lane & 3;
    uint4 o;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(o.x), "=r"(o.y), "=r"(o.z), "=r"(o.w)
                 : "r"(stg + r * 64 + ((j ^ ((r >> 1) & 3)) << 4)));
    if (grow0 + r < M) *reinterpret_cast<uint4*>(dst + (size_t)(grow0 + r) * ldy + j * 8) = o;
  }
  __syncwarp();
}

// affine + leaky done: convert (and, bf16x3, split into hi / lo) and store one 32 x 32 chunk
__device__ __forceinline__ void sk_store_chunk_bf16(const SkArgs& a, uint32_t stg, int lane, const float* f, int col, long long grow0) {
  uint32_t pk[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    pk[i] = *reinterpret_cast<const uint32_t*>(&h);
  }
  __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(a.y) + col;
  sk_store_rows_bf16(stg, lane, pk, dst, grow0, a.M, a.ldy);
  if (a.split_out) {
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const float2 hf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&pk[i]));
      const __nv_bfloat162 l = __floats2bfloat162_rn(f[2 * i] - hf.x, f[2 * i + 1] - hf.y);
      pk[i] = *reinterpret_cast<const uint32_t*>(&l);
    }
    sk_store_rows_bf16(stg, lane, pk, dst + a.lo_off, grow0, a.M, a.ldy);
  }
}

// 512 x 256 pair tiles (two 128-row halves per CTA sharing its half of the filters, 48 KB per K step for twice the flops
// of 32 KB) were measured SLOWER on B200 (L19 149 vs 137 us, L6 116 vs 89 us): the un-overlapped epilogue, the shallower
// 4-stage ring and the coarser tile quantisation cost more than the 1.33x fewer delivered bytes per flop bring.
constexpr uint32_t SK2_A_BYTES = 128 * 128;
// X3 (the bf16x3 precision mode): one pipeline stage holds BOTH halves of a 64-channel chunk of the pixels
// (hi, lo) and of the filters (w_hi, w_lo) -- 64 KB per CTA -- and feeds three MMAs per K = 16 slice (hi*w_hi, lo*w_hi,
// hi*w_lo): 64 KB delivered per 12 MMAs instead of the 96 KB the generic K walk over [hi | lo | hi] x [w_hi | w_hi | w_lo]
// needs.  The kernel is bound by exactly that delivery (above), and the bf16x3 operands (144 MB per head layer) no longer
// fit the L2 beside the output, so fewer re-fetched bytes is what counts.  Same packed weights: w_hi = first, w_lo = third
// block of a tap.
template <bool X3> struct Sk2Cfg {
  static constexpr uint32_t STAGE = X3 ? 4 * SK2_A_BYTES : 2 * SK2_A_BYTES;   // per CTA: pixels (+ lo) + 128 filters (+ lo)
  static constexpr int STAGES = X3 ? 3 : 6;                                  // 192 KB of operands either way
};
constexpr size_t SK2_SMEM = (size_t)Sk2Cfg<false>::STAGES * Sk2Cfg<false>::STAGE + 8 * SK_STG_WARP + 1024;
static_assert(Sk2Cfg<true>::STAGES * Sk2Cfg<true>::STAGE == Sk2Cfg<false>::STAGES * Sk2Cfg<false>::STAGE, "operand smem");

template <bool X3>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(SK_THREADS, 1)
conv_streamk2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const SkArgs a) {
  constexpr int SK2_STAGES = Sk2Cfg<X3>::STAGES;
  constexpr uint32_t SK2_STAGE = Sk2Cfg<X3>::STAGE;
  constexpr int NCHUNK = 4;                                    // 32-column chunks per epilogue warp and segment
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t full_bar[SK2_STAGES], empty_bar[SK2_STAGES], tmem_full[2], tmem_empty[2];
  __shared__ uint32_t s_tmem_base;
  pdl_launch_dependents();                                      // persistent grid: the next kernel may take SMs as my CTAs retire
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem) + 1023u) & ~1023u;
  const uint32_t rank = cluster_ctarank();                      // 0 = leader (issues the MMAs)
  const int pair = (int)(blockIdx.x >> 1), npairs = (int)(gridDim.x >> 1);

  // the pair's contiguous range of (tile, K-step) units
  const long long u_begin = a.units * pair / npairs, u_end = a.units * (pair + 1) / npairs;

  if (warp == 8) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
      for (int s = 0; s < SK2_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
      for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], 16); }   // 8 warps x 2 CTAs
      fence_barrier_init();
    }
  }
  if (warp == 9) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem_base)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                           // the partner's barriers exist before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;
  pdl_wait();                                                   // everything above overlapped the previous kernel's tail

  if (warp == 8) {
    // =========================== TMA producer (both CTAs) ===========================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      long long u = u_begin;
      while (u < u_end) {
        const uint32_t tile = (uint32_t)fdiv((uint32_t)u, a.fd_ks_mul, a.fd_ks_shr);       // units < 2^31 (host-checked)
        const int k0 = (int)(u - (long long)tile * a.ksteps);
        const int k1 = (int)min((long long)a.ksteps, k0 + (u_end - u));
        const uint32_t mt = fdiv(tile, a.fd_nt_mul, a.fd_nt_shr);
        const int nrow0 = (int)(tile - mt * (uint32_t)a.n_tiles) * 256 + (int)rank * 128;   // my half of the filters
        uint32_t m = mt * 256u + rank * 128u;                   // my rows
        if ((long long)m >= a.M) m = 0;                        // entirely past the end: load valid pixels, rows are masked
        const uint32_t row = fdiv(m, a.fd_w_mul, a.fd_w_shr);
        const int w0 = (int)(m - row * (uint32_t)a.W);
        const uint32_t img = fdiv(row, a.fd_h_mul, a.fd_h_shr);
        const int h0 = (int)(row - img * (uint32_t)a.H), n0 = (int)img;
        for (int k = k0; k < k1; ++k) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);             // my own copy: the leader's commit arrives on both
          if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * SK2_STAGE);
          int tap, a_c0, b_k;
          sk_unit(a, k, tap, a_c0, b_k);
          const int kh = a.pad ? (tap * 11) >> 5 : 0, kw = tap - kh * 3;       // tap / 3 for tap < 9 (1x1: tap == 0)
          const uint32_t sA = smem_base + stage * SK2_STAGE;
          const uint32_t bar = smem_u32(&full_bar[stage]) & PEER_BIT_MASK;      // the leader's barrier
          if constexpr (X3) {
            // stage = [pixels hi | pixels lo | filters hi | filters lo]; the lo channels sit one block (of cin_p / 3 = Cin)
            // further, w_lo two blocks further
            const int lo_c = a.cin_p / 3, lo_k = 2 * lo_c;
            tma_load_im2col_4d_2sm(sA, &tmA, bar, a_c0, w0 - a.pad, h0 - a.pad, n0, (uint16_t)kw, (uint16_t)kh);
            tma_load_im2col_4d_2sm(sA + SK2_A_BYTES, &tmA, bar, a_c0 + lo_c, w0 - a.pad, h0 - a.pad, n0, (uint16_t)kw, (uint16_t)kh);
            tma_load_2d_2sm(sA + 2 * SK2_A_BYTES, &tmB, bar, b_k, nrow0);
            tma_load_2d_2sm(sA + 3 * SK2_A_BYTES, &tmB, bar, b_k + lo_k, nrow0);
          } else {
            tma_load_im2col_4d_2sm(sA, &tmA, bar, a_c0, w0 - a.pad, h0 - a.pad, n0, (uint16_t)kw, (uint16_t)kh);
            tma_load_2d_2sm(sA + SK2_A_BYTES, &tmB, bar, b_k, nrow0);
          }
          if (++stage == SK2_STAGES) { stage = 0; phase ^= 1u; }
        }
        u += k1 - k0;
      }
    }
  } else if (warp == 9) {
    // =========================== MMA issuer (leader CTA only) ===========================
    if (rank == 0) {
      uint32_t is_leader;
      asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(is_leader));
      // D=f32, A=B=bf16, K-major both, N = 256, M = 256 (the pair)
      constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      const uint64_t adesc0 = make_smem_desc(smem_base, 16u, 8u * 128u, 2u);                    // SWIZZLE_128B, K-major
      const uint64_t bdesc0 = make_smem_desc(smem_base + (X3 ? 2 : 1) * SK2_A_BYTES, 16u, 8u * 128u, 2u);
      const uint32_t empty0 = smem_u32(&empty_bar[0]), tfull0 = smem_u32(&tmem_full[0]);
      int stage = 0;
      uint32_t phase = 0, seg = 0;
      long long u = u_begin;
      while (u < u_end) {
        const uint32_t tile = (uint32_t)fdiv((uint32_t)u, a.fd_ks_mul, a.fd_ks_shr);
        const int k0 = (int)(u - (long long)tile * a.ksteps);
        const int k1 = (int)min((long long)a.ksteps, k0 + (u_end - u));
        const uint32_t buf = seg & 1u, par = (seg >> 1) & 1u;
        mbar_wait(&tmem_empty[buf], par ^ 1u);                   // both CTAs drained this buffer's previous segment
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + buf * 256u;
        uint32_t accum = 0;
        for (int k = k0; k < k1; ++k) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          if (is_leader) {
            const uint32_t soff = (uint32_t)(stage * SK2_STAGE) >> 4;
            if constexpr (X3) {
              constexpr uint32_t LO = SK2_A_BYTES >> 4;            // the lo block follows the hi block of either operand
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                const uint64_t ah = adesc0 + soff + (uint32_t)(ks * 2), bh = bdesc0 + soff + (uint32_t)(ks * 2);
                umma_bf16_2sm(tmem_d, ah, bh, idesc, accum);        // hi * w_hi
                umma_bf16_2sm(tmem_d, ah + LO, bh, idesc, 1u);      // lo * w_hi
                umma_bf16_2sm(tmem_d, ah, bh + LO, idesc, 1u);      // hi * w_lo
                accum = 1;
              }
            } else {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                umma_bf16_2sm(tmem_d, adesc0 + soff + (uint32_t)(ks * 2), bdesc0 + soff + (uint32_t)(ks * 2), idesc, accum);
                accum = 1;
              }
            }
            umma_commit_2sm_mc(empty0 + 8u * (uint32_t)stage, (uint16_t)3);
          }
          __syncwarp();
          if (++stage == SK2_STAGES) { stage = 0; phase ^= 1u; }
        }
        if (is_leader) umma_commit_2sm_mc(tfull0 + 8u * buf, (uint16_t)3);
        __syncwarp();
        u += k1 - k0;
        ++seg;
      }
    }
  } else {
    // =========================== epilogue (both CTAs, own 128 rows) ===========================
    const int q = warp & 3, chalf = warp >> 2;                 // TMEM lane quarter, column half of the accumulator
    const int et = threadIdx.x;                                // 0..255
    uint32_t seg = 0;
    long long u = u_begin;
    while (u < u_end) {
      const uint32_t tile = (uint32_t)fdiv((uint32_t)u, a.fd_ks_mul, a.fd_ks_shr);
      const int k0 = (int)(u - (long long)tile * a.ksteps);
      const int k1 = (int)min((long long)a.ksteps, k0 + (u_end - u));
      const bool tail = k0 > 0;                                // partial -> workspace slot blockIdx.x
      const bool head = k0 == 0 && k1 < a.ksteps;              // owner: add the partial of CTA blockIdx.x + 2, finalise
      const uint32_t mt = fdiv(tile, a.fd_nt_mul, a.fd_nt_shr);
      const int col0 = (int)(tile - mt * (uint32_t)a.n_tiles) * 256 + chalf * 128;
      const uint32_t buf = seg & 1u, par = (seg >> 1) & 1u;
      if (head) {
        if (et == 0) {
          const int* f = a.ws_flags + blockIdx.x + 2;
          int v;
          long long t0 = clock64();
          do {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
            if (!v) {
              __nanosleep(200);
              if (clock64() - t0 > 6000000000ll) { printf("y2 conv_streamk2: partial of CTA %d never arrived\n", blockIdx.x + 2); __trap(); }
            }
          } while (!v);
          *const_cast<int*>(f) = 0;                             // consumed: the flags are all zero again when the kernel ends
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");          // the 8 epilogue warps
      }
      mbar_wait(&tmem_full[buf], par);
      tc_fence_after();
      const uint32_t stg = smem_base + SK2_STAGES * SK2_STAGE + (uint32_t)warp * SK_STG_WARP;
      float4* part = reinterpret_cast<float4*>(a.ws_partial + (size_t)(tail ? blockIdx.x : blockIdx.x + 2) * 32768) +
                     (size_t)warp * 1024 + lane;                   // + hc * 256 + i * 32
      float4 pv[8];
      if (head) {
#pragma unroll
        for (int i = 0; i < 8; ++i) pv[i] = __ldcg(part + i * 32);
      }
#pragma unroll 1
      for (int hc = 0; hc < NCHUNK; ++hc) {
        const int c = hc * 32;
        const int row0 = (int)rank * 128 + q * 32;                // first tile row of this warp's 32-row slab
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * 256u + (uint32_t)(chalf * 128 + c);
        uint32_t v[32];
        tmem_ld32(taddr, v);
        tmem_ld_wait();
        if (hc == NCHUNK - 1) {                                // my last chunk is in registers
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(smem_u32(&tmem_empty[buf]) & PEER_BIT_MASK);
        }
        if (tail) {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            __stcg(part + hc * 256 + i * 32, make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]),
                                                         __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3])));
          continue;
        }
        float f[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
          if (a.scale) sc = __ldg(reinterpret_cast<const float4*>(a.scale + col0 + c) + i);
          if (a.shift) sh = __ldg(reinterpret_cast<const float4*>(a.shift + col0 + c) + i);
          const float4 p4 = head ? pv[i] : make_float4(0.f, 0.f, 0.f, 0.f);
          f[4 * i + 0] = fmaf(__uint_as_float(v[4 * i + 0]) + p4.x, sc.x, sh.x);
          f[4 * i + 1] = fmaf(__uint_as_float(v[4 * i + 1]) + p4.y, sc.y, sh.y);
          f[4 * i + 2] = fmaf(__uint_as_float(v[4 * i + 2]) + p4.z, sc.z, sh.z);
          f[4 * i + 3] = fmaf(__uint_as_float(v[4 * i + 3]) + p4.w, sc.w, sh.w);
        }
        if (head && hc < NCHUNK - 1) {                         // prefetch the next chunk's partial behind this chunk's stores
#pragma unroll
          for (int i = 0; i < 8; ++i) pv[i] = __ldcg(part + (hc + 1) * 256 + i * 32);
        }
        if (a.leaky) {
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] = fmaxf(f[i], a.alpha * f[i]);
        }
        const long long grow0 = (long long)mt * 256 + row0;       // global row of slab row 0
        if (a.out_f32) {
          // lane = slab row: 8 x 16-byte units, unit j of row r at (j ^ (r & 7))
#pragma unroll
          for (int j = 0; j < 8; ++j)
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(stg + lane * 128 + ((j ^ (lane & 7)) << 4)), "f"(f[4 * j]),
                         "f"(f[4 * j + 1]), "f"(f[4 * j + 2]), "f"(f[4 * j + 3])
                         : "memory");
          __syncwarp();
          float* dst = reinterpret_cast<float*>(a.y) + col0 + c;
#pragma unroll
          for (int t = 0; t < 8; ++t) {
            const int r = t * 4 + (lane >> 3), j = lane & 7;
            float4 o;
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(o.x), "=f"(o.y), "=f"(o.z), "=f"(o.w)
                         : "r"(stg + r * 128 + ((j ^ (r & 7)) << 4)));
            if (grow0 + r < a.M) *reinterpret_cast<float4*>(dst + (size_t)(grow0 + r) * a.ldy + j * 4) = o;
          }
        } else {
          sk_store_chunk_bf16(a, stg, lane, f, col0 + c, grow0);
        }
        __syncwarp();                                           // staging tile free for the next chunk
      }
      if (tail) {
        __threadfence();                                       // my partial is visible device-wide ...
        asm volatile("bar.sync 1, 256;" ::: "memory");          // ... and so is everybody else's
        if (et == 0) {
          int one = 1;
          asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(a.ws_flags + blockIdx.x), "r"(one) : "memory");
        }
      }
      u += k1 - k0;
      ++seg;
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                           // nobody frees TMEM / exits while the partner's MMAs or arrives are in flight
  if (warp == 9) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

static thread_local void* g_sk_ws = nullptr;
static thread_local size_t g_sk_ws_bytes = 0;
constexpr size_t SK_FLAG_BYTES = 4096;

static size_t sk_workspace_bytes(int sms) { return SK_FLAG_BYTES + (size_t)sms * 256 * 256 * sizeof(float); }

// returns Y2_OK and sets *handled = 1 when the layer was issued on this path
int conv_streamk_try(const ConvCall& c, cudaStream_t st, int* handled) {
  *handled = 0;
  if (env().conv_no_streamk || g_sk_ws == nullptr || g_num_sms < 2) return Y2_OK;
  if (c.pool || c.Cin % 64 != 0 || c.Cout % 256 != 0) return Y2_OK;
  if (c.H >= 64 && c.W >= 64) return Y2_OK;                     // large maps: the halo-patch mode of conv_tc_kernel wins
  if (c.ldy % (c.out_f32 ? 4 : 8) != 0 || (reinterpret_cast<uintptr_t>(c.y) & 15) != 0) return Y2_OK;
  if ((c.shift && (reinterpret_cast<uintptr_t>(c.shift) & 15) != 0) || (c.scale && (reinterpret_cast<uintptr_t>(c.scale) & 15) != 0))
    return Y2_OK;
  const bool x3 = c.split_in;                                   // bf16x3: shared-operand stages
  const int cchunks = (x3 ? c.Cin : c.b_cin) / 64, ksteps = c.taps * cchunks;
  if (c.split_out && (c.lo_off & 7) != 0) return Y2_OK;
  const int min_ksteps = x3 ? 6 : 18;                           // short K: the epilogue starts to show (bf16x3 steps are 3x heavier)
  if (ksteps < min_ksteps || ksteps > SK_MAX_UNITS) return Y2_OK;
  SkArgs a;
  memset(&a, 0, sizeof(a));
  a.scale = c.scale;
  a.shift = c.shift;
  a.y = c.y;
  a.alpha = c.alpha;
  a.leaky = c.leaky;
  a.out_f32 = c.out_f32;
  a.M = c.M;
  a.H = c.H; a.W = c.W; a.ldy = c.ldy; a.pad = c.pad;
  a.cin_p = c.b_cin; a.cchunks = cchunks; a.ksteps = ksteps;
  a.split_out = c.split_out ? 1 : 0;
  a.lo_off = c.lo_off;
  fastdiv_init((uint32_t)cchunks, &a.fd_cc_mul, &a.fd_cc_shr);
  a.n_tiles = c.Cout / 256;
  const long long m_tiles = (a.M + 255) / 256;
  a.tiles = (int)(m_tiles * a.n_tiles);
  a.units = (long long)a.tiles * ksteps;
  if ((a.tiles < g_num_sms / 2 && !env().conv_force_streamk) || a.units >= (1ll << 31) || a.M + 256 >= (1ll << 31)) return Y2_OK;
  // 74 pairs, every pair's range at least one tile long (a tile is then shared by at most two pairs)
  const int npairs = a.tiles < g_num_sms / 2 ? a.tiles : g_num_sms / 2;
  if (g_sk_ws_bytes < sk_workspace_bytes(g_num_sms)) return Y2_OK;
  a.ws_flags = reinterpret_cast<int*>(g_sk_ws);
  a.ws_partial = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(g_sk_ws) + SK_FLAG_BYTES);
  fastdiv_init((uint32_t)a.n_tiles, &a.fd_nt_mul, &a.fd_nt_shr);
  fastdiv_init((uint32_t)c.W, &a.fd_w_mul, &a.fd_w_shr);
  fastdiv_init((uint32_t)c.H, &a.fd_h_mul, &a.fd_h_shr);
  fastdiv_init((uint32_t)ksteps, &a.fd_ks_mul, &a.fd_ks_shr);

  static const char* const who = "y2_conv_fwd_bf16 (stream-K)";
  CUtensorMap tmA, tmB;
  int rc = tmap_im2col_nhwc(&tmA, c.x, c.N, c.H, c.W, c.a_cin, c.ksize, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B, who, "A");
  if (rc == Y2_OK)      // each CTA of the pair loads its half of the filters
    rc = tmap_kmajor(&tmB, c.w_packed, c.taps * c.b_cin, c.Cout, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, who, "B");
  if (rc != Y2_OK) return rc;
  // (the flag area was zero when the workspace was registered -- the caller's contract -- and every launch leaves it zero)
  rc = launch_cluster(x3 ? conv_streamk2_kernel<true> : conv_streamk2_kernel<false>, 2 * npairs, SK_THREADS, SK2_SMEM, 2u, st,
                      tmA, tmB, a);
  *handled = rc == Y2_OK;
  return rc;
}

}  // namespace y2

using namespace y2;

extern "C" size_t y2_conv_workspace_bytes(void) {
  if (load_driver_entry_points() != Y2_OK) return 0;
  return sk_workspace_bytes(g_num_sms);
}

extern "C" int y2_conv_set_workspace(void* workspace, size_t bytes) {
  Y2_ARG(workspace == nullptr || (reinterpret_cast<uintptr_t>(workspace) & 255) == 0);
  g_sk_ws = workspace;
  g_sk_ws_bytes = workspace ? bytes : 0;
  return Y2_OK;
}
