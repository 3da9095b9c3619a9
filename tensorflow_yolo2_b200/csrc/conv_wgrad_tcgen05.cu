// conv_wgrad_tcgen05.cu -- a11: weight gradient of the SAME stride-1 convolution (what TF autodiff's
// Conv2DBackpropFilter computes for yolo2_nets/darknet.py:20-21) on the sm_100a tensor cores.
//
//   dW[kh][kw][ci][co] = sum over pixels (n,h,w) of  x[n, h+kh-p, w+kw-p, ci] * dh[n, h, w, co]
//
// GEMM view: D[M = (tap, ci), N = co] = A[K = pixels, M]^T * B[K = pixels, N].  Both operands are consumed
// *MN-major* straight from the NHWC tensors: a pixel's channel chunk is one 128-byte (or 64-byte) smem row, i.e.
// exactly what a TMA box {channels, pixels} with the matching swizzle writes, and the pixel index is the K
// dimension (UMMA instruction descriptor a_major = b_major = MN).  No transposed copy of the activations exists.
//
//   A tile  128 M-rows = `slots` swizzle atoms, each one (filter tap, channel chunk) pair fetched by its own
//           im2col-mode TMA load of KP pixels (the tap shift and the zero halo are done by the TMA unit);
//           for Cin = 64 / 32 two / four taps share one MMA so that M is always 128.
//   B tile  BLOCK_N/64 atoms of dh [pixels, 64 channels], plain 2-D TMA.
//   K loop  KP = 64 pixels per pipeline stage = 4 tcgen05.mma (K = 16); split-K over CTAs: every (m_tile, n_tile,
//           k_split) unit accumulates in TMEM (double-buffered) and is reduced into dW with red.global.add.f32.
//   roles   warps 0-3 epilogue (tcgen05.ld -> vector red), warp 4 TMA producer, warp 5 MMA issuer; persistent grid.
// The caller zeroes dW (the trainer clears its whole gradient arena once per step).
#include "tc_common.cuh"

namespace y2 {

struct WgradArgs {
  float* dw;
  int Cin, Cout, ksize, pad;
  int N, H, W;
  long long M;
  int atom_ch, slots, cchunks, total_slots;
  int m_tiles, n_tiles, n_atoms;
  int kp, kstages, splits, stages;
  uint32_t a_stage_bytes, b_stage_bytes;
  uint32_t fd_w_mul, fd_w_shr, fd_h_mul, fd_h_shr, fd_cch_mul, fd_cch_shr, fd_k_mul, fd_k_shr;
  uint32_t fd_nt_mul, fd_nt_shr, fd_mt_mul, fd_mt_shr;
};

constexpr int WG_THREADS = 6 * 32;
constexpr int WG_WARP_PRODUCER = 4, WG_WARP_MMA = 5;
constexpr int WG_MAX_STAGES = 8;

__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// G: M tiles per scheduling unit that share ONE pass over the dh columns (G accumulators of BLOCK_N columns per TMEM buffer).
// The early layers have few output rows (taps x Cin = 288 .. 1152) and millions of pixels: with one M tile per unit the
// activations are fetched once per tap group and dh once per M tile -- 2.6 GB of DRAM traffic for layer 2's 0.5 GB of operands
// (x and dh no longer fit the L2), which made those layers HBM-bound at 250-500 TFLOP/s.  With G tiles per unit a K stage
// loads dh once and the G tiles' (spatially overlapping) taps of the same pixels together.
template <int BLOCK_N, int ATOM_BYTES, int G = 1>
__global__ void __launch_bounds__(WG_THREADS, 1)
conv_wgrad_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmG, const WgradArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  constexpr int NBUF = 2;
  static_assert(NBUF * G * BLOCK_N <= 512, "TMEM has 512 columns");
  constexpr uint32_t TMEM_COLS = NBUF * G * BLOCK_N <= 128 ? 128 : (NBUF * G * BLOCK_N <= 256 ? 256 : 512);
  __shared__ __align__(8) uint64_t full_bar[WG_MAX_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[WG_MAX_STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar[NBUF];
  __shared__ __align__(8) uint64_t tmem_empty_bar[NBUF];
  __shared__ uint32_t s_tmem_base;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem) + 1023u) & ~1023u;
  const uint32_t stage_bytes = a.a_stage_bytes + a.b_stage_bytes;
  const int m_groups = (a.m_tiles + G - 1) / G;                            // scheduling units along M (G tiles each)
  const int total_units = m_groups * a.n_tiles * a.splits;
  const int unit0 = (int)blockIdx.x, unit_step = (int)gridDim.x;

  if (warp == WG_WARP_PRODUCER && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmX)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmG)) : "memory");
    for (int s = 0; s < a.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int b = 0; b < NBUF; ++b) { mbar_init(&tmem_full_bar[b], 1); mbar_init(&tmem_empty_bar[b], 4); }
    fence_barrier_init();
  }
  if (warp == WG_WARP_MMA) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem_base)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;

  if (warp == WG_WARP_PRODUCER) {
    // =========================== TMA producer ===========================
    int stage = 0;
    uint32_t phase = 0;
    for (int unit = unit0; unit < total_units; unit += unit_step) {
      const uint32_t q1 = fdiv((uint32_t)unit, a.fd_nt_mul, a.fd_nt_shr);
      const int nt = unit - (int)q1 * a.n_tiles;
      const uint32_t sp = fdiv(q1, a.fd_mt_mul, a.fd_mt_shr);
      const int mt = ((int)q1 - (int)sp * m_groups) * G;                                 // first M tile of the unit
      const int ks0 = (int)(((long long)sp * a.kstages) / a.splits), ks1 = (int)(((long long)(sp + 1) * a.kstages) / a.splits);
      // my load: lanes [0, G * slots) fetch A atoms (tile mt + lane / slots), the next n_atoms lanes fetch B atoms
      const int a_lanes = G * a.slots;
      int kw = 0, kh = 0, c0 = 0;
      if (lane < a_lanes) {
        int gs = mt * a.slots + lane;
        if (gs >= a.total_slots) gs = a.total_slots - 1;      // padding slot: any finite data, discarded by the epilogue
        const int tap = (int)fdiv((uint32_t)gs, a.fd_cch_mul, a.fd_cch_shr);
        c0 = (gs - tap * a.cchunks) * a.atom_ch;
        kh = (int)fdiv((uint32_t)tap, a.fd_k_mul, a.fd_k_shr);
        kw = tap - kh * a.ksize;
      } else {
        c0 = nt * BLOCK_N + (lane - a_lanes) * 64;
      }
      for (int ks = ks0; ks < ks1; ++ks) {
        if (lane == 0) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          mbar_expect_tx(&full_bar[stage], stage_bytes);
        }
        __syncwarp();
        const uint32_t p0 = (uint32_t)ks * (uint32_t)a.kp;
        const uint32_t sA = smem_base + stage * stage_bytes;
        const uint32_t bar = smem_u32(&full_bar[stage]);
        if (lane < a_lanes) {
          const uint32_t row = fdiv(p0, a.fd_w_mul, a.fd_w_shr);          // n*H + h
          const int w0 = (int)(p0 - row * (uint32_t)a.W);
          const uint32_t img = fdiv(row, a.fd_h_mul, a.fd_h_shr);
          const int h0 = (int)(row - img * (uint32_t)a.H);
          tma_load_im2col_4d(sA + lane * (a.kp * ATOM_BYTES), &tmX, bar, c0, w0 - a.pad, h0 - a.pad, (int)img, (uint16_t)kw,
                             (uint16_t)kh);
        } else if (lane < a_lanes + a.n_atoms) {
          tma_load_2d(sA + a.a_stage_bytes + (lane - a_lanes) * (a.kp * 128), &tmG, bar, c0, (int)p0);
        }
        __syncwarp();
        if (++stage == a.stages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == WG_WARP_MMA) {
    // =========================== MMA issuer ===========================
    uint32_t is_leader;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(is_leader));
    // D = f32, A = B = bf16, both MN-major (bits 15, 16), N, M = 128
    constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                               ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    constexpr uint32_t a_layout = ATOM_BYTES == 128 ? 2u : 4u;
    // MN-major canonical layout: LBO = byte distance between swizzle atoms along M/N, SBO = between 8-pixel groups
    const uint64_t adesc0 = make_smem_desc(smem_base, (uint32_t)(a.kp * ATOM_BYTES), 8u * ATOM_BYTES, a_layout);
    const uint64_t bdesc0 = make_smem_desc(smem_base + a.a_stage_bytes, (uint32_t)(a.kp * 128), 1024u, 2u);
    constexpr uint32_t a_kstep = (16u * ATOM_BYTES) >> 4, b_kstep = (16u * 128u) >> 4;     // 16 pixels per MMA
    const uint32_t stage16 = stage_bytes >> 4;
    const int ksteps = a.kp >> 4;
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int unit = unit0; unit < total_units; unit += unit_step, ++it) {
      const uint32_t q1 = fdiv((uint32_t)unit, a.fd_nt_mul, a.fd_nt_shr);
      const uint32_t sp = fdiv(q1, a.fd_mt_mul, a.fd_mt_shr);
      const int ks0 = (int)(((long long)sp * a.kstages) / a.splits), ks1 = (int)(((long long)(sp + 1) * a.kstages) / a.splits);
      const int buf = it & 1;
      mbar_wait(&tmem_empty_bar[buf], (((uint32_t)it >> 1) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + (uint32_t)(buf * G * BLOCK_N);
      const uint32_t a_tile16 = (uint32_t)(a.slots * a.kp * ATOM_BYTES) >> 4;          // one M tile's atoms within the stage
      uint32_t accum = 0;
      for (int ks = ks0; ks < ks1; ++ks) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (is_leader) {
          const uint64_t ad = adesc0 + (uint32_t)stage * stage16, bd = bdesc0 + (uint32_t)stage * stage16;
          for (int k = 0; k < ksteps; ++k) {
#pragma unroll
            for (int gi = 0; gi < G; ++gi)
              umma_bf16(tmem_d + (uint32_t)(gi * BLOCK_N), ad + (uint32_t)gi * a_tile16 + (uint32_t)k * a_kstep,
                        bd + (uint32_t)k * b_kstep, idesc, accum);
            accum = 1;
          }
          umma_commit(&empty_bar[stage]);
        }
        __syncwarp();
        if (++stage == a.stages) { stage = 0; phase ^= 1u; }
      }
      if (is_leader) umma_commit(&tmem_full_bar[buf]);
      __syncwarp();
    }
  } else {
    // =========================== epilogue: TMEM -> dW (+=) ===========================
    const int r = warp * 32 + lane;                     // accumulator row = (slot, channel)
    const int slot = r / a.atom_ch, ch = r - slot * a.atom_ch;
    const bool vec_ok = (a.Cout & 3) == 0 && ((reinterpret_cast<uintptr_t>(a.dw) & 15) == 0);
    int it = 0;
    for (int unit = unit0; unit < total_units; unit += unit_step, ++it) {
      const uint32_t q1 = fdiv((uint32_t)unit, a.fd_nt_mul, a.fd_nt_shr);
      const int nt = unit - (int)q1 * a.n_tiles;
      const uint32_t sp = fdiv(q1, a.fd_mt_mul, a.fd_mt_shr);
      const int mt0 = ((int)q1 - (int)sp * m_groups) * G;
      const int buf = it & 1;
      mbar_wait(&tmem_full_bar[buf], ((uint32_t)it >> 1) & 1u);
      tc_fence_after();
#pragma unroll 1
      for (int gi = 0; gi < G; ++gi) {
      const int mt = mt0 + gi;
      const int gs = mt * a.slots + slot;
      const int tap = (int)fdiv((uint32_t)gs, a.fd_cch_mul, a.fd_cch_shr);
      const int ci = (gs - tap * a.cchunks) * a.atom_ch + ch;
      const bool valid = gs < a.total_slots && ci < a.Cin;
      float* const row = a.dw + ((size_t)tap * a.Cin + ci) * a.Cout;
      const uint32_t taddr0 = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * G * BLOCK_N + gi * BLOCK_N);
#pragma unroll 1
      for (int cc = 0; cc < BLOCK_N; cc += 32) {
        uint32_t v[32];
        tmem_ld32(taddr0 + (uint32_t)cc, v);
        tmem_ld_wait();
        if (cc + 32 >= BLOCK_N && gi == G - 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty_bar[buf]);
        }
        const int col0 = nt * BLOCK_N + cc;
        if (valid && col0 < a.Cout) {
          if (vec_ok && col0 + 32 <= a.Cout) {
#pragma unroll
            for (int i = 0; i < 32; i += 4)
              red_add_v4(row + col0 + i, __uint_as_float(v[i]), __uint_as_float(v[i + 1]), __uint_as_float(v[i + 2]),
                         __uint_as_float(v[i + 3]));
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (col0 + i < a.Cout) atomicAdd(row + col0 + i, __uint_as_float(v[i]));
          }
        }
        __syncwarp();
      }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == WG_WARP_MMA) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

template <int BLOCK_N, int ATOM_BYTES>
static int launch_wgrad(const CUtensorMap& tmX, const CUtensorMap& tmG, const WgradArgs& a, size_t smem, cudaStream_t st, int group) {
  if constexpr (BLOCK_N <= 128) {
    constexpr int GG = BLOCK_N == 64 ? 3 : 2;
    if (group == GG) {
      Y2_CUDA(cudaFuncSetAttribute((conv_wgrad_tc_kernel<BLOCK_N, ATOM_BYTES, GG>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)smem));
      const int units = ((a.m_tiles + GG - 1) / GG) * a.n_tiles * a.splits;
      const int grid = units < g_num_sms ? units : g_num_sms;
      conv_wgrad_tc_kernel<BLOCK_N, ATOM_BYTES, GG><<<grid, WG_THREADS, smem, st>>>(tmX, tmG, a);
      Y2_LAUNCHED();
      return Y2_OK;
    }
  }
  Y2_CUDA(cudaFuncSetAttribute(conv_wgrad_tc_kernel<BLOCK_N, ATOM_BYTES>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)smem));
  const int units = a.m_tiles * a.n_tiles * a.splits;
  const int grid = units < g_num_sms ? units : g_num_sms;
  conv_wgrad_tc_kernel<BLOCK_N, ATOM_BYTES><<<grid, WG_THREADS, smem, st>>>(tmX, tmG, a);
  Y2_LAUNCHED();
  return Y2_OK;
}

}  // namespace y2

using namespace y2;

extern "C" int y2_conv_wgrad_bf16(const void* x, const void* dh, int ld_dh, float* dw, int N, int H, int W, int Cin,
                                  int Cout, int ksize, y2_stream_t stream) {
  Y2_ARG(x && dh && dw && N > 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0 && (ksize == 1 || ksize == 3));
  Y2_ARG(ld_dh >= Cout && ld_dh % 64 == 0);
  if (Cin % 32 != 0) {
    set_error("y2_conv_wgrad_bf16: Cin=%d unsupported (multiples of 32; the Cin=3 first layer uses y2_conv_wgrad_c3)", Cin);
    return Y2_ERR_UNSUPPORTED;
  }
  int rc = load_driver_entry_points();
  if (rc != Y2_OK) return rc;
  WgradArgs a;
  memset(&a, 0, sizeof(a));
  a.dw = dw;
  a.Cin = Cin; a.Cout = Cout; a.ksize = ksize; a.pad = ksize / 2;
  a.N = N; a.H = H; a.W = W;
  a.M = (long long)N * H * W;
  Y2_ARG(a.M + 64 < (1ll << 31));
  const int atom_bytes = (Cin % 64 == 0) ? 128 : 64;
  a.atom_ch = atom_bytes / 2;
  a.slots = 128 / a.atom_ch;
  a.cchunks = Cin / a.atom_ch;
  a.total_slots = ksize * ksize * a.cchunks;
  a.m_tiles = (a.total_slots + a.slots - 1) / a.slots;
  const int block_n = ld_dh >= 256 ? 256 : (ld_dh >= 128 ? 128 : 64);
  a.n_tiles = (ld_dh + block_n - 1) / block_n;
  a.n_atoms = block_n / 64;
  a.kp = 64;
  a.kstages = (int)((a.M + a.kp - 1) / a.kp);
  // tile groups for the narrow layers (block_n 64: three M tiles per unit, 128: two) with many pixels per output row
  int group = 1;
  if (ksize == 3 && a.m_tiles >= 2 && a.M >= 2048) group      // (1x1 layers: measured slower)
    = block_n == 64 ? 3 : (block_n == 128 ? 2 : 1);
  a.a_stage_bytes = (uint32_t)(group * a.slots * a.kp * atom_bytes);
  a.b_stage_bytes = (uint32_t)(a.n_atoms * a.kp * 128);
  const size_t SMEM_BUDGET = 200 * 1024;
  int stages = (int)(SMEM_BUDGET / (a.a_stage_bytes + a.b_stage_bytes));
  if (stages > WG_MAX_STAGES) stages = WG_MAX_STAGES;
  a.stages = stages;
  const size_t smem = (size_t)stages * (a.a_stage_bytes + a.b_stage_bytes) + 1024;
  // split-K: enough units to fill the machine ~3 times unless the tiles alone already do
  const int tiles = ((a.m_tiles + group - 1) / group) * a.n_tiles;   // scheduling units before the K split
  int splits = 1;
  if (tiles < g_num_sms * 3 / 2) splits = (g_num_sms * 3 + tiles - 1) / tiles;
  int max_splits = a.kstages / 8;
  if (max_splits < 1) max_splits = 1;
  if (splits > max_splits) splits = max_splits;
  a.splits = splits;
  fastdiv_init((uint32_t)W, &a.fd_w_mul, &a.fd_w_shr);
  fastdiv_init((uint32_t)H, &a.fd_h_mul, &a.fd_h_shr);
  fastdiv_init((uint32_t)a.cchunks, &a.fd_cch_mul, &a.fd_cch_shr);
  fastdiv_init((uint32_t)ksize, &a.fd_k_mul, &a.fd_k_shr);
  fastdiv_init((uint32_t)a.n_tiles, &a.fd_nt_mul, &a.fd_nt_shr);
  fastdiv_init((uint32_t)((a.m_tiles + group - 1) / group), &a.fd_mt_mul, &a.fd_mt_shr);

  CUtensorMap tmX, tmG;
  rc = tmap_im2col_nhwc(&tmX, x, N, H, W, Cin, ksize, a.atom_ch, a.kp, swizzle_for(atom_bytes), "y2_conv_wgrad_bf16", "X");
  if (rc == Y2_OK)
    rc = tmap_kmajor(&tmG, dh, ld_dh, a.M, 64, a.kp, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     "y2_conv_wgrad_bf16", "dh");
  if (rc != Y2_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (atom_bytes == 128) {
    switch (block_n) {
      case 64: return launch_wgrad<64, 128>(tmX, tmG, a, smem, st, group);
      case 128: return launch_wgrad<128, 128>(tmX, tmG, a, smem, st, group);
      default: return launch_wgrad<256, 128>(tmX, tmG, a, smem, st, group);
    }
  }
  switch (block_n) {
    case 64: return launch_wgrad<64, 64>(tmX, tmG, a, smem, st, group);
    case 128: return launch_wgrad<128, 64>(tmX, tmG, a, smem, st, group);
    default: return launch_wgrad<256, 64>(tmX, tmG, a, smem, st, group);
  }
}
