// elementwise.cu -- HBM-bound helpers around the convolutions: input preprocessing (a10),
// weight packing, batch-norm statistics / folding / apply (+leaky, +2x2 pool) (a2, a3), Adam (a11).
// Reference call sites are cited per kernel; the ABI is documented in include/yolo2_b200.h.
#include "common.cuh"

namespace y2 {

// ---------------------------------------------------------------------------------------------
// a10  pascal_detect_darknet.py:36-37 / pascal_voc.py:62-64:  (u8 / 255.0) * 2.0 - 1.0
// Division and multiply kept as separate IEEE ops so the f32 output is bit-identical to NumPy's.
// ---------------------------------------------------------------------------------------------
__global__ void preprocess_u8_f32_kernel(const uint8_t* __restrict__ img, float* __restrict__ out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float v = (float)img[i];
    out[i] = __fsub_rn(__fmul_rn(__fdiv_rn(v, 255.0f), 2.0f), 1.0f);
  }
}

// one thread per pixel: 3 bytes in, 8 bf16 (16 B) out; channels 3..7 are zero padding so the
// first conv can run on the tensor cores with 16-byte TMA rows.
__global__ void preprocess_u8_bf16c8_kernel(const uint8_t* __restrict__ img, uint4* __restrict__ out, size_t npix) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < npix; i += stride) {
    float v0 = (float)img[3 * i + 0], v1 = (float)img[3 * i + 1], v2 = (float)img[3 * i + 2];
    v0 = __fsub_rn(__fmul_rn(__fdiv_rn(v0, 255.0f), 2.0f), 1.0f);
    v1 = __fsub_rn(__fmul_rn(__fdiv_rn(v1, 255.0f), 2.0f), 1.0f);
    v2 = __fsub_rn(__fmul_rn(__fdiv_rn(v2, 255.0f), 2.0f), 1.0f);
    __nv_bfloat162 a = __floats2bfloat162_rn(v0, v1);
    __nv_bfloat162 b = __floats2bfloat162_rn(v2, 0.0f);
    uint4 o;
    o.x = *reinterpret_cast<uint32_t*>(&a);
    o.y = *reinterpret_cast<uint32_t*>(&b);
    o.z = 0u;
    o.w = 0u;
    out[i] = o;
  }
}

__global__ void pad_cast_f32_bf16c8_kernel(const float* __restrict__ x, uint4* __restrict__ out, size_t npix) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < npix; i += stride) {
    __nv_bfloat162 a = __floats2bfloat162_rn(x[3 * i + 0], x[3 * i + 1]);
    __nv_bfloat162 b = __floats2bfloat162_rn(x[3 * i + 2], 0.0f);
    uint4 o;
    o.x = *reinterpret_cast<uint32_t*>(&a);
    o.y = *reinterpret_cast<uint32_t*>(&b);
    o.z = 0u;
    o.w = 0u;
    out[i] = o;
  }
}

// ---------------------------------------------------------------------------------------------
// a10  cv2.resize(image, (IS, IS)) -- pascal_detect_darknet.py:35, img_dataset/pascal_voc.py:61 -- for 8-bit BGR images, default
// interpolation (INTER_LINEAR).  OpenCV (opencv-python 4.13.0 in this image; the algorithm is unchanged since 2.x) computes it
// in fixed point, which makes a bit-exact GPU restatement possible:
//   * per output column: fx = (float)((dx + 0.5) * scale_x - 0.5) (double product), sx = floor(fx), fx -= sx; at the borders
//     (sx < 0 or sx >= W - 1) sx is clamped and fx = 0; coefficients a0 = rint((1 - fx) * 2048), a1 = rint(fx * 2048) as shorts;
//   * per output row: the same WITHOUT zeroing fy at the borders -- the two source ROWS are clamped instead;
//   * horizontal pass in int32: R = S[sx] * a0 + S[sx + 1] * a1; vertical: ((b0 * (R0 >> 4)) >> 16) + ((b1 * (R1 >> 4)) >> 16),
//     then (+ 2) >> 2;
//   * an exact 2x down-scale in both directions is switched to INTER_AREA: (sum of the 2x2 block + 2) >> 2.
// One thread per output pixel (3 channels).  scale_x / scale_y arrive as doubles computed like OpenCV does: 1.0 / (dst / src).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void resize_coef(int d, double scale, int sn, bool clamp, int& s0, int& c0, int& c1) {
  float f = (float)__dadd_rn(__dmul_rn((double)d + 0.5, scale), -0.5);      // (no FMA contraction: two roundings, like the host code)
  s0 = (int)floorf(f);
  f -= (float)s0;
  if (clamp) {
    if (s0 < 0) { f = 0.0f; s0 = 0; }
    if (s0 >= sn - 1) { f = 0.0f; s0 = sn - 1; }
  }
  c0 = __float2int_rn(__fmul_rn(__fsub_rn(1.0f, f), 2048.0f));
  c1 = __float2int_rn(__fmul_rn(f, 2048.0f));
}

__global__ void resize_bilinear_u8c3_kernel(const uint8_t* __restrict__ src, int sh, int sw, size_t src_pitch, uint8_t* __restrict__ dst,
                                            int dh, int dw, double scale_x, double scale_y, int area2) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= dw || y >= dh) return;
  uint8_t* o = dst + ((size_t)y * dw + x) * 3;
  if (area2) {
    const uint8_t* p0 = src + (size_t)(2 * y) * src_pitch + (size_t)(2 * x) * 3;
    const uint8_t* p1 = p0 + src_pitch;
#pragma unroll
    for (int c = 0; c < 3; ++c) o[c] = (uint8_t)(((int)p0[c] + (int)p0[3 + c] + (int)p1[c] + (int)p1[3 + c] + 2) >> 2);
    return;
  }
  int sx, a0, a1, sy, b0, b1;
  resize_coef(x, scale_x, sw, true, sx, a0, a1);
  resize_coef(y, scale_y, sh, false, sy, b0, b1);
  const int x1 = min(sx + 1, sw - 1);
  const int y0 = min(max(sy, 0), sh - 1), y1 = min(max(sy + 1, 0), sh - 1);
  const uint8_t* r0 = src + (size_t)y0 * src_pitch;
  const uint8_t* r1 = src + (size_t)y1 * src_pitch;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int R0 = (int)r0[sx * 3 + c] * a0 + (int)r0[x1 * 3 + c] * a1;
    const int R1 = (int)r1[sx * 3 + c] * a0 + (int)r1[x1 * 3 + c] * a1;
    const int v = (((b0 * (R0 >> 4)) >> 16) + ((b1 * (R1 >> 4)) >> 16) + 2) >> 2;
    o[c] = (uint8_t)min(max(v, 0), 255);
  }
}

// ---------------------------------------------------------------------------------------------
// weight packing: TF HWIO [k,k,Cin,Cout] f32  ->  [Cout_p][Kp] bf16, K index = tap*Cin_p + c
// (K-major rows, the B operand of the implicit GEMM).  Padding rows/columns are zero.
// First layer (Cin 3 -> 8): [10 k-groups][Cout_p][8] instead: taps 0..7, a zero group, tap 8.
// ---------------------------------------------------------------------------------------------
__global__ void pack_weights_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int taps, int Cin,
                                    int Cout, int Cin_p, int Cout_p, int Kp) {
  size_t total = (size_t)Cout_p * Kp;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    int n = (int)(i / Kp);
    int kk = (int)(i % Kp);
    int grp = kk / Cin_p, c = kk % Cin_p;
    // first layer (Cin_p == 8): k-groups are taps 0..7, one all-zero group, then tap 8 (conv_tcgen05.cu pairs the
    // zero group with tap 8 in the last K=16 MMA)
    int tap = (Cin_p == 8) ? (grp < 8 ? grp : (grp == 9 ? 8 : taps)) : grp;
    float v = 0.0f;
    if (n < Cout && tap < taps && c < Cin) v = w[((size_t)tap * Cin + c) * Cout + n];
    // first layer: smem-ready order [k-group][Cout_p][8] (un-swizzled core matrices)
    size_t o = (Cin_p == 8) ? ((size_t)grp * Cout_p + n) * 8 + c : i;
    out[o] = __float2bfloat16_rn(v);
  }
}

// Same packing through a 32 x 32 shared-memory transpose (Cin_p a multiple of 32): the kernel above reads w with a stride of
// Cout floats between consecutive threads (one 32-byte sector per element -- 0.25 ms per training step for the 48 M
// weights); here both the HWIO reads (along Cout) and the K-major writes (along Cin) are coalesced.
// grid (Cout_p / 32 rounded up, Cin_p / 32, taps), block (32, 8).
__global__ void __launch_bounds__(256) pack_weights_tiled_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int Cin,
                                                                int Cout, int Cin_p, int Cout_p, int Kp) {
  __shared__ float t[32][33];
  const int n0 = blockIdx.x * 32, c0 = blockIdx.y * 32, tap = blockIdx.z;
  const int tx = threadIdx.x, ty = threadIdx.y;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = c0 + ty + 8 * j, n = n0 + tx;
    t[ty + 8 * j][tx] = (c < Cin && n < Cout) ? w[((size_t)tap * Cin + c) * Cout + n] : 0.0f;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int n = n0 + ty + 8 * j, c = c0 + tx;
    if (n < Cout_p && c < Cin_p) out[(size_t)n * Kp + (size_t)tap * Cin_p + c] = __float2bfloat16_rn(t[tx][ty + 8 * j]);
  }
}

// "bf16x3" operand (Y2_CONV_IN_SPLIT): [Cout_p][taps][3*Cin] with per tap [w_hi | w_hi | w_lo], w_hi = bf16(w),
// w_lo = bf16(w - w_hi).  The activation side supplies [a_hi | a_lo | a_hi], so one K sweep accumulates
// a_hi*w_hi + a_lo*w_hi + a_hi*w_lo.
__global__ void pack_weights_split_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int taps, int Cin,
                                          int Cout, int Cout_p) {
  const int K3 = 3 * Cin;
  size_t total = (size_t)Cout_p * taps * K3;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    int n = (int)(i / ((size_t)taps * K3));
    int kk = (int)(i % ((size_t)taps * K3));
    int tap = kk / K3, j = kk % K3;
    int part = j / Cin, c = j - part * Cin;
    float v = 0.0f;
    if (n < Cout) {
      const float wv = w[((size_t)tap * Cin + c) * Cout + n];
      const __nv_bfloat16 hi = __float2bfloat16_rn(wv);
      v = part < 2 ? __bfloat162float(hi) : wv - __bfloat162float(hi);
    }
    out[i] = __float2bfloat16_rn(v);
  }
}

// ---------------------------------------------------------------------------------------------
// a2  batch statistics (tf.layers.batch_normalization training=True, darknet.py:42-44):
// per-channel mean and biased variance over M rows.  Shifted sums in float64: with the
// reference's initialiser activations reach 1e9..1e12 and |mean| >> std, where a float32
// E[x^2]-E[x]^2 cancels catastrophically.
// stage 1: grid (ceil(C/32), splits), block (32, 8): partial sum(d), sum(d^2), d = x - x[0][c]
// stage 2: one thread per channel folds the splits in a fixed order (deterministic).
// ---------------------------------------------------------------------------------------------
__global__ void bn_stats_partial_kernel(const float* __restrict__ x, int M, int C, int ld, int rows_per_split,
                                        double* __restrict__ part) {
  __shared__ double s1[8][33], s2[8][33];
  int c = blockIdx.x * 32 + threadIdx.x;
  int split = blockIdx.y;
  int r0 = split * rows_per_split;
  int r1 = min(M, r0 + rows_per_split);
  double a1 = 0.0, a2 = 0.0;
  if (c < C) {
    float k = x[c];
    for (int r = r0 + threadIdx.y; r < r1; r += 8) {
      double d = (double)(x[(size_t)r * ld + c] - k);
      a1 += d;
      a2 += d * d;
    }
  }
  s1[threadIdx.y][threadIdx.x] = a1;
  s2[threadIdx.y][threadIdx.x] = a2;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    for (int y = 1; y < 8; ++y) {
      a1 += s1[y][threadIdx.x];
      a2 += s2[y][threadIdx.x];
    }
    part[((size_t)split * C + c) * 2 + 0] = a1;
    part[((size_t)split * C + c) * 2 + 1] = a2;
  }
}

// Vectorised variant (C % 4 == 0): a thread owns 4 consecutive channels (16-byte loads) and keeps four rows in
// flight; block = TX channel groups x (256/TX) row lanes, so narrow layers (C = 32) still fill 256 threads.
template <int TX, int UNR>
__global__ void __launch_bounds__(256) bn_stats_partial_v4_kernel(const float* __restrict__ x, int M, int C, int ld,
                                                                  int rows_per_split, double* __restrict__ part, int stream_loads) {
  constexpr int TY = 256 / TX;
  __shared__ double sm[TY][TX][8];
  const int tx = threadIdx.x % TX, ty = threadIdx.x / TX;
  const int c0 = (blockIdx.x * TX + tx) * 4;
  // Row tiles of 4*TY rows are dealt to the splits ROUND-ROBIN (split y takes tiles y, y + splits, ...), not as one contiguous
  // range per split: all resident blocks then stream through the same few hundred KB at any moment (DRAM pages stay open)
  // instead of 1024 far-apart streams -- the contiguous version reached 3.9 TB/s of 6.5 (ncu r2n).  Still a fixed assignment:
  // the result does not depend on scheduling.
  (void)rows_per_split;
  const int r1 = M;
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (c0 < C) {
    const float4 k = *reinterpret_cast<const float4*>(x + c0);
    float f[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int cnt = 0;
    // (eight rows in flight instead of four was tried: 17 -> 20 us per head layer under ncu, no gain live)
    for (int rb = blockIdx.y * UNR * TY + ty; rb < r1; rb += gridDim.y * UNR * TY) {
      float4 v[UNR];
#pragma unroll
      for (int j = 0; j < UNR; ++j) {
        const int r = rb + j * TY;
        // default caching when the rows fit in L2 (the affine pass re-reads them), streaming (evict-first) loads otherwise
        const float4* px = reinterpret_cast<const float4*>(x + (size_t)r * ld + c0);
        v[j] = r < r1 ? (stream_loads ? __ldcs(px) : __ldg(px)) : k;
      }
#pragma unroll
      for (int j = 0; j < UNR; ++j) {
        const float d0 = v[j].x - k.x, d1 = v[j].y - k.y, d2 = v[j].z - k.z, d3 = v[j].w - k.w;
        f[0] += d0; f[1] += d1; f[2] += d2; f[3] += d3;
        f[4] = fmaf(d0, d0, f[4]); f[5] = fmaf(d1, d1, f[5]); f[6] = fmaf(d2, d2, f[6]); f[7] = fmaf(d3, d3, f[7]);
      }
      if (++cnt == 32 / UNR) {
#pragma unroll
        for (int i = 0; i < 8; ++i) { acc[i] += (double)f[i]; f[i] = 0.0f; }
        cnt = 0;
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] += (double)f[i];
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) sm[ty][tx][i] = acc[i];
  __syncthreads();
  // fold the TY row lanes: thread (tx, i = ty < 8) handles one of the 8 sums
  if (ty < 8 && c0 < C) {
    double a = 0.0;
    for (int y = 0; y < TY; ++y) a += sm[y][tx][ty];
    const int c = c0 + (ty & 3);
    part[((size_t)blockIdx.y * C + c) * 2 + (ty >> 2)] = a;
  }
}

// grid ceil(C/32), block (32, FIN_TY): the thread rows fold interleaved subsets of the splits (fixed order ->
// deterministic), then one row folds the FIN_TY partials.  32 rows: with 8 each thread walked ~11 dependent L2 round
// trips (8 us for 1.4 MB, ncu r1c).
constexpr int FIN_TY = 32;
// With gamma / beta the same thread also writes the folded affine of the CENTRED form y = (x - mean) * scale + shift
// (scale = gamma * rsqrt(var + eps), shift = beta) -- one launch less per batch-statistics layer.
__global__ void __launch_bounds__(32 * FIN_TY) bn_stats_final_kernel(const float* __restrict__ x, const double* __restrict__ part, int splits, int M,
                                      int C, float* __restrict__ mean, float* __restrict__ var,
                                      const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                      float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ mm,
                                      float* __restrict__ mv, float momentum) {
  __shared__ double s1[FIN_TY][33], s2[FIN_TY][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  double a1 = 0.0, a2 = 0.0;
  if (c < C) {
    // four independent loads in flight per thread (the single-accumulator loop walked up to 19 dependent L2 round trips);
    // the summation order is fixed, so the result stays deterministic
    double b1 = 0.0, b2 = 0.0, c1 = 0.0, c2 = 0.0, d1 = 0.0, d2 = 0.0;
    int s = threadIdx.y;
    for (; s + 3 * FIN_TY < splits; s += 4 * FIN_TY) {
      const double2 p0 = *reinterpret_cast<const double2*>(part + ((size_t)s * C + c) * 2);
      const double2 p1 = *reinterpret_cast<const double2*>(part + ((size_t)(s + FIN_TY) * C + c) * 2);
      const double2 p2 = *reinterpret_cast<const double2*>(part + ((size_t)(s + 2 * FIN_TY) * C + c) * 2);
      const double2 p3 = *reinterpret_cast<const double2*>(part + ((size_t)(s + 3 * FIN_TY) * C + c) * 2);
      a1 += p0.x; a2 += p0.y; b1 += p1.x; b2 += p1.y; c1 += p2.x; c2 += p2.y; d1 += p3.x; d2 += p3.y;
    }
    for (; s < splits; s += FIN_TY) {
      const double2 p = *reinterpret_cast<const double2*>(part + ((size_t)s * C + c) * 2);
      a1 += p.x;
      a2 += p.y;
    }
    a1 = (a1 + b1) + (c1 + d1);
    a2 = (a2 + b2) + (c2 + d2);
  }
  s1[threadIdx.y][threadIdx.x] = a1;
  s2[threadIdx.y][threadIdx.x] = a2;
  __syncthreads();
  if (threadIdx.y != 0 || c >= C) return;
  for (int y = 1; y < FIN_TY; ++y) { a1 += s1[y][threadIdx.x]; a2 += s2[y][threadIdx.x]; }
  double md = a1 / (double)M;
  double v = a2 / (double)M - md * md;
  if (v < 0.0) v = 0.0;
  mean[c] = (float)((double)x[c] + md);
  const float vf = (float)v;
  var[c] = vf;
  if (scale) {
    scale[c] = gamma[c] * rsqrtf(vf + eps);                    // bit-identical to bn_fold_kernel on (mean = 0, bias = 0)
    shift[c] = beta[c];
  }
  if (mm) {                                                    // UPDATE_OPS (same expression as bn_update_moving_kernel)
    mm[c] = mm[c] * momentum + mean[c] * (1.0f - momentum);
    mv[c] = mv[c] * momentum + vf * (1.0f - momentum);
  }
}

__global__ void bn_fold_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                               const float* __restrict__ mean, const float* __restrict__ var,
                               const float* __restrict__ bias, float eps, float* __restrict__ scale,
                               float* __restrict__ shift, int C) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = gamma[c] * rsqrtf(var[c] + eps);
  float b = bias ? bias[c] : 0.0f;
  scale[c] = s;
  shift[c] = beta[c] + (b - mean[c]) * s;
}

__global__ void bn_update_moving_kernel(float* __restrict__ mm, float* __restrict__ mv, const float* __restrict__ mean,
                                        const float* __restrict__ var, float momentum, int C) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  mm[c] = mm[c] * momentum + mean[c] * (1.0f - momentum);
  mv[c] = mv[c] * momentum + var[c] * (1.0f - momentum);
}

// ---------------------------------------------------------------------------------------------
// a2/a3  y = leaky((x - sub)*scale + shift), optional 2x2/2 max-pool (order conv->BN->leaky->pool,
// darknet.py:150-151), f32 or bf16 output.  One thread per output element group of VEC channels.
// ---------------------------------------------------------------------------------------------
template <int VEC, bool BF16OUT>
__global__ void affine_leaky_pool_kernel(const float* __restrict__ x, int ldx, const float* __restrict__ sub,
                                         const float* __restrict__ scale, const float* __restrict__ shift, float alpha, int leaky_on, int pool,
                                         void* __restrict__ out, int N, int H, int W, int C, int ldo, int s2d, int lo_off) {
  int Ho = pool ? H / 2 : H, Wo = pool ? W / 2 : W;
  int CV = C / VEC;
  size_t total = (size_t)N * Ho * Wo * CV;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    int cv = (int)(i % CV);
    size_t pix = i / CV;
    int wo = (int)(pix % Wo);
    int ho = (int)((pix / Wo) % Ho);
    int n = (int)(pix / ((size_t)Wo * Ho));
    int c0 = cv * VEC;
    float r[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) r[v] = -INFINITY;
    int np = pool ? 2 : 1;
    for (int dy = 0; dy < np; ++dy)
      for (int dx = 0; dx < np; ++dx) {
        int h = pool ? ho * 2 + dy : ho, w = pool ? wo * 2 + dx : wo;
        const float* px = x + ((size_t)(n * H + h) * W + w) * ldx + c0;
        float t[VEC];
        if (VEC == 4) {
          float4 q = *reinterpret_cast<const float4*>(px);
          t[0] = q.x; t[1 % VEC] = q.y; t[2 % VEC] = q.z; t[3 % VEC] = q.w;
        } else {
#pragma unroll
          for (int v = 0; v < VEC; ++v) t[v] = px[v];
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          float sc = scale ? scale[c0 + v] : 1.0f, sh = shift ? shift[c0 + v] : 0.0f;
          float sb = sub ? sub[c0 + v] : 0.0f;
          float y = (t[v] - sb) * sc + sh;   // (x - mean) first: exact cancellation when |mean| >> std
          if (leaky_on) y = leaky(y, alpha);
          r[v] = fmaxf(r[v], y);
        }
      }
    // dense rows of stride ldo, or (s2d, passthrough/reorg) tf.space_to_depth(block 2): pixel (h, w) lands in
    // row (h/2, w/2) at channel block (h%2)*2 + (w%2) -- the reorg layer is this store address, never a copy
    size_t o = s2d ? ((size_t)(n * (Ho >> 1) + (ho >> 1)) * (Wo >> 1) + (wo >> 1)) * ldo + (size_t)(((ho & 1) * 2 + (wo & 1)) * C) + c0
                   : pix * ldo + c0;
    if (BF16OUT) {
      __nv_bfloat16* ob = reinterpret_cast<__nv_bfloat16*>(out) + o;
      if (VEC == 4) {
        __nv_bfloat162 a = __floats2bfloat162_rn(r[0], r[1 % VEC]);
        __nv_bfloat162 b = __floats2bfloat162_rn(r[2 % VEC], r[3 % VEC]);
        uint2 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&a);
        pk.y = *reinterpret_cast<uint32_t*>(&b);
        *reinterpret_cast<uint2*>(ob) = pk;
      } else {
#pragma unroll
        for (int v = 0; v < VEC; ++v) ob[v] = __float2bfloat16_rn(r[v]);
      }
      if (lo_off) {                                   // bf16x3: lo = bf16(v - hi) at column lo_off + c
#pragma unroll
        for (int v = 0; v < VEC; ++v) ob[lo_off + v] = __float2bfloat16_rn(r[v] - __bfloat162float(__float2bfloat16_rn(r[v])));
      }
    } else {
      float* of = reinterpret_cast<float*>(out) + o;
      if (VEC == 4) {
        *reinterpret_cast<float4*>(of) = make_float4(r[0], r[1 % VEC], r[2 % VEC], r[3 % VEC]);
      } else {
#pragma unroll
        for (int v = 0; v < VEC; ++v) of[v] = r[v];
      }
    }
  }
}

// bf16x3: the lo halves bf16(v - hi) of 8 values whose hi halves are packed in `hi`
__device__ __forceinline__ uint4 lo_half8(const float* y, const uint4& hi) {
  const uint32_t h[4] = {hi.x, hi.y, hi.z, hi.w};
  uint32_t l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 hf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&h[i]));
    const __nv_bfloat162 l2 = __floats2bfloat162_rn(y[2 * i] - hf.x, y[2 * i + 1] - hf.y);
    l[i] = *reinterpret_cast<const uint32_t*>(&l2);
  }
  return make_uint4(l[0], l[1], l[2], l[3]);
}

// Fast path of the above for the batch-statistics head layers (no pool, dense rows, C % 8 == 0, bf16 out): the generic
// kernel spends its time in 64-bit div/mod per element (30 us for 66 MB, ncu r1c).  Here a thread owns 8 channels --
// their sub / scale / shift live in registers -- and walks rows, four rows of 2 x 16-byte streaming loads in flight,
// one 16-byte store per row.  block = (C/8 rounded to a warp, up to 128) x rows-per-block lanes.
__global__ void __launch_bounds__(256) affine_leaky_rows_bf16_kernel(const float* __restrict__ x, int ldx, const float* __restrict__ sub,
                                                                     const float* __restrict__ scale, const float* __restrict__ shift,
                                                                     float alpha, int leaky_on, __nv_bfloat16* __restrict__ out, int ldo,
                                                                     int M, int C8, int lo_off) {
  const int cx = blockIdx.y * blockDim.x + threadIdx.x;          // channel group
  if (cx >= C8) return;
  const int c0 = cx * 8;
  float sb[8], sc[8], sh[8];
#pragma unroll
  for (int v = 0; v < 8; ++v) {
    sb[v] = sub ? sub[c0 + v] : 0.0f;
    sc[v] = scale ? scale[c0 + v] : 1.0f;
    sh[v] = shift ? shift[c0 + v] : 0.0f;
  }
  const int rstep = gridDim.x * blockDim.y;
  for (int r0 = blockIdx.x * blockDim.y + threadIdx.y; r0 < M; r0 += 4 * rstep) {
    float4 a[4], b[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = r0 + j * rstep;
      if (r < M) {
        const float4* px = reinterpret_cast<const float4*>(x + (size_t)r * ldx + c0);
        a[j] = __ldcs(px);
        b[j] = __ldcs(px + 1);
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = r0 + j * rstep;
      if (r >= M) continue;
      const float t[8] = {a[j].x, a[j].y, a[j].z, a[j].w, b[j].x, b[j].y, b[j].z, b[j].w};
      float y[8];
#pragma unroll
      for (int v = 0; v < 8; ++v) {
        y[v] = (t[v] - sb[v]) * sc[v] + sh[v];                   // same expression as the generic kernel
        if (leaky_on) y[v] = leaky(y[v], alpha);
      }
      const __nv_bfloat162 h0 = __floats2bfloat162_rn(y[0], y[1]), h1 = __floats2bfloat162_rn(y[2], y[3]);
      const __nv_bfloat162 h2 = __floats2bfloat162_rn(y[4], y[5]), h3 = __floats2bfloat162_rn(y[6], y[7]);
      uint4 pk;
      pk.x = *reinterpret_cast<const uint32_t*>(&h0); pk.y = *reinterpret_cast<const uint32_t*>(&h1);
      pk.z = *reinterpret_cast<const uint32_t*>(&h2); pk.w = *reinterpret_cast<const uint32_t*>(&h3);
      *reinterpret_cast<uint4*>(out + (size_t)r * ldo + c0) = pk;
      if (lo_off) *reinterpret_cast<uint4*>(out + (size_t)r * ldo + lo_off + c0) = lo_half8(y, pk);
    }
  }
}

// ... and with the 2x2 max-pool (training forward of the pooled layers: conv -> batch-stat BN -> leaky -> pool): a thread owns
// 8 channels and walks POOLED pixels; eight 16-byte loads in flight per pooled pixel, 32-bit index arithmetic.
__global__ void __launch_bounds__(256) affine_leaky_pool_rows_bf16_kernel(const float* __restrict__ x, int ldx, const float* __restrict__ sub,
                                                                          const float* __restrict__ scale, const float* __restrict__ shift,
                                                                          float alpha, int leaky_on, __nv_bfloat16* __restrict__ out,
                                                                          int ldo, int H, int W, unsigned units, int C8, int lo_off) {
  const int cx = blockIdx.y * blockDim.x + threadIdx.x;
  if (cx >= C8) return;
  const int c0 = cx * 8;
  float sb[8], sc[8], sh[8];
#pragma unroll
  for (int v = 0; v < 8; ++v) {
    sb[v] = sub ? sub[c0 + v] : 0.0f;
    sc[v] = scale ? scale[c0 + v] : 1.0f;
    sh[v] = shift ? shift[c0 + v] : 0.0f;
  }
  const unsigned Wo = (unsigned)W >> 1, Ho = (unsigned)H >> 1;
  const unsigned ustep = gridDim.x * blockDim.y;
  for (unsigned u = blockIdx.x * blockDim.y + threadIdx.y; u < units; u += ustep) {
    const unsigned wo = u % Wo, t = u / Wo, ho = t % Ho, n = t / Ho;
    const size_t base = ((size_t)n * H + 2 * ho) * (size_t)W + 2 * wo;
    const size_t rows[4] = {base, base + 1, base + W, base + W + 1};
    float4 a[4], b[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float4* px = reinterpret_cast<const float4*>(x + rows[k] * ldx + c0);
      a[k] = __ldcs(px);
      b[k] = __ldcs(px + 1);
    }
    float r[8];
#pragma unroll
    for (int v = 0; v < 8; ++v) r[v] = -INFINITY;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float tt[8] = {a[k].x, a[k].y, a[k].z, a[k].w, b[k].x, b[k].y, b[k].z, b[k].w};
#pragma unroll
      for (int v = 0; v < 8; ++v) {
        float y = (tt[v] - sb[v]) * sc[v] + sh[v];               // same expression as the generic kernel
        if (leaky_on) y = leaky(y, alpha);
        r[v] = fmaxf(r[v], y);
      }
    }
    const __nv_bfloat162 h0 = __floats2bfloat162_rn(r[0], r[1]), h1 = __floats2bfloat162_rn(r[2], r[3]);
    const __nv_bfloat162 h2 = __floats2bfloat162_rn(r[4], r[5]), h3 = __floats2bfloat162_rn(r[6], r[7]);
    uint4 pk;
    pk.x = *reinterpret_cast<const uint32_t*>(&h0); pk.y = *reinterpret_cast<const uint32_t*>(&h1);
    pk.z = *reinterpret_cast<const uint32_t*>(&h2); pk.w = *reinterpret_cast<const uint32_t*>(&h3);
    *reinterpret_cast<uint4*>(out + (size_t)u * ldo + c0) = pk;
    if (lo_off) *reinterpret_cast<uint4*>(out + (size_t)u * ldo + lo_off + c0) = lo_half8(r, pk);
  }
}

// Same idea for the float32 output of the detection layer (C = 125, rows padded to 128 in, dense out): one thread per
// channel holds its constants and walks rows; loads and stores are coalesced along the channels.  (The generic kernel
// took 15 us for 5.6 MB.)
__global__ void __launch_bounds__(256) affine_leaky_rows_f32_kernel(const float* __restrict__ x, int ldx, const float* __restrict__ sub,
                                                                    const float* __restrict__ scale, const float* __restrict__ shift,
                                                                    float alpha, int leaky_on, float* __restrict__ out, int ldo, int M,
                                                                    int C) {
  const int c = threadIdx.x;
  if (c >= C) return;
  const float sb = sub ? sub[c] : 0.0f, sc = scale ? scale[c] : 1.0f, sh = shift ? shift[c] : 0.0f;
  const int rstep = gridDim.x * blockDim.y;
  for (int r0 = blockIdx.x * blockDim.y + threadIdx.y; r0 < M; r0 += 4 * rstep) {
    float t[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = r0 + j * rstep;
      t[j] = r < M ? __ldcs(x + (size_t)r * ldx + c) : 0.0f;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = r0 + j * rstep;
      if (r >= M) continue;
      float y = (t[j] - sb) * sc + sh;                           // same expression as the generic kernel
      if (leaky_on) y = leaky(y, alpha);
      out[(size_t)r * ldo + c] = y;
    }
  }
}

// a3  tf.nn.max_pool 2x2/2 (darknet.py:24-25) on a bf16 NHWC tensor, 8 channels (16 B) per thread.  Used when a layer's
// un-pooled output is needed as well (the passthrough source, darknet.py:170) so the pool cannot live in the conv epilogue.
__global__ void maxpool2x2_bf16_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int N, int H, int W, int CV) {
  const int Ho = H / 2, Wo = W / 2;
  const size_t total = (size_t)N * Ho * Wo * CV;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int cv = (int)(i % CV);
    const size_t pix = i / CV;
    const int wo = (int)(pix % Wo), ho = (int)((pix / Wo) % Ho), n = (int)(pix / ((size_t)Wo * Ho));
    const uint4* p = x + ((size_t)(n * H + 2 * ho) * W + 2 * wo) * CV + cv;
    uint4 a = p[0], b = p[CV], c = p[(size_t)W * CV], d = p[(size_t)W * CV + CV];
    uint4 r;
    uint32_t* ra = &a.x; uint32_t* rb = &b.x; uint32_t* rc = &c.x; uint32_t* rd = &d.x; uint32_t* rr = &r.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      __nv_bfloat162 m = __hmax2(__hmax2(*reinterpret_cast<__nv_bfloat162*>(&ra[k]), *reinterpret_cast<__nv_bfloat162*>(&rb[k])),
                                 __hmax2(*reinterpret_cast<__nv_bfloat162*>(&rc[k]), *reinterpret_cast<__nv_bfloat162*>(&rd[k])));
      rr[k] = *reinterpret_cast<uint32_t*>(&m);
    }
    y[i] = r;
  }
}

// a11  tf.train.AdamOptimizer (pascal_train_darknet.py:51): TF1 update form, lr_t from the host.
// tf.nn.avg_pool / tf.layers.average_pooling2d with ksize == stride on an evenly divisible map (darknet.py:28-29,116: the
// 7x7 global pool of the darknet19 classifier): NHWC bf16 or f32 in, f32 out; one thread per output element, window summed
// row-major in float32.
template <typename T>
__global__ void avgpool_kernel(const T* __restrict__ x, float* __restrict__ y, int N, int H, int W, int C, int k) {
  const int Ho = H / k, Wo = W / k;
  const size_t total = (size_t)N * Ho * Wo * C;
  const float inv = 1.0f / (float)(k * k);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    size_t pix = i / C;
    const int wo = (int)(pix % Wo);
    pix /= Wo;
    const int ho = (int)(pix % Ho), n = (int)(pix / Ho);
    float acc = 0.0f;
    for (int dy = 0; dy < k; ++dy)
      for (int dx = 0; dx < k; ++dx)
        acc += (float)x[((size_t)(n * H + ho * k + dy) * W + wo * k + dx) * C + c];
    y[i] = acc * inv;
  }
}

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, size_t n, float lr_t, float b1, float b2, float eps) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float gi = g[i];
    float mi = b1 * m[i] + (1.0f - b1) * gi;
    float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    p[i] -= lr_t * mi / (sqrtf(vi) + eps);
  }
}

// The training step's form of the same update, 16 bytes per access: the gradient is scaled on the fly (the 1/world of the
// data-parallel mean: the all-reduce delivers the SUM), the step size may come from device memory (so that a CUDA graph
// of the step does not bake the bias correction of one iteration in), and the gradient arena is cleared behind the read
// (the weight-gradient kernels accumulate into it, and this kernel is its last reader) -- no separate 193 MB memset / scale.
__global__ void __launch_bounds__(256) adam_ex_kernel(float4* __restrict__ p, float4* __restrict__ g, float4* __restrict__ m,
                                                      float4* __restrict__ v, size_t n4, float lr_t, const float* __restrict__ lr_dev,
                                                      float b1, float b2, float eps, float gscale, int zero_grad) {
  const float lr = lr_dev ? *lr_dev : lr_t;
  const float c1 = 1.0f - b1, c2 = 1.0f - b2;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n4; i += stride) {
    float4 gi = g[i], mi = m[i], vi = v[i], pi = p[i];
    gi.x *= gscale; gi.y *= gscale; gi.z *= gscale; gi.w *= gscale;
    mi.x = b1 * mi.x + c1 * gi.x; mi.y = b1 * mi.y + c1 * gi.y; mi.z = b1 * mi.z + c1 * gi.z; mi.w = b1 * mi.w + c1 * gi.w;
    vi.x = b2 * vi.x + c2 * gi.x * gi.x; vi.y = b2 * vi.y + c2 * gi.y * gi.y;
    vi.z = b2 * vi.z + c2 * gi.z * gi.z; vi.w = b2 * vi.w + c2 * gi.w * gi.w;
    pi.x -= lr * mi.x / (sqrtf(vi.x) + eps); pi.y -= lr * mi.y / (sqrtf(vi.y) + eps);
    pi.z -= lr * mi.z / (sqrtf(vi.z) + eps); pi.w -= lr * mi.w / (sqrtf(vi.w) + eps);
    m[i] = mi; v[i] = vi; p[i] = pi;
    if (zero_grad) g[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// tf.train.MomentumOptimizer (imagenet_train_darknet.py:58; TF's ApplyMomentum without Nesterov): accum = momentum * accum + g,
// p -= lr * accum.  Same conventions as adam_ex_kernel: gradient scaled on the fly, arena cleared behind the read.
__global__ void __launch_bounds__(256) momentum_kernel(float4* __restrict__ p, float4* __restrict__ g, float4* __restrict__ acc,
                                                       size_t n4, float lr, float mom, float gscale, int zero_grad) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n4; i += stride) {
    float4 gi = g[i], ai = acc[i], pi = p[i];
    ai.x = mom * ai.x + gi.x * gscale; ai.y = mom * ai.y + gi.y * gscale;
    ai.z = mom * ai.z + gi.z * gscale; ai.w = mom * ai.w + gi.w * gscale;
    pi.x -= lr * ai.x; pi.y -= lr * ai.y; pi.z -= lr * ai.z; pi.w -= lr * ai.w;
    acc[i] = ai; p[i] = pi;
    if (zero_grad) g[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// dtype plumbing of the drop-in builders (float32 <-> bf16, 8 elements per thread where aligned) and the chain-rule scale of
// get_loss's backward (dnet * upstream scalar, the scalar read from device memory: no host sync)
__global__ void cast_f32_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, size_t n) {
  size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 8, stride = (size_t)gridDim.x * blockDim.x * 8;
  for (; i < n; i += stride) {
    if (i + 8 <= n && ((((uintptr_t)(x + i)) & 15) == 0) && ((((uintptr_t)(y + i)) & 15) == 0)) {
      const float4 a = *reinterpret_cast<const float4*>(x + i), b = *reinterpret_cast<const float4*>(x + i + 4);
      const __nv_bfloat162 h0 = __floats2bfloat162_rn(a.x, a.y), h1 = __floats2bfloat162_rn(a.z, a.w);
      const __nv_bfloat162 h2 = __floats2bfloat162_rn(b.x, b.y), h3 = __floats2bfloat162_rn(b.z, b.w);
      *reinterpret_cast<uint4*>(y + i) = make_uint4(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1),
                                                    *reinterpret_cast<const uint32_t*>(&h2), *reinterpret_cast<const uint32_t*>(&h3));
    } else {
      for (size_t j = i; j < n && j < i + 8; ++j) y[j] = __float2bfloat16_rn(x[j]);
    }
  }
}

__global__ void cast_bf16_f32_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ y, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) y[i] = __bfloat162float(x[i]);
}

__global__ void scale_by_device_scalar_kernel(const float* __restrict__ x, const float* __restrict__ s, float* __restrict__ y, size_t n) {
  const float sv = *s;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) y[i] = x[i] * sv;
}

static int g_sms_elementwise() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  return sms;
}

static int grid_for(size_t n, int block) {
  size_t g = (n + block - 1) / block;
  size_t cap = 148 * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace y2

using namespace y2;

extern "C" {

int y2_preprocess_u8(const uint8_t* img, void* out, int N, int H, int W, int out_dtype, y2_stream_t stream) {
  Y2_ARG(img && out && N > 0 && H > 0 && W > 0 && (out_dtype == 0 || out_dtype == 1));
  cudaStream_t st = (cudaStream_t)stream;
  size_t npix = (size_t)N * H * W;
  if (out_dtype == 0) {
    preprocess_u8_f32_kernel<<<grid_for(npix * 3, 256), 256, 0, st>>>(img, (float*)out, npix * 3);
  } else {
    preprocess_u8_bf16c8_kernel<<<grid_for(npix, 256), 256, 0, st>>>(img, (uint4*)out, npix);
  }
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_resize_bilinear_u8(const uint8_t* src, int src_h, int src_w, uint8_t* dst, int dst_h, int dst_w, y2_stream_t stream) {
  Y2_ARG(src && dst && src_h > 0 && src_w > 0 && dst_h > 0 && dst_w > 0);
  // OpenCV: inv_scale = dsize / ssize (double), scale = 1. / inv_scale
  const double scale_x = 1.0 / ((double)dst_w / (double)src_w), scale_y = 1.0 / ((double)dst_h / (double)src_h);
  const int area2 = (src_w == 2 * dst_w && src_h == 2 * dst_h) ? 1 : 0;
  dim3 grid((unsigned)((dst_w + 127) / 128), (unsigned)dst_h);
  resize_bilinear_u8c3_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(src, src_h, src_w, (size_t)src_w * 3, dst, dst_h, dst_w, scale_x,
                                                                     scale_y, area2);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_pad_cast_f32_to_bf16c8(const float* x, void* out, int N, int H, int W, y2_stream_t stream) {
  Y2_ARG(x && out && N > 0 && H > 0 && W > 0);
  size_t npix = (size_t)N * H * W;
  pad_cast_f32_bf16c8_kernel<<<grid_for(npix, 256), 256, 0, (cudaStream_t)stream>>>(x, (uint4*)out, npix);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_conv_cin_padded(int Cin) { return Cin < 8 ? 8 : Cin; }

static int conv_kp(int ksize, int Cin) {
  int cin_p = y2_conv_cin_padded(Cin);
  int K = ksize * ksize * cin_p;
  if (cin_p == 8) return (K + 15) / 16 * 16;   // first layer: 9 taps x 8 -> 72 -> 80 (whole MMA K steps)
  return K;
}

size_t y2_conv_packed_weight_elems(int ksize, int Cin, int Cout) {
  int cout_p = (Cout + 15) / 16 * 16;
  return (size_t)cout_p * conv_kp(ksize, Cin);
}

int y2_pack_weights_bf16(const float* w_hwio, void* w_packed, int ksize, int Cin, int Cout, y2_stream_t stream) {
  Y2_ARG(w_hwio && w_packed && (ksize == 1 || ksize == 3) && Cin > 0 && Cout > 0);
  int cin_p = y2_conv_cin_padded(Cin);
  Y2_ARG(cin_p == 8 || cin_p % 32 == 0);
  int cout_p = (Cout + 15) / 16 * 16;
  int Kp = conv_kp(ksize, Cin);
  size_t total = (size_t)cout_p * Kp;
  if (cin_p % 32 == 0 && !env().affine_generic) {
    dim3 grid((unsigned)((cout_p + 31) / 32), (unsigned)(cin_p / 32), (unsigned)(ksize * ksize));
    pack_weights_tiled_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(w_hwio, (__nv_bfloat16*)w_packed, Cin, Cout, cin_p,
                                                                              cout_p, Kp);
  } else {
    pack_weights_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
        w_hwio, (__nv_bfloat16*)w_packed, ksize * ksize, Cin, Cout, cin_p, cout_p, Kp);
  }
  Y2_LAUNCHED();
  return Y2_OK;
}

size_t y2_conv_packed_weight_split_elems(int ksize, int Cin, int Cout) {
  int cout_p = (Cout + 15) / 16 * 16;
  return (size_t)cout_p * ksize * ksize * 3 * Cin;
}

int y2_pack_weights_bf16_split(const float* w_hwio, void* w_packed, int ksize, int Cin, int Cout, y2_stream_t stream) {
  Y2_ARG(w_hwio && w_packed && (ksize == 1 || ksize == 3) && Cin > 0 && Cout > 0 && Cin % 32 == 0);
  int cout_p = (Cout + 15) / 16 * 16;
  size_t total = (size_t)cout_p * ksize * ksize * 3 * Cin;
  pack_weights_split_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(w_hwio, (__nv_bfloat16*)w_packed,
                                                                                    ksize * ksize, Cin, Cout, cout_p);
  Y2_LAUNCHED();
  return Y2_OK;
}

static int bn_splits(int M) {
  int s = (M + 127) / 128;
  return s > 1024 ? 1024 : (s < 1 ? 1 : s);
}

size_t y2_bn_stats_workspace_bytes(int M, int C) { return (size_t)bn_splits(M) * C * 2 * sizeof(double); }

static int bn_stats_impl(const float* x, int M, int C, int ld, float* mean, float* var, const float* gamma, const float* beta,
                         float eps, float* scale, float* shift, void* workspace, size_t workspace_bytes, y2_stream_t stream,
                         float* mm = nullptr, float* mv = nullptr, float momentum = 0.0f) {
  Y2_ARG(x && mean && var && M > 0 && C > 0 && ld >= C);
  if (!workspace || workspace_bytes < y2_bn_stats_workspace_bytes(M, C)) {
    set_error("y2_bn_stats: workspace too small (%zu < %zu)", workspace_bytes, y2_bn_stats_workspace_bytes(M, C));
    return Y2_ERR_WORKSPACE;
  }
  Y2_ARG(((uintptr_t)workspace & 15) == 0);
  cudaStream_t st = (cudaStream_t)stream;
  int splits = bn_splits(M);
  int rows = (M + splits - 1) / splits;
  splits = (M + rows - 1) / rows;
  if (C % 4 == 0 && ld % 4 == 0 && (((uintptr_t)x) & 15) == 0) {
    const int cg = C / 4;
    // ONE wave of blocks: registers allow 5 blocks of 256 threads per SM, and the 1024 splits of a large map used to run as
    // 740 + 284 -- the second wave at 38 % occupancy (ncu r2n: 46 % of the warp slots active, 3.9 TB/s).  The round-robin
    // tile assignment balances any number of splits.  Layer 1 at batch 64 (1.4 GB): 382 -> 237 us = 6.0 TB/s.
    {
      const int tx = cg <= 8 ? 8 : (cg <= 16 ? 16 : 32);
      const int wave = g_sms_elementwise() * 5 / ((cg + tx - 1) / tx);
      if (splits > wave) splits = wave > 1 ? wave : 1;
    }
    // large maps: eight rows (128 B per thread) in flight -- with four the kernel sat at 3.9 TB/s (ncu r2n: 47 % of DRAM peak, the
    // affine pass with 128 B per thread in flight reaches 5.7); the deep 13x13 layers keep four (measured: no gain there)
    const bool deep = M >= 32768;
    const int cs = (size_t)M * ld * 4 > (96u << 20) ? 1 : 0;
#define Y2_LAUNCH_STATS(TX_)                                                                                                  \
  do {                                                                                                                        \
    if (deep) bn_stats_partial_v4_kernel<TX_, 8><<<dim3((cg + TX_ - 1) / TX_, splits), 256, 0, st>>>(x, M, C, ld, rows, (double*)workspace, cs); \
    else bn_stats_partial_v4_kernel<TX_, 4><<<dim3((cg + TX_ - 1) / TX_, splits), 256, 0, st>>>(x, M, C, ld, rows, (double*)workspace, cs);      \
  } while (0)
    if (cg <= 8) Y2_LAUNCH_STATS(8);
    else if (cg <= 16) Y2_LAUNCH_STATS(16);
    else Y2_LAUNCH_STATS(32);
#undef Y2_LAUNCH_STATS
  } else {
    dim3 grid((C + 31) / 32, splits), block(32, 8);
    bn_stats_partial_kernel<<<grid, block, 0, st>>>(x, M, C, ld, rows, (double*)workspace);
  }
  Y2_LAUNCHED();
  bn_stats_final_kernel<<<(C + 31) / 32, dim3(32, FIN_TY), 0, st>>>(x, (const double*)workspace, splits, M, C, mean, var, gamma, beta,
                                                               eps, scale, shift, mm, mv, momentum);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_bn_stats(const float* x, int M, int C, int ld, float* mean, float* var, void* workspace, size_t workspace_bytes,
                y2_stream_t stream) {
  return bn_stats_impl(x, M, C, ld, mean, var, nullptr, nullptr, 0.0f, nullptr, nullptr, workspace, workspace_bytes, stream);
}

int y2_bn_stats_fold(const float* x, int M, int C, int ld, float* mean, float* var, const float* gamma, const float* beta,
                     float eps, float* scale, float* shift, void* workspace, size_t workspace_bytes, y2_stream_t stream) {
  Y2_ARG(gamma && beta && scale && shift);
  return bn_stats_impl(x, M, C, ld, mean, var, gamma, beta, eps, scale, shift, workspace, workspace_bytes, stream);
}

int y2_bn_stats_fold_train(const float* x, int M, int C, int ld, float* mean, float* var, const float* gamma, const float* beta,
                           float eps, float* scale, float* shift, float* moving_mean, float* moving_var, float momentum,
                           void* workspace, size_t workspace_bytes, y2_stream_t stream) {
  Y2_ARG(gamma && beta && scale && shift && moving_mean && moving_var);
  return bn_stats_impl(x, M, C, ld, mean, var, gamma, beta, eps, scale, shift, workspace, workspace_bytes, stream, moving_mean,
                       moving_var, momentum);
}

int y2_bn_fold(const float* gamma, const float* beta, const float* mean, const float* var, const float* conv_bias,
               float eps, float* scale, float* shift, int C, y2_stream_t stream) {
  Y2_ARG(gamma && beta && mean && var && scale && shift && C > 0);
  bn_fold_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(gamma, beta, mean, var, conv_bias, eps, scale,
                                                                     shift, C);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_bn_update_moving(float* moving_mean, float* moving_var, const float* mean, const float* var, float momentum,
                        int C, y2_stream_t stream) {
  Y2_ARG(moving_mean && moving_var && mean && var && C > 0);
  bn_update_moving_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(moving_mean, moving_var, mean, var,
                                                                              momentum, C);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_affine_leaky_pool_ex(const float* x, int ldx, const float* sub, const float* scale, const float* shift, float alpha,
                            int leaky_on, int pool, void* out, int out_dtype, int ldo, int space_to_depth, int lo_off, int N, int H,
                            int W, int C, y2_stream_t stream) {
  Y2_ARG(x && out && N > 0 && H > 0 && W > 0 && C > 0 && ldx >= C && (out_dtype == 0 || out_dtype == 1 || out_dtype == 2));
  if (pool) Y2_ARG(H % 2 == 0 && W % 2 == 0);
  const bool split = out_dtype == 2;                // bf16x3: hi at column c, lo at column lo_off + c (0 -> the row's second half)
  if (split) out_dtype = 1;
  if (ldo <= 0) ldo = split ? 2 * C : C;
  if (split && lo_off <= 0) lo_off = space_to_depth ? ldo / 2 : C;
  if (!split) lo_off = 0;
  if (space_to_depth) Y2_ARG(!pool && H % 2 == 0 && W % 2 == 0 && ldo >= (split ? lo_off + 4 * C : 4 * C));
  else Y2_ARG(ldo >= (split ? lo_off + C : C));
  if (split) Y2_ARG(lo_off >= C);
  cudaStream_t st = (cudaStream_t)stream;
  int Ho = pool ? H / 2 : H, Wo = pool ? W / 2 : W;
  if (!pool && !space_to_depth && out_dtype == 1 && C % 8 == 0 && ldx % 4 == 0 && ldo % 8 == 0 && lo_off % 8 == 0 && (((uintptr_t)x | (uintptr_t)out) & 15) == 0 &&
      (long long)N * H * W < (1ll << 30) && !env().affine_generic) {
    const int M = N * H * W, C8 = C / 8;
    const int bx = C8 >= 128 ? 128 : ((C8 + 31) / 32) * 32;       // channel-group lanes per block (whole warps)
    const int by = 256 / bx;                                      // row lanes per block
    int gx = g_sms_elementwise() * 8 / ((C8 + bx - 1) / bx);
    const int need = (M + by - 1) / by;
    if (gx > need) gx = need;
    if (gx < 1) gx = 1;
    affine_leaky_rows_bf16_kernel<<<dim3(gx, (C8 + bx - 1) / bx), dim3(bx, by), 0, st>>>(
        x, ldx, sub, scale, shift, alpha, leaky_on, reinterpret_cast<__nv_bfloat16*>(out), ldo, M, C8, lo_off);
    Y2_LAUNCHED();
    return Y2_OK;
  }
  if (pool && !space_to_depth && out_dtype == 1 && C % 8 == 0 && ldx % 4 == 0 && ldo % 8 == 0 && lo_off % 8 == 0 && (((uintptr_t)x | (uintptr_t)out) & 15) == 0 &&
      (long long)N * H * W < (1ll << 31) && !env().affine_generic) {
    const unsigned units = (unsigned)((long long)N * Ho * Wo);
    const int C8 = C / 8;
    const int bx = C8 >= 32 ? 32 : (C8 >= 16 ? 16 : (C8 >= 8 ? 8 : 4));
    const int by = 256 / bx;
    long long gx = (long long)g_sms_elementwise() * 16 / ((C8 + bx - 1) / bx);
    const long long need = ((long long)units + by - 1) / by;
    if (gx > need) gx = need;
    if (gx < 1) gx = 1;
    affine_leaky_pool_rows_bf16_kernel<<<dim3((unsigned)gx, (unsigned)((C8 + bx - 1) / bx)), dim3(bx, by), 0, st>>>(
        x, ldx, sub, scale, shift, alpha, leaky_on, reinterpret_cast<__nv_bfloat16*>(out), ldo, H, W, units, C8, lo_off);
    Y2_LAUNCHED();
    return Y2_OK;
  }
  if (!pool && !space_to_depth && out_dtype == 0 && C <= 256 && (C % 4 != 0 || ldx % 4 != 0 || ldo % 4 != 0) &&
      (long long)N * H * W < (1ll << 30) && !env().affine_generic) {
    const int M = N * H * W;
    const int bx = ((C + 31) / 32) * 32, by = 256 / bx > 0 ? 256 / bx : 1;
    int gx = g_sms_elementwise() * 8;
    const int need = (M + by - 1) / by;
    if (gx > need) gx = need;
    affine_leaky_rows_f32_kernel<<<gx, dim3(bx, by), 0, st>>>(x, ldx, sub, scale, shift, alpha, leaky_on, reinterpret_cast<float*>(out),
                                                              ldo, M, C);
    Y2_LAUNCHED();
    return Y2_OK;
  }
  bool vec4 = (C % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0) && (lo_off % 4 == 0) && (((uintptr_t)x & 15) == 0) && (((uintptr_t)out & 15) == 0);
  size_t total = (size_t)N * Ho * Wo * (vec4 ? C / 4 : C);
  int g = grid_for(total, 256);
  const int s2d = space_to_depth ? 1 : 0;
  if (vec4) {
    if (out_dtype == 1)
      affine_leaky_pool_kernel<4, true><<<g, 256, 0, st>>>(x, ldx, sub, scale, shift, alpha, leaky_on, pool, out, N, H, W, C, ldo, s2d, lo_off);
    else
      affine_leaky_pool_kernel<4, false><<<g, 256, 0, st>>>(x, ldx, sub, scale, shift, alpha, leaky_on, pool, out, N, H, W, C, ldo, s2d, lo_off);
  } else {
    if (out_dtype == 1)
      affine_leaky_pool_kernel<1, true><<<g, 256, 0, st>>>(x, ldx, sub, scale, shift, alpha, leaky_on, pool, out, N, H, W, C, ldo, s2d, lo_off);
    else
      affine_leaky_pool_kernel<1, false><<<g, 256, 0, st>>>(x, ldx, sub, scale, shift, alpha, leaky_on, pool, out, N, H, W, C, ldo, s2d, lo_off);
  }
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_affine_leaky_pool(const float* x, int ldx, const float* sub, const float* scale, const float* shift, float alpha, int leaky_on,
                         int pool, void* out, int out_dtype, int N, int H, int W, int C, y2_stream_t stream) {
  return y2_affine_leaky_pool_ex(x, ldx, sub, scale, shift, alpha, leaky_on, pool, out, out_dtype, 0, 0, 0, N, H, W, C, stream);
}

int y2_maxpool2x2_bf16(const void* x, void* y, int N, int H, int W, int C, y2_stream_t stream) {
  Y2_ARG(x && y && N > 0 && H > 0 && W > 0 && C > 0 && H % 2 == 0 && W % 2 == 0 && C % 8 == 0);
  Y2_ARG((((uintptr_t)x | (uintptr_t)y) & 15) == 0);
  size_t total = (size_t)N * (H / 2) * (W / 2) * (C / 8);
  maxpool2x2_bf16_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const uint4*)x, (uint4*)y, N, H, W, C / 8);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_avgpool(const void* x, int x_dtype, float* y, int N, int H, int W, int C, int k, y2_stream_t stream) {
  Y2_ARG(x && y && N > 0 && H > 0 && W > 0 && C > 0 && k > 0 && H % k == 0 && W % k == 0 && (x_dtype == 0 || x_dtype == 1));
  const size_t total = (size_t)N * (H / k) * (W / k) * C;
  if (x_dtype == 1) avgpool_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, y, N, H, W, C, k);
  else avgpool_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const float*)x, y, N, H, W, C, k);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_cast(const void* x, int x_dtype, void* y, int y_dtype, size_t n, y2_stream_t stream) {
  Y2_ARG(x && y && n > 0 && (x_dtype == 0 || x_dtype == 1) && (y_dtype == 0 || y_dtype == 1) && x_dtype != y_dtype);
  cudaStream_t st = (cudaStream_t)stream;
  if (x_dtype == 0) cast_f32_bf16_kernel<<<grid_for((n + 7) / 8, 256), 256, 0, st>>>((const float*)x, (__nv_bfloat16*)y, n);
  else cast_bf16_f32_kernel<<<grid_for(n, 256), 256, 0, st>>>((const __nv_bfloat16*)x, (float*)y, n);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_scale_by_device_scalar(const float* x, const float* scalar, float* y, size_t n, y2_stream_t stream) {
  Y2_ARG(x && scalar && y && n > 0);
  scale_by_device_scalar_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(x, scalar, y, n);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_adam_step(float* p, const float* g, float* m, float* v, size_t n, float lr_t, float beta1, float beta2,
                 float eps, y2_stream_t stream) {
  Y2_ARG(p && g && m && v && n > 0);
  adam_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, lr_t, beta1, beta2, eps);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_adam_step_ex(float* p, float* g, float* m, float* v, size_t n, float lr_t, const float* lr_t_dev, float beta1,
                    float beta2, float eps, float grad_scale, int zero_grad, y2_stream_t stream) {
  Y2_ARG(p && g && m && v && n > 0 && n % 4 == 0);
  Y2_ARG(((((uintptr_t)p) | ((uintptr_t)g) | ((uintptr_t)m) | ((uintptr_t)v)) & 15) == 0);
  adam_ex_kernel<<<grid_for(n / 4, 256), 256, 0, (cudaStream_t)stream>>>((float4*)p, (float4*)g, (float4*)m, (float4*)v, n / 4, lr_t,
                                                                         lr_t_dev, beta1, beta2, eps, grad_scale, zero_grad);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_momentum_step(float* p, float* g, float* accum, size_t n, float lr, float momentum, float grad_scale, int zero_grad,
                     void* stream) {
  Y2_ARG(p && g && accum && n > 0 && n % 4 == 0);
  Y2_ARG(((((uintptr_t)p) | ((uintptr_t)g) | ((uintptr_t)accum)) & 15) == 0);
  momentum_kernel<<<grid_for(n / 4, 256), 256, 0, (cudaStream_t)stream>>>((float4*)p, (float4*)g, (float4*)accum, n / 4, lr, momentum,
                                                                          grad_scale, zero_grad);
  Y2_LAUNCHED();
  return Y2_OK;
}

}  // extern "C"
