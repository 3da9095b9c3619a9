// backward.cu -- a11: the HBM-bound half of the training step's backward pass (what TF autodiff emits for
// conv_bn_layer, yolo2_nets/darknet.py:39-46, followed by max_pool, :24-25):
//
//   y2_bn_leaky_pool_bwd     dY (grad of the layer output, after the optional 2x2 max-pool) -> arg-max routing ->
//                            leaky slope -> batch-norm backward (batch statistics):
//                               dz      = dA * (z > 0 ? 1 : alpha)
//                               dbeta   = sum dz          dgamma = sum dz * xhat
//                               dh      = gamma*inv_std * (dz - dbeta/M - xhat * dgamma/M)        -> bf16 [M, ld_dh]
//                            z / xhat / the pooling arg-max are recomputed from the saved fp32 pre-BN rows, so the
//                            forward stores nothing extra.  Two passes over h (reduce in fp64, then apply).
//   y2_bn_leaky_pool_bwd_ex  the same, with dy read as a channel slice of wider rows (row stride ldy), through the inverse
//                            of a space_to_depth(2) store, and / or with an un-pooled addend (a pooled layer whose output
//                            also feeds a second consumer un-pooled): the YOLOv2 passthrough branch's gradients.
//   y2_pack_weights_dgrad_bf16   weights packed transposed + spatially flipped: the data gradient of a SAME stride-1
//                            convolution is the same convolution of dh with those weights, so dgrad runs on
//                            conv_tc_kernel (conv_tcgen05.cu) unchanged.
//   y2_conv_wgrad_c3         weight gradient of the first layer (Cin = 3): K = 11 M pixels, 27 x Cout outputs -- a
//                            shape the tensor cores cannot tile; persistent FFMA kernel with register accumulators.
//   y2_sum_rows_bf16         bias gradient helper (column sums of dh).
#include "common.cuh"

namespace y2 {
int num_sms();                    // conv_tcgen05.cu: SM count of the current device

// ---------------------------------------------------------------------------------------------
// pooled unit -> rows.  unit u indexes output pixels (n, ho, wo); rows are input pixels.
// ---------------------------------------------------------------------------------------------
struct UnitRows { size_t r[4]; int n; };

__device__ __forceinline__ UnitRows unit_rows(size_t u, int H, int W, bool pool) {
  UnitRows o;
  if (!pool) { o.r[0] = u; o.n = 1; return o; }
  const int Ho = H >> 1, Wo = W >> 1;
  const int wo = (int)(u % Wo);
  const size_t t = u / Wo;
  const int ho = (int)(t % Ho);
  const size_t n = t / Ho;
  const size_t base = (n * H + 2 * ho) * (size_t)W + 2 * wo;
  o.r[0] = base; o.r[1] = base + 1; o.r[2] = base + W; o.r[3] = base + W + 1;
  o.n = 4;
  return o;
}

__device__ __forceinline__ float load_dy(const void* dy, int dy_f32, size_t i) {
  return dy_f32 ? reinterpret_cast<const float*>(dy)[i] : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(dy)[i]);
}

// Where the gradient of output unit u (a pixel of the [N,Hu,Wu] map dy is given on) is read, channel c at + c.  The pointer is
// pre-offset to the layer's first column.
//   DY_DENSE  rows of stride C (the layer's own [N,Hu,Wu,C] gradient)
//   DY_ROWS   rows of stride ldy (a channel slice of a wider gradient: conv2's 1024 columns of the [N,S,S,1280] concat)
//   DY_S2D    depth-to-space: the layer's output was stored space_to_depth(2) into rows of stride ldy (the passthrough
//             branch), so pixel (h, w) reads row (h/2, w/2), column ((h%2)*2 + w%2)*C + c -- the inverse of the store
//             address of affine_leaky_pool_kernel's s2d mode (elementwise.cu)
enum { DY_DENSE = 0, DY_ROWS = 1, DY_S2D = 2 };

template <int DYM>
__device__ __forceinline__ size_t dy_row(size_t u, int ldy, int Hu, int Wu, int C) {      // offset of (unit u, channel 0)
  if (DYM == DY_DENSE) return u * C;
  if (DYM == DY_ROWS) return u * ldy;
  const int w = (int)(u % Wu);
  const size_t t = u / Wu;
  const int h = (int)(t % Hu);
  const size_t n = t / Hu;
  return ((n * (Hu >> 1) + (h >> 1)) * (size_t)(Wu >> 1) + (w >> 1)) * ldy + (size_t)(((h & 1) * 2 + (w & 1)) * C);
}

// pass 1: grid (ceil(C/32), splits), block (32, 8).  part[split][c][2] = (sum dz, sum dz*xhat)
// ADD: dy_add (bf16 [N,H,W,C], one value per input row) is added to every row's gradient in front of the leaky slope; the
// pooled dy still goes to the window's first maximum only.
template <int DYM, bool ADD>
__device__ __forceinline__ void bn_bwd_reduce_body(const float* __restrict__ h, int ldh, const void* __restrict__ dy, int dy_f32, int ldy,
                                     const __nv_bfloat16* __restrict__ dy_add,
                                     const float* __restrict__ mean, const float* __restrict__ var,
                                     const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                     float alpha, int leaky_on, int pool, int H, int W, int C, size_t units,
                                     size_t units_per_split, double* __restrict__ part) {
  __shared__ double s1[8][33], s2[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const size_t u0 = (size_t)blockIdx.y * units_per_split;
  const size_t u1 = min(units, u0 + units_per_split);
  double a1 = 0.0, a2 = 0.0;
  if (c < C) {
    const float mu = mean[c], inv = rsqrtf(var[c] + eps), g = gamma[c], b = beta[c];
    float f1 = 0.0f, f2 = 0.0f;
    int cnt = 0;
    for (size_t u = u0 + threadIdx.y; u < u1; u += 8) {
      const UnitRows ur = unit_rows(u, H, W, pool != 0);
      if constexpr (ADD) {
        float xs[4], zs[4], best = -INFINITY;
        int arg = 0;
        for (int k = 0; k < ur.n; ++k) {
          xs[k] = (h[ur.r[k] * ldh + c] - mu) * inv;
          zs[k] = xs[k] * g + b;
          const float a = leaky_on ? fmaxf(zs[k], alpha * zs[k]) : zs[k];
          if (a > best) { best = a; arg = k; }
        }
        const float dp = load_dy(dy, dy_f32, dy_row<DYM>(u, ldy, pool ? H >> 1 : H, pool ? W >> 1 : W, C) + c);
        for (int k = 0; k < ur.n; ++k) {
          float d = __bfloat162float(dy_add[ur.r[k] * C + c]) + (k == arg ? dp : 0.0f);
          if (leaky_on && !(zs[k] > 0.0f)) d *= alpha;
          f1 += d;
          f2 += d * xs[k];
        }
      } else {
        float best = -INFINITY, bx = 0.0f, bz = 0.0f;
        for (int k = 0; k < ur.n; ++k) {
          const float xh = (h[ur.r[k] * ldh + c] - mu) * inv;
          const float z = xh * g + b;
          const float a = leaky_on ? fmaxf(z, alpha * z) : z;
          if (a > best) { best = a; bx = xh; bz = z; }
        }
        float d = load_dy(dy, dy_f32, dy_row<DYM>(u, ldy, pool ? H >> 1 : H, pool ? W >> 1 : W, C) + c);
        if (leaky_on && !(bz > 0.0f)) d *= alpha;
        f1 += d;
        f2 += d * bx;
      }
      if (++cnt == 64) { a1 += (double)f1; a2 += (double)f2; f1 = f2 = 0.0f; cnt = 0; }
    }
    a1 += (double)f1;
    a2 += (double)f2;
  }
  s1[threadIdx.y][threadIdx.x] = a1;
  s2[threadIdx.y][threadIdx.x] = a2;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    for (int y = 1; y < 8; ++y) { a1 += s1[y][threadIdx.x]; a2 += s2[y][threadIdx.x]; }
    part[((size_t)blockIdx.y * C + c) * 2 + 0] = a1;
    part[((size_t)blockIdx.y * C + c) * 2 + 1] = a2;
  }
}
__global__ void bn_bwd_reduce_kernel(const float* __restrict__ h, int ldh, const void* __restrict__ dy, int dy_f32,
                                     const float* __restrict__ mean, const float* __restrict__ var,
                                     const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                     float alpha, int leaky_on, int pool, int H, int W, int C, size_t units,
                                     size_t units_per_split, double* __restrict__ part) {
  bn_bwd_reduce_body<DY_DENSE, false>(h, ldh, dy, dy_f32, C, nullptr, mean, var, gamma, beta, eps, alpha, leaky_on, pool, H, W,
                                      C, units, units_per_split, part);
}
template <int DYM, bool ADD>
__global__ void bn_bwd_reduce_ex_kernel(const float* __restrict__ h, int ldh, const void* __restrict__ dy, int dy_f32, int ldy,
                                        const __nv_bfloat16* __restrict__ dy_add, const float* __restrict__ mean,
                                        const float* __restrict__ var, const float* __restrict__ gamma,
                                        const float* __restrict__ beta, float eps, float alpha, int leaky_on, int pool, int H,
                                        int W, int C, size_t units, size_t units_per_split, double* __restrict__ part) {
  bn_bwd_reduce_body<DYM, ADD>(h, ldh, dy, dy_f32, ldy, dy_add, mean, var, gamma, beta, eps, alpha, leaky_on, pool, H, W, C,
                               units, units_per_split, part);
}

// Vectorised pass 1 (C % 4 == 0): a thread owns 4 channels (16-byte loads of h, 8-byte loads of bf16 dy) and keeps
// UNR units in flight; block = TX channel groups x (256/TX) unit lanes.  Four blocks resident per SM.
// DYM / ADD: the dy read of bn_bwd_reduce_kernel.
template <bool POOL, int TX, int DYM, bool ADD>
__device__ __forceinline__ void bn_bwd_reduce_v4_body(
    const float* __restrict__ h, int ldh, const void* __restrict__ dy, int dy_f32, int ldy,
    const __nv_bfloat16* __restrict__ dy_add, const float* __restrict__ mean,
    const float* __restrict__ var, const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float alpha,
    int leaky_on, int H, int W, int C, size_t units, size_t units_per_split, double* __restrict__ part) {
  constexpr int TY = 256 / TX;
  constexpr int NR = POOL ? 4 : 1;
  constexpr int UNR = POOL ? 2 : 4;
  constexpr int NA = ADD ? NR : 1;
  __shared__ double sm[TY][TX][8];
  const int tx = threadIdx.x % TX, ty = threadIdx.x / TX;
  const int c0 = (blockIdx.x * TX + tx) * 4;
  // unit tiles of UNR*TY units dealt to the splits round-robin (see bn_stats_partial_v4_kernel: DRAM page locality)
  (void)units_per_split;
  const size_t u1 = units;
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (c0 < C) {
    const float4 mu = *reinterpret_cast<const float4*>(mean + c0), vr = *reinterpret_cast<const float4*>(var + c0);
    const float4 g = *reinterpret_cast<const float4*>(gamma + c0), b = *reinterpret_cast<const float4*>(beta + c0);
    const float pm[4] = {mu.x, mu.y, mu.z, mu.w};
    const float pi[4] = {rsqrtf(vr.x + eps), rsqrtf(vr.y + eps), rsqrtf(vr.z + eps), rsqrtf(vr.w + eps)};
    const float pg[4] = {g.x, g.y, g.z, g.w}, pb[4] = {b.x, b.y, b.z, b.w};
    float f[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int cnt = 0;
    for (size_t ub = (size_t)blockIdx.y * UNR * TY + ty; ub < u1; ub += (size_t)gridDim.y * UNR * TY) {
      float4 hv[UNR][NR];
      float dv[UNR][4];
      uint2 av[UNR][NA];                                             // (ADD) bf16 addend of each input row
#pragma unroll
      for (int j = 0; j < UNR; ++j) {
        const size_t u = ub + (size_t)j * TY;
        if (u < u1) {
          const UnitRows ur = unit_rows(u, H, W, POOL);
#pragma unroll
          for (int k = 0; k < NR; ++k) hv[j][k] = __ldg(reinterpret_cast<const float4*>(h + ur.r[k] * ldh + c0));   // (re-read by the apply pass)
          if constexpr (ADD) {
#pragma unroll
            for (int k = 0; k < NR; ++k) av[j][k] = __ldg(reinterpret_cast<const uint2*>(dy_add + ur.r[k] * C + c0));
          }
          if (dy_f32) {
            const float4 q = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(dy) +
                                                                   dy_row<DYM>(u, ldy, POOL ? H >> 1 : H, POOL ? W >> 1 : W, C) + c0));
            dv[j][0] = q.x; dv[j][1] = q.y; dv[j][2] = q.z; dv[j][3] = q.w;
          } else {
            const uint2 q = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(dy) +
                                                                 dy_row<DYM>(u, ldy, POOL ? H >> 1 : H, POOL ? W >> 1 : W, C) + c0));
            const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162*>(&q.x), hi = *reinterpret_cast<const __nv_bfloat162*>(&q.y);
            dv[j][0] = __low2float(lo); dv[j][1] = __high2float(lo); dv[j][2] = __low2float(hi); dv[j][3] = __high2float(hi);
          }
        } else {
#pragma unroll
          for (int k = 0; k < NR; ++k) hv[j][k] = make_float4(0.f, 0.f, 0.f, 0.f);
          dv[j][0] = dv[j][1] = dv[j][2] = dv[j][3] = 0.0f;          // contributes nothing
          if constexpr (ADD) {
#pragma unroll
            for (int k = 0; k < NR; ++k) av[j][k] = make_uint2(0u, 0u);
          }
        }
      }
#pragma unroll
      for (int j = 0; j < UNR; ++j) {
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          if constexpr (ADD) {
            // every input row of the window has a gradient: the addend, plus the pooled dy at the first maximum; the sum
            // (float32) takes the row's own leaky slope
            float xs[NR], zs[NR], best = -INFINITY;
            int arg = 0;
#pragma unroll
            for (int k = 0; k < NR; ++k) {
              const float t = v == 0 ? hv[j][k].x : (v == 1 ? hv[j][k].y : (v == 2 ? hv[j][k].z : hv[j][k].w));
              xs[k] = (t - pm[v]) * pi[v];
              zs[k] = xs[k] * pg[v] + pb[v];
              const float a = leaky_on ? fmaxf(zs[k], alpha * zs[k]) : zs[k];
              if (a > best) { best = a; arg = k; }
            }
#pragma unroll
            for (int k = 0; k < NR; ++k) {
              const __nv_bfloat162 p = *reinterpret_cast<const __nv_bfloat162*>(v < 2 ? &av[j][k].x : &av[j][k].y);
              float d = ((v & 1) ? __high2float(p) : __low2float(p)) + (arg == k ? dv[j][v] : 0.0f);
              if (leaky_on && !(zs[k] > 0.0f)) d *= alpha;
              f[v] += d;
              f[4 + v] = fmaf(d, xs[k], f[4 + v]);
            }
          } else {
            float best = -INFINITY, bx = 0.0f, bz = 0.0f;
#pragma unroll
            for (int k = 0; k < NR; ++k) {
              const float t = v == 0 ? hv[j][k].x : (v == 1 ? hv[j][k].y : (v == 2 ? hv[j][k].z : hv[j][k].w));
              const float xh = (t - pm[v]) * pi[v];
              const float z = xh * pg[v] + pb[v];
              const float a = leaky_on ? fmaxf(z, alpha * z) : z;
              if (a > best) { best = a; bx = xh; bz = z; }
            }
            float d = dv[j][v];
            if (leaky_on && !(bz > 0.0f)) d *= alpha;
            f[v] += d;
            f[4 + v] = fmaf(d, bx, f[4 + v]);
          }
        }
      }
      if (++cnt == 8) {
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
  if (ty < 8 && c0 < C) {
    double a = 0.0;
    for (int y = 0; y < TY; ++y) a += sm[y][tx][ty];
    part[((size_t)blockIdx.y * C + c0 + (ty & 3)) * 2 + (ty >> 2)] = a;
  }
}
template <bool POOL, int TX>
__global__ void __launch_bounds__(256, 4) bn_bwd_reduce_v4_kernel(
    const float* __restrict__ h, int ldh, const void* __restrict__ dy, int dy_f32, const float* __restrict__ mean,
    const float* __restrict__ var, const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float alpha,
    int leaky_on, int H, int W, int C, size_t units, size_t units_per_split, double* __restrict__ part) {
  bn_bwd_reduce_v4_body<POOL, TX, DY_DENSE, false>(h, ldh, dy, dy_f32, C, nullptr, mean, var, gamma, beta, eps, alpha, leaky_on,
                                                   H, W, C, units, units_per_split, part);
}
template <bool POOL, int TX, int DYM, bool ADD>
__global__ void __launch_bounds__(256, 4) bn_bwd_reduce_v4_ex_kernel(
    const float* __restrict__ h, int ldh, const void* __restrict__ dy, int dy_f32, int ldy,
    const __nv_bfloat16* __restrict__ dy_add, const float* __restrict__ mean, const float* __restrict__ var,
    const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float alpha, int leaky_on, int H, int W, int C,
    size_t units, size_t units_per_split, double* __restrict__ part) {
  bn_bwd_reduce_v4_body<POOL, TX, DYM, ADD>(h, ldh, dy, dy_f32, ldy, dy_add, mean, var, gamma, beta, eps, alpha, leaky_on, H, W,
                                            C, units, units_per_split, part);
}

constexpr int BWD_FIN_TY = 32;   // thread rows folding the splits (8 rows walked up to 128 dependent L2 round trips: 22 us per layer)
__global__ void __launch_bounds__(32 * BWD_FIN_TY) bn_bwd_final_kernel(const double* __restrict__ part, int splits, int C, float* __restrict__ dgamma,
                                    float* __restrict__ dbeta) {
  __shared__ double s1[BWD_FIN_TY][33], s2[BWD_FIN_TY][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  double a1 = 0.0, a2 = 0.0;
  if (c < C) {
    double b1 = 0.0, b2 = 0.0, c1 = 0.0, c2 = 0.0, d1 = 0.0, d2 = 0.0;      // four independent loads in flight, fixed order
    int s = threadIdx.y;
    for (; s + 3 * BWD_FIN_TY < splits; s += 4 * BWD_FIN_TY) {
      const double2 p0 = *reinterpret_cast<const double2*>(part + ((size_t)s * C + c) * 2);
      const double2 p1 = *reinterpret_cast<const double2*>(part + ((size_t)(s + BWD_FIN_TY) * C + c) * 2);
      const double2 p2 = *reinterpret_cast<const double2*>(part + ((size_t)(s + 2 * BWD_FIN_TY) * C + c) * 2);
      const double2 p3 = *reinterpret_cast<const double2*>(part + ((size_t)(s + 3 * BWD_FIN_TY) * C + c) * 2);
      a1 += p0.x; a2 += p0.y; b1 += p1.x; b2 += p1.y; c1 += p2.x; c2 += p2.y; d1 += p3.x; d2 += p3.y;
    }
    for (; s < splits; s += BWD_FIN_TY) {
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
  for (int y = 1; y < BWD_FIN_TY; ++y) { a1 += s1[y][threadIdx.x]; a2 += s2[y][threadIdx.x]; }
  dbeta[c] = (float)a1;
  dgamma[c] = (float)a2;
}

// pass 2, fast path (C % 4 == 0, units < 2^31): a thread owns 4 channels -- their seven per-channel constants live in
// registers -- and walks units; 32-bit index arithmetic, 16-byte loads of the pre-BN rows, one 8/16-byte load of dy.
// The generic kernel below spent 3.5 ms of a 17.4 ms training step (ncu launch list) on 64-bit div/mod per element,
// scalar bf16 dy loads and six constant loads + two rsqrt per channel per element.
// DYM / ADD: the dy read of bn_bwd_reduce_kernel.
template <bool POOL, int DYM, bool ADD>
__device__ __forceinline__ void bn_bwd_apply_rows_body(
    const float* __restrict__ h, int ldh, const void* __restrict__ dy, int dy_f32, int ldy,
    const __nv_bfloat16* __restrict__ dy_add, const float* __restrict__ mean,
    const float* __restrict__ var, const float* __restrict__ gamma, const float* __restrict__ beta,
    const float* __restrict__ dgamma, const float* __restrict__ dbeta, float eps, float alpha, int leaky_on, int H, int W, int C,
    unsigned units, float invM, __nv_bfloat16* __restrict__ dh, int ld_dh) {
  const int cx = blockIdx.y * blockDim.x + threadIdx.x;          // group of 4 channels (incl. the zero padding columns)
  const int c0 = cx * 4;
  if (c0 >= ld_dh) return;
  const bool real = c0 < C;                                       // C % 4 == 0: a group is entirely real or entirely padding
  float mu[4], inv[4], ga[4], be[4], gi[4], m1[4], m2[4];
#pragma unroll
  for (int v = 0; v < 4; ++v) {
    const int c = real ? c0 + v : 0;
    mu[v] = mean[c]; inv[v] = rsqrtf(var[c] + eps); ga[v] = gamma[c]; be[v] = beta[c];
    gi[v] = real ? ga[v] * inv[v] : 0.0f;
    m1[v] = dbeta[c] * invM; m2[v] = dgamma[c] * invM;
  }
  const unsigned Wo = POOL ? (unsigned)W >> 1 : (unsigned)W, Ho = POOL ? (unsigned)H >> 1 : (unsigned)H;
  const unsigned ustep = gridDim.x * blockDim.y;
  // (un-pooled layers with four rows in flight per thread: measured no faster -- layer 3 304 -> 328 us -- not kept)
  for (unsigned u = blockIdx.x * blockDim.y + threadIdx.y; u < units; u += ustep) {
    size_t rows[POOL ? 4 : 1];
    if (POOL) {
      const unsigned wo = u % Wo, t = u / Wo, ho = t % Ho, n = t / Ho;
      const size_t base = ((size_t)n * H + 2 * ho) * (size_t)W + 2 * wo;
      rows[0] = base; rows[POOL ? 1 : 0] = base + 1; rows[POOL ? 2 : 0] = base + W; rows[POOL ? 3 : 0] = base + W + 1;
    } else {
      rows[0] = u;
    }
    constexpr int NP = POOL ? 4 : 1;
    float4 q[NP];
    if (real) {
#pragma unroll
      for (int k = 0; k < NP; ++k) q[k] = __ldcs(reinterpret_cast<const float4*>(h + rows[k] * ldh + c0));
    }
    float d[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    if (real) {
      if (dy_f32) {
        const float4 g = __ldcs(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(dy) +
                                                                dy_row<DYM>(u, ldy, (int)Ho, (int)Wo, C) + c0));
        d[0] = g.x; d[1] = g.y; d[2] = g.z; d[3] = g.w;
      } else {
        const uint2 g = __ldcs(reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(dy) +
                                                              dy_row<DYM>(u, ldy, (int)Ho, (int)Wo, C) + c0));
        const __nv_bfloat162 g0 = *reinterpret_cast<const __nv_bfloat162*>(&g.x), g1 = *reinterpret_cast<const __nv_bfloat162*>(&g.y);
        d[0] = __low2float(g0); d[1] = __high2float(g0); d[2] = __low2float(g1); d[3] = __high2float(g1);
      }
    }
    float xh[NP][4];
    int arg[4] = {0, 0, 0, 0};
    float abest[4], zbest[4];
    float zs[ADD ? NP : 1][4];                                      // (ADD) every row's z: each row takes its own slope
#pragma unroll
    for (int v = 0; v < 4; ++v) { abest[v] = -INFINITY; zbest[v] = 0.0f; }
#pragma unroll
    for (int k = 0; k < NP; ++k) {
      const float t[4] = {q[k].x, q[k].y, q[k].z, q[k].w};
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const float x_ = real ? (t[v] - mu[v]) * inv[v] : 0.0f;
        const float z = x_ * ga[v] + be[v];
        const float a = leaky_on ? fmaxf(z, alpha * z) : z;
        xh[k][v] = x_;
        if constexpr (ADD) zs[k][v] = z;
        if (a > abest[v]) { abest[v] = a; arg[v] = k; zbest[v] = z; }      // first maximum wins, as in the generic kernel
      }
    }
    if constexpr (ADD) {
      // every row's gradient: the addend, plus the pooled dy at the first maximum; the float32 sum takes the row's slope
#pragma unroll
      for (int k = 0; k < NP; ++k) {
        float a4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        if (real) {
          const uint2 g = __ldcs(reinterpret_cast<const uint2*>(dy_add + rows[k] * C + c0));
          const __nv_bfloat162 g0 = *reinterpret_cast<const __nv_bfloat162*>(&g.x), g1 = *reinterpret_cast<const __nv_bfloat162*>(&g.y);
          a4[0] = __low2float(g0); a4[1] = __high2float(g0); a4[2] = __low2float(g1); a4[3] = __high2float(g1);
        }
        float o[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          float dk = a4[v] + (arg[v] == k ? d[v] : 0.0f);
          if (leaky_on && !(zs[k][v] > 0.0f)) dk *= alpha;
          o[v] = gi[v] * (dk - m1[v] - xh[k][v] * m2[v]);
        }
        const __nv_bfloat162 a = __floats2bfloat162_rn(o[0], o[1]), b = __floats2bfloat162_rn(o[2], o[3]);
        uint2 pk;
        pk.x = *reinterpret_cast<const uint32_t*>(&a);
        pk.y = *reinterpret_cast<const uint32_t*>(&b);
        *reinterpret_cast<uint2*>(dh + rows[k] * ld_dh + c0) = pk;
      }
    } else {
#pragma unroll
      for (int v = 0; v < 4; ++v)
        if (leaky_on && !(zbest[v] > 0.0f)) d[v] *= alpha;
#pragma unroll
      for (int k = 0; k < NP; ++k) {
        float o[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) o[v] = gi[v] * ((arg[v] == k ? d[v] : 0.0f) - m1[v] - xh[k][v] * m2[v]);
        const __nv_bfloat162 a = __floats2bfloat162_rn(o[0], o[1]), b = __floats2bfloat162_rn(o[2], o[3]);
        uint2 pk;
        pk.x = *reinterpret_cast<const uint32_t*>(&a);
        pk.y = *reinterpret_cast<const uint32_t*>(&b);
        *reinterpret_cast<uint2*>(dh + rows[k] * ld_dh + c0) = pk;
      }
    }
  }
}
template <bool POOL>
__global__ void __launch_bounds__(256, 4) bn_bwd_apply_rows_kernel(
    const float* __restrict__ h, int ldh, const void* __restrict__ dy, int dy_f32, const float* __restrict__ mean,
    const float* __restrict__ var, const float* __restrict__ gamma, const float* __restrict__ beta,
    const float* __restrict__ dgamma, const float* __restrict__ dbeta, float eps, float alpha, int leaky_on, int H, int W, int C,
    unsigned units, float invM, __nv_bfloat16* __restrict__ dh, int ld_dh) {
  bn_bwd_apply_rows_body<POOL, DY_DENSE, false>(h, ldh, dy, dy_f32, C, nullptr, mean, var, gamma, beta, dgamma, dbeta, eps, alpha,
                                                leaky_on, H, W, C, units, invM, dh, ld_dh);
}
template <bool POOL, int DYM, bool ADD>
__global__ void __launch_bounds__(256, 4) bn_bwd_apply_rows_ex_kernel(
    const float* __restrict__ h, int ldh, const void* __restrict__ dy, int dy_f32, int ldy,
    const __nv_bfloat16* __restrict__ dy_add, const float* __restrict__ mean, const float* __restrict__ var,
    const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ dgamma,
    const float* __restrict__ dbeta, float eps, float alpha, int leaky_on, int H, int W, int C, unsigned units, float invM,
    __nv_bfloat16* __restrict__ dh, int ld_dh) {
  bn_bwd_apply_rows_body<POOL, DYM, ADD>(h, ldh, dy, dy_f32, ldy, dy_add, mean, var, gamma, beta, dgamma, dbeta, eps, alpha,
                                         leaky_on, H, W, C, units, invM, dh, ld_dh);
}

// pass 2: one thread per (unit, VEC channels); writes dh for every input pixel of the unit.
// DYM / ADD: the dy read of bn_bwd_reduce_kernel.
template <int VEC, int DYM, bool ADD>
__device__ __forceinline__ void bn_bwd_apply_body(const float* __restrict__ h, int ldh, const void* __restrict__ dy, int dy_f32, int ldy,
                                    const __nv_bfloat16* __restrict__ dy_add, const float* __restrict__ mean, const float* __restrict__ var,
                                    const float* __restrict__ gamma, const float* __restrict__ beta,
                                    const float* __restrict__ dgamma, const float* __restrict__ dbeta, float eps,
                                    float alpha, int leaky_on, int pool, int H, int W, int C, size_t units, float invM,
                                    __nv_bfloat16* __restrict__ dh, int ld_dh) {
  const int CV = ld_dh / VEC;                       // channel groups incl. the zero padding columns
  const size_t total = units * CV;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int cv = (int)(i % CV);
    const size_t u = i / CV;
    const int c0 = cv * VEC;
    const UnitRows ur = unit_rows(u, H, W, pool != 0);
    float xh[4][VEC];
    float zs[ADD ? 4 : 1][VEC];                      // (ADD) every row's z: each row takes its own slope
    int arg[VEC];
    float zbest[VEC], abest[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) { arg[v] = 0; abest[v] = -INFINITY; zbest[v] = 0.0f; }
    for (int k = 0; k < ur.n; ++k) {
      float t[VEC];
      const float* px = h + ur.r[k] * ldh + c0;
      if (VEC == 4 && c0 + 3 < C) {
        const float4 q = *reinterpret_cast<const float4*>(px);
        t[0] = q.x; t[1 % VEC] = q.y; t[2 % VEC] = q.z; t[3 % VEC] = q.w;
      } else {
#pragma unroll
        for (int v = 0; v < VEC; ++v) t[v] = (c0 + v < C) ? px[v] : 0.0f;
      }
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        const int c = c0 + v;
        if (c < C) {
          const float x_ = (t[v] - mean[c]) * rsqrtf(var[c] + eps);
          const float z = x_ * gamma[c] + beta[c];
          const float a = leaky_on ? fmaxf(z, alpha * z) : z;
          xh[k][v] = x_;
          if constexpr (ADD) zs[k][v] = z;
          if (a > abest[v]) { abest[v] = a; arg[v] = k; zbest[v] = z; }
        } else {
          xh[k][v] = 0.0f;
          if constexpr (ADD) zs[k][v] = 0.0f;
        }
      }
    }
    float d[VEC], gi[VEC], m1[VEC], m2[VEC];
    if constexpr (ADD) {
      // every row's gradient: the addend, plus the pooled dy at the first maximum; the float32 sum takes the row's slope
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        const int c = c0 + v;
        d[v] = c < C ? load_dy(dy, dy_f32, dy_row<DYM>(u, ldy, pool ? H >> 1 : H, pool ? W >> 1 : W, C) + c) : 0.0f;
        gi[v] = c < C ? gamma[c] * rsqrtf(var[c] + eps) : 0.0f;
        m1[v] = c < C ? dbeta[c] * invM : 0.0f;
        m2[v] = c < C ? dgamma[c] * invM : 0.0f;
      }
      for (int k = 0; k < ur.n; ++k) {
        __nv_bfloat16* po = dh + ur.r[k] * ld_dh + c0;
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          const int c = c0 + v;
          float dk = c < C ? __bfloat162float(dy_add[ur.r[k] * C + c]) + (arg[v] == k ? d[v] : 0.0f) : 0.0f;
          if (leaky_on && !(zs[k][v] > 0.0f)) dk *= alpha;
          po[v] = __float2bfloat16_rn(gi[v] * (dk - m1[v] - xh[k][v] * m2[v]));
        }
      }
    } else {
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        const int c = c0 + v;
        if (c < C) {
          float g = load_dy(dy, dy_f32, dy_row<DYM>(u, ldy, pool ? H >> 1 : H, pool ? W >> 1 : W, C) + c);
          if (leaky_on && !(zbest[v] > 0.0f)) g *= alpha;
          d[v] = g;
          gi[v] = gamma[c] * rsqrtf(var[c] + eps);
          m1[v] = dbeta[c] * invM;
          m2[v] = dgamma[c] * invM;
        } else {
          d[v] = 0.0f; gi[v] = 0.0f; m1[v] = 0.0f; m2[v] = 0.0f;
        }
      }
      for (int k = 0; k < ur.n; ++k) {
        float o[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) o[v] = gi[v] * ((arg[v] == k ? d[v] : 0.0f) - m1[v] - xh[k][v] * m2[v]);
        __nv_bfloat16* po = dh + ur.r[k] * ld_dh + c0;
        if (VEC == 4) {
          __nv_bfloat162 a = __floats2bfloat162_rn(o[0], o[1 % VEC]);
          __nv_bfloat162 b = __floats2bfloat162_rn(o[2 % VEC], o[3 % VEC]);
          uint2 pk;
          pk.x = *reinterpret_cast<uint32_t*>(&a);
          pk.y = *reinterpret_cast<uint32_t*>(&b);
          *reinterpret_cast<uint2*>(po) = pk;
        } else {
#pragma unroll
          for (int v = 0; v < VEC; ++v) po[v] = __float2bfloat16_rn(o[v]);
        }
      }
    }
  }
}
template <int VEC>
__global__ void bn_bwd_apply_kernel(const float* __restrict__ h, int ldh, const void* __restrict__ dy, int dy_f32,
                                    const float* __restrict__ mean, const float* __restrict__ var,
                                    const float* __restrict__ gamma, const float* __restrict__ beta,
                                    const float* __restrict__ dgamma, const float* __restrict__ dbeta, float eps,
                                    float alpha, int leaky_on, int pool, int H, int W, int C, size_t units, float invM,
                                    __nv_bfloat16* __restrict__ dh, int ld_dh) {
  bn_bwd_apply_body<VEC, DY_DENSE, false>(h, ldh, dy, dy_f32, C, nullptr, mean, var, gamma, beta, dgamma, dbeta, eps, alpha,
                                          leaky_on, pool, H, W, C, units, invM, dh, ld_dh);
}
template <int VEC, int DYM, bool ADD>
__global__ void bn_bwd_apply_ex_kernel(const float* __restrict__ h, int ldh, const void* __restrict__ dy, int dy_f32, int ldy,
                                       const __nv_bfloat16* __restrict__ dy_add, const float* __restrict__ mean,
                                       const float* __restrict__ var, const float* __restrict__ gamma,
                                       const float* __restrict__ beta, const float* __restrict__ dgamma,
                                       const float* __restrict__ dbeta, float eps, float alpha, int leaky_on, int pool, int H,
                                       int W, int C, size_t units, float invM, __nv_bfloat16* __restrict__ dh, int ld_dh) {
  bn_bwd_apply_body<VEC, DYM, ADD>(h, ldh, dy, dy_f32, ldy, dy_add, mean, var, gamma, beta, dgamma, dbeta, eps, alpha, leaky_on,
                                   pool, H, W, C, units, invM, dh, ld_dh);
}

// ---------------------------------------------------------------------------------------------
// dgrad weights: conv'(dh)[n,h,w,ci] = sum_{kh',kw',co} dh[n, h+kh'-p, w+kw'-p, co] * W[k-1-kh', k-1-kw', ci, co]
// packed like y2_pack_weights_bf16 for a convolution with Cin' = ld_dh (>= Cout, zero columns beyond Cout)
// and Cout' = Cin:   out[ci][tap' * ld_dh + co]
// ---------------------------------------------------------------------------------------------
__global__ void pack_weights_dgrad_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int taps, int Cin,
                                          int Cout, int cinp_rows, int ld_dh) {
  const int Kp = taps * ld_dh;
  const size_t total = (size_t)cinp_rows * Kp;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int ci = (int)(i / Kp);
    const int kk = (int)(i % Kp);
    const int tapf = kk / ld_dh, co = kk % ld_dh;
    const int tap = taps - 1 - tapf;                 // (k-1-kh')*k + (k-1-kw') == taps-1-tap'
    float v = 0.0f;
    if (ci < Cin && co < Cout) v = w[((size_t)tap * Cin + ci) * Cout + co];
    out[i] = __float2bfloat16_rn(v);
  }
}

// Same packing, one block per (ci, tap'), 8 output channels per thread: 32-byte reads, 16-byte writes, no 64-bit div/mod per
// element (the generic kernel above took 235 us of a training step for the 48 M weights).  ld_dh % 8 == 0.
__global__ void __launch_bounds__(128) pack_weights_dgrad_v8_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int taps,
                                                                   int Cin, int Cout, int ld_dh) {
  const int ci = blockIdx.x, tapf = blockIdx.y, tap = taps - 1 - tapf;
  const float* src = w + ((size_t)tap * Cin + ci) * Cout;
  __nv_bfloat16* dst = out + ((size_t)ci * taps + tapf) * ld_dh;
  const bool row_ok = ci < Cin;
  const bool vec_ok = (Cout % 4 == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
  for (int c8 = threadIdx.x; c8 * 8 < ld_dh; c8 += blockDim.x) {
    const int co = c8 * 8;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.0f;
    if (row_ok) {
      if (vec_ok && co + 8 <= Cout) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(src + co)), b = __ldg(reinterpret_cast<const float4*>(src + co + 4));
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (co + i < Cout) v[i] = src[co + i];
      }
    }
    const __nv_bfloat162 h0 = __floats2bfloat162_rn(v[0], v[1]), h1 = __floats2bfloat162_rn(v[2], v[3]);
    const __nv_bfloat162 h2 = __floats2bfloat162_rn(v[4], v[5]), h3 = __floats2bfloat162_rn(v[6], v[7]);
    *reinterpret_cast<uint4*>(dst + co) = make_uint4(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1),
                                                     *reinterpret_cast<const uint32_t*>(&h2), *reinterpret_cast<const uint32_t*>(&h3));
  }
}

// ---------------------------------------------------------------------------------------------
// first-layer weight gradient: x bf16 [N,H,W,8] (channels 0..2 real), dh bf16 [N*H*W, ld_dh], Cout <= 32.
// dW[kh][kw][ci][co] += sum_pixels x[n, h+kh-1, w+kw-1, ci] * dh[n,h,w,co]
// Persistent CTAs over 8 x 32 pixel tiles; warp = tile row, lane = co; 27 register accumulators per lane;
// the x halo row slides through registers (3 new smem loads per pixel instead of 9).
// ---------------------------------------------------------------------------------------------
constexpr int W1_TH = 8, W1_TW = 32;

__global__ void __launch_bounds__(256) conv_wgrad_c3_kernel(const __nv_bfloat16* __restrict__ x,
                                                            const __nv_bfloat16* __restrict__ dh, int ld_dh, int N, int H,
                                                            int W, int Cout, float* __restrict__ dw) {
  __shared__ __align__(16) uint2 s_x[W1_TH + 2][W1_TW + 2];          // 4 bf16 per pixel (ch 0..3)
  __shared__ __align__(16) __nv_bfloat16 s_dh[W1_TH][W1_TW][32];
  __shared__ float s_red[8][27][33];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tiles_w = (W + W1_TW - 1) / W1_TW, tiles_h = (H + W1_TH - 1) / W1_TH;
  const int total = N * tiles_h * tiles_w;
  float acc[27];
#pragma unroll
  for (int i = 0; i < 27; ++i) acc[i] = 0.0f;
  for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const int tw = tile % tiles_w, th = (tile / tiles_w) % tiles_h, n = tile / (tiles_w * tiles_h);
    const int h0 = th * W1_TH, w0 = tw * W1_TW;
    __syncthreads();
    for (int i = tid; i < (W1_TH + 2) * (W1_TW + 2); i += 256) {
      const int r = i / (W1_TW + 2), cidx = i % (W1_TW + 2);
      const int hh = h0 + r - 1, ww = w0 + cidx - 1;
      uint2 v = make_uint2(0u, 0u);
      if (hh >= 0 && hh < H && ww >= 0 && ww < W)
        v = *reinterpret_cast<const uint2*>(x + ((size_t)(n * H + hh) * W + ww) * 8);
      s_x[r][cidx] = v;
    }
    for (int i = tid; i < W1_TH * W1_TW * 4; i += 256) {             // 4 x 16-byte chunks per pixel
      const int p = i >> 2, q = i & 3;
      const int r = p / W1_TW, cidx = p % W1_TW;
      const int hh = h0 + r, ww = w0 + cidx;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (hh < H && ww < W && q * 8 < ld_dh)
        v = *reinterpret_cast<const uint4*>(dh + ((size_t)(n * H + hh) * W + ww) * ld_dh + q * 8);
      *reinterpret_cast<uint4*>(&s_dh[r][cidx][q * 8]) = v;
    }
    __syncthreads();
    // warp = tile row; slide a 3-row x 3-column window of x along the row
    float xw[3][3][3];                                               // [kh][kw][ci]
#pragma unroll
    for (int kh = 0; kh < 3; ++kh)
#pragma unroll
      for (int kw = 0; kw < 2; ++kw) {
        const uint2 v = s_x[warp + kh][kw];
        const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&v.x);
        const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&v.y);
        xw[kh][kw + 1][0] = __low2float(a); xw[kh][kw + 1][1] = __high2float(a); xw[kh][kw + 1][2] = __low2float(b);
      }
#pragma unroll 4
    for (int p = 0; p < W1_TW; ++p) {
#pragma unroll
      for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
        for (int ci = 0; ci < 3; ++ci) { xw[kh][0][ci] = xw[kh][1][ci]; xw[kh][1][ci] = xw[kh][2][ci]; }
        const uint2 v = s_x[warp + kh][p + 2];
        const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&v.x);
        const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&v.y);
        xw[kh][2][0] = __low2float(a); xw[kh][2][1] = __high2float(a); xw[kh][2][2] = __low2float(b);
      }
      const float g = __bfloat162float(s_dh[warp][p][lane]);
#pragma unroll
      for (int kh = 0; kh < 3; ++kh)
#pragma unroll
        for (int kw = 0; kw < 3; ++kw)
#pragma unroll
          for (int ci = 0; ci < 3; ++ci) acc[(kh * 3 + kw) * 3 + ci] = fmaf(xw[kh][kw][ci], g, acc[(kh * 3 + kw) * 3 + ci]);
    }
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 27; ++i) s_red[warp][i][lane] = acc[i];
  __syncthreads();
  for (int i = tid; i < 27 * 32; i += 256) {
    const int k = i >> 5, co = i & 31;
    float s = 0.0f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) s += s_red[w8][k][co];
    if (co < Cout) atomicAdd(dw + (size_t)k * Cout + co, s);
  }
}

// The same weight gradient on the warp-level tensor-core instruction (mma.sync.m16n8k16, bf16 x bf16 -> f32): the FFMA
// kernel above issues 27 FMAs + ~45 bookkeeping instructions per pixel and lane (1.0 ms of the 14.5 ms training step for
// 19 GFLOP -- a quarter of the FP32 peak), while the GEMM  D[(tap, ci) = 27 -> 32, co = 32] += A[m][pixel] * B[pixel][co]
// is 8 MMAs per 16 pixels and warp.  tcgen05 cannot tile it (M = 27, K = 11 M pixels, both operands pixel-major), the
// synchronous warp MMA can, and at 0.9 GB of operands the kernel is then HBM-bound (~0.15 ms).
//   smem   x halo tile as bf16 CHANNEL PLANES [ci][10 rows][40], once as is and once shifted by one pixel, so that the two
//          consecutive pixels an A fragment register holds are one aligned 32-bit load for every horizontal tap;
//          dh tile [8 rows][32 px][40 (32 co + pad)] read with ldmatrix.trans (B is pixel-major in memory).
//   warp = tile row (32 pixels = two K blocks); 2 M tiles x 4 N tiles of accumulators per thread; CTA-level reduction
//   through smem, then one atomicAdd per (tap, ci, co) and CTA, as above.
__device__ __forceinline__ void mma_bf16_16816(float* d, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

constexpr int W1_XP = 40;                         // plane pitch (bf16): 34 used, 32-bit loads at even offsets
constexpr int W1_DP = 40;                         // dh row pitch (bf16): 32 co + 8 pad -> conflict-free ldmatrix rows

__global__ void __launch_bounds__(256) conv_wgrad_c3_mma_kernel(const __nv_bfloat16* __restrict__ x,
                                                                const __nv_bfloat16* __restrict__ dh, int ld_dh, int N, int H,
                                                                int W, int Cout, float* __restrict__ dw) {
  // operands and the final cross-warp reduction share one buffer (static shared memory is capped at 48 KB)
  constexpr int SX_ELEMS = 2 * 3 * (W1_TH + 2) * W1_XP, SDH_ELEMS = W1_TH * W1_TW * W1_DP;
  constexpr size_t OPERAND_BYTES = (size_t)(SX_ELEMS + SDH_ELEMS) * 2, RED_BYTES = (size_t)8 * 32 * 33 * 4;
  __shared__ __align__(16) unsigned char s_raw[OPERAND_BYTES > RED_BYTES ? OPERAND_BYTES : RED_BYTES];
  typedef __nv_bfloat16 (*SxT)[3][W1_TH + 2][W1_XP];              // [copy: 0 as is, 1 shifted left by one][ci][row][col]
  typedef __nv_bfloat16 (*SdhT)[W1_TW][W1_DP];
  typedef float (*SredT)[32][33];
  SxT s_x = reinterpret_cast<SxT>(s_raw);
  SdhT s_dh = reinterpret_cast<SdhT>(s_raw + (size_t)SX_ELEMS * 2);
  SredT s_red = reinterpret_cast<SredT>(s_raw);
  static_assert(((size_t)SX_ELEMS * 2) % 16 == 0, "dh tile must stay 16-byte aligned");
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int tiles_w = (W + W1_TW - 1) / W1_TW, tiles_h = (H + W1_TH - 1) / W1_TH;
  const int total = N * tiles_h * tiles_w;
  // per-thread A rows: m = mt * 16 + g + 8 * h  ->  (kh, kw, ci); element offset of the pixel pair (2t, 2t + 1) at p0 = 0
  int a_off[2][2];
  bool a_ok[2][2];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int m = mt * 16 + g + 8 * h;
      a_ok[mt][h] = m < 27;
      const int tap = m / 3, ci = m - tap * 3, kh = tap / 3, kw = tap - kh * 3;
      const int copy = kw == 1 ? 1 : 0, sh = kw == 2 ? 2 : 0;
      a_off[mt][h] = a_ok[mt][h] ? ((copy * 3 + ci) * (W1_TH + 2) + kh) * W1_XP + sh + 2 * t : 0;
    }
  float acc[2][4][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int k = 0; k < 4; ++k) acc[i][j][k] = 0.0f;
  const __nv_bfloat16* sx0 = &s_x[0][0][0][0];
  for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const int tw = tile % tiles_w, th = (tile / tiles_w) % tiles_h, n = tile / (tiles_w * tiles_h);
    const int h0 = th * W1_TH, w0 = tw * W1_TW;
    __syncthreads();
    for (int i = tid; i < (W1_TH + 2) * (W1_TW + 2); i += 256) {
      const int r = i / (W1_TW + 2), cidx = i % (W1_TW + 2);
      const int hh = h0 + r - 1, ww = w0 + cidx - 1;
      uint2 v = make_uint2(0u, 0u);
      if (hh >= 0 && hh < H && ww >= 0 && ww < W)
        v = *reinterpret_cast<const uint2*>(x + ((size_t)(n * H + hh) * W + ww) * 8);
      const __nv_bfloat16* e = reinterpret_cast<const __nv_bfloat16*>(&v);
#pragma unroll
      for (int ci = 0; ci < 3; ++ci) {
        s_x[0][ci][r][cidx] = e[ci];
        if (cidx > 0) s_x[1][ci][r][cidx - 1] = e[ci];
      }
    }
    for (int i = tid; i < W1_TH * W1_TW * 4; i += 256) {             // 4 x 16-byte chunks per pixel
      const int p = i >> 2, q = i & 3;
      const int r = p / W1_TW, cidx = p % W1_TW;
      const int hh = h0 + r, ww = w0 + cidx;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (hh < H && ww < W && q * 8 < ld_dh)
        v = *reinterpret_cast<const uint4*>(dh + ((size_t)(n * H + hh) * W + ww) * ld_dh + q * 8);
      *reinterpret_cast<uint4*>(&s_dh[r][cidx][q * 8]) = v;
    }
    __syncthreads();
#pragma unroll
    for (int kb = 0; kb < 2; ++kb) {                                  // two blocks of 16 pixels of this warp's row
      const int p0 = kb * 16;
      uint32_t a[2][4];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const __nv_bfloat16* q = sx0 + a_off[mt][h] + warp * W1_XP + p0;
          const uint32_t lo = *reinterpret_cast<const uint32_t*>(q), hi = *reinterpret_cast<const uint32_t*>(q + 8);
          a[mt][h] = a_ok[mt][h] ? lo : 0u;                           // a0 / a1: pixels p0 + 2t, + 1
          a[mt][2 + h] = a_ok[mt][h] ? hi : 0u;                       // a2 / a3: pixels p0 + 2t + 8, + 9
        }
      // B fragments: ldmatrix.x4.trans over [16 pixels][16 co]: matrices (k 0-7, n 0-7) (k 8-15, n 0-7) (k 0-7, n 8-15) (k 8-15, n 8-15)
#pragma unroll
      for (int nb = 0; nb < 2; ++nb) {
        const int mi = lane >> 3, rr = lane & 7;
        const __nv_bfloat16* rowp = &s_dh[warp][p0 + (mi & 1) * 8 + rr][nb * 16 + (mi >> 1) * 8];
        uint32_t b[4];
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
                     : "=r"(b[0]), "=r"(b[1]), "=r"(b[2]), "=r"(b[3]) : "r"((uint32_t)__cvta_generic_to_shared(rowp)));
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          mma_bf16_16816(acc[mt][nb * 2 + 0], a[mt], b[0], b[1]);
          mma_bf16_16816(acc[mt][nb * 2 + 1], a[mt], b[2], b[3]);
        }
      }
    }
  }
  __syncthreads();
  // accumulator (mt, j, e): m = mt * 16 + g + 8 * (e >> 1), co = j * 8 + 2 t + (e & 1)
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) s_red[warp][mt * 16 + g + 8 * (e >> 1)][j * 8 + 2 * t + (e & 1)] = acc[mt][j][e];
  __syncthreads();
  for (int i = tid; i < 27 * 32; i += 256) {
    const int k = i >> 5, co = i & 31;
    float s = 0.0f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) s += s_red[w8][k][co];
    if (co < Cout) atomicAdd(dw + (size_t)k * Cout + co, s);
  }
}

// column sums of a bf16 matrix [M, ld] -> out[C] (+=): conv bias gradient
__global__ void sum_rows_bf16_kernel(const __nv_bfloat16* __restrict__ a, int ld, size_t M, int C, size_t rows_per_block,
                                     float* __restrict__ out) {
  __shared__ float s[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const size_t r0 = (size_t)blockIdx.y * rows_per_block, r1 = min(M, r0 + rows_per_block);
  float acc = 0.0f;
  if (c < C)
    for (size_t r = r0 + threadIdx.y; r < r1; r += 8) acc += __bfloat162float(a[r * ld + c]);
  s[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    for (int y = 1; y < 8; ++y) acc += s[y][threadIdx.x];
    atomicAdd(out + c, acc);
  }
}

static int bwd_splits(size_t units) {
  size_t s = (units + 127) / 128;
  return (int)(s > 1024 ? 1024 : (s < 1 ? 1 : s));
}

// The launches of y2_bn_leaky_pool_bwd_ex for one dy read mode (arguments checked by the caller).
template <int DYM, bool ADD>
static int bn_bwd_launch(const float* h_raw, int ldh, const void* dy, int dy_dtype, int ldy, const __nv_bfloat16* dy_add,
                         const float* mean, const float* var, const float* gamma, const float* beta, float eps, float alpha,
                         int leaky_on, int pool, int H, int W, int C, size_t M, size_t units, float* dgamma, float* dbeta,
                         void* dh_bf16, int ld_dh, void* workspace, y2_stream_t stream) {
  constexpr bool DENSE = DYM == DY_DENSE && !ADD;         // the mode of y2_bn_leaky_pool_bwd: its own kernels
  cudaStream_t st = (cudaStream_t)stream;
  int splits = bwd_splits(units);
  size_t ups = (units + splits - 1) / splits;
  splits = (int)((units + ups - 1) / ups);
  if (C % 4 == 0 && ldh % 4 == 0 && (((uintptr_t)h_raw) & 15) == 0 && (((uintptr_t)dy) & 15) == 0 && ldy % 4 == 0 &&
      (((uintptr_t)dy_add) & 7) == 0) {
    const int cg = C / 4;
    {   // one wave of blocks (see bn_stats_impl); tiles are dealt round-robin, so any number of splits is balanced
      const int tx = cg <= 8 ? 8 : (cg <= 16 ? 16 : 32);
      const int wave = num_sms() * 4 / ((cg + tx - 1) / tx);
      if (splits > wave) splits = wave > 1 ? wave : 1;
    }
#define Y2_LAUNCH_RED(POOL_, TX_)                                                                                     \
  if constexpr (DENSE)                                                                                                \
    bn_bwd_reduce_v4_kernel<POOL_, TX_><<<dim3((cg + TX_ - 1) / TX_, splits), 256, 0, st>>>(                          \
        h_raw, ldh, dy, dy_dtype == 0, mean, var, gamma, beta, eps, alpha, leaky_on, H, W, C, units, ups, (double*)workspace); \
  else                                                                                                                \
    bn_bwd_reduce_v4_ex_kernel<POOL_, TX_, DYM, ADD><<<dim3((cg + TX_ - 1) / TX_, splits), 256, 0, st>>>(             \
        h_raw, ldh, dy, dy_dtype == 0, ldy, dy_add, mean, var, gamma, beta, eps, alpha, leaky_on, H, W, C, units, ups,        \
        (double*)workspace)
    if (pool) { if (cg <= 8) { Y2_LAUNCH_RED(true, 8); } else if (cg <= 16) { Y2_LAUNCH_RED(true, 16); } else { Y2_LAUNCH_RED(true, 32); } }
    else      { if (cg <= 8) { Y2_LAUNCH_RED(false, 8); } else if (cg <= 16) { Y2_LAUNCH_RED(false, 16); } else { Y2_LAUNCH_RED(false, 32); } }
#undef Y2_LAUNCH_RED
  } else {
    dim3 grid((C + 31) / 32, splits), block(32, 8);
    if constexpr (DENSE)
      bn_bwd_reduce_kernel<<<grid, block, 0, st>>>(h_raw, ldh, dy, dy_dtype == 0, mean, var, gamma, beta, eps, alpha, leaky_on,
                                                   pool, H, W, C, units, ups, (double*)workspace);
    else
      bn_bwd_reduce_ex_kernel<DYM, ADD><<<grid, block, 0, st>>>(h_raw, ldh, dy, dy_dtype == 0, ldy, dy_add, mean, var, gamma,
                                                                beta, eps, alpha, leaky_on, pool, H, W, C, units, ups,
                                                                (double*)workspace);
  }
  Y2_LAUNCHED();
  bn_bwd_final_kernel<<<(C + 31) / 32, dim3(32, BWD_FIN_TY), 0, st>>>((const double*)workspace, splits, C, dgamma, dbeta);
  Y2_LAUNCHED();
  const bool vec4 = (ld_dh % 4 == 0) && (ldh % 4 == 0) && (((uintptr_t)h_raw & 15) == 0) && (((uintptr_t)dh_bf16 & 7) == 0);
  const float invM = 1.0f / (float)M;
#define Y2_LAUNCH_APPLY(VEC_)                                                                                         \
  if constexpr (DENSE)                                                                                                \
    bn_bwd_apply_kernel<VEC_><<<(int)g, 256, 0, st>>>(h_raw, ldh, dy, dy_dtype == 0, mean, var, gamma, beta, dgamma, dbeta, \
                                                      eps, alpha, leaky_on, pool, H, W, C, units, invM,                     \
                                                      (__nv_bfloat16*)dh_bf16, ld_dh);                                      \
  else                                                                                                                \
    bn_bwd_apply_ex_kernel<VEC_, DYM, ADD><<<(int)g, 256, 0, st>>>(h_raw, ldh, dy, dy_dtype == 0, ldy, dy_add, mean, var,   \
                                                                   gamma, beta, dgamma, dbeta, eps, alpha, leaky_on, pool,  \
                                                                   H, W, C, units, invM, (__nv_bfloat16*)dh_bf16, ld_dh)
  if (vec4 && C % 4 == 0 && units < (1ull << 31) && (((uintptr_t)dy) & 15) == 0 && ldy % 4 == 0 &&
      (((uintptr_t)dy_add) & 7) == 0 && !env().bn_bwd_generic) {
    const int cg = ld_dh / 4;
    const int bx = cg >= 64 ? 64 : (cg >= 32 ? 32 : (cg >= 16 ? 16 : 8));        // channel-group lanes per block
    const int by = 256 / bx;
    long long gx = 148ll * 16 / ((cg + bx - 1) / bx);
    const long long need = ((long long)units + by - 1) / by;
    if (gx > need) gx = need;
    if (gx < 1) gx = 1;
    const dim3 grid((unsigned)gx, (unsigned)((cg + bx - 1) / bx)), block(bx, by);
#define Y2_LAUNCH_ROWS(POOL_)                                                                                         \
  if constexpr (DENSE)                                                                                                \
    bn_bwd_apply_rows_kernel<POOL_><<<grid, block, 0, st>>>(h_raw, ldh, dy, dy_dtype == 0, mean, var, gamma, beta, dgamma,   \
                                                            dbeta, eps, alpha, leaky_on, H, W, C, (unsigned)units, invM,    \
                                                            (__nv_bfloat16*)dh_bf16, ld_dh);                                \
  else                                                                                                                \
    bn_bwd_apply_rows_ex_kernel<POOL_, DYM, ADD><<<grid, block, 0, st>>>(h_raw, ldh, dy, dy_dtype == 0, ldy, dy_add, mean,   \
                                                                         var, gamma, beta, dgamma, dbeta, eps, alpha,       \
                                                                         leaky_on, H, W, C, (unsigned)units, invM,          \
                                                                         (__nv_bfloat16*)dh_bf16, ld_dh)
    if (pool) {
      Y2_LAUNCH_ROWS(true);
    } else {
      Y2_LAUNCH_ROWS(false);
    }
#undef Y2_LAUNCH_ROWS
  } else if (vec4) {
    size_t total = units * (ld_dh / 4);
    size_t g = (total + 255) / 256;
    if (g > 148 * 32) g = 148 * 32;
    Y2_LAUNCH_APPLY(4);
  } else {
    size_t total = units * ld_dh;
    size_t g = (total + 255) / 256;
    if (g > 148 * 32) g = 148 * 32;
    Y2_LAUNCH_APPLY(1);
  }
#undef Y2_LAUNCH_APPLY
  Y2_LAUNCHED();
  return Y2_OK;
}

}  // namespace y2

using namespace y2;

extern "C" {

size_t y2_bn_bwd_workspace_bytes(int M, int C) { return (size_t)bwd_splits((size_t)M) * C * 2 * sizeof(double); }

int y2_bn_leaky_pool_bwd_ex(const float* h_raw, int ldh, const void* dy, int dy_dtype, int ldy, int dy_s2d,
                            const void* dy_add, const float* mean, const float* var, const float* gamma, const float* beta,
                            float eps, float alpha, int leaky_on, int pool, int N, int H, int W, int C, float* dgamma,
                            float* dbeta, void* dh_bf16, int ld_dh, void* workspace, size_t workspace_bytes,
                            y2_stream_t stream) {
  Y2_ARG(h_raw && dy && mean && var && gamma && beta && dgamma && dbeta && dh_bf16);
  Y2_ARG(N > 0 && H > 0 && W > 0 && C > 0 && ldh >= C && ld_dh >= C && (dy_dtype == 0 || dy_dtype == 1));
  if (pool) Y2_ARG(H % 2 == 0 && W % 2 == 0);
  Y2_ARG(ldy >= (dy_s2d ? 4 * C : C));
  if (dy_s2d) Y2_ARG(!pool && H % 2 == 0 && W % 2 == 0);
  if (dy_add) Y2_ARG(pool);
  const size_t M = (size_t)N * H * W;
  const size_t units = pool ? M / 4 : M;
  if (!workspace || workspace_bytes < y2_bn_bwd_workspace_bytes((int)M, C)) {
    set_error("y2_bn_leaky_pool_bwd: workspace too small (%zu < %zu)", workspace_bytes, y2_bn_bwd_workspace_bytes((int)M, C));
    return Y2_ERR_WORKSPACE;
  }
  Y2_ARG(((uintptr_t)workspace & 15) == 0);
  const __nv_bfloat16* add = (const __nv_bfloat16*)dy_add;
#define Y2_BN_BWD(DYM_, ADD_)                                                                                          \
  return bn_bwd_launch<DYM_, ADD_>(h_raw, ldh, dy, dy_dtype, ldy, add, mean, var, gamma, beta, eps, alpha, leaky_on, pool, H, \
                                   W, C, M, units, dgamma, dbeta, dh_bf16, ld_dh, workspace, stream)
  if (dy_s2d) Y2_BN_BWD(DY_S2D, false);
  if (add) { if (ldy == C) Y2_BN_BWD(DY_DENSE, true); else Y2_BN_BWD(DY_ROWS, true); }
  if (ldy == C) Y2_BN_BWD(DY_DENSE, false);
  Y2_BN_BWD(DY_ROWS, false);
#undef Y2_BN_BWD
}

int y2_bn_leaky_pool_bwd(const float* h_raw, int ldh, const void* dy, int dy_dtype, const float* mean, const float* var,
                         const float* gamma, const float* beta, float eps, float alpha, int leaky_on, int pool, int N,
                         int H, int W, int C, float* dgamma, float* dbeta, void* dh_bf16, int ld_dh, void* workspace,
                         size_t workspace_bytes, y2_stream_t stream) {
  return y2_bn_leaky_pool_bwd_ex(h_raw, ldh, dy, dy_dtype, C, 0, nullptr, mean, var, gamma, beta, eps, alpha, leaky_on, pool,
                                 N, H, W, C, dgamma, dbeta, dh_bf16, ld_dh, workspace, workspace_bytes, stream);
}

size_t y2_conv_packed_weight_dgrad_elems(int ksize, int Cin, int ld_dh) {
  const int rows = (Cin + 15) / 16 * 16;
  return (size_t)rows * ksize * ksize * ld_dh;
}

int y2_pack_weights_dgrad_bf16(const float* w_hwio, void* w_packed, int ksize, int Cin, int Cout, int ld_dh,
                               y2_stream_t stream) {
  Y2_ARG(w_hwio && w_packed && (ksize == 1 || ksize == 3) && Cin > 0 && Cout > 0 && ld_dh >= Cout && ld_dh % 32 == 0);
  const int rows = (Cin + 15) / 16 * 16;
  const size_t total = (size_t)rows * ksize * ksize * ld_dh;
  size_t g = (total + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  if ((reinterpret_cast<uintptr_t>(w_packed) & 15) == 0 && !env().bn_bwd_generic)
    pack_weights_dgrad_v8_kernel<<<dim3((unsigned)rows, (unsigned)(ksize * ksize)), (ld_dh / 8 >= 128 ? 128 : ((ld_dh / 8 + 31) / 32 * 32)), 0,
                                   (cudaStream_t)stream>>>(w_hwio, (__nv_bfloat16*)w_packed, ksize * ksize, Cin, Cout, ld_dh);
  else
    pack_weights_dgrad_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(w_hwio, (__nv_bfloat16*)w_packed, ksize * ksize, Cin,
                                                                        Cout, rows, ld_dh);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_conv_wgrad_c3(const void* x_bf16c8, const void* dh_bf16, int ld_dh, int N, int H, int W, int Cout, float* dw,
                     y2_stream_t stream) {
  Y2_ARG(x_bf16c8 && dh_bf16 && dw && N > 0 && H > 0 && W > 0 && Cout > 0 && Cout <= 32 && ld_dh >= Cout && ld_dh % 8 == 0);
  const int tiles = N * ((H + W1_TH - 1) / W1_TH) * ((W + W1_TW - 1) / W1_TW);
  int grid = tiles < 148 * 2 ? tiles : 148 * 2;
  if (!env().bn_bwd_generic) grid = tiles < 148 * 6 ? tiles : 148 * 6;     // 34 KB of smem per CTA: six resident, loads of one hide behind the MMAs of the others
  if (env().bn_bwd_generic)      // (the switch that forces the generic backward kernels: the FFMA version)
    conv_wgrad_c3_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x_bf16c8, (const __nv_bfloat16*)dh_bf16,
                                                                 ld_dh, N, H, W, Cout, dw);
  else
    conv_wgrad_c3_mma_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x_bf16c8, (const __nv_bfloat16*)dh_bf16,
                                                                     ld_dh, N, H, W, Cout, dw);
  Y2_LAUNCHED();
  return Y2_OK;
}

int y2_sum_rows_bf16(const void* a_bf16, int ld, size_t M, int C, float* out, y2_stream_t stream) {
  Y2_ARG(a_bf16 && out && M > 0 && C > 0 && ld >= C);
  size_t blocks = (M + 2047) / 2048;
  if (blocks > 1024) blocks = 1024;
  const size_t rpb = (M + blocks - 1) / blocks;
  blocks = (M + rpb - 1) / rpb;
  dim3 grid((C + 31) / 32, (unsigned)blocks), block(32, 8);
  sum_rows_bf16_kernel<<<grid, block, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)a_bf16, ld, M, C, rpb, out);
  Y2_LAUNCHED();
  return Y2_OK;
}

}  // extern "C"
