// fdx_norm.cu -- GroupNorm(+SiLU) and RMSNorm, forward and backward, NHWC bf16.
//
// Replaces the XLA lowering of
//   nn.GroupNorm(8, eps) + swish      flaxdiff/models/common.py:273-281,286-288,310-312
//   Unet.conv_out_norm + activation   flaxdiff/models/simple_unet.py:24-30,209-210
//   nn.RMSNorm(eps) in TransformerBlock   flaxdiff/models/attention.py:325-326
// flax semantics kept: statistics in f32, fast variance max(0, E[x^2]-E[x]^2),
// y = (x-mean)*rsqrt(var+eps)*scale+bias.
//
// HBM-bound kernels: every thread owns one 16-byte (8 x bf16) channel vector of a pixel,
// fully coalesced; per-(image,group) partial sums are reduced with warp shuffles,
// then shared-memory atomics, then one global atomic per block.
#include "fdx_common.cuh"
#include "../../include/fdx.h"

namespace {

constexpr int kNT = 256;

struct GnGeom {
  int vpp;      // 16-byte vectors per pixel = C/8
  int rows;     // pixel rows per block iteration = kNT / vpp
  int cpg;      // channels per group
};

__device__ __forceinline__ void load8(const __nv_bfloat16* p, float (&f)[8]) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
__device__ __forceinline__ void store8(__nv_bfloat16* p, const float (&f)[8]) {
  uint4 u;
  u.x = pack_bf16x2(f[0], f[1]); u.y = pack_bf16x2(f[2], f[3]);
  u.z = pack_bf16x2(f[4], f[5]); u.w = pack_bf16x2(f[6], f[7]);
  *reinterpret_cast<uint4*>(p) = u;
}

// stats[n][g] = (sum, sumsq) accumulated with atomics (buffer zeroed by the caller)
constexpr int kU = 4;   // pixels in flight per thread (memory-level parallelism)

__global__ void __launch_bounds__(kNT)
gn_stats_kernel(const __nv_bfloat16* __restrict__ x, long long xps, int HW, int C, int G,
                float* __restrict__ stats) {
  const int vpp = C >> 3, rows = kNT / vpp, cpg = C / G;
  const int n = blockIdx.y;
  const int tid = threadIdx.x;
  __shared__ float sh[64];
  if (tid < 2 * G) sh[tid] = 0.f;
  __syncthreads();
  if (tid < rows * vpp) {
    const int cv = tid % vpp, r = tid / vpp;
    const int g = (cv * 8) / cpg;
    float s = 0.f, q = 0.f;
    const __nv_bfloat16* base = x + (long long)n * HW * xps + cv * 8;
    const int stride = gridDim.x * rows;
    int p = blockIdx.x * rows + r;
    for (; p + (kU - 1) * stride < HW; p += kU * stride) {
      uint4 u[kU];
#pragma unroll
      for (int k = 0; k < kU; ++k)
        u[k] = *reinterpret_cast<const uint4*>(base + (long long)(p + k * stride) * xps);
#pragma unroll
      for (int k = 0; k < kU; ++k) {
        const float2 a = unpack_bf16x2(u[k].x), b = unpack_bf16x2(u[k].y), c = unpack_bf16x2(u[k].z),
                     d = unpack_bf16x2(u[k].w);
        s += (a.x + a.y) + (b.x + b.y) + (c.x + c.y) + (d.x + d.y);
        q += a.x * a.x + a.y * a.y + b.x * b.x + b.y * b.y + c.x * c.x + c.y * c.y + d.x * d.x + d.y * d.y;
      }
    }
    for (; p < HW; p += stride) {
      float f[8];
      load8(base + (long long)p * xps, f);
#pragma unroll
      for (int j = 0; j < 8; ++j) { s += f[j]; q += f[j] * f[j]; }
    }
    atomicAdd(&sh[2 * g], s);
    atomicAdd(&sh[2 * g + 1], q);
  }
  __syncthreads();
  if (tid < 2 * G) atomicAdd(&stats[(long long)n * 2 * G + tid], sh[tid]);
}

// y = silu?(a x + b) per channel pair with packed f32x2 ops: h = x*(a/2) + b/2, silu(z) = h*(1 + tanh(h))
template <bool SILU>
__global__ void __launch_bounds__(kNT)
gn_apply_kernel(const __nv_bfloat16* __restrict__ x, long long xps, int HW, int C, int G,
                const float* __restrict__ stats, const float* __restrict__ gamma,
                const float* __restrict__ beta, float eps, __nv_bfloat16* __restrict__ y, long long yps,
                const float* __restrict__ cols, int slots, int ld, int c0, float* __restrict__ stats_out) {
  const int vpp = C >> 3, rows = kNT / vpp, cpg = C / G;
  const int n = blockIdx.y;
  const int tid = threadIdx.x;
  // cols != nullptr: the statistics come straight from the producers' epilogue column sums
  // ([slots][N][2][ld], channels c0 .. c0+C) - every CTA reduces its image's groups itself (one warp per group)
  // instead of a separate stats_from_cols launch; the first CTA of the image stores them for the backward.
  __shared__ float sg[2 * 64];
  if (cols) {
    const int N = gridDim.y;
    const int warp = tid >> 5, lane = tid & 31;
    for (int g = warp; g < G; g += kNT / 32) {
      float s0 = 0.f, s1 = 0.f;
      for (int sl = 0; sl < slots; ++sl) {
        const float* b = cols + (((long long)sl * N + n) * 2) * ld + c0 + g * cpg;
        for (int c = lane; c < cpg; c += 32) { s0 += b[c]; s1 += b[ld + c]; }
      }
      s0 = warp_sum(s0);
      s1 = warp_sum(s1);
      if (lane == 0) {
        sg[2 * g] = s0;
        sg[2 * g + 1] = s1;
        if (blockIdx.x == 0) {
          stats_out[(long long)n * 2 * G + 2 * g] = s0;
          stats_out[(long long)n * 2 * G + 2 * g + 1] = s1;
        }
      }
    }
    __syncthreads();
  }
  if (tid >= rows * vpp) return;
  const int cv = tid % vpp, r = tid / vpp;
  const int g = (cv * 8) / cpg;
  const float cnt = (float)HW * (float)cpg;
  const float sum0 = cols ? sg[2 * g] : stats[(long long)n * 2 * G + 2 * g];
  const float sum1 = cols ? sg[2 * g + 1] : stats[(long long)n * 2 * G + 2 * g + 1];
  const float mean = sum0 / cnt;
  const float var = fmaxf(0.f, sum1 / cnt - mean * mean);
  const float rstd = rsqrtf(var + eps);
  const float sc = SILU ? 0.5f : 1.f;
  f32x2_t a[4], b[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float a0 = rstd * gamma[cv * 8 + 2 * j], a1 = rstd * gamma[cv * 8 + 2 * j + 1];
    a[j] = f2_pack(sc * a0, sc * a1);
    b[j] = f2_pack(sc * (beta[cv * 8 + 2 * j] - mean * a0), sc * (beta[cv * 8 + 2 * j + 1] - mean * a1));
  }
  const __nv_bfloat16* xb = x + (long long)n * HW * xps + cv * 8;
  __nv_bfloat16* yb = y + (long long)n * HW * yps + cv * 8;
  const int stride = gridDim.x * rows;
  for (int p0 = blockIdx.x * rows + r; p0 < HW; p0 += kU * stride) {
    uint4 u[kU];
#pragma unroll
    for (int k = 0; k < kU; ++k) {
      const int p = p0 + k * stride;
      u[k] = make_uint4(0, 0, 0, 0);
      if (p < HW) u[k] = *reinterpret_cast<const uint4*>(xb + (long long)p * xps);
    }
#pragma unroll
    for (int k = 0; k < kU; ++k) {
      const int p = p0 + k * stride;
      if (p < HW) {
        const uint32_t w[4] = {u[k].x, u[k].y, u[k].z, u[k].w};
        uint32_t o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const f32x2_t h = f2_fma(f2_from_bf16x2(w[j]), a[j], b[j]);
          o[j] = f2_to_bf16x2(SILU ? f2_fma(h, f2_tanh(h), h) : h);
        }
        *reinterpret_cast<uint4*>(yb + (long long)p * yps) = make_uint4(o[0], o[1], o[2], o[3]);
      }
    }
  }
}

// ---- GroupNorm(+SiLU) backward ---------------------------------------------------------------
// With a_c = rstd*gamma_c, b_c = beta_c - mean*a_c:  z = a_c*x + b_c,  dz = dy * silu'(z).
// Pass 1 needs only two per-(image, channel) sums, S0 = sum dz and S1 = sum dz*x, because
//   dbeta_c  = sum_n S0                       dgamma_c = sum_n rstd*(S1 - mean*S0)
//   red[n][g] = ( sum_{c in g} gamma_c*S0 ,   sum_{c in g} gamma_c*rstd*(S1 - mean*S0) )
// and pass 2 is  dx = dz*a_c - x*c2 + c3  with per-group c2 = rstd^2*m2, c3 = mean*c2 - rstd*m1.
// Both passes are instruction-issue sensitive (two MUFU per element), hence the reduced algebra.

// The two streaming passes of the backward are written with packed f32x2 arithmetic (FFMA2): with
// scalar ops ncu counted 20-24 instructions per element and an issue-slot utilisation that capped both
// passes at 56-63 % of the HBM rate.  Per channel PAIR: h = x*(a/2) + b/2, t = tanh(h),
//   sigmoid(z) = (1+t)/2,  silu'(z) = sigmoid(z) * (1 + h*(1-t)),  dz = dy * silu'(z)
// = 6 packed ops + 2 MUFU.  Every thread owns 8 channels (16-byte vectors) of kBU pixels per iteration.
constexpr int kBU = 3;   // pixels in flight per thread

struct GnPair4 { f32x2_t v[4]; };

// dz (x 2 when TWICE) for one channel pair
template <bool SILU, bool TWICE>
__device__ __forceinline__ f32x2_t gn_dz_pair(f32x2_t x, f32x2_t dy, f32x2_t ah, f32x2_t bh) {
  if (!SILU) return TWICE ? f2_add(dy, dy) : dy;
  const f32x2_t one = f2_pack(1.f, 1.f);
  const f32x2_t h = f2_fma(x, ah, bh);
  const f32x2_t t = f2_tanh(h);
  const f32x2_t u = f2_fma(h, f2_sub(one, t), one);
  const f32x2_t s = TWICE ? f2_add(t, one) : f2_fma(t, f2_pack(0.5f, 0.5f), f2_pack(0.5f, 0.5f));
  return f2_mul(dy, f2_mul(s, u));
}

// Pass 1 with the finalize step merged in: both of its outputs are linear in the per-(image, channel) sums,
// so every CTA adds its partial's contribution straight into red[n][g][2] (zeroed by the caller), dgamma[c]
// and dbeta[c], and zeroes the column-sum outputs the second pass accumulates into.
template <bool SILU>
__global__ void __launch_bounds__(kNT, 3)
gn_bwd_stats_kernel(const __nv_bfloat16* __restrict__ x, long long xps,
                    const __nv_bfloat16* __restrict__ dy, long long dps, int HW, int C, int G,
                    const float* __restrict__ stats, const float* __restrict__ gamma,
                    const float* __restrict__ beta, float eps,
                    float* __restrict__ red, float* __restrict__ dgamma, float* __restrict__ dbeta,
                    float* __restrict__ csum_img, float* __restrict__ csum_tot) {
  const int vpp = C >> 3, rows = kNT / vpp, cpg = C / G;
  const int n = blockIdx.y;
  const int tid = threadIdx.x;
  extern __shared__ float shm[];   // 2 * [rows*C] + 2 * [C]
  float* part0 = shm;
  float* part1 = part0 + rows * C;
  const float cnt = (float)HW * (float)cpg;
  if (blockIdx.x == 0) {
    if (csum_img) for (int c = tid; c < C; c += kNT) csum_img[(long long)n * C + c] = 0.f;
    if (csum_tot && n == 0) for (int c = tid; c < C; c += kNT) csum_tot[c] = 0.f;
  }
  if (tid < rows * vpp) {
    const int cv = tid % vpp, r = tid / vpp;
    const int g = (cv * 8) / cpg;
    const float mean = stats[(long long)n * 2 * G + 2 * g] / cnt;
    const float var = fmaxf(0.f, stats[(long long)n * 2 * G + 2 * g + 1] / cnt - mean * mean);
    const float rstd = rsqrtf(var + eps);
    GnPair4 ah, bh, s0, s1;      // a/2, b/2 and the two running sums, as channel pairs
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float a0 = rstd * gamma[cv * 8 + 2 * j], a1 = rstd * gamma[cv * 8 + 2 * j + 1];
      ah.v[j] = f2_pack(0.5f * a0, 0.5f * a1);
      bh.v[j] = f2_pack(0.5f * (beta[cv * 8 + 2 * j] - mean * a0), 0.5f * (beta[cv * 8 + 2 * j + 1] - mean * a1));
      s0.v[j] = f2_pack(0.f, 0.f);
      s1.v[j] = f2_pack(0.f, 0.f);
    }
    const __nv_bfloat16* xb = x + (long long)n * HW * xps + cv * 8;
    const __nv_bfloat16* db_ = dy + (long long)n * HW * dps + cv * 8;
    const int stride = gridDim.x * rows;
    for (int p0 = blockIdx.x * rows + r; p0 < HW; p0 += kBU * stride) {
      uint4 xu[kBU], du[kBU];
#pragma unroll
      for (int k = 0; k < kBU; ++k) {
        const int p = p0 + k * stride;
        xu[k] = make_uint4(0, 0, 0, 0);
        du[k] = make_uint4(0, 0, 0, 0);   // dy = 0 contributes nothing to either sum
        if (p < HW) {
          xu[k] = *reinterpret_cast<const uint4*>(xb + (long long)p * xps);
          du[k] = *reinterpret_cast<const uint4*>(db_ + (long long)p * dps);
        }
      }
#pragma unroll
      for (int k = 0; k < kBU; ++k) {
        const uint32_t xw[4] = {xu[k].x, xu[k].y, xu[k].z, xu[k].w};
        const uint32_t dw[4] = {du[k].x, du[k].y, du[k].z, du[k].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const f32x2_t xv = f2_from_bf16x2(xw[j]);
          const f32x2_t dz = gn_dz_pair<SILU, false>(xv, f2_from_bf16x2(dw[j]), ah.v[j], bh.v[j]);
          s0.v[j] = f2_add(s0.v[j], dz);
          s1.v[j] = f2_fma(dz, xv, s1.v[j]);
        }
      }
    }
    // conflict-free partials: part[r][c] (rows x C floats per quantity), then a column sum
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float lo, hi;
      f2_unpack(s0.v[j], lo, hi);
      part0[r * C + cv * 8 + 2 * j] = lo; part0[r * C + cv * 8 + 2 * j + 1] = hi;
      f2_unpack(s1.v[j], lo, hi);
      part1[r * C + cv * 8 + 2 * j] = lo; part1[r * C + cv * 8 + 2 * j + 1] = hi;
    }
  }
  __syncthreads();
  float* gr0 = part1 + rows * C;   // [C] gamma_c * S0,  [C] gamma_c * rstd * (S1 - mean * S0)
  float* gr1 = gr0 + C;
  for (int c = tid; c < C; c += kNT) {
    float t0 = 0.f, t1 = 0.f;
    for (int rr = 0; rr < rows; ++rr) { t0 += part0[rr * C + c]; t1 += part1[rr * C + c]; }
    const int g = c / cpg;
    const float mean = stats[(long long)n * 2 * G + 2 * g] / cnt;
    const float var = fmaxf(0.f, stats[(long long)n * 2 * G + 2 * g + 1] / cnt - mean * mean);
    const float u = rsqrtf(var + eps) * (t1 - mean * t0);
    atomicAdd(&dbeta[c], t0);
    atomicAdd(&dgamma[c], u);
    const float ga = gamma[c];
    gr0[c] = ga * t0;
    gr1[c] = ga * u;
  }
  __syncthreads();
  for (int g = tid; g < G; g += kNT) {
    float r0 = 0.f, r1 = 0.f;
    for (int c = g * cpg; c < (g + 1) * cpg; ++c) { r0 += gr0[c]; r1 += gr1[c]; }
    atomicAdd(&red[(long long)n * 2 * G + 2 * g], r0);
    atomicAdd(&red[(long long)n * 2 * G + 2 * g + 1], r1);
  }
}

// ab[n][0][c] = a = rstd*gamma_c ; ab[n][1][c] = b = beta_c - mean*a   (consumed by the fused dgrad epilogue)
__global__ void __launch_bounds__(256)
gn_coeffs_kernel(const float* __restrict__ stats, const float* __restrict__ gamma,
                 const float* __restrict__ beta, int N, int HW, int C, int G, float eps,
                 float* __restrict__ ab) {
  const int cpg = C / G;
  const float cnt = (float)HW * (float)cpg;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)N * C;
       i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / C), c = (int)(i % C), g = c / cpg;
    const float mean = stats[(long long)n * 2 * G + 2 * g] / cnt;
    const float var = fmaxf(0.f, stats[(long long)n * 2 * G + 2 * g + 1] / cnt - mean * mean);
    const float a = rsqrtf(var + eps) * gamma[c];
    ab[((long long)n * 2) * C + c] = a;
    ab[((long long)n * 2 + 1) * C + c] = beta[c] - mean * a;
  }
}

// stats[n][g] = (sum, sumsq) from the per-(image, channel) sums a convolution epilogue accumulated:
// cols[slot][n][{0,1}][C]; one warp per (image, group)
__global__ void __launch_bounds__(256)
gn_stats_from_cols_kernel(const float* __restrict__ cols, int slots, int N, int ld, int c0, int C, int G,
                          float* __restrict__ stats) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= N * G) return;
  const int lane = threadIdx.x & 31, n = i / G, g = i % G, cpg = C / G;
  float s = 0.f, q = 0.f;
  for (int sl = 0; sl < slots; ++sl) {
    const float* b = cols + (((long long)sl * N + n) * 2) * ld + c0 + g * cpg;
    for (int c = lane; c < cpg; c += 32) { s += b[c]; q += b[ld + c]; }
  }
  s = warp_sum(s);
  q = warp_sum(q);
  if (lane == 0) {
    stats[(long long)n * 2 * G + 2 * g] = s;
    stats[(long long)n * 2 * G + 2 * g + 1] = q;
  }
}

// pass 2: dx (+= if accumulate); optionally the column sums of dx (csum_img[n][c], csum_tot[c]).
//   dx = dz*a - x*c2 + c3 = (2 dz)*(a/2) + (c3 - x*c2)
template <bool SILU, bool ACC, bool CS>
__global__ void __launch_bounds__(kNT, ACC ? 2 : 3)
gn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ x, long long xps,
                    const __nv_bfloat16* __restrict__ dy, long long dps, int HW, int C, int G,
                    const float* __restrict__ stats, const float* __restrict__ red,
                    const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                    __nv_bfloat16* __restrict__ dx, long long dxps, float* __restrict__ csum_img,
                    const __nv_bfloat16* __restrict__ acc, long long accps, float* __restrict__ csum_tot,
                    const float* __restrict__ slot_ws, int slots, float* __restrict__ dgamma,
                    float* __restrict__ dbeta) {
  const int vpp = C >> 3, rows = kNT / vpp, cpg = C / G;
  const int n = blockIdx.y;
  const int tid = threadIdx.x;
  extern __shared__ float sh_cs[];   // [rows*C] when column sums are requested (+ [2C + 2G] with slot_ws)
  // slot_ws != nullptr (fused first pass: the data-gradient epilogue left S0 = sum dz, S1 = sum dz*x per slot):
  // every CTA derives its image's per-group constants itself - no collapse / finalize launches - and the
  // first CTA of each image adds the image's share of dgamma / dbeta.
  float* pro = sh_cs + (CS ? rows * C : 0);
  if (slot_ws) {
    const float cnt_ = (float)HW * (float)cpg;
    const int N = gridDim.y;
    for (int c = tid; c < C; c += kNT) {
      float S0 = 0.f, S1 = 0.f;
      for (int sl = 0; sl < slots; ++sl) {
        const float* b = slot_ws + (((long long)sl * N + n) * 2) * C;
        S0 += b[c];
        S1 += b[C + c];
      }
      const int g = c / cpg;
      const float mean = stats[(long long)n * 2 * G + 2 * g] / cnt_;
      const float var = fmaxf(0.f, stats[(long long)n * 2 * G + 2 * g + 1] / cnt_ - mean * mean);
      const float u = rsqrtf(var + eps) * (S1 - mean * S0);
      if (blockIdx.x == 0) { atomicAdd(&dbeta[c], S0); atomicAdd(&dgamma[c], u); }
      const float ga = gamma[c];
      pro[c] = ga * S0;
      pro[C + c] = ga * u;
    }
    __syncthreads();
    for (int g = tid; g < G; g += kNT) {
      float r0 = 0.f, r1 = 0.f;
      for (int c = g * cpg; c < (g + 1) * cpg; ++c) { r0 += pro[c]; r1 += pro[C + c]; }
      pro[2 * C + 2 * g] = r0;
      pro[2 * C + 2 * g + 1] = r1;
    }
    __syncthreads();
  }
  if (tid < rows * vpp) {
    const int cv = tid % vpp, r = tid / vpp;
    const int g = (cv * 8) / cpg;
    const float cnt = (float)HW * (float)cpg;
    const float mean = stats[(long long)n * 2 * G + 2 * g] / cnt;
    const float var = fmaxf(0.f, stats[(long long)n * 2 * G + 2 * g + 1] / cnt - mean * mean);
    const float rstd = rsqrtf(var + eps);
    const float m1 = (slot_ws ? pro[2 * C + 2 * g] : red[(long long)n * 2 * G + 2 * g]) / cnt;
    const float m2 = (slot_ws ? pro[2 * C + 2 * g + 1] : red[(long long)n * 2 * G + 2 * g + 1]) / cnt;
    const float c2 = rstd * rstd * m2;
    const float c3 = mean * c2 - rstd * m1;
    const f32x2_t nc2 = f2_pack(-c2, -c2), c3p = f2_pack(c3, c3);
    GnPair4 ah, bh, cs;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float a0 = rstd * gamma[cv * 8 + 2 * j], a1 = rstd * gamma[cv * 8 + 2 * j + 1];
      ah.v[j] = f2_pack(0.5f * a0, 0.5f * a1);
      bh.v[j] = SILU ? f2_pack(0.5f * (beta[cv * 8 + 2 * j] - mean * a0),
                               0.5f * (beta[cv * 8 + 2 * j + 1] - mean * a1))
                     : f2_pack(0.f, 0.f);
      cs.v[j] = f2_pack(0.f, 0.f);
    }
    const __nv_bfloat16* xb = x + (long long)n * HW * xps + cv * 8;
    const __nv_bfloat16* db_ = dy + (long long)n * HW * dps + cv * 8;
    __nv_bfloat16* ob = dx + (long long)n * HW * dxps + cv * 8;
    const __nv_bfloat16* ab_ = ACC ? acc + (long long)n * HW * accps + cv * 8 : nullptr;
    const int stride = gridDim.x * rows;
    for (int p0 = blockIdx.x * rows + r; p0 < HW; p0 += kBU * stride) {
      uint4 xu[kBU], du[kBU], ou[kBU];
#pragma unroll
      for (int k = 0; k < kBU; ++k) {
        const int p = p0 + k * stride;
        xu[k] = make_uint4(0, 0, 0, 0);
        du[k] = make_uint4(0, 0, 0, 0);
        ou[k] = make_uint4(0, 0, 0, 0);
        if (p < HW) {
          xu[k] = *reinterpret_cast<const uint4*>(xb + (long long)p * xps);
          du[k] = *reinterpret_cast<const uint4*>(db_ + (long long)p * dps);
          if (ACC) ou[k] = *reinterpret_cast<const uint4*>(ab_ + (long long)p * accps);
        }
      }
#pragma unroll
      for (int k = 0; k < kBU; ++k) {
        const int p = p0 + k * stride;
        if (p < HW) {
          const uint32_t xw[4] = {xu[k].x, xu[k].y, xu[k].z, xu[k].w};
          const uint32_t dw[4] = {du[k].x, du[k].y, du[k].z, du[k].w};
          const uint32_t ow[4] = {ou[k].x, ou[k].y, ou[k].z, ou[k].w};
          uint32_t res[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const f32x2_t xv = f2_from_bf16x2(xw[j]);
            const f32x2_t dz2 = gn_dz_pair<SILU, true>(xv, f2_from_bf16x2(dw[j]), ah.v[j], bh.v[j]);
            f32x2_t v = f2_fma(dz2, ah.v[j], f2_fma(xv, nc2, c3p));
            if (CS) cs.v[j] = f2_add(cs.v[j], v);
            if (ACC) v = f2_add(v, f2_from_bf16x2(ow[j]));
            res[j] = f2_to_bf16x2(v);
          }
          *reinterpret_cast<uint4*>(ob + (long long)p * dxps) = make_uint4(res[0], res[1], res[2], res[3]);
        }
      }
    }
    if (CS) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float lo, hi;
        f2_unpack(cs.v[j], lo, hi);
        sh_cs[r * C + cv * 8 + 2 * j] = lo;
        sh_cs[r * C + cv * 8 + 2 * j + 1] = hi;
      }
    }
  }
  if (CS) {
    __syncthreads();
    for (int c = tid; c < C; c += kNT) {
      float v = 0.f;
      for (int rr = 0; rr < rows; ++rr) v += sh_cs[rr * C + c];
      atomicAdd(&csum_img[(long long)n * C + c], v);
      if (csum_tot) atomicAdd(&csum_tot[c], v);     // zeroed by the first pass (merged finalize)
    }
  }
}

// ---------------------------------------------------------------------------
// RMSNorm over channels, one warp per pixel.
// ---------------------------------------------------------------------------
constexpr int kRmsV = 4;   // up to 4 x 32 x 8 = 1024 channels, one warp per pixel

__global__ void __launch_bounds__(256)
rms_fwd_kernel(const __nv_bfloat16* __restrict__ x, long long xps, long long npix, int C,
               const float* __restrict__ scale, float eps, __nv_bfloat16* __restrict__ y,
               long long yps) {
  const int lane = threadIdx.x & 31;
  const int nv = C >> 3;
  const long long wid = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const long long nw = (long long)gridDim.x * 8;
  for (long long p = wid; p < npix; p += nw) {
    float f[kRmsV][8];
    float q = 0.f;
#pragma unroll
    for (int v = 0; v < kRmsV; ++v) {
      if (v * 32 + lane < nv) {
        load8(x + p * xps + (v * 32 + lane) * 8, f[v]);
#pragma unroll
        for (int j = 0; j < 8; ++j) q += f[v][j] * f[v][j];
      }
    }
    q = warp_sum(q);
    const float r = rsqrtf(q / (float)C + eps);
#pragma unroll
    for (int v = 0; v < kRmsV; ++v) {
      if (v * 32 + lane < nv) {
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = f[v][j] * r * scale[(v * 32 + lane) * 8 + j];
        store8(y + p * yps + (v * 32 + lane) * 8, o);
      }
    }
  }
}

__global__ void __launch_bounds__(256)
rms_bwd_kernel(const __nv_bfloat16* __restrict__ x, long long xps,
               const __nv_bfloat16* __restrict__ dy, long long dps, long long npix, int C,
               const float* __restrict__ scale, float eps, __nv_bfloat16* __restrict__ dx,
               long long dxps, int accumulate, float* __restrict__ dscale) {
  extern __shared__ float sh_ds[];   // [C]
  for (int i = threadIdx.x; i < C; i += 256) sh_ds[i] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int nv = C >> 3;
  const long long wid = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const long long nw = (long long)gridDim.x * 8;
  float ds[kRmsV][8];
#pragma unroll
  for (int v = 0; v < kRmsV; ++v)
#pragma unroll
    for (int j = 0; j < 8; ++j) ds[v][j] = 0.f;
  for (long long p = wid; p < npix; p += nw) {
    float f[kRmsV][8], d[kRmsV][8];
    float q = 0.f;
#pragma unroll
    for (int v = 0; v < kRmsV; ++v) {
      if (v * 32 + lane < nv) {
        load8(x + p * xps + (v * 32 + lane) * 8, f[v]);
        load8(dy + p * dps + (v * 32 + lane) * 8, d[v]);
#pragma unroll
        for (int j = 0; j < 8; ++j) q += f[v][j] * f[v][j];
      }
    }
    q = warp_sum(q);
    const float r = rsqrtf(q / (float)C + eps);
    float m = 0.f;
#pragma unroll
    for (int v = 0; v < kRmsV; ++v) {
      if (v * 32 + lane < nv) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float xh = f[v][j] * r;
          ds[v][j] += d[v][j] * xh;
          d[v][j] *= scale[(v * 32 + lane) * 8 + j];   // g = dy * scale
          m += d[v][j] * xh;
        }
      }
    }
    m = warp_sum(m) / (float)C;
#pragma unroll
    for (int v = 0; v < kRmsV; ++v) {
      if (v * 32 + lane < nv) {
        float o[8];
        if (accumulate) load8(dx + p * dxps + (v * 32 + lane) * 8, o);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float val = r * (d[v][j] - f[v][j] * r * m);
          o[j] = accumulate ? o[j] + val : val;
        }
        store8(dx + p * dxps + (v * 32 + lane) * 8, o);
      }
    }
  }
#pragma unroll
  for (int v = 0; v < kRmsV; ++v)
    if (v * 32 + lane < nv)
#pragma unroll
      for (int j = 0; j < 8; ++j) atomicAdd(&sh_ds[(v * 32 + lane) * 8 + j], ds[v][j]);
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += 256) atomicAdd(&dscale[i], sh_ds[i]);
}

int gn_check(const fdx_act* x, int groups, const char* what) {
  FDX_REQUIRE(x && x->ptr, "%s: null tensor", what);
  FDX_REQUIRE(groups > 0 && groups <= 32 && x->c % groups == 0, "%s: bad group count %d", what, groups);
  FDX_REQUIRE((x->c / groups) % 8 == 0, "%s: channels per group (%d) must be a multiple of 8", what,
              x->c / groups);
  FDX_REQUIRE(x->c / 8 <= kNT, "%s: C=%d too large", what, x->c);
  FDX_REQUIRE(x->pix_stride % 8 == 0, "%s: pix_stride must be a multiple of 8", what);
  return FDX_OK;
}

// Two waves of co-resident blocks (`resident` per SM for the kernel in question): every block then
// amortises its prologue (statistics / gamma / beta loads) and epilogue (partial-sum reduction, atomics)
// over many pixel rows.  Sizing for ~16 blocks per SM made the small deep-level tensors pure launch /
// prologue latency (ncu: 8 MB in 8 us).
dim3 gn_grid(const fdx_act* x, int unroll, int resident) {
  const int HW = x->h * x->w;
  const int rows = kNT / (x->c / 8);
  int bx = (HW + rows * unroll - 1) / (rows * unroll);
  constexpr int kWaves = 2;
  int target = (kWaves * resident * 148) / x->n;
  if (target < 1) target = 1;
  if (bx > target) bx = target;
  if (bx < 1) bx = 1;
  return dim3(bx, x->n);
}

// second pass of the GroupNorm backward: template dispatch on (activation, accumulate, column sums)
void launch_bwd_apply(const fdx_act* x, const fdx_act* dy, int groups, const float* stats, const float* red,
                      const float* gamma, const float* beta, float eps, int silu, const fdx_act* dx,
                      const fdx_act* acc, float* csum_img, cudaStream_t st, float* csum_tot = nullptr,
                      const float* slot_ws = nullptr, int slots = 0, float* dgamma = nullptr, float* dbeta = nullptr) {
  const int accumulate = acc != nullptr;
  const int C = x->c, HW = x->h * x->w;
  const size_t shm = (csum_img ? sizeof(float) * (kNT / (C / 8)) * C : 0) +
                     (slot_ws ? sizeof(float) * (2 * (size_t)C + 2 * groups) : 0);
  const dim3 grid = gn_grid(x, kBU, accumulate ? 2 : 3);
  const __nv_bfloat16* xp = (const __nv_bfloat16*)x->ptr;
  const __nv_bfloat16* dp = (const __nv_bfloat16*)dy->ptr;
  __nv_bfloat16* op = (__nv_bfloat16*)dx->ptr;
#define FDX_GN_APPLY(S, A, CSF)                                                                          \
  gn_bwd_apply_kernel<S, A, CSF><<<grid, kNT, shm, st>>>(xp, x->pix_stride, dp, dy->pix_stride, HW, C,  \
                                                         groups, stats, red, gamma, beta, eps, op,       \
                                                         dx->pix_stride, csum_img,                                 \
                                                         (const __nv_bfloat16*)(acc ? acc->ptr : nullptr),          \
                                                         (long long)(acc ? acc->pix_stride : 0), csum_tot, slot_ws, \
                                                         slots, dgamma, dbeta)
  const int key = (silu ? 4 : 0) | (accumulate ? 2 : 0) | (csum_img ? 1 : 0);
  switch (key) {
    case 0: FDX_GN_APPLY(false, false, false); break;
    case 1: FDX_GN_APPLY(false, false, true); break;
    case 2: FDX_GN_APPLY(false, true, false); break;
    case 3: FDX_GN_APPLY(false, true, true); break;
    case 4: FDX_GN_APPLY(true, false, false); break;
    case 5: FDX_GN_APPLY(true, false, true); break;
    case 6: FDX_GN_APPLY(true, true, false); break;
    default: FDX_GN_APPLY(true, true, true); break;
  }
#undef FDX_GN_APPLY
}

}  // namespace

extern "C" {

int fdx_groupnorm_stats(const fdx_act* x, int groups, float* stats, void* stream) {
  int s = gn_check(x, groups, "groupnorm_stats");
  if (s != FDX_OK) return s;
  cudaStream_t st = (cudaStream_t)stream;
  FDX_CUDA(cudaMemsetAsync(stats, 0, sizeof(float) * 2 * groups * x->n, st));
  gn_stats_kernel<<<gn_grid(x, kU, 5), kNT, 0, st>>>((const __nv_bfloat16*)x->ptr, x->pix_stride,
                                              x->h * x->w, x->c, groups, stats);
  FDX_LAUNCH_CHECK();
  return FDX_OK;
}

int fdx_groupnorm_stats_from_cols(const float* cols, int slots, int N, int ld, int c0, int C, int groups,
                                  float* stats, void* stream) {
  FDX_REQUIRE(cols && stats && slots > 0 && N > 0 && C > 0 && groups > 0 && C % groups == 0 && c0 >= 0 &&
                  c0 + C <= ld,
              "groupnorm_stats_from_cols: bad arguments");
  gn_stats_from_cols_kernel<<<(N * groups + 7) / 8, 256, 0, (cudaStream_t)stream>>>(cols, slots, N, ld, c0, C,
                                                                                    groups, stats);
  FDX_LAUNCH_CHECK();
  return FDX_OK;
}

int fdx_groupnorm_apply_cols(const fdx_act* x, int groups, const float* cols, int slots, int ld, int c0,
                             const float* gamma, const float* beta, float eps, int silu, const fdx_act* y,
                             float* stats_out, void* stream) {
  int s = gn_check(x, groups, "groupnorm_apply_cols");
  if (s != FDX_OK) return s;
  FDX_REQUIRE(y && y->ptr && y->n == x->n && y->h == x->h && y->w == x->w && y->c == x->c,
              "groupnorm_apply_cols: output shape mismatch");
  FDX_REQUIRE(cols && stats_out && slots > 0 && c0 >= 0 && c0 + x->c <= ld && groups <= 64,
              "groupnorm_apply_cols: bad column-sum workspace");
  if (silu)
    gn_apply_kernel<true><<<gn_grid(x, kU, 5), kNT, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)x->ptr, x->pix_stride, x->h * x->w, x->c, groups, nullptr, gamma, beta, eps,
        (__nv_bfloat16*)y->ptr, y->pix_stride, cols, slots, ld, c0, stats_out);
  else
    gn_apply_kernel<false><<<gn_grid(x, kU, 5), kNT, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)x->ptr, x->pix_stride, x->h * x->w, x->c, groups, nullptr, gamma, beta, eps,
        (__nv_bfloat16*)y->ptr, y->pix_stride, cols, slots, ld, c0, stats_out);
  FDX_LAUNCH_CHECK();
  return FDX_OK;
}

int fdx_groupnorm_apply(const fdx_act* x, int groups, const float* stats, const float* gamma,
                        const float* beta, float eps, int silu, const fdx_act* y, void* stream) {
  int s = gn_check(x, groups, "groupnorm_apply");
  if (s != FDX_OK) return s;
  FDX_REQUIRE(y && y->ptr && y->n == x->n && y->h == x->h && y->w == x->w && y->c == x->c,
              "groupnorm_apply: output shape mismatch");
  if (silu)
    gn_apply_kernel<true><<<gn_grid(x, kU, 5), kNT, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)x->ptr, x->pix_stride, x->h * x->w, x->c, groups, stats, gamma, beta, eps,
        (__nv_bfloat16*)y->ptr, y->pix_stride, nullptr, 0, 0, 0, nullptr);
  else
    gn_apply_kernel<false><<<gn_grid(x, kU, 5), kNT, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)x->ptr, x->pix_stride, x->h * x->w, x->c, groups, stats, gamma, beta, eps,
        (__nv_bfloat16*)y->ptr, y->pix_stride, nullptr, 0, 0, 0, nullptr);
  FDX_LAUNCH_CHECK();
  return FDX_OK;
}

static int groupnorm_bwd_impl(const fdx_act* x, const fdx_act* dy, int groups, const float* stats,
                              const float* gamma, const float* beta, float eps, int silu, float* ws,
                              float* dgamma, float* dbeta, const fdx_act* dx, const fdx_act* acc,
                              float* csum_img, float* csum_tot, void* stream) {
  int s = gn_check(x, groups, "groupnorm_bwd");
  if (s != FDX_OK) return s;
  FDX_REQUIRE(dy && dy->ptr && dx && dx->ptr && ws && dgamma && dbeta, "groupnorm_bwd: null tensor");
  FDX_REQUIRE(dy->c == x->c && dx->c == x->c && dy->n == x->n && dx->n == x->n &&
                  dy->h == x->h && dy->w == x->w && dx->h == x->h && dx->w == x->w,
              "groupnorm_bwd: shape mismatch");
  FDX_REQUIRE(!csum_tot || csum_img, "groupnorm_bwd: csum_tot needs csum_img");
  cudaStream_t st = (cudaStream_t)stream;
  const int N = x->n, C = x->c, HW = x->h * x->w;
  float* red = ws;                          // [N][G][2]: the per-group sums of pass 1
  FDX_CUDA(cudaMemsetAsync(red, 0, sizeof(float) * 2 * N * groups, st));
  const size_t shm = sizeof(float) * (2 * (size_t)(kNT / (C / 8)) * C + 2 * C);
  if (silu)
    gn_bwd_stats_kernel<true><<<gn_grid(x, kBU, 3), kNT, shm, st>>>(
        (const __nv_bfloat16*)x->ptr, x->pix_stride, (const __nv_bfloat16*)dy->ptr, dy->pix_stride, HW, C,
        groups, stats, gamma, beta, eps, red, dgamma, dbeta, csum_img, csum_tot);
  else
    gn_bwd_stats_kernel<false><<<gn_grid(x, kBU, 3), kNT, shm, st>>>(
        (const __nv_bfloat16*)x->ptr, x->pix_stride, (const __nv_bfloat16*)dy->ptr, dy->pix_stride, HW, C,
        groups, stats, gamma, beta, eps, red, dgamma, dbeta, csum_img, csum_tot);
  FDX_LAUNCH_CHECK();
  launch_bwd_apply(x, dy, groups, stats, red, gamma, beta, eps, silu, dx, acc, csum_img, st, csum_tot);
  FDX_LAUNCH_CHECK();
  return FDX_OK;
}

int fdx_groupnorm_bwd(const fdx_act* x, const fdx_act* dy, int groups, const float* stats,
                      const float* gamma, const float* beta, float eps, int silu, float* ws,
                      float* dgamma, float* dbeta, const fdx_act* dx, int accumulate,
                      float* csum_img, float* csum_tot, void* stream) {
  return groupnorm_bwd_impl(x, dy, groups, stats, gamma, beta, eps, silu, ws, dgamma, dbeta, dx,
                            accumulate ? dx : nullptr, csum_img, csum_tot, stream);
}

int fdx_groupnorm_bwd_add(const fdx_act* x, const fdx_act* dy, int groups, const float* stats,
                          const float* gamma, const float* beta, float eps, int silu, float* ws,
                          float* dgamma, float* dbeta, const fdx_act* dx, const fdx_act* addend,
                          float* csum_img, float* csum_tot, void* stream) {
  FDX_REQUIRE(addend && addend->ptr, "groupnorm_bwd_add: null addend");
  FDX_REQUIRE(addend->c == x->c && addend->n == x->n && addend->h == x->h && addend->w == x->w,
              "groupnorm_bwd_add: addend shape mismatch");
  return groupnorm_bwd_impl(x, dy, groups, stats, gamma, beta, eps, silu, ws, dgamma, dbeta, dx, addend, csum_img,
                            csum_tot, stream);
}

int fdx_groupnorm_coeffs(const float* stats, const float* gamma, const float* beta, int N, int HW, int C,
                         int groups, float eps, float* ab, void* stream) {
  FDX_REQUIRE(stats && gamma && beta && ab && N > 0 && HW > 0 && C > 0 && groups > 0 && C % groups == 0,
              "groupnorm_coeffs: bad arguments");
  long long grid = ((long long)N * C + 255) / 256;
  if (grid > 148 * 8) grid = 148 * 8;
  gn_coeffs_kernel<<<(int)grid, 256, 0, (cudaStream_t)stream>>>(stats, gamma, beta, N, HW, C, groups, eps, ab);
  FDX_LAUNCH_CHECK();
  return FDX_OK;
}

static int groupnorm_bwd_dz_impl(const fdx_act* x, const fdx_act* dz, int groups, const float* stats,
                                 const float* gamma, float eps, const float* ws_slots, int slots,
                                 float* dgamma, float* dbeta, const fdx_act* dx, const fdx_act* acc,
                                 float* csum_img, float* csum_tot, void* stream) {
  int s = gn_check(x, groups, "groupnorm_bwd_dz");
  if (s != FDX_OK) return s;
  FDX_REQUIRE(dz && dz->ptr && dx && dx->ptr && ws_slots && slots > 0 && dgamma && dbeta,
              "groupnorm_bwd_dz: null tensor");
  FDX_REQUIRE(dz->c == x->c && dx->c == x->c && dz->n == x->n && dx->n == x->n && dz->h == x->h &&
                  dz->w == x->w && dx->h == x->h && dx->w == x->w,
              "groupnorm_bwd_dz: shape mismatch");
  FDX_REQUIRE(!csum_tot || csum_img, "groupnorm_bwd_dz: csum_tot needs csum_img");
  cudaStream_t st = (cudaStream_t)stream;
  const int N = x->n, C = x->c;
  if (csum_img) FDX_CUDA(cudaMemsetAsync(csum_img, 0, sizeof(float) * N * C, st));
  if (csum_tot) FDX_CUDA(cudaMemsetAsync(csum_tot, 0, sizeof(float) * C, st));
  // one launch: the apply kernel's prologue collapses the slots and derives the per-group constants; dz already
  // carries silu'(z), so it is the activation-free second pass (beta is not read)
  launch_bwd_apply(x, dz, groups, stats, nullptr, gamma, gamma, eps, 0, dx, acc, csum_img, st, csum_tot, ws_slots,
                   slots, dgamma, dbeta);
  FDX_LAUNCH_CHECK();
  return FDX_OK;
}

int fdx_groupnorm_bwd_dz(const fdx_act* x, const fdx_act* dz, int groups, const float* stats,
                         const float* gamma, float eps, const float* ws_slots, int slots, float* ws,
                         float* dgamma, float* dbeta, const fdx_act* dx, int accumulate, float* csum_img,
                         float* csum_tot, void* stream) {
  return groupnorm_bwd_dz_impl(x, dz, groups, stats, gamma, eps, ws_slots, slots, dgamma, dbeta, dx,
                               accumulate ? dx : nullptr, csum_img, csum_tot, stream);
}

int fdx_groupnorm_bwd_dz_add(const fdx_act* x, const fdx_act* dz, int groups, const float* stats,
                             const float* gamma, float eps, const float* ws_slots, int slots, float* ws,
                             float* dgamma, float* dbeta, const fdx_act* dx, const fdx_act* addend,
                             float* csum_img, float* csum_tot, void* stream) {
  FDX_REQUIRE(addend && addend->ptr, "groupnorm_bwd_dz_add: null addend");
  FDX_REQUIRE(addend->c == x->c && addend->n == x->n && addend->h == x->h && addend->w == x->w,
              "groupnorm_bwd_dz_add: addend shape mismatch");
  return groupnorm_bwd_dz_impl(x, dz, groups, stats, gamma, eps, ws_slots, slots, dgamma, dbeta, dx, addend,
                               csum_img, csum_tot, stream);
}

int fdx_rmsnorm_fwd(const fdx_act* x, const float* scale, float eps, const fdx_act* y,
                    void* stream) {
  FDX_REQUIRE(x && x->ptr && y && y->ptr && scale, "rmsnorm_fwd: null tensor");
  FDX_REQUIRE(x->c % 8 == 0 && x->c <= 1024, "rmsnorm_fwd: C=%d must be a multiple of 8, <= 1024", x->c);
  const long long npix = (long long)x->n * x->h * x->w;
  int grid = (int)((npix + 7) / 8);
  if (grid > 148 * 8) grid = 148 * 8;
  rms_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x->ptr, x->pix_stride, npix,
                                                         x->c, scale, eps, (__nv_bfloat16*)y->ptr,
                                                         y->pix_stride);
  FDX_LAUNCH_CHECK();
  return FDX_OK;
}

int fdx_rmsnorm_bwd(const fdx_act* x, const fdx_act* dy, const float* scale, float eps,
                    const fdx_act* dx, int accumulate, float* dscale, void* stream) {
  FDX_REQUIRE(x && x->ptr && dy && dy->ptr && dx && dx->ptr && scale && dscale, "rmsnorm_bwd: null tensor");
  FDX_REQUIRE(x->c % 8 == 0 && x->c <= 1024, "rmsnorm_bwd: C=%d must be a multiple of 8, <= 1024", x->c);
  const long long npix = (long long)x->n * x->h * x->w;
  int grid = (int)((npix + 7) / 8);
  if (grid > 148 * 2) grid = 148 * 2;
  rms_bwd_kernel<<<grid, 256, sizeof(float) * x->c, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)x->ptr, x->pix_stride, (const __nv_bfloat16*)dy->ptr, dy->pix_stride, npix, x->c,
      scale, eps, (__nv_bfloat16*)dx->ptr, dx->pix_stride, accumulate, dscale);
  FDX_LAUNCH_CHECK();
  return FDX_OK;
}

}  // extern "C"
