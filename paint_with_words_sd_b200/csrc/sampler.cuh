// Elementwise kernels of the Euler / Euler-ancestral / DPM-Solver++(2M) samplers (sm_100a).
//
// Every one of these samplers updates the latents as
//     x' = a*x + b*eps + c*x0 + d*x0_prev + s*xi,   eps = eps_u + g*(eps_c - eps_u),   x0 = x - sigma*eps
// with per-step scalars read from a device coefficient row (layout: the kCoef* indices below), so a CUDA graph captured
// once sees each step's values after a small copy into the row.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <curand_kernel.h>
#include <stdint.h>

namespace pww {
namespace smp {

// Coefficient row (fp32), shared with paint_with_words_sd_b200/pipeline.py.
enum : int {
  kCoefSigma = 0, kCoefCin = 1, kCoefT = 2, kCoefA = 3, kCoefB = 4, kCoefC = 5, kCoefD = 6, kCoefS = 7,
  kCoefG = 8, kCoefStep = 9, kCoefRow = 12
};

// Four standard normals for elements 4*group .. 4*group+3 of one image's latent at one step: Philox4x32-10 keyed by
// the image seed, counter (group, step), two Box-Muller pairs.  A pure function of (seed, step, element), so the noise
// does not depend on the image's position in a batch or on the GPU.
__device__ __forceinline__ float4 normal4(uint64_t seed, uint32_t step, uint64_t group) {
  const uint4 ctr = make_uint4((uint32_t)group, (uint32_t)(group >> 32), step, 0u);
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  const uint4 r = curand_Philox4x32_10(ctr, key);
  const float2 n0 = _curand_box_muller(r.x, r.y);
  const float2 n1 = _curand_box_muller(r.z, r.w);
  return make_float4(n0.x, n0.y, n1.x, n1.y);
}

__global__ void randn_kernel(float* __restrict__ out, long long n, uint64_t seed, uint32_t step) {
  const long long groups = (n + 3) >> 2;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (long long)gridDim.x * blockDim.x) {
    const float4 zv = normal4(seed, step, (uint64_t)g);
    const long long e = g << 2;
    if (e + 3 < n && ((reinterpret_cast<uintptr_t>(out) & 15u) == 0)) {
      reinterpret_cast<float4*>(out)[g] = zv;
    } else {
      const float z[4] = {zv.x, zv.y, zv.z, zv.w};
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (e + j < n) out[e + j] = z[j];
    }
  }
}

// UNet input of one step: out[n, y, x, ch] (channels-last [2m, C+Ce, H, W] fp16) for n < 2m, image b = n mod m:
// ch < C: fp16(c_in * latents[b, ch, y, x]);  else fp16(extra[b, ch - C, y, x]).
// One thread per (image, 4 consecutive pixels); it writes the cond and the uncond copy.
struct PrepareParams {
  const float* lat;    // [m, C, HW] fp32
  const float* extra;  // [m, Ce, HW] fp32 or null
  const float* coef;
  __half* out;         // [2m, HW, C + Ce] fp16
  int m, C, Ce;
  long long HW;
  bool vec_in;         // 16-byte loads of 4 pixels (HW % 4 == 0, 16-byte aligned inputs)
  bool vec_out;        // 16-byte stores (CT even, 16-byte aligned out, HW % 4 == 0)
};

constexpr int kMaxPrepChannels = 16;

template <int CT>   // C + Ce, a compile-time constant so the staged pixels stay in registers
__global__ void prepare_kernel(const PrepareParams p) {
  const long long quads = (p.HW + 3) >> 2;
  const long long total = (long long)p.m * quads;
  const float cin = p.coef[kCoefCin];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / quads);
    const long long px0 = (i - (long long)b * quads) << 2;
    const int npx = (p.HW - px0) < 4 ? (int)(p.HW - px0) : 4;
    __align__(16) __half v[4 * CT];
#pragma unroll
    for (int ch = 0; ch < CT; ++ch) {
      const bool lat = ch < p.C;
      const float* src = lat ? p.lat + ((long long)b * p.C + ch) * p.HW
                             : p.extra + ((long long)b * p.Ce + (ch - p.C)) * p.HW;
      float f[4] = {0.f, 0.f, 0.f, 0.f};
      if (p.vec_in) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(src + px0));
        f[0] = q.x; f[1] = q.y; f[2] = q.z; f[3] = q.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j < npx) f[j] = __ldg(src + px0 + j);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j * CT + ch] = __float2half_rn(lat ? __fmul_rn(f[j], cin) : f[j]);
    }
#pragma unroll
    for (int copy = 0; copy < 2; ++copy) {
      __half* dst = p.out + (((long long)(b + copy * p.m)) * p.HW + px0) * CT;
      if (p.vec_out) {
#pragma unroll
        for (int k = 0; k < (4 * CT) / 8; ++k) reinterpret_cast<uint4*>(dst)[k] = reinterpret_cast<const uint4*>(v)[k];
      } else {
#pragma unroll
        for (int k = 0; k < 4 * CT; ++k)
          if (k < npx * CT) dst[k] = v[k];
      }
    }
  }
}

// CFG combine + sampler update over the latents [m, C, H, W] fp32 (NCHW contiguous), in place, and x0_prev <- x0.
// eps is [2m, C, H, W] fp16 at element strides (sn, sc, sh, sw): rows 0..m-1 cond, m..2m-1 uncond.
struct StepParams {
  const __half* eps;
  long long sn, sc, sh, sw;
  float* lat;
  float* x0p;
  const float* coef;
  const unsigned long long* seeds;  // [m]
  float guidance;
  int m, C, H, W;
  long long chw;                    // C*H*W
  bool vec;                         // chw % 4 == 0 and lat / x0p 16-byte aligned
};

__device__ __forceinline__ float eps_at(const StepParams& p, long long n, long long e) {
  const long long hw = (long long)p.H * p.W;
  const long long c = e / hw;
  const long long r = e - c * hw;
  const long long y = r / p.W;
  const long long x = r - y * p.W;
  return __half2float(p.eps[n * p.sn + c * p.sc + y * p.sh + x * p.sw]);
}

__global__ void step_kernel(const StepParams p) {
  const float sigma = p.coef[kCoefSigma], ca = p.coef[kCoefA], cb = p.coef[kCoefB], cc = p.coef[kCoefC];
  const float cd = p.coef[kCoefD], cs = p.coef[kCoefS];
  const uint32_t step = (uint32_t)p.coef[kCoefStep];
  const long long groups = (p.chw + 3) >> 2;
  const long long total = (long long)p.m * groups;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / groups);
    const long long g = i - (long long)b * groups;
    const long long e0 = g << 2;
    const int ne = (p.chw - e0) < 4 ? (int)(p.chw - e0) : 4;
    const long long base = (long long)b * p.chw + e0;
    float x[4] = {0.f, 0.f, 0.f, 0.f}, xp[4] = {0.f, 0.f, 0.f, 0.f};
    if (p.vec) {
      const float4 a = reinterpret_cast<const float4*>(p.lat + base)[0];
      const float4 q = reinterpret_cast<const float4*>(p.x0p + base)[0];
      x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w;
      xp[0] = q.x; xp[1] = q.y; xp[2] = q.z; xp[3] = q.w;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < ne) { x[j] = p.lat[base + j]; xp[j] = p.x0p[base + j]; }
    }
    float4 zv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (cs != 0.f) zv = normal4(p.seeds[b], step, (uint64_t)g);
    const float z[4] = {zv.x, zv.y, zv.z, zv.w};
    float xo[4], x0o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      xo[j] = 0.f; x0o[j] = 0.f;
      if (j < ne) {
        const float ec = eps_at(p, b, e0 + j), eu = eps_at(p, (long long)b + p.m, e0 + j);
        const float ehat = eu + p.guidance * (ec - eu);
        const float x0 = x[j] - sigma * ehat;
        x0o[j] = x0;
        xo[j] = ca * x[j] + cb * ehat + cc * x0 + cd * xp[j] + cs * z[j];
      }
    }
    if (p.vec) {
      reinterpret_cast<float4*>(p.lat + base)[0] = make_float4(xo[0], xo[1], xo[2], xo[3]);
      reinterpret_cast<float4*>(p.x0p + base)[0] = make_float4(x0o[0], x0o[1], x0o[2], x0o[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < ne) { p.lat[base + j] = xo[j]; p.x0p[base + j] = x0o[j]; }
    }
  }
}

}  // namespace smp
}  // namespace pww
