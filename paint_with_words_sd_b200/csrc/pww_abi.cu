// extern "C" entry points of libpww_b200.so (declared in include/pww_b200.h).
#include <stdio.h>
#include <string.h>

#include "pww_common.cuh"
#include "xattn_tc.cuh"
#include "xattn_fused.cuh"
#include "xattn_fused2.cuh"
#include "attn_tc.cuh"
#include "unet_ops.cuh"
#include "sampler.cuh"
#include <stdlib.h>

namespace {

thread_local char g_last_cuda_error[640] = "";

int cuda_fail(cudaError_t e);

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

bool aligned4(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; }

// Grid of an elementwise grid-stride kernel over `work` items, 256 threads a block.
unsigned elementwise_grid(long long work) {
  long long blocks = (work + 255) / 256;
  const long long cap = (long long)pww::tc::num_sms() * 8;
  if (blocks > cap) blocks = cap;
  return (unsigned)(blocks < 1 ? 1 : blocks);
}

bool supported_head_dim(int D) { return D == 40 || D == 64 || D == 80 || D == 160; }

int check_common(const void* q, const void* k, int B, int H, int N, int T, int D, int64_t q_bs, int64_t q_rs,
                 int64_t k_bs, int64_t k_rs) {
  if (!q || !k || B <= 0 || H <= 0 || N <= 0 || T <= 0 || D <= 0) return PWW_ERR_BAD_ARG;
  if (!aligned16(q) || !aligned16(k)) return PWW_ERR_BAD_ARG;
  if ((q_bs | q_rs | k_bs | k_rs) & 7) return PWW_ERR_BAD_ARG;  // 16-byte vector access on rows
  if (q_rs < (int64_t)H * D || k_rs < (int64_t)H * D) return PWW_ERR_BAD_ARG;
  if (!supported_head_dim(D) || T > pww::tc::kTP) return PWW_ERR_UNSUPPORTED;
  return PWW_OK;
}

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Partial slots reserved per image (one per CTA of the persistent grid; device independent upper bound so the size
// can be computed without a GPU).
int stats_slots_per_image(int, int) { return 2048; }

int cuda_fail(cudaError_t e) {
  snprintf(g_last_cuda_error, sizeof(g_last_cuda_error), "%s: %s %s", cudaGetErrorName(e), cudaGetErrorString(e),
           pww::tc::tc_error_buf());
  pww::tc::tc_error_buf()[0] = 0;
  return PWW_ERR_CUDA;
}

}  // namespace

extern "C" {

int pww_version(void) { return 100; }  // 0.1.0

const char* pww_status_str(int status) {
  switch (status) {
    case PWW_OK: return "ok";
    case PWW_ERR_BAD_ARG: return "bad argument (null/misaligned pointer, non-positive size or stride not a multiple of 8)";
    case PWW_ERR_UNSUPPORTED: return "unsupported shape (head dim must be 40/64/80/160, T <= 80)";
    case PWW_ERR_CUDA: return "CUDA error (see pww_last_cuda_error)";
    case PWW_ERR_WORKSPACE: return "workspace too small (see pww_xattn_workspace_bytes)";
    default: return "unknown status";
  }
}

const char* pww_last_cuda_error(void) { return g_last_cuda_error; }

int pww_device_supported(void) {
  int dev = 0, major = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e);
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return cuda_fail(e);
  return major == 10 ? 1 : 0;
}

size_t pww_xattn_workspace_bytes(int B, int H, int N, int T, int D) {
  (void)T; (void)D;
  if (B <= 0 || H <= 0 || N <= 0) return 0;
  return align_up((size_t)B * sizeof(unsigned int), 256) +
         (size_t)B * stats_slots_per_image(H, N) * sizeof(pww::StatPartial);
}

int pww_xattn_stats_f16(const void* q, const void* k, int B, int H, int N, int T, int D, int64_t q_batch_stride,
                        int64_t q_row_stride, int64_t k_batch_stride, int64_t k_row_stride, int stat,
                        const int32_t* wmap_index, float* stats, void* workspace, size_t workspace_bytes,
                        void* stream) {
  int rc = check_common(q, k, B, H, N, T, D, q_batch_stride, q_row_stride, k_batch_stride, k_row_stride);
  if (rc) return rc;
  if (!stats || !workspace || (stat != PWW_STAT_MAX && stat != PWW_STAT_STD)) return PWW_ERR_BAD_ARG;
  if (workspace_bytes < pww_xattn_workspace_bytes(B, H, N, T, D)) return PWW_ERR_WORKSPACE;
  pww::XattnParams p;
  memset(&p, 0, sizeof(p));
  p.q = (const __half*)q; p.k = (const __half*)k;
  p.B = B; p.H = H; p.N = N; p.T = T; p.D = D;
  p.q_bs = q_batch_stride; p.q_rs = q_row_stride; p.k_bs = k_batch_stride; p.k_rs = k_row_stride;
  p.wmap_index = wmap_index; p.stat = stat; p.stats_out = stats;
  p.counters = (unsigned int*)workspace;
  p.partials = (pww::StatPartial*)((char*)workspace + align_up((size_t)B * sizeof(unsigned int), 256));
  cudaStream_t s = (cudaStream_t)stream;
  {
    if (pww::tc::stats_slots() > stats_slots_per_image(H, N)) return PWW_ERR_WORKSPACE;
    for (int b0 = 0; b0 < B; b0 += pww::tc::kMaxBatch) {          // <= 256 images per launch
      pww::XattnParams c = p;
      c.B = (B - b0) < pww::tc::kMaxBatch ? (B - b0) : pww::tc::kMaxBatch;
      c.q = p.q + (int64_t)b0 * p.q_bs;
      c.k = p.k + (int64_t)b0 * p.k_bs;
      c.wmap_index = p.wmap_index ? p.wmap_index + b0 : nullptr;
      c.stats_out = p.stats_out + b0;
      cudaError_t e = cudaErrorInvalidValue;
      switch (D) {
        case 40: e = pww::tc::launch_stats<40>(c, s); break;
        case 64: e = pww::tc::launch_stats<64>(c, s); break;
        case 80: e = pww::tc::launch_stats<80>(c, s); break;
        case 160: e = pww::tc::launch_stats<160>(c, s); break;
      }
      if (e != cudaSuccess) return cuda_fail(e);
    }
    return PWW_OK;
  }
}

int pww_xattn_fwd_f16(const void* q, const void* k, const void* v, void* out, int B, int H, int N, int T, int D,
                      int64_t q_batch_stride, int64_t q_row_stride, int64_t k_batch_stride, int64_t k_row_stride,
                      int64_t o_batch_stride, int64_t o_row_stride, const float* wmap, int64_t wmap_batch_stride,
                      const int32_t* wmap_index, const float* stats, const float* g_sigma, float scale,
                      void* stream) {
  int rc = check_common(q, k, B, H, N, T, D, q_batch_stride, q_row_stride, k_batch_stride, k_row_stride);
  if (rc) return rc;
  if (!v || !out || !aligned16(v) || !aligned16(out)) return PWW_ERR_BAD_ARG;
  if ((o_batch_stride | o_row_stride) & 7 || o_row_stride < (int64_t)H * D) return PWW_ERR_BAD_ARG;
  if (wmap && (!stats || !g_sigma)) return PWW_ERR_BAD_ARG;
  pww::XattnParams p;
  memset(&p, 0, sizeof(p));
  p.q = (const __half*)q; p.k = (const __half*)k; p.v = (const __half*)v; p.out = (__half*)out;
  p.B = B; p.H = H; p.N = N; p.T = T; p.D = D;
  p.q_bs = q_batch_stride; p.q_rs = q_row_stride; p.k_bs = k_batch_stride; p.k_rs = k_row_stride;
  p.o_bs = o_batch_stride; p.o_rs = o_row_stride;
  p.wmap = wmap; p.wmap_bs = wmap_batch_stride; p.wmap_index = wmap_index;
  p.stats = stats; p.g_sigma = g_sigma; p.scale = scale;
  cudaStream_t s = (cudaStream_t)stream;
  {
    for (int b0 = 0; b0 < B; b0 += pww::tc::kMaxBatch) {          // <= 256 images per launch
      pww::XattnParams c = p;
      c.B = (B - b0) < pww::tc::kMaxBatch ? (B - b0) : pww::tc::kMaxBatch;
      c.q = p.q + (int64_t)b0 * p.q_bs;
      c.k = p.k + (int64_t)b0 * p.k_bs;
      c.v = p.v + (int64_t)b0 * p.k_bs;
      c.out = p.out + (int64_t)b0 * p.o_bs;
      c.wmap_index = (p.wmap && p.wmap_index) ? p.wmap_index + b0 : nullptr;
      c.stats = p.stats ? p.stats + b0 : nullptr;
      if (p.wmap && !p.wmap_index) c.wmap = p.wmap + (int64_t)b0 * p.wmap_bs;   // identity mapping
      cudaError_t e = cudaErrorInvalidValue;
      switch (D) {
        case 40: e = pww::tc::launch_fwd<40>(c, s); break;
        case 64: e = pww::tc::launch_fwd<64>(c, s); break;
        case 80: e = pww::tc::launch_fwd<80>(c, s); break;
        case 160: e = pww::tc::launch_fwd<160>(c, s); break;
      }
      if (e != cudaSuccess) return cuda_fail(e);
    }
    return PWW_OK;
  }
}

size_t pww_xattn_fused_workspace_bytes(void) { return pww::fx::fused_workspace_bytes(); }

int pww_xattn_fused_f16(const void* q, const void* k, const void* v, void* out, int B, int H, int N, int T, int D,
                        int64_t q_batch_stride, int64_t q_row_stride, int64_t k_batch_stride, int64_t k_row_stride,
                        int64_t o_batch_stride, int64_t o_row_stride, const void* mpack, int64_t mpack_batch_stride,
                        int Bw, const int8_t* cidx, const int32_t* wmap_index, int stat, const float* g_sigma,
                        float scale, float* stats, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_common(q, k, B, H, N, T, D, q_batch_stride, q_row_stride, k_batch_stride, k_row_stride);
  if (rc) return rc;
  if (!v || !out || !aligned16(v) || !aligned16(out)) return PWW_ERR_BAD_ARG;
  if ((o_batch_stride | o_row_stride) & 7 || o_row_stride < (int64_t)H * D || o_batch_stride <= 0) return PWW_ERR_BAD_ARG;
  if (mpack) {
    if (!cidx || !g_sigma || !workspace || Bw <= 0 || !aligned16(mpack)) return PWW_ERR_BAD_ARG;
    if ((mpack_batch_stride & 7) || mpack_batch_stride < (int64_t)N * pww::fx::kMW) return PWW_ERR_BAD_ARG;
    if (stat != PWW_STAT_MAX && stat != PWW_STAT_STD) return PWW_ERR_BAD_ARG;
    if (workspace_bytes < pww_xattn_fused_workspace_bytes()) return PWW_ERR_WORKSPACE;
  }
  pww::XattnParams p;
  memset(&p, 0, sizeof(p));
  p.q = (const __half*)q; p.k = (const __half*)k; p.v = (const __half*)v; p.out = (__half*)out;
  p.B = B; p.H = H; p.N = N; p.T = T; p.D = D;
  p.q_bs = q_batch_stride; p.q_rs = q_row_stride; p.k_bs = k_batch_stride; p.k_rs = k_row_stride;
  p.o_bs = o_batch_stride; p.o_rs = o_row_stride;
  p.g_sigma = g_sigma; p.scale = scale; p.stat = stat;
  p.counters = (unsigned int*)workspace;
  p.partials = workspace ? (pww::StatPartial*)((char*)workspace + 512) : nullptr;   // header: counters @0, per-image maxima @256
  cudaStream_t s = (cudaStream_t)stream;
  // image b is biased iff it has a packed map: with mpack == NULL every index is -1 (the kernel reads wmap_index)
  int chunk = pww::fx::kMaxBatch;                                  // images per launch
  {                                                                // job table of <= 64 units per CTA
    const int tiles = pww::ceil_div(N, pww::fx::kBM);
    const int hg = pww::ceil_div(H, D == 40 ? pww::fx2::Cfg2<40>::G : (D == 64 ? pww::fx2::Cfg2<64>::G : 1));
    while (chunk > 1) {
      const int cb = B < chunk ? B : chunk;
      if (pww::fx2::fused2_fits(cb, hg, tiles, pww::fx::fused_grid(cb * hg * tiles))) break;
      chunk >>= 1;
    }
  }
  for (int b0 = 0; b0 < B; b0 += chunk) {
    pww::XattnParams c = p;
    c.B = (B - b0) < chunk ? (B - b0) : chunk;
    c.q = p.q + (int64_t)b0 * p.q_bs;
    c.k = p.k + (int64_t)b0 * p.k_bs;
    c.v = p.v + (int64_t)b0 * p.k_bs;
    c.out = p.out + (int64_t)b0 * p.o_bs;
    c.stats_out = stats ? stats + b0 : nullptr;
    const void* mp = mpack;
    const int8_t* ci = cidx;
    if (mpack && wmap_index) {
      c.wmap_index = wmap_index + b0;
    } else if (mpack) {                                            // identity mapping: image b uses map b
      c.wmap_index = nullptr;
      mp = (const __half*)mpack + (int64_t)b0 * mpack_batch_stride;
      ci = cidx + (int64_t)b0 * pww::fx::kTP;
    }
    c.wmap = mpack ? (const float*)mp : nullptr;                   // non-null marks "maps present" for the kernel
    cudaError_t e = cudaErrorInvalidValue;
    switch (D) {
      case 40: e = pww::fx2::launch_fused2<40>(c, mp, mpack_batch_stride, Bw, ci, s); break;
      case 64: e = pww::fx2::launch_fused2<64>(c, mp, mpack_batch_stride, Bw, ci, s); break;
      case 80: e = pww::fx2::launch_fused2<80>(c, mp, mpack_batch_stride, Bw, ci, s); break;
      case 160: e = pww::fx2::launch_fused2<160>(c, mp, mpack_batch_stride, Bw, ci, s); break;
    }
    if (e == cudaErrorInvalidConfiguration) return PWW_ERR_UNSUPPORTED;
    if (e != cudaSuccess) return cuda_fail(e);
  }
  return PWW_OK;
}

size_t pww_groupnorm_workspace_bytes(int B, int HW, int G) {
  if (B <= 0 || HW <= 0 || G <= 0) return 0;
  return align_up((size_t)B * sizeof(unsigned int), 256) + align_up((size_t)B * G * 2 * sizeof(float), 256) +
         (size_t)B * pww::uops::gn_chunks(HW) * G * 2 * sizeof(float);
}

int pww_groupnorm_nhwc_f16(const void* x, const void* add, int64_t add_batch_stride, const void* gamma, const void* beta,
                           void* y, int B, int HW, int C, int G, float eps, int silu, void* workspace,
                           size_t workspace_bytes, void* stream) {
  if (!x || !gamma || !beta || !y || !workspace || B <= 0 || HW <= 0 || C <= 0 || G <= 0) return PWW_ERR_BAD_ARG;
  if (!aligned16(x) || !aligned16(y) || !aligned16(gamma) || !aligned16(beta) || (add && !aligned16(add)))
    return PWW_ERR_BAD_ARG;
  if ((C & 7) || (C % G) || G > 64 || (C >> 3) > 1024) return PWW_ERR_UNSUPPORTED;
  if (add && ((add_batch_stride & 7) || add_batch_stride < C)) return PWW_ERR_BAD_ARG;
  if (workspace_bytes < pww_groupnorm_workspace_bytes(B, HW, G)) return PWW_ERR_WORKSPACE;
  pww::uops::GnParams p;
  p.x = (const __half*)x; p.add = (const __half*)add; p.add_bs = add_batch_stride; p.gamma = (const __half*)gamma; p.beta = (const __half*)beta;
  p.y = (__half*)y;
  char* w = (char*)workspace;
  p.counters = (unsigned int*)w;
  w += align_up((size_t)B * sizeof(unsigned int), 256);
  p.stats = (float*)w;
  w += align_up((size_t)B * G * 2 * sizeof(float), 256);
  p.partial = (float*)w;
  p.B = B; p.HW = HW; p.C = C; p.G = G; p.eps = eps; p.silu = silu;
  p.chunks = pww::uops::gn_chunks(HW);
  p.rows_per_chunk = (HW + p.chunks - 1) / p.chunks;
  cudaStream_t s = (cudaStream_t)stream;
  const int nvec = C >> 3;
  const int rpp = nvec >= 256 ? 1 : 256 / nvec;
  const size_t smem1 = (size_t)rpp * C * 2 * sizeof(float);
  if (smem1 > 48 * 1024) return PWW_ERR_UNSUPPORTED;
  pww::uops::gn_stats_kernel<<<dim3(p.chunks, B), nvec * rpp, smem1, s>>>(p);
  // enough row chunks to fill the machine even at 8x8 resolution
  int rows_per_block = (int)(((long long)HW * B + 2 * pww::tc::num_sms() - 1) / (2 * pww::tc::num_sms()));
  if (rows_per_block < rpp) rows_per_block = rpp;
  if (rows_per_block > 32) rows_per_block = 32;
  pww::uops::gn_apply_kernel<<<dim3((HW + rows_per_block - 1) / rows_per_block, B), nvec * rpp, 0, s>>>(p, rows_per_block);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PWW_OK : cuda_fail(e);
}

int pww_geglu_f16(const void* in, void* out, int64_t M, int I, void* stream) {
  if (!in || !out || M <= 0 || I <= 0 || !aligned16(in) || !aligned16(out)) return PWW_ERR_BAD_ARG;
  if (I & 7) return PWW_ERR_UNSUPPORTED;
  const long long total = (long long)M * (I >> 3);
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)pww::tc::num_sms() * 16;
  if (blocks > cap) blocks = cap;
  pww::uops::geglu_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((const __half*)in, (__half*)out, M, I);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PWW_OK : cuda_fail(e);
}

int pww_add_layernorm_f16(const void* x, const void* res, const void* gamma, const void* beta, void* sum_out, void* y,
                          int64_t M, int C, float eps, void* stream) {
  if (!x || !gamma || !beta || !y || M <= 0 || C <= 0) return PWW_ERR_BAD_ARG;
  if (!aligned16(x) || !aligned16(y) || !aligned16(gamma) || !aligned16(beta) || (res && !aligned16(res)) ||
      (sum_out && !aligned16(sum_out)))
    return PWW_ERR_BAD_ARG;
  if ((C & 7) || C > 2048) return PWW_ERR_UNSUPPORTED;
  const int vpl = ((C >> 3) + 31) / 32;
  const int warps = 8;
  const unsigned grid = (unsigned)((M + warps - 1) / warps);
  cudaStream_t s = (cudaStream_t)stream;
  const __half *xp = (const __half*)x, *rp = (const __half*)res, *gp = (const __half*)gamma, *bp = (const __half*)beta;
  __half *sp = (__half*)sum_out, *yp = (__half*)y;
  switch (vpl) {
    case 1: pww::uops::add_layernorm_kernel<1><<<grid, warps * 32, 0, s>>>(xp, rp, gp, bp, sp, yp, M, C, eps); break;
    case 2: pww::uops::add_layernorm_kernel<2><<<grid, warps * 32, 0, s>>>(xp, rp, gp, bp, sp, yp, M, C, eps); break;
    case 3: pww::uops::add_layernorm_kernel<3><<<grid, warps * 32, 0, s>>>(xp, rp, gp, bp, sp, yp, M, C, eps); break;
    case 4: pww::uops::add_layernorm_kernel<4><<<grid, warps * 32, 0, s>>>(xp, rp, gp, bp, sp, yp, M, C, eps); break;
    case 5: pww::uops::add_layernorm_kernel<5><<<grid, warps * 32, 0, s>>>(xp, rp, gp, bp, sp, yp, M, C, eps); break;
    case 6: pww::uops::add_layernorm_kernel<6><<<grid, warps * 32, 0, s>>>(xp, rp, gp, bp, sp, yp, M, C, eps); break;
    case 7: pww::uops::add_layernorm_kernel<7><<<grid, warps * 32, 0, s>>>(xp, rp, gp, bp, sp, yp, M, C, eps); break;
    case 8: pww::uops::add_layernorm_kernel<8><<<grid, warps * 32, 0, s>>>(xp, rp, gp, bp, sp, yp, M, C, eps); break;
    default: return PWW_ERR_UNSUPPORTED;
  }
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PWW_OK : cuda_fail(e);
}

// Test infrastructure (not declared in the public header): point the kernels' debug timeline at a device buffer of
// kTlTags*kTlIts int64 clock64 stamps [tag][iteration] written by CTA 0; pass NULL to disable.
int pww_debug_set_timeline(void* device_buffer) {
  pww::tc::debug_timeline() = (long long*)device_buffer;
  return PWW_OK;
}

// Test infrastructure (not declared in the public header): structure of the tcgen05 forward kernel, for A/B timing.
// 0 = per-thread global stores, 1 = TMA-store epilogue at D = 40 (default), 3 = TMA-store epilogue at every head dim
// (see xattn_tc.cuh).
int pww_debug_set_variant(int variant) {
  if (variant != 0 && variant != 1 && variant != 3) return PWW_ERR_BAD_ARG;
  pww::tc::fwd_variant() = variant;
  return PWW_OK;
}

// Test infrastructure (not declared in the public header): replay the forward kernel's unit schedule on the host.
// wmap_index and out are HOST pointers; out receives 8 int32 per unit (see fwd_schedule_host); returns the number of
// units written or a negative value for bad arguments.  No GPU needed.
int pww_debug_fwd_schedule(int B, int H, int tiles, int grid, const int* wmap_index, int* out) {
  if (!wmap_index || !out) return PWW_ERR_BAD_ARG;
  return pww::tc::fwd_schedule_host(B, H, tiles, grid, wmap_index, out);
}

// Test infrastructure (not declared in the public header): cap the persistent grid of the fused kernel (0 = all SMs) so
// small shapes exercise long job lists; does CTA `cta` contribute a partial to image b's statistic (H = head GROUPS)?
int pww_debug_set_fused_grid(int grid) {
  pww::fx::debug_grid() = grid < 0 ? 0 : grid;
  return PWW_OK;
}
// Test infrastructure: clock64 timeline of one CTA of the fused kernel ([16][64] int64 device buffer, NULL = off).
int pww_debug_set_fused_timeline(void* device_buffer, int cta) {
  pww::fx::debug_timeline() = (long long*)device_buffer;
  pww::fx::debug_timeline_cta() = cta;
  return PWW_OK;
}
// Host replay of the grouped-head kernel's job lists (14 int32 per job, see fused2_schedule_host).
int pww_debug_fused2_schedule(int B, int H, int G, int tiles, int grid, const int* wmap_index, int* out, int max_jobs) {
  if (!wmap_index || !out) return PWW_ERR_BAD_ARG;
  return pww::fx2::fused2_schedule_host(B, H, G, tiles, grid, wmap_index, out, max_jobs);
}
// Test infrastructure: device buffer of grid * (2 + 1024) uint32 the grouped-head kernel copies every CTA's job table to.
// Heads per unit of the grouped-head kernel (a build-time constant).
int pww_debug_fused2_heads_per_unit(void) { return pww::fx2::Cfg2<40>::G; }
int pww_debug_set_fused_jobs_dump(void* device_buffer) {
  pww::fx::debug_jobs_dump() = (unsigned*)device_buffer;
  return PWW_OK;
}
int pww_debug_fused_cta_has_image(int cta, int grid, int B, int H, int tiles, const int* wmap_index, int b) {
  if (!wmap_index) return PWW_ERR_BAD_ARG;
  return pww::fx::fused_cta_has_image_host(cta, grid, B, H, tiles, wmap_index, b);
}

int pww_attn_fwd_f16(const void* q, const void* k, const void* v, void* out, int B, int H, int N, int D,
                     int64_t qkv_batch_stride, int64_t qkv_row_stride, int64_t o_batch_stride, int64_t o_row_stride,
                     float scale, void* stream) {
  if (!q || !k || !v || !out || B <= 0 || H <= 0 || N <= 0 || D <= 0) return PWW_ERR_BAD_ARG;
  if (!aligned16(q) || !aligned16(k) || !aligned16(v) || !aligned16(out)) return PWW_ERR_BAD_ARG;
  if ((qkv_batch_stride | qkv_row_stride | o_batch_stride | o_row_stride) & 7) return PWW_ERR_BAD_ARG;
  if (qkv_row_stride < (int64_t)H * D || o_row_stride < (int64_t)H * D) return PWW_ERR_BAD_ARG;
  if (!supported_head_dim(D)) return PWW_ERR_UNSUPPORTED;
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaErrorInvalidValue;
  switch (D) {
    case 40: e = pww::fa::launch<40>(q, k, v, out, B, H, N, qkv_batch_stride, qkv_row_stride, o_batch_stride, o_row_stride, scale, s); break;
    case 64: e = pww::fa::launch<64>(q, k, v, out, B, H, N, qkv_batch_stride, qkv_row_stride, o_batch_stride, o_row_stride, scale, s); break;
    case 80: e = pww::fa::launch<80>(q, k, v, out, B, H, N, qkv_batch_stride, qkv_row_stride, o_batch_stride, o_row_stride, scale, s); break;
    case 160: e = pww::fa::launch<160>(q, k, v, out, B, H, N, qkv_batch_stride, qkv_row_stride, o_batch_stride, o_row_stride, scale, s); break;
  }
  return e == cudaSuccess ? PWW_OK : cuda_fail(e);
}

int pww_sampler_prepare_f16(const float* latents, const float* extra, const float* coef, void* out, int m, int C, int Ce,
                            int H, int W, void* stream) {
  if (!latents || !coef || !out || m <= 0 || C <= 0 || Ce < 0 || H <= 0 || W <= 0) return PWW_ERR_BAD_ARG;
  if ((Ce > 0) != (extra != nullptr)) return PWW_ERR_BAD_ARG;
  if (!aligned4(latents) || !aligned4(coef) || (extra && !aligned4(extra)) || (reinterpret_cast<uintptr_t>(out) & 1u))
    return PWW_ERR_BAD_ARG;
  const int Ct = C + Ce;
  const long long HW = (long long)H * W;
  if (Ct > pww::smp::kMaxPrepChannels || HW > (1LL << 40) || (long long)m > (1LL << 20)) return PWW_ERR_UNSUPPORTED;
  pww::smp::PrepareParams p;
  p.lat = latents; p.extra = extra; p.coef = coef; p.out = (__half*)out;
  p.m = m; p.C = C; p.Ce = Ce; p.HW = HW;
  p.vec_in = (HW % 4) == 0 && aligned16(latents) && (!extra || aligned16(extra));
  p.vec_out = (HW % 4) == 0 && (Ct % 2) == 0 && aligned16(out);
  const unsigned grid = elementwise_grid((long long)m * ((HW + 3) / 4));
  cudaStream_t s = (cudaStream_t)stream;
  switch (Ct) {
#define PWW_PREP_CASE(n) case n: pww::smp::prepare_kernel<n><<<grid, 256, 0, s>>>(p); break;
    PWW_PREP_CASE(1) PWW_PREP_CASE(2) PWW_PREP_CASE(3) PWW_PREP_CASE(4) PWW_PREP_CASE(5) PWW_PREP_CASE(6)
    PWW_PREP_CASE(7) PWW_PREP_CASE(8) PWW_PREP_CASE(9) PWW_PREP_CASE(10) PWW_PREP_CASE(11) PWW_PREP_CASE(12)
    PWW_PREP_CASE(13) PWW_PREP_CASE(14) PWW_PREP_CASE(15) PWW_PREP_CASE(16)
#undef PWW_PREP_CASE
    default: return PWW_ERR_UNSUPPORTED;
  }
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PWW_OK : cuda_fail(e);
}

int pww_sampler_step_f32(const void* eps, int64_t eps_n_stride, int64_t eps_c_stride, int64_t eps_h_stride,
                         int64_t eps_w_stride, float* latents, float* x0_prev, const float* coef, const uint64_t* seeds,
                         float guidance_scale, int m, int C, int H, int W, void* stream) {
  if (!eps || !latents || !x0_prev || !coef || !seeds || m <= 0 || C <= 0 || H <= 0 || W <= 0) return PWW_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(eps) & 1u) || !aligned4(latents) || !aligned4(x0_prev) || !aligned4(coef) ||
      (reinterpret_cast<uintptr_t>(seeds) & 7u))
    return PWW_ERR_BAD_ARG;
  if (eps_n_stride <= 0 || eps_c_stride <= 0 || eps_h_stride <= 0 || eps_w_stride <= 0) return PWW_ERR_BAD_ARG;
  const long long chw = (long long)C * H * W;
  if (chw > (1LL << 40) || (long long)m > (1LL << 20)) return PWW_ERR_UNSUPPORTED;
  pww::smp::StepParams p;
  p.eps = (const __half*)eps;
  p.sn = eps_n_stride; p.sc = eps_c_stride; p.sh = eps_h_stride; p.sw = eps_w_stride;
  p.lat = latents; p.x0p = x0_prev; p.coef = coef; p.seeds = (const unsigned long long*)seeds;
  p.guidance = guidance_scale;
  p.m = m; p.C = C; p.H = H; p.W = W; p.chw = chw;
  p.vec = (chw % 4) == 0 && aligned16(latents) && aligned16(x0_prev);
  pww::smp::step_kernel<<<elementwise_grid((long long)m * ((chw + 3) / 4)), 256, 0, (cudaStream_t)stream>>>(p);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PWW_OK : cuda_fail(e);
}

int pww_randn_f32(float* out, int64_t n, uint64_t seed, int step, void* stream) {
  if (!out || n <= 0 || step < 0 || !aligned4(out)) return PWW_ERR_BAD_ARG;
  if (n > (1LL << 42)) return PWW_ERR_UNSUPPORTED;
  pww::smp::randn_kernel<<<elementwise_grid((n + 3) / 4), 256, 0, (cudaStream_t)stream>>>(out, n, seed, (uint32_t)step);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PWW_OK : cuda_fail(e);
}

}  // extern "C"
