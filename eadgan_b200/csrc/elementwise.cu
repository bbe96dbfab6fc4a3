// Pointwise activations, row softmax, nearest 2x upsample, fill, and the error /
// version plumbing of the C ABI.  All kernels are HBM-bound streaming passes:
// 128-bit vectorised loads/stores, grid sized to a multiple of the SM count.
// Reference call sites: nn.LeakyReLU / nn.ReLU / nn.Tanh / F.sigmoid / F.softmax /
// nn.Softmax / nn.Upsample in celebA/EAD-GAN_celebA.py:80-92,111-134,
// dSprites/rp.py:67-183, MNIST/EAD-GAN_rpqmnxy.py:81-91,107,161.
#include <stdarg.h>

#include <atomic>
#include <string.h>

#include "common.cuh"

// ---------------------------------------------------------------------------
static thread_local char g_err[512] = "";

int eadgan_set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int eg_sm_count() {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != cached_dev) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    cached = v;
    cached_dev = dev;
  }
  return cached;
}

static std::atomic<long long> g_launches{0};
void eg_count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
extern "C" int64_t eadgan_kernel_launches(void) { return (int64_t)g_launches.load(); }

extern "C" const char* eadgan_last_error(void) { return g_err; }
extern "C" int eadgan_version(void) { return EADGAN_VERSION; }
extern "C" int eadgan_sm_count(void) { return eg_sm_count(); }

namespace {

int stream_grid(int64_t work_items, int per_block) {
  int64_t b = (work_items + per_block - 1) / per_block;
  const int64_t cap = 16 * (int64_t)eg_sm_count();
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

__global__ void __launch_bounds__(256) act_fwd_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                      int64_t n, int act, float slope) {
  const int64_t n4 = n >> 2;
  const bool al = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  if (al) {
    for (int64_t i = tid; i < n4; i += nth) {
      float4 v = reinterpret_cast<const float4*>(x)[i];
      v.x = eg_act(v.x, act, slope); v.y = eg_act(v.y, act, slope);
      v.z = eg_act(v.z, act, slope); v.w = eg_act(v.w, act, slope);
      reinterpret_cast<float4*>(y)[i] = v;
    }
    for (int64_t i = (n4 << 2) + tid; i < n; i += nth) y[i] = eg_act(x[i], act, slope);
  } else {
    for (int64_t i = tid; i < n; i += nth) y[i] = eg_act(x[i], act, slope);
  }
}

__global__ void __launch_bounds__(256) act_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ y,
                                                      float* __restrict__ dx, int64_t n, int act, float slope) {
  const int64_t n4 = n >> 2;
  const bool al = ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(y) |
                    reinterpret_cast<uintptr_t>(dx)) & 15) == 0;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  if (al) {
    for (int64_t i = tid; i < n4; i += nth) {
      const float4 g = reinterpret_cast<const float4*>(dy)[i];
      const float4 o = reinterpret_cast<const float4*>(y)[i];
      float4 r;
      r.x = g.x * eg_act_grad(o.x, act, slope); r.y = g.y * eg_act_grad(o.y, act, slope);
      r.z = g.z * eg_act_grad(o.z, act, slope); r.w = g.w * eg_act_grad(o.w, act, slope);
      reinterpret_cast<float4*>(dx)[i] = r;
    }
    for (int64_t i = (n4 << 2) + tid; i < n; i += nth) dx[i] = dy[i] * eg_act_grad(y[i], act, slope);
  } else {
    for (int64_t i = tid; i < n; i += nth) dx[i] = dy[i] * eg_act_grad(y[i], act, slope);
  }
}

// one warp per row; cols small (<= 1024)
__global__ void softmax_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int rows, int cols) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + (int64_t)row * cols;
  float mx = -INFINITY;
  for (int j = lane; j < cols; j += 32) mx = fmaxf(mx, xr[j]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float s = 0.f;
  for (int j = lane; j < cols; j += 32) s += expf(xr[j] - mx);
  s = eg_warp_sum(s);
  const float inv = 1.f / s;
  for (int j = lane; j < cols; j += 32) y[(int64_t)row * cols + j] = expf(xr[j] - mx) * inv;
}

// dx = y * (dy - sum_j dy_j y_j)
__global__ void softmax_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ y,
                                   float* __restrict__ dx, int rows, int cols) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int64_t off = (int64_t)row * cols;
  float s = 0.f;
  for (int j = lane; j < cols; j += 32) s += dy[off + j] * y[off + j];
  s = eg_warp_sum(s);
  for (int j = lane; j < cols; j += 32) dx[off + j] = y[off + j] * (dy[off + j] - s);
}

__global__ void __launch_bounds__(256) upsample2x_fwd_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                             int nc, int h, int w) {
  const int64_t total = (int64_t)nc * h * w;  // one thread per INPUT element, writes 2x2
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int xx = (int)(i % w);
    const int64_t r = i / w;
    const int yy = (int)(r % h);
    const int64_t p = r / h;
    const float v = x[i];
    float* o = y + (p * (2 * h) + 2 * yy) * (int64_t)(2 * w) + 2 * xx;
    *reinterpret_cast<float2*>(o) = make_float2(v, v);
    *reinterpret_cast<float2*>(o + 2 * w) = make_float2(v, v);
  }
}

__global__ void __launch_bounds__(256) upsample2x_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx,
                                                             int nc, int h, int w) {
  const int64_t total = (int64_t)nc * h * w;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int xx = (int)(i % w);
    const int64_t r = i / w;
    const int yy = (int)(r % h);
    const int64_t p = r / h;
    const float* o = dy + (p * (2 * h) + 2 * yy) * (int64_t)(2 * w) + 2 * xx;
    const float2 a = *reinterpret_cast<const float2*>(o);
    const float2 b = *reinterpret_cast<const float2*>(o + 2 * w);
    dx[i] = (a.x + a.y) + (b.x + b.y);
  }
}

__global__ void fill_kernel(float* p, int64_t n, float v) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    p[i] = v;
}

}  // namespace

extern "C" int eadgan_act_fwd(const float* x, float* y, int64_t numel, int act, float slope, void* stream) {
  EG_REQUIRE(x && y && numel >= 0, EADGAN_ERR_INVALID, "act_fwd: bad arguments");
  if (numel == 0) return 0;
  act_fwd_kernel<<<stream_grid(numel, 1024), 256, 0, (cudaStream_t)stream>>>(x, y, numel, act, slope);
  EG_LAUNCH_CHECK("act_fwd_kernel");
  return 0;
}

extern "C" int eadgan_act_bwd(const float* dy, const float* y, float* dx, int64_t numel, int act, float slope,
                              void* stream) {
  EG_REQUIRE(dy && y && dx && numel >= 0, EADGAN_ERR_INVALID, "act_bwd: bad arguments");
  if (numel == 0) return 0;
  act_bwd_kernel<<<stream_grid(numel, 1024), 256, 0, (cudaStream_t)stream>>>(dy, y, dx, numel, act, slope);
  EG_LAUNCH_CHECK("act_bwd_kernel");
  return 0;
}

extern "C" int eadgan_softmax_fwd(const float* x, float* y, int rows, int cols, void* stream) {
  EG_REQUIRE(x && y && rows > 0 && cols > 0, EADGAN_ERR_INVALID, "softmax_fwd: bad arguments");
  softmax_fwd_kernel<<<(rows + 7) / 8, 256, 0, (cudaStream_t)stream>>>(x, y, rows, cols);
  EG_LAUNCH_CHECK("softmax_fwd_kernel");
  return 0;
}

extern "C" int eadgan_softmax_bwd(const float* dy, const float* y, float* dx, int rows, int cols, void* stream) {
  EG_REQUIRE(dy && y && dx && rows > 0 && cols > 0, EADGAN_ERR_INVALID, "softmax_bwd: bad arguments");
  softmax_bwd_kernel<<<(rows + 7) / 8, 256, 0, (cudaStream_t)stream>>>(dy, y, dx, rows, cols);
  EG_LAUNCH_CHECK("softmax_bwd_kernel");
  return 0;
}

extern "C" int eadgan_upsample2x_fwd(const float* x, float* y, int nc, int h, int w, void* stream) {
  EG_REQUIRE(x && y && nc > 0 && h > 0 && w > 0, EADGAN_ERR_INVALID, "upsample2x_fwd: bad arguments");
  upsample2x_fwd_kernel<<<stream_grid((int64_t)nc * h * w, 256), 256, 0, (cudaStream_t)stream>>>(x, y, nc, h, w);
  EG_LAUNCH_CHECK("upsample2x_fwd_kernel");
  return 0;
}

extern "C" int eadgan_upsample2x_bwd(const float* dy, float* dx, int nc, int h, int w, void* stream) {
  EG_REQUIRE(dy && dx && nc > 0 && h > 0 && w > 0, EADGAN_ERR_INVALID, "upsample2x_bwd: bad arguments");
  upsample2x_bwd_kernel<<<stream_grid((int64_t)nc * h * w, 256), 256, 0, (cudaStream_t)stream>>>(dy, dx, nc, h, w);
  EG_LAUNCH_CHECK("upsample2x_bwd_kernel");
  return 0;
}

extern "C" int eadgan_fill_f32(float* p, int64_t numel, float value, void* stream) {
  EG_REQUIRE(p && numel >= 0, EADGAN_ERR_INVALID, "fill_f32: bad arguments");
  if (numel == 0) return 0;
  fill_kernel<<<stream_grid(numel, 1024), 256, 0, (cudaStream_t)stream>>>(p, numel, value);
  EG_LAUNCH_CHECK("fill_kernel");
  return 0;
}

namespace {
__global__ void f64_to_f32_kernel(const double* __restrict__ src, float* __restrict__ dst, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dst[i] = (float)src[i];
}

// one thread per (image, halo pixel, 8-channel vector): 16-byte zero stores
__global__ void zero_halo_kernel(uint4* __restrict__ xp, int n, int h, int w, int cv) {
  const int per_img = 2 * (w + 2) + 2 * h;
  const int64_t total = (int64_t)n * per_img * cv;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int v = (int)(i % cv);
    const int64_t r = i / cv;
    const int hp = (int)(r % per_img);
    const int64_t b = r / per_img;
    int y, x;
    if (hp < w + 2) { y = 0; x = hp; }
    else if (hp < 2 * (w + 2)) { y = h + 1; x = hp - (w + 2); }
    else { const int q = hp - 2 * (w + 2); y = 1 + (q >> 1); x = (q & 1) ? w + 1 : 0; }
    xp[((b * (h + 2) + y) * (int64_t)(w + 2) + x) * cv + v] = make_uint4(0u, 0u, 0u, 0u);
  }
}
}  // namespace

extern "C" int eadgan_f64_to_f32(const double* src, float* dst, int64_t numel, void* stream) {
  EG_REQUIRE(src && dst && numel > 0, EADGAN_ERR_INVALID, "f64_to_f32: bad arguments");
  f64_to_f32_kernel<<<stream_grid(numel, 256), 256, 0, (cudaStream_t)stream>>>(src, dst, numel);
  EG_LAUNCH_CHECK("f64_to_f32_kernel");
  return 0;
}

extern "C" int eadgan_zero_halo(void* xp, int n, int h, int w, int c, void* stream) {
  EG_REQUIRE(xp && n > 0 && h > 0 && w > 0 && c > 0 && c % 8 == 0, EADGAN_ERR_INVALID,
             "zero_halo: bad arguments (c must be a multiple of 8)");
  const int64_t total = (int64_t)n * (2 * (w + 2) + 2 * h) * (c / 8);
  zero_halo_kernel<<<stream_grid(total, 256), 256, 0, (cudaStream_t)stream>>>((uint4*)xp, n, h, w, c / 8);
  EG_LAUNCH_CHECK("zero_halo_kernel");
  return 0;
}
