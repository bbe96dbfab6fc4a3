// BatchNorm2d (training + eval) as HBM-bound streaming kernels, split into
// reduce / finalize / apply halves so a cross-rank all-reduce of the [2C] fp64
// partial sums can be placed between them (SyncBN, SURVEY.md section 5.9b).
// Reference call sites: nn.BatchNorm2d at celebA/EAD-GAN_celebA.py:79,83,87,
// dSprites/rp.py:130,134,138, MNIST/EAD-GAN_rpqmnxy.py:80,83,87,145 (eps = 0.8 there).
// Semantics follow torch F.batch_norm: biased variance for normalisation, unbiased
// for running_var, momentum 0.1 (SURVEY.md section 7.3-7).
//
// Two memory layouts are handled without per-element integer division:
//   kind 0  dense NCHW   : a "row" is one (n,c) plane of h*w contiguous elements
//   kind 1  NHWC rows    : a "row" is one (n,y) line of w*c contiguous elements
//                          (halo-padded private buffers: sc==1, sw==c, any sh/sn)
// Algorithmic bytes / element: stats 4 (fp32) or 2 (bf16) read; apply read+write;
// bwd_reduce 2 reads; bwd_apply 2 reads + 1 write.  Eval mode (running statistics) has no
// batch-wide dependency: its backward is ONE pass (eval_bwd, 2 reads + 1 write) plus a
// per-channel finalize of dgamma / dbeta / conv-bias gradient.
#include <cstdlib>
#include "common.cuh"

namespace {

struct Geo {
  int kind, n, c, h, w;
  int rows, inner;
};

int classify(const eadgan_tensor4* t, int c, int h, int w) {
  if (t->sw == 1 && t->sh == w) return 0;
  if (t->sc == 1 && t->sw == c) return 1;
  if (h == 1 && w == 1) return 0;  // [N,C,1,1]: any strides, inner run of length 1
  return -1;
}

__device__ __forceinline__ int64_t row_base(const eadgan_tensor4& t, const Geo& g, int row) {
  if (g.kind == 0) {
    const int b = row / g.c, ch = row - b * g.c;
    return (int64_t)b * t.sn + (int64_t)ch * t.sc;
  }
  const int b = row / g.h, y = row - b * g.h;
  return (int64_t)b * t.sn + (int64_t)y * t.sh;
}

constexpr int CHUNK = 2048;  // inner elements per warp job (kind 0)

// ---------------- per-channel reductions -------------------------------------------------
// F(i_global_offsets...) returns the two values to accumulate for one element.
// kind 0: warp job = (row, chunk); lanes stride the contiguous run; one channel per job.
template <class F>
__device__ void reduce_kind0(const Geo g, double* sums, F f) {
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  const int chunks = (g.inner + CHUNK - 1) / CHUNK;
  const int64_t jobs = (int64_t)g.rows * chunks;
  for (int64_t job = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5); job < jobs;
       job += (int64_t)gridDim.x * warps_per_block) {
    const int row = (int)(job / chunks);
    const int ck = (int)(job - (int64_t)row * chunks);
    const int ch = row % g.c;
    const int i_end = min(g.inner, (ck + 1) * CHUNK);
    double s0 = 0.0, s1 = 0.0;
    float a0 = 0.f, a1 = 0.f;
    int cnt = 0;
    for (int i = ck * CHUNK + lane; i < i_end; i += 32) {
      float v0, v1;
      f(row, i, ch, v0, v1);
      a0 += v0;
      a1 += v1;
      if (++cnt == 16) { s0 += a0; s1 += a1; a0 = a1 = 0.f; cnt = 0; }
    }
    s0 += a0;
    s1 += a1;
    s0 = eg_warp_sum_d(s0);
    s1 = eg_warp_sum_d(s1);
    if (lane == 0) {
      atomicAdd(&sums[ch], s0);
      atomicAdd(&sums[g.c + ch], s1);
    }
  }
}

// kind 1: thread <-> channel (channels contiguous); blockDim.x = 256 covers `cb` channels
// times 256/cb pixel lanes; a block walks pixels in grid-stride; smem reduce; atomics.
template <class F>
__device__ void reduce_kind1(const Geo g, double* sums, F f) {
  __shared__ double sh0[256], sh1[256];
  const int cb = g.c < 256 ? g.c : 256;      // channels per pass; the last pass of c > 256 may be partial
  const int lanes = 256 / cb;                // pixel lanes per block (>=1)
  const int tch = threadIdx.x % cb, tl = threadIdx.x / cb;
  const int64_t pixels = (int64_t)g.rows * g.w;
  for (int c0 = 0; c0 < g.c; c0 += cb) {
    const int ch = c0 + tch;
    double s0 = 0.0, s1 = 0.0;
    if (tl < lanes && ch < g.c) {
      float a0 = 0.f, a1 = 0.f;
      int cnt = 0;
      for (int64_t p = (int64_t)blockIdx.x * lanes + tl; p < pixels; p += (int64_t)gridDim.x * lanes) {
        const int row = (int)(p / g.w);
        const int x = (int)(p - (int64_t)row * g.w);
        float v0, v1;
        f(row, x * g.c + ch, ch, v0, v1);
        a0 += v0;
        a1 += v1;
        if (++cnt == 16) { s0 += a0; s1 += a1; a0 = a1 = 0.f; cnt = 0; }
      }
      s0 += a0;
      s1 += a1;
    }
    sh0[threadIdx.x] = s0;
    sh1[threadIdx.x] = s1;
    __syncthreads();
    if (threadIdx.x < cb && ch < g.c) {
      double r0 = 0.0, r1 = 0.0;
      for (int l = 0; l < lanes; ++l) { r0 += sh0[l * cb + threadIdx.x]; r1 += sh1[l * cb + threadIdx.x]; }
      atomicAdd(&sums[ch], r0);
      atomicAdd(&sums[g.c + ch], r1);
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256) bn_stats_kernel(eadgan_tensor4 x, Geo g, double* sums) {
  auto f = [&](int row, int i, int ch, float& v0, float& v1) {
    const float v = eg_ld(x.ptr, row_base(x, g, row) + i, x.dtype);
    v0 = v;
    v1 = v * v;
  };
  if (g.kind == 0) reduce_kind0(g, sums, f); else reduce_kind1(g, sums, f);
}

struct BwdArgs {
  eadgan_tensor4 dy, x, y, dx;
  const float *mean, *invstd, *gamma, *beta;
  const double* sums;
  double count;
  int act;
  float slope;
};

// dz = dy * act'(y);  xhat = (x - mean) * invstd
__global__ void __launch_bounds__(256) bn_bwd_reduce_kernel(BwdArgs a, Geo g, double* sums) {
  auto f = [&](int row, int i, int ch, float& v0, float& v1) {
    float dz = eg_ld(a.dy.ptr, row_base(a.dy, g, row) + i, a.dy.dtype);
    if (a.act != EADGAN_ACT_NONE) {
      const float yv = eg_ld(a.y.ptr, row_base(a.y, g, row) + i, a.y.dtype);
      dz *= eg_act_grad(yv, a.act, a.slope);
    }
    const float xv = eg_ld(a.x.ptr, row_base(a.x, g, row) + i, a.x.dtype);
    v0 = dz;
    v1 = dz * (xv - a.mean[ch]) * a.invstd[ch];
  };
  if (g.kind == 0) reduce_kind0(g, sums, f); else reduce_kind1(g, sums, f);
}

// eval-mode backward, one pass: nothing depends on the batch's statistics, so the per-element gradient is written
// while the per-channel sums are accumulated.  dz = dy * act'(y), dx = dz * gamma * rsqrt(rv + eps),
// sums = [S dz | S dz * xhat] with xhat = (x - rm) * rsqrt(rv + eps).  Every element is read and written by the same
// thread, so dx may alias dy.  (a.mean = running_mean, a.invstd = running_var here.)
__global__ void __launch_bounds__(256) bn_eval_bwd_kernel(BwdArgs a, Geo g, float eps, double* sums) {
  auto f = [&](int row, int i, int ch, float& v0, float& v1) {
    float dz = eg_ld(a.dy.ptr, row_base(a.dy, g, row) + i, a.dy.dtype);
    if (a.act != EADGAN_ACT_NONE) {
      const float yv = eg_ld(a.y.ptr, row_base(a.y, g, row) + i, a.y.dtype);
      dz *= eg_act_grad(yv, a.act, a.slope);
    }
    const float is = rsqrtf(a.invstd[ch] + eps);
    const float ga = a.gamma ? a.gamma[ch] : 1.f;
    const float xv = eg_ld(a.x.ptr, row_base(a.x, g, row) + i, a.x.dtype);
    eg_st(a.dx.ptr, row_base(a.dx, g, row) + i, a.dx.dtype, dz * ga * is);
    v0 = dz;
    v1 = dz * (xv - a.mean[ch]) * is;
  };
  if (g.kind == 0) reduce_kind0(g, sums, f); else reduce_kind1(g, sums, f);
}

// ---------------- elementwise passes -----------------------------------------------------
template <class F>
__device__ void foreach_elem(const Geo g, F f) {
  // block job = (row, 1024-element chunk); threads stride the contiguous run
  const int chunks = (g.inner + 1023) / 1024;
  const int64_t jobs = (int64_t)g.rows * chunks;
  for (int64_t job = blockIdx.x; job < jobs; job += gridDim.x) {
    const int row = (int)(job / chunks);
    const int ck = (int)(job - (int64_t)row * chunks);
    const int i_end = min(g.inner, (ck + 1) * 1024);
    const int ch_row = row % g.c;
    for (int i = ck * 1024 + threadIdx.x; i < i_end; i += blockDim.x)
      f(row, i, g.kind == 0 ? ch_row : i % g.c);
  }
}

struct ApplyArgs {
  eadgan_tensor4 x, y;
  const float *mean, *invstd, *gamma, *beta;
  int act;
  float slope;
  float eps;
  int eval;  // mean=running_mean, invstd=running_var (converted on the fly)
};

__global__ void __launch_bounds__(256) bn_apply_kernel(ApplyArgs a, Geo g) {
  foreach_elem(g, [&](int row, int i, int ch) {
    const float xv = eg_ld(a.x.ptr, row_base(a.x, g, row) + i, a.x.dtype);
    const float is = a.eval ? rsqrtf(a.invstd[ch] + a.eps) : a.invstd[ch];
    const float ga = a.gamma ? a.gamma[ch] : 1.f, be = a.beta ? a.beta[ch] : 0.f;
    float v = (xv - a.mean[ch]) * is * ga + be;
    v = eg_act(v, a.act, a.slope);
    eg_st(a.y.ptr, row_base(a.y, g, row) + i, a.y.dtype, v);
  });
}

__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(BwdArgs a, Geo g) {
  const double inv_count = 1.0 / a.count;
  foreach_elem(g, [&](int row, int i, int ch) {
    float dz = eg_ld(a.dy.ptr, row_base(a.dy, g, row) + i, a.dy.dtype);
    if (a.act != EADGAN_ACT_NONE) {
      const float yv = eg_ld(a.y.ptr, row_base(a.y, g, row) + i, a.y.dtype);
      dz *= eg_act_grad(yv, a.act, a.slope);
    }
    const float xv = eg_ld(a.x.ptr, row_base(a.x, g, row) + i, a.x.dtype);
    const float is = a.invstd[ch];
    const float xhat = (xv - a.mean[ch]) * is;
    const float m_dz = (float)(a.sums[ch] * inv_count);
    const float m_dzx = (float)(a.sums[g.c + ch] * inv_count);
    const float ga = a.gamma ? a.gamma[ch] : 1.f;
    const float v = ga * is * (dz - m_dz - xhat * m_dzx);
    eg_st(a.dx.ptr, row_base(a.dx, g, row) + i, a.dx.dtype, v);
  });
}


// ---------------- NHWC bf16 fast paths (the private halo-padded buffers of the chain executor) --------
// A row (n, y) of the interior is one contiguous run of w*c bf16 = w*c/8 16-byte vectors.  256 threads per
// block, grid-stride over rows; vector v of a row holds channels 8*(v % (c/8)).., and because c/8 divides
// 256 every thread keeps ONE channel group for the whole kernel, so the per-channel parameters live in
// registers.  Bytes per element: apply 2R+2W, bwd_reduce 4R (dy, x; the ReLU/LeakyReLU gate is recomputed
// from x with the forward's own expression instead of reading y), bwd_apply 4R+2W.
struct Nhwc8 {
  int n, c, h, w;
  int cv;         // c / 8
  int row_vecs;   // w * c / 8
};

__device__ __forceinline__ void bf8_to_f32(const uint4 u, float* f) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    f[2 * e] = __uint_as_float(w[e] << 16);
    f[2 * e + 1] = __uint_as_float(w[e] & 0xffff0000u);
  }
}
__device__ __forceinline__ uint4 f32_to_bf8(const float* f) {
  uint32_t w[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    __nv_bfloat162 h2 = __floats2bfloat162_rn(f[2 * e], f[2 * e + 1]);
    w[e] = *reinterpret_cast<uint32_t*>(&h2);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ const uint4* row_ptr(const eadgan_tensor4& t, int b, int y) {
  return reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(t.ptr) + (int64_t)b * t.sn + (int64_t)y * t.sh);
}

constexpr int NHWC8_U = 4;   // rows processed together by a block (independent loads in flight per thread)
struct ChanParams { float mean[8], is[8], ga[8], be[8], sc[8], sh[8], nm[8]; };   // sc = is*ga, sh = be - mean*sc, nm = -mean*is
__device__ __forceinline__ void load_params(ChanParams& p, int ch0, const float* mean, const float* invstd,
                                            const float* gamma, const float* beta) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    p.mean[j] = mean[ch0 + j];
    p.is[j] = invstd[ch0 + j];
    p.ga[j] = gamma ? gamma[ch0 + j] : 1.f;
    p.be[j] = beta ? beta[ch0 + j] : 0.f;
  }
}
// one FMA per element instead of sub/mul/mul/add: y = x*sc + sh, xhat = x*is + nm (bf16 buffers: the fp32
// re-association is far below the output rounding; apply and the recomputed gate use the SAME expression)
__device__ __forceinline__ void derive_params(ChanParams& p) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    p.sc[j] = p.is[j] * p.ga[j];
    p.sh[j] = p.be[j] - p.mean[j] * p.sc[j];
    p.nm[j] = -p.mean[j] * p.is[j];
  }
}

__global__ void __launch_bounds__(256) bn_apply_nhwc8_kernel(ApplyArgs a, Nhwc8 g) {
  ChanParams p;
  const int ch0 = (threadIdx.x % g.cv) * 8;
  load_params(p, ch0, a.mean, a.invstd, a.gamma, a.beta);
  if (a.eval) {
#pragma unroll
    for (int j = 0; j < 8; ++j) p.is[j] = rsqrtf(p.is[j] + a.eps);
  }
  derive_params(p);
  const bool leaky = a.act == EADGAN_ACT_RELU || a.act == EADGAN_ACT_LRELU;
  const float neg = a.act == EADGAN_ACT_RELU ? 0.f : a.slope;
  // NHWC8_U rows per block iteration: every thread keeps NHWC8_U independent 16-byte loads in flight (one load
  // per thread left the kernel latency-bound at ~3 TB/s: 2048 threads x 16 B per SM per memory round trip)
  const int rows = g.n * g.h;
  for (int row0 = blockIdx.x * NHWC8_U; row0 < rows; row0 += gridDim.x * NHWC8_U) {
    const uint4* xr[NHWC8_U];
    uint4* yr[NHWC8_U];
#pragma unroll
    for (int u = 0; u < NHWC8_U; ++u) {
      const int row = min(row0 + u, rows - 1);
      const int b = row / g.h, y = row - b * g.h;
      xr[u] = row_ptr(a.x, b, y);
      yr[u] = const_cast<uint4*>(row_ptr(a.y, b, y));
    }
    for (int v = threadIdx.x; v < g.row_vecs; v += 256) {
      uint4 raw[NHWC8_U];
#pragma unroll
      for (int u = 0; u < NHWC8_U; ++u) raw[u] = __ldg(xr[u] + v);
#pragma unroll
      for (int u = 0; u < NHWC8_U; ++u) {
        if (row0 + u < rows) {
          float f[8];
          bf8_to_f32(raw[u], f);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float t = fmaf(f[j], p.sc[j], p.sh[j]);
            f[j] = leaky ? (t > 0.f ? t : t * neg) : eg_act(t, a.act, a.slope);
          }
          yr[u][v] = f32_to_bf8(f);
        }
      }
    }
  }
}

// gate of a ReLU / LeakyReLU that follows the affine transform, recomputed from x exactly as apply did
__device__ __forceinline__ float bn_gate(float x, const ChanParams& p, int j, float slope_neg) {
  return fmaf(x, p.sc[j], p.sh[j]) > 0.f ? 1.f : slope_neg;
}

template <bool GATE_FROM_X>
__global__ void __launch_bounds__(256) bn_bwd_reduce_nhwc8_kernel(BwdArgs a, Nhwc8 g, double* sums) {
  __shared__ double sh[2 * 1024];
  for (int i = threadIdx.x; i < 2 * g.c; i += 256) sh[i] = 0.0;
  __syncthreads();
  ChanParams p;
  const int ch0 = (threadIdx.x % g.cv) * 8;
  load_params(p, ch0, a.mean, a.invstd, a.gamma, a.beta);
  derive_params(p);
  const float slope_neg = a.act == EADGAN_ACT_RELU ? 0.f : a.slope;
  float s0[8], s1[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s0[j] = s1[j] = 0.f;
  const int rows = g.n * g.h;
  for (int row0 = blockIdx.x * NHWC8_U; row0 < rows; row0 += gridDim.x * NHWC8_U) {
    const uint4 *dyr[NHWC8_U], *xr[NHWC8_U], *yr[NHWC8_U];
#pragma unroll
    for (int u = 0; u < NHWC8_U; ++u) {
      const int row = min(row0 + u, rows - 1);
      const int b = row / g.h, y = row - b * g.h;
      dyr[u] = row_ptr(a.dy, b, y);
      xr[u] = row_ptr(a.x, b, y);
      yr[u] = GATE_FROM_X ? nullptr : row_ptr(a.y, b, y);
    }
    for (int v = threadIdx.x; v < g.row_vecs; v += 256) {
      uint4 rdz[NHWC8_U], rx[NHWC8_U], ry[NHWC8_U];
#pragma unroll
      for (int u = 0; u < NHWC8_U; ++u) {
        rdz[u] = __ldg(dyr[u] + v);
        rx[u] = __ldg(xr[u] + v);
        if (!GATE_FROM_X) ry[u] = __ldg(yr[u] + v);
      }
#pragma unroll
      for (int u = 0; u < NHWC8_U; ++u) {
        if (row0 + u < rows) {
          float dz[8], xv[8];
          bf8_to_f32(rdz[u], dz);
          bf8_to_f32(rx[u], xv);
          if (GATE_FROM_X) {
            if (a.act != EADGAN_ACT_NONE) {
#pragma unroll
              for (int j = 0; j < 8; ++j) dz[j] *= bn_gate(xv[j], p, j, slope_neg);
            }
          } else {
            float yv[8];
            bf8_to_f32(ry[u], yv);
#pragma unroll
            for (int j = 0; j < 8; ++j) dz[j] *= eg_act_grad(yv[j], a.act, a.slope);
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            s0[j] += dz[j];
            s1[j] = fmaf(dz[j], fmaf(xv[j], p.is[j], p.nm[j]), s1[j]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    atomicAdd(&sh[ch0 + j], (double)s0[j]);
    atomicAdd(&sh[g.c + ch0 + j], (double)s1[j]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * g.c; i += 256) atomicAdd(&sums[i], sh[i]);
}

// forward statistics (sum x, sum x^2) of a bf16 NHWC buffer whose producer could not fuse them (dense 1x1 -> 4x4
// layers): same access pattern as the kernels above instead of one 2-byte load per thread and iteration
__global__ void __launch_bounds__(256) bn_stats_nhwc8_kernel(eadgan_tensor4 x, Nhwc8 g, double* sums) {
  __shared__ double sh[2 * 1024];
  for (int i = threadIdx.x; i < 2 * g.c; i += 256) sh[i] = 0.0;
  __syncthreads();
  const int ch0 = (threadIdx.x % g.cv) * 8;
  float s0[8], s1[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s0[j] = s1[j] = 0.f;
  const int rows = g.n * g.h;
  for (int row0 = blockIdx.x * NHWC8_U; row0 < rows; row0 += gridDim.x * NHWC8_U) {
    const uint4* xr[NHWC8_U];
#pragma unroll
    for (int u = 0; u < NHWC8_U; ++u) {
      const int row = min(row0 + u, rows - 1);
      const int b = row / g.h, y = row - b * g.h;
      xr[u] = row_ptr(x, b, y);
    }
    for (int v = threadIdx.x; v < g.row_vecs; v += 256) {
      uint4 raw[NHWC8_U];
#pragma unroll
      for (int u = 0; u < NHWC8_U; ++u) raw[u] = __ldg(xr[u] + v);
#pragma unroll
      for (int u = 0; u < NHWC8_U; ++u) {
        if (row0 + u < rows) {
          float f[8];
          bf8_to_f32(raw[u], f);
#pragma unroll
          for (int j = 0; j < 8; ++j) { s0[j] += f[j]; s1[j] = fmaf(f[j], f[j], s1[j]); }
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    atomicAdd(&sh[ch0 + j], (double)s0[j]);
    atomicAdd(&sh[g.c + ch0 + j], (double)s1[j]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * g.c; i += 256) atomicAdd(&sums[i], sh[i]);
}

template <bool GATE_FROM_X>
__global__ void __launch_bounds__(256) bn_bwd_apply_nhwc8_kernel(BwdArgs a, Nhwc8 g) {
  ChanParams p;
  const int ch0 = (threadIdx.x % g.cv) * 8;
  load_params(p, ch0, a.mean, a.invstd, a.gamma, a.beta);
  const float slope_neg = a.act == EADGAN_ACT_RELU ? 0.f : a.slope;
  const double inv_count = 1.0 / a.count;
  derive_params(p);
  float c2[8], c3[8];   // dx = sc*dz - sc*mean(dz) - xhat*sc*mean(dz*xhat)
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    c2[j] = p.sc[j] * (float)(a.sums[ch0 + j] * inv_count);
    c3[j] = p.sc[j] * (float)(a.sums[g.c + ch0 + j] * inv_count);
  }
  const int rows = g.n * g.h;
  for (int row0 = blockIdx.x * NHWC8_U; row0 < rows; row0 += gridDim.x * NHWC8_U) {
    const uint4 *dyr[NHWC8_U], *xr[NHWC8_U], *yr[NHWC8_U];
    uint4* dxr[NHWC8_U];
#pragma unroll
    for (int u = 0; u < NHWC8_U; ++u) {
      const int row = min(row0 + u, rows - 1);
      const int b = row / g.h, y = row - b * g.h;
      dyr[u] = row_ptr(a.dy, b, y);
      xr[u] = row_ptr(a.x, b, y);
      yr[u] = GATE_FROM_X ? nullptr : row_ptr(a.y, b, y);
      dxr[u] = const_cast<uint4*>(row_ptr(a.dx, b, y));
    }
    for (int v = threadIdx.x; v < g.row_vecs; v += 256) {
      uint4 rdz[NHWC8_U], rx[NHWC8_U], ry[NHWC8_U];
#pragma unroll
      for (int u = 0; u < NHWC8_U; ++u) {
        rdz[u] = __ldg(dyr[u] + v);
        rx[u] = __ldg(xr[u] + v);
        if (!GATE_FROM_X) ry[u] = __ldg(yr[u] + v);
      }
#pragma unroll
      for (int u = 0; u < NHWC8_U; ++u) {
        if (row0 + u < rows) {
          float dz[8], xv[8];
          bf8_to_f32(rdz[u], dz);
          bf8_to_f32(rx[u], xv);
          if (GATE_FROM_X) {
            if (a.act != EADGAN_ACT_NONE) {
#pragma unroll
              for (int j = 0; j < 8; ++j) dz[j] *= bn_gate(xv[j], p, j, slope_neg);
            }
          } else {
            float yv[8];
            bf8_to_f32(ry[u], yv);
#pragma unroll
            for (int j = 0; j < 8; ++j) dz[j] *= eg_act_grad(yv[j], a.act, a.slope);
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float xhat = fmaf(xv[j], p.is[j], p.nm[j]);
            dz[j] = fmaf(-xhat, c3[j], fmaf(dz[j], p.sc[j], -c2[j]));
          }
          dxr[u][v] = f32_to_bf8(dz);
        }
      }
    }
  }
}

// eval-mode backward on the padded bf16 buffers: bn_bwd_reduce_nhwc8 and the dx store in one pass (dx = dz * sc).
// The parameters are the running statistics, converted exactly as bn_apply_nhwc8_kernel converts them, so the
// recomputed ReLU / LeakyReLU gate equals the stored output's gate bit for bit.  dx may alias dy: every 16-byte
// vector is loaded before the same thread stores it.  Bytes per element: 4R+2W (6R+2W with the gate read from y).
template <bool GATE_FROM_X>
__global__ void __launch_bounds__(256) bn_eval_bwd_nhwc8_kernel(BwdArgs a, Nhwc8 g, float eps, double* sums) {
  __shared__ double sh[2 * 1024];
  for (int i = threadIdx.x; i < 2 * g.c; i += 256) sh[i] = 0.0;
  __syncthreads();
  ChanParams p;
  const int ch0 = (threadIdx.x % g.cv) * 8;
  load_params(p, ch0, a.mean, a.invstd, a.gamma, a.beta);
#pragma unroll
  for (int j = 0; j < 8; ++j) p.is[j] = rsqrtf(p.is[j] + eps);
  derive_params(p);
  const float slope_neg = a.act == EADGAN_ACT_RELU ? 0.f : a.slope;
  float s0[8], s1[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s0[j] = s1[j] = 0.f;
  const int rows = g.n * g.h;
  for (int row0 = blockIdx.x * NHWC8_U; row0 < rows; row0 += gridDim.x * NHWC8_U) {
    const uint4 *dyr[NHWC8_U], *xr[NHWC8_U], *yr[NHWC8_U];
    uint4* dxr[NHWC8_U];
#pragma unroll
    for (int u = 0; u < NHWC8_U; ++u) {
      const int row = min(row0 + u, rows - 1);
      const int b = row / g.h, y = row - b * g.h;
      dyr[u] = row_ptr(a.dy, b, y);
      xr[u] = row_ptr(a.x, b, y);
      yr[u] = GATE_FROM_X ? nullptr : row_ptr(a.y, b, y);
      dxr[u] = const_cast<uint4*>(row_ptr(a.dx, b, y));
    }
    for (int v = threadIdx.x; v < g.row_vecs; v += 256) {
      uint4 rdz[NHWC8_U], rx[NHWC8_U], ry[NHWC8_U];
#pragma unroll
      for (int u = 0; u < NHWC8_U; ++u) {
        rdz[u] = dyr[u][v];     // plain loads: dy may be the buffer this kernel writes
        rx[u] = __ldg(xr[u] + v);
        if (!GATE_FROM_X) ry[u] = __ldg(yr[u] + v);
      }
#pragma unroll
      for (int u = 0; u < NHWC8_U; ++u) {
        if (row0 + u < rows) {
          float dz[8], xv[8];
          bf8_to_f32(rdz[u], dz);
          bf8_to_f32(rx[u], xv);
          if (GATE_FROM_X) {
            if (a.act != EADGAN_ACT_NONE) {
#pragma unroll
              for (int j = 0; j < 8; ++j) dz[j] *= bn_gate(xv[j], p, j, slope_neg);
            }
          } else {
            float yv[8];
            bf8_to_f32(ry[u], yv);
#pragma unroll
            for (int j = 0; j < 8; ++j) dz[j] *= eg_act_grad(yv[j], a.act, a.slope);
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            s0[j] += dz[j];
            s1[j] = fmaf(dz[j], fmaf(xv[j], p.is[j], p.nm[j]), s1[j]);
            dz[j] *= p.sc[j];
          }
          dxr[u][v] = f32_to_bf8(dz);
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    atomicAdd(&sh[ch0 + j], (double)s0[j]);
    atomicAdd(&sh[g.c + ch0 + j], (double)s1[j]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * g.c; i += 256) atomicAdd(&sums[i], sh[i]);
}

// all tensors channel-fastest bf16 rows with 16-byte aligned runs, and c/8 divides 256
bool nhwc8_ok(const Geo& g, const eadgan_tensor4* const* ts, int nt) {
  if (g.kind != 1 || g.c % 8 != 0 || g.c > 1024 || 256 % (g.c / 8) != 0) return false;
  for (int i = 0; i < nt; ++i) {
    if (!ts[i]) continue;
    if (ts[i]->dtype != EADGAN_BF16 || (ts[i]->sn % 8) != 0 || (ts[i]->sh % 8) != 0) return false;
    if ((reinterpret_cast<uintptr_t>(ts[i]->ptr) & 15) != 0) return false;
  }
  return true;
}
Nhwc8 make_nhwc8(const Geo& g) { return Nhwc8{g.n, g.c, g.h, g.w, g.c / 8, g.w * g.c / 8}; }
int nhwc8_grid(const Geo& g) {
  const int groups = (g.n * g.h + NHWC8_U - 1) / NHWC8_U, cap = 2 * eg_sm_count();   // 2 blocks per SM (profiles/r02ab_*)
  return groups < cap ? groups : cap;
}

__global__ void bn_finalize_kernel(const double* sums, double count, int c, float eps, float momentum,
                                   float* mean, float* invstd, float* rmean, float* rvar) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  const double m = sums[ch] / count;
  double var = sums[c + ch] / count - m * m;
  if (var < 0.0) var = 0.0;
  mean[ch] = (float)m;
  invstd[ch] = (float)(1.0 / sqrt(var + (double)eps));
  if (rmean) rmean[ch] = (1.f - momentum) * rmean[ch] + momentum * (float)m;
  if (rvar) {
    const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
    rvar[ch] = (1.f - momentum) * rvar[ch] + momentum * (float)unbiased;
  }
}


// dgamma / dbeta (local sums) and the gradient of a conv bias feeding this BatchNorm, all from the
// fp64 partial sums -- no extra pass over the activation.  sum(dx) over the local elements is
//   gamma*invstd*(S_dz_loc - n_loc*S_dz/count - S_xhat_loc*S_dzxhat/count),  S_xhat_loc = (S_x_loc - n_loc*mean)*invstd
// (mathematically zero on one rank: torch's own value there is fp32 summation noise).
__global__ void bn_bwd_finalize_kernel(const double* loc, const double* glob, const double* fwd_loc, double n_loc,
                                       double count, const float* mean, const float* invstd, const float* gamma,
                                       int c, float* dgamma, float* dbeta, float* dbias) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  if (dbeta) dbeta[ch] = (float)loc[ch];
  if (dgamma) dgamma[ch] = (float)loc[c + ch];
  if (dbias) {
    const double is = (double)invstd[ch];
    const double sxhat = fwd_loc ? (fwd_loc[ch] - n_loc * (double)mean[ch]) * is : 0.0;
    const double ga = gamma ? (double)gamma[ch] : 1.0;
    dbias[ch] = (float)(ga * is * (loc[ch] - n_loc * glob[ch] / count - sxhat * glob[c + ch] / count));
  }
}

// eval mode: dbeta = S dz, dgamma = S dz*xhat, and the gradient of a conv bias feeding the BatchNorm, sum of dx =
// gamma * rsqrt(rv + eps) * S dz (not zero in eval mode: the normalisation does not depend on the batch)
__global__ void bn_eval_bwd_finalize_kernel(const double* sums, const float* rvar, float eps, const float* gamma,
                                            int c, float* dgamma, float* dbeta, float* dbias) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  if (dbeta) dbeta[ch] = (float)sums[ch];
  if (dgamma) dgamma[ch] = (float)sums[c + ch];
  if (dbias) {
    const double ga = gamma ? (double)gamma[ch] : 1.0;
    dbias[ch] = (float)(ga * (double)rsqrtf(rvar[ch] + eps) * sums[ch]);
  }
}

int make_geo(Geo* g, int n, int c, int h, int w, const eadgan_tensor4* const* ts, int nt,
             const char* who) {
  EG_REQUIRE(n > 0 && c > 0 && h > 0 && w > 0, EADGAN_ERR_INVALID, "%s: bad extents", who);
  int kind = -2;
  for (int i = 0; i < nt; ++i) {
    if (!ts[i]) continue;
    EG_REQUIRE(ts[i]->ptr != nullptr, EADGAN_ERR_INVALID, "%s: NULL tensor", who);
    const int k = classify(ts[i], c, h, w);
    EG_REQUIRE(k >= 0, EADGAN_ERR_UNSUPPORTED,
               "%s: tensor is neither dense NCHW nor channel-fastest NHWC rows", who);
    EG_REQUIRE(kind == -2 || kind == k, EADGAN_ERR_UNSUPPORTED, "%s: mixed layouts", who);
    kind = k;
  }
  g->kind = kind; g->n = n; g->c = c; g->h = h; g->w = w;
  // kind 1 takes any channel count: reduce_kind1 masks the channels past c of a partial last 256-channel pass, and
  // foreach_elem derives the channel of every element as i % c
  if (kind == 0) { g->rows = n * c; g->inner = h * w; }
  else { g->rows = n * h; g->inner = w * c; }
  return 0;
}

int reduce_grid(const Geo& g) {
  int64_t jobs;
  if (g.kind == 0) jobs = ((int64_t)g.rows * ((g.inner + CHUNK - 1) / CHUNK) + 7) / 8;
  else jobs = ((int64_t)g.rows * g.w + 63) / 64;
  const int cap = 16 * eg_sm_count();
  return (int)(jobs < 1 ? 1 : (jobs > cap ? cap : jobs));
}
int elem_grid(const Geo& g) {
  const int64_t jobs = (int64_t)g.rows * ((g.inner + 1023) / 1024);
  const int cap = 32 * eg_sm_count();
  return (int)(jobs > cap ? cap : jobs);
}

}  // namespace

extern "C" int eadgan_bn_stats(const eadgan_tensor4* x, int n, int c, int h, int w, double* sums,
                               void* stream) {
  Geo g;
  const eadgan_tensor4* ts[] = {x};
  EG_REQUIRE(x && sums, EADGAN_ERR_INVALID, "bn_stats: NULL argument");
  if (int e = make_geo(&g, n, c, h, w, ts, 1, "bn_stats")) return e;
  if (nhwc8_ok(g, ts, 1)) {
    const int groups = (g.n * g.h + NHWC8_U - 1) / NHWC8_U, cap = 4 * eg_sm_count();   // one wave, four blocks per SM
    bn_stats_nhwc8_kernel<<<groups < cap ? groups : cap, 256, 0, (cudaStream_t)stream>>>(*x, make_nhwc8(g), sums);
    EG_LAUNCH_CHECK("bn_stats_nhwc8_kernel");
    return 0;
  }
  bn_stats_kernel<<<reduce_grid(g), 256, 0, (cudaStream_t)stream>>>(*x, g, sums);
  EG_LAUNCH_CHECK("bn_stats_kernel");
  return 0;
}

extern "C" int eadgan_bn_finalize(const double* sums, double count, int c, float eps, float momentum,
                                  float* mean, float* invstd, float* running_mean,
                                  float* running_var, void* stream) {
  EG_REQUIRE(sums && mean && invstd && c > 0 && count > 0, EADGAN_ERR_INVALID, "bn_finalize: bad arguments");
  bn_finalize_kernel<<<(c + 127) / 128, 128, 0, (cudaStream_t)stream>>>(sums, count, c, eps, momentum, mean,
                                                                       invstd, running_mean, running_var);
  EG_LAUNCH_CHECK("bn_finalize_kernel");
  return 0;
}

extern "C" int eadgan_bn_apply(const eadgan_tensor4* x, int n, int c, int h, int w, const float* mean,
                               const float* invstd, const float* gamma, const float* beta, int act,
                               float slope, const eadgan_tensor4* y, void* stream) {
  Geo g;
  const eadgan_tensor4* ts[] = {x, y};
  EG_REQUIRE(x && y && mean && invstd, EADGAN_ERR_INVALID, "bn_apply: NULL argument");
  if (int e = make_geo(&g, n, c, h, w, ts, 2, "bn_apply")) return e;
  ApplyArgs a{*x, *y, mean, invstd, gamma, beta, act, slope, 0.f, 0};
  if (nhwc8_ok(g, ts, 2)) {
    bn_apply_nhwc8_kernel<<<nhwc8_grid(g), 256, 0, (cudaStream_t)stream>>>(a, make_nhwc8(g));
    EG_LAUNCH_CHECK("bn_apply_nhwc8_kernel");
    return 0;
  }
  bn_apply_kernel<<<elem_grid(g), 256, 0, (cudaStream_t)stream>>>(a, g);
  EG_LAUNCH_CHECK("bn_apply_kernel");
  return 0;
}

extern "C" int eadgan_bn_eval(const eadgan_tensor4* x, int n, int c, int h, int w,
                              const float* running_mean, const float* running_var, float eps,
                              const float* gamma, const float* beta, int act, float slope,
                              const eadgan_tensor4* y, void* stream) {
  Geo g;
  const eadgan_tensor4* ts[] = {x, y};
  EG_REQUIRE(x && y && running_mean && running_var, EADGAN_ERR_INVALID, "bn_eval: NULL argument");
  if (int e = make_geo(&g, n, c, h, w, ts, 2, "bn_eval")) return e;
  ApplyArgs a{*x, *y, running_mean, running_var, gamma, beta, act, slope, eps, 1};
  if (nhwc8_ok(g, ts, 2)) {
    bn_apply_nhwc8_kernel<<<nhwc8_grid(g), 256, 0, (cudaStream_t)stream>>>(a, make_nhwc8(g));
    EG_LAUNCH_CHECK("bn_apply_nhwc8_kernel(eval)");
    return 0;
  }
  bn_apply_kernel<<<elem_grid(g), 256, 0, (cudaStream_t)stream>>>(a, g);
  EG_LAUNCH_CHECK("bn_apply_kernel(eval)");
  return 0;
}

extern "C" int eadgan_bn_eval_bwd(const eadgan_tensor4* dy, const eadgan_tensor4* x, const eadgan_tensor4* y,
                                  int n, int c, int h, int w, const float* running_mean, const float* running_var,
                                  float eps, const float* gamma, const float* beta, int act, float slope,
                                  double* sums, const eadgan_tensor4* dx, float* dgamma, float* dbeta, float* dbias,
                                  void* stream) {
  Geo g;
  EG_REQUIRE(dy && x && dx && running_mean && running_var && sums, EADGAN_ERR_INVALID,
             "bn_eval_bwd: NULL argument");
  EG_REQUIRE(act == EADGAN_ACT_NONE || y, EADGAN_ERR_INVALID, "bn_eval_bwd: fused activation needs y");
  const eadgan_tensor4* ts[] = {dy, x, dx, act != EADGAN_ACT_NONE ? y : nullptr};
  if (int e = make_geo(&g, n, c, h, w, ts, 4, "bn_eval_bwd")) return e;
  BwdArgs a{};
  a.dy = *dy; a.x = *x; if (y) a.y = *y; a.dx = *dx;
  a.mean = running_mean; a.invstd = running_var; a.gamma = gamma; a.beta = beta; a.act = act; a.slope = slope;
  cudaStream_t s = (cudaStream_t)stream;
  const bool gate_x = act == EADGAN_ACT_NONE || act == EADGAN_ACT_RELU || act == EADGAN_ACT_LRELU;
  const eadgan_tensor4* fs[] = {dy, x, dx, gate_x ? nullptr : y};
  if (nhwc8_ok(g, fs, 4)) {
    if (gate_x) bn_eval_bwd_nhwc8_kernel<true><<<nhwc8_grid(g), 256, 0, s>>>(a, make_nhwc8(g), eps, sums);
    else bn_eval_bwd_nhwc8_kernel<false><<<nhwc8_grid(g), 256, 0, s>>>(a, make_nhwc8(g), eps, sums);
    EG_LAUNCH_CHECK("bn_eval_bwd_nhwc8_kernel");
  } else {
    bn_eval_bwd_kernel<<<reduce_grid(g), 256, 0, s>>>(a, g, eps, sums);
    EG_LAUNCH_CHECK("bn_eval_bwd_kernel");
  }
  if (dgamma || dbeta || dbias) {
    bn_eval_bwd_finalize_kernel<<<(c + 127) / 128, 128, 0, s>>>(sums, running_var, eps, gamma, c, dgamma, dbeta,
                                                                dbias);
    EG_LAUNCH_CHECK("bn_eval_bwd_finalize_kernel");
  }
  return 0;
}

extern "C" int eadgan_bn_bwd_reduce(const eadgan_tensor4* dy, const eadgan_tensor4* x,
                                    const eadgan_tensor4* y, int n, int c, int h, int w,
                                    const float* mean, const float* invstd, const float* gamma,
                                    const float* beta, int act, float slope, double* sums,
                                    void* stream) {
  Geo g;
  EG_REQUIRE(dy && x && mean && invstd && sums, EADGAN_ERR_INVALID, "bn_bwd_reduce: NULL argument");
  EG_REQUIRE(act == EADGAN_ACT_NONE || y, EADGAN_ERR_INVALID, "bn_bwd_reduce: fused activation needs y");
  const eadgan_tensor4* ts[] = {dy, x, act != EADGAN_ACT_NONE ? y : nullptr};
  if (int e = make_geo(&g, n, c, h, w, ts, 3, "bn_bwd_reduce")) return e;
  BwdArgs a{};
  a.dy = *dy; a.x = *x; if (y) a.y = *y;
  a.mean = mean; a.invstd = invstd; a.gamma = gamma; a.beta = beta; a.act = act; a.slope = slope;
  const bool gate_x = act == EADGAN_ACT_NONE || act == EADGAN_ACT_RELU || act == EADGAN_ACT_LRELU;
  const eadgan_tensor4* fs[] = {dy, x, gate_x ? nullptr : y};
  if (nhwc8_ok(g, fs, 3)) {
    if (gate_x) bn_bwd_reduce_nhwc8_kernel<true><<<nhwc8_grid(g), 256, 0, (cudaStream_t)stream>>>(a, make_nhwc8(g), sums);
    else bn_bwd_reduce_nhwc8_kernel<false><<<nhwc8_grid(g), 256, 0, (cudaStream_t)stream>>>(a, make_nhwc8(g), sums);
    EG_LAUNCH_CHECK("bn_bwd_reduce_nhwc8_kernel");
    return 0;
  }
  bn_bwd_reduce_kernel<<<reduce_grid(g), 256, 0, (cudaStream_t)stream>>>(a, g, sums);
  EG_LAUNCH_CHECK("bn_bwd_reduce_kernel");
  return 0;
}

extern "C" int eadgan_bn_bwd_apply(const eadgan_tensor4* dy, const eadgan_tensor4* x,
                                   const eadgan_tensor4* y, int n, int c, int h, int w,
                                   const float* mean, const float* invstd, const float* gamma,
                                   const float* beta, int act, float slope, const double* sums,
                                   double count, const eadgan_tensor4* dx, void* stream) {
  Geo g;
  EG_REQUIRE(dy && x && dx && mean && invstd && sums && count > 0, EADGAN_ERR_INVALID,
             "bn_bwd_apply: NULL argument");
  EG_REQUIRE(act == EADGAN_ACT_NONE || y, EADGAN_ERR_INVALID, "bn_bwd_apply: fused activation needs y");
  const eadgan_tensor4* ts[] = {dy, x, dx, act != EADGAN_ACT_NONE ? y : nullptr};
  if (int e = make_geo(&g, n, c, h, w, ts, 4, "bn_bwd_apply")) return e;
  BwdArgs a{};
  a.dy = *dy; a.x = *x; if (y) a.y = *y; a.dx = *dx;
  a.mean = mean; a.invstd = invstd; a.gamma = gamma; a.beta = beta; a.act = act; a.slope = slope;
  a.sums = sums; a.count = count;
  const bool gate_x = act == EADGAN_ACT_NONE || act == EADGAN_ACT_RELU || act == EADGAN_ACT_LRELU;
  const eadgan_tensor4* fs[] = {dy, x, dx, gate_x ? nullptr : y};
  if (nhwc8_ok(g, fs, 4)) {
    if (gate_x) bn_bwd_apply_nhwc8_kernel<true><<<nhwc8_grid(g), 256, 0, (cudaStream_t)stream>>>(a, make_nhwc8(g));
    else bn_bwd_apply_nhwc8_kernel<false><<<nhwc8_grid(g), 256, 0, (cudaStream_t)stream>>>(a, make_nhwc8(g));
    EG_LAUNCH_CHECK("bn_bwd_apply_nhwc8_kernel");
    return 0;
  }
  bn_bwd_apply_kernel<<<elem_grid(g), 256, 0, (cudaStream_t)stream>>>(a, g);
  EG_LAUNCH_CHECK("bn_bwd_apply_kernel");
  return 0;
}

extern "C" int eadgan_bn_bwd_finalize(const double* local_sums, const double* global_sums,
                                      const double* fwd_local_sum_x, double n_local, double count,
                                      const float* mean, const float* invstd, const float* gamma, int c,
                                      float* dgamma, float* dbeta, float* dbias, void* stream) {
  EG_REQUIRE(local_sums && global_sums && mean && invstd && c > 0 && count > 0 && n_local > 0, EADGAN_ERR_INVALID,
             "bn_bwd_finalize: bad arguments");
  bn_bwd_finalize_kernel<<<(c + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      local_sums, global_sums, fwd_local_sum_x, n_local, count, mean, invstd, gamma, c, dgamma, dbeta, dbias);
  EG_LAUNCH_CHECK("bn_bwd_finalize_kernel");
  return 0;
}
