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

// The three backward passes.  BWD_REDUCE (training, first half): sums = [S dz | S dz*xhat] for the cross-rank
// all-reduce.  BWD_APPLY (training, second half): dx from the all-reduced sums.  BWD_EVAL (running statistics): nothing
// depends on the batch, so dx = dz * gamma * rsqrt(rv + eps) is written while the sums are accumulated, in one pass;
// there mean / invstd are running_mean / running_var, with eps.  dz = dy * act'(y), xhat = (x - mean) * invstd.
enum BwdMode { BWD_REDUCE, BWD_APPLY, BWD_EVAL };

struct BwdArgs {
  eadgan_tensor4 dy, x, y, dx;
  const float *mean, *invstd, *gamma, *beta;
  double* sums;   // written by BWD_REDUCE / BWD_EVAL, read by BWD_APPLY
  double count;
  int act;
  float slope;
  float eps;
};

__device__ __forceinline__ float bn_dz(const BwdArgs& a, const Geo& g, int row, int i) {
  float dz = eg_ld(a.dy.ptr, row_base(a.dy, g, row) + i, a.dy.dtype);
  if (a.act != EADGAN_ACT_NONE) {
    const float yv = eg_ld(a.y.ptr, row_base(a.y, g, row) + i, a.y.dtype);
    dz *= eg_act_grad(yv, a.act, a.slope);
  }
  return dz;
}

// BWD_REDUCE or BWD_EVAL.  In eval mode every element is read and written by the same thread, so dx may alias dy.
template <int MODE>
__global__ void __launch_bounds__(256) bn_bwd_reduce_kernel(BwdArgs a, Geo g) {
  auto f = [&](int row, int i, int ch, float& v0, float& v1) {
    const float dz = bn_dz(a, g, row, i);
    const float is = MODE == BWD_EVAL ? rsqrtf(a.invstd[ch] + a.eps) : a.invstd[ch];
    const float xv = eg_ld(a.x.ptr, row_base(a.x, g, row) + i, a.x.dtype);
    if (MODE == BWD_EVAL) {
      const float ga = a.gamma ? a.gamma[ch] : 1.f;
      eg_st(a.dx.ptr, row_base(a.dx, g, row) + i, a.dx.dtype, dz * ga * is);
    }
    v0 = dz;
    v1 = dz * (xv - a.mean[ch]) * is;
  };
  if (g.kind == 0) reduce_kind0(g, a.sums, f); else reduce_kind1(g, a.sums, f);
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
    const float dz = bn_dz(a, g, row, i);
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
// registers.  Bytes per element: apply 2R+2W, bwd reduce 4R (dy, x; the ReLU/LeakyReLU gate is recomputed
// from x with the forward's own expression instead of reading y), bwd apply and eval bwd 4R+2W.
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

// The row walk of every nhwc8 kernel.  A block takes NHWC8_U rows at a time (the pointers of a partial last group are
// clamped to the last row) and, for each of its 16-byte vectors v, issues the loads of the NIN tensors `in` for all
// NHWC8_U rows before it calls body(raw, dst) for each row that exists: raw[k] is vector v of in[k], dst points at
// vector v of `out` (nullptr without OUT).  NHWC8_U independent loads per thread are in flight: one load per thread
// left the kernels latency-bound at ~3 TB/s (2048 threads x 16 B per SM per memory round trip).  in[0] is read with a
// plain load when PLAIN0 (it may be the buffer `out` aliases), every other input through __ldg.
template <int NIN, bool PLAIN0, bool OUT, class Body>
__device__ __forceinline__ void nhwc8_rows(const Nhwc8& g, const eadgan_tensor4* in, const eadgan_tensor4& out,
                                           Body body) {
  const int rows = g.n * g.h;
  for (int row0 = blockIdx.x * NHWC8_U; row0 < rows; row0 += gridDim.x * NHWC8_U) {
    const uint4* r[NHWC8_U][NIN];
    uint4* o[NHWC8_U];
#pragma unroll
    for (int u = 0; u < NHWC8_U; ++u) {
      const int row = min(row0 + u, rows - 1);
      const int b = row / g.h, y = row - b * g.h;
#pragma unroll
      for (int k = 0; k < NIN; ++k) r[u][k] = row_ptr(in[k], b, y);
      o[u] = OUT ? const_cast<uint4*>(row_ptr(out, b, y)) : nullptr;
    }
    for (int v = threadIdx.x; v < g.row_vecs; v += 256) {
      uint4 raw[NHWC8_U][NIN];
#pragma unroll
      for (int u = 0; u < NHWC8_U; ++u) {
#pragma unroll
        for (int k = 0; k < NIN; ++k) raw[u][k] = PLAIN0 && k == 0 ? r[u][k][v] : __ldg(r[u][k] + v);
      }
#pragma unroll
      for (int u = 0; u < NHWC8_U; ++u) {
        if (row0 + u < rows) body(raw[u], OUT ? o[u] + v : nullptr);
      }
    }
  }
}

// the per-channel sums [S s0 | S s1] of the block: 8 channels per thread into shared memory, then one global fp64
// atomic per block and entry
__device__ __forceinline__ void block_sums(int c, int ch0, const float* s0, const float* s1, double* sums) {
  __shared__ double sh[2 * 1024];
  for (int i = threadIdx.x; i < 2 * c; i += 256) sh[i] = 0.0;
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    atomicAdd(&sh[ch0 + j], (double)s0[j]);
    atomicAdd(&sh[c + ch0 + j], (double)s1[j]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * c; i += 256) atomicAdd(&sums[i], sh[i]);
}

struct ChanParams { float mean[8], is[8], ga[8], be[8], sc[8], sh[8], nm[8]; };   // sc = is*ga, sh = be - mean*sc, nm = -mean*is
// eval: mean / invstd are running_mean / running_var, converted to the inverse standard deviation here
__device__ __forceinline__ void load_params(ChanParams& p, int ch0, const float* mean, const float* invstd,
                                            const float* gamma, const float* beta, bool eval, float eps) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    p.mean[j] = mean[ch0 + j];
    p.is[j] = invstd[ch0 + j];
    p.ga[j] = gamma ? gamma[ch0 + j] : 1.f;
    p.be[j] = beta ? beta[ch0 + j] : 0.f;
  }
  if (eval) {
#pragma unroll
    for (int j = 0; j < 8; ++j) p.is[j] = rsqrtf(p.is[j] + eps);
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
  load_params(p, ch0, a.mean, a.invstd, a.gamma, a.beta, a.eval, a.eps);
  derive_params(p);
  const bool leaky = a.act == EADGAN_ACT_RELU || a.act == EADGAN_ACT_LRELU;
  const float neg = a.act == EADGAN_ACT_RELU ? 0.f : a.slope;
  nhwc8_rows<1, false, true>(g, &a.x, a.y, [&](const uint4* raw, uint4* dst) {
    float f[8];
    bf8_to_f32(raw[0], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float t = fmaf(f[j], p.sc[j], p.sh[j]);
      f[j] = leaky ? (t > 0.f ? t : t * neg) : eg_act(t, a.act, a.slope);
    }
    *dst = f32_to_bf8(f);
  });
}

// forward statistics (sum x, sum x^2) of a bf16 NHWC buffer whose producer could not fuse them (dense 1x1 -> 4x4
// layers): same access pattern as the kernels around it instead of one 2-byte load per thread and iteration
__global__ void __launch_bounds__(256) bn_stats_nhwc8_kernel(eadgan_tensor4 x, Nhwc8 g, double* sums) {
  const int ch0 = (threadIdx.x % g.cv) * 8;
  float s0[8], s1[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s0[j] = s1[j] = 0.f;
  nhwc8_rows<1, false, false>(g, &x, x, [&](const uint4* raw, uint4*) {
    float f[8];
    bf8_to_f32(raw[0], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) { s0[j] += f[j]; s1[j] = fmaf(f[j], f[j], s1[j]); }
  });
  block_sums(g.c, ch0, s0, s1, sums);
}

// gate of a ReLU / LeakyReLU that follows the affine transform, recomputed from x exactly as apply did
__device__ __forceinline__ float bn_gate(float x, const ChanParams& p, int j, float slope_neg) {
  return fmaf(x, p.sc[j], p.sh[j]) > 0.f ? 1.f : slope_neg;
}

// The three backward passes (see BwdMode) on the padded bf16 buffers.  GATE_FROM_X: the activation is none, ReLU or
// LeakyReLU, and its gate is recomputed from x (bn_gate) instead of reading y.  In eval mode the parameters are the
// running statistics, converted exactly as bn_apply_nhwc8_kernel converts them, so the recomputed gate equals the
// stored output's gate bit for bit; and dx may alias dy: dy is read with plain loads, and every 16-byte vector is
// loaded before the same thread stores it.
template <int MODE, bool GATE_FROM_X>
__global__ void __launch_bounds__(256) bn_bwd_nhwc8_kernel(BwdArgs a, Nhwc8 g) {
  ChanParams p;
  const int ch0 = (threadIdx.x % g.cv) * 8;
  load_params(p, ch0, a.mean, a.invstd, a.gamma, a.beta, MODE == BWD_EVAL, a.eps);
  derive_params(p);
  const float slope_neg = a.act == EADGAN_ACT_RELU ? 0.f : a.slope;
  const double inv_count = MODE == BWD_APPLY ? 1.0 / a.count : 0.0;
  float s0[8], s1[8];   // BWD_REDUCE / BWD_EVAL: the sums; BWD_APPLY: dx = sc*dz - s0 - xhat*s1
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (MODE == BWD_APPLY) {
      s0[j] = p.sc[j] * (float)(a.sums[ch0 + j] * inv_count);
      s1[j] = p.sc[j] * (float)(a.sums[g.c + ch0 + j] * inv_count);
    } else {
      s0[j] = s1[j] = 0.f;
    }
  }
  const eadgan_tensor4 in[3] = {a.dy, a.x, a.y};
  nhwc8_rows<GATE_FROM_X ? 2 : 3, MODE == BWD_EVAL, MODE != BWD_REDUCE>(g, in, a.dx, [&](const uint4* raw, uint4* dst) {
    float dz[8], xv[8];
    bf8_to_f32(raw[0], dz);
    bf8_to_f32(raw[1], xv);
    if constexpr (GATE_FROM_X) {
      if (a.act != EADGAN_ACT_NONE) {
#pragma unroll
        for (int j = 0; j < 8; ++j) dz[j] *= bn_gate(xv[j], p, j, slope_neg);
      }
    } else {
      float yv[8];
      bf8_to_f32(raw[2], yv);
#pragma unroll
      for (int j = 0; j < 8; ++j) dz[j] *= eg_act_grad(yv[j], a.act, a.slope);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (MODE == BWD_APPLY) {
        const float xhat = fmaf(xv[j], p.is[j], p.nm[j]);
        dz[j] = fmaf(-xhat, s1[j], fmaf(dz[j], p.sc[j], -s0[j]));
      } else {
        s0[j] += dz[j];
        s1[j] = fmaf(dz[j], fmaf(xv[j], p.is[j], p.nm[j]), s1[j]);
        if (MODE == BWD_EVAL) dz[j] *= p.sc[j];
      }
    }
    if (MODE != BWD_REDUCE) *dst = f32_to_bf8(dz);
  });
  if (MODE != BWD_APPLY) block_sums(g.c, ch0, s0, s1, a.sums);
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

// the apply pass of eadgan_bn_apply (batch statistics) and eadgan_bn_eval (running statistics, a.eval)
int bn_apply(const eadgan_tensor4* x, const eadgan_tensor4* y, int n, int c, int h, int w, const ApplyArgs& a,
             void* stream, const char* who) {
  Geo g;
  const eadgan_tensor4* ts[] = {x, y};
  if (int e = make_geo(&g, n, c, h, w, ts, 2, who)) return e;
  if (nhwc8_ok(g, ts, 2)) {
    bn_apply_nhwc8_kernel<<<nhwc8_grid(g), 256, 0, (cudaStream_t)stream>>>(a, make_nhwc8(g));
    EG_LAUNCH_CHECK("bn_apply_nhwc8_kernel");
    return 0;
  }
  bn_apply_kernel<<<elem_grid(g), 256, 0, (cudaStream_t)stream>>>(a, g);
  EG_LAUNCH_CHECK("bn_apply_kernel");
  return 0;
}

// one backward pass (BwdMode) of eadgan_bn_bwd_reduce (dx NULL), eadgan_bn_bwd_apply or eadgan_bn_eval_bwd
template <int MODE>
int bn_bwd(const eadgan_tensor4* dy, const eadgan_tensor4* x, const eadgan_tensor4* y, const eadgan_tensor4* dx,
           int n, int c, int h, int w, const float* mean, const float* invstd, float eps, const float* gamma,
           const float* beta, int act, float slope, double* sums, double count, void* stream, const char* who) {
  EG_REQUIRE(act == EADGAN_ACT_NONE || y, EADGAN_ERR_INVALID, "%s: fused activation needs y", who);
  Geo g;
  const eadgan_tensor4* ts[] = {dy, x, dx, act != EADGAN_ACT_NONE ? y : nullptr};
  if (int e = make_geo(&g, n, c, h, w, ts, 4, who)) return e;
  BwdArgs a{};
  a.dy = *dy; a.x = *x; if (y) a.y = *y; if (dx) a.dx = *dx;
  a.mean = mean; a.invstd = invstd; a.gamma = gamma; a.beta = beta; a.act = act; a.slope = slope; a.eps = eps;
  a.sums = sums; a.count = count;
  cudaStream_t s = (cudaStream_t)stream;
  // the nhwc8 kernels recompute a ReLU / LeakyReLU gate from x and then do not read y
  const bool gate_x = act == EADGAN_ACT_NONE || act == EADGAN_ACT_RELU || act == EADGAN_ACT_LRELU;
  const eadgan_tensor4* fs[] = {dy, x, dx, gate_x ? nullptr : y};
  if (nhwc8_ok(g, fs, 4)) {
    (gate_x ? bn_bwd_nhwc8_kernel<MODE, true> : bn_bwd_nhwc8_kernel<MODE, false>)<<<nhwc8_grid(g), 256, 0, s>>>(
        a, make_nhwc8(g));
    EG_LAUNCH_CHECK("bn_bwd_nhwc8_kernel");
  } else if constexpr (MODE == BWD_APPLY) {
    bn_bwd_apply_kernel<<<elem_grid(g), 256, 0, s>>>(a, g);
    EG_LAUNCH_CHECK("bn_bwd_apply_kernel");
  } else {
    bn_bwd_reduce_kernel<MODE><<<reduce_grid(g), 256, 0, s>>>(a, g);
    EG_LAUNCH_CHECK("bn_bwd_reduce_kernel");
  }
  return 0;
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
  EG_REQUIRE(x && y && mean && invstd, EADGAN_ERR_INVALID, "bn_apply: NULL argument");
  return bn_apply(x, y, n, c, h, w, ApplyArgs{*x, *y, mean, invstd, gamma, beta, act, slope, 0.f, 0}, stream,
                  "bn_apply");
}

extern "C" int eadgan_bn_eval(const eadgan_tensor4* x, int n, int c, int h, int w,
                              const float* running_mean, const float* running_var, float eps,
                              const float* gamma, const float* beta, int act, float slope,
                              const eadgan_tensor4* y, void* stream) {
  EG_REQUIRE(x && y && running_mean && running_var, EADGAN_ERR_INVALID, "bn_eval: NULL argument");
  return bn_apply(x, y, n, c, h, w, ApplyArgs{*x, *y, running_mean, running_var, gamma, beta, act, slope, eps, 1},
                  stream, "bn_eval");
}

extern "C" int eadgan_bn_eval_bwd(const eadgan_tensor4* dy, const eadgan_tensor4* x, const eadgan_tensor4* y,
                                  int n, int c, int h, int w, const float* running_mean, const float* running_var,
                                  float eps, const float* gamma, const float* beta, int act, float slope,
                                  double* sums, const eadgan_tensor4* dx, float* dgamma, float* dbeta, float* dbias,
                                  void* stream) {
  EG_REQUIRE(dy && x && dx && running_mean && running_var && sums, EADGAN_ERR_INVALID,
             "bn_eval_bwd: NULL argument");
  if (int e = bn_bwd<BWD_EVAL>(dy, x, y, dx, n, c, h, w, running_mean, running_var, eps, gamma, beta, act, slope,
                               sums, 0.0, stream, "bn_eval_bwd"))
    return e;
  if (dgamma || dbeta || dbias) {
    bn_eval_bwd_finalize_kernel<<<(c + 127) / 128, 128, 0, (cudaStream_t)stream>>>(sums, running_var, eps, gamma, c,
                                                                                  dgamma, dbeta, dbias);
    EG_LAUNCH_CHECK("bn_eval_bwd_finalize_kernel");
  }
  return 0;
}

extern "C" int eadgan_bn_bwd_reduce(const eadgan_tensor4* dy, const eadgan_tensor4* x,
                                    const eadgan_tensor4* y, int n, int c, int h, int w,
                                    const float* mean, const float* invstd, const float* gamma,
                                    const float* beta, int act, float slope, double* sums,
                                    void* stream) {
  EG_REQUIRE(dy && x && mean && invstd && sums, EADGAN_ERR_INVALID, "bn_bwd_reduce: NULL argument");
  return bn_bwd<BWD_REDUCE>(dy, x, y, nullptr, n, c, h, w, mean, invstd, 0.f, gamma, beta, act, slope, sums, 0.0,
                            stream, "bn_bwd_reduce");
}

extern "C" int eadgan_bn_bwd_apply(const eadgan_tensor4* dy, const eadgan_tensor4* x,
                                   const eadgan_tensor4* y, int n, int c, int h, int w,
                                   const float* mean, const float* invstd, const float* gamma,
                                   const float* beta, int act, float slope, const double* sums,
                                   double count, const eadgan_tensor4* dx, void* stream) {
  EG_REQUIRE(dy && x && dx && mean && invstd && sums && count > 0, EADGAN_ERR_INVALID,
             "bn_bwd_apply: NULL argument");
  return bn_bwd<BWD_APPLY>(dy, x, y, dx, n, c, h, w, mean, invstd, 0.f, gamma, beta, act, slope,
                           const_cast<double*>(sums), count, stream, "bn_bwd_apply");   // BWD_APPLY only reads sums
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
