// tcgen05 / TMEM / TMA implicit-GEMM convolution for kernel 4, stride 2, pad 1 (the
// geometry of every heavy layer of EAD-GAN: celebA/EAD-GAN_celebA.py:78-87,113-119,
// dSprites/rp.py:66-75,95-104,129-141,165-174).  bf16 operands, fp32 accumulation
// in tensor memory.  Written for sm_100a only.
//
// Data layout.  Every activation lives in a private halo-padded NHWC bf16 buffer
// X[n][H+2][W+2][C] whose 1-pixel halo is zero.  With the halo in memory there is no
// boundary special case, and both operand gathers become plain TMA *tiled* boxes:
//
//  * FPROP (Conv2d forward, ConvTranspose2d input-grad): y[oy,ox] = sum_{ky,kx,c}
//    Xp[2oy+ky][2ox+kx][c] w[ky][kx][c].  Writing ky=2a+dy, kx=2b+dx, the padded map
//    is viewed as a 5-D tensor (dx*C+c, j, dy, i, n) with Xp[2i+dy][2j+dx] (space to
//    depth by strides only, no copy); tap (a,b,dy) of an output tile is the box
//    [64 ch] x [Tw] x [1] x [Th] x [Tb] at (q*64, ox0+b, dy, oy0+a, n0).
//    GEMM: M = n*p*q pixels, N = k, K = 16*c ordered (a,b,dy,dx,c).
//  * DGRAD (ConvTranspose2d forward, Conv2d input-grad): four output-parity
//    sub-convolutions with 2x2 taps (SURVEY.md appendix D.1); tap (ty,tx) of parity
//    (py,px) is the 4-D box at (q*64, j0+1+dx, i0+1+dy, n0) of the small map.
//    GEMM per parity: M = n*p*q, N = c, K = 4*k.
//  * WGRAD: dw[ko][kk] = sum_pixels dy[pix][ko] * patch[pix][kk]; both operands are
//    "MN-major" (the reduction runs over smem rows), 64 pixels per pipeline stage,
//    split over the pixel dimension, fp32 partials reduced + permuted to [k,c,4,4].
//
// Kernel anatomy (all three): 192 threads = warp 0 TMA producer (one elected lane),
// warp 1 TMEM allocator + single-thread tcgen05.mma issuer, warps 2..5 epilogue
// (tcgen05.ld 32x32b, one TMEM lane quadrant each).  smem ring of STAGES x (A|B)
// tiles with 128-byte swizzle, full/empty mbarriers, tcgen05.commit releases slots.
#include <cuda.h>

#include <atomic>
#include <mutex>
#include <cstdio>
#include <cstdlib>

#include "common.cuh"

namespace {

// ------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%0], %1;\n\t"
      "@P bra.uni WAIT_DONE;\n\t"
      "bra.uni WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// TMA tiled loads.  `bar` is a shared::cluster ADDRESS (uint32): the CTA's own barrier for cta_group::1 kernels,
// the LEADER CTA's barrier (mapa to rank 0) for cta_group::2 kernels, whose loads land in the issuing CTA's shared
// memory but signal their bytes on the pair leader's full barrier (CUTLASS SM100_TMA_2SM_LOAD_*).
template <int CG>
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  if constexpr (CG == 1)
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
  else
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
        "%4}], [%2];" ::"r"(smem_u32(dst)), "l"(map), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
template <int CG>
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  if constexpr (CG == 1)
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
        "[%2];" ::"r"(smem_u32(dst)),
        "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
  else
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
        "%4, %5, %6}], [%2];" ::"r"(smem_u32(dst)),
        "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
template <int CG>
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  if constexpr (CG == 1)
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, "
        "%7}], [%2];" ::"r"(smem_u32(dst)),
        "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
  else
    asm volatile(
        "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
        "%4, %5, %6, %7}], [%2];" ::"r"(smem_u32(dst)),
        "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
// ---- thread-block cluster / CTA pair (cta_group::2) helpers ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa(uint32_t local_smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on a barrier given by its shared::cluster address (possibly in the peer CTA)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

template <int CG = 1>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  if constexpr (CG == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {   // issued by the same warp of BOTH CTAs of the pair, same destination offset
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
}
template <int CG = 1>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  if constexpr (CG == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate
// cta_group::2: issued by the pair LEADER only; the instruction spans both SMs (M = 256: rows 0..127 from the
// leader's A tile, 128..255 from the peer's, at the same shared-memory offsets; each CTA holds half of the B rows)
template <int CG = 1>
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  if constexpr (CG == 1)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on `bar` once every MMA issued so far has completed; cta_group::2: on the barrier at the same
// shared-memory offset in BOTH CTAs of the pair (multicast, mask 0b11)
template <int CG = 1>
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  if constexpr (CG == 1)
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
  else
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3)
                 : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// UMMA shared-memory descriptor, 128-byte swizzle (cute::UMMA::SmemDescriptor, version 1)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;  // LayoutType::SWIZZLE_128B
  return d;
}
// cute::UMMA::InstrDescriptor for kind::f16: bf16 x bf16 -> fp32
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ------------------------------------------------------------------------------------
// kernel parameters
// ------------------------------------------------------------------------------------
enum { MODE_GEMM = 0, MODE_FPROP = 1, MODE_DGRAD = 2, MODE_DENSE_GATHER = 3 };

struct TcParams {
  int mode;
  int n, p, q;        // GEMM pixel grid: n images of p x q positions
  int Tw, Th, Tb;     // tile of 128 positions = Tb x Th x Tw
  int tiles_y;        // p / Th
  int N_total;        // output channels of this direction (k for fprop, c for dgrad)
  int K_ch;           // operand channels: fprop c (big map), dgrad k (small map); gemm: K
  int nkb;            // number of 64-wide k blocks
  int qblocks;        // fprop: 2c/64 ; dgrad: k/64
  // epilogue
  int act; float slope;
  int out_f32_nchw, want_stats, mask_mode;
  int OH, OW;         // output map extents (fprop: p,q ; dgrad: 2p,2q)
  const float* bias;
  void* out;
  const __nv_bfloat16* mask;
  double* stats;
  int gemm_m, gemm_n;  // MODE_GEMM extents
  int n_store;         // real output channels (<= N_total; the rest is zero padding of the operand)
  int dense_C;         // > 0: 4x4 <-> 1x1 "dense" layers; channels of the padded [n,6,6,C] map
  int m_tiles, n_tiles, parities;  // persistent tile space: tile = (m_tile * parities + parity) * n_tiles + n_tile
  int stat_channels;   // length of one statistics vector (stats = [sum | sum of squares])
  int thin;            // fprop on a <= 4-channel image: ONE 64-wide k block, A boxes from the row-expanded buffer
  int bias_len;        // number of bias entries (n_store, or dense_C for the scatter GEMM)
  const float* sigma;  // spectral-norm sigma (device scalar) or NULL: accumulators are multiplied by 1/sigma, so the
                       // packed bf16 operand can be the UN-normalised weight_orig (cached across forwards)
};

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;
constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KB
constexpr int STAT_MAX_CH = 1024;               // per-CTA running statistics cover up to this many channels

// MT = number of 128-row M tiles per CTA tile (1 or 2): MT = 2 halves the B re-reads.
// CG = tcgen05 cta_group: 1 = one CTA computes a (MT x 128) x BLOCK_N tile; 2 = a CTA PAIR (cluster of two SMs of one
// TPC) computes (2 x MT x 128) x BLOCK_N with one MMA stream issued by the pair leader: each CTA stages its own A rows
// and only HALF of the B rows, so the shared-memory traffic per MAC (TMA writes + MMA operand reads) drops by a third
// at BLOCK_N = 256 (125 instead of 188 B/clk/SM at full tensor rate), and the ring is 6 stages of 32 KB instead of 4 of 48.
template <int BLOCK_N, int MT, int CG>
struct Cfg {
  static_assert(CG == 1 || CG == 2, "cta_group");
  static constexpr int B_BYTES = (BLOCK_N / CG) * BLOCK_K * 2;  // this CTA's share of the B tile
  static constexpr int STAGE_BYTES = MT * A_BYTES + B_BYTES;
  static constexpr int ACC_COLS = BLOCK_N < 32 ? 32 : BLOCK_N;  // TMEM columns of ONE 128-row accumulator
  static constexpr int BUF_COLS = MT * ACC_COLS;                // one accumulator buffer (MT sub-tiles)
  static constexpr int TMEM_COLS = 2 * BUF_COLS;                // two buffers: epilogue(i) overlaps mainloop(i+1)
  static_assert(TMEM_COLS <= 512, "accumulators exceed tensor memory");
  static constexpr int BAR_BYTES = 256;
  static constexpr int STAT_PART_BYTES = 4 * BLOCK_N * 2 * 4;   // float [4 warps][BLOCK_N][2]
  static constexpr int STAT_ACC_BYTES = STAT_MAX_CH * 2 * 8;    // double [channels][2]
  static constexpr int BIAS_BYTES = STAT_MAX_CH * 4;            // float [channels]: the bias vector, staged once
  static constexpr int FIXED_BYTES = 1024 /*align*/ + BAR_BYTES + STAT_PART_BYTES + STAT_ACC_BYTES + BIAS_BYTES;
  static constexpr int RING_BUDGET = 227 * 1024 - FIXED_BYTES;
  static constexpr int STAGES = RING_BUDGET / STAGE_BYTES < 8 ? RING_BUDGET / STAGE_BYTES : 8;
  static_assert(2 * STAGES + 4 <= BAR_BYTES / 8 - 1, "barrier block too small");
  static constexpr int SMEM = STAGES * STAGE_BYTES + FIXED_BYTES;
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// per-channel totals over the 32 rows of a warp: butterfly transpose-reduce; lane l ends up with channel l
template <bool SQ>
__device__ __forceinline__ void warp_col_sums(const float* v, bool valid, int lane, float& o1, float& o2) {
  float s1[32], s2[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) { s1[j] = valid ? v[j] : 0.f; s2[j] = SQ ? s1[j] * s1[j] : 0.f; }
#pragma unroll
  for (int w = 16; w >= 1; w >>= 1) {
#pragma unroll
    for (int j = 0; j < w; ++j) {
      const bool up = (lane & w) != 0;
      const float a1 = up ? s1[j] : s1[j + w], k1 = up ? s1[j + w] : s1[j];
      s1[j] = k1 + __shfl_xor_sync(0xffffffffu, a1, w);
      if (SQ) {
        const float a2 = up ? s2[j] : s2[j + w], k2 = up ? s2[j + w] : s2[j];
        s2[j] = k2 + __shfl_xor_sync(0xffffffffu, a2, w);
      }
    }
  }
  o1 = s1[0];
  o2 = s2[0];
}


// where row `row` of sub-tile h of persistent tile `tile` lives in the output / mask tensors
struct RowInfo {
  bool valid, f32_out;
  int n0, bias_base;
  int64_t out_off, ch_stride, mask_off;
};
template <int BLOCK_N, int MT, int CG>
__device__ __forceinline__ RowInfo row_info(const TcParams& P, int tile, int h, int row, int rank) {
  RowInfo ri;
  const int n_tile = tile % P.n_tiles, r = tile / P.n_tiles;
  const int parity = r % P.parities, m_tile = ((r / P.parities) * CG + rank) * MT + h;
  const int py = parity >> 1, px = parity & 1;
  const int n0 = n_tile * BLOCK_N;
  ri.n0 = n0; ri.bias_base = n0; ri.out_off = 0; ri.ch_stride = 1; ri.mask_off = 0;
  if (P.mode == MODE_GEMM || P.mode == MODE_DENSE_GATHER) {
    const int m = m_tile * BLOCK_M + row;
    ri.valid = m < P.gemm_m;
    if (P.mode == MODE_GEMM && P.dense_C > 0) {
      // scatter: GEMM column n = tap * C + ch  ->  padded map [m][1+ky][1+kx][ch]
      const int tap = n0 / P.dense_C, ch0 = n0 - tap * P.dense_C;
      ri.out_off = (((int64_t)m * 6 + 1 + (tap >> 2)) * 6 + 1 + (tap & 3)) * P.dense_C + ch0;
      ri.mask_off = ri.out_off;
      ri.bias_base = ch0;
      ri.f32_out = false;
    } else {
      ri.out_off = (int64_t)m * P.n_store + n0;
      if (P.mode == MODE_DENSE_GATHER) ri.out_off += (int64_t)parity * P.gemm_m * P.n_store;   // split-K slab
      ri.f32_out = true;
    }
  } else {
    const int b0 = (m_tile / P.tiles_y) * P.Tb, y0 = (m_tile % P.tiles_y) * P.Th;
    const int xl = row % P.Tw, yl = (row / P.Tw) % P.Th, bl = row / (P.Tw * P.Th);
    const int b = b0 + bl;
    ri.valid = b < P.n;
    int oy, ox;
    if (P.mode == MODE_FPROP) { oy = y0 + yl; ox = xl; }
    else { oy = 2 * (y0 + yl) + py; ox = 2 * xl + px; }
    const int64_t pad_off = (((int64_t)b * (P.OH + 2) + oy + 1) * (P.OW + 2) + ox + 1) * P.N_total + n0;
    ri.mask_off = pad_off;
    ri.f32_out = P.out_f32_nchw != 0;
    if (ri.f32_out) {
      ri.out_off = (((int64_t)b * P.n_store + n0) * P.OH + oy) * P.OW + ox;
      ri.ch_stride = (int64_t)P.OH * P.OW;
    } else {
      ri.out_off = pad_off;
    }
  }
  return ri;
}

// ------------------------------------------------------------------------------------
// fprop / dgrad / gemm kernel.  PERSISTENT: grid <= number of SMs, CTA c runs tiles c, c+grid, ...
// (n-tile fastest so concurrently running CTAs share the streamed A operand through L2).
// ------------------------------------------------------------------------------------
template <int BLOCK_N, int MT, int CG>
__global__ void __launch_bounds__(320, 1)
tc_conv_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
               const TcParams P) {
  using C = Cfg<BLOCK_N, MT, CG>;
  extern __shared__ uint8_t smem_raw[];
  // align by OFFSETTING the shared array (not by integer round trip): the compiler keeps the shared address
  // space, so every access below is LDS/STS instead of a generic LD/ST through the L1TEX path
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* tiles = smem;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tmem_full_bar = empty_bar + C::STAGES;   // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;      // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
  float* stat_part = reinterpret_cast<float*>(smem + C::STAGES * C::STAGE_BYTES + C::BAR_BYTES);
  double* stat_acc = reinterpret_cast<double*>(smem + C::STAGES * C::STAGE_BYTES + C::BAR_BYTES + C::STAT_PART_BYTES);
  float* bias_s = reinterpret_cast<float*>(smem + C::STAGES * C::STAGE_BYTES + C::BAR_BYTES + C::STAT_PART_BYTES +
                                           C::STAT_ACC_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_tiles = P.parities * P.m_tiles * P.n_tiles;
  // cta_group::2: the two CTAs of a pair walk the SAME tile list (first = pair index, step = number of pairs);
  // rank 0 is the leader (issues the MMAs, owns the full / accumulator-empty barriers both CTAs signal)
  const int rank = CG == 2 ? (int)cluster_ctarank() : 0;
  const int first_tile = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int tile_step = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
  }
  if (warp == 1) {
    if (lane == 0) {
      // full: ONE arrival -- the leader's arrive.expect_tx of the bytes of BOTH CTAs; the peer only issues its loads,
      // whose bytes complete on the leader's barrier (a peer load can land before the leader's expect_tx of the same
      // phase: the transaction count is then transiently negative, which mbarriers allow; it cannot land in an
      // earlier phase, because the slot is only released once the MMAs that consumed that phase have completed)
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
      // accumulator empty: the 8 epilogue warps of every CTA of the group
      for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full_bar[b], 1); mbar_init(&tmem_empty_bar[b], 8 * CG); }
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc<CG>(tmem_ptr, C::TMEM_COLS);
  }
  if (warp >= 2) {
    if (P.want_stats) {
      for (int i = threadIdx.x - 64; i < 2 * P.stat_channels; i += 256) stat_acc[i] = 0.0;
      for (int i = threadIdx.x - 64; i < 4 * BLOCK_N * 2; i += 256) stat_part[i] = 0.f;
    }
    if (P.bias) {  // bias_len <= STAT_MAX_CH (checked on the host)
      for (int i = threadIdx.x - 64; i < P.bias_len; i += 256) bias_s[i] = __ldg(&P.bias[i]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CG == 2) cluster_sync();   // the peer's barriers exist before anybody signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===== TMA producer (one per CTA: its own A rows and its share of the B rows) =====
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = first_tile; tile < total_tiles; tile += tile_step) {
        const int n_tile = tile % P.n_tiles, r = tile / P.n_tiles;
        // parity next-fastest: the 4 output parities of an M tile read the SAME input tile (shifted taps), so they
        // run back to back / side by side and share it through L2 instead of re-streaming it from HBM 4 times
        const int parity = r % P.parities;
        const int m_grp = (r / P.parities) * CG + rank;   // this CTA's group of MT consecutive 128-row tiles
        const int py = parity >> 1, px = parity & 1;
        const int n0 = n_tile * BLOCK_N + rank * (BLOCK_N / CG);      // first B row this CTA stages
        const int b_row = (P.mode == MODE_DGRAD ? parity * P.N_total : 0) + n0;
        // Everything that needs an integer division is computed ONCE PER TILE: this single thread issues every load
        // of the CTA, and with divisions inside the k loop it was the instruction-bound stage of the whole pipeline
        // (ncu r02a: the producer never waited for a free slot while the MMA warp waited for data a quarter of the time)
        int b0[MT], y0[MT];
#pragma unroll
        for (int h = 0; h < MT; ++h) {
          const int m_tile = m_grp * MT + h;
          if (P.mode == MODE_GEMM || P.mode == MODE_DENSE_GATHER) { b0[h] = m_tile * BLOCK_M; y0[h] = 0; }
          else { b0[h] = (m_tile / P.tiles_y) * P.Tb; y0[h] = (m_tile % P.tiles_y) * P.Th; }
        }
        // k block -> (tap t, 64-channel block qi); dense gather: the K range is split over the "parity" index (split-K)
        const int kb0 = P.mode == MODE_DENSE_GATHER ? parity * P.nkb : 0;
        int qi = kb0 % P.qblocks, t = kb0 / P.qblocks;
#pragma unroll 1
        for (int kb = 0; kb < P.nkb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = tiles + stage * C::STAGE_BYTES;
          uint8_t* sb = sa + MT * A_BYTES;
          uint32_t fb = smem_u32(&full_bar[stage]);
          if constexpr (CG == 2) {
            fb = mapa(fb, 0);
            if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * C::STAGE_BYTES);
          } else {
            mbar_expect_tx(&full_bar[stage], C::STAGE_BYTES);
          }
          const int kcol = qi * BLOCK_K;
          int b_col = (kb0 + kb) * BLOCK_K;
          if (P.mode == MODE_GEMM) {
#pragma unroll
            for (int h = 0; h < MT; ++h) tma_load_2d<CG>(sa + h * A_BYTES, &map_a, fb, kb * BLOCK_K, b0[h]);
          } else if (P.mode == MODE_DENSE_GATHER) {
            // A[b][(tap, c)] = Y[b][1+ky][1+kx][c]: box [64 ch] x 1 x 1 x [128 images]  (t = tap)
#pragma unroll
            for (int h = 0; h < MT; ++h) tma_load_4d<CG>(sa + h * A_BYTES, &map_a, fb, kcol, 1 + (t & 3), 1 + (t >> 2), b0[h]);
          } else if (P.mode == MODE_FPROP && P.thin) {
            // R[n][oy][X][ky][4]: the 4x4x4 patch of output (oy, ox) is the 64 contiguous elements at X = 2 ox
#pragma unroll
            for (int h = 0; h < MT; ++h) tma_load_4d<CG>(sa + h * A_BYTES, &map_a, fb, 0, 0, y0[h], b0[h]);
          } else if (P.mode == MODE_FPROP) {
            const int dy = t & 1, bt = (t >> 1) & 1, at = t >> 2;
#pragma unroll
            for (int h = 0; h < MT; ++h) tma_load_5d<CG>(sa + h * A_BYTES, &map_a, fb, kcol, bt, dy, y0[h] + at, b0[h]);
          } else {  // dgrad: t = ty*2+tx
            const int ty = t >> 1, tx = t & 1;
            const int dy = py == 0 ? (ty == 0 ? 0 : -1) : (ty == 0 ? 1 : 0);
            const int dx = px == 0 ? (tx == 0 ? 0 : -1) : (tx == 0 ? 1 : 0);
#pragma unroll
            for (int h = 0; h < MT; ++h) tma_load_4d<CG>(sa + h * A_BYTES, &map_a, fb, kcol, 1 + dx, y0[h] + 1 + dy, b0[h]);
            // tap t's weights start at column t * K_ch (= kb * 64 whenever K_ch is a multiple of 64; for K_ch = 32 the
            // box also covers 32 columns of the next tap, multiplied by the zero-filled half of A)
            b_col = t * P.K_ch + kcol;
          }
          tma_load_2d<CG>(sb, &map_b, fb, b_col, b_row);
          if (++qi == P.qblocks) { qi = 0; ++t; }
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (cta_group::2: the pair leader only; its instructions drive both SMs) =====
    constexpr uint32_t idesc = make_idesc(BLOCK_M * CG, BLOCK_N, 0, 0);
    int stage = 0; uint32_t phase = 0;
    int it = 0;
    for (int tile = first_tile; tile < total_tiles && rank == 0; tile += tile_step, ++it) {
      const int buf = it & 1;
      mbar_wait(&tmem_empty_bar[buf], ((it >> 1) & 1) ^ 1);  // epilogue has drained this accumulator
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(buf * C::BUF_COLS);
      for (int kb = 0; kb < P.nkb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_u32(tiles + stage * C::STAGE_BYTES);
          const uint32_t sb = sa + MT * A_BYTES;
#pragma unroll
          for (int k = 0; k < BLOCK_K / 16; ++k) {
            const uint64_t db = make_desc(sb + k * 32, 16, 1024);
#pragma unroll
            for (int h = 0; h < MT; ++h) {
              const uint64_t da = make_desc(sa + h * A_BYTES + k * 32, 16, 1024);
              umma_bf16<CG>(d_tmem + (uint32_t)(h * C::ACC_COLS), da, db, idesc, (kb > 0 || k > 0) ? 1u : 0u);
            }
          }
          umma_commit<CG>(&empty_bar[stage]);                         // frees the slot in both CTAs
          if (kb == P.nkb - 1) umma_commit<CG>(&tmem_full_bar[buf]);  // wakes the epilogue warps of both CTAs
        }
        __syncwarp();
        if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ===== epilogue: TMEM -> registers -> global.  8 warps: two per TMEM lane quadrant, splitting the
    // 32-column chunks of the tile between them (chunk ci belongs to warp-half ci & 1) =====
    const int quad = warp & 3;            // TMEM lane quadrant this warp may read
    const int half = (warp - 2) >> 2;     // 0: warps 2..5, 1: warps 6..9
    const int row = quad * 32 + lane;     // row of the 128-row tile
    const int et = threadIdx.x - 64;      // 0..255
    constexpr int NCHUNK = BLOCK_N / 32;
    const float inv_sigma = P.sigma ? 1.f / __ldg(P.sigma) : 1.f;
    // the accumulator-empty barriers live in the pair leader (the MMA issuer waits on them)
    uint32_t te_bar[2] = {smem_u32(&tmem_empty_bar[0]), smem_u32(&tmem_empty_bar[1])};
    if constexpr (CG == 2) { te_bar[0] = mapa(te_bar[0], 0); te_bar[1] = mapa(te_bar[1], 0); }
    auto te_arrive = [&](int b) {
      if constexpr (CG == 2) mbar_arrive_cluster(te_bar[b]);
      else mbar_arrive(&tmem_empty_bar[b]);
    };
    int it = 0;
    for (int tile = first_tile; tile < total_tiles; tile += tile_step, ++it) {
      if (P.mask_mode) {
        // pull the NEXT tile's mask rows into L2 now: by the time its accumulator is ready the loads below
        // are L2 hits instead of DRAM round trips (the epilogue is latency-bound otherwise)
        const int nt = tile + tile_step;
        if (nt < total_tiles) {
#pragma unroll
          for (int h = 0; h < MT; ++h) {
            const RowInfo ri = row_info<BLOCK_N, MT, CG>(P, nt, h, row, rank);
            if (ri.valid) {
              for (int l = half; l < (BLOCK_N >= 64 ? BLOCK_N / 64 : 1); l += 2)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(P.mask + ri.mask_off + l * 64));
            }
          }
        }
      }
      const int buf = it & 1;
      mbar_wait(&tmem_full_bar[buf], (it >> 1) & 1);
      tc_fence_after();
      if (half >= NCHUNK) {  // BLOCK_N = 32: the second warp of each quadrant has no columns
        if (lane == 0) te_arrive(buf);
      }
#pragma unroll 1
      for (int h = 0; h < MT; ++h) {
        const RowInfo ri = row_info<BLOCK_N, MT, CG>(P, tile, h, row, rank);
        const bool valid = ri.valid, f32_out = ri.f32_out;
        const int n0 = ri.n0, bias_base = ri.bias_base;
        const int64_t ch_stride = ri.ch_stride;
        const uint32_t acc = tmem_base + (uint32_t)(buf * C::BUF_COLS + h * C::ACC_COLS) + ((uint32_t)(quad * 32) << 16);

#pragma unroll 1
        for (int ci = half; ci < NCHUNK; ci += 2) {
          const int c0 = ci * 32;
          const int n_left = P.n_store - (n0 + c0);  // real channels remaining from this column on
          const bool live = valid && (n_left > 0 || P.dense_C > 0);
          uint4 mv[4];
          if (P.mask_mode && live) {  // issue the mask loads before waiting for the accumulator
            const uint4* mp = reinterpret_cast<const uint4*>(P.mask + ri.mask_off + c0);
#pragma unroll
            for (int g = 0; g < 4; ++g) mv[g] = __ldg(mp + g);
          }
          float v[32];
          tmem_ld32(acc + (uint32_t)c0, v);
          if (ci + 2 >= NCHUNK && h == MT - 1) {
            // all of this warp's columns are in registers: hand the TMEM buffer back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) te_arrive(buf);
          }
          if (P.sigma) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= inv_sigma;
          }
          if (P.bias) {
            if (n_left >= 32 || P.dense_C > 0) {  // 32 consecutive channels: eight 16-byte broadcast LDS
              const float4* bp = reinterpret_cast<const float4*>(bias_s + bias_base + c0);
#pragma unroll
              for (int g = 0; g < 8; ++g) {
                const float4 b4 = bp[g];
                v[g * 4 + 0] += b4.x; v[g * 4 + 1] += b4.y; v[g * 4 + 2] += b4.z; v[g * 4 + 3] += b4.w;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (j < n_left) v[j] += bias_s[bias_base + c0 + j];
            }
          }
          if (P.want_stats == 1) {  // BatchNorm statistics of the pre-activation output
            float o1, o2;
            warp_col_sums<true>(v, valid, lane, o1, o2);
            stat_part[(quad * BLOCK_N + c0 + lane) * 2 + 0] += o1;   // entry owned by this warp alone
            stat_part[(quad * BLOCK_N + c0 + lane) * 2 + 1] += o2;
          }
          if (live) {
            // the activation kind is uniform for the launch: branch ONCE, outside the element loops
            if (P.act == EADGAN_ACT_RELU || P.act == EADGAN_ACT_LRELU) {
              const float sl = P.act == EADGAN_ACT_RELU ? 0.f : P.slope;
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = v[j] > 0.f ? v[j] : v[j] * sl;
            } else if (P.act == EADGAN_ACT_TANH) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = tanhf(v[j]);
            } else if (P.act == EADGAN_ACT_SIGMOID) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = 1.f / (1.f + expf(-v[j]));
            }
            if (P.mask_mode == EADGAN_ACT_RELU || P.mask_mode == EADGAN_ACT_LRELU) {
              const float sl = P.mask_mode == EADGAN_ACT_RELU ? 0.f : P.slope;
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                const uint32_t mw[4] = {mv[g].x, mv[g].y, mv[g].z, mv[g].w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  // saved OUTPUT y > 0  <=>  pre-activation > 0; bf16 sign/zero test on the raw bits
                  const bool lo_pos = (mw[e] & 0x8000u) == 0 && (mw[e] & 0x7fffu) != 0;
                  const bool hi_pos = (mw[e] & 0x80000000u) == 0 && (mw[e] & 0x7fff0000u) != 0;
                  if (!lo_pos) v[g * 8 + e * 2 + 0] *= sl;
                  if (!hi_pos) v[g * 8 + e * 2 + 1] *= sl;
                }
              }
            } else if (P.mask_mode) {
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                const uint32_t mw[4] = {mv[g].x, mv[g].y, mv[g].z, mv[g].w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float m_lo = __uint_as_float(mw[e] << 16), m_hi = __uint_as_float(mw[e] & 0xffff0000u);
                  v[g * 8 + e * 2 + 0] *= eg_act_grad(m_lo, P.mask_mode, P.slope);
                  v[g * 8 + e * 2 + 1] *= eg_act_grad(m_hi, P.mask_mode, P.slope);
                }
              }
            }
          }
          if (P.want_stats == 2) {  // per-channel sums of the FINAL value (bias gradient of the layer below)
            float o1, o2;
            warp_col_sums<false>(v, live, lane, o1, o2);
            stat_part[(quad * BLOCK_N + c0 + lane) * 2 + 0] += o1;
          }
          if (live) {
            if (f32_out) {
              float* op = reinterpret_cast<float*>(P.out) + ri.out_off + (int64_t)c0 * ch_stride;
              if (ch_stride == 1 && n_left >= 32 && (P.n_store & 3) == 0) {
#pragma unroll
                for (int g = 0; g < 8; ++g)
                  *reinterpret_cast<float4*>(op + g * 4) = make_float4(v[g * 4], v[g * 4 + 1], v[g * 4 + 2], v[g * 4 + 3]);
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (j < n_left) op[(int64_t)j * ch_stride] = v[j];
              }
            } else {
              // (measured, r02o: exchanging 16-byte pieces inside lane quads so that every store instruction writes
              // eight 64-byte runs instead of 32 scattered 16-byte pieces made the step 1 ms SLOWER -- this epilogue
              // is bound by instruction issue and latency, not by the number of lines its stores touch)
              __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(P.out) + ri.out_off + c0;
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                uint32_t pk[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  __nv_bfloat162 h2 = __floats2bfloat162_rn(v[g * 8 + e * 2], v[g * 8 + e * 2 + 1]);
                  pk[e] = *reinterpret_cast<uint32_t*>(&h2);
                }
                *reinterpret_cast<uint4*>(op + g * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
              }
            }
          }
        }
        if (P.want_stats && h == MT - 1) {
          // Each warp keeps fp32 running column sums of ITS rows / chunks in stat_part (no sharing, no barrier).
          // They are folded into the CTA's fp64 per-channel totals only when the next tile of this CTA covers a
          // different channel block (or there is no next tile): thread et owns channel bias_base + et [+ 256 ...]
          const int nt = tile + tile_step;
          const bool fold = nt >= total_tiles || (nt % P.n_tiles) != (tile % P.n_tiles) ||
                            (P.dense_C > 0);
          if (fold) {
            asm volatile("bar.sync 1, 256;" ::: "memory");
            for (int ch = et; ch < BLOCK_N; ch += 256) {
              const int gch = bias_base + ch;
              float a = 0.f, b2 = 0.f;
#pragma unroll
              for (int w = 0; w < 4; ++w) {
                a += stat_part[(w * BLOCK_N + ch) * 2]; b2 += stat_part[(w * BLOCK_N + ch) * 2 + 1];
                stat_part[(w * BLOCK_N + ch) * 2] = 0.f; stat_part[(w * BLOCK_N + ch) * 2 + 1] = 0.f;
              }
              if (gch < P.stat_channels) {
                stat_acc[gch * 2 + 0] += (double)a;
                stat_acc[gch * 2 + 1] += (double)b2;
              }
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
          }
        }
      }  // sub-tile h
    }
    if (P.want_stats) {
      // one flush per CTA: 2 fp64 atomics per channel
      for (int ch = et; ch < P.stat_channels; ch += 256) {
        const double a = stat_acc[ch * 2], b2 = stat_acc[ch * 2 + 1];
        if (a != 0.0 || b2 != 0.0) {
          atomicAdd(&P.stats[ch], a);
          if (P.want_stats == 1) atomicAdd(&P.stats[P.stat_channels + ch], b2);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (CG == 2) cluster_sync();   // the leader's MMAs read the peer's shared memory: nobody leaves early
  if (warp == 1) tmem_dealloc<CG>(tmem_base, C::TMEM_COLS);
}

// ------------------------------------------------------------------------------------
// CHANNEL-MAJOR kernel ("transposed" GEMM) for layers with 128 output channels: the c = 128 dgrad below, and the thin
// image-layer fprop Conv2d(3,128) (celebA/EAD-GAN_celebA.py:110; one 64-wide k block per tile, purely epilogue- /
// HBM-bound: the per-lane-scalar epilogue below needs a third of the instructions of the pixel-major one).
// TRANSPOSED dgrad for layers with 128 output channels per parity (ConvTranspose2d(256,128) forward / Conv2d(128,256)
// input gradient: the dominant kernel of the CelebA step, celebA/EAD-GAN_celebA.py:86,113).
//
// With N = c = 128 the pixel-major formulation is stuck with 128-wide UMMAs, whose operand reads alone need the full
// 128 B/clk of shared-memory bandwidth, on top of the TMA writes of the same data (ncu r02a: 45 % tensor-pipe, the
// pipeline waits on shared memory, not on L2 or DRAM).  Here the SAME staged tiles are multiplied the other way round:
//     D^T[channel][pixel] = Wd[128 channels][K] . X[256 pixels][K]^T        (M = 128, N = 256, K = 4 k per parity)
// i.e. the packed weight tile is the A operand and the two 128-pixel tiles are ONE 256-row B operand: half as many,
// twice as wide UMMAs (96 instead of 128 B/clk of operand reads), nothing else changes up to the accumulator.
// In tensor memory a lane is now an output CHANNEL and a column a pixel, which makes the epilogue simpler: bias and
// BatchNorm statistics are per-lane scalars (plain register accumulation, no cross-lane reduction), and for a given
// pixel the 32 lanes of a warp hold 32 consecutive channels = one 64-byte run of the NHWC tensors, so the fused
// activation-backward mask is read, and the result written, as full 32-byte sectors.
// ------------------------------------------------------------------------------------
struct DgTCfg {
  static constexpr int STAGE_BYTES = 3 * A_BYTES;                 // two pixel tiles + one weight tile, 48 KB
  static constexpr int STAGES = 4;
  static constexpr int EW = 16;                                   // epilogue warps
  static constexpr int CH = 16;                                   // pixels per epilogue chunk
  static constexpr int STG_BYTES = CH * 64;                       // per warp: [CH pixels][32 channels] bf16
  static constexpr int STAT_BYTES = (EW / 4) * 128 * 2 * 4;       // [column group][channel][sum, sum of squares] fp32
  static constexpr int SMEM = STAGES * STAGE_BYTES + 1024 + 256 + EW * STG_BYTES + STAT_BYTES;
};

// 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// SPEC fixes the epilogue's mode switches at compile time for the three shapes the training step launches (the
// epilogue is bound by its instruction stream: ncu r02y, 414 instructions per 32x32 chunk of which 160 are the
// arithmetic and the stores): 0 = generic (every switch read from P), 1 = bias + (Leaky)ReLU (the thin fprop),
// 2 = fused (Leaky)ReLU-backward mask, 3 = BatchNorm statistics; ReLU is LeakyReLU with slope 0 (set by the launcher).
// Epilogue warp (quad, group) owns channels quad*32.. and 256 / (EW/4) pixel columns.
template <int SPEC>
__global__ void __launch_bounds__(64 + DgTCfg::EW * 32, 1)
tc_dgradT_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, const TcParams P) {
  using C = DgTCfg;
  constexpr int EW = C::EW;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tmem_full_bar = empty_bar + C::STAGES;   // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;      // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // tile = (pixel-tile pair * parities + parity) * n_tiles + channel block; P.m_tiles counts PAIRS of 128-pixel tiles
  const int total_tiles = P.parities * P.m_tiles * P.n_tiles;

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&map_x); tma_prefetch_desc(&map_w); }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
      for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full_bar[b], 1); mbar_init(&tmem_empty_bar[b], EW); }
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_ptr, 512);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int n_tile = tile % P.n_tiles, r = tile / P.n_tiles;
        const int parity = r % P.parities, m_pair = r / P.parities;
        const int py = parity >> 1, px = parity & 1;
        int b0[2], y0[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int m_tile = m_pair * 2 + h;
          b0[h] = (m_tile / P.tiles_y) * P.Tb; y0[h] = (m_tile % P.tiles_y) * P.Th;
        }
        const int w_row = parity * P.N_total + n_tile * 128;
        int qi = 0, t = 0;
#pragma unroll 1
        for (int kb = 0; kb < P.nkb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sx = smem + stage * C::STAGE_BYTES;
          const uint32_t fb = smem_u32(&full_bar[stage]);
          mbar_expect_tx(&full_bar[stage], C::STAGE_BYTES);
          if (P.thin) {   // thin fprop: the whole 4x4x(4) patch of an output pixel is ONE 64-element box row (K = 64)
#pragma unroll
            for (int h = 0; h < 2; ++h) tma_load_4d<1>(sx + h * A_BYTES, &map_x, fb, 0, 0, y0[h], b0[h]);
            tma_load_2d<1>(sx + 2 * A_BYTES, &map_w, fb, 0, n_tile * 128);
            if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
            continue;
          }
          const int ty = t >> 1, tx = t & 1;
          const int dy = py == 0 ? (ty == 0 ? 0 : -1) : (ty == 0 ? 1 : 0);
          const int dx = px == 0 ? (tx == 0 ? 0 : -1) : (tx == 0 ? 1 : 0);
#pragma unroll
          for (int h = 0; h < 2; ++h)
            tma_load_4d<1>(sx + h * A_BYTES, &map_x, fb, qi * BLOCK_K, 1 + dx, y0[h] + 1 + dy, b0[h]);
          tma_load_2d<1>(sx + 2 * A_BYTES, &map_w, fb, t * P.K_ch + qi * BLOCK_K, w_row);
          if (++qi == P.qblocks) { qi = 0; ++t; }
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc(128, 256, 0, 0);
    int stage = 0; uint32_t phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      mbar_wait(&tmem_empty_bar[buf], ((it >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(buf * 256);
      for (int kb = 0; kb < P.nkb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sx = smem_u32(smem + stage * C::STAGE_BYTES);
          const uint32_t sw = sx + 2 * A_BYTES;
#pragma unroll
          for (int k = 0; k < BLOCK_K / 16; ++k)   // A = weights (128 channel rows), B = pixels (256 rows, two tiles back to back)
            umma_bf16(d_tmem, make_desc(sw + k * 32, 16, 1024), make_desc(sx + k * 32, 16, 1024), idesc,
                      (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit(&empty_bar[stage]);
          if (kb == P.nkb - 1) umma_commit(&tmem_full_bar[buf]);
        }
        __syncwarp();
        if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ===== epilogue: lane = output channel, column = pixel.  Warp (quad, grp): channels quad*32.., columns grp*GCOLS.. =====
    // Global traffic goes through a per-warp staging tile [CH pixels][32 channels] bf16: the fused mask is read, and
    // the result written, with 16-byte accesses (lane -> pixel lane/4 + 8 i, channel octet lane%4: every instruction
    // covers eight 64-byte runs), while the per-channel view (lane = channel) uses 2-byte shared-memory accesses.
    constexpr int GROUPS = EW / 4, GCOLS = 256 / GROUPS, CH = C::CH, NI = CH / 8;
    const int act = SPEC == 0 ? P.act : (SPEC == 1 ? (int)EADGAN_ACT_LRELU : 0);
    const int mask_mode = SPEC == 0 ? P.mask_mode : (SPEC == 2 ? (int)EADGAN_ACT_LRELU : 0);
    const int want_stats = SPEC == 0 ? P.want_stats : (SPEC == 3 ? 1 : 0);
    // dgrad writes every second pixel of the big map (one parity), fprop all of them
    const int up = P.mode == MODE_DGRAD ? 2 : 1;
    const int quad = warp & 3, grp = (warp - 2) >> 2;
    const int h = (grp * GCOLS) >> 7, cbase = (grp * GCOLS) & 127;   // pixel-tile half and first column inside it
    const float inv_sigma = P.sigma ? 1.f / __ldg(P.sigma) : 1.f;
    const int lTw = 31 - __clz(P.Tw), lTh = 31 - __clz(P.Th);
    const int row_stride = (P.OW + 2) * P.N_total, img_stride = (P.OH + 2) * row_stride;   // elements, < 2^31
    __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(P.out);
    uint8_t* stg = smem + C::STAGES * C::STAGE_BYTES + 256 + (warp - 2) * C::STG_BYTES;
    float* stat_s = reinterpret_cast<float*>(smem + C::STAGES * C::STAGE_BYTES + 256 + EW * C::STG_BYTES);   // [grp][128][2]
    const int et = threadIdx.x - 64;
    float s1 = 0.f, s2 = 0.f;      // running per-channel statistics of this lane's channel (fp32 per CTA, fp64 across)
    int cur_blk = -1;
    auto flush = [&]() {           // all epilogue warps: fold the column groups, one fp64 atomic per channel
      stat_s[(grp * 128 + quad * 32 + lane) * 2 + 0] = s1;
      stat_s[(grp * 128 + quad * 32 + lane) * 2 + 1] = s2;
      asm volatile("bar.sync 1, %0;" ::"n"(EW * 32) : "memory");
      if (et < 128 && cur_blk >= 0) {
        const int gch = cur_blk * 128 + et;
        if (gch < P.stat_channels) {
          double a1 = 0.0, a2 = 0.0;
#pragma unroll
          for (int g = 0; g < GROUPS; ++g) { a1 += (double)stat_s[(g * 128 + et) * 2]; a2 += (double)stat_s[(g * 128 + et) * 2 + 1]; }
          atomicAdd(&P.stats[gch], a1);
          if (want_stats == 1) atomicAdd(&P.stats[P.stat_channels + gch], a2);
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(EW * 32) : "memory");
      s1 = 0.f; s2 = 0.f;
    };
    const int pl = lane >> 2, oct = lane & 3;          // 16-byte view: pixel pl + 8 i of the chunk, channel octet oct
    uint8_t* stg16 = stg + pl * 64 + oct * 16;         // ... its slot in the staging tile (+ 512 i)
    uint8_t* stg2 = stg + lane * 2;                    // channel view: pixel j of the chunk at + 64 j
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int n_tile = tile % P.n_tiles, r = tile / P.n_tiles;
      const int parity = r % P.parities, m_tile = (r / P.parities) * 2 + h;
      const int py = parity >> 1, px = parity & 1;
      const int b0 = (m_tile / P.tiles_y) * P.Tb, y0 = (m_tile % P.tiles_y) * P.Th;
      if (want_stats && n_tile != cur_blk) {           // tile -> channel block is the same for every warp of the CTA
        if (cur_blk >= 0) flush();
        cur_blk = n_tile;
      }
      const int ch = n_tile * 128 + quad * 32 + lane;
      const float bias = P.bias ? __ldg(&P.bias[ch]) : 0.f;
      // columns are ordered (image, row, x): the valid ones (image < n) are a prefix
      int nvalid = (P.n - b0) << (lTw + lTh);
      nvalid = nvalid < 0 ? 0 : (nvalid > 128 ? 128 : nvalid);
      // element offset of (first pixel of the tile, this lane's channel octet); pixels of the tile are 32-bit offsets from it
      const int64_t tbase = (int64_t)b0 * img_stride + (int64_t)(up * y0 + py + 1) * row_stride +
                            (int64_t)((px + 1) * P.N_total + n_tile * 128 + quad * 32 + oct * 8);
      __nv_bfloat16* out_t = out + tbase;
      const __nv_bfloat16* mask_t = P.mask + tbase;
      auto rel = [&](int col) -> int {
        const int xl = col & (P.Tw - 1), yl = (col >> lTw) & (P.Th - 1), bl = col >> (lTw + lTh);
        return bl * img_stride + up * (yl * row_stride + xl * P.N_total);
      };
      // the fused mask is software-pipelined one chunk ahead: its loads are in flight while the accumulator of the
      // current chunk is read and processed (the first chunk's while this warp still waits for the MMAs)
      uint4 mreg[NI];
      auto load_mask = [&](int cn) {
#pragma unroll
        for (int i = 0; i < NI; ++i) {
          mreg[i] = make_uint4(0u, 0u, 0u, 0u);
          if (cn + pl + 8 * i < nvalid) mreg[i] = __ldg(reinterpret_cast<const uint4*>(mask_t + rel(cn + pl + 8 * i)));
        }
      };
      if (mask_mode) load_mask(cbase);
      const int buf = it & 1;
      mbar_wait(&tmem_full_bar[buf], (it >> 1) & 1);
      tc_fence_after();
      const uint32_t acc = tmem_base + (uint32_t)(buf * 256 + h * 128) + ((uint32_t)(quad * 32) << 16);
#pragma unroll 1
      for (int c0 = cbase; c0 < cbase + GCOLS; c0 += CH) {
        int goff[NI];
#pragma unroll
        for (int i = 0; i < NI; ++i) goff[i] = rel(c0 + pl + 8 * i);
        if (mask_mode) {
#pragma unroll
          for (int i = 0; i < NI; ++i) *reinterpret_cast<uint4*>(stg16 + 512 * i) = mreg[i];
          if (c0 + CH < cbase + GCOLS) load_mask(c0 + CH);
        }
        float v[CH];
        tmem_ld16(acc + (uint32_t)c0, v);
        if (c0 + CH >= cbase + GCOLS) {   // this warp's columns are all in registers: hand the accumulator back
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty_bar[buf]);
        }
        __syncwarp();
        // every mode switch is uniform for the launch: decided ONCE per chunk, outside the element loops
        const bool all_valid = c0 + CH <= nvalid;
#pragma unroll
        for (int j = 0; j < CH; ++j) v[j] = fmaf(v[j], inv_sigma, bias);
        if (want_stats == 1) {
          if (all_valid) {
#pragma unroll
            for (int j = 0; j < CH; ++j) { s1 += v[j]; s2 = fmaf(v[j], v[j], s2); }
          } else {
#pragma unroll
            for (int j = 0; j < CH; ++j)
              if (c0 + j < nvalid) { s1 += v[j]; s2 = fmaf(v[j], v[j], s2); }
          }
        }
        if (act == EADGAN_ACT_RELU || act == EADGAN_ACT_LRELU) {
          const float sl = act == EADGAN_ACT_RELU ? 0.f : P.slope;
#pragma unroll
          for (int j = 0; j < CH; ++j) v[j] = v[j] > 0.f ? v[j] : v[j] * sl;
        } else if (act == EADGAN_ACT_TANH) {
#pragma unroll
          for (int j = 0; j < CH; ++j) v[j] = tanhf(v[j]);
        } else if (act == EADGAN_ACT_SIGMOID) {
#pragma unroll
          for (int j = 0; j < CH; ++j) v[j] = 1.f / (1.f + expf(-v[j]));
        }
        if (mask_mode == EADGAN_ACT_RELU || mask_mode == EADGAN_ACT_LRELU) {
          const float sl = mask_mode == EADGAN_ACT_RELU ? 0.f : P.slope;
#pragma unroll
          for (int j = 0; j < CH; ++j) {   // saved OUTPUT y > 0 <=> pre-activation > 0: sign / zero test on the raw bf16 bits
            const uint32_t mb = *reinterpret_cast<const uint16_t*>(stg2 + j * 64);
            if ((mb & 0x8000u) != 0 || (mb & 0x7fffu) == 0) v[j] *= sl;
          }
        } else if (mask_mode) {
#pragma unroll
          for (int j = 0; j < CH; ++j) {
            const float m = __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(stg2 + j * 64));
            v[j] *= eg_act_grad(m, mask_mode, P.slope);
          }
        }
        if (want_stats == 2) {
          if (all_valid) {
#pragma unroll
            for (int j = 0; j < CH; ++j) s1 += v[j];
          } else {
#pragma unroll
            for (int j = 0; j < CH; ++j)
              if (c0 + j < nvalid) s1 += v[j];
          }
        }
        if (mask_mode) __syncwarp();   // every lane has read its mask column: the staging tile can take the result
#pragma unroll
        for (int j = 0; j < CH; ++j)
          *reinterpret_cast<__nv_bfloat16*>(stg2 + j * 64) = __float2bfloat16_rn(v[j]);
        __syncwarp();
        if (all_valid) {
#pragma unroll
          for (int i = 0; i < NI; ++i)
            *reinterpret_cast<uint4*>(out_t + goff[i]) = *reinterpret_cast<const uint4*>(stg16 + 512 * i);
        } else {
#pragma unroll
          for (int i = 0; i < NI; ++i)
            if (c0 + pl + 8 * i < nvalid)
              *reinterpret_cast<uint4*>(out_t + goff[i]) = *reinterpret_cast<const uint4*>(stg16 + 512 * i);
        }
        __syncwarp();           // ... before the next chunk overwrites the tile
      }
    }
    if (want_stats) flush();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------
// wgrad kernel: acc[ko][kk] = sum_pixels dy[pix][ko] * patch[pix][kk]
// ------------------------------------------------------------------------------------
struct WgParams {
  int n, p, q;
  int Tw, Th, Tb;       // 64 pixels per stage
  int tiles_y;          // p / Th
  int k, c;             // small-map / big-map channels
  int qblocks;          // 2c/64
  int steps_total;      // number of 64-pixel steps
  int steps_per_split;
  int Ktot;             // 16*c
  float* partial;       // [splits][k][16c]
  int dense;            // 1: "pixels" are batch rows; A boxes from a [n][Mp] matrix, B boxes from [n,6,6,C]
  int thin;             // 1: big map is a <= 4-channel image; B = one 64-wide patch box of the row-expanded buffer
  int kk_tiles, ko_tiles, splits;   // persistent item space (filled by launch_wgrad from the logical grid)
};

// BLOCK_N columns of kk per tile (multiple of 64).  CG = 2: a CTA pair computes 256 ko rows x BLOCK_N columns; each
// CTA stages the dy box of ITS 128 ko rows and HALF of the patch columns (32 KB per stage instead of 48).
template <int BLOCK_N, int CG>
struct WgCfg {
  static constexpr int A_B = 2 * 64 * 128;               // two 64-channel boxes x 64 pixels
  static constexpr int NB = BLOCK_N / 64 / CG;           // 64-column patch boxes this CTA stages
  static constexpr int B_B = NB * 64 * 128;
  static constexpr int STAGE_BYTES = A_B + B_B;
  static constexpr int STAGES = CG == 2 ? 6 : (BLOCK_N >= 256 ? 4 : 6);
  static constexpr int SMEM = STAGES * STAGE_BYTES + 1024 + 256;
  static_assert(SMEM <= 227 * 1024, "wgrad ring exceeds shared memory");
};

template <int BLOCK_N, int CG>
__global__ void __launch_bounds__(192, 1)
tc_wgrad_kernel(const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_x,
                const WgParams P) {
  // PERSISTENT: work items are (split, ko tile, kk tile) triples, kk fastest; CTA c runs items c, c + grid, ...
  // Two TMEM accumulators: the epilogue of item i (128 x BLOCK_N fp32 partial -> global) overlaps the
  // mainloop of item i + 1, and barrier / TMEM / tensor-map set-up is paid once per CTA instead of per item.
  using C = WgCfg<BLOCK_N, CG>;
  extern __shared__ uint8_t smem_raw[];
  // align by OFFSETTING the shared array (not by integer round trip): the compiler keeps the shared address
  // space, so every access below is LDS/STS instead of a generic LD/ST through the L1TEX path
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tmem_full_bar = empty_bar + C::STAGES;   // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;      // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles = P.kk_tiles * P.ko_tiles;
  const int total_items = tiles * P.splits;
  // cta_group::2: both CTAs of a pair walk the same item list; rank 0 leads (see tc_conv_kernel)
  const int rank = CG == 2 ? (int)cluster_ctarank() : 0;
  const int first_item = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int item_step = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&map_dy); tma_prefetch_desc(&map_x); }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
      for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full_bar[b], 1); mbar_init(&tmem_empty_bar[b], 4 * CG); }
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc<CG>(tmem_ptr, 2 * BLOCK_N);
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CG == 2) cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int item = first_item; item < total_items; item += item_step) {
        const int kk_tile = item % P.kk_tiles, ko_tile = (item / P.kk_tiles) % P.ko_tiles, split = item / tiles;
        const int ko0 = (ko_tile * CG + rank) * 128;                 // this CTA's 128 dy channels
        const int nb0 = (kk_tile * CG + rank) * C::NB;               // ... and its first 64-column patch block
        const int step0 = split * P.steps_per_split;
        const int step1 = min(P.steps_total, step0 + P.steps_per_split);
        // per-item constants (no integer division inside the step loop: this one thread issues every load of the CTA)
        int qis[C::NB], taps[C::NB];
#pragma unroll
        for (int i = 0; i < C::NB; ++i) { qis[i] = ((nb0 + i) % P.qblocks) * 64; taps[i] = (nb0 + i) / P.qblocks; }
        int ty_i = P.dense ? 0 : step0 % P.tiles_y, tb_i = P.dense ? 0 : step0 / P.tiles_y;
#pragma unroll 1
        for (int st = step0; st < step1; ++st) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * C::STAGE_BYTES;
          uint8_t* sb = sa + C::A_B;
          uint32_t fb = smem_u32(&full_bar[stage]);
          if constexpr (CG == 2) {
            fb = mapa(fb, 0);
            if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * C::STAGE_BYTES);
          } else {
            mbar_expect_tx(&full_bar[stage], C::STAGE_BYTES);
          }
          if (P.dense) {
#pragma unroll
            for (int h = 0; h < 2; ++h)
              tma_load_2d<CG>(sa + h * 8192, &map_dy, fb, ko0 + h * 64, st * 64);
#pragma unroll
            for (int i = 0; i < C::NB; ++i)   // tap = ky*4+kx
              tma_load_4d<CG>(sb + i * 8192, &map_x, fb, qis[i], 1 + (taps[i] & 3), 1 + (taps[i] >> 2), st * 64);
          } else {
            const int b0 = tb_i * P.Tb;
            const int y0 = ty_i * P.Th;
            if (++ty_i == P.tiles_y) { ty_i = 0; ++tb_i; }
#pragma unroll
            for (int h = 0; h < 2; ++h)
              tma_load_4d<CG>(sa + h * 8192, &map_dy, fb, ko0 + h * 64, 1, y0 + 1, b0);
            if (P.thin) {
              tma_load_4d<CG>(sb, &map_x, fb, 0, 0, y0, b0);
            } else {
#pragma unroll
              for (int i = 0; i < C::NB; ++i) {
                const int t = taps[i];
                tma_load_5d<CG>(sb + i * 8192, &map_x, fb, qis[i], (t >> 1) & 1, t & 1, y0 + (t >> 2), b0);
              }
            }
          }
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc(128 * CG, BLOCK_N, 1, 1);  // both operands MN-major
    int stage = 0; uint32_t phase = 0;
    int use = 0;   // accumulator uses so far (items with at least one step)
    for (int item = first_item; item < total_items && rank == 0; item += item_step) {
      const int split = item / tiles;
      const int step0 = split * P.steps_per_split;
      const int nsteps = min(P.steps_total, step0 + P.steps_per_split) - step0;
      if (nsteps <= 0) continue;
      const int buf = use & 1;
      mbar_wait(&tmem_empty_bar[buf], ((use >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BLOCK_N);
      for (int it = 0; it < nsteps; ++it) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + stage * C::STAGE_BYTES);
          const uint32_t sb = sa + C::A_B;
#pragma unroll
          for (int k = 0; k < 4; ++k) {  // 16 pixel rows per MMA
            const uint64_t da = make_desc(sa + k * 2048, 8192, 1024);
            const uint64_t db = make_desc(sb + k * 2048, 8192, 1024);
            umma_bf16<CG>(d_tmem, da, db, idesc, (it > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit<CG>(&empty_bar[stage]);
          if (it == nsteps - 1) umma_commit<CG>(&tmem_full_bar[buf]);
        }
        __syncwarp();
        if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
      }
      ++use;
    }
  } else {
    const int quad = warp & 3;
    uint32_t te_bar[2] = {smem_u32(&tmem_empty_bar[0]), smem_u32(&tmem_empty_bar[1])};
    if constexpr (CG == 2) { te_bar[0] = mapa(te_bar[0], 0); te_bar[1] = mapa(te_bar[1], 0); }
    int use = 0;
    for (int item = first_item; item < total_items; item += item_step) {
      const int kk_tile = item % P.kk_tiles, ko_tile = (item / P.kk_tiles) % P.ko_tiles, split = item / tiles;
      const int step0 = split * P.steps_per_split;
      const int nsteps = min(P.steps_total, step0 + P.steps_per_split) - step0;
      const int ko = (ko_tile * CG + rank) * 128 + quad * 32 + lane;
      const int buf = use & 1;
      if (nsteps > 0) {
        mbar_wait(&tmem_full_bar[buf], (use >> 1) & 1);
        tc_fence_after();
      }
      float* dst = P.partial + ((int64_t)split * P.k + ko) * P.Ktot + (int64_t)kk_tile * BLOCK_N;
#pragma unroll 1
      for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
        float v[32];
        if (nsteps > 0) {
          tmem_ld32(tmem_base + (uint32_t)(buf * BLOCK_N) + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, v);
          if (c0 + 32 >= BLOCK_N) {   // every column of this warp's rows is in registers: release the accumulator
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if constexpr (CG == 2) mbar_arrive_cluster(te_bar[buf]);
              else mbar_arrive(&tmem_empty_bar[buf]);
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0.f;
        }
        if (ko < P.k) {
#pragma unroll
          for (int g = 0; g < 8; ++g)
            *reinterpret_cast<float4*>(dst + c0 + g * 4) = make_float4(v[g * 4], v[g * 4 + 1], v[g * 4 + 2], v[g * 4 + 3]);
        }
      }
      if (nsteps > 0) ++use;
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CG == 2) cluster_sync();
  if (warp == 1) tmem_dealloc<CG>(tmem_base, 2 * BLOCK_N);
}

// sum split partials and permute GEMM column order (a,b,dy,dx,c) -> dw[ko][c][ky][kx]
// block = (ko, 64-channel group); coalesced reads of 16 x 64-float runs, one 4 KB write
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ partial, int splits, int k, int c,
                                                           int c_real, float* __restrict__ dw) {
  __shared__ float tile[16][65];
  const int ko = blockIdx.y, c0 = blockIdx.x * 64;
  const int Ktot = 16 * c;
  {   // one float4 (4 channels of one tap) per thread, the split loop unrolled: 4 x 16 B in flight per thread
    const int tap = threadIdx.x >> 4, cl = (threadIdx.x & 15) * 4;  // tap = ((a*2+b)*2+dy)*2+dx
    if (c0 + cl < c) {                                              // c is a multiple of 32: whole float4s
      const int t3 = tap >> 1, dx = tap & 1;
      const int64_t col = (int64_t)t3 * 2 * c + (int64_t)dx * c + c0 + cl;
      const float4* src = reinterpret_cast<const float4*>(partial + (int64_t)ko * Ktot + col);
      const int64_t sp_stride = (int64_t)k * Ktot / 4;
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
      for (int sp = 0; sp < splits; ++sp) {
        const float4 v = __ldg(src + sp * sp_stride);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      }
      const int dy = t3 & 1, bt = (t3 >> 1) & 1, at = t3 >> 2;
      const int ky = 2 * at + dy, kx = 2 * bt + dx;
      float* trow = tile[ky * 4 + kx];
      trow[cl] = s.x; trow[cl + 1] = s.y; trow[cl + 2] = s.z; trow[cl + 3] = s.w;
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 64 * 16; e += 256) {
    const int cl = e / 16, tp = e % 16;
    if (c0 + cl < c_real) dw[((int64_t)ko * c_real + c0 + cl) * 16 + tp] = tile[tp][cl];
  }
}

// dense layers: partial[m][tap*C + ch] (tap = ky*4+kx) -> dw[m][ch][ky][kx]
__global__ void __launch_bounds__(256) dense_wgrad_reduce_kernel(const float* __restrict__ partial, int m_pad, int C,
                                                                 float* __restrict__ dw) {
  __shared__ float tile[16][65];
  const int m = blockIdx.y, c0 = blockIdx.x * 64;
  for (int e = threadIdx.x; e < 16 * 64; e += 256) {
    const int tap = e / 64, cl = e % 64;
    tile[tap][cl] = partial[(int64_t)m * 16 * C + (int64_t)tap * C + c0 + cl];
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 64 * 16; e += 256) {
    const int cl = e / 16, tp = e % 16;
    dw[((int64_t)m * C + c0 + cl) * 16 + tp] = tile[tp][cl];
  }
}

// dense weight packs from w[m][ch][tap] (m_real x C x 16, fp32):
//   rows_major = 1:  out[m][tap*C + ch]   (m padded to m_pad rows)      -- B operand of the gather GEMM
//   rows_major = 0:  out[tap*C + ch][m]   (m padded to m_pad columns)   -- B operand of the scatter GEMM
__global__ void dense_pack_kernel(const float* __restrict__ w, int m_real, int m_pad, int C, int rows_major,
                                  __nv_bfloat16* __restrict__ out) {
  const int64_t total = (int64_t)m_pad * 16 * C;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int m, tap, ch;
    if (rows_major) {
      m = (int)(i / (16 * C));
      const int r = (int)(i - (int64_t)m * 16 * C);
      tap = r / C; ch = r - tap * C;
    } else {
      const int64_t r = i / m_pad;
      m = (int)(i - r * m_pad);
      tap = (int)(r / C); ch = (int)(r - (int64_t)tap * C);
    }
    out[i] = __float2bfloat16_rn(m < m_real ? w[((int64_t)m * C + ch) * 16 + tap] : 0.f);
  }
}

// ------------------------------------------------------------------------------------
// weight packing
// ------------------------------------------------------------------------------------
// Wf[ko][((a*2+b)*2+dy)*2c + dx*c + ci] = w[ko][ci][2a+dy][2b+dx] / sigma, i.e. per ko a [c][16] -> [16][c]
// transpose with a tap permutation.  Block = (64-channel chunk, ko): coalesced 4 KB read, sixteen 128-byte writes.
__global__ void __launch_bounds__(256) pack_w_fprop_kernel(const float* __restrict__ w, const float* __restrict__ sigma,
                                                           int k, int c_real, int c, __nv_bfloat16* __restrict__ out) {
  __shared__ float tile[64][17];
  const float inv = sigma ? 1.f / *sigma : 1.f;
  const int ko = blockIdx.y, c0 = blockIdx.x * 64;
  for (int e = threadIdx.x; e < 64 * 16; e += 256) {
    const int cl = e >> 4, tp = e & 15;   // tp = ky*4 + kx
    tile[cl][tp] = (c0 + cl < c_real) ? w[((int64_t)ko * c_real + c0 + cl) * 16 + tp] * inv : 0.f;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 16 * 64; e += 256) {
    const int tap = e >> 6, cl = e & 63;  // tap = ((a*2+b)*2+dy)*2+dx
    if (c0 + cl < c) {
      const int dx = tap & 1, dy = (tap >> 1) & 1, bt = (tap >> 2) & 1, at = tap >> 3;
      out[(int64_t)ko * 16 * c + (int64_t)tap * c + c0 + cl] = __float2bfloat16_rn(tile[cl][(2 * at + dy) * 4 + 2 * bt + dx]);
    }
  }
}
// Wd[(py*2+px)*c + co][(ty*2+tx)*k + ki] = w[ki][co][ky(py,ty)][kx(px,tx)] / sigma.  Block = (64 ki, 8 co): reads
// 512-byte runs (8 co x 16 taps of one ki), writes 128-byte runs (64 ki of one (parity, co, tap)).
__global__ void __launch_bounds__(256) pack_w_dgrad_kernel(const float* __restrict__ w, const float* __restrict__ sigma,
                                                           int k, int c_real, int c, __nv_bfloat16* __restrict__ out) {
  __shared__ float tile[64][129];
  const float inv = sigma ? 1.f / *sigma : 1.f;
  const int ki0 = blockIdx.x * 64, co0 = blockIdx.y * 8;
  for (int e = threadIdx.x; e < 64 * 128; e += 256) {
    const int kl = e >> 7, r = e & 127;   // r = co_local*16 + ky*4 + kx
    const int co = co0 + (r >> 4);
    tile[kl][r] = (ki0 + kl < k && co < c_real) ? w[((int64_t)(ki0 + kl) * c_real + co) * 16 + (r & 15)] * inv : 0.f;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 128 * 64; e += 256) {
    const int combo = e >> 6, kl = e & 63;     // combo = (co_local*4 + par)*4 + t
    const int t = combo & 3, par = (combo >> 2) & 3, col = combo >> 4;
    const int co = co0 + col;
    if (co < c && ki0 + kl < k) {
      const int py = par >> 1, px = par & 1, ty = t >> 1, tx = t & 1;
      const int ky = py == 0 ? (ty == 0 ? 1 : 3) : (ty == 0 ? 0 : 2);
      const int kx = px == 0 ? (tx == 0 ? 1 : 3) : (tx == 0 ? 0 : 2);
      out[((int64_t)par * c + co) * 4 * k + (int64_t)t * k + ki0 + kl] = __float2bfloat16_rn(tile[kl][col * 16 + ky * 4 + kx]);
    }
  }
}

// ------------------------------------------------------------------------------------
// host: tensor maps
// ------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

int encode_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
               const uint32_t* box) {
  EncodeTiledFn enc = get_encode();
  EG_REQUIRE(enc != nullptr, EADGAN_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t gd[5], gs[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  EG_REQUIRE(r == CUDA_SUCCESS, EADGAN_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rank %d)", (int)r,
             rank);
  return 0;
}

// 5-D space-to-depth view of the big padded map [n][h+2][w+2][c]
int map_big_s2d(CUtensorMap* m, const void* base, int n, int c, int h, int w, int Tw, int Th, int Tb) {
  const uint64_t dims[5] = {(uint64_t)2 * c, (uint64_t)(w + 2) / 2, 2, (uint64_t)(h + 2) / 2, (uint64_t)n};
  const uint64_t st[4] = {(uint64_t)2 * c * 2, (uint64_t)(w + 2) * c * 2, (uint64_t)2 * (w + 2) * c * 2,
                          (uint64_t)(h + 2) * (w + 2) * c * 2};
  const uint32_t box[5] = {64, (uint32_t)Tw, 1, (uint32_t)Th, (uint32_t)Tb};
  return encode_map(m, base, 5, dims, st, box);
}
// 4-D view of the small padded map [n][p+2][q+2][k]
int map_small(CUtensorMap* m, const void* base, int n, int k, int p, int q, int Tw, int Th, int Tb) {
  const uint64_t dims[4] = {(uint64_t)k, (uint64_t)(q + 2), (uint64_t)(p + 2), (uint64_t)n};
  const uint64_t st[3] = {(uint64_t)k * 2, (uint64_t)(q + 2) * k * 2, (uint64_t)(p + 2) * (q + 2) * k * 2};
  const uint32_t box[4] = {64, (uint32_t)Tw, (uint32_t)Th, (uint32_t)Tb};
  return encode_map(m, base, 4, dims, st, box);
}
int map_matrix(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  const uint64_t dims[2] = {cols, rows};
  const uint64_t st[1] = {cols * 2};
  const uint32_t box[2] = {64, box_rows};
  return encode_map(m, base, 2, dims, st, box);
}


// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies PER DEVICE: remember which devices have been opted in
// (bit d of an atomic mask; devices >= 64 simply set the attribute on every launch).  Safe from any thread
// (backward runs on autograd's per-device worker threads).
template <typename K>
int opt_in_smem(K kernel, int bytes, std::atomic<uint64_t>& done) {
  int dev = 0;
  EG_CUDA(cudaGetDevice(&dev));
  const uint64_t bit = dev < 64 ? (1ull << dev) : 0ull;
  if (bit && (done.load(std::memory_order_acquire) & bit)) return 0;
  EG_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  if (bit) done.fetch_or(bit, std::memory_order_release);
  return 0;
}

template <int SPEC>
int launch_channel_major_t(const CUtensorMap& mx, const CUtensorMap& mw, const TcParams& P, cudaStream_t st) {
  static std::atomic<uint64_t> opted{0};
  if (int e = opt_in_smem(tc_dgradT_kernel<SPEC>, DgTCfg::SMEM, opted)) return e;
  const int total = P.parities * P.m_tiles * P.n_tiles;
  const int units = eg_sm_count();
  const int waves = (total + units - 1) / units;
  const int grid = (total + waves - 1) / waves;
  tc_dgradT_kernel<SPEC><<<grid, 64 + DgTCfg::EW * 32, DgTCfg::SMEM, st>>>(mx, mw, P);
  EG_LAUNCH_CHECK("tc_dgradT_kernel");
  return 0;
}

int launch_channel_major(const CUtensorMap& mx, const CUtensorMap& mw, TcParams P, cudaStream_t st) {
  // the three epilogue shapes of the training step get a specialised instance (see tc_dgradT_kernel)
  const bool act_lrelu = P.act == EADGAN_ACT_RELU || P.act == EADGAN_ACT_LRELU;
  const bool mask_lrelu = P.mask_mode == EADGAN_ACT_RELU || P.mask_mode == EADGAN_ACT_LRELU;
  int spec = 0;
  if (act_lrelu && !P.mask_mode && !P.want_stats) {
    spec = 1;
    if (P.act == EADGAN_ACT_RELU) { P.act = EADGAN_ACT_LRELU; P.slope = 0.f; }
  } else if (mask_lrelu && !P.want_stats && !P.act) {
    spec = 2;
    if (P.mask_mode == EADGAN_ACT_RELU) { P.mask_mode = EADGAN_ACT_LRELU; P.slope = 0.f; }
  } else if (!P.mask_mode && P.want_stats == 1 && !P.act) {
    spec = 3;
  }
  switch (spec) {
    case 1: return launch_channel_major_t<1>(mx, mw, P, st);
    case 2: return launch_channel_major_t<2>(mx, mw, P, st);
    case 3: return launch_channel_major_t<3>(mx, mw, P, st);
  }
  return launch_channel_major_t<0>(mx, mw, P, st);
}

bool pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

// tile of `pixels` positions of a p x q grid: Tw = q, Th rows, Tb images
int pick_tile(int p, int q, int pixels, int* Tw, int* Th, int* Tb) {
  if (!pow2(q) || !pow2(p) || q > pixels) return -1;
  *Tw = q;
  int th = pixels / q;
  if (th > p) th = p;
  *Th = th;
  *Tb = pixels / (q * th);
  return 0;
}

template <int BN, int MT, int CG>
int launch_conv(const CUtensorMap& ma, const CUtensorMap& mb, const TcParams& P, cudaStream_t st) {
  static std::atomic<uint64_t> opted{0};
  if (int e = opt_in_smem(tc_conv_kernel<BN, MT, CG>, Cfg<BN, MT, CG>::SMEM, opted)) return e;
  // persistent grid: every CTA (CTA pair) runs the same number of tiles (+-1), at most one CTA per SM
  const int total = P.parities * P.m_tiles * P.n_tiles;
  const int units = eg_sm_count() / CG;
  const int waves = (total + units - 1) / units;
  const int grid = ((total + waves - 1) / waves) * CG;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(320); cfg.dynamicSmemBytes = Cfg<BN, MT, CG>::SMEM; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = CG == 2 ? 1 : 0;
  EG_CUDA(cudaLaunchKernelEx(&cfg, tc_conv_kernel<BN, MT, CG>, ma, mb, P));
  EG_LAUNCH_CHECK("tc_conv_kernel");
  return 0;
}

// tile configuration of one launch: BLOCK_N, M tiles per CTA, cta_group
struct TileCfg { int bn, mt, cg; };

int pick_bn_tiles(int nch, int m_tiles_x_par);

// cg = 2 (CTA pairs, see Cfg) for the layers with enough tiles to keep every pair busy for several tiles; the small /
// ragged launches (dSprites 32..64-channel layers, dense and thin GEMMs) stay on the single-CTA path.
TileCfg pick_cfg(int nch, int m_tiles, int parities, bool allow_pair, int force_bn = 0) {
  TileCfg t;
  t.bn = force_bn ? force_bn : pick_bn_tiles(nch, m_tiles * parities);
  if (t.bn <= 0) return t;
  const int sms = eg_sm_count();
  const int64_t tiles = (int64_t)m_tiles * parities * (nch / t.bn);
  t.cg = (allow_pair && t.bn >= 128 && m_tiles >= 2 && tiles >= 2 * sms) ? 2 : 1;
  // test hook: force CTA pairs on (2) / off (1), so that small, ragged shapes exercise the pair protocol
  if (const char* e = getenv("EADGAN_TC_CG")) { if (allow_pair && t.bn >= 128 && (atoi(e) == 1 || atoi(e) == 2)) t.cg = atoi(e); }
  // two 128-row tiles per CTA tile (sharing every B load) when BLOCK_N <= 128 and there is enough work
  t.mt = (t.bn <= 128 && tiles >= 4 * sms * t.cg) ? 2 : 1;
  return t;
}

int dispatch_conv(const TileCfg& t, const CUtensorMap& ma, const CUtensorMap& mb, TcParams& P, int m_tiles, int n_total,
                  int parities, cudaStream_t st) {
  const int bn = t.bn, mt = t.mt, per = t.mt * t.cg;
  P.m_tiles = (m_tiles + per - 1) / per; P.n_tiles = n_total / bn; P.parities = parities;
  if (P.qblocks <= 0) P.qblocks = 1;   // plain GEMMs: the producer's (tap, channel block) counters are unused
  P.bias_len = P.bias ? (P.dense_C > 0 ? P.dense_C : P.n_store) : 0;
  EG_REQUIRE(P.bias_len <= STAT_MAX_CH, EADGAN_ERR_UNSUPPORTED, "tc conv: fused bias supports at most %d channels (got %d)",
             STAT_MAX_CH, P.bias_len);
  EG_REQUIRE(!P.want_stats || (P.stat_channels > 0 && P.stat_channels <= STAT_MAX_CH), EADGAN_ERR_UNSUPPORTED,
             "tc conv: fused statistics support at most %d channels (got %d)", STAT_MAX_CH, P.stat_channels);
  switch ((bn * 10 + mt) * 10 + t.cg) {
    case 3211: return launch_conv<32, 1, 1>(ma, mb, P, st);
    case 3221: return launch_conv<32, 2, 1>(ma, mb, P, st);
    case 6411: return launch_conv<64, 1, 1>(ma, mb, P, st);
    case 6421: return launch_conv<64, 2, 1>(ma, mb, P, st);
    case 12811: return launch_conv<128, 1, 1>(ma, mb, P, st);
    case 12821: return launch_conv<128, 2, 1>(ma, mb, P, st);
    case 25611: return launch_conv<256, 1, 1>(ma, mb, P, st);
    case 12812: return launch_conv<128, 1, 2>(ma, mb, P, st);
    case 12822: return launch_conv<128, 2, 2>(ma, mb, P, st);
    case 25612: return launch_conv<256, 1, 2>(ma, mb, P, st);
  }
  return eadgan_set_error(EADGAN_ERR_UNSUPPORTED, "tc conv: unsupported tile configuration BLOCK_N %d, MT %d, cta_group %d",
                          bn, mt, t.cg);
}

// BLOCK_N: 256 halves the A re-reads and the smem traffic per MAC; keep 128 while the tile count is too
// small to fill the machine twice
int pick_bn_tiles(int nch, int m_tiles_x_par) {
  if (nch % 256 == 0 && (int64_t)m_tiles_x_par * (nch / 256) >= 2 * eg_sm_count()) return 256;
  if (nch % 128 == 0) return 128;
  if (nch % 64 == 0) return 64;
  if (nch % 32 == 0) return 32;
  return -1;
}

int pick_bn(int nch) {
  if (nch % 128 == 0) return 128;
  if (nch % 64 == 0) return 64;
  if (nch % 32 == 0) return 32;
  return -1;
}

int check_tc(const eadgan_tc_desc* d, const char* who) {
  EG_REQUIRE(d != nullptr, EADGAN_ERR_INVALID, "%s: NULL desc", who);
  EG_REQUIRE(d->n > 0 && d->c > 0 && d->k > 0 && d->h >= 2 && d->w >= 2 && (d->h % 2) == 0 && (d->w % 2) == 0,
             EADGAN_ERR_INVALID, "%s: bad extents", who);
  return 0;
}

}  // namespace

extern "C" int eadgan_tc_pack_w_fprop(const float* w, const float* sigma, int k, int c_real, int c, void* w_packed,
                                      void* stream) {
  EG_REQUIRE(w && w_packed && k > 0 && c > 0 && c_real > 0 && c_real <= c, EADGAN_ERR_INVALID,
             "tc_pack_w_fprop: bad arguments");
  pack_w_fprop_kernel<<<dim3((c + 63) / 64, k), 256, 0, (cudaStream_t)stream>>>(w, sigma, k, c_real, c,
                                                                                (__nv_bfloat16*)w_packed);
  EG_LAUNCH_CHECK("pack_w_fprop_kernel");
  return 0;
}

extern "C" int eadgan_tc_pack_w_dgrad(const float* w, const float* sigma, int k, int c_real, int c, void* w_packed,
                                      void* stream) {
  EG_REQUIRE(w && w_packed && k > 0 && c > 0 && c_real > 0 && c_real <= c, EADGAN_ERR_INVALID,
             "tc_pack_w_dgrad: bad arguments");
  pack_w_dgrad_kernel<<<dim3((k + 63) / 64, (c + 7) / 8), 256, 0, (cudaStream_t)stream>>>(w, sigma, k, c_real, c,
                                                                                          (__nv_bfloat16*)w_packed);
  EG_LAUNCH_CHECK("pack_w_dgrad_kernel");
  return 0;
}

extern "C" int eadgan_tc_fprop(const eadgan_tc_desc* d, const void* x_pad, const void* w_packed, const float* bias,
                               void* y, const void* mask, double* stats, const float* sigma, void* stream) {
  if (int e = check_tc(d, "tc_fprop")) return e;
  EG_REQUIRE(x_pad && w_packed && y, EADGAN_ERR_INVALID, "tc_fprop: NULL pointer");
  const int p = d->h / 2, q = d->w / 2;
  EG_REQUIRE((2 * d->c) % 64 == 0, EADGAN_ERR_UNSUPPORTED, "tc_fprop: c=%d must be a multiple of 32", d->c);
  TcParams P{};
  P.mode = MODE_FPROP; P.n = d->n; P.p = p; P.q = q;
  EG_REQUIRE(pick_tile(p, q, 128, &P.Tw, &P.Th, &P.Tb) == 0, EADGAN_ERR_UNSUPPORTED,
             "tc_fprop: output map %dx%d must be a power of two <= 128 wide", p, q);
  const int m_tiles = ((d->n + P.Tb - 1) / P.Tb) * (p / P.Th);
  const TileCfg tcfg = pick_cfg(d->k, m_tiles, 1, true);
  const int bn = tcfg.bn;
  EG_REQUIRE(bn > 0, EADGAN_ERR_UNSUPPORTED, "tc_fprop: k=%d must be a multiple of 32", d->k);
  P.tiles_y = p / P.Th; P.N_total = d->k; P.K_ch = d->c; P.qblocks = 2 * d->c / 64; P.nkb = 8 * P.qblocks;
  P.act = d->act; P.slope = d->slope; P.out_f32_nchw = d->out_f32_nchw; P.want_stats = d->want_stats;
  P.mask_mode = d->mask_mode; P.OH = p; P.OW = q; P.bias = bias; P.out = y;
  P.mask = (const __nv_bfloat16*)mask; P.stats = stats; P.n_store = d->k; P.stat_channels = d->k; P.sigma = sigma;
  EG_REQUIRE(!P.mask_mode || mask, EADGAN_ERR_INVALID, "tc_fprop: mask_mode without mask");
  EG_REQUIRE(!P.want_stats || stats, EADGAN_ERR_INVALID, "tc_fprop: want_stats without stats");
  CUtensorMap ma, mb;
  if (int e = map_big_s2d(&ma, x_pad, d->n, d->c, d->h, d->w, P.Tw, P.Th, P.Tb)) return e;
  if (int e = map_matrix(&mb, w_packed, d->k, (uint64_t)16 * d->c, bn / tcfg.cg)) return e;
  return dispatch_conv(tcfg, ma, mb, P, m_tiles, d->k, 1, (cudaStream_t)stream);
}

extern "C" int eadgan_tc_dgrad(const eadgan_tc_desc* d, const void* dy_pad, const void* w_packed, const float* bias,
                               void* dx, const void* mask, double* stats, const float* sigma, void* stream) {
  if (int e = check_tc(d, "tc_dgrad")) return e;
  EG_REQUIRE(dy_pad && w_packed && dx, EADGAN_ERR_INVALID, "tc_dgrad: NULL pointer");
  const int p = d->h / 2, q = d->w / 2;
  // k = 32: the 64-channel TMA boxes run past the tensor and are zero-filled (half of each k block is idle)
  EG_REQUIRE(d->k % 64 == 0 || d->k == 32, EADGAN_ERR_UNSUPPORTED, "tc_dgrad: k=%d must be 32 or a multiple of 64", d->k);
  TcParams P{};
  P.mode = MODE_DGRAD; P.n = d->n; P.p = p; P.q = q;
  EG_REQUIRE(pick_tile(p, q, 128, &P.Tw, &P.Th, &P.Tb) == 0, EADGAN_ERR_UNSUPPORTED,
             "tc_dgrad: small map %dx%d must be a power of two <= 128 wide", p, q);
  const int m_tiles = ((d->n + P.Tb - 1) / P.Tb) * (p / P.Th);
  const TileCfg tcfg = pick_cfg(d->c, m_tiles, 4, true);
  const int bn = tcfg.bn;
  EG_REQUIRE(bn > 0, EADGAN_ERR_UNSUPPORTED, "tc_dgrad: c=%d must be a multiple of 32", d->c);
  P.tiles_y = p / P.Th; P.N_total = d->c; P.K_ch = d->k; P.qblocks = (d->k + 63) / 64; P.nkb = 4 * P.qblocks;
  P.act = d->act; P.slope = d->slope; P.out_f32_nchw = d->out_f32_nchw; P.want_stats = d->want_stats;
  P.mask_mode = d->mask_mode; P.OH = d->h; P.OW = d->w; P.bias = bias; P.out = dx;
  P.mask = (const __nv_bfloat16*)mask; P.stats = stats; P.sigma = sigma;
  P.n_store = (d->c_real > 0 && d->c_real < d->c) ? d->c_real : d->c;
  P.stat_channels = P.n_store;
  EG_REQUIRE(P.n_store == d->c || d->out_f32_nchw, EADGAN_ERR_UNSUPPORTED,
             "tc_dgrad: zero-padded output channels (c_real < c) need out_f32_nchw");
  EG_REQUIRE(!P.mask_mode || mask, EADGAN_ERR_INVALID, "tc_dgrad: mask_mode without mask");
  EG_REQUIRE(!P.want_stats || stats, EADGAN_ERR_INVALID, "tc_dgrad: want_stats without stats");
  CUtensorMap ma, mb;
  if (int e = map_small(&ma, dy_pad, d->n, d->k, p, q, P.Tw, P.Th, P.Tb)) return e;
  // 128-channel outputs with a long pixel dimension: the transposed kernel (see tc_dgradT_kernel), 128 channels x 256
  // pixels per tile.  It shares P: its conditions k % 64 == 0, c_real == c and no out_f32_nchw are what make
  // qblocks, n_store and out_f32_nchw above right for it too.
  bool transposed = d->c == 128 && d->k % 64 == 0 && !d->out_f32_nchw && (d->c_real <= 0 || d->c_real == d->c);
  bool enough = (int64_t)m_tiles * 4 >= 8 * eg_sm_count();
  // test hook: 0 / 2 = never / always use the transposed kernel where it applies
  if (const char* e = getenv("EADGAN_TC_DGRADT")) { if (atoi(e) == 0) transposed = false; else if (atoi(e) == 2) enough = true; }
  if (transposed && enough) {
    P.m_tiles = (m_tiles + 1) / 2; P.n_tiles = d->c / 128; P.parities = 4;
    if (int e = map_matrix(&mb, w_packed, (uint64_t)4 * d->c, (uint64_t)4 * d->k, 128)) return e;
    return launch_channel_major(ma, mb, P, (cudaStream_t)stream);
  }
  if (int e = map_matrix(&mb, w_packed, (uint64_t)4 * d->c, (uint64_t)4 * d->k, bn / tcfg.cg)) return e;
  return dispatch_conv(tcfg, ma, mb, P, m_tiles, d->c, 4, (cudaStream_t)stream);
}

namespace {
int wgrad_plan(const eadgan_tc_desc* d, WgParams* P, int* bn, int* splits, int* cg) {
  const int p = d->h / 2, q = d->w / 2;
  // dy channel boxes past k are zero-filled by TMA and the matching partial rows are never read
  EG_REQUIRE(d->k % 32 == 0, EADGAN_ERR_UNSUPPORTED, "tc_wgrad: k=%d must be a multiple of 32", d->k);
  EG_REQUIRE((2 * d->c) % 64 == 0, EADGAN_ERR_UNSUPPORTED, "tc_wgrad: c=%d must be a multiple of 32", d->c);
  P->n = d->n; P->p = p; P->q = q; P->k = d->k; P->c = d->c;
  EG_REQUIRE(pick_tile(p, q, 64, &P->Tw, &P->Th, &P->Tb) == 0, EADGAN_ERR_UNSUPPORTED,
             "tc_wgrad: small map %dx%d must be a power of two <= 64 wide", p, q);
  P->tiles_y = p / P->Th;
  P->qblocks = 2 * d->c / 64;
  P->Ktot = 16 * d->c;
  P->steps_total = ((d->n + P->Tb - 1) / P->Tb) * P->tiles_y;
  *bn = (P->Ktot % 256 == 0) ? 256 : (P->Ktot % 128 == 0 ? 128 : 64);
  // CTA pairs (256 ko rows per tile, see WgCfg) when there are whole 256-row tiles and a long reduction
  *cg = (*bn == 256 && d->k % 256 == 0 && P->steps_total >= 256) ? 2 : 1;
  // test hook: force CTA pairs on (2) / off (1), as in pick_cfg
  if (const char* e = getenv("EADGAN_TC_CG")) { if (*bn == 256 && d->k % 256 == 0 && (atoi(e) == 1 || atoi(e) == 2)) *cg = atoi(e); }
  const int tiles = (P->Ktot / *bn) * ((d->k + 127) / 128) / *cg;
  // split of the pixel reduction: one CTA per (tile, split) and one CTA per SM at a time, so the kernel runs in
  // waves of sm_count CTAs.  Pick the split count minimising  waves * steps_per_split  (tensor time, a 64-pixel
  // step of a 128 x bn tile is bn*2 clocks) plus the fp32 partial-sum traffic (written once, read once).
  const int sms = eg_sm_count() / *cg;   // concurrently running CTAs (CTA pairs)
  const int max_s = (P->steps_total + 7) / 8;
  const int k_pad = ((d->k + 127) / 128) * 128;
  double best = 1e300;
  int best_s = 1;
  for (int s = 1; s <= max_s && s <= 4 * sms; ++s) {
    const int sps = (P->steps_total + s - 1) / s;
    const int s_eff = (P->steps_total + sps - 1) / sps;
    const int64_t ctas = (int64_t)tiles * s_eff;
    const int64_t waves = (ctas + sms - 1) / sms;
    const double t_mma = (double)waves * (sps * (*bn) * 2.0 + 1500.0) / 1.9e9 / 0.9;  // + pipeline refill per item
    const double t_part = (double)s_eff * k_pad * (double)P->Ktot * 8.0 / 6.0e12;
    if (t_mma + t_part < best) { best = t_mma + t_part; best_s = s_eff; }
  }
  P->steps_per_split = (P->steps_total + best_s - 1) / best_s;
  *splits = (P->steps_total + P->steps_per_split - 1) / P->steps_per_split;
  return 0;
}

template <int BN, int CG = 1>
int launch_wgrad(const CUtensorMap& mdy, const CUtensorMap& mx, const WgParams& P, dim3 grid, cudaStream_t st) {
  static std::atomic<uint64_t> opted{0};
  if (int e = opt_in_smem(tc_wgrad_kernel<BN, CG>, WgCfg<BN, CG>::SMEM, opted)) return e;
  // `grid` is the logical item space (kk tiles, ko tiles, splits); the launch is one CTA per SM at most, every
  // CTA running the same number of items (+-1)
  WgParams Q = P;
  Q.kk_tiles = (int)grid.x; Q.ko_tiles = (int)grid.y; Q.splits = (int)grid.z;
  const int total = Q.kk_tiles * Q.ko_tiles * Q.splits;
  const int units = eg_sm_count() / CG;
  const int waves = (total + units - 1) / units;
  const int ctas = ((total + waves - 1) / waves) * CG;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(ctas); cfg.blockDim = dim3(192); cfg.dynamicSmemBytes = WgCfg<BN, CG>::SMEM; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = CG == 2 ? 1 : 0;
  EG_CUDA(cudaLaunchKernelEx(&cfg, tc_wgrad_kernel<BN, CG>, mdy, mx, Q));
  EG_LAUNCH_CHECK("tc_wgrad_kernel");
  return 0;
}
}  // namespace

extern "C" size_t eadgan_tc_workspace_bytes(const eadgan_tc_desc* d, int direction) {
  if (direction != 2 || !d) return 0;
  WgParams P{};
  int bn = 0, splits = 0, cg = 1;
  if (wgrad_plan(d, &P, &bn, &splits, &cg) != 0) return 0;
  const int k_pad = ((d->k + 127) / 128) * 128;
  return (size_t)splits * k_pad * (size_t)P.Ktot * sizeof(float);
}

extern "C" int eadgan_tc_wgrad(const eadgan_tc_desc* d, const void* x_pad, const void* dy_pad, float* dw,
                               void* workspace, size_t ws_bytes, void* stream) {
  if (int e = check_tc(d, "tc_wgrad")) return e;
  EG_REQUIRE(x_pad && dy_pad && dw && workspace, EADGAN_ERR_INVALID, "tc_wgrad: NULL pointer");
  WgParams P{};
  int bn = 0, splits = 0, cg = 1;
  if (int e = wgrad_plan(d, &P, &bn, &splits, &cg)) return e;
  const int k_pad = ((d->k + 127) / 128) * 128;
  const size_t need = (size_t)splits * k_pad * (size_t)P.Ktot * sizeof(float);
  EG_REQUIRE(ws_bytes >= need, EADGAN_ERR_WORKSPACE, "tc_wgrad: workspace %zu < %zu bytes", ws_bytes, need);
  P.partial = (float*)workspace;
  // partial rows are indexed with stride P.k: use the padded k so out-of-range rows stay in bounds
  WgParams PK = P;
  PK.k = k_pad;
  CUtensorMap mdy, mx;
  if (int e = map_small(&mdy, dy_pad, d->n, d->k, P.p, P.q, P.Tw, P.Th, P.Tb)) return e;
  if (int e = map_big_s2d(&mx, x_pad, d->n, d->c, d->h, d->w, P.Tw, P.Th, P.Tb)) return e;
  dim3 grid(P.Ktot / bn, k_pad / (128 * cg), splits);
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  switch (bn) {
    case 64: rc = launch_wgrad<64>(mdy, mx, PK, grid, st); break;
    case 128: rc = launch_wgrad<128>(mdy, mx, PK, grid, st); break;
    default: rc = cg == 2 ? launch_wgrad<256, 2>(mdy, mx, PK, grid, st) : launch_wgrad<256>(mdy, mx, PK, grid, st); break;
  }
  if (rc) return rc;
  const int c_real = (d->c_real > 0 && d->c_real < d->c) ? d->c_real : d->c;
  wgrad_reduce_kernel<<<dim3((d->c + 63) / 64, d->k), 256, 0, st>>>(P.partial, splits, k_pad, d->c, c_real, dw);
  EG_LAUNCH_CHECK("wgrad_reduce_kernel");
  return 0;
}

extern "C" int eadgan_tc_gemm(const void* a_bf16, const void* b_bf16, float* c_f32, int m, int n, int kk,
                              void* stream) {
  EG_REQUIRE(a_bf16 && b_bf16 && c_f32 && m > 0 && n > 0 && kk > 0, EADGAN_ERR_INVALID, "tc_gemm: bad arguments");
  EG_REQUIRE(kk % 64 == 0, EADGAN_ERR_UNSUPPORTED, "tc_gemm: K=%d must be a multiple of 64", kk);
  const TileCfg tcfg = pick_cfg(n, (m + 127) / 128, 1, true);
  const int bn = tcfg.bn;
  EG_REQUIRE(bn > 0, EADGAN_ERR_UNSUPPORTED, "tc_gemm: N=%d must be a multiple of 32", n);
  TcParams P{};
  P.mode = MODE_GEMM; P.nkb = kk / 64; P.gemm_m = m; P.gemm_n = n; P.out = c_f32; P.N_total = n; P.n_store = n;
  CUtensorMap ma, mb;
  if (int e = map_matrix(&ma, a_bf16, m, kk, 128)) return e;
  if (int e = map_matrix(&mb, b_bf16, n, kk, bn / tcfg.cg)) return e;
  return dispatch_conv(tcfg, ma, mb, P, (m + 127) / 128, n, 1, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------
// "dense" 4x4 <-> 1x1 layers as GEMMs over the batch:
//   ConvTranspose2d(m, C, 4, 1, 0) on a 1x1 input (celebA/EAD-GAN_celebA.py:76) and
//   Conv2d(C, m, 4, 1, 0) on a 4x4 input (the D/Q head, celebA/EAD-GAN_celebA.py:122)
// ------------------------------------------------------------------------------------
namespace {
int map_pad6(CUtensorMap* m, const void* base, int n, int C, int rows_box) {
  const uint64_t dims[4] = {(uint64_t)C, 6, 6, (uint64_t)n};
  const uint64_t st[3] = {(uint64_t)C * 2, (uint64_t)6 * C * 2, (uint64_t)36 * C * 2};
  const uint32_t box[4] = {64, 1, 1, (uint32_t)rows_box};
  return encode_map(m, base, 4, dims, st, box);
}
}  // namespace

extern "C" int eadgan_tc_dense_pack(const float* w, int m_real, int m_pad, int C, int rows_major, void* out,
                                    void* stream) {
  EG_REQUIRE(w && out && m_real > 0 && m_pad >= m_real && C > 0, EADGAN_ERR_INVALID, "tc_dense_pack: bad arguments");
  const int64_t total = (int64_t)m_pad * 16 * C;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 16 * eg_sm_count()) blocks = 16 * eg_sm_count();
  dense_pack_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(w, m_real, m_pad, C, rows_major, (__nv_bfloat16*)out);
  EG_LAUNCH_CHECK("dense_pack_kernel");
  return 0;
}

namespace {
constexpr int GATHER_SPLITS = 16;   // one split per tap: 8 M tiles x 16 splits fill the machine at batch 1024
__global__ void dense_gather_sum_kernel(const float* __restrict__ partial, const float* __restrict__ bias, int n,
                                        int m_real, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * m_real) return;
  const int b = i / m_real, j = i - b * m_real;
  float s = bias ? bias[j] : 0.f;
  for (int sp = 0; sp < GATHER_SPLITS; ++sp) s += partial[((int64_t)sp * n + b) * 32 + j];
  out[i] = s;
}
}  // namespace

extern "C" size_t eadgan_tc_dense_gather_workspace(int n) { return (size_t)GATHER_SPLITS * n * 32 * sizeof(float); }

// out[b][j] (fp32, j < m_real) = bias[j] + sum_{tap,c} Y[b][tap][c] * Wp[j][tap*C + c].  K = 16 C is long and
// M = n, N = 32 give only n/128 tiles, so the K range is split per tap over CTAs (fp32 slabs in the caller's
// workspace, summed in a fixed order: deterministic).
extern "C" int eadgan_tc_dense_gather(const void* y_pad, const void* w_rows, const float* bias, float* out, int n,
                                      int C, int m_real, void* workspace, size_t ws_bytes, void* stream) {
  EG_REQUIRE(y_pad && w_rows && out && n > 0 && m_real > 0, EADGAN_ERR_INVALID, "tc_dense_gather: bad arguments");
  EG_REQUIRE(C % 64 == 0 && m_real <= 32, EADGAN_ERR_UNSUPPORTED, "tc_dense_gather: needs C%%64==0 and m<=32");
  EG_REQUIRE(workspace && ws_bytes >= eadgan_tc_dense_gather_workspace(n), EADGAN_ERR_WORKSPACE,
             "tc_dense_gather: workspace %zu < %zu bytes", ws_bytes, eadgan_tc_dense_gather_workspace(n));
  TcParams P{};
  P.mode = MODE_DENSE_GATHER; P.qblocks = C / 64; P.nkb = P.qblocks /* per split: one tap */; P.gemm_m = n; P.gemm_n = 32;
  P.N_total = 32; P.n_store = 32; P.bias = nullptr; P.out = workspace;
  CUtensorMap ma, mb;
  if (int e = map_pad6(&ma, y_pad, n, C, 128)) return e;
  if (int e = map_matrix(&mb, w_rows, 32, (uint64_t)16 * C, 32)) return e;
  if (int e = dispatch_conv(pick_cfg(32, (n + 127) / 128, GATHER_SPLITS, false, 32), ma, mb, P, (n + 127) / 128, 32,
                            GATHER_SPLITS, (cudaStream_t)stream)) return e;
  dense_gather_sum_kernel<<<(n * m_real + 255) / 256, 256, 0, (cudaStream_t)stream>>>((const float*)workspace, bias, n,
                                                                                      m_real, out);
  EG_LAUNCH_CHECK("dense_gather_sum_kernel");
  return 0;
}

// Out[b][1+ky][1+kx][ch] (padded NHWC bf16) = (bias[ch] + sum_j A[b][j] * Wp[tap*C + ch][j]) * mask'(.)
extern "C" int eadgan_tc_dense_scatter(const void* a_bf16, const void* w_cols, const float* bias, void* out_pad,
                                       const void* mask, int mask_act, float slope, int n, int C, int m_pad,
                                       double* chan_sums, void* stream) {
  EG_REQUIRE(a_bf16 && w_cols && out_pad && n > 0, EADGAN_ERR_INVALID, "tc_dense_scatter: bad arguments");
  EG_REQUIRE(C % 128 == 0 && m_pad % 64 == 0, EADGAN_ERR_UNSUPPORTED, "tc_dense_scatter: needs C%%128==0, m_pad%%64==0");
  TcParams P{};
  P.mode = MODE_GEMM; P.nkb = m_pad / 64; P.gemm_m = n; P.gemm_n = 16 * C; P.N_total = 16 * C; P.n_store = 16 * C;
  P.dense_C = C; P.bias = bias; P.out = out_pad; P.mask = (const __nv_bfloat16*)mask; P.mask_mode = mask ? mask_act : 0;
  P.slope = slope;
  if (chan_sums) { P.want_stats = 2; P.stats = chan_sums; P.stat_channels = C; }
  CUtensorMap ma, mb;
  if (int e = map_matrix(&ma, a_bf16, n, m_pad, 128)) return e;
  if (int e = map_matrix(&mb, w_cols, (uint64_t)16 * C, m_pad, 128)) return e;
  return dispatch_conv(pick_cfg(16 * C, (n + 127) / 128, 1, false, 128), ma, mb, P, (n + 127) / 128, 16 * C, 1,
                       (cudaStream_t)stream);
}

extern "C" size_t eadgan_tc_dense_wgrad_workspace(int C, int m_pad) {
  const int mp = ((m_pad + 127) / 128) * 128;
  return (size_t)mp * 16 * C * sizeof(float);
}

// dw[j][ch][ky][kx] (fp32, j < m_real) = sum_b A[b][j] * Y[b][1+ky][1+kx][ch]
extern "C" int eadgan_tc_dense_wgrad(const void* a_bf16, const void* y_pad, float* dw, void* workspace,
                                     size_t ws_bytes, int n, int C, int m_real, int m_pad, void* stream) {
  EG_REQUIRE(a_bf16 && y_pad && dw && workspace && n > 0, EADGAN_ERR_INVALID, "tc_dense_wgrad: bad arguments");
  EG_REQUIRE(C % 64 == 0 && m_pad % 64 == 0 && m_real <= m_pad, EADGAN_ERR_UNSUPPORTED,
             "tc_dense_wgrad: needs C%%64==0 and m_pad%%64==0");
  const int mp = ((m_pad + 127) / 128) * 128;
  EG_REQUIRE(ws_bytes >= (size_t)mp * 16 * C * sizeof(float), EADGAN_ERR_WORKSPACE, "tc_dense_wgrad: workspace too small");
  WgParams P{};
  P.dense = 1; P.n = n; P.k = mp; P.c = C; P.qblocks = C / 64; P.Ktot = 16 * C;
  P.steps_total = (n + 63) / 64; P.steps_per_split = P.steps_total; P.partial = (float*)workspace;
  CUtensorMap ma, mx;
  if (int e = map_matrix(&ma, a_bf16, n, m_pad, 64)) return e;
  if (int e = map_pad6(&mx, y_pad, n, C, 64)) return e;
  dim3 grid(P.Ktot / 256, mp / 128, 1);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = launch_wgrad<256>(ma, mx, P, grid, st)) return rc;
  dense_wgrad_reduce_kernel<<<dim3(C / 64, m_real), 256, 0, st>>>(P.partial, mp, C, dw);
  EG_LAUNCH_CHECK("dense_wgrad_reduce_kernel");
  return 0;
}

// ------------------------------------------------------------------------------------
// "Thin" image layers: the k4 s2 p1 convolutions whose big map is the IMAGE (1..4 channels) --
// D's first Conv2d(3,128) (celebA/EAD-GAN_celebA.py:110), G's last ConvTranspose2d(128,3) (:90), the
// dSprites trunks' Conv2d(1|3,32) (dSprites/rp.py:66,95,165) and G's ConvTranspose2d(64,1|3) (:141).
// Padding 3 channels to 32 made these layers stream 8x the bytes they need; here
//   * the image lives in a ROW-EXPANDED bf16 buffer R[n][p][W+2][ky 4][c 4]: R[n][oy][X][ky][c] =
//     Xpad[n][2 oy + ky][X][c].  The whole 4x4x(4) patch of output pixel (oy, ox) is then the 64
//     CONTIGUOUS elements starting at X = 2 ox, so one TMA box (64 elems, q pixels at a 64-byte stride,
//     rows, images) is a ready 128-byte-swizzled K-major operand with K = 64 = (kx, ky, c);
//   * Conv2d forward / ConvTranspose2d input-gradient: ONE k block per 128-pixel tile (thin fprop);
//   * weight gradient: dw[ko][kk] = sum_pixels dy[pix][ko] R_patch[pix][kk], N = 64 (thin wgrad);
//   * ConvTranspose2d forward / Conv2d input-gradient: Z[pixel][(ky,kx,c)] = y[pixel][:] . W, N = 64,
//     K = k, followed by the col2im overlap-add IN THE EPILOGUE (shuffles along x, shared memory along y):
//     the small map is read once instead of once per output parity and tap.
// ------------------------------------------------------------------------------------
namespace {

// fp32 image (any strides) [* act'(mask)]  ->  R[n][p][W+2][4][4] bf16 (zero halo, zero padding channels)
__global__ void __launch_bounds__(256) thin_expand_kernel(eadgan_tensor4 src, eadgan_tensor4 mask, int act, float slope,
                                                          int n, int c_real, int h, int w,
                                                          __nv_bfloat16* __restrict__ R) {
  // one thread per (n, oy, X): up to 12 independent loads in flight, one 32-byte store
  const int p = h / 2, wp = w + 2;
  const int64_t total = (int64_t)n * p * wp;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i;
    const int X = (int)(r % wp); r /= wp;
    const int oy = (int)(r % p);
    const int b = (int)(r / p);
    const int x = X - 1;
    float v[4][4], m[4][4];
#pragma unroll
    for (int ky = 0; ky < 4; ++ky) {
      const int y = 2 * oy + ky - 1;
      const bool in = y >= 0 && y < h && x >= 0 && x < w;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        v[ky][c] = 0.f; m[ky][c] = 0.f;
        if (in && c < c_real) {
          v[ky][c] = eg_ld(src.ptr, (int64_t)b * src.sn + (int64_t)c * src.sc + (int64_t)y * src.sh + (int64_t)x * src.sw,
                           src.dtype);
          if (act != EADGAN_ACT_NONE)
            m[ky][c] = eg_ld(mask.ptr, (int64_t)b * mask.sn + (int64_t)c * mask.sc + (int64_t)y * mask.sh +
                                           (int64_t)x * mask.sw, mask.dtype);
        }
      }
    }
    uint32_t pk[8];
#pragma unroll
    for (int ky = 0; ky < 4; ++ky) {
      if (act != EADGAN_ACT_NONE) {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[ky][c] *= eg_act_grad(m[ky][c], act, slope);
      }
      __nv_bfloat162 lo = __floats2bfloat162_rn(v[ky][0], v[ky][1]), hi = __floats2bfloat162_rn(v[ky][2], v[ky][3]);
      pk[2 * ky] = *reinterpret_cast<uint32_t*>(&lo);
      pk[2 * ky + 1] = *reinterpret_cast<uint32_t*>(&hi);
    }
    uint4* dst = reinterpret_cast<uint4*>(R + i * 16);
    dst[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    dst[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
  }
}

// direction 0: Wf[ko][kx*16 + ky*4 + c] = w[ko][c][ky][kx]           (bf16 [k][64])      thin fprop B operand
// direction 1: Wt[ky*16 + kx*4 + c][ki] = w[ki][c][ky][kx]           (bf16 [64][k])      thin dgrad B operand
__global__ void thin_pack_kernel(const float* __restrict__ w, int k, int c_real, int direction,
                                 __nv_bfloat16* __restrict__ out) {
  const int total = k * 64;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int ko, ky, kx, c;
    if (direction == 0) { ko = i >> 6; const int kk = i & 63; kx = kk >> 4; ky = (kk >> 2) & 3; c = kk & 3; }
    else { const int row = i / k; ko = i - row * k; ky = row >> 4; kx = (row >> 2) & 3; c = row & 3; }
    out[i] = __float2bfloat16_rn(c < c_real ? w[(((int64_t)ko * c_real + c) * 4 + ky) * 4 + kx] : 0.f);
  }
}

// thin wgrad: sum split partials [splits][k_pad][64] (column kx*16+ky*4+c) -> dw[ko][c][ky][kx]
__global__ void thin_wgrad_reduce_kernel(const float* __restrict__ partial, int splits, int k_pad, int k, int c_real,
                                         float* __restrict__ dw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= k * 64) return;
  const int ko = i >> 6, kk = i & 63;
  const int kx = kk >> 4, ky = (kk >> 2) & 3, c = kk & 3;
  if (c >= c_real) return;
  float s = 0.f;
  for (int sp = 0; sp < splits; ++sp) s += partial[((int64_t)sp * k_pad + ko) * 64 + kk];
  dw[(((int64_t)ko * c_real + c) * 4 + ky) * 4 + kx] = s;
}

// 4-D view of the row-expanded image buffer: (64-element window, ox at a 32-element stride, oy, n)
int map_thin(CUtensorMap* m, const void* base, int n, int h, int w, int Tw, int Th, int Tb) {
  const int p = h / 2, q = w / 2;
  const uint64_t row = (uint64_t)(w + 2) * 16;   // elements per (n, oy) row of R
  const uint64_t dims[4] = {64, (uint64_t)q, (uint64_t)p, (uint64_t)n};
  const uint64_t st[3] = {64, row * 2, row * 2 * p};
  const uint32_t box[4] = {64, (uint32_t)Tw, (uint32_t)Th, (uint32_t)Tb};
  return encode_map(m, base, 4, dims, st, box);
}

struct ThinDgParams {
  int n, p;               // images, small-map rows (q == 32)
  int nkb;                // k / 64
  int tiles_per_img;      // p / 2: a tile is rows [r0-1, r0+2] of one image and OWNS rows r0, r0+1
  int c_real;
  int act; float slope;
  const float* bias;      // [c_real] or NULL
  const float* sigma;
  float* out;             // fp32 NCHW [n][c_real][2p][64]
};

constexpr int THIN_STAGES = 6;
constexpr int THIN_STAGE_BYTES = A_BYTES + 64 * BLOCK_K * 2;   // 16 KB + 8 KB
constexpr int THIN_SMEM = THIN_STAGES * THIN_STAGE_BYTES + 1024 + 256 + 2 * 2 * 4 * 12 * 32 * 4;

// Z[128 pixels][64] = y_tile[128][k] . Wt^T, then col2im.  320 threads: warp 0 TMA, warp 1 MMA, warps 2..5 and 6..9
// two epilogue groups, one per accumulator buffer (even / odd tiles of the CTA): the kernel is bound by the epilogue
// (ncu r02aa: 9 % occupancy, 0.25 eligible warps per scheduler with a single group), two tiles are drained at once.
// (TMEM lane quadrant q = warp & 3 = tile row q; lane = x).  Input row m owns output rows 2m, 2m+1:
//   out[2m  ][2j+b] = Xr_m[ky 1][b] + Xr_{m-1}[ky 3][b]        Xr[ky][0] = Z[ky][kx 1] + Z_{j-1}[ky][kx 3]
//   out[2m+1][2j+b] = Xr_m[ky 2][b] + Xr_{m+1}[ky 0][b]        Xr[ky][1] = Z[ky][kx 2] + Z_{j+1}[ky][kx 0]
__global__ void __launch_bounds__(320, 1)
tc_thin_dgrad_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                     const ThinDgParams P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + THIN_STAGES * THIN_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + THIN_STAGES;
  uint64_t* tmem_full_bar = empty_bar + THIN_STAGES;   // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;        // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
  float* xs = reinterpret_cast<float*>(smem + THIN_STAGES * THIN_STAGE_BYTES + 256);  // [2 groups][2][4 rows][12][32]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_tiles = P.n * P.tiles_per_img;

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&map_a); tma_prefetch_desc(&map_b); }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < THIN_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
      for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full_bar[b], 1); mbar_init(&tmem_empty_bar[b], 4); }
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_ptr, 128);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int b = tile / P.tiles_per_img, r0 = (tile % P.tiles_per_img) * 2;
        for (int kb = 0; kb < P.nkb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * THIN_STAGE_BYTES;
          mbar_expect_tx(&full_bar[stage], THIN_STAGE_BYTES);
          // padded small map rows r0 .. r0+3  =  image rows r0-1 .. r0+2 (row -1 / row p are the zero halo)
          tma_load_4d<1>(sa, &map_a, smem_u32(&full_bar[stage]), kb * BLOCK_K, 1, r0, b);
          tma_load_2d<1>(sa + A_BYTES, &map_b, smem_u32(&full_bar[stage]), kb * BLOCK_K, 0);
          if (++stage == THIN_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc(BLOCK_M, 64, 0, 0);
    int stage = 0; uint32_t phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      mbar_wait(&tmem_empty_bar[buf], ((it >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(buf * 64);
      for (int kb = 0; kb < P.nkb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + stage * THIN_STAGE_BYTES);
          const uint32_t sb = sa + A_BYTES;
#pragma unroll
          for (int k = 0; k < BLOCK_K / 16; ++k)
            umma_bf16(d_tmem, make_desc(sa + k * 32, 16, 1024), make_desc(sb + k * 32, 16, 1024), idesc,
                      (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit(&empty_bar[stage]);
          if (kb == P.nkb - 1) umma_commit(&tmem_full_bar[buf]);
        }
        __syncwarp();
        if (++stage == THIN_STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    const int quad = warp & 3;   // tile row: 0 = r0-1 (halo), 1 = r0, 2 = r0+1, 3 = r0+2 (halo)
    const int grp = (warp - 2) >> 2;   // epilogue group = accumulator buffer = parity of the CTA's tile counter
    const float inv_sigma = P.sigma ? 1.f / __ldg(P.sigma) : 1.f;
    float bias[4] = {0.f, 0.f, 0.f, 0.f};
    if (P.bias) {
#pragma unroll
      for (int c = 0; c < 4; ++c) if (c < P.c_real) bias[c] = __ldg(&P.bias[c]);
    }
    const int OW = 64, OH = 2 * P.p;
    int it = grp;
    for (int tile = blockIdx.x + grp * gridDim.x; tile < total_tiles; tile += 2 * gridDim.x, it += 2) {
      const int buf = grp;             // == it & 1
      const int b = tile / P.tiles_per_img, r0 = (tile % P.tiles_per_img) * 2;
      mbar_wait(&tmem_full_bar[buf], (it >> 1) & 1);
      tc_fence_after();
      float z[64];   // z[ky*16 + kx*4 + c]
      const uint32_t acc = tmem_base + (uint32_t)(buf * 64) + ((uint32_t)(quad * 32) << 16);
      tmem_ld32(acc, z);
      tmem_ld32(acc + 32, z + 32);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty_bar[buf]);
      // ---- x direction (neighbouring lanes); edges of the 32-wide map contribute zero ----
      float xr[4][2][3];
#pragma unroll
      for (int ky = 0; ky < 4; ++ky) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          float left = __shfl_up_sync(0xffffffffu, z[ky * 16 + 3 * 4 + c], 1);
          float right = __shfl_down_sync(0xffffffffu, z[ky * 16 + 0 * 4 + c], 1);
          if (lane == 0) left = 0.f;
          if (lane == 31) right = 0.f;
          xr[ky][0][c] = z[ky * 16 + 1 * 4 + c] + left;
          xr[ky][1][c] = z[ky * 16 + 2 * 4 + c] + right;
        }
      }
      // ---- y direction (neighbouring warps) through shared memory ----
      // exchange buffer alternates per use: the group's barrier of use i+1 separates the reads of use i from the writes of use i+2
      float* xg = xs + ((grp * 2 + ((it >> 1) & 1)) * 4 * 12) * 32;
      float* mine = xg + (quad * 12) * 32;
#pragma unroll
      for (int bb = 0; bb < 2; ++bb)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          mine[(0 * 6 + bb * 3 + c) * 32 + lane] = xr[0][bb][c];   // what the row ABOVE needs (its out[2m+1])
          mine[(1 * 6 + bb * 3 + c) * 32 + lane] = xr[3][bb][c];   // what the row BELOW needs (its out[2m])
        }
      if (grp == 0) asm volatile("bar.sync 1, 128;" ::: "memory"); else asm volatile("bar.sync 2, 128;" ::: "memory");
      if (quad == 1 || quad == 2) {
        const int m = r0 + quad - 1;
        const float* above = xg + ((quad - 1) * 12) * 32;   // row m-1: its ky = 3 sums
        const float* below = xg + ((quad + 1) * 12) * 32;   // row m+1: its ky = 0 sums
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          if (c < P.c_real) {
            float o[2][2];
#pragma unroll
            for (int bb = 0; bb < 2; ++bb) {
              o[0][bb] = (xr[1][bb][c] + above[(1 * 6 + bb * 3 + c) * 32 + lane]) * inv_sigma + bias[c];
              o[1][bb] = (xr[2][bb][c] + below[(0 * 6 + bb * 3 + c) * 32 + lane]) * inv_sigma + bias[c];
            }
            if (P.act != EADGAN_ACT_NONE) {
#pragma unroll
              for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int bb = 0; bb < 2; ++bb) o[a][bb] = eg_act(o[a][bb], P.act, P.slope);
            }
            float* op = P.out + (((int64_t)b * P.c_real + c) * OH + 2 * m) * OW + 2 * lane;
            *reinterpret_cast<float2*>(op) = make_float2(o[0][0], o[0][1]);
            *reinterpret_cast<float2*>(op + OW) = make_float2(o[1][0], o[1][1]);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 128);
}

int check_thin(const eadgan_tc_desc* d, const char* who) {
  if (int e = check_tc(d, who)) return e;
  EG_REQUIRE(d->c >= 1 && d->c <= 4, EADGAN_ERR_UNSUPPORTED, "%s: the image must have 1..4 channels (got %d)", who, d->c);
  return 0;
}

}  // namespace

extern "C" size_t eadgan_tc_thin_buffer_elems(int n, int h, int w) { return (size_t)n * (h / 2) * (w + 2) * 16; }

extern "C" int eadgan_tc_thin_expand(const eadgan_tensor4* src, const eadgan_tensor4* mask, int act, float slope, int n,
                                     int c_real, int h, int w, void* r_out, void* stream) {
  EG_REQUIRE(src && src->ptr && r_out && n > 0 && c_real >= 1 && c_real <= 4 && h >= 2 && w >= 2 && h % 2 == 0 &&
                 w % 2 == 0, EADGAN_ERR_INVALID, "tc_thin_expand: bad arguments");
  EG_REQUIRE(act == EADGAN_ACT_NONE || (mask && mask->ptr), EADGAN_ERR_INVALID, "tc_thin_expand: act without mask");
  const int64_t total = (int64_t)n * (h / 2) * (w + 2);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 32 * eg_sm_count()) blocks = 32 * eg_sm_count();
  eadgan_tensor4 mk = mask ? *mask : *src;
  thin_expand_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(*src, mk, mask ? act : EADGAN_ACT_NONE, slope, n, c_real, h,
                                                               w, (__nv_bfloat16*)r_out);
  EG_LAUNCH_CHECK("thin_expand_kernel");
  return 0;
}

extern "C" int eadgan_tc_thin_pack_w(const float* w, int k, int c_real, int direction, void* out, void* stream) {
  EG_REQUIRE(w && out && k > 0 && c_real >= 1 && c_real <= 4 && (direction == 0 || direction == 1), EADGAN_ERR_INVALID,
             "tc_thin_pack_w: bad arguments");
  thin_pack_kernel<<<(k * 64 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, k, c_real, direction, (__nv_bfloat16*)out);
  EG_LAUNCH_CHECK("thin_pack_kernel");
  return 0;
}

// y[n,p+2,q+2,k] (padded NHWC bf16) or fp32 NCHW = act(conv(image, W / sigma) + bias) [* mask'(.)]
extern "C" int eadgan_tc_thin_fprop(const eadgan_tc_desc* d, const void* r_buf, const void* w_packed, const float* bias,
                                    void* y, const void* mask, double* stats, const float* sigma, void* stream) {
  if (int e = check_thin(d, "tc_thin_fprop")) return e;
  EG_REQUIRE(r_buf && w_packed && y, EADGAN_ERR_INVALID, "tc_thin_fprop: NULL pointer");
  const int p = d->h / 2, q = d->w / 2;
  TcParams P{};
  P.mode = MODE_FPROP; P.thin = 1; P.n = d->n; P.p = p; P.q = q;
  EG_REQUIRE(pick_tile(p, q, 128, &P.Tw, &P.Th, &P.Tb) == 0, EADGAN_ERR_UNSUPPORTED,
             "tc_thin_fprop: output map %dx%d must be a power of two <= 128 wide", p, q);
  const int m_tiles = ((d->n + P.Tb - 1) / P.Tb) * (p / P.Th);
  const int bn = pick_bn(d->k);
  EG_REQUIRE(bn > 0, EADGAN_ERR_UNSUPPORTED, "tc_thin_fprop: k=%d must be a multiple of 32", d->k);
  const TileCfg tcfg = pick_cfg(d->k, m_tiles, 1, false, bn);
  P.tiles_y = p / P.Th; P.N_total = d->k; P.K_ch = 4; P.qblocks = 1; P.nkb = 1;
  bool channel_major = d->k % 128 == 0 && !d->out_f32_nchw && (int64_t)m_tiles * (d->k / 128) >= 8 * eg_sm_count();
  if (const char* e = getenv("EADGAN_TC_DGRADT")) {   // test hook: 0 / 2 = never / always channel-major where it applies
    if (atoi(e) == 0) channel_major = false;
    else if (atoi(e) == 2) channel_major = d->k % 128 == 0 && !d->out_f32_nchw;
  }
  P.act = d->act; P.slope = d->slope; P.out_f32_nchw = d->out_f32_nchw; P.want_stats = d->want_stats;
  P.mask_mode = d->mask_mode; P.OH = p; P.OW = q; P.bias = bias; P.out = y;
  P.mask = (const __nv_bfloat16*)mask; P.stats = stats; P.n_store = d->k; P.stat_channels = d->k; P.sigma = sigma;
  EG_REQUIRE(!P.mask_mode || mask, EADGAN_ERR_INVALID, "tc_thin_fprop: mask_mode without mask");
  EG_REQUIRE(!P.want_stats || stats, EADGAN_ERR_INVALID, "tc_thin_fprop: want_stats without stats");
  CUtensorMap ma, mb;
  if (int e = map_thin(&ma, r_buf, d->n, d->h, d->w, P.Tw, P.Th, P.Tb)) return e;
  if (channel_major) {   // tc_dgradT_kernel: 128 channels x 256 pixels per tile
    P.m_tiles = (m_tiles + 1) / 2; P.n_tiles = d->k / 128; P.parities = 1;
    if (int e = map_matrix(&mb, w_packed, d->k, 64, 128)) return e;
    return launch_channel_major(ma, mb, P, (cudaStream_t)stream);
  }
  if (int e = map_matrix(&mb, w_packed, d->k, 64, bn)) return e;
  return dispatch_conv(tcfg, ma, mb, P, m_tiles, d->k, 1, (cudaStream_t)stream);
}

namespace {
int thin_wgrad_plan(const eadgan_tc_desc* d, WgParams* P, int* splits) {
  const int p = d->h / 2, q = d->w / 2;
  EG_REQUIRE(d->k % 32 == 0, EADGAN_ERR_UNSUPPORTED, "tc_thin_wgrad: k=%d must be a multiple of 32", d->k);
  P->n = d->n; P->p = p; P->q = q; P->k = d->k; P->c = 4; P->thin = 1;
  EG_REQUIRE(pick_tile(p, q, 64, &P->Tw, &P->Th, &P->Tb) == 0, EADGAN_ERR_UNSUPPORTED,
             "tc_thin_wgrad: small map %dx%d must be a power of two <= 64 wide", p, q);
  P->tiles_y = p / P->Th; P->qblocks = 1; P->Ktot = 64;
  P->steps_total = ((d->n + P->Tb - 1) / P->Tb) * P->tiles_y;
  // the only parallelism is the split of the pixel reduction: one CTA per SM (per 128-row ko tile)
  const int ko_tiles = (d->k + 127) / 128;
  int s = eg_sm_count() / ko_tiles;
  const int max_s = (P->steps_total + 7) / 8;
  if (s > max_s) s = max_s;
  if (s < 1) s = 1;
  P->steps_per_split = (P->steps_total + s - 1) / s;
  *splits = (P->steps_total + P->steps_per_split - 1) / P->steps_per_split;
  return 0;
}
}  // namespace

extern "C" size_t eadgan_tc_thin_wgrad_workspace(const eadgan_tc_desc* d) {
  if (!d) return 0;
  WgParams P{};
  int splits = 0;
  if (thin_wgrad_plan(d, &P, &splits) != 0) return 0;
  return (size_t)splits * (((d->k + 127) / 128) * 128) * 64 * sizeof(float);
}

// dw[k][c][4][4] fp32 = sum over pixels of dy (padded NHWC bf16 small map) x image patch (row-expanded buffer)
extern "C" int eadgan_tc_thin_wgrad(const eadgan_tc_desc* d, const void* r_buf, const void* dy_pad, float* dw,
                                    void* workspace, size_t ws_bytes, void* stream) {
  if (int e = check_thin(d, "tc_thin_wgrad")) return e;
  EG_REQUIRE(r_buf && dy_pad && dw && workspace, EADGAN_ERR_INVALID, "tc_thin_wgrad: NULL pointer");
  WgParams P{};
  int splits = 0;
  if (int e = thin_wgrad_plan(d, &P, &splits)) return e;
  const int k_pad = ((d->k + 127) / 128) * 128;
  const size_t need = (size_t)splits * k_pad * 64 * sizeof(float);
  EG_REQUIRE(ws_bytes >= need, EADGAN_ERR_WORKSPACE, "tc_thin_wgrad: workspace %zu < %zu bytes", ws_bytes, need);
  P.partial = (float*)workspace;
  WgParams PK = P;
  PK.k = k_pad;
  CUtensorMap mdy, mx;
  if (int e = map_small(&mdy, dy_pad, d->n, d->k, P.p, P.q, P.Tw, P.Th, P.Tb)) return e;
  if (int e = map_thin(&mx, r_buf, d->n, d->h, d->w, P.Tw, P.Th, P.Tb)) return e;
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = launch_wgrad<64>(mdy, mx, PK, dim3(1, k_pad / 128, splits), st)) return rc;
  thin_wgrad_reduce_kernel<<<(d->k * 64 + 255) / 256, 256, 0, st>>>(P.partial, splits, k_pad, d->k, d->c, dw);
  EG_LAUNCH_CHECK("thin_wgrad_reduce_kernel");
  return 0;
}

// out fp32 NCHW [n][c][2p][64] = act(conv_transpose(dy, W / sigma) + bias): GEMM over input pixels + col2im epilogue
extern "C" int eadgan_tc_thin_dgrad(const eadgan_tc_desc* d, const void* dy_pad, const void* w_packed, const float* bias,
                                    float* out, const float* sigma, void* stream) {
  if (int e = check_thin(d, "tc_thin_dgrad")) return e;
  EG_REQUIRE(dy_pad && w_packed && out, EADGAN_ERR_INVALID, "tc_thin_dgrad: NULL pointer");
  const int p = d->h / 2, q = d->w / 2;
  EG_REQUIRE(q == 32 && p >= 2 && p % 2 == 0, EADGAN_ERR_UNSUPPORTED,
             "tc_thin_dgrad: the small map must be 32 wide with an even number of rows (got %dx%d)", p, q);
  EG_REQUIRE(d->k % 64 == 0 || d->k == 32, EADGAN_ERR_UNSUPPORTED, "tc_thin_dgrad: k=%d must be 32 or a multiple of 64", d->k);
  EG_REQUIRE(d->c <= 3, EADGAN_ERR_UNSUPPORTED, "tc_thin_dgrad: at most 3 image channels");
  ThinDgParams P{};
  P.n = d->n; P.p = p; P.nkb = (d->k + 63) / 64; P.tiles_per_img = p / 2; P.c_real = d->c; P.act = d->act; P.slope = d->slope;
  P.bias = bias; P.sigma = sigma; P.out = out;
  CUtensorMap ma, mb;
  if (int e = map_small(&ma, dy_pad, d->n, d->k, p, q, 32, 4, 1)) return e;
  if (int e = map_matrix(&mb, w_packed, 64, (uint64_t)d->k, 64)) return e;
  static std::atomic<uint64_t> opted{0};
  if (int e = opt_in_smem(tc_thin_dgrad_kernel, THIN_SMEM, opted)) return e;
  const int total = d->n * (p / 2);
  const int sms = eg_sm_count();
  const int waves = (total + sms - 1) / sms;
  const int grid = (total + waves - 1) / waves;
  tc_thin_dgrad_kernel<<<grid, 320, THIN_SMEM, (cudaStream_t)stream>>>(ma, mb, P);
  EG_LAUNCH_CHECK("tc_thin_dgrad_kernel");
  return 0;
}
