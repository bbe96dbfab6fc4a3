/*
 * eadgan.h -- C ABI of libeadgan.so: the sm_100a kernels behind the drop-in
 * torch.nn / torch.optim surface that EAD-GAN's training scripts construct.
 *
 * The reference (letao1991/EAD-GAN) is pure Python; its "plugin boundary" is the
 * torch operator API (SURVEY.md section 8b).  Each entry point below names the
 * reference call site(s) whose device work it replaces (paths relative to the
 * reference checkout) and the torch operator that implements it there.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch types.  All pointers are DEVICE
 *     pointers unless the name ends in _host.
 *   - `stream` is a cudaStream_t passed as void* (the caller's current stream).
 *   - the library never allocates or frees device memory and keeps no reference
 *     to caller buffers; scratch space is passed in as `workspace`.
 *   - every function returns 0 on success or a negative eadgan_status; the
 *     message is available (thread-local) from eadgan_last_error().
 *   - no silent fallback: an unsupported geometry is EADGAN_ERR_UNSUPPORTED.
 *   - functions are re-entrant; backward is called from autograd worker threads.
 */
#ifndef EADGAN_H_
#define EADGAN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EADGAN_VERSION 100

typedef enum {
  EADGAN_OK = 0,
  EADGAN_ERR_INVALID = -1,     /* bad argument */
  EADGAN_ERR_UNSUPPORTED = -2, /* geometry / dtype not implemented by this path */
  EADGAN_ERR_CUDA = -3,        /* a CUDA runtime / driver call failed */
  EADGAN_ERR_WORKSPACE = -4    /* workspace too small */
} eadgan_status;

typedef enum { EADGAN_F32 = 0, EADGAN_BF16 = 1 } eadgan_dtype;

/* fused pointwise epilogues (nn.ReLU / nn.LeakyReLU / nn.Tanh / F.sigmoid) */
typedef enum {
  EADGAN_ACT_NONE = 0,
  EADGAN_ACT_RELU = 1,
  EADGAN_ACT_LRELU = 2,
  EADGAN_ACT_TANH = 3,
  EADGAN_ACT_SIGMOID = 4
} eadgan_act;

/* A 4-D activation tensor with explicit element strides, so the same kernels read
 * fp32 NCHW module-boundary tensors and the private halo-padded NHWC bf16 buffers. */
typedef struct {
  void* ptr;
  int64_t sn, sc, sh, sw; /* element strides of the n, c, h, w axes */
  int32_t dtype;          /* eadgan_dtype */
  int32_t _pad;
} eadgan_tensor4;

/* Geometry of ONE convolution, always stated in the direction of the forward
 * convolution  x[n,c,h,w] (*) w[k,c,r,s] -> y[n,k,p,q].
 * nn.Conv2d(c,k,...)          : forward = fprop, input-grad = dgrad
 * nn.ConvTranspose2d(k,c,...) : forward = dgrad, input-grad = fprop
 * (same weight memory layout [k,c,r,s] in both cases; SURVEY.md appendix D.2). */
typedef struct {
  int32_t n, c, h, w;
  int32_t k, r, s;
  int32_t p, q;
  int32_t stride, pad;
} eadgan_conv_desc;

const char* eadgan_last_error(void);
int eadgan_version(void);
/* number of SMs of the current device (grid sizing on the host side) */
int eadgan_sm_count(void);
/* total number of kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t eadgan_kernel_launches(void);

/* ------------------------------------------------------------------------- */
/* Generic fp32-accumulate SIMT implicit-GEMM convolution (any r,s,stride,pad) */
/* Replaces F.conv2d / F.conv_transpose2d / F.linear and their autograd       */
/* (ConvolutionBackward0, AddmmBackward0) at every call site of               */
/* celebA/EAD-GAN_celebA.py:75-90,110-122; dSprites/rp.py:66-80,95-110,129-146,*/
/* 165-183; MNIST/EAD-GAN_rpqmnxy.py:77-91,105-124,141-163.                    */
/* nn.Linear(i,o) is the r=s=h=w=1 case.                                      */
/* ------------------------------------------------------------------------- */
/* y = act(conv(x, w) + bias) [* mask_act'(mask)]   -- mask: optional tensor of y's shape holding a
 * saved post-activation output; multiplies the result by that activation's derivative (fused
 * activation backward when this call computes an input gradient).  mask may be NULL. */
int eadgan_conv_fprop(const eadgan_conv_desc* d, const eadgan_tensor4* x, const float* w,
                      const float* bias, int act, float slope, const eadgan_tensor4* y,
                      const eadgan_tensor4* mask, int mask_act, float mask_slope, void* stream);
/* dx = act(conv_transpose(dy, w) + bias)   (bias/act used when this IS a ConvTranspose2d forward) */
int eadgan_conv_dgrad(const eadgan_conv_desc* d, const eadgan_tensor4* dy, const float* w,
                      const float* bias, int act, float slope, const eadgan_tensor4* dx,
                      const eadgan_tensor4* mask, int mask_act, float mask_slope, void* stream);
/* dw[k,c,r,s] = sum_{n,p,q} dy * patch(x)  (overwrites dw).  The reduction is split over CTAs; each split
 * writes its own slab of the caller's workspace and the slabs are summed in a fixed order, so the result is
 * run-to-run deterministic (no floating-point atomics).  eadgan_conv_wgrad_workspace() = bytes required. */
size_t eadgan_conv_wgrad_workspace(const eadgan_conv_desc* d);
int eadgan_conv_wgrad(const eadgan_conv_desc* d, const eadgan_tensor4* x, const eadgan_tensor4* dy,
                      float* dw, void* workspace, size_t ws_bytes, void* stream);
/* out[ch] = sum over n,h,w of t[n,ch,h,w]   (bias gradients) */
int eadgan_channel_sum(const eadgan_tensor4* t, int n, int c, int h, int w, float* out,
                       void* stream);

/* ------------------------------------------------------------------------- */
/* tcgen05 / TMEM / TMA implicit-GEMM convolution, k4 s2 p1, bf16 operands,   */
/* fp32 accumulation.  Operates on PRIVATE halo-padded NHWC bf16 buffers       */
/* [n, h+2, w+2, c] (zero halo).  Same three directions as above.             */
/* Replaces the cuDNN kernels torch dispatches for the 134-MMAC layers of      */
/* celebA/EAD-GAN_celebA.py:78-87 (G ConvT 1024-512-256-128) and :113-119      */
/* (D Conv 128-256-512-1024) and the dSprites 32/64-channel trunks.            */
/* ------------------------------------------------------------------------- */
typedef struct {
  int32_t n, c, h, w; /* big map  : [n, h+2, w+2, c] bf16 padded NHWC */
  int32_t k;          /* small map: [n, p+2, q+2, k] bf16 padded NHWC, p=h/2, q=w/2 */
  int32_t act;        /* eadgan_act fused into the epilogue */
  float slope;
  int32_t out_f32_nchw; /* 1: write the result as dense fp32 NCHW instead of padded NHWC bf16 */
  int32_t want_stats;   /* 1: accumulate per-channel sum / sum-of-squares of the pre-activation
                              output into fp64 stats[2*C] (BatchNorm statistics fused in the epilogue);
                           2: accumulate per-channel sums of the FINAL value (after activation / mask) into
                              fp64 stats[C] -- the bias gradient of the layer below, fused into the kernel
                              that produces that layer's output gradient */
  int32_t c_real;       /* 0 or c: all big-map channels are real.  0 < c_real < c: channels >= c_real of the
                              big map are zero padding (the 3-channel image layers run with c = 32); weights
                              are given / returned as [k, c_real, 4, 4] */
  int32_t mask_mode;    /* eadgan_act kind A != NONE: multiply the result by A'(mask), mask being the
                              saved padded NHWC bf16 post-activation tensor of the output's shape
                              (activation backward fused into the dgrad epilogue); 0 = off */
} eadgan_tc_desc;

/* weight repacks (fp32 [k,c,4,4] -> bf16 GEMM operand layouts); weights are divided by
 * *sigma for spectral-normalised layers (pointer to a device float, or NULL for 1) */
int eadgan_tc_pack_w_fprop(const float* w, const float* sigma, int k, int c_real, int c,
                           void* w_packed, void* stream);
int eadgan_tc_pack_w_dgrad(const float* w, const float* sigma, int k, int c_real, int c,
                           void* w_packed, void* stream);
size_t eadgan_tc_workspace_bytes(const eadgan_tc_desc* d, int direction);
/* sigma: NULL, or a device scalar -- the accumulators are multiplied by 1/sigma before bias/activation, i.e.
 * the layer computed is conv(x, W / sigma) with W the packed (un-normalised) operand.  This lets the bf16 pack
 * of a spectral-normalised weight_orig be cached across the forwards of a phase (sigma changes per forward). */
int eadgan_tc_fprop(const eadgan_tc_desc* d, const void* x_pad, const void* w_packed,
                    const float* bias, void* y, const void* mask, double* stats, const float* sigma,
                    void* stream);
int eadgan_tc_dgrad(const eadgan_tc_desc* d, const void* dy_pad, const void* w_packed,
                    const float* bias, void* dx, const void* mask, double* stats, const float* sigma,
                    void* stream);
/* dw[k,c,4,4] fp32 = sum dy (x) patch(x); workspace holds split partial sums */
int eadgan_tc_wgrad(const eadgan_tc_desc* d, const void* x_pad, const void* dy_pad, float* dw,
                    void* workspace, size_t ws_bytes, void* stream);
/* plain bf16 GEMM C[m,n] = A[m,kk] * B[n,kk]^T through the same mainloop (self-test hook
 * and the 1x1-input ConvTranspose2d(218,1024,4,1,0) of celebA/EAD-GAN_celebA.py:76) */
int eadgan_tc_gemm(const void* a_bf16, const void* b_bf16, float* c_f32, int m, int n, int kk,
                   void* stream);

/* ------------------------------------------------------------------------- */
/* "Thin" image layers: k4 s2 p1 convolutions whose big map is the IMAGE       */
/* (1..4 channels): D's first nn.Conv2d(3,128,4,2,1) (celebA/EAD-GAN_celebA.py */
/* :110), G's last nn.ConvTranspose2d(128,3,4,2,1) (:90), the dSprites trunks'  */
/* nn.Conv2d(1|3,32,4,2,1) (dSprites/rp.py:66,95,165; colored rp_color.py) and  */
/* G's nn.ConvTranspose2d(64,1|3,4,2,1) (rp.py:141).  The image is held in a    */
/* row-expanded bf16 buffer R[n][h/2][w+2][ky 4][c 4] (R[n][oy][X][ky][c] =     */
/* Xpad[n][2 oy + ky][X][c]) so that the 4x4x4 patch of an output pixel is 64   */
/* contiguous elements = one 128-byte K-major tcgen05 operand row (K = 64).     */
/* desc: c = image channels (1..4), h, w = image size, k = small-map channels.  */
/* ------------------------------------------------------------------------- */
size_t eadgan_tc_thin_buffer_elems(int n, int h, int w);   /* bf16 elements of R */
/* src: fp32/bf16 image tensor (any strides); mask/act: optional fused activation backward,
 * R <- src * act'(mask) with mask the saved post-activation output (act = 0: plain copy) */
int eadgan_tc_thin_expand(const eadgan_tensor4* src, const eadgan_tensor4* mask, int act, float slope,
                          int n, int c_real, int h, int w, void* r_out, void* stream);
/* fp32 [k,c,4,4] -> bf16 [k][64] (direction 0, fprop operand) or [64][k] (direction 1, dgrad operand) */
int eadgan_tc_thin_pack_w(const float* w, int k, int c_real, int direction, void* out, void* stream);
/* Conv2d forward / ConvTranspose2d input-gradient: y = act(conv(image, W/sigma) + bias) [* mask'] */
int eadgan_tc_thin_fprop(const eadgan_tc_desc* d, const void* r_buf, const void* w_packed,
                         const float* bias, void* y, const void* mask, double* stats, const float* sigma,
                         void* stream);
/* weight gradient dw[k,c,4,4] fp32; deterministic (split partials summed in a fixed order) */
size_t eadgan_tc_thin_wgrad_workspace(const eadgan_tc_desc* d);
int eadgan_tc_thin_wgrad(const eadgan_tc_desc* d, const void* r_buf, const void* dy_pad, float* dw,
                         void* workspace, size_t ws_bytes, void* stream);
/* ConvTranspose2d forward / Conv2d input-gradient onto the image: fp32 NCHW [n,c,h,w] =
 * act(conv_transpose(dy, W/sigma) + bias); one GEMM over the small map's pixels (N = 16 taps x 4),
 * col2im overlap-add in the epilogue.  Needs a 32-wide small map and c <= 3. */
int eadgan_tc_thin_dgrad(const eadgan_tc_desc* d, const void* dy_pad, const void* w_packed,
                         const float* bias, float* out, const float* sigma, void* stream);

/* "dense" 4x4 <-> 1x1 layers as batch GEMMs on the same tcgen05 mainloop:
 * nn.ConvTranspose2d(218,1024,4,1,0) on the 1x1 latent (celebA/EAD-GAN_celebA.py:76) and the D/Q head
 * nn.Conv2d(1024,19,4,1,0) on the 4x4 map (celebA/EAD-GAN_celebA.py:122).  The weight is always viewed
 * as w[m][ch][tap] (m = 218 latent dims, or 19 head outputs; tap = ky*4+kx), the map as padded
 * NHWC bf16 [n,6,6,C].
 *   pack   : rows_major=1 -> bf16 [m_pad][16*C] ; rows_major=0 -> bf16 [16*C][m_pad]
 *   gather : out[n][m_real] fp32 = bias + Y . w           (head forward)
 *   scatter: Y[n,6,6,C] bf16 = (bias + A . w) * mask'      (ConvT forward; head input-gradient)
 *   wgrad  : dw[m_real][C][4][4] fp32 = A^T . Y            (both weight gradients) */
int eadgan_tc_dense_pack(const float* w, int m_real, int m_pad, int C, int rows_major, void* out,
                         void* stream);
size_t eadgan_tc_dense_gather_workspace(int n);
int eadgan_tc_dense_gather(const void* y_pad, const void* w_rows, const float* bias, float* out, int n,
                           int C, int m_real, void* workspace, size_t ws_bytes, void* stream);
int eadgan_tc_dense_scatter(const void* a_bf16, const void* w_cols, const float* bias, void* out_pad,
                            const void* mask, int mask_act, float slope, int n, int C, int m_pad,
                            double* chan_sums /* NULL, or fp64 [C]: per-channel sums of the result */,
                            void* stream);
size_t eadgan_tc_dense_wgrad_workspace(int C, int m_pad);
int eadgan_tc_dense_wgrad(const void* a_bf16, const void* y_pad, float* dw, void* workspace,
                          size_t ws_bytes, int n, int C, int m_real, int m_pad, void* stream);

/* ------------------------------------------------------------------------- */
/* layout / dtype conversion between module-boundary and private buffers      */
/* ------------------------------------------------------------------------- */
/* dst[n,c,h,w] = src[n,c,h,w] with arbitrary strides/dtypes (halo not touched) */
int eadgan_copy4(const eadgan_tensor4* src, const eadgan_tensor4* dst, int n, int c, int h, int w,
                 void* stream);

/* ------------------------------------------------------------------------- */
/* BatchNorm2d, training mode (nn.BatchNorm2d at celebA/EAD-GAN_celebA.py:     */
/* 79,83,87; dSprites/rp.py:130,134,138; MNIST/EAD-GAN_rpqmnxy.py:80,83,87,145)*/
/* split so that a cross-rank all-reduce of the [2C] partial sums can sit      */
/* between the reduce and the apply halves (SyncBN).                           */
/* ------------------------------------------------------------------------- */
/* sums[0:C] = sum x, sums[C:2C] = sum x^2 over (n,h,w), fp64 accumulators -- sums must be zeroed.
 * Tensors must be dense NCHW (sw==1, sh==w) or channel-fastest NHWC rows (sc==1, sw==c). */
int eadgan_bn_stats(const eadgan_tensor4* x, int n, int c, int h, int w, double* sums, void* stream);
/* mean/invstd from global sums; running_mean/var momentum update (unbiased var),
 * torch/nn/functional.py batch_norm semantics.  running_* may be NULL. */
int eadgan_bn_finalize(const double* sums, double count, int c, float eps, float momentum,
                       float* mean, float* invstd, float* running_mean, float* running_var,
                       void* stream);
/* y = act(gamma * (x - mean) * invstd + beta) */
int eadgan_bn_apply(const eadgan_tensor4* x, int n, int c, int h, int w, const float* mean,
                    const float* invstd, const float* gamma, const float* beta, int act, float slope,
                    const eadgan_tensor4* y, void* stream);
/* sums[0:C] = sum dz, sums[C:2C] = sum dz * xhat, with dz = dy * act'(y) when act != NONE
 * (y is the saved post-activation output).  sums must be zeroed. */
int eadgan_bn_bwd_reduce(const eadgan_tensor4* dy, const eadgan_tensor4* x, const eadgan_tensor4* y,
                         int n, int c, int h, int w, const float* mean, const float* invstd,
                         const float* gamma, const float* beta, int act, float slope, double* sums,
                         void* stream);
/* dx = gamma*invstd*(dz - sum_dz/count - xhat*sum_dz_xhat/count); dgamma = sum_dz_xhat; dbeta = sum_dz */
int eadgan_bn_bwd_apply(const eadgan_tensor4* dy, const eadgan_tensor4* x, const eadgan_tensor4* y,
                        int n, int c, int h, int w, const float* mean, const float* invstd,
                        const float* gamma, const float* beta, int act, float slope,
                        const double* sums, double count, const eadgan_tensor4* dx, void* stream);
/* dgamma = local S(dz*xhat), dbeta = local S(dz) as fp32, and (dbias != NULL) the gradient of a conv
 * bias feeding this BatchNorm = sum over the local elements of dx, in closed form from the sums
 * (fwd_local_sum_x = this rank's S(x) of the forward; n_local = local n*h*w; count = global). */
int eadgan_bn_bwd_finalize(const double* local_sums, const double* global_sums,
                           const double* fwd_local_sum_x, double n_local, double count,
                           const float* mean, const float* invstd, const float* gamma, int c,
                           float* dgamma, float* dbeta, float* dbias, void* stream);
/* eval mode: y = act(gamma*(x-running_mean)/sqrt(running_var+eps)+beta) */
int eadgan_bn_eval(const eadgan_tensor4* x, int n, int c, int h, int w, const float* running_mean,
                   const float* running_var, float eps, const float* gamma, const float* beta,
                   int act, float slope, const eadgan_tensor4* y, void* stream);
/* eval-mode backward (torch NativeBatchNormBackward0 with training=False, plus the fused activation's
 * backward), one pass: dz = dy * act'(.), dx = dz * gamma * rsqrt(running_var + eps), and
 * sums[0:C] = sum dz, sums[C:2C] = sum dz * xhat with xhat = (x - running_mean) * rsqrt(running_var + eps)
 * (fp64, sums must be zeroed).  dx may alias dy.  The ReLU / LeakyReLU gate is recomputed from x on
 * bf16 NHWC buffers whose c / 8 divides 256, else read from y (y is the saved post-activation output).
 * Then, for each of dgamma / dbeta / dbias that is not NULL: dgamma = sum dz*xhat, dbeta = sum dz, and the
 * gradient of a conv bias feeding this BatchNorm, dbias = gamma * rsqrt(running_var + eps) * sum dz. */
int eadgan_bn_eval_bwd(const eadgan_tensor4* dy, const eadgan_tensor4* x, const eadgan_tensor4* y,
                       int n, int c, int h, int w, const float* running_mean, const float* running_var,
                       float eps, const float* gamma, const float* beta, int act, float slope, double* sums,
                       const eadgan_tensor4* dx, float* dgamma, float* dbeta, float* dbias, void* stream);

/* ------------------------------------------------------------------------- */
/* pointwise activations and row softmax (nn.LeakyReLU/ReLU/Tanh, F.sigmoid,   */
/* F.softmax / nn.Softmax with implicit dim=1)                                 */
/* ------------------------------------------------------------------------- */
int eadgan_act_fwd(const float* x, float* y, int64_t numel, int act, float slope, void* stream);
/* dx = dy * act'(.) expressed through the OUTPUT y (valid for all five kinds) */
int eadgan_act_bwd(const float* dy, const float* y, float* dx, int64_t numel, int act, float slope,
                   void* stream);
int eadgan_softmax_fwd(const float* x, float* y, int rows, int cols, void* stream);
int eadgan_softmax_bwd(const float* dy, const float* y, float* dx, int rows, int cols, void* stream);
/* nn.Upsample(scale_factor=2), nearest (MNIST/EAD-GAN_rpqmnxy.py:81,85) */
int eadgan_upsample2x_fwd(const float* x, float* y, int nc, int h, int w, void* stream);
int eadgan_upsample2x_bwd(const float* dy, float* dx, int nc, int h, int w, void* stream);

/* ------------------------------------------------------------------------- */
/* legacy torch.nn.utils.spectral_norm (torch/nn/utils/spectral_norm.py        */
/* SpectralNorm.compute_weight) as used at celebA/EAD-GAN_celebA.py:110-119,   */
/* dSprites/rp.py:95-109,165-183, MNIST/EAD-GAN_rpqmnxy.py:107,124,143,161-163 */
/* ------------------------------------------------------------------------- */
/* one power iteration in place on u[rows], v[cols] (skipped when do_power_iter == 0),
 * sigma = u^T W v, w_sn = W / sigma.  scratch: eadgan_spectral_norm_scratch_floats(rows, cols, 0) floats
 * (split partial sums are kept there and added in a fixed order: the result is run-to-run deterministic). */
size_t eadgan_spectral_norm_scratch_floats(int rows, int cols, int backward);
int eadgan_spectral_norm_fwd(const float* w_orig, int rows, int cols, float* u, float* v,
                             int do_power_iter, float eps, float* sigma, float* w_sn,
                             float* scratch, void* stream);
/* dW_orig = dW/sigma - (<dW, W_orig>/sigma^2) u v^T     (SURVEY.md appendix D.3) */
/* W_sn = W / sigma alone (eadgan_spectral_norm_fwd skips it when w_sn == NULL) */
int eadgan_spectral_norm_scale(const float* w_orig, const float* sigma, float* w_sn, long long n, void* stream);
int eadgan_spectral_norm_bwd(const float* dw_sn, const float* w_orig, const float* u,
                             const float* v, const float* sigma, int rows, int cols,
                             float* dw_orig, float* scratch, void* stream);

/* ------------------------------------------------------------------------- */
/* losses, forward + backward (celebA/EAD-GAN_celebA.py:161-164;               */
/* dSprites/rp.py:225-232,249-251; MNIST/EAD-GAN_rpqmnxy.py:195-198)           */
/* loss outputs are single device floats; *_bwd multiply by the upstream       */
/* gradient read from the device scalar gout.                                  */
/* ------------------------------------------------------------------------- */
int eadgan_bce_fwd(const float* p, const float* target, int64_t numel, float* loss, void* stream);
int eadgan_bce_bwd(const float* p, const float* target, const float* gout, int64_t numel,
                   float* dp, void* stream);
int eadgan_mse_fwd(const float* a, const float* b, int64_t numel, float* loss, void* stream);
/* da = 2 (a-b) / numel * gout; db = -da when db != NULL */
int eadgan_mse_bwd(const float* a, const float* b, const float* gout, int64_t numel, float* da,
                   float* db, void* stream);
/* nn.CrossEntropyLoss()(x, labels) = mean_i(-log_softmax(x_i)[labels_i]) */
int eadgan_ce_fwd(const float* x, const int64_t* labels, int rows, int cols, float* loss,
                  void* stream);
int eadgan_ce_bwd(const float* x, const int64_t* labels, const float* gout, int rows, int cols,
                  float* dx, void* stream);
/* mutual_info_loss(c_given_x, c) of dSprites/rp.py:225-232 (eps = 1e-8 inside both logs) */
int eadgan_mi_fwd(const float* q, const float* c, int rows, int cols, float* loss, void* stream);
int eadgan_mi_bwd(const float* q, const float* c, const float* gout, int rows, int cols, float* dq,
                  void* stream);

/* ------------------------------------------------------------------------- */
/* torch.optim.Adam.step (celebA/EAD-GAN_celebA.py:211-217,345,366,401), fused */
/* multi-tensor; op order of torch/optim/adam.py::_single_tensor_adam          */
/* (SURVEY.md appendix D.4).  28 bytes of HBM traffic per parameter.           */
/* ------------------------------------------------------------------------- */
#define EADGAN_ADAM_MAX_TENSORS 48
typedef struct {
  float* p[EADGAN_ADAM_MAX_TENSORS];
  const float* g[EADGAN_ADAM_MAX_TENSORS];
  float* m[EADGAN_ADAM_MAX_TENSORS];
  float* v[EADGAN_ADAM_MAX_TENSORS];
  int64_t numel[EADGAN_ADAM_MAX_TENSORS];
  int32_t count;
  int32_t _pad;
} eadgan_adam_tensors;
/* step_size = lr / (1-beta1^t), bc2_sqrt = sqrt(1-beta2^t), both computed in double on the
 * host exactly as torch does; grad_scale multiplies g on load (1/world_size for DP sums). */
int eadgan_adam_step(const eadgan_adam_tensors* t, double beta1, double beta2, double eps,
                     double step_size, double bc2_sqrt, float grad_scale, void* stream);
/* CUDA-graph form: the step count t is a DEVICE int64 (advanced by eadgan_adam_advance inside the captured
 * step), and lr/(1-beta1^t), sqrt(1-beta2^t) are formed on the device in double -- so a captured
 * optimiser step stays correct across replays (the host form bakes t into the kernel arguments). */
int eadgan_adam_step_dev(const eadgan_adam_tensors* t, double beta1, double beta2, double eps, double lr,
                         const int64_t* step_dev, float grad_scale, void* stream);
int eadgan_adam_advance(int64_t* step_dev, void* stream);

/* fill / scale helpers used by the host layer (buffer zeroing stays on our stream) */
int eadgan_fill_f32(float* p, int64_t numel, float value, void* stream);
int eadgan_f64_to_f32(const double* src, float* dst, int64_t numel, void* stream);
/* zero the 1-pixel halo of a padded NHWC bf16 buffer [n, h+2, w+2, c] (c % 8 == 0); the interior is
 * left untouched (it is fully overwritten by the producing kernel's epilogue) */
int eadgan_zero_halo(void* xp, int n, int h, int w, int c, void* stream);

/* ------------------------------------------------------------------------- */
/* Affine glue (SURVEY.md section 8f ranks 1-2).                               */
/* stn_fwd: transformation_2D.stn = F.grid_sample(x, F.affine_grid(theta, x.size()),
 * padding_mode) with align_corners = False (celebA/EAD-GAN_celebA.py:149-153; 'border' everywhere
 * but colored_dSprites/pxy_color.py:90).  img/out fp32 NCHW contiguous, theta fp32 [n,2,3].
 * relcode: "affine_regularzier" in closed form with its Jacobian (forward-mode), mode 0 =
 * celebA/utils_rpqxy.py:82-116 (5 codes -> 5), 1 = dSprites/utils_rp.py:117-147 (4 -> 4), 2 = the 2x3
 * rows of trans @ inverse(real) fed to MNIST's approximator (MNIST/utils_rpqmnxy.py:117-129; 7 -> 6).
 * real/trans: rows of >= k_in floats at the given row strides; out [n,k_out]; jac [n,k_out,2*k_in].  */
/* ------------------------------------------------------------------------- */
int eadgan_stn_fwd(const float* img, const float* theta, int n, int c, int h, int w, int padding_border,
                   float* out, void* stream);
/* F.affine_grid / F.grid_sample (bilinear, align_corners = False, padding 'border' (1) | 'zeros' (0)) as separate
 * differentiable operators, for the unmodified scripts (dSprites/rp.py:200-211,374-377,399-400 reach their backward).
 * grid [n,oh,ow,2] fp32; grid_sample_bwd: dimg must be ZEROED by the caller (scatter-add), either output may be NULL. */
int eadgan_affine_grid_fwd(const float* theta, int n, int h, int w, float* grid, void* stream);
int eadgan_affine_grid_bwd(const float* dgrid, int n, int h, int w, float* dtheta, void* stream);
int eadgan_grid_sample_fwd(const float* img, const float* grid, int n, int c, int h, int w, int oh, int ow,
                           int padding_border, float* out, void* stream);
int eadgan_grid_sample_bwd(const float* gout, const float* img, const float* grid, int n, int c, int h, int w, int oh,
                           int ow, int padding_border, float* dimg_zeroed, float* dgrid, void* stream);
int eadgan_relcode_dims(int mode, int* k_in, int* k_out);
int eadgan_relcode_fwd(int mode, const float* real, long long real_stride, const float* trans,
                       long long trans_stride, int n, float* out, float* jac, void* stream);
int eadgan_relcode_bwd(int mode, const float* g, const float* jac, int n, float* d_real, float* d_trans,
                       void* stream);

/* ------------------------------------------------------------------------- */
/* Device-side sampling of the per-iteration latent draws (SURVEY.md section 8f rank 3): replaces the host
 * NumPy sampling + H2D copies of celebA/EAD-GAN_celebA.py:308-318, dSprites/rp.py:389-396,424-434.
 * Philox4x32-10, counter = (group of 4 elements of the GLOBAL [*, cols] array, stream_id, step), key = seed:
 * rows [row0, row0+rows) of a sharded batch are exactly the rows a single device draws.
 * kind 0: uniform [lo, hi) fp32; 1: standard normal fp32 (Box-Muller); 2: integers in [0, n) as int64.
 * step: *step_dev when step_dev != NULL (CUDA-graph replay), else step_host.  See csrc/sample.cu.           */
/* ------------------------------------------------------------------------- */
int eadgan_philox(int kind, unsigned long long seed, const int64_t* step_dev, long long step_host, int stream_id,
                  long long row0, long long rows, long long cols, float lo, float hi, int n, void* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EADGAN_H_ */
