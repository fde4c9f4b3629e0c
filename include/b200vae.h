/* b200vae.h -- C ABI of libb200vae.so: the B200 (sm_100a) decoder-and-loss hot path of vae-song.
 *
 * The reference (claviclecrusher/vae-song) is pure Python/PyTorch and has NO FFI of its own
 * (SURVEY.md section 8(b)); each entry point below replaces a block of PyTorch-eager ops and names
 * the reference lines it stands in for.  The Python host side (vae_song_b200/_C.py) binds these
 * with ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to contiguous row-major data (fp32 unless noted),
 *     16-byte aligned; the caller owns every buffer, the library allocates nothing persistent.
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it.
 *   - return value: 0 OK, <0 error (B200VAE_E*); nothing is launched on error.
 *   - thread-safe for distinct streams/workspaces; no global state except a device-attribute cache.
 *   - there is NO CPU path: without a CUDA device every compute entry returns B200VAE_ECUDA.
 */
#ifndef B200VAE_H
#define B200VAE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200VAE_OK 0
#define B200VAE_ESHAPE (-1)   /* bad / inconsistent sizes                                 */
#define B200VAE_EUNSUP (-2)   /* configuration not supported by this build                */
#define B200VAE_EALIGN (-3)   /* null or misaligned pointer                               */
#define B200VAE_ECUDA (-4)    /* CUDA launch / runtime error, see b200vae_last_cuda_error  */
#define B200VAE_EWS (-5)      /* workspace too small (see b200vae_icnn_workspace_bytes)    */

/* weight reparameterisation of PositiveLinear, module.py:110 (exp) / module.py:114 (clamp) */
#define B200VAE_WEIGHT_EXP 0
#define B200VAE_WEIGHT_CLAMP 1

/* arithmetic of the two H x H contractions */
#define B200VAE_PREC_FP32 0   /* FP32 SIMT FMA: the parity path (rtol 1e-5)                */
#define B200VAE_PREC_TF32 1   /* tcgen05 kind::tf32, fp32 accumulate in TMEM               */
/* value 2 is RESERVED and rejected with B200VAE_EUNSUP: version 0.1 declared a bf16 (tcgen05 kind::f16) mode here that was
 * never built.  It is not coming back for the d <= 3 kernels -- they GENERATE their A operands, so halving the tensor time
 * per MAC would make operand generation the bound, at an 8-bit mantissa -- see DESIGN.md "Out of scope". */
#define B200VAE_PREC_TF32X3 3 /* tcgen05 3xTF32 split (hi*hi + hi*lo + lo*hi): fp32-grade  */
/* fp32-grade at half the tensor time of 3xTF32: both operands split into FP16 hi/lo pairs (22 mantissa bits, like a tf32
 * pair), three tcgen05 kind::f16 MMAs per K step, every operand scaled by an exact power of two into the fp16 range (per
 * tensor for the prepared weights, per sample row for the generated operands) and unscaled in the epilogue.  Same bounds as
 * TF32X3 / FP32.  The wide-input entry points run TF32X3 for it.
 * Every tensor-core precision (TF32, TF32X3, F16X3) of the d <= 4 entry points needs d <= 3 and H <= 1024; FP32 takes
 * d <= 4, H <= 4096.  Outside that, b200vae_icnn_workspace_bytes returns 0 and b200vae_icnn_prepare, _decode_fwd,
 * _decode_bwd and _decode_bwd_params return B200VAE_EUNSUP. */
#define B200VAE_PREC_F16X3 4

/* Parameters of one module.ICNN(in_channel=d, hidden_channel=H) -- module.py:117-140.
 * Field <- state_dict key:  A0w<-A0.weight [H,d]  A0b<-A0.bias [H]  A1w<-A.0.weight [H,d]
 * A1b<-A.0.bias [H]  A2w<-A.1.weight [1,d]  A2b<-A.1.bias [1]  W0<-W.0.param [H,H] (raw)
 * W1<-W.1.param [1,H] (raw). */
typedef struct b200vae_icnn_params {
  const float *A0w, *A0b, *A1w, *A1b, *A2w, *A2b, *W0, *W1;
} b200vae_icnn_params;

/* Same shapes; every non-null field is OVERWRITTEN with the batch-summed gradient. */
typedef struct b200vae_icnn_grads {
  float *A0w, *A0b, *A1w, *A1b, *A2w, *A2b, *W0, *W1;
} b200vae_icnn_grads;

/* Bytes of caller-owned workspace needed by prepare/fwd/bwd for these sizes. `for_backward`=0
 * sizes it for prepare+fwd only.  0 for sizes or a precision the entry points refuse. */
size_t b200vae_icnn_workspace_bytes(int B, int d, int H, int precision, int for_backward);

/* Materialise the positive weights P = exp(W) | clamp(W,1e-2) (module.py:110/114) and the padded,
 * kernel-layout copies of all parameters into `ws`.  Must precede fwd/bwd whenever parameters
 * changed.  Replaces: the per-call `self.param.exp()` of PositiveLinear.forward. */
int b200vae_icnn_prepare(const b200vae_icnn_params* p, int d, int H, int weight_mode, int precision,
                         void* ws, size_t ws_bytes, void* stream);

/* Fused potential + Brenier map:  psi[b] = ICNN(z_b)  (module.py:142-148)  and
 * xhat[b,:] = grad_z( psi(z_b) + kappa*|z_b|^2 )      (model.py:820-822 / :826-828),
 * one forward-then-reverse sweep, activations never leave the SM.
 *   z [B,d]; psi [B] or NULL; xhat [B,d] or NULL;
 *   mask1 [B, Hp/32] uint32 (bit n of row b = h1[b,n] > 0; Hp = H rounded up to 128) or NULL;
 *   mask2 [B] uint8 (h2 > 0) or NULL.  Save both masks when a backward will follow. */
int b200vae_icnn_decode_fwd(const float* z, int B, int d, int H, int weight_mode, float kappa,
                            float* psi, float* xhat, uint32_t* mask1, uint8_t* mask2,
                            int precision, const void* ws, size_t ws_bytes, void* stream);

/* Double-backward of the Brenier map (what autograd runs for lipschitz.py:41 through
 * model.py:822/828):  gradients of  L = sum_b <v_b, xhat_b> + sum_b gpsi_b * psi_b.
 *   v [B,d] (dL/dxhat) or NULL; gpsi [B] (dL/dpsi) or NULL; masks as written by decode_fwd;
 *   dz [B,d] or NULL; grads: see b200vae_icnn_grads (raw-parameter gradients, i.e. already
 *   chained through exp / clamp). */
int b200vae_icnn_decode_bwd(const float* z, const float* v, const float* gpsi, const uint32_t* mask1,
                            const uint8_t* mask2, int B, int d, int H,
                            const b200vae_icnn_params* p, int weight_mode, float kappa,
                            const b200vae_icnn_grads* grads, float* dz, int precision, void* ws,
                            size_t ws_bytes, void* stream);

/* Second half of b200vae_icnn_decode_bwd for the tensor-core precisions, so that a training step can take it off its critical
 * path: call b200vae_icnn_decode_bwd with grads = NULL first (dz + the ordered column partials, left in the workspace), hand
 * dz to the encoder's backward, and run THIS call -- the batch-reduced H x H weight gradient and the finalize kernels, about
 * 40 % of the backward's time -- on another stream while the encoder's small kernels leave the GPU mostly idle.  Same z, v,
 * masks, sizes and workspace as the first call; the caller orders the two calls (this one after the first) and joins the
 * streams before reading `grads`.  Replaces nothing new in the reference: it is the parameter half of what autograd runs
 * for lipschitz.py:41.  FP32 precision: B200VAE_EUNSUP (use the one-call form). */
int b200vae_icnn_decode_bwd_params(const float* z, const float* v, const uint32_t* mask1, const uint8_t* mask2, int B,
                                   int d, int H, const b200vae_icnn_params* p, int weight_mode,
                                   const b200vae_icnn_grads* grads, int precision, void* ws, size_t ws_bytes,
                                   void* stream);

/* Exact Jacobian of the Brenier map, from the same fused forward.  With the LeakyReLU masks fixed xhat is affine in z, so
 *   jac[b] = d xhat_b / d z_b = A0^T diag(2 s0^2 gx1) A0 + 2 kappa I          (d x d, symmetric, >= 2 kappa I)
 * where gx1 = g1 . P0 is the forward's second contraction; it is the derivative almost everywhere (wherever no pre-
 * activation sits exactly on its kink) and NOT differentiable itself.  psi, xhat and the masks are bitwise those of
 * b200vae_icnn_decode_fwd on the same inputs and precision; the saved-accumulator state of a for_backward workspace is left
 * alone, so a Jacobian call may sit between a training forward and its backward.
 *   ws: prepared by b200vae_icnn_prepare (a for_backward workspace is accepted); jac [B,d,d] (required);
 *   jac_scratch: caller-owned, at least b200vae_icnn_jac_scratch_bytes(B, d, H, precision) bytes, 16-byte aligned (the
 *   tensor-core precisions publish per-(row, pass, column half) partials there: Bp * ceil(H/256) * 2 * (d <= 2 ? 1 : 2)
 *   float4, Bp = B rounded up to 256; FP32 needs none and may pass NULL).
 * Same shape / precision rules as b200vae_icnn_decode_fwd; _scratch_bytes returns 0 where the entry refuses (and for FP32,
 * which needs no scratch). */
size_t b200vae_icnn_jac_scratch_bytes(int B, int d, int H, int precision);
int b200vae_icnn_decode_jac(const float* z, int B, int d, int H, float kappa, float* psi, float* xhat, float* jac,
                            uint32_t* mask1, uint8_t* mask2, int precision, const void* ws, size_t ws_bytes,
                            void* jac_scratch, size_t jac_scratch_bytes, void* stream);

/* Chain rule of the decoder's two Brenier maps and its singular values, one thread per sample, fp64 inside:
 *   J[b] = J2[b] . M . J1[b]      J2 [B,Dx,Dx], M [Dx,D] (LIDVAE's B buffer), J1 [B,D,D]  ->  J [B,Dx,D] or NULL
 *   svals [B,min(Dx,D)] or NULL: singular values of J[b] in descending order (one-sided Jacobi, fixed sweeps).
 * 1 <= D, Dx <= 4; anything else returns B200VAE_EUNSUP. */
int b200vae_jacobian_chain(const float* J2, const float* M, const float* J1, int B, int Dx, int D, float* J, float* svals,
                           void* stream);

/* Left inverse of the Brenier map: z = T^{-1}(x), T = grad(psi + kappa|.|^2), by batched Newton steps (csrc/inverse.cu).
 * z* is the unique minimiser of f(z) = psi(z) + kappa|z|^2 - <x, z>; its gradient xhat(z) - x and Hessian jac come from
 * b200vae_icnn_decode_jac.  One ROUND is
 *     b200vae_icnn_decode_jac(z_trial, ...) -> xhat, jac;   b200vae_brenier_newton_step(x, xhat, jac, ..., round, ...)
 * after one b200vae_brenier_inverse_init.  The step kernel takes a Newton step by Cholesky with a line search on the sign
 * of (xhat - x)^T p (psi is not used), one thread per row in fp64, and writes the next trial point, the accepted z [B,d],
 * status [B] int32 (B200VAE_INV_*) and err_bound [B] = ||xhat(z) - x|| / (2 kappa) >= ||z - z*|| (+inf at kappa = 0).
 * A finished row keeps z and its trial point equals z; final_round != 0 turns rows still active into MAXITER.
 *   state: caller-owned, b200vae_brenier_inverse_state_bytes(B, d) bytes, 16-byte aligned, set by _init; its first four
 *   bytes after round k hold, at int32 index (k & 1), the number of rows still active (integer atomics: deterministic).
 *   tolerance: a row converges when ||xhat(z) - x|| <= tol_rel ||x|| + tol_abs.  z0 [B,d] or NULL (start at 0).
 * 1 <= d <= 4 (B200VAE_EUNSUP above), B >= 1; null pointers (z0 excepted) B200VAE_EALIGN; a short state B200VAE_EWS. */
#define B200VAE_INV_ACTIVE 0
#define B200VAE_INV_CONVERGED 1   /* ||xhat(z) - x|| <= tol                                                        */
#define B200VAE_INV_MAXITER 2     /* still active after the last round                                             */
#define B200VAE_INV_STALLED 3     /* line search collapsed at t = 0 (x in a jump of the gradient / at a kink), or  */
                                  /* the step no longer moves z in fp32                                            */
#define B200VAE_INV_SINGULAR 4    /* Cholesky of jac failed (kappa = 0 only)                                       */
#define B200VAE_INV_NONFINITE 5   /* x, z0 or xhat(z) not finite                                                   */
size_t b200vae_brenier_inverse_state_bytes(int B, int d);
int b200vae_brenier_inverse_init(const float* x, const float* z0, int B, int d, float tol_rel, float tol_abs, void* state,
                                 size_t state_bytes, float* z_trial, float* z, int* status, float* err_bound, void* stream);
int b200vae_brenier_newton_step(const float* x, const float* xhat, const float* jac, int B, int d, float kappa, int round,
                                int final_round, void* state, size_t state_bytes, float* z_trial, float* z, int* status,
                                float* err_bound, void* stream);

/* Fused reparameterisation + Gaussian KL + reconstruction (+ latent reconstruction).
 * Replaces model.py:843 / :423-424 (z = mu + eps*exp(lv/2)), :884/:550/:606 (KL), :870/:542/:589
 * (MSE) or :872-882 (log-MSE), :551/:603 (latent recon, mean over dim 0 = L).
 *   reparam:  mu, lv [B,D]; eps [L,B,D]; z [L,B,D]   (any may be NULL to skip)
 *   KL:       out[1] = sum_{b,j} -0.5(1+lv-mu^2-e^lv) / B
 *   recon:    x, xhat [B,Dx];  logmse=0: out[0] = sum (x-xhat)^2 / B
 *                              logmse=1: out[0] = mean_b 0.5*Dx*(log(2*pi*mse_b+1e-5)+1);
 *             mse_rows [B] scratch (needed when logmse=1, else may be NULL)
 *   latent:   z_in, z_rec [Lz,Bz,Dz]: out[2] = sum (z_in-z_rec)^2 / Lz
 *   out: B200VAE_LOSS_OUT_FLOATS fp32; out[0..2] = (recon, kl, latent).  The tail is reduction scratch
 *   (ordered block partials + a ticket): it must be ZERO before the first call and is left zeroed by
 *   every call, so one zero-initialised buffer can be reused; results are bit-reproducible. */
#define B200VAE_LOSS_OUT_FLOATS 2048
int b200vae_loss_fwd(const float* mu, const float* lv, const float* eps, float* z, int L, int B, int D,
                     const float* x, const float* xhat, int Dx, int logmse, float* mse_rows,
                     const float* z_in, const float* z_rec, int Lz, int Bz, int Dz, float* out,
                     void* stream);

/* Backward of the above given upstream scalars (device pointers, fp32):
 *   g_recon, g_kl, g_lat : dL/d out[0..2]  (NULL = 0)
 *   gz [L,B,D] : dL/dz from the decoder (NULL = 0)
 *   writes d_mu, d_lv [B,D] (KL + reparam paths), d_xhat [B,Dx], d_zrec [Lz,Bz,Dz] (NULL to skip) */
int b200vae_loss_bwd(const float* mu, const float* lv, const float* eps, const float* gz, int L, int B,
                     int D, const float* x, const float* xhat, int Dx, int logmse, const float* mse_rows,
                     const float* z_in, const float* z_rec, int Lz, int Bz, int Dz, const float* g_recon,
                     const float* g_kl, const float* g_lat, float* d_mu, float* d_lv, float* d_xhat,
                     float* d_zrec, void* stream);

/* Random-pair Lipschitz ratios, utils.py:548-562:
 *   ratio[p] = clamp(|Y[i1]-Y[i2]|_2, eps) / clamp(|X[i1]-X[i2]|_2, eps);  X [N,dx], Y [N,dy]. */
int b200vae_lipschitz_pairs(const float* X, const float* Y, const int64_t* i1, const int64_t* i2, int P,
                            int N, int dx, int dy, float eps, float* ratio, void* stream);

/* Tiled all-pairs estimator (north_star kernel 4; replaces the random-pair sampling of utils.py:544-562 by EVERY pair,
 * same per-pair formula utils.py:560-562): over unordered pairs i<j whose 64x64 tile index t (row-major over the upper
 * triangle incl. diagonal tiles) satisfies tile_begin <= t < tile_end.
 *   stats [4] fp64: max, min, sum, count -- overwritten (an empty range gives 0, DBL_MAX, 0, 0);
 *   hist [nbins] uint32 or NULL: log2-spaced histogram of ratios over [2^hist_lo, 2^hist_hi) -- overwritten;
 *   scratch: b200vae_lipschitz_scratch_bytes() bytes, 16-byte aligned: ordered per-CTA partials + a ticket.  It must be
 *   ZERO before the first call and is left ready by every call (one zero-initialised buffer per stream can be reused).
 * ONE kernel launch; max/min/sum are combined in a fixed order (bit-reproducible).  Shard tiles across ranks and combine
 * the per-rank stats with MAX/MIN/SUM. */
size_t b200vae_lipschitz_scratch_bytes(void);
int b200vae_lipschitz_allpairs(const float* X, const float* Y, int N, int dx, int dy, float eps,
                               long long tile_begin, long long tile_end, double* stats, uint32_t* hist,
                               int nbins, float hist_lo, float hist_hi, void* scratch, void* stream);
long long b200vae_lipschitz_num_tiles(int N);

/* Exact quantiles of the same keys over every pair i<j: the all-pairs version of the reference's figure, utils.py:563-567
 * (A = quantile(r, q), B = quantile(r, 1-q) of the ratios).  A pair's key is exactly the value the entry above feeds into
 * its min / max, so quantile 0 / 1 equal its min / max bit for bit.  Quantiles use torch.quantile's "linear" rule with the
 * rank arithmetic in fp64 (torch does it in the tensor's dtype, which cannot address ranks beyond 2^24):
 *   n = N(N-1)/2, pos = q (n-1), k = floor(pos), w = pos - k,  v(q) = key[k] + w (key[min(k+1, n-1)] - key[k])  (fp64).
 * A radix select on the keys' bit patterns in B200VAE_LIPSCHITZ_SELECT_PASSES = 3 passes; per pass p = 0, 1, 2:
 *   select_count(..., tile_begin, tile_end, p, state, hist)  on every rank (tiles split like the entry above): OVERWRITES
 *       hist with the counts of its pairs' keys in the bins of pass p (integer atomics only: the same at any grid size);
 *   sum hist over ranks (uint64 element-wise; skip on one rank);
 *   select_locate(N, q0, q1, p, hist, state, out)  on every rank: narrows the targets (ranks k and k+1 of q0 and q1) in
 *       `state`; pass 0 sets them from (N, q0, q1).  After pass 2: out [6] fp64 = (v(q0), v(q1), key[k0], key[k0+1],
 *       key[k1], key[k1+1]).
 * No host synchronisation inside, so a one-rank sequence can be captured into a CUDA graph.
 *   state: b200vae_lipschitz_select_state_bytes(), hist: b200vae_lipschitz_select_hist_bytes() (uint64), both 16-byte
 *   aligned, caller-owned, no initialisation needed.  Requires N >= 2 and eps > 0; B200VAE_EUNSUP when one CTA would count
 *   2^32 or more pairs (N above about 2 million points). */
#define B200VAE_LIPSCHITZ_SELECT_PASSES 3
size_t b200vae_lipschitz_select_state_bytes(void);
size_t b200vae_lipschitz_select_hist_bytes(void);
/* host only: (k, w) of the rule above for n >= 1 keys and q in [0, 1] (else B200VAE_ESHAPE) */
int b200vae_lipschitz_quantile_ranks(long long n, double q, long long* k, double* w);
int b200vae_lipschitz_select_count(const float* X, const float* Y, int N, int dx, int dy, float eps,
                                   long long tile_begin, long long tile_end, int pass, const void* state, uint64_t* hist,
                                   void* stream);
int b200vae_lipschitz_select_locate(int N, double q0, double q1, int pass, const uint64_t* hist, void* state, double* out,
                                    void* stream);

/* Fused Adam step over a flat fp32 parameter buffer (torch.optim.Adam semantics, lipschitz.py:25,43):
 *   m,v moments; step = 1-based step count; grad_scale multiplies g first (e.g. 1/world_size). */
int b200vae_adam_step(float* param, const float* grad, float* m, float* v, long long n, float lr,
                      float beta1, float beta2, float eps, float weight_decay, long long step,
                      float grad_scale, void* stream);

/* Same, with the 1-based step counter on the device (*step_dev is incremented, then used): the whole train
 * step can then be captured in a CUDA graph and replayed. */
int b200vae_adam_step_dev(float* param, const float* grad, float* m, float* v, long long n, float lr,
                          float beta1, float beta2, float eps, float weight_decay, long long* step_dev,
                          float grad_scale, void* stream);

/* Same, with the learning rate following a schedule evaluated ON THE DEVICE from the step counter (graph replay needs no
 * host-side scheduler): sched_kind 0 = constant lr0, 1 = CosineAnnealingLR(T_max = sched_T, eta_min = 0) stepped after
 * every optimiser step -- main.py:200-203, 286-287. */
int b200vae_adam_step_sched(float* param, const float* grad, float* m, float* v, long long n, float lr0, float beta1,
                            float beta2, float eps, float weight_decay, long long* step_dev, float grad_scale,
                            int sched_kind, long long sched_T, void* stream);

/* ---- fused [Linear -> BatchNorm1d -> LeakyReLU] encoder layers (model.py:711-734; SURVEY.md 8(f) rank 1) ------------
 * Widths <= 128 (backward: powers of two).  A layer INPUT is described by the previous layer's pre-BN output
 * `*_y` [B,w] plus its BatchNorm statistics `*_stats` [4][w] = (mean, biased var, invstd, count), gamma, beta; the
 * LeakyReLU(BN(.)) is applied while loading.  `*_stats` == NULL means "raw input, no BN/activation".
 * `scratch`: b200vae_mlp_scratch_bytes(B) bytes of caller-owned device memory -- ordered per-CTA partials plus, in its last
 * 256 bytes, the ticket with which the LAST CTA of a layer kernel finalises the layer's statistics / sums / weight gradient
 * itself (no separate finalize launch on one GPU), and the grid-barrier counters of the stack entries below.  They must be
 * ZERO before the first call and are left zero by
 * every call: zero-initialise the buffer once and reuse it (per stream). */
size_t b200vae_mlp_scratch_bytes(int B);
/* y_out [B,wo] = act(in) W^T + bias, W [wo,wi]; if stats_out != NULL also the batch statistics of y_out (and, when
 * running_mean/var != NULL, their momentum update with the unbiased variance -- torch.nn.BatchNorm1d semantics). */
int b200vae_mlp_layer_fwd(const float* in_y, const float* in_stats, const float* in_gamma, const float* in_beta,
                          float slope, const float* W, const float* bias, int B, int wi, int wo, float* y_out,
                          float* stats_out, float eps, float* running_mean, float* running_var, float momentum,
                          void* scratch, void* stream);
/* da [B,w] = dL/d act(y).  Writes dyhat = da*lrelu'(.) [B,w] and sums [2][w] = (sum dyhat, sum dyhat*xhat)
 * (= dbeta, dgamma).  stats == NULL: no BN (dyhat = da, sums[0] = bias gradient). */
int b200vae_mlp_layer_bwd_reduce(const float* da, const float* y, const float* stats, const float* gamma,
                                 const float* beta, float slope, int B, int w, float* dyhat, float* sums,
                                 void* scratch, void* stream);
/* With dy = gamma*invstd*(dyhat - sums[0]*inv_n - xhat*sums[1]*inv_n) (or dyhat when stats == NULL):
 * da_prev [B,wi] = dy W (NULL to skip) and dW [wo,wi] = dy^T act(prev) (NULL to skip). */
int b200vae_mlp_layer_bwd(const float* dyhat, const float* y, const float* stats, const float* gamma,
                          const float* beta, const float* sums, float inv_n, float slope, const float* W,
                          const float* prev_y, const float* prev_stats, const float* prev_gamma,
                          const float* prev_beta, int B, int wo, int wi, float* da_prev, float* dW,
                          void* scratch, void* stream);

/* ---- a whole narrow stack in one launch per direction -----------------------------------------------------------------
 * Layer l: y_l = act_{l-1}(y_{l-1}) W_l^T + bias_l with act = LeakyReLU(slope) . BatchNorm_l (y_{-1} = x, no act); every
 * layer but the last feeds a BatchNorm.  Every wi, wo <= 8, 1 <= nl <= 16.  The kernels are cooperative (all CTAs
 * co-resident; capturable into a CUDA graph) and use the same `scratch` as the layer entries above.  In training the
 * forward gives the same bits as the layer entries at the same batch. */
typedef struct {
  const float* W;                 /* [wo][wi] */
  const float* bias;              /* [wo] */
  const float* gamma;             /* [wo] BatchNorm affine (not read for the last layer) */
  const float* beta;
  float* y;                       /* [B][wo] pre-BatchNorm output: written by the forward, read by the backward */
  float* stats;                   /* [4][wo] (mean, biased var, invstd, count): training writes it, eval reads it */
  float* running_mean;            /* training: momentum update (may be NULL) */
  float* running_var;
  long long* num_batches_tracked; /* training: += 1 (may be NULL) */
  float eps, momentum;
  int wi, wo;
} b200vae_mlp_layer_t;
typedef struct {
  float* dW;                      /* [wo][wi] */
  float* db;                      /* [wo]: exactly zero for a layer that feeds a BatchNorm */
  float* dgamma;                  /* [wo] (not written for the last layer) */
  float* dbeta;
} b200vae_mlp_grad_t;
/* head > 0 (2 head == last wo): mu [B][head] = y_last[:, :head] and lv [B][head] = softplus(y_last[:, head:]) as well. */
int b200vae_mlp_stack_fwd(const b200vae_mlp_layer_t* layers, int nl, const float* x, int B, float slope, int training,
                          int head, float* mu, float* lv, void* scratch, void* stream);
/* Gradients of every parameter and (dx != NULL) of x.  head > 0: g0 = dL/dmu, g1 = dL/dlv [B][head] (NULL = zero), the
 * softplus derivative is applied inside; head == 0: g0 = dL/dy_last [B][wo]. */
int b200vae_mlp_stack_bwd(const b200vae_mlp_layer_t* layers, const b200vae_mlp_grad_t* grads, int nl, const float* x,
                          int B, float slope, int training, int head, const float* g0, const float* g1, float* dx,
                          void* scratch, void* stream);

/* ---- nearest-neighbour squared distances (chamfer_distance, model.py:896-912; SURVEY.md 8(f) rank 2) -------------------
 * minv[b,i] = min_j |A[b,i,:] - Bp[b,j,:]|^2, argm[b,i] = a minimiser.  A [B,Na,dim], Bp [B,Nb,dim], dim <= 4.  The
 * [B,Na,Nb] matrix of torch.cdist is never formed. */
int b200vae_nn_sqdist_fwd(const float* A, const float* Bp, int B, int Na, int Nb, int dim, float* minv, int* argm,
                          void* stream);
/* dA[b,i,:] = gA[b,i]*2(A_i - Bp_argA(i)) + sum_{j: argB(j)=i} gB[b,j]*2(A_i - Bp_j): gradient w.r.t. A of
 * sum gA*min_j|A_i-Bp_j|^2 + sum gB*min_i|Bp_j-A_i|^2 (argB = minimisers of the reversed query).  gA or gB may be NULL. */
int b200vae_nn_sqdist_bwd(const float* A, const float* Bp, const int* argA, const int* argB, const float* gA,
                          const float* gB, int B, int Na, int Nb, int dim, float* dA, void* stream);

/* ---- wide-input ICNN (d > 4): MNIST-shaped LIDVAE decoder, ICNN(32,512) + ICNN(784,1024) (model.py:766-805) ----------
 * Same mathematics as b200vae_icnn_decode_fwd/bwd (module.py:142-148 + the autograd.grad of model.py:822,828 and its
 * double-backward), FP32, as a chain of fused tile GEMMs whose operands are generated while loading (csrc/icnn_wide.cu).
 * Caller-owned activations: h0 [B,H] fp32, mask1 [B,H] uint8 (h1 > 0), s2 [B] fp32 (1 or 0.2) are SAVED by the forward
 * for the backward; g0 (fwd) and u0,q1,g0,t0 (bwd) are [B,H] fp32 scratch.  psi may be NULL; xhat NULL = psi only.
 * b200vae_icnn_wide_bwd takes v = dL/dxhat (the psi-gradient path is b200vae_icnn_wide_bwd_psi below) and OVERWRITES every
 * non-null field of `g` and dz.
 * `precision`: FP32 = the tile-GEMM chain above; TF32 / TF32X3 = every GEMM of the call on tcgen05 (csrc/icnn_wide_tc.cu:
 * TMA-fed 128x256 tiles, transform + hi/lo split of the A tile in shared memory, accumulators in TMEM) -- in the backward
 * the sample-stationary GEMMs (u0, w1, gx1, dz) and the batch-reduction GEMMs (dA0, dA1, dP0) alike; F16X3 runs as
 * TF32X3 (the operands come from HBM: there is no fp16 variant).  A tensor-core precision falls back to the FP32 chain
 * when d, nz or H is not a multiple of 4, and in the forward also when A0b, A1b or A2w is not 16-byte aligned (the
 * tensor-core epilogues read them with 16-byte loads).  Either backward works on whatever forward produced h0/mask1/s2.
 * b200vae_icnn_wide_workspace_bytes returns 0 for a shape or precision the entries refuse; for a tensor-core precision
 * it is the larger of the two paths' workspaces, since it sees neither nz nor the parameters' alignment.
 * `nz` (1 <= nz <= d): z is [B,nz] and the ICNN input is z ZERO-PADDED to d columns -- the x = x1 B^T step of
 * model.py:824 with B = eye(Dx, D) fused away (nz = D = 32, d = Dx = 784): products with z run over nz columns only,
 * xhat is [B,d], v is [B,d], dz is [B,nz].  nz = d is the plain case. */
size_t b200vae_icnn_wide_workspace_bytes(int B, int d, int H, int precision, int for_backward);
int b200vae_icnn_wide_fwd(const float* z, int B, int d, int nz, int H, const b200vae_icnn_params* p, int weight_mode, float kappa,
                          float* psi, float* xhat, float* h0, uint8_t* mask1, float* s2, float* g0, int precision,
                          void* workspace, size_t ws_bytes, void* stream);
int b200vae_icnn_wide_bwd(const float* z, const float* v, const float* h0, const uint8_t* mask1, const float* s2, int B,
                          int d, int nz, int H, const b200vae_icnn_params* p, int weight_mode, float kappa,
                          const b200vae_icnn_grads* g, float* dz, float* u0, float* q1, float* g0, float* t0, int precision,
                          void* workspace, size_t ws_bytes, void* stream);

/* First-order backward of psi for wide inputs (what autograd runs when module.ICNN.forward's output carries a gradient,
 * module.py:142-148; SURVEY Appendix A last line): gradients of L = sum_b gpsi[b]*psi[b] w.r.t. z (dz [B,nz], may be NULL)
 * and every parameter (non-null fields of `g` are OVERWRITTEN; A1b / A2b are NOT zero on this path).  h0 / mask1 / s2 as
 * saved by b200vae_icnn_wide_fwd (any precision); x1, g0 [B,H] fp32 and s2g [B] fp32 are caller-owned scratch; workspace
 * as for b200vae_icnn_wide_bwd with precision FP32 (this path runs on the FP32 tile kernels). */
int b200vae_icnn_wide_bwd_psi(const float* z, const float* gpsi, const float* h0, const uint8_t* mask1, const float* s2, int B,
                              int d, int nz, int H, const b200vae_icnn_params* p, int weight_mode,
                              const b200vae_icnn_grads* g, float* dz, float* x1, float* g0, float* s2g, void* workspace,
                              size_t ws_bytes, void* stream);

/* ---- aggregate-posterior log-density for calc_mi (utils.py:87-107; SURVEY.md 8(f) rank 4) ------------------------------------
 * logqz[i] = logsumexp_j log N(z[i]; mu[j], diag exp(lv[j])) - log B for z, mu, lv [B,nz]: tiled all-pairs with an online
 * logsumexp; the [B,B,nz] tensor of the reference is never formed. */
int b200vae_mi_logqz(const float* z, const float* mu, const float* lv, int B, int nz, float* logqz, void* stream);

/* Importance-weighted likelihood bound, utils.py:109-120 (nll_iw): out[0] = logsumexp over all (b, s) of
 * log p(z[b,s]) - log q(z[b,s] | x_b) with z = mu + eps*exp(lv/2); mu, lv [B,nz], eps [B,S,nz] (the caller draws eps so that
 * the random stream stays torch's).  The caller finishes  nll = -(out[0] - loss_rec - log S).  The reference materialises
 * z [B,S,nz] and three [B,S] log-density tensors; here it is one pass with an online logsumexp (ordered: reproducible).
 * scratch: b200vae_nll_iw_scratch_bytes() bytes, zero before the first call, left ready by every call. */
size_t b200vae_nll_iw_scratch_bytes(void);
int b200vae_nll_iw_lse(const float* mu, const float* lv, const float* eps, int B, int S, int nz, float* out, void* scratch,
                       void* stream);

/* ---- peer-memory exchange between the GPUs of one node (SURVEY.md 8(e): the data-parallel exchange steps) ---------------
 * The reference has no multi-GPU path; these replace what torch.distributed/NCCL would do for the LATENCY-bound
 * collectives of the sharded train step (BatchNorm statistics of model.py:711-734's encoder, 1 KB each, ten per step)
 * and for the gradient all-reduce + Adam of lipschitz.py:41-43, as kernels that read/write the other GPUs' memory
 * directly over NVLink / NVSwitch.
 *
 * Set-up (host, once): every rank calls b200vae_peer_alloc (cudaMalloc + zero fill + CUDA IPC handle), exchanges the
 * 64-byte handles out of band (torch.distributed.all_gather_object), maps the others with b200vae_peer_open and
 * fills a b200vae_peer_t with buf[r] = rank r's buffer as addressable from THIS process (own buffer at buf[rank]).
 * A host barrier must separate set-up from the first exchange.  Every rank must issue the same sequence of
 * exchanges per slot (they are collective).  NO RANK MAY LAG ANOTHER BY MORE THAN THE TIMEOUT (20 s; environment variable
 * B200VAE_PEER_TIMEOUT_S, read once per process, overrides): a peer that does not arrive in time sets a sticky per-rank
 * flag (no GPU hang) readable with b200vae_peer_timed_out; later exchanges on that rank no longer wait, and from then on
 * every exchange returns NaN payloads and b200vae_peer_allreduce_adam writes NaN parameters, so the failure cannot go
 * unnoticed. */
#define B200VAE_PEER_MAX_WORLD 16
#define B200VAE_PEER_HANDLE_BYTES 64
typedef struct b200vae_peer {
  int world, rank;
  void* buf[B200VAE_PEER_MAX_WORLD];
} b200vae_peer_t;
size_t b200vae_peer_exchange_bytes(void);  /* size of the exchange buffer (b200vae_peer_num_slots() slots)          */
int b200vae_peer_num_slots(void);
int b200vae_peer_max_payload(void);        /* floats per rank per exchange                                         */
int b200vae_peer_alloc(size_t bytes, void** buf, unsigned char* handle /*[64]*/);
int b200vae_peer_open(const unsigned char* handle /*[64]*/, void** mapped);
int b200vae_peer_close(void* mapped);
int b200vae_peer_free(void* buf);
int b200vae_peer_timed_out(const b200vae_peer_t* comm, int* out /*host*/);
/* out [world][n] = every rank's `in` [n] (n <= b200vae_peer_max_payload()); one CTA, a few microseconds. */
int b200vae_peer_allgather(const b200vae_peer_t* comm, int slot, const float* in, int n, float* out, void* stream);

/* b200vae_mlp_layer_fwd with CROSS-RANK BatchNorm statistics: the kernel that finalises this rank's (count, mean, M2)
 * publishes them to every peer, waits for theirs and Chan-combines in rank order, so stats_out / running stats are the
 * global-batch values, bit-identical on every rank.  stats_out must be non-NULL. */
int b200vae_mlp_layer_fwd_peer(const float* in_y, const float* in_stats, const float* in_gamma, const float* in_beta,
                               float slope, const float* W, const float* bias, int B, int wi, int wo, float* y_out,
                               float* stats_out, float eps, float* running_mean, float* running_var, float momentum,
                               void* scratch, const b200vae_peer_t* comm, int slot, void* stream);
/* b200vae_mlp_layer_bwd_reduce that also all-reduces the two sums over the ranks: sums_local [2][w] (this rank's
 * dbeta, dgamma contribution) and sums_global [2][w] (what b200vae_mlp_layer_bwd needs, with inv_n = 1/global batch). */
int b200vae_mlp_layer_bwd_reduce_peer(const float* da, const float* y, const float* stats, const float* gamma,
                                      const float* beta, float slope, int B, int w, float* dyhat, float* sums_local,
                                      float* sums_global, void* scratch, const b200vae_peer_t* comm, int slot,
                                      void* stream);

/* Gradient all-reduce FUSED with Adam (lipschitz.py:41-43 across ranks), two-shot over peer memory: rank r sums chunk r
 * of every rank's gradient buffer (peer loads, rank order => deterministic), applies Adam to chunk r of the parameters
 * (moments m, v: only chunk r is touched on rank r) and stores the updated chunk into EVERY rank's parameter buffer.
 * grads[r] / params[r]: rank r's flat fp32 buffers (n floats, b200vae_peer_alloc'ed and opened like the exchange
 * buffer; n % 4 == 0).  Bracketed by two exchanges on `slot`, `slot`+1 (gradients complete / parameters written).
 * grad_scale multiplies the summed gradient (1/world for a batch mean). */
int b200vae_peer_allreduce_adam(const b200vae_peer_t* comm, int slot, void* const* grads, void* const* params,
                                float* m, float* v, long long n, float lr, float beta1, float beta2, float eps,
                                float weight_decay, long long* step_dev, float grad_scale, void* stream);

int b200vae_last_cuda_error(void);
const char* b200vae_version(void);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches claim) */
long long b200vae_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* B200VAE_H */
