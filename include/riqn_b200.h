/* riqn_b200.h -- C-ABI of the B200-native Rainbow-IQN Ape-X learner hot path.
 *
 * The reference (valeoai/rainbow-iqn-apex) is pure Python/PyTorch and has no FFI or operator registry:
 * its boundary for this path is the Python class surface Agent / Learner / DQN / NoisyLinear /
 * ReplayRedisMemory (SURVEY.md section 8b).  This header is the boundary a native replacement exports
 * underneath that surface; rainbow_iqn_apex_b200/*.py binds it with ctypes (see INTEGRATION.md) and
 * re-creates the reference classes on top.
 *
 * Conventions
 *   - every function returns 0 on success or a cudaError_t value; nothing is allocated inside, all
 *     buffers are caller-owned DEVICE pointers unless stated; work is enqueued on `stream`
 *     (a cudaStream_t passed as void*) and is stream-ordered, re-entrant per stream;
 *   - fp32 tensors row-major.  tau, q and dtheta use the reference's quantile-major rows r = q * batch + b
 *     (rainbowiqn/model.py:149, compute_loss_iqn.py:238-310); the head-internal matrices (cos, x, h, dh, dz and
 *     their bf16 images) use sample-major rows r' = b * num_quantiles + q, which makes the Hadamard operand
 *     feat[b,:] a warp-broadcast and the reduction over a sample's quantiles contiguous;
 *   - `long long*` index buffers are int64 like the reference's torch.int64 / numpy int64.
 *
 * Each entry point cites the reference code it replaces (paths relative to /root/reference).
 */
#ifndef RIQN_B200_H
#define RIQN_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define RIQN_B200_ABI_VERSION 1

/* Library / build identification.  Returns RIQN_B200_ABI_VERSION. */
int riqn_version(void);
/* Number of CUDA kernels this library has launched in this process (bench.py's gpu_launches). */
long long riqn_launch_count(void);
/* 1 if the running device is compute capability 10.x (sm_100a cubins only), else 0; <0 on CUDA error. */
int riqn_device_ok(void);

/* Per-step scalars that change from one learner step to the next, kept in DEVICE memory so that a whole step can be
 * captured once in a CUDA graph and replayed: entry points taking `dyn` read these instead of their by-value arguments
 * when dyn != NULL (the host rewrites the 32-byte struct with one async copy before each replay). */
typedef struct riqn_dyn_state {
  unsigned long long rng_offset;   /* added to every Philox stream id (advance by >= 64 per step)          */
  float adam_neg_step_size;        /* -(lr / (1 - beta1^t))                                                 */
  float adam_sqrt_bc2;             /* sqrt(1 - beta2^t)                                                     */
  double is_capacity;              /* current replay fill, ReplayRedisMemory.sample_byte capacity (:467)    */
  double is_beta;                  /* priority_weight beta (annealed by the caller, launch_learner.py:167)  */
} riqn_dyn_state;

/* ------------------------------------------------------------------------------------------------
 * Conv trunk                                     replaces nn.Conv2d x3 + ReLU, rainbowiqn/model.py:65-67,115-118
 * ---------------------------------------------------------------------------------------------- */
typedef struct riqn_conv_geom {
  int B, Cin, H, W;          /* input  (B, Cin, H, W), NCHW                                     */
  int Cout, KH, KW;          /* weight (Cout, Cin, KH, KW)                                       */
  int stride, pad;
  int OH, OW;                /* output (B, Cout, OH, OW), NCHW (flattens C-major, model.py:118)  */
  long in_bstride;           /* elements between consecutive samples of the input (>= Cin*H*W):
                                lets conv1 read states / next_states as strided views of the
                                (B, history+n, 84, 84) replay window                             */
} riqn_conv_geom;

/* out = relu(conv(in) + bias).  `in` is uint8 frames (x/255 applied on the fly, reproducing
 * redis_memory.py:527-536) when in_is_u8 != 0, else fp32.  `col` (B*OH*OW, Cin*KH*KW) is workspace
 * that riqn_conv_bwd re-uses. */
int riqn_conv_fwd(const riqn_conv_geom* g, const void* in, int in_is_u8, const float* w, const float* bias,
                  float* col, float* out, void* stream);
/* Backward of the above: dout is dL/d(out) (post-ReLU), `out` the forward output (ReLU mask).
 * dw/dbias are ACCUMULATED into (zero them first, like zero_grad -- learner.py:22); din (may be NULL
 * for the first layer) is overwritten with dL/d(in).  dY (B*OH*OW, Cout) and dcol (like col) are
 * workspaces. */
int riqn_conv_bwd(const riqn_conv_geom* g, const float* dout, const float* out, const float* col, const float* w,
                  float* dY, float* dcol, float* dw, float* dbias, float* din, void* stream);

/* fp32 im2col alone: col (B*OH*OW, Cin*KH*KW), the workspace riqn_conv_bwd expects. */
int riqn_im2col_f32(const riqn_conv_geom* g, const void* in, int in_is_u8, float* col, void* stream);

/* Tensor-core variants (tcgen05 GEMM on bf16 im2col operands written straight from the uint8 / fp32 input).
 * w_hi / w_lo: bf16 images of the (Cout, Cin*KH*KW) weight (riqn_split_bf16); col_lo == NULL selects the
 * single-bf16 product, otherwise split-bf16 x3 (fp32-faithful).  col_hi/col_lo (M, K) bf16 workspaces; colT_hi
 * (K, M), if non-NULL, is also written for riqn_conv_bwd_tc (needs B*OH*OW % 8 == 0). */
int riqn_conv_fwd_tc(const riqn_conv_geom* g, const void* in, int in_is_u8, const void* w_hi, const void* w_lo,
                     const float* bias, void* col_hi, void* col_lo, void* colT_hi, float* out, void* stream);
/* Strip convolution: the forward of nn.Conv2d + ReLU (model.py:65-67,115-118) with NO im2col matrix.  With kernel edge
 * k = t*stride the padded input is cut into stride x stride blocks (block matrix: B*G*G rows of stride^2*Cin values,
 * G = OH + t - 1) and the outputs are laid on the same G x G grid, so that every k-block of the implicit im2col matrix
 * is a 2-D tile of the block matrix at a row offset (TMA).  Requires stride^2*Cin % 64 == 0, Cout <= 64.
 *   riqn_s2d_u8: uint8 frame stack -> block matrix a_px (B*G*G, stride^2*Cin) bf16 of raw pixel values, within-block
 *                order (c, iy, ix); the 1/255 of redis_memory.py:527-536 is folded into the weights.
 *   riqn_conv_fwd_strip: a_hi / a_lo (lo may be NULL) block matrices; w_hi / w_lo (Cout, K) bf16 weights with K
 *                ordered (dy, dx, within-block); out (B, Cout, OH, OW) fp32 = relu(conv + bias), or NULL when only the
 *                next layer's images are wanted (no-grad passes); next_hi / next_lo (may be
 *                NULL) receive the result as the NEXT layer's block matrix (block edge next_stride, grid next_grid,
 *                within-block order (iy, ix, c)).
 *   riqn_im2col_bf16_t: the transposed bf16 im2col (K, M) alone, the wgrad operand of riqn_conv_bwd_tc. */
int riqn_s2d_u8(const riqn_conv_geom* g, const unsigned char* in, void* a_px, void* stream);
int riqn_conv_fwd_strip(const riqn_conv_geom* g, const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo,
                        const float* bias, float* out, void* next_hi, void* next_lo, int next_stride, int next_grid,
                        const void* w2_hi, const void* w2_lo, const float* bias2, int share_a, void* stream);
/* w2_hi != NULL: TWO networks in one launch (the online and the target trunk over the same next_states): g->B counts both
 * halves of a stacked batch, samples [0, B/2) use w_hi / w_lo / bias, samples [B/2, B) use w2_hi / w2_lo / bias2; outputs and
 * next-layer images are the stacked (B, ...) tensors.  share_a != 0: the A image holds B/2 samples read by both halves (first
 * layer: the pixel block matrix).  Needs (B/2)*G*G % 128 == 0. */
int riqn_im2col_bf16_t(const riqn_conv_geom* g, const void* in, int in_is_u8, void* colT_hi, void* stream);
/* Backward of a strip convolution on the tensor cores, again without im2col matrices: a_hi is the block matrix the
 * forward read (riqn_s2d_u8 / the previous layer's next_hi); w_hi (Cout, K) bf16 weight in the ORIGINAL k order (data
 * gradient, read as an MN-major operand); perm (K ints): strip k order -> original k; dYg (B*G*G, Cout) bf16 and dwp_scratch (Cout*K floats)
 * workspaces; dw / dbias accumulated; din (may be NULL; pad == 0 only) overwritten.  wgrad_scale = 1/255 when a_hi
 * holds raw pixel values. */
int riqn_conv_bwd_strip(const riqn_conv_geom* g, const float* dout, const float* out, const void* a_hi, const void* w_hi,
                        const int* perm, void* dYg, float* dwp_scratch, float* dw, float* dbias, float* din,
                        float wgrad_scale, void* stream);

/* Backward on the tensor cores (bf16 operands, fp32 accumulate): wT_hi (K, Cout) bf16; dY_hi (M, Cout) and dYT_hi
 * (Cout, M) bf16 workspaces; dcol fp32 (M, K) workspace; dw/dbias accumulated; din may be NULL. */
int riqn_conv_bwd_tc(const riqn_conv_geom* g, const float* dout, const float* out, const void* colT_hi, const void* wT_hi,
                     void* dY_hi, void* dYT_hi, float* dcol, float* dw, float* dbias, float* din, float wgrad_scale,
                     void* stream);
/* First layer on raw uint8 frames: pixel values 0..255 are exact in bf16, so the im2col operand has no lo image and the
 * reference's /255 (redis_memory.py:527-536) is folded into the weights: ws_hi / ws_lo = bf16 images of weight/255
 * (ws_lo == NULL: single-bf16 product).  col_px (M, K) and colT_px (K, M; may be NULL) hold pixel values; pass
 * wgrad_scale = 1/255 to riqn_conv_bwd_tc when it consumes colT_px.  in: 16-byte aligned, in_bstride % 16 == 0.
 * reuse_col != 0: col_px already holds the im2col of `in` (the online and target passes over next_states share it). */
int riqn_conv_fwd_tc_u8(const riqn_conv_geom* g, const unsigned char* in, const void* ws_hi, const void* ws_lo,
                        const float* bias, void* col_px, void* colT_px, float* out, int reuse_col, void* stream);
/* split of (src * scale): bf16 hi / lo images of a scaled matrix (e.g. weight/255). */
int riqn_split_bf16_scaled(long rows, int cols, const float* src, float scale, void* hi, void* lo, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Randomness                       replaces torch normal_/uniform_ draws, model.py:32-37 and :131-134
 * ---------------------------------------------------------------------------------------------- */
/* out[i] ~ U(0,1): the quantile fractions tau.  Philox4x32-10 keyed by (seed, stream_id). */
int riqn_fill_uniform(long n, unsigned long long seed, unsigned long long stream_id, float* out,
                      const riqn_dyn_state* dyn, void* stream);
/* out[i] = sign(x) sqrt|x|, x ~ N(0,1): NoisyLinear._scale_noise (model.py:32-37). */
int riqn_noisy_sample(long n, unsigned long long seed, unsigned long long stream_id, float* out,
                      const riqn_dyn_state* dyn, void* stream);

/* ------------------------------------------------------------------------------------------------
 * NoisyLinear                                             replaces rainbowiqn/model.py:9-53
 * ---------------------------------------------------------------------------------------------- */
/* reset_noise + effective weights in one pass.  If eps_in/eps_out are non-NULL, weight_epsilon :=
 * eps_out (x) eps_in and bias_epsilon := eps_out are (re)written (model.py:39-43); otherwise the
 * stored epsilons are used.  w_eff = mu + sigma*eps, b_eff likewise (training != 0, model.py:46-51)
 * or the mu's alone (eval, model.py:52-53). */
int riqn_noisy_compose(int out_features, int in_features, const float* weight_mu, const float* weight_sigma,
                       float* weight_epsilon, const float* eps_in, const float* eps_out, const float* bias_mu,
                       const float* bias_sigma, float* bias_epsilon, float* w_eff, float* b_eff, int training,
                       void* stream);

/* One NoisyLinear layer of a network-wide noise reset (riqn_noisy_reset_net). */
typedef struct riqn_noisy_layer {
  int out_features, in_features;                 /* in_features % 4 == 0 */
  const float* weight_mu;
  const float* weight_sigma;
  float* weight_epsilon;                         /* (out, in): eps_out (x) eps_in is written here */
  const float* bias_mu;
  const float* bias_sigma;
  float* bias_epsilon;                           /* (out) */
  float* eps_in;                                 /* (in)  factor vector f(eps_in): drawn here when sample != 0 */
  float* eps_out;                                /* (out) factor vector f(eps_out) */
  float* w_eff;                                  /* (out, in) mu + sigma * eps   (mu when training == 0) */
  float* b_eff;                                  /* (out) */
  unsigned long long stream_in, stream_out;      /* Philox stream ids of the two draws */
  void* w_hi;                                    /* (out, in) bf16 image of w_eff for the tensor-core products, or NULL */
  void* w_lo;                                    /* (out, in) bf16(w_eff - hi), or NULL */
  int w_fp16;                                    /* != 0: w_hi = fp16(w_eff), w_lo (or NULL) = bf16(w_eff) -- fp16 head forward */
} riqn_noisy_layer;

/* DQN.reset_noise() for all NoisyLinear layers of one network in two launches (model.py:159-162 -> :39-43 -> :32-37):
 * draw every factor vector (sample != 0; same values as riqn_noisy_sample on the same seed / stream ids), then
 * compose every layer like riqn_noisy_compose.  layers is a HOST array of n_layers <= 8 descriptors. */
int riqn_noisy_reset_net(int n_layers, const riqn_noisy_layer* layers, unsigned long long seed, int sample, int training,
                         const riqn_dyn_state* dyn, void* stream);
/* h = relu(x w_eff^T + b_eff)   (the hidden layers fcnoisy_h_v | fcnoisy_h_a concatenated along out_features,
 * model.py:153-154 with the F.relu folded in). */
int riqn_noisy_linear_fwd(long rows, int in_features, int out_features, const float* x, const float* w_eff,
                          const float* b_eff, float* h, void* stream);
/* dx = dh w_eff   (dh already masked by the ReLU). */
int riqn_noisy_linear_dgrad(long rows, int in_features, int out_features, const float* dh, const float* w_eff,
                            float* dx, void* stream);
/* grad_weight_mu += dh^T x ; grad_weight_sigma += (dh^T x) * weight_epsilon ; bias grads likewise.
 * db_scratch: out_features floats. */
int riqn_noisy_linear_wgrad(long rows, int in_features, int out_features, const float* dh, const float* x,
                            const float* weight_epsilon, const float* bias_epsilon, float* db_scratch,
                            float* grad_weight_mu, float* grad_weight_sigma, float* grad_bias_mu,
                            float* grad_bias_sigma, void* stream);

/* Bias half of the above alone (used when the weight half runs on the tensor cores).  dh == NULL: db_scratch already holds
 * the column sums of dh (riqn_dueling_bwd_bf16). */
int riqn_noisy_bias_grad(long rows, int out_features, const float* dh, const float* bias_epsilon, float* db_scratch,
                         float* grad_bias_mu, float* grad_bias_sigma, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Quantile embedding                                      replaces rainbowiqn/model.py:136-151
 * ---------------------------------------------------------------------------------------------- */
/* cosv[r',i] = cos(fl(fl(i+1)*fl(pi)) * tau[q*batch+b]);  x[r',:] = feat[b,:] * relu(cosv[r',:] iqn_w^T + iqn_b),
 * r' = b*num_quantiles + q (sample-major output rows, quantile-major tau).
 * tau (rows), feat (batch, feat_dim), iqn_w (feat_dim, embed_dim); cosv (rows, embed_dim) and
 * x (rows, feat_dim) are outputs, rows = batch * num_quantiles. */
int riqn_quantile_embed_fwd(int batch, int num_quantiles, int embed_dim, int feat_dim, const float* tau,
                            const float* feat, const float* iqn_w, const float* iqn_b, float* cosv, float* x,
                            void* stream);
/* Given dL/dx in dx_inout (overwritten with dL/d(pre-activation of iqn_fc)): dfeat (batch, feat_dim) is
 * overwritten; grad_iqn_w / grad_iqn_b are accumulated into. */
int riqn_quantile_embed_bwd(int batch, int num_quantiles, int embed_dim, int feat_dim, const float* x,
                            const float* feat, const float* cosv, float* dx_inout, float* dfeat, float* grad_iqn_w,
                            float* grad_iqn_b, void* stream);

/* Tensor-core variants.  Forward: the tcgen05 GEMM's epilogue applies relu / bias / the Hadamard with feat and writes
 * the bf16 operand images of x directly: x_hi, x_lo (rows, feat_dim) for the NoisyLinear product, x_hi_t / x_lo_t
 * (feat_dim, rows) for its weight gradient in the cross-check arithmetic modes (each may be NULL; the transposed images
 * are split from x32 by a second launch and therefore need x32 != NULL); x32 (may be NULL) is the fp32 matrix.  cos_hi / cos_lo
 * (rows, embed_dim) and cos_t_hi (embed_dim, rows; may be NULL) are outputs too.  cos_lo == NULL selects the
 * single-bf16 product.  iqn_w_hi / iqn_w_lo: bf16 images of iqn_fc.weight (riqn_split_bf16). */
int riqn_quantile_embed_fwd_tc(int batch, int num_quantiles, int embed_dim, int feat_dim, const float* tau,
                               const float* feat, const void* iqn_w_hi, const void* iqn_w_lo, const float* iqn_b,
                               void* cos_hi, void* cos_lo, void* cos_t_hi, float* x32, void* x_hi, void* x_lo, void* x_hi_t,
                               void* x_lo_t, int x_fp16, void* stream);
/* x_fp16 != 0: x_hi = fp16(x), the operand of the single-pass fp16 head product (same tensor-core rate as bf16, 11-bit
 * significand), and x_lo (or NULL) = bf16(x), the operand of the bf16 backward; x_hi_t / x_lo_t must be NULL. */
/* Backward on bf16 operands (rows % 8 == 0): dx (rows, feat_dim) from the head dgrad, fp32 or (dx_is_bf16 != 0) bf16;
 * x_lo may be NULL (x = x_hi); cos_hi (rows, embed_dim) bf16 row-major (the forward's image); dpre (rows, feat_dim) bf16
 * workspace; dfeat overwritten; grad_iqn_w / grad_iqn_b accumulated. */
int riqn_quantile_embed_bwd_tc(int batch, int num_quantiles, int embed_dim, int feat_dim, const void* x_hi, const void* x_lo,
                               const float* feat, const void* cos_hi, const void* dx, int dx_is_bf16, void* dpre,
                               float* dfeat, float* grad_iqn_w, float* grad_iqn_b, void* stream);

/* ------------------------------------------------------------------------------------------------
 * z-layers + dueling aggregation                          replaces rainbowiqn/model.py:153-156
 * ---------------------------------------------------------------------------------------------- */
/* Domain of the three dueling entry points: hidden in {128, 256, ..., 1024} (a multiple of 128), 1 <= A <= 31, and the
 * shared memory of the kernel the call selects within 227 KB; anything else returns cudaErrorInvalidValue before a launch.
 * h (rows, 2*hidden) = [value-stream hidden | advantage-stream hidden]; wz (1+A, hidden) = effective
 * weights of fcnoisy_z_v (row 0) and fcnoisy_z_a; bz (1+A).  q (rows, A) = v + a - mean_a a. */
int riqn_dueling_fwd(long rows, int batch, int hidden, int action_space, const float* h, const float* wz,
                     const float* bz, float* q, void* stream);
/* Backward for the gathered action: dq[r, actions[b]] = dtheta[r] * gscale[b].  Writes dh (rows, 2*hidden),
 * already masked by h > 0, and dz (rows, 32) = [dv, da_0.., 0..] for riqn_z_wgrad; dz_bf16 (may be NULL) is its bf16
 * image (rows, 32) for riqn_z_wgrad_tc. */
int riqn_dueling_bwd(long rows, int batch, int hidden, int action_space, const float* h, const float* wz,
                     const float* dtheta, const float* gscale, float gscale_mul, const long long* actions, float* dh,
                     float* dz, void* dz_bf16, void* stream);
/* (gscale_mul multiplies gscale[b]: the learner passes the IS weights and 1/B, learner.py:23's .mean(), without an extra
 * elementwise launch) */
/* Same backward for bf16 tensor-core consumers (rows % 8 == 0): instead of the fp32 dh it writes dh_hi (rows, 2*hidden)
 * as bf16 (and its transpose dh_hi_t (2*hidden, rows) if non-NULL), dh_colsum (2*hidden) = the fp32 column sums of dh
 * (zeroed here; pass it to riqn_noisy_bias_grad with dh == NULL) and dz_bf16 (rows, 32), if non-NULL, the bf16 image of
 * dz for riqn_z_wgrad_tc.  Only the sign of h matters here (ReLU mask): h_bf16 (rows, 2*hidden), if non-NULL, is read
 * instead of h.  The transposed image needs a 32 x 2*hidden bf16 tile (128*hidden bytes) beside the
 * ((1+A)*hidden + 3*hidden) floats of the weights and sums; where that exceeds 227 KB (e.g. hidden 1024 with A = 24) a
 * non-NULL dh_hi_t is refused. */
int riqn_dueling_bwd_bf16(long rows, int batch, int hidden, int action_space, const float* h, const void* h_bf16,
                          const float* wz,
                          const float* dtheta, const float* gscale, float gscale_mul, const long long* actions, void* dh_hi,
                          void* dh_hi_t,
                          float* dh_colsum, float* dz, void* dz_bf16, void* stream);
/* Parameter gradients of the two z-layers (accumulated): dwz_scratch 32*2*hidden floats, dbz_scratch 32. */
/* Same with the reduction dz^T h on the tensor cores, straight from the row-major bf16 images dz_bf16 (rows, 32) and
 * h_bf16 (rows, 2*hidden) (rows % 8 == 0). */
int riqn_z_wgrad_tc(long rows, int hidden, int action_space, const void* dz_bf16, const void* h_bf16, const float* dz,
                    float* dwz_scratch, float* dbz_scratch, const float* eps_w_zv, const float* eps_b_zv,
                    const float* eps_w_za, const float* eps_b_za, float* g_mu_zv, float* g_sig_zv, float* g_bmu_zv,
                    float* g_bsig_zv, float* g_mu_za, float* g_sig_za, float* g_bmu_za, float* g_bsig_za, void* stream);
int riqn_z_wgrad(long rows, int hidden, int action_space, const float* dz, const float* h, float* dwz_scratch,
                 float* dbz_scratch, const float* eps_w_zv, const float* eps_b_zv, const float* eps_w_za,
                 const float* eps_b_za, float* g_mu_zv, float* g_sig_zv, float* g_bmu_zv, float* g_bsig_zv,
                 float* g_mu_za, float* g_sig_za, float* g_bmu_za, float* g_bsig_za, void* stream);

/* ------------------------------------------------------------------------------------------------
 * IQN loss                                     replaces rainbowiqn/compute_loss_iqn.py:216-358
 * ---------------------------------------------------------------------------------------------- */
/* a_star[b] = argmax_a mean_k q[k*batch+b, a]            (compute_loss_iqn.py:238-245) */
int riqn_argmax_mean(int batch, int num_quantiles, int action_space, const float* q, long long* a_star, void* stream);
/* Fused n-step target + pairwise quantile-Huber loss and its gradient (compute_loss_iqn.py:262-357):
 *   target[b,j] = returns[b] + gamma_n*nonterminals[b]*q_target[j*batch+b, a_star[b]]
 *   theta[b,i]  = q_online[i*batch+b, actions[b]]
 *   loss[b]     = mean_j sum_i |tau[i*batch+b] - 1{d<0}| huber_kappa(d)/kappa ,  d = target_j - theta_i
 *   dtheta[i*batch+b] = d loss[b] / d theta[b,i]
 * theta_out (batch, n_tau) / target_out (batch, n_tau_prime) are optional debug outputs (may be NULL). */
int riqn_iqn_loss_fwd_bwd(int batch, int n_tau, int n_tau_prime, int action_space, const float* q_online,
                          const float* q_target, const float* tau, const long long* actions, const long long* a_star,
                          const float* returns, const float* nonterminals, float gamma_n, float kappa, float* loss,
                          float* dtheta, float* theta_out, float* target_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Rainbow-only (C51) head and loss            replaces rainbowiqn/model.py:120-129, rainbowiqn/agent.py:77-141
 * ---------------------------------------------------------------------------------------------- */
/* zv (batch, atoms), za (batch, A*atoms) -> q = v + a - mean_a a; p / logp (batch, A, atoms) = (log_)softmax over
 * atoms (either may be NULL); a_star (may be NULL) = argmax_a sum_j support[j] p[b,a,j]  (agent.py:92-99). */
int riqn_c51_head_fwd(int batch, int action_space, int atoms, const float* zv, const float* za, const float* support,
                      float* p, float* logp, long long* a_star, void* stream);
/* Bellman projection of p_target[b, a_star[b], :] onto the support (agent.py:104-133, incl. the l == u fix),
 * loss[b] = -sum_j m_j logp_online[b, actions[b], j] (agent.py:141) and dq (batch, atoms) = dloss/dq[b, actions[b], :].
 * m_out (batch, atoms) optional. */
int riqn_c51_loss_fwd_bwd(int batch, int action_space, int atoms, const float* logp_online, const float* p_target,
                          const long long* actions, const long long* a_star, const float* returns,
                          const float* nonterminals, const float* support, float gamma_n, float v_min, float v_max,
                          float delta_z, float* loss, float* dq, float* m_out, void* stream);
/* dzv (batch, atoms), dza (batch, A*atoms) from dq scaled by gscale[b] (dueling backward). */
int riqn_c51_head_bwd(int batch, int action_space, int atoms, const float* dq, const float* gscale, float gscale_mul,
                      const long long* actions, float* dzv, float* dza, void* stream);
/* n floats <- 0 (the gradient arena's zero_grad, learner.py:22): cudaMemsetAsync on the caller's stream. */
int riqn_zero_f32(float* p, long n, void* stream);
/* grad[i] = 0 where act[i] <= 0. */
int riqn_relu_mask(long n, const float* act, float* grad, void* stream);
/* Strided fp32 linear-layer helpers for the small z-layers: y = x w^T + bias (optional ReLU); dx = dy w;
 * grad_mu += dy^T x, grad_sigma += (dy^T x) * weight_epsilon. */
int riqn_linear_fwd_ld(long rows, int in_features, int out_features, const float* x, long ldx, const float* w,
                       const float* bias, float* y, long ldy, int relu, void* stream);
int riqn_linear_dgrad_ld(long rows, int in_features, int out_features, const float* dy, long lddy, const float* w,
                         float* dx, long lddx, void* stream);
int riqn_noisy_wgrad_ld(long rows, int in_features, int out_features, const float* dy, long lddy, const float* x, long ldx,
                        const float* weight_epsilon, float* grad_mu, float* grad_sigma, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Optimiser                              replaces torch.optim.Adam.step, agent.py:43 / learner.py:24
 * ---------------------------------------------------------------------------------------------- */
/* One Adam step over a flat arena of n fp32 parameters; `step` is the 1-based step count; grads are
 * multiplied by grad_scale first (1/world_size after a gradient all-reduce). */
int riqn_adam_step(long n, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int step, float lr,
                   float beta1, float beta2, float eps, float grad_scale, const riqn_dyn_state* dyn, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Prioritized replay: sum-tree          replaces RedisSegmentTree / ReplayRedisMemory, redis_memory.py
 * tree: 2*capacity-1 float64 nodes in HBM, leaf of data index d at d + capacity - 1.
 * ---------------------------------------------------------------------------------------------- */
/* Stratified sample values, one per segment of total/n, shuffled (redis_memory.py:276-287). n <= 12000. */
int riqn_sumtree_stratified(int n, unsigned long long seed, unsigned long long stream_id, const double* tree,
                            double* values, const riqn_dyn_state* dyn, void* stream);
/* Descent (_retrieve_multiple_values :205-229) + transform_to_valid_tree_indexes (:242-264) + priority
 * read (:315-321).  index_actor: per-actor write heads (int64).  Bit-exact with the reference. */
int riqn_sumtree_sample(int n, long capacity, int actor_capacity, const double* tree, const double* values,
                        const long long* index_actor, int history, int n_step, long long* tree_idx,
                        long long* data_idx, double* priorities, void* stream);
/* Importance-sampling weights (sample_byte :465-475); n_nonpositive (device int, may be NULL) counts the
 * priorities <= 0 that were replaced by 1/capacity (:446-456). */
int riqn_sumtree_is_weights(int n, const double* tree, const double* priorities, double current_capacity,
                            double priority_weight, double* w64, float* w32, int* n_nonpositive,
                            const riqn_dyn_state* dyn, void* stream);
/* update_priorities / update_multiple_value / _propagate_multiple_values (:557-573,139-151,94-105).
 * apply_pow != 0: new = np.power(loss, float32(priority_exponent)) first.  new_priorities (n floats) and
 * diff_scratch (n doubles) are outputs/workspace; *max_priority (device double) is raised if needed.
 * n <= 4096.  The tree arithmetic is bit-exact with the reference (including duplicated indices) given the
 * float32 priorities; the power itself is the correctly rounded float32 value, which numpy/libm powf only
 * approximates (<= 1 ulp apart, platform dependent). */
int riqn_sumtree_update(int n, long capacity, double* tree, const long long* tree_idx, const float* loss,
                        float priority_exponent, int apply_pow, float* new_priorities, double* diff_scratch,
                        double* max_priority, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Prioritized replay: frame store            replaces the Redis hashes "transitions<i>" (:184-193)
 * ---------------------------------------------------------------------------------------------- */
/* Frame half of append_actor_buffer (:159-199): n consecutive transitions of one actor into its ring. */
int riqn_replay_append(int n, int actor_capacity, int id_actor, int start, const unsigned char* frames,
                       const int* timestep, const int* action, const float* reward, const unsigned char* nonterminal,
                       unsigned char* s_frames, int* s_timestep, int* s_action, float* s_reward,
                       unsigned char* s_nonterminal, void* stream);
/* Transition assembly (:347-369, :479-541): window (batch, history+n_step, 84, 84) uint8 with blank frames
 * across episode boundaries; states = window[:, :history], next_states = window[:, n_step:].
 * gamma_pow: n_step doubles, discount**k. */
int riqn_frame_gather(int batch, int actor_capacity, int history, int n_step, const long long* data_idx,
                      const unsigned char* s_frames, const int* s_timestep, const int* s_action, const float* s_reward,
                      const unsigned char* s_nonterminal, const double* gamma_pow, unsigned char* window,
                      long long* actions, float* returns, float* nonterminals, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Tensor-core building blocks of the NoisyLinear products (tcgen05.mma + TMA; csrc/gemm_tc.cu).
 * ---------------------------------------------------------------------------------------------- */
/* fp32 (rows, cols) -> bf16 hi and lo = bf16(x - hi) (either may be NULL); hi_t / lo_t (may be NULL) receive the
 * transposed (cols, rows) copies the weight-gradient product consumes. */
int riqn_split_bf16(long rows, int cols, const float* src, void* hi, void* lo, void* hi_t, void* lo_t, int fp16, void* stream);
/* fp16 != 0: hi = fp16(x) and lo (or NULL) = bf16(x) instead (hi_t / lo_t must be NULL). */
/* Several small splits in ONE launch (the per-step refresh of the noise-free weight images): for each job
 * out[r, c] = src[r, perm ? perm[c] : c] / div (div == 1: unscaled), written as hi / lo = bf16(x - hi) (lo, hi_t may be
 * NULL; hi_t is the transposed (cols, rows) hi image).  Same values as riqn_split_bf16 / riqn_split_bf16_scaled on a
 * column-permuted source.  jobs: HOST array of n_jobs <= 12. */
typedef struct riqn_split_job {
  const float* src;     /* (rows, cols) fp32 */
  const int* perm;      /* cols ints or NULL */
  int rows, cols;
  float div;
  void* hi;
  void* lo;
  void* hi_t;
} riqn_split_job;
int riqn_split_bf16_multi(int n_jobs, const riqn_split_job* jobs, void* stream);
/* C (+)= A B^T with A (M,K), B (N,K) row-major bf16, K % 8 == 0, fp32 accumulation in TMEM.  a_lo/b_lo non-NULL
 * selects the split-bf16 x3 (fp32-faithful) product.  epilogue: 0 store, 1 relu(acc+bias[n]), 2 atomicAdd into C,
 * 3 atomicAdd into C and acc*eps[m,n] into out2 (NoisyLinear dmu / dsigma).  split_k > 1 needs 2 or 3.
 * c_t_bf16 / c_bf16 (may be NULL; epilogue 1 only): bf16 transposed (N, M) / row-major (M, N) images of the result. */
int riqn_gemm_bf16_tc(int M, int N, int K, const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo,
                      float* c, long ldc, int epilogue, const float* bias, float* out2, const float* eps, int split_k,
                      void* c_t_bf16, void* c_bf16, int fmt, void* stream);
/* fmt (both GEMM entry points): 0 = both operand images hold bf16, 3 = both hold fp16 (single-pass: a_lo == b_lo == NULL).
 * 1 / 2 (mixed) are rejected: tcgen05 kind::f16 raises an illegal-instruction fault when A and B formats differ. */
/* Products whose B operand is (K, N) row-major bf16 (MN-major tcgen05 operand, N % 8 == 0) -- no transposed copies:
 *   a_is_km != 0: C (+)= A^T B with A (K, M) row-major (M % 8 == 0): the reduction runs over the ROWS of both, i.e. a
 *                 weight gradient dW = dY^T X straight from the row-major activations;
 *   a_is_km == 0: C (+)= A B with A (M, K) row-major (K % 8 == 0): a data gradient dX = dY W from the untransposed W.
 * epilogue 0 / 2 / 3 as above (2, 3 scale the accumulator by alpha); single-bf16 product.  c_bf16 (may be NULL; epilogue 0,
 * N % 32 == 0): write the result as bf16 (M, N) there INSTEAD of fp32 into c. */
int riqn_gemm_bf16_tc_mn(int M, int N, int K, const void* a, const void* b_kn, int a_is_km, float* c, long ldc, int epilogue,
                         float* out2, const float* eps, float alpha, int split_k, void* c_bf16, int fmt, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Test hook: plain strided fp32 product C[m,n] = sum_k A[m*sAm + k*sAk] * B[n*sBn + k*sBk].
 * ---------------------------------------------------------------------------------------------- */
int riqn_gemm_f32(int M, int N, int K, const float* A, long sAm, long sAk, const float* B, long sBn, long sBk,
                  float* C, long ldc, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RIQN_B200_H */
