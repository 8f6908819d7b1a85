/*
 * lsnf.h -- C ABI of the B200-native short-run Langevin posterior-inference path.
 *
 * The reference (jianwen-xie/Latent-Space-Normalizing-Flow) is pure Python and has no FFI; the entry
 * points below are what a binding for its hot path would call, one per reference call site
 * (paths relative to the reference tree):
 *
 *   lsnf_generator_forward   <- netG(z)                                   train.py:312, model.py:156-157
 *   lsnf_generator_dgrad     <- torch.autograd.grad(g_log_lkhd, z)        train.py:313-314
 *   lsnf_flow_forward        <- netF(z, objective) + log-prior + its grad train.py:316-323, model.py:473-483
 *   lsnf_flow_inverse        <- netF(z, objective, reverse=True)          train.py:434, :569; model.py:484-498
 *   lsnf_langevin_update     <- z update + noise + diagnostics            train.py:324-329
 *   lsnf_langevin_run        <- sample_langevin_post_z_with_flow          train.py:307-335, :602-634
 *   lsnf_sample_prior        <- sample_x(): eps -> F^-1 -> G -> [0,1]     train.py:565-576, :433-437, :472-478
 *   lsnf_generator_param_grads <- loss_g = mse(G(z_k), x) / B; loss_g.backward()  train.py:390-394
 *   lsnf_flow_param_grads    <- loss_f = -ll.mean(); loss_f.backward()    train.py:403-411, model.py:182
 *   lsnf_adam_step           <- optG.step() / optF.step() (torch.optim.Adam) train.py:294-295, :398, :415
 *   lsnf_*_masked            <- the same three generator-loss entry points with a per-pixel likelihood weight
 *   lsnf_*_measured          <- the same generator-loss entry points and AIS with y = A vec(G(z)) + noise in place of x
 *   lsnf_generator_vjp       <- backward of netG(z) for any loss (torch.autograd through lsnf_b200.kernel_autograd)
 *   lsnf_flow_vjp            <- backward of netF(z, objective) for any loss (same)
 *   lsnf_pack_*              <- parameters of _netG / _netF               model.py:48-157, :460-498
 *
 * Conventions: every function returns 0 on success and a negative lsnf_status otherwise;
 * lsnf_last_error() returns a thread-local message for the last failure.  All tensor arguments are raw
 * DEVICE pointers to contiguous fp32 data in the reference's own layouts (NCHW images, [B,nz] latents,
 * [C_in,C_out,k,k] ConvTranspose2d weights) unless stated otherwise.  `stream` is a cudaStream_t; all work
 * is enqueued on it and no call synchronises the device.  The caller owns every buffer, including the
 * workspace; inputs are never modified.  A plan is tied to one device (the current device of lsnf_plan_bind) and one
 * batch size and is not thread-safe; distinct plans -- on the same or on different devices of one process -- may be
 * used concurrently from distinct threads / streams (per-device kernel attributes are set up under a lock at bind
 * time, nothing on the launch path is process-global).
 *
 * There is no CPU fallback: on a machine without a CUDA device every compute entry point fails with
 * LSNF_ERR_CUDA.
 */
#ifndef LSNF_H_
#define LSNF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LSNF_ABI_VERSION 1

typedef struct lsnf_plan lsnf_plan;
typedef void* lsnf_stream; /* cudaStream_t */

typedef enum lsnf_status {
  LSNF_OK = 0,
  LSNF_ERR_INVALID = -1,     /* bad argument / unsupported configuration */
  LSNF_ERR_CUDA = -2,        /* CUDA runtime or driver error (message has the detail) */
  LSNF_ERR_STATE = -3,       /* call order violated (e.g. weights not packed, workspace not bound) */
  LSNF_ERR_UNSUPPORTED = -4  /* configuration the reference itself rejects or never implemented */
} lsnf_status;

/* generator architectures of model.py:52-151 (args.dataset) */
typedef enum lsnf_arch {
  LSNF_ARCH_NONE = -1,        /* flow prior only (no generator stages) */
  LSNF_ARCH_SVHN = 0,         /* model.py:56-71  */
  LSNF_ARCH_CIFAR10 = 1,      /* model.py:77-92  */
  LSNF_ARCH_CELEBA_CROP = 2,  /* model.py:98-117 */
  LSNF_ARCH_CELEBA_HQ256 = 3  /* model.py:123-151 */
} lsnf_arch;

typedef enum lsnf_gemm_impl {
  LSNF_GEMM_TCGEN05 = 0, /* product path: TMA-fed tcgen05 tensor-core tiles on 16-bit hi|lo operand pairs (value =
                            hi + lo): fp16 pairs with power-of-two-scaled weights in the forward pass, bf16 pairs in the
                            data gradient; three MMAs per K step (hi*hi + hi*lo + lo*hi), fp32 accumulation in TMEM */
  LSNF_GEMM_SIMT = 1     /* debugging twin on CUDA cores over the same buffers (tests only) */
} lsnf_gemm_impl;

typedef struct lsnf_config {
  int32_t arch;          /* lsnf_arch */
  int32_t batch;         /* samples held by this plan (this rank's shard) */
  int32_t nz;            /* --nz, a multiple of 4 in 4..256 (even: model.py:383) */
  int32_t ngf;           /* --ngf */
  int32_t nc;            /* --nc (3) */
  int32_t f_depth;       /* --f_depth, 1..32 */
  int32_t f_width;       /* --f_width, a multiple of 4 in 4..256.  Accepted flow range: one step of the fused flow kernels
                            must fit the 227 KB of shared memory of one CTA at one sample per CTA -- its largest matrix
                            (f_width^2 floats, or nz^2 with f_flow_permutation 2) plus f_depth * (2 f_width + nz) floats of
                            activations plus ~3 KB.  So f_width <= 232 (192 at nz 100, f_depth 32); with
                            f_flow_permutation 2 nz <= 228 (224 at f_width 64, f_depth 5; 204 at f_depth 32); the shuffle
                            permutation takes every nz up to 256 (f_width <= 196 there).  lsnf_plan_create refuses a
                            configuration outside it with LSNF_ERR_INVALID.  A configuration it accepts runs at every batch:
                            the kernels take fewer samples per CTA where the preferred number does not fit. */
  int32_t f_permutation; /* --f_flow_permutation: 2 = invertible 1x1 (default), 1 = fixed shuffle */
  int32_t f_coupling;    /* --f_flow_coupling: 1 = affine (default), 0 = additive */
  float leak;            /* --g_activation_leak of the LeakyReLU (0.2) */
  int32_t gemm_impl;     /* lsnf_gemm_impl */
  int32_t bwd_passes;    /* tensor-core passes of the data-gradient stages: 0 or 3 (default) = bf16 hi|lo split, 3 MMAs
                            per K step, 16 significant bits per operand: z_T at the reference's own fp32 noise floor.
                            1 = explicit opt-in to a single fp16 pass (11-bit significands, gradient good to ~2e-4): a
                            reduced-precision mode, measured margins in DESIGN.md section 4.1 */
  int32_t train;         /* != 0: the workspace also holds the buffers of lsnf_generator_param_grads (transposed
                            operands and split-K partials of the weight-gradient GEMMs); 0 for inference-only plans */
  int32_t meas_rows;     /* m > 0: rows of a dense linear measurement operator A [m, nc*H*W] (lsnf_*_measured below);
                            the workspace then also holds A packed twice (about 8 m n bytes, n = nc*H*W) plus the
                            split-K partials of its two GEMMs.  0 = no operator: the plan is exactly that of a config
                            without this field */
  int32_t reserved[2];
} lsnf_config;

/* number of per-step flow parameter pointers expected by lsnf_pack_flow_weights, in this order:
 * actnorm.b, actnorm.logs, invertible_1x1_conv.w, f.fc_1.w, f.fc_1.actnorm.b, f.fc_1.actnorm.logs,
 * f.fc_2.w, f.fc_2.actnorm.b, f.fc_2.actnorm.logs, f.fc_zeros.w, f.fc_zeros.b, f.fc_zeros.logs
 * (state_dict names under revnet2d_s.0.revnet2d_step_s.<i>., model.py:367-387) */
#define LSNF_FLOW_PTRS_PER_STEP 12

int lsnf_abi_version(void);
const char* lsnf_last_error(void);

/* ---- plan ------------------------------------------------------------------------------------------- */
/* Pure host work: validates the configuration, lays out the workspace and builds the stage tables. */
int lsnf_plan_create(const lsnf_config* cfg, lsnf_plan** out);
void lsnf_plan_destroy(lsnf_plan* plan);
size_t lsnf_workspace_bytes(const lsnf_plan* plan);
/* `workspace` is device memory of at least lsnf_workspace_bytes(), 1024-byte aligned, zero-initialised by
 * the caller once.  Encodes the TMA descriptors that point into it. */
int lsnf_plan_bind(lsnf_plan* plan, void* workspace, size_t bytes);

/* ---- parameters ------------------------------------------------------------------------------------- */
/* weights[i]: [C_in,C_out,k,k], biases[i]: [C_out] of the i-th ConvTranspose2d (gen.{3i}.weight|bias).
 * Re-packs into the 16-bit hi|lo K-major operand layouts of every stage: fp16 pairs times a per-layer power of two for
 * the forward stages, bf16 pairs for the data-gradient stages (single fp16 halves when bwd_passes == 1). */
int lsnf_pack_generator_weights(lsnf_plan* plan, const float* const* weights, const float* const* biases,
                                int32_t n_layers, lsnf_stream stream);
/* params: f_depth * LSNF_FLOW_PTRS_PER_STEP device pointers (order above).  For f_permutation == 1 the
 * third pointer of each step is ignored and perm / perm_inverse hold f_depth device pointers to int32[nz].
 * log_abs_det: DEVICE array [f_depth] of log|det W_i| evaluated in fp64 as model.py:182 does (ignored for shuffle);
 * w_inverse: f_depth device pointers to [nz,nz] inverses (model.py:193), or NULL if lsnf_flow_inverse is
 * not going to be called.  Both are hoisted out of the Langevin loop: parameters are constant during it.
 * log_abs_det == NULL (f_permutation 2, nz <= 160): the library evaluates both itself in one launch (fp64 Gauss-Jordan
 * with partial pivoting, one CTA per step) and w_inverse is ignored. */
int lsnf_pack_flow_weights(lsnf_plan* plan, const float* const* params, const int32_t* const* perm,
                           const int32_t* const* perm_inverse, const float* log_abs_det,
                           const float* const* w_inverse, lsnf_stream stream);

/* ---- stages of one Langevin step -------------------------------------------------------------------- */
/* z [B,nz] -> x_hat [B,nc,H,W]; keeps the activations in the workspace for lsnf_generator_dgrad. */
int lsnf_generator_forward(lsnf_plan* plan, const float* z, float* x_hat, lsnf_stream stream);
/* grad_z [B,nz] = d/dz [ 1/(2 sigma^2) * sum (G(z) - x)^2 ] for the z of the last lsnf_generator_forward. */
int lsnf_generator_dgrad(lsnf_plan* plan, const float* x, float sigma, float* grad_z, lsnf_stream stream);
/* z [B,nz] -> z_out [B,nz], logdet [B], logp [B] (= sum(-z_out^2/2) + log(2 pi) + logdet, train.py:317-319),
 * grad_z [B,nz] = d/dz [ -sum_b logp_b ] (train.py:320-323).  Any output pointer may be NULL. */
int lsnf_flow_forward(lsnf_plan* plan, const float* z, float* z_out, float* logdet, float* logp,
                      float* grad_z, lsnf_stream stream);
/* eps [B,nz] -> z [B,nz] = F^-1(eps); neg_objective [B] (nullable) is what the reference returns with
 * return_obj=True for objective=0 (model.py:498).  Does not modify eps (the reference does, model.py:436). */
int lsnf_flow_inverse(lsnf_plan* plan, const float* eps, float* z, float* neg_objective, lsnf_stream stream);
/* z <- z - s^2/2 (grad_g + grad_f) [+ s * noise]  (train.py:324-326).  noise = eps [B,nz] when eps != NULL,
 * else (with_noise != 0) Philox4x32-10 keyed by (seed, sample_offset + b, step), else none.
 * gnorms (nullable, device float[2]) receives mean_b |grad_g_b|_2 and mean_b |grad_f_b|_2 (train.py:328-329). */
int lsnf_langevin_update(lsnf_plan* plan, float* z, const float* grad_g, const float* grad_f, float step_size,
                         const float* eps, int32_t with_noise, uint64_t seed, uint64_t sample_offset,
                         uint32_t step, float* gnorms, lsnf_stream stream);

/* ---- the whole loop --------------------------------------------------------------------------------- */
/* sample_langevin_post_z_with_flow: z0 [B,nz], x [B,nc,H,W] -> z_out [B,nz] after `steps` iterations and
 * gnorms[2] (device) from the last one.  eps: [steps,B,nz] injected noise or NULL; see lsnf_langevin_update.
 * z0 and z_out may alias. */
int lsnf_langevin_run(lsnf_plan* plan, const float* z0, const float* x, int32_t steps, float step_size,
                      float sigma, int32_t with_noise, const float* eps, uint64_t seed, uint64_t sample_offset,
                      float* z_out, float* gnorms, lsnf_stream stream);
/* Prior sampling, train.py:565-576 (also :433-437, :472-478): eps [B,nz] ~ N(0,I) -> z = F^-1(eps) -> x = G(z)
 * [B,nc,H,W]; with to_unit_range != 0 the store applies to_range_0_1 and the clamp of train.py:573,
 * x = clamp((G(z) + 1) / 2, 0, 1).  z (nullable) receives the latents [B,nz].  eps is not modified.  Needs flow
 * weights packed with w_inverse. */
int lsnf_sample_prior(lsnf_plan* plan, const float* eps, float* x, float* z, int32_t to_unit_range, lsnf_stream stream);
/* ---- parameter updates (training mode) ---------------------------------------------------------------- */
/* Generator parameter gradients of loss_g = (1 / global_batch) * sum (G(z) - x)^2 over this plan's batch
 * (train.py:390-394): z [B,nz] (the inferred latents z_k), x [B,nc,H,W].  Needs a plan created with
 * lsnf_config.train != 0.  grads: device buffer of lsnf_generator_grad_floats() floats; layer l's weight gradient
 * occupies [offsets[2l], +sizes[2l]) in the parameter's own [C_in,C_out,k,k] layout and its bias gradient
 * [offsets[2l+1], +sizes[2l+1]) (lsnf_generator_grad_layout).  With several ranks each passes its shard and the GLOBAL
 * batch size; the buffers are then summed (one all-reduce).  loss (nullable, device float): this rank's share of
 * loss_g.  Runs the forward pass, the data-gradient chain and one weight-gradient tap-GEMM per layer; deterministic.
 * part: -1 = everything; -2 = only the forward pass, the loss and the data-gradient chain; l >= 0 = only layer l's
 * weight and bias gradient (after a -2 call on the same inputs) -- so that a data-parallel caller can start the
 * all-reduce of a layer's gradients while the next layer's are being computed. */
size_t lsnf_generator_grad_floats(const lsnf_plan* plan);
int lsnf_generator_grad_layout(const lsnf_plan* plan, int64_t* offsets, int64_t* sizes);
int lsnf_generator_param_grads(lsnf_plan* plan, const float* z, const float* x, int32_t global_batch, float* grads,
                               float* loss, int32_t part, lsnf_stream stream);
/* Flow parameter gradients of loss_f = -(1 / global_batch) * sum_b ll_b(z_b) over this plan's batch z [B,nz]
 * (train.py:403-411; ll_b = log p(z_b) of lsnf_flow_forward).  grads: device buffer of lsnf_flow_grad_floats()
 * floats, ZERO-INITIALISED by the caller once (alignment padding is never written); tensor (step, i) -- i in the order
 * of LSNF_FLOW_PTRS_PER_STEP -- occupies [offsets[step*12+i], +sizes[step*12+i]) in its natural row-major shape
 * (lsnf_flow_grad_layout).  With several ranks each passes its shard and the GLOBAL batch size; the buffers are then
 * summed (one all-reduce).  d log|det W| / dW = W^-T (model.py:182) uses the W^-1 given to lsnf_pack_flow_weights.
 * loss (nullable, device float): this rank's share of loss_f.  Deterministic (fixed summation order). */
size_t lsnf_flow_grad_floats(const lsnf_plan* plan);
int lsnf_flow_grad_layout(const lsnf_plan* plan, int64_t* offsets, int64_t* sizes);
int lsnf_flow_param_grads(lsnf_plan* plan, const float* z, int32_t global_batch, float* grads, float* loss,
                          lsnf_stream stream);
/* Fused multi-tensor Adam, semantics of torch.optim.Adam (no amsgrad; weight_decay is added to the gradient):
 * for each of n_tensors fp32 device tensors  g' = g * (*grad_scale) + weight_decay * p;  m = lerp(m, g', 1-beta1);
 * v = beta2 v + (1-beta2) g'^2;  p -= lr / (1-beta1^step) * m / (sqrt(v) / sqrt(1-beta2^step) + eps).
 * `step` is the 1-based count AFTER this update.  grad_scale: nullable device scalar (gradient-norm clipping).
 * grad_kk / grad_inner (nullable): gradient i is stored tap-major [kk][outer][inner] for a parameter laid out
 * [outer][inner][kk] (ConvTranspose2d weights); kk <= 1 means same layout as the parameter.  No plan needed. */
/* ---- vector-Jacobian products for any loss (autograd through the kernels) ------------------------------ */
/* dL/dz [B,nz] (nullable) and, on a plan created with train != 0, the parameter gradients (nullable; layout of
 * lsnf_generator_grad_layout, overwritten) of L for upstream grad_x_hat = dL/dx_hat [B,nc,H,W], at the z of the last
 * lsnf_generator_forward on this plan.  Runs the data-gradient chain of lsnf_generator_dgrad and the weight-gradient
 * GEMMs of lsnf_generator_param_grads from the seed grad_x_hat * (1 - x_hat^2), at scale 1.  Needs the 3-pass data
 * gradient: a plan with bwd_passes == 1 returns LSNF_ERR_UNSUPPORTED.  Deterministic. */
int lsnf_generator_vjp(lsnf_plan* plan, const float* grad_x_hat, float* grad_z, float* grads, lsnf_stream stream);

/* ---- masked reconstruction loss (inpainting, occluded pixels, images with missing regions) -------------- */
/* The three calls below are lsnf_langevin_run, lsnf_generator_dgrad and lsnf_generator_param_grads with a nullable
 * `mask`: fp32 [B,nc,H,W], the layout of x, a per-pixel likelihood weight m (1 = observed, 0 = missing, fractions
 * allowed).  mask == NULL is exactly the unmasked call (which is implemented as this call with NULL).
 *   Langevin energy  1/(2 sigma^2) sum m (G(z) - x)^2 - log p(z)     (so m_i = sigma^2 / sigma_i^2 is a per-pixel
 *                                                                      noise precision)
 *   generator loss   loss_g = sum m (G(z) - x)^2 / global_batch      (the flow prior and its update are unchanged)
 * The weight multiplies (G(z) - x) before any other factor, so an all-ones mask reproduces the unmasked results bit
 * for bit.  The gradient norms of lsnf_langevin_run_masked are those of the masked gradient.  Supported weights lie in
 * [0, 1]: the data-gradient tensors are sized for that range (a larger common weight can be folded into sigma).  The
 * library does not read device values, so it does not check this.
 * lsnf_langevin_run_masked: a call that replays a CUDA graph first copies the mask into the workspace (as it does x),
 * so the mask's contents and address may change between calls; masked and unmasked loops never share a graph.
 * lsnf_generator_param_grads_masked: the mask is read by the part -1 and -2 calls only (the forward pass, the loss and
 * the data-gradient chain); a layer's call (part >= 0) ignores it. */
int lsnf_langevin_run_masked(lsnf_plan* plan, const float* z0, const float* x, const float* mask, int32_t steps,
                             float step_size, float sigma, int32_t with_noise, const float* eps, uint64_t seed,
                             uint64_t sample_offset, float* z_out, float* gnorms, lsnf_stream stream);
int lsnf_generator_dgrad_masked(lsnf_plan* plan, const float* x, const float* mask, float sigma, float* grad_z,
                                lsnf_stream stream);
int lsnf_generator_param_grads_masked(lsnf_plan* plan, const float* z, const float* x, const float* mask,
                                      int32_t global_batch, float* grads, float* loss, int32_t part,
                                      lsnf_stream stream);
/* z [B,nz]; upstream grad_z_out [B,nz] and grad_logdet [B] (either nullable = 0) -> grad_z [B,nz] (nullable) and the
 * flow parameter gradients (nullable; layout of lsnf_flow_grad_layout; needs w_inverse for W). Deterministic. */
int lsnf_flow_vjp(lsnf_plan* plan, const float* z, const float* grad_z_out, const float* grad_logdet, float* grad_z,
                  float* grads, lsnf_stream stream);

/* ---- annealed importance sampling (AIS) with Metropolis-adjusted Langevin transitions ------------------ */
/* Estimates log p(x) = log int p(x|z) p(z) dz.  With l(z) = -sum m (G(z) - x)^2 / (2 sigma^2) (m = mask, NULL = 1) and
 * pi_beta(z) ~ p(z) exp(beta l(z)), every chain b runs, for t = 1..steps:
 *   log w += (betas[t] - betas[t-1]) l(z_{t-1})                                  (fp64 accumulator)
 *   z_t = one MALA step on pi_{betas[t]} from z_{t-1}: proposal z' = z - (s^2/2) grad U(z) + s eps, accepted iff
 *         log u < U(z) - U(z') - |z - z' + (s^2/2) grad U(z')|^2 / (2 s^2) + |eps|^2 / 2   (NaN / inf energies reject)
 * with U = -log p - beta l.  Forward AIS (betas 0 -> 1, z0 exact prior samples) gives a stochastic lower bound:
 * log p(x) >= E[log w] + C, C = -1/2 sum_{m_i > 0} log(2 pi sigma^2 / m_i), which the caller adds.  A decreasing
 * schedule started from an exact posterior sample is BDMC's reverse chain, whose -log w bounds from above.  With a
 * constant schedule of ones the call is a Metropolis-adjusted posterior sampler.
 *   z0 [B,nz], x and mask [B,nc,H,W], betas: device array of steps + 1 values in [0, 1] (not checked: the library
 *   does not read device values on the host); steps >= 1; step_size > 0 is the initial step s of every chain; with
 *   target_accept > 0 each chain adapts it after every decision, log s += 0.05 (min(1, alpha) - target_accept), s
 *   clamped to [1e-5, 10]; target_accept <= 0 keeps it fixed.
 *   eps [steps,B,nz] (the t-th proposal's noise) and u [steps,B] (the t-th decision's uniform), both nullable: Philox
 *   keyed by (seed, sample_offset + b, iteration) otherwise.  Injected noise runs eagerly; other calls after a plan's
 *   first replay CUDA graphs of the loop (the schedule, x and mask are copied into the workspace before each replay).
 *   Outputs: z_out [B,nz] the last state, log_w [B] without C, accept_rate [B] accepted / steps.
 * Each proposal is stored rounded to the fp16 hi|lo value the first generator layer reads, so the generator, the
 * flow and the acceptance test all see the same z.  steps transitions take steps + 1 loop iterations. */
int lsnf_ais_run(lsnf_plan* plan, const float* z0, const float* x, const float* mask, const float* betas,
                 int32_t steps, float step_size, float target_accept, float sigma, const float* eps, const float* u,
                 uint64_t seed, uint64_t sample_offset, float* z_out, float* log_w, float* accept_rate,
                 lsnf_stream stream);

/* ---- linear measurements y = A vec(G(z)) + sigma noise (compressed sensing, super-resolution, deblurring) ------- */
/* A plan created with lsnf_config.meas_rows = m > 0 runs the energy
 *   U(z) = |A vec(x_hat) - y|^2 / (2 sigma^2) - log p(z),   x_hat = G(z),
 * with vec the NCHW flattening of x_hat [B,nc,H,W] (n = nc*H*W elements per sample; torch's x.view(B, -1)), A a dense
 * fp32 [m, n] row-major device matrix and y [B, m].  Heteroscedastic noise needs nothing extra: scaling row i of A and
 * of y by sigma / sigma_i gives the same energy.
 * Workspace: A is kept as two K-major 16-bit hi|lo copies, about 8 m n bytes, plus fp32 split-K partials of
 * A x_hat and A^T r (r = A x_hat - y).  A dense operator grows fast with the image: at CelebA-HQ256 (n = 196 608) a
 * 4x-downsampling A (m = n / 16) takes 19 GB.
 * lsnf_pack_measurement: packs A (read once; the caller may free or change it afterwards) into both copies, times one
 *   power of two 2^k computed on the device (max|A| 2^k in [1, 2)).  The 16-bit tensors of the measured path carry
 *   2^k and 2^2k, so they do not depend on the units of A, y and sigma; 2^-2k is undone exactly in fp32.  The call
 *   reads k back and synchronises `stream`.  Pack again after A changes.
 * lsnf_langevin_run_measured, lsnf_generator_dgrad_measured and lsnf_ais_run_measured have the contracts of
 *   lsnf_langevin_run, lsnf_generator_dgrad and lsnf_ais_run (injected noise, Philox keying, gradient norms, graph
 *   replay with y copied into the workspace before each replay; measured and unmeasured loops never share a graph)
 *   with y [B, m] in place of x (and the mask).  For AIS, l(z) = -|A vec(G(z)) - y|^2 / (2 sigma^2) and the caller adds
 *   C = -(m/2) log(2 pi sigma^2).
 * lsnf_generator_param_grads_measured has the contract of lsnf_generator_param_grads (flat gradient layout, part
 *   -1 / -2 / l, loss nullable and this rank's share, GLOBAL batch, deterministic) for the measured loss
 *     loss_g = (1 / global_batch) * sum_b |A vec(G(z_b)) - y_b|^2        (no sigma, as the unmeasured loss_g has none)
 *   on a plan created with train != 0; y [B, m] is read by the part -1 and -2 calls only.  The 16-bit gradient tensors
 *   carry the operator's 2^2k; the weight and bias gradients and the loss undo it in fp32, so scaling A and y by 2^j
 *   scales loss_g and every gradient by exactly 2^2j.  Layer calls (part >= 0) must follow a part -2 call of this
 *   entry point, not of the unmeasured one (and vice versa): LSNF_ERR_STATE otherwise.
 * The four return LSNF_ERR_UNSUPPORTED on a plan with meas_rows == 0 or bwd_passes == 1 (the single-pass data
 * gradient writes an fp16 seed and A^T r has no bounded range), and LSNF_ERR_INVALID until an operator is packed.
 * lsnf_generator_param_grads_measured also returns LSNF_ERR_STATE on a plan without train and LSNF_ERR_UNSUPPORTED on
 * the SIMT path, as lsnf_generator_param_grads_masked does. */
int lsnf_pack_measurement(lsnf_plan* plan, const float* A, lsnf_stream stream);
int lsnf_langevin_run_measured(lsnf_plan* plan, const float* z0, const float* y, int32_t steps, float step_size,
                               float sigma, int32_t with_noise, const float* eps, uint64_t seed, uint64_t sample_offset,
                               float* z_out, float* gnorms, lsnf_stream stream);
int lsnf_generator_dgrad_measured(lsnf_plan* plan, const float* y, float sigma, float* grad_z, lsnf_stream stream);
int lsnf_generator_param_grads_measured(lsnf_plan* plan, const float* z, const float* y, int32_t global_batch,
                                        float* grads, float* loss, int32_t part, lsnf_stream stream);
int lsnf_ais_run_measured(lsnf_plan* plan, const float* z0, const float* y, const float* betas, int32_t steps,
                          float step_size, float target_accept, float sigma, const float* eps, const float* u,
                          uint64_t seed, uint64_t sample_offset, float* z_out, float* log_w, float* accept_rate,
                          lsnf_stream stream);

int lsnf_adam_step(int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                   float* const* exp_avg_sq, const int64_t* sizes, const int32_t* grad_kk, const int32_t* grad_inner,
                   float lr, float beta1, float beta2, float eps, float weight_decay, int64_t step,
                   const float* grad_scale, lsnf_stream stream);

/* Launches generator stage `index` alone (0..L-1 forward, L..2L-1 data gradient, and on a plan with meas_rows > 0
 * 2L = A x_hat, 2L+1 = A^T r) on the buffers currently in the
 * workspace.  Profiling / test hook: bench.py times the dominant tap-GEMM with CUDA events through it.  A stage whose
 * launch record has cross_fp8 set reads the e4m3 operand the last data-gradient call converted (the conversion is
 * not part of the stage), and no stage run this way changes the scales a later call uses. */
int lsnf_plan_run_stage(lsnf_plan* plan, int32_t index, lsnf_stream stream);
/* how many kernels one lsnf_langevin_run of `steps` iterations launches (for bench.py's gpu_launches). */
int lsnf_langevin_launch_count(const lsnf_plan* plan, int32_t steps);

/* ---- introspection (host only; used by the CPU tests to emulate the stage tables) -------------------- */
#define LSNF_MAX_TAPS 16
#define LSNF_MAX_PHASES 4

typedef struct lsnf_tap {
  int32_t dy, dx; /* shift of the operand box in the stage's row grid */
  int32_t plane;  /* phase plane of a phase-split operand (0 for plain NHWC) */
  int32_t brow;   /* first row of this tap's block in the packed weight matrix */
} lsnf_tap;

typedef struct lsnf_stage_info {
  int32_t kind;          /* 0 forward, 1 data-gradient, 3 measurement operator (A x_hat or A^T r; layer = the last) */
  int32_t layer;         /* generator layer index */
  int32_t grid_h, grid_w;/* row grid: M = batch * grid_h * grid_w */
  int32_t box_b, box_h, box_w; /* M tile = box_b*box_h*box_w = 128 rows */
  int32_t k_per_tap;     /* channels contracted per tap (multiple of 64) */
  int32_t n_valid, n_pad;/* output columns, and padded to the N tile */
  int32_t block_n;       /* N tile */
  int32_t n_phases;
  int32_t n_taps[LSNF_MAX_PHASES];
  lsnf_tap taps[LSNF_MAX_PHASES][LSNF_MAX_TAPS];
  int32_t out_mul;       /* output position = row position * out_mul + out_off[phase] */
  int32_t out_off_y[LSNF_MAX_PHASES], out_off_x[LSNF_MAX_PHASES];
  int32_t out_phase_split; /* output written in phase-split layout */
  int32_t out_channels;  /* channels per output position (n_pad may span several positions) */
  int32_t epilogue;      /* 0 bias+lrelu -> fp16 hi|lo + sign bits, 1 bias+tanh -> fp32 NCHW, 2 *lrelu' -> bf16 hi|lo (fp16
                            hi only when bwd_passes == 1), 3 raw fp32 rows (split-K partials / per-tap products of the
                            last forward layer) */
  int32_t k_splits;
  int32_t a_planes;      /* planes of the A operand (4 when phase-split) */
  int32_t a_h, a_w;      /* spatial extent of the A operand (== grid except for the first layer's data gradient) */
  int32_t tap_gen_k;     /* != 0: taps are generated, tap t = (dy, dx) = (t / k, t % k), weight column offset t*k_per_tap */
  int32_t b_k;           /* columns of the hi half of the packed weight matrix (lo half follows) */
  int32_t b_rows;        /* rows of the packed weight matrix */
  int32_t operand_fp16;  /* operands are fp16 hi|lo (forward stages) rather than bf16 hi|lo (data-gradient stages) */
  int32_t passes;        /* MMAs per K step: 3 (hi*hi + hi*lo + lo*hi) or 1 (hi*hi only) */
  int64_t a_offset, b_offset, out_offset; /* byte offsets into the workspace */
  int64_t flops;         /* 2*M*N*K over all phases and taps (nominal, padded taps included) */
} lsnf_stage_info;

int lsnf_plan_num_stages(const lsnf_plan* plan);
int lsnf_plan_stage_info(const lsnf_plan* plan, int32_t index, lsnf_stage_info* out);
/* (row, col) of ConvTranspose2d weight element W[ci][co][ky][kx] of `layer` inside the packed operand of
 * stage `index` (hi half; the lo half sits k_total columns further).  Returns <0 if the stage does not use it. */
int lsnf_plan_pack_index(const lsnf_plan* plan, int32_t index, int32_t ci, int32_t co, int32_t ky, int32_t kx,
                         int64_t* row, int64_t* col);

/* How the tcgen05 path launches stage `index` on a device with `num_sms` SMs: which kernel, grid, operand ring and
 * shared memory, resident CTAs per SM, tensor-store map kind, stream-K.  Host only (no device, no bound workspace
 * needed): the CPU tests check the launch geometry of every BASELINE configuration against the hardware limits
 * (227 KiB shared memory per CTA, 512 TMEM columns per SM) with it. */
#define LSNF_KERNEL_SINGLE 0 /* tapgemm_tc_kernel<block_n>: one CTA per tile, ring sized per launch */
#define LSNF_KERNEL_PAIR 1   /* tapgemm_tc2_kernel: persistent CTA pairs (cta_group::2), N tile 256 */
typedef struct lsnf_launch_info {
  int32_t kernel;                 /* LSNF_KERNEL_* */
  int32_t grid_x, grid_y, grid_z, block;
  int32_t ring_stages;            /* depth of the shared-memory operand ring */
  int32_t stage_bytes;            /* bytes of one ring stage (per CTA) */
  int32_t smem_bytes;             /* dynamic shared memory requested per CTA */
  int32_t ctas_per_sm;            /* CTAs that fit one SM with that request */
  int32_t tmem_columns;           /* TMEM columns one CTA allocates */
  int32_t tma_store;              /* 0 per-thread stores, 1..4 tensor-store map kind of the 16-bit output */
  int32_t stream_k;               /* 1 if the K range of tiles is split across CTA pairs */
  int32_t cross_fp8;              /* 1 if the cross terms run as one e4m3 stream (fp16 hi*hi + kind::f8f6f4) */
  int32_t reserved[3];
} lsnf_launch_info;
int lsnf_plan_stage_launch_info(const lsnf_plan* plan, int32_t index, int32_t num_sms, lsnf_launch_info* out);

#ifdef __cplusplus
}
#endif
#endif /* LSNF_H_ */
