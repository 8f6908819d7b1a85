// Internal structures shared by the host plan code and the kernels.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "lsnf.h"

namespace lsnf {

constexpr int BLOCK_M = 128;  // rows (batch x grid positions) per tile
constexpr int BLOCK_K = 64;   // bf16 channels per K block = one 128-byte swizzle span

enum Epilogue : int32_t {
  EPI_ACT_HL = 0,    // + bias, LeakyReLU, split to bf16 hi|lo                 (hidden forward layers)
  EPI_OUT_TANH = 1,  // + bias, tanh, fp32 NCHW                                 (last forward layer)
  EPI_GRAD_HL = 2,   // * LeakyReLU'(saved activation), split to bf16 hi|lo     (hidden data-gradient layers)
  EPI_PARTIAL = 3    // raw fp32 [split][row][n_pad]: split-K partials of the first layer's data gradient,
                     // and the per-tap products of the last forward layer (gathered by last_gather_tanh)
};

struct TapDev {
  int16_t dy, dx, plane;
  int16_t bsh;   // column shift of the B operand box (weight-gradient stages: the tap's offset in the flattened,
                 // zero-haloed position axis); 0 everywhere else
  int32_t brow;
};

struct PhaseDev {
  int32_t ntaps;
  int32_t mo, no;  // output position offset of this phase
  TapDev taps[LSNF_MAX_TAPS];
};

// One tap-GEMM launch: D[row, n] = sum_taps sum_k A[plane][b][m+dy][n+dx][k] * Bmat[brow + n][k]
// with A, Bmat stored as bf16 hi|lo halves (value = hi + lo) concatenated along the channel axis.
struct StageDev {
  const __nv_bfloat16* a;  // [aP][B][Hg][Wg][2*Ka]
  const __nv_bfloat16* b;  // [b_rows][2*Ka]
  int32_t aP, B, Hg, Wg, Ka, b_rows;
  int32_t aH, aW, tap_gen, b_k;      // A spatial extent, generated-tap mode (k), hi-half width of B
  int32_t bB, bH, bW;                // M tile box, bB*bH*bW == 128
  int32_t tiles_b, tiles_h, tiles_w; // M tiles per axis
  int32_t n_valid, n_pad, block_n;
  int32_t nphase, ksplit, it_per_split;
  // epilogue
  int32_t epi, bias_mod, oC, ms, split;
  float leak;
  const float* bias;
  void* out;
  uint32_t* mbits;                    // sign bits of a saved activation, [B*H*W][oC/32] words (bit c%32 of word c/32):
                                      // written by the EPI_ACT_HL stage producing the activation, read by the
                                      // EPI_GRAD_HL stage that applies LeakyReLU' (train.py:314)
  int64_t sP, sB, sH, sW, sPos;       // output strides in elements
  int32_t nc, Ho, Wo, pad_;
  int32_t fp16, out_fp16;             // operand / hi|lo-output element format: 1 = fp16, 0 = bf16
  int32_t passes, out_single;         // MMAs per K step (3 or 1: hi halves only); output written as hi half only
  const float* descale;               // accumulators are multiplied by *descale (weights packed times 2^k), or null
  int64_t rows_total;                 // B*Hg*Wg (row stride of one split in EPI_PARTIAL)
  float* sk_slots;                    // stream-K: one fp32 partial accumulator [128][256] per CTA of the pair grid
  int32_t* sk_flags;                  // stream-K: one flag per (CTA, epilogue warp), 0 = empty, 1 = partial ready
  int32_t sk_enable;                  // stream-K on/off for this launch
  int32_t wgrad;                      // weight-gradient stage (train.py:394): rows = C_in, columns = C_out, K = the
                                      // flattened zero-haloed positions; every blockIdx.z slice is ONE tap (x split)
  int32_t out_tma, nst;               // hi|lo output written by TMA tensor stores (1 up2 forward, 2 first layer,
                                      // 3 plain gradient, 4 phase-split gradient; 0 = per-thread stores); ring depth
                                      // of this launch (1-CTA kernel)
  int32_t cross8;                     // operands are an fp16 hi half plus an e4m3 cross-term half (see
                                      // tc_cross_fp8, tapgemm_tc.cu); 0 = 16-bit hi|lo halves
  uint32_t* amax_out;                 // the epilogue atomicMax-es max |output| (fp32 bits) into this word: the
                                      // consumer stage converts the output to e4m3 with that scale; or null
  uint32_t* amax_reset;               // this stage's input amax word, zeroed once the conversion that read it is
                                      // complete; or null
  PhaseDev ph[LSNF_MAX_PHASES];
};

// How one tap-GEMM stage launches on a device with a given SM count: decided by tc_plan_launch (tapgemm_tc.cu) alone.
using TcKernel = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, StageDev);
struct TcLaunch {
  TcKernel kernel = nullptr;   // tapgemm_tc2_kernel<passes == 1> or tapgemm_tc_kernel<block_n>; null: no such N tile
  lsnf_launch_info info;       // what lsnf_plan_stage_launch_info reports: grid, block, shared memory, ring depth,
                               // stream-K, tensor-store kind, TMEM columns
};

struct StageHost {
  lsnf_stage_info info;   // layer, kind (0 forward, 1 data gradient, 2 weight gradient), workspace offsets, tables
  StageDev dev;           // derived from info by fill_dev (plan.cu); lsnf_plan_bind adds the workspace pointers and
                          // nst, sk_enable and out_tma from `launch`
  TcLaunch launch;        // for the plan's device (lsnf_plan_bind)
  CUtensorMap tmA, tmB, tmO;
  bool maps_ready = false;
  int k = 0, s = 0, p = 0, ci = 0, co = 0;  // the ConvTranspose2d this stage belongs to
  bool last = false, first = false;
  size_t mbits_off = 0, bias_off = 0;       // workspace offsets of the sign bits and the bias, where the stage has them
  // cross8 stages: workspace offsets of the bf16 hi|lo gradient the conversion reads (the converted operand is at
  // info.a_offset) and of the two words [amax bits of that gradient, descale of the accumulator]
  size_t x8_src_off = 0, x8_off = 0;
};

struct FlowLayout {
  // float offsets inside one step's packed block
  int nz, w, n_out, half;
  size_t an_b, an_e, an_ei, W, WT, Winv, W1, W1T, b1, e1, W2, W2T, b2, e2, W3, W3T, b3, e3, perm, perm_inv, ld_const;
  size_t step_floats;
  size_t vec_floats;  // the per-step vectors come first in a step's block, [0, vec_floats)
  size_t max_mat;     // floats of the largest matrix a flow kernel streams (W counts only with the 1x1 permutation)
  size_t step_mat;    // floats of the matrices one step streams in one pass (likewise)
};

// Training stash of the flow prior (flow parameter update, train.py:403-415): per step, per slot a [B][dim] block.
// Offsets are cumulative dims ("floats per sample before this slot"); element (L, slot, b, j) sits at
// L * layer_floats * B + slot * B + b * dim + j.
struct FlowStash {
  size_t y, u1, a1, a2, h, gu, gp1, gp2, gp3, gx, gl0, gl1, gl2, gl3;
  size_t layer_floats;
};

// Flat parameter-gradient layout of one flow step (floats), in the order of LSNF_FLOW_PTRS_PER_STEP:
// actnorm.b, actnorm.logs, W, fc_1.w, fc_1.actnorm.b, fc_1.actnorm.logs, fc_2.w, ..., fc_zeros.w, .b, .logs
struct FlowGradLayout {
  size_t off[LSNF_FLOW_PTRS_PER_STEP];
  size_t size[LSNF_FLOW_PTRS_PER_STEP];
  size_t step_floats;
};

// arguments of the weight-gradient helper kernels (wgrad.cu)
struct TransArgs {
  const uint16_t* src;
  uint16_t* dst;
  int P, B, H, W, C;
  long long s_plane, s_b, s_h, s_w;   // source strides (elements)
  int src_fp16, src_single;           // halves are fp16 (else bf16); the lo half is absent
  int Hp, Wp, halo;                   // destination grid of one sample: Hp x Wp, `halo` zero rows above and below
  long long Kp;                       // columns of one half of a destination row
  int c_rows;                         // destination rows per plane (>= C)
  int xvar;                           // != 0: every source plane p is written twice -- as is (destination plane 2p) and
                                      // shifted by one column (2p+1): to the right for odd p (reading column x yields
                                      // g(x-1)), to the left for even p (g(x+1)); columns shifted in are zero
};

struct FinalizeArgs {
  const float* part;
  float* out;
  long long s_tap, s_split, s_ci;
  int ksplit, kk, C_in, C_out;
  float scale;
};

struct RowSumArgs {
  const uint16_t* src;
  float* out;
  long long Kp;
  int nsel, C;
  float scale;
  int sel[64];
};

// One layer of the generator parameter update: transposed operand buffers, the weight-gradient tap-GEMM and where
// its results go in the flat gradient buffer.
struct WgradLayer {
  StageHost st;
  TransArgs ta, tg;          // act_{l-1} -> aT, gpre_l (or the im2col seed) -> gT
  size_t off_aT = 0, off_gT = 0, off_part = 0;
  int a_rows = 0, g_rows = 0, planes = 1, ntaps = 1, kk = 1, ksplit = 1;
  long long Kp = 0;
  size_t grad_w_off = 0, grad_b_off = 0;   // floats, in the flat gradient buffer
  FinalizeArgs fin;
  RowSumArgs rs;
};

// State and per-call values of annealed importance sampling (lsnf_ais_run, ais_update_kernel).  The state lives in the
// plan's workspace: the chain's current point z, its reconstruction gradient -dl/dz and its prior gradient
// -dlog p/dz kept apart (so that grad U_beta = gp + beta gr can be formed for any beta), [B][nz] each; log w (fp64);
// and the rows of `scal` [7][B]: l(z), log p(z), step size, accepted proposals, |eps|^2/2 of the pending proposal, and
// the outputs float log w and acceptance rate.
struct AisArgs {
  float* zc;
  float* gr;
  float* gp;
  float* scal;
  double* logw;
  float* epart;          // [B][tiles]: sum m (G(z) - x)^2 over the pixels of one fused last-layer tile
  float* logp;           // [B]: log p(z) from the flow kernel
  const float* betas;    // betas[t] is the schedule value of the call's (or replayed chunk's) iteration t
  const float* eps;      // injected proposal noise [T][B][nz] (eager calls only), or null: Philox
  const float* u;        // injected uniforms of the decisions [T][B] (eager calls only), or null: Philox
  int tiles, total;      // tiles per sample; T (eager calls; a replayed graph reads it from dyn[3])
  float step0, target, inv2s2;   // initial step size, target acceptance rate (<= 0: fixed step), 1 / (2 sigma^2)
};
// step-size adaptation after every decision: log s += AIS_KAPPA (min(1, alpha) - target), s clamped
constexpr double AIS_KAPPA = 0.05, AIS_STEP_MIN = 1e-5, AIS_STEP_MAX = 10.0;
constexpr int AIS_BETA_FLOATS = 1024;   // workspace copy of a replayed chunk's schedule values (<= 1023 iterations)

}  // namespace lsnf

struct lsnf_plan {
  lsnf_config cfg;
  int n_layers = 0;
  int img = 0;
  int kp = 0;   // nz rounded up to BLOCK_K
  int nzp = 0;  // nz rounded up to 128 (N tile of the first layer's data gradient)
  struct Layer { int ci, co, k, s, p, hin, hout; } layers[8];
  std::vector<lsnf::StageHost> stages;  // forward stages 0..L-1, then data-gradient stages L-1..0
  lsnf::FlowLayout fl;
  std::vector<lsnf::WgradLayer> wg;     // training plans only (cfg.train)
  size_t gen_grad_floats = 0;
  bool wg_ready = false;                // the forward pass + data-gradient chain of lsnf_generator_param_grads ran
  lsnf::FlowStash fstash;
  lsnf::FlowGradLayout fgrad;
  size_t off_fstash = 0, off_fgrad = 0, off_floss = 0, off_flinalg = 0;
  // workspace layout (byte offsets)
  size_t ws_bytes = 0;
  size_t off_zhl = 0, off_act[8] = {0}, off_gpre[8] = {0}, off_mbits[8] = {0}, off_xhat = 0, off_im2col = 0, off_partial = 0;
  size_t off_bias[8] = {0};
  size_t off_norms = 0, off_wscale = 0, off_dlast = 0;
  int dlast_pad = 0;
  size_t off_gradg = 0, off_gradf = 0, off_z = 0, off_flow = 0, off_scalars = 0, off_flow_out = 0;
  int ksplit_first = 1;
  char* ws = nullptr;
  bool bound = false, g_packed = false, f_packed = false, have_winv = false;
  int device = -1;
  int num_sms = 148;
  // side stream + fork/join events: the flow prior of a Langevin iteration depends only on z, so it runs
  // concurrently with the generator stages
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  // CUDA graphs of the g_l_steps loop, one per chunk length of at most `graph_chunk` (plan.cu) iterations.  Per-call
  // values (seed, sample offset, the step index of the chunk's first iteration) are read from device memory (dyn) and
  // inputs are staged into the workspace, so a chain of any length replays the same few graphs (train.py:606: 8 000
  // steps).
  // Every value a captured launch bakes in must be part of the key.  An AIS run's step count is not baked in:
  // ais_update_kernel reads it from dyn[3] under replay.  A Langevin loop keys with target = 0, an AIS loop
  // (lsnf_ais_run) with with_noise = 1, and `ais` keeps the two apart.
  struct LoopKey {
    int steps; float step_size, sigma; int with_noise; bool masked, ais; float target;
    bool operator==(const LoopKey& o) const {
      return steps == o.steps && step_size == o.step_size && sigma == o.sigma && with_noise == o.with_noise &&
             masked == o.masked && ais == o.ais && target == o.target;
    }
  };
  struct LoopGraph { LoopKey key; cudaGraphExec_t exec; };
  std::vector<LoopGraph> graphs;
  cudaStream_t cap_stream = nullptr;
  size_t off_x = 0, off_mask = 0, off_gnorms = 0, off_dyn = 0, off_sk_slots = 0, off_sk_flags = 0;
  // annealed importance sampling (lsnf::AisArgs): chain state, energy partials, log p, schedule copy of a replay
  size_t off_ais_z = 0, off_ais_gr = 0, off_ais_gp = 0, off_ais_logw = 0, off_ais_scal = 0, off_ais_epart = 0,
         off_ais_logp = 0, off_ais_beta = 0;
  int fused_tiles = 0;   // CTAs of the fused last-layer kernel per sample
  long long runs = 0;
  bool use_graphs = true;
};

namespace lsnf {

// ---- 16-bit hi|lo splitting: value = hi + lo, both halves in the same 16-bit float format ----
// fp16 (11-bit significands, 22 bits together) is used where the value range is known -- activations, latents
// and power-of-two-scaled weights of the forward pass -- so that LeakyReLU pre-activations are as exact as an fp32
// computation; bf16 (8+8 bits, fp32 range) is used for the gradients of the backward pass.
__device__ __forceinline__ void split16(float v, bool fp16, uint16_t& hi, uint16_t& lo) {
  if (fp16) {
    const __half h = __float2half_rn(v);
    const __half l = __float2half_rn(v - __half2float(h));
    hi = __half_as_ushort(h); lo = __half_as_ushort(l);
  } else {
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
    hi = __bfloat16_as_ushort(h); lo = __bfloat16_as_ushort(l);
  }
}
// e4m3 scale of a tensor whose max |value| is amax: the exponent k with amax * 2^k in [128, 256) (e4m3 reaches 448),
// clamped so that every power of two the cross8 stages build from it stays a normal fp32 number; 0 for zeros
__host__ __device__ inline int fp8_scale_exp(float amax) {
  if (!(amax > 0.f) || !(amax <= 3.4e38f)) return 0;
  int e = 0;
  frexpf(amax, &e);   // amax = f * 2^e, f in [0.5, 1)
  const int k = 8 - e;
  return k < -40 ? -40 : (k > 40 ? 40 : k);
}
__device__ __forceinline__ float join16(uint16_t hi, uint16_t lo, bool fp16) {
  if (fp16) return __half2float(__ushort_as_half(hi)) + __half2float(__ushort_as_half(lo));
  return __bfloat162float(__ushort_as_bfloat16(hi)) + __bfloat162float(__ushort_as_bfloat16(lo));
}

void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what);
#define LSNF_CUDA(call)                                       \
  do {                                                        \
    cudaError_t e__ = (call);                                 \
    if (e__ != cudaSuccess) return ::lsnf::cuda_fail(e__, #call); \
  } while (0)

// ---- programmatic dependent launch (PDL) inside the Langevin loop ----
// Every kernel of the loop calls pdl_wait() before its first access to global memory (it returns at once unless the
// launch carried the attribute below, in which case it returns when the stream predecessor has completed and its
// writes are visible) and then pdl_trigger(), which lets the NEXT kernel's CTAs become resident as soon as every CTA
// of this grid has got that far: the next launch and its prologue (barrier init, TMEM allocation, tensor-map
// prefetch) then overlap this kernel's body instead of following its last CTA.  Nothing is written to global memory
// before pdl_wait(), so there is no write-after-read hazard with the predecessor.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Set by the loop (plan.cu) around a launch that may start before its stream predecessor has completed; thread-local
// because plans are driven from several host threads.  Every other launch of the library leaves it 0.
extern thread_local int g_launch_pdl;
struct PdlScope {
  explicit PdlScope(bool on) { g_launch_pdl = on ? 1 : 0; }
  ~PdlScope() { g_launch_pdl = 0; }
};

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                            Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  if (g_launch_pdl) {
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
  }
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// kernels / launchers implemented in the other translation units
int launch_tapgemm_simt(const StageHost& st, cudaStream_t s);
int launch_tapgemm_tc(const StageHost& st, cudaStream_t s);
int tc_encode_maps(lsnf_plan* plan, StageHost& st);
// What launch_tapgemm_tc does for this stage on a device with `num_sms` SMs (no device needed)
TcLaunch tc_plan_launch(const StageHost& st, int num_sms);
// Whether a 3-pass bf16 data-gradient stage runs its cross terms as one e4m3 stream (operand format of the stage)
bool tc_cross_fp8(const StageDev& d);
// bf16 hi|lo gradient -> the hi16 / e4m3 operand of a cross8 stage, and the stage's descale word
int launch_convert_fp8(const lsnf_plan* plan, const StageHost& st, cudaStream_t s);
int launch_pack_stage(const lsnf_plan* plan, const StageHost& st, const float* w, cudaStream_t s);
int launch_split_z(const lsnf_plan* plan, const float* z, cudaStream_t s);
int launch_weight_scales(const lsnf_plan* plan, const float* const* weights, cudaStream_t s);
int launch_last_gather(const lsnf_plan* plan, float* out, int to_unit_range, cudaStream_t s);
// mask (nullable): per-pixel likelihood weight [B,nc,H,W] of the loss-gradient seed (ignored with upstream != 0)
int launch_recon_grad_im2col(const lsnf_plan* plan, const float* x, const float* mask, float seed_scale, int upstream,
                             cudaStream_t s);
// epart (nullable): [B][tiles] sum m (x_hat - x)^2 over the pixels each CTA owns (tiles = last_fused_tiles)
int launch_last_fused(const lsnf_plan* plan, const float* x, const float* mask, float* epart, float seed_scale,
                      cudaStream_t s);
int last_fused_tiles(const lsnf_plan* plan, int* TR, int* TC);
int launch_ais_begin(const lsnf_plan* plan, float* z, cudaStream_t s);
int launch_ais_update(const lsnf_plan* plan, const AisArgs& a, const float* gf, float gscale, uint64_t seed,
                      uint64_t sample_offset, uint32_t t, const uint64_t* dyn, cudaStream_t s);
int launch_transpose_hl(const TransArgs& a, cudaStream_t s);
int launch_wgrad_finalize(const FinalizeArgs& a, cudaStream_t s);
int launch_bias_rowsum(const RowSumArgs& a, cudaStream_t s);
int launch_mse_sum(const float* xh, const float* x, const float* mask, long long n, float scale, float* partial,
                   unsigned int* ticket, float* out, cudaStream_t s);
int launch_reduce_partial(const lsnf_plan* plan, float* grad_z, float scale, cudaStream_t s);
int launch_flow_pack(lsnf_plan* plan, const float* const* params, const int32_t* const* perm,
                     const int32_t* const* perm_inv, const float* log_abs_det, const float* const* winv,
                     cudaStream_t s);
int launch_flow_forward(const lsnf_plan* plan, const float* z, float* z_out, float* logdet, float* logp,
                        float* grad_z, cudaStream_t s);
int launch_flow_inverse(const lsnf_plan* plan, const float* eps, float* z, float* negobj, cudaStream_t s);
// Dynamic shared memory of one fused flow launch at S samples per CTA: the fixed part (with the forward kernel's
// per-step activation stash when `stash`) plus the matrix ring (sized for both passes when `both_passes`).  Returns 0
// and sets *ring_floats and *smem_bytes when that fits the 227 KB a CTA may opt in to, -1 otherwise.  The launchers
// and lsnf_plan_create both decide with it.
int flow_smem(const FlowLayout& f, int S, int depth, bool stash, bool both_passes, uint32_t* ring_floats,
              size_t* smem_bytes);
constexpr int FLOW_SMEM_BYTES = 227 * 1024;
int launch_adam(int n, float* const* params, const float* const* grads, float* const* m, float* const* v,
                const int64_t* sizes, const int32_t* grad_kk, const int32_t* grad_inner, float lr, float beta1,
                float beta2, float eps, float weight_decay, int64_t step, const float* grad_scale, cudaStream_t s);
int launch_flow_logdet_inverse(const lsnf_plan* plan, const float* const* params, float* winv, float* logdet,
                               cudaStream_t s);
int launch_flow_param_grads(const lsnf_plan* plan, const float* z, float inv_global_batch, float* grads, float* loss,
                            cudaStream_t s);
// lsnf_flow_vjp: the fused forward + backward seeded with seed_g = dL/dz_out and seed_ld = dL/dlogdet (either nullable
// = 0, not both), then -- when grads != nullptr -- the parameter-gradient reductions at scale 1
int launch_flow_vjp(const lsnf_plan* plan, const float* z, const float* seed_g, const float* seed_ld, float* grad_z,
                    float* grads, cudaStream_t s);
int launch_update(const lsnf_plan* plan, float* z, const float* gg, const float* partial, int nsplit, float gscale,
                  const float* gf, float step, const float* eps, int with_noise, uint64_t seed,
                  uint64_t sample_offset, uint32_t step_idx, const uint64_t* dyn, float* gnorms,
                  int write_zhl, cudaStream_t s);
// dyn[0..3] = (seed, sample offset, first iteration of the replayed chunk, total iterations of an AIS run)
int launch_set_dyn(const lsnf_plan* plan, uint64_t seed, uint64_t sample_offset, uint32_t base_step, cudaStream_t s,
                   uint32_t total = 0);
// Per-device one-time setup (opt-in shared-memory limits of every kernel instantiation).  Called by
// lsnf_plan_bind for the plan's device; thread-safe; nothing on the launch path touches function attributes.
int tc_prepare_device(int device);
int aux_prepare_device(int device);
int flow_prepare_device(int device);

// The loss-gradient seed (x_hat - x) / sigma^2 * (1 - x_hat^2) carries 1/sigma^2 (train.py:313).  Only a power of
// two of at most 16 of it is baked into the 16-bit gradient tensors (so a small --g_llhd_sigma cannot overflow
// them); the remaining factor is applied in fp32 where the first layer's split-K partials are summed.
inline float sigma_seed_scale(float sigma) {
  const float inv = 1.f / (sigma * sigma);
  float s = 1.f;
  while (s * 2.f <= inv && s < 16.f) s *= 2.f;
  return s;
}
inline float sigma_post_scale(float sigma) { return 1.f / (sigma * sigma) / sigma_seed_scale(sigma); }

// (row, col) of W[ci][co][ky][kx] in the packed B operand of a stage; shared by host and device
struct PackGeom {
  int kind, first, last, k, ci, co, n_pad, ka;  // ka = columns of the hi half
};

__host__ __device__ inline bool pack_index(const PackGeom& g, int ci, int co, int ky, int kx, long long* row,
                                           long long* col) {
  const int tap = ky * g.k + kx;
  if (g.kind == 0) {
    if (g.first || g.last) {  // rows = (tap, co), cols = ci
      *row = (long long)tap * g.co + co;
      *col = ci;
    } else {        // rows = tap * n_pad + co, cols = ci
      *row = (long long)tap * g.n_pad + co;
      *col = ci;
    }
  } else {
    if (g.first) {  // rows = ci, cols = (tap, co): K runs over the flattened NHWC activation
      *row = ci;
      *col = (long long)tap * g.co + co;
    } else if (g.last) {  // rows = ci, cols = tap * nc + co (explicit im2col operand)
      *row = ci;
      *col = (long long)tap * g.co + co;
    } else {        // rows = tap * n_pad + ci, cols = co
      *row = (long long)tap * g.n_pad + ci;
      *col = co;
    }
  }
  return true;
}

inline PackGeom geom_of(const StageHost& st) {
  return {st.info.kind, st.first, st.last, st.k, st.ci, st.co, st.info.n_pad, st.info.b_k};
}

}  // namespace lsnf
