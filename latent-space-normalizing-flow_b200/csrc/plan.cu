// Host side of the C ABI: plan construction (stage tables, workspace layout) and the entry points.
// Reference call sites are cited in include/lsnf.h.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>

#include "lsnf_internal.cuh"

namespace lsnf {

thread_local int g_launch_pdl = 0;   // see lsnf_internal.cuh
static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
int cuda_fail(cudaError_t e, const char* what) {
  g_err = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
  return LSNF_ERR_CUDA;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static int fail(int code, const std::string& msg) {
  set_error(msg);
  return code;
}

// model.py:52-151
static int arch_layers(const lsnf_config& c, lsnf_plan::Layer* L) {
  const int nz = c.nz, g = c.ngf, nc = c.nc;
  auto set = [&](int i, int ci, int co, int k, int s, int p) { L[i] = {ci, co, k, s, p, 0, 0}; };
  switch (c.arch) {
    case LSNF_ARCH_NONE:
      return 0;
    case LSNF_ARCH_SVHN:
      set(0, nz, g * 8, 4, 1, 0); set(1, g * 8, g * 4, 4, 2, 1); set(2, g * 4, g * 2, 4, 2, 1);
      set(3, g * 2, nc, 4, 2, 1);
      return 4;
    case LSNF_ARCH_CIFAR10:
      set(0, nz, g * 8, 8, 1, 0); set(1, g * 8, g * 4, 4, 2, 1); set(2, g * 4, g * 2, 4, 2, 1);
      set(3, g * 2, nc, 3, 1, 1);
      return 4;
    case LSNF_ARCH_CELEBA_CROP:
      set(0, nz, g * 8, 4, 1, 0); set(1, g * 8, g * 4, 4, 2, 1); set(2, g * 4, g * 2, 4, 2, 1);
      set(3, g * 2, g, 4, 2, 1); set(4, g, nc, 4, 2, 1);
      return 5;
    case LSNF_ARCH_CELEBA_HQ256:
      set(0, nz, g * 16, 4, 1, 0); set(1, g * 16, g * 8, 4, 2, 1); set(2, g * 8, g * 4, 4, 2, 1);
      set(3, g * 4, g * 2, 4, 2, 1); set(4, g * 2, g, 4, 2, 1); set(5, g, g, 4, 2, 1); set(6, g, nc, 4, 2, 1);
      return 7;
    default:
      return -1;
  }
}

static int pick_block_n(int n) {
  if (n % 256 == 0) return 256;
  if (n % 128 == 0) return 128;
  return 64;
}

// Hidden stages whose 256 x 256 CTA-pair tiles would leave more than half of the 74 pairs idle AND whose K loop is
// short (<= 32 blocks: nothing for the persistent ring to amortise) take 128-wide tiles on the 1-CTA kernel instead,
// which spreads them over 2-4x as many SMs.  Measured in round 2 (B200): SVHN B=100 forward layer 1 44.6 -> 29.6 us and
// data gradient of layer 2 41.9 -> 27.5 us (437 k -> 504 k latent-steps/s); with longer K loops (>= 64 blocks: CelebA,
// the deep HQ256 layers) the same switch LOSES 10-80 us per stage -- the pair kernel halves the weight traffic per
// CTA -- hence the bound.
static int pick_block_n_hidden(int n, int rows, int phases, int k_blocks) {
  const int bn = pick_block_n(n);
  if (bn != 256 || k_blocks > 32) return bn;
  const int mtiles = (rows + BLOCK_M - 1) / BLOCK_M;
  const int pair_tiles = (mtiles + 1) / 2 * (n / 256) * phases;
  const int small_tiles = mtiles * (n / 128) * phases;
  return (pair_tiles <= 37 && small_tiles <= 2 * 148) ? 128 : 256;
}

static void make_box(int hg, int wg, int* bb, int* bh, int* bw) {
  *bw = std::min(wg, BLOCK_M);
  *bh = std::min(hg, BLOCK_M / *bw);
  *bb = BLOCK_M / (*bw * *bh);
}

// taps of a k4/s2/p1 transposed convolution for output parity (py, px): oy = 2*iy - 1 + ky
static int up2_fwd_taps(int py, int px, int n_pad, lsnf_tap* t) {
  int n = 0;
  for (int ky = 0; ky < 4; ++ky) {
    if (((ky + 1) & 1) != py) continue;  // oy + 1 - ky must be even
    const int dy = (py + 1 - ky) / 2;    // iy = m + dy for oy = 2m + py
    for (int kx = 0; kx < 4; ++kx) {
      if (((kx + 1) & 1) != px) continue;
      const int dx = (px + 1 - kx) / 2;
      t[n++] = {dy, dx, 0, (ky * 4 + kx) * n_pad};
    }
  }
  return n;
}

// data gradient of the same layer: gin[iy] = sum_ky g[2*iy - 1 + ky] * W[ky]; g is stored phase-split
static int up2_bwd_taps(int n_pad, lsnf_tap* t) {
  int n = 0;
  for (int ky = 0; ky < 4; ++ky) {
    const int oy_off = ky - 1;                       // oy = 2*iy + oy_off
    const int py = oy_off & 1, dy = (oy_off - py) / 2;
    for (int kx = 0; kx < 4; ++kx) {
      const int ox_off = kx - 1;
      const int px = ox_off & 1, dx = (ox_off - px) / 2;
      t[n++] = {dy, dx, py * 2 + px, (ky * 4 + kx) * n_pad};
    }
  }
  return n;
}

// The kernel parameter of a stage, derived from its record for all three kinds; lsnf_plan_bind adds only the workspace
// pointers and nst, sk_enable and out_tma of the launch record.
static void fill_dev(const lsnf_plan* p, StageHost& st) {
  const lsnf_stage_info& I = st.info;
  const lsnf_plan::Layer& y = p->layers[I.layer];
  const bool wg = I.kind == 2;   // weight gradient: one M axis of C_in rows; every blockIdx.z slice is one tap
  StageDev& d = st.dev;
  memset(&d, 0, sizeof(d));
  d.aP = I.a_planes; d.B = wg ? 1 : p->cfg.batch; d.Hg = I.grid_h; d.Wg = I.grid_w; d.Ka = I.k_per_tap;
  d.bB = I.box_b; d.bH = I.box_h; d.bW = I.box_w;
  d.aH = I.a_h; d.aW = I.a_w; d.tap_gen = I.tap_gen_k; d.b_k = I.b_k; d.b_rows = I.b_rows;
  // (the C_in rows of a weight-gradient stage need not fill its last tile)
  d.tiles_b = (d.B + d.bB - 1) / d.bB; d.tiles_h = d.Hg / d.bH; d.tiles_w = (d.Wg + d.bW - 1) / d.bW;
  d.n_valid = I.n_valid; d.n_pad = I.n_pad; d.block_n = I.block_n;
  d.nphase = I.n_phases; d.ksplit = I.k_splits;
  {
    const int ntaps0 = I.tap_gen_k ? I.tap_gen_k * I.tap_gen_k : I.n_taps[0];
    const int total = (wg ? 1 : ntaps0) * (I.k_per_tap / BLOCK_K);
    d.it_per_split = (total + I.k_splits - 1) / I.k_splits;
  }
  d.epi = I.epilogue; d.bias_mod = I.kind == 0 ? y.co : 0; d.oC = I.out_channels; d.ms = I.out_mul;
  d.split = I.out_phase_split;
  d.leak = p->cfg.leak;
  d.fp16 = I.operand_fp16; d.passes = I.passes;
  // single-pass data gradients carry fp16 tensors (hi half only) end to end
  const bool single_bwd = p->cfg.bwd_passes == 1;
  d.out_fp16 = (I.epilogue == EPI_ACT_HL || single_bwd) ? 1 : 0;
  d.out_single = (I.epilogue == EPI_GRAD_HL && single_bwd) ? 1 : 0;
  d.rows_total = (int64_t)d.B * I.grid_h * I.grid_w;
  d.wgrad = wg ? 1 : 0;
  for (int ph = 0; ph < I.n_phases; ++ph) {
    d.ph[ph].ntaps = I.tap_gen_k ? I.tap_gen_k * I.tap_gen_k : I.n_taps[ph];
    d.ph[ph].mo = I.out_off_y[ph]; d.ph[ph].no = I.out_off_x[ph];
    for (int t = 0; t < I.n_taps[ph]; ++t) {
      const lsnf_tap& s = I.taps[ph][t];
      d.ph[ph].taps[t] = {(int16_t)s.dy, (int16_t)s.dx, (int16_t)s.plane, 0, s.brow};
    }
  }
  if (I.kind == 0 && st.last) {
    d.nc = p->cfg.nc; d.Ho = y.hout; d.Wo = y.hout;
  } else if (I.kind == 0) {
    d.sW = 2 * y.co; d.sH = (int64_t)y.hout * d.sW; d.sB = (int64_t)y.hout * d.sH; d.sPos = d.sW;
  } else if (I.kind == 1 && !st.first) {
    const int hg = I.grid_h;
    d.sW = 2 * y.ci;
    if (I.out_phase_split) {
      d.sH = (int64_t)(hg / 2) * d.sW; d.sB = (int64_t)(hg / 2) * d.sH; d.sP = (int64_t)d.B * d.sB;
    } else {
      d.sH = (int64_t)hg * d.sW; d.sB = (int64_t)hg * d.sH;
    }
  } else if (wg && !st.first && !st.last) {
    // plane and (dy, dx) of every tap: brow = plane * C_out in the transposed gradient, its as-is or column-shifted
    // copy by dx (TransArgs::xvar); dy shifts the K range by dy zero-haloed rows of Wp positions
    lsnf_tap tp[16];
    up2_bwd_taps(y.co, tp);
    const int wp = p->wg[I.layer].tg.Wp;
    for (int t = 0; t < 16; ++t)
      d.ph[0].taps[t] = {0, 0, 0, (int16_t)(tp[t].dy * wp), (tp[t].plane * 2 + (tp[t].dx != 0 ? 1 : 0)) * y.co};
  }
}

// Next 1024-byte aligned workspace region; ws_bytes is the running total.
static size_t take(lsnf_plan* p, size_t bytes) {
  const size_t o = p->ws_bytes;
  p->ws_bytes = align_up(o + bytes, 1024);
  return o;
}

// Checks the config, then the generator's geometry, in this order.  Derives what the checks read: the layer table
// (with image size, kp, nzp) and the flow layout.
static int check_config(lsnf_plan* p) {
  const lsnf_config& c = p->cfg;
  if (c.batch <= 0) return fail(LSNF_ERR_INVALID, "batch must be positive");
  if (c.nz <= 0 || (c.nz & 1)) return fail(LSNF_ERR_INVALID, "nz must be even (model.py:383)");
  if (c.nz % 4) return fail(LSNF_ERR_INVALID, "nz must be a multiple of 4 (128-bit latent rows)");
  if (c.nz > 256) return fail(LSNF_ERR_INVALID, "nz > 256 is not supported");
  if (c.f_depth <= 0 || c.f_depth > 32) return fail(LSNF_ERR_INVALID, "f_depth out of range");
  if (c.f_width <= 0 || c.f_width > 256 || c.f_width % 4) return fail(LSNF_ERR_INVALID, "f_width must be a multiple of 4, <= 256");
  if (c.f_permutation != 1 && c.f_permutation != 2)
    return fail(LSNF_ERR_UNSUPPORTED, "f_flow_permutation must be 1 or 2 (model.py:372-379)");
  if (c.f_coupling != 0 && c.f_coupling != 1)
    return fail(LSNF_ERR_UNSUPPORTED, "f_flow_coupling must be 0 or 1 (model.py:384-387)");
  if (c.gemm_impl != LSNF_GEMM_TCGEN05 && c.gemm_impl != LSNF_GEMM_SIMT) return fail(LSNF_ERR_INVALID, "bad gemm_impl");
  if (c.bwd_passes != 0 && c.bwd_passes != 1 && c.bwd_passes != 3) return fail(LSNF_ERR_INVALID, "bwd_passes must be 0, 1 or 3");
  if (c.meas_rows < 0) return fail(LSNF_ERR_INVALID, "meas_rows must not be negative");
  if (c.meas_rows > 0 && c.arch == LSNF_ARCH_NONE) return fail(LSNF_ERR_INVALID, "a measurement operator needs a generator");

  const int L = arch_layers(c, p->layers);
  if (L < 0) return fail(LSNF_ERR_INVALID, "unknown arch (model.py:154 raises ValueError)");
  p->n_layers = L;
  p->kp = (int)align_up(c.nz, BLOCK_K);
  p->nzp = (int)align_up(c.nz, 128);
  if (L > 0) {
    if (c.nc <= 0 || c.nc > 4) return fail(LSNF_ERR_INVALID, "nc must be in 1..4");
    if (c.ngf <= 0) return fail(LSNF_ERR_INVALID, "ngf must be positive");
    int h = 1;
    for (int l = 0; l < L; ++l) {
      auto& y = p->layers[l];
      y.hin = h;
      y.hout = (h - 1) * y.s - 2 * y.p + y.k;
      h = y.hout;
      if (l < L - 1 && y.co % BLOCK_K)
        return fail(LSNF_ERR_INVALID, "hidden generator channel counts must be multiples of 64 (raise --ngf)");
      if (y.hin > 128) return fail(LSNF_ERR_INVALID, "layer grid wider than 128 not supported");
    }
    p->img = h;
  }

  {  // flow parameter block (floats)
    FlowLayout& f = p->fl;
    f.nz = c.nz; f.w = c.f_width; f.half = c.nz / 2; f.n_out = c.f_coupling ? c.nz : c.nz / 2;
    size_t o = 0;
    auto tk = [&](size_t n) { size_t r = o; o += (n + 3) / 4 * 4; return r; };
    // vectors first (they are staged into shared memory as one block), then the matrices
    f.an_b = tk(f.nz); f.an_e = tk(f.nz); f.an_ei = tk(f.nz);
    f.b1 = tk(f.w); f.e1 = tk(f.w); f.b2 = tk(f.w); f.e2 = tk(f.w); f.b3 = tk(f.n_out); f.e3 = tk(f.n_out);
    f.perm = tk(f.nz); f.perm_inv = tk(f.nz); f.ld_const = tk(4);
    f.vec_floats = o;
    f.W = tk((size_t)f.nz * f.nz); f.WT = tk((size_t)f.nz * f.nz); f.Winv = tk((size_t)f.nz * f.nz);
    f.W1 = tk((size_t)f.half * f.w); f.W1T = tk((size_t)f.half * f.w);
    f.W2 = tk((size_t)f.w * f.w); f.W2T = tk((size_t)f.w * f.w);
    f.W3 = tk((size_t)f.w * f.n_out); f.W3T = tk((size_t)f.w * f.n_out);
    // what the flow kernels stream: the shuffle permutation has no matrix
    const size_t w_floats = c.f_permutation == 2 ? (size_t)f.nz * f.nz : 0;
    f.max_mat = std::max({w_floats, (size_t)f.half * f.w, (size_t)f.w * f.w, (size_t)f.w * f.n_out});
    f.step_mat = w_floats + (size_t)f.half * f.w + (size_t)f.w * f.w + (size_t)f.w * f.n_out;
    f.step_floats = o;
    // every flow entry point must be able to launch: the forward kernel (with its activation stash, both passes) at
    // one sample per CTA is the largest footprint; the inverse kernel needs less
    uint32_t ring_floats;
    size_t smem_bytes;
    if (flow_smem(f, 1, c.f_depth, true, true, &ring_floats, &smem_bytes))
      return fail(LSNF_ERR_INVALID,
                  "flow prior exceeds the " + std::to_string(FLOW_SMEM_BYTES / 1024) +
                      " KB of shared memory of one CTA even at one sample per CTA: its largest matrix (f_width^2, or "
                      "nz^2 with f_flow_permutation 2) plus f_depth * (2 f_width + nz) stashed activations must fit "
                      "(include/lsnf.h, lsnf_config)");
  }

  // the ConvTranspose2d geometries the stage builders implement: forward stages first, then data gradients
  for (int l = 0; l < L; ++l) {
    const auto& y = p->layers[l];
    const bool up2 = y.k == 4 && y.s == 2 && y.p == 1, same = y.k == 3 && y.s == 1 && y.p == 1;
    if (l == 0 && !(y.s == 1 && y.p == 0)) return fail(LSNF_ERR_INVALID, "first layer must be s1 p0");
    if (l == 0 && L == 1) return fail(LSNF_ERR_INVALID, "single-layer generator not supported");
    if (l > 0 && !(up2 || same))
      return fail(LSNF_ERR_INVALID, l == L - 1 ? "unsupported last-layer geometry" : "unsupported ConvTranspose2d geometry");
  }
  for (int l = L - 1; l >= 0; --l) {
    const auto& y = p->layers[l];
    if (l == L - 1 && y.k * y.k * y.co > BLOCK_K) return fail(LSNF_ERR_INVALID, "k*k*nc must be <= 64");
    if (l > 0 && l < L - 1 && !(y.k == 4 && y.s == 2 && y.p == 1))
      return fail(LSNF_ERR_INVALID, "unsupported hidden layer geometry");
  }
  return LSNF_OK;
}

// Every region but the tap-GEMM operands and results of the stage builders and the AIS state.
static void take_regions(lsnf_plan* p) {
  const lsnf_config& c = p->cfg;
  const int L = p->n_layers, B = c.batch;
  const FlowLayout& f = p->fl;
  p->off_z = take(p, (size_t)B * c.nz * 4);
  p->off_gradg = take(p, (size_t)B * c.nz * 4);
  p->off_gradf = take(p, (size_t)B * c.nz * 4);
  p->off_scalars = take(p, 256);
  p->off_dyn = take(p, 64);
  p->off_gnorms = take(p, 64);
  p->off_norms = take(p, (size_t)2 * B * 4);
  p->off_flow_out = take(p, (size_t)B * (c.nz + 2) * 4);
  p->off_flow = take(p, f.step_floats * 4 * c.f_depth);
  {  // training stash and flat gradient layout of the flow parameter update (train.py:403-415)
    FlowStash& t = p->fstash;
    size_t so = 0;
    auto ts = [&](size_t n) { size_t r = so; so += n; return r; };
    t.y = ts(f.nz); t.u1 = ts(f.half); t.a1 = ts(f.w); t.a2 = ts(f.w); t.h = ts(f.n_out);
    t.gu = ts(f.nz); t.gp1 = ts(f.w); t.gp2 = ts(f.w); t.gp3 = ts(f.n_out); t.gx = ts(f.nz);
    t.gl0 = ts(f.nz); t.gl1 = ts(f.w); t.gl2 = ts(f.w); t.gl3 = ts(f.n_out);
    t.layer_floats = so;
    p->off_fstash = take(p, so * 4 * (size_t)B * c.f_depth);
    // W^-1 [f_depth][nz][nz] and log|det W| [f_depth] when the library evaluates them itself
    p->off_flinalg = take(p, ((size_t)c.f_depth * f.nz * f.nz + 32) * 4);
    FlowGradLayout& gl = p->fgrad;
    const size_t sizes[LSNF_FLOW_PTRS_PER_STEP] = {
        (size_t)f.nz, (size_t)f.nz, (size_t)f.nz * f.nz, (size_t)f.half * f.w, (size_t)f.w, (size_t)f.w,
        (size_t)f.w * f.w, (size_t)f.w, (size_t)f.w, (size_t)f.w * f.n_out, (size_t)f.n_out, (size_t)f.n_out};
    size_t go = 0;
    for (int i = 0; i < LSNF_FLOW_PTRS_PER_STEP; ++i) { gl.off[i] = go; gl.size[i] = sizes[i]; go += (sizes[i] + 3) / 4 * 4; }
    gl.step_floats = go;
  }
  if (L == 0) return;
  p->off_zhl = take(p, (size_t)B * 2 * p->kp * 2);
  p->off_sk_slots = take(p, (size_t)160 * 128 * 256 * 4);   // stream-K partial accumulators (<= 160 CTAs)
  p->off_sk_flags = take(p, (size_t)160 * 8 * 4);
  p->off_x = take(p, (size_t)B * c.nc * p->img * p->img * 4);
  p->off_mask = take(p, (size_t)B * c.nc * p->img * p->img * 4);   // the graph-replayed loop's copy of a mask
  for (int l = 0; l < L - 1; ++l) {
    const auto& y = p->layers[l];
    const size_t bytes = (size_t)B * y.hout * y.hout * 2 * y.co * 2;
    p->off_act[l] = take(p, bytes);
    p->off_gpre[l] = take(p, bytes);
    p->off_mbits[l] = take(p, (size_t)B * y.hout * y.hout * y.co / 8);   // LeakyReLU sign bits of act[l]
  }
  for (int l = 0; l < L; ++l) p->off_bias[l] = take(p, (size_t)p->layers[l].co * 4);
  p->off_xhat = take(p, (size_t)B * c.nc * p->img * p->img * 4);
  p->off_wscale = take(p, (size_t)L * 16);   // per layer: |w|max bits, scale 2^k, descale 2^-k
  const auto& yl = p->layers[L - 1];
  const int kk = yl.k * yl.k * yl.co;
  p->off_dlast = take(p, (size_t)B * yl.hin * yl.hin * (kk <= 32 ? 32 : 64) * 4);
  p->off_im2col = take(p, (size_t)B * yl.hin * yl.hin * 2 * BLOCK_K * 2);
}

// A cleared record of `kind` for layer l, and the ConvTranspose2d it belongs to.
static void set_conv(StageHost& st, const lsnf_plan* p, int kind, int l) {
  const auto& y = p->layers[l];
  memset(&st.info, 0, sizeof(st.info));
  st.info.kind = kind; st.info.layer = l;
  st.k = y.k; st.s = y.s; st.p = y.p; st.ci = y.ci; st.co = y.co;
  st.first = l == 0; st.last = l == p->n_layers - 1;
}

// Forward stage of layer l (train.py:312): stages[l].
static void build_forward_stage(lsnf_plan* p, int l) {
  const lsnf_config& c = p->cfg;
  const int B = c.batch;
  const auto& y = p->layers[l];
  StageHost& st = p->stages[l];
  set_conv(st, p, 0, l);
  lsnf_stage_info& I = st.info;
  I.a_planes = 1;
  I.k_splits = 1;
  if (st.first) {
    I.grid_h = I.grid_w = 1;
    I.k_per_tap = p->kp;
    I.n_valid = y.k * y.k * y.co; I.n_pad = I.n_valid; I.block_n = pick_block_n(y.co);
    I.n_phases = 1; I.n_taps[0] = 1; I.taps[0][0] = {0, 0, 0, 0};
    I.out_mul = 1; I.out_channels = y.co; I.epilogue = EPI_ACT_HL;
    I.a_offset = p->off_zhl;
  } else {
    I.grid_h = I.grid_w = y.hin;
    I.k_per_tap = y.ci;
    I.out_channels = y.co;
    if (st.last) {
      // direct product D[pos][(tap, c)] = act[pos][:] . W[:, c, tap]; last_gather_tanh sums the taps that land
      // on each output pixel (col2im without atomics), adds the bias and applies tanh
      I.n_valid = y.k * y.k * y.co; I.n_pad = I.n_valid <= 32 ? 32 : 64; I.block_n = I.n_pad;
      I.epilogue = EPI_PARTIAL; I.out_channels = I.n_pad;
      I.n_phases = 1; I.out_mul = 1; I.n_taps[0] = 1; I.taps[0][0] = {0, 0, 0, 0};
      p->dlast_pad = I.n_pad;
    } else {
      I.n_valid = I.n_pad = y.co; I.epilogue = EPI_ACT_HL;
      I.block_n = pick_block_n_hidden(y.co, B * y.hin * y.hin, (y.k == 4 && y.s == 2) ? 4 : 1,
                                      ((y.k == 4 && y.s == 2) ? 4 : y.k * y.k) * (y.ci / BLOCK_K));
      if (y.k == 4 && y.s == 2 && y.p == 1) {
        I.n_phases = 4; I.out_mul = 2;
        for (int ph = 0; ph < 4; ++ph) {
          I.n_taps[ph] = up2_fwd_taps(ph >> 1, ph & 1, I.n_pad, I.taps[ph]);
          I.out_off_y[ph] = ph >> 1; I.out_off_x[ph] = ph & 1;
        }
      } else {   // k3 s1 p1
        I.n_phases = 1; I.out_mul = 1; I.n_taps[0] = 9;
        for (int ky = 0; ky < 3; ++ky)
          for (int kx = 0; kx < 3; ++kx) I.taps[0][ky * 3 + kx] = {1 - ky, 1 - kx, 0, (ky * 3 + kx) * I.n_pad};
      }
    }
    I.a_offset = p->off_act[l - 1];
  }
  make_box(I.grid_h, I.grid_w, &I.box_b, &I.box_h, &I.box_w);
  const size_t b_rows = (st.first || st.last) ? (size_t)I.n_pad : (size_t)y.k * y.k * I.n_pad;
  I.operand_fp16 = 1; I.passes = 3;
  I.a_h = I.grid_h; I.a_w = I.grid_w; I.tap_gen_k = 0; I.b_k = I.k_per_tap; I.b_rows = (int)b_rows;
  I.b_offset = take(p, b_rows * 2 * I.k_per_tap * 2);
  I.out_offset = st.last ? p->off_dlast : p->off_act[l];
  st.mbits_off = st.last ? 0 : p->off_mbits[l];
  st.bias_off = p->off_bias[l];
  int taps_sum = 0;
  for (int ph = 0; ph < I.n_phases; ++ph) taps_sum += I.n_taps[ph];
  I.flops = 2LL * B * I.grid_h * I.grid_w * (long long)I.n_valid * I.k_per_tap * taps_sum;
  if (st.first) I.flops = 2LL * B * (long long)I.n_valid * c.nz;
  if (st.last) I.flops = 2LL * B * I.grid_h * I.grid_w * (long long)y.k * y.k * y.co * y.ci;
  fill_dev(p, st);
}

// K splits of a split-K stage over `tiles` output tiles: about one wave of CTAs, at least two K blocks per split, and
// every split non-empty
static int split_count(int kblocks, int tiles) {
  const int want = std::max(1, (148 + tiles - 1) / tiles);
  int per = std::max(2, (kblocks + want - 1) / want);
  const int s = (kblocks + per - 1) / per;
  per = (kblocks + s - 1) / s;                            // what the kernels use (it_per_split)
  return (kblocks + per - 1) / per;
}

// Data-gradient stage of layer l (train.py:314): stages[L + (L - 1 - l)], run from the last layer down to the first.
// The first layer's stage writes split-K partials whose region lsnf_plan_create takes after all data-gradient stages.
static void build_dgrad_stage(lsnf_plan* p, int l) {
  const lsnf_config& c = p->cfg;
  const int L = p->n_layers, B = c.batch;
  const auto& y = p->layers[l];
  StageHost& st = p->stages[L + (L - 1 - l)];
  set_conv(st, p, 1, l);
  lsnf_stage_info& I = st.info;
  I.a_planes = 1; I.k_splits = 1;
  I.n_phases = 1; I.out_mul = 1;
  size_t b_rows;
  if (st.last) {
    I.grid_h = I.grid_w = y.hin;
    I.k_per_tap = BLOCK_K;
    I.n_valid = I.n_pad = y.ci; I.block_n = pick_block_n(y.ci);
    I.n_taps[0] = 1; I.taps[0][0] = {0, 0, 0, 0};
    I.a_offset = p->off_im2col;
    b_rows = I.n_pad;
  } else if (st.first) {
    I.grid_h = I.grid_w = 1;
    I.k_per_tap = y.co;           // per output position of the first layer; taps run over the k*k positions
    I.n_valid = c.nz; I.n_pad = p->nzp; I.block_n = 128;
    I.n_taps[0] = 0;              // generated: tap t -> (dy, dx) = (t / k, t % k), B column offset t*co
    I.a_offset = p->off_gpre[0];
    b_rows = I.n_pad;
    I.k_splits = split_count(y.k * y.k * y.co / BLOCK_K, (B + BLOCK_M - 1) / BLOCK_M);
    p->ksplit_first = I.k_splits;
  } else {   // k4 s2 p1
    I.grid_h = I.grid_w = y.hin;
    I.k_per_tap = y.co;
    I.n_valid = I.n_pad = y.ci; I.block_n = pick_block_n_hidden(y.ci, B * y.hin * y.hin, 1, 16 * (y.co / BLOCK_K));
    I.a_planes = 4;
    I.n_taps[0] = up2_bwd_taps(I.n_pad, I.taps[0]);
    I.a_offset = p->off_gpre[l];
    b_rows = (size_t)16 * I.n_pad;
  }
  make_box(I.grid_h, I.grid_w, &I.box_b, &I.box_h, &I.box_w);
  const size_t b_k = st.first ? (size_t)y.k * y.k * y.co : (size_t)I.k_per_tap;
  I.operand_fp16 = c.bwd_passes == 1 ? 1 : 0; I.passes = c.bwd_passes == 1 ? 1 : 3;
  I.a_h = st.first ? y.k : I.grid_h; I.a_w = st.first ? y.k : I.grid_w;
  I.tap_gen_k = st.first ? y.k : 0; I.b_k = (int)b_k; I.b_rows = (int)b_rows;
  I.b_offset = take(p, b_rows * 2 * b_k * 2);
  if (st.first) {
    I.epilogue = EPI_PARTIAL; I.out_channels = I.n_pad;
  } else {
    I.epilogue = EPI_GRAD_HL; I.out_channels = y.ci;
    // the consumer (data gradient of layer l-1) reads phase-split when it is a stride-2 layer
    I.out_phase_split = (l - 1 > 0) ? 1 : 0;
    I.out_offset = p->off_gpre[l - 1];
    st.mbits_off = p->off_mbits[l - 1];
  }
  I.flops = 2LL * B * I.grid_h * I.grid_w * (long long)I.n_valid *
            (st.last ? y.k * y.k * y.co : (st.first ? (long long)y.k * y.k * y.co : 16LL * y.co));
  fill_dev(p, st);
  // the tcgen05 path runs this stage's cross terms in e4m3: it reads gpre[l] converted to the hi16 / e4m3 format
  // (launch_convert_fp8) from a region of its own, and keeps gpre[l]'s amax and its accumulator descale beside it
  if (c.gemm_impl == LSNF_GEMM_TCGEN05 && tc_cross_fp8(st.dev)) {
    st.dev.cross8 = 1;
    st.x8_src_off = I.a_offset;
    I.a_offset = take(p, (size_t)B * y.hout * y.hout * 2 * y.co * 2);
    st.x8_off = take(p, 16);
  }
}

// Generator parameter update of layer l (train.py:390-394): transposed operands, the weight-gradient tap-GEMM and where
// its results go in the flat gradient buffer (gen_grad_floats is the running total).
static void build_wgrad_layer(lsnf_plan* p, int l) {
  const lsnf_config& c = p->cfg;
  const int L = p->n_layers, B = c.batch;
  const auto& y = p->layers[l];
  WgradLayer& w = p->wg[l];
  const bool first = (l == 0), last = (l == L - 1);
  const int kk = y.k * y.k;
  const bool single = c.bwd_passes == 1;   // gradient tensors hold fp16 hi halves only
  w.kk = kk;
  int n_cols, hp, wp, halo, block_n;
  TransArgs& ta = w.ta;
  TransArgs& tg = w.tg;
  memset(&ta, 0, sizeof(ta)); memset(&tg, 0, sizeof(tg));
  if (first) {
    // dW0[ci][(tap, co)] = sum_b z[b][ci] * gpre_0[b][tap][co]
    w.a_rows = (int)align_up(c.nz, 128); hp = wp = 1; halo = 0;
    w.Kp = (long long)align_up(B, BLOCK_K);
    w.planes = 1; w.g_rows = kk * y.co; w.ntaps = 1; n_cols = kk * y.co; block_n = pick_block_n(n_cols);
    ta.P = 1; ta.B = B; ta.H = ta.W = 1; ta.C = p->kp; ta.s_b = 2 * p->kp; ta.src_fp16 = 1; ta.c_rows = w.a_rows;
    tg.P = kk; tg.B = B; tg.H = tg.W = 1; tg.C = y.co; tg.s_plane = 2 * y.co; tg.s_b = (long long)kk * 2 * y.co;
    tg.c_rows = y.co;
  } else if (last) {
    // dW[ci][(tap, c)] = sum_pos act[pos][ci] * im2col_seed[pos][(tap, c)]   (the seed already holds the taps)
    w.a_rows = y.ci; hp = wp = y.hin; halo = 0;
    w.Kp = (long long)align_up((size_t)B * y.hin * y.hin, BLOCK_K);
    w.planes = 1; w.g_rows = BLOCK_K; w.ntaps = 1; n_cols = BLOCK_K; block_n = 64;
    ta.P = 1; ta.B = B; ta.H = ta.W = y.hin; ta.C = y.ci; ta.s_w = 2 * y.ci; ta.s_h = (long long)y.hin * ta.s_w;
    ta.s_b = (long long)y.hin * ta.s_h; ta.src_fp16 = 1; ta.c_rows = y.ci;
    tg.P = 1; tg.B = B; tg.H = tg.W = y.hin; tg.C = BLOCK_K; tg.s_w = 2 * BLOCK_K; tg.s_h = (long long)y.hin * tg.s_w;
    tg.s_b = (long long)y.hin * tg.s_h; tg.c_rows = BLOCK_K;
  } else {
    // k4/s2/p1: per tap, dW[ci][co] = sum_pos act[pos][ci] * gpre[plane_tap][pos + (dy, dx)][co].  One zero halo
    // row above and below every sample (dy becomes the K offset dy * Wp, a multiple of 8 elements = 16 bytes as
    // TMA box origins must be); dx picks the as-is or the column-shifted copy of the phase plane (TransArgs::xvar)
    w.a_rows = y.ci; hp = y.hin + 2; wp = (int)align_up(y.hin, 8); halo = 1;
    w.Kp = (long long)align_up((size_t)B * hp * wp, BLOCK_K);
    w.planes = 8; w.g_rows = y.co; w.ntaps = 16; n_cols = y.co; block_n = pick_block_n(y.co);
    ta.P = 1; ta.B = B; ta.H = ta.W = y.hin; ta.C = y.ci; ta.s_w = 2 * y.ci; ta.s_h = (long long)y.hin * ta.s_w;
    ta.s_b = (long long)y.hin * ta.s_h; ta.src_fp16 = 1; ta.c_rows = y.ci;
    tg.P = 4; tg.B = B; tg.H = tg.W = y.hin; tg.C = y.co; tg.s_w = 2 * y.co; tg.s_h = (long long)y.hin * tg.s_w;
    tg.s_b = (long long)y.hin * tg.s_h; tg.s_plane = (long long)B * tg.s_b; tg.c_rows = y.co; tg.xvar = 1;
  }
  ta.Hp = tg.Hp = hp; ta.Wp = tg.Wp = wp; ta.halo = tg.halo = halo; ta.Kp = tg.Kp = w.Kp;
  tg.src_fp16 = single ? 1 : 0; tg.src_single = single ? 1 : 0;
  w.off_aT = take(p, (size_t)w.a_rows * 2 * w.Kp * 2);
  w.off_gT = take(p, (size_t)w.planes * w.g_rows * 2 * w.Kp * 2);
  // the tap-GEMM: rows = C_in, columns = C_out (or (tap, co) / the 64 seed columns), K = flattened positions
  StageHost& st = w.st;
  set_conv(st, p, 2, l);
  lsnf_stage_info& I = st.info;
  I.grid_h = 1; I.grid_w = w.a_rows; I.box_b = 1; I.box_h = 1; I.box_w = BLOCK_M;
  I.k_per_tap = (int)w.Kp; I.n_valid = n_cols; I.block_n = block_n; I.n_pad = (int)align_up(n_cols, block_n);
  I.n_phases = 1; I.n_taps[0] = w.ntaps; I.out_mul = 1; I.out_channels = I.n_pad; I.epilogue = EPI_PARTIAL;
  I.a_planes = 1; I.a_h = 1; I.a_w = w.a_rows; I.b_k = (int)w.Kp; I.b_rows = w.planes * w.g_rows;
  I.operand_fp16 = 0; I.passes = 3;
  const int kblocks = (int)(w.Kp / BLOCK_K);
  const int tiles = ((w.a_rows + BLOCK_M - 1) / BLOCK_M) * (I.n_pad / block_n) * w.ntaps;
  int want = std::max(1, (2 * 148 + tiles - 1) / tiles);
  want = std::min(want, std::max(1, kblocks / 4));          // at least four K blocks per split
  const int per = (kblocks + want - 1) / want;
  w.ksplit = (kblocks + per - 1) / per;                     // every split is non-empty: it_per_split = per
  I.k_splits = w.ksplit;
  for (int t = 0; t < w.ntaps; ++t) I.taps[0][t] = {0, 0, 0, 0};
  I.flops = 2LL * w.a_rows * (long long)n_cols * w.Kp * w.ntaps;
  I.a_offset = w.off_aT; I.b_offset = w.off_gT;
  w.off_part = take(p, (size_t)w.ntaps * w.ksplit * w.a_rows * I.n_pad * 4);
  I.out_offset = w.off_part;
  fill_dev(p, st);
  // results: dW in the parameter's own layout, then db
  w.grad_w_off = p->gen_grad_floats; p->gen_grad_floats += align_up((size_t)y.ci * y.co * kk, 4);
  w.grad_b_off = p->gen_grad_floats; p->gen_grad_floats += align_up((size_t)y.co, 4);
  FinalizeArgs& f = w.fin;
  memset(&f, 0, sizeof(f));
  f.ksplit = w.ksplit; f.kk = kk; f.C_in = y.ci; f.C_out = y.co;
  if (first) { f.s_tap = y.co; f.s_split = 0; f.s_ci = I.n_pad; f.ksplit = 1; }
  else if (last) { f.s_tap = y.co; f.s_split = (long long)w.a_rows * I.n_pad; f.s_ci = I.n_pad; }
  else { f.s_tap = (long long)w.ksplit * w.a_rows * I.n_pad; f.s_split = (long long)w.a_rows * I.n_pad; f.s_ci = I.n_pad; }
  RowSumArgs& r = w.rs;
  memset(&r, 0, sizeof(r));
  r.Kp = w.Kp; r.C = y.co;
  if (first) { r.nsel = kk; for (int t = 0; t < kk; ++t) r.sel[t] = t * y.co; }
  else if (last) {
    // every output pixel is produced by exactly one of these taps (oy = iy*s - p + ky covers each oy once)
    r.nsel = 0;
    for (int ky = 0; ky < y.k; ++ky)
      for (int kx = 0; kx < y.k; ++kx) {
        const bool once_y = y.s == 1 ? ky == y.p : (ky == 1 || ky == 2);
        const bool once_x = y.s == 1 ? kx == y.p : (kx == 1 || kx == 2);
        if (once_y && once_x) r.sel[r.nsel++] = (ky * y.k + kx) * y.co;
      }
  } else { r.nsel = 4; for (int q = 0; q < 4; ++q) r.sel[q] = 2 * q * y.co; }   // the as-is copy of every plane
}

// The two measurement-operator stages of a plan with meas_rows = m > 0, after every other region: stages[2L] = A x_hat
// (M = B, N = m, K = n; fp16 operands, A scaled by a power of two) and stages[2L+1] = A^T r (M = B, N = n, K = m; bf16
// operands).  Each is a plain GEMM over a flattened operand with split-K partials [S][B][n_pad] -- the kind of the
// first layer's data-gradient stage with one generated tap of the whole K extent -- and with only one or a few
// 128-row M tiles the K splits fill the SMs.
static void take_meas_regions(lsnf_plan* p) {
  const lsnf_config& c = p->cfg;
  const int L = p->n_layers, B = c.batch, m = c.meas_rows, n = c.nc * p->img * p->img;
  p->meas_m = m;
  p->meas_kx = (int)align_up(n, BLOCK_K);
  p->meas_km = (int)align_up(m, BLOCK_K);
  p->meas_tiles = (m + 255) / 256;
  p->off_meas_xhl = take(p, (size_t)B * 2 * p->meas_kx * 2);
  p->off_meas_r = take(p, (size_t)B * 2 * p->meas_km * 2);
  p->off_meas_y = take(p, (size_t)B * m * 4);
  p->off_meas_epart = take(p, (size_t)B * p->meas_tiles * 4);
  p->off_meas_scale = take(p, 16);
  for (int which = 1; which <= 2; ++which) {
    StageHost& st = p->stages[2 * L + which - 1];
    memset(&st.info, 0, sizeof(st.info));
    st.meas = which;
    lsnf_stage_info& I = st.info;
    I.kind = 3; I.layer = L - 1;
    const int rows = which == 1 ? m : n, k = which == 1 ? p->meas_kx : p->meas_km;
    I.grid_h = I.grid_w = 1;
    I.k_per_tap = k;
    I.n_valid = rows; I.block_n = 128; I.n_pad = (int)align_up(rows, 128);
    I.n_phases = 1; I.n_taps[0] = 0; I.out_mul = 1; I.out_channels = I.n_pad; I.epilogue = EPI_PARTIAL;
    I.a_planes = 1; I.a_h = I.a_w = 1; I.tap_gen_k = 1; I.b_k = k; I.b_rows = I.n_pad;
    I.operand_fp16 = which == 1 ? 1 : 0; I.passes = 3;
    make_box(1, 1, &I.box_b, &I.box_h, &I.box_w);
    I.k_splits = split_count(k / BLOCK_K, ((B + BLOCK_M - 1) / BLOCK_M) * (I.n_pad / I.block_n));
    I.a_offset = which == 1 ? p->off_meas_xhl : p->off_meas_r;
    I.b_offset = take(p, (size_t)I.b_rows * 2 * k * 2);
    I.out_offset = take(p, (size_t)I.k_splits * B * I.n_pad * 4);
    I.flops = 2LL * B * m * (long long)n;
    fill_dev(p, st);
  }
}

// Annealed importance sampling (lsnf_ais_run): chain state and energies, after every other region.
static void take_ais_regions(lsnf_plan* p) {
  const int B = p->cfg.batch, nz = p->cfg.nz;
  int tr, tc;
  p->fused_tiles = last_fused_tiles(p, &tr, &tc);
  p->off_ais_z = take(p, (size_t)B * nz * 4);
  p->off_ais_gr = take(p, (size_t)B * nz * 4);
  p->off_ais_gp = take(p, (size_t)B * nz * 4);
  p->off_ais_logw = take(p, (size_t)B * 8);
  p->off_ais_scal = take(p, (size_t)7 * B * 4);
  p->off_ais_epart = take(p, (size_t)B * p->fused_tiles * 4);
  p->off_ais_logp = take(p, (size_t)B * 4);
  p->off_ais_beta = take(p, (size_t)AIS_BETA_FLOATS * 4);
}

}  // namespace lsnf

using namespace lsnf;

extern "C" int lsnf_abi_version(void) { return LSNF_ABI_VERSION; }
extern "C" const char* lsnf_last_error(void) { return g_err.c_str(); }

extern "C" int lsnf_plan_create(const lsnf_config* cfg, lsnf_plan** out) {
  if (!cfg || !out) return fail(LSNF_ERR_INVALID, "null argument");
  std::unique_ptr<lsnf_plan> p(new lsnf_plan());
  p->cfg = *cfg;
  if (int rc = check_config(p.get())) return rc;
  take_regions(p.get());
  const int L = p->n_layers;
  if (L > 0) {
    p->stages.resize(2 * L);
    for (int l = 0; l < L; ++l) build_forward_stage(p.get(), l);
    for (int l = L - 1; l >= 0; --l) build_dgrad_stage(p.get(), l);
    // partial sums of the first layer's split-K data gradient
    p->off_partial = take(p.get(), (size_t)p->ksplit_first * p->cfg.batch * p->nzp * 4);
    p->stages[2 * L - 1].info.out_offset = p->off_partial;
    if (p->cfg.train) {
      p->wg.resize(L);
      for (int l = 0; l < L; ++l) build_wgrad_layer(p.get(), l);
    }
    take_ais_regions(p.get());
    if (p->cfg.meas_rows > 0) {
      p->stages.resize(2 * L + 2);
      take_meas_regions(p.get());
    }
  }
  *out = p.release();
  return LSNF_OK;
}

extern "C" void lsnf_plan_destroy(lsnf_plan* plan) {
  if (!plan) return;
  if (plan->side) cudaStreamDestroy(plan->side);
  if (plan->ev_fork) cudaEventDestroy(plan->ev_fork);
  if (plan->ev_join) cudaEventDestroy(plan->ev_join);
  for (auto& g : plan->graphs) cudaGraphExecDestroy(g.exec);
  if (plan->cap_stream) cudaStreamDestroy(plan->cap_stream);
  delete plan;
}

extern "C" size_t lsnf_workspace_bytes(const lsnf_plan* plan) { return plan ? plan->ws_bytes : 0; }

extern "C" int lsnf_plan_num_stages(const lsnf_plan* plan) { return plan ? (int)plan->stages.size() : 0; }

extern "C" int lsnf_plan_stage_info(const lsnf_plan* plan, int32_t index, lsnf_stage_info* out) {
  if (!plan || !out || index < 0 || index >= (int)plan->stages.size()) return fail(LSNF_ERR_INVALID, "bad stage index");
  *out = plan->stages[index].info;
  return LSNF_OK;
}

extern "C" int lsnf_plan_stage_launch_info(const lsnf_plan* plan, int32_t index, int32_t num_sms,
                                           lsnf_launch_info* out) {
  if (!plan || !out || index < 0 || index >= (int)plan->stages.size()) return fail(LSNF_ERR_INVALID, "bad stage index");
  if (num_sms < 2) return fail(LSNF_ERR_INVALID, "num_sms must be at least 2");
  *out = tc_plan_launch(plan->stages[index], num_sms).info;
  return LSNF_OK;
}

extern "C" int lsnf_plan_pack_index(const lsnf_plan* plan, int32_t index, int32_t ci, int32_t co, int32_t ky,
                                    int32_t kx, int64_t* row, int64_t* col) {
  if (!plan || index < 0 || index >= (int)plan->stages.size() || !row || !col) return fail(LSNF_ERR_INVALID, "bad argument");
  const StageHost& st = plan->stages[index];
  if (ci < 0 || ci >= st.ci || co < 0 || co >= st.co || ky < 0 || ky >= st.k || kx < 0 || kx >= st.k)
    return fail(LSNF_ERR_INVALID, "weight index out of range");
  long long r, c;
  pack_index(geom_of(st), ci, co, ky, kx, &r, &c);
  *row = r; *col = c;
  return LSNF_OK;
}

// Operand and output pointers of a stage in the bound workspace, and its launch on the plan's device; with
// `encode`, its tensor maps.
static int bind_stage(lsnf_plan* plan, StageHost& st, bool encode) {
  StageDev& d = st.dev;
  d.a = (const __nv_bfloat16*)(plan->ws + st.info.a_offset);
  d.b = (const __nv_bfloat16*)(plan->ws + st.info.b_offset);
  d.out = plan->ws + st.info.out_offset;
  st.launch = tc_plan_launch(st, plan->num_sms);
  d.nst = st.launch.info.ring_stages;
  d.sk_enable = st.launch.info.stream_k;
  d.out_tma = st.launch.info.tma_store;
  return encode ? tc_encode_maps(plan, st) : LSNF_OK;
}

extern "C" int lsnf_plan_bind(lsnf_plan* plan, void* workspace, size_t bytes) {
  if (!plan || !workspace) return fail(LSNF_ERR_INVALID, "null argument");
  if (bytes < plan->ws_bytes) return fail(LSNF_ERR_INVALID, "workspace too small");
  if ((uintptr_t)workspace % 1024) return fail(LSNF_ERR_INVALID, "workspace must be 1024-byte aligned");
  int dev = -1;
  LSNF_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  LSNF_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) return fail(LSNF_ERR_CUDA, "this library is built for sm_100a (B200) only");
  plan->device = dev;
  plan->num_sms = prop.multiProcessorCount;
  plan->ws = (char*)workspace;
  {
    int rc;
    if ((rc = tc_prepare_device(dev)) || (rc = aux_prepare_device(dev)) || (rc = flow_prepare_device(dev))) return rc;
  }
  for (size_t i = 0; i < plan->stages.size(); ++i) {
    StageHost& st = plan->stages[i];
    const lsnf_stage_info& I = st.info;
    StageDev& d = st.dev;
    d.bias = (I.kind == 0 && !st.last) ? (const float*)(plan->ws + st.bias_off) : nullptr;
    d.sk_slots = (float*)(plan->ws + plan->off_sk_slots);
    d.sk_flags = (int32_t*)(plan->ws + plan->off_sk_flags);
    d.descale = (I.kind == 0 || plan->cfg.bwd_passes == 1) ? (const float*)(plan->ws + plan->off_wscale + (size_t)I.layer * 16 + 8) : nullptr;
    if (d.cross8) d.descale = (const float*)(plan->ws + st.x8_off + 4);
    d.amax_reset = d.cross8 ? (uint32_t*)(plan->ws + st.x8_off) : nullptr;
    // the data-gradient stage before a cross8 stage writes that stage's input
    const bool feeds8 = i + 1 < plan->stages.size() && plan->stages[i + 1].dev.cross8;
    d.amax_out = feeds8 ? (uint32_t*)(plan->ws + plan->stages[i + 1].x8_off) : nullptr;
    d.mbits = ((I.kind == 0 && !st.last) || (I.kind == 1 && !st.first)) ? (uint32_t*)(plan->ws + st.mbits_off) : nullptr;
    if (st.meas) d.descale = nullptr;   // the operator's 2^k is carried to the fp32 post-scale (meas_post_scale)
    int rc = bind_stage(plan, st, plan->cfg.gemm_impl == LSNF_GEMM_TCGEN05);
    if (rc) return rc;
  }
  for (auto& w : plan->wg) {
    int rc = bind_stage(plan, w.st, true);
    if (rc) return rc;
    w.ta.dst = (uint16_t*)(plan->ws + w.off_aT);
    w.tg.dst = (uint16_t*)(plan->ws + w.off_gT);
    w.fin.part = (const float*)(plan->ws + w.off_part);
    w.rs.src = (const uint16_t*)(plan->ws + w.off_gT);
  }
  if (!plan->side) {
    LSNF_CUDA(cudaStreamCreateWithFlags(&plan->side, cudaStreamNonBlocking));
    LSNF_CUDA(cudaEventCreateWithFlags(&plan->ev_fork, cudaEventDisableTiming));
    LSNF_CUDA(cudaEventCreateWithFlags(&plan->ev_join, cudaEventDisableTiming));
    LSNF_CUDA(cudaStreamCreateWithFlags(&plan->cap_stream, cudaStreamNonBlocking));
  }
  for (auto& g : plan->graphs) cudaGraphExecDestroy(g.exec);
  plan->graphs.clear();
  plan->runs = 0;
  {
    const char* e = getenv("LSNF_NO_GRAPH");
    plan->use_graphs = !(e && e[0] == '1');
  }
  plan->bound = true;
  plan->g_packed = plan->f_packed = plan->meas_packed = false;
  return LSNF_OK;
}

static int need(const lsnf_plan* p, bool gen, bool flow) {
  if (!p) return fail(LSNF_ERR_INVALID, "null plan");
  if (!p->bound) return fail(LSNF_ERR_STATE, "lsnf_plan_bind has not been called");
  if (gen && p->n_layers == 0) return fail(LSNF_ERR_STATE, "plan has no generator (arch = none)");
  if (gen && !p->g_packed) return fail(LSNF_ERR_STATE, "generator weights not packed");
  if (flow && !p->f_packed) return fail(LSNF_ERR_STATE, "flow weights not packed");
  return 0;
}

static int run_stage(const lsnf_plan* p, const StageHost& st, cudaStream_t s) {
  return p->cfg.gemm_impl == LSNF_GEMM_TCGEN05 ? launch_tapgemm_tc(st, s) : launch_tapgemm_simt(st, s);
}

// A data-gradient stage of a chain: a cross8 stage first converts the gradient its predecessor just wrote.
// (lsnf_plan_run_stage runs the tap-GEMM alone, on the operand the last chain call converted.)
static int run_dgrad_stage(const lsnf_plan* p, const StageHost& st, cudaStream_t s) {
  if (st.dev.cross8) {
    const int rc = launch_convert_fp8(p, st, s);
    if (rc) return rc;
  }
  return run_stage(p, st, s);
}

extern "C" int lsnf_pack_generator_weights(lsnf_plan* plan, const float* const* weights, const float* const* biases,
                                           int32_t n_layers, lsnf_stream stream) {
  if (!plan || !plan->bound) return fail(LSNF_ERR_STATE, "plan not bound");
  if (n_layers != plan->n_layers || !weights || !biases) return fail(LSNF_ERR_INVALID, "layer count mismatch");
  cudaStream_t s = (cudaStream_t)stream;
  {
    int rc = launch_weight_scales(plan, weights, s);
    if (rc) return rc;
  }
  for (auto& st : plan->stages) {
    if (st.meas) continue;   // packed by lsnf_pack_measurement
    int rc = launch_pack_stage(plan, st, weights[st.info.layer], s);
    if (rc) return rc;
    // a cross8 stage's input amax starts at 0; from then on the stage zeroes it after each conversion
    if (st.dev.cross8) LSNF_CUDA(cudaMemsetAsync(plan->ws + st.x8_off, 0, 16, s));
  }
  for (int l = 0; l < plan->n_layers; ++l)
    LSNF_CUDA(cudaMemcpyAsync(plan->ws + plan->off_bias[l], biases[l], (size_t)plan->layers[l].co * 4,
                              cudaMemcpyDeviceToDevice, s));
  plan->g_packed = true;
  plan->wg_ready = false;   // activations and gradients in the workspace belong to the old weights
  return LSNF_OK;
}

extern "C" int lsnf_pack_flow_weights(lsnf_plan* plan, const float* const* params, const int32_t* const* perm,
                                      const int32_t* const* perm_inverse, const float* log_abs_det,
                                      const float* const* w_inverse, lsnf_stream stream) {
  if (!plan || !plan->bound) return fail(LSNF_ERR_STATE, "plan not bound");
  if (!params) return fail(LSNF_ERR_INVALID, "null argument");
  if (plan->cfg.f_permutation == 1 && (!perm || !perm_inverse)) return fail(LSNF_ERR_INVALID, "permutation indices missing");
  int rc;
  const float* winv_ptrs[32];
  if (!log_abs_det && plan->cfg.f_permutation == 2) {
    // the library evaluates log|det W| (fp64) and W^-1 itself: one launch, one CTA per step
    float* winv = (float*)(plan->ws + plan->off_flinalg);
    float* ld = winv + (size_t)plan->cfg.f_depth * plan->cfg.nz * plan->cfg.nz;
    if ((rc = launch_flow_logdet_inverse(plan, params, winv, ld, (cudaStream_t)stream))) return rc;
    for (int i = 0; i < plan->cfg.f_depth; ++i) winv_ptrs[i] = winv + (size_t)i * plan->cfg.nz * plan->cfg.nz;
    log_abs_det = ld;
    w_inverse = winv_ptrs;
  }
  rc = launch_flow_pack(plan, params, perm, perm_inverse, log_abs_det, w_inverse, (cudaStream_t)stream);
  if (rc) return rc;
  plan->f_packed = true;
  plan->have_winv = (w_inverse != nullptr) || plan->cfg.f_permutation == 1;
  return LSNF_OK;
}

static int gen_forward(lsnf_plan* p, const float* z, float* x_hat, cudaStream_t s, bool split) {
  int rc;
  if (split && (rc = launch_split_z(p, z, s))) return rc;
  for (int l = 0; l < p->n_layers; ++l)
    if ((rc = run_stage(p, p->stages[l], s))) return rc;
  uint16_t* xhl = p->meas_m ? (uint16_t*)(p->ws + p->off_meas_xhl) : nullptr;   // for lsnf_generator_dgrad_measured
  if ((rc = launch_last_gather(p, nullptr, 0, s, xhl))) return rc;
  if (x_hat) {
    const size_t bytes = (size_t)p->cfg.batch * p->cfg.nc * p->img * p->img * 4;
    LSNF_CUDA(cudaMemcpyAsync(x_hat, p->ws + p->off_xhat, bytes, cudaMemcpyDeviceToDevice, s));
  }
  return LSNF_OK;
}

static int gen_dgrad_partial(lsnf_plan* p, const float* x, const float* mask, float sigma, cudaStream_t s) {
  int rc;
  if ((rc = launch_recon_grad_im2col(p, x, mask, sigma_seed_scale(sigma), 0, s))) return rc;
  for (int i = p->n_layers; i < 2 * p->n_layers; ++i)
    if ((rc = run_dgrad_stage(p, p->stages[i], s))) return rc;
  return LSNF_OK;
}

// Loss-gradient seed of a measured iteration, from the last forward stage's per-tap products: x_hat (with its fp16 rows),
// A x_hat, r = A x_hat - y (and the |r|^2 partials into epart, nullable), A^T r, and the last layer's im2col seed
// A^T r (1 - x_hat^2).  r carries seed_scale, the share of 1/sigma^2 kept in the 16-bit tensors, and the operator's
// 2^k (A^T r 2^2k): see meas_post_scale.
static int meas_seed(const lsnf_plan* p, const float* y, float* epart, float seed_scale, cudaStream_t s) {
  const int L = p->n_layers;
  const StageHost& bw = p->stages[2 * L + 1];
  int rc;
  if ((rc = launch_last_gather(p, nullptr, 0, s, (uint16_t*)(p->ws + p->off_meas_xhl))) ||
      (rc = run_stage(p, p->stages[2 * L], s)) || (rc = launch_meas_finish(p, y, seed_scale, epart, s)) ||
      (rc = run_stage(p, bw, s)))
    return rc;
  return launch_recon_grad_im2col(p, nullptr, nullptr, 1.f, 1, s, (const float*)(p->ws + bw.info.out_offset),
                                  bw.info.k_splits, bw.info.n_pad);
}

// The fp32 factor of the first layer's split-K sum of a measured gradient: the share of 1/sigma^2 the seed did not
// apply, and 2^-2k for the operator's scale that r (2^k) and A^T r (2^2k) carry.
static float meas_post_scale(const lsnf_plan* p, float sigma) {
  return ldexpf(sigma_post_scale(sigma), -2 * p->meas_k);
}

// The measured entry points' own conditions (after need()).
static int need_measured(const lsnf_plan* p) {
  if (p->cfg.meas_rows == 0) return fail(LSNF_ERR_UNSUPPORTED, "plan was created without lsnf_config.meas_rows");
  if (p->cfg.bwd_passes == 1)
    return fail(LSNF_ERR_UNSUPPORTED, "measurements need the 3-pass bf16 data gradient (bwd_passes 1 writes an fp16 "
                                      "seed, and A^T r has no bounded range)");
  if (!p->meas_packed) return fail(LSNF_ERR_INVALID, "no measurement operator packed (lsnf_pack_measurement)");
  return LSNF_OK;
}

extern "C" int lsnf_pack_measurement(lsnf_plan* plan, const float* A, lsnf_stream stream) {
  if (!plan || !plan->bound) return fail(LSNF_ERR_STATE, "plan not bound");
  if (plan->cfg.meas_rows == 0) return fail(LSNF_ERR_UNSUPPORTED, "plan was created without lsnf_config.meas_rows");
  if (!A) return fail(LSNF_ERR_INVALID, "null operator");
  int rc = launch_meas_pack(plan, A, &plan->meas_k, (cudaStream_t)stream);
  if (rc) return rc;
  plan->meas_packed = true;
  return LSNF_OK;
}

extern "C" int lsnf_generator_dgrad_measured(lsnf_plan* plan, const float* y, float sigma, float* grad_z,
                                             lsnf_stream stream) {
  int rc = need(plan, true, false);
  if (rc || (rc = need_measured(plan))) return rc;
  if (!y || !grad_z || !(sigma > 0.f)) return fail(LSNF_ERR_INVALID, "bad argument");
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = meas_seed(plan, y, nullptr, sigma_seed_scale(sigma), s))) return rc;
  for (int i = plan->n_layers; i < 2 * plan->n_layers; ++i)
    if ((rc = run_dgrad_stage(plan, plan->stages[i], s))) return rc;
  return launch_reduce_partial(plan, grad_z, meas_post_scale(plan, sigma), s);
}

extern "C" int lsnf_plan_run_stage(lsnf_plan* plan, int32_t index, lsnf_stream stream) {
  int rc = need(plan, true, false);
  if (rc) return rc;
  if (index < 0 || index >= (int)plan->stages.size()) return fail(LSNF_ERR_INVALID, "bad stage index");
  // a stage run alone leaves the amax words of the chain alone: the next chain call's e4m3 scales depend on that
  // call's gradients only
  StageHost alone = plan->stages[index];
  alone.dev.amax_out = alone.dev.amax_reset = nullptr;
  return run_stage(plan, alone, (cudaStream_t)stream);
}

extern "C" int lsnf_generator_forward(lsnf_plan* plan, const float* z, float* x_hat, lsnf_stream stream) {
  int rc = need(plan, true, false);
  if (rc) return rc;
  if (!z) return fail(LSNF_ERR_INVALID, "null z");
  return gen_forward(plan, z, x_hat, (cudaStream_t)stream, true);
}

extern "C" int lsnf_generator_dgrad_masked(lsnf_plan* plan, const float* x, const float* mask, float sigma,
                                           float* grad_z, lsnf_stream stream) {
  int rc = need(plan, true, false);
  if (rc) return rc;
  if (!x || !grad_z || !(sigma > 0.f)) return fail(LSNF_ERR_INVALID, "bad argument");
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = gen_dgrad_partial(plan, x, mask, sigma, s))) return rc;
  return launch_reduce_partial(plan, grad_z, sigma_post_scale(sigma), s);
}

extern "C" int lsnf_generator_dgrad(lsnf_plan* plan, const float* x, float sigma, float* grad_z, lsnf_stream stream) {
  return lsnf_generator_dgrad_masked(plan, x, nullptr, sigma, grad_z, stream);
}

extern "C" int lsnf_flow_forward(lsnf_plan* plan, const float* z, float* z_out, float* logdet, float* logp,
                                 float* grad_z, lsnf_stream stream) {
  int rc = need(plan, false, true);
  if (rc) return rc;
  if (!z) return fail(LSNF_ERR_INVALID, "null z");
  return launch_flow_forward(plan, z, z_out, logdet, logp, grad_z, (cudaStream_t)stream);
}

extern "C" int lsnf_flow_inverse(lsnf_plan* plan, const float* eps, float* z, float* neg_objective, lsnf_stream stream) {
  int rc = need(plan, false, true);
  if (rc) return rc;
  if (!eps || !z) return fail(LSNF_ERR_INVALID, "null argument");
  if (!plan->have_winv) return fail(LSNF_ERR_STATE, "flow weights were packed without w_inverse");
  return launch_flow_inverse(plan, eps, z, neg_objective, (cudaStream_t)stream);
}

extern "C" size_t lsnf_generator_grad_floats(const lsnf_plan* plan) { return plan ? plan->gen_grad_floats : 0; }

extern "C" int lsnf_generator_grad_layout(const lsnf_plan* plan, int64_t* offsets, int64_t* sizes) {
  if (!plan || !offsets || !sizes) return fail(LSNF_ERR_INVALID, "null argument");
  if (plan->wg.empty()) return fail(LSNF_ERR_STATE, "plan was created without lsnf_config.train");
  for (int l = 0; l < plan->n_layers; ++l) {
    const auto& y = plan->layers[l];
    offsets[2 * l] = (int64_t)plan->wg[l].grad_w_off; sizes[2 * l] = (int64_t)y.ci * y.co * y.k * y.k;
    offsets[2 * l + 1] = (int64_t)plan->wg[l].grad_b_off; sizes[2 * l + 1] = y.co;
  }
  return LSNF_OK;
}

// LSNF_SYNC_DEBUG=1: synchronise after every step of the generator's parameter gradients and name the one that failed
static int sync_check(cudaStream_t s, const char* what, int l) {
  static const bool dbg = [] { const char* e = getenv("LSNF_SYNC_DEBUG"); return e && e[0] == '1'; }();
  if (!dbg) return 0;
  cudaError_t e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) return 0;
  set_error(std::string("CUDA error: ") + cudaGetErrorString(e) + " after " + what + " of layer " + std::to_string(l));
  return LSNF_ERR_CUDA;
}

// weight and bias gradient of layer l from the activations and the data-gradient tensors in the workspace, times scale
static int gen_layer_grads(lsnf_plan* plan, int l, float* grads, float scale, cudaStream_t s) {
  const int L = plan->n_layers;
  int rc;
  WgradLayer& w = plan->wg[l];
  TransArgs ta = w.ta, tg = w.tg;
  ta.src = (const uint16_t*)(plan->ws + (l == 0 ? plan->off_zhl : plan->off_act[l - 1]));
  tg.src = (const uint16_t*)(plan->ws + (l == L - 1 ? plan->off_im2col : plan->off_gpre[l]));
  if ((rc = launch_transpose_hl(ta, s)) || (rc = sync_check(s, "activation transpose", l))) return rc;
  if ((rc = launch_transpose_hl(tg, s)) || (rc = sync_check(s, "gradient transpose", l))) return rc;
  if ((rc = launch_tapgemm_tc(w.st, s)) || (rc = sync_check(s, "weight-gradient tap-GEMM", l))) return rc;
  FinalizeArgs f = w.fin;
  f.out = grads + w.grad_w_off; f.scale = scale;
  if ((rc = launch_wgrad_finalize(f, s)) || (rc = sync_check(s, "finalize", l))) return rc;
  RowSumArgs r = w.rs;
  r.out = grads + w.grad_b_off; r.scale = scale;
  if ((rc = launch_bias_rowsum(r, s)) || (rc = sync_check(s, "bias row sums", l))) return rc;
  return LSNF_OK;
}

extern "C" int lsnf_generator_param_grads_masked(lsnf_plan* plan, const float* z, const float* x, const float* mask,
                                                 int32_t global_batch, float* grads, float* loss, int32_t part,
                                                 lsnf_stream stream) {
  int rc = need(plan, true, false);
  if (rc) return rc;
  if (plan->wg.empty()) return fail(LSNF_ERR_STATE, "plan was created without lsnf_config.train");
  if (plan->cfg.gemm_impl != LSNF_GEMM_TCGEN05) return fail(LSNF_ERR_UNSUPPORTED, "weight gradients need the tcgen05 path");
  if (!z || !x || !grads || global_batch <= 0) return fail(LSNF_ERR_INVALID, "bad argument");
  if (part < -2 || part >= plan->n_layers) return fail(LSNF_ERR_INVALID, "part must be -1 (all), -2 (prologue) or a layer");
  cudaStream_t s = (cudaStream_t)stream;
  const lsnf_config& c = plan->cfg;
  const int L = plan->n_layers;
  const bool prologue = part < 0, layers_all = part == -1;
  if (prologue) {
    // x_hat = G(z_k) (train.py:392) and loss_g = mse_sum / B (train.py:393)
    if ((rc = gen_forward(plan, z, nullptr, s, true))) return rc;
    if ((rc = sync_check(s, "generator forward", -1))) return rc;
    const long long npix = (long long)c.batch * c.nc * plan->img * plan->img;
    // partial sums in the (idle) norm scratch of the update kernel, ticket next to its own
    if (loss && (rc = launch_mse_sum((const float*)(plan->ws + plan->off_xhat), x, mask, npix, 1.f / (float)global_batch,
                                     (float*)(plan->ws + plan->off_flow_out),
                                     (unsigned int*)(plan->ws + plan->off_scalars + 64), loss, s)))
      return rc;
    // backward through the generator: seed (x_hat - x)(1 - x_hat^2) unscaled; the factor 2 / B of the loss is applied
    // in fp32 when the gradients are finalized.  The first layer's data gradient is not needed.
    if ((rc = launch_last_fused(plan, x, mask, nullptr, 1.f, s))) return rc;
    for (int i = L; i < 2 * L - 1; ++i)
      if ((rc = run_dgrad_stage(plan, plan->stages[i], s))) return rc;
    if ((rc = sync_check(s, "data-gradient chain", -1))) return rc;
    plan->wg_ready = true;
    plan->wg_measured = false;
    if (!layers_all) return LSNF_OK;
  }
  if (!plan->wg_ready || plan->wg_measured)
    return fail(LSNF_ERR_STATE, "a layer's gradients were requested before the forward / data-gradient part (part = -2)");
  const float scale = 2.f / (float)global_batch;
  for (int l = L - 1; l >= 0; --l) {
    if (!layers_all && l != part) continue;
    if ((rc = gen_layer_grads(plan, l, grads, scale, s))) return rc;
  }
  return LSNF_OK;
}

extern "C" int lsnf_generator_param_grads(lsnf_plan* plan, const float* z, const float* x, int32_t global_batch,
                                          float* grads, float* loss, int32_t part, lsnf_stream stream) {
  return lsnf_generator_param_grads_masked(plan, z, x, nullptr, global_batch, grads, loss, part, stream);
}

// The measured loss loss_g = |A vec(G(z)) - y|^2 / global_batch.  The prologue is the measured Langevin iteration's
// generator half at seed scale 1: r carries 2^k and the last layer's im2col seed A^T r (1 - x_hat^2) carries 2^2k, so
// the factor 2 / global_batch of the loss and 2^-2k are applied together in fp32 when the gradients are finalized, and
// 2^-2k / global_batch to the |r 2^k|^2 partials the finisher leaves in the measured regions.
extern "C" int lsnf_generator_param_grads_measured(lsnf_plan* plan, const float* z, const float* y,
                                                   int32_t global_batch, float* grads, float* loss, int32_t part,
                                                   lsnf_stream stream) {
  int rc = need(plan, true, false);
  if (rc || (rc = need_measured(plan))) return rc;
  if (plan->wg.empty()) return fail(LSNF_ERR_STATE, "plan was created without lsnf_config.train");
  if (plan->cfg.gemm_impl != LSNF_GEMM_TCGEN05) return fail(LSNF_ERR_UNSUPPORTED, "weight gradients need the tcgen05 path");
  if (part < -2 || part >= plan->n_layers) return fail(LSNF_ERR_INVALID, "part must be -1 (all), -2 (prologue) or a layer");
  const bool prologue = part < 0, layers_all = part == -1;
  if (!z || (prologue && !y) || !grads || global_batch <= 0) return fail(LSNF_ERR_INVALID, "bad argument");
  cudaStream_t s = (cudaStream_t)stream;
  const int L = plan->n_layers;
  if (prologue) {
    if ((rc = launch_split_z(plan, z, s))) return rc;
    for (int l = 0; l < L; ++l)
      if ((rc = run_stage(plan, plan->stages[l], s))) return rc;
    float* epart = (float*)(plan->ws + plan->off_meas_epart);
    if ((rc = meas_seed(plan, y, epart, 1.f, s))) return rc;
    if ((rc = sync_check(s, "generator forward and measurement seed", -1))) return rc;
    if (loss && (rc = launch_meas_loss(epart, plan->cfg.batch * plan->meas_tiles,
                                       ldexpf(1.f / (float)global_batch, -2 * plan->meas_k), loss, s)))
      return rc;
    for (int i = L; i < 2 * L - 1; ++i)
      if ((rc = run_dgrad_stage(plan, plan->stages[i], s))) return rc;
    if ((rc = sync_check(s, "data-gradient chain", -1))) return rc;
    plan->wg_ready = plan->wg_measured = true;
    if (!layers_all) return LSNF_OK;
  }
  if (!plan->wg_ready || !plan->wg_measured)
    return fail(LSNF_ERR_STATE, "a layer's gradients were requested before the measured forward / data-gradient part "
                                "(part = -2)");
  const float scale = ldexpf(2.f / (float)global_batch, -2 * plan->meas_k);
  for (int l = L - 1; l >= 0; --l) {
    if (!layers_all && l != part) continue;
    if ((rc = gen_layer_grads(plan, l, grads, scale, s))) return rc;
  }
  return LSNF_OK;
}

extern "C" int lsnf_generator_vjp(lsnf_plan* plan, const float* grad_x_hat, float* grad_z, float* grads,
                                  lsnf_stream stream) {
  int rc = need(plan, true, false);
  if (rc) return rc;
  if (!grad_x_hat) return fail(LSNF_ERR_INVALID, "null grad_x_hat");
  if (plan->cfg.bwd_passes == 1)
    return fail(LSNF_ERR_UNSUPPORTED, "the vector-Jacobian product needs the 3-pass bf16 data gradient (bwd_passes 1 "
                                      "has fp16's range, too narrow for an arbitrary upstream gradient)");
  if (grads && plan->wg.empty()) return fail(LSNF_ERR_STATE, "plan was created without lsnf_config.train");
  if (grads && plan->cfg.gemm_impl != LSNF_GEMM_TCGEN05)
    return fail(LSNF_ERR_UNSUPPORTED, "weight gradients need the tcgen05 path");
  cudaStream_t s = (cudaStream_t)stream;
  const int L = plan->n_layers;
  // seed g = dL/dx_hat * (1 - x_hat^2) at scale 1 (bf16 keeps fp32's exponent range), x_hat of the last forward pass
  if ((rc = launch_recon_grad_im2col(plan, grad_x_hat, nullptr, 1.f, 1, s))) return rc;
  const int end = grad_z ? 2 * L : 2 * L - 1;   // the first layer's data gradient only feeds dL/dz
  for (int i = L; i < end; ++i)
    if ((rc = run_dgrad_stage(plan, plan->stages[i], s))) return rc;
  if (grad_z && (rc = launch_reduce_partial(plan, grad_z, 1.f, s))) return rc;
  // the gradient tensors no longer hold the part = -2 state of lsnf_generator_param_grads
  plan->wg_ready = false;
  if (grads)
    for (int l = L - 1; l >= 0; --l)
      if ((rc = gen_layer_grads(plan, l, grads, 1.f, s))) return rc;
  return LSNF_OK;
}

extern "C" size_t lsnf_flow_grad_floats(const lsnf_plan* plan) {
  return plan ? plan->fgrad.step_floats * (size_t)plan->cfg.f_depth : 0;
}

extern "C" int lsnf_flow_grad_layout(const lsnf_plan* plan, int64_t* offsets, int64_t* sizes) {
  if (!plan || !offsets || !sizes) return fail(LSNF_ERR_INVALID, "null argument");
  for (int L = 0; L < plan->cfg.f_depth; ++L)
    for (int i = 0; i < LSNF_FLOW_PTRS_PER_STEP; ++i) {
      offsets[L * LSNF_FLOW_PTRS_PER_STEP + i] = (int64_t)(L * plan->fgrad.step_floats + plan->fgrad.off[i]);
      sizes[L * LSNF_FLOW_PTRS_PER_STEP + i] = (int64_t)plan->fgrad.size[i];
    }
  return LSNF_OK;
}

extern "C" int lsnf_flow_param_grads(lsnf_plan* plan, const float* z, int32_t global_batch, float* grads, float* loss,
                                     lsnf_stream stream) {
  int rc = need(plan, false, true);
  if (rc) return rc;
  if (!z || !grads || global_batch <= 0) return fail(LSNF_ERR_INVALID, "bad argument");
  if (plan->cfg.f_permutation == 2 && !plan->have_winv)
    return fail(LSNF_ERR_STATE, "flow weights were packed without w_inverse (needed for d log|det W| / dW = W^-T)");
  return launch_flow_param_grads(plan, z, 1.f / (float)global_batch, grads, loss, (cudaStream_t)stream);
}

extern "C" int lsnf_flow_vjp(lsnf_plan* plan, const float* z, const float* grad_z_out, const float* grad_logdet,
                             float* grad_z, float* grads, lsnf_stream stream) {
  int rc = need(plan, false, true);
  if (rc) return rc;
  if (!z) return fail(LSNF_ERR_INVALID, "null z");
  if (grads && plan->cfg.f_permutation == 2 && !plan->have_winv)
    return fail(LSNF_ERR_STATE, "flow weights were packed without w_inverse (needed for d log|det W| / dW = W^-T)");
  cudaStream_t s = (cudaStream_t)stream;
  if (!grad_z_out && !grad_logdet) {
    // a zero upstream gradient (the fused kernel reads two null seeds as those of -sum_b log p)
    if (grad_z) LSNF_CUDA(cudaMemsetAsync(grad_z, 0, (size_t)plan->cfg.batch * plan->cfg.nz * 4, s));
    if (grads) LSNF_CUDA(cudaMemsetAsync(grads, 0, lsnf_flow_grad_floats(plan) * 4, s));
    return LSNF_OK;
  }
  if (!grad_z && !grads) return LSNF_OK;
  return launch_flow_vjp(plan, z, grad_z_out, grad_logdet, grad_z, grads, s);
}

extern "C" int lsnf_adam_step(int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                              float* const* exp_avg_sq, const int64_t* sizes, const int32_t* grad_kk,
                              const int32_t* grad_inner, float lr, float beta1, float beta2, float eps,
                              float weight_decay, int64_t step, const float* grad_scale, lsnf_stream stream) {
  if (n_tensors <= 0 || !params || !grads || !exp_avg || !exp_avg_sq || !sizes || step <= 0)
    return fail(LSNF_ERR_INVALID, "bad argument");
  return launch_adam(n_tensors, params, grads, exp_avg, exp_avg_sq, sizes, grad_kk, grad_inner, lr, beta1, beta2, eps,
                     weight_decay, step, grad_scale, (cudaStream_t)stream);
}

extern "C" int lsnf_sample_prior(lsnf_plan* plan, const float* eps, float* x, float* z, int32_t to_unit_range,
                                 lsnf_stream stream) {
  int rc = need(plan, true, true);
  if (rc) return rc;
  if (!eps || !x) return fail(LSNF_ERR_INVALID, "null argument");
  if (!plan->have_winv) return fail(LSNF_ERR_STATE, "flow weights were packed without w_inverse");
  cudaStream_t s = (cudaStream_t)stream;
  float* zw = (float*)(plan->ws + plan->off_z);
  if ((rc = launch_flow_inverse(plan, eps, zw, nullptr, s))) return rc;          // train.py:568-569
  if ((rc = launch_split_z(plan, zw, s))) return rc;
  for (int l = 0; l < plan->n_layers; ++l)                                        // train.py:572
    if ((rc = run_stage(plan, plan->stages[l], s))) return rc;
  if ((rc = launch_last_gather(plan, x, to_unit_range, s))) return rc;            // train.py:573 fused into the store
  if (z) LSNF_CUDA(cudaMemcpyAsync(z, zw, (size_t)plan->cfg.batch * plan->cfg.nz * 4, cudaMemcpyDeviceToDevice, s));
  return LSNF_OK;
}

extern "C" int lsnf_langevin_update(lsnf_plan* plan, float* z, const float* grad_g, const float* grad_f,
                                    float step_size, const float* eps, int32_t with_noise, uint64_t seed,
                                    uint64_t sample_offset, uint32_t step, float* gnorms, lsnf_stream stream) {
  if (!plan || !plan->bound) return fail(LSNF_ERR_STATE, "plan not bound");
  if (!z || !grad_g || !grad_f) return fail(LSNF_ERR_INVALID, "null argument");
  return launch_update(plan, z, grad_g, nullptr, 0, 1.f, grad_f, step_size, eps, with_noise, seed, sample_offset, step,
                       nullptr, gnorms, 0, (cudaStream_t)stream);
}

// Loop iterations per captured graph.  An AIS chunk reads graph_chunk + 1 schedule values from the workspace.
constexpr int graph_chunk = 40;
static_assert(graph_chunk < AIS_BETA_FLOATS, "the workspace schedule copy must hold a chunk's values");

extern "C" int lsnf_langevin_launch_count(const lsnf_plan* plan, int32_t steps) {
  if (!plan) return 0;
  // per step: L forward + fused gather/tanh/seed/im2col + L data-gradient (each cross8 stage with its operand
  // conversion) + flow + update; once: split_z; per replayed graph chunk: the kernel that sets (seed, sample offset,
  // first step index) in device memory
  const int chunks = steps > 0 ? (steps + graph_chunk - 1) / graph_chunk : 0;
  int conversions = 0;
  for (const auto& st : plan->stages) conversions += st.dev.cross8;
  return 1 + steps * (2 * plan->n_layers + 3 + conversions) + chunks;
}

// the g_l_steps loop on stream s: inputs are the workspace copies of z and x (and of the mask, nullable)
// LSNF_TRACE=1: time every launch of the second iteration in situ with CUDA events and print the table to stderr
struct LoopTrace {
  std::vector<cudaEvent_t> ev;
  std::vector<std::string> name;
  cudaStream_t s;
  bool on = false;
  void mark(const char* n) {
    if (!on) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, s);
    ev.push_back(e);
    name.push_back(n);
  }
  void report() {
    if (!on || ev.empty()) return;
    cudaEventSynchronize(ev.back());
    float total = 0.f;
    cudaEventElapsedTime(&total, ev.front(), ev.back());
    fprintf(stderr, "[lsnf trace] one Langevin iteration: %.1f us\n", total * 1e3f);
    for (size_t i = 1; i < ev.size(); ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
      fprintf(stderr, "[lsnf trace]   %-28s %8.1f us\n", name[i].c_str(), ms * 1e3f);
    }
    for (auto e : ev) cudaEventDestroy(e);
    ev.clear();
    name.clear();
  }
};

// With `ais` (lsnf_ais_run) the same stages also write the per-tile energy partials and log p(z), and the iteration
// ends with the AIS update instead of the Langevin update.
static int langevin_loop(lsnf_plan* plan, const float* x, const float* mask, bool measured, int steps, float step_size,
                         float sigma, int with_noise,
                         const float* eps, uint64_t seed, uint64_t sample_offset, const uint64_t* dyn, float* gnorms,
                         cudaStream_t s, const AisArgs* ais) {
  const float gscale = measured ? meas_post_scale(plan, sigma) : sigma_post_scale(sigma);
  int rc;
  static int trace_env = -1;
  if (trace_env < 0) { const char* e = getenv("LSNF_TRACE"); trace_env = (e && e[0] == '1') ? 1 : 0; }
  LoopTrace tr;
  tr.s = s;
  const lsnf_config& c = plan->cfg;
  float* z = (float*)(plan->ws + plan->off_z);
  float* gf = (float*)(plan->ws + plan->off_gradf);
  const float* partial = (const float*)(plan->ws + plan->off_partial);
  // Programmatic dependent launch across the kernel boundaries of the loop's main stream (lsnf_internal.cuh), on the
  // tcgen05 path unless LSNF_PDL=0.  The update kernel is never launched this way (it also waits for the flow prior's
  // stream), nor is the first kernel of a call or of a captured graph (no kernel precedes it there).
  static const bool pdl_env = [] { const char* e = getenv("LSNF_PDL"); return !(e && strcmp(e, "0") == 0); }();
  const bool use_pdl = pdl_env && c.gemm_impl == LSNF_GEMM_TCGEN05;
  for (int t = 0; t < steps; ++t) {
    tr.on = trace_env == 1 && t == 1 && !dyn;
    tr.mark("start");
    // The flow prior (train.py:316-323) only needs z and runs on the side stream.  It is forked right before the
    // last forward layer so that it overlaps the short, non-persistent kernels (last layer, gather, loss-gradient
    // seed): its few CTAs hold whole SMs for tens of microseconds, which would otherwise delay the cluster launch
    // of the persistent CTA-pair GEMMs.
    const int fork_at = plan->n_layers - 1;
    for (int l = 0; l < plan->n_layers; ++l) {
      if (l == fork_at) {
        LSNF_CUDA(cudaEventRecord(plan->ev_fork, s));
        LSNF_CUDA(cudaStreamWaitEvent(plan->side, plan->ev_fork, 0));
        if ((rc = launch_flow_forward(plan, z, nullptr, nullptr, ais ? ais->logp : nullptr, gf, plan->side))) return rc;
        LSNF_CUDA(cudaEventRecord(plan->ev_join, plan->side));
      }
      {
        PdlScope pdl(use_pdl && (t > 0 || l > 0));
        if ((rc = run_stage(plan, plan->stages[l], s))) return rc;
      }
      tr.mark(("forward layer " + std::to_string(l)).c_str());
    }
    {
      PdlScope pdl(use_pdl);
      float* epart = ais ? ais->epart : nullptr;
      if ((rc = measured ? meas_seed(plan, x, epart, sigma_seed_scale(sigma), s)
                         : launch_last_fused(plan, x, mask, epart, sigma_seed_scale(sigma), s)))
        return rc;
    }
    tr.mark(measured ? "gather + tanh + A x_hat + r + A^T r + im2col" : "gather + tanh + recon grad + im2col");
    for (int i = plan->n_layers; i < 2 * plan->n_layers; ++i) {
      {
        PdlScope pdl(use_pdl);
        if ((rc = run_dgrad_stage(plan, plan->stages[i], s))) return rc;
      }
      tr.mark(("dgrad layer " + std::to_string(plan->stages[i].info.layer)).c_str());
    }
    LSNF_CUDA(cudaStreamWaitEvent(s, plan->ev_join, 0));
    tr.mark("join flow prior");
    const float* e = eps ? eps + (size_t)t * c.batch * c.nz : nullptr;
    if (ais) {
      if ((rc = launch_ais_update(plan, *ais, gf, gscale, seed, sample_offset, (uint32_t)t, dyn, s))) return rc;
    } else if ((rc = launch_update(plan, z, nullptr, partial, plan->ksplit_first, gscale, gf, step_size, e, with_noise,
                                   seed, sample_offset, (uint32_t)t, dyn, t == steps - 1 ? gnorms : nullptr, 1, s))) {
      return rc;
    }
    tr.mark("update");
    tr.report();
  }
  return LSNF_OK;
}

// Runs `iters` loop iterations on the workspace z, with the Langevin update or, with `ais`, the AIS update.  The
// first call of a plan runs eagerly (module load, kernel attributes), and so do calls with injected noise: parity
// runs pass a different eps pointer every time.  Later calls replay CUDA graphs of the loop in chunks of at most
// graph_chunk iterations: one graph per chunk length, the index of a chunk's first iteration (Philox counter) read
// from device memory, so test mode's 8 000-step chains (train.py:606) reuse one 40-iteration graph 200 times instead
// of instantiating 88 000 kernel nodes.  Graphs read the workspace copies of x and the mask, and an AIS graph that of
// its chunk's schedule values, which are staged before each replay.  With `measured`, x is y [B][m].
static int run_chain(lsnf_plan* plan, const float* x, const float* mask, bool measured, int iters, float step_size,
                     float sigma, int with_noise, const float* eps, uint64_t seed, uint64_t sample_offset,
                     float* gnorms, cudaStream_t s, const AisArgs* ais = nullptr) {
  const bool injected = eps || (ais && (ais->eps || ais->u));
  const bool graph_ok = plan->use_graphs && !injected && iters > 0 && plan->runs > 0;
  plan->runs++;
  if (!graph_ok)
    return langevin_loop(plan, x, mask, measured, iters, step_size, sigma, with_noise, eps, seed, sample_offset,
                         nullptr, gnorms, s, ais);
  const lsnf_config& c = plan->cfg;
  float* x_ws = (float*)(plan->ws + (measured ? plan->off_meas_y : plan->off_x));
  float* mask_ws = mask ? (float*)(plan->ws + plan->off_mask) : nullptr;
  float* gn_ws = (float*)(plan->ws + plan->off_gnorms);
  float* beta_ws = (float*)(plan->ws + plan->off_ais_beta);
  const uint64_t* dyn = (const uint64_t*)(plan->ws + plan->off_dyn);
  const size_t xbytes = (size_t)c.batch * (measured ? plan->meas_m : c.nc * plan->img * plan->img) * 4;
  LSNF_CUDA(cudaMemcpyAsync(x_ws, x, xbytes, cudaMemcpyDeviceToDevice, s));
  if (mask) LSNF_CUDA(cudaMemcpyAsync(mask_ws, mask, xbytes, cudaMemcpyDeviceToDevice, s));
  AisArgs ag = {};
  if (ais) { ag = *ais; ag.betas = beta_ws; }
  int rc;
  for (int done = 0; done < iters;) {
    const int n = std::min(iters - done, graph_chunk);
    const lsnf_plan::LoopKey key = {n, step_size, sigma, with_noise, mask != nullptr, ais != nullptr,
                                    ais ? ais->target : 0.f, measured, measured ? plan->meas_k : 0};
    cudaGraphExec_t exec = nullptr;
    for (auto& g : plan->graphs)
      if (g.key == key) exec = g.exec;
    if (!exec) {
      cudaGraph_t graph = nullptr;
      cudaStream_t cs = plan->cap_stream;
      LSNF_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
      rc = langevin_loop(plan, x_ws, mask_ws, measured, n, step_size, sigma, with_noise, nullptr, 0, 0, dyn, gn_ws, cs,
                         ais ? &ag : nullptr);
      cudaError_t ce = cudaStreamEndCapture(cs, &graph);
      if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
      if (ce != cudaSuccess) return cuda_fail(ce, "cudaStreamEndCapture");
      ce = cudaGraphInstantiate(&exec, graph, 0);
      cudaGraphDestroy(graph);
      if (ce != cudaSuccess) return cuda_fail(ce, "cudaGraphInstantiate");
      if (plan->graphs.size() >= 8) { cudaGraphExecDestroy(plan->graphs.front().exec); plan->graphs.erase(plan->graphs.begin()); }
      plan->graphs.push_back({key, exec});
    }
    if (ais) {
      const int nb = std::min(n + 1, iters - done);   // the last iteration reads no next value
      LSNF_CUDA(cudaMemcpyAsync(beta_ws, ais->betas + done, (size_t)nb * 4, cudaMemcpyDeviceToDevice, s));
    }
    if ((rc = launch_set_dyn(plan, seed, sample_offset, (uint32_t)done, s, ais ? (uint32_t)ais->total : 0))) return rc;
    LSNF_CUDA(cudaGraphLaunch(exec, s));
    done += n;
  }
  if (gnorms) LSNF_CUDA(cudaMemcpyAsync(gnorms, gn_ws, 8, cudaMemcpyDeviceToDevice, s));
  return LSNF_OK;
}

static int langevin_run(lsnf_plan* plan, const float* z0, const float* x, const float* mask, bool measured,
                        int32_t steps, float step_size, float sigma, int32_t with_noise, const float* eps,
                        uint64_t seed, uint64_t sample_offset, float* z_out, float* gnorms, lsnf_stream stream) {
  int rc = need(plan, true, true);
  if (rc || (measured && (rc = need_measured(plan)))) return rc;
  if (!z0 || !x || !z_out || steps < 0 || !(sigma > 0.f)) return fail(LSNF_ERR_INVALID, "bad argument");
  cudaStream_t s = (cudaStream_t)stream;
  const lsnf_config& c = plan->cfg;
  float* z = (float*)(plan->ws + plan->off_z);
  const size_t zbytes = (size_t)c.batch * c.nz * 4;
  LSNF_CUDA(cudaMemcpyAsync(z, z0, zbytes, cudaMemcpyDeviceToDevice, s));
  if ((rc = launch_split_z(plan, z, s))) return rc;
  if ((rc = run_chain(plan, x, mask, measured, steps, step_size, sigma, with_noise, eps, seed, sample_offset, gnorms,
                      s)))
    return rc;
  LSNF_CUDA(cudaMemcpyAsync(z_out, z, zbytes, cudaMemcpyDeviceToDevice, s));
  return LSNF_OK;
}

extern "C" int lsnf_langevin_run_masked(lsnf_plan* plan, const float* z0, const float* x, const float* mask,
                                        int32_t steps, float step_size, float sigma, int32_t with_noise,
                                        const float* eps, uint64_t seed, uint64_t sample_offset, float* z_out,
                                        float* gnorms, lsnf_stream stream) {
  return langevin_run(plan, z0, x, mask, false, steps, step_size, sigma, with_noise, eps, seed, sample_offset, z_out,
                      gnorms, stream);
}

extern "C" int lsnf_langevin_run_measured(lsnf_plan* plan, const float* z0, const float* y, int32_t steps,
                                          float step_size, float sigma, int32_t with_noise, const float* eps,
                                          uint64_t seed, uint64_t sample_offset, float* z_out, float* gnorms,
                                          lsnf_stream stream) {
  return langevin_run(plan, z0, y, nullptr, true, steps, step_size, sigma, with_noise, eps, seed, sample_offset, z_out,
                      gnorms, stream);
}

extern "C" int lsnf_langevin_run(lsnf_plan* plan, const float* z0, const float* x, int32_t steps, float step_size,
                                 float sigma, int32_t with_noise, const float* eps, uint64_t seed,
                                 uint64_t sample_offset, float* z_out, float* gnorms, lsnf_stream stream) {
  return lsnf_langevin_run_masked(plan, z0, x, nullptr, steps, step_size, sigma, with_noise, eps, seed, sample_offset,
                                  z_out, gnorms, stream);
}

static int ais_run(lsnf_plan* plan, const float* z0, const float* x, const float* mask, bool measured,
                   const float* betas, int32_t steps, float step_size, float target_accept, float sigma, const float* eps,
                   const float* u, uint64_t seed, uint64_t sample_offset, float* z_out, float* log_w, float* accept_rate,
                   lsnf_stream stream) {
  int rc = need(plan, true, true);
  if (rc || (measured && (rc = need_measured(plan)))) return rc;
  if (!z0 || !x || !betas || !z_out || !log_w || !accept_rate) return fail(LSNF_ERR_INVALID, "null argument");
  if (steps < 1) return fail(LSNF_ERR_INVALID, "steps must be at least 1");
  if (!(sigma > 0.f)) return fail(LSNF_ERR_INVALID, "sigma must be positive");
  if (!(step_size > 0.f)) return fail(LSNF_ERR_INVALID, "step_size must be positive");
  cudaStream_t s = (cudaStream_t)stream;
  const lsnf_config& c = plan->cfg;
  const int B = c.batch;
  float* z = (float*)(plan->ws + plan->off_z);
  const size_t zbytes = (size_t)B * c.nz * 4;
  LSNF_CUDA(cudaMemcpyAsync(z, z0, zbytes, cudaMemcpyDeviceToDevice, s));
  if ((rc = launch_ais_begin(plan, z, s))) return rc;
  AisArgs a;
  a.zc = (float*)(plan->ws + plan->off_ais_z);
  a.gr = (float*)(plan->ws + plan->off_ais_gr);
  a.gp = (float*)(plan->ws + plan->off_ais_gp);
  a.scal = (float*)(plan->ws + plan->off_ais_scal);
  a.logw = (double*)(plan->ws + plan->off_ais_logw);
  a.epart = (float*)(plan->ws + (measured ? plan->off_meas_epart : plan->off_ais_epart));
  a.logp = (float*)(plan->ws + plan->off_ais_logp);
  a.betas = betas; a.eps = eps; a.u = u;
  a.tiles = measured ? plan->meas_tiles : plan->fused_tiles; a.total = steps;
  a.step0 = step_size; a.target = target_accept > 0.f ? target_accept : 0.f;
  a.inv2s2 = measured ? ldexpf(0.5f / (sigma * sigma), -2 * plan->meas_k) : 0.5f / (sigma * sigma);   // |r 2^k|^2
  // steps + 1 iterations: iteration 0 only initialises and proposes, the last one only decides
  if ((rc = run_chain(plan, x, mask, measured, steps + 1, step_size, sigma, 1, nullptr, seed, sample_offset, nullptr, s,
                      &a)))
    return rc;
  LSNF_CUDA(cudaMemcpyAsync(z_out, z, zbytes, cudaMemcpyDeviceToDevice, s));
  LSNF_CUDA(cudaMemcpyAsync(log_w, a.scal + 5 * B, (size_t)B * 4, cudaMemcpyDeviceToDevice, s));
  LSNF_CUDA(cudaMemcpyAsync(accept_rate, a.scal + 6 * B, (size_t)B * 4, cudaMemcpyDeviceToDevice, s));
  return LSNF_OK;
}

extern "C" int lsnf_ais_run(lsnf_plan* plan, const float* z0, const float* x, const float* mask, const float* betas,
                            int32_t steps, float step_size, float target_accept, float sigma, const float* eps,
                            const float* u, uint64_t seed, uint64_t sample_offset, float* z_out, float* log_w,
                            float* accept_rate, lsnf_stream stream) {
  return ais_run(plan, z0, x, mask, false, betas, steps, step_size, target_accept, sigma, eps, u, seed, sample_offset,
                 z_out, log_w, accept_rate, stream);
}

extern "C" int lsnf_ais_run_measured(lsnf_plan* plan, const float* z0, const float* y, const float* betas,
                                     int32_t steps, float step_size, float target_accept, float sigma, const float* eps,
                                     const float* u, uint64_t seed, uint64_t sample_offset, float* z_out, float* log_w,
                                     float* accept_rate, lsnf_stream stream) {
  return ais_run(plan, z0, y, nullptr, true, betas, steps, step_size, target_accept, sigma, eps, u, seed,
                 sample_offset, z_out, log_w, accept_rate, stream);
}
