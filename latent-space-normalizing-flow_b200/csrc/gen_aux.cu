// Small HBM-bound kernels around the generator tap-GEMMs: weight packing, latent splitting, the
// reconstruction-gradient seed (with its im2col), split-K reduction and the fused Langevin update.
#include <cuda_fp8.h>

#include <mutex>

#include "lsnf_internal.cuh"

namespace lsnf {

__device__ __forceinline__ void split_bf16(float v, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(v);
  lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}

// ---------------------------------------------------------------------------------------------------
// weight packing: ConvTranspose2d weight [ci][co][k][k] fp32 -> K-major bf16 hi|lo operand of one stage
// (model.py:57-149 weights; layouts documented at pack_index in lsnf_internal.cuh)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint8_t e4m3(float v) {   // round to nearest, out of range -> +-448
  return (uint8_t)__nv_cvt_float_to_fp8(v, __NV_SATFINITE, __NV_E4M3);
}

// cross8 stages (tc_cross_fp8) split w 2^kw (kw: the e4m3 scale of the layer's max |w|, `wmax`) into fp16 halves
// w_hi + w_lo and take, per 64-column K block of a row, w_hi 2^6 in the hi half's columns and the 128 bytes
// [w_lo8 x 64 | w_hi8 x 64] in the lo half's, w_hi8 = e4m3(w_hi), w_lo8 = e4m3(w_lo 2^11).
__global__ void pack_stage_kernel(const float* __restrict__ w, uint16_t* __restrict__ out, PackGeom g, int rows,
                                  int nz_valid, int fp16, const float* __restrict__ scale,
                                  const unsigned int* __restrict__ wmax) {
  const float sc = scale ? *scale : 1.f;
  const int kw = wmax ? fp8_scale_exp(__uint_as_float(*wmax)) : 0;
  const long long total = (long long)rows * g.ka;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int row = (int)(i / g.ka), col = (int)(i % g.ka);
    int ci = -1, co = -1, tap = -1;
    if (g.kind == 0) {
      ci = col;
      if (g.first || g.last) { tap = row / g.co; co = row % g.co; }
      else { tap = row / g.n_pad; co = row % g.n_pad; }
    } else if (g.first || g.last) {
      ci = row; tap = col / g.co; co = col % g.co;
    } else {
      tap = row / g.n_pad; ci = row % g.n_pad; co = col;
    }
    float v = 0.f;
    if (ci < g.ci && co < g.co && tap < g.k * g.k && ci < nz_valid)
      v = w[((long long)ci * g.co + co) * g.k * g.k + tap] * sc;
    uint16_t hi, lo;
    if (wmax) {
      split16(ldexpf(v, kw), true, hi, lo);
      const float h = __half2float(__ushort_as_half(hi)), l = __half2float(__ushort_as_half(lo));
      out[(long long)row * 2 * g.ka + col] = __half_as_ushort(__float2half_rn(h * 64.f));
      uint8_t* x8 = reinterpret_cast<uint8_t*>(out + (long long)row * 2 * g.ka + g.ka) + (col / 64) * 128 + col % 64;
      x8[0] = e4m3(l * 2048.f);
      x8[64] = e4m3(h);
      continue;
    }
    split16(v, fp16 != 0, hi, lo);
    out[(long long)row * 2 * g.ka + col] = hi;
    out[(long long)row * 2 * g.ka + g.ka + col] = lo;
  }
}

int launch_pack_stage(const lsnf_plan* plan, const StageHost& st, const float* w, cudaStream_t s) {
  const PackGeom g = geom_of(st);
  const int rows = st.info.b_rows;
  const long long total = (long long)rows * g.ka;
  const int threads = 256;
  const int blocks = (int)std::min<long long>((total + threads - 1) / threads, 148 * 16);
  const float* scale = (st.info.kind == 0 || plan->cfg.bwd_passes == 1)
                           ? (const float*)(plan->ws + plan->off_wscale + (size_t)st.info.layer * 16 + 4) : nullptr;
  const unsigned int* wmax =
      st.dev.cross8 ? (const unsigned int*)(plan->ws + plan->off_wscale + (size_t)st.info.layer * 16) : nullptr;
  pack_stage_kernel<<<blocks, threads, 0, s>>>(w, (uint16_t*)(plan->ws + st.info.b_offset), g, rows, st.ci,
                                               st.info.operand_fp16, scale, wmax);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// A operand of a cross8 stage from the bf16 hi|lo gradient its producer wrote, element by element (the phase-split
// layout is kept): the value (hi + lo, exact in fp32) times 2^ka is split into fp16 halves a_hi + a_lo, and each
// 64-channel block of a position holds a_hi 2^5 in the hi half's place and the 128 bytes [a_hi8 x 64 | a_lo8 x 64] in
// the lo half's, a_hi8 = e4m3(a_hi), a_lo8 = e4m3(a_lo 2^11); ka is the e4m3 scale of the gradient's max |value|
// (atomicMax-ed by the producer's epilogue).  With the weights' 2^kw and lifts (pack_stage_kernel) every product of
// the stage carries 2^(ka+kw+11): hi*hi as (a_hi 2^5)(w_hi 2^6), which fp16 holds (2^8 * 2^6 < 65504), the cross
// terms as a_hi8 w_lo8 and a_lo8 w_hi8.  One thread writes 2^-(ka+kw+11) to the stage's descale word; the stage
// zeroes the amax word.
// ---------------------------------------------------------------------------------------------------
// One thread per 16 channels of a position (two 64-channel blocks fill a warp's 512-byte reads), threadIdx.y picks
// the position: every load and store is a 16-byte vector and no index needs a division.
__global__ void __launch_bounds__(256) convert_fp8_kernel(const uint16_t* __restrict__ src, uint16_t* __restrict__ dst,
                                                          int rows, int C, const unsigned int* amax,
                                                          const unsigned int* __restrict__ wmax, float* descale) {
  pdl_wait();
  pdl_trigger();
  const int ka = fp8_scale_exp(__uint_as_float(*amax));
  if (blockIdx.x == 0 && threadIdx.x == 0 && threadIdx.y == 0)
    *descale = ldexpf(1.f, -(ka + fp8_scale_exp(__uint_as_float(*wmax)) + 11));
  const int row = blockIdx.x * blockDim.y + threadIdx.y;
  if (row >= rows) return;
  const float sa = ldexpf(1.f, ka);
  const int c = threadIdx.x * 16;
  const uint16_t* in = src + (size_t)row * 2 * C + c;
  __align__(16) uint16_t h16[16], l16[16];
  *reinterpret_cast<uint4*>(h16) = __ldcs(reinterpret_cast<const uint4*>(in));
  *reinterpret_cast<uint4*>(h16 + 8) = __ldcs(reinterpret_cast<const uint4*>(in + 8));
  *reinterpret_cast<uint4*>(l16) = __ldcs(reinterpret_cast<const uint4*>(in + C));
  *reinterpret_cast<uint4*>(l16 + 8) = __ldcs(reinterpret_cast<const uint4*>(in + C + 8));
  __align__(16) uint16_t hs[16];
  __align__(16) uint8_t h8[16], l8[16];
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const float v = (__bfloat162float(__ushort_as_bfloat16(h16[q])) + __bfloat162float(__ushort_as_bfloat16(l16[q]))) * sa;
    const float h = __half2float(__float2half_rn(v)), l = v - h;
    hs[q] = __half_as_ushort(__float2half_rn(h * 32.f));
    h8[q] = e4m3(h);
    l8[q] = e4m3(l * 2048.f);
  }
  uint16_t* o = dst + (size_t)row * 2 * C;
  *reinterpret_cast<uint4*>(o + c) = *reinterpret_cast<const uint4*>(hs);
  *reinterpret_cast<uint4*>(o + c + 8) = *reinterpret_cast<const uint4*>(hs + 8);
  uint8_t* x8 = reinterpret_cast<uint8_t*>(o + C) + (c / 64) * 128 + c % 64;
  *reinterpret_cast<uint4*>(x8) = *reinterpret_cast<const uint4*>(h8);
  *reinterpret_cast<uint4*>(x8 + 64) = *reinterpret_cast<const uint4*>(l8);
}

int launch_convert_fp8(const lsnf_plan* plan, const StageHost& st, cudaStream_t s) {
  const lsnf_plan::Layer& y = plan->layers[st.info.layer];
  const int C = st.info.k_per_tap;   // a multiple of 64
  const int rows = plan->cfg.batch * y.hout * y.hout;
  const dim3 block(C / 16, std::max(1, 256 / (C / 16)));
  uint32_t* words = (uint32_t*)(plan->ws + st.x8_off);
  LSNF_CUDA(launch_k(convert_fp8_kernel, dim3((rows + block.y - 1) / block.y), block, 0, s,
                     (const uint16_t*)(plan->ws + st.x8_src_off), (uint16_t*)(plan->ws + st.info.a_offset), rows, C,
                     (const unsigned int*)words,
                     (const unsigned int*)(plan->ws + plan->off_wscale + (size_t)st.info.layer * 16),
                     (float*)(words + 1)));
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// per-layer power-of-two weight scale for the fp16 forward operands: 2^k with max|w| * 2^k in [1, 2), so that both
// halves of every weight are normal fp16 numbers; the accumulators are multiplied by 2^-k in the epilogue (exact)
// ---------------------------------------------------------------------------------------------------
__global__ void wmax_kernel(const float* __restrict__ w, long long n, unsigned int* __restrict__ maxbits) {
  float m = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(w[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(maxbits, __float_as_uint(m));  // non-negative floats order like uints
}

// The scale exponent is clamped to [emin, emax]: [-14, 30] for the weights (whose fp16 halves must stay normal fp16
// numbers), [-126, 126] for the measurement operator (whose scale is carried through the measured path, so 2^k and
// 2^-k only have to be normal fp32 numbers).
__global__ void wscale_finalize_kernel(unsigned int* __restrict__ blk, int n_layers, int emin, int emax) {
  const int l = threadIdx.x;
  if (l >= n_layers) return;
  const float m = __uint_as_float(blk[4 * l]);
  int e = 0;
  if (m > 0.f && isfinite(m)) frexpf(m, &e);      // m = f * 2^e, f in [0.5, 1)
  e = max(emin, min(emax, 1 - e));                // scale = 2^(1-e): max|w| * scale in [1, 2)
  reinterpret_cast<float*>(blk)[4 * l + 1] = ldexpf(1.f, e);
  reinterpret_cast<float*>(blk)[4 * l + 2] = ldexpf(1.f, -e);
}

int launch_weight_scales(const lsnf_plan* plan, const float* const* weights, cudaStream_t s) {
  unsigned int* blk = (unsigned int*)(plan->ws + plan->off_wscale);
  LSNF_CUDA(cudaMemsetAsync(blk, 0, (size_t)plan->n_layers * 16, s));
  for (int l = 0; l < plan->n_layers; ++l) {
    const auto& y = plan->layers[l];
    const long long n = (long long)y.ci * y.co * y.k * y.k;
    const int blocks = (int)std::min<long long>((n + 255) / 256, 148 * 8);
    wmax_kernel<<<blocks, 256, 0, s>>>(weights[l], n, blk + 4 * l);
    LSNF_CUDA(cudaGetLastError());
  }
  wscale_finalize_kernel<<<1, 32, 0, s>>>(blk, plan->n_layers, -14, 30);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// linear measurement operator A [m, n] (lsnf_pack_measurement): the B operands of the two measurement stages,
//   stage 2L (A x_hat):   rows i < m, K = n:  fp16 hi|lo of A[i][j] 2^k, 2^k the power of two with max|A| 2^k in [1, 2)
//                         (wmax_kernel / wscale_finalize_kernel on the operator's scale block)
//   stage 2L+1 (A^T r):   rows j < n, K = m:  bf16 hi|lo of A[i][j] 2^k (the format of the data-gradient stages' operands)
// Padding rows and columns are written as zeros.  2^k is not undone in the 16-bit path: stage 2L writes A x_hat 2^k,
// the finisher scales y by 2^k, stage 2L+1 writes A^T r 2^2k, and 2^-2k is folded into the fp32 post-scale of the
// first layer's split-K sum and into the AIS energy (meas_post_scale, plan.cu).  So the 16-bit tensors of the
// measured path do not depend on the units of A, y and sigma, and k is read back to the host (*k_out).
// ---------------------------------------------------------------------------------------------------
__global__ void meas_pack_kernel(const float* __restrict__ A, int m, int n, uint16_t* __restrict__ fwd, int fwd_rows,
                                 int kx, uint16_t* __restrict__ bwd, int bwd_rows, int km,
                                 const float* __restrict__ scale) {
  const float sc = *scale;
  const long long nf = (long long)fwd_rows * kx, total = nf + (long long)bwd_rows * km;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    uint16_t hi, lo;
    if (e < nf) {
      const int i = (int)(e / kx), j = (int)(e % kx);
      split16(i < m && j < n ? A[(size_t)i * n + j] * sc : 0.f, true, hi, lo);
      fwd[(size_t)i * 2 * kx + j] = hi;
      fwd[(size_t)i * 2 * kx + kx + j] = lo;
    } else {
      const int j = (int)((e - nf) / km), i = (int)((e - nf) % km);
      split16(i < m && j < n ? A[(size_t)i * n + j] * sc : 0.f, false, hi, lo);
      bwd[(size_t)j * 2 * km + i] = hi;
      bwd[(size_t)j * 2 * km + km + i] = lo;
    }
  }
}

int launch_meas_pack(const lsnf_plan* plan, const float* A, int* k_out, cudaStream_t s) {
  const StageHost& f = plan->stages[2 * plan->n_layers];
  const StageHost& b = plan->stages[2 * plan->n_layers + 1];
  const int m = plan->meas_m, n = plan->cfg.nc * plan->img * plan->img;
  unsigned int* blk = (unsigned int*)(plan->ws + plan->off_meas_scale);
  LSNF_CUDA(cudaMemsetAsync(blk, 0, 16, s));
  const long long na = (long long)m * n;
  wmax_kernel<<<(int)std::min<long long>((na + 255) / 256, 148 * 8), 256, 0, s>>>(A, na, blk);
  LSNF_CUDA(cudaGetLastError());
  wscale_finalize_kernel<<<1, 32, 0, s>>>(blk, 1, -126, 126);
  LSNF_CUDA(cudaGetLastError());
  const long long total = (long long)f.info.b_rows * plan->meas_kx + (long long)b.info.b_rows * plan->meas_km;
  meas_pack_kernel<<<(int)std::min<long long>((total + 255) / 256, 148 * 16), 256, 0, s>>>(
      A, m, n, (uint16_t*)(plan->ws + f.info.b_offset), f.info.b_rows, plan->meas_kx,
      (uint16_t*)(plan->ws + b.info.b_offset), b.info.b_rows, plan->meas_km, (const float*)(blk + 1));
  LSNF_CUDA(cudaGetLastError());
  float sc = 0.f;
  LSNF_CUDA(cudaMemcpyAsync(&sc, blk + 1, 4, cudaMemcpyDeviceToHost, s));
  LSNF_CUDA(cudaStreamSynchronize(s));
  *k_out = ilogbf(sc);
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// Between the two measurement stages: r = A x_hat - y, with A x_hat the fixed-order sum of stage 2L's split-K partials
// [S][B][n_pad], which carry the operator's scale 2^k (yscale; y is multiplied by it, exact).  One CTA per (256 rows of
// r, sample): writes r 2^k seed_scale as the bf16 hi|lo row [B][2 km] stage 2L+1 reads (seed_scale =
// sigma_seed_scale(sigma): the share of 1/sigma^2 the 16-bit gradient tensors carry, as in the unmeasured seed) and,
// when epart is given, the CTA's fixed-order partial of |r 2^k|^2 into epart[b][blockIdx.x] (annealed importance
// sampling: l(z) = -|r|^2 / (2 sigma^2), with 2^-2k in the caller's 1 / (2 sigma^2)).
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) meas_finish_kernel(const float* __restrict__ part, int nsplit, int pitch,
                                                          const float* __restrict__ y, int B, int m,
                                                          uint16_t* __restrict__ r_hl, int km, float yscale,
                                                          float seed_scale, float* __restrict__ epart) {
  __shared__ float red[256];
  pdl_wait();
  pdl_trigger();
  const int b = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
  float e = 0.f;
  if (i < m) {
    float v = 0.f;
    for (int q = 0; q < nsplit; ++q) v += __ldcg(part + ((size_t)q * B + b) * pitch + i);
    const float r = v - y[(size_t)b * m + i] * yscale;
    e = r * r;
    uint16_t hi, lo;
    split16(r * seed_scale, false, hi, lo);
    r_hl[(size_t)b * 2 * km + i] = hi;
    r_hl[(size_t)b * 2 * km + km + i] = lo;
  }
  if (!epart) return;
  red[threadIdx.x] = e;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) epart[(size_t)b * gridDim.x + blockIdx.x] = red[0];
}

int launch_meas_finish(const lsnf_plan* plan, const float* y, float seed_scale, float* epart, cudaStream_t s) {
  const StageHost& f = plan->stages[2 * plan->n_layers];
  LSNF_CUDA(launch_k(meas_finish_kernel, dim3(plan->meas_tiles, plan->cfg.batch), dim3(256), 0, s,
                     (const float*)(plan->ws + f.info.out_offset), f.info.k_splits, f.info.n_pad, y, plan->cfg.batch,
                     plan->meas_m, (uint16_t*)(plan->ws + plan->off_meas_r), plan->meas_km,
                     ldexpf(1.f, plan->meas_k), seed_scale, epart));
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// last forward layer, second half (model.py:69-70 / :90-91 / :115-116 / :149-150): the tap-GEMM left the per-tap
// products D[b][iy][ix][tap*nc + c]; each output pixel sums the taps that land on it (fixed order), adds the bias
// and applies tanh.   x_hat[b][c][oy][ox] = tanh(bias[c] + sum_{ky,kx} D[b][(oy+p-ky)/s][(ox+p-kx)/s][...])
// ---------------------------------------------------------------------------------------------------
template <int K, int S>
__global__ void __launch_bounds__(256) last_gather_tanh_kernel(const float* __restrict__ d,
                                                               const float* __restrict__ bias,
                                                               float* __restrict__ xhat, int B, int nc, int img,
                                                               int hin, int p, int n_pad, int to_unit_range,
                                                               uint16_t* __restrict__ xhl, int kx) {
  pdl_wait();
  pdl_trigger();
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long total = (long long)B * nc * img * img;
  if (i >= total) return;
  const int ox = (int)(i % img), oy = (int)((i / img) % img), c = (int)((i / ((long long)img * img)) % nc);
  const int b = (int)(i / ((long long)img * img * nc));
  // taps along one axis that can land on this pixel: ky = (o + p) % S + S*j, j < K/S (rounded up)
  constexpr int T = (K + S - 1) / S;
  float v[T * T];
  const int ky0 = (oy + p) % S, kx0 = (ox + p) % S;
#pragma unroll
  for (int a = 0; a < T; ++a) {
#pragma unroll
    for (int e = 0; e < T; ++e) {
      const int ky = ky0 + S * a, kx = kx0 + S * e;
      const int iy = (oy + p - ky) / S, ix = (ox + p - kx) / S;   // exact: the numerators are multiples of S
      const bool ok = ky < K && kx < K && oy + p - ky >= 0 && ox + p - kx >= 0 && iy < hin && ix < hin;
      v[a * T + e] = ok ? __ldcg(d + (((size_t)b * hin + iy) * hin + ix) * n_pad + (ky * K + kx) * nc + c) : 0.f;
    }
  }
  float acc = bias[c];
#pragma unroll
  for (int t = 0; t < T * T; ++t) acc += v[t];
  const float t = tanhf(acc);
  // prior sampling (train.py:562, :573): to_range_0_1(x).clamp(0, 1) fused into the same store
  xhat[i] = to_unit_range ? fminf(fmaxf((t + 1.f) / 2.f, 0.f), 1.f) : t;
  if (xhl) {
    // the A operand of the measurement GEMM A x_hat: row b holds vec(x_hat_b) (NCHW order); |x_hat| <= 1 fits fp16
    const long long n = (long long)nc * img * img;
    uint16_t hi, lo;
    split16(t, true, hi, lo);
    uint16_t* row = xhl + (size_t)b * 2 * kx;
    row[i - b * n] = hi;
    row[kx + i - b * n] = lo;
  }
}

int launch_last_gather(const lsnf_plan* plan, float* out, int to_unit_range, cudaStream_t s, uint16_t* xhl) {
  const auto& y = plan->layers[plan->n_layers - 1];
  const long long total = (long long)plan->cfg.batch * plan->cfg.nc * plan->img * plan->img;
  const float* d = (const float*)(plan->ws + plan->off_dlast);
  const float* bias = (const float*)(plan->ws + plan->off_bias[plan->n_layers - 1]);
  float* xh = out ? out : (float*)(plan->ws + plan->off_xhat);
  const unsigned blocks = (unsigned)((total + 255) / 256);
  LSNF_CUDA(launch_k(y.k == 3 && y.s == 1 ? last_gather_tanh_kernel<3, 1> : last_gather_tanh_kernel<4, 2>, dim3(blocks),
                     dim3(256), 0, s, d, bias, xh, plan->cfg.batch, plan->cfg.nc, plan->img, y.hin, y.p,
                     plan->dlast_pad, to_unit_range, xhl, plan->meas_kx));
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// z [B][nz] fp32 -> fp16 hi|lo [B][2*kp] (operand of the first generator layer, train.py:312)
// ---------------------------------------------------------------------------------------------------
__global__ void split_z_kernel(const float* __restrict__ z, uint16_t* __restrict__ zhl, int B, int nz, int kp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * kp) return;
  const int b = i / kp, j = i % kp;
  const float v = j < nz ? z[(size_t)b * nz + j] : 0.f;
  uint16_t hi, lo;
  split16(v, true, hi, lo);
  zhl[(size_t)b * 2 * kp + j] = hi;
  zhl[(size_t)b * 2 * kp + kp + j] = lo;
}

int launch_split_z(const lsnf_plan* plan, const float* z, cudaStream_t s) {
  const int n = plan->cfg.batch * plan->kp;
  split_z_kernel<<<(n + 255) / 256, 256, 0, s>>>(z, (uint16_t*)(plan->ws + plan->off_zhl), plan->cfg.batch,
                                                 plan->cfg.nz, plan->kp);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// seed of the reconstruction gradient (train.py:313-314):
//   g[b,c,oy,ox] = (x_hat - x) / sigma^2 * (1 - x_hat^2)          (MSE-sum derivative times tanh')
// of which only seed_scale = sigma_seed_scale(sigma) <= 16 (a power of two) is applied here; the rest of 1/sigma^2
// multiplies the fp32 sum of the first layer's split-K partials (langevin_update_kernel / reduce_partial_kernel).
// With upstream != 0, `x` is a caller-supplied dL/dx_hat and the seed is g = x * seed_scale * (1 - x_hat^2) (the
// vector-Jacobian product of lsnf_generator_vjp, seed_scale 1).  With upstream == 0 and a likelihood mask m (nullable,
// [B,nc,H,W] like x) the loss is the weighted 1/(2 sigma^2) sum m (x_hat - x)^2 and the seed (m * (x_hat - x)) * ...:
// the weight multiplies the difference before any other factor, so an all-ones mask reproduces the unmasked seed bit
// for bit.  Either seed is
// written directly as the im2col operand of the last layer's data gradient:
//   A[b][iy][ix][tap*nc + c] = g[b][c][iy*s - p + ky][ix*s - p + kx]  (0 outside the image), 64 columns.
// ---------------------------------------------------------------------------------------------------
// One CTA per (sample, input row, segment of <= 32 input columns): the loss-gradient values the segment's taps touch
// are computed once into shared memory (coalesced reads of x_hat and x), then written out as 64-column im2col rows
// (coalesced 2-byte stores).
constexpr int IM2COL_SEG = 32;
__global__ void __launch_bounds__(128) recon_grad_im2col_kernel(const float* __restrict__ xhat,
                                                                const float* __restrict__ x,
                                                                const float* __restrict__ mask,
                                                                uint16_t* __restrict__ a, int B, int nc, int img,
                                                                int hin, int k, int s, int p, float seed_scale,
                                                                int fp16, int upstream, const float* __restrict__ part,
                                                                int nsplit, int pitch) {
  extern __shared__ float g[];   // [nc][k][span], span = (seg-1)*s + k
  pdl_wait();
  pdl_trigger();
  const int segs = (hin + IM2COL_SEG - 1) / IM2COL_SEG;
  const int seg = blockIdx.x % segs, iy = (blockIdx.x / segs) % hin, b = blockIdx.x / (segs * hin);
  const int ix0 = seg * IM2COL_SEG, nseg = min(IM2COL_SEG, hin - ix0);
  const int span = (nseg - 1) * s + k;
  const int oy0 = iy * s - p, ox0 = ix0 * s - p;
  for (int i = threadIdx.x; i < nc * k * span; i += blockDim.x) {
    const int xx = i % span, ky = (i / span) % k, c = i / (span * k);
    const int oy = oy0 + ky, ox = ox0 + xx;
    float v = 0.f;
    if (oy >= 0 && oy < img && ox >= 0 && ox < img) {
      const size_t o = (((size_t)b * nc + c) * img + oy) * img + ox;
      const float xh = xhat[o];
      float d;
      if (part) {   // dL/dx_hat = A^T r: its split-K partials summed in a fixed order
        const size_t col = o - (size_t)b * nc * img * img;
        d = 0.f;
        for (int q = 0; q < nsplit; ++q) d += __ldcg(part + ((size_t)q * B + b) * pitch + col);
      } else {
        d = upstream ? x[o] : xh - x[o];
      }
      if (mask) d = mask[o] * d;   // read only with upstream == 0 (the launcher passes null otherwise)
      v = d * seed_scale * (1.f - xh * xh);
    }
    g[i] = v;
  }
  __syncthreads();
  const size_t row0 = ((size_t)b * hin + iy) * hin + ix0;
  for (int i = threadIdx.x; i < nseg * BLOCK_K; i += blockDim.x) {
    const int col = i % BLOCK_K, r = i / BLOCK_K;
    float v = 0.f;
    if (col < k * k * nc) {
      const int tap = col / nc, c = col % nc;
      v = g[(c * k + tap / k) * span + r * s + tap % k];
    }
    uint16_t hi, lo;
    split16(v, fp16 != 0, hi, lo);   // operand of the data-gradient stages (bf16 hi|lo, or fp16 for one pass)
    a[(row0 + r) * 2 * BLOCK_K + col] = hi;
    a[(row0 + r) * 2 * BLOCK_K + BLOCK_K + col] = lo;
  }
}

int launch_recon_grad_im2col(const lsnf_plan* plan, const float* x, const float* mask, float seed_scale, int upstream,
                             cudaStream_t s, const float* part, int nsplit, int pitch) {
  const auto& y = plan->layers[plan->n_layers - 1];
  const int segs = (y.hin + IM2COL_SEG - 1) / IM2COL_SEG;
  const int span = (std::min(IM2COL_SEG, y.hin) - 1) * y.s + y.k;
  const size_t smem = (size_t)plan->cfg.nc * y.k * span * 4;
  LSNF_CUDA(launch_k(recon_grad_im2col_kernel, dim3(plan->cfg.batch * y.hin * segs), dim3(128), smem, s,
                     (const float*)(plan->ws + plan->off_xhat), x, upstream ? nullptr : mask,
                     (uint16_t*)(plan->ws + plan->off_im2col), plan->cfg.batch, plan->cfg.nc, plan->img, y.hin, y.k, y.s,
                     y.p, seed_scale, plan->cfg.bwd_passes == 1 ? 1 : 0, upstream, part, nsplit, pitch));
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// The two kernels above fused for the Langevin loop (train.py:312-314 back to back): one CTA owns a TR x TC tile of
// last-layer input positions.  It stages the direct-product rows of the tile and a 2-position halo in shared memory
// (coalesced 128-bit reads; the per-position stride is padded to an odd word count so the tap gathers that follow
// are bank-conflict free), computes x_hat and the loss-gradient seed for the output window the tile's taps touch,
// and writes the tile's 64-column im2col rows.  x_hat is written by the tile that owns pixel (oy/s, ox/s); the tap
// summation order equals last_gather_tanh_kernel's, so x_hat is bit-identical to the unfused path.  With a mask
// (nullable) the CTA also stages the mask window next to the x window and weights the seed as
// recon_grad_im2col_kernel does.
// ---------------------------------------------------------------------------------------------------
constexpr int FUSE_HALO = 2;   // ceil((k-1)/s) for both supported geometries (k3/s1, k4/s2)
// x / d for the small index ranges of this kernel (x * d < 2^32) as one multiply-high: the kernel is all index
// arithmetic, and hardware-less 32-bit division made it instruction-bound
struct FastDiv {
  uint32_t d, m;
  __device__ __forceinline__ explicit FastDiv(int d_) : d((uint32_t)d_), m(d_ > 1 ? 0xFFFFFFFFu / (uint32_t)d_ + 1u : 0u) {}
  __device__ __forceinline__ int div(int x) const { return d > 1 ? (int)__umulhi((uint32_t)x, m) : x; }
};

template <int K, int S>
__global__ void __launch_bounds__(256) last_fused_kernel(const float* __restrict__ d, const float* __restrict__ bias,
                                                         const float* __restrict__ x, const float* __restrict__ mask,
                                                         float* __restrict__ epart,
                                                         float* __restrict__ xhat, uint16_t* __restrict__ a, int B,
                                                         int nc, int img, int hin,
                                                         int p, int n_pad, int TR, int TC, float seed_scale, int fp16,
                                                         int write_lo) {
  extern __shared__ float fs[];
  pdl_wait();      // the last forward layer's per-tap products must be complete (no-op without the launch attribute)
  pdl_trigger();
  constexpr int T = (K + S - 1) / S;
  const int tiles_c = (hin + TC - 1) / TC, tiles_r = (hin + TR - 1) / TR;
  const int tc = blockIdx.x % tiles_c, tr = (blockIdx.x / tiles_c) % tiles_r, b = blockIdx.x / (tiles_c * tiles_r);
  const int r0 = tr * TR, c0 = tc * TC;
  const int nr = min(TR, hin - r0), ncol = min(TC, hin - c0);
  const int DW = TC + 2 * FUSE_HALO, DH = TR + 2 * FUSE_HALO, PS = n_pad + 1;
  const int GH = (TR - 1) * S + K, GW = (TC - 1) * S + K;
  float* Dt = fs;                         // [DH][DW][PS]
  float* G = fs + (size_t)DH * DW * PS;   // [nc][GH][GW]
  float* M = G + (size_t)nc * GH * GW;    // [nc][GH][GW], mask window (only with a mask)
  const int tid = threadIdx.x;
  const int qs = n_pad == 32 ? 3 : 4;     // log2 of the float4 count per position (n_pad is 32 or 64)
  const int dr0 = max(0, r0 - FUSE_HALO), dr1 = min(hin, r0 + nr + FUSE_HALO);
  const int dc0 = max(0, c0 - FUSE_HALO), dc1 = min(hin, c0 + ncol + FUSE_HALO);
  const int dwc = dc1 - dc0;
  const FastDiv by_dwc(dwc), by_gw(GW), by_gwh(GW * GH), by_ncol(ncol);
  // All global reads of the CTA are issued here, four independent loads per thread at a time: the target pixels of
  // the output window go to G, which the next phase overwrites in place with the seed; then the direct-product rows
  // (tile + halo, clipped to the grid).
  constexpr int U = 4;
  const int oy_lo = r0 * S - p, ox_lo = c0 * S - p;
  const int nwin = nc * GH * GW;
  for (int i0 = tid; i0 < nwin; i0 += U * blockDim.x) {
    float xv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u * blockDim.x;
      const int c = by_gwh.div(i), rem = i - c * GW * GH, yy = by_gw.div(rem), xx = rem - yy * GW;
      const int oy = oy_lo + yy, ox = ox_lo + xx;
      xv[u] = (i < nwin && oy >= 0 && oy < img && ox >= 0 && ox < img)
                  ? __ldg(x + (((size_t)b * nc + c) * img + oy) * img + ox) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u * blockDim.x;
      if (i < nwin) G[i] = xv[u];
    }
  }
  if (mask) {
    for (int i0 = tid; i0 < nwin; i0 += U * blockDim.x) {
      float mv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = i0 + u * blockDim.x;
        const int c = by_gwh.div(i), rem = i - c * GW * GH, yy = by_gw.div(rem), xx = rem - yy * GW;
        const int oy = oy_lo + yy, ox = ox_lo + xx;
        mv[u] = (i < nwin && oy >= 0 && oy < img && ox >= 0 && ox < img)
                    ? __ldg(mask + (((size_t)b * nc + c) * img + oy) * img + ox) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = i0 + u * blockDim.x;
        if (i < nwin) M[i] = mv[u];
      }
    }
  }
  const int nd = ((dr1 - dr0) * dwc) << qs;
  const float* dbase = d + ((size_t)b * hin * hin) * n_pad;
  for (int i0 = tid; i0 < nd; i0 += U * blockDim.x) {
    float4 v[U];
    int so[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u * blockDim.x;
      so[u] = -1;
      if (i < nd) {
        const int q = i & ((1 << qs) - 1), pos = i >> qs;
        const int row = by_dwc.div(pos), cl = pos - row * dwc;
        const int ix = dc0 + cl, iy = dr0 + row;
        v[u] = __ldcg(reinterpret_cast<const float4*>(dbase + ((size_t)iy * hin + ix) * n_pad) + q);
        so[u] = ((iy - (r0 - FUSE_HALO)) * DW + (ix - (c0 - FUSE_HALO))) * PS + 4 * q;
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (so[u] >= 0) {
        float* o = Dt + so[u];
        o[0] = v[u].x; o[1] = v[u].y; o[2] = v[u].z; o[3] = v[u].w;
      }
    }
  }
  __syncthreads();
  // ---- x_hat and the seed g = (m * (x_hat - x)) / sigma^2 * (1 - x_hat^2) on the output window of the tile ----
  float esum = 0.f;   // sum m (x_hat - x)^2 over the pixels this thread visits that the tile owns (epart only)
  for (int i = tid; i < nwin; i += blockDim.x) {
    const int c = by_gwh.div(i), rem = i - c * GW * GH, yy = by_gw.div(rem), xx = rem - yy * GW;
    const int oy = oy_lo + yy, ox = ox_lo + xx;
    float g = 0.f;
    if (oy >= 0 && oy < img && ox >= 0 && ox < img) {
      const int ky0 = (oy + p) % S, kx0 = (ox + p) % S;
      // local coordinates of the tap (ky0, kx0) in the staged tile; tap (e, f) lies e, f positions before it
      const int ly = (oy + p - ky0) / S - (r0 - FUSE_HALO), lx = (ox + p - kx0) / S - (c0 - FUSE_HALO);
      const int gy = (oy + p - ky0) / S, gx = (ox + p - kx0) / S;
      float acc = bias[c];
      float v[T * T];
#pragma unroll
      for (int e = 0; e < T; ++e) {
#pragma unroll
        for (int f = 0; f < T; ++f) {
          const int ky = ky0 + S * e, kx = kx0 + S * f;
          const int iy = gy - e, ix = gx - f;
          const bool ok = ky < K && kx < K && iy >= 0 && ix >= 0 && iy < hin && ix < hin;
          v[e * T + f] = ok ? Dt[((ly - e) * DW + (lx - f)) * PS + (ky * K + kx) * nc + c] : 0.f;
        }
      }
#pragma unroll
      for (int t = 0; t < T * T; ++t) acc += v[t];
      const float xh = tanhf(acc);
      const int iyo = oy / S, ixo = ox / S;   // the tile that owns this pixel writes x_hat
      const bool own = iyo >= r0 && iyo < r0 + nr && ixo >= c0 && ixo < c0 + ncol;
      if (own) xhat[(((size_t)b * nc + c) * img + oy) * img + ox] = xh;
      const float d0 = xh - G[i];
      float dv = d0;
      if (mask) dv = M[i] * dv;
      if (own) esum += dv * d0;
      g = dv * seed_scale * (1.f - xh * xh);
    }
    G[i] = g;
  }
  if (epart) {
    // per-sample energy partial of the tile (annealed importance sampling): a fixed-order block sum, one float per CTA
    __shared__ float ered[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) esum += __shfl_xor_sync(0xffffffffu, esum, o);
    if ((tid & 31) == 0) ered[tid >> 5] = esum;
    __syncthreads();
    if (tid == 0) {
      float e = 0.f;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) e += ered[w];
      epart[blockIdx.x] = e;
    }
  }
  __syncthreads();
  // ---- im2col rows of the tile: A[pos][tap*nc + c] = g[c][iy*s - p + ky][ix*s - p + kx] ----
  // eight threads per position, eight columns (one 16-byte store per half) per thread; a thread's columns are fixed,
  // so their offsets into the seed window are computed once
  const int sub = tid & 7;
  int goff[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int col = 8 * sub + j;
    const int tap = col / nc, c = col % nc;
    goff[j] = col < K * K * nc ? (c * GH + tap / K) * GW + tap % K : -1;
  }
  const bool f16 = fp16 != 0;
  for (int pos = tid >> 3; pos < nr * ncol; pos += blockDim.x >> 3) {
    const int r = by_ncol.div(pos), cc = pos - r * ncol;
    const int base = r * S * GW + cc * S;
    __align__(16) uint16_t hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) split16(goff[j] >= 0 ? G[goff[j] + base] : 0.f, f16, hi[j], lo[j]);
    uint16_t* row = a + (((size_t)b * hin + r0 + r) * hin + c0 + cc) * 2 * BLOCK_K + 8 * sub;
    *reinterpret_cast<uint4*>(row) = *reinterpret_cast<const uint4*>(hi);
    if (write_lo) *reinterpret_cast<uint4*>(row + BLOCK_K) = *reinterpret_cast<const uint4*>(lo);
  }
}

int last_fused_tiles(const lsnf_plan* plan, int* TR, int* TC) {
  const auto& y = plan->layers[plan->n_layers - 1];
  *TC = std::min(32, y.hin);
  *TR = std::min(plan->dlast_pad <= 32 ? 8 : 4, y.hin);
  return ((y.hin + *TR - 1) / *TR) * ((y.hin + *TC - 1) / *TC);
}

int launch_last_fused(const lsnf_plan* plan, const float* x, const float* mask, float* epart, float seed_scale,
                      cudaStream_t s) {
  const auto& y = plan->layers[plan->n_layers - 1];
  const int n_pad = plan->dlast_pad;
  int TR, TC;
  const int tiles = last_fused_tiles(plan, &TR, &TC);
  const int DW = TC + 2 * FUSE_HALO, DH = TR + 2 * FUSE_HALO;
  const int GH = (TR - 1) * y.s + y.k, GW = (TC - 1) * y.s + y.k;
  const size_t smem = ((size_t)DH * DW * (n_pad + 1) + (size_t)plan->cfg.nc * GH * GW * (mask ? 2 : 1)) * 4;
  const float* d = (const float*)(plan->ws + plan->off_dlast);
  const float* bias = (const float*)(plan->ws + plan->off_bias[plan->n_layers - 1]);
  float* xh = (float*)(plan->ws + plan->off_xhat);
  uint16_t* a = (uint16_t*)(plan->ws + plan->off_im2col);
  const int one = plan->cfg.bwd_passes == 1 ? 1 : 0;
  if (smem > 160 * 1024) { set_error("fused last-layer kernel: tile does not fit shared memory"); return LSNF_ERR_INVALID; }
  const dim3 grid(plan->cfg.batch * tiles), block(256);
  if (y.k == 3 && y.s == 1)
    LSNF_CUDA(launch_k(last_fused_kernel<3, 1>, grid, block, smem, s, d, bias, x, mask, epart, xh, a, plan->cfg.batch,
                       plan->cfg.nc, plan->img, y.hin, y.p, n_pad, TR, TC, seed_scale, one, !one));
  else
    LSNF_CUDA(launch_k(last_fused_kernel<4, 2>, grid, block, smem, s, d, bias, x, mask, epart, xh, a, plan->cfg.batch,
                       plan->cfg.nc, plan->img, y.hin, y.p, n_pad, TR, TC, seed_scale, one, !one));
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// split-K partials [S][B][nzp] -> grad_z [B][nz]  (standalone lsnf_generator_dgrad only; the Langevin loop
// folds this sum into the update kernel)
// ---------------------------------------------------------------------------------------------------
__global__ void reduce_partial_kernel(const float* __restrict__ part, float* __restrict__ g, int S, int B, int nz,
                                      int nzp, float scale) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * nz) return;
  const int b = i / nz, j = i % nz;
  float acc = 0.f;
  for (int s = 0; s < S; ++s) acc += part[((size_t)s * B + b) * nzp + j];
  g[i] = acc * scale;
}

int launch_reduce_partial(const lsnf_plan* plan, float* grad_z, float scale, cudaStream_t s) {
  const int n = plan->cfg.batch * plan->cfg.nz;
  reduce_partial_kernel<<<(n + 255) / 256, 256, 0, s>>>((const float*)(plan->ws + plan->off_partial), grad_z,
                                                       plan->ksplit_first, plan->cfg.batch, plan->cfg.nz, plan->nzp, scale);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// fused Langevin update (train.py:324-329): one CTA per sample, 4 latent elements per lane
//   z <- z - s^2/2 (grad_g + grad_f) + s * noise ;  per-sample |grad_g|, |grad_f| ; next step's bf16 hi|lo z
// Noise: injected eps, or Philox4x32-10 keyed by (seed, global sample index, step, element quad) drawn in
// registers (oracle/philox.py is the checker).
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float& n0, float& n1) {
  const float u0 = ((float)(a >> 8) + 0.5f) * 5.9604644775390625e-8f;  // 2^-24
  const float u1 = ((float)(b >> 8) + 0.5f) * 5.9604644775390625e-8f;
  const float r = sqrtf(-2.f * logf(u0));
  float sn, cs;
  sincospif(2.f * u1, &sn, &cs);
  n0 = r * cs; n1 = r * sn;
}

// One CTA per sample: 8 thread groups x 32 lanes; lane q owns latent elements [4q, 4q+4) and the groups share the
// split-K partial sums of the reconstruction gradient (fixed summation order -> deterministic).
__global__ void __launch_bounds__(256) langevin_update_kernel(
    float* __restrict__ z, const float* __restrict__ gg, const float* __restrict__ partial, int nsplit, int nzp,
    float gscale, const float* __restrict__ gf, const float* __restrict__ eps, uint16_t* __restrict__ zhl, int B, int nz,
    int kp, float step, int with_noise, uint64_t seed, uint64_t sample_offset, uint32_t step_idx,
    const uint64_t* __restrict__ dyn, float* __restrict__ norm_scratch, unsigned int* __restrict__ ticket,
    float* __restrict__ gnorms) {
  __shared__ float4 part[8][64];
  pdl_wait();      // launched without the attribute (it joins the flow prior's stream): returns at once
  pdl_trigger();   // the next iteration's first layer may set itself up while this kernel runs
  if (dyn) { seed = dyn[0]; sample_offset = dyn[1]; step_idx += (uint32_t)dyn[2]; }   // per-call values of a replayed CUDA graph
  __shared__ float red[2][256];
  __shared__ bool is_last;
  const int b = blockIdx.x, tid = threadIdx.x;
  const int nq = nz / 4;
  const int grp = tid >> 5, lane = tid & 31;
  // ---- reconstruction gradient of this sample: sum of the split-K partials (or a ready gradient) ----
  for (int q = lane; q < nq; q += 32) {
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    if (partial) {
#pragma unroll 4
      for (int s = grp; s < nsplit; s += 8) {
        const float4 p = __ldcg(reinterpret_cast<const float4*>(partial + ((size_t)s * B + b) * nzp + 4 * q));
        g.x += p.x; g.y += p.y; g.z += p.z; g.w += p.w;
      }
    } else if (grp == 0) {
      g = *reinterpret_cast<const float4*>(gg + (size_t)b * nz + 4 * q);
    }
    part[grp][q] = g;
  }
  __syncthreads();
  float sg = 0.f, sf = 0.f;
  if (tid < nq) {
    const int q = tid;
    float4 g = part[0][q];
#pragma unroll
    for (int k = 1; k < 8; ++k) {
      const float4 p = part[k][q];
      g.x += p.x; g.y += p.y; g.z += p.z; g.w += p.w;
    }
    g.x *= gscale; g.y *= gscale; g.z *= gscale; g.w *= gscale;   // the part of 1/sigma^2 kept out of the 16-bit tensors
    const size_t o = (size_t)b * nz + 4 * q;
    const float4 f = *reinterpret_cast<const float4*>(gf + o);
    float4 v = *reinterpret_cast<const float4*>(z + o);
    const float h = 0.5f * step * step;
    v.x = v.x - h * (g.x + f.x); v.y = v.y - h * (g.y + f.y);
    v.z = v.z - h * (g.z + f.z); v.w = v.w - h * (g.w + f.w);
    if (eps) {
      const float4 e = *reinterpret_cast<const float4*>(eps + o);
      v.x += step * e.x; v.y += step * e.y; v.z += step * e.z; v.w += step * e.w;
    } else if (with_noise) {
      const uint64_t sample = sample_offset + (uint64_t)b;
      uint32_t r[4];
      philox4x32_10((uint32_t)sample, (uint32_t)(sample >> 32), step_idx, (uint32_t)q, (uint32_t)seed,
                    (uint32_t)(seed >> 32), r);
      float n0, n1, n2, n3;
      box_muller(r[0], r[1], n0, n1);
      box_muller(r[2], r[3], n2, n3);
      v.x += step * n0; v.y += step * n1; v.z += step * n2; v.w += step * n3;
    }
    *reinterpret_cast<float4*>(z + o) = v;
    sg = g.x * g.x + g.y * g.y + g.z * g.z + g.w * g.w;
    sf = f.x * f.x + f.y * f.y + f.z * f.z + f.w * f.w;
    if (zhl) {
      __align__(8) uint16_t hi[4], lo[4];   // fp16 hi|lo operand of the first forward layer
      split16(v.x, true, hi[0], lo[0]); split16(v.y, true, hi[1], lo[1]);
      split16(v.z, true, hi[2], lo[2]); split16(v.w, true, hi[3], lo[3]);
      uint16_t* row = zhl + (size_t)b * 2 * kp;
      *reinterpret_cast<uint2*>(row + 4 * q) = *reinterpret_cast<uint2*>(hi);
      *reinterpret_cast<uint2*>(row + kp + 4 * q) = *reinterpret_cast<uint2*>(lo);
    }
  }
  if (!gnorms) return;
  // per-sample norms (train.py:328-329), then the last CTA to finish averages them in a fixed order
  red[0][tid] = sg; red[1][tid] = sf;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) { red[0][tid] += red[0][tid + o]; red[1][tid] += red[1][tid + o]; }
    __syncthreads();
  }
  if (tid == 0) {
    norm_scratch[b] = sqrtf(red[0][0]);
    norm_scratch[B + b] = sqrtf(red[1][0]);
    __threadfence();
    is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  float a = 0.f, c = 0.f;
  for (int i = tid; i < B; i += blockDim.x) {
    a += __ldcg(norm_scratch + i);
    c += __ldcg(norm_scratch + B + i);
  }
  red[0][tid] = a; red[1][tid] = c;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) { red[0][tid] += red[0][tid + o]; red[1][tid] += red[1][tid + o]; }
    __syncthreads();
  }
  if (tid == 0) {
    gnorms[0] = red[0][0] / (float)B;
    gnorms[1] = red[1][0] / (float)B;
    *ticket = 0u;
  }
}

int launch_update(const lsnf_plan* plan, float* z, const float* gg, const float* partial, int nsplit, float gscale,
                  const float* gf, float step, const float* eps, int with_noise, uint64_t seed,
                  uint64_t sample_offset, uint32_t step_idx, const uint64_t* dyn, float* gnorms, int write_zhl,
                  cudaStream_t s) {
  const int B = plan->cfg.batch;
  unsigned int* ticket = (unsigned int*)(plan->ws + plan->off_scalars);  // last-block-done counter
  float* scratch = (float*)(plan->ws + plan->off_norms);
  uint16_t* zhl = (write_zhl && plan->n_layers) ? (uint16_t*)(plan->ws + plan->off_zhl) : nullptr;
  langevin_update_kernel<<<B, 256, 0, s>>>(z, gg, partial, nsplit, plan->nzp, gscale, gf, eps, zhl, B, plan->cfg.nz,
                                           plan->kp, step, with_noise, seed, sample_offset, step_idx, dyn, scratch,
                                           ticket, gnorms);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

__global__ void set_dyn_kernel(uint64_t* dyn, uint64_t seed, uint64_t sample_offset, uint64_t base_step,
                               uint64_t total) {
  dyn[0] = seed; dyn[1] = sample_offset; dyn[2] = base_step; dyn[3] = total;
}

int launch_set_dyn(const lsnf_plan* plan, uint64_t seed, uint64_t sample_offset, uint32_t base_step, cudaStream_t s,
                   uint32_t total) {
  set_dyn_kernel<<<1, 1, 0, s>>>((uint64_t*)(plan->ws + plan->off_dyn), seed, sample_offset, base_step, total);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// Annealed importance sampling with Metropolis-adjusted Langevin (MALA) transitions (lsnf_ais_run).
// The loop evaluates, at the point z the generator saw, l(z) = -sum m (G(z) - x)^2 / (2 sigma^2) (from the fused
// last-layer kernel's per-tile partials), log p(z) and both gradients; this kernel keeps the chain's state and
//   iteration k = 0      initialises the state with the evaluated point,
//   iteration 1 <= k     accepts or rejects the proposal of step k (target pi_{beta_k}),
//   iteration k < T      adds (beta_{k+1} - beta_k) l(z_k) to log w and proposes step k+1 on pi_{beta_{k+1}},
// so T transitions take T+1 iterations.  k is the global iteration index (dyn[2] + t under graph replay) and T is
// read from dyn[3] there.  The proposal is stored rounded to its fp16 hi|lo value, the point the first generator layer
// reads, so that G, the flow and the Metropolis-Hastings test all see the same z.  The same stored gradient proposes
// and enters the acceptance density, so the test is exact with respect to the computed energies.
// ---------------------------------------------------------------------------------------------------
__global__ void ais_begin_kernel(float* __restrict__ z, uint16_t* __restrict__ zhl, int B, int nz, int kp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * kp) return;
  const int b = i / kp, j = i % kp;
  const float v = j < nz ? z[(size_t)b * nz + j] : 0.f;
  uint16_t hi, lo;
  split16(v, true, hi, lo);
  zhl[(size_t)b * 2 * kp + j] = hi;
  zhl[(size_t)b * 2 * kp + kp + j] = lo;
  if (j < nz) z[(size_t)b * nz + j] = join16(hi, lo, true);
}

int launch_ais_begin(const lsnf_plan* plan, float* z, cudaStream_t s) {
  const int n = plan->cfg.batch * plan->kp;
  ais_begin_kernel<<<(n + 255) / 256, 256, 0, s>>>(z, (uint16_t*)(plan->ws + plan->off_zhl), plan->cfg.batch,
                                                   plan->cfg.nz, plan->kp);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

// fixed-order sum over the 256 threads of a CTA (every thread gets the result)
__device__ __forceinline__ float block_sum256(float v, float* red) {
  __syncthreads();
  red[threadIdx.x] = v;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  return red[0];
}

__device__ __forceinline__ float4 f4_fma(float4 a, float s, float4 b) {   // a + s * b
  return make_float4(a.x + s * b.x, a.y + s * b.y, a.z + s * b.z, a.w + s * b.w);
}

__global__ void __launch_bounds__(256) ais_update_kernel(
    AisArgs A, float* __restrict__ z, uint16_t* __restrict__ zhl, const float* __restrict__ partial, int nsplit,
    int nzp, float gscale, const float* __restrict__ gf, int B, int nz, int kp, uint64_t seed, uint64_t sample_offset,
    uint32_t t, const uint64_t* __restrict__ dyn) {
  __shared__ float4 part[8][64];
  __shared__ float red[256];
  __shared__ int s_accept;
  __shared__ float s_step;
  pdl_wait();
  pdl_trigger();
  uint32_t k = t, total = (uint32_t)A.total;
  if (dyn) { seed = dyn[0]; sample_offset = dyn[1]; k += (uint32_t)dyn[2]; total = (uint32_t)dyn[3]; }
  const int b = blockIdx.x, tid = threadIdx.x;
  const int nq = nz / 4;
  const int grp = tid >> 5, lane = tid & 31;
  for (int q = lane; q < nq; q += 32) {
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
    for (int s = grp; s < nsplit; s += 8) {
      const float4 p = __ldcg(reinterpret_cast<const float4*>(partial + ((size_t)s * B + b) * nzp + 4 * q));
      g.x += p.x; g.y += p.y; g.z += p.z; g.w += p.w;
    }
    part[grp][q] = g;
  }
  __syncthreads();
  const bool act = tid < nq;
  const size_t o = (size_t)b * nz + 4 * (act ? tid : 0);
  float4 gr1 = make_float4(0.f, 0.f, 0.f, 0.f), gp1 = gr1, z1 = gr1;   // the point evaluated by this iteration
  if (act) {
    gr1 = part[0][tid];
#pragma unroll
    for (int j = 1; j < 8; ++j) {
      const float4 p = part[j][tid];
      gr1.x += p.x; gr1.y += p.y; gr1.z += p.z; gr1.w += p.w;
    }
    gr1.x *= gscale; gr1.y *= gscale; gr1.z *= gscale; gr1.w *= gscale;   // -dl/dz
    gp1 = *reinterpret_cast<const float4*>(gf + o);                         // -dlog p/dz
    z1 = *reinterpret_cast<const float4*>(z + o);
  }
  float* ell = A.scal;              // state: l(z)
  float* lp = A.scal + B;           //        log p(z) (the flow's, with its constant)
  float* stp = A.scal + 2 * B;      //        step size
  float* acc = A.scal + 3 * B;      //        accepted proposals
  float* e2 = A.scal + 4 * B;       //        |eps|^2 / 2 of the pending proposal
  float ell_cur = 0.f;              // thread 0 only
  float4 zc = z1, grc = gr1, gpc = gp1;
  float step;
  if (k == 0) {
    if (act) {
      *reinterpret_cast<float4*>(A.zc + o) = z1;
      *reinterpret_cast<float4*>(A.gr + o) = gr1;
      *reinterpret_cast<float4*>(A.gp + o) = gp1;
    }
    step = A.step0;
    if (tid == 0) {
      float e = 0.f;
      for (int i = 0; i < A.tiles; ++i) e += A.epart[(size_t)b * A.tiles + i];
      ell_cur = -e * A.inv2s2;
      ell[b] = ell_cur; lp[b] = A.logp[b]; stp[b] = step; acc[b] = 0.f; A.logw[b] = 0.0;
    }
  } else {
    const float beta = A.betas[t];
    step = stp[b];
    if (act) {
      zc = *reinterpret_cast<const float4*>(A.zc + o);
      grc = *reinterpret_cast<const float4*>(A.gr + o);
      gpc = *reinterpret_cast<const float4*>(A.gp + o);
    }
    // reverse-move density: |z - z' + (s^2/2) grad U(z')|^2 / (2 s^2)
    const float h = 0.5f * step * step;
    float rk = 0.f;
    if (act) {
      const float4 gu = f4_fma(gp1, beta, gr1);
      const float4 r = f4_fma(make_float4(zc.x - z1.x, zc.y - z1.y, zc.z - z1.z, zc.w - z1.w), h, gu);
      rk = r.x * r.x + r.y * r.y + r.z * r.z + r.w * r.w;
    }
    rk = block_sum256(rk, red);
    if (tid == 0) {
      float e = 0.f;
      for (int i = 0; i < A.tiles; ++i) e += A.epart[(size_t)b * A.tiles + i];
      const float ell1 = -e * A.inv2s2, lp1 = A.logp[b];
      const double u0 = -(double)lp[b] - (double)beta * ell[b], u1 = -(double)lp1 - (double)beta * ell1;
      const double la = u0 - u1 - (double)rk / (2.0 * (double)step * step) + (double)e2[b];
      float u;
      if (A.u) {
        u = A.u[(size_t)(k - 1) * B + b];
      } else {
        const uint64_t sample = sample_offset + (uint64_t)b;
        uint32_t r[4];
        philox4x32_10((uint32_t)sample, (uint32_t)(sample >> 32), k, 0xFFFFFFFFu, (uint32_t)seed,
                      (uint32_t)(seed >> 32), r);
        u = ((float)(r[0] >> 8) + 0.5f) * 5.9604644775390625e-8f;
      }
      const bool ok = isfinite(u1) && isfinite(la) && log((double)u) < la;
      ell_cur = ok ? ell1 : ell[b];
      if (ok) { ell[b] = ell1; lp[b] = lp1; acc[b] += 1.f; }
      double sn = step;
      if (A.target > 0.f) {
        const double a = isfinite(u1) && !isnan(la) ? (la >= 0.0 ? 1.0 : exp(la)) : 0.0;
        sn = fmin(fmax(sn * exp(AIS_KAPPA * (a - (double)A.target)), AIS_STEP_MIN), AIS_STEP_MAX);
      }
      s_accept = ok ? 1 : 0;
      s_step = (float)sn;
      stp[b] = (float)sn;
    }
    __syncthreads();
    step = s_step;
    if (s_accept) {
      zc = z1; grc = gr1; gpc = gp1;
      if (act) {
        *reinterpret_cast<float4*>(A.zc + o) = z1;
        *reinterpret_cast<float4*>(A.gr + o) = gr1;
        *reinterpret_cast<float4*>(A.gp + o) = gp1;
      }
    }
  }
  if (k >= total) {
    // the chain's result: z_T in the workspace latent, log w and the acceptance rate in the output rows
    if (act) *reinterpret_cast<float4*>(z + o) = zc;
    if (tid == 0) {
      A.scal[5 * B + b] = (float)A.logw[b];
      A.scal[6 * B + b] = acc[b] / (float)total;
    }
    return;
  }
  const float beta0 = A.betas[t], beta1 = A.betas[t + 1];
  if (tid == 0) A.logw[b] += ((double)beta1 - (double)beta0) * (double)ell_cur;
  // proposal of step k+1 on pi_{beta_{k+1}}: z' = z - (s^2/2) grad U(z) + s eps, rounded to its fp16 hi|lo value
  float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
  if (act) {
    if (A.eps) {
      e = *reinterpret_cast<const float4*>(A.eps + (size_t)k * B * nz + o);
    } else {
      const uint64_t sample = sample_offset + (uint64_t)b;
      uint32_t r[4];
      philox4x32_10((uint32_t)sample, (uint32_t)(sample >> 32), k, (uint32_t)tid, (uint32_t)seed,
                    (uint32_t)(seed >> 32), r);
      box_muller(r[0], r[1], e.x, e.y);
      box_muller(r[2], r[3], e.z, e.w);
    }
    const float h = 0.5f * step * step;
    const float4 gu = f4_fma(gpc, beta1, grc);
    float v[4] = {zc.x - h * gu.x + step * e.x, zc.y - h * gu.y + step * e.y, zc.z - h * gu.z + step * e.z,
                  zc.w - h * gu.w + step * e.w};
    __align__(8) uint16_t hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      split16(v[j], true, hi[j], lo[j]);
      v[j] = join16(hi[j], lo[j], true);
    }
    *reinterpret_cast<float4*>(z + o) = make_float4(v[0], v[1], v[2], v[3]);
    uint16_t* row = zhl + (size_t)b * 2 * kp;
    *reinterpret_cast<uint2*>(row + 4 * tid) = *reinterpret_cast<uint2*>(hi);
    *reinterpret_cast<uint2*>(row + kp + 4 * tid) = *reinterpret_cast<uint2*>(lo);
  }
  const float ee = block_sum256(e.x * e.x + e.y * e.y + e.z * e.z + e.w * e.w, red);
  if (tid == 0) e2[b] = 0.5f * ee;
}

int launch_ais_update(const lsnf_plan* plan, const AisArgs& a, const float* gf, float gscale, uint64_t seed,
                      uint64_t sample_offset, uint32_t t, const uint64_t* dyn, cudaStream_t s) {
  ais_update_kernel<<<plan->cfg.batch, 256, 0, s>>>(
      a, (float*)(plan->ws + plan->off_z), (uint16_t*)(plan->ws + plan->off_zhl),
      (const float*)(plan->ws + plan->off_partial), plan->ksplit_first, plan->nzp, gscale, gf, plan->cfg.batch,
      plan->cfg.nz, plan->kp, seed, sample_offset, t, dyn);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

int aux_prepare_device(int device) {
  static std::mutex mu;
  static bool done[64] = {false};
  std::lock_guard<std::mutex> lock(mu);
  if (device < 0 || device >= 64) { set_error("device index out of range"); return LSNF_ERR_INVALID; }
  if (done[device]) return LSNF_OK;
  LSNF_CUDA(cudaFuncSetAttribute(last_fused_kernel<3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
  LSNF_CUDA(cudaFuncSetAttribute(last_fused_kernel<4, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
  done[device] = true;
  return LSNF_OK;
}

}  // namespace lsnf
