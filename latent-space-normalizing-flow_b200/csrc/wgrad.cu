// Generator parameter gradients (train.py:390-394: loss_g = mse_sum(G(z_k), x) / B; loss_g.backward()).
//
// The data-gradient chain of the Langevin loop already leaves, for every layer l, the gradient w.r.t. its
// pre-activation output (gpre_l, LeakyReLU' applied) next to the layer's input activation act_{l-1}.  The weight
// gradient of a ConvTranspose2d is then, per kernel tap (ky, kx),
//     dW[ci][co][ky][kx] = sum_{b, iy, ix} act[b][iy][ix][ci] * gpre[b][iy*s - p + ky][ix*s - p + kx][co]
// i.e. a GEMM whose K axis is (batch x positions).  The tcgen05 tap-GEMM wants K-major operands, so both tensors are
// first TRANSPOSED to [channel][position] with the positions of every sample laid out on a grid with one zero halo
// row above and below (Hp = H + 2, Wp = W rounded up to 8): a vertical tap shift dy then is the constant offset dy*Wp
// along the flattened K axis and reads the zero halo outside the image.  TMA box origins must be 16-byte aligned
// along the innermost axis (an odd element offset raises an illegal-instruction fault), so the horizontal shift
// dx = +-1 cannot be a coordinate offset: the transposed gradient is stored twice per phase plane, as is and
// pre-shifted by one column (`xvar`), and each tap picks its copy.  One 2-D TMA box per K block feeds each operand
// (wgrad stages of tapgemm_tc_kernel).  Values are re-split to bf16 hi|lo pairs (fp32 range, 16 significant bits; 3 MMA passes).
// A finalize kernel sums the split-K partials and writes the gradient in the parameter's own [C_in][C_out][k][k]
// layout; bias gradients are row sums of the transposed gradient.
#include <algorithm>

#include "lsnf_internal.cuh"

namespace lsnf {

// ---------------------------------------------------------------------------------------------------
// [P][B][H][W][2C] 16-bit hi|lo (position-major)  ->  [P][c_rows][2*Kp] bf16 hi|lo (channel-major, zero halo)
// ---------------------------------------------------------------------------------------------------

constexpr int TR_POS = 32, TR_CH = 64;

// One CTA moves a tile of 32 positions x 64 channels through shared memory: coalesced 16-byte reads along the channel
// axis, then 16-byte stores along the position axis whenever eight consecutive positions are eight consecutive,
// 16-byte-aligned K indices (rows of a grid whose width is a multiple of 8, or an unpadded flat layout); narrower grids
// fall back to 2-byte stores.  The tile carries one halo position on either side so that the column-shifted copy
// (TransArgs::xvar) is written with aligned vectors too.
__global__ void __launch_bounds__(256) transpose_hl_kernel(TransArgs a) {
  __shared__ __align__(16) uint16_t hi[TR_CH][TR_POS + 8], lo[TR_CH][TR_POS + 8];   // column 1 + i = position pos0 + i
  const int tid = threadIdx.x;
  const long long npos = (long long)a.B * a.H * a.W;
  const long long pos0 = (long long)blockIdx.x * TR_POS;
  const int c0 = blockIdx.y * TR_CH, p = blockIdx.z;
  // ---- load: 32 positions (+ 2 halo positions) x 8 channels per thread ----
  for (int task = tid; task < (TR_POS + 2) * 8; task += blockDim.x) {
    const int col = task >> 3, cq = task & 7;        // col 0 / 33 are the halo positions pos0 - 1 / pos0 + 32
    const long long pos = pos0 + col - 1;
    const int c = c0 + cq * 8;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = 0.f;
    const bool halo_col = col == 0 || col == TR_POS + 1;
    if (pos >= 0 && pos < npos && c < a.C && (!halo_col || a.xvar)) {
      const int x = (int)(pos % a.W), y = (int)((pos / a.W) % a.H), b = (int)(pos / ((long long)a.W * a.H));
      const uint16_t* src = a.src + (long long)p * a.s_plane + (long long)b * a.s_b + (long long)y * a.s_h + (long long)x * a.s_w + c;
      __align__(16) uint16_t h8[8], l8[8];
      *reinterpret_cast<uint4*>(h8) = *reinterpret_cast<const uint4*>(src);
      if (!a.src_single) *reinterpret_cast<uint4*>(l8) = *reinterpret_cast<const uint4*>(src + a.C);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = join16(h8[j], a.src_single ? (uint16_t)0 : l8[j], a.src_fp16 != 0);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      uint16_t h, l;
      split16(v[j], false, h, l);
      hi[cq * 8 + j][col] = h; lo[cq * 8 + j][col] = l;
    }
  }
  __syncthreads();
  // ---- store: one channel row x 8 positions per thread ----
  const int cr = tid >> 2, pq = tid & 3;
  const int c = c0 + cr;
  if (c >= a.C) return;
  const int nvar = a.xvar ? 2 : 1;
  uint16_t* row = a.dst + ((long long)p * nvar * a.c_rows + c) * 2 * a.Kp;
  uint16_t* row1 = row + (long long)a.c_rows * 2 * a.Kp;   // the column-shifted copy
  const int sh = (p & 1) ? 1 : -1;
  const long long g0 = pos0 + pq * 8;                     // first position of this thread's group
  const bool flat = a.halo == 0 && a.Hp == a.H && a.Wp == a.W;   // K index == position index
  if ((flat || a.W % 8 == 0) && !(a.xvar && flat)) {
    if (g0 >= npos && !flat) return;
    if (flat && g0 >= a.Kp) return;
    long long k;
    int x0 = 0;
    if (flat) k = g0;   // positions past the end of the batch hold zeros in the tile: they fill the K padding
    else {
      x0 = (int)(g0 % a.W);
      const int y = (int)((g0 / a.W) % a.H), b = (int)(g0 / ((long long)a.W * a.H));
      k = ((long long)b * a.Hp + y + a.halo) * a.Wp + x0;
    }
    __align__(16) uint16_t vh[8], vl[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { vh[j] = hi[cr][1 + pq * 8 + j]; vl[j] = lo[cr][1 + pq * 8 + j]; }
    *reinterpret_cast<uint4*>(row + k) = *reinterpret_cast<const uint4*>(vh);
    *reinterpret_cast<uint4*>(row + a.Kp + k) = *reinterpret_cast<const uint4*>(vl);
    if (a.xvar) {   // column x of the shifted copy holds source column x - sh (zero outside the row)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int xs = x0 + j - sh;
        const bool ok = xs >= 0 && xs < a.W;
        vh[j] = ok ? hi[cr][1 + pq * 8 + j - sh] : (uint16_t)0;
        vl[j] = ok ? lo[cr][1 + pq * 8 + j - sh] : (uint16_t)0;
      }
      *reinterpret_cast<uint4*>(row1 + k) = *reinterpret_cast<const uint4*>(vh);
      *reinterpret_cast<uint4*>(row1 + a.Kp + k) = *reinterpret_cast<const uint4*>(vl);
    }
    return;
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const long long pos = g0 + j;
    if (pos < npos) {
      const int x = (int)(pos % a.W), y = (int)((pos / a.W) % a.H), b = (int)(pos / ((long long)a.W * a.H));
      const long long k = ((long long)b * a.Hp + y + a.halo) * a.Wp + x;
      row[k] = hi[cr][1 + pq * 8 + j];
      row[a.Kp + k] = lo[cr][1 + pq * 8 + j];
      if (a.xvar && x + sh >= 0 && x + sh < a.W) {
        row1[k + sh] = hi[cr][1 + pq * 8 + j];
        row1[a.Kp + k + sh] = lo[cr][1 + pq * 8 + j];
      }
    }
  }
}

int launch_transpose_hl(const TransArgs& a, cudaStream_t s) {
  const long long npos = (long long)a.B * a.H * a.W;
  dim3 grid((unsigned)((npos + TR_POS - 1) / TR_POS), (unsigned)((a.C + TR_CH - 1) / TR_CH), (unsigned)a.P);
  transpose_hl_kernel<<<grid, 256, 0, s>>>(a);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// split-K partials [tap][split][C_in][n_pad] -> dW in the parameter's layout [C_in][C_out][kk], times `scale`
// generic source index: tap * s_tap + split * s_split + ci * s_ci + co
// ---------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(256) wgrad_finalize_kernel(FinalizeArgs a) {
  __shared__ float tile[64][33];   // [tap][co]
  const int ci = blockIdx.y, co0 = blockIdx.x * 32;
  const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const int co = co0 + lane;
  for (int tap = grp; tap < a.kk; tap += 8) {
    float v = 0.f;
    if (co < a.C_out) {
      const float* p = a.part + (long long)tap * a.s_tap + (long long)ci * a.s_ci + co;
      for (int s = 0; s < a.ksplit; ++s) v += __ldcg(p + (long long)s * a.s_split);   // fixed order: deterministic
    }
    tile[tap][lane] = v * a.scale;
  }
  __syncthreads();
  const int ncol = min(32, a.C_out - co0);
  float* o = a.out + ((long long)ci * a.C_out + co0) * a.kk;
  for (int i = threadIdx.x; i < ncol * a.kk; i += blockDim.x) o[i] = tile[i % a.kk][i / a.kk];
}

int launch_wgrad_finalize(const FinalizeArgs& a, cudaStream_t s) {
  if (a.kk > 64) { set_error("wgrad finalize: more than 64 taps"); return LSNF_ERR_INVALID; }
  dim3 grid((unsigned)((a.C_out + 31) / 32), (unsigned)a.C_in);
  wgrad_finalize_kernel<<<grid, 256, 0, s>>>(a);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// bias gradient: db[c] = scale * sum over the selected rows (sel[j] + c) of a transposed hi|lo matrix of ALL their
// 2*Kp elements (value = hi + lo, the halo is zero).  One CTA per output channel.
// ---------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(256) bias_rowsum_kernel(RowSumArgs a) {
  __shared__ float red[256];
  const int c = blockIdx.x;
  float acc = 0.f;
  for (int j = 0; j < a.nsel; ++j) {
    const uint4* row = reinterpret_cast<const uint4*>(a.src + (long long)(a.sel[j] + c) * 2 * a.Kp);
    const long long n16 = 2 * a.Kp / 8;   // Kp is a multiple of 64
    for (long long i = threadIdx.x; i < n16; i += blockDim.x) {
      const uint4 q = __ldg(row + i);
      const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        acc += __uint_as_float(w[t] << 16);            // bf16 -> fp32: the low element
        acc += __uint_as_float(w[t] & 0xFFFF0000u);    // the high element
      }
    }
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) a.out[c] = red[0] * a.scale;
}

int launch_bias_rowsum(const RowSumArgs& a, cudaStream_t s) {
  bias_rowsum_kernel<<<a.C, 256, 0, s>>>(a);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// loss_g = scale * sum (x_hat - x)^2 (train.py:393), or scale * sum m (x_hat - x)^2 with a mask (nullable): 64 CTAs leave
// fixed-order partial sums, the last one to finish adds them in index order (deterministic).  fmaf(m*d, d, acc) equals
// fmaf(d, d, acc) for m = 1, so an all-ones mask reproduces the unmasked loss bit for bit.
// ---------------------------------------------------------------------------------------------------
constexpr int MSE_CTAS = 64;
__global__ void __launch_bounds__(256) mse_sum_kernel(const float* __restrict__ xh, const float* __restrict__ x,
                                                      const float* __restrict__ mask, long long n, float scale, float* __restrict__ partial,
                                                      unsigned int* __restrict__ ticket, float* __restrict__ out) {
  __shared__ float red[256];
  __shared__ bool last;
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float d = xh[i] - x[i];
    acc = fmaf(mask ? mask[i] * d : d, d, acc);
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    partial[blockIdx.x] = red[0];
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (unsigned i = 0; i < gridDim.x; ++i) t += __ldcg(partial + i);
    *out = t * scale;
    *ticket = 0u;
  }
}

int launch_mse_sum(const float* xh, const float* x, const float* mask, long long n, float scale, float* partial,
                   unsigned int* ticket, float* out, cudaStream_t s) {
  mse_sum_kernel<<<MSE_CTAS, 256, 0, s>>>(xh, x, mask, n, scale, partial, ticket, out);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

// ---------------------------------------------------------------------------------------------------
// loss_g of a measured update = scale * sum of the n fixed-order partials of |r 2^k|^2 that meas_finish_kernel left
// ([B][meas_tiles]); scale = 2^-2k / global_batch.  One CTA: thread t sums partials t, t + 256, ... in index order,
// then a fixed tree, so the result does not depend on timing (no atomics).
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) meas_loss_kernel(const float* __restrict__ part, int n, float scale,
                                                        float* __restrict__ out) {
  __shared__ float red[256];
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) acc += part[i];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = red[0] * scale;
}

int launch_meas_loss(const float* part, int n, float scale, float* out, cudaStream_t s) {
  meas_loss_kernel<<<1, 256, 0, s>>>(part, n, scale, out);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

}  // namespace lsnf
