// Fused flow-prior kernels (fp32 CUDA cores): actnorm -> invertible 1x1 (or fixed shuffle) -> coupling,
// all f_depth steps in one launch, per-sample log-det and log p(z) reduced in-kernel, followed (same launch)
// by the analytic backward d(-sum_b log p(z_b))/dz.  Reference: model.py:357-365 (revnet2d), :389-458
// (revnet2d_step), :280-294 (actnorm), :179-198 (invertible_1x1_conv), :306-350 (coupling MLP),
// train.py:316-323 (log-prior and its gradient).  Backward formulas: SURVEY.md section 8a, row A5
// (pinned against autograd in fp64 by tests/test_oracle_golden.py).
#include <mutex>

#include "lsnf_internal.cuh"

namespace lsnf {

struct FlowArgs {
  const float* params;  // f_depth blocks of FlowLayout::step_floats
  FlowLayout fl;
  int depth, B, coupling, permutation;
  const float* in;      // z (forward) or eps (inverse), [B][nz]
  float* z_out;         // forward: z_out; inverse: z
  float* logdet;        // forward: logdet; inverse: -objective
  float* logp;
  float* grad;
  uint32_t ring_floats;  // shared-memory ring that streams the matrices
  float* stash;          // TRAIN instantiation: per-layer, per-sample vectors the parameter gradients are built from
  FlowStash sl;
  // upstream gradients of the backward (lsnf_flow_vjp): dL/dz_out [B][nz] and dL/dlogdet [B].  Both null: the seeds of
  // -sum_b log p(z_b), g = z_out and dL/dlogdet = -1; otherwise a null one stands for zero
  const float* seed_g;
  const float* seed_ld;
};

constexpr int FLOW_THREADS = 256;

// ---- shared-memory staging of the parameters: cp.async.bulk (1-D TMA) + mbarrier, double-buffered ----
// Every matrix of the coupling layers is streamed global -> shared while the previous mat-vec computes, and the
// per-step vectors (actnorm b / exp(3 logs), MLP biases and scales) travel as one block per step; the mat-vecs then
// read shared memory only ("the small coupling MLPs stay SMEM-resident").
__device__ __forceinline__ uint32_t f_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void f_mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void f_bulk_load(uint32_t dst, const float* src, uint32_t bytes, uint32_t bar) {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

constexpr int FEED_SLOTS = 8;      // matrices that may be in flight at once (mbarrier slots)
constexpr int FEED_MAX_ITEMS = 320; // f_depth <= 32, at most 2 passes x 4 matrices per step (+ slack)

// Streams the matrices of the whole pass through a shared-memory byte ring: thread 0 keeps issuing bulk copies for
// as many upcoming matrices as fit (typically 4-6 in flight, > 100 KB), so the mat-vec chain never waits for a
// copy.  Space is reclaimed in FIFO order when the mat-vec that used it has passed its closing __syncthreads.
// The (source offset, size) of every item is tabulated once in shared memory.
struct Feeder {
  const float* params;
  float* ring;            // [ring_floats]
  float* vbase;           // two per-step vector blocks, back to back
  uint2* items;           // [n_mat] (float offset into params, floats)
  uint32_t* item_off;     // [FEED_SLOTS] placement of each in-flight matrix (floats from `ring`)
  uint32_t* item_fp;      // [FEED_SLOTS] footprint incl. wrap waste
  uint32_t bar0, vbar0;   // shared addresses of the mbarrier arrays
  uint32_t ring_floats, vec_floats, step_floats;
  uint32_t m, v;          // next matrix / vector-block item to be consumed
  uint32_t next_issue, head, used;   // producer state (meaningful in thread 0 only)
  int n_mat, n_vec, depth, inverse;

  __device__ __forceinline__ int vec_layer(int idx) const {
    if (inverse) return depth - 1 - idx;
    return idx < depth ? idx : 2 * depth - 1 - idx;
  }
  // thread 0: issue every upcoming matrix that fits into the ring (FIFO allocation with wrap-around)
  __device__ __forceinline__ void pump(uint32_t consumer) {
    while ((int)next_issue < n_mat && next_issue < consumer + FEED_SLOTS - 1) {
      const uint2 it = items[next_issue];
      const uint32_t n = it.y;
      uint32_t place, fp;
      if (used == 0) head = 0;   // empty ring: restart at the beginning (guarantees progress when ring < 2 matrices)
      if (head + n > ring_floats) {
        const uint32_t waste = ring_floats - head;
        if (used + waste + n > ring_floats) break;
        place = 0; fp = waste + n; head = n;
      } else {
        if (used + n > ring_floats) break;
        place = head; fp = n; head += n;
      }
      const uint32_t slot = next_issue % FEED_SLOTS;
      item_off[slot] = place; item_fp[slot] = fp;
      used += fp;
      f_bulk_load(f_smem_u32(ring + place), params + it.x, n * 4u, bar0 + 8u * slot);
      ++next_issue;
    }
  }
  __device__ __forceinline__ void issue_vec(int idx) {
    if (idx >= n_vec) return;
    f_bulk_load(f_smem_u32(vbase + (idx & 1) * vec_floats), params + (size_t)vec_layer(idx) * step_floats,
                vec_floats * 4u, vbar0 + 8u * (idx & 1));
  }
  // Returns the staged matrix of the current item.  The previous item's space is reclaimed here: its mat-vec has
  // passed its closing __syncthreads, so no thread reads it any more.
  __device__ __forceinline__ const float* next_mat() {
    const uint32_t i = m++;
    if (threadIdx.x == 0) {
      if (i > 0) used -= item_fp[(i - 1) % FEED_SLOTS];
      pump(i);
    }
    const uint32_t slot = i % FEED_SLOTS;
    f_mbar_wait(bar0 + 8u * slot, (i / FEED_SLOTS) & 1u);
    return ring + item_off[slot];
  }
  __device__ __forceinline__ const float* next_vec() {
    const uint32_t i = v++;
    f_mbar_wait(vbar0 + 8u * (i & 1), (i >> 1) & 1u);
    if (threadIdx.x == 0) issue_vec((int)i + 1);
    return vbase + (i & 1) * vec_floats;
  }
};

// matrix item -> (offset, floats).  forward pass: per step [W] W1 W2 W3; backward: per step (descending) W3T W2T
// W1T [WT]; inverse pass: per step (descending) W1 W2 W3 [Winv]
__device__ __forceinline__ uint2 flow_mat_item(const FlowLayout& f, int depth, bool perm2, bool inverse, int idx) {
  const int nz = f.nz, w = f.w, half = f.half, n_out = f.n_out;
  const int ipl = perm2 ? 4 : 3;
  int L, j;
  bool bwd = false;
  if (inverse) { L = depth - 1 - idx / ipl; j = idx % ipl; }
  else if (idx < depth * ipl) { L = idx / ipl; j = idx % ipl + (perm2 ? 0 : 1); }
  else { bwd = true; idx -= depth * ipl; L = depth - 1 - idx / ipl; j = idx % ipl; }
  size_t o; uint32_t c;
  if (inverse) {
    if (j == 0) { o = f.W1; c = half * w; } else if (j == 1) { o = f.W2; c = w * w; }
    else if (j == 2) { o = f.W3; c = w * n_out; } else { o = f.Winv; c = nz * nz; }
  } else if (!bwd) {
    if (j == 0) { o = f.W; c = nz * nz; } else if (j == 1) { o = f.W1; c = half * w; }
    else if (j == 2) { o = f.W2; c = w * w; } else { o = f.W3; c = w * n_out; }
  } else {
    if (j == 0) { o = f.W3T; c = w * n_out; } else if (j == 1) { o = f.W2T; c = w * w; }
    else if (j == 2) { o = f.W1T; c = half * w; } else { o = f.WT; c = nz * nz; }
  }
  return make_uint2((uint32_t)((size_t)L * f.step_floats + o), c);
}

// carve the dynamic shared memory; returns the first free float
__device__ __forceinline__ float* feeder_init(Feeder& fd, float* sm, const FlowArgs& a, bool with_bwd, bool inverse) {
  const FlowLayout& f = a.fl;
  const bool perm2 = a.permutation == 2;
  const int ipl = perm2 ? 4 : 3;
  fd.params = a.params; fd.depth = a.depth; fd.inverse = inverse;
  fd.n_mat = a.depth * ipl * ((with_bwd && !inverse) ? 2 : 1);
  fd.n_vec = a.depth * ((with_bwd && !inverse) ? 2 : 1);
  fd.m = fd.v = 0;
  fd.next_issue = fd.head = fd.used = 0;
  fd.ring_floats = a.ring_floats; fd.vec_floats = (uint32_t)f.vec_floats; fd.step_floats = (uint32_t)f.step_floats;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm);   // FEED_SLOTS + 2 mbarriers (the buffer is 16-byte aligned)
  fd.bar0 = f_smem_u32(bars);
  fd.vbar0 = f_smem_u32(bars + FEED_SLOTS);
  fd.item_off = reinterpret_cast<uint32_t*>(bars + FEED_SLOTS + 2);
  fd.item_fp = fd.item_off + FEED_SLOTS;
  fd.items = reinterpret_cast<uint2*>(fd.item_fp + FEED_SLOTS);
  float* p = sm + 2 * (FEED_SLOTS + 2) + 2 * FEED_SLOTS + 2 * FEED_MAX_ITEMS;
  fd.vbase = p; p += 2 * f.vec_floats;
  fd.ring = p; p += a.ring_floats;
  for (int i = threadIdx.x; i < fd.n_mat; i += blockDim.x) fd.items[i] = flow_mat_item(f, a.depth, perm2, inverse, i);
  if (threadIdx.x == 0) {
    for (int i = 0; i < FEED_SLOTS + 2; ++i)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(f_smem_u32(bars + i)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) { fd.issue_vec(0); fd.pump(0); }
  return p;
}

// Activations live in shared memory SAMPLE-MINOR: element (sample s, feature j) of a buffer is buf[j*S + s], so a
// mat-vec reads the S samples of one feature with ONE broadcast vector load.
template <int S>
struct SVec { float v[S]; };
template <int S>
__device__ __forceinline__ SVec<S> load_samples(const float* p) {
  SVec<S> r;
  if constexpr (S == 1) { r.v[0] = p[0]; }
  else if constexpr (S == 2) { const float2 t = *reinterpret_cast<const float2*>(p); r.v[0] = t.x; r.v[1] = t.y; }
  else {
#pragma unroll
    for (int q = 0; q < S; q += 4) {
      const float4 t = *reinterpret_cast<const float4*>(p + q);
      r.v[q] = t.x; r.v[q + 1] = t.y; r.v[q + 2] = t.z; r.v[q + 3] = t.w;
    }
  }
  return r;
}

// epi(s, j, sum_k in[k][s] * M[k*N + j]) for s < S, j < N.  M is row-major [K][N] in SHARED memory (conflict-free
// along j); `in` is a sample-minor [K][S] shared-memory buffer.  The K range is split across 256/Nr thread groups
// whose partial sums meet in `scratch`.
template <int S, class Epi>
__device__ __forceinline__ void matvec(const float* M, int K, int N, const float* in, float* scratch, Epi epi) {
  const int Nr = (N + 31) & ~31;
  const int G = FLOW_THREADS / Nr > 0 ? FLOW_THREADS / Nr : 1;
  const int tid = threadIdx.x;
  const int Kc = (K + G - 1) / G;
  for (int j0 = 0; j0 < N; j0 += FLOW_THREADS) {   // only loops when N > 256 (never: nz, f_width <= 256)
    const int g = tid / Nr, j = j0 + tid % Nr;
    if (g < G && j < N) {
      float acc[S];
#pragma unroll
      for (int s = 0; s < S; ++s) acc[s] = 0.f;
      const int k0 = g * Kc, k1 = min(K, k0 + Kc);
      const float* m = M + (size_t)k0 * N + j;
      const float* x = in + (size_t)k0 * S;
#pragma unroll 8
      for (int k = k0; k < k1; ++k, m += N, x += S) {
        const float w = *m;
        const SVec<S> xv = load_samples<S>(x);
#pragma unroll
        for (int s = 0; s < S; ++s) acc[s] = fmaf(xv.v[s], w, acc[s]);
      }
#pragma unroll
      for (int s = 0; s < S; ++s) scratch[(g * S + s) * Nr + (j - j0)] = acc[s];
    }
    __syncthreads();
    for (int i = tid; i < S * Nr; i += FLOW_THREADS) {
      const int s = i / Nr, jj = i % Nr;
      if (j0 + jj < N) {
        float v = 0.f;
        for (int g2 = 0; g2 < G; ++g2) v += scratch[(g2 * S + s) * Nr + jj];
        epi(s, j0 + jj, v);
      }
    }
    __syncthreads();
  }
}

// sum over the threads of the CTA of one value per sample slot (warp shuffles, then one shared-memory pass)
template <int S>
__device__ __forceinline__ void block_sum(float (&v)[S], float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int s = 0; s < S; ++s) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[s] += __shfl_xor_sync(0xffffffffu, v[s], o);
    if (lane == 0) red[warp * S + s] = v[s];
  }
  __syncthreads();
#pragma unroll
  for (int s = 0; s < S; ++s) {
    float t = 0.f;
    for (int w = 0; w < FLOW_THREADS / 32; ++w) t += red[w * S + s];
    v[s] = t;
  }
  __syncthreads();
}

#define AT(buf, s, j) (buf)[(j) * S + (s)]

// element (layer L, slot offset `slot`, sample b, feature j) of the training stash
__device__ __forceinline__ float* stash_at(const FlowArgs& a, int L, size_t slot, int dim, int b, int j) {
  return a.stash + (size_t)L * a.sl.layer_floats * a.B + slot * a.B + (size_t)b * dim + j;
}

// TRAIN = true (flow parameter update, train.py:403-415): the same forward + analytic backward, additionally
// writing for every step and sample the vectors whose batch outer products are the parameter gradients
// (flow_param_grad_kernel): layer inputs y, u1, a1, a2, the MLP output h, the gradients w.r.t. the four matmul
// outputs g_u, g_p1, g_p2, g_p3, w.r.t. the step input g_x, and the per-element log-scale terms gl0..gl3.
template <int S, bool TRAIN>
__global__ void __launch_bounds__(FLOW_THREADS) flow_forward_kernel(FlowArgs a) {
  extern __shared__ __align__(16) float sm[];
  const FlowLayout& f = a.fl;
  const int nz = f.nz, w = f.w, half = f.half, n_out = f.n_out;
  const int nmax = max(nz, max(w, n_out));
  const int nr_max = (nmax + 31) & ~31;
  const int stash_step = 2 * w + nz;  // a1[w], a2[w], scale[half], x2+shift[half]  (each x S samples)
  Feeder fd;
  float* cur = feeder_init(fd, sm, a, a.grad != nullptr, false);   // [nz][S]
  float* ta = cur + S * nz;                // [nmax][S]
  float* tb = ta + S * nmax;               // [nmax][S]
  float* scratch = tb + S * nmax;          // partial sums: G*S*Nr <= 256*S
  float* red = scratch + S * max(FLOW_THREADS, nr_max);
  float* stash = red + (FLOW_THREADS / 32) * S;  // [depth][stash_step][S]
  const int tid = threadIdx.x;
  const int b0 = blockIdx.x * S;
  const int ns = min(S, a.B - b0);

  for (int i = tid; i < S * nz; i += FLOW_THREADS) {
    const int s = i / nz, j = i % nz;     // coalesced global read
    AT(cur, s, j) = s < ns ? a.in[(size_t)(b0 + s) * nz + j] : 0.f;
  }
  __syncthreads();

  float ld[S];  // per-thread partial of sum_j log(scale); constants are added by thread 0 only
#pragma unroll
  for (int s = 0; s < S; ++s) ld[s] = 0.f;

  for (int L = 0; L < a.depth; ++L) {
    const float* P = fd.next_vec();   // this step's vectors, in shared memory
    float* st = stash + (size_t)L * S * stash_step;
    // actnorm (model.py:282-284): (x + b) * exp(3 logs)
    for (int i = tid; i < S * nz; i += FLOW_THREADS) {
      const int j = i / S;
      ta[i] = (cur[i] + P[f.an_b + j]) * P[f.an_e + j];
    }
    __syncthreads();
    if constexpr (TRAIN) {
      for (int i = tid; i < S * nz; i += FLOW_THREADS) {
        const int s = i / nz, j = i % nz;
        if (s < ns) *stash_at(a, L, a.sl.y, nz, b0 + s, j) = AT(ta, s, j);
      }
    }
    if (a.permutation == 2) {   // model.py:187: z @ W
      matvec<S>(fd.next_mat(), nz, nz, ta, scratch, [&](int s, int j, float v) { AT(cur, s, j) = v; });
    } else {                    // intended shuffle_features: h[:, idx]
      const int* idx = reinterpret_cast<const int*>(P + f.perm);
      for (int i = tid; i < S * nz; i += FLOW_THREADS) cur[i] = AT(ta, i % S, idx[i / S]);
      __syncthreads();
    }
    if (tid == 0) {
#pragma unroll
      for (int s = 0; s < S; ++s) ld[s] += P[f.ld_const] , ld[s] += P[f.ld_const + 1];
    }
    if constexpr (TRAIN) {
      for (int i = tid; i < S * half; i += FLOW_THREADS) {
        const int s = i / half, j = i % half;
        if (s < ns) *stash_at(a, L, a.sl.u1, half, b0 + s, j) = AT(cur, s, j);
      }
    }
    // coupling MLP on x1 = cur[:half] (model.py:306-310)
    float* a1 = st;             // [w][S]
    float* a2 = st + S * w;     // [w][S]
    float* sc = a2 + S * w;     // [half][S]
    float* xs = sc + S * half;  // [half][S]
    matvec<S>(fd.next_mat(), half, w, cur, scratch,
              [&](int s, int j, float v) { AT(a1, s, j) = fmaxf((v + P[f.b1 + j]) * P[f.e1 + j], 0.f); });
    matvec<S>(fd.next_mat(), w, w, a1, scratch,
              [&](int s, int j, float v) { AT(a2, s, j) = fmaxf((v + P[f.b2 + j]) * P[f.e2 + j], 0.f); });
    matvec<S>(fd.next_mat(), w, n_out, a2, scratch,
              [&](int s, int j, float v) { AT(ta, s, j) = (v + P[f.b3 + j]) * P[f.e3 + j]; });
    if constexpr (TRAIN) {
      for (int i = tid; i < S * w; i += FLOW_THREADS) {
        const int s = i / w, j = i % w;
        if (s < ns) {
          *stash_at(a, L, a.sl.a1, w, b0 + s, j) = AT(a1, s, j);
          *stash_at(a, L, a.sl.a2, w, b0 + s, j) = AT(a2, s, j);
        }
      }
      for (int i = tid; i < S * n_out; i += FLOW_THREADS) {
        const int s = i / n_out, j = i % n_out;
        if (s < ns) *stash_at(a, L, a.sl.h, n_out, b0 + s, j) = AT(ta, s, j);
      }
    }
    float* x2 = cur + S * half;   // [half][S]
    if (a.coupling == 1) {      // model.py:410-418
      for (int i = tid; i < S * half; i += FLOW_THREADS) {
        const int s = i % S, j = i / S;
        const float shift = AT(ta, s, 2 * j);
        const float scale = 1.f / (1.f + expf(-(AT(ta, s, 2 * j + 1) + 2.f)));
        const float x2s = x2[i] + shift;
        x2[i] = x2s * scale;
        sc[i] = scale; xs[i] = x2s;
#pragma unroll
        for (int q = 0; q < S; ++q) if (q == s) ld[q] += logf(scale);
      }
    } else {                    // model.py:407-408
      for (int i = tid; i < S * half; i += FLOW_THREADS) x2[i] += ta[i];
    }
    __syncthreads();
  }

  // log-det and log p(z) (train.py:317-319), warp-shuffle reductions
  block_sum<S>(ld, red);
  float sq[S];
#pragma unroll
  for (int s = 0; s < S; ++s) sq[s] = 0.f;
  for (int i = tid; i < S * nz; i += FLOW_THREADS) {
    const int s = i % S;
    const float v = cur[i];
#pragma unroll
    for (int q = 0; q < S; ++q) if (q == s) sq[q] += -0.5f * v * v;
  }
  block_sum<S>(sq, red);
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < S; ++s) {
      if (s < ns) {
        if (a.logdet) a.logdet[b0 + s] = ld[s];
        if (a.logp) a.logp[b0 + s] = sq[s] + 1.8378770664093453f + ld[s];  // log(2 pi), train.py:318
      }
    }
  }
  if (a.z_out)
    for (int i = tid; i < S * nz; i += FLOW_THREADS) {
      const int s = i / nz, j = i % nz;
      if (s < ns) a.z_out[(size_t)(b0 + s) * nz + j] = AT(cur, s, j);
    }
  if (!a.grad) return;
  // the backward overwrites cur in place (g2p below, with another thread-to-element mapping): every thread must be
  // done reading it for the z_out store first
  if (a.z_out) __syncthreads();

  // ---- analytic backward of -sum_b ll_b: seed g = z_out, d/dlogdet = -1 (or the caller's seeds) ----
  float* g = cur;  // in place, [nz][S]
  float* g2p = g + S * half;
  const bool seeded = a.seed_g || a.seed_ld;
  if (seeded) {
    for (int i = tid; i < S * nz; i += FLOW_THREADS) {
      const int s = i / nz, j = i % nz;
      AT(g, s, j) = (a.seed_g && s < ns) ? a.seed_g[(size_t)(b0 + s) * nz + j] : 0.f;
    }
    __syncthreads();
  }
  for (int L = a.depth - 1; L >= 0; --L) {
    const float* P = fd.next_vec();
    float* st = stash + (size_t)L * S * stash_step;
    const float* a1 = st;
    const float* a2 = st + S * w;
    const float* sc = a2 + S * w;
    const float* xs = sc + S * half;
    // gradient w.r.t. the MLP output h, already multiplied by e3 = exp(3 logs_zeros)
    if (a.coupling == 1) {
      // d/dscale of the step's output and of logdet += log(scale) is g2 * x2s - (-dL/dlogdet) / scale.  The default
      // seed's loop and the caller-seeded one are separate instances of the same expression, so that the default keeps
      // its own rounding and a caller seed of -1 reproduces it bit for bit.
      auto coupling_bwd = [&](auto g_scale_of) {
        for (int i = tid; i < S * half; i += FLOW_THREADS) {
          const int s = i % S, j = i / S;
          const float g2 = g2p[i], scale = sc[i];
          const float g_shift = g2 * scale;
          const float g_scale = g_scale_of(g2, xs[i], scale, s);
          const float gh0 = g_shift, gh1 = g_scale * scale * (1.f - scale);
          AT(ta, s, 2 * j) = gh0 * P[f.e3 + 2 * j];
          AT(ta, s, 2 * j + 1) = gh1 * P[f.e3 + 2 * j + 1];
          g2p[i] = g_shift;  // = g_x2
          if constexpr (TRAIN) {
            if (s < ns) {   // d/dlogs of h = (p + b) * exp(3 logs) is 3 h (model.py:348)
              const float* hrow = stash_at(a, L, a.sl.h, n_out, b0 + s, 2 * j);
              float* gl = stash_at(a, L, a.sl.gl3, n_out, b0 + s, 2 * j);
              gl[0] = 3.f * gh0 * hrow[0];
              gl[1] = 3.f * gh1 * hrow[1];
            }
          }
        }
      };
      if (seeded)
        coupling_bwd([&](float g2, float x2s, float scale, int s) {
          const float neg_ld = (a.seed_ld && s < ns) ? -a.seed_ld[b0 + s] : 0.f;
          return g2 * x2s - neg_ld / scale;
        });
      else
        coupling_bwd([](float g2, float x2s, float scale, int) { return g2 * x2s - 1.f / scale; });
    } else {
      for (int i = tid; i < S * half; i += FLOW_THREADS) {
        const int s = i % S, j = i / S;
        const float gh = g2p[i];
        ta[i] = gh * P[f.e3 + j];
        if constexpr (TRAIN) {
          if (s < ns) *stash_at(a, L, a.sl.gl3, n_out, b0 + s, j) = 3.f * gh * *stash_at(a, L, a.sl.h, n_out, b0 + s, j);
        }
      }
    }
    __syncthreads();
    if constexpr (TRAIN) {
      for (int i = tid; i < S * n_out; i += FLOW_THREADS) {
        const int s = i / n_out, j = i % n_out;
        if (s < ns) *stash_at(a, L, a.sl.gp3, n_out, b0 + s, j) = AT(ta, s, j);
      }
    }
    matvec<S>(fd.next_mat(), n_out, w, ta, scratch, [&](int s, int j, float v) {
      const float act = AT(a2, s, j);
      const float gq = act > 0.f ? v : 0.f;   // gradient w.r.t. the actnorm output of fc_2 (ReLU mask applied)
      AT(tb, s, j) = gq * P[f.e2 + j];
      if constexpr (TRAIN) {
        if (s < ns) {
          *stash_at(a, L, a.sl.gp2, w, b0 + s, j) = gq * P[f.e2 + j];
          *stash_at(a, L, a.sl.gl2, w, b0 + s, j) = 3.f * gq * act;
        }
      }
    });
    matvec<S>(fd.next_mat(), w, w, tb, scratch, [&](int s, int j, float v) {
      const float act = AT(a1, s, j);
      const float gq = act > 0.f ? v : 0.f;
      AT(ta, s, j) = gq * P[f.e1 + j];
      if constexpr (TRAIN) {
        if (s < ns) {
          *stash_at(a, L, a.sl.gp1, w, b0 + s, j) = gq * P[f.e1 + j];
          *stash_at(a, L, a.sl.gl1, w, b0 + s, j) = 3.f * gq * act;
        }
      }
    });
    matvec<S>(fd.next_mat(), w, half, ta, scratch, [&](int s, int j, float v) { AT(g, s, j) += v; });
    for (int i = tid; i < S * nz; i += FLOW_THREADS) ta[i] = g[i];
    __syncthreads();
    if constexpr (TRAIN) {
      for (int i = tid; i < S * nz; i += FLOW_THREADS) {
        const int s = i / nz, j = i % nz;
        if (s < ns) *stash_at(a, L, a.sl.gu, nz, b0 + s, j) = AT(ta, s, j);
      }
    }
    // g_y = g_u @ W^T (or the inverse shuffle), g_x = g_y * exp(3 logs); d/dlogs of y = (x + b) exp(3 logs) is 3 y
    auto actnorm_bwd = [&](int s, int j, float gy) {
      const float gx = gy * P[f.an_e + j];
      AT(g, s, j) = gx;
      if constexpr (TRAIN) {
        if (s < ns) {
          *stash_at(a, L, a.sl.gx, nz, b0 + s, j) = gx;
          *stash_at(a, L, a.sl.gl0, nz, b0 + s, j) = 3.f * gy * *stash_at(a, L, a.sl.y, nz, b0 + s, j);
        }
      }
    };
    if (a.permutation == 2) {   // g @ W^T, then the actnorm scale
      matvec<S>(fd.next_mat(), nz, nz, ta, scratch, actnorm_bwd);
    } else {
      const int* inv = reinterpret_cast<const int*>(P + f.perm_inv);
      for (int i = tid; i < S * nz; i += FLOW_THREADS) {
        const int s = i % S, j = i / S;
        actnorm_bwd(s, j, AT(ta, s, inv[j]));
      }
      __syncthreads();
    }
  }
  for (int i = tid; i < S * nz; i += FLOW_THREADS) {
    const int s = i / nz, j = i % nz;
    if (s < ns) a.grad[(size_t)(b0 + s) * nz + j] = AT(g, s, j);
  }
}

// reverse pass (model.py:424-456, :361-363, :484-498)
template <int S>
__global__ void __launch_bounds__(FLOW_THREADS) flow_inverse_kernel(FlowArgs a) {
  extern __shared__ __align__(16) float sm[];
  const FlowLayout& f = a.fl;
  const int nz = f.nz, w = f.w, half = f.half, n_out = f.n_out;
  const int nmax = max(nz, max(w, n_out));
  const int nr_max = (nmax + 31) & ~31;
  Feeder fd;
  float* cur = feeder_init(fd, sm, a, false, true);   // [nz][S]
  float* ta = cur + S * nz;
  float* tb = ta + S * nmax;
  float* scratch = tb + S * nmax;
  float* red = scratch + S * max(FLOW_THREADS, nr_max);
  const int tid = threadIdx.x;
  const int b0 = blockIdx.x * S;
  const int ns = min(S, a.B - b0);
  for (int i = tid; i < S * nz; i += FLOW_THREADS) {
    const int s = i / nz, j = i % nz;
    AT(cur, s, j) = s < ns ? a.in[(size_t)(b0 + s) * nz + j] : 0.f;
  }
  __syncthreads();
  float ld[S];
#pragma unroll
  for (int s = 0; s < S; ++s) ld[s] = 0.f;
  float* x2 = cur + S * half;
  for (int L = a.depth - 1; L >= 0; --L) {
    const float* P = fd.next_vec();
    matvec<S>(fd.next_mat(), half, w, cur, scratch,
              [&](int s, int j, float v) { AT(ta, s, j) = fmaxf((v + P[f.b1 + j]) * P[f.e1 + j], 0.f); });
    matvec<S>(fd.next_mat(), w, w, ta, scratch,
              [&](int s, int j, float v) { AT(tb, s, j) = fmaxf((v + P[f.b2 + j]) * P[f.e2 + j], 0.f); });
    matvec<S>(fd.next_mat(), w, n_out, tb, scratch,
              [&](int s, int j, float v) { AT(ta, s, j) = (v + P[f.b3 + j]) * P[f.e3 + j]; });
    if (a.coupling == 1) {      // model.py:432-438
      for (int i = tid; i < S * half; i += FLOW_THREADS) {
        const int s = i % S, j = i / S;
        const float shift = AT(ta, s, 2 * j);
        const float scale = 1.f / (1.f + expf(-(AT(ta, s, 2 * j + 1) + 2.f)));
        x2[i] = x2[i] / scale - shift;
#pragma unroll
        for (int q = 0; q < S; ++q) if (q == s) ld[q] -= logf(scale);
      }
    } else {                    // model.py:429-430
      for (int i = tid; i < S * half; i += FLOW_THREADS) x2[i] -= ta[i];
    }
    __syncthreads();
    for (int i = tid; i < S * nz; i += FLOW_THREADS) tb[i] = cur[i];
    __syncthreads();
    if (a.permutation == 2) {   // model.py:193-196: z @ inverse(W), then actnorm reverse (:288-291)
      matvec<S>(fd.next_mat(), nz, nz, tb, scratch,
                [&](int s, int j, float v) { AT(cur, s, j) = v * P[f.an_ei + j] - P[f.an_b + j]; });
    } else {
      const int* inv = reinterpret_cast<const int*>(P + f.perm_inv);
      for (int i = tid; i < S * nz; i += FLOW_THREADS) {
        const int s = i % S, j = i / S;
        cur[i] = AT(tb, s, inv[j]) * P[f.an_ei + j] - P[f.an_b + j];
      }
      __syncthreads();
    }
    if (tid == 0) {
#pragma unroll
      for (int s = 0; s < S; ++s) ld[s] -= P[f.ld_const + 1], ld[s] -= P[f.ld_const];
    }
    __syncthreads();   // every read of this step's vector block is done before its buffer is refilled
  }
  block_sum<S>(ld, red);
  if (tid == 0 && a.logdet) {
#pragma unroll
    for (int s = 0; s < S; ++s)
      if (s < ns) a.logdet[b0 + s] = -ld[s];   // the reference returns -objective (model.py:498)
  }
  for (int i = tid; i < S * nz; i += FLOW_THREADS) {
    const int s = i / nz, j = i % nz;
    if (s < ns) a.z_out[(size_t)(b0 + s) * nz + j] = AT(cur, s, j);
  }
}
#undef AT

// ---------------------------------------------------------------------------------------------------
// parameter packing: one launch per flow step; builds transposes, exp(+-3 logs) and the log-det constants
// ---------------------------------------------------------------------------------------------------
struct FlowPackPtrs {
  const float* p[LSNF_FLOW_PTRS_PER_STEP];
  const float* winv;
  const int32_t* perm;
  const int32_t* perm_inv;
  const float* log_abs_det;  // device scalar (nullptr -> 0)
};

__global__ void flow_pack_kernel(FlowPackPtrs q, FlowLayout f, float* __restrict__ out, int permutation) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  const int nz = f.nz, w = f.w, half = f.half, n_out = f.n_out;
  for (int i = tid; i < nz; i += nt) {
    out[f.an_b + i] = q.p[0][i];
    out[f.an_e + i] = expf(q.p[1][i] * 3.f);
    out[f.an_ei + i] = expf(-(q.p[1][i] * 3.f));
    if (permutation == 1) {
      reinterpret_cast<int*>(out + f.perm)[i] = q.perm[i];
      reinterpret_cast<int*>(out + f.perm_inv)[i] = q.perm_inv[i];
    }
  }
  if (permutation == 2)
    for (int i = tid; i < nz * nz; i += nt) {
      const int r = i / nz, c = i % nz;
      out[f.W + i] = q.p[2][i];
      out[f.WT + (size_t)c * nz + r] = q.p[2][i];
      if (q.winv) out[f.Winv + i] = q.winv[i];
    }
  for (int i = tid; i < half * w; i += nt) {
    const int r = i / w, c = i % w;
    out[f.W1 + i] = q.p[3][i];
    out[f.W1T + (size_t)c * half + r] = q.p[3][i];
  }
  for (int i = tid; i < w * w; i += nt) {
    const int r = i / w, c = i % w;
    out[f.W2 + i] = q.p[6][i];
    out[f.W2T + (size_t)c * w + r] = q.p[6][i];
  }
  for (int i = tid; i < w * n_out; i += nt) {
    const int r = i / n_out, c = i % n_out;
    out[f.W3 + i] = q.p[9][i];
    out[f.W3T + (size_t)c * w + r] = q.p[9][i];
  }
  for (int i = tid; i < w; i += nt) {
    out[f.b1 + i] = q.p[4][i]; out[f.e1 + i] = expf(q.p[5][i] * 3.f);
    out[f.b2 + i] = q.p[7][i]; out[f.e2 + i] = expf(q.p[8][i] * 3.f);
  }
  for (int i = tid; i < n_out; i += nt) {
    out[f.b3 + i] = q.p[10][i]; out[f.e3 + i] = expf(q.p[11][i] * 3.f);
  }
  if (tid == 0) {
    float s = 0.f;
    for (int i = 0; i < nz; ++i) s += q.p[1][i] * 3.f;   // torch.sum(logs * 3), model.py:264-273
    out[f.ld_const] = s;
    out[f.ld_const + 1] = q.log_abs_det ? *q.log_abs_det : 0.f;
  }
}

// ---------------------------------------------------------------------------------------------------
// log|det W| (fp64, model.py:182) and W^-1 (model.py:193) of every step's invertible 1x1 matrix in ONE launch: one CTA
// per matrix, in-place Gauss-Jordan elimination with partial pivoting on an fp64 copy in shared memory; the log-abs
// pivots sum to log|det W|, the result is W^-1 (cast to fp32).  Replaces torch.linalg.det(w.double()) + torch.linalg
// .inv(w) -- two batched LU factorisations, ~1 ms of small kernels per parameter version -- when the caller passes no
// log_abs_det to lsnf_pack_flow_weights.  A singular W yields -inf / non-finite entries, as the reference's
// log(abs(det)) does.
// ---------------------------------------------------------------------------------------------------
constexpr int LINALG_THREADS = 512;
constexpr int LINALG_MAX_N = 160;   // n*n fp64 must fit the 227 KB of shared memory

struct LinalgArgs {
  const float* w[32];
  float* winv;      // [depth][n][n]
  float* logdet;    // [depth]
  int n;
};

__global__ void __launch_bounds__(LINALG_THREADS) flow_logdet_inverse_kernel(LinalgArgs a) {
  extern __shared__ __align__(16) double A[];   // [n][n] row-major
  __shared__ double rowk[LINALG_MAX_N], colk[LINALG_MAX_N];
  __shared__ double red_v[LINALG_THREADS / 32];
  __shared__ int red_i[LINALG_THREADS / 32];
  __shared__ int piv[LINALG_MAX_N];
  __shared__ int s_p;
  const int n = a.n, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* __restrict__ W = a.w[blockIdx.x];
  for (int i = tid; i < n * n; i += LINALG_THREADS) A[i] = (double)W[i];
  __syncthreads();
  double logdet = 0.0;   // meaningful in thread 0
  for (int k = 0; k < n; ++k) {
    // ---- partial pivoting: row of the largest |A[i][k]|, i >= k (ties: smallest i, deterministic) ----
    double bv = -1.0;
    int bi = k;
    for (int i = k + tid; i < n; i += LINALG_THREADS) {
      const double v = fabs(A[i * n + k]);
      if (v > bv) { bv = v; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) { red_v[warp] = bv; red_i[warp] = bi; }
    __syncthreads();
    if (tid == 0) {
      double v = red_v[0];
      int p = red_i[0];
      for (int w2 = 1; w2 < LINALG_THREADS / 32; ++w2)
        if (red_v[w2] > v || (red_v[w2] == v && red_i[w2] < p)) { v = red_v[w2]; p = red_i[w2]; }
      s_p = p; piv[k] = p;
      logdet += log(v);
    }
    __syncthreads();
    const int p = s_p;
    if (p != k)
      for (int j = tid; j < n; j += LINALG_THREADS) {
        const double t = A[k * n + j]; A[k * n + j] = A[p * n + j]; A[p * n + j] = t;
      }
    __syncthreads();
    // ---- new pivot row and the old pivot column ----
    const double pv = A[k * n + k];
    for (int j = tid; j < n; j += LINALG_THREADS) {
      rowk[j] = (j == k ? 1.0 : A[k * n + j]) / pv;
      colk[j] = A[j * n + k];
    }
    __syncthreads();
    // ---- eliminate column k from every other row; row k becomes the scaled pivot row (a warp per row) ----
    for (int i = warp; i < n; i += LINALG_THREADS / 32) {
      double* row = A + i * n;
      if (i == k) {
        for (int j = lane; j < n; j += 32) row[j] = rowk[j];
      } else {
        const double f = colk[i];
        for (int j = lane; j < n; j += 32) row[j] = (j == k ? 0.0 : row[j]) - f * rowk[j];
      }
    }
    __syncthreads();
  }
  // ---- undo the row interchanges: (P W)^-1 = W^-1 P^-1, i.e. swap the columns back in reverse order ----
  for (int k = n - 1; k >= 0; --k) {
    const int p = piv[k];
    if (p != k)
      for (int i = tid; i < n; i += LINALG_THREADS) {
        const double t = A[i * n + k]; A[i * n + k] = A[i * n + p]; A[i * n + p] = t;
      }
    __syncthreads();
  }
  float* out = a.winv + (size_t)blockIdx.x * n * n;
  for (int i = tid; i < n * n; i += LINALG_THREADS) out[i] = (float)A[i];
  if (tid == 0) a.logdet[blockIdx.x] = (float)logdet;
}

int launch_flow_logdet_inverse(const lsnf_plan* plan, const float* const* params, float* winv, float* logdet,
                               cudaStream_t s) {
  const int n = plan->cfg.nz, depth = plan->cfg.f_depth;
  if (n > LINALG_MAX_N || depth > 32) {
    set_error("built-in log|det W| / W^-1 supports nz <= 160: pass log_abs_det and w_inverse to lsnf_pack_flow_weights");
    return LSNF_ERR_UNSUPPORTED;
  }
  LinalgArgs a;
  for (int i = 0; i < depth; ++i) a.w[i] = params[i * LSNF_FLOW_PTRS_PER_STEP + 2];
  a.winv = winv; a.logdet = logdet; a.n = n;
  flow_logdet_inverse_kernel<<<depth, LINALG_THREADS, (size_t)n * n * sizeof(double), s>>>(a);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

int launch_flow_pack(lsnf_plan* plan, const float* const* params, const int32_t* const* perm,
                     const int32_t* const* perm_inv, const float* log_abs_det, const float* const* winv,
                     cudaStream_t s) {
  const FlowLayout& f = plan->fl;
  for (int i = 0; i < plan->cfg.f_depth; ++i) {
    FlowPackPtrs q;
    for (int k = 0; k < LSNF_FLOW_PTRS_PER_STEP; ++k) q.p[k] = params[i * LSNF_FLOW_PTRS_PER_STEP + k];
    q.winv = winv ? winv[i] : nullptr;
    q.perm = perm ? perm[i] : nullptr;
    q.perm_inv = perm_inv ? perm_inv[i] : nullptr;
    q.log_abs_det = plan->cfg.f_permutation == 2 ? log_abs_det + i : nullptr;
    flow_pack_kernel<<<32, 256, 0, s>>>(q, f, (float*)(plan->ws + plan->off_flow) + (size_t)i * f.step_floats,
                                        plan->cfg.f_permutation);
    LSNF_CUDA(cudaGetLastError());
  }
  return LSNF_OK;
}

// preferred samples per CTA: every CTA streams all the parameters (~1.3 MB per pass) through its shared memory, so a
// few samples share one stream; 4 keeps the reference batch of 100 on 25 SMs for ~20 us.  Where that tier's shared
// memory does not fit, the launchers take the next smaller one (fitting_s)
static int pick_s(int B) {
  if (B <= 32) return 1;
  if (B <= 64) return 2;
  if (B <= 1200) return 4;
  return 8;
}

// shared-memory floats besides the matrix ring
static size_t flow_fixed_floats(const FlowLayout& f, int S, int depth, bool stash) {
  const int nmax = std::max(f.nz, std::max(f.w, f.n_out));
  const int nr_max = (nmax + 31) & ~31;
  size_t n = 2 * (FEED_SLOTS + 2) + 2 * FEED_SLOTS + 2 * FEED_MAX_ITEMS + 2 * f.vec_floats +   // mbarriers, ring bookkeeping, item table, vector blocks
             (size_t)S * f.nz + 2 * (size_t)S * nmax + (size_t)S * std::max(FLOW_THREADS, nr_max) +
             (size_t)(FLOW_THREADS / 32) * S;
  if (stash) n += (size_t)depth * S * (2 * f.w + f.nz);
  return n;
}

// ring size: everything one pass streams if it fits, else whatever the 227 KB budget leaves (>= the largest matrix)
int flow_smem(const FlowLayout& f, int S, int depth, bool stash, bool both_passes, uint32_t* ring_floats,
              size_t* smem_bytes) {
  const size_t budget = (size_t)FLOW_SMEM_BYTES / 4;
  const size_t fixed = flow_fixed_floats(f, S, depth, stash);
  if (fixed + f.max_mat > budget) return -1;
  const size_t want = f.step_mat * depth * (both_passes ? 2 : 1);
  size_t r = std::min(budget - fixed, want + 4);
  r = std::max(r, f.max_mat) / 4 * 4;
  *ring_floats = (uint32_t)r;
  *smem_bytes = (fixed + r) * 4;
  return 0;
}

// the largest samples-per-CTA tier <= pick_s(B) whose footprint fits (0: none, not even S = 1)
static int fitting_s(const FlowArgs& a, bool stash, bool both_passes, uint32_t* ring_floats, size_t* smem_bytes) {
  for (int S = pick_s(a.B); S >= 1; S /= 2)
    if (flow_smem(a.fl, S, a.depth, stash, both_passes, ring_floats, smem_bytes) == 0) return S;
  set_error("flow kernel shared memory budget exceeded");
  return 0;
}

template <int S>
static int launch_fwd_t(const FlowArgs& a, size_t smem, cudaStream_t s) {
  if (a.stash)
    flow_forward_kernel<S, true><<<(a.B + S - 1) / S, FLOW_THREADS, smem, s>>>(a);
  else
    flow_forward_kernel<S, false><<<(a.B + S - 1) / S, FLOW_THREADS, smem, s>>>(a);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}
template <int S>
static int launch_inv_t(const FlowArgs& a, size_t smem, cudaStream_t s) {
  flow_inverse_kernel<S><<<(a.B + S - 1) / S, FLOW_THREADS, smem, s>>>(a);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

static int launch_flow_fwd_args(FlowArgs& a, cudaStream_t s) {
  size_t smem;
  const int S = fitting_s(a, true, a.grad != nullptr, &a.ring_floats, &smem);
  switch (S) {
    case 0: return LSNF_ERR_INVALID;
    case 1: return launch_fwd_t<1>(a, smem, s);
    case 2: return launch_fwd_t<2>(a, smem, s);
    case 4: return launch_fwd_t<4>(a, smem, s);
    default: return launch_fwd_t<8>(a, smem, s);
  }
}

// opt-in shared-memory limit of every instantiation, once per device (lsnf_plan_bind)
int flow_prepare_device(int device) {
  static std::mutex mu;
  static bool done[64] = {false};
  std::lock_guard<std::mutex> lock(mu);
  if (device < 0 || device >= 64) { set_error("device index out of range"); return LSNF_ERR_INVALID; }
  if (done[device]) return LSNF_OK;
  const int lim = 227 * 1024;
  LSNF_CUDA(cudaFuncSetAttribute(flow_forward_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  LSNF_CUDA(cudaFuncSetAttribute(flow_forward_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  LSNF_CUDA(cudaFuncSetAttribute(flow_forward_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  LSNF_CUDA(cudaFuncSetAttribute(flow_forward_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  LSNF_CUDA(cudaFuncSetAttribute(flow_forward_kernel<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  LSNF_CUDA(cudaFuncSetAttribute(flow_forward_kernel<4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  LSNF_CUDA(cudaFuncSetAttribute(flow_forward_kernel<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  LSNF_CUDA(cudaFuncSetAttribute(flow_forward_kernel<8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  LSNF_CUDA(cudaFuncSetAttribute(flow_inverse_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  LSNF_CUDA(cudaFuncSetAttribute(flow_inverse_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  LSNF_CUDA(cudaFuncSetAttribute(flow_inverse_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  LSNF_CUDA(cudaFuncSetAttribute(flow_inverse_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  LSNF_CUDA(cudaFuncSetAttribute(flow_logdet_inverse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 LINALG_MAX_N * LINALG_MAX_N * (int)sizeof(double)));
  done[device] = true;
  return LSNF_OK;
}

int launch_flow_forward(const lsnf_plan* plan, const float* z, float* z_out, float* logdet, float* logp,
                        float* grad_z, cudaStream_t s) {
  FlowArgs a;
  a.params = (const float*)(plan->ws + plan->off_flow);
  a.fl = plan->fl; a.depth = plan->cfg.f_depth; a.B = plan->cfg.batch;
  a.coupling = plan->cfg.f_coupling; a.permutation = plan->cfg.f_permutation;
  a.in = z; a.z_out = z_out; a.logdet = logdet; a.logp = logp; a.grad = grad_z;
  a.stash = nullptr;
  a.seed_g = a.seed_ld = nullptr;
  return launch_flow_fwd_args(a, s);
}

// ---------------------------------------------------------------------------------------------------
// flow parameter gradients (train.py:403-411): loss_f = -(1 / B_global) sum_b ll_b.  After the TRAIN instantiation
// of the fused kernel has left the per-sample vectors in the stash, every parameter gradient is a reduction over
// the batch: matrices dM[k][n] = sum_b X[b][k] G[b][n], vectors = column sums.
//   d invertible_1x1_conv.w = y^T g_u - B_local * W^-T     (d log|det W| / dW = W^-T, model.py:182)
//   d actnorm.b = colsum(g_x),  d actnorm.logs = colsum(gl0) - 3 B_local   (logdet += sum 3 logs, model.py:273-276)
// (with the caller's dL/dlogdet seeds of lsnf_flow_vjp, -B_local becomes sum_b seed_ld[b], summed in a fixed order)
//   d fc_k.w = in_k^T g_pk,  d fc_k.actnorm.b = colsum(g_pk),  d fc_k.actnorm.logs = colsum(gl_k)   (k = 1, 2)
//   d fc_zeros.w = a2^T g_p3,  d fc_zeros.b = colsum(g_p3),  d fc_zeros.logs = colsum(gl3)
// all multiplied by 1 / B_global.  Summation over the batch is in a fixed order: deterministic.
// Grid: (row blocks of the four matrices + 4 vector CTAs + 1 loss CTA, f_depth).
// ---------------------------------------------------------------------------------------------------
constexpr int PG_ROWS = 8;   // matrix rows per CTA

struct ParamGradArgs {
  const float* stash;
  const float* params;   // packed flow parameters (W^-1 of every step)
  const float* logp;     // [B]
  float* grads;          // flat, FlowGradLayout per step
  float* loss;           // -(1 / B_global) sum_b logp_b
  int seeded;            // lsnf_flow_vjp: the log-det coefficients come from seed_ld (nullable = 0)
  const float* seed_ld;  // [B]
  FlowLayout fl;
  FlowStash sl;
  FlowGradLayout gl;
  int B, permutation, blocks_w, blocks_w1, blocks_w2, blocks_w3;
  float inv_bg;
};

__device__ __forceinline__ void pg_matrix(const float* X, int K, const float* G, int N, int B, int k0, float scale,
                                          float* out, const float* winv, int nz, float winv_coef) {
  // rows [k0, k0 + PG_ROWS) of out[K][N] = scale * (sum_b X[b][k] G[b][n] + winv_coef * Winv[n][k])
  const int rows = min(PG_ROWS, K - k0);
  for (int o = threadIdx.x; o < rows * N; o += blockDim.x) {
    const int k = k0 + o / N, n = o % N;
    float acc = 0.f;
#pragma unroll 4
    for (int b = 0; b < B; ++b) acc = fmaf(__ldg(X + (size_t)b * K + k), __ldg(G + (size_t)b * N + n), acc);
    if (winv) acc += winv_coef * winv[(size_t)n * nz + k];
    out[(size_t)k * N + n] = acc * scale;
  }
}

__device__ __forceinline__ void pg_colsum(const float* V, int N, int B, float scale, float add, float* out) {
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc += __ldg(V + (size_t)b * N + n);
    out[n] = (acc + add) * scale;
  }
}

// sum of v[0..n) over the CTA in a fixed order (strided partial sums, then a tree): deterministic; every thread gets it
__device__ __forceinline__ float fixed_order_sum(const float* v, int n) {
  __shared__ float red[256];
  float acc = 0.f;
  for (int b = threadIdx.x; b < n; b += blockDim.x) acc += v[b];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  const float r = red[0];
  __syncthreads();
  return r;
}

// d loss / d logdet summed over the batch: -B for -sum_b ll_b, or sum_b seed_ld[b]
__device__ __forceinline__ float logdet_coef(const ParamGradArgs& a) {
  if (!a.seeded) return -(float)a.B;
  return a.seed_ld ? fixed_order_sum(a.seed_ld, a.B) : 0.f;
}

__global__ void __launch_bounds__(256) flow_param_grad_kernel(ParamGradArgs a) {
  const int L = blockIdx.y;
  const FlowLayout& f = a.fl;
  const int nz = f.nz, w = f.w, half = f.half, n_out = f.n_out, B = a.B;
  const float* st = a.stash + (size_t)L * a.sl.layer_floats * B;
  auto slot = [&](size_t off) { return st + off * B; };
  float* g = a.grads + (size_t)L * a.gl.step_floats;
  int blk = blockIdx.x;
  if (blk < a.blocks_w) {
    if (a.permutation == 2)
      pg_matrix(slot(a.sl.y), nz, slot(a.sl.gu), nz, B, blk * PG_ROWS, a.inv_bg, g + a.gl.off[2],
                a.params + (size_t)L * f.step_floats + f.Winv, nz, logdet_coef(a));
    return;
  }
  blk -= a.blocks_w;
  if (blk < a.blocks_w1) {
    pg_matrix(slot(a.sl.u1), half, slot(a.sl.gp1), w, B, blk * PG_ROWS, a.inv_bg, g + a.gl.off[3], nullptr, 0, 0.f);
    return;
  }
  blk -= a.blocks_w1;
  if (blk < a.blocks_w2) {
    pg_matrix(slot(a.sl.a1), w, slot(a.sl.gp2), w, B, blk * PG_ROWS, a.inv_bg, g + a.gl.off[6], nullptr, 0, 0.f);
    return;
  }
  blk -= a.blocks_w2;
  if (blk < a.blocks_w3) {
    pg_matrix(slot(a.sl.a2), w, slot(a.sl.gp3), n_out, B, blk * PG_ROWS, a.inv_bg, g + a.gl.off[9], nullptr, 0, 0.f);
    return;
  }
  blk -= a.blocks_w3;
  if (blk == 0) {
    pg_colsum(slot(a.sl.gx), nz, B, a.inv_bg, 0.f, g + a.gl.off[0]);
    pg_colsum(slot(a.sl.gl0), nz, B, a.inv_bg, 3.f * logdet_coef(a), g + a.gl.off[1]);
  } else if (blk == 1) {
    pg_colsum(slot(a.sl.gp1), w, B, a.inv_bg, 0.f, g + a.gl.off[4]);
    pg_colsum(slot(a.sl.gl1), w, B, a.inv_bg, 0.f, g + a.gl.off[5]);
  } else if (blk == 2) {
    pg_colsum(slot(a.sl.gp2), w, B, a.inv_bg, 0.f, g + a.gl.off[7]);
    pg_colsum(slot(a.sl.gl2), w, B, a.inv_bg, 0.f, g + a.gl.off[8]);
  } else if (blk == 3) {
    pg_colsum(slot(a.sl.gp3), n_out, B, a.inv_bg, 0.f, g + a.gl.off[10]);
    pg_colsum(slot(a.sl.gl3), n_out, B, a.inv_bg, 0.f, g + a.gl.off[11]);
  } else if (L == 0 && a.loss) {
    // loss_f = -mean_b ll_b over the global batch (this rank's partial sum), fixed-order tree
    const float sum = fixed_order_sum(a.logp, B);
    if (threadIdx.x == 0) *a.loss = -sum * a.inv_bg;
  }
}

// the TRAIN instantiation of the fused kernel (stash written), then the parameter-gradient reductions
static int flow_grads(const lsnf_plan* plan, const float* z, const float* seed_g, const float* seed_ld, float* grad_z,
                      float inv_global_batch, float* grads, float* loss, cudaStream_t s) {
  FlowArgs a;
  a.params = (const float*)(plan->ws + plan->off_flow);
  a.fl = plan->fl; a.depth = plan->cfg.f_depth; a.B = plan->cfg.batch;
  a.coupling = plan->cfg.f_coupling; a.permutation = plan->cfg.f_permutation;
  float* fo = (float*)(plan->ws + plan->off_flow_out);   // z_out [B][nz], logdet [B], logp [B]
  a.in = z; a.z_out = nullptr; a.logdet = nullptr; a.logp = fo + (size_t)a.B * a.fl.nz + a.B;
  // the kernel's backward needs a destination even when the caller does not want dL/dz
  a.grad = grad_z ? grad_z : (float*)(plan->ws + plan->off_gradf);
  a.stash = (float*)(plan->ws + plan->off_fstash);
  a.sl = plan->fstash;
  a.seed_g = seed_g; a.seed_ld = seed_ld;
  int rc = launch_flow_fwd_args(a, s);
  if (rc) return rc;
  ParamGradArgs p;
  p.stash = a.stash; p.params = a.params; p.logp = a.logp; p.grads = grads; p.loss = loss;
  p.seeded = (seed_g || seed_ld) ? 1 : 0; p.seed_ld = seed_ld;
  p.fl = plan->fl; p.sl = plan->fstash; p.gl = plan->fgrad;
  p.B = a.B; p.permutation = a.permutation; p.inv_bg = inv_global_batch;
  p.blocks_w = (a.fl.nz + PG_ROWS - 1) / PG_ROWS;
  p.blocks_w1 = (a.fl.half + PG_ROWS - 1) / PG_ROWS;
  p.blocks_w2 = (a.fl.w + PG_ROWS - 1) / PG_ROWS;
  p.blocks_w3 = (a.fl.w + PG_ROWS - 1) / PG_ROWS;
  dim3 grid(p.blocks_w + p.blocks_w1 + p.blocks_w2 + p.blocks_w3 + 5, a.depth);
  flow_param_grad_kernel<<<grid, 256, 0, s>>>(p);
  LSNF_CUDA(cudaGetLastError());
  return LSNF_OK;
}

int launch_flow_param_grads(const lsnf_plan* plan, const float* z, float inv_global_batch, float* grads, float* loss,
                            cudaStream_t s) {
  return flow_grads(plan, z, nullptr, nullptr, nullptr, inv_global_batch, grads, loss, s);
}

int launch_flow_vjp(const lsnf_plan* plan, const float* z, const float* seed_g, const float* seed_ld, float* grad_z,
                    float* grads, cudaStream_t s) {
  if (grads) return flow_grads(plan, z, seed_g, seed_ld, grad_z, 1.f, grads, nullptr, s);
  FlowArgs a;
  a.params = (const float*)(plan->ws + plan->off_flow);
  a.fl = plan->fl; a.depth = plan->cfg.f_depth; a.B = plan->cfg.batch;
  a.coupling = plan->cfg.f_coupling; a.permutation = plan->cfg.f_permutation;
  a.in = z; a.z_out = nullptr; a.logdet = nullptr; a.logp = nullptr; a.grad = grad_z;
  a.stash = nullptr;
  a.seed_g = seed_g; a.seed_ld = seed_ld;
  return launch_flow_fwd_args(a, s);
}

int launch_flow_inverse(const lsnf_plan* plan, const float* eps, float* z, float* negobj, cudaStream_t s) {
  FlowArgs a;
  a.params = (const float*)(plan->ws + plan->off_flow);
  a.fl = plan->fl; a.depth = plan->cfg.f_depth; a.B = plan->cfg.batch;
  a.coupling = plan->cfg.f_coupling; a.permutation = plan->cfg.f_permutation;
  a.in = eps; a.z_out = z; a.logdet = negobj; a.logp = nullptr; a.grad = nullptr; a.stash = nullptr;
  a.seed_g = a.seed_ld = nullptr;
  size_t smem;
  const int S = fitting_s(a, false, false, &a.ring_floats, &smem);
  switch (S) {
    case 0: return LSNF_ERR_INVALID;
    case 1: return launch_inv_t<1>(a, smem, s);
    case 2: return launch_inv_t<2>(a, smem, s);
    case 4: return launch_inv_t<4>(a, smem, s);
    default: return launch_inv_t<8>(a, smem, s);
  }
}

}  // namespace lsnf
