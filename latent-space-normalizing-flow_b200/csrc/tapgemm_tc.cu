// tcgen05 / TMEM / TMA tap-GEMM for sm_100a: the generator's transposed convolutions (forward, train.py:312)
// and their data gradients (train.py:314) as implicit GEMMs.
//
//   D[row, n] = sum_{tap} sum_{k} A[plane_tap][b][m + dy_tap][n + dx_tap][k] * W[brow_tap + n][k]
//
// * A rows are 128 grid positions (b, m, n) fetched by ONE 5-D TMA box per tap and K block; the (dy, dx) shift
//   moves the box, and TMA's out-of-bounds zero fill supplies the convolution padding and the ragged batch.
// * Operands are 16-bit hi|lo pairs (value = hi + lo; fp16 for the forward pass, bf16 for 3-pass data gradients); each
//   K step issues three tcgen05.mma (lo*hi, hi*lo, hi*hi) into one fp32 TMEM accumulator -- the 3-pass split that
//   keeps z_T within the 1e-4 parity budget.  Single-pass stages (passes == 1: the data gradient of noisy chains)
//   load and multiply the hi halves only.  The wide 3-pass data-gradient stages (cross8, tc_cross_fp8) instead hold an
//   fp16 hi half and, in the lo half's bytes, the two cross terms as e4m3 along K: per K block one kind::f16 pass on
//   the hi halves and one kind::f8f6f4 pass (twice the 16-bit rate) over the 128-element e4m3 row.
// * Warp roles: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..9 = epilogue
//   (tcgen05.ld -> bias / LeakyReLU / LeakyReLU' from bit-packed signs -> 16-bit hi|lo through TMA tensor stores,
//   or fp32 rows).  Two kernels: tapgemm_tc_kernel<BN> (one CTA per tile, ring sized per launch) and
//   tapgemm_tc2_kernel<DEEP> (persistent cta_group::2 pairs for the 256-wide stages).  tc_plan_launch picks the
//   kernel, grid, ring and epilogue of each stage; lsnf_plan_bind stores that record and launch_tapgemm_tc launches
//   from it, and lsnf_plan_stage_launch_info reports it.
#include <algorithm>
#include <mutex>
#include <type_traits>

#include "tapgemm_common.cuh"

namespace lsnf {

constexpr int TC_EPI_WARPS = 8;                       // two warps per TMEM lane quarter, each owning half the columns
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS;
constexpr int A_TILE_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KiB per hi or lo half
// L2 eviction-priority hints (the encodings createpolicy.fractional.L2::evict_{first,last} produce for fraction 1.0)
constexpr uint64_t L2_EVICT_FIRST = 0x12F0000000000000ull;
constexpr uint64_t L2_EVICT_LAST = 0x14F0000000000000ull;

// The 1-CTA kernel's operand ring is sized per launch (ring_geometry below): a stage holds the hi halves of the A and
// B tiles, plus the lo halves for a 3-pass stage; short K loops get shallow rings so that several CTAs share an SM
// and one CTA's prologue / epilogue overlaps another's loads.
constexpr int TC_MAX_STAGES = 8;
constexpr int TC_SMEM_EXTRA = 1024 /*alignment slack*/ + 256 /*barriers*/;
constexpr int TC_SMEM_MAX = 232448;   // 227 KiB
template <int BN>
struct TcCfg {
  static constexpr int B_TILE_BYTES = BN * BLOCK_K * 2;
  static constexpr int SPAN = BN >= 64 ? BN / 2 : BN;   // columns per epilogue warp
  static constexpr int TMEM_COLS = BN < 32 ? 32 : BN;
  static constexpr bool TMA_EPI = BN >= 128;            // hi|lo outputs may leave through tensor stores
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
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
// One lane of a converged warp.  The producer and MMA warps run their loops with ALL lanes (so addresses,
// descriptors and coordinates stay warp-uniform and live in uniform registers) and only issue under this predicate;
// issuing from inside an `if (lane == 0)` region makes every operand thread-varying and costs an
// elect / R2UR.BROADCAST loop around each UTMALDG / UTCHMMA.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred P;\n"
      "elect.sync _|P, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, P;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

// K-major, 128-byte swizzled operand tile: rows of 128 B, 8-row groups 1024 B apart (SBO), descriptor version 1
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;             // leading byte offset (unused for swizzled K-major), encoded 16 B
  d |= (uint64_t)(1024 >> 4) << 32;   // stride byte offset between 8-row groups
  d |= (uint64_t)1 << 46;             // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;             // SWIZZLE_128B
  return d;
}

template <int BN>
__device__ __forceinline__ uint32_t umma_idesc(bool fp16) {
  // c_format F32 (bits 4-5 = 1), a/b format (bits 7-9, 10-12): 0 = F16, 1 = BF16; K-major A and B;
  // N>>3 at bit 17, M>>4 at bit 24
  const uint32_t fmt = fp16 ? 0u : 1u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}

__device__ __forceinline__ void epi_bar_sync() {   // the 8 epilogue warps only
  asm volatile("bar.sync 1, %0;" ::"n"(32 * TC_EPI_WARPS) : "memory");
}

// max |value| of a warp's gradient outputs into the consumer's amax word (non-negative floats order like their bits)
__device__ __forceinline__ void warp_amax(uint32_t* word, float m, int lane) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) atomicMax(word, __float_as_uint(m));
}

// element i of a small register array without dynamic indexing (which would push the array to local memory)
template <int N>
__device__ __forceinline__ uint32_t pick_word(const uint32_t (&a)[N], int i) {
  uint32_t r = a[0];
#pragma unroll
  for (int k = 1; k < N; ++k) r = (i == k) ? a[k] : r;
  return r;
}

// The column loops of the epilogues are deliberately NOT unrolled: unrolled they made the CTA-pair kernel 240 KB of
// SASS, far beyond the instruction cache, and the producer / MMA loops kept missing in it.
// Epilogue of one 128-row accumulator tile.  Warp w may touch TMEM lanes [32*(w%4), 32*(w%4)+32); warps w and w+4
// split the columns.  Row-invariant addressing is hoisted out of the column loop, and the saved-activation signs a
// data-gradient row needs are fetched BEFORE waiting for the accumulator, i.e. while the main loop still runs.
// Reference semantics: bias + LeakyReLU of model.py:56-151; LeakyReLU' for the data gradient (train.py:314).
// Stream-K (CTA-pair kernel): `sk_mode` 1 = this CTA computed only the head of the tile's K range: the raw fp32
// accumulator goes to this CTA's slot and the warp's flag is raised; 2 = this CTA computed the tail: the partials
// of the CTAs [sk_first, sk_self) are added before the normal epilogue.  Flags are per (CTA, epilogue warp) -- the
// warps of the two CTAs own the same rows and columns -- and are reset by their single consumer, so they are 0
// again at the next launch (CUDA-graph replays included).
template <int BN>
__device__ __forceinline__ void tc_epilogue(const StageDev& st, int mtile, int n0, int phase, int split, int warp,
                                            int lane, uint32_t tmem_acc, uint32_t full_bar, uint32_t parity,
                                            bool have_acc, int sk_mode = 0, int sk_self = 0, int sk_first = 0,
                                            int sk_stride = 2) {
  using Cfg = TcCfg<BN>;
  const int quarter = warp & 3;
  const int half = (warp - 2) >> 2;
  const int r = quarter * 32 + lane;
  const RowCtx rc = tile_row(st, mtile, r);
  constexpr int SPAN = Cfg::SPAN;
  constexpr int CH = SPAN >= 32 ? 32 : 16;
  const int c_begin = half * SPAN;
  const bool active = c_begin < BN;
  const int col0 = n0 + c_begin;
  const int epi = st.epi;
  const bool ok = active && rc.valid && col0 < st.n_pad;
  const int lo_off = st.oC;
  const float leak = st.leak;
  const bool out16 = st.out_fp16 != 0;
  uint16_t* o16 = nullptr;
  float* o32 = nullptr;
  const float* bias = nullptr;
  constexpr int NW = (SPAN + 31) / 32;
  uint32_t mb[NW];            // LeakyReLU sign bits of this thread's columns (data gradient)
  uint32_t* obits = nullptr;  // where the sign bits of this thread's outputs go (forward)
  if (ok) {
    if (epi == EPI_ACT_HL) {
      const int pos = col0 / st.oC, cb = col0 % st.oC;
      const int mo = rc.m * st.ms + st.ph[phase].mo, no = rc.n * st.ms + st.ph[phase].no;
      const size_t off = (size_t)rc.b * st.sB + (size_t)mo * st.sH + (size_t)no * st.sW + (size_t)pos * st.sPos;
      o16 = (uint16_t*)st.out + off + cb;
      obits = act_bits_word(st, off, cb);
      bias = st.bias + cb;
    } else if (epi == EPI_GRAD_HL) {
      size_t off;
      if (st.split)
        off = (size_t)((rc.m & 1) * 2 + (rc.n & 1)) * st.sP + (size_t)rc.b * st.sB + (size_t)(rc.m >> 1) * st.sH +
              (size_t)(rc.n >> 1) * st.sW;
      else
        off = (size_t)rc.b * st.sB + (size_t)rc.m * st.sH + (size_t)rc.n * st.sW;
      o16 = (uint16_t*)st.out + off + col0;
      const uint32_t* mp = grad_bits_row(st, rc) + (col0 >> 5);
#pragma unroll
      for (int j = 0; j < NW; ++j) mb[j] = __ldg(mp + j);
    } else {
      const size_t row = ((size_t)rc.b * st.Hg + rc.m) * st.Wg + rc.n;
      o32 = (float*)st.out + ((size_t)split * st.rows_total + row) * st.n_pad + col0;
    }
  }
  const float descale = st.descale ? __ldg(st.descale) : 1.f;
  if (have_acc) mbar_wait(full_bar, parity);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  if (!active) return;
  const int ewarp = warp - 2;
  if (sk_mode == 1) {
    // helper: raw accumulator -> slot[sk_self], stored COLUMN-major ([256 columns][128 rows]) so that the 32 lanes
    // of a warp (32 consecutive rows) write 128 contiguous bytes per column; then raise this warp's flag
    float* slot = st.sk_slots + ((size_t)sk_self * 256 + c_begin) * BLOCK_M + r;
#pragma unroll 1
    for (int cc = 0; cc < SPAN; cc += CH) {
      uint32_t v[CH];
      const uint32_t taddr = tmem_acc + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(c_begin + cc);
      if constexpr (CH == 32) tmem_ld32(taddr, v); else tmem_ld16(taddr, v);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int j = 0; j < CH; ++j) slot[(size_t)(cc + j) * BLOCK_M] = __uint_as_float(v[j]);
    }
    __threadfence();
    __syncwarp();
    if (lane == 0) {
      volatile int32_t* flag = st.sk_flags + sk_self * TC_EPI_WARPS + ewarp;
      asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(flag), "r"(1) : "memory");
    }
    return;
  }
  if (sk_mode == 2) {
    // finisher: wait until every helper CTA of this tile has published this warp's part
    if (lane == 0) {
      for (int h = sk_first; h < sk_self; h += sk_stride) {
        const int32_t* flag = st.sk_flags + h * TC_EPI_WARPS + ewarp;
        int32_t f;
        do {
          asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(f) : "l"(flag) : "memory");
        } while (f == 0);
      }
    }
    __syncwarp();
    __threadfence();
  }
  float amax = 0.f;
#pragma unroll 1
  for (int cc = 0; cc < SPAN; cc += CH) {
    uint32_t v[CH];
    const uint32_t taddr = tmem_acc + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(c_begin + cc);
    if constexpr (CH == 32) tmem_ld32(taddr, v); else tmem_ld16(taddr, v);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    const uint32_t mword = pick_word(mb, cc >> 5);
    if (sk_mode == 2) {
      for (int h = sk_first; h < sk_self; h += sk_stride) {
        const float* slot = st.sk_slots + ((size_t)h * 256 + c_begin + cc) * BLOCK_M + r;
#pragma unroll
        for (int j = 0; j < CH; ++j)
          v[j] = __float_as_uint(__uint_as_float(v[j]) + __ldcg(slot + (size_t)j * BLOCK_M));
      }
    }
    if (!ok) continue;
    uint32_t signs = 0u;
#pragma unroll
    for (int j = 0; j < CH; j += 8) {
      float f[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) f[q] = have_acc ? __uint_as_float(v[j + q]) * descale : 0.f;
      if (epi == EPI_ACT_HL) {
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + cc + j));
        const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + cc + j + 4));
        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        __align__(16) uint16_t hi[8], lo[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          float t = f[q] + bb[q];
          t = t > 0.f ? t : t * leak;
          split16(t, out16, hi[q], lo[q]);
          signs |= (uint32_t)(hi[q] >> 15) << ((j + q) & 31);
        }
        *reinterpret_cast<uint4*>(o16 + cc + j) = *reinterpret_cast<uint4*>(hi);
        *reinterpret_cast<uint4*>(o16 + lo_off + cc + j) = *reinterpret_cast<uint4*>(lo);
      } else if (epi == EPI_GRAD_HL) {
        const uint32_t mw = mword >> ((cc + j) & 31);
        __align__(16) uint16_t hi[8], lo[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float t = ((mw >> q) & 1u) ? f[q] * leak : f[q];   // sign of the saved activation
          amax = fmaxf(amax, fabsf(t));
          split16(t, out16, hi[q], lo[q]);
        }
        *reinterpret_cast<uint4*>(o16 + cc + j) = *reinterpret_cast<uint4*>(hi);
        if (!st.out_single) *reinterpret_cast<uint4*>(o16 + lo_off + cc + j) = *reinterpret_cast<uint4*>(lo);
      } else {
        *reinterpret_cast<float4*>(o32 + cc + j) = make_float4(f[0], f[1], f[2], f[3]);
        *reinterpret_cast<float4*>(o32 + cc + j + 4) = make_float4(f[4], f[5], f[6], f[7]);
      }
    }
    if constexpr (CH == 32) {
      if (epi == EPI_ACT_HL) obits[cc >> 5] = signs;   // hidden widths are multiples of 64: whole words
    }
  }
  if (epi == EPI_GRAD_HL && st.amax_out) warp_amax(st.amax_out, amax, lane);
  if (sk_mode == 2) {
    __syncwarp();
    if (lane == 0)
      for (int h = sk_first; h < sk_self; h += sk_stride) st.sk_flags[h * TC_EPI_WARPS + ewarp] = 0;
  }
}

template <int BN, bool SINGLE>
__device__ __forceinline__ void tc_epilogue_tma(const StageDev& st, const CUtensorMap* tmO, uint32_t stage_smem,
                                                int mtile, int n0, int phase, int warp, int lane, uint32_t tmem_acc,
                                                uint32_t full_bar, uint32_t parity, int sk_mode, int sk_self,
                                                int sk_first);

template <int BN>
__global__ void __launch_bounds__(TC_THREADS, 2)
tapgemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ CUtensorMap tmO, const __grid_constant__ StageDev st) {
  using Cfg = TcCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t tiles = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const bool three = st.passes != 1;   // single pass: hi halves only, compact stages
  const uint32_t nst = (uint32_t)st.nst;
  const uint32_t a_bytes = three ? 2 * A_TILE_BYTES : A_TILE_BYTES;
  const uint32_t stage_bytes = a_bytes + (three ? 2 : 1) * Cfg::B_TILE_BYTES;
  const uint32_t bars = tiles + nst * stage_bytes;
  // barrier block: full[MAX], empty[MAX], tmem_full, then the TMEM base address slot
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (TC_MAX_STAGES + s); };
  const uint32_t tmem_full_bar = bars + 8u * (2 * TC_MAX_STAGES);
  const uint32_t tmem_slot = bars + 8u * (2 * TC_MAX_STAGES + 1);
  uint8_t* gen_base = smem_raw + (tiles - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(gen_base + nst * stage_bytes + 8 * (2 * TC_MAX_STAGES + 1));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int mtile = blockIdx.x, n0 = blockIdx.y * BN;
  const int zphase = blockIdx.z / st.ksplit, split = blockIdx.z % st.ksplit;
  const bool wg = st.wgrad != 0;                 // weight gradient: slice zphase is tap zphase of phase 0, alone
  const int phase = wg ? 0 : zphase, tap0 = wg ? zphase : 0;
  const int kblocks = st.Ka / BLOCK_K;
  const int total = (wg ? 1 : st.ph[phase].ntaps) * kblocks;
  const int it0 = split * st.it_per_split, it1 = min(total, it0 + st.it_per_split);

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    if (Cfg::TMA_EPI && st.out_tma) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmO) : "memory");
    for (int s = 0; s < TC_MAX_STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                 "r"((uint32_t)Cfg::TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot_ptr;
  // everything above touched shared / tensor memory only; operands, sign bits and scales are read below
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    {
      // ===== TMA producer =====
      int b0, h0, w0;
      tile_origin(st, mtile, b0, h0, w0);
      uint32_t s = 0, par = 0, sa = tiles;
      int tp = it0 / kblocks, kc = (it0 - tp * kblocks) * BLOCK_K;
      tp += tap0;
      int dy = 0, dx = 0, plane = 0, brow = 0, bcol = 0;
      if (it1 > it0) get_tap(st, phase, tp, dy, dx, plane, brow, bcol);
      for (int it = it0; it < it1; ++it) {
        mbar_wait(empty_bar(s), par ^ 1u);
        const uint32_t sb = sa + a_bytes;
        if (elect_one()) {
          mbar_expect_tx(full_bar(s), stage_bytes);
          tma_load_5d(sa, &tmA, full_bar(s), kc, w0 + dx, h0 + dy, b0, plane);
          if (three) tma_load_5d(sa + A_TILE_BYTES, &tmA, full_bar(s), st.Ka + kc, w0 + dx, h0 + dy, b0, plane);
          tma_load_2d(sb, &tmB, full_bar(s), bcol + kc, brow + n0);
          if (three) tma_load_2d(sb + Cfg::B_TILE_BYTES, &tmB, full_bar(s), st.b_k + bcol + kc, brow + n0);
        }
        kc += BLOCK_K;
        if (kc == st.Ka) {
          kc = 0; ++tp;
          if (it + 1 < it1) get_tap(st, phase, tp, dy, dx, plane, brow, bcol);
        }
        sa += stage_bytes;
        if (++s == nst) { s = 0; par ^= 1u; sa = tiles; }
      }
    }
  } else if (warp == 1) {
    {
      // ===== MMA issuer =====
      const uint32_t idesc = umma_idesc<BN>(st.fp16 != 0);
      uint32_t s = 0, par = 0, sa = tiles;
      for (int it = it0; it < it1; ++it) {
        mbar_wait(full_bar(s), par);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint64_t da = umma_desc(sa), db = umma_desc(sa + a_bytes);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BLOCK_K / 16; ++k) {
            const uint64_t a_hi = da + 2 * k, a_lo = a_hi + (A_TILE_BYTES >> 4);
            const uint64_t b_hi = db + 2 * k, b_lo = b_hi + (Cfg::B_TILE_BYTES >> 4);
            if (three) {
              umma_bf16(tmem_base, a_lo, b_hi, idesc, (it > it0 || k > 0) ? 1u : 0u);
              umma_bf16(tmem_base, a_hi, b_lo, idesc, 1u);
              umma_bf16(tmem_base, a_hi, b_hi, idesc, 1u);
            } else {
              umma_bf16(tmem_base, a_hi, b_hi, idesc, (it > it0 || k > 0) ? 1u : 0u);
            }
          }
          umma_commit(empty_bar(s));  // frees the smem slot once the MMAs above have read it
        }
        sa += stage_bytes;
        if (++s == nst) { s = 0; par ^= 1u; sa = tiles; }
      }
      if (elect_one()) umma_commit(tmem_full_bar);   // accumulator complete (same lane as the MMAs: elect is deterministic)
    }
  } else {
    bool done = false;
    if constexpr (Cfg::TMA_EPI) {
      // hi|lo outputs of a wide tile leave through tensor stores; the operand ring is idle once the accumulator is
      // complete, so its first 32 KiB serve as the staging tile
      if (st.out_tma) {
        if (st.out_single)
          tc_epilogue_tma<BN, true>(st, &tmO, tiles, mtile, n0, phase, warp, lane, tmem_base, tmem_full_bar, 0u, 0, 0, 0);
        else
          tc_epilogue_tma<BN, false>(st, &tmO, tiles, mtile, n0, phase, warp, lane, tmem_base, tmem_full_bar, 0u, 0, 0, 0);
        if (warp == 2 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        done = true;
      }
    }
    // weight-gradient slices land at [tap][split][C_in][C_out]: blockIdx.z IS tap * ksplit + split
    if (!done) tc_epilogue<BN>(st, mtile, n0, phase, wg ? (int)blockIdx.z : split, warp, lane, tmem_base, tmem_full_bar,
                               0u, it1 > it0);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"((uint32_t)Cfg::TMEM_COLS)
                 : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------
// CTA-pair variant (cta_group::2) for the wide stages (N tile 256): two CTAs of one cluster compute a 256 x 256
// output tile.  Each CTA loads its own 128 A rows and HALF of the 256 weight rows, so operand traffic per CTA drops
// from 384 to 256 rows per K block (the 3-pass hi|lo split doubles operand bytes per FLOP and makes the single-CTA
// kernel L2-bound); the leader CTA issues the MMAs for both and commits to the barriers of both.
// ---------------------------------------------------------------------------------------------------
constexpr int P_BN = 256;
constexpr int P_B_TILE_BYTES = (P_BN / 2) * BLOCK_K * 2;                 // this CTA's half of the weight rows
constexpr int P_STAGE_BYTES = 2 * A_TILE_BYTES + 2 * P_B_TILE_BYTES;      // 64 KiB per CTA
constexpr int P_STAGES = 3;                                                // 64 KiB stages (hi and lo halves) ...
constexpr int P_MAX_STAGES = 2 * P_STAGES;                                 // ... or twice as many 32 KiB ones (hi only)
constexpr int P_EPI_STAGING = 2 * BLOCK_M * 128;                           // hi + lo slab of 128 rows x 64 channels
constexpr int P_SMEM_BYTES = P_STAGES * P_STAGE_BYTES + P_EPI_STAGING + 1024 + 256;   // ring + staging + align + barriers
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;                            // clears the CTA-rank bit of a shared::cluster address

__device__ __forceinline__ void tma2_load_5d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                             int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6, %7}], [%2], %8;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "l"(L2_EVICT_LAST)
      : "memory");
}
__device__ __forceinline__ void tma2_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "l"(L2_EVICT_LAST)
      : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma2_f8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma2_commit_both(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"((uint16_t)3)
      : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__device__ __forceinline__ void cluster_sync_relaxed() {
  asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in the LEADER CTA of the pair
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar & PEER_BIT_MASK) : "memory");
}

// Outputs are written once and not re-read by this kernel: evict-first keeps them from displacing the operands,
// which every tap re-reads from L2.
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3,
                                             int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3, %4, %5, %6}], [%1], %7;" ::"l"(map),
      "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "l"(L2_EVICT_FIRST)
      : "memory");
}

// Epilogue of the CTA-pair kernel for the hi|lo outputs, through shared memory and TMA tensor stores.
// Per-thread 16-byte stores of a thread-per-row layout touch 32 different 1 KB-strided rows per instruction; they
// cost the wide stages ~20 % and made the last layer's data gradient store-bound.  Here the 8 warps cooperate on one
// 64-channel slab at a time: warp (quarter, half) converts rows [32*quarter, +32) x channels [32*half, +32) into the
// 128-byte-swizzled staging tile (hi and lo, 16 KiB each), then one thread issues two 5-D tensor stores (the box
// scatters rows to their strided / phase-split positions and clips the ragged batch).
// SINGLE (outputs keep only their hi half: the single-pass data gradient): the two 16 KiB buffers alternate between
// consecutive slabs, so a slab's tensor store drains while the next slab is converted.
__device__ __forceinline__ uint32_t pack2_16(float a, float b, bool fp16) {
  if (fp16) { const __half2 h = __floats2half2_rn(a, b); return *reinterpret_cast<const uint32_t*>(&h); }
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

template <int BN, bool SINGLE>
__device__ __forceinline__ void tc_epilogue_tma(const StageDev& st, const CUtensorMap* tmO, uint32_t stage_smem,
                                                int mtile, int n0, int phase, int warp, int lane, uint32_t tmem_acc,
                                                uint32_t full_bar, uint32_t parity, int sk_mode, int sk_self,
                                                int sk_first) {
  const int quarter = warp & 3;
  const int half = (warp - 2) >> 2;
  const int ewarp = warp - 2;
  const int r = quarter * 32 + lane;
  const RowCtx rc = tile_row(st, mtile, r);
  const int epi = st.epi;
  const float leak = st.leak;
  const bool out16 = st.out_fp16 != 0;
  constexpr int NCH = BN / 64;   // 64-channel slabs per tile
  // saved-activation signs for this thread's 32 channels of every slab (fetched while the main loop runs), or the
  // place where the signs of this thread's outputs go
  uint32_t mb[NCH];
  uint32_t* obits = nullptr;
#pragma unroll
  for (int ch = 0; ch < NCH; ++ch) mb[ch] = 0u;
  if (epi == EPI_GRAD_HL && rc.valid) {
    const uint32_t* mrow = grad_bits_row(st, rc) + (n0 >> 5) + half;
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) mb[ch] = __ldg(mrow + 2 * ch);
  } else if (epi == EPI_ACT_HL && rc.valid) {
    const int pos = n0 / st.oC;
    const int mo = rc.m * st.ms + st.ph[phase].mo, no = rc.n * st.ms + st.ph[phase].no;
    const size_t off = (size_t)rc.b * st.sB + (size_t)mo * st.sH + (size_t)no * st.sW + (size_t)pos * st.sPos;
    obits = act_bits_word(st, off, n0 % st.oC) + half;
  }
  // tensor-store coordinates of this tile
  int b0, h0, w0;
  tile_origin(st, mtile, b0, h0, w0);
  const int cb = n0 % st.oC;
  int c1, c2, c3, c4;
  if (st.out_tma == 1) { c1 = st.ph[phase].no; c2 = w0; c3 = st.ph[phase].mo; c4 = b0 * st.Hg + h0; }
  else if (st.out_tma == 2) { c1 = n0 / st.oC; c2 = 0; c3 = 0; c4 = b0; }
  else if (st.out_tma == 3) { c1 = w0; c2 = h0; c3 = b0; c4 = 0; }
  else { c1 = w0 >> 1; c2 = b0 * (st.Hg >> 1) + (h0 >> 1); c3 = 0; c4 = 0; }
  // staging row of this thread's tile row: identity, except for the phase-split gradient whose box is ordered
  // (py, px, b*H/2 + m/2, n/2) so that the tensor map's strides increase monotonically
  int srow = r;
  if (st.out_tma == 4) {
    const int nl = r % st.bW, ml = (r / st.bW) % st.bH, bl = r / (st.bW * st.bH);
    srow = (((ml & 1) * 2 + (nl & 1)) * (st.bB * (st.bH >> 1)) + bl * (st.bH >> 1) + (ml >> 1)) * (st.bW >> 1) + (nl >> 1);
  }
  const float* bias = (epi == EPI_ACT_HL) ? st.bias + cb + half * 32 : nullptr;
  const float descale = st.descale ? __ldg(st.descale) : 1.f;
  const uint32_t buf0 = stage_smem, buf1 = stage_smem + 128 * 128;

  mbar_wait(full_bar, parity);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  if (sk_mode == 2) {
    if (lane == 0) {
      for (int h = sk_first; h < sk_self; h += 2) {
        const int32_t* flag = st.sk_flags + h * TC_EPI_WARPS + ewarp;
        int32_t f;
        do {
          asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(f) : "l"(flag) : "memory");
        } while (f == 0);
      }
    }
    __syncwarp();
    __threadfence();
  }
  float amax = 0.f;
#pragma unroll 1
  for (int ch = 0; ch < NCH; ++ch) {
    const int col = ch * 64 + half * 32;   // column of the accumulator tile
    uint32_t v[32];
    tmem_ld32(tmem_acc + ((uint32_t)(quarter * 32) << 16) + (uint32_t)col, v);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    if (sk_mode == 2) {
      for (int h = sk_first; h < sk_self; h += 2) {
        // column-major slot: coalesced across the warp's 32 rows
        const float* slot = st.sk_slots + ((size_t)h * 256 + col) * BLOCK_M + r;
#pragma unroll
        for (int j = 0; j < 32; ++j)
          v[j] = __float_as_uint(__uint_as_float(v[j]) + __ldcg(slot + (size_t)j * BLOCK_M));
      }
    }
    // SINGLE: this slab's buffer was last used two slabs ago; at most the previous slab's store may still be
    // reading.  Otherwise the issuing thread already waited for the previous slab's stores before arriving here.
    const uint32_t hi_buf = SINGLE ? ((ch & 1) ? buf1 : buf0) : buf0;
    const uint32_t lo_buf = buf1;
    if (SINGLE && warp == 2 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
    epi_bar_sync();
    uint32_t signs = 0u;
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      float t[8];
      if (epi == EPI_ACT_HL) {
        const float4 q0 = __ldg(reinterpret_cast<const float4*>(bias + ch * 64 + j));
        const float4 q1 = __ldg(reinterpret_cast<const float4*>(bias + ch * 64 + j + 4));
        const float bb[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float a = __uint_as_float(v[j + q]) * descale + bb[q];
          t[q] = a > 0.f ? a : a * leak;
          signs |= (__float_as_uint(t[q]) >> 31) << (j + q);   // rounding to 16 bits keeps the sign
        }
      } else {
        const uint32_t mw = pick_word(mb, ch) >> j;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float a = __uint_as_float(v[j + q]) * descale;
          t[q] = ((mw >> q) & 1u) ? a * leak : a;   // sign of the saved activation
          amax = fmaxf(amax, fabsf(t[q]));
        }
      }
      // row r of the slab is 128 B; the 16-byte chunk index is XORed with (row % 8) -- the 128-byte TMA swizzle
      const uint32_t chunk = (uint32_t)(half * 4 + j / 8) ^ (uint32_t)(srow & 7);
      const uint32_t off = (uint32_t)srow * 128u + chunk * 16u;
      if constexpr (SINGLE) {
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(hi_buf + off), "r"(pack2_16(t[0], t[1], out16)),
                     "r"(pack2_16(t[2], t[3], out16)), "r"(pack2_16(t[4], t[5], out16)),
                     "r"(pack2_16(t[6], t[7], out16))
                     : "memory");
      } else {
        __align__(16) uint16_t hi[8], lo[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) split16(t[q], out16, hi[q], lo[q]);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(hi_buf + off), "r"(((uint32_t*)hi)[0]),
                     "r"(((uint32_t*)hi)[1]), "r"(((uint32_t*)hi)[2]), "r"(((uint32_t*)hi)[3])
                     : "memory");
        if (!st.out_single)
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(lo_buf + off), "r"(((uint32_t*)lo)[0]),
                       "r"(((uint32_t*)lo)[1]), "r"(((uint32_t*)lo)[2]), "r"(((uint32_t*)lo)[3])
                       : "memory");
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    epi_bar_sync();
    if (warp == 2 && lane == 0) {
      const int c0 = cb + ch * 64;
      tma_store_5d(tmO, hi_buf, c0, c1, c2, c3, c4);
      if (!SINGLE && !st.out_single) tma_store_5d(tmO, lo_buf, c0 + st.oC, c1, c2, c3, c4);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      if (!SINGLE) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    if (obits) obits[2 * ch] = signs;   // after the barrier: the store's latency stays off the slab's critical path
  }
  if (epi == EPI_GRAD_HL && st.amax_out) warp_amax(st.amax_out, amax, lane);
  if (sk_mode == 2) {
    __syncwarp();
    if (lane == 0)
      for (int h = sk_first; h < sk_self; h += 2) st.sk_flags[h * TC_EPI_WARPS + ewarp] = 0;
  }
}

// Work list of one CTA pair under stream-K.  The stage's tiles (m-pair fastest, so consecutive tiles share weights
// in L2) times their K blocks form one linear range of units, cut into equal contiguous shares; a share that ends
// inside a tile makes its owner a HELPER for that tile (it publishes a raw partial accumulator), one that starts
// inside a tile a FINISHER (it adds the helpers' partials, then runs the normal epilogue).  The helper item is
// processed FIRST and the finisher item LAST, so nobody ever waits long for a partial.
struct SkItem { int tile, ka, kb, mode; };   // mode 0 full, 1 helper, 2 finisher
struct SkPlan {
  int total, t_lo, t_hi, ka_lo, kb_hi, first_fin, last_help, first_help_only, n_items, full_lo, full_hi;
  long long u0, u1;
  int strided, pair_, npairs_;
  __device__ __forceinline__ void init(int pair, int num_pairs, int num_tiles, int total_, bool stream_k) {
    total = total_;
    strided = !stream_k; pair_ = pair; npairs_ = num_pairs;
    if (strided) {   // whole tiles: pair, pair + P, pair + 2P, ...
      n_items = pair < num_tiles ? (num_tiles - pair + num_pairs - 1) / num_pairs : 0;
      first_fin = last_help = first_help_only = 0;
      return;
    }
    const long long U = (long long)num_tiles * total;
    u0 = U * pair / num_pairs; u1 = U * (pair + 1) / num_pairs;
    n_items = 0; first_fin = last_help = first_help_only = 0; full_lo = 0; full_hi = -1;
    if (u1 <= u0) return;
    t_lo = (int)(u0 / total); t_hi = (int)((u1 - 1) / total);
    ka_lo = (int)(u0 - (long long)t_lo * total);
    kb_hi = (int)(u1 - (long long)t_hi * total);          // in (0, total]
    const bool first_cut = ka_lo != 0, last_cut = kb_hi != total;
    if (t_lo == t_hi) {
      if (last_cut) { last_help = 1; }                     // a share inside one tile that does not reach its end
      else if (first_cut) { first_fin = 1; }
      else { full_lo = full_hi = t_lo; }
    } else {
      last_help = last_cut; first_fin = first_cut;
      full_lo = first_cut ? t_lo + 1 : t_lo;
      full_hi = last_cut ? t_hi - 1 : t_hi;
    }
    n_items = last_help + (full_hi >= full_lo ? full_hi - full_lo + 1 : 0) + first_fin;
  }
  __device__ __forceinline__ SkItem item(int j) const {
    SkItem it;
    if (strided) { it.tile = pair_ + j * npairs_; it.ka = 0; it.kb = total; it.mode = 0; return it; }
    if (last_help) {
      if (j == 0) { it.tile = t_hi; it.ka = (t_lo == t_hi) ? ka_lo : 0; it.kb = kb_hi; it.mode = 1; return it; }
      --j;
    }
    const int nfull = full_hi >= full_lo ? full_hi - full_lo + 1 : 0;
    if (j < nfull) { it.tile = full_lo + j; it.ka = 0; it.kb = total; it.mode = 0; return it; }
    it.tile = t_lo; it.ka = ka_lo; it.kb = total; it.mode = 2;
    return it;
  }
};

// first pair whose share contains unit u (shares are [U*p/P, U*(p+1)/P))
__device__ __forceinline__ int sk_pair_of(long long u, long long U, int P) {
  int p = (int)((u * P) / U);
  while (p > 0 && U * p / P > u) --p;
  while (p + 1 < P && U * (p + 1) / P <= u) ++p;
  return p;
}

// Persistent: one CTA pair per SM pair.  The shared-memory ring keeps streaming across tile boundaries, and the 512
// TMEM columns hold TWO 256-column accumulators so the epilogue of item i overlaps the main loop of item i+1.
// DEEP (single-pass stages: hi halves only) splits the same ring memory into twice as many half-sized stages.  The
// ring geometry is a compile-time constant on purpose: with run-time stage counts / sizes the 3-pass stages measured
// 6 % slower.
template <bool DEEP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
tapgemm_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ CUtensorMap tmO, const __grid_constant__ StageDev st) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t tiles = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t stage_smem = tiles + P_STAGES * P_STAGE_BYTES;   // 32 KiB epilogue staging (hi, lo slabs)
  const uint32_t bars = stage_smem + P_EPI_STAGING;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (P_MAX_STAGES + s); };
  auto tmem_full_bar = [&](int a) { return bars + 8u * (2 * P_MAX_STAGES + a); };
  auto tmem_empty_bar = [&](int a) { return bars + 8u * (2 * P_MAX_STAGES + 2 + a); };
  const uint32_t tmem_slot = bars + 8u * (2 * P_MAX_STAGES + 4);
  uint8_t* gen_base = smem_raw + (tiles - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(
      gen_base + P_STAGES * P_STAGE_BYTES + P_EPI_STAGING + 8 * (2 * P_MAX_STAGES + 4));
  // A single-pass stage loads hi halves only: the same ring memory then holds twice as many, half-sized stages --
  // the bytes in flight, not the stage count, are what hides the L2 latency
  constexpr bool three = !DEEP;
  constexpr uint32_t nst = DEEP ? P_MAX_STAGES : P_STAGES;
  constexpr uint32_t stage_bytes = DEEP ? P_STAGE_BYTES / 2 : P_STAGE_BYTES;
  constexpr uint32_t b_off = DEEP ? A_TILE_BYTES : 2 * A_TILE_BYTES;

  uint32_t cta_rank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(cta_rank));
  const bool leader = cta_rank == 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kblocks = st.Ka / BLOCK_K;
  // tile list: t = (phase * n_tiles + ntile) * m_pairs + mpair
  const int mtiles = st.tiles_b * st.tiles_h * st.tiles_w;
  const int m_pairs = (mtiles + 1) >> 1, n_tiles = st.n_pad / P_BN;
  const int num_tiles = m_pairs * n_tiles * st.nphase;
  const int pair_id = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int total = st.ph[0].ntaps * kblocks;   // identical for every phase of a stage (checked on the host)
  SkPlan sk;
  sk.init(pair_id, num_pairs, num_tiles, total, st.sk_enable != 0);

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    if (st.out_tma) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmO) : "memory");
    for (int s = 0; s < P_MAX_STAGES; ++s) {
      mbar_init(full_bar(s), 1);    // leader's producer arrives once per use (+ the bytes of both CTAs)
      mbar_init(empty_bar(s), 1);   // one multicast commit per use
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tmem_full_bar(a), 1);                     // multicast commit of the item's last MMA
      mbar_init(tmem_empty_bar(a), 2 * TC_EPI_WARPS);     // every epilogue warp of both CTAs (leader's copy is used)
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();   // the peer's barriers are initialised before anything can arrive on them
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_wait();      // see lsnf_internal.cuh: the set-up above overlaps the tail of the previous kernel
  pdl_trigger();
  // the conversion that read this stage's input amax is complete: zero the word for the next producer
  if (st.amax_reset && blockIdx.x == 0 && threadIdx.x == 0) *st.amax_reset = 0u;

  if (warp == 0) {
    {
      // ===== TMA producer (both CTAs); completions of both land on the LEADER's full barrier =====
      // Nothing but the barrier wait and the copies sits between a slot becoming free and its refill: the ring is
      // only as deep as shared memory allows, so every cycle spent here shows up as an idle tensor pipe.
      uint32_t s = 0, par = 0, sa = tiles;   // ring slot, its use parity and address: no drain between items
      constexpr uint32_t tx_bytes = three ? 2 * P_STAGE_BYTES : P_STAGE_BYTES;   // both CTAs' bytes land on the leader
      for (int j = 0; j < sk.n_items; ++j) {
        const SkItem w = sk.item(j);
        const int t = w.tile;
        const int mp = t % m_pairs, nt = (t / m_pairs) % n_tiles, phase = t / (m_pairs * n_tiles);
        const int mtile = 2 * mp + (int)cta_rank;
        int b0, h0, w0;
        tile_origin(st, mtile, b0, h0, w0);
        const int nb = nt * P_BN + (int)cta_rank * (P_BN / 2);
        int tp = w.ka / kblocks, kc = (w.ka - tp * kblocks) * BLOCK_K;
        int dy, dx, plane, brow, bcol;
        get_tap(st, phase, tp, dy, dx, plane, brow, bcol);
        for (int it = w.ka; it < w.kb; ++it) {
          mbar_wait(empty_bar(s), par ^ 1u);
          const uint32_t sb = sa + b_off;
          const uint32_t fb = full_bar(s) & PEER_BIT_MASK;
          if (elect_one()) {
            if (leader) mbar_expect_tx(full_bar(s), tx_bytes);
            tma2_load_5d(sa, &tmA, fb, kc, w0 + dx, h0 + dy, b0, plane);
            if (three) tma2_load_5d(sa + A_TILE_BYTES, &tmA, fb, st.Ka + kc, w0 + dx, h0 + dy, b0, plane);
            tma2_load_2d(sb, &tmB, fb, bcol + kc, brow + nb);
            if (three) tma2_load_2d(sb + P_B_TILE_BYTES, &tmB, fb, st.b_k + bcol + kc, brow + nb);
          }
          kc += BLOCK_K;
          if (kc == st.Ka) {
            kc = 0; ++tp;
            if (it + 1 < w.kb) get_tap(st, phase, tp, dy, dx, plane, brow, bcol);
          }
          sa += stage_bytes;
          if (++s == nst) { s = 0; par ^= 1u; sa = tiles; }
        }
      }
    }
  } else if (warp == 1) {
    if (leader) {
      // ===== MMA issuer (leader CTA only): M = 256 over both CTAs, N = 256 =====
      const bool cross8 = st.cross8 != 0;
      const uint32_t fmt = (st.fp16 || cross8) ? 0u : 1u;   // the hi halves of a cross8 stage are fp16
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(P_BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      // kind::f8f6f4 with E4M3 (format 0) A and B, fp32 accumulator
      const uint32_t idesc8 = (1u << 4) | ((uint32_t)(P_BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      uint32_t s = 0, par = 0, sa = tiles;
      for (int j = 0; j < sk.n_items; ++j) {
        const SkItem w = sk.item(j);
        const uint32_t acc = (uint32_t)j & 1u;
        // the epilogues of both CTAs must have drained this accumulator (two items ago)
        mbar_wait(tmem_empty_bar(acc), (((uint32_t)j >> 1) & 1u) ^ 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t d_tmem = tmem_base + acc * P_BN;
        for (int it = w.ka; it < w.kb; ++it) {
          mbar_wait(full_bar(s), par);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          // descriptors differ only in their 16-byte-unit address field: K step k starts 32 bytes further
          const uint64_t da = umma_desc(sa), db = umma_desc(sa + b_off);
          if (elect_one()) {
            if (three && cross8) {
              // hi*hi on the fp16 halves (K = 16 per MMA), then the e4m3 rows [a_hi8 | a_lo8] . [w_lo8 | w_hi8]
              // (K = 32 per MMA): the same 32-byte descriptor steps cover the 128-byte rows
#pragma unroll
              for (int k = 0; k < BLOCK_K / 16; ++k)
                umma2_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (it > w.ka || k > 0) ? 1u : 0u);
#pragma unroll
              for (int k = 0; k < BLOCK_K / 16; ++k)
                umma2_f8(d_tmem, da + (A_TILE_BYTES >> 4) + 2 * k, db + (P_B_TILE_BYTES >> 4) + 2 * k, idesc8, 1u);
            } else {
#pragma unroll
              for (int k = 0; k < BLOCK_K / 16; ++k) {
                const uint64_t a_hi = da + 2 * k, a_lo = a_hi + (A_TILE_BYTES >> 4);
                const uint64_t b_hi = db + 2 * k, b_lo = b_hi + (P_B_TILE_BYTES >> 4);
                if (three) {
                  umma2_bf16(d_tmem, a_lo, b_hi, idesc, (it > w.ka || k > 0) ? 1u : 0u);
                  umma2_bf16(d_tmem, a_hi, b_lo, idesc, 1u);
                  umma2_bf16(d_tmem, a_hi, b_hi, idesc, 1u);
                } else {
                  umma2_bf16(d_tmem, a_hi, b_hi, idesc, (it > w.ka || k > 0) ? 1u : 0u);
                }
              }
            }
            umma2_commit_both(empty_bar(s));      // frees the slot in both CTAs
          }
          sa += stage_bytes;
          if (++s == nst) { s = 0; par ^= 1u; sa = tiles; }
        }
        if (elect_one()) umma2_commit_both(tmem_full_bar(acc));  // this accumulator is complete in both CTAs
      }
    }
  } else {
    // ===== epilogue warps: item j reads accumulator j & 1, then hands it back to the MMA issuer =====
    const long long U = (long long)num_tiles * total;
    for (int j = 0; j < sk.n_items; ++j) {
      const SkItem w = sk.item(j);
      const int t = w.tile;
      const int mp = t % m_pairs, nt = (t / m_pairs) % n_tiles, phase = t / (m_pairs * n_tiles);
      const int mtile = 2 * mp + (int)cta_rank;
      const uint32_t acc = (uint32_t)j & 1u;
      const int self = 2 * pair_id + (int)cta_rank;       // slot / flag index of this CTA
      int first = self;
      if (w.mode == 2) first = 2 * sk_pair_of((long long)t * total, U, num_pairs) + (int)cta_rank;
      if (st.out_tma && w.mode != 1) {
        if (st.out_single)
          tc_epilogue_tma<P_BN, true>(st, &tmO, stage_smem, mtile, nt * P_BN, phase, warp, lane,
                                      tmem_base + acc * P_BN, tmem_full_bar(acc), ((uint32_t)j >> 1) & 1u, w.mode,
                                      self, first);
        else
          tc_epilogue_tma<P_BN, false>(st, &tmO, stage_smem, mtile, nt * P_BN, phase, warp, lane,
                                       tmem_base + acc * P_BN, tmem_full_bar(acc), ((uint32_t)j >> 1) & 1u, w.mode,
                                       self, first);
      } else
        tc_epilogue<P_BN>(st, mtile, nt * P_BN, phase, 0, warp, lane, tmem_base + acc * P_BN, tmem_full_bar(acc),
                          ((uint32_t)j >> 1) & 1u, true, w.mode, self, first, 2);
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(tmem_empty_bar(acc));
    }
    // the staging tile must outlive the tensor stores that still read it
    if (st.out_tma && warp == 2 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_relaxed();   // neither CTA may free TMEM or exit while the pair is still working
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------
// host: tensor-map encoding (driver entry point fetched at run time; the library does not link libcuda)
// ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = (EncodeTiledFn)p;
  return fn;
}

// The CTA-pair kernel serves every stage with 256-wide N tiles.  A stage with a single M tile still uses it: the
// second CTA of each pair then owns an all-padding tile (its A boxes are out of bounds -> zero fill, no traffic; its
// stores are clipped), which wastes half of a tensor pipe that such weight-streaming stages leave idle anyway, and
// buys the persistent schedule, the halved weight traffic per CTA and stream-K over the K range.
// Stages whose K loop is only one or two blocks long (the first layer, the last layer's data gradient) are all
// prologue and epilogue: they run on the 1-CTA kernel with shallow rings and several CTAs per SM instead (measured in
// round 2: the last layer's data gradient at CIFAR-10, one K block per tile, takes 64 us on the pair kernel against
// 44 us here).
static bool use_pair(const StageDev& d) {
  const int mtiles = d.tiles_b * d.tiles_h * d.tiles_w;
  const int total = d.ph[0].ntaps * (d.Ka / BLOCK_K);
  return !d.wgrad && d.block_n == 256 && d.n_pad % 256 == 0 && d.ksplit == 1 && total >= 3 &&
         (mtiles >= 2 || total >= 8);
}

// The 3-pass bf16 data-gradient stages that run on the pair kernel with at least 8 M tiles take the fp16 / e4m3
// cross-term operands (DESIGN.md section 4.1): two pass-equivalents per K block instead of three.  With fewer rows
// (CelebA-HQ256 B=8: 1 and 4 M tiles, 128 and 512 rows) a stage streams far more weight bytes than it multiplies
// (2048 x 1024 x 16 taps for 128 rows), fewer MMA passes buy little, and the operand conversion costs more than they
// save.  lsnf_plan_create gives a selected stage that operand format (StageDev::cross8) and the conversion of its
// input; the pair kernel's main loop follows it.
bool tc_cross_fp8(const StageDev& d) {
  const int mtiles = d.tiles_b * d.tiles_h * d.tiles_w;
  return use_pair(d) && d.epi == EPI_GRAD_HL && d.passes == 3 && !d.fp16 && mtiles >= 8;
}

// Ring of the 1-CTA kernel for one launch: stage bytes, depth, dynamic shared memory to request.
struct RingGeom { int nst; size_t stage_bytes, smem; };
static RingGeom ring_geometry(const StageDev& d, int out_tma) {
  const bool three = d.passes != 1;
  const size_t stage = (size_t)(three ? 2 : 1) * (A_TILE_BYTES + (size_t)d.block_n * BLOCK_K * 2);
  const int total = d.ph[0].ntaps * (d.Ka / BLOCK_K);
  const int iters = d.ksplit > 1 ? d.it_per_split : total;
  // short loops: half an SM's shared memory at most, so two CTAs are resident; long loops: all of it
  // (round-2 sweep at CIFAR-10: a third or all of the shared memory instead of half changes the short stages by
  // -1 / +11 us; 128- or 64-wide tiles for the last layer's data gradient cost +10 / +43 us -- half it stays)
  const size_t budget = (iters <= 4 ? TC_SMEM_MAX / 2 : TC_SMEM_MAX) - TC_SMEM_EXTRA;
  int nst = (int)std::min<size_t>(budget / stage, (size_t)std::min(iters, TC_MAX_STAGES));
  nst = std::max(nst, 1);
  while (out_tma && nst * stage < 32768) ++nst;   // the tensor-store epilogue stages 32 KiB in the idle ring
  size_t smem = nst * stage + TC_SMEM_EXTRA;
  // never more resident CTAs than tensor memory can hold (the allocation of one more would spin)
  const int tmem_cols = d.block_n < 32 ? 32 : d.block_n;
  const int tmem_ctas = 512 / tmem_cols;
  smem = std::max(smem, (size_t)TC_SMEM_MAX / (tmem_ctas + 1) + 16);
  return {nst, stage, smem};
}

// Which tensor-store map the 16-bit output of a stage gets: 1 stride-2 forward [B][2H][2W][2C], 2 first layer
// [B][k*k][2C], 3 plain gradient [B][H][W][2C], 4 phase-split gradient; 0 = per-thread stores.
static int out_tma_kind(const StageHost& sh, bool pair) {
  const StageDev& d = sh.dev;
  const bool wide_single = d.block_n >= 128 && d.n_pad % d.block_n == 0 && d.ksplit == 1;   // 1-CTA kernel, wide N tile
  if (!(pair || wide_single) || !(d.epi == EPI_ACT_HL || d.epi == EPI_GRAD_HL)) return 0;
  if (d.epi == EPI_ACT_HL && sh.first) return 2;
  if (d.epi == EPI_ACT_HL && d.ms == 2) return 1;
  if (d.epi == EPI_GRAD_HL && !d.split) return 3;
  if (d.epi == EPI_GRAD_HL && d.split && d.bW >= 2 && d.bH >= 2 && (d.bH % 2) == 0) return 4;
  return 0;
}

// Stream-K (equal shares of tiles x K blocks per pair, partial accumulators exchanged through L2) pays only when
// whole-tile scheduling would leave the pairs badly balanced: it costs a partial-tile round trip per pair.
// One K block costs about 1 us of tensor time; the partial-tile round trip of stream-K about 35 of them.
static bool pair_stream_k(const StageDev& st, int max_pairs) {
  const int mtiles = st.tiles_b * st.tiles_h * st.tiles_w;
  const int num_tiles = (mtiles + 1) / 2 * (st.n_pad / P_BN) * st.nphase;
  const int total = st.ph[0].ntaps * (st.Ka / BLOCK_K);
  const int rounds = (num_tiles + max_pairs - 1) / max_pairs;
  const long long static_units = (long long)rounds * total;                        // critical path, whole tiles
  const long long sk_units = ((long long)num_tiles * total + max_pairs - 1) / max_pairs + 35;
  return sk_units < static_units && total >= 8 &&
         (long long)num_tiles * total >= 4LL * max_pairs && max_pairs <= 80;
}

TcLaunch tc_plan_launch(const StageHost& sh, int num_sms) {
  const StageDev& d = sh.dev;
  const bool pair = use_pair(d);
  const int mtiles = d.tiles_b * d.tiles_h * d.tiles_w;
  TcLaunch l;
  lsnf_launch_info& o = l.info;
  memset(&o, 0, sizeof(o));
  o.block = TC_THREADS;
  o.tma_store = out_tma_kind(sh, pair);   // before the ring: the tensor-store epilogue stages in it
  if (pair) {
    const int max_pairs = num_sms / 2;
    const int num_tiles = (mtiles + 1) / 2 * (d.n_pad / P_BN) * d.nphase;   // an odd tail pairs with an empty tile
    l.kernel = d.passes == 1 ? &tapgemm_tc2_kernel<true> : &tapgemm_tc2_kernel<false>;
    o.kernel = LSNF_KERNEL_PAIR;
    o.stream_k = pair_stream_k(d, max_pairs) ? 1 : 0;
    o.grid_x = 2 * (o.stream_k ? max_pairs : std::min(num_tiles, max_pairs));
    o.grid_y = o.grid_z = 1;
    o.ring_stages = d.passes == 1 ? P_MAX_STAGES : P_STAGES;
    o.stage_bytes = d.passes == 1 ? P_STAGE_BYTES / 2 : P_STAGE_BYTES;
    o.smem_bytes = P_SMEM_BYTES;
    o.ctas_per_sm = 1;
    o.tmem_columns = 512;
    o.cross_fp8 = d.cross8;
  } else {
    switch (d.block_n) {
      case 256: l.kernel = &tapgemm_tc_kernel<256>; break;
      case 128: l.kernel = &tapgemm_tc_kernel<128>; break;
      case 64: l.kernel = &tapgemm_tc_kernel<64>; break;
      case 32: l.kernel = &tapgemm_tc_kernel<32>; break;
      case 16: l.kernel = &tapgemm_tc_kernel<16>; break;
    }
    const RingGeom g = ring_geometry(d, o.tma_store);
    o.kernel = LSNF_KERNEL_SINGLE;
    // every blockIdx.z slice of a weight-gradient stage is one tap (x split)
    o.grid_x = mtiles; o.grid_y = d.n_pad / d.block_n; o.grid_z = (d.wgrad ? d.ph[0].ntaps : d.nphase) * d.ksplit;
    o.ring_stages = g.nst;
    o.stage_bytes = (int32_t)g.stage_bytes;
    o.smem_bytes = (int32_t)g.smem;
    // shared memory (1 KiB per CTA is reserved by the system), the 2048-thread and 64 Ki-register limits
    const int by_smem = (TC_SMEM_MAX + 1024) / ((int)g.smem + 1024);
    o.ctas_per_sm = std::max(1, std::min(by_smem, 2048 / TC_THREADS));
    o.tmem_columns = d.block_n < 32 ? 32 : d.block_n;
  }
  return l;
}

int tc_encode_maps(lsnf_plan* plan, StageHost& sh) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return LSNF_ERR_CUDA; }
  const StageDev& d = sh.dev;
  const lsnf_launch_info& li = sh.launch.info;
  auto failed = [&](const char* map, CUresult r) {
    set_error(std::string("cuTensorMapEncodeTiled(") + map + ") failed with code " + std::to_string((int)r) +
              " for stage layer " + std::to_string(sh.info.layer) + " kind " + std::to_string(sh.info.kind));
    return LSNF_ERR_CUDA;
  };
  {
    const cuuint64_t row = (cuuint64_t)2 * d.Ka * 2;  // bytes per position (hi|lo)
    cuuint64_t dims[5] = {(cuuint64_t)2 * d.Ka, (cuuint64_t)d.aW, (cuuint64_t)d.aH, (cuuint64_t)d.B, (cuuint64_t)d.aP};
    cuuint64_t strides[4] = {row, row * d.aW, row * d.aW * d.aH, row * d.aW * d.aH * d.B};
    cuuint32_t box[5] = {BLOCK_K, (cuuint32_t)d.bW, (cuuint32_t)d.bH, (cuuint32_t)d.bB, 1};
    cuuint32_t es[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(&sh.tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)d.a, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return failed("A", r);
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)2 * d.b_k, (cuuint64_t)d.b_rows};
    cuuint64_t strides[1] = {(cuuint64_t)2 * d.b_k * 2};
    const bool pair = li.kernel == LSNF_KERNEL_PAIR;   // each CTA of a pair loads half the N tile
    cuuint32_t box[2] = {BLOCK_K, (cuuint32_t)(pair ? d.block_n / 2 : d.block_n)};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&sh.tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)d.b, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return failed("B", r);
  }
  // output map of the 16-bit epilogues (tensor stores)
  if (li.tma_store) {
    const cuuint64_t C2 = (cuuint64_t)2 * d.oC, eb = 2;   // channels per position (hi|lo), bytes per element
    cuuint64_t dims[5], strides[4];
    cuuint32_t box[5], es[5] = {1, 1, 1, 1, 1};
    if (li.tma_store == 2) {                               // [B][k*k][2C]
      const cuuint64_t kk = (cuuint64_t)sh.k * sh.k;
      dims[0] = C2; dims[1] = kk; dims[2] = 1; dims[3] = 1; dims[4] = d.B;
      strides[0] = C2 * eb; strides[1] = C2 * kk * eb; strides[2] = C2 * kk * eb; strides[3] = C2 * kk * eb;
      box[0] = 64; box[1] = 1; box[2] = 1; box[3] = 1; box[4] = 128;
    } else if (li.tma_store == 1) {                        // [B][2H][2W][2C] as (c, px, w, py, b*H + h)
      const cuuint64_t W = d.Wg, H = d.Hg;
      dims[0] = C2; dims[1] = 2; dims[2] = W; dims[3] = 2; dims[4] = (cuuint64_t)d.B * H;
      strides[0] = C2 * eb; strides[1] = 2 * C2 * eb; strides[2] = 2 * W * C2 * eb; strides[3] = 4 * W * C2 * eb;
      box[0] = 64; box[1] = 1; box[2] = d.bW; box[3] = 1; box[4] = d.bB * d.bH;
    } else if (li.tma_store == 3) {                        // [B][H][W][2C]
      const cuuint64_t W = d.Wg, H = d.Hg;
      dims[0] = C2; dims[1] = W; dims[2] = H; dims[3] = d.B; dims[4] = 1;
      strides[0] = C2 * eb; strides[1] = W * C2 * eb; strides[2] = H * W * C2 * eb; strides[3] = (cuuint64_t)d.B * H * W * C2 * eb;
      box[0] = 64; box[1] = d.bW; box[2] = d.bH; box[3] = d.bB; box[4] = 1;
    } else {
      // 4: [4 = (py,px)][B][H/2][W/2][2C] as (c, w/2, b*(H/2) + h/2, px, py): strides increase monotonically; the
      // epilogue permutes its staging rows accordingly
      const cuuint64_t Wh = d.Wg / 2, Hh = d.Hg / 2;
      const cuuint64_t plane = (cuuint64_t)d.B * Hh * Wh * C2;
      dims[0] = C2; dims[1] = Wh; dims[2] = (cuuint64_t)d.B * Hh; dims[3] = 2; dims[4] = 2;
      strides[0] = C2 * eb; strides[1] = Wh * C2 * eb; strides[2] = plane * eb; strides[3] = 2 * plane * eb;
      box[0] = 64; box[1] = d.bW / 2; box[2] = d.bB * d.bH / 2; box[3] = 2; box[4] = 2;
    }
    CUresult r = enc(&sh.tmO, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, d.out, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return failed("out", r);
  } else {
    sh.tmO = sh.tmA;   // placeholder, never dereferenced
  }
  sh.maps_ready = true;
  return LSNF_OK;
}

// opt-in shared-memory limit of every instantiation, once per device (lsnf_plan_bind); function attributes are per
// device, so a process that drives several GPUs prepares each of them
int tc_prepare_device(int device) {
  static std::mutex mu;
  static bool done[64] = {false};
  std::lock_guard<std::mutex> lock(mu);
  if (device < 0 || device >= 64) { set_error("device index out of range"); return LSNF_ERR_INVALID; }
  if (done[device]) return LSNF_OK;
  LSNF_CUDA(cudaFuncSetAttribute(tapgemm_tc_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_MAX));
  LSNF_CUDA(cudaFuncSetAttribute(tapgemm_tc_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_MAX));
  LSNF_CUDA(cudaFuncSetAttribute(tapgemm_tc_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_MAX));
  LSNF_CUDA(cudaFuncSetAttribute(tapgemm_tc_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_MAX));
  LSNF_CUDA(cudaFuncSetAttribute(tapgemm_tc_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_MAX));
  LSNF_CUDA(cudaFuncSetAttribute(tapgemm_tc2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM_BYTES));
  LSNF_CUDA(cudaFuncSetAttribute(tapgemm_tc2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM_BYTES));
  done[device] = true;
  return LSNF_OK;
}

int launch_tapgemm_tc(const StageHost& sh, cudaStream_t s) {
  if (!sh.maps_ready) { set_error("tensor maps not encoded"); return LSNF_ERR_STATE; }
  const TcLaunch& l = sh.launch;
  if (!l.kernel) { set_error("unsupported N tile"); return LSNF_ERR_INVALID; }
  LSNF_CUDA(launch_k(l.kernel, dim3(l.info.grid_x, l.info.grid_y, l.info.grid_z), dim3(l.info.block),
                     l.info.smem_bytes, s, sh.tmA, sh.tmB, sh.tmO, sh.dev));
  return LSNF_OK;
}

}  // namespace lsnf
