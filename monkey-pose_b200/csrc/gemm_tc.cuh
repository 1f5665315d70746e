// Split-K GEMM on tcgen05 for the readout's first dense layer (reference: hgru_pose.py:91,156-163,
// `tf.matmul(reshape(x,[-1,in]), weights)`):   part[z][m][n] = sum_{k in slice z} A[m][k] * B[n][k]
//   A [M][K]  bf16, K-major  = batch-norm'ed hGRU output, flattened (h, w, c)
//   B [Nn][K] bf16, K-major  = fc_1 weights, transposed once at set_params
// The layer is weight-streaming bound at these batch sizes (K = 262 144, M <= 512): the grid is
// (N tiles) x (M tiles) x (K splits) ~ one CTA per SM so every SM streams a disjoint slice of B
// exactly once; partial sums are reduced by the readout tail kernel.
//
// CTA tile 128 x 256 x 64; operands land in shared memory through 2-D TMA boxes with the 128-byte
// swizzle (box = 64 bf16 = 128 B per row), the canonical K-major SW128 UMMA layout; 4-stage ring;
// one accumulator (256 TMEM columns); warps: w0 TMA, w1 MMA, w2 TMEM alloc, w4..7 epilogue.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "op_format.cuh"
#include "sm100_ptx.cuh"

namespace hgru {

// Precision (template parameter Op, op_format.cuh):
//   OpBf16x3: both operands are stored as bf16 hi + lo halves (hi = bf16(x), lo = bf16(x - hi)), the hi parts in
//     columns [0, Kpad) and the lo parts in [Kpad, 2*Kpad) of A and B.  Each k-block is accumulated as three products
//     A_hi*B_hi + A_lo*B_hi + A_hi*B_lo  (fp32-class accuracy: K = 262 144 bf16 products would otherwise contribute
//     ~2.5e-3 relative error, the largest single error of the bf16 path).  A stage holds the four tiles so B_hi is
//     fetched once for two products; 2 stages x 96 KB (BN = 256) / 3 x 64 KB (BN = 128).
//   OpFp16: one fp16 operand per value (11 significand bits, row pitch Kpad), one product per k-step at the bf16
//     rate; a stage is one A and one B tile, so the same shared memory holds 4 x 48 KB / 7 x 32 KB stages.
constexpr int kGemmBM = 128, kGemmBN = 256, kGemmBK = 64;
constexpr int kGemmABytes = kGemmBM * kGemmBK * 2;    // 16 KB
template <int BN, class Op = OpBf16x3>
struct GemmCfg {
  static_assert(BN == 128 || BN == 256, "N tile");
  static constexpr int kParts = Op::kParts;
  static constexpr int kStages = kParts == 2 ? (BN == 256 ? 2 : 3) : (BN == 256 ? 4 : 7);
  static constexpr int kBBytes = BN * kGemmBK * 2;                       // 32 / 16 KB
  static constexpr int kStageBytes = kParts * (kGemmABytes + kBBytes);   // A_hi, A_lo, B_hi, B_lo / A, B
  static constexpr int kSmemBytes = kStages * kStageBytes + 256 + 1024;
  static_assert(kSmemBytes <= 227 * 1024, "shared memory");
};
constexpr int kGemmSmemBytes = GemmCfg<kGemmBN>::kSmemBytes;

struct GemmArgs {
  int M, Nn, K;          // problem size
  int Kpad;              // K rounded up to the k-block: the column where the lo halves start (OpBf16x3)
  int kblocks_per_split; // K blocks (of 64) handled by one z slice
  float* part;           // [splits][M][Nn] fp32
  // implicit-GEMM convolution (CONV = true): A rows are the pixels (n, y, x) of a bf16 NHWC activation, K runs
  // over (dy, dx, ci); a 128-row tile is `by` image rows of `nf` frames
  int S, Cin, H, W, by, nf;
};

// K-major operand tile written by TMA with CU_TENSOR_MAP_SWIZZLE_128B: rows of 128 B, 8-row groups
// of 1024 B (SBO), 16-byte chunks XOR-swizzled inside each 1024-B atom.  Tile base 1024-B aligned.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>(1) << 16;                 // LBO (ignored for swizzled K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;         // SBO: 8 rows x 128 B
  d |= static_cast<uint64_t>(1) << 46;                 // descriptor version (sm_100)
  d |= static_cast<uint64_t>(2) << 61;                 // SWIZZLE_128B
  return d;
}

// BN = 256 for wide outputs; BN = 128 where the output has <= 128 columns, so that half of every MMA is not spent on
// zero-filled B rows.
// CONV = true: stride-1 SAME convolution as an implicit GEMM -- the A tile of k-block (tap, 64-channel block) is
// one 4-D TMA box of the NHWC activation shifted by the tap (zero fill = padding); map_a / map_a_lo are the hi
// and lo activation tensors.  CONV = false: plain GEMM, map_a_lo is ignored (lo halves sit at column Kpad).
// map_a_lo is not read when Op has one part.
template <int BN, bool CONV = false, class Op = OpBf16x3>
__global__ void __launch_bounds__(256, 1)
gemm_tc_splitk_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_a_lo,
                      const __grid_constant__ CUtensorMap map_b, const GemmArgs g) {
  using namespace sm100;
  using Cfg = GemmCfg<BN, Op>;
  constexpr bool kHiLo = Cfg::kParts == 2;
  constexpr int kGemmBN = BN, kGemmStages = Cfg::kStages, kGemmBBytes = Cfg::kBBytes;
  constexpr int kGemmStageBytes = Cfg::kStageBytes;
  // stage layout: A_hi, [A_lo], B_hi, [B_lo]
  constexpr int kBOff = Cfg::kParts * kGemmABytes;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = base + kGemmStages * kGemmStageBytes;
  const uint32_t bar_full = bars, bar_empty = bars + 8 * kGemmStages, bar_acc = bar_empty + 8 * kGemmStages;
  const uint32_t tmem_slot = bar_acc + 8;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);   // provably warp-uniform
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kGemmStages; ++i) {
      mbar_init(bar_full + 8 * i, 1);
      mbar_init(bar_empty + 8 * i, 1);
    }
    mbar_init(bar_acc, 1);
    fence_barrier_init();
    tma_prefetch_desc(&map_a);
    if constexpr (CONV && kHiLo) tma_prefetch_desc(&map_a_lo);
    tma_prefetch_desc(&map_b);
  }
  if (warp == 2) tmem_alloc<BN>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_ptr, 0);

  const int n0 = blockIdx.x * kGemmBN, m0 = blockIdx.y * kGemmBM, z = blockIdx.z;
  const int total_kb = (g.K + kGemmBK - 1) / kGemmBK;
  const int kb0 = z * g.kblocks_per_split;
  int nkb = total_kb - kb0;
  if (nkb > g.kblocks_per_split) nkb = g.kblocks_per_split;
  if (nkb < 0) nkb = 0;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t st = 0, ph = 0;
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(bar_empty + 8 * st, ph ^ 1);
        mbar_arrive_expect_tx(bar_full + 8 * st, kGemmStageBytes);
        const uint32_t sa = base + st * kGemmStageBytes;
        const int kc = (kb0 + kb) * kGemmBK;
        if constexpr (CONV) {
          const int cblks = g.Cin / kGemmBK, kbi = kb0 + kb;
          const int tap = kbi / cblks, cb = kbi - tap * cblks, pad = (g.S - 1) / 2;
          const int ppf = g.H * g.W;                      // pixels per frame
          const int tile = blockIdx.y;
          const int f0 = ppf >= kGemmBM ? tile / (ppf / kGemmBM) : tile * g.nf;
          const int y0 = ppf >= kGemmBM ? (tile % (ppf / kGemmBM)) * g.by : 0;
          const int cx = tap % g.S - pad, cy = y0 + tap / g.S - pad;
          tma_load_4d(sa, &map_a, bar_full + 8 * st, cb * kGemmBK, cx, cy, f0);                  // A_hi
          if constexpr (kHiLo)
            tma_load_4d(sa + kGemmABytes, &map_a_lo, bar_full + 8 * st, cb * kGemmBK, cx, cy, f0); // A_lo
        } else {
          tma_load_2d(sa, &map_a, bar_full + 8 * st, kc, m0);                                     // A_hi
          if constexpr (kHiLo)
            tma_load_2d(sa + kGemmABytes, &map_a, bar_full + 8 * st, g.Kpad + kc, m0);            // A_lo
        }
        tma_load_2d(sa + kBOff, &map_b, bar_full + 8 * st, kc, n0);                              // B_hi
        if constexpr (kHiLo)
          tma_load_2d(sa + kBOff + kGemmBBytes, &map_b, bar_full + 8 * st, g.Kpad + kc, n0);     // B_lo
        if (++st == kGemmStages) { st = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    const bool leader = elect_one();
    constexpr uint32_t idesc = make_idesc(Op::kIdescFmt, kGemmBM, kGemmBN);
    const uint64_t a_hi = make_smem_desc_sw128(base);
    const uint64_t a_lo = make_smem_desc_sw128(base + kGemmABytes);
    const uint64_t b_hi = make_smem_desc_sw128(base + kBOff);
    const uint64_t b_lo = make_smem_desc_sw128(base + kBOff + kGemmBBytes);
    uint32_t st = 0, ph = 0;
    for (int kb = 0; kb < nkb; ++kb) {
      mbar_wait_warp(bar_full + 8 * st, ph);
      tc_fence_after();
      const uint64_t so = static_cast<uint64_t>((st * kGemmStageBytes) >> 4);
#pragma unroll
      for (int ks = 0; ks < kGemmBK / 16; ++ks) {
        // advance 16 K-elements = 32 bytes inside the 128-byte swizzle row
        if (leader) {
          mma_bf16_ss(tmem_base, a_hi + so + ks * 2, b_hi + so + ks * 2, idesc, (kb | ks) != 0);
          if constexpr (kHiLo) {
            mma_bf16_ss(tmem_base, a_lo + so + ks * 2, b_hi + so + ks * 2, idesc, 1);
            mma_bf16_ss(tmem_base, a_hi + so + ks * 2, b_lo + so + ks * 2, idesc, 1);
          }
        }
      }
      if (leader) tc_commit(bar_empty + 8 * st);
      if (++st == kGemmStages) { st = 0; ph ^= 1; }
    }
    if (leader) tc_commit(bar_acc);
    __syncwarp();
  } else if (warp >= 4) {
    const int ew = warp & 3;
    const int m = m0 + ew * 32 + lane;
    float* dst = g.part + (static_cast<size_t>(z) * g.M + m) * g.Nn + n0;
    if (nkb > 0) {
      mbar_wait(bar_acc, 0);
      tc_fence_after();
    }
#pragma unroll 1
    for (int c0 = 0; c0 < kGemmBN; c0 += 16) {
      uint32_t v[16];
      if (nkb > 0) {
        tmem_ld16(tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + c0, v);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0u;
      }
      if (m < g.M) {
        if (n0 + c0 + 16 <= g.Nn && (g.Nn & 3) == 0) {
#pragma unroll
          for (int j = 0; j < 16; j += 4)
            *reinterpret_cast<float4*>(dst + c0 + j) =
                make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                            __uint_as_float(v[j + 3]));
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (n0 + c0 + j < g.Nn) dst[c0 + j] = __uint_as_float(v[j]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<BN>(tmem_base);
  }
}

// fc_1 weights [K][F] fp32 -> bf16 [F][hi(0..K) | pad | lo(0..K) | pad] (K-major B operand, row pitch 2*Kpad;
// OpBf16x3) or fp16 [F][0..K | pad] (row pitch Kpad; OpFp16); 32x32 tiles through shared memory.  The reference's K
// index (pin*k + c, tf.reshape of NHWC) is permuted to channel-major (c*HW + pin), the order in which the H2 epilogue
// emits the A operand (kch = 1: no permutation).
template <class Op = OpBf16x3>
__global__ void __launch_bounds__(256)
transpose_operand_kernel(const float* __restrict__ w, typename Op::T* __restrict__ wt, int K, int F, int Kpad,
                         int kch) {
  __shared__ float tile[32][33];
  const int k0 = blockIdx.x * 32, f0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // 32 x 8
  for (int r = ty; r < 32; r += 8) {
    const int kk = k0 + r, f = f0 + tx;
    tile[r][tx] = (kk < K && f < F) ? w[static_cast<size_t>(kk) * F + f] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int f = f0 + r, kk = k0 + tx;
    if (f < F && kk < K) {
      const float v = tile[tx][r];
      const int pin_ = kk / kch, c_ = kk - pin_ * kch;
      const int kd = c_ * (K / kch) + pin_;
      if constexpr (Op::kParts == 2) {
        const __nv_bfloat16 hi = __float2bfloat16(v);
        __nv_bfloat16* row = wt + static_cast<size_t>(f) * (2 * static_cast<size_t>(Kpad));
        row[kd] = hi;
        row[Kpad + kd] = __float2bfloat16(v - __bfloat162float(hi));
      } else {
        wt[static_cast<size_t>(f) * Kpad + kd] = Op::cvt(v);
      }
    }
  }
}

}  // namespace hgru
