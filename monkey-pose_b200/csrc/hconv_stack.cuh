// Tap-stacked implicit-GEMM 15x15 convolution for narrow layers (k <= 32) on tcgen05.
//
// Why: an M=128 UMMA reads 4 KB of A from shared memory whatever N is, and shared memory delivers
// 128 B/clk (profiles/r01_mma_shape_microbench.log): N = 32 runs at 35 % of the tensor issue rate,
// N >= 128 at 100 %.  With k = 25 output channels the N dimension is filled by stacking T
// horizontally adjacent filter taps into one B operand:
//     B[(s, c)][ci] = W[dy][T*g + T-1-s][ci][c]          (s = 0..T-1,  N = T*KC <= 128)
// One MMA with the pixel window at tap (dy, T*g + T-1) then yields, for every window position
// `pos`, the T partial products  D[pos][s] = in[pos + T*g + T-1 - PAD] * W[dy][T*g+T-1-s],
// and the convolution is  out[x] = sum_s D[x - s][s].  The shift by s is undone in the epilogue:
// a pixel row of a tile lives in 8 consecutive TMEM lanes of one warp, so a rotate-by-s shuffle
// delivers D[x-s][s] from the same tile when x%8 >= s and otherwise produces exactly the value
// lane x%8 of the NEXT tile needs -- kept in registers as a carry while the CTA walks the tiles
// of a 16-row block from left to right (one extra leading tile per block supplies the first carry).
//
// Unit = 16 rows x 64 columns of one frame = 1 carry tile + 8 output tiles, whole halo window
// (30 x ~82 pixels x KP channels) resident in shared memory.  TMEM holds four 128-column
// accumulators: tiles are processed in pairs, two accumulating while two drain, so the epilogue
// (shuffles + fused gate/integration math + global I/O) hides behind the MMAs.  The stacked
// weights (288 KB at k = 25 with the remainder-packed schedule) stream through a ring (5 stages at k = 25) once per
// tile pair.  Tap group 0 of a row's first carry tile only reads zero-filled window columns and is not issued.
//
// Narrow units (TcConvArgs::unit_tiles = 1): 16 rows x 8 columns = 1 carry tile + 1 output tile, one tile pair, for
// batches too small to fill the SMs with wide units.  The window, its TMA box and the weight schedule are those of
// the wide unit (the unused columns cost nothing at such batch sizes).  A narrow unit's carry tile is an output tile
// of a wide unit: it gets every tap group (unless it starts at image column 0, where the wide unit's carry tile
// skips group 0 too) through the same stage sequence, so its accumulator, the carry taken from it and every output
// are bitwise those of the wide unit -- a frame's result does not depend on the unit width.
//
// Launch chaining: the launches of one forward depend on each other only frame by frame (a unit needs the four
// units of its frame from the previous launch), so instead of grid-wide stream order each unit's epilogue counts
// itself done in a per-launch, per-frame counter (TcConvArgs::done_flags) and the next launch -- started early by
// programmatic dependent launch, its CTAs taking SMs as this launch's CTAs exit -- waits per frame
// (wait_flags) in its window producer and epilogue warps.
//
// Warps: w0 weight producer, w1 MMA issuer, w2 TMEM alloc, w3 window producer, w4.. epilogue warpgroups.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "hconv_tc.cuh"
#include "sm100_ptx.cuh"

namespace hgru {

// GX3: the epilogue-issued 1x1 gate conv runs on bf16 hi/lo splits too (bf16x3 mode): staging tiles for both halves
// of the new state, gate weights as [w_hi | w_lo] stacked along N plus w_hi (the SPLIT3 packing of hconv_tc.cuh).
// F_: format of the 16-bit operands, window, weights and gate staging tile (op_format.cuh).
template <int KP_, int T_, int KC_, bool GX3_ = false, class F_ = OpBf16>
struct StackCfg {
  static constexpr int KP = KP_, T = T_, KC = KC_;
  static constexpr bool GX3 = GX3_;
  using Fmt = F_;
  static constexpr int S = 15, PAD = 7;
  static constexpr int KSTEPS = KP / 16;
  static constexpr int CG = KP / 8;
  static constexpr int NG = (S + T - 1) / T;             // tap groups per filter row
  static constexpr int NPAD = 128;                        // UMMA N
  static constexpr int MAXNTO = 8;                        // output tiles per unit (64 columns)
  static constexpr int ROWS = kTileRows + S - 1;          // 30
  static constexpr int COLS = 8 * MAXNTO + T * (NG - 1) + 8;
  static constexpr int ROW_PITCH = COLS * 16;
  static constexpr int CHUNK_PITCH = ROWS * ROW_PITCH;
  static constexpr int WIN_BYTES = CG * CHUNK_PITCH;
  static constexpr int MIN_COL = T - 16;                  // image column of window column 0, minus x0
  // Epilogue warpgroups split each tile's channels in 8-channel chunks (the last group takes the rest): the
  // epilogue is latency-bound per thread, so more, lighter warps per SM sub-partition is what speeds it up.
#ifdef HGRU_STACK_NGRP4
  // development switch: at k = 25 give the 25th channel (the row-packed remainder plane with its 8 scattered operand
  // stores) a warpgroup of its own.  It balances the groups (no more waiting at the gate barrier) but the fifth warp
  // per SM sub-partition slows the MMA issuer: +8 % cycles, same time (profiles/r01_stack_kernel_v27_ngrp4_ab.log).
  static constexpr int NGRP = (KC == 25) ? 4 : ((KC > 16) ? 3 : 2);
#elif defined(HGRU_STACK_NGRP4_K32)
  static constexpr int NGRP = (KC == 32) ? 4 : ((KC > 16) ? 3 : 2);      // development switch: 8/8/8/8 instead of 8/8/16
#else
  static constexpr int NGRP = (KC > 16) ? 3 : 2;
#endif
  static constexpr int NEPI = 128 * NGRP;                 // epilogue threads
  static constexpr int NTHREADS = 128 + NEPI;             // 4 service warps + NGRP x 4 epilogue warps
  static constexpr int BLK_BYTES = 2 * NPAD * 16;         // one (dy, q, g) weight block
  static constexpr int STAGE_BYTES = NG * BLK_BYTES;      // all tap groups of one (dy, q)
  // Remainder packing (k = 25 = 3 full 8-channel chunks + ONE channel): instead of padding K to 32 for every
  // filter row, the last channel is stored as a plane whose 8 "channels" are that channel at 8 consecutive
  // rows, P[y][x][j] = in[y + j][x][c = 24] (written that way by the producing epilogues, 7 pad rows on top).
  // One K = 16 step then covers all 15 filter rows of that channel, and chunk 2 pairs up across filter rows:
  // 15 + 7 + 1 + 1 = 24 weight stages per tile pair instead of 30 -- a fifth fewer MMAs for the same result.
#ifdef HGRU_STACK_NO_REM
  static constexpr bool REM = false;      // development switch: A/B against the plain K schedule
#else
  static constexpr bool REM = (KC == 25) && (KP == 32);
#endif
  static constexpr int ACT_PAD = REM ? 7 : 0;             // zero rows on top of every operand chunk plane
  static constexpr int PASS_STAGES = REM ? (S + S / 2 + 2) : S * KSTEPS;   // weight stages per tile pair
  static constexpr int GATE_A_HALF = CG * 128 * 16;       // staging tile of the new state (bf16, K-major)
  static constexpr int GATE_A_BYTES = GATE_A_HALF * (GX3 ? 2 : 1);      // (GX3: hi tile, lo tile)
  static constexpr int GATE_W_BYTES = KSTEPS * 2 * KP * 16 * (GX3 ? 3 : 1);
  static constexpr int GATE_BYTES = GATE_A_BYTES + GATE_W_BYTES;
  // ring depth: as deep as the 227 KB allow
#ifdef HGRU_STACK_WSTAGES
  static constexpr int WSTAGES = HGRU_STACK_WSTAGES;      // development switch
#else
  // as many as fit next to the window (3..6).  The issuer's wait for a weight stage is the round trip
  // MMA completion -> commit -> producer -> bulk copy, not bandwidth: it is the same with the refills disabled,
  // and a fifth stage at k = 25 cut it from 50K to 37K cycles per launch (profiles/r01_stack_kernel_v19_*.log).
  static constexpr int WFIT = (232448 - WIN_BYTES - GATE_BYTES - 2048) / STAGE_BYTES;
  static constexpr int WSTAGES = WFIT > 6 ? 6 : (WFIT < 3 ? 3 : WFIT);
#endif
  // The window is loaded in WPARTS parts with their own barriers.  With the remainder-packed schedule the first
  // 15 stages of a pass read chunk planes 0-1 only and the last 9 read planes 2-3 only, so the next unit's first
  // half is loaded under the current unit's last 9 stages and its second half under the next unit's first 15.
  static constexpr int WPARTS = REM ? 2 : 1;
  static constexpr int PART_CHUNKS = CG / WPARTS;
  static constexpr int PART_BYTES = WIN_BYTES / WPARTS;
  static constexpr int NUM_BARS = 4 + 2 * WSTAGES + 8 + 1;
  static constexpr int PAR_FLOATS = 5 * KP + 4;           // bias, v0, v1, v2, gate_bias (KP each) + rho_t
  static constexpr int SMEM_BYTES =
      WIN_BYTES + WSTAGES * STAGE_BYTES + GATE_BYTES + NUM_BARS * 8 + 32 + PAR_FLOATS * 4 + 1024;
  static_assert(T * KC <= NPAD, "stacked taps must fit N = 128");
  static_assert(KC <= KP && KP % 16 == 0, "channel padding");
  static_assert((CHUNK_PITCH >> 4) < 16384, "LBO range");
  static_assert(2 * COLS <= 256, "TMA box limit");
  static_assert(!GX3 || Fmt::kIdescFmt == OpBf16::kIdescFmt, "hi/lo gate splits are bf16");
};

// Stacked weight packing: HWIO fp32 [15][15][k][k] -> F [dy][q][g][2 chunks][128 n][8 ci],
// n = s*KC + c  <->  tap dx = T*g + T-1-s, output channel c (zero where dx >= 15 or c, ci >= k).
// `lo_part` = 1 packs the remainder  F(w - F(w))  instead (second weight set of the bf16x3 mode).
template <class F = OpBf16>
__global__ void pack_weights_stack_kernel(const float* __restrict__ w, typename F::T* __restrict__ wpk,
                                          int k, int ksteps, int T, int KC, int NG, int lo_part = 0) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  const size_t total = static_cast<size_t>(15) * ksteps * NG * 2 * 128 * 8;
  if (i >= total) return;
  const int j = i & 7;
  size_t r = i >> 3;
  const int n = r % 128; r /= 128;
  const int ch = r & 1; r >>= 1;
  const int g = r % NG; r /= NG;
  const int q = r % ksteps;
  const int dy = r / ksteps;
  const int s = n / KC, c = n - s * KC;
  const int dx = T * g + T - 1 - s;
  const int ci = q * 16 + ch * 8 + j;
  float v = 0.f;
  if (s < T && dx >= 0 && dx < 15 && c < k && ci < k) v = w[((static_cast<size_t>(dy) * 15 + dx) * k + ci) * k + c];
  const typename F::T hi = F::cvt(v);
  wpk[i] = lo_part ? F::cvt(v - F::to_float(hi)) : hi;
}

// Same for the remainder-packed schedule (StackCfg::REM, KC = 25): [stage 24][g][2 chunks][128 n'][8 j] with the
// K elements of a stage drawn from
//   stage dy        (0..14): chunk 0 = channels 0..7, chunk 1 = channels 8..15 of filter row dy
//   stage 15 + i    (0..6) : chunks = channels 16..23 of filter rows 2i and 2i + 1
//   stage 22               : chunk 0 = channels 16..23 of row 14, chunk 1 = channel 24 of rows 0..7
//   stage 23               : chunk 0 = channel 24 of rows 8..14 (+ one zero), chunk 1 = zero
template <class F = OpBf16>
__global__ void pack_weights_stack_rem_kernel(const float* __restrict__ w, typename F::T* __restrict__ wpk, int k,
                                              int T, int KC, int NG, int lo_part = 0) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  const size_t total = static_cast<size_t>(24) * NG * 2 * 128 * 8;
  if (i >= total) return;
  const int j = i & 7;
  size_t r = i >> 3;
  const int np = r % 128; r /= 128;
  const int ch = r & 1; r >>= 1;
  const int g = r % NG;
  const int st = static_cast<int>(r / NG);
  const int s = np / KC, c = np - s * KC;
  const int dx = T * g + T - 1 - s;
  int dy = -1, ci = -1;
  if (st < 15) { dy = st; ci = ch * 8 + j; }
  else if (st < 22) { dy = 2 * (st - 15) + ch; ci = 16 + j; }
  else if (st == 22) { if (ch == 0) { dy = 14; ci = 16 + j; } else { dy = j; ci = 24; } }
  else if (ch == 0 && 8 + j < 15) { dy = 8 + j; ci = 24; }
  float v = 0.f;
  if (dy >= 0 && s < T && dx >= 0 && dx < 15 && c < k && ci < k)
    v = w[((static_cast<size_t>(dy) * 15 + dx) * k + ci) * k + c];
  const typename F::T hi = F::cvt(v);
  wpk[i] = lo_part ? F::cvt(v - F::to_float(hi)) : hi;
}

namespace detail {
template <int N>
__device__ __forceinline__ void tmem_ld_f(uint32_t taddr, float* v);
template <>
__device__ __forceinline__ void tmem_ld_f<16>(uint32_t taddr, float* v) {
  uint32_t u[16];
  sm100::tmem_ld16(taddr, u);
  sm100::tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(u[i]);
}
template <>
__device__ __forceinline__ void tmem_ld_f<8>(uint32_t taddr, float* v) {
  uint32_t u[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
               : "r"(taddr));
  sm100::tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(u[i]);
}
template <>
__device__ __forceinline__ void tmem_ld_f<1>(uint32_t taddr, float* v) {
  uint32_t u;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(u) : "r"(taddr));
  sm100::tmem_ld_wait();
  v[0] = __uint_as_float(u);
}
// Issue-only variants (no tcgen05.wait::ld): the caller batches several loads behind one wait.
template <int N>
__device__ __forceinline__ void tmem_ld_issue(uint32_t taddr, uint32_t* u);
template <>
__device__ __forceinline__ void tmem_ld_issue<16>(uint32_t taddr, uint32_t* u) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
        "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
      : "r"(taddr));
}
template <>
__device__ __forceinline__ void tmem_ld_issue<8>(uint32_t taddr, uint32_t* u) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
               : "r"(taddr));
}
template <>
__device__ __forceinline__ void tmem_ld_issue<1>(uint32_t taddr, uint32_t* u) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(u[0]) : "r"(taddr));
}
template <int CN>
__device__ __forceinline__ void tmem_ld_range_issue(uint32_t taddr, uint32_t (&u)[CN]) {
  static_assert(CN == 1 || CN == 8 || CN == 9 || CN == 16, "supported channel-range widths");
  if constexpr (CN == 1) {
    tmem_ld_issue<1>(taddr, u);
  } else if constexpr (CN == 16) {
    tmem_ld_issue<16>(taddr, u);
  } else if constexpr (CN == 8) {
    tmem_ld_issue<8>(taddr, u);
  } else {
    tmem_ld_issue<8>(taddr, u);
    tmem_ld_issue<1>(taddr + 8, u + 8);
  }
}
// KC consecutive fp32 columns of this thread's TMEM lane
template <int KC>
__device__ __forceinline__ void tmem_ld_block(uint32_t taddr, float (&v)[KC]) {
  static_assert(KC == 16 || KC == 25 || KC == 32, "supported stacked channel strides");
  if constexpr (KC == 16) {
    tmem_ld_f<16>(taddr, v);
  } else if constexpr (KC == 32) {
    tmem_ld_f<16>(taddr, v);
    tmem_ld_f<16>(taddr + 16, v + 16);
  } else {
    tmem_ld_f<16>(taddr, v);
    tmem_ld_f<8>(taddr + 16, v + 16);
    tmem_ld_f<1>(taddr + 24, v + 24);
  }
}
// CN consecutive fp32 columns (CN in {8, 9, 16}) of this thread's TMEM lane
template <int CN>
__device__ __forceinline__ void tmem_ld_range(uint32_t taddr, float (&v)[CN]) {
  static_assert(CN == 8 || CN == 9 || CN == 16, "supported channel-range widths");
  if constexpr (CN == 16) {
    tmem_ld_f<16>(taddr, v);
  } else if constexpr (CN == 8) {
    tmem_ld_f<8>(taddr, v);
  } else {
    tmem_ld_f<8>(taddr, v);
    tmem_ld_f<1>(taddr + 8, v + 8);
  }
}
}  // namespace detail

// MMA issue loop of the stacked kernel.  The whole warp runs it convergently (addresses and descriptors
// stay warp-uniform); one elected lane issues the tcgen05 instructions.
template <class Cfg, bool PROF, int WSETS = 1>
__device__ __forceinline__ void stack_mma_issuer(const TcConvArgs& a, uint32_t tmem_base, uint32_t win,
                                                 uint32_t w_buf, uint32_t bar_win_full, uint32_t bar_win_empty,
                                                 uint32_t bar_w_full, uint32_t bar_w_empty, uint32_t bar_acc_full,
                                                 uint32_t bar_acc_empty, int iters, int NT, int npairs) {
  using namespace sm100;
  constexpr int T = Cfg::T;
  const bool leader = elect_one();
  tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);      // read from shared memory: mark it warp-uniform
  constexpr uint32_t idesc = make_idesc(Cfg::Fmt::kIdescFmt, 128, Cfg::NPAD);
  const uint64_t adesc0 = make_smem_desc(win, Cfg::CHUNK_PITCH, Cfg::ROW_PITCH);
  const uint64_t bdesc0 = make_smem_desc(w_buf, Cfg::NPAD * 16, 128);
  uint32_t st = 0, ph = 0;
  bool w_ready = false;       // the current weight stage was already seen complete by the previous stage's probe
  uint32_t tc = 0;            // running tile counter: TMEM slot = tc & 3, use count = tc >> 2
  int vit = 0;
  long long t_win = 0, t_acc = 0, t_w = 0, t_begin = 0, t0 = 0;
  unsigned long long g_begin = 0;
  if constexpr (PROF) {
    t_begin = clock64();
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(g_begin));
  }
  for (int it = 0; it < iters; ++it) {
    const int u = it * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);
    if (u >= a.num_units) break;      // idle tail
    // Left-most unit of an image row: tap group 0 of the carry tile reads window columns 0..7 = image columns
    // T-16 .. T-9 < 0, all zero-filled by TMA, so those MMAs add nothing and are not issued.
    const bool carry_zero = (u % a.units_x) == 0;
    if constexpr (PROF) t0 = clock64();
    mbar_wait_warp(bar_win_full, vit & 1);
    if constexpr (PROF) t_win += clock64() - t0;
    tc_fence_after();
    bool part1_ready = Cfg::WPARTS == 1;
    for (int pr = 0; pr < npairs; ++pr) {
      // tiles are accumulated in pairs; with an odd count the single tile goes FIRST, so the last pass of a unit
      // is a full pair and the next unit's first window part has the longest possible time to land
      const bool odd = (NT & 1) != 0;
      const int j0 = odd ? (pr == 0 ? 0 : 2 * pr - 1) : 2 * pr;
      const bool two = odd ? (pr != 0) : true;
      const bool last_pass = pr + 1 == npairs;
      const uint32_t s0 = tc & 3, s1 = (tc + 1) & 3;
      if constexpr (PROF) t0 = clock64();
      mbar_wait_warp(bar_acc_empty + 8 * s0, ((tc >> 2) & 1) ^ 1);
      if (two) mbar_wait_warp(bar_acc_empty + 8 * s1, (((tc + 1) >> 2) & 1) ^ 1);
      if constexpr (PROF) t_acc += clock64() - t0;
      tc_fence_after();
      const uint32_t acc0 = tmem_base + s0 * Cfg::NPAD, acc1 = tmem_base + s1 * Cfg::NPAD;
      const uint64_t a_tile0 = adesc0 + static_cast<uint64_t>(8 * j0);      // 8 pixels = 8 x 16 B
      // one weight stage: wait for it, NG tap groups x (1 or 2) tiles, release it
      const bool skip0 = carry_zero && j0 == 0;      // tile j0 (accumulator 0) is the carry tile
      auto issue_stage = [&](uint64_t adesc_st, bool first) {
        if constexpr (PROF) t0 = clock64();
        if (!w_ready) mbar_wait_warp(bar_w_full + 8 * st, ph);
        if constexpr (PROF) t_w += clock64() - t0;
        tc_fence_after();
        // Probe the NEXT stage's barrier now and read the answer only after this stage's MMAs are issued:
        // the tensor queue is shallow (~2 MMAs), so a barrier round trip between stages otherwise drains it.
        const uint32_t nst = (st + 1 == Cfg::WSTAGES) ? 0 : st + 1;
        const bool probe = mbar_test(bar_w_full + 8 * nst, (st + 1 == Cfg::WSTAGES) ? ph ^ 1 : ph);
        if (leader) {
          const uint64_t bdesc_st = bdesc0 + static_cast<uint64_t>((st * Cfg::STAGE_BYTES) >> 4);
#pragma unroll
          for (int g = 0; g < Cfg::NG; ++g) {
            const uint64_t bdesc = bdesc_st + static_cast<uint64_t>((g * Cfg::BLK_BYTES) >> 4);
            const uint64_t adesc = adesc_st + static_cast<uint64_t>(T * g);
            const uint32_t accum = (!first || g != 0) ? 1u : 0u;
            // (with g = 0 skipped, g = 1 of the first stage is the MMA that overwrites the accumulator)
            if (!(skip0 && g == 0)) mma_bf16_ss(acc0, adesc, bdesc, idesc, (!first || g > (skip0 ? 1 : 0)) ? 1u : 0u);
            if (two) mma_bf16_ss(acc1, adesc + 8, bdesc, idesc, accum);
          }
          // release the weight stage when these MMAs have read it
          tc_commit(bar_w_empty + 8 * st);
        }
        w_ready = __all_sync(0xffffffffu, probe);
        if (++st == Cfg::WSTAGES) { st = 0; ph ^= 1; }
      };
      if constexpr (Cfg::REM) {
        // remainder-packed K schedule (see StackCfg::REM / pack_weights_stack_rem_kernel); the K = 16 chunk
        // pair of a stage is (start address, LBO): any two 16-byte pixel columns of the resident window
        constexpr uint32_t RP = Cfg::ROW_PITCH, CP = Cfg::CHUNK_PITCH;
        const uint64_t tile_off = static_cast<uint64_t>(8 * j0);
        const uint64_t dB = make_smem_desc(win + 2 * CP, RP, RP) + tile_off;                  // chunk 2 @ dy, dy+1
        const uint64_t dC = make_smem_desc(win + 2 * CP + 14 * RP, CP - 14 * RP, RP) + tile_off;   // chunk 2 @ 14 | P @ 0
        const uint64_t dD = make_smem_desc(win + 3 * CP + 8 * RP, RP, RP) + tile_off;         // P @ 8 | (zero weights)
        // (WSETS = 2: the same operand schedule twice, against the w_hi and then the w_lo weight set)
#pragma unroll 1
        for (int ws = 0; ws < WSETS; ++ws) {
          const bool last_set = ws + 1 == WSETS;
          for (int dy = 0; dy < Cfg::S; ++dy)
            issue_stage(a_tile0 + static_cast<uint64_t>((dy * RP) >> 4), (ws | dy) == 0);
          // chunk planes 0-1 are not read again by this unit: hand them to the window producer already
          if (last_set && last_pass && leader) tc_commit(bar_win_empty);
          if (!part1_ready) {        // planes 2-3 of this unit were loading under the stages above
            if constexpr (PROF) t0 = clock64();
            mbar_wait_warp(bar_win_full + 8, vit & 1);
            if constexpr (PROF) t_win += clock64() - t0;
            tc_fence_after();
            part1_ready = true;
          }
          for (int i = 0; i < Cfg::S / 2; ++i) issue_stage(dB + static_cast<uint64_t>((2 * i * RP) >> 4), false);
          issue_stage(dC, false);
          issue_stage(dD, false);
          if (last_set && last_pass && leader) tc_commit(bar_win_empty + 8);
        }
      } else {
        // stage order: (weight set,) filter row dy, then k-step q
#pragma unroll 1
        for (int ws = 0; ws < WSETS; ++ws)
          for (int dy = 0; dy < Cfg::S; ++dy) {
#pragma unroll
            for (int q = 0; q < Cfg::KSTEPS; ++q)
              issue_stage(a_tile0 + static_cast<uint64_t>((dy * Cfg::ROW_PITCH + q * 2 * Cfg::CHUNK_PITCH) >> 4),
                          (ws | dy | q) == 0);
          }
      }
      if (leader) {
        tc_commit(bar_acc_full + 8 * s0);
        if (two) tc_commit(bar_acc_full + 8 * s1);
      }
      tc += two ? 2 : 1;
    }
    // release the window (the two-part schedule released its parts inside the last pass)
    if constexpr (Cfg::WPARTS == 1) {
      if (leader) tc_commit(bar_win_empty);
    }
    ++vit;
  }
  if (PROF && a.prof && leader) {
    long long* o = a.prof + static_cast<size_t>(blockIdx.x) * 8;
    o[0] = clock64() - t_begin; o[1] = t_win; o[2] = t_acc; o[3] = t_w;
    unsigned long long g_end;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(g_end));
    o[6] = static_cast<long long>(g_end - g_begin);      // nanoseconds: o[0] / o[6] = the SM clock in GHz
  }
  __syncwarp();
}

// Epilogue of one warpgroup for the channel range [C0, C0+CN) of every tile: un-stack (rotate +
// carry), fused math, stores.  Two warpgroups split the channels so that each SM sub-partition has
// two epilogue warps to overlap TMEM / global-memory latencies; they never need to talk to each
// other (un-stacking and the integration math are per channel).
// C0 is a run-time value: warpgroups with the same channel count CN execute ONE copy of this code (the epilogue is
// the bulk of the kernel's instructions, and per-group copies thrash the instruction caches: `stall_no_inst` was
// 31 % of the H2 kernel's samples, profiles/r02_ncu_source_stalls_stack_k25_v39_v40.txt).
template <class Cfg, class Epi, int CN, bool PROF, bool PART = false>
__device__ __forceinline__ void stack_epilogue(const TcConvArgs& a, const int C0, uint32_t tmem_base, uint32_t bar_acc_full,
                                               uint32_t bar_acc_empty, int iters, int NT,
                                               int units_per_frame, int warp, int lane, bool profile,
                                               uint8_t* smem_raw, uint32_t gate_a, uint32_t gate_w,
                                               uint32_t bar_gate) {
  using namespace sm100;
  constexpr int KC = Cfg::KC, T = Cfg::T, KP = Cfg::KP;
  const bool gated = Epi::kGate && a.do_gate;
  uint32_t gate_uses = 0;
  constexpr int NCH = (CN + 7) / 8 * 8;            // channels handed to the fused epilogue (8-aligned)
  const int ew = warp & 3;
  const int m = ew * 32 + lane;
  const int prow = m >> 3, pcol = m & 7;
  uint32_t tc = 0;
  long long e_wait = 0, e_begin = 0, e0 = 0, e_tm = 0, e_fin = 0, e_gw = 0, e_gm = 0;
  if constexpr (PROF) e_begin = clock64();
  for (int it = 0; it < iters; ++it) {
    const int u = it * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);
    if (u >= a.num_units) break;      // idle tail: every role of the CTA stops at the same iteration
    const int nl = u / units_per_frame;
    const int r = u - nl * units_per_frame;
    const int n = a.n0 + nl;
    const int uy = r / a.units_x, ux = r - uy * a.units_x;
    const int y = uy * kTileRows + prow;
    if (a.wait_flags) {
      // chained launch: this frame's tensors are ready once all its units finished in the previous launch
      if (lane == 0)
        while (ld_acquire_gpu(a.wait_flags + n) < a.flag_target) {}
      __syncwarp();
    }
    float carry[CN];
#pragma unroll
    for (int c = 0; c < CN; ++c) carry[c] = 0.f;
#pragma unroll 1
    for (int j = 0; j < NT; ++j, ++tc) {
      const uint32_t slot = tc & 3;
      // this thread's output pixel; its global inputs are fetched while the MMAs still run
      const int x = ux * (8 * a.unit_tiles) + 8 * (j - 1) + pcol;
      const bool store = j >= 1 && y < a.H && x < a.W;
      const size_t pin = static_cast<size_t>(y) * a.W + x;
      typename Epi::template Pre<NCH> pre;
      if (store) Epi::template load<NCH, CN>(a, n, pin, C0, pre);
      // second launch of a two-launch (bf16x3) conv: the first launch's sums of this pixel, requested now
      float4 part[PART ? NCH / 4 : 1];
      if constexpr (PART) {
        if (store) {
#pragma unroll
          for (int i = 0; i < NCH / 4; ++i)
            if (4 * i < CN) part[i] = ld_stream(a.partial + quad_off(a, n, (C0 >> 2) + i, pin));
        }
      }
      if constexpr (PROF) e0 = clock64();
      mbar_wait(bar_acc_full + 8 * slot, (tc >> 2) & 1);
      if constexpr (PROF) { const long long t = clock64(); e_wait += t - e0; e0 = t; }
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + slot * Cfg::NPAD + C0;
      float out[NCH], nxt[CN];
      // all T tap slots of this thread's channels: loads issued back to back behind ONE wait
      uint32_t blk[T][CN];
#pragma unroll
#ifdef HGRU_DBG_ONE_TMEM_LD
      detail::tmem_ld_range_issue<CN>(taddr, blk[0]);
#pragma unroll
      for (int s = 1; s < T; ++s)
#pragma unroll
        for (int c = 0; c < CN; ++c) blk[s][c] = blk[0][c] + s;
#else
#pragma unroll
      for (int s = 0; s < T; ++s) detail::tmem_ld_range_issue<CN>(taddr + s * KC, blk[s]);
#endif
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < NCH; ++c) out[c] = (c < CN) ? __uint_as_float(blk[0][c < CN ? c : 0]) + carry[c < CN ? c : 0] : 0.f;
#pragma unroll
      for (int c = 0; c < CN; ++c) nxt[c] = 0.f;
#pragma unroll
      for (int s = 1; s < T; ++s) {
        const int src = (lane & ~7) | ((pcol - s) & 7);
        const bool own = pcol >= s;
#pragma unroll
        for (int c = 0; c < CN; ++c) {
#ifdef HGRU_DBG_NO_SHFL
          const float v = __uint_as_float(blk[s][c] + src);
#else
          const float v = __uint_as_float(__shfl_sync(0xffffffffu, blk[s][c], src));
#endif
          if (own) out[c] += v; else nxt[c] += v;
        }
      }
#pragma unroll
      for (int c = 0; c < CN; ++c) carry[c] = nxt[c];
      if constexpr (PART) {
        if (store) {
#pragma unroll
          for (int i = 0; i < NCH / 4; ++i)
            if (4 * i < CN) {
              out[4 * i] += part[i].x;
              out[4 * i + 1] += part[i].y;
              out[4 * i + 2] += part[i].z;
              out[4 * i + 3] += part[i].w;
            }
        }
      }
      if constexpr (PROF) { const long long t = clock64(); e_tm += t - e0; e0 = t; }
      const bool gate_follows = gated && j >= 1;
      if (!gate_follows) {
        tc_fence_before();
        mbar_arrive(bar_acc_empty + 8 * slot);      // accumulator drained: MMAs may reuse it
      }
      // the fused math + stores: ONE inlined copy serves both paths (the new state also stays in registers for the gate)
      float hv[NCH];
#pragma unroll
      for (int c = 0; c < NCH; ++c) hv[c] = 0.f;
      if (store) Epi::template finish<NCH, CN>(a, n, pin, C0, out, pre, hv);
      if constexpr (PROF) { const long long t = clock64(); e_fin += t - e0; e0 = t; }
      if (gate_follows) {
        // ---- fused gate: new state -> 16-bit (Cfg::Fmt) staging tile -> 1x1 conv on the tensor core -> sigmoid ----
        {
          uint8_t* stg = smem_raw + (gate_a - smem_u32(smem_raw));
#pragma unroll
          for (int i = 0; i < NCH / 8; ++i) {
            typename Cfg::Fmt::T2 h[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) h[q] = Cfg::Fmt::cvt2(hv[8 * i + 2 * q], hv[8 * i + 2 * q + 1]);
            *reinterpret_cast<uint4*>(stg + ((C0 >> 3) + i) * 2048 + m * 16) = *reinterpret_cast<const uint4*>(h);
            if constexpr (Cfg::GX3) {      // the bf16 remainders, as a second tile
              __nv_bfloat162 l[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float2 hf = __bfloat1622float2(h[q]);
                l[q] = __floats2bfloat162_rn(hv[8 * i + 2 * q] - hf.x, hv[8 * i + 2 * q + 1] - hf.y);
              }
              *reinterpret_cast<uint4*>(stg + Cfg::GATE_A_HALF + ((C0 >> 3) + i) * 2048 + m * 16) =
                  *reinterpret_cast<const uint4*>(l);
            }
          }
        }
        fence_proxy_async();          // staging writes -> visible to the async (tensor core) proxy
        tc_fence_before();            // our tcgen05.ld of this accumulator precede the barrier
        asm volatile("bar.sync 1, %0;" ::"n"(Cfg::NEPI) : "memory");
        if (warp == 4) {
          // the tile's own accumulator columns [0, KP) are free now: gate pre-activations land there
          const bool leader = elect_one();
          tc_fence_after();
          if (leader) {
            constexpr uint32_t gdesc = make_idesc(Cfg::Fmt::kIdescFmt, 128, KP);
            const uint64_t ad = make_smem_desc(gate_a, 2048, 128);
            if constexpr (Cfg::GX3) {
              // hi * [w_hi | w_lo] -> columns [0, 2 KP), then lo * w_hi added into columns [0, KP)
              constexpr uint32_t gdesc_w = make_idesc(Cfg::Fmt::kIdescFmt, 128, 2 * KP);
              const uint64_t ad_lo = make_smem_desc(gate_a + Cfg::GATE_A_HALF, 2048, 128);
              const uint64_t bd_w = make_smem_desc(gate_w, 2 * KP * 16, 128);
              const uint64_t bd_n = make_smem_desc(gate_w + 4 * KP * 16, KP * 16, 128);
#pragma unroll
              for (int q = 0; q < Cfg::KSTEPS; ++q) {
                mma_bf16_ss(tmem_base + slot * Cfg::NPAD, ad + static_cast<uint64_t>((q * 2 * 2048) >> 4),
                            bd_w + static_cast<uint64_t>((q * 6 * KP * 16) >> 4), gdesc_w, q != 0);
                mma_bf16_ss(tmem_base + slot * Cfg::NPAD, ad_lo + static_cast<uint64_t>((q * 2 * 2048) >> 4),
                            bd_n + static_cast<uint64_t>((q * 6 * KP * 16) >> 4), gdesc, 1u);
              }
            } else {
              const uint64_t bd = make_smem_desc(gate_w, KP * 16, 128);
#pragma unroll
              for (int q = 0; q < Cfg::KSTEPS; ++q)
                mma_bf16_ss(tmem_base + slot * Cfg::NPAD, ad + static_cast<uint64_t>((q * 2 * 2048) >> 4),
                            bd + static_cast<uint64_t>((q * 2 * KP * 16) >> 4), gdesc, q != 0);
            }
            tc_commit(bar_gate);
          }
          __syncwarp();
        }
        mbar_wait(bar_gate, gate_uses & 1);
        ++gate_uses;
        tc_fence_after();
        if constexpr (PROF) { const long long t = clock64(); e_gw += t - e0; e0 = t; }
        float gacc[NCH];
#pragma unroll
        for (int c = 0; c < NCH; c += 8) detail::tmem_ld_f<8>(taddr + c, gacc + c);   // columns C0 + c of the slot
        if constexpr (Cfg::GX3) {      // + the hi * w_lo products in columns [KP, 2 KP)
#pragma unroll
          for (int c = 0; c < NCH; c += 8) {
            float g2[8];
            detail::tmem_ld_f<8>(taddr + KP + c, g2);
#pragma unroll
            for (int j = 0; j < 8; ++j) gacc[c + j] += g2[j];
          }
        }
        tc_fence_before();
        mbar_arrive(bar_acc_empty + 8 * slot);
        if (store) Epi::template gate<NCH, CN>(a, n, pin, C0, gacc, hv);
        if constexpr (PROF) { const long long t = clock64(); e_gm += t - e0; e0 = t; }
      }
    }
    if (a.done_flags) {
      // all epilogue stores of this unit are issued: publish them, then count the unit as done
      asm volatile("bar.sync 2, %0;" ::"n"(Cfg::NEPI) : "memory");
      if (threadIdx.x == 128) {
        __threadfence();
        atomicAdd(a.done_flags + n, 1);
      }
    }
  }
  if (PROF && a.prof && (threadIdx.x & 127) == 0) {
    if (profile) {
      long long* o = a.prof + static_cast<size_t>(blockIdx.x) * 8;
      o[4] = clock64() - e_begin; o[5] = e_wait;
    }
    // per-warpgroup phase split, after the per-CTA records: [total, wait, tmem+unstack, finish, gate wait, gate math]
    long long* g = a.prof + static_cast<size_t>(gridDim.x) * 8 +
                   (static_cast<size_t>(blockIdx.x) * Cfg::NGRP + ((warp - 4) >> 2)) * 8;
    g[0] = clock64() - e_begin; g[1] = e_wait; g[2] = e_tm; g[3] = e_fin; g[4] = e_gw; g[5] = e_gm;
  }
}

// F: 16-bit operand format (op_format.cuh); Epi writes the next launch's operands in the same format.
template <int KP, int T, int KC, class Epi, bool PROF = false, int WSETS = 1, bool PART = false, bool GX3 = false,
          class F = OpBf16>
__global__ void __launch_bounds__((StackCfg<KP, T, KC, GX3, F>::NTHREADS), 1)
hconv_stack_kernel(const __grid_constant__ CUtensorMap in_map, const TcConvArgs a) {
  using namespace sm100;
  using Cfg = StackCfg<KP, T, KC, GX3, F>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t win = base;
  const uint32_t w_buf = win + Cfg::WIN_BYTES;
  const uint32_t gate_a = w_buf + Cfg::WSTAGES * Cfg::STAGE_BYTES;   // staging tile [CG][128 px][16 B]
  const uint32_t gate_w = gate_a + Cfg::GATE_A_BYTES;                // 1x1 gate weights
  const uint32_t bars = gate_w + Cfg::GATE_W_BYTES;
  const uint32_t bar_win_full = bars, bar_win_empty = bars + 16;     // [2] each (one per window part)
  const uint32_t bar_w_full = bars + 32;                             // [WSTAGES]
  const uint32_t bar_w_empty = bar_w_full + 8 * Cfg::WSTAGES;        // [WSTAGES]
  const uint32_t bar_acc_full = bar_w_empty + 8 * Cfg::WSTAGES;      // [4]
  const uint32_t bar_acc_empty = bar_acc_full + 32;                  // [4]
  const uint32_t bar_gate = bar_acc_empty + 32;
  const uint32_t tmem_slot = bar_gate + 8;
  const uint32_t par_off = (tmem_slot + 16 + 15u) & ~15u;            // per-channel parameter vectors (fp32)
  float* par = reinterpret_cast<float*>(smem_raw + (par_off - smem_u32(smem_raw)));
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  // warp index through a shuffle: tells the compiler it is warp-uniform, so the role branches below are
  // uniform branches and the MMA issuer's addresses can live in uniform registers
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_win_full + 8 * i, 1);
      mbar_init(bar_win_empty + 8 * i, 1);
    }
    for (int i = 0; i < Cfg::WSTAGES; ++i) {
      mbar_init(bar_w_full + 8 * i, 1);
      mbar_init(bar_w_empty + 8 * i, 1);
    }
    for (int i = 0; i < 4; ++i) {
      mbar_init(bar_acc_full + 8 * i, 1);
      mbar_init(bar_acc_empty + 8 * i, Cfg::NEPI);     // all epilogue threads
    }
    mbar_init(bar_gate, 1);
    fence_barrier_init();
    tma_prefetch_desc(&in_map);
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  if (warp >= 4) {
    // Per-channel parameter vectors -> shared memory.  With ~220 KB of the SM's SRAM carved out as shared
    // memory the L1 is a few KB, so every per-tile __ldg of these vectors was an L2 round trip on the
    // epilogue's critical path.
    for (int i = threadIdx.x - 128; i < 5 * KP; i += Cfg::NEPI) {
      const int v = i / KP;
      const float* sp = v == 0 ? a.bias : v == 1 ? a.v0 : v == 2 ? a.v1 : v == 3 ? a.v2 : a.gate_bias;
      par[i] = sp ? __ldg(sp + (i % KP)) : 0.f;
    }
    if (threadIdx.x == 128) par[5 * KP] = a.rho_t ? __ldg(a.rho_t) : 1.f;
  }
  if (Epi::kGate && a.do_gate && warp >= 4) {
    // 1x1 gate weights -> shared memory (generic-proxy writes, made visible to the tensor core)
    const uint4* src = reinterpret_cast<const uint4*>(a.gate_wpk);
    uint8_t* dst = smem_raw + (gate_w - smem_u32(smem_raw));
    for (int i = threadIdx.x - 128; i < Cfg::GATE_W_BYTES / 16; i += Cfg::NEPI)
      reinterpret_cast<uint4*>(dst)[i] = __ldg(src + i);
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  grid_launch_dependents();      // a chained next launch may take SMs as they free up (no effect otherwise)

  const int iters = (a.num_units + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int units_per_frame = a.units_x * a.units_y;
  const int ucols = 8 * a.unit_tiles;              // image columns per unit
  const int wseg = a.W < ucols ? a.W : ucols;
  const int NT = 1 + (wseg + 7) / 8;               // carry tile + output tiles, uniform over units
  const int npairs = (NT + 1) / 2;

  if (warp == 0) {
    // ---------------- weight producer ----------------
    if (lane == 0) {
      uint32_t st = 0, ph = 0;
      const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(a.wpk);
      for (int it = 0; it < iters; ++it) {
        if (it * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x) >= a.num_units) break;
        for (int pr = 0; pr < npairs; ++pr)
          for (int sg = 0; sg < Cfg::PASS_STAGES * WSETS; ++sg) {
            mbar_wait(bar_w_empty + 8 * st, ph ^ 1);
            if ((a.dbg_flags & 1) && (it | pr | (sg >= Cfg::WSTAGES))) {
              mbar_arrive(bar_w_full + 8 * st);      // development: reuse the resident (stale) stage
            } else {
              mbar_arrive_expect_tx(bar_w_full + 8 * st, Cfg::STAGE_BYTES);
              bulk_load(w_buf + st * Cfg::STAGE_BYTES, wsrc + static_cast<size_t>(sg) * Cfg::STAGE_BYTES,
                        Cfg::STAGE_BYTES, bar_w_full + 8 * st);
            }
            if (++st == Cfg::WSTAGES) { st = 0; ph ^= 1; }
          }
      }
    }
  } else if (warp == 3) {
    // ---------------- window producer: one TMA box per unit ----------------
    if (lane == 0) {
      int vit = 0;
      for (int it = 0; it < iters; ++it) {
        const int u = it * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);
        if (u >= a.num_units) continue;
        const int nl = u / units_per_frame;
        const int r = u - nl * units_per_frame;
        const int n = a.n0 + nl;
        const int uy = r / a.units_x, ux = r - uy * a.units_x;
        if (a.wait_flags) {
          while (ld_acquire_gpu(a.wait_flags + n) < a.flag_target) {}
          fence_proxy_async_global();
        }
        mbar_wait(bar_win_empty, (vit & 1) ^ 1);
        mbar_arrive_expect_tx(bar_win_full, Cfg::PART_BYTES);
        tma_load_4d(win, &in_map, bar_win_full, 2 * (ux * ucols + Cfg::MIN_COL),
                    uy * kTileRows - Cfg::PAD + Cfg::ACT_PAD, 0, n);
        if constexpr (Cfg::WPARTS == 2) {
          mbar_wait(bar_win_empty + 8, (vit & 1) ^ 1);
          mbar_arrive_expect_tx(bar_win_full + 8, Cfg::PART_BYTES);
          tma_load_4d(win + Cfg::PART_BYTES, &in_map, bar_win_full + 8, 2 * (ux * ucols + Cfg::MIN_COL),
                      uy * kTileRows - Cfg::PAD + Cfg::ACT_PAD, Cfg::PART_CHUNKS, n);
        }
        ++vit;
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer (convergent warp, one elected lane issues) ----------------
    const long long clk0 = a.clk_out ? clock64() : 0;
    const unsigned long long ns0 = a.clk_out ? global_timer_ns() : 0ull;
    stack_mma_issuer<Cfg, PROF, WSETS>(a, tmem_base, win, w_buf, bar_win_full, bar_win_empty, bar_w_full, bar_w_empty,
                                bar_acc_full, bar_acc_empty, iters, NT, npairs);
    if (a.clk_out && lane == 0) {      // cycles / nanoseconds of this CTA's MMA loop = its SM clock in GHz
      a.clk_out[2 * blockIdx.x] = static_cast<unsigned long long>(clock64() - clk0);
      a.clk_out[2 * blockIdx.x + 1] = global_timer_ns() - ns0;
    }
  } else if (warp >= 4) {
    // the epilogue functors read the parameter vectors through the arguments: point them at the staged copies
    TcConvArgs ae = a;
    ae.bias = par; ae.v0 = par + KP; ae.v1 = par + 2 * KP; ae.v2 = par + 3 * KP; ae.gate_bias = par + 4 * KP;
    ae.rho_t = par + 5 * KP;
    // ---------------- epilogue: NGRP warpgroups, 8-channel chunks each, the last one takes the rest ----------
#define HGRU_STACK_EPI(C0_, CN_)                                                                                 \
  stack_epilogue<Cfg, Epi, CN_, PROF, PART>(ae, C0_, tmem_base, bar_acc_full, bar_acc_empty, iters, NT,                 \
                                            units_per_frame, warp, lane, warp < 8, smem_raw, gate_a, gate_w, bar_gate)
    // all groups but the last take 8 channels and share one copy of the code
    constexpr int kLastGrp = Cfg::NGRP - 1;
    const int grp = (warp - 4) >> 2;
    if (grp < kLastGrp) HGRU_STACK_EPI(8 * grp, 8);
    else HGRU_STACK_EPI(8 * kLastGrp, KC - 8 * kLastGrp);
#undef HGRU_STACK_EPI
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace hgru
