// 1x1 gate convolutions of the hGRU step on tcgen05 (reference: hgru_module.py:696-711, 729-740),
// as a light non-persistent kernel: the op is HBM-bound (one bf16 operand read, one fp32 or bf16
// write per pixel, a k x k contraction in between), so instead of one persistent CTA per SM it runs
// many small CTAs per SM (10-24 KB of shared memory, 32-64 TMEM columns each) and lets occupancy
// hide the load -> MMA -> store latency chain.
//
// CTA = 128 consecutive pixels of one frame (one UMMA M tile).  The chunked operand layout
// [n][cg][pix][8] makes every channel chunk of the tile a contiguous 2 KB run, so CG 1-D bulk
// copies land the tile in shared memory directly in the canonical K-major UMMA layout.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "hconv_tc.cuh"
#include "sm100_ptx.cuh"

namespace hgru {

namespace detail_gate {
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t u[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
               : "r"(taddr));
  sm100::tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(u[i]);
}
}  // namespace detail_gate

template <int KP>
struct GateCfg {
  static constexpr int KSTEPS = KP / 16, CG = KP / 8;
  static constexpr int A_BYTES = CG * 128 * 16;
  static constexpr int W_BYTES = KSTEPS * 2 * KP * 16;
  static constexpr int SMEM_BYTES = A_BYTES + W_BYTES + 64 + 128;
  static constexpr uint32_t TMEM_COLS = KP < 32 ? 32 : KP;
};

template <int KP, class Epi>
__global__ void __launch_bounds__(128)
gate_tc_kernel(const __nv_bfloat16* __restrict__ act /*[N][CG][HW][8]*/, const TcConvArgs a) {
  using namespace sm100;
  using Cfg = GateCfg<KP>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 127u) & ~127u;
  const uint32_t a_buf = base, w_buf = base + Cfg::A_BYTES;
  const uint32_t bar_ld = w_buf + Cfg::W_BYTES, bar_mma = bar_ld + 8, tmem_slot = bar_ld + 16;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);   // provably warp-uniform
  const int lane = threadIdx.x & 31;
  const int HW = a.H * a.W;
  const int tiles_per_frame = (HW + 127) / 128;
  const int n = blockIdx.x / tiles_per_frame;
  const int p0 = (blockIdx.x - n * tiles_per_frame) * 128;
  const int valid = min(128, HW - p0);

  if (threadIdx.x == 0) {
    mbar_init(bar_ld, 1);
    mbar_init(bar_mma, 1);
    fence_barrier_init();
    mbar_arrive_expect_tx(bar_ld, static_cast<uint32_t>(Cfg::CG * valid * 16 + Cfg::W_BYTES));
    bulk_load(w_buf, a.wpk, Cfg::W_BYTES, bar_ld);
#pragma unroll
    for (int cg = 0; cg < Cfg::CG; ++cg)
      bulk_load(a_buf + cg * 2048, act + ((static_cast<size_t>(n) * Cfg::CG + cg) * HW + p0) * 8,
                static_cast<uint32_t>(valid * 16), bar_ld);
  }
  if (warp == 1) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_ptr, 0);

  if (warp == 0) {
    const bool leader = elect_one();
    mbar_wait(bar_ld, 0);
    tc_fence_after();
    constexpr uint32_t idesc = make_idesc(1, 128, KP);
    const uint64_t adesc = make_smem_desc(a_buf, 2048, 128);        // LBO: chunk plane, SBO: 8 pixels
    const uint64_t bdesc = make_smem_desc(w_buf, KP * 16, 128);
#pragma unroll
    for (int q = 0; q < Cfg::KSTEPS; ++q)
      if (leader) mma_bf16_ss(tmem_base, adesc + static_cast<uint64_t>((q * 2 * 2048) >> 4),
                              bdesc + static_cast<uint64_t>((q * 2 * KP * 16) >> 4), idesc, q != 0);
    if (leader) tc_commit(bar_mma);
    __syncwarp();
  }
  mbar_wait(bar_mma, 0);
  tc_fence_after();
  float acc[KP];
#pragma unroll
  for (int c0 = 0; c0 < KP; c0 += 16) {
    uint32_t v[16];
    tmem_ld16(tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + c0, v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 16; ++j) acc[c0 + j] = __uint_as_float(v[j]);
  }
  const int m = warp * 32 + lane;
  if (m < valid) {
    const int pin = p0 + m;
    Epi::template apply<KP>(a, n, pin / a.W, pin % a.W, acc);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

// Initial state of the tensor-core path in one pass (hgru_module.py:884-887, 696-711): O_0 (NHWC fp32, k channels, or
// null = zeros) -> H2 (quad-chunked fp32, zero padded) + the first timestep's gated operand
// A = F(sigmoid(O_0 *1x1 i_r + i_b) . O_0) (F: the 16-bit operand format, op_format.cuh; the packed i_r is in F too).
// Same shape as gate_tc_kernel: CTA = 128 pixels of one frame, the
// 1x1 conv is one UMMA tile; the 16-bit K-major operand tile is written to shared memory by the threads that
// convert the state, so the state is read from HBM exactly once.  (The SIMT version of this pass was bound by its
// shared-memory weight reads: 148 us per 256 frames at k = 25.)
// a.wpk = packed i_r, a.bias = i_b, a.H2 = H2 out, a.out_bf16 = operand out, a.act_pad as for the stacked conv.
template <int KP>
struct InitCfg {
  static constexpr int KSTEPS = KP / 16, CG = KP / 8;
  static constexpr int A_BYTES = CG * 128 * 16;
  static constexpr int W_BYTES = KSTEPS * 2 * KP * 16;
  static constexpr int STG_BYTES = 128 * (KP + 1) * 4;
  static constexpr int SMEM_BYTES = A_BYTES + W_BYTES + 64 + STG_BYTES + 128;
  static constexpr uint32_t TMEM_COLS = KP < 32 ? 32 : KP;
};

template <int KP, class F = OpBf16>
__global__ void __launch_bounds__(128)
init_state_tc_kernel(const float* __restrict__ h0 /*[N][HW][k] or nullptr*/, const TcConvArgs a) {
  using namespace sm100;
  using Cfg = InitCfg<KP>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 127u) & ~127u;
  const uint32_t a_buf = base, w_buf = base + Cfg::A_BYTES;
  const uint32_t bar_ld = w_buf + Cfg::W_BYTES, bar_mma = bar_ld + 8, tmem_slot = bar_ld + 16;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));      // generic pointer to `base`
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(gen + Cfg::A_BYTES + Cfg::W_BYTES + 16);
  float* stg = reinterpret_cast<float*>(gen + Cfg::A_BYTES + Cfg::W_BYTES + 64);
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int HW = a.H * a.W, k = a.kreal;
  const int tiles_per_frame = (HW + 127) / 128;
  const int n = blockIdx.x / tiles_per_frame;
  const int p0 = (blockIdx.x - n * tiles_per_frame) * 128;
  const int valid = min(128, HW - p0);

  if (threadIdx.x == 0) {
    mbar_init(bar_ld, 1);
    mbar_init(bar_mma, 1);
    fence_barrier_init();
    mbar_arrive_expect_tx(bar_ld, static_cast<uint32_t>(Cfg::W_BYTES));
    bulk_load(w_buf, a.wpk, Cfg::W_BYTES, bar_ld);
  }
  if (warp == 1) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  // the tile's pixels are contiguous in O_0: stream them in flat order into rows of KP + 1 floats
  {
    const float* src = h0 ? h0 + (static_cast<size_t>(n) * HW + p0) * k : nullptr;
    const unsigned magic = 0xFFFFFFFFu / static_cast<unsigned>(k) + 1u;      // e / k for e < 2^16
    const int tot = valid * k;
#pragma unroll 4
    for (int e = threadIdx.x; e < tot; e += 128) {
      const int pp = static_cast<int>(__umulhi(static_cast<unsigned>(e), magic));
      stg[pp * (KP + 1) + (e - pp * k)] = src ? __ldg(src + e) : 0.f;
    }
  }
  __syncthreads();
  const int m = threadIdx.x;
  const bool live = m < valid;
  const size_t pin = static_cast<size_t>(p0 + m);
  float hv[KP];
#pragma unroll
  for (int c = 0; c < KP; ++c) hv[c] = (live && c < k) ? stg[m * (KP + 1) + c] : 0.f;
#pragma unroll
  for (int cg = 0; cg < Cfg::CG; ++cg) {
    if (live) {
      st_stream(a.H2 + quad_off(a, n, 2 * cg, pin), make_float4(hv[8 * cg], hv[8 * cg + 1], hv[8 * cg + 2], hv[8 * cg + 3]));
      st_stream(a.H2 + quad_off(a, n, 2 * cg + 1, pin),
                make_float4(hv[8 * cg + 4], hv[8 * cg + 5], hv[8 * cg + 6], hv[8 * cg + 7]));
    }
    typename F::T2 h[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) h[q] = F::cvt2(hv[8 * cg + 2 * q], hv[8 * cg + 2 * q + 1]);
    *reinterpret_cast<uint4*>(gen + cg * 2048 + m * 16) = *reinterpret_cast<const uint4*>(h);   // K-major operand tile
  }
  fence_proxy_async();          // operand tile -> visible to the tensor core
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_ptr, 0);

  if (warp == 0) {
    const bool leader = elect_one();
    mbar_wait(bar_ld, 0);
    tc_fence_after();
    constexpr uint32_t idesc = make_idesc(F::kIdescFmt, 128, KP);
    const uint64_t adesc = make_smem_desc(a_buf, 2048, 128);        // LBO: chunk plane, SBO: 8 pixels
    const uint64_t bdesc = make_smem_desc(w_buf, KP * 16, 128);
#pragma unroll
    for (int q = 0; q < Cfg::KSTEPS; ++q)
      if (leader) mma_bf16_ss(tmem_base, adesc + static_cast<uint64_t>((q * 2 * 2048) >> 4),
                              bdesc + static_cast<uint64_t>((q * 2 * KP * 16) >> 4), idesc, q != 0);
    if (leader) tc_commit(bar_mma);
    __syncwarp();
  }
  mbar_wait(bar_mma, 0);
  tc_fence_after();
#pragma unroll
  for (int c0 = 0; c0 < KP; c0 += 8) {
    float acc[8], r[8];
    detail_gate::tmem_ld8(tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + c0, acc);
#pragma unroll
    for (int j = 0; j < 8; ++j)      // pad channels: hv = 0
      r[j] = (c0 + j < k) ? fast_sigmoid(acc[j] + __ldg(a.bias + c0 + j)) * hv[c0 + j] : 0.f;
    if (live) store_act_chunk<F>(a, a.out_bf16, n, c0 >> 3, pin, r);
  }
  (void)lane;
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

}  // namespace hgru
