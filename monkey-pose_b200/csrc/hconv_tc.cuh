// Implicit-GEMM SxS "SAME" convolution on tcgen05 tensor cores (sm_100a), bf16 operands, fp32
// accumulation in TMEM.  This is kernel K8 of SURVEY.md 2b: the 15x15 horizontal convolutions
// C1 = W * (G1 . H2) and C2 = W * H1 of the hGRU step (reference: hgru_module.py:615-624 via
// tf.nn.conv2d at :531-535), and it also serves the 3x3 stem convs (hgru_pose.py:146).
//
// GEMM view: M = output pixels, N = output channels, K = (tap, input channel).
//
// Data layout in HBM
//   activations (operand copy): bf16 "chunked NHWC"  [n][cg][y][x][8]   (cg = channel / 8)
//       -> one TMA box load brings a (rows+S-1) x (cols+S-1) halo window of 2 channel-chunks into
//          shared memory as [cg][row][col][16 B]; out-of-image pixels are zero-filled by TMA,
//          which IS the SAME padding.
//   weights: bf16 packed per (kstep, tap) as [2 chunks][CO_PAD][8 ci]  (2 KB at CO_PAD = 64)
//       -> streamed with 1-D bulk copies through a small ring.
//
// Shared-memory operand form: the no-swizzle K-major canonical layout (8-row x 16-byte core
// matrices).  A pixel's 8 channels are one 16-byte row, 8 horizontally adjacent pixels form one
// core matrix, so an M = 128 operand is a 16-row x 8-column pixel patch: SBO = window row pitch,
// LBO = chunk plane pitch.  A filter tap (dy, dx) is then nothing but a different descriptor
// start address into the SAME resident window -- the input is read from HBM/L2 once per unit and
// reused by all S*S taps.
//
// CTA = 8 warps: w0 weight producer, w1 MMA issuer, w2 TMEM allocator, w3 input producer,
// w4..7 epilogue (TMEM -> registers -> global).  Persistent over "units" (16 x 8*TILES_X pixels
// of one frame); two TMEM accumulator sets so unit u's epilogue overlaps unit u+1's MMAs.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "op_format.cuh"
#include "sm100_ptx.cuh"

namespace hgru {

constexpr int kTileRows = 16;   // M tile = 16 rows x 8 cols of pixels

// SPLIT3: operands carry bf16 hi and lo halves (window parts [0,KSTEPS) = hi, [KSTEPS,2*KSTEPS) = lo) and
// every 16-channel k-step is accumulated as three products  a_hi*w_hi + a_hi*w_lo + a_lo*w_hi
// (fp32-class accuracy from bf16 tensor cores; used for the stem, whose smooth inputs make plain bf16
// rounding errors add up coherently, and for the hGRU's own convs in the bf16x3 mode).  The three products are
// TWO instructions: the weights of the a_hi pass are [w_hi | w_lo] stacked along N (accumulator columns [0, CO) and
// [CO, 2 CO), summed in the epilogue), the a_lo pass adds a_lo*w_hi into columns [0, CO).  An M = 128 MMA costs the
// same shared-memory operand fetch whatever its N, so one N = 2 CO instruction replaces two N = CO ones
// (N = 32: 35 % of the issue rate, N = 64: 67 %; profiles/r01_mma_shape_microbench.log).
// FUSE: the 1x1 gate conv that follows the integration (G2 after H1, the next step's G1 after H2) is issued from
// the epilogue as tcgen05.mma on a shared-memory staging tile of the new state (as in hconv_stack.cuh), and the
// launches of a forward are chained through per-frame completion counters (TcConvArgs::wait_flags / done_flags):
// two launches per timestep instead of four, no grid-wide stream order between them.
template <int S, int KSTEPS, int CO_PAD, int TILES_X, int G, int WSTAGES, bool SPLIT3 = false, bool FUSE = false>
struct TcConvCfg {
  static constexpr int kParts = SPLIT3 ? 2 * KSTEPS : KSTEPS;      // window parts (TMA boxes / barriers)
  static constexpr int kWSteps = SPLIT3 ? 2 * KSTEPS : KSTEPS;     // weight k-steps (SPLIT3: wide a_hi pass, a_lo pass)
  static constexpr int kS = S;
  static constexpr int kTaps = S * S;
  static constexpr int kPad = (S - 1) / 2;
  static constexpr int kRows = kTileRows + S - 1;           // window rows
  static constexpr int kCols = 8 * TILES_X + S - 1;         // window cols
  static constexpr int kRowPitch = kCols * 16;              // bytes (SBO of A)
  static constexpr int kChunkPitch = kRows * kRowPitch;     // bytes (LBO of A)
  static constexpr int kPartBytes = 2 * kChunkPitch;        // one kstep = 2 chunks
  static constexpr int kInBytes = kParts * kPartBytes;
  static constexpr int kTapBytes = 2 * CO_PAD * 16;         // one (kstep, tap) weight block
  static constexpr int kTapBytesWide = SPLIT3 ? 2 * kTapBytes : kTapBytes;   // [w_hi | w_lo] stacked along N
  static constexpr int kGroupBytes = kTaps * (kTapBytesWide + kTapBytes);     // SPLIT3: both passes of a 16-channel group
  // PAIRTAP (the fused 64-channel 15x15 kernel): taps dx and dx + 8 of a filter row share their A operand -- window
  // offset 8 t + dx serves tile t with tap dx AND tile t - 1 with tap dx + 8 -- and the accumulators of neighbouring
  // tiles are neighbouring TMEM columns, so ONE N = 128 instruction with B = [W[dx+8] ; W[dx]] feeds both: 39
  // instructions per filter row and k-step instead of 60, 21 of them at the full issue rate (an M = 128 MMA fetches
  // the same 4 KB of A whatever its N; at N = 64 that fetch, not the math, sets the pace).  Weights are packed in
  // 4 KB blocks [2 chunks][128 rows][8 ci]: block 0 = tap 7 (rows 64.. zero), block 1 + dx = rows 0-63 tap dx + 8,
  // rows 64-127 tap dx; a ring stage = two blocks.
  static constexpr bool kPairTap = FUSE;
  static constexpr int kPairBlockBytes = 2 * 128 * 16;
  static constexpr int kStageBytes = kPairTap ? 2 * kPairBlockBytes : G * kTapBytesWide;
  static constexpr int kStagesPerKstep = kPairTap ? S * 4 : kTaps / G;
  static constexpr int kAccN = SPLIT3 ? 2 * CO_PAD : CO_PAD; // accumulator columns per tile
  static constexpr int kAccCols = TILES_X * kAccN;          // TMEM columns per accumulator set
  static constexpr int kGateABytes = FUSE ? (CO_PAD / 8) * 128 * 16 : 0;   // staging tile of the new state (bf16, K-major)
  static constexpr int kGateWBytes = FUSE ? KSTEPS * 2 * CO_PAD * 16 : 0;   // packed 1x1 gate weights
  static constexpr int kGateBytes = kGateABytes + kGateWBytes;
  static constexpr int kNumBars = 2 * kParts + 2 * WSTAGES + 4 + (FUSE ? 1 : 0);
  // (no-swizzle operands and TMA boxes need 128-byte alignment; the fused configuration has no kilobyte to spare)
  static constexpr int kAlign = FUSE ? 128 : 1024;
  static constexpr int kSmemBytes = kInBytes + WSTAGES * kStageBytes + kGateBytes + kNumBars * 8 + 16 + kAlign;
  static_assert(kSmemBytes <= 232448, "shared memory per CTA");
  static_assert(kPairTap || kTaps % G == 0, "taps per stage must divide S*S");
  static_assert(!kPairTap || (S == 15 && CO_PAD == 64 && TILES_X == 4 && !SPLIT3), "paired-tap schedule: 64 channels, 15x15");
  static_assert(2 * kAccCols <= 512, "two accumulator sets must fit TMEM");
  static_assert(CO_PAD % 16 == 0 && CO_PAD >= 16 && kAccN <= 256, "UMMA N constraint (M=128)");
  static_assert(kChunkPitch % 16 == 0 && (kChunkPitch >> 4) < 16384, "LBO range");
};

struct TcConvArgs {
  int N, H, W;              // frames, image height / width
  int KP;                   // padded channel count of the fp32 NHWC tensors (== CO_PAD)
  int kreal;                // real channel count (pad channels are written as zero)
  int units_x, units_y;     // units per frame
  int num_units;
  // (16-bit tensors are typed bf16 here; in the fp16 mode the hGRU conv operands and weights hold fp16,
  //  see op_format.cuh -- the kernels only move their bytes or write them through the launch's format)
  const __nv_bfloat16* wpk; // packed weights [KSTEPS][taps][2][CO_PAD][8]
  const float* bias;        // [KP] lateral bias / conv bias (zero padded)
  const float* scale;       // [KP] (EpiBiasReluAffine) batch-norm scale, zero padded
  const float* shift;       // [KP]
  float* out;               // fp32 quad-chunked [N][KP/4][H][W][4]
  __nv_bfloat16* out_bf16;  // optional bf16 chunked copy [N][KP/8][H][W][8]
  // fused hGRU epilogues (all fp32 quad-chunked [N][KP/4][H][W][4] unless noted)
  const float* X;           // feed-forward drive
  const float* H1;          // EpiH2: inhibited state of this timestep
  const float* G;           // EpiH2: mix gate G2
  float* H2;                // EpiH1/EpiGate1: read; EpiH2: read + written in place
  const float* v0;          // per-channel vectors [KP], meaning depends on the epilogue
  const float* v1;
  const float* v2;
  const float* rho_t;       // device pointer to the adaptation scale rho[t] of this timestep
  // gate fused behind the integration (stacked kernel): 1x1 conv of the new state on tensor cores
  const __nv_bfloat16* gate_wpk;   // packed 1x1 weights [KSTEPS][2][KP][8] (o_r after H1, i_r after H2)
  const float* gate_bias;          // [KP] (o_b / i_b)
  float* gate_out;                 // EpiH1: G2 fp32 quad-chunked
  __nv_bfloat16* gate_act_out;     // EpiH2: next step's gated operand bf16(G1 . H2), chunked
  int do_gate;                     // 0: skip (last timestep's H2, or the unfused pipeline)
  // readout operand fused behind the last H2 update: bf16 hi + lo halves of batch_norm(H2) in the fc_1
  // GEMM's A layout, row n = [hi: c*HW + pin | ... | lo at +fc_kpad], row pitch 2*fc_kpad (nullptr: skip)
  __nv_bfloat16* fc_a;
  const float* fc_scale;           // [KP] folded inference batch-norm of the hGRU output (hgru_pose.py:82-90)
  const float* fc_shift;
  int fc_kpad;
  long long* prof;          // optional per-CTA cycle counters (development; nullptr in production)
  int dbg_flags;            // development only: bit 0 = do not re-stream weights after the first ring fill
  // bf16 operand tensors written by this launch (out_bf16 / gate_act_out) in the remainder-packed layout of
  // the stacked kernel (StackCfg::REM): act_pad zero rows on top of every chunk plane, and the last chunk
  // holds channel KP-8 at the 8 rows y..y+7.  0 = plain chunked layout.
  int act_pad;
  // operand tensors written by this launch carry bf16 hi AND lo halves.  1: chunk planes [0,CG) and [CG,2CG) of one
  // tensor (the SPLIT3 kernels of hconv_tc.cuh read both through one window; not with act_pad).  2: two separate
  // tensors in the stacked kernel's layout (act_pad honoured), the lo tensor lo_off elements behind the hi one (the
  // bf16x3 mode on the tap-stacked kernel reads them in two launches).
  int split_out;
  size_t lo_off;
  // bf16x3 on the tap-stacked kernel: the conv is two launches.  The first (EpiPartial, a_hi window, weight sets
  // w_hi then w_lo accumulated in TMEM) writes its un-stacked fp32 sums to `out`; the second (a_lo window, w_hi) adds
  // them back from `partial` before the integration epilogue.  nullptr: the ordinary single launch.
  const float* partial;
  // Launch chaining (stacked kernel): per-frame completion counters.  A unit of frame n may touch that frame's
  // tensors once wait_flags[n] == flag_target (all units of the frame finished in the previous launch), and adds 1
  // to done_flags[n] when its own stores are out.  nullptr = ordinary stream order.
  const int* wait_flags;
  int* done_flags;
  int flag_target;
  // A launch covers frames [n0, n0 + N) of the tensors (N = frames of this launch; tensor strides do not depend on
  // it): the stem convs run chunk by chunk behind the upload of the crops.
  int n0;
  // Optional in-kernel SM clock measurement (nvidia-smi keeps reporting the nominal clock while the kernel runs at
  // its power-limited one): the MMA issuer of CTA b stores {clock64 cycles, %globaltimer nanoseconds} it spent in
  // its loop at clk_out[2b], clk_out[2b + 1].  nullptr = off.
  unsigned long long* clk_out;
};

__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// fp32 state tensors of the tensor-core path are "quad-chunked": [n][c/4][y][x][4].  A thread owns
// one pixel (its TMEM lane) and a warp covers 8 horizontally adjacent pixels x 4 rows, so one 16-byte
// access per thread makes each warp request 4 fully used 128-byte lines (NHWC would touch 32 lines).
__device__ __forceinline__ size_t quad_off(const TcConvArgs& a, int n, int quad, size_t pin) {
  return ((static_cast<size_t>(n) * (a.KP >> 2) + quad) * (static_cast<size_t>(a.H) * a.W) + pin) * 4;
}

// H1 and G2 of the fused bf16 pipeline travel between its two launches as fp16 "oct-chunked" tensors
// [n][c/8][y][x][8] (one 16-byte access per pixel and 8 channels): both are bounded (tanh / sigmoid outputs), fp16
// keeps 11 significand bits of them, and their rounding (<= 4.9e-4 relative) sits well below the bf16 rounding of the
// conv operands the same launches consume (2e-3); state (H2), drive (X) and all arithmetic stay fp32.  The fp32-class
// modes (fp32, bf16x3) keep fp32 tensors.
__device__ __forceinline__ size_t oct_off(const TcConvArgs& a, int n, int oct, size_t pin) {
  return ((static_cast<size_t>(n) * (a.KP >> 3) + oct) * (static_cast<size_t>(a.H) * a.W) + pin) * 8;
}
__device__ __forceinline__ uint4 pack_half8(const float* r) {
  __half2 h[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) h[j] = __floats2half2_rn(r[2 * j], r[2 * j + 1]);
  return *reinterpret_cast<const uint4*>(h);
}
__device__ __forceinline__ void unpack_half8(const uint4& u, float* r) {
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 f = __half22float2(h[j]);
    r[2 * j] = f.x;
    r[2 * j + 1] = f.y;
  }
}

// streaming accesses of the epilogues: every state byte is touched once per launch, so keep it out of
// L1 (whose SRAM and datapath the UMMA operand fetch needs)
__device__ __forceinline__ float4 ld_stream(const float* p) {
  float4 r;
#ifdef HGRU_DBG_NO_GLOBAL
  return make_float4(0.f, 0.f, 0.f, 0.f);
#endif
  // (not .nc: a chained launch reads tensors that the previous launch, possibly still running, wrote)
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ float4 ld_stream_rw(const float* p) {   // data also written by this kernel (H2)
  float4 r;
#ifdef HGRU_DBG_NO_GLOBAL
  return make_float4(0.f, 0.f, 0.f, 0.f);
#endif
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p) : "memory");
  return r;
}
__device__ __forceinline__ uint4 ld_stream_u4(const void* p) {
  uint4 r;
#ifdef HGRU_DBG_NO_GLOBAL
  return make_uint4(0u, 0u, 0u, 0u);
#endif
  asm volatile("ld.global.L1::no_allocate.v4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream(float* p, const float4& v) {
#ifdef HGRU_DBG_NO_GLOBAL
  if (v.x != 123.456f) return;
#endif
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};"
               ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_stream(void* p, const uint4& v) {
#ifdef HGRU_DBG_NO_GLOBAL
  if (v.x != 0x12345678u) return;
#endif
  asm volatile("st.global.L1::no_allocate.v4.b32 [%0], {%1, %2, %3, %4};"
               ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ float fast_sigmoid(float x) { return 1.f / (1.f + __expf(-x)); }
// tanh via one exp: (1 - e^-2x) / (1 + e^-2x); |err| ~ 1e-7 abs, far inside the bf16-path budget
__device__ __forceinline__ float fast_tanh(float x) {
  const float e = __expf(-2.f * fabsf(x));
  const float t = __fdividef(1.f - e, 1.f + e);
  return copysignf(t, x);
}
// per-channel parameter quad; generic load: the stacked kernel stages these vectors in shared memory
__device__ __forceinline__ float4 ld_par4(const float* p) { return *reinterpret_cast<const float4*>(p); }
// 8 channels of one pixel -> a chunked 16-bit operand tensor in format F (see op_format.cuh)
template <class F = OpBf16>
__device__ __forceinline__ void store_chunk16(__nv_bfloat16* base, int KP, int HWp, int n, int cg, size_t pin,
                                              const float* r) {
  typename F::T2 h[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) h[j] = F::cvt2(r[2 * j], r[2 * j + 1]);
  __nv_bfloat16* o = base + ((static_cast<size_t>(n) * (KP >> 3) + cg) * HWp + pin) * 8;
  st_stream(o, *reinterpret_cast<const uint4*>(h));
}
// Operand store that honours TcConvArgs::act_pad (remainder-packed layout, see StackCfg::REM): chunk planes
// have act_pad zero rows on top; the last chunk is the row-packed plane P[y][x][j] = v(y + j, x) of channel
// KP - 8, so this pixel's value goes to the 8 planes rows y - j (j = 0..7), element j.
// (F: the operand format, op_format.cuh; the hi / lo splits of split_out are made in it too)
template <class F = OpBf16>
__device__ __forceinline__ void store_act_chunk1(const TcConvArgs& a, __nv_bfloat16* base, int n, int cg,
                                                 size_t pin, const float* r);
template <class F = OpBf16>
__device__ __forceinline__ void store_act_chunk(const TcConvArgs& a, __nv_bfloat16* base, int n, int cg,
                                                size_t pin, const float* r) {
  if (a.split_out) {
    float hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      hi[j] = F::to_float(F::cvt(r[j]));
      lo[j] = r[j] - hi[j];
    }
    if (a.split_out == 2) {      // two tensors in the stacked kernel's own layout
      store_act_chunk1<F>(a, base, n, cg, pin, hi);
      store_act_chunk1<F>(a, base + a.lo_off, n, cg, pin, lo);
      return;
    }
    store_chunk16<F>(base, 2 * a.KP, a.H * a.W, n, cg, pin, hi);
    store_chunk16<F>(base, 2 * a.KP, a.H * a.W, n, (a.KP >> 3) + cg, pin, lo);
    return;
  }
  store_act_chunk1<F>(a, base, n, cg, pin, r);
}
template <class F>
__device__ __forceinline__ void store_act_chunk1(const TcConvArgs& a, __nv_bfloat16* base, int n, int cg,
                                                 size_t pin, const float* r) {
  if (a.act_pad == 0) {
    store_chunk16<F>(base, a.KP, a.H * a.W, n, cg, pin, r);
    return;
  }
  const size_t plane = static_cast<size_t>(a.H + a.act_pad) * a.W;
  const size_t pp = pin + static_cast<size_t>(a.act_pad) * a.W;
  if (cg != (a.KP >> 3) - 1) {
    store_chunk16<F>(base, a.KP, static_cast<int>(plane), n, cg, pp, r);
  } else {
    typename F::T* o = reinterpret_cast<typename F::T*>(base) + ((static_cast<size_t>(n) * (a.KP >> 3) + cg) * plane + pp) * 8;
    const typename F::T v = F::cvt(r[0]);
#ifdef HGRU_DBG_REM_ONE_STORE
    o[0] = v;      // development: upper bound of what a cheaper remainder-plane write could give (wrong results)
#else
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j - static_cast<ptrdiff_t>(j) * a.W * 8] = v;
#endif
  }
}

// ---- epilogue functors: consume one pixel's CO_PAD accumulators --------------------------------
// out = acc + bias                       (P = conv + lateral_bias, hgru_module.py:657)
struct EpiBias {
  static constexpr bool kGate = false;
  template <int NCH> struct Pre {};
  template <int NCH, int NREAL = NCH>
  __device__ static __forceinline__ void load(const TcConvArgs&, int, size_t, int, Pre<NCH>&) {}
  template <int NCH, int NREAL = NCH>
  __device__ static __forceinline__ void gate(const TcConvArgs&, int, size_t, int, const float*, const float*) {}
  template <int NCH, int NREAL = NCH>
  __device__ static __forceinline__ void finish(const TcConvArgs& a, int n, size_t pin, int c0,
                                                const float* acc, const Pre<NCH>&, float* = nullptr) {
#pragma unroll
    for (int c = 0; c < NCH; c += 4) {
      const float4 b = ld_par4(a.bias + c0 + c);
      *reinterpret_cast<float4*>(a.out + quad_off(a, n, (c0 + c) >> 2, pin)) =
          make_float4(acc[c] + b.x, acc[c + 1] + b.y, acc[c + 2] + b.z, acc[c + 3] + b.w);
    }
  }
  template <int CO_PAD>
  __device__ static __forceinline__ void apply(const TcConvArgs& a, int n, int y, int x,
                                               float (&acc)[CO_PAD]) {
    Pre<CO_PAD> p;
    finish<CO_PAD>(a, n, static_cast<size_t>(y) * a.W + x, 0, acc, p);
  }
};
// out = acc: the raw fp32 sums of a partial convolution (first launch of a two-launch bf16x3 conv on the stacked kernel)
struct EpiPartial {
  static constexpr bool kGate = false;
  template <int NCH> struct Pre {};
  template <int NCH, int NREAL = NCH>
  __device__ static __forceinline__ void load(const TcConvArgs&, int, size_t, int, Pre<NCH>&) {}
  template <int NCH, int NREAL = NCH>
  __device__ static __forceinline__ void gate(const TcConvArgs&, int, size_t, int, const float*, const float*) {}
  template <int NCH, int NREAL = NCH>
  __device__ static __forceinline__ void finish(const TcConvArgs& a, int n, size_t pin, int c0,
                                                const float* acc, const Pre<NCH>&, float* = nullptr) {
#pragma unroll
    for (int c = 0; c < NCH; c += 4)
      if (c < NREAL)
        st_stream(a.out + quad_off(a, n, (c0 + c) >> 2, pin), make_float4(acc[c], acc[c + 1], acc[c + 2], acc[c + 3]));
  }
};
// out = relu(acc + bias) * scale + shift  (conv_layer + inference batch-norm, hgru_pose.py:61-80),
// fp32 NHWC plus the bf16 chunked operand copy for the next tensor-core conv.
struct EpiBiasReluAffine {
  template <int CO_PAD>
  __device__ static __forceinline__ void apply(const TcConvArgs& a, int n, int y, int x,
                                               float (&acc)[CO_PAD]) {
    const size_t pin = static_cast<size_t>(y) * a.W + x;
#pragma unroll
    for (int c = 0; c < CO_PAD; c += 8) {
      float r[8];
#pragma unroll
      for (int j = 0; j < 8; ++j)
        r[j] = fmaxf(acc[c + j] + __ldg(a.bias + c + j), 0.f) * __ldg(a.scale + c + j) + __ldg(a.shift + c + j);
      if (a.out) {
        *reinterpret_cast<float4*>(a.out + quad_off(a, n, c >> 2, pin)) = make_float4(r[0], r[1], r[2], r[3]);
        *reinterpret_cast<float4*>(a.out + quad_off(a, n, (c >> 2) + 1, pin)) = make_float4(r[4], r[5], r[6], r[7]);
      }
      if (a.out_bf16) {
        // hi + lo bf16 split of the operand copy (see stem_conv1_pool_bn_kernel): planes [0,CG), [CG,2CG)
        float hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          hi[j] = __bfloat162float(__float2bfloat16(r[j]));
          lo[j] = r[j] - hi[j];
        }
        store_chunk16(a.out_bf16, 2 * a.KP, a.H * a.W, n, c >> 3, pin, hi);
        store_chunk16(a.out_bf16, 2 * a.KP, a.H * a.W, n, (a.KP >> 3) + (c >> 3), pin, lo);
      }
    }
  }
};

// ---- fused integration epilogues -----------------------------------------------------------------
// Both are split into `load` (every global read of a pixel's NCH channels, issued back to back so
// their latencies overlap, and callable BEFORE the accumulator is ready) and `finish` (math + stores).
// The split matters: H2 is updated in place, so without it the compiler must order each chunk's
// loads after the previous chunk's stores and the epilogue becomes a chain of DRAM round trips.
//
// input_integration fused into the C1 conv (hgru_module.py:657, 795-804):
//   C1 = acc + lateral_bias;  H1 = tanh(X - (beta*H2 + nu) * C1)
// writes H1 fp32 and its chunked operand copy (format F, op_format.cuh).  bias = lateral_bias, v0 = beta, v1 = nu.
template <bool HALF, class F = OpBf16>
struct EpiH1T {
  static constexpr bool kGate = true;
  template <int NCH>
  struct Pre { float4 x[NCH / 4], h[NCH / 4]; };
  // NREAL (compile time): channels [NREAL, NCH) of this range are layout padding -- never loaded, no math
  template <int NCH, int NREAL = NCH>
  __device__ static __forceinline__ void load(const TcConvArgs& a, int n, size_t pin, int c0, Pre<NCH>& p) {
#pragma unroll
    for (int i = 0; i < NCH / 4; ++i) {
      if (4 * i < NREAL) {
        const size_t o = quad_off(a, n, (c0 >> 2) + i, pin);
        p.x[i] = ld_stream(a.X + o);
        p.h[i] = ld_stream(a.H2 + o);
      } else {
        p.x[i] = p.h[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  }
  // mix gate on the tensor-core result of H1 *1x1 o_r (hgru_module.py:729-740): G2 = sigmoid(. + o_b)
  template <int NCH, int NREAL = NCH>
  __device__ static __forceinline__ void gate(const TcConvArgs& a, int n, size_t pin, int c0, const float* gacc,
                                              const float*) {
    if constexpr (HALF) {
#pragma unroll
      for (int c = 0; c < NCH; c += 8) {
        if (c >= NREAL) continue;                 // a chunk of layout padding is never read back
        float g[8];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float bv[4] = {0.f, 0.f, 0.f, 0.f};
          if (c + 4 * h < NREAL) {
            const float4 b = ld_par4(a.gate_bias + c0 + c + 4 * h);
            bv[0] = b.x; bv[1] = b.y; bv[2] = b.z; bv[3] = b.w;
          }
#pragma unroll
          for (int j = 0; j < 4; ++j)
            g[4 * h + j] = (c + 4 * h + j < NREAL && c0 + c + 4 * h + j < a.kreal)
                               ? fast_sigmoid(gacc[c + 4 * h + j] + bv[j]) : 0.f;
        }
        st_stream(reinterpret_cast<__half*>(a.gate_out) + oct_off(a, n, (c0 + c) >> 3, pin), pack_half8(g));
      }
    } else {
#pragma unroll
      for (int c = 0; c < NCH; c += 4) {
        float g[4] = {0.f, 0.f, 0.f, 0.f};
        if (c < NREAL) {
          const float4 b = ld_par4(a.gate_bias + c0 + c);
          const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (c + j < NREAL && c0 + c + j < a.kreal) g[j] = fast_sigmoid(gacc[c + j] + bv[j]);
        }
        st_stream(a.gate_out + quad_off(a, n, (c0 + c) >> 2, pin), make_float4(g[0], g[1], g[2], g[3]));
      }
    }
  }
  template <int NCH, int NREAL = NCH>
  __device__ static __forceinline__ void finish(const TcConvArgs& a, int n, size_t pin, int c0,
                                                const float* acc, const Pre<NCH>& p, float* hout = nullptr) {
#pragma unroll
    for (int c = 0; c < NCH; c += 8) {
      float r[8];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int i = (c >> 2) + h, cc = c0 + c + 4 * h;
        const float xv[4] = {p.x[i].x, p.x[i].y, p.x[i].z, p.x[i].w};
        const float hv[4] = {p.h[i].x, p.h[i].y, p.h[i].z, p.h[i].w};
        float lbv[4] = {0.f, 0.f, 0.f, 0.f}, bev[4] = {0.f, 0.f, 0.f, 0.f}, nuv[4] = {0.f, 0.f, 0.f, 0.f};
        if (c + 4 * h < NREAL) {     // per-channel parameters: one vector load per quad (zero padded)
          const float4 lb = ld_par4(a.bias + cc);
          const float4 be = ld_par4(a.v0 + cc);
          const float4 nu = ld_par4(a.v1 + cc);
          lbv[0] = lb.x; lbv[1] = lb.y; lbv[2] = lb.z; lbv[3] = lb.w;
          bev[0] = be.x; bev[1] = be.y; bev[2] = be.z; bev[3] = be.w;
          nuv[0] = nu.x; nuv[1] = nu.y; nuv[2] = nu.z; nuv[3] = nu.w;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          r[4 * h + j] = 0.f;
          if (c + 4 * h + j < NREAL)
            r[4 * h + j] = fast_tanh(xv[j] - (bev[j] * hv[j] + nuv[j]) * (acc[c + 4 * h + j] + lbv[j]));
        }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (c0 + c + j >= a.kreal) r[j] = 0.f;
      if constexpr (HALF) {
        st_stream(reinterpret_cast<__half*>(a.out) + oct_off(a, n, (c0 + c) >> 3, pin), pack_half8(r));
      } else {
        st_stream(a.out + quad_off(a, n, (c0 + c) >> 2, pin), make_float4(r[0], r[1], r[2], r[3]));
        st_stream(a.out + quad_off(a, n, ((c0 + c) >> 2) + 1, pin), make_float4(r[4], r[5], r[6], r[7]));
      }
      store_act_chunk<F>(a, a.out_bf16, n, (c0 + c) >> 3, pin, r);
      if (hout) {
#pragma unroll
        for (int j = 0; j < 8; ++j) hout[c + j] = r[j];
      }
    }
  }
  template <int CO_PAD>
  __device__ static __forceinline__ void apply(const TcConvArgs& a, int n, int y, int x,
                                               float (&acc)[CO_PAD]) {
    constexpr int NCH = CO_PAD < 32 ? CO_PAD : 32;
    const size_t pin = static_cast<size_t>(y) * a.W + x;
#pragma unroll
    for (int c0 = 0; c0 < CO_PAD; c0 += NCH) {
      Pre<NCH> p;
      load<NCH>(a, n, pin, c0, p);
      finish<NCH>(a, n, pin, c0, acc + c0, p);
    }
  }
};
using EpiH1 = EpiH1T<false>;
using EpiH1h = EpiH1T<true>;      // fused bf16 pipeline: H1 and G2 leave as fp16
using EpiH1hF16 = EpiH1T<true, OpFp16>;      // ... with fp16 conv operands (the fp16 mode)
// output_integration + adaptation fused into the C2 conv (hgru_module.py:657, 806-823, 847-849):
//   C2 = acc + lateral_bias; e = gamma*C2; Ht = tanh(kappa*(H1+e) + omega*(H1*e));
//   H2 = (G2*H2 + (1-G2)*Ht) * rho_t      (in place) + chunked operand copy of the new H2 (format F).
// bias = lateral_bias, v0 = gamma, v1 = kappa, v2 = omega.
template <bool HALF, class F = OpBf16>
struct EpiH2T {
  static constexpr bool kGate = true;
  // HALF: h1 / g hold the raw 16-byte fp16 chunks (8 channels each) until `finish` unpacks them
  template <int NCH>
  struct Pre { float4 h1[NCH / 4], g[NCH / 4], h2[NCH / 4]; };
  template <int NCH, int NREAL = NCH>
  __device__ static __forceinline__ void load(const TcConvArgs& a, int n, size_t pin, int c0, Pre<NCH>& p) {
    if constexpr (HALF) {
#pragma unroll
      for (int i = 0; i < NCH / 8; ++i) {
        if (8 * i < NREAL) {
          const size_t o = oct_off(a, n, (c0 >> 3) + i, pin);
          const uint4 uh = ld_stream_u4(reinterpret_cast<const __half*>(a.H1) + o);
          const uint4 ug = ld_stream_u4(reinterpret_cast<const __half*>(a.G) + o);
          p.h1[2 * i] = make_float4(__uint_as_float(uh.x), __uint_as_float(uh.y), __uint_as_float(uh.z), __uint_as_float(uh.w));
          p.g[2 * i] = make_float4(__uint_as_float(ug.x), __uint_as_float(ug.y), __uint_as_float(ug.z), __uint_as_float(ug.w));
        }
      }
#pragma unroll
      for (int i = 0; i < NCH / 4; ++i)
        p.h2[i] = (4 * i < NREAL) ? ld_stream_rw(a.H2 + quad_off(a, n, (c0 >> 2) + i, pin)) : make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
#pragma unroll
      for (int i = 0; i < NCH / 4; ++i) {
        if (4 * i < NREAL) {
          const size_t o = quad_off(a, n, (c0 >> 2) + i, pin);
          p.h1[i] = ld_stream(a.H1 + o);
          p.g[i] = ld_stream(a.G + o);
          p.h2[i] = ld_stream_rw(a.H2 + o);
        } else {
          p.h1[i] = p.g[i] = p.h2[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    }
  }
  // input gate of the NEXT timestep on the tensor-core result of H2 *1x1 i_r (hgru_module.py:696-711):
  // G1 = sigmoid(. + i_b); gated operand = F(G1 . H2) for the next C1 conv.
  template <int NCH, int NREAL = NCH>
  __device__ static __forceinline__ void gate(const TcConvArgs& a, int n, size_t pin, int c0, const float* gacc,
                                              const float* hv) {
#pragma unroll
    for (int c = 0; c < NCH; c += 8) {
      float r[8];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float bv[4] = {0.f, 0.f, 0.f, 0.f};
        if (c + 4 * h < NREAL) {
          const float4 b = ld_par4(a.gate_bias + c0 + c + 4 * h);
          bv[0] = b.x; bv[1] = b.y; bv[2] = b.z; bv[3] = b.w;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)   // pad channels: hv = 0
          r[4 * h + j] = (c + 4 * h + j < NREAL) ? fast_sigmoid(gacc[c + 4 * h + j] + bv[j]) * hv[c + 4 * h + j] : 0.f;
      }
      store_act_chunk<F>(a, a.gate_act_out, n, (c0 + c) >> 3, pin, r);
    }
  }
  template <int NCH, int NREAL = NCH>
  __device__ static __forceinline__ void finish(const TcConvArgs& a, int n, size_t pin, int c0,
                                                const float* acc, const Pre<NCH>& p, float* hout = nullptr) {
    const float rho = *a.rho_t;
#pragma unroll
    for (int c = 0; c < NCH; c += 8) {
      float r[8];
      float h1h[8], gh[8];      // HALF: this chunk's fp16 inputs, unpacked
      if constexpr (HALF) {
        if (c < NREAL) {
          const float4 uh = p.h1[c >> 2], ug = p.g[c >> 2];
          unpack_half8(make_uint4(__float_as_uint(uh.x), __float_as_uint(uh.y), __float_as_uint(uh.z), __float_as_uint(uh.w)), h1h);
          unpack_half8(make_uint4(__float_as_uint(ug.x), __float_as_uint(ug.y), __float_as_uint(ug.z), __float_as_uint(ug.w)), gh);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) h1h[j] = gh[j] = 0.f;
        }
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int i = (c >> 2) + h, cc = c0 + c + 4 * h;
        const float4 h1 = p.h1[i], g = p.g[i], h2 = p.h2[i];
        float h1v[4] = {h1.x, h1.y, h1.z, h1.w}, gv[4] = {g.x, g.y, g.z, g.w};
        if constexpr (HALF) {
#pragma unroll
          for (int j = 0; j < 4; ++j) { h1v[j] = h1h[4 * h + j]; gv[j] = gh[4 * h + j]; }
        }
        const float h2v[4] = {h2.x, h2.y, h2.z, h2.w};
        float lbv[4] = {0.f, 0.f, 0.f, 0.f}, gav[4] = {0.f, 0.f, 0.f, 0.f}, kav[4] = {0.f, 0.f, 0.f, 0.f};
        float omv[4] = {0.f, 0.f, 0.f, 0.f};
        if (c + 4 * h < NREAL) {     // per-channel parameters: one vector load per quad (zero padded)
          const float4 lb = ld_par4(a.bias + cc);
          const float4 ga = ld_par4(a.v0 + cc);
          const float4 ka = ld_par4(a.v1 + cc);
          const float4 om = ld_par4(a.v2 + cc);
          lbv[0] = lb.x; lbv[1] = lb.y; lbv[2] = lb.z; lbv[3] = lb.w;
          gav[0] = ga.x; gav[1] = ga.y; gav[2] = ga.z; gav[3] = ga.w;
          kav[0] = ka.x; kav[1] = ka.y; kav[2] = ka.z; kav[3] = ka.w;
          omv[0] = om.x; omv[1] = om.y; omv[2] = om.z; omv[3] = om.w;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          r[4 * h + j] = 0.f;
          if (c + 4 * h + j < NREAL) {
            const float e = gav[j] * (acc[c + 4 * h + j] + lbv[j]);
            const float ht = fast_tanh(kav[j] * (h1v[j] + e) + omv[j] * (h1v[j] * e));
            r[4 * h + j] = (gv[j] * h2v[j] + (1.f - gv[j]) * ht) * rho;
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (c0 + c + j >= a.kreal) r[j] = 0.f;
      st_stream(a.H2 + quad_off(a, n, (c0 + c) >> 2, pin), make_float4(r[0], r[1], r[2], r[3]));
      if (c + 4 < NREAL)      // (a quad of pure layout padding is never read back: it stays at its initial zeros)
        st_stream(a.H2 + quad_off(a, n, ((c0 + c) >> 2) + 1, pin), make_float4(r[4], r[5], r[6], r[7]));
      if (a.out_bf16) store_chunk16<F>(a.out_bf16, a.KP, a.H * a.W, n, (c0 + c) >> 3, pin, r);
      if (a.fc_a) {
        // last timestep: emit the fc_1 operand (channel-major K order c*HW + pin, bf16 hi/lo split)
        const size_t HWp = static_cast<size_t>(a.H) * a.W;
        __nv_bfloat16* row = a.fc_a + static_cast<size_t>(n) * (2 * static_cast<size_t>(a.fc_kpad));
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int ch = c0 + c + j;
          if (ch < a.kreal) {
            const float v = r[j] * __ldg(a.fc_scale + ch) + __ldg(a.fc_shift + ch);
            const __nv_bfloat16 hi = __float2bfloat16(v);
            row[ch * HWp + pin] = hi;
            row[a.fc_kpad + ch * HWp + pin] = __float2bfloat16(v - __bfloat162float(hi));
          }
        }
      }
      if (hout) {
#pragma unroll
        for (int j = 0; j < 8; ++j) hout[c + j] = r[j];
      }
    }
  }
  template <int CO_PAD>
  __device__ static __forceinline__ void apply(const TcConvArgs& a, int n, int y, int x,
                                               float (&acc)[CO_PAD]) {
    constexpr int NCH = CO_PAD < 32 ? CO_PAD : 32;
    const size_t pin = static_cast<size_t>(y) * a.W + x;
#pragma unroll
    for (int c0 = 0; c0 < CO_PAD; c0 += NCH) {
      Pre<NCH> p;
      load<NCH>(a, n, pin, c0, p);
      finish<NCH>(a, n, pin, c0, acc + c0, p);
    }
  }
};
using EpiH2 = EpiH2T<false>;
using EpiH2h = EpiH2T<true>;
using EpiH2hF16 = EpiH2T<true, OpFp16>;
// mix gate as a 1x1 tensor-core conv (hgru_module.py:729-740): G2 = sigmoid(acc + o_b) -> fp32.
struct EpiGateOut {
  template <int CO_PAD>
  __device__ static __forceinline__ void apply(const TcConvArgs& a, int n, int y, int x,
                                               float (&acc)[CO_PAD]) {
    const size_t pin = static_cast<size_t>(y) * a.W + x;
#pragma unroll
    for (int c = 0; c < CO_PAD; c += 4) {
      const float4 b = ld_par4(a.bias + c);
      float4 g = make_float4(fast_sigmoid(acc[c] + b.x), fast_sigmoid(acc[c + 1] + b.y),
                             fast_sigmoid(acc[c + 2] + b.z), fast_sigmoid(acc[c + 3] + b.w));
      if (c + 0 >= a.kreal) g.x = 0.f;
      if (c + 1 >= a.kreal) g.y = 0.f;
      if (c + 2 >= a.kreal) g.z = 0.f;
      if (c + 3 >= a.kreal) g.w = 0.f;
      *reinterpret_cast<float4*>(a.out + quad_off(a, n, c >> 2, pin)) = g;
    }
  }
};
// input gate as a 1x1 tensor-core conv + gated operand (hgru_module.py:696-711):
//   G1 = sigmoid(acc + i_b);  operand = bf16(G1 . H2)   (chunked copy consumed by the C1 conv).
struct EpiGateIn {
  template <int CO_PAD>
  __device__ static __forceinline__ void apply(const TcConvArgs& a, int n, int y, int x,
                                               float (&acc)[CO_PAD]) {
    const size_t pin = static_cast<size_t>(y) * a.W + x;
    float4 hv[CO_PAD / 4];
#pragma unroll
    for (int i = 0; i < CO_PAD / 4; ++i) hv[i] = *reinterpret_cast<const float4*>(a.H2 + quad_off(a, n, i, pin));
#pragma unroll
    for (int c = 0; c < CO_PAD; c += 8) {
      float r[8];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(a.bias + c + 4 * h));
        const float4 v = hv[(c >> 2) + h];
        r[4 * h + 0] = fast_sigmoid(acc[c + 4 * h + 0] + b.x) * v.x;
        r[4 * h + 1] = fast_sigmoid(acc[c + 4 * h + 1] + b.y) * v.y;
        r[4 * h + 2] = fast_sigmoid(acc[c + 4 * h + 2] + b.z) * v.z;
        r[4 * h + 3] = fast_sigmoid(acc[c + 4 * h + 3] + b.w) * v.w;
      }
      store_chunk16(a.out_bf16, a.KP, a.H * a.W, n, c >> 3, pin, r);   // pad channels: H2 pad is 0
    }
  }
};

// F: format of the 16-bit operands (op_format.cuh); fp16 exists for the FUSE path (its Epi writes the same format).
template <int S, int KSTEPS, int CO_PAD, int TILES_X, int G, int WSTAGES, class Epi, bool SPLIT3 = false,
          bool FUSE = false, class F = OpBf16>
__global__ void __launch_bounds__(256, 1)
hconv_tc_kernel(const __grid_constant__ CUtensorMap in_map, const TcConvArgs a) {
  using namespace sm100;
  using Cfg = TcConvCfg<S, KSTEPS, CO_PAD, TILES_X, G, WSTAGES, SPLIT3, FUSE>;
  constexpr int NP = Cfg::kParts, NW = Cfg::kWSteps;
  static_assert(!FUSE || !SPLIT3, "the fused-gate epilogue serves the plain bf16 path");
  static_assert(FUSE || F::kIdescFmt == OpBf16::kIdescFmt, "16-bit operand formats other than bf16: FUSE path only");
  extern __shared__ uint8_t smem_raw[];
  // aligned carve-up
  const uint32_t base = (smem_u32(smem_raw) + static_cast<uint32_t>(Cfg::kAlign - 1)) & ~static_cast<uint32_t>(Cfg::kAlign - 1);
  const uint32_t in_buf = base;
  const uint32_t w_buf = in_buf + Cfg::kInBytes;
  const uint32_t gate_a = w_buf + WSTAGES * Cfg::kStageBytes;      // [CO_PAD/8][128 px][16 B]   (FUSE)
  const uint32_t gate_w = gate_a + Cfg::kGateABytes;               // packed 1x1 weights          (FUSE)
  const uint32_t bars = gate_w + Cfg::kGateWBytes;
  const uint32_t bar_in_full = bars;                               // [NP]
  const uint32_t bar_in_empty = bar_in_full + 8 * NP;              // [NP]
  const uint32_t bar_w_full = bar_in_empty + 8 * NP;               // [WSTAGES]
  const uint32_t bar_w_empty = bar_w_full + 8 * WSTAGES;           // [WSTAGES]
  const uint32_t bar_acc_full = bar_w_empty + 8 * WSTAGES;         // [2]
  const uint32_t bar_acc_empty = bar_acc_full + 16;                // [2]
  const uint32_t bar_gate = bar_acc_empty + 16;                    // (FUSE)
  const uint32_t tmem_slot = bar_gate + (FUSE ? 8 : 0);
  uint32_t* tmem_slot_ptr =
      reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);   // provably warp-uniform
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < NP; ++i) {
      mbar_init(bar_in_full + 8 * i, 1);
      mbar_init(bar_in_empty + 8 * i, 1);
    }
    for (int i = 0; i < WSTAGES; ++i) {
      mbar_init(bar_w_full + 8 * i, 1);
      mbar_init(bar_w_empty + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_acc_full + 8 * i, 1);
      mbar_init(bar_acc_empty + 8 * i, 128);
    }
    if constexpr (FUSE) mbar_init(bar_gate, 1);
    fence_barrier_init();
    tma_prefetch_desc(&in_map);
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  if constexpr (FUSE) {
    if (a.do_gate && warp >= 4) {
      // 1x1 gate weights -> shared memory (generic-proxy writes, made visible to the tensor core)
      const uint4* src = reinterpret_cast<const uint4*>(a.gate_wpk);
      uint8_t* dst = smem_raw + (gate_w - smem_u32(smem_raw));
      for (int i = threadIdx.x - 128; i < Cfg::kGateWBytes / 16; i += 128)
        reinterpret_cast<uint4*>(dst)[i] = __ldg(src + i);
      fence_proxy_async();
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_ptr, 0);
  if constexpr (FUSE) grid_launch_dependents();   // a chained next launch may take SMs as they free up

  const int units_per_frame = a.units_x * a.units_y;
  const int first = blockIdx.x;
  const int stride = gridDim.x;

  if (warp == 0) {
    // ---------------- weight producer: ring of WSTAGES stages, G taps each ----------------
    if (lane == 0) {
      uint32_t st = 0, ph = 0;
      for (int u = first; u < a.num_units; u += stride) {
        for (int q = 0; q < NW; ++q) {
          // SPLIT3 layout per 16-channel group: [taps] wide blocks ([w_hi | w_lo]) then [taps] w_hi blocks
          const bool wide = SPLIT3 && !(q & 1);
          const uint32_t sbytes = Cfg::kPairTap ? Cfg::kStageBytes : G * (wide ? Cfg::kTapBytesWide : Cfg::kTapBytes);
          const uint8_t* src = reinterpret_cast<const uint8_t*>(a.wpk) +
                               (Cfg::kPairTap ? static_cast<size_t>(q) * Cfg::kStagesPerKstep * Cfg::kStageBytes
                                : SPLIT3 ? static_cast<size_t>(q >> 1) * Cfg::kGroupBytes +
                                               ((q & 1) ? static_cast<size_t>(Cfg::kTaps) * Cfg::kTapBytesWide : 0)
                                         : static_cast<size_t>(q) * Cfg::kTaps * Cfg::kTapBytes);
          for (int sg = 0; sg < Cfg::kStagesPerKstep; ++sg) {
            mbar_wait(bar_w_empty + 8 * st, ph ^ 1);
            mbar_arrive_expect_tx(bar_w_full + 8 * st, sbytes);
            bulk_load(w_buf + st * Cfg::kStageBytes, src + static_cast<size_t>(sg) * sbytes, sbytes,
                      bar_w_full + 8 * st);
            if (++st == WSTAGES) { st = 0; ph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 3) {
    // ---------------- input producer: one TMA box per (unit, kstep) ----------------
    if (lane == 0) {
      int it = 0;
      for (int u = first; u < a.num_units; u += stride, ++it) {
        const int nl = u / units_per_frame;
        const int r = u - nl * units_per_frame;
        const int n = a.n0 + nl;
        const int uy = r / a.units_x, ux = r - uy * a.units_x;
        const int y0 = uy * kTileRows - Cfg::kPad;
        const int x0 = ux * (8 * TILES_X) - Cfg::kPad;
        if constexpr (FUSE) {
          if (a.wait_flags) {
            // chained launch: this frame's operand is complete once all its units finished in the previous launch
            while (ld_acquire_gpu(a.wait_flags + n) < a.flag_target) {}
            fence_proxy_async_global();
          }
        }
        for (int q = 0; q < NP; ++q) {
          mbar_wait(bar_in_empty + 8 * q, (it & 1) ^ 1);
          mbar_arrive_expect_tx(bar_in_full + 8 * q, Cfg::kPartBytes);
          // tensor viewed as 8-byte elements: dim0 = 2*x, dim1 = y, dim2 = chunk, dim3 = frame
          tma_load_4d(in_buf + q * Cfg::kPartBytes, &in_map, bar_in_full + 8 * q, 2 * x0, y0,
                      2 * q, n);
        }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer ----------------
    // The whole warp runs this loop convergently so every address / descriptor stays in uniform
    // registers; one elected lane issues the tcgen05 instructions (the same lane every time, so
    // its commits track all of its MMAs).
    const bool leader = elect_one();
    const long long clk0 = a.clk_out ? clock64() : 0;
    const unsigned long long ns0 = a.clk_out ? global_timer_ns() : 0ull;
    constexpr uint32_t idesc_n = make_idesc(F::kIdescFmt, 128, CO_PAD);
    constexpr uint32_t idesc_w = make_idesc(F::kIdescFmt, 128, Cfg::kAccN);      // SPLIT3: the wide a_hi pass
    // descriptor templates: only the 14-bit start-address field changes per instruction
    const uint64_t adesc0 = make_smem_desc(in_buf, Cfg::kChunkPitch, Cfg::kRowPitch);
    const uint64_t bdesc0_n = make_smem_desc(w_buf, CO_PAD * 16, 128);
    const uint64_t bdesc0_w = make_smem_desc(w_buf, Cfg::kAccN * 16, 128);
    uint32_t st = 0, ph = 0;
    int it = 0;
    for (int u = first; u < a.num_units; u += stride, ++it) {
      const uint32_t s = it & 1;
      const uint32_t acc = tmem_base + s * Cfg::kAccCols;
      mbar_wait_warp(bar_acc_empty + 8 * s, ((it >> 1) & 1) ^ 1);
      tc_fence_after();
      for (int wq = 0; wq < NW; ++wq) {
        // window part used by weight k-step wq; SPLIT3 order per 16-channel group: (a_hi, [w_hi | w_lo]), (a_lo, w_hi)
        const int q = SPLIT3 ? ((wq & 1) ? KSTEPS + (wq >> 1) : (wq >> 1)) : wq;
        const bool wide = SPLIT3 && !(wq & 1);
        const uint32_t idesc = wide ? idesc_w : idesc_n;
        const uint64_t bdesc0 = wide ? bdesc0_w : bdesc0_n;
        const uint32_t tapb = wide ? Cfg::kTapBytesWide : Cfg::kTapBytes;
        mbar_wait_warp(bar_in_full + 8 * q, it & 1);
        const uint64_t adesc_q = adesc0 + static_cast<uint64_t>((q * Cfg::kPartBytes) >> 4);
        uint32_t tap_off = 0;            // (dy * kRowPitch + dx * 16) >> 4, advanced incrementally
        uint32_t dx = 0;
        if constexpr (Cfg::kPairTap) {
          // ---- paired-tap schedule (see TcConvCfg::kPairTap): stage = blocks (2 sg', 2 sg' + 1) of filter row dy ----
          constexpr uint32_t idesc_p = make_idesc(F::kIdescFmt, 128, 128);
          const uint64_t bdesc0_p = make_smem_desc(w_buf, 2048, 128);      // block: chunk pitch 2 KB, 128 rows
          for (int sg = 0; sg < Cfg::kStagesPerKstep; ++sg) {
            const int dy = sg >> 2, sb = sg & 3;
            mbar_wait_warp(bar_w_full + 8 * st, ph);
            tc_fence_after();
            const uint64_t a_row = adesc_q + static_cast<uint64_t>((dy * Cfg::kRowPitch) >> 4);
            const uint64_t b_st = bdesc0_p + static_cast<uint64_t>((st * Cfg::kStageBytes) >> 4);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int blk = 2 * sb + h;
              const uint64_t b_blk = b_st + static_cast<uint64_t>((h * Cfg::kPairBlockBytes) >> 4);
              if (blk == 0) {
                // tap 7 alone, every tile: the first instructions of a unit (they overwrite the accumulators)
                const uint32_t accum = (wq | dy) != 0;
#pragma unroll
                for (int t = 0; t < 4; ++t)
                  if (leader) mma_bf16_ss(acc + t * 64, a_row + static_cast<uint64_t>(8 * t + 7), b_blk, idesc_n, accum);
              } else {
                const int pdx = blk - 1;      // rows 0-63 of the block: tap pdx + 8, rows 64-127: tap pdx
                if (leader) {
                  // tile 0 has no left neighbour for its low taps, tile 3 no right neighbour for its high taps
                  mma_bf16_ss(acc, a_row + static_cast<uint64_t>(pdx), b_blk + (1024 >> 4), idesc_n, 1u);
#pragma unroll
                  for (int t = 1; t < 4; ++t)
                    mma_bf16_ss(acc + (t - 1) * 64, a_row + static_cast<uint64_t>(8 * t + pdx), b_blk, idesc_p, 1u);
                  mma_bf16_ss(acc + 3 * 64, a_row + static_cast<uint64_t>(24 + pdx + 8), b_blk, idesc_n, 1u);
                }
              }
            }
            if (leader) tc_commit(bar_w_empty + 8 * st);
            if (++st == WSTAGES) { st = 0; ph ^= 1; }
          }
        } else
        for (int sg = 0; sg < Cfg::kStagesPerKstep; ++sg) {
          mbar_wait_warp(bar_w_full + 8 * st, ph);
          tc_fence_after();
          const uint64_t bdesc_st = bdesc0 + static_cast<uint64_t>((st * Cfg::kStageBytes) >> 4);
#pragma unroll
          for (int g = 0; g < G; ++g) {
            const uint64_t bdesc = bdesc_st + static_cast<uint64_t>((g * tapb) >> 4);
            const uint64_t adesc_tap = adesc_q + tap_off;
            const uint32_t accum = (wq | sg | g) != 0;
#pragma unroll
            for (int t = 0; t < TILES_X; ++t) {
              if (leader) mma_bf16_ss(acc + t * Cfg::kAccN, adesc_tap + static_cast<uint64_t>(t * 8), bdesc, idesc, accum);
            }
            // next tap: dx+1, wrapping to the next filter row
            if (++dx == S) { dx = 0; tap_off += (Cfg::kRowPitch - (S - 1) * 16) >> 4; }
            else tap_off += 1;
          }
          if (leader) tc_commit(bar_w_empty + 8 * st);
          if (++st == WSTAGES) { st = 0; ph ^= 1; }
        }
        if (leader) tc_commit(bar_in_empty + 8 * q);
      }
      if (leader) tc_commit(bar_acc_full + 8 * s);
    }
    if (a.clk_out && leader) {
      a.clk_out[2 * blockIdx.x] = static_cast<unsigned long long>(clock64() - clk0);
      a.clk_out[2 * blockIdx.x + 1] = global_timer_ns() - ns0;
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ---------------- epilogue: TMEM -> registers -> fp32 NHWC ----------------
    const int ew = warp & 3;                      // TMEM lane quarter this warp may access
    const int m = ew * 32 + lane;                 // accumulator row = pixel within the M tile
    const int prow = m >> 3, pcol = m & 7;
    int it = 0;
    uint32_t gate_uses = 0;
    (void)gate_uses;
    for (int u = first; u < a.num_units; u += stride, ++it) {
      const uint32_t s = it & 1;
      const int nl = u / units_per_frame;
      const int r = u - nl * units_per_frame;
      const int n = a.n0 + nl;
      const int uy = r / a.units_x, ux = r - uy * a.units_x;
      const int y = uy * kTileRows + prow;
      if constexpr (FUSE) {
        if (a.wait_flags) {
          // chained launch: the state tensors of this frame are final once its units of the previous launch are done
          if (lane == 0)
            while (ld_acquire_gpu(a.wait_flags + n) < a.flag_target) {}
          __syncwarp();
        }
      }
      mbar_wait(bar_acc_full + 8 * s, (it >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int t = 0; t < TILES_X; ++t) {
        const int x = ux * (8 * TILES_X) + t * 8 + pcol;
        const bool ok = (y < a.H) && (x < a.W);
        const uint32_t taddr =
            tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + s * Cfg::kAccCols + t * Cfg::kAccN;
        if constexpr (FUSE) {
          // integration in 16-channel pieces (accumulator columns, global inputs and parameters of one piece live
          // at a time); the new state stays in registers for the gate that follows
          const size_t pin = static_cast<size_t>(y) * a.W + x;
          float hv[CO_PAD];
#pragma unroll
          for (int c0 = 0; c0 < CO_PAD; c0 += 16) {
            typename Epi::template Pre<16> pre;
            if (ok) Epi::template load<16>(a, n, pin, c0, pre);
            uint32_t v[16];
            tmem_ld16(taddr + c0, v);
            tmem_ld_wait();
            float acc[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) { acc[j] = __uint_as_float(v[j]); hv[c0 + j] = 0.f; }
            if (ok) Epi::template finish<16>(a, n, pin, c0, acc, pre, hv + c0);
          }
          if (a.do_gate) {
            // ---- fused gate: new state -> 16-bit (F) staging tile -> 1x1 conv on the tensor core -> sigmoid ----
            uint8_t* stg = smem_raw + (gate_a - smem_u32(smem_raw));
#pragma unroll
            for (int i = 0; i < CO_PAD / 8; ++i) {
              typename F::T2 h[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) h[q] = F::cvt2(hv[8 * i + 2 * q], hv[8 * i + 2 * q + 1]);
              *reinterpret_cast<uint4*>(stg + i * 2048 + m * 16) = *reinterpret_cast<const uint4*>(h);
            }
            fence_proxy_async();          // staging writes -> visible to the async (tensor core) proxy
            tc_fence_before();            // our tcgen05.ld of this tile's columns precede the barrier
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (warp == 4) {
              // the tile's own accumulator columns are drained: the gate pre-activations land there
              const bool leader = elect_one();
              tc_fence_after();
              if (leader) {
                constexpr uint32_t gdesc = make_idesc(F::kIdescFmt, 128, CO_PAD);
                const uint64_t ad = make_smem_desc(gate_a, 2048, 128);
                const uint64_t bd = make_smem_desc(gate_w, CO_PAD * 16, 128);
#pragma unroll
                for (int q = 0; q < KSTEPS; ++q)
                  mma_bf16_ss(tmem_base + s * Cfg::kAccCols + t * Cfg::kAccN, ad + static_cast<uint64_t>((q * 2 * 2048) >> 4),
                              bd + static_cast<uint64_t>((q * 2 * CO_PAD * 16) >> 4), gdesc, q != 0);
                tc_commit(bar_gate);
              }
              __syncwarp();
            }
            mbar_wait(bar_gate, gate_uses & 1);
            ++gate_uses;
            tc_fence_after();
#pragma unroll
            for (int c0 = 0; c0 < CO_PAD; c0 += 16) {
              uint32_t v[16];
              tmem_ld16(taddr + c0, v);
              tmem_ld_wait();
              float gacc[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) gacc[j] = __uint_as_float(v[j]);
              if (ok) Epi::template gate<16>(a, n, pin, c0, gacc, hv + c0);
            }
          }
        } else {
        float acc[CO_PAD];
#pragma unroll
        for (int c0 = 0; c0 < CO_PAD; c0 += 16) {
          uint32_t v[16];
          tmem_ld16(taddr + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) acc[c0 + j] = __uint_as_float(v[j]);
          if constexpr (SPLIT3) {      // + the a_hi * w_lo products accumulated in columns [CO, 2 CO)
            tmem_ld16(taddr + CO_PAD + c0, v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) acc[c0 + j] += __uint_as_float(v[j]);
          }
        }
        if (ok) Epi::template apply<CO_PAD>(a, n, y, x, acc);
        }
      }
      tc_fence_before();
      mbar_arrive(bar_acc_empty + 8 * s);
      if constexpr (FUSE) {
        if (a.done_flags) {
          // all epilogue stores of this unit are issued: publish them, then count the unit as done
          asm volatile("bar.sync 2, 128;" ::: "memory");
          if (threadIdx.x == 128) {
            __threadfence();
            atomicAdd(a.done_flags + n, 1);
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace hgru
