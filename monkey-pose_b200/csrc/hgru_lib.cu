// libhgru_b200.so -- plans, parameter packing, kernel orchestration and the C ABI declared in
// include/hgru_b200.h.  Pure CUDA runtime; no framework types cross this boundary.
#include "lib_common.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "crop.cuh"
#include "gate_tc.cuh"
#include "gemm_tc.cuh"
#include "post.cuh"
#include "hconv_tc.cuh"
#include "layers.cuh"
#include "simt_kernels.cuh"
#include <algorithm>
#include <array>

#include "attn.cuh"
#include "tc_host.cuh"

namespace {
thread_local std::string g_err;
int g_timing = 0;
}  // namespace

namespace hgru_host {
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
}  // namespace hgru_host

using namespace hgru_host;

// the frame count of a *_batch forward: 1 <= n <= N, the capacity the plan was created with
static int check_batch(const char* fn, int n, int N) {
  if (n >= 1 && n <= N) return 0;
  return fail(HGRU_E_INVALID, std::string(fn) + ": n = " + std::to_string(n) + " is outside [1, " + std::to_string(N) +
                                  "], the plan's capacity");
}

namespace {

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  int alloc(size_t b) {
    bytes = b;
    cudaError_t e = cudaMalloc(&p, b ? b : 16);
    if (e != cudaSuccess) return fail(HGRU_E_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
  }
  template <class T> T* as() const { return static_cast<T*>(p); }
};

// ---------------------------------------------------------------- 1x1 gate convs (light kernel)
template <int KP, class Epi>
int launch_gate(const __nv_bfloat16* act, const hgru::TcConvArgs& a, cudaStream_t st) {
  using Cfg = hgru::GateCfg<KP>;
  const int tiles_per_frame = (a.H * a.W + 127) / 128;
  hgru::gate_tc_kernel<KP, Epi><<<a.N * tiles_per_frame, 128, Cfg::SMEM_BYTES, st>>>(act, a);
  CUDA_TRY(cudaGetLastError());
  return 0;
}
template <class Epi>
int dispatch_gate(int KP, const __nv_bfloat16* act, const hgru::TcConvArgs& a, cudaStream_t st) {
  if (KP == 64) return launch_gate<64, Epi>(act, a, st);
  if (KP == 32) return launch_gate<32, Epi>(act, a, st);
  if (KP == 16) return launch_gate<16, Epi>(act, a, st);
  return fail(HGRU_E_UNSUPPORTED, "tensor-core gate: unsupported padded channel count");
}

template <int S>
int launch_simt_conv(const float* in, const float* w, const float* bias, const float* scale,
                     const float* shift, float* out, int N, int H, int W, int Ci, int Co, int relu,
                     cudaStream_t st) {
  using Cfg = hgru::ConvSimtCfg<S>;
  auto kern = hgru::conv_simt_kernel<S>;
  SMEM_ATTR_ONCE(kern, Cfg::kSmemBytes);
  dim3 grid(((W + 15) / 16) * ((H + 15) / 16), (Co + 63) / 64, N);
  kern<<<grid, 256, Cfg::kSmemBytes, st>>>(in, w, bias, scale, shift, out, N, H, W, Ci, Co, relu);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int dispatch_simt_conv(int S, const float* in, const float* w, const float* bias, const float* scale,
                       const float* shift, float* out, int N, int H, int W, int Ci, int Co, int relu,
                       cudaStream_t st) {
  switch (S) {
    case 1: return launch_simt_conv<1>(in, w, bias, scale, shift, out, N, H, W, Ci, Co, relu, st);
    case 3: return launch_simt_conv<3>(in, w, bias, scale, shift, out, N, H, W, Ci, Co, relu, st);
    case 5: return launch_simt_conv<5>(in, w, bias, scale, shift, out, N, H, W, Ci, Co, relu, st);
    case 7: return launch_simt_conv<7>(in, w, bias, scale, shift, out, N, H, W, Ci, Co, relu, st);
    case 9: return launch_simt_conv<9>(in, w, bias, scale, shift, out, N, H, W, Ci, Co, relu, st);
    case 11: return launch_simt_conv<11>(in, w, bias, scale, shift, out, N, H, W, Ci, Co, relu, st);
    case 13: return launch_simt_conv<13>(in, w, bias, scale, shift, out, N, H, W, Ci, Co, relu, st);
    case 15: return launch_simt_conv<15>(in, w, bias, scale, shift, out, N, H, W, Ci, Co, relu, st);
    default: return fail(HGRU_E_UNSUPPORTED, "conv: filter size must be odd and <= 15");
  }
}

// copies a [rows][k] (or [k]) fp32 device array into a zero-padded [rows][KP] one
__global__ void pad_matrix_kernel(const float* in, float* out, int rows, int k, int KP, int rows_pad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows_pad * KP) return;
  const int c = i % KP, r = i / KP;
  out[i] = (r < rows && c < k) ? in[static_cast<size_t>(r) * k + c] : 0.f;
}
// HWIO [taps][k][k] -> [taps][KP][KP] zero padded
__global__ void pad_hwio_kernel(const float* in, float* out, int taps, int k, int KP) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= static_cast<size_t>(taps) * KP * KP) return;
  const int co = i % KP;
  const int ci = (i / KP) % KP;
  const int t = i / (static_cast<size_t>(KP) * KP);
  out[i] = (ci < k && co < k) ? in[(static_cast<size_t>(t) * k + ci) * k + co] : 0.f;
}

struct KernelTimer {
  std::vector<cudaEvent_t> ev;
  int used = 0;
  int kernels = 0;        // horizontal-conv launches inside the recorded intervals
  bool open = false;
  void begin(cudaStream_t st) {
    if (!g_timing || open) return;
    open = true;
    while (static_cast<int>(ev.size()) < used + 2) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      ev.push_back(e);
    }
    cudaEventRecord(ev[used], st);
  }
  void end(cudaStream_t st, int n = 1) {
    if (!g_timing || !open) return;
    cudaEventRecord(ev[used + 1], st);
    used += 2;
    kernels += n;
    open = false;
  }
  void reset() { used = 0; kernels = 0; open = false; }
  int collect(float* total_ms) {
    float t = 0.f;
    for (int i = 0; i + 1 < used; i += 2) {
      cudaEventSynchronize(ev[i + 1]);
      float ms = 0.f;
      cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
      t += ms;
    }
    *total_ms = t;
    return used ? kernels : 0;
  }
  ~KernelTimer() {
    for (auto e : ev) cudaEventDestroy(e);
  }
};

}  // namespace

// =================================================================================================
// hGRU plan
// =================================================================================================
struct hgru_plan_s {
  int N, H, W, k, KP, CG, S, T, mode;   // N: capacity, the frames every buffer and tensor map is sized for
  size_t npix, nelem;        // pixels, padded elements (of N frames)
  int n = 0;                 // frames of the current (or last) forward, 1 <= n <= N: the first n frames of every buffer
  bool params_set = false;
  int launches = 0;
  // parameters (zero padded to KP)
  DevBuf p_r, i_r, o_r, vecs, rho, wpk, wpk_i, wpk_o;   // vecs: 8 x [KP]: i_b o_b beta nu gamma kappa omega lateral_bias
  // activations, fp32 [N,H,W,KP]
  DevBuf Xp, H2, H1, C, G, A;
  // bf16 chunked operand copies (tensor-core mode)
  DevBuf actA, actH1, actH2;
  DevBuf flags;                     // launch chaining: [conv launches per timestep x T][N] per-frame completion counters
  DevBuf clk;                       // in-kernel clock samples of the last conv launch: [CTA][2] (cycles, ns)
  bool chain = false;
  CUtensorMap mapA, mapH1;          // SxS halo-window boxes (horizontal convs)
  CUtensorMap mapA_lo, mapH1_lo;    // bf16x3 on the stacked kernel: the lo halves are tensors of their own
  size_t lo_off = 0;                // ... lo_off elements behind the hi tensors
  CUtensorMap mapH1_g, mapH2_g;     // 1x1 boxes (gate convs)
  // readout operand emitted by the last H2 epilogue (set by the pose plan; nullptr for the bare layer)
  __nv_bfloat16* fc_a = nullptr;
  const float* fc_scale = nullptr;
  const float* fc_shift = nullptr;
  int fc_kpad = 0;
  bool stacked = false;             // narrow layers: tap-stacked kernel (hconv_stack.cuh)
  bool fused_tc = false;            // 64 channels, 15x15: hconv_tc_kernel with epilogue-issued gates, chained (FUSE)
  bool epi_gates = false;           // the 1x1 gates run in the conv launches' epilogues (else as launches of their own)
  int stack_T = 0;
  int act_pad = 0;                  // pad rows of the bf16 operand planes (remainder-packed layout)
  bool state_ready = false;         // the caller already ran hgru_init_state_bf16 for the coming forward
  KernelTimer timer;
  // bf16 and fp16 modes: one pipeline (16-bit operands, no hi/lo splits), parameterised by the operand format
  bool op16() const { return mode == HGRU_MODE_BF16 || mode == HGRU_MODE_FP16; }
  OpFormat fmt() const { return mode == HGRU_MODE_FP16 ? FMT_FP16 : FMT_BF16; }
  float* vec(int i) const { return vecs.as<float>() + static_cast<size_t>(i) * KP; }
  size_t npix_n() const { return static_cast<size_t>(n) * H * W; }      // pixels, padded elements of n frames
  size_t nelem_n() const { return npix_n() * KP; }
  // launches per conv: two on the bf16x3 tap-stacked path (EPI_PARTIAL into C, then the launch that adds C), else one
  int conv_parts() const { return mode == HGRU_MODE_BF16X3 && stacked ? 2 : 1; }
  // every device buffer: what workspace() counts is what hgru_plan_free releases
  template <class P> static auto buffers(P* p) {
    return std::array{&p->p_r, &p->i_r, &p->o_r, &p->vecs, &p->rho, &p->wpk, &p->wpk_i, &p->wpk_o, &p->Xp, &p->H2,
                      &p->H1, &p->C, &p->G, &p->A, &p->actA, &p->actH1, &p->actH2, &p->flags, &p->clk};
  }
  size_t workspace() const {
    size_t b = 0;
    for (auto buf : buffers(this)) b += buf->bytes;
    return b;
  }
};

enum { V_IB = 0, V_OB, V_BETA, V_NU, V_GAMMA, V_KAPPA, V_OMEGA, V_LBIAS };

static int hgru_plan_init(hgru_plan_s* p, int N, int H, int W, int k, int S, int T, int mode) {
  if (N < 1 || H < 1 || W < 1 || k < 1 || T < 1) return fail(HGRU_E_INVALID, "hgru_plan_create: non-positive shape");
  if (S < 1 || (S % 2) == 0 || S > 15) return fail(HGRU_E_UNSUPPORTED, "hgru_plan_create: S must be odd and <= 15");
  if (mode != HGRU_MODE_FP32 && mode != HGRU_MODE_BF16 && mode != HGRU_MODE_BF16X3 && mode != HGRU_MODE_FP16)
    return fail(HGRU_E_UNSUPPORTED, "hgru_plan_create: unknown mode");
  // fp16 operands exist for the 15x15 kernels only: tap-stacked (k <= 32) and fused paired-tap (k <= 64)
  if (mode == HGRU_MODE_FP16 && (S != 15 || k > 64))
    return fail(HGRU_E_UNSUPPORTED, "hgru_plan_create: fp16 mode supports S = 15 and k <= 64");
  p->N = N; p->n = N; p->H = H; p->W = W; p->k = k; p->S = S; p->T = T; p->mode = mode;
  p->KP = round_up(k, 16);
  if (mode != HGRU_MODE_FP32 && p->KP == 48) p->KP = 64;      // tensor-core kernels exist for 16 / 32 / 64 padded channels
  // exact path: the 1x1 gate kernel keeps the k x k matrix and a 64-pixel tile in <= 64 KB of shared memory
  if (mode == HGRU_MODE_FP32 && p->KP > 96)
    return fail(HGRU_E_UNSUPPORTED, "hgru_plan_create: fp32 mode supports k <= 96 channels");
  p->CG = p->KP / 8;
  p->npix = static_cast<size_t>(N) * H * W;
  p->nelem = p->npix * p->KP;
  int rc = 0;
  const size_t act = p->nelem * sizeof(float);
  if ((rc = p->Xp.alloc(act)) || (rc = p->H2.alloc(act)) || (rc = p->H1.alloc(act)) ||
      (rc = p->G.alloc(act)))
    return rc;
  if ((rc = p->i_r.alloc(sizeof(float) * p->KP * p->KP)) || (rc = p->o_r.alloc(sizeof(float) * p->KP * p->KP)) ||
      (rc = p->vecs.alloc(sizeof(float) * 8 * p->KP)) || (rc = p->rho.alloc(sizeof(float) * T)))
    return rc;
  if (mode == HGRU_MODE_FP32) {
    if ((rc = p->A.alloc(act)) || (rc = p->C.alloc(act)) ||
        (rc = p->p_r.alloc(sizeof(float) * S * S * p->KP * p->KP)))
      return rc;
    return 0;
  }
  // tensor-core modes: the tap-stacked kernel for narrow 15x15 layers, else hconv_tc_kernel (FUSE at 64 channels in
  // the bf16 / fp16 modes, SPLIT3 in the bf16x3 mode)
  const bool x3 = mode == HGRU_MODE_BF16X3;
  StackGeom sg{};
  TcGeom g{};
  p->stacked = stack_geometry(S, p->KP, k, &sg);
  if (!p->stacked && !(x3 ? x3_geometry(S, p->KP, &g) : tc_geometry(S, p->KP, &g)))
    return fail(HGRU_E_UNSUPPORTED, x3 ? "hgru_plan_create: bf16x3 mode supports S = 15 and k <= 64"
                                      : "hgru_plan_create: bf16 mode supports S in {1,3,5,7,15} and k <= 64");
  p->fused_tc = !x3 && !p->stacked && S == 15 && p->KP == 64;
  // bf16x3 at 32 channels keeps its gates in the exact SIMT kernel: see launch_stack
  p->epi_gates = x3 ? p->stacked && !(p->KP == 32 && sg.T == 4) : p->stacked || p->fused_tc;
  int box_cols = g.box_cols, box_rows = g.box_rows, box_chunks = 2;
  if (p->stacked) {
    p->stack_T = sg.T;
    p->act_pad = sg.act_pad;
    box_cols = sg.box_cols; box_rows = sg.box_rows;
    box_chunks = sg.act_pad ? p->CG / 2 : p->CG;      // remainder-packed kernel loads the window in two parts
  }
  if (p->stacked || p->fused_tc) {
    // consecutive conv launches are chained through per-frame counters (HGRU_NO_CHAIN=1: plain stream order)
    const char* nc = getenv("HGRU_NO_CHAIN");
    p->chain = !(nc && nc[0] == '1');
    const size_t launches = 2 * static_cast<size_t>(p->conv_parts()) * T;
    if (p->chain && (rc = p->flags.alloc(sizeof(int) * launches * N))) return rc;
  }
  // 16-bit operand planes.  bf16x3 carries hi and lo halves: on the stacked kernel two tensors, the lo one lo_off
  // elements behind the hi one (the first launch of a conv reads a_lo, the second a_hi), else 2 * CG chunk planes per
  // frame.  In the remainder-packed layout the planes carry act_pad zero rows on top; they (and the never written tail
  // elements of the row-packed plane) must read as zero, so the buffers are cleared once.
  const int HA = H + p->act_pad;
  const size_t plane = static_cast<size_t>(N) * p->CG * HA * W * 8 * sizeof(__nv_bfloat16);
  const size_t ab = x3 ? 2 * plane : plane;
  if ((rc = p->actA.alloc(ab)) || (rc = p->actH1.alloc(ab)) || (!x3 && (rc = p->actH2.alloc(ab)))) return rc;
  // (cudaMemset on device memory is asynchronous and the kernels run on non-blocking streams: hgru_plan_init's
  // caller synchronises the device once after all clears, see plan_clears_done)
  CUDA_TRY(cudaMemset(p->actA.p, 0, ab));
  CUDA_TRY(cudaMemset(p->actH1.p, 0, ab));
  if (p->conv_parts() == 2) {
    p->lo_off = plane / sizeof(__nv_bfloat16);
    if ((rc = p->C.alloc(act))) return rc;
  }
  // packed weights: the 15x15 (or SxS) conv, and the 1x1 gates where a tensor-core kernel issues them
  const int ksteps = p->KP / 16;
  const size_t tapb = sizeof(__nv_bfloat16) * ksteps * 2 * p->KP * 8;      // one tap, 16-bit operands
  const size_t stack_set = p->stacked ? sizeof(__nv_bfloat16) * sg.stages * sg.NG * 2 * 128 * 8 : 0;
  size_t wbytes = tapb * S * S, gbytes = tapb;
  if (x3) {      // SPLIT3: w_hi and w_lo sets on the stacked kernel, [w_hi, w_lo, w_hi] per k-step else
    wbytes = p->stacked ? 2 * stack_set : 3 * tapb * S * S;
    gbytes = p->stacked ? 3 * tapb : 0;      // ([w_hi | w_lo] wide block + w_hi per 16 input channels)
  } else if (p->stacked) {
    wbytes = stack_set;
  } else if (p->fused_tc) {
    wbytes = sizeof(__nv_bfloat16) * ksteps * 15 * 8 * 2 * 128 * 8;      // paired-tap blocks
  }
  if ((rc = p->wpk.alloc(wbytes))) return rc;
  if (gbytes && ((rc = p->wpk_i.alloc(gbytes)) || (rc = p->wpk_o.alloc(gbytes)))) return rc;
  if (!x3) {
    if ((rc = p->clk.alloc(sizeof(unsigned long long) * 2 * 1024))) return rc;
    CUDA_TRY(cudaMemset(p->clk.p, 0, p->clk.bytes));
  }
  // operand windows of the convs (SxS halo boxes) and, for the separate gate kernels, 1x1 boxes
  char* a0 = static_cast<char*>(p->actA.p);
  char* h0 = static_cast<char*>(p->actH1.p);
  const int planes = x3 && !p->stacked ? 2 * p->CG : p->CG;
  bool bad = hgru::make_act_tensor_map(&p->mapA, a0, N, planes, HA, W, box_cols, box_rows, box_chunks) ||
             hgru::make_act_tensor_map(&p->mapH1, h0, N, planes, HA, W, box_cols, box_rows, box_chunks);
  if (p->conv_parts() == 2)
    bad = bad || hgru::make_act_tensor_map(&p->mapA_lo, a0 + plane, N, planes, HA, W, box_cols, box_rows, box_chunks) ||
          hgru::make_act_tensor_map(&p->mapH1_lo, h0 + plane, N, planes, HA, W, box_cols, box_rows, box_chunks);
  if (!x3) {
    TcGeom g1;
    tc_geometry(1, p->KP, &g1);
    bad = bad || hgru::make_act_tensor_map(&p->mapH1_g, h0, N, p->CG, HA, W, g1.box_cols, g1.box_rows) ||
          hgru::make_act_tensor_map(&p->mapH2_g, p->actH2.p, N, p->CG, HA, W, g1.box_cols, g1.box_rows);
  }
  if (bad) return fail(HGRU_E_CUDA, "cuTensorMapEncodeTiled failed");
  return 0;
}

static void hgru_plan_free(hgru_plan_s* p) {
  for (auto b : hgru_plan_s::buffers(p)) b->release();
}

// weights of the bf16 / fp16 modes in their operand format F: p_r for the plan's 15x15 kernel, i_r and o_r for the
// 1x1 gates
template <class F>
static void pack_op16_weights(hgru_plan_s* p, const float* p_r, const float* i_r, const float* o_r, cudaStream_t st) {
  const int k = p->k, KP = p->KP, taps = p->S * p->S, ksteps = KP / 16;
  auto out = [](DevBuf& b) { return b.as<typename F::T>(); };
  if (p->fused_tc) {
    const size_t tp = static_cast<size_t>(ksteps) * 15 * 8 * 2 * 128 * 8;
    hgru::pack_weights_pairtap_kernel<F><<<nblk(tp), 256, 0, st>>>(p_r, out(p->wpk), k, ksteps);
  } else if (!p->stacked) {
    const size_t total = static_cast<size_t>(ksteps) * taps * 2 * KP * 8;
    hgru::pack_weights_kernel<F><<<nblk(total), 256, 0, st>>>(p_r, out(p->wpk), taps, k, ksteps, KP);
  }
  const size_t t1 = static_cast<size_t>(ksteps) * 2 * KP * 8;
  hgru::pack_weights_kernel<F><<<nblk(t1), 256, 0, st>>>(i_r, out(p->wpk_i), 1, k, ksteps, KP);
  hgru::pack_weights_kernel<F><<<nblk(t1), 256, 0, st>>>(o_r, out(p->wpk_o), 1, k, ksteps, KP);
}

static int hgru_set_params_impl(hgru_plan_s* p, const float* p_r, const float* i_r, const float* i_b,
                                const float* o_r, const float* o_b, const float* beta, const float* nu,
                                const float* gamma, const float* kappa, const float* omega,
                                const float* rho, const float* lateral_bias, cudaStream_t st) {
  const float* ptrs[] = {p_r, i_r, i_b, o_r, o_b, beta, nu, gamma, kappa, omega, rho, lateral_bias};
  for (auto q : ptrs)
    if (!q) return fail(HGRU_E_INVALID, "hgru_set_params: null parameter pointer");
  const int k = p->k, KP = p->KP;
  pad_matrix_kernel<<<nblk(KP * KP), 256, 0, st>>>(i_r, p->i_r.as<float>(), k, k, KP, KP);
  pad_matrix_kernel<<<nblk(KP * KP), 256, 0, st>>>(o_r, p->o_r.as<float>(), k, k, KP, KP);
  const float* v[8] = {i_b, o_b, beta, nu, gamma, kappa, omega, lateral_bias};
  for (int i = 0; i < 8; ++i) pad_matrix_kernel<<<nblk(KP), 256, 0, st>>>(v[i], p->vec(i), 1, k, KP, 1);
  CUDA_TRY(cudaMemcpyAsync(p->rho.p, rho, sizeof(float) * p->T, cudaMemcpyDeviceToDevice, st));
  const int taps = p->S * p->S;
  if (p->mode == HGRU_MODE_FP32) {
    pad_hwio_kernel<<<nblk(static_cast<size_t>(taps) * KP * KP), 256, 0, st>>>(p_r, p->p_r.as<float>(), taps, k, KP);
  } else if (p->mode == HGRU_MODE_BF16X3 && p->stacked) {
    StackGeom sg;
    stack_geometry(p->S, KP, k, &sg);
    const size_t ts = static_cast<size_t>(sg.stages) * sg.NG * 2 * 128 * 8;      // elements of one weight set
    for (int part = 0; part < 2; ++part) {      // set 0 = bf16(w), set 1 = bf16(w - bf16(w))
      int rc = stack_pack_weights(p_r, p->wpk.as<__nv_bfloat16>() + part * ts, k, sg, part, FMT_BF16, st);
      if (rc) return rc;
    }
    const size_t tg = static_cast<size_t>(3 * (KP / 16)) * 2 * KP * 8;
    hgru::pack_weights_split3_kernel<<<nblk(tg), 256, 0, st>>>(i_r, p->wpk_i.as<__nv_bfloat16>(), 1, k, KP / 16, KP);
    hgru::pack_weights_split3_kernel<<<nblk(tg), 256, 0, st>>>(o_r, p->wpk_o.as<__nv_bfloat16>(), 1, k, KP / 16, KP);
  } else if (p->mode == HGRU_MODE_BF16X3) {
    const int ksteps = KP / 16;
    const size_t total = static_cast<size_t>(3 * ksteps) * taps * 2 * KP * 8;
    hgru::pack_weights_split3_kernel<<<nblk(total), 256, 0, st>>>(p_r, p->wpk.as<__nv_bfloat16>(), taps, k, ksteps, KP);
  } else {      // bf16 / fp16
    StackGeom sg;
    if (p->stacked && stack_geometry(p->S, KP, k, &sg)) {
      int rc = stack_pack_weights(p_r, p->wpk.as<__nv_bfloat16>(), k, sg, 0, p->fmt(), st);
      if (rc) return rc;
    }
    if (p->fmt() == FMT_FP16) pack_op16_weights<hgru::OpFp16>(p, p_r, i_r, o_r, st);
    else pack_op16_weights<hgru::OpBf16>(p, p_r, i_r, o_r, st);
  }
  CUDA_TRY(cudaGetLastError());
  p->params_set = true;
  return 0;
}

// API boundary <-> internal state layout (fp32 mode: channel-padded NHWC; bf16 modes: quad-chunked)
static void state_from_nhwc(const hgru_plan_s* p, const float* in, float* out, cudaStream_t st) {
  if (p->mode != HGRU_MODE_FP32)
    hgru::nhwc_to_quad_kernel<<<nblk(p->nelem_n() / 4), 256, 0, st>>>(in, out, p->npix_n(), p->k, p->KP, p->H * p->W);
  else
    hgru::pad_channels_kernel<<<nblk(p->nelem_n()), 256, 0, st>>>(in, out, p->npix_n(), p->k, p->KP);
}
static void state_to_nhwc(const hgru_plan_s* p, const float* in, float* out, cudaStream_t st) {
  if (p->mode != HGRU_MODE_FP32)
    hgru::quad_to_nhwc_kernel<<<nblk(p->npix_n() * p->k), 256, 0, st>>>(in, out, p->npix_n(), p->k, p->KP, p->H * p->W);
  else
    hgru::unpad_channels_kernel<<<nblk(p->npix_n() * p->k), 256, 0, st>>>(in, out, p->npix_n(), p->k, p->KP);
}

// H1 or H2 of timestep t -> its trace [T][n][H][W][k], if there is one (half: H1 of the bf16 / fp16 pipeline with
// epilogue-issued gates, an fp16 oct-chunked tensor)
static void copy_trace(hgru_plan_s* p, const void* src, bool half, float* trace, int t, cudaStream_t st) {
  if (!trace) return;
  float* dst = trace + static_cast<size_t>(t) * p->npix_n() * p->k;
  if (half)
    hgru::oct_half_to_nhwc_kernel<<<nblk(p->npix_n() * p->k), 256, 0, st>>>(static_cast<const __half*>(src), dst,
                                                                              p->npix_n(), p->k, p->KP, p->H * p->W);
  else
    state_to_nhwc(p, static_cast<const float*>(src), dst, st);
  ++p->launches;
}

// ---- fp32 path: SIMT kernels, unfused (the <= 1e-4 anchor) --------------------------------------
static int hgru_run_fp32(hgru_plan_s* p, const float* Xp, float* H1_trace, float* H2_trace, cudaStream_t st) {
  const int KP = p->KP, HW = p->H * p->W;
  const size_t nchunks = p->nelem_n() / 8;
  const size_t gate_smem = sizeof(float) * (KP * KP + 64 * (KP + 1));
  SMEM_ATTR_ONCE(hgru::gate1x1_kernel, 64 * 1024);
  int rc;
  for (int t = 0; t < p->T; ++t) {
    // circuit_input (hgru_module.py:692-724): G1, gated copy, C1 = conv + lateral_bias (:657)
    hgru::gate1x1_kernel<<<nblk(p->npix_n(), 64), 256, gate_smem, st>>>(
        p->H2.as<float>(), p->i_r.as<float>(), p->vec(V_IB), nullptr, p->A.as<float>(), nullptr, p->npix_n(), KP,
        p->k, HW);
    p->timer.begin(st);
    if ((rc = dispatch_simt_conv(p->S, p->A.as<float>(), p->p_r.as<float>(), p->vec(V_LBIAS), nullptr, nullptr,
                                 p->C.as<float>(), p->n, p->H, p->W, KP, KP, 0, st)))
      return rc;
    p->timer.end(st);
    // input_integration (:795-804)
    hgru::h1_kernel<<<nblk(nchunks), 256, 0, st>>>(Xp, p->H2.as<float>(), p->C.as<float>(), p->vec(V_BETA),
                                                  p->vec(V_NU), p->H1.as<float>(), nullptr, nchunks, KP, p->k, HW);
    // circuit_output (:726-756): G2, C2
    hgru::gate1x1_kernel<<<nblk(p->npix_n(), 64), 256, gate_smem, st>>>(
        p->H1.as<float>(), p->o_r.as<float>(), p->vec(V_OB), p->G.as<float>(), nullptr, nullptr, p->npix_n(), KP,
        p->k, HW);
    p->timer.begin(st);
    if ((rc = dispatch_simt_conv(p->S, p->H1.as<float>(), p->p_r.as<float>(), p->vec(V_LBIAS), nullptr, nullptr,
                                 p->C.as<float>(), p->n, p->H, p->W, KP, KP, 0, st)))
      return rc;
    p->timer.end(st);
    // output_integration + rho (:806-823, 847-849)
    hgru::h2_kernel<<<nblk(nchunks), 256, 0, st>>>(p->H1.as<float>(), p->C.as<float>(), p->G.as<float>(),
                                                  p->vec(V_GAMMA), p->vec(V_KAPPA), p->vec(V_OMEGA),
                                                  p->rho.as<float>(), t, p->H2.as<float>(), nchunks, KP, p->k);
    p->launches += 6;
    copy_trace(p, p->H1.p, false, H1_trace, t, st);
    copy_trace(p, p->H2.p, false, H2_trace, t, st);
  }
  return 0;
}

// Initial state of the bf16 / fp16 path: O_0 (NHWC, or zeros) -> H2 (quad-chunked fp32) + the first gated operand.
// Touches only H2 / actA, so it can run before (and concurrently with the input copy of) the stem.
template <int KP, class F>
static int launch_init_tc(const float* h0, const hgru::TcConvArgs& a, cudaStream_t st) {
  using Cfg = hgru::InitCfg<KP>;
  if (KP == 64) SMEM_ATTR_ONCE((hgru::init_state_tc_kernel<KP, F>), Cfg::SMEM_BYTES);
  const int tiles_per_frame = (a.H * a.W + 127) / 128;
  hgru::init_state_tc_kernel<KP, F><<<a.N * tiles_per_frame, 128, Cfg::SMEM_BYTES, st>>>(h0, a);
  CUDA_TRY(cudaGetLastError());
  return 0;
}
template <class F>
static int launch_init_tc(int KP, const float* h0, const hgru::TcConvArgs& a, cudaStream_t st) {
  if (KP == 64) return launch_init_tc<64, F>(h0, a, st);
  if (KP == 32) return launch_init_tc<32, F>(h0, a, st);
  return launch_init_tc<16, F>(h0, a, st);
}

static int hgru_init_state_bf16(hgru_plan_s* p, const float* H2_init_nhwc, cudaStream_t st) {
  // the 1x1 gate conv as one UMMA tile per 128 pixels (16-bit operands like every later gate)
  hgru::TcConvArgs a{};
  a.N = p->n; a.H = p->H; a.W = p->W; a.KP = p->KP; a.kreal = p->k; a.act_pad = p->act_pad;
  a.wpk = p->wpk_i.as<__nv_bfloat16>(); a.bias = p->vec(V_IB); a.H2 = p->H2.as<float>();
  a.out_bf16 = p->actA.as<__nv_bfloat16>();
  return p->fmt() == FMT_FP16 ? launch_init_tc<hgru::OpFp16>(p->KP, H2_init_nhwc, a, st)
                              : launch_init_tc<hgru::OpBf16>(p->KP, H2_init_nhwc, a, st);
}

// The conv launch of one half-step, on the plan's kernel family: c = 0 for C1 + input integration (-> H1), 1 for C2 +
// output integration (-> H2); partial: the first launch of a bf16x3 conv on the stacked kernel (a_lo * w_hi -> C).
static int conv_launch(const hgru_plan_s* p, int c, bool partial, const hgru::TcConvArgs& a, cudaStream_t st) {
  const CUtensorMap& map = c == 0 ? (partial ? p->mapA_lo : p->mapA) : (partial ? p->mapH1_lo : p->mapH1);
  if (p->stacked && p->mode == HGRU_MODE_BF16X3)
    return stack_launch(partial ? EPI_PARTIAL : c ? EPI_H2 : EPI_H1, p->KP, p->stack_T, FMT_BF16, map, a, st);
  // (fused pipeline: H1 and G2 travel to the H2 launch as fp16, EpiH1h / EpiH2h)
  if (p->stacked) return stack_launch(c ? EPI_H2_HALF : EPI_H1_HALF, p->KP, p->stack_T, p->fmt(), map, a, st);
  if (p->fused_tc)
    return c ? tc_fused64_launch<EPI_H2_HALF>(p->fmt(), map, a, st) : tc_fused64_launch<EPI_H1_HALF>(p->fmt(), map, a, st);
  if (p->mode == HGRU_MODE_BF16X3)
    return c ? tc_x3_launch<EPI_H2>(p->S, p->KP, map, a, st) : tc_x3_launch<EPI_H1>(p->S, p->KP, map, a, st);
  return c ? tc_hconv_launch<EPI_H2>(p->S, p->KP, map, a, st) : tc_hconv_launch<EPI_H1>(p->S, p->KP, map, a, st);
}

// A 1x1 gate as a launch of its own (where the conv epilogues do not issue it): c = 0 for circuit_input
// (hgru_module.py:696-711), operand A = F(sigmoid(H2 *1x1 i_r + i_b) . H2); c = 1 for circuit_output (:729-740),
// G2 = sigmoid(H1 *1x1 o_r + o_b).  On tensor cores in the bf16 / fp16 modes, exact fp32 (SIMT) in the bf16x3 mode.
static int gate_launch(hgru_plan_s* p, int c, const hgru::TcConvArgs& base, cudaStream_t st) {
  const int KP = p->KP, HW = p->H * p->W;
  int rc = 0;
  if (p->mode == HGRU_MODE_BF16X3) {
    SMEM_ATTR_ONCE(hgru::gate_quad_split_kernel, 100 * 1024);
    const size_t smem = sizeof(float) * (KP * KP + hgru::kInitPix * (KP + 1));
    const dim3 grid = nblk(p->npix_n(), hgru::kInitPix);
    if (c == 0)
      hgru::gate_quad_split_kernel<<<grid, 256, smem, st>>>(p->H2.as<float>(), p->i_r.as<float>(), p->vec(V_IB), nullptr,
                                                            p->actA.as<__nv_bfloat16>(), p->npix_n(), p->k, KP, HW,
                                                            p->lo_off, p->W, p->act_pad);
    else
      hgru::gate_quad_split_kernel<<<grid, 256, smem, st>>>(p->H1.as<float>(), p->o_r.as<float>(), p->vec(V_OB),
                                                            p->G.as<float>(), nullptr, p->npix_n(), p->k, KP, HW);
  } else {
    hgru::TcConvArgs a = base;
    if (c == 0) {
      a.wpk = p->wpk_i.as<__nv_bfloat16>(); a.bias = p->vec(V_IB); a.H2 = p->H2.as<float>();
      a.out_bf16 = p->actA.as<__nv_bfloat16>();
      rc = dispatch_gate<hgru::EpiGateIn>(KP, p->actH2.as<__nv_bfloat16>(), a, st);
    } else {
      a.wpk = p->wpk_o.as<__nv_bfloat16>(); a.bias = p->vec(V_OB); a.out = p->G.as<float>();
      rc = dispatch_gate<hgru::EpiGateOut>(KP, p->actH1.as<__nv_bfloat16>(), a, st);
    }
  }
  ++p->launches;
  return rc;
}

// ---- tensor-core paths: bf16, fp16 and bf16x3 ------------------------------------------------------------------
// Per timestep: [circuit_input gate], C1 conv + input integration -> H1, [circuit_output gate], C2 conv + output
// integration -> H2, traces.  All integration math happens on TMEM accumulators.  The gates are epilogue-issued MMAs
// inside the conv launches where the plan has epi_gates, else launches of their own.  bf16x3: every conv operand is a
// bf16 hi + lo pair and each k-step is three products (hi*hi + hi*w_lo + lo*w_hi); on the stacked kernel the first
// launch of a conv reads a_lo against w_hi and leaves fp32 sums in C, the second reads a_hi against w_hi and w_lo and
// adds C -- the launch with the heavy epilogue is the one with twice the MMAs to hide it behind.
static int hgru_run_tc(hgru_plan_s* p, const float* Xp, const float* H2_init_nhwc, float* H1_trace, float* H2_trace,
                       cudaStream_t st) {
  int rc;
  // initial state O_0 (NHWC or zeros) -> H2 (quad-chunked fp32).  bf16 / fp16: + the first gated operand, in one pass
  // (unless the caller already ran it: the pose plan overlaps it with the upload of the crops)
  if (p->op16()) {
    if (!p->state_ready && (rc = hgru_init_state_bf16(p, H2_init_nhwc, st))) return rc;
    p->state_ready = false;
  } else if (H2_init_nhwc) {
    state_from_nhwc(p, H2_init_nhwc, p->H2.as<float>(), st);
  } else {
    CUDA_TRY(cudaMemsetAsync(p->H2.p, 0, p->nelem_n() * sizeof(float), st));
  }
  ++p->launches;
  const bool x3 = p->mode == HGRU_MODE_BF16X3;
  const int parts = p->conv_parts();
  hgru::TcConvArgs base{};
  base.N = p->n; base.H = p->H; base.W = p->W; base.KP = p->KP; base.kreal = p->k;
  base.act_pad = p->act_pad; base.lo_off = p->lo_off;
  base.split_out = x3 ? parts : 0;      // bf16x3: hi / lo operand splits, two tensors on the stacked kernel
  // (a weight ring of 5 stages x 3 taps instead of 3 stages x 5 taps for the fused 64-channel kernel measured the
  // same: profiles/r02_bench_k64_fused_ring_5x3taps.json)
  // Chained launches (see TcConvArgs::wait_flags): launch l waits per frame on launch l-1's counters instead of on
  // the whole grid.  Not with traces (their copy kernels sit between the launches), and not where a gate is a launch
  // of its own.
  const bool chain = p->chain && p->epi_gates && !H1_trace && !H2_trace;
  int* flags = chain ? p->flags.as<int>() : nullptr;
  if (chain) CUDA_TRY(cudaMemsetAsync(flags, 0, p->flags.bytes, st));
  // conv c of timestep t; a: the arguments of its (last) launch
  auto conv = [&](int t, int c, const hgru::TcConvArgs& a) -> int {
    // kernel timer: chained, one interval around all launches, counted as 2T passes over the whole batch; else one
    // interval per conv
    if (!chain || (t == 0 && c == 0)) p->timer.begin(st);
    for (int i = 0; i < parts; ++i) {
      const bool partial = i + 1 < parts;
      hgru::TcConvArgs la = a;
      if (partial) {
        la = base;
        la.wpk = p->wpk.as<__nv_bfloat16>(); la.out = p->C.as<float>();
      }
      if (chain) {
        const size_t l = static_cast<size_t>(2 * t + c) * parts + i;
        la.done_flags = flags + l * p->N;
        la.wait_flags = l > 0 ? flags + (l - 1) * p->N : nullptr;
      }
      if (int r = conv_launch(p, c, partial, la, st)) return r;
    }
    if (!chain || (t + 1 == p->T && c == 1)) p->timer.end(st, chain ? 2 * p->T : 1);
    p->launches += parts;
    return 0;
  };
  for (int t = 0; t < p->T; ++t) {
    // at t = 0 the operand comes from the initial-state pass in the bf16 / fp16 modes
    if ((t == 0 ? !p->op16() : !p->epi_gates) && (rc = gate_launch(p, 0, base, st))) return rc;
    // C1 conv (:714-718, 657) + input_integration (:795-804) -> H1 (fp32 + 16-bit operand copy)
    // [epi_gates: + circuit_output gate (:729-740) -> G2]
    hgru::TcConvArgs a = base;
    a.wpk = p->wpk.as<__nv_bfloat16>(); a.partial = parts == 2 ? p->C.as<float>() : nullptr;
    a.bias = p->vec(V_LBIAS); a.X = Xp; a.H2 = p->H2.as<float>(); a.v0 = p->vec(V_BETA); a.v1 = p->vec(V_NU);
    a.out = p->H1.as<float>(); a.out_bf16 = p->actH1.as<__nv_bfloat16>();
    a.gate_wpk = p->wpk_o.as<__nv_bfloat16>(); a.gate_bias = p->vec(V_OB); a.gate_out = p->G.as<float>();
    a.do_gate = p->epi_gates ? 1 : 0;
    if ((rc = conv(t, 0, a))) return rc;
    if (!p->epi_gates && (rc = gate_launch(p, 1, base, st))) return rc;
    // C2 conv (:746-750, 657) + output_integration + rho (:806-823, 847-849) -> H2 in place
    // [epi_gates: + the next timestep's circuit_input gate -> operand A]
    a = base;
    a.wpk = p->wpk.as<__nv_bfloat16>(); a.partial = parts == 2 ? p->C.as<float>() : nullptr;
    a.bias = p->vec(V_LBIAS); a.H1 = p->H1.as<float>(); a.G = p->G.as<float>(); a.H2 = p->H2.as<float>();
    a.v0 = p->vec(V_GAMMA); a.v1 = p->vec(V_KAPPA); a.v2 = p->vec(V_OMEGA);
    a.rho_t = p->rho.as<float>() + t;
    a.out_bf16 = p->epi_gates ? nullptr : p->actH2.as<__nv_bfloat16>();      // (the bf16 / fp16 gate kernel's operand)
    a.gate_wpk = p->wpk_i.as<__nv_bfloat16>(); a.gate_bias = p->vec(V_IB);
    a.gate_act_out = p->actA.as<__nv_bfloat16>();
    a.do_gate = (p->epi_gates && t + 1 < p->T) ? 1 : 0;
    if (t + 1 == p->T) {
      if (g_timing) a.clk_out = p->clk.as<unsigned long long>();      // (bf16 / fp16; grids are <= 1024 CTAs)
      if (p->fc_a) {      // the last update also emits the readout's bf16 hi/lo operand
        a.fc_a = p->fc_a; a.fc_scale = p->fc_scale; a.fc_shift = p->fc_shift; a.fc_kpad = p->fc_kpad;
      }
    }
    if ((rc = conv(t, 1, a))) return rc;
    copy_trace(p, p->H1.p, p->op16() && p->epi_gates, H1_trace, t, st);
    copy_trace(p, p->H2.p, false, H2_trace, t, st);
  }
  return 0;
}

// The recurrence on padded buffers: X = Xp, state in p->H2 (in/out).
static int hgru_run_padded(hgru_plan_s* p, const float* Xp, const float* H2_init_nhwc, float* H1_trace,
                           float* H2_trace, cudaStream_t st) {
  if (!p->params_set) return fail(HGRU_E_STATE, "hgru_forward before hgru_set_params");
  p->launches = 0;
  p->timer.reset();
  int rc;
  if (p->mode != HGRU_MODE_FP32) {
    rc = hgru_run_tc(p, Xp, H2_init_nhwc, H1_trace, H2_trace, st);
  } else {
    if (H2_init_nhwc) state_from_nhwc(p, H2_init_nhwc, p->H2.as<float>(), st);
    else CUDA_TRY(cudaMemsetAsync(p->H2.p, 0, p->nelem_n() * sizeof(float), st));
    rc = hgru_run_fp32(p, Xp, H1_trace, H2_trace, st);
  }
  if (rc) return rc;
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// =================================================================================================
// pose plan
// =================================================================================================
struct pose_plan_s {
  int N, HW, C, KP, S, T, F, O, mode;
  bool params_set = false;
  int launches = 0;
  int nsplit = 16;
  hgru_plan_s hg;
  DevBuf depth, pool1, conv2, w1, b1, w2, b2, w3, b3, fc1_w, fc1_b, fc2_w, fc2_b, bn, part, fc1, out;
  DevBuf act_pool1, act_conv2, wpk2, wpk3;         // tensor-core stem
  CUtensorMap map_pool1, map_conv2;
  bool h0_identity = false;                        // hidden_init='identity': the initial state is conv3 (hgru_module.py:876-878)
  DevBuf h0_tmp;                                   // ... in the reference's layout, filled after the stem
  DevBuf fc1_wt, fc1_a;                            // tensor-core fc_1: bf16 [F][K] weights, bf16 [N][K] input
  CUtensorMap map_fc_a, map_fc_b;
  bool fc1_tc = false;
  int fc_splits = 1, fc_kbps = 1, fc_kpad = 0;
  cudaStream_t copy_st = nullptr;                  // pose_forward_host: upload of the crops overlaps the initial-state pass
  cudaEvent_t ev_begin = nullptr;
  static constexpr int kUploadChunks = 4;          // the crops are uploaded in frame chunks; the stem follows chunk by chunk
  static constexpr int kUploadChunkFrames = 32;    // ... of at least this many frames (smaller launches are latency-bound)
  cudaEvent_t ev_chunk[kUploadChunks] = {};
  cudaStream_t side_st = nullptr;                  // the initial-state pass runs beside the stem (independent inputs)
  cudaEvent_t ev_fork = nullptr, ev_init = nullptr;
  float* bn_scale(int i) const { return bn.as<float>() + static_cast<size_t>(i) * 2 * bnw; }
  float* bn_shift(int i) const { return bn_scale(i) + bnw; }
  int bnw = 0;
  // every device buffer besides the hGRU plan's: what workspace() counts is what pose_plan_free releases
  template <class P> static auto buffers(P* p) {
    return std::array{&p->depth, &p->pool1, &p->conv2, &p->w1, &p->b1, &p->w2, &p->b2, &p->w3, &p->b3,
                      &p->fc1_w, &p->fc1_b, &p->fc2_w, &p->fc2_b, &p->bn, &p->part, &p->fc1, &p->out,
                      &p->act_pool1, &p->act_conv2, &p->wpk2, &p->wpk3, &p->fc1_wt, &p->fc1_a, &p->h0_tmp};
  }
  size_t workspace() const {
    size_t b = hg.workspace();
    for (auto buf : buffers(this)) b += buf->bytes;
    return b;
  }
};

static void pose_plan_free(pose_plan_s* p) {
  hgru_plan_free(&p->hg);
  if (p->copy_st) cudaStreamDestroy(p->copy_st);
  if (p->ev_begin) cudaEventDestroy(p->ev_begin);
  for (auto e : p->ev_chunk) if (e) cudaEventDestroy(e);
  if (p->side_st) cudaStreamDestroy(p->side_st);
  if (p->ev_fork) cudaEventDestroy(p->ev_fork);
  if (p->ev_init) cudaEventDestroy(p->ev_init);
  for (auto b : pose_plan_s::buffers(p)) b->release();
}

// A forward over the first n frames of the plan (n <= N; buffers, tensor maps and the chaining counters keep the
// capacity N as their size and stride).  Every per-forward size derives from n, so the result equals that of a plan
// created for n frames, bit for bit.
static int pose_forward_impl(pose_plan_s* p, int n, const float* depth, const float* H2_init, float* out,
                             cudaStream_t st, const cudaEvent_t* chunk_ready = nullptr, int nchunks = 1) {
  if (!p->params_set) return fail(HGRU_E_STATE, "pose_forward before pose_set_params");
  if (!depth || !out) return fail(HGRU_E_INVALID, "pose_forward: null pointer");
  hgru_plan_s* h = &p->hg;
  h->n = n;
  const int HW = p->HW, KP = p->KP, C = p->C;
  const bool tc = p->mode != HGRU_MODE_FP32;      // stem + fc_1 on tensor cores (hi/lo splits) in both bf16 modes
  int rc;
  p->launches = 0;
  if (p->h0_identity && !p->h0_tmp.p) {
    if (int r = p->h0_tmp.alloc(static_cast<size_t>(p->N) * HW * HW * C * sizeof(float))) return r;
  }
  if (h->op16() && !p->h0_identity) {
    // the hGRU's initial-state pass does not depend on the crops: run it first (under their upload, when the
    // caller copies them on another stream)
    // ... and beside the stem: both are latency-bound passes of ~0.1 ms that leave most of the chip idle
    if (!p->side_st) {
      CUDA_TRY(cudaStreamCreateWithFlags(&p->side_st, cudaStreamNonBlocking));
      CUDA_TRY(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&p->ev_init, cudaEventDisableTiming));
    }
    CUDA_TRY(cudaEventRecord(p->ev_fork, st));            // after everything earlier in `st` (the previous forward)
    CUDA_TRY(cudaStreamWaitEvent(p->side_st, p->ev_fork, 0));
    if ((rc = hgru_init_state_bf16(h, H2_init, p->side_st))) return rc;
    CUDA_TRY(cudaEventRecord(p->ev_init, p->side_st));
    h->state_ready = true;
  }
  // conv_1 + relu + pool_1 + BN (hgru_pose.py:50-60), conv_2 + relu + BN (:61-70), conv_3 + relu + BN (:71-80; its
  // output is X of the hGRU).  Frames are independent, so with a chunked upload (pose_forward_host) the stem of a
  // chunk runs as soon as the chunk has landed, under the upload of the next one; per-frame results do not depend
  // on the chunking.
  const int per = (n + nchunks - 1) / nchunks;
  const size_t pix = static_cast<size_t>(HW) * HW;
  auto conv1 = [&](int n0, int nn) {
    float* o32 = tc ? nullptr : p->pool1.as<float>() + static_cast<size_t>(n0) * pix * KP;
    __nv_bfloat16* o16 = tc ? p->act_pool1.as<__nv_bfloat16>() + static_cast<size_t>(n0) * 2 * KP * pix : nullptr;
    hgru::stem_conv1_pool_bn_kernel<<<dim3(nblk(static_cast<size_t>(nn) * HW * ((HW + hgru::kStemPix - 1) / hgru::kStemPix)), KP / 8),
                                      256, 0, st>>>(
        depth + static_cast<size_t>(n0) * 4 * pix, p->w1.as<float>(), p->b1.as<float>(), p->bn_scale(0), p->bn_shift(0),
        o32, o16, nn, HW, HW, C, KP, tc ? 1 : 0);
    ++p->launches;
  };
  auto conv23_tc = [&](int n0, int nn) -> int {
    hgru::TcConvArgs a{};
    a.N = nn; a.n0 = n0; a.H = HW; a.W = HW; a.KP = KP; a.kreal = C;
    a.wpk = p->wpk2.as<__nv_bfloat16>(); a.bias = p->b2.as<float>();
    a.scale = p->bn_scale(1); a.shift = p->bn_shift(1);
    a.out = nullptr; a.out_bf16 = p->act_conv2.as<__nv_bfloat16>();      // (no fp32 copy: see pose_plan_create)
    int r = tc_stem_launch(KP, p->map_pool1, a, st);
    if (r) return r;
    a.wpk = p->wpk3.as<__nv_bfloat16>(); a.bias = p->b3.as<float>();
    a.scale = p->bn_scale(2); a.shift = p->bn_shift(2);
    a.out = h->Xp.as<float>(); a.out_bf16 = nullptr;
    p->launches += 2;
    return tc_stem_launch(KP, p->map_conv2, a, st);
  };
  for (int c = 0; c < nchunks; ++c) {
    const int n0 = c * per, nn = (n0 + per <= n ? per : n - n0);
    if (nn <= 0) break;
    if (chunk_ready) CUDA_TRY(cudaStreamWaitEvent(st, chunk_ready[c], 0));
    conv1(n0, nn);
    if (tc && (rc = conv23_tc(n0, nn))) return rc;
  }
  if (!tc) {
    if ((rc = dispatch_simt_conv(3, p->pool1.as<float>(), p->w2.as<float>(), p->b2.as<float>(), p->bn_scale(1),
                                 p->bn_shift(1), p->conv2.as<float>(), n, HW, HW, KP, KP, 1, st)))
      return rc;
    if ((rc = dispatch_simt_conv(3, p->conv2.as<float>(), p->w3.as<float>(), p->b3.as<float>(), p->bn_scale(2),
                                 p->bn_shift(2), h->Xp.as<float>(), n, HW, HW, KP, KP, 1, st)))
      return rc;
    p->launches += 2;
  }
  // hGRU (:81, R-D4)
  if (p->fc1_tc) {   // the last H2 epilogue writes the fc_1 operand directly
    h->fc_a = p->fc1_a.as<__nv_bfloat16>(); h->fc_scale = p->bn_scale(3); h->fc_shift = p->bn_shift(3);
    h->fc_kpad = p->fc_kpad;
  }
  if (p->h0_identity) {      // O_0 = X (hgru_module.py:876-878): conv3 in the reference's layout, then the usual path
    state_to_nhwc(h, h->Xp.as<float>(), p->h0_tmp.as<float>(), st);
    H2_init = p->h0_tmp.as<float>();
    ++p->launches;
  } else if (h->op16()) {
    CUDA_TRY(cudaStreamWaitEvent(st, p->ev_init, 0));      // join the initial-state pass
  }
  if ((rc = hgru_run_padded(h, h->Xp.as<float>(), H2_init, nullptr, nullptr, st))) return rc;
  p->launches += h->launches;
  // BN (:82-90) folded into the A-operand of fc_1 (:91); split-K partial sums
  const int K = HW * HW * C;
  int nsplit = p->nsplit;
  if (p->fc1_tc) {
    hgru::GemmArgs g{n, p->F, K, p->fc_kpad, p->fc_kbps, p->part.as<float>(), 0, 0, 0, 0, 0, 0};
    dim3 grid((p->F + hgru::kGemmBN - 1) / hgru::kGemmBN, (n + hgru::kGemmBM - 1) / hgru::kGemmBM, p->fc_splits);
    hgru::gemm_tc_splitk_kernel<hgru::kGemmBN><<<grid, 256, hgru::kGemmSmemBytes, st>>>(p->map_fc_a, p->map_fc_a, p->map_fc_b, g);
    nsplit = p->fc_splits;
    ++p->launches;
  } else {
    const int kslice = round_up((K + p->nsplit - 1) / p->nsplit, 16);
    dim3 g1((p->F + 63) / 64, (n + 63) / 64, p->nsplit);
    hgru::fc1_splitk_kernel<<<g1, 256, 0, st>>>(h->H2.as<float>(), p->fc1_w.as<float>(), p->bn_scale(3),
                                                p->bn_shift(3), p->part.as<float>(), n, K, p->F, C, KP, kslice);
    ++p->launches;
  }
  // + bias, relu (:92), BN (:95-103), fc_out (:104)
  hgru::fc_tail_kernel<<<n, 256, sizeof(float) * (p->F + hgru::kFcTailScratch), st>>>(
      p->part.as<float>(), nsplit, p->fc1_b.as<float>(), p->bn_scale(4), p->bn_shift(4),
      p->fc2_w.as<float>(), p->fc2_b.as<float>(), p->fc1.as<float>(), out, n, p->F, p->O);
  ++p->launches;      // (one per kernel: the count is checked against the ncu launch list)
  CUDA_TRY(cudaGetLastError());
  return 0;
}

#include "attn_plan.inl"

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

const char* hgru_last_error(void) { return g_err.c_str(); }
int hgru_version(void) { return 100; }
int hgru_enable_kernel_timing(int on) {
  g_timing = on ? 1 : 0;
  return 0;
}

int hgru_plan_create(int N, int H, int W, int k, int S, int T, int mode, hgru_plan_t* out) {
  if (!out) return fail(HGRU_E_INVALID, "hgru_plan_create: out is null");
  *out = nullptr;
  hgru_plan_s* p = new hgru_plan_s();
  int rc = hgru_plan_init(p, N, H, W, k, S, T, mode);
  if (!rc && cudaDeviceSynchronize() != cudaSuccess)      // the workspace clears are done before any stream uses it
    rc = fail(HGRU_E_CUDA, "hgru_plan_create: device synchronisation failed");
  if (rc) {
    hgru_plan_free(p);
    delete p;
    return rc;
  }
  *out = p;
  return 0;
}

int hgru_plan_destroy(hgru_plan_t plan) {
  if (!plan) return 0;
  hgru_plan_free(plan);
  delete plan;
  return 0;
}

int hgru_set_params(hgru_plan_t plan, const float* p_r, const float* i_r, const float* i_b,
                    const float* o_r, const float* o_b, const float* beta, const float* nu,
                    const float* gamma, const float* kappa, const float* omega, const float* rho,
                    const float* lateral_bias, void* stream) {
  if (!plan) return fail(HGRU_E_INVALID, "hgru_set_params: null plan");
  return hgru_set_params_impl(plan, p_r, i_r, i_b, o_r, o_b, beta, nu, gamma, kappa, omega, rho,
                              lateral_bias, static_cast<cudaStream_t>(stream));
}

int hgru_forward(hgru_plan_t p, const float* X, const float* H2_init, float* H2_out, float* H1_trace,
                 float* H2_trace, void* stream) {
  if (!p) return fail(HGRU_E_INVALID, "hgru_forward: null plan");
  return hgru_forward_batch(p, p->N, X, H2_init, H2_out, H1_trace, H2_trace, stream);
}

int hgru_forward_batch(hgru_plan_t p, int n, const float* X, const float* H2_init, float* H2_out, float* H1_trace,
                       float* H2_trace, void* stream) {
  if (!p) return fail(HGRU_E_INVALID, "hgru_forward_batch: null plan");
  if (int rc = check_batch("hgru_forward_batch", n, p->N)) return rc;
  if (!X || !H2_out) return fail(HGRU_E_INVALID, "hgru_forward: null tensor pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  p->n = n;
  state_from_nhwc(p, X, p->Xp.as<float>(), st);
  int rc = hgru_run_padded(p, p->Xp.as<float>(), H2_init, H1_trace, H2_trace, st);
  if (rc) return rc;
  state_to_nhwc(p, p->H2.as<float>(), H2_out, st);
  p->launches += 3;
  CUDA_TRY(cudaGetLastError());
  return 0;
}

size_t hgru_plan_workspace_bytes(hgru_plan_t plan) { return plan ? plan->workspace() : 0; }
int hgru_plan_launch_count(hgru_plan_t plan) { return plan ? plan->launches : 0; }

int pose_plan_create(int N, int HW, int C, int S, int T, int F, int O, int mode, pose_plan_t* out) {
  if (!out) return fail(HGRU_E_INVALID, "pose_plan_create: out is null");
  *out = nullptr;
  if (N < 1 || HW < 1 || C < 1 || F < 1 || O < 1) return fail(HGRU_E_INVALID, "pose_plan_create: non-positive shape");
  pose_plan_s* p = new pose_plan_s();
  p->N = N; p->HW = HW; p->C = C; p->S = S; p->T = T; p->F = F; p->O = O; p->mode = mode;
  int rc = hgru_plan_init(&p->hg, N, HW, HW, C, S, T, mode);
  const int KP = p->hg.KP;
  p->KP = KP;
  p->bnw = F > KP ? F : KP;
  const size_t act = static_cast<size_t>(N) * HW * HW * KP * sizeof(float);
  const size_t K = static_cast<size_t>(HW) * HW * C;
  auto A = [&](DevBuf& b, size_t bytes) { if (!rc) rc = b.alloc(bytes); };
  A(p->depth, static_cast<size_t>(N) * 4 * HW * HW * sizeof(float));
  // fp32 copies of pool1 / conv2 exist only on the exact path: the tensor-core stem consumes bf16 hi/lo operand
  // copies, and pose_get_activation rebuilds the fp32 tensors from those (hi + lo, 16 mantissa bits)
  if (mode == HGRU_MODE_FP32) { A(p->pool1, act); A(p->conv2, act); }
  A(p->w1, sizeof(float) * 9 * C); A(p->b1, sizeof(float) * KP);
  A(p->b2, sizeof(float) * KP); A(p->b3, sizeof(float) * KP);
  // fc_1 on tensor cores (operand rows are padded to whole k-blocks, so any K works)
  p->fc1_tc = (mode != HGRU_MODE_FP32);
  if (p->fc1_tc) {
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int total_kb = static_cast<int>((K + hgru::kGemmBK - 1) / hgru::kGemmBK);
    // The K split depends on K and F only (not on the batch), so a frame's result is bitwise
    // independent of its batch neighbours: ~2 M-tiles x N-tiles x splits CTAs fill the SMs.
    const int ntiles_n = (F + hgru::kGemmBN - 1) / hgru::kGemmBN;
    int splits = sms / (2 * ntiles_n);
    if (splits < 1) splits = 1;
    if (splits > total_kb) splits = total_kb;
    p->fc_kbps = (total_kb + splits - 1) / splits;
    p->fc_splits = (total_kb + p->fc_kbps - 1) / p->fc_kbps;
    p->fc_kpad = total_kb * hgru::kGemmBK;                       // lo halves start here; row pitch 2*Kpad
    const size_t pitch = 2 * static_cast<size_t>(p->fc_kpad);
    A(p->fc1_wt, sizeof(__nv_bfloat16) * pitch * F);
    A(p->fc1_a, sizeof(__nv_bfloat16) * pitch * N);
    if (!rc) {
      cudaMemset(p->fc1_wt.p, 0, p->fc1_wt.bytes);               // pad columns stay zero
      cudaMemset(p->fc1_a.p, 0, p->fc1_a.bytes);
    }
    if (!rc && (hgru::make_kmajor_bf16_map(&p->map_fc_a, p->fc1_a.p, N, pitch, hgru::kGemmBM) ||
                hgru::make_kmajor_bf16_map(&p->map_fc_b, p->fc1_wt.p, F, pitch, hgru::kGemmBN)))
      rc = fail(HGRU_E_CUDA, "cuTensorMapEncodeTiled (fc_1) failed");
    if (!rc && cudaFuncSetAttribute(hgru::gemm_tc_splitk_kernel<hgru::kGemmBN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    hgru::kGemmSmemBytes) != cudaSuccess)
      rc = fail(HGRU_E_CUDA, "cudaFuncSetAttribute(gemm_tc_splitk_kernel) failed");
  } else {
    A(p->fc1_w, sizeof(float) * K * F);
  }
  A(p->fc1_b, sizeof(float) * F);
  A(p->fc2_w, sizeof(float) * F * O); A(p->fc2_b, sizeof(float) * O);
  A(p->bn, sizeof(float) * 5 * 2 * p->bnw);
  A(p->part, sizeof(float) * (p->fc1_tc ? p->fc_splits : p->nsplit) * N * F); A(p->fc1, sizeof(float) * N * F); A(p->out, sizeof(float) * N * O);
  if (mode == HGRU_MODE_FP32) {
    A(p->w2, sizeof(float) * 9 * KP * KP); A(p->w3, sizeof(float) * 9 * KP * KP);
  } else if (!rc) {
    const size_t ab = 2 * static_cast<size_t>(N) * HW * HW * KP * sizeof(__nv_bfloat16);   // hi + lo halves
    A(p->act_pool1, ab); A(p->act_conv2, ab);
    const size_t wb = sizeof(__nv_bfloat16) * (3 * KP / 16) * 9 * 2 * KP * 8;        // [w_hi, w_lo, w_hi] per k-step
    A(p->wpk2, wb); A(p->wpk3, wb);
    TcGeom g;
    if (!rc && !stem_geometry(KP, &g)) rc = fail(HGRU_E_UNSUPPORTED, "pose_plan_create: unsupported channel count for bf16 mode");
    if (!rc && (hgru::make_act_tensor_map(&p->map_pool1, p->act_pool1.p, N, 2 * KP / 8, HW, HW, g.box_cols, g.box_rows) ||
                hgru::make_act_tensor_map(&p->map_conv2, p->act_conv2.p, N, 2 * KP / 8, HW, HW, g.box_cols, g.box_rows)))
      rc = fail(HGRU_E_CUDA, "cuTensorMapEncodeTiled failed");
  }
  if (!rc && cudaDeviceSynchronize() != cudaSuccess)      // the workspace clears are done before any stream uses it
    rc = fail(HGRU_E_CUDA, "pose_plan_create: device synchronisation failed");
  if (rc) {
    pose_plan_free(p);
    delete p;
    return rc;
  }
  *out = p;
  return 0;
}

int pose_plan_destroy(pose_plan_t plan) {
  if (!plan) return 0;
  pose_plan_free(plan);
  delete plan;
  return 0;
}

int pose_set_params(pose_plan_t p, const pose_params_t* q, float eps, void* stream) {
  if (!p || !q) return fail(HGRU_E_INVALID, "pose_set_params: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int C = p->C, KP = p->KP, F = p->F, O = p->O;
  const float* req[] = {q->conv_1_filters, q->conv_1_biases, q->conv_2_filters, q->conv_2_biases,
                        q->conv_3_filters, q->conv_3_biases, q->fc_1_weights, q->fc_1_biases,
                        q->fc_out_weights, q->fc_out_biases};
  for (auto r : req)
    if (!r) return fail(HGRU_E_INVALID, "pose_set_params: null parameter pointer");
  for (int i = 0; i < 5; ++i)
    for (int j = 0; j < 4; ++j)
      if (!q->bn[i][j]) return fail(HGRU_E_INVALID, "pose_set_params: null batch-norm pointer");
  CUDA_TRY(cudaMemcpyAsync(p->w1.p, q->conv_1_filters, sizeof(float) * 9 * C, cudaMemcpyDeviceToDevice, st));
  pad_matrix_kernel<<<nblk(KP), 256, 0, st>>>(q->conv_1_biases, p->b1.as<float>(), 1, C, KP, 1);
  pad_matrix_kernel<<<nblk(KP), 256, 0, st>>>(q->conv_2_biases, p->b2.as<float>(), 1, C, KP, 1);
  pad_matrix_kernel<<<nblk(KP), 256, 0, st>>>(q->conv_3_biases, p->b3.as<float>(), 1, C, KP, 1);
  if (p->mode == HGRU_MODE_FP32) {
    pad_hwio_kernel<<<nblk(static_cast<size_t>(9) * KP * KP), 256, 0, st>>>(q->conv_2_filters, p->w2.as<float>(), 9, C, KP);
    pad_hwio_kernel<<<nblk(static_cast<size_t>(9) * KP * KP), 256, 0, st>>>(q->conv_3_filters, p->w3.as<float>(), 9, C, KP);
  } else {
    const size_t total = static_cast<size_t>(3 * KP / 16) * 9 * 2 * KP * 8;
    hgru::pack_weights_split3_kernel<<<nblk(total), 256, 0, st>>>(q->conv_2_filters, p->wpk2.as<__nv_bfloat16>(), 9,
                                                                 C, KP / 16, KP);
    hgru::pack_weights_split3_kernel<<<nblk(total), 256, 0, st>>>(q->conv_3_filters, p->wpk3.as<__nv_bfloat16>(), 9,
                                                                 C, KP / 16, KP);
  }
  const size_t K = static_cast<size_t>(p->HW) * p->HW * C;
  if (p->fc1_tc) {
    dim3 tg(static_cast<unsigned>((K + 31) / 32), (F + 31) / 32);
    hgru::transpose_operand_kernel<<<tg, 256, 0, st>>>(q->fc_1_weights, p->fc1_wt.as<__nv_bfloat16>(),
                                                     static_cast<int>(K), F, p->fc_kpad, C);
  } else {
    CUDA_TRY(cudaMemcpyAsync(p->fc1_w.p, q->fc_1_weights, sizeof(float) * K * F, cudaMemcpyDeviceToDevice, st));
  }
  CUDA_TRY(cudaMemcpyAsync(p->fc1_b.p, q->fc_1_biases, sizeof(float) * F, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(p->fc2_w.p, q->fc_out_weights, sizeof(float) * F * O, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(p->fc2_b.p, q->fc_out_biases, sizeof(float) * O, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(cudaMemsetAsync(p->bn.p, 0, p->bn.bytes, st));
  for (int i = 0; i < 5; ++i) {
    const int c = (i == 4) ? F : C;
    hgru::bn_fold_kernel<<<nblk(c), 256, 0, st>>>(q->bn[i][0], q->bn[i][1], q->bn[i][2], q->bn[i][3], eps,
                                                  p->bn_scale(i), p->bn_shift(i), c);
  }
  CUDA_TRY(cudaGetLastError());
  int rc = hgru_set_params_impl(&p->hg, q->p_r, q->i_r, q->i_b, q->o_r, q->o_b, q->beta, q->nu, q->gamma,
                                q->kappa, q->omega, q->rho, q->lateral_bias, st);
  if (rc) return rc;
  p->params_set = true;
  return 0;
}

int pose_forward(pose_plan_t p, const float* depth, const float* H2_init, float* out, void* stream) {
  if (!p) return fail(HGRU_E_INVALID, "pose_forward: null plan");
  return pose_forward_impl(p, p->N, depth, H2_init, out, static_cast<cudaStream_t>(stream));
}

int pose_forward_batch(pose_plan_t p, int n, const float* depth, const float* H2_init, float* out, void* stream) {
  if (!p) return fail(HGRU_E_INVALID, "pose_forward_batch: null plan");
  if (int rc = check_batch("pose_forward_batch", n, p->N)) return rc;
  return pose_forward_impl(p, n, depth, H2_init, out, static_cast<cudaStream_t>(stream));
}

int pose_forward_host(pose_plan_t p, const float* depth_host, const float* H2_init, float* out_host, void* stream) {
  if (!p) return fail(HGRU_E_INVALID, "pose_forward_host: null plan");
  return pose_forward_host_batch(p, p->N, depth_host, H2_init, out_host, stream);
}

int pose_forward_host_batch(pose_plan_t p, int n, const float* depth_host, const float* H2_init, float* out_host,
                            void* stream) {
  if (!p) return fail(HGRU_E_INVALID, "pose_forward_host_batch: null plan");
  if (int rc = check_batch("pose_forward_host_batch", n, p->N)) return rc;
  if (!depth_host || !out_host) return fail(HGRU_E_INVALID, "pose_forward_host: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // upload on the plan's copy stream (ordered after the work already queued on `st`), so that the copy engine
  // runs under the initial-state kernel; the stem waits for the copy
  if (!p->copy_st) {
    CUDA_TRY(cudaStreamCreateWithFlags(&p->copy_st, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&p->ev_begin, cudaEventDisableTiming));
    for (auto& e : p->ev_chunk) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  CUDA_TRY(cudaEventRecord(p->ev_begin, st));
  CUDA_TRY(cudaStreamWaitEvent(p->copy_st, p->ev_begin, 0));
  // frame chunks, one event each: conv_1 of chunk c runs while chunk c+1 is still on the bus
  int nchunks = n / pose_plan_s::kUploadChunkFrames;
  nchunks = nchunks < 1 ? 1 : (nchunks > pose_plan_s::kUploadChunks ? pose_plan_s::kUploadChunks : nchunks);
  {
    const int per = (n + nchunks - 1) / nchunks;
    const size_t frame = static_cast<size_t>(4) * p->HW * p->HW;      // floats per 2HW x 2HW crop
    for (int c = 0; c < nchunks; ++c) {
      const int n0 = c * per, nn = (n0 + per <= n ? per : n - n0);
      if (nn > 0)
        CUDA_TRY(cudaMemcpyAsync(p->depth.as<float>() + n0 * frame, depth_host + n0 * frame, nn * frame * sizeof(float),
                                 cudaMemcpyHostToDevice, p->copy_st));
      CUDA_TRY(cudaEventRecord(p->ev_chunk[c], p->copy_st));
    }
  }
  int rc = pose_forward_impl(p, n, p->depth.as<float>(), H2_init, p->out.as<float>(), st, p->ev_chunk, nchunks);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(out_host, p->out.p, sizeof(float) * n * p->O, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}

int pose_set_hidden_init(pose_plan_t p, int identity) {
  if (!p) return fail(HGRU_E_INVALID, "pose_set_hidden_init: null plan");
  p->h0_identity = identity != 0;
  return 0;
}

int pose_get_activation(pose_plan_t p, const char* name, float* dst, void* stream) {
  if (!p || !name || !dst) return fail(HGRU_E_INVALID, "pose_get_activation: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float* src = nullptr;
  const bool is_pool1 = !strcmp(name, "pool1"), is_conv2 = !strcmp(name, "conv2");
  if ((is_pool1 || is_conv2) && p->mode != HGRU_MODE_FP32) {
    // tensor-core stem: the activation lives as bf16 hi | lo chunk planes
    const hgru_plan_s* h = &p->hg;
    hgru::split_chunks_to_nhwc_kernel<<<nblk(h->npix_n() * h->k), 256, 0, st>>>(
        (is_pool1 ? p->act_pool1 : p->act_conv2).as<__nv_bfloat16>(), dst, h->npix_n(), h->k, h->KP / 8, h->H * h->W);
    CUDA_TRY(cudaGetLastError());
    return 0;
  }
  if (is_pool1) src = p->pool1.as<float>();
  else if (is_conv2) src = p->conv2.as<float>();
  else if (!strcmp(name, "conv3")) src = p->hg.Xp.as<float>();
  else if (!strcmp(name, "hgru")) src = p->hg.H2.as<float>();
  else if (!strcmp(name, "fc1")) {
    CUDA_TRY(cudaMemcpyAsync(dst, p->fc1.p, sizeof(float) * p->hg.n * p->F, cudaMemcpyDeviceToDevice, st));
    return 0;
  } else return fail(HGRU_E_INVALID, std::string("pose_get_activation: unknown name ") + name);
  state_to_nhwc(&p->hg, src, dst, st);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

size_t pose_plan_workspace_bytes(pose_plan_t plan) { return plan ? plan->workspace() : 0; }
int pose_plan_launch_count(pose_plan_t plan) { return plan ? plan->launches : 0; }

int pose_plan_sm_clock_ghz(pose_plan_t plan, float* ghz_mean, float* ghz_min) {
  if (!plan || !ghz_mean || !ghz_min) return fail(HGRU_E_INVALID, "pose_plan_sm_clock_ghz: null argument");
  *ghz_mean = *ghz_min = 0.f;
  const hgru_plan_s* h = &plan->hg;
  if (!h->clk.p) return 0;                       // (the exact fp32 path has no tensor-core launch to sample)
  std::vector<unsigned long long> v(h->clk.bytes / sizeof(unsigned long long));
  CUDA_TRY(cudaMemcpy(v.data(), h->clk.p, h->clk.bytes, cudaMemcpyDeviceToHost));   // (synchronises the device)
  double sum = 0.0, mn = 1e30;
  int n = 0;
  for (size_t i = 0; i + 1 < v.size(); i += 2) {
    if (!v[i + 1]) continue;
    const double g = static_cast<double>(v[i]) / static_cast<double>(v[i + 1]);
    sum += g; mn = g < mn ? g : mn; ++n;
  }
  if (n) { *ghz_mean = static_cast<float>(sum / n); *ghz_min = static_cast<float>(mn); }
  return 0;
}

int pose_plan_kernel_times(pose_plan_t plan, float* hconv_ms_total, int* hconv_launches) {
  if (!plan || !hconv_ms_total || !hconv_launches) return fail(HGRU_E_INVALID, "pose_plan_kernel_times: null argument");
  *hconv_launches = plan->hg.timer.collect(hconv_ms_total);
  return 0;
}

int crop_area3d_forward(const float* frames, int N, int H, int W, float frame_scale, const int* ip,
                        const float* zp, float background, double out_divisor, float* out, int dh, int dw,
                        void* stream) {
  if (!frames || !ip || !zp || !out) return fail(HGRU_E_INVALID, "crop_area3d_forward: null pointer");
  if (N < 1 || H < 1 || W < 1 || dh < 1 || dw < 1) return fail(HGRU_E_INVALID, "crop_area3d_forward: non-positive shape");
  if (!(out_divisor > 0.0)) return fail(HGRU_E_INVALID, "crop_area3d_forward: out_divisor must be positive");
  const size_t total = static_cast<size_t>(N) * dh * dw;
  hgru::crop_area3d_kernel<<<nblk(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      frames, frame_scale, ip, zp, background, out_divisor, out, N, H, W, dh, dw);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int depth_preprocess_forward(const unsigned short* raw, size_t count, unsigned int near_mm, unsigned int far_mm,
                             double fill, double max_depth, float* out, void* stream) {
  if (!raw || !out) return fail(HGRU_E_INVALID, "depth_preprocess_forward: null pointer");
  if (count < 1 || !(max_depth > 0.0)) return fail(HGRU_E_INVALID, "depth_preprocess_forward: bad size or divisor");
  hgru::depth_preprocess_kernel<<<nblk(count), 256, 0, static_cast<cudaStream_t>(stream)>>>(raw, count, near_mm, far_mm,
                                                                                         fill, max_depth, out);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int crop_windows_forward(const float* tr, const double* com_in, double s0, double s1, double s2, int N, int H, int W,
                         int dw, int dh, double fx, double fy, double cube_x, double cube_y, double cube_z,
                         double* coms, int* iparams, float* zparams, double* Ms, int* invalid, void* stream) {
  if ((!tr && !com_in) || !coms || !iparams || !zparams || !Ms || !invalid)
    return fail(HGRU_E_INVALID, "crop_windows_forward: null pointer");
  if (N < 1 || H < 1 || W < 1 || dw < 1 || dh < 1) return fail(HGRU_E_INVALID, "crop_windows_forward: non-positive shape");
  hgru::crop_windows_kernel<<<nblk(N, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      tr, com_in, s0, s1, s2, N, H, W, dw, dh, fx, fy, cube_x, cube_y, cube_z, coms, iparams, zparams, Ms, invalid);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// An 8-lane group sums a subtree of 2^leaves_log2 blocks of numpy's pairwise tree (16 when the batch alone fills the
// GPU, 4 for a few frames); only the subtree sums reach the workspace: 2^(L + 1) heap slots per frame, L = the level
// of those subtrees in the tree of the largest image allowed.
// (deeper trees than 12 + that: bigger subtrees, so that the top levels always fit 32 KB of shared memory)
static int com_leaves_log2(int N, long long max_pixels) {
  const int d = hgru::np_pairwise_depth(max_pixels < 1 ? 1 : max_pixels);
  return std::max(N >= 32 ? 4 : 2, d - 12);
}
static int com_top_levels(int N, long long max_pixels, long long pixels) {
  const int d = hgru::np_pairwise_depth(pixels < 1 ? 1 : pixels), l = com_leaves_log2(N, max_pixels);
  return d > l ? d - l : 0;
}
// workspace: [N][4] uint64 statistics, then [N][heap slots] floats
size_t calculate_com_workspace_bytes(int N, long long max_pixels) {
  if (N < 1 || max_pixels < 1 || max_pixels > 0x7fffffffLL) return 0;
  return static_cast<size_t>(N) * (4 * sizeof(unsigned long long) + (2u << com_top_levels(N, max_pixels, max_pixels)) * sizeof(float));
}
int calculate_com_forward(const float* frames, int N, int H, int W, float frame_scale, float min_depth, float max_depth,
                          const int* iparams, const float* zparams, long long max_pixels, void* ws, double* coms,
                          int* overflow, void* stream) {
  if (!frames || !ws || !coms || !overflow) return fail(HGRU_E_INVALID, "calculate_com_forward: null pointer");
  if ((iparams == nullptr) != (zparams == nullptr))
    return fail(HGRU_E_INVALID, "calculate_com_forward: iparams and zparams go together");
  if (N < 1 || H < 1 || W < 1 || N > 65535) return fail(HGRU_E_INVALID, "calculate_com_forward: bad shape (1 <= N <= 65535)");
  if (max_pixels < 1 || max_pixels > 0x7fffffffLL)
    return fail(HGRU_E_INVALID, "calculate_com_forward: max_pixels must be in [1, 2^31)");
  if (!iparams && static_cast<long long>(H) * W > max_pixels)
    return fail(HGRU_E_INVALID, "calculate_com_forward: max_pixels is smaller than a frame");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned long long* stats = static_cast<unsigned long long*>(ws);
  float* heap = reinterpret_cast<float*>(stats + 4 * static_cast<size_t>(N));
  const int leaves_log2 = com_leaves_log2(N, max_pixels);
  const int top = com_top_levels(N, max_pixels, max_pixels);
  const unsigned slots = 2u << top;                               // <= 8192: 32 KB of shared memory in the second kernel
  CUDA_TRY(cudaMemsetAsync(stats, 0, 4 * sizeof(unsigned long long) * static_cast<size_t>(N), st));
  // the grid covers the deepest tree the workspace allows (whole frames: the frame's own); groups beyond a frame's
  // own tree idle
  const int grid_levels = iparams ? top : com_top_levels(N, max_pixels, static_cast<long long>(H) * W);
  const unsigned parts = ((1u << grid_levels) * 8u + 255u) / 256u;
  const dim3 grid(parts, N);
#define HGRU_COM_BLOCKS(WIN, POS)                                                                                   \
  hgru::com_blocks_kernel<WIN, POS><<<grid, 256, 0, st>>>(frames, H, W, frame_scale, min_depth, max_depth, iparams, \
                                                          zparams, heap, slots, leaves_log2, stats)
  if (iparams) { if (min_depth > 0.f) HGRU_COM_BLOCKS(true, true); else HGRU_COM_BLOCKS(true, false); }
  else         { if (min_depth > 0.f) HGRU_COM_BLOCKS(false, true); else HGRU_COM_BLOCKS(false, false); }
#undef HGRU_COM_BLOCKS
  hgru::com_finish_kernel<<<N, 256, slots * sizeof(float), st>>>(frames, H, W, frame_scale, min_depth, max_depth,
                                                                iparams, zparams, heap, slots, leaves_log2, stats, coms,
                                                                overflow);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int pose_postprocess_forward(const float* out_put, const double* com_uvd, int N, int J, double fx, double fy,
                             double ux, double uy, float scale, float* xyz, float* uvd, void* stream) {
  if (!out_put || !com_uvd || !xyz || !uvd) return fail(HGRU_E_INVALID, "pose_postprocess_forward: null pointer");
  if (N < 1 || J < 1) return fail(HGRU_E_INVALID, "pose_postprocess_forward: non-positive shape");
  hgru::pose_postprocess_kernel<<<nblk(static_cast<size_t>(N) * J), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      out_put, com_uvd, N, J, fx, fy, ux, uy, scale, xyz, uvd);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int joint_error_forward(const float* labels, const float* results, int N, int J, double* frame_mean_ws,
                        float* frame_max_ws, double* result, void* stream) {
  if (!labels || !results || !frame_mean_ws || !frame_max_ws || !result)
    return fail(HGRU_E_INVALID, "joint_error_forward: null pointer");
  if (N < 1 || J < 1) return fail(HGRU_E_INVALID, "joint_error_forward: non-positive shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  hgru::joint_error_frame_kernel<<<N, 128, 0, st>>>(labels, results, J, frame_mean_ws, frame_max_ws);
  hgru::joint_error_final_kernel<<<1, 32, 0, st>>>(frame_mean_ws, frame_max_ws, N, result);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int joint_error_stats_forward(const float* labels, const float* results, int N, int J, int skip_nan, float* err,
                              float* frame_mean, float* frame_max, float* joint_mean, float* summary, void* stream) {
  if (!labels || !results || !err || !frame_mean || !frame_max || !joint_mean || !summary)
    return fail(HGRU_E_INVALID, "joint_error_stats_forward: null pointer");
  if (N < 1 || J < 1) return fail(HGRU_E_INVALID, "joint_error_stats_forward: non-positive shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t NJ = static_cast<size_t>(N) * J;
  hgru::joint_error_matrix_kernel<<<nblk(NJ), 256, 0, st>>>(labels, results, NJ, err);
  hgru::joint_error_reduce_kernel<<<nblk(static_cast<size_t>(N) + J, 128), 128, 0, st>>>(err, N, J, skip_nan ? 1 : 0,
                                                                                        frame_mean, frame_max, joint_mean);
  hgru::joint_error_summary_kernel<<<1, 32, 0, st>>>(frame_mean, frame_max, N, skip_nan ? 1 : 0, summary);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int joint_error_count_within_forward(const float* frame_stat, int N, float dist, int* count, void* stream) {
  if (!frame_stat || !count) return fail(HGRU_E_INVALID, "joint_error_count_within_forward: null pointer");
  if (N < 1) return fail(HGRU_E_INVALID, "joint_error_count_within_forward: non-positive shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaMemsetAsync(count, 0, sizeof(int), st));
  hgru::count_within_kernel<<<nblk(N), 256, 0, st>>>(frame_stat, N, dist, count);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int axis1_error_mean_forward(const float* a, const float* b, int N, int M, int C, int skip_nan, float* rows_ws,
                             float* out, void* stream) {
  if (!a || !b || !rows_ws || !out) return fail(HGRU_E_INVALID, "axis1_error_mean_forward: null pointer");
  if (N < 1 || M < 1 || C < 1) return fail(HGRU_E_INVALID, "axis1_error_mean_forward: non-positive shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  hgru::axis1_error_rows_kernel<<<nblk(static_cast<size_t>(N) * C), 256, 0, st>>>(a, b, N, M, C, rows_ws);
  hgru::axis0_mean_kernel<<<nblk(C, 64), 64, 0, st>>>(rows_ws, N, C, skip_nan ? 1 : 0, out);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ---- stand-alone layers (the reference model's layer methods; exact fp32, unfused) -----------------------------
int layer_conv2d_forward(const float* x, int N, int H, int W, int Cin, const float* filters, int S, int Cout,
                         const float* biases, int relu, float* out, void* stream) {
  if (!x || !filters || !biases || !out) return fail(HGRU_E_INVALID, "layer_conv2d_forward: null pointer");
  if (N < 1 || H < 1 || W < 1 || Cin < 1 || Cout < 1) return fail(HGRU_E_INVALID, "layer_conv2d_forward: non-positive shape");
  if (S < 1 || (S % 2) == 0) return fail(HGRU_E_UNSUPPORTED, "layer_conv2d_forward: filter size must be odd");
  const size_t total = static_cast<size_t>(N) * H * W * Cout;
  hgru::conv2d_direct_kernel<<<nblk(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, filters, biases, out, N, H,
                                                                                       W, Cin, Cout, S, relu ? 1 : 0);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int circuit_gate_forward(const float* x, size_t rows, int k, const float* w, const float* b, float* gate, float* gated,
                         void* stream) {
  if (!x || !w || !b || !gate) return fail(HGRU_E_INVALID, "circuit_gate_forward: null pointer");
  if (rows < 1 || k < 1) return fail(HGRU_E_INVALID, "circuit_gate_forward: non-positive shape");
  hgru::circuit_gate_kernel<<<nblk(rows * k), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, w, b, gate, gated, rows, k);
  CUDA_TRY(cudaGetLastError());
  return 0;
}
int circuit_input_integration_forward(const float* X, const float* O, const float* P, const float* beta,
                                      const float* nu, float xi, size_t rows, int k, float* I, void* stream) {
  if (!X || !O || !P || !beta || !nu || !I) return fail(HGRU_E_INVALID, "circuit_input_integration_forward: null pointer");
  if (rows < 1 || k < 1) return fail(HGRU_E_INVALID, "circuit_input_integration_forward: non-positive shape");
  hgru::circuit_input_integration_kernel<<<nblk(rows * k), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      X, O, P, beta, nu, xi, rows * k, k, I);
  CUDA_TRY(cudaGetLastError());
  return 0;
}
int circuit_output_integration_forward(const float* I, const float* P, const float* O, const float* G,
                                       const float* gamma, const float* kappa, const float* omega, float zeta,
                                       const float* rho, size_t rows, int k, float* O_out, void* stream) {
  if (!I || !P || !O || !G || !gamma || !kappa || !omega || !O_out)
    return fail(HGRU_E_INVALID, "circuit_output_integration_forward: null pointer");
  if (rows < 1 || k < 1) return fail(HGRU_E_INVALID, "circuit_output_integration_forward: non-positive shape");
  hgru::circuit_output_integration_kernel<<<nblk(rows * k), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      I, P, O, G, gamma, kappa, omega, zeta, rho, rows * k, k, O_out);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int layer_max_pool2x2_forward(const float* x, int N, int H, int W, int C, float* out, void* stream) {
  if (!x || !out) return fail(HGRU_E_INVALID, "layer_max_pool2x2_forward: null pointer");
  if (N < 1 || H < 1 || W < 1 || C < 1) return fail(HGRU_E_INVALID, "layer_max_pool2x2_forward: non-positive shape");
  const size_t total = static_cast<size_t>(N) * ((H + 1) / 2) * ((W + 1) / 2) * C;
  hgru::max_pool2x2_kernel<<<nblk(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, out, N, H, W, C);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int layer_pool_same_forward(const float* x, int N, int H, int W, int C, int ksize, int average, float* out,
                            void* stream) {
  if (!x || !out) return fail(HGRU_E_INVALID, "layer_pool_same_forward: null pointer");
  if (N < 1 || H < 1 || W < 1 || C < 1 || ksize < 1) return fail(HGRU_E_INVALID, "layer_pool_same_forward: non-positive shape");
  const size_t total = static_cast<size_t>(N) * ((H + ksize - 1) / ksize) * ((W + ksize - 1) / ksize) * C;
  hgru::pool_same_kernel<<<nblk(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, out, N, H, W, C, ksize,
                                                                                     average ? 1 : 0);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int layer_batchnorm_moments0_forward(const float* x, int N, size_t inner, float epsilon, float* out, void* stream) {
  if (!x || !out) return fail(HGRU_E_INVALID, "layer_batchnorm_moments0_forward: null pointer");
  if (N < 1 || inner < 1) return fail(HGRU_E_INVALID, "layer_batchnorm_moments0_forward: non-positive shape");
  hgru::batchnorm_moments0_kernel<<<nblk(inner), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, N, inner, epsilon, out);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int layer_fc_forward(const float* x, int M, int K, const float* weights, const float* biases, int F, float* out,
                     void* stream) {
  if (!x || !weights || !biases || !out) return fail(HGRU_E_INVALID, "layer_fc_forward: null pointer");
  if (M < 1 || K < 1 || F < 1) return fail(HGRU_E_INVALID, "layer_fc_forward: non-positive shape");
  hgru::fc_direct_kernel<<<nblk(static_cast<size_t>(M) * F), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, weights, biases, out, M, K, F);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int layer_resize_bilinear_forward(const float* x, int N, int H, int W, int OH, int OW, float* out, void* stream) {
  if (!x || !out) return fail(HGRU_E_INVALID, "layer_resize_bilinear_forward: null pointer");
  if (N < 1 || H < 1 || W < 1 || OH < 1 || OW < 1) return fail(HGRU_E_INVALID, "layer_resize_bilinear_forward: non-positive shape");
  const size_t total = static_cast<size_t>(N) * OH * OW;
  // TF 1.x: scale = in / out in float32 (kernels/resize_bilinear_op.cc CalculateResizeScale)
  const float sh = static_cast<float>(H) / static_cast<float>(OH), sw = static_cast<float>(W) / static_cast<float>(OW);
  hgru::resize_bilinear_kernel<<<nblk(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, out, N, H, W, OH, OW, sh, sw);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int layer_batch_norm_forward(const float* x, size_t rows, int C, const float* gamma, const float* beta,
                             const float* moving_mean, const float* moving_var, float eps, int training,
                             int relu_first, float dropout_keep, unsigned long long dropout_seed, float momentum,
                             float* new_moving_mean, float* new_moving_var, double* sums_ws, float* y, void* stream) {
  if (!x || !gamma || !beta || !moving_mean || !moving_var || !y)
    return fail(HGRU_E_INVALID, "layer_batch_norm_forward: null pointer");
  if (rows < 1 || C < 1) return fail(HGRU_E_INVALID, "layer_batch_norm_forward: non-positive shape");
  if (!(dropout_keep > 0.f)) return fail(HGRU_E_INVALID, "layer_batch_norm_forward: dropout_keep must be positive");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t total = rows * static_cast<size_t>(C);
  if (!training) {
    if (dropout_keep < 1.f) return fail(HGRU_E_INVALID, "layer_batch_norm_forward: dropout is a training-mode op");
    hgru::bn_inference_kernel<<<nblk(total), 256, 0, st>>>(x, y, total, C, gamma, beta, moving_mean, moving_var, eps,
                                                          relu_first ? 1 : 0);
    CUDA_TRY(cudaGetLastError());
    return 0;
  }
  if (!sums_ws) return fail(HGRU_E_INVALID, "layer_batch_norm_forward: training mode needs the 2*C doubles of workspace");
  if ((new_moving_mean == nullptr) != (new_moving_var == nullptr))
    return fail(HGRU_E_INVALID, "layer_batch_norm_forward: give both new moving statistics or neither");
  CUDA_TRY(cudaMemsetAsync(sums_ws, 0, sizeof(double) * 2 * C, st));
  size_t chunks = (rows + 2047) / 2048;
  if (chunks > 2048) chunks = 2048;
  hgru::bn_batch_sums_kernel<<<dim3((C + 31) / 32, static_cast<unsigned>(chunks)), 256, 0, st>>>(
      x, rows, C, sums_ws, relu_first ? 1 : 0, dropout_keep, dropout_seed);
  hgru::bn_apply_batch_kernel<<<nblk(total > static_cast<size_t>(C) ? total : C), 256, 0, st>>>(
      x, y, rows, C, sums_ws, gamma, beta, eps, moving_mean, moving_var, momentum, new_moving_mean, new_moving_var,
      relu_first ? 1 : 0, dropout_keep, dropout_seed);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ---- attention (centre-of-mass) CNN ----------------------------------------------------------------
int attn_plan_create(int N, int H, int W, const int* widths, int fc_hidden, int O, attn_plan_t* out) {
  return attn_plan_create_mode(N, H, W, widths, fc_hidden, O, HGRU_MODE_BF16X3, out);
}

int attn_plan_create_mode(int N, int H, int W, const int* widths, int fc_hidden, int O, int mode, attn_plan_t* out) {
  if (!out || !widths) return fail(HGRU_E_INVALID, "attn_plan_create: null pointer");
  *out = nullptr;
  if (N < 1 || H < 1 || W < 1 || fc_hidden < 1 || O < 1)
    return fail(HGRU_E_INVALID, "attn_plan_create: non-positive shape");
  for (int i = 0; i < 5; ++i)
    if (widths[i] < 8 || widths[i] % 8) return fail(HGRU_E_UNSUPPORTED, "attn_plan_create: widths must be multiples of 8");
  if (mode != HGRU_MODE_BF16X3 && mode != HGRU_MODE_FP16)
    return fail(HGRU_E_UNSUPPORTED, "attn_plan_create_mode: mode must be HGRU_MODE_BF16X3 or HGRU_MODE_FP16");
  attn_plan_s* p = new attn_plan_s();
  p->N = N; p->n = N; p->H = H; p->W = W; p->F = fc_hidden; p->O = O; p->mode = mode;
  for (int i = 0; i < 5; ++i) p->w[i] = widths[i];
  const int rc = attn_plan_build(p);
  if (rc) {
    attn_plan_free(p);
    delete p;
    return rc;
  }
  *out = p;
  return 0;
}

int attn_plan_destroy(attn_plan_t plan) {
  if (!plan) return 0;
  attn_plan_free(plan);
  delete plan;
  return 0;
}

int attn_set_params(attn_plan_t plan, const attn_params_t* params, float bn_epsilon, void* stream) {
  if (!plan) return fail(HGRU_E_INVALID, "attn_set_params: null plan");
  return attn_set_params_impl(plan, params, bn_epsilon, static_cast<cudaStream_t>(stream));
}

int attn_forward(attn_plan_t plan, const float* frames_dev, float* out_dev, void* stream) {
  if (!plan) return fail(HGRU_E_INVALID, "attn_forward: null plan");
  return attn_forward_impl(plan, plan->N, frames_dev, out_dev, static_cast<cudaStream_t>(stream));
}

int attn_forward_batch(attn_plan_t plan, int n, const float* frames_dev, float* out_dev, void* stream) {
  if (!plan) return fail(HGRU_E_INVALID, "attn_forward_batch: null plan");
  if (int rc = check_batch("attn_forward_batch", n, plan->N)) return rc;
  return attn_forward_impl(plan, n, frames_dev, out_dev, static_cast<cudaStream_t>(stream));
}

int attn_get_activation(attn_plan_t plan, const char* name, float* dst, void* stream) {
  if (!plan || !name || !dst) return fail(HGRU_E_INVALID, "attn_get_activation: null pointer");
  const std::string n(name);
  const void* src = nullptr;
  size_t bytes = 0;      // (of the capacity N; the copy takes the last forward's n frames)
  if (n == "resized") { src = plan->resized.p; bytes = plan->resized.bytes; }
  else if (n == "fc1") { src = plan->fc1.p; bytes = plan->fc1.bytes; }
  else if (n.size() == 5 && n.compare(0, 4, "pool") == 0 && n[4] >= '1' && n[4] <= '5') {
    src = plan->pool[n[4] - '1'].p; bytes = plan->pool[n[4] - '1'].bytes;
  }
  if (!src) return fail(HGRU_E_INVALID, "attn_get_activation: unknown tensor name '" + n + "'");
  bytes = bytes / plan->N * plan->n;
  CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return 0;
}

size_t attn_plan_workspace_bytes(attn_plan_t plan) { return plan ? plan->workspace_bytes() : 0; }
int attn_plan_launch_count(attn_plan_t plan) { return plan ? plan->launches : 0; }

}  // extern "C"
