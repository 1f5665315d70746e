// Development harness (GPU box only): tap-stacked tcgen05 conv vs a naive fp32 conv.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include <vector>
#include "../hconv_stack.cuh"
#include "../tc_host.cuh"
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e_), __LINE__); exit(2);} } while (0)

__global__ void naive_conv(const float* in, const float* w, const float* bias, float* out, int N, int H, int W, int k, int S) {
  size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t total = (size_t)N * H * W * k;
  if (idx >= total) return;
  int co = idx % k; size_t p = idx / k; int x = p % W; int y = (p / W) % H; int n = p / ((size_t)W * H);
  int pad = (S - 1) / 2; float acc = 0.f;
  for (int dy = 0; dy < S; ++dy) { int yy = y + dy - pad; if (yy < 0 || yy >= H) continue;
    for (int dx = 0; dx < S; ++dx) { int xx = x + dx - pad; if (xx < 0 || xx >= W) continue;
      const float* ip = in + ((size_t)(n * H + yy) * W + xx) * k; const float* wp = w + ((size_t)(dy * S + dx) * k) * k + co;
      for (int ci = 0; ci < k; ++ci) acc += ip[ci] * wp[(size_t)ci * k]; } }
  out[idx] = acc + bias[co];
}
__global__ void fill_f32(float* p, size_t n, float lo, float hi, unsigned seed) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
  unsigned h = (unsigned)(i * 2654435761u) ^ seed; h ^= h << 13; h ^= h >> 17; h ^= h << 5;
  p[i] = lo + (hi - lo) * (h & 0xFFFFFF) / 16777216.f;
}
__global__ void fill_bf16(__nv_bfloat16* p, size_t n, float lo, float hi, unsigned seed) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
  unsigned h = (unsigned)(i * 2654435761u) ^ seed; h ^= h << 13; h ^= h >> 17; h ^= h << 5;
  p[i] = __float2bfloat16(lo + (hi - lo) * (h & 0xFFFFFF) / 16777216.f);
}
static int g_random_data = 0, g_check_layout = 0, g_audit_fail = 0;
static float bf16r(float v) { return __bfloat162float(__float2bfloat16(v)); }

template <int KP, int T, int KC>
int run_case(int N, int H, int W, int k, int grid_override, int iters) {
  using Cfg = hgru::StackCfg<KP, T, KC>;
  const int S = 15, CG = KP / 8;
  printf("stack case KP=%d T=%d KC=%d k=%d N=%d H=%d W=%d smem=%d cols=%d\n", KP, T, KC, k, N, H, W, Cfg::SMEM_BYTES, Cfg::COLS);
  size_t npix = (size_t)N * H * W;
  std::vector<float> in(npix * k), w((size_t)S * S * k * k), bias(KP, 0.f);
  srand(123);
  for (auto& v : in) v = bf16r((rand() / (float)RAND_MAX) * 2.f - 1.f);
  for (auto& v : w) v = bf16r(((rand() / (float)RAND_MAX) * 2.f - 1.f) * 0.05f);
  for (int c = 0; c < k; ++c) bias[c] = (rand() / (float)RAND_MAX) - 0.5f;
  const int PADR = Cfg::ACT_PAD, HA = H + PADR;     // remainder-packed operand layout (StackCfg::REM)
  std::vector<__nv_bfloat16> act((size_t)N * CG * HA * W * 8, __float2bfloat16(0.f));
  for (int n = 0; n < N; ++n) for (int y = 0; y < H; ++y) for (int x = 0; x < W; ++x) for (int c = 0; c < k; ++c) {
    const __nv_bfloat16 v = __float2bfloat16(in[(((size_t)n * H + y) * W + x) * k + c]);
    if (Cfg::REM && c / 8 == CG - 1) {
      if (c % 8 == 0) for (int j = 0; j < 8; ++j) act[((((size_t)n * CG + CG - 1) * HA + (y + PADR - j)) * W + x) * 8 + j] = v;
    } else {
      act[((((size_t)n * CG + c / 8) * HA + y + PADR) * W + x) * 8 + (c % 8)] = v;
    }
  }
  float *d_in, *d_w, *d_bias, *d_ref, *d_out; __nv_bfloat16 *d_act, *d_wpk;
  size_t wpk_elems = (size_t)Cfg::PASS_STAGES * Cfg::NG * 2 * 128 * 8;
  CK(cudaMalloc(&d_in, in.size() * 4)); CK(cudaMalloc(&d_w, w.size() * 4)); CK(cudaMalloc(&d_bias, KP * 4));
  CK(cudaMalloc(&d_ref, npix * k * 4)); CK(cudaMalloc(&d_out, npix * KP * 4));
  CK(cudaMalloc(&d_act, act.size() * 2)); CK(cudaMalloc(&d_wpk, wpk_elems * 2));
  CK(cudaMemcpy(d_in, in.data(), in.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_w, w.data(), w.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_bias, bias.data(), KP * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_act, act.data(), act.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemset(d_out, 0xFF, npix * KP * 4));
  if (Cfg::REM) hgru::pack_weights_stack_rem_kernel<<<(unsigned)((wpk_elems + 255) / 256), 256>>>(d_w, d_wpk, k, T, KC, Cfg::NG);
  else hgru::pack_weights_stack_kernel<<<(unsigned)((wpk_elems + 255) / 256), 256>>>(d_w, d_wpk, k, Cfg::KSTEPS, T, KC, Cfg::NG);
  CK(cudaDeviceSynchronize());
  CUtensorMap map;
  if (hgru::make_act_tensor_map(&map, d_act, N, CG, HA, W, Cfg::COLS, Cfg::ROWS, Cfg::PART_CHUNKS)) { printf("map fail\n"); return 1; }
  hgru::TcConvArgs a{};
  a.N = N; a.H = H; a.W = W; a.KP = KP; a.kreal = k; a.act_pad = PADR;
  a.units_x = (W + 63) / 64; a.units_y = (H + 15) / 16; a.num_units = N * a.units_x * a.units_y;
  a.wpk = d_wpk; a.bias = d_bias; a.out = d_out;
  auto kern = hgru::hconv_stack_kernel<KP, T, KC, hgru::EpiBias>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  int sms = 0; CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
  const int grid = grid_override > 0 ? grid_override : (a.num_units < sms ? a.num_units : sms);
  cudaLaunchConfig_t cfg{}; cfg.gridDim = dim3(grid); cfg.blockDim = dim3(Cfg::NTHREADS); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  CK(cudaLaunchKernelEx(&cfg, kern, map, a));
  CK(cudaDeviceSynchronize());
  size_t total = npix * k;
  naive_conv<<<(unsigned)((total + 255) / 256), 256>>>(d_in, d_w, d_bias, d_ref, N, H, W, k, S);
  CK(cudaDeviceSynchronize());
  std::vector<float> outp(npix * KP), ref(total);
  CK(cudaMemcpy(outp.data(), d_out, npix * KP * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(ref.data(), d_ref, total * 4, cudaMemcpyDeviceToHost));
  double maxerr = 0, maxref = 0; size_t bad = 0, nan = 0;
  for (size_t p = 0; p < npix; ++p) for (int c = 0; c < k; ++c) {
    size_t nn = p / ((size_t)H * W), pin = p % ((size_t)H * W);
    float o = outp[((nn * (KP / 4) + c / 4) * (size_t)H * W + pin) * 4 + (c % 4)], r = ref[p * k + c];
    if (!(o == o)) { ++nan; continue; }
    double e = fabs((double)o - r); if (e > maxerr) maxerr = e; if (fabs(r) > maxref) maxref = fabs(r);
    if (e > 1e-3 * (1.0 + fabs(r))) ++bad; }
  printf("  grid=%d units=%d maxerr=%.3e maxref=%.3e bad=%zu nan=%zu\n", grid, a.num_units, maxerr, maxref, bad, nan);
  if (bad || nan) {
    for (int y = 0; y < (H < 32 ? H : 32); ++y) { for (int x = 0; x < (W < 64 ? W : 64); ++x) {
      float o = outp[((size_t)y * W + x) * 4], r = ref[(((size_t)0 * H + y) * W + x) * k];
      putchar(!(o == o) ? 'N' : (fabs(o - r) > 1e-3 * (1 + fabs(r)) ? 'x' : '.')); } putchar('\n'); }
  }
  if (iters > 0 && !bad && !nan) {
    long long* d_prof; CK(cudaMalloc(&d_prof, grid * 40 * sizeof(long long))); CK(cudaMemset(d_prof, 0, grid * 40 * sizeof(long long)));
    hgru::TcConvArgs ap = a; ap.prof = d_prof;
    CK(cudaLaunchKernelEx(&cfg, kern, map, ap)); CK(cudaDeviceSynchronize());
    std::vector<long long> pr(grid * 8); CK(cudaMemcpy(pr.data(), d_prof, grid * 8 * sizeof(long long), cudaMemcpyDeviceToHost));
    double av[6] = {0, 0, 0, 0, 0, 0}; for (int b = 0; b < grid; ++b) for (int i = 0; i < 6; ++i) av[i] += pr[b * 8 + i] / (double)grid;
    printf("  prof (avg cycles/CTA): mma_total=%.0f wait_win=%.0f wait_acc_empty=%.0f wait_w_full=%.0f | epi_total=%.0f epi_wait_acc_full=%.0f\n", av[0], av[1], av[2], av[3], av[4], av[5]);
    cudaFree(d_prof);
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int i = 0; i < 2; ++i) cudaLaunchKernelEx(&cfg, kern, map, a);
    cudaEventRecord(e0);
    for (int i = 0; i < iters; ++i) cudaLaunchKernelEx(&cfg, kern, map, a);
    cudaEventRecord(e1); CK(cudaDeviceSynchronize());
    float ms; cudaEventElapsedTime(&ms, e0, e1); ms /= iters;
    printf("  time %.3f ms -> %.1f TFLOP/s algorithmic\n", ms, 2.0 * npix * 225.0 * k * k / ms * 1e-9);
  }
  cudaFree(d_in); cudaFree(d_w); cudaFree(d_bias); cudaFree(d_ref); cudaFree(d_out); cudaFree(d_act); cudaFree(d_wpk);
  return (bad || nan) ? 1 : 0;
}
template <int KP, int T, int KC, class Epi>
void time_real_epilogue(const char* name, int N, int H, int W, int k, int gate = 1, int dbg = 0) {
  using Cfg = hgru::StackCfg<KP, T, KC>;
  const int CG = KP / 8;
  size_t npix = (size_t)N * H * W;
  float *X, *H1, *G, *H2, *vec; __nv_bfloat16 *act, *actout, *wpk;
  size_t wpk_elems = (size_t)Cfg::PASS_STAGES * Cfg::NG * 2 * 128 * 8;
  const int HA = H + Cfg::ACT_PAD; const size_t actb = (size_t)N * CG * HA * W * 8 * 2;
  CK(cudaMalloc(&X, npix * KP * 4)); CK(cudaMalloc(&H1, npix * KP * 4)); CK(cudaMalloc(&G, npix * KP * 4)); CK(cudaMalloc(&H2, npix * KP * 4));
  CK(cudaMalloc(&vec, 8 * KP * 4)); CK(cudaMalloc(&act, actb));
  const size_t GUARD = 1 << 20; uint8_t* actout_raw; CK(cudaMalloc(&actout_raw, actb + 2 * GUARD)); CK(cudaMemset(actout_raw, 0xA5, actb + 2 * GUARD));
  actout = reinterpret_cast<__nv_bfloat16*>(actout_raw + GUARD); CK(cudaMalloc(&wpk, wpk_elems * 2));
  CK(cudaMemset(X, 0, npix * KP * 4)); CK(cudaMemset(H1, 0, npix * KP * 4)); CK(cudaMemset(G, 0, npix * KP * 4)); CK(cudaMemset(H2, 0, npix * KP * 4));
  CK(cudaMemset(vec, 0, 8 * KP * 4)); CK(cudaMemset(act, 0, actb)); CK(cudaMemset(actout, 0, actb)); CK(cudaMemset(wpk, 0, wpk_elems * 2));
  if (g_random_data) {   // realistic operand / state values instead of zeros (switching power, real tanh inputs)
    size_t ns = npix * KP;
    fill_f32<<<(unsigned)((ns + 255) / 256), 256>>>(X, ns, -1.f, 1.f, 1u); fill_f32<<<(unsigned)((ns + 255) / 256), 256>>>(H1, ns, -1.f, 1.f, 2u);
    fill_f32<<<(unsigned)((ns + 255) / 256), 256>>>(G, ns, 0.f, 1.f, 3u); fill_f32<<<(unsigned)((ns + 255) / 256), 256>>>(H2, ns, -1.f, 1.f, 4u);
    fill_f32<<<(8 * KP + 255) / 256, 256>>>(vec, 8 * KP, 0.5f, 1.f, 5u);
    fill_bf16<<<(unsigned)((actb / 2 + 255) / 256), 256>>>(act, actb / 2, -1.f, 1.f, 6u);
    fill_bf16<<<(unsigned)((wpk_elems + 255) / 256), 256>>>(wpk, wpk_elems, -0.05f, 0.05f, 7u);
    CK(cudaDeviceSynchronize());
  }
  CUtensorMap map;
  hgru::make_act_tensor_map(&map, act, N, CG, HA, W, Cfg::COLS, Cfg::ROWS, Cfg::PART_CHUNKS);
  hgru::TcConvArgs a{};
  a.N = N; a.H = H; a.W = W; a.KP = KP; a.kreal = k; a.act_pad = Cfg::ACT_PAD;
  a.units_x = (W + 63) / 64; a.units_y = (H + 15) / 16; a.num_units = N * a.units_x * a.units_y;
  a.wpk = wpk; a.bias = vec; a.v0 = vec + KP; a.v1 = vec + 2 * KP; a.v2 = vec + 3 * KP; a.rho_t = vec + 4 * KP;
  a.X = X; a.H1 = H1; a.G = G; a.H2 = H2; a.out = H1; a.out_bf16 = actout;
  a.gate_wpk = wpk; a.gate_bias = vec; a.gate_out = G; a.gate_act_out = actout; a.do_gate = gate; a.dbg_flags = dbg;
  if (std::is_same<Epi, hgru::EpiH2>::value) a.out_bf16 = nullptr;   // fused pipeline: H2's operand copy comes from the gate
  auto kern = hgru::hconv_stack_kernel<KP, T, KC, Epi, false>;
  auto kern_prof = hgru::hconv_stack_kernel<KP, T, KC, Epi, true>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  CK(cudaFuncSetAttribute(kern_prof, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  int grid = 148;
  cudaLaunchConfig_t cfg{}; cfg.gridDim = dim3(grid); cfg.blockDim = dim3(Cfg::NTHREADS); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  long long* d_prof; CK(cudaMalloc(&d_prof, grid * 40 * sizeof(long long))); CK(cudaMemset(d_prof, 0, grid * 40 * sizeof(long long)));
  hgru::TcConvArgs ap = a; ap.prof = d_prof;
  CK(cudaLaunchKernelEx(&cfg, kern_prof, map, ap)); CK(cudaDeviceSynchronize());
  std::vector<long long> pr(grid * 40); CK(cudaMemcpy(pr.data(), d_prof, grid * 40 * sizeof(long long), cudaMemcpyDeviceToHost));
  double av[6] = {0, 0, 0, 0, 0, 0}; int nl = 0;
  for (int b = 0; b < grid; ++b) { if (pr[b * 8]) ++nl; for (int i = 0; i < 6; ++i) av[i] += pr[b * 8 + i]; }
  { long long mx = 0, mxe = 0; double ns = 0; for (int b = 0; b < grid; ++b) { if (pr[b * 8] > mx) mx = pr[b * 8]; if (pr[b * 8 + 4] > mxe) mxe = pr[b * 8 + 4]; ns += pr[b * 8 + 6]; }
    printf("    max over CTAs: mma_total=%lld epi_total=%lld | mean CTA wall %.1f us -> SM clock %.3f GHz\n", mx, mxe, ns / nl * 1e-3, av[0] / ns); }
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  cudaEventRecord(e0);
  for (int i = 0; i < 20; ++i) cudaLaunchKernelEx(&cfg, kern, map, a);
  cudaEventRecord(e1); CK(cudaDeviceSynchronize());
  float ms; cudaEventElapsedTime(&ms, e0, e1); ms /= 20;
  { // the same PROF launch again, right behind 40 more back-to-back launches: clock under sustained load
    for (int i = 0; i < 40; ++i) cudaLaunchKernelEx(&cfg, kern, map, a);
    CK(cudaMemset(d_prof, 0, grid * 40 * sizeof(long long)));
    CK(cudaLaunchKernelEx(&cfg, kern_prof, map, ap)); CK(cudaDeviceSynchronize());
    std::vector<long long> p2(grid * 8); CK(cudaMemcpy(p2.data(), d_prof, grid * 8 * sizeof(long long), cudaMemcpyDeviceToHost));
    double cyc = 0, ns = 0; long long mx = 0; for (int b = 0; b < grid; ++b) { cyc += p2[b * 8]; ns += p2[b * 8 + 6]; if (p2[b * 8] > mx) mx = p2[b * 8]; }
    printf("    sustained: mma_total avg %.0f max %lld cycles, mean CTA wall %.1f us -> SM clock %.3f GHz\n", cyc / grid, mx, ns / grid * 1e-3, cyc / ns); }
  printf("%s gate=%d: %.3f ms | avg cycles: mma_total=%.0f wait_win=%.0f wait_acc_empty=%.0f wait_w=%.0f | epi_total=%.0f epi_wait=%.0f\n", name, gate, ms,
         av[0] / nl, av[1] / nl, av[2] / nl, av[3] / nl, av[4] / grid, av[5] / grid);
  if (g_check_layout) {
    // Bounds / layout audit of the operand tensor the epilogue wrote (stands in for a memory checker):
    // guard bands untouched; pad rows and never-written elements still zero; in the remainder-packed plane every
    // value appears at its 8 (row - j, lane j) positions.
    std::vector<uint8_t> hb(actb + 2 * GUARD);
    CK(cudaMemcpy(hb.data(), actout_raw, hb.size(), cudaMemcpyDeviceToHost));
    size_t guard_bad = 0, pad_bad = 0, pack_bad = 0, nonzero = 0;
    for (size_t i = 0; i < GUARD; ++i) { if (hb[i] != 0xA5) ++guard_bad; if (hb[GUARD + actb + i] != 0xA5) ++guard_bad; }
    const uint16_t* o = reinterpret_cast<const uint16_t*>(hb.data() + GUARD);
    const int PADR = Cfg::ACT_PAD;
    auto at = [&](int n, int cg, int r, int x, int j) { return o[((((size_t)n * CG + cg) * HA + r) * W + x) * 8 + j]; };
    for (int n = 0; n < N; n += 37) for (int cg = 0; cg < CG; ++cg) for (int r = 0; r < HA; ++r) for (int x = 0; x < W; ++x) for (int j = 0; j < 8; ++j) {
      const uint16_t v = at(n, cg, r, x, j);
      if (v) ++nonzero;
      const bool rem_plane = Cfg::REM && cg == CG - 1;
      if (!rem_plane) {
        if (r < PADR && v) ++pad_bad;                                       // top pad rows stay zero
        if (cg * 8 + j >= k && v) ++pad_bad;                                // pad channels stay zero
      } else {
        const int y = r - PADR + j;                                         // source pixel row of this element
        if ((y < 0 || y >= H) && v) ++pad_bad;                              // never written -> still zero
        if (y >= 0 && y < H && v != at(n, cg, y + PADR, x, 0)) ++pack_bad;  // == the value stored at (y, lane 0)
      }
    }
    printf("    layout audit: guard_bad=%zu pad_bad=%zu pack_bad=%zu (nonzero elements seen %zu)\n", guard_bad, pad_bad, pack_bad, nonzero);
    if (guard_bad || pad_bad || pack_bad || !nonzero) g_audit_fail = 1;
  }
  for (int g = 0; g < Cfg::NGRP; ++g) {
    double ph[6] = {0, 0, 0, 0, 0, 0};
    for (int b = 0; b < grid; ++b) for (int i = 0; i < 6; ++i) ph[i] += pr[grid * 8 + (b * Cfg::NGRP + g) * 8 + i] / (double)grid;
    printf("    epilogue group %d: total=%.0f wait=%.0f tmem+unstack=%.0f finish=%.0f gate_wait=%.0f gate_math=%.0f\n", g, ph[0], ph[1], ph[2], ph[3], ph[4], ph[5]);
  }
  cudaFree(X); cudaFree(H1); cudaFree(G); cudaFree(H2); cudaFree(vec); cudaFree(act); cudaFree(actout_raw); cudaFree(wpk); cudaFree(d_prof);
}

int main(int argc, char** argv) {
  int which = argc > 1 ? atoi(argv[1]) : 0, f = 0;
  if (which == 0 || which == 1) f += run_case<32, 5, 25>(2, 64, 64, 25, 0, 0);
  if (which == 0 || which == 2) f += run_case<32, 5, 25>(3, 64, 64, 25, 5, 0);      // several units per CTA, idle tail
  if (which == 0 || which == 3) f += run_case<32, 5, 25>(2, 40, 24, 20, 0, 0);      // ragged, k < KC
  if (which == 0 || which == 4) f += run_case<32, 4, 32>(2, 64, 64, 32, 0, 0);
  if (which == 0 || which == 5) f += run_case<16, 8, 16>(2, 32, 48, 16, 0, 0);
  if (which == 0 || which == 7) f += run_case<32, 5, 25>(256, 64, 64, 25, 0, 5);
  if (which == 21) {   // weight ring refills on / off (dbg bit 0), random operand data: what the L2 -> SM weight stream costs
    g_random_data = 1;
    time_real_epilogue<32, 5, 25, hgru::EpiBias>("EpiBias", 256, 64, 64, 25, 0, 0);
    time_real_epilogue<32, 5, 25, hgru::EpiBias>("EpiBias noWstream", 256, 64, 64, 25, 0, 1);
    time_real_epilogue<32, 5, 25, hgru::EpiH2>("EpiH2", 256, 64, 64, 25, 1, 0);
    time_real_epilogue<32, 5, 25, hgru::EpiH2>("EpiH2 noWstream", 256, 64, 64, 25, 1, 1);
    g_random_data = 0;
  }
  if (which == 23) {   // epilogue-written operand tensors: guard bands, zero padding, remainder-plane consistency
    g_random_data = 1; g_check_layout = 1;
    time_real_epilogue<32, 5, 25, hgru::EpiH1>("EpiH1", 256, 64, 64, 25, 1);
    time_real_epilogue<32, 5, 25, hgru::EpiH2>("EpiH2", 256, 64, 64, 25, 1);
    time_real_epilogue<32, 5, 25, hgru::EpiH2>("EpiH2 ragged", 37, 40, 24, 25, 1);
    time_real_epilogue<32, 4, 32, hgru::EpiH2>("EpiH2 k32", 64, 64, 64, 32, 1);
    g_random_data = 0; g_check_layout = 0; f += g_audit_fail;
  }
  if (which == 22) {
    for (g_random_data = 0; g_random_data < 2; ++g_random_data) {
      printf("---- %s data\n", g_random_data ? "random" : "zero");
      time_real_epilogue<32, 5, 25, hgru::EpiBias>("EpiBias", 256, 64, 64, 25, 0);
      time_real_epilogue<32, 5, 25, hgru::EpiH1>("EpiH1", 256, 64, 64, 25, 1);
      time_real_epilogue<32, 5, 25, hgru::EpiH2>("EpiH2", 256, 64, 64, 25, 1);
    }
  }
  if (which == 20) {   // each epilogue with and without its fused gate, random data
    g_random_data = 1;
    time_real_epilogue<32, 5, 25, hgru::EpiBias>("EpiBias", 256, 64, 64, 25, 0);
    time_real_epilogue<32, 5, 25, hgru::EpiH1>("EpiH1", 256, 64, 64, 25, 0);
    time_real_epilogue<32, 5, 25, hgru::EpiH1>("EpiH1", 256, 64, 64, 25, 1);
    time_real_epilogue<32, 5, 25, hgru::EpiH2>("EpiH2", 256, 64, 64, 25, 0);
    time_real_epilogue<32, 5, 25, hgru::EpiH2>("EpiH2", 256, 64, 64, 25, 1);
  }
  printf(f ? "FAILED %d\n" : "ALL OK\n", f);
  return f;
}
