// Launchers of hconv_tc_kernel for the hGRU convs, shared by tc_launch_h1.cu and tc_launch_h2.cu: each of the two
// translation units instantiates them for its own epilogues only (see lib_common.cuh for the interfaces).
#pragma once
#include "lib_common.cuh"

namespace hgru_host {

// the epilogue types of an EpiKind (Fp16: the fp16 mode's, where it has one)
template <EpiKind E> struct TcEpi;
template <> struct TcEpi<EPI_H1> { using Bf16 = hgru::EpiH1; };
template <> struct TcEpi<EPI_H2> { using Bf16 = hgru::EpiH2; };
template <> struct TcEpi<EPI_H1_HALF> { using Bf16 = hgru::EpiH1h; using Fp16 = hgru::EpiH1hF16; };
template <> struct TcEpi<EPI_H2_HALF> { using Bf16 = hgru::EpiH2h; using Fp16 = hgru::EpiH2hF16; };

namespace {

template <int S, int KSTEPS, int CO_PAD, int TILES_X, int G, class Epi, bool SPLIT3 = false, int WS = 4>
int launch_tc(const CUtensorMap& map, hgru::TcConvArgs a, cudaStream_t st) {
  using Cfg = hgru::TcConvCfg<S, KSTEPS, CO_PAD, TILES_X, G, WS, SPLIT3>;
  auto kern = hgru::hconv_tc_kernel<S, KSTEPS, CO_PAD, TILES_X, G, WS, Epi, SPLIT3>;
  SMEM_ATTR_ONCE(kern, Cfg::kSmemBytes);
  a.units_x = (a.W + 8 * TILES_X - 1) / (8 * TILES_X);
  a.units_y = (a.H + hgru::kTileRows - 1) / hgru::kTileRows;
  a.num_units = a.N * a.units_x * a.units_y;
  int sms = 0, rc = sm_count(&sms);
  if (rc) return rc;
  const int grid = a.num_units < sms ? a.num_units : sms;
  kern<<<grid, 256, Cfg::kSmemBytes, st>>>(map, a);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// (S, KP) instances.  KP -> (KSTEPS, TILES_X): 64 -> (4,4), 32 -> (2,8), 16 -> (1,8); G taps per stage.
#define TC_CASE(Epi_, S_, KP_, KS_, TX_, G_) \
  if (S == S_ && KP == KP_) return launch_tc<S_, KS_, KP_, TX_, G_, Epi_>(map, a, st);
#define TC_CASES_S(Epi_, S_, G64_, G32_)  \
  TC_CASE(Epi_, S_, 64, 4, 4, G64_)       \
  TC_CASE(Epi_, S_, 32, 2, 8, G32_)       \
  TC_CASE(Epi_, S_, 16, 1, 8, G32_)

// the horizontal convs with the fused integration epilogues, S < 15 (15 x 15 runs on the tap-stacked kernel or, at
// 64 channels, on the fused one below)
template <class Epi>
int dispatch_tc_hconv(int S, int KP, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st) {
  TC_CASES_S(Epi, 7, 7, 7)
  TC_CASES_S(Epi, 5, 5, 5)
  TC_CASES_S(Epi, 3, 9, 9)
  TC_CASES_S(Epi, 1, 1, 1)
  return fail(HGRU_E_UNSUPPORTED, "tensor-core conv: unsupported (S, padded channels)");
}
#undef TC_CASES_S
#undef TC_CASE

// 64 channels, 15x15 (the reference's own width): the same kernel with the 1x1 gate convs issued from its epilogue
// and the launches of a forward chained per frame (TcConvCfg FUSE) -- two launches per timestep.  Three weight
// stages instead of four make room for the gate's staging tile and weights.
// UT: tiles per unit, 4 (wide) or 2 (narrow, see launch_tc_fused64).
template <class Epi, class F, int UT, int G = 5, int WS = 3>
int launch_tc_fused64_ut(const CUtensorMap& map, hgru::TcConvArgs a, int sms, cudaStream_t st) {
  using Cfg = hgru::TcConvCfg<15, 4, 64, 4, G, WS, false, true, UT>;
  auto kern = hgru::hconv_tc_kernel<15, 4, 64, 4, G, WS, Epi, false, true, F, UT>;
  SMEM_ATTR_ONCE(kern, Cfg::kSmemBytes);
  a.units_x = (a.W + 8 * UT - 1) / (8 * UT);
  a.units_y = (a.H + hgru::kTileRows - 1) / hgru::kTileRows;
  a.num_units = a.N * a.units_x * a.units_y;
  a.flag_target = a.units_x * a.units_y;
  const int grid = a.num_units < sms ? a.num_units : sms;
  return launch_chainable(kern, grid, 256, Cfg::kSmemBytes, map, a, st);
}
// Wide units (4 tiles) or narrow ones (2 tiles); work = paired-tap instructions per filter row, 8 UT + 7.
template <class Epi, class F = hgru::OpBf16>
int launch_tc_fused64(const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st) {
  int sms = 0, rc = sm_count(&sms);
  if (rc) return rc;
  const int units_y = (a.H + hgru::kTileRows - 1) / hgru::kTileRows;
  if (narrow_units_faster(a.N * ((a.W + 31) / 32) * units_y, 39, a.N * ((a.W + 15) / 16) * units_y, 23, sms))
    return launch_tc_fused64_ut<Epi, F, 2>(map, a, sms, st);
  return launch_tc_fused64_ut<Epi, F, 4>(map, a, sms, st);
}

}  // namespace

template <EpiKind E>
int tc_hconv_launch(int S, int KP, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st) {
  return dispatch_tc_hconv<typename TcEpi<E>::Bf16>(S, KP, map, a, st);
}

template <EpiKind E>
int tc_fused64_launch(OpFormat fmt, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st) {
  if (fmt == FMT_FP16) return launch_tc_fused64<typename TcEpi<E>::Fp16, hgru::OpFp16>(map, a, st);
  return launch_tc_fused64<typename TcEpi<E>::Bf16>(map, a, st);
}

// bf16x3 mode at 64 channels: the 15x15 horizontal convs on hi/lo operand splits (narrower layers run it on the
// tap-stacked kernel)
template <EpiKind E>
int tc_x3_launch(int S, int KP, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st) {
  if (S == 15 && KP == 64)      // (wide stages: 3 taps each)
    return launch_tc<15, 4, 64, 1, 3, typename TcEpi<E>::Bf16, true>(map, a, st);
  return fail(HGRU_E_UNSUPPORTED, "bf16x3 conv: unsupported (S, padded channels)");
}

}  // namespace hgru_host
