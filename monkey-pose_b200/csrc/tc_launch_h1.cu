// libhgru_b200.so, translation unit tc_launch_h1 (C1 + input-integration epilogues, the stem convs, the geometries): instantiations and launchers of hconv_tc_kernel
// (see lib_common.cuh for the interfaces).
#include "lib_common.cuh"

namespace hgru_host {
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
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = Cfg::kSmemBytes; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = a.wait_flags ? 1 : 0;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, map, a));
  return 0;
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

// bf16x3 mode at 64 channels: the 15x15 horizontal convs on hi/lo operand splits (narrower layers run it on the
// tap-stacked kernel)
template <class Epi>
int dispatch_tc_hconv_x3(int S, int KP, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st) {
  if (S == 15 && KP == 64) return launch_tc<15, 4, 64, 1, 3, Epi, true>(map, a, st);   // (wide stages: 3 taps each)
  return fail(HGRU_E_UNSUPPORTED, "bf16x3 conv: unsupported (S, padded channels)");
}

}  // namespace

int tc_launch_h1(int family, int S, int KP, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st) {
  if (family == 0) return dispatch_tc_hconv<hgru::EpiH1>(S, KP, map, a, st);
  if (family == 1) return launch_tc_fused64<hgru::EpiH1h>(map, a, st);
  if (family == 3) return launch_tc_fused64<hgru::EpiH1hF16, hgru::OpFp16>(map, a, st);      // fp16 mode
  return dispatch_tc_hconv_x3<hgru::EpiH1>(S, KP, map, a, st);
}

// geometry of the window box for a given (S, KP)
bool tc_geometry(int S, int KP, TcGeom* g) {
  if (!(S == 1 || S == 3 || S == 5 || S == 7 || S == 15)) return false;
  if (!(KP == 16 || KP == 32 || KP == 64)) return false;
  g->tiles_x = (KP == 64) ? 4 : 8;
  g->box_cols = 8 * g->tiles_x + S - 1;
  g->box_rows = hgru::kTileRows + S - 1;
  return true;
}
// 3x3 stem convs: bf16 hi + lo operand halves, three products per k-step (SPLIT3): fp32-class accuracy.
// A SPLIT3 tile owns 2 * KP accumulator columns ([w_hi | w_lo] stacked along N), so two accumulator sets hold
// 2 / 4 / 8 tiles of 8 columns at 64 / 32 / 16 channels.
bool stem_geometry(int KP, TcGeom* g) {
  if (!(KP == 16 || KP == 32 || KP == 64)) return false;
  g->tiles_x = (KP == 64) ? 2 : (KP == 32) ? 4 : 8;
  g->box_cols = 8 * g->tiles_x + 2;
  g->box_rows = hgru::kTileRows + 2;
  return true;
}
// bf16x3 on hconv_tc_kernel (64 channels): the window holds both operand halves, so a unit is one tile of 8 columns
bool x3_geometry(int S, int KP, TcGeom* g) {
  if (S != 15 || KP != 64) return false;
  g->tiles_x = 1;
  g->box_cols = 8 * g->tiles_x + S - 1;
  g->box_rows = hgru::kTileRows + S - 1;
  return true;
}
int tc_stem_launch(int KP, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st) {
  if (KP == 64) return launch_tc<3, 4, 64, 2, 3, hgru::EpiBiasReluAffine, true>(map, a, st);
  if (KP == 32) return launch_tc<3, 2, 32, 4, 9, hgru::EpiBiasReluAffine, true>(map, a, st);
  if (KP == 16) return launch_tc<3, 1, 16, 8, 9, hgru::EpiBiasReluAffine, true>(map, a, st);
  return fail(HGRU_E_UNSUPPORTED, "tensor-core stem conv: unsupported padded channel count");
}
int tc_launch_h2(int family, int S, int KP, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st);
int tc_hconv_launch(EpiKind epi, int S, int KP, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st) {
  return epi == EPI_H1 ? tc_launch_h1(0, S, KP, map, a, st) : tc_launch_h2(0, S, KP, map, a, st);
}
int tc_fused64_launch(EpiKind epi, OpFormat fmt, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st) {
  const int family = fmt == FMT_FP16 ? 3 : 1;
  return epi == EPI_H1_HALF ? tc_launch_h1(family, 15, 64, map, a, st) : tc_launch_h2(family, 15, 64, map, a, st);
}
int tc_x3_launch(EpiKind epi, int S, int KP, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st) {
  return epi == EPI_H1 ? tc_launch_h1(2, S, KP, map, a, st) : tc_launch_h2(2, S, KP, map, a, st);
}

}  // namespace hgru_host
