// libhgru_b200.so, translation unit tc_launch_h1 (C1 + input-integration epilogues, the stem convs, the geometries): instantiations and launchers of hconv_tc_kernel
// (see tc_launch.cuh and lib_common.cuh).
#include "tc_launch.cuh"

namespace hgru_host {

template int tc_hconv_launch<EPI_H1>(int, int, const CUtensorMap&, const hgru::TcConvArgs&, cudaStream_t);
template int tc_fused64_launch<EPI_H1_HALF>(OpFormat, const CUtensorMap&, const hgru::TcConvArgs&, cudaStream_t);
template int tc_x3_launch<EPI_H1>(int, int, const CUtensorMap&, const hgru::TcConvArgs&, cudaStream_t);

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

}  // namespace hgru_host
