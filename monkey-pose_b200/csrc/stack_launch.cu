// libhgru_b200.so, translation unit stack_launch: instantiations and launchers of the tap-stacked conv
// (hconv_stack.cuh) and its weight packing (see lib_common.cuh for the interfaces).
#include "lib_common.cuh"

#include "hconv_stack.cuh"

namespace hgru_host {

bool stack_geometry(int S, int KP, int k, StackGeom* g) {
  if (S != 15) return false;
  if (KP == 32 && k <= 25) { g->T = 5; g->KC = 25; }
  else if (KP == 32) { g->T = 4; g->KC = 32; }
  else if (KP == 16) { g->T = 8; g->KC = 16; }
  else return false;
  g->NG = (15 + g->T - 1) / g->T;
  g->ksteps = KP / 16;
  g->box_cols = 64 + g->T * (g->NG - 1) + 8;
  g->box_rows = hgru::kTileRows + 14;
  // KC = 25: remainder-packed K schedule (hgru::StackCfg::REM) -- 24 weight stages, 7 pad rows per plane
  const bool rem = hgru::StackCfg<32, 5, 25>::REM && g->KC == 25;
  g->stages = rem ? hgru::StackCfg<32, 5, 25>::PASS_STAGES : 15 * g->ksteps;
  g->act_pad = rem ? hgru::StackCfg<32, 5, 25>::ACT_PAD : 0;
  return true;
}

namespace {

template <class F>
void pack_stack(const float* p_r, __nv_bfloat16* dst, int k, const StackGeom& sg, int lo_part, cudaStream_t st) {
  const size_t ts = static_cast<size_t>(sg.stages) * sg.NG * 2 * 128 * 8;
  auto* o = reinterpret_cast<typename F::T*>(dst);
  if (sg.act_pad)
    hgru::pack_weights_stack_rem_kernel<F><<<nblk(ts), 256, 0, st>>>(p_r, o, k, sg.T, sg.KC, sg.NG, lo_part);
  else
    hgru::pack_weights_stack_kernel<F><<<nblk(ts), 256, 0, st>>>(p_r, o, k, sg.ksteps, sg.T, sg.KC, sg.NG, lo_part);
}

template <int KP, int T, int KC, class Epi, int WSETS = 1, bool PART = false, class F = hgru::OpBf16>
int launch_stack(const CUtensorMap& map, hgru::TcConvArgs a, cudaStream_t st) {
  // The second launch of a bf16x3 conv (PART) is also the one whose epilogue issues the gate, on hi/lo splits (GX3)
  // -- except at 32 channels, where the two staging tiles do not fit next to a 3-stage weight ring: that
  // configuration keeps its gates in the exact SIMT kernel.
  constexpr bool GX3 = PART && !(KP == 32 && T == 4);
  using Cfg = hgru::StackCfg<KP, T, KC, GX3, F>;
  auto kern = hgru::hconv_stack_kernel<KP, T, KC, Epi, false, WSETS, PART, GX3, F>;
  SMEM_ATTR_ONCE(kern, Cfg::SMEM_BYTES);
  a.units_x = (a.W + 63) / 64;
  a.units_y = (a.H + hgru::kTileRows - 1) / hgru::kTileRows;
  a.num_units = a.N * a.units_x * a.units_y;
  int sms = 0, rc = sm_count(&sms);
  if (rc) return rc;
  const int grid = a.num_units < sms ? a.num_units : sms;
  a.flag_target = a.units_x * a.units_y;
  // A launch that waits on the previous launch's per-frame counters is chained to it (programmatic dependent
  // launch): its CTAs take SMs as the previous launch's CTAs exit instead of waiting for the whole grid.
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(Cfg::NTHREADS); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = a.wait_flags ? 1 : 0;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, map, a));
  return 0;
}

template <class Epi, int WSETS = 1, bool PART = false, class F = hgru::OpBf16>
int dispatch_stack(int KP, int T, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st) {
  if (KP == 32 && T == 5) return launch_stack<32, 5, 25, Epi, WSETS, PART, F>(map, a, st);
  if (KP == 32 && T == 4) return launch_stack<32, 4, 32, Epi, WSETS, PART, F>(map, a, st);
  if (KP == 16 && T == 8) return launch_stack<16, 8, 16, Epi, WSETS, PART, F>(map, a, st);
  return fail(HGRU_E_UNSUPPORTED, "stacked conv: unsupported configuration");
}

}  // namespace

int stack_pack_weights(const float* p_r, __nv_bfloat16* dst, int k, const StackGeom& sg, int lo_part, OpFormat fmt,
                       cudaStream_t st) {
  if (fmt == FMT_FP16) pack_stack<hgru::OpFp16>(p_r, dst, k, sg, lo_part, st);
  else pack_stack<hgru::OpBf16>(p_r, dst, k, sg, lo_part, st);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int stack_launch(EpiKind epi, int wsets, bool part, int KP, int T, OpFormat fmt, const CUtensorMap& map,
                 const hgru::TcConvArgs& a, cudaStream_t st) {
  if (fmt == FMT_FP16) {      // fp16 mode: the fused pipeline's two launches per timestep
    if (!part && wsets == 1 && epi == EPI_H1_HALF)
      return dispatch_stack<hgru::EpiH1hF16, 1, false, hgru::OpFp16>(KP, T, map, a, st);
    if (!part && wsets == 1 && epi == EPI_H2_HALF)
      return dispatch_stack<hgru::EpiH2hF16, 1, false, hgru::OpFp16>(KP, T, map, a, st);
    return fail(HGRU_E_UNSUPPORTED, "stacked conv: no fp16 variant of this kernel");
  }
  if (!part && wsets == 1) {
    switch (epi) {
      case EPI_H1_HALF: return dispatch_stack<hgru::EpiH1h>(KP, T, map, a, st);      // fused bf16 pipeline
      case EPI_H2_HALF: return dispatch_stack<hgru::EpiH2h>(KP, T, map, a, st);
      case EPI_PARTIAL: return dispatch_stack<hgru::EpiPartial>(KP, T, map, a, st);  // bf16x3, first launch of a conv
      default: break;
    }
  } else if (part && wsets == 2) {                                                   // bf16x3, second launch
    if (epi == EPI_H1) return dispatch_stack<hgru::EpiH1, 2, true>(KP, T, map, a, st);
    if (epi == EPI_H2) return dispatch_stack<hgru::EpiH2, 2, true>(KP, T, map, a, st);
  }
  return fail(HGRU_E_UNSUPPORTED, "stacked conv: no such kernel variant");
}

}  // namespace hgru_host
