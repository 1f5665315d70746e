// libhgru_b200.so, translation unit tc_launch_h2 (C2 + output-integration epilogues): instantiations and launchers of hconv_tc_kernel
// (see tc_launch.cuh and lib_common.cuh).
#include "tc_launch.cuh"

namespace hgru_host {

template int tc_hconv_launch<EPI_H2>(int, int, const CUtensorMap&, const hgru::TcConvArgs&, cudaStream_t);
template int tc_fused64_launch<EPI_H2_HALF>(OpFormat, const CUtensorMap&, const hgru::TcConvArgs&, cudaStream_t);
template int tc_x3_launch<EPI_H2>(int, int, const CUtensorMap&, const hgru::TcConvArgs&, cudaStream_t);

}  // namespace hgru_host
