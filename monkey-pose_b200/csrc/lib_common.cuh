// Host-side plumbing shared by the translation units of libhgru_b200.so (the library is compiled as several .cu files
// so that the template instantiations of the big kernels build in parallel): error reporting, per-device caches, the
// launch geometries and the non-template launcher interfaces.
#pragma once
#include "../../include/hgru_b200.h"

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <string>

#include "hconv_tc.cuh"

namespace hgru_host {

// message of the last failure on the calling thread (defined in hgru_lib.cu)
int fail(int code, const std::string& msg);

#define CUDA_TRY(expr)                                                                        \
  do {                                                                                        \
    cudaError_t e_ = (expr);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return hgru_host::fail(HGRU_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));\
  } while (0)

// Function attributes (the dynamic shared-memory opt-in) and the SM count belong to a DEVICE, and one process may
// drive several: remember per device what was done / read, not per process.
struct PerDeviceOnce {
  std::atomic<unsigned long long> mask{0};
  bool seen(int dev) const { return dev >= 0 && dev < 64 && ((mask.load(std::memory_order_acquire) >> dev) & 1ull); }
  void mark(int dev) { if (dev >= 0 && dev < 64) mask.fetch_or(1ull << dev, std::memory_order_release); }
};
#define SMEM_ATTR_ONCE(kern, bytes)                                                                       \
  do {                                                                                                    \
    static hgru_host::PerDeviceOnce once_;                                                                \
    int dev_ = 0;                                                                                         \
    CUDA_TRY(cudaGetDevice(&dev_));                                                                       \
    if (!once_.seen(dev_)) {      /* (idempotent: a race only sets the attribute twice) */                \
      CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));           \
      once_.mark(dev_);                                                                                   \
    }                                                                                                     \
  } while (0)

// multiprocessor count of the current device
inline int sm_count(int* out) {
  static std::atomic<int> cache[64];
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  int v = (dev >= 0 && dev < 64) ? cache[dev].load(std::memory_order_relaxed) : 0;
  if (!v) {
    CUDA_TRY(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev));
    if (dev >= 0 && dev < 64) cache[dev].store(v, std::memory_order_relaxed);
  }
  *out = v;
  return 0;
}

inline unsigned nblk(size_t n, int b = 256) { return static_cast<unsigned>((n + b - 1) / b); }
inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

// ---- launch geometries (must match the template instances in tc_launch_*.cu / stack_launch.cu) ----
struct TcGeom { int tiles_x, box_cols, box_rows; };
bool tc_geometry(int S, int KP, TcGeom* g);        // plain bf16 hconv_tc_kernel
bool stem_geometry(int KP, TcGeom* g);             // 3x3 stem convs (SPLIT3)
bool x3_geometry(int S, int KP, TcGeom* g);        // bf16x3 on hconv_tc_kernel (SPLIT3)
struct StackGeom { int T, KC, NG, ksteps, box_cols, box_rows, stages, act_pad; };
bool stack_geometry(int S, int KP, int k, StackGeom* g);

// ---- launchers (one translation unit per kernel family) ----
// format of the hGRU convs' 16-bit operands and weights (hgru::OpBf16 / hgru::OpFp16): bf16 mode / fp16 mode
enum OpFormat { FMT_BF16 = 0, FMT_FP16 = 1 };
enum EpiKind { EPI_H1 = 0, EPI_H2 = 1, EPI_H1_HALF = 2, EPI_H2_HALF = 3, EPI_PARTIAL = 4 };
// hconv_stack_kernel<..., Epi, WSETS, PART>: tap-stacked 15x15 conv (k <= 32); FMT_FP16 exists for EPI_H*_HALF
int stack_launch(EpiKind epi, int wsets, bool part, int KP, int T, OpFormat fmt, const CUtensorMap& map,
                 const hgru::TcConvArgs& a, cudaStream_t st);
// its weight packing: HWIO fp32 -> the stacked (or remainder-packed) 16-bit stage layout; lo_part = the remainder
int stack_pack_weights(const float* p_r, __nv_bfloat16* dst, int k, const StackGeom& sg, int lo_part, OpFormat fmt,
                       cudaStream_t st);
// hconv_tc_kernel: plain (EPI_H1 / EPI_H2), FUSE at 64 channels (EPI_H1_HALF / EPI_H2_HALF), SPLIT3 stem, SPLIT3 x3
int tc_hconv_launch(EpiKind epi, int S, int KP, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st);
int tc_fused64_launch(EpiKind epi, OpFormat fmt, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st);
int tc_stem_launch(int KP, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st);
int tc_x3_launch(EpiKind epi, int S, int KP, const CUtensorMap& map, const hgru::TcConvArgs& a, cudaStream_t st);

}  // namespace hgru_host
