// Kernels of the attention (centre-of-mass) CNN forward, reference `attn_model_struct.build`
// (train_cnn_networks_hgru.py:440-525): the network that runs right before the crop stage.
//
// Convolutions 2..5 and afc_1 run as GEMMs on the tcgen05 split-K kernel of gemm_tc.cuh, fp32 accumulation, in one
// of two operand formats (template parameter Op, op_format.cuh): OpBf16x3 (bf16 hi/lo, three products per k-step:
// fp32-class accuracy) or OpFp16 (one fp16 product: 11 significand bits at the bf16 rate).  Everything around them
// is HBM-bound glue written here:
//   resize_bilinear_kernel   tf.image.resize_images(x, [128,128])                       :442   bit-exact float32
//   im2col_split_kernel      fp32 NHWC activation -> K-major GEMM operand (hi|lo / fp16) (conv2d SAME, :552)
//   bias_relu_pool_bn_kernel bias_add + relu (:553-554), max_pool 2x2 (:540-543), inference batch-norm (:446-454)
// The first layer (1 input channel) reuses stem_conv1_pool_bn_kernel, the dense head reuses fc_tail_kernel.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "op_format.cuh"

namespace hgru {

// TF 1.x ResizeBilinear (kernels/resize_bilinear_op.cc), align_corners = false: src = dst * (in / out),
// lower = floor(src), upper = min(lower + 1, in - 1), lerp = src - lower;
// top = tl + (tr - tl) * xl; bottom = bl + (br - bl) * xl; out = top + (bottom - top) * yl  -- all float32,
// no fused multiply-adds so the result equals the numpy float32 restatement bit for bit.
__global__ void __launch_bounds__(256)
resize_bilinear_kernel(const float* __restrict__ in, float* __restrict__ out, int N, int H, int W, int OH, int OW,
                       float sh, float sw) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  const size_t total = static_cast<size_t>(N) * OH * OW;
  if (i >= total) return;
  const int ox = i % OW;
  const int oy = (i / OW) % OH;
  const size_t n = i / (static_cast<size_t>(OW) * OH);
  const float* f = in + n * static_cast<size_t>(H) * W;
  if (OH == H && OW == W) {
    out[i] = f[static_cast<size_t>(oy) * W + ox];
    return;
  }
  const float sy = __fmul_rn(static_cast<float>(oy), sh), sx = __fmul_rn(static_cast<float>(ox), sw);
  const int y0 = static_cast<int>(floorf(sy)), x0 = static_cast<int>(floorf(sx));
  const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
  const float yl = __fsub_rn(sy, static_cast<float>(y0)), xl = __fsub_rn(sx, static_cast<float>(x0));
  const float tl = __ldg(f + static_cast<size_t>(y0) * W + x0), tr = __ldg(f + static_cast<size_t>(y0) * W + x1);
  const float bl = __ldg(f + static_cast<size_t>(y1) * W + x0), br = __ldg(f + static_cast<size_t>(y1) * W + x1);
  const float top = __fadd_rn(tl, __fmul_rn(__fsub_rn(tr, tl), xl));
  const float bot = __fadd_rn(bl, __fmul_rn(__fsub_rn(br, bl), xl));
  out[i] = __fadd_rn(top, __fmul_rn(__fsub_rn(bot, top), yl));
}

// im2col for a stride-1 SAME SxS convolution (tf.nn.conv2d, :552): row m = pixel (n, y, x), column
// k = (dy*S + dx)*Cin + ci  (the flatten order of the HWIO filter), written as bf16 hi at [k] and lo at
// [Kpad + k] (OpBf16x3, row pitch 2*Kpad) or as fp16 at [k] (OpFp16, row pitch Kpad); columns [K, Kpad) were zeroed.
// Cin % 8 == 0; one thread = 8 channels of one tap: 32 contiguous input bytes in, Op::kParts x 16 contiguous bytes out.
template <class Op = OpBf16x3>
__global__ void __launch_bounds__(256)
im2col_split_kernel(const float* __restrict__ in, typename Op::T* __restrict__ a, int N, int H, int W, int Cin,
                    int S, int Kpad) {
  const int c8n = Cin >> 3, taps = S * S, pad = (S - 1) / 2;
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  const size_t total = static_cast<size_t>(N) * H * W * taps * c8n;
  if (i >= total) return;
  const int c8 = i % c8n;
  const int t = (i / c8n) % taps;
  const size_t m = i / (static_cast<size_t>(c8n) * taps);
  const int x = m % W;
  const int y = (m / W) % H;
  const size_t n = m / (static_cast<size_t>(W) * H);
  const int yy = y + t / S - pad, xx = x + t % S - pad;
  float v[8];
  if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
    const float4* p = reinterpret_cast<const float4*>(in + ((n * H + yy) * W + xx) * Cin + c8 * 8);
    const float4 a0 = __ldg(p), a1 = __ldg(p + 1);
    v[0] = a0.x; v[1] = a0.y; v[2] = a0.z; v[3] = a0.w; v[4] = a1.x; v[5] = a1.y; v[6] = a1.z; v[7] = a1.w;
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = 0.f;
  }
  if constexpr (Op::kParts == 2) {
    __nv_bfloat162 hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat16 h0 = __float2bfloat16(v[2 * j]), h1 = __float2bfloat16(v[2 * j + 1]);
      hi[j] = __halves2bfloat162(h0, h1);
      lo[j] = __floats2bfloat162_rn(v[2 * j] - __bfloat162float(h0), v[2 * j + 1] - __bfloat162float(h1));
    }
    __nv_bfloat16* row = a + m * (2 * static_cast<size_t>(Kpad)) + static_cast<size_t>(t) * Cin + c8 * 8;
    *reinterpret_cast<uint4*>(row) = *reinterpret_cast<const uint4*>(hi);
    *reinterpret_cast<uint4*>(row + Kpad) = *reinterpret_cast<const uint4*>(lo);
  } else {
    typename Op::T2 h[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) h[j] = Op::cvt2(v[2 * j], v[2 * j + 1]);
    typename Op::T* row = a + m * static_cast<size_t>(Kpad) + static_cast<size_t>(t) * Cin + c8 * 8;
    *reinterpret_cast<uint4*>(row) = *reinterpret_cast<const uint4*>(h);
  }
}

// conv epilogue: sum of the split-K partials + bias, relu, 2x2/2 max-pool (even H, W: SAME needs no padding),
// inference batch-norm affine.  part [nsplit][N*H*W][C] fp32 -> out [N][H/2][W/2][C] fp32.  C % 4 == 0.
template <class Op = OpBf16x3>
__global__ void __launch_bounds__(256)
bias_relu_pool_bn_kernel(const float* __restrict__ part, int nsplit, const float* __restrict__ bias,
                         const float* __restrict__ scale, const float* __restrict__ shift, float* __restrict__ out,
                         typename Op::T* __restrict__ out_hi, typename Op::T* __restrict__ out_lo /* optional 16-bit
                         copies (same NHWC layout): the next layer's implicit-GEMM operand; out_lo: OpBf16x3 only */,
                         int N, int H, int W, int C) {
  const int c4n = C >> 2, PH = H >> 1, PW = W >> 1;
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  const size_t total = static_cast<size_t>(N) * PH * PW * c4n;
  if (i >= total) return;
  const int c4 = i % c4n;
  const size_t p = i / c4n;
  const int px = p % PW;
  const int py = (p / PW) % PH;
  const size_t n = p / (static_cast<size_t>(PW) * PH);
  const size_t M = static_cast<size_t>(N) * H * W;
  const float4 b = __ldg(reinterpret_cast<const float4*>(bias) + c4);
  float4 m = make_float4(0.f, 0.f, 0.f, 0.f);        // relu output is >= 0, so 0 is the identity of this max
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      const size_t row = (n * H + 2 * py + dy) * W + 2 * px + dx;
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int z = 0; z < nsplit; ++z) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(part + (z * M + row) * C) + c4);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      }
      m.x = fmaxf(m.x, s.x + b.x); m.y = fmaxf(m.y, s.y + b.y);
      m.z = fmaxf(m.z, s.z + b.z); m.w = fmaxf(m.w, s.w + b.w);
    }
  const float4 sc = __ldg(reinterpret_cast<const float4*>(scale) + c4);
  const float4 sf = __ldg(reinterpret_cast<const float4*>(shift) + c4);
  const float r[4] = {m.x * sc.x + sf.x, m.y * sc.y + sf.y, m.z * sc.z + sf.z, m.w * sc.w + sf.w};
  reinterpret_cast<float4*>(out + p * C)[c4] = make_float4(r[0], r[1], r[2], r[3]);
  if (out_hi) {
    if constexpr (Op::kParts == 2) {
      __nv_bfloat162 hi[2], lo[2];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const __nv_bfloat16 h0 = __float2bfloat16(r[2 * j]), h1 = __float2bfloat16(r[2 * j + 1]);
        hi[j] = __halves2bfloat162(h0, h1);
        lo[j] = __floats2bfloat162_rn(r[2 * j] - __bfloat162float(h0), r[2 * j + 1] - __bfloat162float(h1));
      }
      reinterpret_cast<uint2*>(out_hi + p * C)[c4] = *reinterpret_cast<const uint2*>(hi);
      reinterpret_cast<uint2*>(out_lo + p * C)[c4] = *reinterpret_cast<const uint2*>(lo);
    } else {
      const typename Op::T2 h[2] = {Op::cvt2(r[0], r[1]), Op::cvt2(r[2], r[3])};
      reinterpret_cast<uint2*>(out_hi + p * C)[c4] = *reinterpret_cast<const uint2*>(h);
    }
  }
}

// fp32 -> bf16 hi + lo (x ~ hi + lo to ~16 mantissa bits; OpBf16x3) or -> fp16 (OpFp16, lo unused), 8 elements per
// thread; n % 8 == 0.
template <class Op = OpBf16x3>
__global__ void __launch_bounds__(256)
split_operand_kernel(const float* __restrict__ in, typename Op::T* __restrict__ hi, typename Op::T* __restrict__ lo,
                  size_t n8) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= n8) return;
  const float4 a = __ldg(reinterpret_cast<const float4*>(in) + 2 * i), b = __ldg(reinterpret_cast<const float4*>(in) + 2 * i + 1);
  const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  if constexpr (Op::kParts == 2) {
    __nv_bfloat162 h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat16 h0 = __float2bfloat16(v[2 * j]), h1 = __float2bfloat16(v[2 * j + 1]);
      h[j] = __halves2bfloat162(h0, h1);
      l[j] = __floats2bfloat162_rn(v[2 * j] - __bfloat162float(h0), v[2 * j + 1] - __bfloat162float(h1));
    }
    reinterpret_cast<uint4*>(hi)[i] = *reinterpret_cast<const uint4*>(h);
    reinterpret_cast<uint4*>(lo)[i] = *reinterpret_cast<const uint4*>(l);
  } else {
    typename Op::T2 h[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) h[j] = Op::cvt2(v[2 * j], v[2 * j + 1]);
    reinterpret_cast<uint4*>(hi)[i] = *reinterpret_cast<const uint4*>(h);
  }
}

}  // namespace hgru
