// fp32 SIMT kernels for the hGRU-pose forward: the exact (<= 1e-4) path and the glue around the
// tensor-core convolutions.  All activations are NHWC fp32 (the reference's layout), weights HWIO.
// Reference call sites are cited per kernel (paths relative to /root/reference).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "op_format.cuh"

namespace hgru {

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + __expf(-x)); }
// tanh with ~1e-7 relative error (tanhf from libdevice; NOT tanh.approx, the 1e-4 path needs it)
__device__ __forceinline__ float tanhf_(float x) { return tanhf(x); }

// ------------------------------------------------------------------------------------------------
// Generic direct convolution, stride 1, SAME zero padding, fp32 (tf.nn.conv2d: hgru_module.py:531-548,
// hgru_pose.py:146), with the epilogue  y = act(conv + bias) * scale + shift  (bias_add + relu of
// hgru_pose.py:147-148 and the inference-mode batch_normalization that follows, :52-80).
// Block = 256 threads = 32 pixel-groups (8 px along x) x 8 channel-groups (8 co): a 16x16 pixel tile
// times 64 output channels; input patch and one filter row are staged in shared memory.
// ------------------------------------------------------------------------------------------------
template <int S>
struct ConvSimtCfg {
  static constexpr int PH = 16 + S - 1;
  static constexpr int PWraw = 16 + S - 1;
  static constexpr int PW = ((8 + ((8 + S - 1 + 3) / 4) * 4) + 3) / 4 * 4;   // room for float4 window loads
  static constexpr int NWIN = ((8 + S - 1 + 3) / 4) * 4;                       // window floats per thread
  static constexpr int kPatchFloats = 8 * PH * PW;
  static constexpr int kWFloats = S * 8 * 64;
  static constexpr int kSmemBytes = (kPatchFloats + kWFloats) * 4;
};

template <int S>
__global__ void __launch_bounds__(256)
conv_simt_kernel(const float* __restrict__ in, const float* __restrict__ w,
                 const float* __restrict__ bias, const float* __restrict__ scale,
                 const float* __restrict__ shift, float* __restrict__ out, int N, int H, int W,
                 int Ci, int Co, int relu) {
  using Cfg = ConvSimtCfg<S>;
  extern __shared__ float smem_f[];
  float* patch = smem_f;                       // [8 ci][PH][PW]
  float* wsm = smem_f + Cfg::kPatchFloats;     // [S dx][8 ci][64 co]
  constexpr int PAD = (S - 1) / 2;
  const int tiles_x = (W + 15) / 16;
  const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
  const int co0 = blockIdx.y * 64;
  const int n = blockIdx.z;
  const int tid = threadIdx.x;
  const int cg = tid & 7;            // channel group -> co0 + cg*8 .. +8
  const int pg = tid >> 3;           // pixel group 0..31
  const int prow = pg >> 1;          // 0..15
  const int pxg = (pg & 1) * 8;      // 0 or 8
  const int y_base = ty * 16 - PAD, x_base = tx * 16 - PAD;

  float acc[8][8];
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[j][c] = 0.f;

  for (int ci0 = 0; ci0 < Ci; ci0 += 8) {
    __syncthreads();
    // stage the input patch (zero fill outside the image / beyond Ci)
    for (int e = tid; e < Cfg::PH * Cfg::PWraw * 8; e += 256) {
      const int ci = e & 7;
      const int p = e >> 3;
      const int px = p % Cfg::PWraw, py = p / Cfg::PWraw;
      const int y = y_base + py, x = x_base + px;
      float v = 0.f;
      if (y >= 0 && y < H && x >= 0 && x < W && ci0 + ci < Ci)
        v = in[((static_cast<size_t>(n) * H + y) * W + x) * Ci + ci0 + ci];
      patch[(ci * Cfg::PH + py) * Cfg::PW + px] = v;
    }
    for (int dy = 0; dy < S; ++dy) {
      __syncthreads();
      for (int e = tid; e < S * 8 * 64; e += 256) {
        const int co = e & 63;
        const int ci = (e >> 6) & 7;
        const int dx = e >> 9;
        float v = 0.f;
        if (ci0 + ci < Ci && co0 + co < Co)
          v = w[((static_cast<size_t>(dy) * S + dx) * Ci + ci0 + ci) * Co + co0 + co];
        wsm[e] = v;
      }
      __syncthreads();
#pragma unroll 1
      for (int ci = 0; ci < 8; ++ci) {
        float win[Cfg::NWIN];
        const float4* src =
            reinterpret_cast<const float4*>(patch + (ci * Cfg::PH + prow + dy) * Cfg::PW + pxg);
#pragma unroll
        for (int j = 0; j < Cfg::NWIN / 4; ++j) {
          const float4 v = src[j];
          win[4 * j] = v.x; win[4 * j + 1] = v.y; win[4 * j + 2] = v.z; win[4 * j + 3] = v.w;
        }
#pragma unroll
        for (int dx = 0; dx < S; ++dx) {
          const float4* wp = reinterpret_cast<const float4*>(wsm + (dx * 8 + ci) * 64 + cg * 8);
          const float4 w0 = wp[0], w1 = wp[1];
          const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
          for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[j][c] = fmaf(win[j + dx], wv[c], acc[j][c]);
        }
      }
    }
  }
  const int y = ty * 16 + prow;
  if (y >= H) return;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int x = tx * 16 + pxg + j;
    if (x >= W) continue;
    float* dst = out + ((static_cast<size_t>(n) * H + y) * W + x) * Co;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const int co = co0 + cg * 8 + c;
      if (co < Co) {
        float v = acc[j][c] + (bias ? bias[co] : 0.f);
        if (relu) v = fmaxf(v, 0.f);
        if (scale) v = v * scale[co] + shift[co];
        dst[co] = v;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Internal activation layout: fp32 NHWC with the channel dimension padded to KP (a multiple of 16,
// pad channels are zero) so every pixel-chunk of 8 channels is 32 B (fp32) / 16 B (bf16) aligned.
// Elementwise kernels below: one thread = one pixel-chunk (8 channels).
// ------------------------------------------------------------------------------------------------
struct F8 { float v[8]; };
__device__ __forceinline__ F8 ld8(const float* p) {
  const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
  return F8{{a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}};
}
__device__ __forceinline__ void st8(float* p, const F8& f) {
  reinterpret_cast<float4*>(p)[0] = make_float4(f.v[0], f.v[1], f.v[2], f.v[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(f.v[4], f.v[5], f.v[6], f.v[7]);
}
__device__ __forceinline__ void st8_bf16(__nv_bfloat16* p, const F8& f) {
  __nv_bfloat162 h[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f.v[2 * i], f.v[2 * i + 1]);
  *reinterpret_cast<uint4*>(p) = *reinterpret_cast<const uint4*>(h);
}
// bf16 chunked operand copy [n][cg][pix][8]: address of chunk cg of pixel `pin` of frame n
__device__ __forceinline__ __nv_bfloat16* chunk_ptr(__nv_bfloat16* base, int n, int cg, size_t pin,
                                                    int HW, int CG) {
  return base + ((static_cast<size_t>(n) * CG + cg) * HW + pin) * 8;
}

// ------------------------------------------------------------------------------------------------
// Stem head: conv 3x3 (1 -> C) + bias + ReLU (hgru_pose.py:50,146-148), 2x2/2 max-pool (:51,134-137)
// and the inference batch-norm affine (:52-60), fused: [N,2H,2W,1] -> [N,H,W,KP] (+ bf16 hi/lo chunked copy).
// One thread = 4 horizontally adjacent pooled pixels x one chunk of 8 channels (blockIdx.y = the chunk, so a
// chunk of layout padding costs nothing and a warp writes 128 consecutive pixels of one chunk plane).  Every
// filter tap read from shared memory feeds 16 FMAs (4 pixels x the 2x2 pooling window); with one pixel per
// thread the kernel was bound by those shared-memory reads (145 us per 256 frames, now HBM-bound).
// `out` (fp32) may be null: the tensor-core path only consumes the bf16 hi/lo copy.
// ------------------------------------------------------------------------------------------------
constexpr int kStemPix = 4;      // pooled pixels per thread
__global__ void __launch_bounds__(256)
stem_conv1_pool_bn_kernel(const float* __restrict__ depth, const float* __restrict__ w /*[3][3][1][C]*/,
                          const float* __restrict__ bias, const float* __restrict__ scale,
                          const float* __restrict__ shift, float* __restrict__ out,
                          __nv_bfloat16* __restrict__ out_bf16, int N, int H, int W, int C, int KP, int quad) {
  __shared__ float wsm[9][8];      // this chunk's filter taps
  __shared__ float bsm[3][8];      // bias, scale, shift
  const int cg = blockIdx.y, CG = KP >> 3;
  if (threadIdx.x < 72) {
    const int t = threadIdx.x >> 3, c = cg * 8 + (threadIdx.x & 7);
    wsm[t][threadIdx.x & 7] = (c < C) ? w[t * C + c] : 0.f;
  } else if (threadIdx.x < 96) {
    const int v = (threadIdx.x - 72) >> 3, c = cg * 8 + (threadIdx.x & 7);
    const float* src = v == 0 ? bias : v == 1 ? scale : shift;
    bsm[v][threadIdx.x & 7] = (c < C) ? src[c] : 0.f;
  }
  __syncthreads();
  const int WQ = (W + kStemPix - 1) / kStemPix;
  const size_t g = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (g >= static_cast<size_t>(N) * H * WQ) return;
  const int xq = g % WQ;
  const int y = (g / WQ) % H;
  const int n = g / (static_cast<size_t>(WQ) * H);
  const int x0 = xq * kStemPix;
  const int IH = 2 * H, IW = 2 * W;
  float v[4][2 * kStemPix + 2];     // input rows 2y-1 .. 2y+2, columns 2x0-1 .. 2x0+8
  // the 8 inner columns start at a multiple of 8 floats: two 16-byte loads when the row pitch allows it
  const bool vec = (IW & 3) == 0 && 2 * x0 + 2 * kStemPix <= IW && (reinterpret_cast<uintptr_t>(depth) & 15) == 0;
#pragma unroll
  for (int rr = 0; rr < 4; ++rr) {
    const int yy = 2 * y - 1 + rr;
    const bool rowok = yy >= 0 && yy < IH;
    const float* row = depth + (static_cast<size_t>(n) * IH + yy) * IW;
    if (vec) {
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      const float4 lo = rowok ? __ldg(reinterpret_cast<const float4*>(row + 2 * x0)) : z4;
      const float4 hi = rowok ? __ldg(reinterpret_cast<const float4*>(row + 2 * x0 + 4)) : z4;
      v[rr][0] = (rowok && x0 > 0) ? __ldg(row + 2 * x0 - 1) : 0.f;
      v[rr][1] = lo.x; v[rr][2] = lo.y; v[rr][3] = lo.z; v[rr][4] = lo.w;
      v[rr][5] = hi.x; v[rr][6] = hi.y; v[rr][7] = hi.z; v[rr][8] = hi.w;
      v[rr][9] = (rowok && 2 * x0 + 8 < IW) ? __ldg(row + 2 * x0 + 8) : 0.f;
    } else {
#pragma unroll
      for (int q = 0; q < 2 * kStemPix + 2; ++q) {
        const int xx = 2 * x0 - 1 + q;
        v[rr][q] = (rowok && xx >= 0 && xx < IW) ? __ldg(row + xx) : 0.f;
      }
    }
  }
  const int nreal = C - cg * 8;     // real channels of this chunk (uniform over the block)
  float r[kStemPix][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (j < nreal) {
      float wt[9];
#pragma unroll
      for (int t = 0; t < 9; ++t) wt[t] = wsm[t][j];
      const float bj = bsm[0][j], sj = bsm[1][j], hj = bsm[2][j];
#pragma unroll
      for (int px = 0; px < kStemPix; ++px) {
        float m = -INFINITY;
#pragma unroll
        for (int py = 0; py < 2; ++py)
#pragma unroll
          for (int qx = 0; qx < 2; ++qx) {
            float a = 0.f;
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
              for (int dx = 0; dx < 3; ++dx) a = fmaf(v[py + dy][2 * px + qx + dx], wt[dy * 3 + dx], a);
            m = fmaxf(m, a);
          }
        r[px][j] = fmaxf(m + bj, 0.f) * sj + hj;      // relu and max commute
      }
    } else {
#pragma unroll
      for (int px = 0; px < kStemPix; ++px) r[px][j] = 0.f;     // layout padding
    }
  }
  const size_t HW = static_cast<size_t>(H) * W;
#pragma unroll
  for (int px = 0; px < kStemPix; ++px) {
    const int x = x0 + px;
    if (x >= W) break;
    const size_t pin = static_cast<size_t>(y) * W + x;
    F8 rv;
#pragma unroll
    for (int j = 0; j < 8; ++j) rv.v[j] = r[px][j];
    if (out) {
      if (quad) {   // quad-chunked fp32 [n][c/4][pix][4] (tensor-core path)
        float* o = out + ((static_cast<size_t>(n) * (KP >> 2) + 2 * cg) * HW + pin) * 4;
        *reinterpret_cast<float4*>(o) = make_float4(rv.v[0], rv.v[1], rv.v[2], rv.v[3]);
        *reinterpret_cast<float4*>(o + HW * 4) = make_float4(rv.v[4], rv.v[5], rv.v[6], rv.v[7]);
      } else {
        st8(out + (static_cast<size_t>(n) * HW + pin) * KP + cg * 8, rv);
      }
    }
    if (out_bf16) {
      // operand copy for the tensor-core conv_2, split into bf16 hi + lo parts (chunk planes [0,CG) and
      // [CG,2CG)): the pooled depth map is smooth, so plain bf16 rounding errors add up coherently
      F8 hi, lo;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        hi.v[j] = __bfloat162float(__float2bfloat16(rv.v[j]));
        lo.v[j] = rv.v[j] - hi.v[j];
      }
      st8_bf16(chunk_ptr(out_bf16, n, cg, pin, H * W, 2 * CG), hi);
      st8_bf16(chunk_ptr(out_bf16, n, CG + cg, pin, H * W, 2 * CG), lo);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// 1x1 gate convolution + sigmoid (hgru_module.py:696-707 and :729-740):
//   G = sigmoid(in *1x1 wg + bg);  optional gated copy  out_mul = in . G  (:709-711).
// Block = 64 pixels; wg [KP][KP] and the pixel tile in shared memory; thread = pixel x 8 outputs.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gate1x1_kernel(const float* __restrict__ in, const float* __restrict__ wg /*[ci][co] KPxKP*/,
               const float* __restrict__ bg, float* __restrict__ out_g, float* __restrict__ out_mul,
               __nv_bfloat16* __restrict__ out_mul_bf16, size_t npix, int KP, int kreal, int HW) {
  extern __shared__ float smem_f[];
  float* wsm = smem_f;                 // [KP][KP]
  float* xin = smem_f + KP * KP;       // [64][KP+1]
  const int tid = threadIdx.x;
  const int CG = KP >> 3;
  const size_t p0 = blockIdx.x * static_cast<size_t>(64);
  for (int e = tid; e < KP * KP; e += 256) wsm[e] = wg[e];
  for (int e = tid; e < 64 * KP; e += 256) {
    const int pp = e / KP, c = e - pp * KP;
    xin[pp * (KP + 1) + c] = (p0 + pp < npix) ? in[(p0 + pp) * KP + c] : 0.f;
  }
  __syncthreads();
  const int pp = tid & 63;
  const size_t p = p0 + pp;
  if (p >= npix) return;
  const int n = p / HW;
  const size_t pin = p - static_cast<size_t>(n) * HW;
  for (int cg = tid >> 6; cg < CG; cg += 4) {
    F8 a;
#pragma unroll
    for (int j = 0; j < 8; ++j) a.v[j] = 0.f;
    for (int ci = 0; ci < KP; ++ci) {
      const float xv = xin[pp * (KP + 1) + ci];
      const float4 w0 = *reinterpret_cast<const float4*>(wsm + ci * KP + cg * 8);
      const float4 w1 = *reinterpret_cast<const float4*>(wsm + ci * KP + cg * 8 + 4);
      a.v[0] = fmaf(xv, w0.x, a.v[0]); a.v[1] = fmaf(xv, w0.y, a.v[1]);
      a.v[2] = fmaf(xv, w0.z, a.v[2]); a.v[3] = fmaf(xv, w0.w, a.v[3]);
      a.v[4] = fmaf(xv, w1.x, a.v[4]); a.v[5] = fmaf(xv, w1.y, a.v[5]);
      a.v[6] = fmaf(xv, w1.z, a.v[6]); a.v[7] = fmaf(xv, w1.w, a.v[7]);
    }
    F8 g, mv;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = cg * 8 + j;
      g.v[j] = (c < kreal) ? sigmoidf_(a.v[j] + bg[c]) : 0.f;
      mv.v[j] = xin[pp * (KP + 1) + c] * g.v[j];
    }
    if (out_g) st8(out_g + p * KP + cg * 8, g);
    if (out_mul) st8(out_mul + p * KP + cg * 8, mv);
    if (out_mul_bf16) st8_bf16(chunk_ptr(out_mul_bf16, n, cg, pin, HW, CG), mv);
  }
}

// ------------------------------------------------------------------------------------------------
// input_integration (hgru_module.py:795-804):  H1 = tanh(X - (beta*H2 + nu) * C1),  C1 already
// includes lateral_bias (:657).  Optionally emits the bf16 chunked operand copy of H1.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
h1_kernel(const float* __restrict__ X, const float* __restrict__ H2, const float* __restrict__ C1,
          const float* __restrict__ beta, const float* __restrict__ nu, float* __restrict__ H1,
          __nv_bfloat16* __restrict__ H1_bf16, size_t nchunks, int KP, int kreal, int HW) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= nchunks) return;
  const int CG = KP >> 3;
  const int cg = i % CG;
  const size_t p = i / CG;
  const F8 x = ld8(X + i * 8), h2 = ld8(H2 + i * 8), c1 = ld8(C1 + i * 8);
  const F8 b = ld8(beta + cg * 8), nv = ld8(nu + cg * 8);
  F8 h1;
#pragma unroll
  for (int j = 0; j < 8; ++j)
    h1.v[j] = (cg * 8 + j < kreal) ? tanhf_(x.v[j] - (b.v[j] * h2.v[j] + nv.v[j]) * c1.v[j]) : 0.f;
  st8(H1 + i * 8, h1);
  if (H1_bf16) {
    const int n = p / HW;
    st8_bf16(chunk_ptr(H1_bf16, n, cg, p - static_cast<size_t>(n) * HW, HW, CG), h1);
  }
}

// ------------------------------------------------------------------------------------------------
// output_integration + adaptation (hgru_module.py:806-823, 847-849):
//   e = gamma*C2; Ht = tanh(kappa*(H1+e) + omega*(H1*e)); H2 = (G2*H2 + (1-G2)*Ht) * rho_t
// In place on H2; optional trace copies are taken by the caller afterwards.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
h2_kernel(const float* __restrict__ H1, const float* __restrict__ C2, const float* __restrict__ G2,
          const float* __restrict__ gamma, const float* __restrict__ kappa,
          const float* __restrict__ omega, const float* __restrict__ rho, int t,
          float* __restrict__ H2, size_t nchunks, int KP, int kreal) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= nchunks) return;
  const int CG = KP >> 3;
  const int cg = i % CG;
  const F8 h1 = ld8(H1 + i * 8), c2 = ld8(C2 + i * 8), g = ld8(G2 + i * 8), h2 = ld8(H2 + i * 8);
  const F8 ga = ld8(gamma + cg * 8), ka = ld8(kappa + cg * 8), om = ld8(omega + cg * 8);
  const float r = rho[t];
  F8 o;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float e = ga.v[j] * c2.v[j];
    const float ht = tanhf_(ka.v[j] * (h1.v[j] + e) + om.v[j] * (h1.v[j] * e));
    o.v[j] = (cg * 8 + j < kreal) ? (g.v[j] * h2.v[j] + (1.f - g.v[j]) * ht) * r : 0.f;
  }
  st8(H2 + i * 8, o);
}

// NHWC [.., k] -> NHWC [.., KP] (zero pad channels) and back; optional per-channel affine on unpad.
__global__ void __launch_bounds__(256)
pad_channels_kernel(const float* __restrict__ in, float* __restrict__ out, size_t npix, int k, int KP) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= npix * KP) return;
  const int c = i % KP;
  const size_t p = i / KP;
  out[i] = (c < k) ? in[p * k + c] : 0.f;
}
__global__ void __launch_bounds__(256)
unpad_channels_kernel(const float* __restrict__ in, float* __restrict__ out, size_t npix, int k, int KP) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= npix * k) return;
  const int c = i % k;
  const size_t p = i / k;
  out[i] = in[p * KP + c];
}
// fp32 padded NHWC -> bf16 chunked operand copy
__global__ void __launch_bounds__(256)
to_chunked_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, size_t nchunks,
                       int KP, int HW) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= nchunks) return;
  const int CG = KP >> 3;
  const int cg = i % CG;
  const size_t p = i / CG;
  const int n = p / HW;
  st8_bf16(chunk_ptr(out, n, cg, p - static_cast<size_t>(n) * HW, HW, CG), ld8(in + i * 8));
}

// ------------------------------------------------------------------------------------------------
// Layout conversions at the boundary of the tensor-core path, whose fp32 state tensors are
// quad-chunked [n][c/4][pix][4] (see hconv_tc.cuh).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
nhwc_to_quad_kernel(const float* __restrict__ in, float* __restrict__ out, size_t npix, int k, int KP, int HW) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;   // over [n][quad][pin]
  const int Q = KP >> 2;
  if (i >= npix * Q) return;
  const size_t pin = i % HW;
  const int q = (i / HW) % Q;
  const size_t n = i / (static_cast<size_t>(HW) * Q);
  const float* src = in + (n * HW + pin) * k + 4 * q;
  float4 v;
  v.x = (4 * q + 0 < k) ? src[0] : 0.f;
  v.y = (4 * q + 1 < k) ? src[1] : 0.f;
  v.z = (4 * q + 2 < k) ? src[2] : 0.f;
  v.w = (4 * q + 3 < k) ? src[3] : 0.f;
  reinterpret_cast<float4*>(out)[i] = v;
}
__global__ void __launch_bounds__(256)
quad_to_nhwc_kernel(const float* __restrict__ in, float* __restrict__ out, size_t npix, int k, int KP, int HW) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;   // over [npix][k]
  if (i >= npix * k) return;
  const int c = i % k;
  const size_t p = i / k;
  const size_t n = p / HW, pin = p - n * HW;
  out[i] = in[((n * (KP >> 2) + (c >> 2)) * HW + pin) * 4 + (c & 3)];
}

// fp16 oct-chunked [n][c/8][pix][8] (H1 / G2 of the fused bf16 pipeline, see hconv_tc.cuh) -> fp32 NHWC
__global__ void __launch_bounds__(256)
oct_half_to_nhwc_kernel(const __half* __restrict__ in, float* __restrict__ out, size_t npix, int k, int KP, int HW) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;   // over [npix][k]
  if (i >= npix * k) return;
  const int c = i % k;
  const size_t p = i / k;
  const size_t n = p / HW, pin = p - n * HW;
  out[i] = __half2float(in[((n * (KP >> 3) + (c >> 3)) * HW + pin) * 8 + (c & 7)]);
}

// bf16 hi | lo chunk planes [n][2*CG][pix][8] (the operand copies of the tensor-core stem) -> fp32 NHWC
__global__ void __launch_bounds__(256)
split_chunks_to_nhwc_kernel(const __nv_bfloat16* __restrict__ in, float* __restrict__ out, size_t npix, int k, int CG,
                            int HW) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;   // over [npix][k]
  if (i >= npix * k) return;
  const int c = i % k;
  const size_t p = i / k;
  const size_t n = p / HW, pin = p - n * HW;
  const size_t hi = ((n * 2 * CG + (c >> 3)) * HW + pin) * 8 + (c & 7);
  const size_t lo = ((n * 2 * CG + CG + (c >> 3)) * HW + pin) * 8 + (c & 7);
  out[i] = __bfloat162float(in[hi]) + __bfloat162float(in[lo]);
}

// ------------------------------------------------------------------------------------------------
// Exact fp32 1x1 gate on the quad-chunked state layout (bf16x3 mode; hgru_module.py:696-711, 729-740):
//   g = sigmoid(in *1x1 wg + bg);  out_g (quad fp32) = g              when out_g  != nullptr   (G2)
//                                  out_act = bf16 hi | lo of g . in   when out_act != nullptr  (gated operand)
// 256 pixels per block (i_r in shared memory), thread = 4 pixels x 8 output channels.
// ------------------------------------------------------------------------------------------------
constexpr int kInitPix = 256;     // pixels per block of gate_quad_split_kernel (4 per thread)
// `lo_off` > 0: the operand goes to TWO tensors in the tap-stacked kernel's layout instead (hi at out_act, lo lo_off
// elements behind it; `act_pad` zero rows on top of every chunk plane of width W, and with act_pad > 0 the last chunk
// is the row-packed plane P[y][x][j] = v(y + j, x) of channel KP - 8: see StackCfg::REM in hconv_stack.cuh).
__device__ __forceinline__ void st8_stacked(__nv_bfloat16* base, int n, int cg, int CG, size_t pin, int HW, int W,
                                            int act_pad, const F8& v) {
  const size_t plane = static_cast<size_t>(HW) + static_cast<size_t>(act_pad) * W;
  const size_t pp = pin + static_cast<size_t>(act_pad) * W;
  __nv_bfloat16* o = base + ((static_cast<size_t>(n) * CG + cg) * plane + pp) * 8;
  if (act_pad == 0 || cg != CG - 1) {
    st8_bf16(o, v);
  } else {
    const __nv_bfloat16 b = __float2bfloat16(v.v[0]);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j - static_cast<ptrdiff_t>(j) * W * 8] = b;
  }
}

__global__ void __launch_bounds__(256)
gate_quad_split_kernel(const float* __restrict__ inq, const float* __restrict__ wg /*[KP][KP]*/,
                       const float* __restrict__ bg, float* __restrict__ out_g, __nv_bfloat16* __restrict__ out_act,
                       size_t npix, int k, int KP, int HW, size_t lo_off = 0, int W = 0, int act_pad = 0) {
  extern __shared__ float smem_f[];
  float* wsm = smem_f;                 // [KP][KP]
  float* xin = smem_f + KP * KP;       // [kInitPix][KP+1]
  const int tid = threadIdx.x;
  const int CG = KP >> 3;
  const size_t p0 = blockIdx.x * static_cast<size_t>(kInitPix);
  for (int e = tid; e < KP * KP; e += 256) wsm[e] = wg[e];
  for (int e = tid; e < kInitPix * (KP >> 2); e += 256) {        // one float4 = 4 channels of one pixel
    const int pp = e % kInitPix, q = e / kInitPix;
    const size_t p = p0 + pp;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p < npix) {
      const size_t n = p / HW, pin = p - n * HW;
      v = *reinterpret_cast<const float4*>(inq + ((n * (KP >> 2) + q) * HW + pin) * 4);
    }
    float* d = xin + pp * (KP + 1) + 4 * q;
    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
  }
  __syncthreads();
  const int pq = tid & 63;
  for (int cg = tid >> 6; cg < CG; cg += 4) {
    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    for (int ci = 0; ci < KP; ++ci) {
      const float4 w0 = *reinterpret_cast<const float4*>(wsm + ci * KP + cg * 8);
      const float4 w1 = *reinterpret_cast<const float4*>(wsm + ci * KP + cg * 8 + 4);
      const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float xv = xin[(pq + 64 * i) * (KP + 1) + ci];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(xv, wv[j], acc[i][j]);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int pp = pq + 64 * i;
      const size_t p = p0 + pp;
      if (p >= npix) continue;
      const size_t n = p / HW, pin = p - n * HW;
      F8 g, hi, lo;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int c = cg * 8 + j;
        g.v[j] = (c < k) ? sigmoidf_(acc[i][j] + bg[c]) : 0.f;
        const float a = g.v[j] * xin[pp * (KP + 1) + c];
        hi.v[j] = __bfloat162float(__float2bfloat16(a));
        lo.v[j] = a - hi.v[j];
      }
      if (out_g) {
        float* o = out_g + ((n * (KP >> 2) + 2 * cg) * HW + pin) * 4;
        *reinterpret_cast<float4*>(o) = make_float4(g.v[0], g.v[1], g.v[2], g.v[3]);
        *reinterpret_cast<float4*>(o + static_cast<size_t>(HW) * 4) = make_float4(g.v[4], g.v[5], g.v[6], g.v[7]);
      }
      if (out_act && lo_off) {
        st8_stacked(out_act, static_cast<int>(n), cg, CG, pin, HW, W, act_pad, hi);
        st8_stacked(out_act + lo_off, static_cast<int>(n), cg, CG, pin, HW, W, act_pad, lo);
      } else if (out_act) {
        st8_bf16(chunk_ptr(out_act, static_cast<int>(n), cg, pin, HW, 2 * CG), hi);
        st8_bf16(chunk_ptr(out_act, static_cast<int>(n), CG + cg, pin, HW, 2 * CG), lo);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Readout FC1 (hgru_pose.py:91,156-163): part[z][m][j] = sum_{kk in slice z} (a[m][kk]*sc[kk%k]+sh[kk%k]) * Wt[kk][j]
// (a is read from the channel-padded activation buffer; kk enumerates (h, w, c) like tf.reshape)
// The per-channel affine on A is the inference batch-norm of the hGRU output (:82-90).
// Split-K SGEMM: block tile 64(m) x 64(j), 256 threads, 4x4 per thread, K step 16.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
fc1_splitk_kernel(const float* __restrict__ A, const float* __restrict__ Wt,
                  const float* __restrict__ sc, const float* __restrict__ sh,
                  float* __restrict__ part, int M, int K, int Nout, int kch, int KP, int kslice) {
  __shared__ float As[16][64 + 4];
  __shared__ float Bs[16][64 + 4];
  const int tid = threadIdx.x;
  const int j0 = blockIdx.x * 64, m0 = blockIdx.y * 64, z = blockIdx.z;
  const int kb = z * kslice, ke = min(K, kb + kslice);
  const int tm = (tid >> 4) * 4, tj = (tid & 15) * 4;
  float acc[4][4] = {};
  for (int k0 = kb; k0 < ke; k0 += 16) {
    // A tile: 64 rows x 16 k  (row-major A[m][K]); each thread loads 4 elements
    {
      const int r = tid >> 2, kk = (tid & 3) * 4;
      const int m = m0 + r;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int kidx = k0 + kk + q;
        float v = 0.f;
        if (m < M && kidx < ke) {
          // A is the channel-padded activation [M][K/kch pixels][KP]; kidx runs over (pixel, real channel)
          const int pix = kidx / kch, c = kidx - pix * kch;
          v = A[(static_cast<size_t>(m) * (K / kch) + pix) * KP + c] * sc[c] + sh[c];
        }
        As[kk + q][r] = v;
      }
    }
    {
      const int kk = tid >> 4, jj = (tid & 15) * 4;
      const int kidx = k0 + kk;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int j = j0 + jj + q;
        Bs[kk][jj + q] = (kidx < ke && j < Nout) ? Wt[static_cast<size_t>(kidx) * Nout + j] : 0.f;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) { a[q] = As[kk][tm + q]; b[q] = Bs[kk][tj + q]; }
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int r = 0; r < 4; ++r) acc[q][r] = fmaf(a[q], b[r], acc[q][r]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int m = m0 + tm + q;
    if (m >= M) continue;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int j = j0 + tj + r;
      if (j < Nout) part[(static_cast<size_t>(z) * M + m) * Nout + j] = acc[q][r];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Readout tail: fc1 = sum_z part + b1 (hgru_pose.py:91); relu (:92); batch-norm affine (:95-103,
// resolution R-D5); fc_out (:104, R-D6): out[m][o] = sum_j r[j] * W2[j][o] + b2[o].
// One block per frame.
// ------------------------------------------------------------------------------------------------
constexpr int kFcTailScratch = 256;      // floats of shared memory behind r[Hid]
__global__ void __launch_bounds__(256)
fc_tail_kernel(const float* __restrict__ part, int nsplit, const float* __restrict__ b1,
               const float* __restrict__ sc, const float* __restrict__ sh,
               const float* __restrict__ W2, const float* __restrict__ b2, float* __restrict__ fc1_out,
               float* __restrict__ out, int M, int Hid, int Nout) {
  extern __shared__ float r[];      // [Hid] + [kFcTailScratch]
  float* scratch = r + Hid;
  const int m = blockIdx.x;
  // split-K partial sums, added in slice order.  Everything here is latency-bound (a few hundred KB per frame),
  // so the loops are shaped to keep many independent loads in flight: 4 columns per thread as one 16-byte load,
  // six slices per round.
  const size_t zs = static_cast<size_t>(M) * Hid;
  if ((Hid & 3) == 0) {
    for (int j = 4 * threadIdx.x; j < Hid; j += 4 * blockDim.x) {
      const float* pj = part + static_cast<size_t>(m) * Hid + j;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
      int z = 0;
      for (; z + 6 <= nsplit; z += 6) {
        float4 v[6];
#pragma unroll
        for (int q = 0; q < 6; ++q) v[q] = __ldg(reinterpret_cast<const float4*>(pj + (z + q) * zs));
#pragma unroll
        for (int q = 0; q < 6; ++q) { a.x += v[q].x; a.y += v[q].y; a.z += v[q].z; a.w += v[q].w; }
      }
      for (; z < nsplit; ++z) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(pj + z * zs));
        a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
      }
      const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float t = av[q] + b1[j + q];
        if (fc1_out) fc1_out[static_cast<size_t>(m) * Hid + j + q] = t;
        r[j + q] = fmaxf(t, 0.f) * sc[j + q] + sh[j + q];
      }
    }
  } else {
    for (int j = threadIdx.x; j < Hid; j += blockDim.x) {
      const float* pj = part + static_cast<size_t>(m) * Hid + j;
      float a = 0.f;
      for (int z = 0; z < nsplit; ++z) a += pj[z * zs];
      a += b1[j];
      if (fc1_out) fc1_out[static_cast<size_t>(m) * Hid + j] = a;
      r[j] = fmaxf(a, 0.f) * sc[j] + sh[j];
    }
  }
  __syncthreads();
  // fc_out: thread = (group g, output o); a group walks the rows j = g, g + G, ... of W2 [Hid][Nout], so a warp
  // reads consecutive outputs of one row (the old lane-per-row mapping touched 32 cache lines per load)
  for (int o0 = 0; o0 < Nout; o0 += kFcTailScratch) {
    const int no = min(Nout - o0, kFcTailScratch);
    const int G = kFcTailScratch / no;
    const int g = threadIdx.x / no, o = threadIdx.x - g * no;
    if (g < G) {
      const float* wcol = W2 + o0 + o;
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      int j = g;
      for (; j + 15 * G < Hid; j += 16 * G) {      // 16 independent loads per round
        float w[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) w[q] = __ldg(wcol + static_cast<size_t>(j + q * G) * Nout);
#pragma unroll
        for (int q = 0; q < 16; ++q) acc[q & 3] = fmaf(r[j + q * G], w[q], acc[q & 3]);
      }
      for (; j < Hid; j += G) acc[0] = fmaf(r[j], __ldg(wcol + static_cast<size_t>(j) * Nout), acc[0]);
      scratch[g * no + o] = (acc[0] + acc[1]) + (acc[2] + acc[3]);
    }
    __syncthreads();
    if (threadIdx.x < no) {
      float a = 0.f;
      for (int gg = 0; gg < G; ++gg) a += scratch[gg * no + threadIdx.x];
      out[static_cast<size_t>(m) * Nout + o0 + threadIdx.x] = a + b2[o0 + threadIdx.x];
    }
    __syncthreads();
  }
}

// batch-norm inference fold: scale = gamma / sqrt(var + eps), shift = beta - mean * scale
__global__ void bn_fold_kernel(const float* gamma, const float* beta, const float* mean,
                               const float* var, float eps, float* scale, float* shift, int c) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c) return;
  const float s = gamma[i] / sqrtf(var[i] + eps);
  scale[i] = s;
  shift[i] = beta[i] - mean[i] * s;
}

// Weight packing for the tcgen05 conv: HWIO fp32 [S][S][k][k] -> F [KSTEPS][taps][2][CO_PAD][8 ci]
// (F: the 16-bit operand format, op_format.cuh).
// `ci_wrap` > 0: input channel index wraps at ci_wrap (the operand carries hi and lo bf16 halves of the
// same channels in consecutive chunk planes, both multiplied by the same weights).
template <class F = OpBf16>
__global__ void pack_weights_kernel(const float* __restrict__ w, typename F::T* __restrict__ wpk,
                                    int taps, int k, int ksteps, int co_pad, int ci_wrap = 0) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  const size_t total = static_cast<size_t>(ksteps) * taps * 2 * co_pad * 8;
  if (i >= total) return;
  const int j = i & 7;
  size_t r = i >> 3;
  const int co = r % co_pad; r /= co_pad;
  const int ch = r & 1; r >>= 1;
  const int tap = r % taps;
  const int q = r / taps;
  int ci = q * 16 + ch * 8 + j;
  if (ci_wrap > 0 && ci >= ci_wrap) ci -= ci_wrap;
  float v = 0.f;
  if (ci < k && co < k) v = w[(static_cast<size_t>(tap) * k + ci) * k + co];
  wpk[i] = F::cvt(v);
}

// Weight packing for the paired-tap schedule of the fused 64-channel 15x15 kernel (TcConvCfg::kPairTap):
// HWIO fp32 [15][15][k][k] -> F [kstep q][dy][block b = 0..7][2 chunks][128 rows][8 ci]
//   block 0: rows 0-63 = tap dx = 7 (output channels), rows 64-127 = zero
//   block 1 + p (p = 0..6): rows 0-63 = tap dx = p + 8, rows 64-127 = tap dx = p
template <class F = OpBf16>
__global__ void pack_weights_pairtap_kernel(const float* __restrict__ w, typename F::T* __restrict__ wpk, int k,
                                            int ksteps) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  const size_t total = static_cast<size_t>(ksteps) * 15 * 8 * 2 * 128 * 8;
  if (i >= total) return;
  const int j = i & 7;
  size_t r = i >> 3;
  const int row = r % 128; r /= 128;
  const int ch = r & 1; r >>= 1;
  const int b = r % 8; r /= 8;
  const int dy = r % 15;
  const int q = static_cast<int>(r / 15);
  int dx = -1;
  if (b == 0) { if (row < 64) dx = 7; }
  else dx = (row < 64) ? (b - 1 + 8) : (b - 1);
  const int co = row & 63;
  const int ci = q * 16 + ch * 8 + j;
  float v = 0.f;
  if (dx >= 0 && ci < k && co < k) v = w[((static_cast<size_t>(dy) * 15 + dx) * k + ci) * k + co];
  wpk[i] = F::cvt(v);
}

// Weight packing for the SPLIT3 tensor-core conv (hi = bf16(w), lo = bf16(w - hi)): per 16-channel group q
//   [taps][2 chunks][2*co_pad n][8 ci]   n < co_pad: w_hi[.., co = n],  n >= co_pad: w_lo[.., co = n - co_pad]   (a_hi pass)
//   [taps][2 chunks][co_pad n][8 ci]     w_hi                                                                  (a_lo pass)
// i.e. 3 * taps * 2 * co_pad * 8 elements per group.
__global__ void pack_weights_split3_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wpk,
                                           int taps, int k, int ksteps, int co_pad) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  const size_t group = static_cast<size_t>(3) * taps * 2 * co_pad * 8;
  if (i >= group * ksteps) return;
  const int q = static_cast<int>(i / group);
  size_t r = i - q * group;
  const size_t wide_elems = static_cast<size_t>(taps) * 2 * (2 * co_pad) * 8;
  int tap, ch, n, j, lo;
  if (r < wide_elems) {
    j = r & 7; r >>= 3;
    n = r % (2 * co_pad); r /= (2 * co_pad);
    ch = r & 1; tap = static_cast<int>(r >> 1);
    lo = n >= co_pad;
    if (lo) n -= co_pad;
  } else {
    r -= wide_elems;
    j = r & 7; r >>= 3;
    n = r % co_pad; r /= co_pad;
    ch = r & 1; tap = static_cast<int>(r >> 1);
    lo = 0;
  }
  const int ci = q * 16 + ch * 8 + j;
  float v = 0.f;
  if (ci < k && n < k) v = w[(static_cast<size_t>(tap) * k + ci) * k + n];
  const __nv_bfloat16 hi = __float2bfloat16(v);
  wpk[i] = lo ? __float2bfloat16(v - __bfloat162float(hi)) : hi;
}

}  // namespace hgru
