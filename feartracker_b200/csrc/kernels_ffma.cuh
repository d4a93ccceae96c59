// CUDA-core (FFMA) kernels of the FEAR-XS hot path, channels-last (NHWC) fp32.
//
// These are the always-correct implementations every stage can run on; the tcgen05 kernels in
// kernels_tc.cuh replace the dense contractions (1x1 convs, correlation) where they apply.
// Layout: activations [B][H][W][C] fp32, C a multiple of 4 (float4 over channels); 1x1 weights
// torch-native [Cout][Cin] ("K-major"); depthwise weights [k*k][C]; stem weights [27][16].
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/fear_b200.h"

namespace fear {

// ------------------------------------------------------------------------------------------
// Stem: conv3x3 stride 2 pad 1, 3 -> 16, + folded BN bias + ReLU.   NCHW in -> NHWC out.
// (fbnet_c xif0_0; reference call site fear_net.py:58-61.)  One thread per output pixel, all 16
// output channels in registers; the 432 weights are broadcast from shared memory.
// ------------------------------------------------------------------------------------------
// U8 = true: img is a uint8 HWC crop (B,H,W,3) as the tracker holds it; the ImageNet normalisation of
// Tracker._preprocess_image (reference base_tracker.py:69-81,97-103: (x - mean*255) * (1/(std*255)), float32,
// subtract then multiply) is applied on the fly with the same two roundings, so the result is bit-identical
// to normalising on the host while the host->device copy shrinks 4x.
struct StemNorm {
  float mean[3], inv[3];
};
template <bool U8>
__global__ void __launch_bounds__(128) stem_conv3x3s2_kernel(const void* __restrict__ img_, const float* __restrict__ w,
                                                             const float* __restrict__ bias, float* __restrict__ out,
                                                             int B, int H, int W, StemNorm nrm) {
  __shared__ float sw[27 * 16];
  __shared__ float sb[16];
  for (int i = threadIdx.x; i < 27 * 16; i += blockDim.x) sw[i] = w[i];
  if (threadIdx.x < 16) sb[threadIdx.x] = bias[threadIdx.x];
  __syncthreads();
  // CTA = 32 output columns x 4 output rows (one warp per row): vertically adjacent rows share an input
  // row, which now hits L1 instead of being re-read from L2 by another CTA.
  const int Ho = H >> 1, Wo = W >> 1;
  const int xg = (Wo + 31) / 32, yg = (Ho + 3) / 4;
  int t = blockIdx.x;
  const int bx = t % xg;
  t /= xg;
  const int by = t % yg;
  const int b = t / yg;
  const int ox = bx * 32 + (threadIdx.x & 31);
  const int oy = by * 4 + (threadIdx.x >> 5);
  if (ox >= Wo || oy >= Ho || b >= B) return;
  const long long idx = ((long long)b * Ho + oy) * Wo + ox;
  float acc[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) acc[c] = sb[c];
  const float* base = static_cast<const float*>(img_) + (long long)b * 3 * H * W;
  const uint8_t* base8 = static_cast<const uint8_t*>(img_) + (long long)b * 3 * H * W;
#pragma unroll
  for (int ci = 0; ci < 3; ++ci) {
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int iy = oy * 2 - 1 + ky;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int ix = ox * 2 - 1 + kx;
        float v = 0.f;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
          if (U8)
            v = __fmul_rn(__fsub_rn((float)__ldg(base8 + ((long long)iy * W + ix) * 3 + ci), nrm.mean[ci]), nrm.inv[ci]);
          else
            v = __ldg(base + ((long long)ci * H + iy) * W + ix);
        }
        const float* wr = sw + (ci * 9 + ky * 3 + kx) * 16;
#pragma unroll
        for (int c = 0; c < 16; ++c) acc[c] = fmaf(v, wr[c], acc[c]);
      }
    }
  }
  float4* o = reinterpret_cast<float4*>(out + idx * 16);
#pragma unroll
  for (int q = 0; q < 4; ++q)
    o[q] = make_float4(fmaxf(acc[4 * q], 0.f), fmaxf(acc[4 * q + 1], 0.f), fmaxf(acc[4 * q + 2], 0.f),
                       fmaxf(acc[4 * q + 3], 0.f));
}

// ------------------------------------------------------------------------------------------
// Depthwise KxK conv (pad K/2, stride S) NHWC, optional bias / ReLU.  One thread per
// (pixel, 4 channels): neighbouring threads walk the channel dimension => 16-byte coalesced
// loads; the K*K taps of a pixel hit L1 (each input value is reused by up to K*K/S^2 outputs).
// Backbone dw (+BN+ReLU): mobile_cv IRF block; head dw: SepConv.depthwise, blocks.py:57-66.
// ------------------------------------------------------------------------------------------
template <int K, int S, bool RELU, bool BIAS>
__global__ void __launch_bounds__(256) dw_conv_nhwc_kernel(const float4* __restrict__ in, const float4* __restrict__ w,
                                                           const float4* __restrict__ bias, float4* __restrict__ out,
                                                           int B, int H, int W, int C4) {
  const int Ho = H / S, Wo = W / S;
  const long long total = (long long)B * Ho * Wo * C4;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c4 = (int)(idx % C4);
  const long long pix = idx / C4;
  const int ox = (int)(pix % Wo);
  const int oy = (int)((pix / Wo) % Ho);
  const int b = (int)(pix / ((long long)Wo * Ho));
  constexpr int P = K / 2;
  float4 acc = BIAS ? __ldg(bias + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
  const float4* inb = in + (long long)b * H * W * C4;
#pragma unroll
  for (int ky = 0; ky < K; ++ky) {
    const int iy = oy * S - P + ky;
    if (iy < 0 || iy >= H) continue;
#pragma unroll
    for (int kx = 0; kx < K; ++kx) {
      const int ix = ox * S - P + kx;
      if (ix < 0 || ix >= W) continue;
      const float4 v = __ldg(inb + ((long long)iy * W + ix) * C4 + c4);
      const float4 k = __ldg(w + (ky * K + kx) * C4 + c4);
      acc.x = fmaf(v.x, k.x, acc.x);
      acc.y = fmaf(v.y, k.y, acc.y);
      acc.z = fmaf(v.z, k.z, acc.z);
      acc.w = fmaf(v.w, k.w, acc.w);
    }
  }
  if (RELU) {
    acc.x = fmaxf(acc.x, 0.f);
    acc.y = fmaxf(acc.y, 0.f);
    acc.z = fmaxf(acc.z, 0.f);
    acc.w = fmaxf(acc.w, 0.f);
  }
  out[idx] = acc;
}

// ------------------------------------------------------------------------------------------
// Depthwise KxK conv, register-strip version: one thread produces TX consecutive output pixels of a
// row for 4 channels.  Each input row segment (TX*S + K - S float4) and the K weights of that row are
// loaded once and reused by all TX outputs, cutting L1 wavefronts per output ~3x against the
// one-pixel-per-thread kernel above (which is L1-wavefront bound, not HBM bound).
// Requires Wo % TX == 0.
// ------------------------------------------------------------------------------------------
template <int K, int S, int TX, bool RELU, bool BIAS>
__global__ void __launch_bounds__(TX >= 16 ? 128 : 256) dw_conv_strip_kernel(const float4* __restrict__ in, const float4* __restrict__ w,
                                                            const float4* __restrict__ bias, float4* __restrict__ out,
                                                            int B, int H, int W, int C4) {
  const int Ho = H / S, Wo = W / S;
  const int strips = Wo / TX;
  const long long total = (long long)B * Ho * strips * C4;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c4 = (int)(idx % C4);
  long long rest = idx / C4;
  const int sx = (int)(rest % strips);
  rest /= strips;
  const int oy = (int)(rest % Ho);
  const int b = (int)(rest / Ho);
  constexpr int P = K / 2;
  constexpr int NIN = (TX - 1) * S + K;  // input columns feeding TX outputs
  const int ox0 = sx * TX;
  const int ix0 = ox0 * S - P;
  float4 acc[TX];
  const float4 b4 = BIAS ? __ldg(bias + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int t = 0; t < TX; ++t) acc[t] = b4;
  const float4* inb = in + (long long)b * H * W * C4 + c4;
#pragma unroll
  for (int ky = 0; ky < K; ++ky) {
    const int iy = oy * S - P + ky;
    if (iy < 0 || iy >= H) continue;
    const float4* row = inb + (long long)iy * W * C4;
    float4 v[NIN];
#pragma unroll
    for (int i = 0; i < NIN; ++i) {
      const int ix = ix0 + i;
      v[i] = (ix >= 0 && ix < W) ? __ldg(row + (long long)ix * C4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int kx = 0; kx < K; ++kx) {
      const float4 k = __ldg(w + (ky * K + kx) * C4 + c4);
#pragma unroll
      for (int t = 0; t < TX; ++t) {
        const float4 x = v[t * S + kx];
        acc[t].x = fmaf(x.x, k.x, acc[t].x);
        acc[t].y = fmaf(x.y, k.y, acc[t].y);
        acc[t].z = fmaf(x.z, k.z, acc[t].z);
        acc[t].w = fmaf(x.w, k.w, acc[t].w);
      }
    }
  }
  float4* o = out + (((long long)b * Ho + oy) * Wo + ox0) * C4 + c4;
#pragma unroll
  for (int t = 0; t < TX; ++t) {
    float4 r = acc[t];
    if (RELU) {
      r.x = fmaxf(r.x, 0.f);
      r.y = fmaxf(r.y, 0.f);
      r.z = fmaxf(r.z, 0.f);
      r.w = fmaxf(r.w, 0.f);
    }
    o[(long long)t * C4] = r;
  }
}

// ------------------------------------------------------------------------------------------
// Depthwise KxK conv, rolling-window version.  One thread owns (4 channels, TX output columns) and
// walks ROWS output rows top to bottom: all K*K weights live in registers, every input row segment
// is loaded ONCE and scattered into a ring of ceil(K/S) live output-row accumulators, so a 5x5 conv
// issues ~3 loads per output float4 instead of ~16 (strip) / 50 (per-pixel).  That moves the kernel
// from L1-wavefront-bound to FFMA/HBM-bound.  Fully unrolled => all ring indices are compile time.
// Accumulation order per output (bias, then ky, kx ascending) is identical to the other two kernels.
// ------------------------------------------------------------------------------------------
template <int K, int S, int TX, int ROWS, bool RELU, bool BIAS>
__global__ void __launch_bounds__(128) dw_conv_roll_kernel(const float4* __restrict__ in, const float4* __restrict__ w,
                                                           const float4* __restrict__ bias, float4* __restrict__ out,
                                                           int B, int H, int W, int C4) {
  constexpr int P = K / 2;
  constexpr int NIN = (TX - 1) * S + K;
  constexpr int LIVE = (K + S - 1) / S;
  constexpr int NR = (ROWS - 1) * S + K;  // input rows feeding ROWS output rows
  const int Ho = H / S, Wo = W / S;
  const int strips = Wo / TX, segs = (Ho + ROWS - 1) / ROWS;
  const long long total = (long long)B * segs * strips * C4;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c4 = (int)(idx % C4);
  long long rest = idx / C4;
  const int sx = (int)(rest % strips);
  rest /= strips;
  const int seg = (int)(rest % segs);
  const int b = (int)(rest / segs);
  const int oy0 = seg * ROWS, ox0 = sx * TX;
  const int iy0 = oy0 * S - P, ix0 = ox0 * S - P;

  float4 wr[K * K];
#pragma unroll
  for (int i = 0; i < K * K; ++i) wr[i] = __ldg(w + i * C4 + c4);
  const float4 b4 = BIAS ? __ldg(bias + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
  float4 acc[LIVE][TX];
#pragma unroll
  for (int l = 0; l < LIVE; ++l)
#pragma unroll
    for (int t = 0; t < TX; ++t) acc[l][t] = b4;

  const float4* inb = in + (long long)b * H * W * C4 + c4;
  float4* outb = out + (long long)b * Ho * Wo * C4 + c4;
#pragma unroll
  for (int r = 0; r < NR; ++r) {
    const int iy = iy0 + r;
    if (iy >= 0 && iy < H) {
      const float4* row = inb + (long long)iy * W * C4;
      float4 v[NIN];
#pragma unroll
      for (int i = 0; i < NIN; ++i) {
        const int ix = ix0 + i;
        v[i] = (ix >= 0 && ix < W) ? __ldg(row + (long long)ix * C4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int ky = K - 1; ky >= 0; --ky) {  // descending ky = ascending output row; order per output unchanged
        if ((r - ky) >= 0 && (r - ky) % S == 0 && (r - ky) / S < ROWS) {
          constexpr int dummy = 0;
          (void)dummy;
          const int slot = ((r - ky) / S) % LIVE;
#pragma unroll
          for (int kx = 0; kx < K; ++kx) {
            const float4 k = wr[ky * K + kx];
#pragma unroll
            for (int t = 0; t < TX; ++t) {
              const float4 x = v[t * S + kx];
              acc[slot][t].x = fmaf(x.x, k.x, acc[slot][t].x);
              acc[slot][t].y = fmaf(x.y, k.y, acc[slot][t].y);
              acc[slot][t].z = fmaf(x.z, k.z, acc[slot][t].z);
              acc[slot][t].w = fmaf(x.w, k.w, acc[slot][t].w);
            }
          }
        }
      }
    }
    if (r >= K - 1 && (r - (K - 1)) % S == 0) {  // output row o is complete after input row r
      const int o = (r - (K - 1)) / S;
      const int slot = o % LIVE;
      if (oy0 + o < Ho) {
        float4* orow = outb + ((long long)(oy0 + o) * Wo + ox0) * C4;
#pragma unroll
        for (int t = 0; t < TX; ++t) {
          float4 res = acc[slot][t];
          if (RELU) {
            res.x = fmaxf(res.x, 0.f);
            res.y = fmaxf(res.y, 0.f);
            res.z = fmaxf(res.z, 0.f);
            res.w = fmaxf(res.w, 0.f);
          }
          orow[(long long)t * C4] = res;
        }
      }
#pragma unroll
      for (int t = 0; t < TX; ++t) acc[slot][t] = b4;
    }
  }
}

// ------------------------------------------------------------------------------------------
// 1x1 conv / correlation as a GEMM on CUDA cores:  C[M][N] = A[M][K] * Bw[N][K]^T (+bias)(+R)(ReLU)
// A rows = pixels (lda floats apart), Bw rows = output channels (ldb apart), both K-contiguous.
// Tile 128 x BN x 16, 256 threads as 32 (rows, 4 each) x 8 (cols, TN = BN/8 each).
// gridDim.z batches independent problems (per-frame correlation: A/C strided per frame, Bw
// strided per frame or shared when strideB == 0 -- template batch-1 broadcast, blocks.py:123).
// ------------------------------------------------------------------------------------------
template <int TN>
__global__ void __launch_bounds__(256) gemm_nt_ffma_kernel(const float* __restrict__ A, int lda, long long strideA,
                                                           const float* __restrict__ Bw, int ldb, long long strideB,
                                                           const float* __restrict__ bias, const float* __restrict__ R,
                                                           int ldr, float* __restrict__ C, int ldc, long long strideC,
                                                           int M, int N, int K, int relu) {
  constexpr int BM = 128, BK = 16, BN = 8 * TN, TM = 4;
  constexpr int AS = BM + 4;  // padded row length of the k-major A tile
  __shared__ __align__(16) float As[BK][AS];
  __shared__ __align__(16) float Bs[BK][BN + 1];
  const int tid = threadIdx.x;
  const int tx = tid & 7, ty = tid >> 3;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  A += (long long)blockIdx.z * strideA;
  Bw += (long long)blockIdx.z * strideB;
  C += (long long)blockIdx.z * strideC;
  if (R) R += (long long)blockIdx.z * strideC;

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += BK) {
    // A tile: 128 rows x 16 k = 512 float4, two per thread; stored transposed (k-major).
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int id = tid + it * 256;
      const int r = id >> 2, kq = (id & 3) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m0 + r < M && k0 + kq < K) v = __ldg(reinterpret_cast<const float4*>(A + (long long)(m0 + r) * lda + k0 + kq));
      As[kq + 0][r] = v.x;
      As[kq + 1][r] = v.y;
      As[kq + 2][r] = v.z;
      As[kq + 3][r] = v.w;
    }
    // B tile: BN rows (output channels) x 16 k.
    for (int id = tid; id < BN * 4; id += 256) {
      const int n = id >> 2, kq = (id & 3) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (n0 + n < N && k0 + kq < K) v = __ldg(reinterpret_cast<const float4*>(Bw + (long long)(n0 + n) * ldb + k0 + kq));
      Bs[kq + 0][n] = v.x;
      Bs[kq + 1][n] = v.y;
      Bs[kq + 2][n] = v.z;
      Bs[kq + 3][n] = v.w;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * TM]);
      const float a[TM] = {a4.x, a4.y, a4.z, a4.w};
      float bv[TN];
#pragma unroll
      for (int j = 0; j < TN; ++j) bv[j] = Bs[kk][tx * TN + j];
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int row = m0 + ty * TM + i;
    if (row >= M) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int col = n0 + tx * TN + j;
      if (col >= N) continue;
      float v = acc[i][j];
      if (bias) v += __ldg(bias + col);
      if (R) v += __ldg(R + (long long)row * ldr + col);
      if (relu) v = fmaxf(v, 0.f);
      C[(long long)row * ldc + col] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------
// Context crop + constant-colour padding + bilinear resize of the tracking loop, on the device
// (reference model_training/utils/utils.py:215-253 get_extended_crop: cv2.copyMakeBorder + albumentations.Resize =
// cv2.resize(INTER_LINEAR) on uint8).  The frame is uploaded once; this kernel reads the context window straight out
// of it (pixels outside the frame = the padding colour) and reproduces OpenCV's 8-bit fixed-point bilinear kernel
// bit for bit: 11-bit coefficients, horizontal pass in int32, vertical pass
//     ((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2
// (cv::VResizeLinear<uchar> / VResizeLinearVec_32s8u).  The per-axis source offsets and coefficients are computed on
// the host in float32 exactly as cv::resize does (feartracker_b200/image_ops.py:resize_tables) and passed in
// `params`:  [0..3] context x, y, w, h (frame coordinates, may leave the frame); [4..6] padding colour RGB; [7] unused;
// then xofs[S], xa0[S], xa1[S], yofs[S], ya0[S], ya1[S] for an S x S output.  out: [S][S][3] uint8 (HWC).
// ------------------------------------------------------------------------------------------
// One output pixel (all three channels) of the padded, resized context window (cx, cy, cw, ch): x0 / a0 / a1 are the
// column's source offset and coefficients, yo / b0 / b1 the row's.  Shared with track_crops_u8_kernel.
__device__ __forceinline__ void crop_resize_pixel(const uint8_t* __restrict__ frame, int H, int W, int cx, int cy,
                                                  int cw, int ch, const int (&pad)[3], int x0, int a0, int a1, int yo,
                                                  int b0, int b1, uint8_t* __restrict__ out_px) {
  const int x1 = min(x0 + 1, cw - 1);
  const int y0 = min(max(yo, 0), ch - 1), y1 = min(max(yo + 1, 0), ch - 1);
  auto px = [&](int y, int x, int c) -> int {  // padded context window
    const int fy = cy + y, fx = cx + x;
    return (fy >= 0 && fy < H && fx >= 0 && fx < W) ? (int)__ldg(frame + ((long long)fy * W + fx) * 3 + c) : pad[c];
  };
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int s0 = px(y0, x0, c) * a0 + px(y0, x1, c) * a1;
    const int s1 = px(y1, x0, c) * a0 + px(y1, x1, c) * a1;
    const int v = (((b0 * (s0 >> 4)) >> 16) + ((b1 * (s1 >> 4)) >> 16) + 2) >> 2;
    out_px[c] = (uint8_t)min(max(v, 0), 255);
  }
}

__global__ void __launch_bounds__(256) crop_resize_u8_kernel(const uint8_t* __restrict__ frame, int H, int W,
                                                             const int* __restrict__ params, uint8_t* __restrict__ out,
                                                             int S) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= S * S) return;
  const int dy = idx / S, dx = idx - dy * S;
  const int cx = __ldg(params), cy = __ldg(params + 1), cw = __ldg(params + 2), ch = __ldg(params + 3);
  const int* tx = params + 8;
  const int* ty = params + 8 + 3 * S;
  const int pad[3] = {__ldg(params + 4), __ldg(params + 5), __ldg(params + 6)};
  crop_resize_pixel(frame, H, W, cx, cy, cw, ch, pad, __ldg(tx + dx), __ldg(tx + S + dx), __ldg(tx + 2 * S + dx),
                    __ldg(ty + dy), __ldg(ty + S + dy), __ldg(ty + 2 * S + dy), out + (long long)idx * 3);
}

// ------------------------------------------------------------------------------------------
// Pixel-wise correlation straight on the reference's layouts (MobileCorrelation.forward, blocks.py:121-123):
//   out[b, 256 + k, p] = sum_c z[b, c, k] * x[b, c, p],  z (Bz,256,64), x (B,256,256), out (B,320,256).
// Compatibility kernel of the workspace-free C entry point fear_corr_concat_f32; the hot path runs
// tc::corr_ts_kernel on the channels-last concat buffer instead.  grid (4, B), 256 threads: 64 pixels x 4 groups
// of 16 template cells, the template streamed through shared memory in 64-channel slices.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) corr_nchw_ffma_kernel(const float* __restrict__ z, long long z_stride,
                                                             const float* __restrict__ x, float* __restrict__ out) {
  __shared__ float sz[64 * 64];  // [channel within the slice][template cell]
  const int b = blockIdx.y, p = blockIdx.x * 64 + (threadIdx.x & 63), kq = threadIdx.x >> 6;
  const float* zb = z + (long long)b * z_stride;
  const float* xb = x + (long long)b * 256 * 256;
  float acc[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) acc[j] = 0.f;
  for (int c0 = 0; c0 < 256; c0 += 64) {
    __syncthreads();
    for (int i = threadIdx.x; i < 64 * 64; i += 256) sz[i] = __ldg(zb + c0 * 64 + i);
    __syncthreads();
    for (int cc = 0; cc < 64; ++cc) {
      const float xv = __ldg(xb + (c0 + cc) * 256 + p);
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[j] = fmaf(sz[cc * 64 + kq * 16 + j], xv, acc[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 16; ++j) out[((long long)b * 320 + 256 + kq * 16 + j) * 256 + p] = acc[j];
}

// ------------------------------------------------------------------------------------------
// Tiny 1x1 convs (xif1_0.pwl 16->16, xif2_2/2_3.pwl 24->24) are pure streaming: ~1 FLOP per byte, millions of
// pixels.  A tensor-core tile pipeline only adds per-tile latency there, so these run one pixel per thread on CUDA
// cores with the [Cin][Cout] weights passed BY VALUE (kernel parameter = constant bank): every FFMA takes its weight
// as a uniform-register / constant operand.  (A broadcast LDS costs one LSU wavefront per 4 bytes even when all
// lanes read the same address, which made a shared-memory version LSU-bound.)   out = act(x * W^T + b (+ residual)).
// ------------------------------------------------------------------------------------------
template <int CIN, int COUT>
struct PwSmallWeights {
  float w[CIN * COUT];  // [k][o]
  float b[COUT];
};
template <int CIN, int COUT>
__global__ void __launch_bounds__(256) pw_small_const_kernel(const float* __restrict__ x, const float* __restrict__ res,
                                                             float* __restrict__ out, long long M, int relu,
                                                             const __grid_constant__ PwSmallWeights<CIN, COUT> wts) {
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  float xin[CIN];
  const float4* xp = reinterpret_cast<const float4*>(x + m * CIN);
#pragma unroll
  for (int i = 0; i < CIN / 4; ++i) {
    const float4 v = __ldg(xp + i);
    xin[4 * i] = v.x;
    xin[4 * i + 1] = v.y;
    xin[4 * i + 2] = v.z;
    xin[4 * i + 3] = v.w;
  }
  float4 q[COUT / 4];
  const float4* rp = res ? reinterpret_cast<const float4*>(res + m * COUT) : nullptr;
  if (rp) {
#pragma unroll
    for (int o4 = 0; o4 < COUT / 4; ++o4) q[o4] = __ldg(rp + o4);  // issued early: overlaps the FMAs
  }
  float acc[COUT];
#pragma unroll
  for (int o = 0; o < COUT; ++o) acc[o] = wts.b[o];
#pragma unroll
  for (int k = 0; k < CIN; ++k)
#pragma unroll
    for (int o = 0; o < COUT; ++o) acc[o] = fmaf(xin[k], wts.w[k * COUT + o], acc[o]);
  float4* op = reinterpret_cast<float4*>(out + m * COUT);
#pragma unroll
  for (int o4 = 0; o4 < COUT / 4; ++o4) {
    float4 r = make_float4(acc[4 * o4], acc[4 * o4 + 1], acc[4 * o4 + 2], acc[4 * o4 + 3]);
    if (rp) {
      r.x += q[o4].x;
      r.y += q[o4].y;
      r.z += q[o4].z;
      r.w += q[o4].w;
    }
    if (relu) {
      r.x = fmaxf(r.x, 0.f);
      r.y = fmaxf(r.y, 0.f);
      r.z = fmaxf(r.z, 0.f);
      r.w = fmaxf(r.w, 0.f);
    }
    op[o4] = r;
  }
}

// ------------------------------------------------------------------------------------------
// Batched 2-D transpose with leading dimensions: out[b][j][i] = in[b][i][j], i < R, j < Cn.
// Used for NCHW <-> NHWC at the API boundary (the reference API is NCHW, fear_net.py:58-96).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) transpose_kernel(const float* __restrict__ in, int ldin, long long strideIn,
                                                        float* __restrict__ out, int ldout, long long strideOut, int R,
                                                        int Cn) {
  __shared__ float tile[32][33];
  in += (long long)blockIdx.z * strideIn;
  out += (long long)blockIdx.z * strideOut;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
#pragma unroll
  for (int i = ty; i < 32; i += 8) {
    const int r = r0 + i, c = c0 + tx;
    if (r < R && c < Cn) tile[i][tx] = in[(long long)r * ldin + c];
  }
  __syncthreads();
#pragma unroll
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, r = r0 + tx;
    if (r < R && c < Cn) out[(long long)c * ldout + r] = tile[tx][i];
  }
}

// ------------------------------------------------------------------------------------------
// Prediction 1x1 conv (256 -> NOUT, NOUT = 4 | 1) fused with the BoxTower epilogue
// (blocks.py:187-188,192):  bbox = exp(adjust * pred + bias), cls = 0.1 * pred.  adjust / 0.1 /
// biases are folded into w, b on the host, so this is  out = f(w . t + b).  One warp per pixel,
// NHWC in, NCHW out (B, NOUT, 16, 16) -- the layout FEARNet returns.
// ------------------------------------------------------------------------------------------
template <int NOUT, bool EXP>
__global__ void __launch_bounds__(256) pred_pw_kernel(const float* __restrict__ t, const float* __restrict__ w,
                                                      const float* __restrict__ b, float* __restrict__ out, int B) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= B * 256) return;
  const float4* tp = reinterpret_cast<const float4*>(t + (long long)warp * 256);
  const float4 v0 = __ldg(tp + lane), v1 = __ldg(tp + 32 + lane);
  float acc[NOUT];
#pragma unroll
  for (int o = 0; o < NOUT; ++o) {
    const float4* wp = reinterpret_cast<const float4*>(w + o * 256);
    const float4 w0 = __ldg(wp + lane), w1 = __ldg(wp + 32 + lane);
    float s = v0.x * w0.x;
    s = fmaf(v0.y, w0.y, s);
    s = fmaf(v0.z, w0.z, s);
    s = fmaf(v0.w, w0.w, s);
    s = fmaf(v1.x, w1.x, s);
    s = fmaf(v1.y, w1.y, s);
    s = fmaf(v1.z, w1.z, s);
    s = fmaf(v1.w, w1.w, s);
    acc[o] = s;
  }
#pragma unroll
  for (int o = 0; o < NOUT; ++o)
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], d);
  if (lane < NOUT) {
    float v = 0.f;
#pragma unroll
    for (int o = 0; o < NOUT; ++o)
      if (lane == o) v = acc[o];
    v += __ldg(b + lane);
    if (EXP) v = expf(v);
    const int frame = warp >> 8, p = warp & 255;
    out[((long long)frame * NOUT + lane) * 256 + p] = v;
  }
}

// ------------------------------------------------------------------------------------------
// Box decode (FEARTracker._postprocess + FEARBoxCoder.decode, fear_tracker.py:74-86,
// box_coder.py:75-107): score = sigmoid(cls) in fp32, argmax = first maximum in row-major
// order, box = [gx - l, gy - t, (gx + r) - (gx - l), (gy + b) - (gy - t)] evaluated in double
// (the reference's grid is float64, utils/utils.py:183-199, so torch promotes).  One 256-thread
// block per frame.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) decode_kernel(const float* __restrict__ bbox, const float* __restrict__ cls,
                                                     int apply_sigmoid, FearBox* __restrict__ boxes) {
  __shared__ float sv[8];
  __shared__ int si[8];
  const int f = blockIdx.x, t = threadIdx.x;
  float v = cls[(long long)f * 256 + t];
  if (apply_sigmoid) v = 1.0f / (1.0f + expf(-v));
  int i = t;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, d);
    const int oi = __shfl_xor_sync(0xffffffffu, i, d);
    if (ov > v || (ov == v && oi < i)) {
      v = ov;
      i = oi;
    }
  }
  if ((t & 31) == 0) {
    sv[t >> 5] = v;
    si[t >> 5] = i;
  }
  __syncthreads();
  if (t == 0) {
    for (int k = 1; k < 8; ++k)
      if (sv[k] > v || (sv[k] == v && si[k] < i)) {
        v = sv[k];
        i = si[k];
      }
    const int r = i >> 4, c = i & 15;
    const double gx = (double)((c - 8) * 16 + 128), gy = (double)((r - 8) * 16 + 128);
    const float* bb = bbox + (long long)f * 4 * 256 + i;
    const double x1 = gx - (double)bb[0], y1 = gy - (double)bb[256];
    const double x2 = gx + (double)bb[512], y2 = gy + (double)bb[768];
    FearBox o;
    o.x = x1;
    o.y = y1;
    o.w = x2 - x1;
    o.h = y2 - y1;
    o.score = v;
    o.row = r;
    o.col = c;
    o.flat = i;
    boxes[f] = o;
  }
}

}  // namespace fear
