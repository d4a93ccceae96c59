// Batched tracking loop with the per-track state on the device (FearTrack, include/fear_b200.h): the host crop math of
// FEARTracker.update (image_ops.context_box / resize_tables before the network, rescale_bbox + clamp_bbox after it)
// reproduced to the last bit, so one step for N tracks is crop -> network -> advance with no host arithmetic.
//
// Exactness: nvcc contracts a*b+c into FMA by default, numpy never does, so every float64 / float32 operation below
// is an explicit round-to-nearest intrinsic.  Python's round() on a float64 rounds half to even (rint, not CUDA's
// round()); numpy's .astype("int32") truncates toward zero (__double2int_rz).
#pragma once

#include <cstdint>

namespace fear {

// image_ops.context_box: [x - w*off, y - h*off, w*(1 + 2*off), h*(1 + 2*off)] in float64, truncated to int32.
__device__ __forceinline__ int4 context_box_dev(int4 box, double off) {
  const double grow = __dadd_rn(1.0, __dmul_rn(2.0, off));
  return make_int4(__double2int_rz(__dsub_rn((double)box.x, __dmul_rn((double)box.z, off))),
                   __double2int_rz(__dsub_rn((double)box.y, __dmul_rn((double)box.w, off))),
                   __double2int_rz(__dmul_rn((double)box.z, grow)), __double2int_rz(__dmul_rn((double)box.w, grow)));
}

// image_ops._axis_table for one destination index d: float64 position (d + 0.5) * (src / dst) - 0.5 rounded once to
// float32, floor, float32 fraction, 11-bit coefficients rint((1 - f) * 2048) and rint(f * 2048).  Along x (clamp) the
// offset is clamped into the row and the fraction zeroed; along y the kernel clamps the row index instead.
__device__ __forceinline__ void resize_coef(int d, int src, int dst, bool clamp, int& s, int& a0, int& a1) {
  const double pos = __dsub_rn(__dmul_rn(__dadd_rn((double)d, 0.5), __ddiv_rn((double)src, (double)dst)), 0.5);
  const float f = __double2float_rn(pos);
  const float fl = floorf(f);
  float fr = __fsub_rn(f, fl);
  s = (int)fl;
  if (clamp && (s < 0 || s >= src - 1)) {
    s = s < 0 ? 0 : src - 1;
    fr = 0.f;
  }
  a0 = (int)rintf(__fmul_rn(__fsub_rn(1.f, fr), 2048.f));
  a1 = (int)rintf(__fmul_rn(fr, 2048.f));
}

// grid (ceil(S*S / 256), N): crop n of `crops` ([N][S][S][3]) around track n's box in frame frames[frame_of_track[n]].
// Every thread derives the context box and its own column / row coefficients (no table buffer); thread 0 of track n
// stores the context box.  Only x..h and the padding colour are read, so that store races with nothing.
__global__ void __launch_bounds__(256) track_crops_u8_kernel(const FearFrame* __restrict__ frames, int F,
                                                             const int32_t* __restrict__ frame_of_track,
                                                             FearTrack* tracks, int S, double context,
                                                             uint8_t* __restrict__ crops) {
  const int n = blockIdx.y;
  const int f = __ldg(frame_of_track + n);
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (f < 0 || f >= F || idx >= S * S) return;
  const FearFrame fr = frames[f];
  const int4 box = *reinterpret_cast<const int4*>(&tracks[n].x);
  const int4 pv = *reinterpret_cast<const int4*>(&tracks[n].pad_r);
  const int4 ctx = context_box_dev(box, context);
  if (idx == 0) *reinterpret_cast<int4*>(&tracks[n].cx) = ctx;
  const int dy = idx / S, dx = idx - dy * S;
  int x0, a0, a1, yo, b0, b1;
  resize_coef(dx, ctx.z, S, true, x0, a0, a1);
  resize_coef(dy, ctx.w, S, false, yo, b0, b1);
  const int pad[3] = {pv.x, pv.y, pv.z};
  crop_resize_pixel(fr.data, fr.h, fr.w, ctx.x, ctx.y, ctx.z, ctx.w, pad, x0, a0, a1, yo, b0, b1,
                    crops + ((long long)n * S * S + idx) * 3);
}

// python round() of a float64 (half to even), kept inside +-2^40 so the integer conversion is defined for any input.
__device__ __forceinline__ long long round_half_even(double v) {
  return (long long)fmin(fmax(rint(v), -1099511627776.0), 1099511627776.0);
}

// One thread per track: image_ops.rescale_bbox (search crop -> frame pixels through the stored context box) followed
// by image_ops.clamp_bbox against that track's frame (trim_box, then sides below 3 grown back inside the frame).
__global__ void __launch_bounds__(128) track_advance_kernel(const FearBox* __restrict__ boxes,
                                                            const FearFrame* __restrict__ frames,
                                                            const int32_t* __restrict__ frame_of_track,
                                                            FearTrack* __restrict__ tracks, int N, int instance_size) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const int f = frame_of_track[n];
  if (f < 0) return;
  const FearBox b = boxes[n];
  const FearFrame fr = frames[f];
  const int4 ctx = *reinterpret_cast<const int4*>(&tracks[n].cx);
  const double sx = __ddiv_rn((double)ctx.z, (double)instance_size);
  const double sy = __ddiv_rn((double)ctx.w, (double)instance_size);
  const long long x = round_half_even(__dadd_rn(__dmul_rn(b.x, sx), (double)ctx.x));
  const long long y = round_half_even(__dadd_rn(__dmul_rn(b.y, sy), (double)ctx.y));
  const long long w = max(3LL, round_half_even(__dmul_rn(b.w, sx)));
  const long long h = max(3LL, round_half_even(__dmul_rn(b.h, sy)));
  const long long W = fr.w, H = fr.h;
  const long long x1 = min(max(0LL, x), W), y1 = min(max(0LL, y), H);
  const long long x2 = min(max(0LL, x1 + w), W), y2 = min(max(0LL, y1 + h), H);
  int ox = (int)x1, oy = (int)y1, ow = (int)(x2 - x1), oh = (int)(y2 - y1);
  if (ow < 3) {
    ow = 3;
    ox -= max(0, ox + ow - (int)W);
  }
  if (oh < 3) {
    oh = 3;
    oy -= max(0, oy + oh - (int)H);
  }
  *reinterpret_cast<int4*>(&tracks[n].x) = make_int4(ox, oy, ow, oh);
}

}  // namespace fear
