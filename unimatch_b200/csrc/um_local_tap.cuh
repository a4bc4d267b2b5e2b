// Tap geometry and the 8-lanes-per-pixel dot product of the local-window kernels (um_local.cu, um_local_tc.cu).
//
// Coordinates replicate the reference's fp32 arithmetic (normalise to [-1,1], ATen un-normalise with align_corners=True,
// floor, 4 weights), so every kernel that includes this header forms the same taps and weights to the last bit.
#pragma once
#include "um_common.cuh"

namespace um {
namespace local {

constexpr float SQRT_C = 11.313708498984761f;

struct Tap { int x0, y0; float wnw, wne, wsw, wse; };

__device__ __forceinline__ float unnormalize(float g, int size) { return ((g + 1.0f) / 2.0f) * (float)(size - 1); }

// geometry.py:49-51 normalisation (bilinear_sample): g = 2*p/(size-1) - 1
__device__ __forceinline__ float norm_sample(float p, int size) { return 2.0f * p / (float)(size - 1) - 1.0f; }
// geometry.py:35-38 normalisation (normalize_coords): g = (p - c)/c, c = (size-1)/2
__device__ __forceinline__ float norm_window(float p, int size) { float c = (float)(size - 1) / 2.0f; return (p - c) / c; }

__device__ __forceinline__ Tap make_tap(float ix, float iy) {
  Tap t;
  float fx = floorf(ix), fy = floorf(iy);
  t.x0 = (int)fx; t.y0 = (int)fy;
  float xe = fx + 1.0f, ye = fy + 1.0f;
  t.wnw = (xe - ix) * (ye - iy);
  t.wne = (ix - fx) * (ye - iy);
  t.wsw = (xe - ix) * (iy - fy);
  t.wse = (ix - fx) * (iy - fy);
  return t;
}

__device__ __forceinline__ void read_flow(const float* flow, long long pix, int flow_dim, float* u, float* v) {
  if (flow_dim == 2) { float2 f = __ldg(reinterpret_cast<const float2*>(flow) + pix); *u = f.x; *v = f.y; }
  else { *u = -__ldg(flow + pix); *v = 0.0f; }     // disparity -> (-d, 0)  (unimatch.py:160-166, :277-287)
}

// local_correlation_with_flow (matching.py:86-123): the integer tap origin of the window centre, (x + dx) + u with dx = 0
__device__ __forceinline__ Tap corr_center_tap(const float* flow, long long pix, int flow_dim, int x, int y, int h, int w) {
  float u, v;
  read_flow(flow, pix, flow_dim, &u, &v);
  const float cx = unnormalize(norm_window((float)x + u, w), w);
  const float cy = unnormalize(norm_window((float)y + v, h), h);
  return make_tap(cx, cy);
}

// 4 -> 1 blend of the integer-tap dots d[0], d[1] (row iy) and d[GRID], d[GRID + 1] (row iy + 1), in the reference order
__device__ __forceinline__ float blend(float nw, float ne, float sw, float se, const Tap& t) {
  float r = nw * t.wnw;
  r = fmaf(ne, t.wne, r);
  r = fmaf(sw, t.wsw, r);
  r = fmaf(se, t.wse, r);
  return r / SQRT_C;
}

struct Vec16 { float4 v[4]; };

// 8 lanes per pixel: lane `sub` owns channels {sub*4 + 32*i .. +3}, i = 0..3
__device__ __forceinline__ Vec16 load_row(const float* row, int sub) {
  Vec16 r;
  const float4* p = reinterpret_cast<const float4*>(row);
#pragma unroll
  for (int i = 0; i < 4; ++i) r.v[i] = __ldg(p + sub + 8 * i);
  return r;
}
__device__ __forceinline__ float dot_partial(const Vec16& a, const Vec16& b) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    s = fmaf(a.v[i].x, b.v[i].x, s); s = fmaf(a.v[i].y, b.v[i].y, s);
    s = fmaf(a.v[i].z, b.v[i].z, s); s = fmaf(a.v[i].w, b.v[i].w, s);
  }
  return s;
}
// sum over the 8 lanes of one pixel group; only that group's lanes are named in the mask, so groups whose
// pixel is out of range may have exited
__device__ __forceinline__ float reduce8(float s) {
  const unsigned gmask = 0xFFu << (threadIdx.x & 24);
  s += __shfl_xor_sync(gmask, s, 4);
  s += __shfl_xor_sync(gmask, s, 2);
  s += __shfl_xor_sync(gmask, s, 1);
  return s;
}

}  // namespace local
}  // namespace um
