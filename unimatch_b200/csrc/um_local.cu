// HBM/L2-bound gather kernels of the matching path (channel-last, C = 128):
//   flow_warp, local 9x9 correlation (+softmax / +flow), 3x3 local propagation, depth plane sweep.
//
// Mapping: 8 lanes per pixel, 4 pixels per warp.  A lane owns channels {sub*4 + 32*i .. +3}, i = 0..3, so
// every bilinear / integer tap is 4 fully coalesced 128-byte requests per pixel and a dot product needs a
// 3-step xor-shuffle.  The 81 (or 100) taps of a window are re-read from L1/L2, never materialised: the
// reference's [B,128,H*W,81] grid_sample output (1.04 GB/pair/call, SURVEY.md §8a a7/a8) does not exist here.
//
// Coordinates replicate the reference's fp32 arithmetic (normalise to [-1,1], ATen un-normalise with
// align_corners=True, floor, 4 weights) so taps and weights agree to the last bit wherever possible.
#include <limits.h>
#include <math_constants.h>

#include "um_common.cuh"
#include "um_local_tap.cuh"

namespace {

using namespace um::local;

constexpr int PIX_PER_CTA = 32;     // 256 threads = 8 warps x 4 pixels

__device__ __forceinline__ void store_row(float* row, int sub, const Vec16& r) {
  float4* p = reinterpret_cast<float4*>(row);
#pragma unroll
  for (int i = 0; i < 4; ++i) p[sub + 8 * i] = r.v[i];
}
__device__ __forceinline__ Vec16 zero16() {
  Vec16 r;
#pragma unroll
  for (int i = 0; i < 4; ++i) r.v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  return r;
}
__device__ __forceinline__ void axpy(Vec16& acc, float w, const Vec16& x) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    acc.v[i].x = fmaf(w, x.v[i].x, acc.v[i].x); acc.v[i].y = fmaf(w, x.v[i].y, acc.v[i].y);
    acc.v[i].z = fmaf(w, x.v[i].z, acc.v[i].z); acc.v[i].w = fmaf(w, x.v[i].w, acc.v[i].w);
  }
}
// bilinear sample of a 128-channel row (zeros padding), ATen order nw, ne, sw, se.  A tap whose weight is exactly zero
// is not fetched: w * x with w == 0 adds +-0 to a finite accumulator, so the result is bit-identical -- and the integer
// windows of local_correlation_softmax (matching.py:58-67) land exactly on pixel centres almost everywhere, which makes
// three of the four fetches of every window position vanish (the kernel was 4x over-fetching: 1.26 ms at 8x120x208).
__device__ __forceinline__ Vec16 sample(const float* img, int h, int w, const Tap& t, int sub) {
  Vec16 acc = zero16();
  const bool xl = (t.x0 >= 0 && t.x0 < w), xr = (t.x0 + 1 >= 0 && t.x0 + 1 < w);
  const bool yt = (t.y0 >= 0 && t.y0 < h), yb = (t.y0 + 1 >= 0 && t.y0 + 1 < h);
  if (yt && xl && t.wnw != 0.0f) axpy(acc, t.wnw, load_row(img + ((long long)t.y0 * w + t.x0) * UM_C, sub));
  if (yt && xr && t.wne != 0.0f) axpy(acc, t.wne, load_row(img + ((long long)t.y0 * w + t.x0 + 1) * UM_C, sub));
  if (yb && xl && t.wsw != 0.0f) axpy(acc, t.wsw, load_row(img + ((long long)(t.y0 + 1) * w + t.x0) * UM_C, sub));
  if (yb && xr && t.wse != 0.0f) axpy(acc, t.wse, load_row(img + ((long long)(t.y0 + 1) * w + t.x0 + 1) * UM_C, sub));
  return acc;
}

// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) flow_warp_kernel(const float* __restrict__ f, const float* __restrict__ flow,
                                                        float* __restrict__ out, int h, int w, int flow_dim,
                                                        long long npix) {
  const int sub = threadIdx.x & 7;
  const long long pix = (long long)blockIdx.x * PIX_PER_CTA + (threadIdx.x >> 3);
  if (pix >= npix) return;
  const long long hw = (long long)h * w;
  const int b = (int)(pix / hw);
  const int rem = (int)(pix - (long long)b * hw);
  const int y = rem / w, x = rem - y * w;
  float u, v;
  read_flow(flow, pix, flow_dim, &u, &v);
  const float px = (float)x + u, py = (float)y + v;
  Tap t = make_tap(unnormalize(norm_sample(px, w), w), unnormalize(norm_sample(py, h), h));
  Vec16 r = sample(f + (long long)b * hw * UM_C, h, w, t, sub);
  store_row(out + pix * UM_C, sub, r);
}

// ---------------------------------------------------------------------------------------------------------
// local_correlation_softmax (matching.py:39-83) / _stereo (:154-200): integer window, online softmax.
__global__ void __launch_bounds__(256) local_corr_softmax_kernel(const float* __restrict__ f0, const float* __restrict__ f1,
                                                                 float* __restrict__ out, int h, int w, int ry, int rx,
                                                                 int stereo, long long npix) {
  const int sub = threadIdx.x & 7;
  const long long pix = (long long)blockIdx.x * PIX_PER_CTA + (threadIdx.x >> 3);
  if (pix >= npix) return;
  const long long hw = (long long)h * w;
  const int b = (int)(pix / hw);
  const int rem = (int)(pix - (long long)b * hw);
  const int y = rem / w, x = rem - y * w;
  const Vec16 a = load_row(f0 + pix * UM_C, sub);
  const float* img = f1 + (long long)b * hw * UM_C;
  float m = -CUDART_INF_F, l = 0.f, ax = 0.f, ay = 0.f;
  for (int dy = -ry; dy <= ry; ++dy) {
    for (int dx = -rx; dx <= rx; ++dx) {
      const float sx = (float)x + (float)dx, sy = (float)y + (float)dy;
      const bool valid = (sx >= 0.f) && (sx < (float)w) && (sy >= 0.f) && (sy < (float)h);
      float logit = -1e9f;
      if (valid) {
        Tap t = make_tap(unnormalize(norm_window(sx, w), w), unnormalize(norm_window(sy, h), h));
        Vec16 s = sample(img, h, w, t, sub);
        logit = reduce8(dot_partial(a, s)) / SQRT_C;
      }
      const float m_new = fmaxf(m, logit);
      const float alpha = expf(m - m_new), p = expf(logit - m_new);
      l = l * alpha + p;
      ax = ax * alpha + p * sx;
      ay = ay * alpha + p * sy;
      m = m_new;
    }
  }
  if (sub == 0) {
    const float fx = ax / l - (float)x, fy = ay / l - (float)y;
    if (stereo) out[pix] = -fx;
    else reinterpret_cast<float2*>(out)[pix] = make_float2(fx, fy);
  }
}

// ---------------------------------------------------------------------------------------------------------
// local_correlation_with_flow (matching.py:86-123).  All (2r+1)^2 taps share the fractional offset of
// (x+u, y+v), so the (2r+2)^2 integer-tap dot products are computed once and blended 4 -> 1.
// (Tried in round 2 and measured slower, so not kept: one warp per 2 x 2 pixel block walking the UNION of the four windows so
// that one 512-byte row fetch serves four dot products -- 3x fewer L1 bytes, 1.4x more dot products: 0.66 ms against 0.52 ms
// for this version at 8 x 120 x 208.  The kernel is bound by the latency of its load -> 16 FMA -> 3 shuffle chain per tap,
// not by L1 bandwidth.)
template <int R>
__global__ void __launch_bounds__(256) local_corr_volume_kernel(const float* __restrict__ f0, const float* __restrict__ f1,
                                                                const float* __restrict__ flow, float* __restrict__ corr,
                                                                int h, int w, int flow_dim, long long npix) {
  constexpr int WIN = 2 * R + 1, GRID = WIN + 1;
  __shared__ float dots[PIX_PER_CTA][GRID * GRID + 1];
  const int sub = threadIdx.x & 7, slot = threadIdx.x >> 3;
  const long long pix = (long long)blockIdx.x * PIX_PER_CTA + slot;
  const bool active = pix < npix;
  const long long hw = (long long)h * w;
  int b = 0, y = 0, x = 0;
  float u = 0.f, v = 0.f;
  if (active) {
    b = (int)(pix / hw);
    const int rem = (int)(pix - (long long)b * hw);
    y = rem / w; x = rem - y * w;
    read_flow(flow, pix, flow_dim, &u, &v);
  }
  // centre tap position, exactly as the reference forms it: (x + dx) + u with dx = 0
  const float cx = unnormalize(norm_window((float)x + u, w), w);
  const float cy = unnormalize(norm_window((float)y + v, h), h);
  const Tap t = make_tap(cx, cy);
  if (active) {
    const Vec16 a = load_row(f0 + pix * UM_C, sub);
    const float* img = f1 + (long long)b * hw * UM_C;
    for (int iy = 0; iy < GRID; ++iy) {
      const int yy = t.y0 - R + iy;
      for (int ix = 0; ix < GRID; ++ix) {
        const int xx = t.x0 - R + ix;
        float d = 0.f;
        if (yy >= 0 && yy < h && xx >= 0 && xx < w)     // warp-uniform per 8-lane group
          d = dot_partial(a, load_row(img + ((long long)yy * w + xx) * UM_C, sub));
        d = reduce8(d);
        if (sub == 0) dots[slot][iy * GRID + ix] = d;
      }
    }
  }
  __syncwarp();
  if (active) {
    float* dst = corr + pix * (WIN * WIN);
    for (int k = sub; k < WIN * WIN; k += 8) {
      const int iy = k / WIN, ix = k - iy * WIN;
      const float* d = &dots[slot][iy * GRID + ix];
      float r = d[0] * t.wnw;
      r = fmaf(d[1], t.wne, r);
      r = fmaf(d[GRID], t.wsw, r);
      r = fmaf(d[GRID + 1], t.wse, r);
      dst[k] = r / SQRT_C;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// SelfAttnPropagation.forward_local_window_attn (attention.py:217-253), zero-padded unfold semantics.
__global__ void __launch_bounds__(256) propagate_local_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                              const float* __restrict__ flow, float* __restrict__ out,
                                                              int h, int w, int r, int flow_dim, long long ldq,
                                                              long long ldk, long long npix) {
  const int sub = threadIdx.x & 7;
  const long long pix = (long long)blockIdx.x * PIX_PER_CTA + (threadIdx.x >> 3);
  if (pix >= npix) return;
  const long long hw = (long long)h * w;
  const int b = (int)(pix / hw);
  const int rem = (int)(pix - (long long)b * hw);
  const int y = rem / w, x = rem - y * w;
  const Vec16 a = load_row(q + pix * ldq, sub);
  float m = -CUDART_INF_F, l = 0.f, a0 = 0.f, a1 = 0.f;
  for (int dy = -r; dy <= r; ++dy) {
    for (int dx = -r; dx <= r; ++dx) {
      const int yy = y + dy, xx = x + dx;
      float logit = 0.f, v0 = 0.f, v1 = 0.f;
      if (yy >= 0 && yy < h && xx >= 0 && xx < w) {
        const long long np = (long long)b * hw + (long long)yy * w + xx;
        logit = reduce8(dot_partial(a, load_row(k + np * ldk, sub))) / SQRT_C;
        v0 = __ldg(flow + np * flow_dim);
        if (flow_dim > 1) v1 = __ldg(flow + np * flow_dim + 1);
      }
      const float m_new = fmaxf(m, logit);
      const float alpha = expf(m - m_new), p = expf(logit - m_new);
      l = l * alpha + p;
      a0 = a0 * alpha + p * v0;
      a1 = a1 * alpha + p * v1;
      m = m_new;
    }
  }
  if (sub == 0) {
    out[pix * flow_dim] = a0 / l;
    if (flow_dim > 1) out[pix * flow_dim + 1] = a1 / l;
  }
}

// ---------------------------------------------------------------------------------------------------------
// correlation_softmax_depth (matching.py:203-236) + warp_with_pose_depth_candidates (:239-282)
__global__ void __launch_bounds__(256) depth_corr_kernel(const float* __restrict__ f0, const float* __restrict__ f1,
                                                         const float* __restrict__ Kmat, const float* __restrict__ Kinv,
                                                         const float* __restrict__ pose, const float* __restrict__ cand,
                                                         float* __restrict__ out, int h, int w, int D, int from_argmax,
                                                         long long npix) {
  const int sub = threadIdx.x & 7;
  const long long pix = (long long)blockIdx.x * PIX_PER_CTA + (threadIdx.x >> 3);
  if (pix >= npix) return;
  const long long hw = (long long)h * w;
  const int b = (int)(pix / hw);
  const int rem = (int)(pix - (long long)b * hw);
  const int y = rem / w, x = rem - y * w;
  const float* Ki = Kinv + b * 9;
  const float* Kb = Kmat + b * 9;
  const float* P = pose + b * 16;
  const float fx = (float)x, fy = (float)y;
  // X = K^-1 [x, y, 1];  Xr = R X                                   (matching.py:259-262)
  float X[3], Xr[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) X[r] = fmaf(Ki[r * 3 + 2], 1.0f, fmaf(Ki[r * 3 + 1], fy, Ki[r * 3] * fx));
#pragma unroll
  for (int r = 0; r < 3; ++r) Xr[r] = fmaf(P[r * 4 + 2], X[2], fmaf(P[r * 4 + 1], X[1], P[r * 4] * X[0]));
  const Vec16 a = load_row(f0 + pix * UM_C, sub);
  const float* img = f1 + (long long)b * hw * UM_C;
  float m = -CUDART_INF_F, l = 0.f, acc = 0.f, best = 0.f;
  for (int d = 0; d < D; ++d) {
    const float c = __ldg(cand + d);
    const float depth = 1.0f / c;
    float Pt[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) Pt[r] = Xr[r] * depth + P[r * 4 + 3];           // :262-264
    float pr[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) pr[r] = fmaf(Kb[r * 3 + 2], Pt[2], fmaf(Kb[r * 3 + 1], Pt[1], Kb[r * 3] * Pt[0]));   // :266
    const float z = fmaxf(pr[2], 1e-3f);
    const float uu = pr[0] / z, vv = pr[1] / z;                                    // :267
    Tap t = make_tap(unnormalize(norm_sample(uu, w), w), unnormalize(norm_sample(vv, h), h));
    const float logit = reduce8(dot_partial(a, sample(img, h, w, t, sub))) / SQRT_C;
    if (logit > m) best = c;                       // first maximum wins, like torch.argmax
    const float m_new = fmaxf(m, logit);
    const float alpha = expf(m - m_new), p = expf(logit - m_new);
    l = l * alpha + p;
    acc = acc * alpha + p * c;
    m = m_new;
  }
  if (sub == 0) out[pix] = from_argmax ? best : acc / l;
}

}  // namespace
namespace um {
int local_corr_softmax_stencil(const float* f0, const float* f1, float* flow, int batch, int h, int w, cudaStream_t st);
}
namespace {

inline int grid_for(long long npix) { return (int)((npix + PIX_PER_CTA - 1) / PIX_PER_CTA); }

// ---------------------------------------------------------------------------------------------------------
// forward_backward_consistency_check (geometry.py:75-96) fused into one pass over the two PLANAR flow fields
// [B,2,H,W] the module returns: occ = |flow + warp(other flow, flow)| > alpha (|fwd| + |bwd|) + beta, both directions.
__device__ __forceinline__ float2 sample_flow(const float* f, long long plane, int h, int w, float px, float py) {
  // bilinear_sample(geometry.py:41-62): normalise, ATen un-normalise (align_corners=True), zeros outside
  const Tap t = make_tap(unnormalize(norm_sample(px, w), w), unnormalize(norm_sample(py, h), h));
  const bool xl = (t.x0 >= 0 && t.x0 < w), xr = (t.x0 + 1 >= 0 && t.x0 + 1 < w);
  const bool yt = (t.y0 >= 0 && t.y0 < h), yb = (t.y0 + 1 >= 0 && t.y0 + 1 < h);
  float2 r = make_float2(0.f, 0.f);
  auto tap = [&](bool ok, int yy, int xx, float wgt) {
    if (!ok) return;
    const long long o = (long long)yy * w + xx;
    r.x = fmaf(wgt, __ldg(f + o), r.x);
    r.y = fmaf(wgt, __ldg(f + plane + o), r.y);
  };
  tap(yt && xl, t.y0, t.x0, t.wnw);
  tap(yt && xr, t.y0, t.x0 + 1, t.wne);
  tap(yb && xl, t.y0 + 1, t.x0, t.wsw);
  tap(yb && xr, t.y0 + 1, t.x0 + 1, t.wse);
  return r;
}

__global__ void __launch_bounds__(256) fb_consistency_kernel(const float* __restrict__ fwd, const float* __restrict__ bwd,
                                                             float alpha, float beta, float* __restrict__ fwd_occ,
                                                             float* __restrict__ bwd_occ, int h, int w, long long npix) {
  const long long pix = (long long)blockIdx.x * 256 + threadIdx.x;
  if (pix >= npix) return;
  const long long plane = (long long)h * w;
  const int b = (int)(pix / plane);
  const int rem = (int)(pix - (long long)b * plane);
  const int y = rem / w, x = rem - y * w;
  const float* fb = fwd + (long long)b * 2 * plane;
  const float* bb = bwd + (long long)b * 2 * plane;
  const float fu = __ldg(fb + rem), fv = __ldg(fb + plane + rem);
  const float bu = __ldg(bb + rem), bv = __ldg(bb + plane + rem);
  const float mag = sqrtf(fu * fu + fv * fv) + sqrtf(bu * bu + bv * bv);
  const float2 wb = sample_flow(bb, plane, h, w, (float)x + fu, (float)y + fv);   // flow_warp(bwd, fwd)
  const float2 wf = sample_flow(fb, plane, h, w, (float)x + bu, (float)y + bv);   // flow_warp(fwd, bwd)
  const float dfx = fu + wb.x, dfy = fv + wb.y, dbx = bu + wf.x, dby = bv + wf.y;
  const float thr = alpha * mag + beta;
  fwd_occ[pix] = sqrtf(dfx * dfx + dfy * dfy) > thr ? 1.0f : 0.0f;
  bwd_occ[pix] = sqrtf(dbx * dbx + dby * dby) > thr ? 1.0f : 0.0f;
}

}  // namespace

extern "C" {

int um_flow_warp(const float* f, const float* flow, float* out, int32_t batch, int32_t h, int32_t w,
                 int32_t flow_dim, void* stream) {
  UM_REQUIRE(f && flow && out && batch > 0 && h > 1 && w > 1, "um_flow_warp: bad arguments");
  UM_REQUIRE(flow_dim == 1 || flow_dim == 2, "um_flow_warp: flow_dim must be 1 or 2");
  const long long npix = (long long)batch * h * w;
  flow_warp_kernel<<<grid_for(npix), 256, 0, (cudaStream_t)stream>>>(f, flow, out, h, w, flow_dim, npix);
  return um::check_launch("um_flow_warp");
}

int um_fb_consistency(const float* fwd_flow, const float* bwd_flow, float alpha, float beta, float* fwd_occ,
                      float* bwd_occ, int32_t batch, int32_t h, int32_t w, void* stream) {
  UM_REQUIRE(fwd_flow && bwd_flow && fwd_occ && bwd_occ && batch > 0 && h > 1 && w > 1, "um_fb_consistency: bad arguments");
  const long long npix = (long long)batch * h * w;
  fb_consistency_kernel<<<(unsigned)((npix + 255) / 256), 256, 0, (cudaStream_t)stream>>>(fwd_flow, bwd_flow, alpha, beta,
                                                                                      fwd_occ, bwd_occ, h, w, npix);
  return um::check_launch("um_fb_consistency");
}

int um_local_corr_softmax(const float* f0, const float* f1, float* flow, int32_t batch, int32_t h, int32_t w,
                          int32_t ry, int32_t rx, int32_t stereo, void* stream) {
  UM_REQUIRE(f0 && f1 && flow && batch > 0 && h > 1 && w > 1 && ry >= 0 && rx >= 0,
             "um_local_corr_softmax: bad arguments");
  if (!stereo && ry == 4 && rx == 4)          // the 9x9 flow window (unimatch.py: corr_radius 4): register-tiled stencil
    return um::local_corr_softmax_stencil(f0, f1, flow, batch, h, w, (cudaStream_t)stream);
  const long long npix = (long long)batch * h * w;
  local_corr_softmax_kernel<<<grid_for(npix), 256, 0, (cudaStream_t)stream>>>(f0, f1, flow, h, w, ry, rx, stereo, npix);
  return um::check_launch("um_local_corr_softmax");
}

int um_local_corr_volume(const float* f0, const float* f1, const float* flow, float* corr, int32_t batch, int32_t h,
                         int32_t w, int32_t radius, int32_t flow_dim, void* stream) {
  UM_REQUIRE(f0 && f1 && flow && corr && batch > 0 && h > 1 && w > 1, "um_local_corr_volume: bad arguments");
  UM_REQUIRE(radius == 4, "um_local_corr_volume: only radius 4 is built (unimatch.py:308-313 uses local_radius=4)");
  UM_REQUIRE(flow_dim == 1 || flow_dim == 2, "um_local_corr_volume: flow_dim must be 1 or 2");
  const long long npix = (long long)batch * h * w;
  local_corr_volume_kernel<4><<<grid_for(npix), 256, 0, (cudaStream_t)stream>>>(f0, f1, flow, corr, h, w, flow_dim, npix);
  return um::check_launch("um_local_corr_volume");
}

int um_propagate_local(const float* q, const float* k, const float* flow, float* out, int32_t batch, int32_t h,
                       int32_t w, int32_t radius, int32_t flow_dim, int64_t ldq, int64_t ldk, void* stream) {
  UM_REQUIRE(q && k && flow && out && batch > 0 && h > 0 && w > 0 && radius > 0, "um_propagate_local: bad arguments");
  UM_REQUIRE(flow_dim == 1 || flow_dim == 2, "um_propagate_local: flow_dim must be 1 or 2");
  UM_REQUIRE(ldq % 4 == 0 && ldk % 4 == 0 && ldq >= UM_C && ldk >= UM_C, "um_propagate_local: bad row strides");
  const long long npix = (long long)batch * h * w;
  propagate_local_kernel<<<grid_for(npix), 256, 0, (cudaStream_t)stream>>>(q, k, flow, out, h, w, radius, flow_dim,
                                                                          ldq, ldk, npix);
  return um::check_launch("um_propagate_local");
}

int um_depth_corr_softmax(const float* f0, const float* f1, const float* Kmat, const float* Kinv, const float* pose,
                          const float* cand, float* out, int32_t batch, int32_t h, int32_t w, int32_t num_cand,
                          int32_t from_argmax, void* stream) {
  UM_REQUIRE(f0 && f1 && Kmat && Kinv && pose && cand && out && batch > 0 && h > 1 && w > 1 && num_cand > 0,
             "um_depth_corr_softmax: bad arguments");
  const long long npix = (long long)batch * h * w;
  depth_corr_kernel<<<grid_for(npix), 256, 0, (cudaStream_t)stream>>>(f0, f1, Kmat, Kinv, pose, cand, out, h, w,
                                                                     num_cand, from_argmax, npix);
  return um::check_launch("um_depth_corr_softmax");
}

}  // extern "C"
