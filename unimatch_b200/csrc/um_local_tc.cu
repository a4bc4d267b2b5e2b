// local_correlation_with_flow (matching.py:86-123) on the tcgen05 tensor cores: the 10 x 10 integer-tap dot products of
// every pixel as one small GEMM per 16 x 8 pixel tile, fp32-faithful (3xFP16: hi*hi + hi*lo + lo*hi, fp32 accumulate).
//
// The CUDA-core kernel (um_local.cu, local_corr_volume_kernel) re-reads every tap of every window from L1 and is bound by
// the latency of its load -> FMA -> shuffle chain.  Within a pixel tile the windows overlap almost completely when the flow
// is smooth, so the tile instead multiplies
//   A = the tile's 128 f0 rows (128 x 128 channels, resident for the tile)
//   B = f1 over the bounding box of the tile's integer-tap windows, in chunks of 32 columns x 8 rows (N = 256)
// into TMEM, and the epilogue (thread = TMEM lane = pixel) picks its own 10 x 10 taps out of the accumulator rows and blends
// them 4 -> 1 exactly as the CUDA-core kernel does.  The chunks are 4-D TMA boxes of the fp16 (hi, lo) feature planes at
// dynamic, possibly negative origins; TMA's out-of-bounds zero fill is the reference's zero padding.
//
// Chunk columns overlap (stride 23 = 32 - 10 + 1), so every window row of a pixel lies in exactly one chunk column; chunk
// rows are disjoint and visited top to bottom, so each window row arrives once, in order, and only two rows of 10 dots stay
// live per pixel.  A tile whose box needs more than MAX_CHUNKS chunks (a rough flow) is computed by the epilogue warps on
// CUDA cores instead (the gather of local_corr_volume_kernel, reading the planes); the launch counts those tiles.
//
// Roles (320 threads, one persistent CTA per SM): warp 0 = flow -> bounding box + TMA producer, warp 1 = MMA issuer into two
// 256-column TMEM accumulators (the epilogue of chunk c overlaps the MMAs of chunk c + 1), warps 2-9 = epilogue, two warps
// per TMEM lane quarter that split the window rows (0-5 and 5-9): the epilogue is latency bound, not issue bound.
#include <limits.h>

#include "um_common.cuh"
#include "um_local_tap.cuh"
#include "um_tc.cuh"

namespace um {

using namespace tc;
using namespace local;

namespace {

constexpr int TW = 16, TH = 8;                 // pixel tile = 128 pixels = the MMA's M
constexpr int R = 4, GRID = 2 * R + 2, NOUT = (2 * R + 1) * (2 * R + 1);
constexpr int CW = 32, CH = 8;                 // chunk of f1 pixels = the MMA's N = 256
constexpr int CSTEP = CW - GRID + 1;           // 23: column stride of the overlapping chunk columns
constexpr int MAX_CHUNKS = 6;                  // larger boxes take the CUDA-core path
constexpr int MAX_SPREAD = 256;                // tap-origin spread (pixels) beyond which the box is not even sized
constexpr int STAGES = 2;
constexpr int NEPI = 8;                        // epilogue warps: two per TMEM lane quarter
constexpr int NTHREADS = 64 + 32 * NEPI;
constexpr int INFO_SLOTS = 4;
constexpr int ROWBUF_LD = 33;                  // warp-private row buffer: 32 lanes x 32 dots (+1: conflict-free stores)
constexpr uint32_t A_BYTES = 4 * 16384;        // [channel half][hi, lo] 128 pixels x 64 channels fp16
constexpr uint32_t STAGE_BYTES = 32768;        // one channel half of one plane of a chunk: 256 pixels x 64 channels fp16
constexpr uint32_t STAGING_BYTES = 128 * NOUT * 4;
constexpr uint32_t ROWBUF_BYTES = NEPI * 32 * ROWBUF_LD * 4;
constexpr uint32_t TAIL_BYTES = 256;
constexpr uint32_t SMEM_BYTES = A_BYTES + STAGES * STAGE_BYTES + STAGING_BYTES + ROWBUF_BYTES + TAIL_BYTES;
static_assert(SMEM_BYTES <= 232448, "shared memory budget");

struct TileInfo { int X0, Y0, nr, nc; };       // box origin (tap-origin minimum - R); nr == 0: CUDA-core tile

struct CorrParams {
  int B, H, W, tiles_x, tiles_y, ntiles, flow_dim;
  const float* flow;
  const __half* f0; const __half* f1; long long plane;     // (hi, lo) planes, `plane` halves apart
  float* out_f32;
  __half* out_split; int cp_split, off_split; long long plane_split;
  int* fallback;
};

__device__ __forceinline__ bool tile_pixel_tap(const CorrParams& p, int b, int y0, int x0, int m, Tap* t) {
  const int y = y0 + (m >> 4), x = x0 + (m & 15);
  if (y >= p.H || x >= p.W) return false;
  *t = corr_center_tap(p.flow, ((long long)b * p.H + y) * p.W + x, p.flow_dim, x, y, p.H, p.W);
  return true;
}

// 16 channels of a (hi, lo) plane row as fp32 hi + lo, in the lane layout of load_row
__device__ __forceinline__ Vec16 load_row_planes(const __half* hi, long long plane, int sub) {
  Vec16 r;
  const uint2* ph = reinterpret_cast<const uint2*>(hi);
  const uint2* pl = reinterpret_cast<const uint2*>(hi + plane);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint2 h = __ldg(ph + sub + 8 * i), l = __ldg(pl + sub + 8 * i);
    const float2 h01 = __half22float2(*reinterpret_cast<const __half2*>(&h.x));
    const float2 h23 = __half22float2(*reinterpret_cast<const __half2*>(&h.y));
    const float2 l01 = __half22float2(*reinterpret_cast<const __half2*>(&l.x));
    const float2 l23 = __half22float2(*reinterpret_cast<const __half2*>(&l.y));
    r.v[i] = make_float4(h01.x + l01.x, h01.y + l01.y, h23.x + l23.x, h23.y + l23.y);
  }
  return r;
}

__global__ void __launch_bounds__(NTHREADS, 1)
local_corr_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, CorrParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sa = smem;
  uint8_t* sb = smem + A_BYTES;
  float* staging = reinterpret_cast<float*>(smem + A_BYTES + STAGES * STAGE_BYTES);     // [128 pixels][81]
  float* rowbufs = reinterpret_cast<float*>(smem + A_BYTES + STAGES * STAGE_BYTES + STAGING_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + A_BYTES + STAGES * STAGE_BYTES + STAGING_BYTES + ROWBUF_BYTES);
  uint64_t* full = bars;                          // [STAGES]
  uint64_t* empty = full + STAGES;                // [STAGES]
  uint64_t* acc_full = empty + STAGES;            // [2]
  uint64_t* acc_empty = acc_full + 2;             // [2]
  uint64_t* a_full = acc_empty + 2;
  uint64_t* a_empty = a_full + 1;
  uint64_t* info_full = a_empty + 1;              // [INFO_SLOTS]
  uint64_t* info_empty = info_full + INFO_SLOTS;  // [INFO_SLOTS]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(info_empty + INFO_SLOTS);
  TileInfo* info = reinterpret_cast<TileInfo*>(bars + 24);
  static_assert((2 * STAGES + 6 + 2 * INFO_SLOTS) * 8 + 4 <= 24 * 8 && 24 * 8 + INFO_SLOTS * 16 <= TAIL_BYTES, "tail layout");

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(acc_full + i, 1); mbar_init(acc_empty + i, 32 * NEPI); }
    mbar_init(a_full, 1); mbar_init(a_empty, 1);
    for (int i = 0; i < INFO_SLOTS; ++i) { mbar_init(info_full + i, 1); mbar_init(info_empty + i, 1 + 32 * NEPI); }
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&map_a); tma_prefetch_desc(&map_b); }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int tiles_img = p.tiles_x * p.tiles_y;

  if (warp == 0) {
    // ---- producer: tap origins of the tile -> bounding box -> tile info; then A once and B chunk by chunk ----
    int it = 0, na = 0, lt = 0;
    for (int t = blockIdx.x; t < p.ntiles; t += gridDim.x, ++lt) {
      const int b = t / tiles_img, rem = t - b * tiles_img;
      const int y0 = (rem / p.tiles_x) * TH, x0 = (rem % p.tiles_x) * TW;
      int mnx = INT_MAX, mxx = INT_MIN, mny = INT_MAX, mxy = INT_MIN;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        Tap tp;
        if (tile_pixel_tap(p, b, y0, x0, lane + 32 * i, &tp)) {
          mnx = min(mnx, tp.x0); mxx = max(mxx, tp.x0); mny = min(mny, tp.y0); mxy = max(mxy, tp.y0);
        }
      }
      mnx = __reduce_min_sync(0xffffffffu, mnx); mxx = __reduce_max_sync(0xffffffffu, mxx);
      mny = __reduce_min_sync(0xffffffffu, mny); mxy = __reduce_max_sync(0xffffffffu, mxy);
      const long long sx = (long long)mxx - mnx, sy = (long long)mxy - mny;
      TileInfo ti{mnx - R, mny - R, 0, 0};
      const bool boxed = sx <= MAX_SPREAD && sy <= MAX_SPREAD && mnx > -(1 << 24) && mnx < (1 << 24) &&
                         mny > -(1 << 24) && mny < (1 << 24);
      if (boxed) {
        const int nc = (int)sx / CSTEP + 1, nr = ((int)sy + GRID + CH - 1) / CH;
        if (nc * nr <= MAX_CHUNKS) { ti.nr = nr; ti.nc = nc; }
      }
      const int slot = lt % INFO_SLOTS;
      mbar_wait(info_empty + slot, ((lt / INFO_SLOTS) & 1) ^ 1);
      if (lane == 0) {
        info[slot] = ti;
        mbar_arrive(info_full + slot);
        if (ti.nr == 0 && p.fallback) atomicAdd(p.fallback, 1);
      }
      __syncwarp();
      if (ti.nr == 0) continue;
      mbar_wait(a_empty, (na & 1) ^ 1);
      ++na;
      if (elect_one()) {
        mbar_arrive_expect_tx(a_full, A_BYTES);
#pragma unroll
        for (int kc = 0; kc < 2; ++kc)
#pragma unroll
          for (int part = 0; part < 2; ++part)
            tma_load_4d(sa + (kc * 2 + part) * 16384, &map_a, a_full, kc * 64, x0, y0, part * p.B + b);
      }
      __syncwarp();
      for (int cr = 0; cr < ti.nr; ++cr)
        for (int cc = 0; cc < ti.nc; ++cc)
          for (int s = 0; s < 4; ++s, ++it) {                // (channel half, plane) = (0, hi) (0, lo) (1, hi) (1, lo)
            const int st = it % STAGES;
            mbar_wait(empty + st, ((it / STAGES) & 1) ^ 1);
            if (elect_one()) {
              mbar_arrive_expect_tx(full + st, STAGE_BYTES);
              tma_load_4d(sb + st * STAGE_BYTES, &map_b, full + st, (s >> 1) * 64, ti.X0 + cc * CSTEP, ti.Y0 + cr * CH,
                          (s & 1) * p.B + b);
            }
            __syncwarp();
          }
    }
  } else if (warp == 1) {
    // ---- MMA issuer: per chunk 2 channel halves x (lo*hi + hi*hi, hi*lo) x 4 K-steps of 128 x 256 x 16 ----
    constexpr uint32_t IDESC = idesc_f16(128, 256, 0, 0);
    int it = 0, ch = 0, na = 0, lt = 0;
    for (int t = blockIdx.x; t < p.ntiles; t += gridDim.x, ++lt) {
      const int slot = lt % INFO_SLOTS;
      mbar_wait(info_full + slot, (lt / INFO_SLOTS) & 1);
      const TileInfo ti = info[slot];
      __syncwarp();
      if (elect_one()) mbar_arrive(info_empty + slot);
      __syncwarp();
      if (ti.nr == 0) continue;
      mbar_wait(a_full, na & 1);
      ++na;
      tc_fence_after();
      const int nch = ti.nr * ti.nc;
      for (int c = 0; c < nch; ++c, ++ch) {
        const int buf = ch & 1;
        mbar_wait(acc_empty + buf, ((ch >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d = tmem + buf * 256;
        for (int s = 0; s < 4; ++s, ++it) {
          const int st = it % STAGES, kc = s >> 1;
          mbar_wait(full + st, (it / STAGES) & 1);
          tc_fence_after();
          const uint32_t b_base = smem_u32(sb + st * STAGE_BYTES);
          const uint32_t a_hi = smem_u32(sa + (kc * 2) * 16384), a_lo = a_hi + 16384;
          if (elect_one()) {
            if ((s & 1) == 0) {                              // B hi: small term first
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) umma_f16(d, desc_kmajor(a_lo + ks * 32), desc_kmajor(b_base + ks * 32), IDESC, s > 0 || ks > 0);
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) umma_f16(d, desc_kmajor(a_hi + ks * 32), desc_kmajor(b_base + ks * 32), IDESC, true);
            } else {                                         // B lo
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) umma_f16(d, desc_kmajor(a_hi + ks * 32), desc_kmajor(b_base + ks * 32), IDESC, true);
            }
            umma_commit(empty + st);
            if (s == 3 && c == nch - 1) umma_commit(a_empty);   // before acc_full: nothing arrives after the last wait
            if (s == 3) umma_commit(acc_full + buf);
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ---- epilogue: thread = pixel m = TMEM lane; half 0 takes window rows 0-5 (output rows 0-4), half 1 rows 5-9 ----
    const int quarter = warp & 3, ew = warp - 2, half = ew >> 2;
    const int iy_lo = half ? GRID / 2 : 0, iy_hi = half ? GRID - 1 : GRID / 2;
    const int m = quarter * 32 + lane;
    const int e = ew * 32 + lane;                          // 0..255 for the cooperative stores
    float* rowbuf = rowbufs + ew * 32 * ROWBUF_LD;
    auto epi_sync = [&]() { asm volatile("bar.sync 1, %0;" ::"n"(32 * NEPI) : "memory"); };
    int ch = 0, lt = 0;
    for (int t = blockIdx.x; t < p.ntiles; t += gridDim.x, ++lt) {
      const int b = t / tiles_img, rem = t - b * tiles_img;
      const int y0 = (rem / p.tiles_x) * TH, x0 = (rem % p.tiles_x) * TW;
      const int slot = lt % INFO_SLOTS;
      mbar_wait(info_full + slot, (lt / INFO_SLOTS) & 1);
      const TileInfo ti = info[slot];
      mbar_arrive(info_empty + slot);
      if (ti.nr > 0) {
        Tap tp{};
        const bool valid = tile_pixel_tap(p, b, y0, x0, m, &tp);
        const int oxr = tp.x0 - R - ti.X0, oyr = tp.y0 - R - ti.Y0;
        const int mycc = valid ? oxr / CSTEP : -1;
        const int off = oxr - mycc * CSTEP;
        float* orow = staging + m * NOUT;
        float prev[GRID], cur[GRID];
        for (int cr = 0; cr < ti.nr; ++cr) {
          for (int cc = 0; cc < ti.nc; ++cc, ++ch) {
            const int buf = ch & 1;
            mbar_wait(acc_full + buf, (ch >> 1) & 1);
            tc_fence_after();
            const uint32_t taddr = tmem + ((uint32_t)(quarter * 32) << 16) + buf * 256;
#pragma unroll 1
            for (int ry = 0; ry < CH; ++ry) {
              const int iy = cr * CH + ry - oyr;               // window row of this accumulator row
              const bool need = cc == mycc && iy >= iy_lo && iy <= iy_hi;
              if (!__any_sync(0xffffffffu, need)) continue;
              float v[32];
              tmem_ld32(taddr + ry * 32, v);
              tmem_wait_ld();
#pragma unroll
              for (int i = 0; i < 32; ++i) rowbuf[lane * ROWBUF_LD + i] = v[i];
              __syncwarp();
              if (need) {                                      // registers cannot be indexed by `off`: go through the row buffer
#pragma unroll
                for (int j = 0; j < GRID; ++j) cur[j] = rowbuf[lane * ROWBUF_LD + off + j];
                if (iy > iy_lo) {
                  float* o = orow + (iy - 1) * (GRID - 1);
#pragma unroll
                  for (int ix = 0; ix < GRID - 1; ++ix) o[ix] = blend(prev[ix], prev[ix + 1], cur[ix], cur[ix + 1], tp);
                }
#pragma unroll
                for (int j = 0; j < GRID; ++j) prev[j] = cur[j];
              }
              __syncwarp();
            }
            tc_fence_before();
            mbar_arrive(acc_empty + buf);
          }
        }
      } else {
        // CUDA-core tile: 8 lanes per pixel, 32 pixels per pass (the gather of local_corr_volume_kernel on the planes)
        const int sub = lane & 7, grp = lane >> 3;
        float* dots = rowbuf + grp * GRID * GRID;
        const __half* img = p.f1 + (long long)b * p.H * p.W * UM_C;
#pragma unroll 1
        for (int pass = 0; pass < 128 / (4 * NEPI); ++pass) {
          const int mm = pass * 4 * NEPI + ew * 4 + grp;
          Tap tq;
          const bool ok = tile_pixel_tap(p, b, y0, x0, mm, &tq);      // uniform over the 8 lanes of the pixel
          if (ok) {
            const long long pix = ((long long)b * p.H + y0 + (mm >> 4)) * p.W + x0 + (mm & 15);
            const Vec16 a = load_row_planes(p.f0 + pix * UM_C, p.plane, sub);
            for (int iy = 0; iy < GRID; ++iy) {
              const int yy = tq.y0 - R + iy;
              for (int ix = 0; ix < GRID; ++ix) {
                const int xx = tq.x0 - R + ix;
                float d = 0.f;
                if (yy >= 0 && yy < p.H && xx >= 0 && xx < p.W)
                  d = dot_partial(a, load_row_planes(img + ((long long)yy * p.W + xx) * UM_C, p.plane, sub));
                d = reduce8(d);
                if (sub == 0) dots[iy * GRID + ix] = d;
              }
            }
          }
          __syncwarp();
          if (ok) {
            for (int k = sub; k < NOUT; k += 8) {
              const int iy = k / (GRID - 1), ix = k - iy * (GRID - 1);
              const float* d = dots + iy * GRID + ix;
              staging[mm * NOUT + k] = blend(d[0], d[1], d[GRID], d[GRID + 1], tq);
            }
          }
          __syncwarp();
        }
      }
      // ---- the tile's 128 x 81 results -> global: each pixel row of the tile is one contiguous run ----
      epi_sync();
      const int nvx = min(TW, p.W - x0);
      for (int py = 0; py < TH && y0 + py < p.H; ++py) {
        const long long pix0 = ((long long)b * p.H + y0 + py) * p.W + x0;
        const int n = nvx * NOUT;
        const float* src = staging + py * TW * NOUT;
        if (p.out_f32) {
          float* dst = p.out_f32 + pix0 * NOUT;
#pragma unroll 4
          for (int i = e; i < n; i += 32 * NEPI) dst[i] = src[i];
        }
        if (p.out_split) {
#pragma unroll 4
          for (int i = e; i < n; i += 32 * NEPI) {
            const int px = i / NOUT, k = i - px * NOUT;
            __half hi, lo;
            split_f16(src[i], &hi, &lo);
            __half* dh = p.out_split + (pix0 + px) * p.cp_split + p.off_split + k;
            dh[0] = hi;
            dh[p.plane_split] = lo;
          }
        }
      }
      epi_sync();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// f1 planes [2][B][H][W][128] viewed as (c, W, H, 2B): box = 64 channels x 32 x 8 pixels (one chunk), 128B swizzle;
// out-of-bounds boxes read as zero
int make_map_chunk(CUtensorMap* map, const void* base, uint64_t W, uint64_t H, uint64_t NB) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) { set_error("cuTensorMapEncodeTiled unavailable"); return UM_ECUDA; }
  cuuint64_t dims[4] = {UM_C, W, H, NB};
  cuuint64_t strides[3] = {UM_C * 2, UM_C * W * 2, UM_C * W * H * 2};
  cuuint32_t box[4] = {64, CW, CH, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(corr chunk) failed (%d)", (int)r); return UM_ECUDA; }
  return UM_OK;
}

}  // namespace
}  // namespace um

extern "C" {

int um_local_corr_volume_planes(const void* f0_planes, const void* f1_planes, const float* flow, float* corr,
                                void* out_split, int32_t cp_split, int32_t off_split, int32_t batch, int32_t h, int32_t w,
                                int32_t radius, int32_t flow_dim, int32_t* fallback_tiles, void* stream) {
  using namespace um;
  UM_REQUIRE(f0_planes && f1_planes && flow && batch > 0 && h > 1 && w > 1, "um_local_corr_volume_planes: bad arguments");
  UM_REQUIRE(radius == R, "um_local_corr_volume_planes: only radius 4 is built (unimatch.py:308-313 uses local_radius=4)");
  UM_REQUIRE(flow_dim == 1 || flow_dim == 2, "um_local_corr_volume_planes: flow_dim must be 1 or 2");
  UM_REQUIRE(corr || out_split, "um_local_corr_volume_planes: no output");
  UM_REQUIRE(((reinterpret_cast<uintptr_t>(f0_planes) | reinterpret_cast<uintptr_t>(f1_planes)) & 15) == 0,
             "um_local_corr_volume_planes: feature planes must be 16-byte aligned");
  if (out_split)
    UM_REQUIRE(off_split >= 0 && cp_split >= off_split + NOUT, "um_local_corr_volume_planes: split output needs cp >= off + 81");
  CorrParams p{};
  p.B = batch; p.H = h; p.W = w; p.flow_dim = flow_dim;
  p.tiles_x = (w + TW - 1) / TW; p.tiles_y = (h + TH - 1) / TH;
  p.ntiles = p.tiles_x * p.tiles_y * batch;
  p.flow = flow;
  p.f0 = reinterpret_cast<const __half*>(f0_planes); p.f1 = reinterpret_cast<const __half*>(f1_planes);
  p.plane = (long long)batch * h * w * UM_C;
  p.out_f32 = corr;
  p.out_split = reinterpret_cast<__half*>(out_split); p.cp_split = cp_split; p.off_split = off_split;
  p.plane_split = (long long)batch * h * w * cp_split;
  p.fallback = fallback_tiles;
  CUtensorMap ma, mb;
  int rc;
  if ((rc = make_map_4d_f16(&ma, f0_planes, UM_C, w, h, 2ull * batch, 1))) return rc;
  if ((rc = make_map_chunk(&mb, f1_planes, w, h, 2ull * batch))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (fallback_tiles && cudaMemsetAsync(fallback_tiles, 0, sizeof(int32_t), st) != cudaSuccess)
    return check_launch("um_local_corr_volume_planes(counter)");
  static PerDeviceBytes configured;
  if ((rc = ensure_smem(configured, local_corr_tc_kernel, SMEM_BYTES, "local_corr_tc"))) return rc;
  const int sms = device_sm_count();
  const int grid = p.ntiles < sms ? p.ntiles : sms;            // persistent: one CTA per SM, tiles in raster order
  local_corr_tc_kernel<<<grid, NTHREADS, SMEM_BYTES, st>>>(ma, mb, p);
  return check_launch("um_local_corr_volume_planes");
}

}  // extern "C"
