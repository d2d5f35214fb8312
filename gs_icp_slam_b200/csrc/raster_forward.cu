// raster_forward.cu — forward pass of the B200 Gaussian-splat rasterizer.
//
// Replaces CudaRasterizer::Rasterizer::forward (DGR/cuda_rasterizer/rasterizer_impl.cu:201-347):
//   preprocess -> scan -> duplicateWithKeys -> 64-bit radix sort of all R instances -> identifyTileRanges -> render
// with a pipeline re-designed around launch count and HBM traffic (DESIGN.md §4):
//   preprocess   writes one 48-B splat record per visible Gaussian and COUNTS the tiles it touches (atomics on T counters)
//   tile_scan    one CTA: exclusive scan of the T counts -> per-tile ranges, LPT launch order, R published to the host
//   emit_binned  every instance is dropped into its tile's range (atomic cursor) as a 64-bit key (depth bits << 32 | id)
//   tile_sort    one CTA per tile sorts its own range in shared memory (bitonic) and writes the ids to point_list
//   render
// The reference's single global sort on (tile << 32 | depth bits) with a stable radix sort orders the instances of a
// tile by depth and equal depths by Gaussian index; sorting each tile's bucket on (depth bits, index) yields exactly the
// same list, so point_list is bit-identical (tests/test_raster_gpu.py) — without moving the R x 12-byte pairs through
// 6 radix passes, and with 5 launches instead of 17.  Tiles holding more than kTileSortCap instances fall back to a
// segmented radix sort (cub::DeviceSegmentedRadixSort) of the same 64-bit keys.
#include <cub/cub.cuh>
#include <mutex>
#include "host_common.h"
#include "raster_common.cuh"

namespace gsicp {

// ------------------------------------------------------------------------------------------
// preprocess: one thread per Gaussian (DGR/cuda_rasterizer/forward.cu:171-274)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ F3 sh_to_rgb(int idx, int deg, int max_coeffs, const float* __restrict__ means,
                                        const float* __restrict__ campos, const float* __restrict__ shs,
                                        uint8_t& clamp_mask) {
  const F3 pos = {means[3 * idx], means[3 * idx + 1], means[3 * idx + 2]};
  const F3 cam = {campos[0], campos[1], campos[2]};
  F3 dir = pos - cam;
  const float len = sqrtf(dot3(dir, dir));
  dir = {dir.x / len, dir.y / len, dir.z / len};
  const F3* sh = reinterpret_cast<const F3*>(shs) + (size_t)idx * max_coeffs;
  F3 res = kShC0 * sh[0];
  if (deg > 0) {
    const float x = dir.x, y = dir.y, z = dir.z;
    res = res - kShC1 * y * sh[1] + kShC1 * z * sh[2] - kShC1 * x * sh[3];
    if (deg > 1) {
      const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
      res = res + kShC2[0] * xy * sh[4] + kShC2[1] * yz * sh[5] + kShC2[2] * (2.0f * zz - xx - yy) * sh[6] +
            kShC2[3] * xz * sh[7] + kShC2[4] * (xx - yy) * sh[8];
      if (deg > 2) {
        res = res + kShC3[0] * y * (3.0f * xx - yy) * sh[9] + kShC3[1] * xy * z * sh[10] +
              kShC3[2] * y * (4.0f * zz - xx - yy) * sh[11] +
              kShC3[3] * z * (2.0f * zz - 3.0f * xx - 3.0f * yy) * sh[12] +
              kShC3[4] * x * (4.0f * zz - xx - yy) * sh[13] + kShC3[5] * z * (xx - yy) * sh[14] +
              kShC3[6] * x * (xx - 3.0f * yy) * sh[15];
      }
    }
  }
  res = {res.x + 0.5f, res.y + 0.5f, res.z + 0.5f};
  clamp_mask = (uint8_t)((res.x < 0.f ? 1 : 0) | (res.y < 0.f ? 2 : 0) | (res.z < 0.f ? 4 : 0));
  return {fmaxf(res.x, 0.f), fmaxf(res.y, 0.f), fmaxf(res.z, 0.f)};
}

struct PreArgs {
  int P, D, M, W, H, tiles_x, tiles_y;
  float tan_fovx, tan_fovy, focal_x, focal_y, scale_modifier;
  const float *means, *scales, *rots, *opac, *shs, *cov_pre, *col_pre, *view, *proj, *campos;
  int prefiltered, shard_count, shard_index;
};

// Per-Gaussian part of preprocess.  Returns true (and the tile rectangle) when the Gaussian is visible.
__device__ __forceinline__ bool preprocess_one(const PreArgs& a, int idx, int32_t* __restrict__ radii,
                                               uint8_t* __restrict__ is_used, Splat* __restrict__ splats,
                                               float* __restrict__ moments, uint8_t* __restrict__ clamped, int& x0,
                                               int& y0, int& x1, int& y1) {
  radii[idx] = 0;
  is_used[idx] = 0;

  const float3 p = make_float3(a.means[3 * idx], a.means[3 * idx + 1], a.means[3 * idx + 2]);
  const float3 pv = xform_point_4x3(p, a.view);
  if (pv.z <= 0.2f) {  // near cull only; no x/y frustum test (auxiliary.h:159)
    if (a.prefiltered) {
      printf("Point is filtered although prefiltered is set. This shouldn't happen!");
      __trap();
    }
    return false;
  }
  const float4 ph = xform_point_4x4(p, a.proj);
  const float pw = 1.0f / (ph.w + 0.0000001f);
  const float3 pp = make_float3(ph.x * pw, ph.y * pw, ph.z * pw);

  float cov3[6];
  if (a.cov_pre) {
#pragma unroll
    for (int i = 0; i < 6; i++) cov3[i] = a.cov_pre[6 * (size_t)idx + i];
  } else {
    const float3 s = make_float3(a.scales[3 * idx], a.scales[3 * idx + 1], a.scales[3 * idx + 2]);
    const float4 q = reinterpret_cast<const float4*>(a.rots)[idx];
    cov3d_from_scale_rot(s, a.scale_modifier, q, cov3);
  }

  const Ewa e = ewa_project(p, a.focal_x, a.focal_y, a.tan_fovx, a.tan_fovy, cov3, a.view);
  const float cxx = e.cov.m[0][0] + 0.3f;  // low-pass: at least one pixel wide
  const float cxy = e.cov.m[0][1];
  const float czx = e.cov.m[0][2];
  const float cyy = e.cov.m[1][1] + 0.3f;
  const float cyz = e.cov.m[1][2];

  const float det = (cxx * cyy - cxy * cxy);
  if (det == 0.0f) return false;
  const float det_inv = 1.f / det;
  const float conx = cyy * det_inv, cony = -cxy * det_inv, conz = cxx * det_inv;

  const float mid = 0.5f * (cxx + cyy);
  const float lambda1 = mid + sqrtf(fmaxf(0.1f, mid * mid - det));
  const float lambda2 = mid - sqrtf(fmaxf(0.1f, mid * mid - det));
  const float my_radius = ceilf(3.f * sqrtf(fmaxf(lambda1, lambda2)));
  const float px = ndc_to_pix(pp.x, a.W), py = ndc_to_pix(pp.y, a.H);
  tile_rect(px, py, (int)my_radius, a.tiles_x, a.tiles_y, x0, y0, x1, y1);
  if ((x1 - x0) * (y1 - y0) == 0) return false;

  F3 rgb;
  uint8_t cm = 0;
  if (a.col_pre) {
    rgb = {a.col_pre[3 * idx], a.col_pre[3 * idx + 1], a.col_pre[3 * idx + 2]};
  } else {
    rgb = sh_to_rgb(idx, a.D, a.M, a.means, a.campos, a.shs, cm);
  }
  clamped[idx] = cm;

  Splat s;
  s.a = make_float4(px, py, conx, cony);
  s.b = make_float4(conz, a.opac[idx], czx, cyz);
  s.c = make_float4(rgb.x, rgb.y, rgb.z, pv.z);
  splats[idx] = s;
  // the render-backward accumulators of this Gaussian start at zero (GeomState::moments)
  float4* mz = reinterpret_cast<float4*>(moments) + 3 * (size_t)idx;
  mz[0] = mz[1] = mz[2] = make_float4(0.f, 0.f, 0.f, 0.f);
  radii[idx] = (int)my_radius;
  is_used[idx] = 1;
  return true;
}

// Visits, warp-cooperatively, every (visible Gaussian, owned tile) pair of the warp's 32 Gaussians: the rectangle of
// one visible Gaussian at a time is broadcast and its tiles are spread over the lanes, so the per-tile atomics of a
// Gaussian are issued in ONE parallel round instead of a serial per-thread loop of dependent atomics.
// f(payload of that Gaussian, tile) is called by the lane that owns the pair; returns the number of owned tiles of the
// caller's own Gaussian.
template <typename F>
__device__ __forceinline__ uint32_t for_each_owned_tile(bool vis, int x0, int y0, int x1, int y1, int tiles_x,
                                                        int shard_count, int shard_index, unsigned long long payload, F f) {
  const int lane = threadIdx.x & 31;
  uint32_t mine = 0;
  unsigned m = __ballot_sync(0xffffffffu, vis);
  while (m) {
    const int src = __ffs(m) - 1;
    m &= m - 1;
    const int rx0 = __shfl_sync(0xffffffffu, x0, src), ry0 = __shfl_sync(0xffffffffu, y0, src);
    const int rx1 = __shfl_sync(0xffffffffu, x1, src), ry1 = __shfl_sync(0xffffffffu, y1, src);
    const unsigned long long pl = __shfl_sync(0xffffffffu, payload, src);
    const int w = rx1 - rx0, n = w * (ry1 - ry0);
    uint32_t owned = 0;
    for (int k = lane; k < n; k += 32) {
      const int t = (ry0 + k / w) * tiles_x + rx0 + k % w;
      if (shard_count > 1 && (t % shard_count) != shard_index) continue;
      f(pl, t);
      owned++;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) owned += __shfl_xor_sync(0xffffffffu, owned, o);
    if (lane == src) mine = owned;
  }
  return mine;
}

__global__ void __launch_bounds__(256)
preprocess_kernel(PreArgs a, int32_t* __restrict__ radii, uint8_t* __restrict__ is_used, Splat* __restrict__ splats,
                  float* __restrict__ moments, uint8_t* __restrict__ clamped, uint32_t* __restrict__ tiles_touched,
                  uint32_t* __restrict__ tile_count) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // blockDim is a multiple of 32: whole warps stay together
  int x0 = 0, y0 = 0, x1 = 0, y1 = 0;
  const bool vis = (idx < a.P) && preprocess_one(a, idx, radii, is_used, splats, moments, clamped, x0, y0, x1, y1);
  // count this Gaussian in every tile it touches that this rank owns (tile % shard_count == shard_index)
  const uint32_t n = for_each_owned_tile(vis, x0, y0, x1, y1, a.tiles_x, a.shard_count, a.shard_index, 0ull,
                                         [&](unsigned long long, int t) { atomicAdd(&tile_count[t], 1u); });
  if (idx < a.P) tiles_touched[idx] = n;
}

// Shared-memory tile sort, two size classes (tiles are already ordered by decreasing count in `order`):
//   small: < 1024 instances — 256 threads, 8 KB of keys (most tiles; many CTAs per SM)
//   big:   1024 .. kTileSortCap instances — 1024 threads, up to 128 KB of keys
constexpr int kBigTileBin = 32;                          // sqrt-count bucket where the big class starts
constexpr int kSmallTileCap = kBigTileBin * kBigTileBin;  // 1024
constexpr int kTileSortCap = 16384;                      // instances one CTA sorts in shared memory (128 KB of 64-bit keys)

// One CTA: exclusive scan of the per-tile counts -> ranges and emit cursors, launch order of the render CTAs (tiles by
// decreasing instance count, bucketed by sqrt(count): the hardware dispatches CTAs in index order, so the longest
// tiles start first and the short ones fill the tail), and (R, largest tile) published to the host through mapped
// pinned memory + a sequence word (no memcpy / stream-synchronize calls on the host).
__global__ void __launch_bounds__(1024)
tile_scan_kernel(int tiles, const uint32_t* __restrict__ tile_count, uint2* __restrict__ ranges, uint32_t* __restrict__ cursor,
                 uint32_t* __restrict__ seg_begin, uint32_t* __restrict__ seg_end, uint32_t* __restrict__ order,
                 volatile unsigned long long* host_map, unsigned long long seq) {
  __shared__ uint32_t s_warp[32], s_hist[64], s_start[64], s_max[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < 64) s_hist[tid] = 0;
  const int per = (tiles + 1023) / 1024;
  const int t0 = tid * per, t1 = min(t0 + per, tiles);
  uint32_t local = 0, lmax = 0;
  for (int t = t0; t < t1; t++) {
    const uint32_t c = tile_count[t];
    local += c;
    lmax = max(lmax, c);
  }
  uint32_t incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
    lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
  }
  if (lane == 31) s_warp[warp] = incl;
  if (lane == 0) s_max[warp] = lmax;
  __syncthreads();
  if (warp == 0) {
    uint32_t v = s_warp[lane], m = s_max[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t u = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += u;
      m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    }
    s_warp[lane] = v;
    s_max[lane] = m;
  }
  __syncthreads();
  uint32_t run = (incl - local) + (warp > 0 ? s_warp[warp - 1] : 0u);
  for (int t = t0; t < t1; t++) {
    const uint32_t c = tile_count[t];
    ranges[t] = c ? make_uint2(run, run + c) : make_uint2(0u, 0u);  // empty tiles read (0,0) like the reference's zero-filled ranges
    cursor[t] = run;
    seg_begin[t] = run;
    seg_end[t] = run + c;
    atomicAdd(&s_hist[min(63, (int)sqrtf((float)c))], 1u);
    run += c;
  }
  __syncthreads();
  if (tid == 0) {
    uint32_t acc = 0;
    for (int b = 63; b >= 0; b--) {
      s_start[b] = acc;
      acc += s_hist[b];
    }
    uint32_t n_big = 0;
    for (int b = kBigTileBin; b < 64; b++) n_big += s_hist[b];
    host_map[0] = (unsigned long long)s_warp[31];  // R
    host_map[2] = (unsigned long long)s_max[0];    // largest tile
    host_map[3] = (unsigned long long)n_big;       // tiles with >= kBigTileBin^2 instances (they lead `order`)
    __threadfence_system();
    host_map[1] = seq;
    __threadfence_system();
  }
  __syncthreads();
  for (int t = t0; t < t1; t++) order[atomicAdd(&s_start[min(63, (int)sqrtf((float)tile_count[t]))], 1u)] = (uint32_t)t;
}

// Drop a (depth bits << 32 | id) key into the range of every owned tile of each visible Gaussian's rectangle
// (reference: duplicateWithKeys, rasterizer_impl.cu:70-111; here the tile is implied by the slot), warp-cooperatively.
__global__ void __launch_bounds__(256)
emit_binned_kernel(int P, const uint32_t* __restrict__ tiles_touched, const Splat* __restrict__ splats,
                   const int32_t* __restrict__ radii, int tiles_x, int tiles_y, int shard_count,
                   int shard_index, uint32_t* __restrict__ cursor, unsigned long long* __restrict__ keys) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  const bool vis = (g < P) && tiles_touched[g] != 0;
  int x0 = 0, y0 = 0, x1 = 0, y1 = 0;
  unsigned long long key = 0;
  if (vis) {
    const Splat* sp = splats + g;
    const float4 a = sp->a;
    key = ((unsigned long long)__float_as_uint(sp->c.w) << 32) | (unsigned long long)(uint32_t)g;
    tile_rect(a.x, a.y, radii[g], tiles_x, tiles_y, x0, y0, x1, y1);
  }
  // (Measured and dropped, r2p: keeping the slot atomics of four Gaussians in flight before the dependent key stores did
  // not shorten the kernel — it waits on the gathered splat / radius loads, not on the atomics' return values.)
  for_each_owned_tile(vis, x0, y0, x1, y1, tiles_x, shard_count, shard_index, key,
                      [&](unsigned long long k, int t) { keys[atomicAdd(&cursor[t], 1u)] = k; });
}

// One CTA per tile: bitonic sort of the tile's keys in shared memory, ids written to point_list.  CTA b sorts tile
// order[first + b] (the size classes are ranges of `order`); a tile above cap is left to the segmented-sort fallback.
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
tile_sort_kernel(const uint32_t* __restrict__ order, int first, int cap, const uint2* __restrict__ ranges,
                 const unsigned long long* __restrict__ keys, uint32_t* __restrict__ point_list) {
  extern __shared__ unsigned long long sk[];
  const uint2 r = ranges[order[first + blockIdx.x]];
  const int n = (int)(r.y - r.x);
  if (n <= 0 || n > cap) return;
  if (n == 1) {
    if (threadIdx.x == 0) point_list[r.x] = (uint32_t)keys[r.x];
    return;
  }
  int N = 2;
  while (N < n) N <<= 1;
  for (int i = threadIdx.x; i < N; i += THREADS) sk[i] = (i < n) ? keys[r.x + i] : ~0ull;
  __syncthreads();
  for (int k = 2; k <= N; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < (N >> 1); i += THREADS) {
        const int lo = ((i & ~(j - 1)) << 1) | (i & (j - 1));  // insert a 0 bit at position log2(j)
        const int hi = lo | j;
        const bool up = ((lo & k) == 0);
        const unsigned long long x = sk[lo], y = sk[hi];
        if ((x > y) == up) {
          sk[lo] = y;
          sk[hi] = x;
        }
      }
      // With this indexing the 32 compare-exchanges of a warp touch exactly the 64 keys [64 w, 64 w + 64) whenever j <= 32
      // (w = i / 32, the same in every stage): between two such stages only the warp itself has to be in step.  A stage with
      // j > 32 crosses warps, and so does the final copy-out.  512 keys: 9 block barriers instead of 45.
      const int next_j = (j > 1) ? (j >> 1) : ((k < N) ? k : 0);
      if (j > 32 || next_j > 32 || next_j == 0)
        __syncthreads();
      else
        __syncwarp();
    }
  }
  for (int i = threadIdx.x; i < n; i += THREADS) point_list[r.x + i] = (uint32_t)sk[i];
}

__global__ void keys_to_ids_kernel(int R, const unsigned long long* __restrict__ keys, uint32_t* __restrict__ point_list) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < R) point_list[i] = (uint32_t)keys[i];
}

// ------------------------------------------------------------------------------------------
// render forward: one CTA per 16x16 tile, each warp owns an 8x4 sub-tile.
//
// Per batch of 256 tile instances the CTA stages the 48-B splat records in shared memory with
// 128-bit loads (one instance per thread).  Each warp then culls the batch against its own 8x4
// pixel rectangle — lane l tests instance 32*chunk+l: the exact minimum of the conic's
// quadratic form over the rectangle against ln(255*opacity) (raster_common.cuh: subtile_hit) — and only the survivors (ballot mask) are evaluated by all 32 lanes.
// Culled instances are exactly those the reference skips for every pixel of the sub-tile
// (power > 0 or alpha < 1/255, forward.cu:359-366), so the blend result is unchanged while the
// pixel-Gaussian pair count drops by the ratio (bounding-square tiles) / (ellipse ∩ sub-tiles).
// ------------------------------------------------------------------------------------------
template <bool kCull>
__global__ void __launch_bounds__(kTilePixels)
render_forward_kernel(const uint32_t* __restrict__ tile_order, const uint2* __restrict__ ranges,
                      const uint32_t* __restrict__ point_list, int W, int H,
                      int tiles_x, const Splat* __restrict__ splats, const float* __restrict__ bg,
                      float* __restrict__ out_color, float* __restrict__ out_depth, float* __restrict__ final_T,
                      uint32_t* __restrict__ n_contrib, uint32_t* __restrict__ hit_out, int shard_count, int shard_index) {
  const int tile = (int)tile_order[blockIdx.x];
  if (shard_count > 1 && (tile % shard_count) != shard_index) return;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tile_x = tile % tiles_x, tile_y = tile / tiles_x;
  const int wx0 = tile_x * kTile + (warp & 1) * 8, wy0 = tile_y * kTile + (warp >> 1) * 4;
  const int px = wx0 + (lane & 7), py = wy0 + (lane >> 3);
  const bool inside = px < W && py < H;
  const float pxf = (float)px, pyf = (float)py;

  // double-buffered staging of 256 instances: one barrier per batch, loads of batch k+1 overlap the blending of batch k
  __shared__ __align__(16) float4 sA2[2][kTilePixels], sB2[2][kTilePixels], sC2[2][kTilePixels];

  const uint2 range = ranges[tile];
  const int total = (int)(range.y - range.x);
  bool done = !inside;
  float T = 1.f, Cr = 0.f, Cg = 0.f, Cb = 0.f, D = 0.f;
  uint32_t last = 0;

  auto stage = [&](int base, int buf) {
    const int n = min(kTilePixels, total - base);
    if (tid < n) {
      const uint32_t g = point_list[range.x + base + tid];
      const Splat* sp = splats + g;
      cp_async16(&sA2[buf][tid], &sp->a);
      cp_async16(&sB2[buf][tid], &sp->b);
      cp_async16(&sC2[buf][tid], &sp->c);
    }
    cp_async_commit();
  };
  if (total > 0) stage(0, 0);

  for (int base = 0, buf = 0; base < total; base += kTilePixels, buf ^= 1) {
    // barrier: batch `base` is staged (each thread's asynchronous copies have landed) and every warp is done with the
    // other buffer; also the block-wide early exit
    cp_async_wait_all();
    if (__syncthreads_count(done) == kTilePixels) break;
    if (base + kTilePixels < total) stage(base + kTilePixels, buf ^ 1);
    const int n = min(kTilePixels, total - base);
    const float4* sA = sA2[buf];
    const float4* sB = sB2[buf];
    const float4* sC = sC2[buf];
    if (__all_sync(0xffffffffu, done)) continue;

    for (int c0 = 0; c0 < n; c0 += 32) {
      uint32_t mask;
      if (kCull) {
        const int j = c0 + lane;
        const bool hit = (j < n) && subtile_hit(sA[j], sB[j], (float)wx0, (float)wy0, 7.f, 3.f);
        mask = __ballot_sync(0xffffffffu, hit);
      } else {
        mask = (n - c0 >= 32) ? 0xffffffffu : ((1u << (n - c0)) - 1u);
      }
      // kept for the backward pass (BinState::hit): every chunk this warp evaluates reaches at least its last contributor
      if (lane == 0) hit_out[(hit_word(range.x, tile) + (size_t)((base + c0) >> 5)) * 8 + warp] = mask;
      while (mask) {
        const int bit = __ffs(mask) - 1;
        mask &= mask - 1;
        const int j = c0 + bit;
        // Branch-free blend step: every lane evaluates the instance, the state update is predicated.  The
        // expressions keep the reference's shape ((c * alpha) * T, forward.cu:373-375,400) so results match bit for bit.
        const float4 a = sA[j], b = sB[j], c = sC[j];
        const float dx = a.x - pxf, dy = a.y - pyf;
        const float power = -0.5f * (a.z * dx * dx + b.x * dy * dy) - a.w * dx * dy;
        const float alpha = fminf(0.99f, b.y * expf(power));
        const float test_T = T * (1 - alpha);
        const bool hit = !done && !(power > 0.0f) && !(alpha < 1.0f / 255.0f);
        const bool blend = hit && !(test_T < 0.0001f);
        done = done || (hit && !blend);  // colour and depth both stop here (forward.cu:367-383,392-393)
        // depth conditioned on the pixel offset through the z cross-covariances (forward.cu:395-399)
        const float dcond = c.w - (b.z * a.z + b.w * a.w) * dx - (b.z * a.w + b.w * b.x) * dy;
        Cr = blend ? (Cr + c.x * alpha * T) : Cr;
        Cg = blend ? (Cg + c.y * alpha * T) : Cg;
        Cb = blend ? (Cb + c.z * alpha * T) : Cb;
        D = blend ? (D + dcond * alpha * T) : D;
        T = blend ? test_T : T;
        last = blend ? (uint32_t)(base + j + 1) : last;
      }
      if (__all_sync(0xffffffffu, done)) break;
    }
  }

  if (inside) {
    const int pix = py * W + px;
    final_T[pix] = T;
    n_contrib[pix] = last;
    out_depth[pix] = D + T * 15.f;  // background depth 15 m (forward.cu:419-421)
    const size_t HW = (size_t)H * W;
    out_color[0 * HW + pix] = Cr + T * bg[0];
    out_color[1 * HW + pix] = Cg + T * bg[1];
    out_color[2 * HW + pix] = Cb + T * bg[2];
  }
}

__global__ void mark_visible_kernel(int P, const float* __restrict__ means, const float* __restrict__ view,
                                    uint8_t* __restrict__ present) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P) return;
  const float3 p = make_float3(means[3 * idx], means[3 * idx + 1], means[3 * idx + 2]);
  present[idx] = xform_point_4x3(p, view).z > 0.2f;
}

__global__ void copy_ranges_kernel(int tiles, const uint2* __restrict__ ranges, uint32_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < tiles) {
    out[2 * i] = ranges[i].x;
    out[2 * i + 1] = ranges[i].y;
  }
}

// Library-internal scratch (not needed by backward), one set PER DEVICE: one rasterization in flight per device (the mutex
// is held until the forward's launches are enqueued; streams of one device share the scratch and are serialised by the
// host-side wait on the instance count).  The reference launches everything on the legacy default stream.
constexpr int kMaxDevices = 32;
struct FwdScratch {
  std::mutex mu;
  Scratch per_gaussian, per_instance, cub_tmp;
  HostMailbox box;  // [0] num_rendered, [1] sequence word, [2] largest tile, [3] tiles of >= kSmallTileCap instances
  bool sort_attr_set = false;  // cudaFuncSetAttribute of the big tile sort, per device
};
static FwdScratch g_fwd_dev[kMaxDevices];

float* raster_moment_accumulator(const gsicp_raster_args* args, float* geom_moments);  // raster_backward.cu

int g_render_cull = 1;  // test hook: 0 renders without sub-tile culling (must give identical output)

}  // namespace gsicp

using namespace gsicp;

extern "C" int gsicp_raster_forward(const gsicp_raster_args* args, float* d_out_color, float* d_out_depth,
                                    int32_t* d_radii, uint8_t* d_is_used, gsicp_alloc_fn geom_alloc,
                                    gsicp_alloc_fn binning_alloc, gsicp_alloc_fn image_alloc, void* user,
                                    void* stream_v) {
  if (!args || !geom_alloc || !binning_alloc || !image_alloc) {
    set_error("gsicp_raster_forward: null argument");
    return GSICP_EINVAL;
  }
  const int P = args->P, W = args->width, H = args->height;
  if (P < 0 || W <= 0 || H <= 0) {
    set_error("gsicp_raster_forward: bad sizes P=%d W=%d H=%d", P, W, H);
    return GSICP_EINVAL;
  }
  if (!args->d_shs && !args->d_colors_precomp && P > 0) {
    set_error("gsicp_raster_forward: provide SHs or precomputed colours");
    return GSICP_EINVAL;
  }
  if (!args->d_cov3D_precomp && (!args->d_scales || !args->d_rotations) && P > 0) {
    set_error("gsicp_raster_forward: provide scale/rotation or precomputed 3D covariance");
    return GSICP_EINVAL;
  }
  cudaStream_t stream = (cudaStream_t)stream_v;
  const int shard_count = args->tile_shard_count > 1 ? args->tile_shard_count : 1;
  const int shard_index = shard_count > 1 ? args->tile_shard_index : 0;
  const int tiles_x = (W + kTile - 1) / kTile, tiles_y = (H + kTile - 1) / kTile;
  const int tiles = tiles_x * tiles_y;
  const size_t N = (size_t)W * H;

  char* geom_p = (char*)geom_alloc(GeomState::bytes(P), user);
  char* img_p = (char*)image_alloc(ImgState::bytes(N, tiles), user);
  if (!geom_p || !img_p) {
    set_error("gsicp_raster_forward: workspace callback returned NULL");
    return GSICP_ENOMEM;
  }
  GeomState geom = GeomState::from(geom_p, P);
  ImgState img = ImgState::from(img_p, N, tiles);

  int dev = 0;
  GSICP_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices) {
    set_error("gsicp_raster_forward: device index %d out of range", dev);
    return GSICP_EINVAL;
  }
  FwdScratch& g_fwd = g_fwd_dev[dev];
  std::lock_guard<std::mutex> lock(g_fwd.mu);
  HostMailbox& box = g_fwd.box;
  if (int e = box.ensure(4 * sizeof(unsigned long long))) return e;

  int R = 0;
  unsigned long long max_tile = 0;
  int n_big = 0;
  uint32_t *tiles_touched = nullptr, *tile_count = nullptr, *cursor = nullptr, *seg_begin = nullptr, *seg_end = nullptr;
  if (P > 0) {
    // scratch: u32[P] owned-tile counts + 4 x u32[tiles]
    const size_t pstride = ((size_t)P * 4 + 127) & ~size_t(127);
    const size_t tstride = ((size_t)tiles * 4 + 127) & ~size_t(127);
    if (int e = g_fwd.per_gaussian.ensure(pstride + 4 * tstride)) return e;
    char* base = g_fwd.per_gaussian.as<char>();
    tiles_touched = (uint32_t*)base;
    tile_count = (uint32_t*)(base + pstride);
    cursor = (uint32_t*)(base + pstride + tstride);
    seg_begin = (uint32_t*)(base + pstride + 2 * tstride);
    seg_end = (uint32_t*)(base + pstride + 3 * tstride);
    GSICP_CUDA(cudaMemsetAsync(tile_count, 0, (size_t)tiles * 4, stream));

    PreArgs pa;
    pa.P = P; pa.D = args->D; pa.M = args->M; pa.W = W; pa.H = H; pa.tiles_x = tiles_x; pa.tiles_y = tiles_y;
    pa.tan_fovx = args->tan_fovx; pa.tan_fovy = args->tan_fovy;
    pa.focal_y = H / (2.0f * args->tan_fovy);
    pa.focal_x = W / (2.0f * args->tan_fovx);
    pa.scale_modifier = args->scale_modifier;
    pa.means = args->d_means3D; pa.scales = args->d_scales; pa.rots = args->d_rotations; pa.opac = args->d_opacities;
    pa.shs = args->d_shs; pa.cov_pre = args->d_cov3D_precomp; pa.col_pre = args->d_colors_precomp;
    pa.view = args->d_viewmatrix; pa.proj = args->d_projmatrix; pa.campos = args->d_campos;
    pa.prefiltered = args->prefiltered; pa.shard_count = shard_count; pa.shard_index = shard_index;
    {
      ProfScope ps(kProfPreprocess, stream);
      // the rows preprocess zeroes are where render_backward will accumulate: the geometry buffer, or this rank's exchange
      // segment in a sharded run (comm.cuh)
      GSICP_LAUNCH(preprocess_kernel, (P + 255) / 256, 256, 0, stream, pa, d_radii, d_is_used, geom.splats,
                   raster_moment_accumulator(args, geom.moments), geom.clamped, tiles_touched, tile_count);
    }
    if (args->debug) GSICP_CUDA(cudaStreamSynchronize(stream));

    // The Python API returns num_rendered as a host int (DGR/diff_gaussian_rasterization/__init__.py:96) and the instance
    // buffers are sized by it (rasterizer_impl.cu:286-287 does a blocking 4-byte memcpy).  Here the scan kernel publishes
    // it into mapped pinned memory and the host spins on a sequence word.
    const unsigned long long seq = ++box.seq;
    {
      ProfScope ps(kProfDepthSort, stream);  // slot reused: "tile_scan"
      GSICP_LAUNCH(tile_scan_kernel, 1, 1024, 0, stream, tiles, tile_count, img.ranges, cursor, seg_begin, seg_end,
                   img.tile_order, (volatile unsigned long long*)box.dev, seq);
    }
    GSICP_CUDA(cudaGetLastError());
    if (int e = box.wait(1, seq, stream, "rasterizer instance count")) return e;
    if (box.host[0] > 0x7fffffffull) {
      set_error("gsicp_raster_forward: instance count overflow");
      return GSICP_EINVAL;
    }
    R = (int)box.host[0];
    max_tile = box.host[2];
    n_big = (int)box.host[3];
  } else {
    GSICP_CUDA(cudaMemsetAsync(img.ranges, 0, sizeof(uint2) * tiles, stream));
  }

  char* bin_p = (char*)binning_alloc(BinState::bytes(R, (size_t)tiles), user);
  if (!bin_p) {
    set_error("gsicp_raster_forward: binning callback returned NULL");
    return GSICP_ENOMEM;
  }
  BinState bin = BinState::from(bin_p, R, (size_t)tiles);

  if (R > 0) {
    const size_t kbytes = ((size_t)R * 8 + 127) & ~size_t(127);
    const bool big = max_tile > (unsigned long long)kTileSortCap;
    if (int e = g_fwd.per_instance.ensure(big ? 2 * kbytes : kbytes)) return e;
    unsigned long long* keys = g_fwd.per_instance.as<unsigned long long>();
    {
      ProfScope ps(kProfEmit, stream);
      GSICP_LAUNCH(emit_binned_kernel, (P + 255) / 256, 256, 0, stream, P, tiles_touched, geom.splats, d_radii, tiles_x, tiles_y,
                   shard_count, shard_index, cursor, keys);
    }
    {
      ProfScope ps(kProfTileSort, stream);
      if (!big) {
        if (n_big > 0) {
          bool& attr_set = g_fwd.sort_attr_set;
          if (!attr_set) {
            GSICP_CUDA(cudaFuncSetAttribute(tile_sort_kernel<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTileSortCap * 8));
            attr_set = true;
          }
          int cap = kSmallTileCap;
          while ((unsigned long long)cap < max_tile) cap <<= 1;
          GSICP_LAUNCH(tile_sort_kernel<1024>, n_big, 1024, (size_t)cap * 8, stream, img.tile_order, 0, cap, img.ranges,
                       keys, bin.point_list);
        }
        if (tiles > n_big)
          GSICP_LAUNCH(tile_sort_kernel<256>, tiles - n_big, 256, (size_t)kSmallTileCap * 8, stream, img.tile_order, n_big,
                       kSmallTileCap, img.ranges, keys, bin.point_list);
      } else {
        // some tile exceeds the shared-memory sort: segmented radix sort of the same 64-bit keys (31 depth bits + id bits)
        unsigned long long* keys_out = (unsigned long long*)((char*)keys + kbytes);
        int id_bits = 1;
        while ((1ull << id_bits) < (unsigned long long)P) id_bits++;
        size_t tmp = 0;
        cub::DeviceSegmentedRadixSort::SortKeys(nullptr, tmp, keys, keys_out, R, tiles, seg_begin, seg_end, 0, 64, stream);
        if (int e = g_fwd.cub_tmp.ensure(tmp)) return e;
        tmp = g_fwd.cub_tmp.cap;
        GSICP_CUDA(cub::DeviceSegmentedRadixSort::SortKeys(g_fwd.cub_tmp.ptr, tmp, keys, keys_out, R, tiles, seg_begin, seg_end,
                                                          0, 64, stream));
        (void)id_bits;
        GSICP_LAUNCH(keys_to_ids_kernel, (R + 255) / 256, 256, 0, stream, R, keys_out, bin.point_list);
      }
    }
    if (args->debug) GSICP_CUDA(cudaStreamSynchronize(stream));
  }

  if (P > 0) {
    ProfScope ps(kProfRenderFwd, stream);
    if (g_render_cull) {
      GSICP_LAUNCH(render_forward_kernel<true>, tiles, kTilePixels, 0, stream, img.tile_order, img.ranges, bin.point_list, W, H, tiles_x,
                   geom.splats, args->d_background, d_out_color, d_out_depth, img.final_T, img.n_contrib, bin.hit, shard_count,
                   shard_index);
    } else {
      GSICP_LAUNCH(render_forward_kernel<false>, tiles, kTilePixels, 0, stream, img.tile_order, img.ranges, bin.point_list, W, H, tiles_x,
                   geom.splats, args->d_background, d_out_color, d_out_depth, img.final_T, img.n_contrib, bin.hit, shard_count,
                   shard_index);
    }
    if (args->debug) GSICP_CUDA(cudaStreamSynchronize(stream));
  }
  GSICP_CUDA(cudaGetLastError());
  return R;
}

extern "C" int gsicp_raster_export_binning(const gsicp_raster_args* args, int num_rendered, const void* d_binning,
                                           const void* d_image, uint32_t* d_point_list, uint32_t* d_ranges,
                                           void* stream_v) {
  if (!args || !d_binning || !d_image) return GSICP_EINVAL;
  cudaStream_t stream = (cudaStream_t)stream_v;
  const int W = args->width, H = args->height;
  const int tiles_x = (W + kTile - 1) / kTile, tiles_y = (H + kTile - 1) / kTile, tiles = tiles_x * tiles_y;
  BinState bin = BinState::from((char*)d_binning, num_rendered, (size_t)tiles);
  ImgState img = ImgState::from((char*)d_image, (size_t)W * H, tiles);
  if (d_point_list && num_rendered > 0)
    GSICP_CUDA(cudaMemcpyAsync(d_point_list, bin.point_list, sizeof(uint32_t) * (size_t)num_rendered,
                               cudaMemcpyDeviceToDevice, stream));
  if (d_ranges) GSICP_LAUNCH(copy_ranges_kernel, (tiles + 255) / 256, 256, 0, stream, tiles, img.ranges, d_ranges);
  GSICP_CUDA(cudaGetLastError());
  return GSICP_OK;
}

extern "C" int gsicp_mark_visible(int P, const float* d_means3D, const float* d_viewmatrix, const float* d_projmatrix,
                                  uint8_t* d_present, void* stream_v) {
  (void)d_projmatrix;
  if (P < 0) return GSICP_EINVAL;
  if (P == 0) return GSICP_OK;
  GSICP_LAUNCH(mark_visible_kernel, (P + 255) / 256, 256, 0, (cudaStream_t)stream_v, P, d_means3D, d_viewmatrix,
               d_present);
  GSICP_CUDA(cudaGetLastError());
  return GSICP_OK;
}

extern "C" void gsicp_test_set_render_cull(int on) { gsicp::g_render_cull = on; }
