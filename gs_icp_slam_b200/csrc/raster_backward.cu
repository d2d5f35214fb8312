// raster_backward.cu — backward pass of the B200 Gaussian-splat rasterizer.
//
// Replaces CudaRasterizer::Rasterizer::backward (DGR/cuda_rasterizer/rasterizer_impl.cu:351-454):
//   BACKWARD::render (backward.cu:429-657)  +  computeCov2DCUDA (:144-294)  +  preprocessCUDA (:369-426)
//
// render backward: the reference issues up to 12 global float atomicAdd per contributing pixel-Gaussian pair.  Here each
// warp owns an 8x4 sub-tile, culls the staged batch exactly as the forward does, replays the blend back to front, and per
// surviving (sub-tile, instance) only TWO per-pixel scalars are formed: t = G * dL/dalpha and w = alpha * T.  The
// reference's 12 per-pair gradient expressions (backward.cu:575-654) are linear in twelve MOMENTS of those two fields over
// the pixels (t against {1, dx, dy, dx^2, dx dy, dy^2}; w against dL/dpix_depth {1, dx, dy} and dL/dpix_{r,g,b}), and a sum
// over the 32 pixels of a warp against fixed per-pixel weights is a small matrix product: the (t, w) values of 8 survivors
// are transposed through 2.3 KB of shared memory per warp and reduced by the tensor cores
// (mma.sync.m16n8k8 tf32, fp32 accumulate; values split hi/lo so the products carry 22 mantissa bits):
//     D[12 moments x 8 instances] = A[12 x 32 pixels] * B[32 pixels x 8 instances]
// with the pixel-offset basis taken in the warp's own integer frame (exact in tf32) and shifted to the Gaussian's centre
// afterwards.  20 MMAs + 4 REDs serve 8 instances, instead of 13 shuffles + 26 selects + 13 adds + 1 RED per instance.
// Global atomics: 12 per (sub-tile, instance) that blended anything, vs 12 per (pixel, Gaussian) pair in the reference.
//
// per-Gaussian backward: computeCov2D backward and the preprocess backward are one kernel (the
// intermediate dL_dcov3D / dL_dmeans never round-trip through HBM between two launches).
#include <cstdlib>
#include <mutex>
#include "host_common.h"
#include "raster_common.cuh"
#include "comm.cuh"

namespace gsicp {

constexpr int kG = 12;    // moments per Gaussian (see below)
constexpr int kGrp = 8;   // survivors reduced per MMA group (the N dimension of m16n8k8)
constexpr int kRow = 36;  // words per staged row: 32 pixels + 4 pad (conflict-free 128-bit fragment loads)
constexpr int kWarps = kTilePixels / 32;

// Dynamic shared memory of render_backward_kernel (59 392 B; three CTAs per SM):
template <int kStage>
struct __align__(16) BwdSmemT {
  float4 a[2][kStage], b[2][kStage], c[2][kStage];  // double-buffered staging of kStage splat records
  float tq[kWarps][kGrp * kRow], wq[kWarps][kGrp * kRow];          // per-warp transposition buffers of the MMA reduction
  float4 aw[kWarps][4][32];                                        // per-warp constant A fragments of the w-block
};
using BwdSmem = BwdSmemT<kTilePixels>;

// D += A * B, A 16x8 (row major), B 8x8 (column major), tf32 inputs (the low 13 mantissa bits are ignored), fp32 accumulate.
// Fragment layout (PTX ISA, mma.m16n8k8 .tf32), g = lane >> 2, t = lane & 3:
//   a0 = A[g][t], a1 = A[g+8][t], a2 = A[g][t+4], a3 = A[g+8][t+4];  b0 = B[t][g], b1 = B[t+4][g];
//   d0 = D[g][2t], d1 = D[g][2t+1], d2 = D[g+8][2t], d3 = D[g+8][2t+1].
__device__ __forceinline__ void mma_tf32(float (&d)[4], float a0, float a1, float a2, float a3, float b0, float b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(__float_as_uint(a0)), "r"(__float_as_uint(a1)), "r"(__float_as_uint(a2)), "r"(__float_as_uint(a3)),
        "r"(__float_as_uint(b0)), "r"(__float_as_uint(b1)));
}
// Shared-memory accesses by 32-bit window address + immediate offset: with the addresses formed once per chunk / per thread
// the survivor loop carries no address arithmetic (the compiler otherwise rebuilds the window base every iteration
// under the 64-register cap).
template <int kOff>
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4+%5];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr), "n"(kOff));
  return v;
}
template <int kOff>
__device__ __forceinline__ void sts32(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0+%1], %2;" ::"r"(addr), "n"(kOff), "f"(v) : "memory");
}
__device__ __forceinline__ float rcp_approx(float x) {  // MUFU.RCP, 1 ulp; the backward's tolerance is 2e-4 of the maximum
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// x = hi + lo with hi exactly representable in tf32 (lo keeps the next 11 bits once the MMA drops its own low bits)
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }

// moments[P][12], summed over every pixel the Gaussian was blended into (dx = mean2D.x - pixel.x, dy likewise):
//   [0..5]  sum t {1, dx, dy, dx^2, dx dy, dy^2}     t = G (dL/dalpha + dL/dalpha_d)     ([0] = dL/dopacity)
//   [6..8]  sum v {1, dx, dy}                         v = w dL/dpix_depth, w = alpha T   ([6] = dL/ddepth)
//   [9..11] sum w dL/dpix_{r,g,b}                                                         (= dL/dcolour)
// gaussian_backward_kernel forms the reference's gradients from them with per-Gaussian coefficients.
// Measured and dropped (profiles/r2b_notes.md): a software-pipelined survivor loop (alpha evaluation of candidate k+1
// interleaved with the blend chain of candidate k in one predicated basic block: 240 us vs 226 us) and a 128-register /
// 2-CTA-per-SM build (262-276 us): the kernel wants resident warps, not more ILP per warp.
// kStage / kMinBlocks: (256, 3) = 80 registers, 58 KB of shared memory, 3 CTAs per SM (default);
// (128, 4) = 64 registers, 46 KB, 4 CTAs per SM (experiment: GSICP_BWD_VARIANT=1).
template <bool kCull, int kStage = kTilePixels, int kMinBlocks = 3>
__global__ void __launch_bounds__(kTilePixels, kMinBlocks)
render_backward_kernel(const uint32_t* __restrict__ tile_order, const uint2* __restrict__ ranges,
                       const uint32_t* __restrict__ point_list, int W, int H,
                       int tiles_x, const float* __restrict__ bg, const Splat* __restrict__ splats,
                       const float* __restrict__ final_T, const uint32_t* __restrict__ n_contrib,
                       const float* __restrict__ dL_dpix_color, const float* __restrict__ dL_dpix_depth,
                       float* __restrict__ moments, const uint32_t* __restrict__ hit_in, int shard_count, int shard_index) {
  const int tile = (int)tile_order[blockIdx.x];
  if (shard_count > 1 && (tile % shard_count) != shard_index) return;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tile_x = tile % tiles_x, tile_y = tile / tiles_x;
  const int wx0 = tile_x * kTile + (warp & 1) * 8, wy0 = tile_y * kTile + (warp >> 1) * 4;
  const int px = wx0 + (lane & 7), py = wy0 + (lane >> 3);
  const bool inside = px < W && py < H;
  const float pxf = (float)px, pyf = (float)py;
  const float wx0f = (float)wx0, wy0f = (float)wy0;
  const int pix = py * W + px;

  extern __shared__ __align__(16) unsigned char smem_raw[];
  BwdSmemT<kStage>& sm = *reinterpret_cast<BwdSmemT<kStage>*>(smem_raw);

  const uint2 range = ranges[tile];
  const int total = (int)(range.y - range.x);

  const float T_final = inside ? final_T[pix] : 0.f;
  float T = T_final;
  const int last_contributor = inside ? (int)n_contrib[pix] : 0;
  // instances behind the deepest contributor of this warp's pixels are never touched
  int warp_last = last_contributor;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) warp_last = max(warp_last, __shfl_xor_sync(0xffffffffu, warp_last, o));

  float dpr = 0.f, dpg = 0.f, dpb = 0.f, dpd = 0.f;
  if (inside) {
    const size_t HW = (size_t)H * W;
    dpr = dL_dpix_color[0 * HW + pix];
    dpg = dL_dpix_color[1 * HW + pix];
    dpb = dL_dpix_color[2 * HW + pix];
    dpd = dL_dpix_depth[pix];
  }
  const float bg_dot_dpixel = bg[0] * dpr + bg[1] * dpg + bg[2] * dpb;
  const float bg_dot_ddepth = 15.f * dpd;
  const float bg_term = T_final * (bg_dot_dpixel + bg_dot_ddepth);  // background share of dL/dalpha + dL/dalpha_d

  // ---- A operand of the reduction: rows = moments, columns = the warp's 32 pixels (k = lane; i = k & 7, j = k >> 3) ----
  // Thread (g8, t4) supplies, for k-step ks, the columns k = 8 ks + t4 and k + 4 (i = t4 / t4 + 4, j = ks) of its rows.
  //   t-block (B = t values):  row g8 < 6 = {1, i, j, i^2, i j, j^2} in the warp's integer frame — exact in tf32, and a
  //     polynomial in j = ks: at = alpha + j (beta + gamma j) with per-thread constants (5 registers).
  //   w-block (B = w values):  row g8 < 6 = HIGH tf32 part of {dpd, dpd i, dpd j, dpr, dpg, dpb}(pixel k), row 8 + g8 = the
  //     LOW part (dp* = dL/dpix_*): both parts ride the same MMA and are added in the epilogue.  Kept in shared memory.
  const int g8 = lane >> 2, t4 = lane & 3;
  const float fi0 = (float)t4, fi1 = (float)(t4 + 4);
  const float t_al0 = g8 == 0 ? 1.f : g8 == 1 ? fi0 : g8 == 3 ? fi0 * fi0 : 0.f;
  const float t_al1 = g8 == 0 ? 1.f : g8 == 1 ? fi1 : g8 == 3 ? fi1 * fi1 : 0.f;
  const float t_be0 = g8 == 2 ? 1.f : g8 == 4 ? fi0 : 0.f;
  const float t_be1 = g8 == 2 ? 1.f : g8 == 4 ? fi1 : 0.f;
  const float t_ga = g8 == 5 ? 1.f : 0.f;
#pragma unroll
  for (int ks = 0; ks < 4; ks++) {
    float hi[2], lo[2];
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int k = 8 * ks + t4 + 4 * h;
      const float fi = (float)(k & 7), fj = (float)(k >> 3);
      const float kr = __shfl_sync(0xffffffffu, dpr, k), kg = __shfl_sync(0xffffffffu, dpg, k);
      const float kb = __shfl_sync(0xffffffffu, dpb, k), kd = __shfl_sync(0xffffffffu, dpd, k);
      const float v = g8 == 0 ? kd : g8 == 1 ? kd * fi : g8 == 2 ? kd * fj : g8 == 3 ? kr : g8 == 4 ? kg : g8 == 5 ? kb : 0.f;
      hi[h] = tf32_hi(v);
      lo[h] = v - hi[h];
    }
    sm.aw[warp][ks][lane] = make_float4(hi[0], lo[0], hi[1], lo[1]);  // {a0, a1, a2, a3} of k-step ks
  }
  float* const myT = sm.tq[warp];
  float* const myW = sm.wq[warp];
  const int wpos = (lane & 3) * 8 + (lane >> 2);  // pixel k = lane sits at word (k & 3) * 8 + (k >> 2): the 8 pixels a
                                                  // thread needs for its B fragments are 8 consecutive words
  constexpr int kOffB = 2 * kStage * 16, kOffC = 4 * kStage * 16;           // sm.b / sm.c relative to sm.a (same buffer)
  constexpr int kOffW = kWarps * kGrp * kRow * 4;                           // sm.wq relative to sm.tq
  const uint32_t s_base = (uint32_t)__cvta_generic_to_shared(smem_raw);
  uint32_t s_slot = (uint32_t)__cvta_generic_to_shared(myT + wpos);         // this lane's word of survivor slot 0
  asm volatile("" : "+r"(s_slot));                                          // opaque: one register, never rebuilt in the loop
  int cnt = 0;                                    // survivors staged in the current group (warp-uniform)
  float m_cx = 0.f, m_cy = 0.f;                   // lane s: centre of survivor s in the warp's frame, and its Gaussian
  uint32_t m_id = 0;

  // Reduce the staged group: D = A * B on the tensor cores, shift the pixel-frame moments to each Gaussian's centre,
  // one fp32 RED per moment.
  const bool r_1 = g8 == 1, r_2 = g8 == 2, r_3 = g8 == 3, r_4 = g8 == 4, r_5 = g8 == 5;
  auto flush = [&]() {
    for (int s2 = cnt; s2 < kGrp; s2++) {  // unused slots contribute zero
      myT[s2 * kRow + wpos] = 0.f;
      myW[s2 * kRow + wpos] = 0.f;
    }
    __syncwarp();
    const float4* rt = reinterpret_cast<const float4*>(myT + g8 * kRow + t4 * 8);
    const float4* rw = reinterpret_cast<const float4*>(myW + g8 * kRow + t4 * 8);
    float dT[4] = {0.f, 0.f, 0.f, 0.f}, dW[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int half = 0; half < 2; half++) {  // words 4 half .. 4 half + 3 of the row feed the k-steps 2 half and 2 half + 1
      const float4 tv = rt[half], wv = rw[half];
      const float bt[4] = {tv.x, tv.y, tv.z, tv.w}, bw[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int q = 0; q < 2; q++) {
        const int ks = 2 * half + q;
        const float fj = (float)ks;
        const float at0 = t_al0 + fj * (t_be0 + t_ga * fj), at1 = t_al1 + fj * (t_be1 + t_ga * fj);
        const float th0 = tf32_hi(bt[2 * q]), th1 = tf32_hi(bt[2 * q + 1]);
        mma_tf32(dT, at0, at0, at1, at1, th0, th1);                                // rows 8..15 of dT are not used
        mma_tf32(dT, at0, at0, at1, at1, bt[2 * q] - th0, bt[2 * q + 1] - th1);
        const float4 aw = sm.aw[warp][ks][lane];
        const float wh0 = tf32_hi(bw[2 * q]), wh1 = tf32_hi(bw[2 * q + 1]);
        mma_tf32(dW, aw.x, aw.y, aw.z, aw.w, wh0, wh1);
        mma_tf32(dW, aw.x, aw.y, aw.z, aw.w, bw[2 * q] - wh0, bw[2 * q + 1] - wh1);
      }
    }
    __syncwarp();  // every lane has read its fragments: the slots may be overwritten
    // thread (g8, t4) holds moment row g8 of the instances 2 t4 (index 0) and 2 t4 + 1 (index 1):
    // t-block dT[h]; w-block high + low part dW[h] + dW[2 + h]
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int n = 2 * t4 + h;
      const float own_t = dT[h], own_w = dW[h] + dW[2 + h];
      // pixel-frame sums of rows 0, 1, 2 of this instance live in the threads (0, t4), (1, t4), (2, t4)
      const float S0 = __shfl_sync(0xffffffffu, own_t, t4), S1 = __shfl_sync(0xffffffffu, own_t, 4 + t4);
      const float S2 = __shfl_sync(0xffffffffu, own_t, 8 + t4);
      const float V0 = __shfl_sync(0xffffffffu, own_w, t4);
      const float cx = __shfl_sync(0xffffffffu, m_cx, n), cy = __shfl_sync(0xffffffffu, m_cy, n);
      const uint32_t gid = __shfl_sync(0xffffffffu, m_id, n);
      // dx = cx - i, dy = cy - j: sum f dx = cx S0 - S_i, sum f dx^2 = cx^2 S0 - 2 cx S_i + S_ii, ... as one branch-free
      // form  gt = +-own_t + p q S0 - (p Sb + q Sa)  with per-row selections of p, q in {0, 1, cx, cy}:
      //   row 0: own_t | 1: cx S0 - own_t | 2: cy S0 - own_t | 3: own_t + cx^2 S0 - 2 cx S1
      //   row 4: own_t + cx cy S0 - cx S2 - cy S1 | 5: own_t + cy^2 S0 - 2 cy S2
      const float p = (r_1 | r_3 | r_4) ? cx : (r_2 | r_5) ? cy : 0.f;
      const float q = r_3 ? cx : (r_4 | r_5) ? cy : 1.f;
      const float cross = (g8 >= 3) ? p * (r_3 ? S1 : S2) + q * (r_5 ? S2 : S1) : 0.f;
      const float gt = ((r_1 | r_2) ? -own_t : own_t) + (p * q) * S0 - cross;
      const float gw = (r_1 | r_2) ? p * V0 - own_w : own_w;
      if (g8 < 6 && n < cnt) {
        float* dst = moments + (size_t)gid * kG;
        atomicAdd(dst + g8, gt);
        atomicAdd(dst + 6 + g8, gw);
      }
    }
    cnt = 0;
  };

  float last_alpha = 0.f, last_r = 0.f, last_g = 0.f, last_b = 0.f, last_depth = 0.f;
  float acc_r = 0.f, acc_g = 0.f, acc_b = 0.f, acc_d = 0.f;

  // Back to front: batch `base` covers list positions [total-base-n, total-base), staged reversed
  // (slot k = position total-base-1-k) like backward.cu:519-531.
  auto stage = [&](int base, int buf) {
    const int n = min(kStage, total - base);
    if (tid < n) {
      const Splat* sp = splats + point_list[range.y - 1 - base - tid];
      cp_async16(&sm.a[buf][tid], &sp->a);
      cp_async16(&sm.b[buf][tid], &sp->b);
      cp_async16(&sm.c[buf][tid], &sp->c);
    }
    cp_async_commit();
  };
  if (total > 0) stage(0, 0);

  // The forward pass recorded, per 32 list positions of the tile and per sub-tile, which instances survive the exact cull
  // (BinState::hit): replayed here instead of evaluating the cull again.  A batch spans at most kStage / 32 + 1 words;
  // lane l holds the word of positions 32 (top - l) .. (top = word of the batch's first slot), loaded before the barrier.
  const uint32_t* const hit_tile = hit_in + hit_word(range.x, tile) * 8 + warp;

  for (int base = 0, buf = 0; base < total; base += kStage, buf ^= 1) {
    const int n = min(kStage, total - base);
    const int p_top = total - 1 - base;  // list position (0-based, front to back) of slot 0 of this batch
    uint32_t hit_words = 0;
    if (kCull) {
      const int w = (p_top >> 5) - lane;
      if (lane <= kStage / 32 && w >= 0) hit_words = __ldg(hit_tile + (size_t)w * 8);
    }
    cp_async_wait_all();
    __syncthreads();  // batch `base` is staged; every warp has finished reading the other buffer
    if (base + kStage < total) stage(base + kStage, buf ^ 1);

    const int first_pos = total - base;  // 1-based contributor id of slot 0
    if (first_pos - (n - 1) > warp_last) continue;  // the whole batch lies behind this warp's last contributor
    for (int c0 = 0; c0 < n; c0 += 32) {
      if (first_pos - c0 - 31 > warp_last && c0 + 32 <= n) continue;  // whole chunk behind the last contributor
      uint32_t s_chunk = s_base + (uint32_t)(buf * kStage + c0) * 16u;  // sm.a[buf][c0]
      asm volatile("" : "+r"(s_chunk));  // opaque: keep it in a register instead of rebuilding it per survivor
      uint32_t mask;
      {
        const int j = c0 + lane;
        mask = __ballot_sync(0xffffffffu, (j < n) && (first_pos - j <= warp_last));
        if (kCull) {
          // slot c0 + i is list position p_hi - i: bits p_hi - 31 .. p_hi of the recorded masks, reversed
          const int p_hi = p_top - c0, l1 = (p_top >> 5) - (p_hi >> 5);
          const uint32_t hi = __shfl_sync(0xffffffffu, hit_words, l1), lo = __shfl_sync(0xffffffffu, hit_words, l1 + 1);
          mask &= __brev(__funnelshift_rc(lo, hi, (p_hi & 31) + 1));
        }
      }
      while (mask) {
        const int bit = __ffs(mask) - 1;
        mask &= mask - 1;
        const int j = c0 + bit;
        const int contributor = first_pos - j;  // 1-based; reference compares (contributor-1) >= last (backward.cu:540-542)
        const uint32_t s_j = s_chunk + (uint32_t)bit * 16u;
        const float4 a = lds128<0>(s_j), b = lds128<kOffB>(s_j);
        const float dx = a.x - pxf, dy = a.y - pyf;
        const float power = -0.5f * (a.z * dx * dx + b.x * dy * dy) - a.w * dx * dy;
        const float G = expf(power);
        const float alpha = fminf(0.99f, b.y * G);
        const bool active = inside && (contributor <= last_contributor) && !(power > 0.0f) && !(alpha < 1.0f / 255.0f);

        if (!__any_sync(0xffffffffu, active)) continue;  // no pixel of this sub-tile blended the instance

        float tq = 0.f, wq = 0.f;
        if (active) {
          const float4 c = lds128<kOffC>(s_j);
          const float inv = rcp_approx(1.f - alpha);  // one reciprocal shared by the three divisions
          T = T * inv;                               // transmittance in front of this Gaussian (backward.cu:555)
          wq = alpha * T;                            // d(pixel channel)/d(colour), also d(pixel depth)/d(depth)

          // colour and depth blended behind this Gaussian (backward.cu:563-576, 617-620)
          acc_r = last_alpha * last_r + (1.f - last_alpha) * acc_r;
          acc_g = last_alpha * last_g + (1.f - last_alpha) * acc_g;
          acc_b = last_alpha * last_b + (1.f - last_alpha) * acc_b;
          acc_d = last_alpha * last_depth + (1.f - last_alpha) * acc_d;
          const float czx = b.z, cyz = b.w;
          const float depth = c.w - (czx * a.z + cyz * a.w) * dx - (czx * a.w + cyz * b.x) * dy;
          last_r = c.x; last_g = c.y; last_b = c.z; last_depth = depth;
          last_alpha = alpha;
          // dL/dalpha (colour) + dL/dalpha_d (depth; same alpha and transmittance, T_d == T bit for bit, DESIGN.md)
          const float dsum = ((c.x - acc_r) * dpr + (c.y - acc_g) * dpg + (c.z - acc_b) * dpb + (depth - acc_d) * dpd) * T -
                             bg_term * inv;
          tq = G * dsum;
        }
        {
          const uint32_t s_dst = s_slot + (uint32_t)cnt * (kRow * 4);
          sts32<0>(s_dst, tq);
          sts32<kOffW>(s_dst, wq);
        }
        if (lane == cnt) {
          m_cx = a.x - wx0f;
          m_cy = a.y - wy0f;
          m_id = point_list[range.y - 1 - base - j];
        }
        if (++cnt == kGrp) flush();
      }
    }
  }
  if (cnt > 0) flush();
}

// ------------------------------------------------------------------------------------------
// per-Gaussian backward (backward.cu:144-294 + 298-364 + 369-426 + 20-139 fused)
// ------------------------------------------------------------------------------------------
struct BwdArgs {
  int P, D, M;
  float tan_fovx, tan_fovy, focal_x, focal_y, scale_modifier;
  const float *means, *scales, *rots, *shs, *cov_pre, *view, *proj, *campos;
};

__device__ __forceinline__ F3 dnormv(F3 v, F3 dv) {  // gradient through v/|v| (auxiliary.h:113-124)
  const float sum2 = v.x * v.x + v.y * v.y + v.z * v.z;
  const float invsum32 = 1.0f / sqrtf(sum2 * sum2 * sum2);
  F3 r;
  r.x = ((+sum2 - v.x * v.x) * dv.x - v.y * v.x * dv.y - v.z * v.x * dv.z) * invsum32;
  r.y = (-v.x * v.y * dv.x + (sum2 - v.y * v.y) * dv.y - v.z * v.y * dv.z) * invsum32;
  r.z = (-v.x * v.z * dv.x - v.y * v.z * dv.y + (sum2 - v.z * v.z) * dv.z) * invsum32;
  return r;
}

__device__ __forceinline__ F3 sh_backward(int idx, const BwdArgs& a, uint8_t clamp_mask, F3 dL_dRGB,
                                          float* __restrict__ dL_dsh_out) {
  const F3 pos = {a.means[3 * idx], a.means[3 * idx + 1], a.means[3 * idx + 2]};
  const F3 cam = {a.campos[0], a.campos[1], a.campos[2]};
  const F3 dir_orig = pos - cam;
  const float len = sqrtf(dot3(dir_orig, dir_orig));
  const F3 dir = {dir_orig.x / len, dir_orig.y / len, dir_orig.z / len};
  const F3* sh = reinterpret_cast<const F3*>(a.shs) + (size_t)idx * a.M;
  F3* dL_dsh = reinterpret_cast<F3*>(dL_dsh_out) + (size_t)idx * a.M;

  dL_dRGB.x *= (clamp_mask & 1) ? 0.f : 1.f;
  dL_dRGB.y *= (clamp_mask & 2) ? 0.f : 1.f;
  dL_dRGB.z *= (clamp_mask & 4) ? 0.f : 1.f;

  F3 dRGBdx = {0, 0, 0}, dRGBdy = {0, 0, 0}, dRGBdz = {0, 0, 0};
  const float x = dir.x, y = dir.y, z = dir.z;
  dL_dsh[0] = kShC0 * dL_dRGB;
  if (a.D > 0) {
    dL_dsh[1] = (-kShC1 * y) * dL_dRGB;
    dL_dsh[2] = (kShC1 * z) * dL_dRGB;
    dL_dsh[3] = (-kShC1 * x) * dL_dRGB;
    dRGBdx = -kShC1 * sh[3];
    dRGBdy = -kShC1 * sh[1];
    dRGBdz = kShC1 * sh[2];
    if (a.D > 1) {
      const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
      dL_dsh[4] = (kShC2[0] * xy) * dL_dRGB;
      dL_dsh[5] = (kShC2[1] * yz) * dL_dRGB;
      dL_dsh[6] = (kShC2[2] * (2.f * zz - xx - yy)) * dL_dRGB;
      dL_dsh[7] = (kShC2[3] * xz) * dL_dRGB;
      dL_dsh[8] = (kShC2[4] * (xx - yy)) * dL_dRGB;
      dRGBdx = dRGBdx + (kShC2[0] * y * sh[4] + kShC2[2] * 2.f * -x * sh[6] + kShC2[3] * z * sh[7] + kShC2[4] * 2.f * x * sh[8]);
      dRGBdy = dRGBdy + (kShC2[0] * x * sh[4] + kShC2[1] * z * sh[5] + kShC2[2] * 2.f * -y * sh[6] + kShC2[4] * 2.f * -y * sh[8]);
      dRGBdz = dRGBdz + (kShC2[1] * y * sh[5] + kShC2[2] * 2.f * 2.f * z * sh[6] + kShC2[3] * x * sh[7]);
      if (a.D > 2) {
        dL_dsh[9] = (kShC3[0] * y * (3.f * xx - yy)) * dL_dRGB;
        dL_dsh[10] = (kShC3[1] * xy * z) * dL_dRGB;
        dL_dsh[11] = (kShC3[2] * y * (4.f * zz - xx - yy)) * dL_dRGB;
        dL_dsh[12] = (kShC3[3] * z * (2.f * zz - 3.f * xx - 3.f * yy)) * dL_dRGB;
        dL_dsh[13] = (kShC3[4] * x * (4.f * zz - xx - yy)) * dL_dRGB;
        dL_dsh[14] = (kShC3[5] * z * (xx - yy)) * dL_dRGB;
        dL_dsh[15] = (kShC3[6] * x * (xx - 3.f * yy)) * dL_dRGB;
        dRGBdx = dRGBdx + (kShC3[0] * sh[9] * 3.f * 2.f * xy + kShC3[1] * sh[10] * yz + kShC3[2] * sh[11] * -2.f * xy +
                           kShC3[3] * sh[12] * -3.f * 2.f * xz + kShC3[4] * sh[13] * (-3.f * xx + 4.f * zz - yy) +
                           kShC3[5] * sh[14] * 2.f * xz + kShC3[6] * sh[15] * 3.f * (xx - yy));
        dRGBdy = dRGBdy + (kShC3[0] * sh[9] * 3.f * (xx - yy) + kShC3[1] * sh[10] * xz +
                           kShC3[2] * sh[11] * (-3.f * yy + 4.f * zz - xx) + kShC3[3] * sh[12] * -3.f * 2.f * yz +
                           kShC3[4] * sh[13] * -2.f * xy + kShC3[5] * sh[14] * -2.f * yz + kShC3[6] * sh[15] * -3.f * 2.f * xy);
        dRGBdz = dRGBdz + (kShC3[1] * sh[10] * xy + kShC3[2] * sh[11] * 4.f * 2.f * yz +
                           kShC3[3] * sh[12] * 3.f * (2.f * zz - xx - yy) + kShC3[4] * sh[13] * 4.f * 2.f * xz +
                           kShC3[5] * sh[14] * (xx - yy));
      }
    }
  }
  // coefficients above the active degree get no gradient (the caller's buffer is uninitialised: write the zeros)
  for (int c = (a.D + 1) * (a.D + 1); c < a.M; c++) dL_dsh[c] = {0.f, 0.f, 0.f};
  const F3 dL_ddir = {dot3(dRGBdx, dL_dRGB), dot3(dRGBdy, dL_dRGB), dot3(dRGBdz, dL_dRGB)};
  return dnormv(dir_orig, dL_ddir);
}

// Clears rows [wbase, wbase + 32) of a row-major [P][k] float array with one warp: 128-bit stores when the block is 16-byte
// aligned (always, for 16-byte aligned arrays: the block starts 128 k bytes into the array), 32-bit coalesced stores otherwise.
__device__ __forceinline__ void zero_rows(float* __restrict__ out, int k, int wbase, int lane) {
  float* base = out + (size_t)wbase * k;
  if ((reinterpret_cast<uintptr_t>(base) & 15) == 0) {
    float4* b4 = reinterpret_cast<float4*>(base);
    for (int i = lane; i < 8 * k; i += 32) b4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  } else {
    for (int i = lane; i < 32 * k; i += 32) base[i] = 0.f;
  }
}

__global__ void __launch_bounds__(256)
gaussian_backward_kernel(BwdArgs a, const int32_t* __restrict__ radii, const uint8_t* __restrict__ clamped,
                         float* __restrict__ moments, const Splat* __restrict__ splats, int W, int H,
                         float* __restrict__ dL_dmean2D, float* __restrict__ dL_dcolors,
                         float* __restrict__ dL_dopacity, float* __restrict__ dL_dmeans3D,
                         float* __restrict__ dL_dcov3D, float* __restrict__ dL_dsh, float* __restrict__ dL_dscales,
                         float* __restrict__ dL_drots, float* __restrict__ xmom) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  // Every gradient row of an invisible Gaussian is exactly zero, and the kernel writes those zeros itself: the caller hands
  // over uninitialised memory and no P-sized fill launch precedes the backward (the reference zero-fills ten tensors,
  // rasterize_points.cu:158-167).  89 % of the rows are such rows, so a warp first clears the 32-row block of every output
  // with coalesced (128-bit where aligned) stores; the visible lanes then overwrite their own rows.
  const int lane = threadIdx.x & 31;
  const int wbase = idx - lane;
  const bool full = wbase + 32 <= a.P;  // warp-uniform; the last, partial warp takes the per-row path
  if (full) {
    zero_rows(dL_dmean2D, 3, wbase, lane);
    zero_rows(dL_dcolors, 3, wbase, lane);
    zero_rows(dL_dopacity, 1, wbase, lane);
    zero_rows(dL_dmeans3D, 3, wbase, lane);
    zero_rows(dL_dcov3D, 6, wbase, lane);
    if (dL_dsh) zero_rows(dL_dsh, 3 * a.M, wbase, lane);
    zero_rows(dL_dscales, 3, wbase, lane);
    zero_rows(dL_drots, 4, wbase, lane);
    __syncwarp();  // orders the block clear before the visible lanes' own stores
  }
  if (idx >= a.P) return;
  if (!(radii[idx] > 0)) {
    if (!full) {
#pragma unroll
      for (int i = 0; i < 3; i++) {
        dL_dmean2D[3 * (size_t)idx + i] = 0.f;
        dL_dcolors[3 * (size_t)idx + i] = 0.f;
        dL_dmeans3D[3 * (size_t)idx + i] = 0.f;
        dL_dscales[3 * (size_t)idx + i] = 0.f;
      }
      dL_dopacity[idx] = 0.f;
#pragma unroll
      for (int i = 0; i < 6; i++) dL_dcov3D[6 * (size_t)idx + i] = 0.f;
#pragma unroll
      for (int i = 0; i < 4; i++) dL_drots[4 * (size_t)idx + i] = 0.f;
      if (dL_dsh)
        for (int i = 0; i < 3 * a.M; i++) dL_dsh[(size_t)idx * 3 * a.M + i] = 0.f;
    }
    return;
  }
  // dL_dmean2D is [P][3]; the third component is never written by the reference either (stays zero)
  dL_dmean2D[3 * (size_t)idx + 2] = 0.f;

  const float3 mean = make_float3(a.means[3 * idx], a.means[3 * idx + 1], a.means[3 * idx + 2]);
  float cov3[6];
  float3 scale = make_float3(0, 0, 0);
  float4 q = make_float4(0, 0, 0, 1);
  if (a.cov_pre) {
#pragma unroll
    for (int i = 0; i < 6; i++) cov3[i] = a.cov_pre[6 * (size_t)idx + i];
  } else {
    if (a.scales) scale = make_float3(a.scales[3 * idx], a.scales[3 * idx + 1], a.scales[3 * idx + 2]);
    if (a.rots) q = reinterpret_cast<const float4*>(a.rots)[idx];
    cov3d_from_scale_rot(scale, a.scale_modifier, q, cov3);
  }
  // ---- render gradients from the moments (reference expressions: backward.cu:604-654) ----
  float4* mrow = reinterpret_cast<float4*>(moments) + 3 * (size_t)idx;
  const float4 m0 = mrow[0], m1 = mrow[1], m2 = mrow[2];
  mrow[0] = mrow[1] = mrow[2] = make_float4(0.f, 0.f, 0.f, 0.f);  // consumed: a second backward on the same state starts from zero
  if (xmom) {  // sharded run: this rank's accumulator row in the exchange segment (every peer has read it by now)
    float4* xr = reinterpret_cast<float4*>(xmom) + 3 * (size_t)idx;
    xr[0] = xr[1] = xr[2] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const Splat sp = splats[idx];
  const float cA = sp.a.z, cB = sp.a.w, cC = sp.b.x, opac = sp.b.y, czx = sp.b.z, cyz = sp.b.w;
  // u = opacity * t (backward.cu:606-612 multiply by con_o.w per pair; here once per Gaussian)
  const float tt = m0.x, ux = opac * m0.y, uy = opac * m0.z, uxx = opac * m0.w, uxy = opac * m1.x, uyy = opac * m1.y;
  const float v0 = m1.z, vx = m1.w, vy = m2.x;
  dL_dcolors[3 * (size_t)idx + 0] = m2.y;
  dL_dcolors[3 * (size_t)idx + 1] = m2.z;
  dL_dcolors[3 * (size_t)idx + 2] = m2.w;
  dL_dopacity[idx] = tt;
  const float g2x = (-cA * ux - cB * uy - (czx * cA + cyz * cB) * v0) * (0.5f * W);
  const float g2y = (-cC * uy - cB * ux - (czx * cB + cyz * cC) * v0) * (0.5f * H);
  dL_dmean2D[3 * (size_t)idx + 0] = g2x;
  dL_dmean2D[3 * (size_t)idx + 1] = g2y;
  const float dc_x = -0.5f * uxx - czx * vx;             // dL/dconic_xx
  const float dc_y = -0.5f * uxy - cyz * vx - czx * vy;  // dL/dconic_xy
  const float dc_z = -0.5f * uyy - cyz * vy;             // dL/dconic_yy
  const float dL_dcovzx = -cA * vx - cB * vy;
  const float dL_dcovyz = -cB * vx;  // the reference omits the conic_yy * dy term (backward.cu:616)
  const float dL_ddepth = v0;

  // ---- 2D covariance backward (backward.cu:144-294) ----
  const Ewa e = ewa_project(mean, a.focal_x, a.focal_y, a.tan_fovx, a.tan_fovy, cov3, a.view);
  const float limx = 1.3f * a.tan_fovx, limy = 1.3f * a.tan_fovy;
  const float x_grad_mul = (e.txtz < -limx || e.txtz > limx) ? 0.f : 1.f;
  const float y_grad_mul = (e.tytz < -limy || e.tytz > limy) ? 0.f : 1.f;
  const M3& T = e.T;
  const M3& V = e.Vrk;
  const M3& Wm = e.W;
  const float ca = e.cov.m[0][0] + 0.3f, cb = e.cov.m[0][1], cc = e.cov.m[1][1] + 0.3f;
  const float denom = ca * cc - cb * cb;
  float dL_da = 0, dL_db = 0, dL_dc = 0;
  const float denom2inv = 1.0f / ((denom * denom) + 0.0000001f);
  float dcov[6];
  if (denom2inv != 0) {
    dL_da = denom2inv * (-cc * cc * dc_x + 2 * cb * cc * dc_y + (denom - ca * cc) * dc_z);
    dL_dc = denom2inv * (-ca * ca * dc_z + 2 * ca * cb * dc_y + (denom - ca * cc) * dc_x);
    dL_db = denom2inv * 2 * (cb * cc * dc_x - (denom + 2 * cb * cb) * dc_y + ca * cb * dc_z);
    dcov[0] = (T.m[0][0] * T.m[0][0] * dL_da + T.m[0][0] * T.m[1][0] * dL_db + T.m[0][0] * T.m[2][0] * dL_dcovzx +
               T.m[1][0] * T.m[1][0] * dL_dc + T.m[1][0] * T.m[2][0] * dL_dcovyz);
    dcov[3] = (T.m[0][1] * T.m[0][1] * dL_da + T.m[0][1] * T.m[1][1] * dL_db + T.m[0][1] * T.m[2][1] * dL_dcovzx +
               T.m[1][1] * T.m[1][1] * dL_dc + T.m[1][1] * T.m[2][1] * dL_dcovyz);
    dcov[5] = (T.m[0][2] * T.m[0][2] * dL_da + T.m[0][2] * T.m[1][2] * dL_db + T.m[0][2] * T.m[2][2] * dL_dcovzx +
               T.m[1][2] * T.m[1][2] * dL_dc + T.m[1][2] * T.m[2][2] * dL_dcovyz);
    dcov[1] = 2 * T.m[0][0] * T.m[0][1] * dL_da + (T.m[0][0] * T.m[1][1] + T.m[0][1] * T.m[1][0]) * dL_db +
              (T.m[0][1] * T.m[2][0] + T.m[0][0] * T.m[2][1]) * dL_dcovzx +
              (T.m[1][1] * T.m[2][0] + T.m[1][0] * T.m[2][1]) * dL_dcovyz + 2 * T.m[1][0] * T.m[1][1] * dL_dc;
    dcov[2] = 2 * T.m[0][0] * T.m[0][2] * dL_da + (T.m[0][0] * T.m[1][2] + T.m[0][2] * T.m[1][0]) * dL_db +
              (T.m[0][2] * T.m[2][0] + T.m[0][0] * T.m[2][2]) * dL_dcovzx +
              (T.m[1][2] * T.m[2][0] + T.m[1][0] * T.m[2][2]) * dL_dcovyz + 2 * T.m[1][0] * T.m[1][2] * dL_dc;
    dcov[4] = 2 * T.m[0][2] * T.m[0][1] * dL_da + (T.m[0][1] * T.m[1][2] + T.m[0][2] * T.m[1][1]) * dL_db +
              (T.m[0][2] * T.m[2][1] + T.m[0][1] * T.m[2][2]) * dL_dcovzx +
              (T.m[1][2] * T.m[2][1] + T.m[1][1] * T.m[2][2]) * dL_dcovyz + 2 * T.m[1][1] * T.m[1][2] * dL_dc;
  } else {
#pragma unroll
    for (int i = 0; i < 6; i++) dcov[i] = 0.f;
  }
#pragma unroll
  for (int i = 0; i < 6; i++) dL_dcov3D[6 * (size_t)idx + i] = dcov[i];

  // gradient w.r.t. the upper 2x3 of T.  Reference quirk reproduced: the cov_yz terms of
  // dL_dT11 / dL_dT12 are dropped by stray ';' (backward.cu:263-268).
  const float dL_dT00 = 2 * (T.m[0][0] * V.m[0][0] + T.m[0][1] * V.m[0][1] + T.m[0][2] * V.m[0][2]) * dL_da +
                        (T.m[1][0] * V.m[0][0] + T.m[1][1] * V.m[0][1] + T.m[1][2] * V.m[0][2]) * dL_db +
                        (T.m[2][0] * V.m[0][0] + T.m[2][1] * V.m[0][1] + T.m[2][2] * V.m[0][2]) * dL_dcovzx;
  const float dL_dT01 = 2 * (T.m[0][0] * V.m[1][0] + T.m[0][1] * V.m[1][1] + T.m[0][2] * V.m[1][2]) * dL_da +
                        (T.m[1][0] * V.m[1][0] + T.m[1][1] * V.m[1][1] + T.m[1][2] * V.m[1][2]) * dL_db +
                        (T.m[2][0] * V.m[1][0] + T.m[2][1] * V.m[1][1] + T.m[2][2] * V.m[1][2]) * dL_dcovzx;
  const float dL_dT02 = 2 * (T.m[0][0] * V.m[2][0] + T.m[0][1] * V.m[2][1] + T.m[0][2] * V.m[2][2]) * dL_da +
                        (T.m[1][0] * V.m[2][0] + T.m[1][1] * V.m[2][1] + T.m[1][2] * V.m[2][2]) * dL_db +
                        (T.m[2][0] * V.m[2][0] + T.m[2][1] * V.m[2][1] + T.m[2][2] * V.m[2][2]) * dL_dcovzx;
  const float dL_dT10 = 2 * (T.m[1][0] * V.m[0][0] + T.m[1][1] * V.m[0][1] + T.m[1][2] * V.m[0][2]) * dL_dc +
                        (T.m[0][0] * V.m[0][0] + T.m[0][1] * V.m[0][1] + T.m[0][2] * V.m[0][2]) * dL_db +
                        (T.m[2][0] * V.m[0][0] + T.m[2][1] * V.m[0][1] + T.m[2][2] * V.m[0][2]) * dL_dcovyz;
  const float dL_dT11 = 2 * (T.m[1][0] * V.m[1][0] + T.m[1][1] * V.m[1][1] + T.m[1][2] * V.m[1][2]) * dL_dc +
                        (T.m[0][0] * V.m[1][0] + T.m[0][1] * V.m[1][1] + T.m[0][2] * V.m[1][2]) * dL_db;
  const float dL_dT12 = 2 * (T.m[1][0] * V.m[2][0] + T.m[1][1] * V.m[2][1] + T.m[1][2] * V.m[2][2]) * dL_dc +
                        (T.m[0][0] * V.m[2][0] + T.m[0][1] * V.m[2][1] + T.m[0][2] * V.m[2][2]) * dL_db;

  const float dL_dJ00 = Wm.m[0][0] * dL_dT00 + Wm.m[0][1] * dL_dT01 + Wm.m[0][2] * dL_dT02;
  const float dL_dJ02 = Wm.m[2][0] * dL_dT00 + Wm.m[2][1] * dL_dT01 + Wm.m[2][2] * dL_dT02;
  const float dL_dJ11 = Wm.m[1][0] * dL_dT10 + Wm.m[1][1] * dL_dT11 + Wm.m[1][2] * dL_dT12;
  const float dL_dJ12 = Wm.m[2][0] * dL_dT10 + Wm.m[2][1] * dL_dT11 + Wm.m[2][2] * dL_dT12;

  const float tz = 1.f / e.t.z, tz2 = tz * tz, tz3 = tz2 * tz;
  const float hx = a.focal_x, hy = a.focal_y;
  const float dL_dtx = x_grad_mul * -hx * tz2 * dL_dJ02;
  const float dL_dty = y_grad_mul * -hy * tz2 * dL_dJ12;
  const float dL_dtz = -hx * tz2 * dL_dJ00 - hy * tz2 * dL_dJ11 + (2 * hx * e.t.x) * tz3 * dL_dJ02 +
                       (2 * hy * e.t.y) * tz3 * dL_dJ12;
  const float* vm = a.view;
  F3 dmean = {vm[0] * dL_dtx + vm[1] * dL_dty + vm[2] * dL_dtz, vm[4] * dL_dtx + vm[5] * dL_dty + vm[6] * dL_dtz,
              vm[8] * dL_dtx + vm[9] * dL_dty + vm[10] * dL_dtz};

  // ---- depth and 2D-mean paths (backward.cu:393-417) ----
  const float* proj = a.proj;
  const float4 mh = xform_point_4x4(mean, proj);
  const float m_w = 1.0f / (mh.w + 0.0000001f);
  const float mul = vm[2] * mean.x + vm[6] * mean.y + vm[10] * mean.z + vm[14];
  dmean.x += dL_ddepth * (vm[2] - vm[3] * mul);
  dmean.y += dL_ddepth * (vm[6] - vm[7] * mul);
  dmean.z += dL_ddepth * (vm[10] - vm[11] * mul);
  const float mul1 = (proj[0] * mean.x + proj[4] * mean.y + proj[8] * mean.z + proj[12]) * m_w * m_w;
  const float mul2 = (proj[1] * mean.x + proj[5] * mean.y + proj[9] * mean.z + proj[13]) * m_w * m_w;
  dmean.x += (proj[0] * m_w - proj[3] * mul1) * g2x + (proj[1] * m_w - proj[3] * mul2) * g2y;
  dmean.y += (proj[4] * m_w - proj[7] * mul1) * g2x + (proj[5] * m_w - proj[7] * mul2) * g2y;
  dmean.z += (proj[8] * m_w - proj[11] * mul1) * g2x + (proj[9] * m_w - proj[11] * mul2) * g2y;

  // ---- SH path ----
  if (a.shs) {
    const F3 dRGB = {m2.y, m2.z, m2.w};
    const F3 dm = sh_backward(idx, a, clamped[idx], dRGB, dL_dsh);
    dmean = dmean + dm;
  }
  dL_dmeans3D[3 * (size_t)idx + 0] = dmean.x;
  dL_dmeans3D[3 * (size_t)idx + 1] = dmean.y;
  dL_dmeans3D[3 * (size_t)idx + 2] = dmean.z;

  // ---- scale / rotation (backward.cu:298-364; no quaternion-normalisation backward) ----
  if (!a.scales) {  // precomputed 3D covariance: no scale / rotation gradient (rows stay zero like the reference's)
    dL_dscales[3 * (size_t)idx + 0] = dL_dscales[3 * (size_t)idx + 1] = dL_dscales[3 * (size_t)idx + 2] = 0.f;
    reinterpret_cast<float4*>(dL_drots)[idx] = make_float4(0.f, 0.f, 0.f, 0.f);
  } else {
    const M3 R = quat_to_m3(q.x, q.y, q.z, q.w);
    const float3 s = make_float3(a.scale_modifier * scale.x, a.scale_modifier * scale.y, a.scale_modifier * scale.z);
    M3 S;
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
      for (int r = 0; r < 3; r++) S.m[c][r] = 0.f;
    S.m[0][0] = s.x; S.m[1][1] = s.y; S.m[2][2] = s.z;
    const M3 Mx = m3_mul(S, R);
    M3 dSig;
    dSig.m[0][0] = dcov[0];        dSig.m[0][1] = 0.5f * dcov[1]; dSig.m[0][2] = 0.5f * dcov[2];
    dSig.m[1][0] = 0.5f * dcov[1]; dSig.m[1][1] = dcov[3];        dSig.m[1][2] = 0.5f * dcov[4];
    dSig.m[2][0] = 0.5f * dcov[2]; dSig.m[2][1] = 0.5f * dcov[4]; dSig.m[2][2] = dcov[5];
    M3 M2;
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
      for (int r = 0; r < 3; r++) M2.m[c][r] = 2.0f * Mx.m[c][r];
    const M3 dL_dM = m3_mul(M2, dSig);
    const M3 Rt = m3_transpose(R);
    M3 dMt = m3_transpose(dL_dM);
    dL_dscales[3 * (size_t)idx + 0] = Rt.m[0][0] * dMt.m[0][0] + Rt.m[0][1] * dMt.m[0][1] + Rt.m[0][2] * dMt.m[0][2];
    dL_dscales[3 * (size_t)idx + 1] = Rt.m[1][0] * dMt.m[1][0] + Rt.m[1][1] * dMt.m[1][1] + Rt.m[1][2] * dMt.m[1][2];
    dL_dscales[3 * (size_t)idx + 2] = Rt.m[2][0] * dMt.m[2][0] + Rt.m[2][1] * dMt.m[2][1] + Rt.m[2][2] * dMt.m[2][2];
#pragma unroll
    for (int r = 0; r < 3; r++) {
      dMt.m[0][r] *= s.x;
      dMt.m[1][r] *= s.y;
      dMt.m[2][r] *= s.z;
    }
    const float x = q.x, y = q.y, z = q.z, w = q.w;
    float4 dq;
    dq.x = 2 * y * (dMt.m[1][0] + dMt.m[0][1]) + 2 * z * (dMt.m[2][0] + dMt.m[0][2]) + 2 * w * (dMt.m[1][2] - dMt.m[2][1]) -
           4 * x * (dMt.m[2][2] + dMt.m[1][1]);
    dq.y = 2 * x * (dMt.m[1][0] + dMt.m[0][1]) + 2 * w * (dMt.m[2][0] - dMt.m[0][2]) + 2 * z * (dMt.m[1][2] + dMt.m[2][1]) -
           4 * y * (dMt.m[2][2] + dMt.m[0][0]);
    dq.z = 2 * w * (dMt.m[0][1] - dMt.m[1][0]) + 2 * x * (dMt.m[2][0] + dMt.m[0][2]) + 2 * y * (dMt.m[1][2] + dMt.m[2][1]) -
           4 * z * (dMt.m[1][1] + dMt.m[0][0]);
    dq.w = 2 * z * (dMt.m[0][1] - dMt.m[1][0]) + 2 * y * (dMt.m[2][0] - dMt.m[0][2]) + 2 * x * (dMt.m[1][2] - dMt.m[2][1]);
    reinterpret_cast<float4*>(dL_drots)[idx] = dq;
  }
}

extern int g_render_cull;
// 0 (default): 256-entry staging, 80 registers, 3 CTAs/SM; 1: 128-entry staging, 64 registers, 4 CTAs/SM.  Measured (r2j, with
// the recorded hit masks): 176.2 vs 185.5 us at C3, 912 vs 930 us at C4 — fewer, longer batches win once the cull is gone.
// Same arithmetic per survivor; the switch exists for tools/bench_raster.py and the parity tests.
int g_bwd_variant = [] { const char* e = getenv("GSICP_BWD_VARIANT"); return e ? atoi(e) : 0; }();

// ---- multi-GPU: all-reduce of the render moments of the VISIBLE Gaussians (SURVEY §8e) ----
// Every rank preprocesses all Gaussians, so the set {radii > 0} and its index order are identical on all ranks; only the
// moments of those Gaussians are summed over the ranks, and the per-Gaussian backward then runs replicated.
//
// Sharded run through the exchange layer (comm.cuh): every rank's render_backward accumulated the moments of ITS tiles in
// its own segment.  The all-reduce over the ranks is two P2P passes over NVLink, both inside our kernels:
//   reduce-scatter: rank r adds, in rank order, the world's rows of the visible Gaussians of ITS slice of the table
//                   (slice = ceil(P / world) consecutive Gaussians) into the upper half of its own segment;
//   all-gather:     every rank copies each visible row from the rank that owns its slice into its private moments buffer.
// 2 (N-1)/N * 48 B per visible Gaussian cross the links per rank (a one-pass "read everything from everybody" is
// (N-1) * 48 B: 4x more at 8 ranks).  Every sum is formed once, by one rank, in rank order: identical bits everywhere.
// No compaction, no host-side count, no host-launched collective.
__global__ void moments_reduce_slice_kernel(CommView c, int P, int slice, const int32_t* __restrict__ radii, size_t red_off) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = c.rank * slice + k;
  if (k >= slice || i >= P || !(radii[i] > 0)) return;
  float4 acc[3] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
  for (int r = 0; r < c.world; r++) {
    const float4* src = reinterpret_cast<const float4*>(c.seg[r] + kCommHeapOff) + 3 * (size_t)i;
#pragma unroll
    for (int q = 0; q < 3; q++) {
      const float4 v = __ldcv(src + q);  // written by another GPU since the last read: never from a cached line
      acc[q].x += v.x; acc[q].y += v.y; acc[q].z += v.z; acc[q].w += v.w;
    }
  }
  float4* dst = reinterpret_cast<float4*>(c.seg[c.rank] + kCommHeapOff + red_off) + 3 * (size_t)k;
  dst[0] = acc[0]; dst[1] = acc[1]; dst[2] = acc[2];
}

__global__ void moments_gather_slices_kernel(CommView c, int P, int slice, const int32_t* __restrict__ radii, size_t red_off,
                                             float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P || !(radii[i] > 0)) return;
  const int owner = i / slice, k = i - owner * slice;
  const float4* src = reinterpret_cast<const float4*>(c.seg[owner] + kCommHeapOff + red_off) + 3 * (size_t)k;
  float4* dst = reinterpret_cast<float4*>(out) + 3 * (size_t)i;
  dst[0] = __ldcv(src); dst[1] = __ldcv(src + 1); dst[2] = __ldcv(src + 2);
}

gsicp_comm* g_raster_comm = nullptr;  // set by gsicp_raster_set_comm; also read by the forward pass (raster_forward.cu)
static std::mutex g_raster_comm_mu;   // serialises gsicp_raster_set_comm

// Where this rank's render moments accumulate: the exchange segment in a sharded run, else the geometry buffer.
float* raster_moment_accumulator(const gsicp_raster_args* args, float* geom_moments) {
  gsicp_comm* c = g_raster_comm;
  if (!c || c->world <= 1 || args->tile_shard_count <= 1) return geom_moments;
  return reinterpret_cast<float*>(c->local + kCommHeapOff);
}

}  // namespace gsicp

using namespace gsicp;

// render_backward_kernel needs more than the 48 KB of shared memory a kernel gets by default: opt in once per device.
static int ensure_bwd_smem_attr() {
  static std::mutex mu;
  static bool done[64] = {};
  int dev = 0;
  GSICP_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  if (dev < 0 || dev >= 64 || done[dev]) return GSICP_OK;
  GSICP_CUDA(cudaFuncSetAttribute(render_backward_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BwdSmem)));
  GSICP_CUDA(cudaFuncSetAttribute(render_backward_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BwdSmem)));
  GSICP_CUDA(cudaFuncSetAttribute((render_backward_kernel<true, 128, 4>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)sizeof(BwdSmemT<128>)));
  done[dev] = true;
  return GSICP_OK;
}

// The render moments live in the geometry buffer the forward pass allocated (GeomState::moments, zeroed for the visible
// Gaussians by preprocess): the backward needs no caller-provided work buffer any more.  Kept for ABI stability.
extern "C" int gsicp_raster_set_comm(gsicp_comm* comm) {
  if (comm && !comm->connected) {
    set_error("gsicp_raster_set_comm: the exchange group is not connected");
    return GSICP_ESTATE;
  }
  std::lock_guard<std::mutex> lock(g_raster_comm_mu);
  g_raster_comm = comm;
  return GSICP_OK;
}

extern "C" size_t gsicp_raster_backward_work_bytes(int P) { (void)P; return 0; }

extern "C" int gsicp_raster_backward(const gsicp_raster_args* args, int num_rendered, const int32_t* d_radii,
                                     const void* d_geom, const void* d_binning, const void* d_image,
                                     const float* d_dL_dout_color, const float* d_dL_dout_depth, float* d_dL_dmeans2D,
                                     float* d_dL_dcolors, float* d_dL_dopacity, float* d_dL_dmeans3D, float* d_dL_dcov3D,
                                     float* d_dL_dsh, float* d_dL_dscales, float* d_dL_drotations, void* d_work,
                                     void* stream_v) {
  (void)d_work;
  if (!args) return GSICP_EINVAL;
  const int P = args->P, W = args->width, H = args->height;
  if (P == 0) return GSICP_OK;
  if (!d_geom || !d_binning || !d_image || !d_radii) {
    set_error("gsicp_raster_backward: null state buffer");
    return GSICP_EINVAL;
  }
  if (!d_dL_dmeans2D || !d_dL_dcolors || !d_dL_dopacity || !d_dL_dmeans3D || !d_dL_dcov3D || !d_dL_dscales ||
      !d_dL_drotations || (args->M > 0 && args->d_shs && !d_dL_dsh)) {
    set_error("gsicp_raster_backward: null gradient buffer");
    return GSICP_EINVAL;
  }
  cudaStream_t stream = (cudaStream_t)stream_v;
  const int shard_count = args->tile_shard_count > 1 ? args->tile_shard_count : 1;
  const int shard_index = shard_count > 1 ? args->tile_shard_index : 0;
  const int tiles_x = (W + kTile - 1) / kTile, tiles_y = (H + kTile - 1) / kTile, tiles = tiles_x * tiles_y;
  GeomState geom = GeomState::from((char*)d_geom, P);
  BinState bin = BinState::from((char*)d_binning, num_rendered, (size_t)tiles);
  ImgState img = ImgState::from((char*)d_image, (size_t)W * H, tiles);
  gsicp_comm* comm = (g_raster_comm && g_raster_comm->world > 1 && shard_count > 1) ? g_raster_comm : nullptr;
  if (comm && (size_t)P * kG * sizeof(float) > comm->heap_bytes() / 2) {
    set_error("gsicp_raster_backward: exchange heap too small for %d Gaussians (needs %zu bytes in its lower half)", P,
              (size_t)P * kG * sizeof(float));
    return GSICP_ENOMEM;
  }
  float* work = raster_moment_accumulator(args, geom.moments);  // [P][12]

  if (num_rendered > 0) {
    if (int e = ensure_bwd_smem_attr()) return e;
    ProfScope ps(kProfRenderBwd, stream);
    if (!g_render_cull) {  // test hook: no sub-tile culling
      GSICP_LAUNCH(render_backward_kernel<false>, tiles, kTilePixels, sizeof(BwdSmem), stream, img.tile_order, img.ranges, bin.point_list,
                   W, H, tiles_x, args->d_background, geom.splats, img.final_T, img.n_contrib, d_dL_dout_color, d_dL_dout_depth,
                   work, bin.hit, shard_count, shard_index);
    } else if (g_bwd_variant == 1) {
      GSICP_LAUNCH((render_backward_kernel<true, 128, 4>), tiles, kTilePixels, sizeof(BwdSmemT<128>), stream, img.tile_order, img.ranges,
                   bin.point_list, W, H, tiles_x, args->d_background, geom.splats, img.final_T, img.n_contrib, d_dL_dout_color,
                   d_dL_dout_depth, work, bin.hit, shard_count, shard_index);
    } else {
      GSICP_LAUNCH(render_backward_kernel<true>, tiles, kTilePixels, sizeof(BwdSmem), stream, img.tile_order, img.ranges, bin.point_list,
                   W, H, tiles_x, args->d_background, geom.splats, img.final_T, img.n_contrib, d_dL_dout_color, d_dL_dout_depth,
                   work, bin.hit, shard_count, shard_index);
    }
    if (args->debug) GSICP_CUDA(cudaStreamSynchronize(stream));
  }

  float* xmom = nullptr;
  if (comm) {
    // exchange: barrier (all ranks have finished their render_backward) -> reduce own slice -> barrier (every slice is
    // reduced; nobody reads a peer's accumulator any more, so gaussian_backward may clear it) -> gather the slices.  The
    // reduced slices are overwritten only after the first barrier of the NEXT exchange, which every rank reaches after its
    // gather in stream order: no third barrier.
    const int slice = (P + comm->world - 1) / comm->world;
    const size_t red_off = (comm->heap_bytes() / 2) & ~size_t(255);
    ProfScope ps_x(kProfExchange, stream);
    if (int e = comm_stream_barrier(comm, stream)) return e;
    GSICP_LAUNCH(moments_reduce_slice_kernel, (slice + 255) / 256, 256, 0, stream, comm->view(), P, slice, d_radii, red_off);
    if (int e = comm_stream_barrier(comm, stream)) return e;
    GSICP_LAUNCH(moments_gather_slices_kernel, (P + 255) / 256, 256, 0, stream, comm->view(), P, slice, d_radii, red_off, geom.moments);
    xmom = work;
    work = geom.moments;
  }

  BwdArgs ba;
  ba.P = P; ba.D = args->D; ba.M = args->M;
  ba.tan_fovx = args->tan_fovx; ba.tan_fovy = args->tan_fovy;
  ba.focal_y = H / (2.0f * args->tan_fovy);
  ba.focal_x = W / (2.0f * args->tan_fovx);
  ba.scale_modifier = args->scale_modifier;
  ba.means = args->d_means3D; ba.scales = args->d_scales; ba.rots = args->d_rotations;
  ba.shs = args->d_shs; ba.cov_pre = args->d_cov3D_precomp; ba.view = args->d_viewmatrix; ba.proj = args->d_projmatrix;
  ba.campos = args->d_campos;
  ProfScope ps_gb(kProfGaussBwd, stream);
  GSICP_LAUNCH(gaussian_backward_kernel, (P + 255) / 256, 256, 0, stream, ba, d_radii, geom.clamped, work, geom.splats, W, H,
               d_dL_dmeans2D, d_dL_dcolors, d_dL_dopacity, d_dL_dmeans3D, d_dL_dcov3D, d_dL_dsh, d_dL_dscales, d_dL_drotations, xmom);
  if (args->debug) GSICP_CUDA(cudaStreamSynchronize(stream));
  GSICP_CUDA(cudaGetLastError());
  return GSICP_OK;
}

extern "C" void gsicp_test_set_bwd_variant(int v) { gsicp::g_bwd_variant = v; }
