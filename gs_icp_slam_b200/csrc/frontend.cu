// frontend.cu — the tracker's per-frame front-end on the device (SURVEY.md §8f row N1).
//
// Replaces the torch-CPU / numpy code around pygicp in mp_Tracker.py:
//   gsicp_frontend_cloud      set_downsample_filter + downsample_and_make_pointcloud2 (mp_Tracker.py:394-413, 415-431):
//                             pick every `step`-th pixel, z = depth / depth_scale, drop z == 0 (raster order kept), x = x_pre z,
//                             y = y_pre z, colours / 255, trackable = z <= depth_trunc -> the 1-based filter slots pygicp takes
//                             (mp_Tracker.py:159-161): one scan + one kernel, outputs stay on the device and feed
//                             gsicp_gicp_set_input_source_device / gsicp_gicp_set_source_filter_device directly.
//   gsicp_frontend_keyframe   the keyframe branch (mp_Tracker.py:229, 256-274): points to the world frame
//                             (R p - R T with the INVERSE pose's R, T as the script forms them), q_cam (x) rots for every
//                             point (quaternion_multiply, :385-392), and eliminate_overlapped2 (:374-380): the trackable
//                             slots whose squared NN distance exceeds the threshold, compacted.
#include <mutex>
#include "host_common.h"
#include "scan.cuh"

namespace gsicp {

struct CloudArgs {
  int W, H, step, rows, cols;  // rows = H / step + 1, cols = ceil(W / step)
  float fx, fy, cx, cy, depth_scale, depth_trunc;
  const uint16_t* depth;
  const uint8_t* rgb;  // [H][W][3] as the caller holds it
};

__device__ __forceinline__ int sample_pixel(const CloudArgs& a, int s) {
  const int r = s / a.cols, c = s % a.cols;
  const int v = (r == 0) ? 0 : (a.step * r - 1);  // h_val = step * arange - 1, h_val[0] = 0 (mp_Tracker.py:397-399)
  const int u = c * a.step;
  return (v < a.H) ? v * a.W + u : -1;
}

struct NonZeroDepth {
  CloudArgs a;
  __host__ __device__ int operator()(int s) const {
#ifdef __CUDA_ARCH__
    const int p = sample_pixel(a, s);
    return (p >= 0 && a.depth[p] != 0) ? 1 : 0;
#else
    return 0;
#endif
  }
};

__global__ void __launch_bounds__(256)
cloud_kernel(CloudArgs a, int n_samples, const int* __restrict__ excl, float* __restrict__ points, float* __restrict__ colors,
             float* __restrict__ zvals, int32_t* __restrict__ filter, unsigned int* __restrict__ trk_counter) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_samples) return;
  const int p = sample_pixel(a, s);
  if (p < 0) return;
  const uint16_t d = a.depth[p];
  if (d == 0) return;
  const int o = excl[s];
  const float z = __fdiv_rn((float)d, a.depth_scale);
  const int v = p / a.W, u = p % a.W;
  const float xp = __fdiv_rn((float)u - a.cx, a.fx), yp = __fdiv_rn((float)v - a.cy, a.fy);
  points[3 * (size_t)o + 0] = __fmul_rn(xp, z);
  points[3 * (size_t)o + 1] = __fmul_rn(yp, z);
  points[3 * (size_t)o + 2] = z;
  colors[3 * (size_t)o + 0] = __fdiv_rn((float)a.rgb[3 * (size_t)p + 0], 255.f);
  colors[3 * (size_t)o + 1] = __fdiv_rn((float)a.rgb[3 * (size_t)p + 1], 255.f);
  colors[3 * (size_t)o + 2] = __fdiv_rn((float)a.rgb[3 * (size_t)p + 2], 255.f);
  zvals[o] = z;
  filter[o] = (z <= a.depth_trunc) ? 1 : 0;  // turned into 1-based slots by the second scan
  (void)trk_counter;
}

struct FlagAt {
  const int32_t* f;
  __host__ __device__ int operator()(int i) const { return f[i] != 0 ? 1 : 0; }
};

// filter[i] = 0 or (rank among the trackable points) + 1; trackable[j] = i for the j-th trackable point
__global__ void __launch_bounds__(256)
slots_kernel(int n, const int* __restrict__ excl, int32_t* __restrict__ filter, int32_t* __restrict__ trackable,
             unsigned long long* host_map, unsigned long long seq, int n_points_slot) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int on = filter[i] != 0;
  if (on) {
    filter[i] = excl[i] + 1;
    trackable[excl[i]] = i;
  }
  if (i == n - 1 && host_map) {
    host_map[n_points_slot] = (unsigned long long)(excl[i] + on);
    __threadfence_system();
    host_map[3] = seq;
  }
}

__global__ void publish_count_kernel(int n_samples, const int* __restrict__ excl, CloudArgs a, unsigned long long* host_map,
                                     unsigned long long seq) {
  const int s = n_samples - 1;
  const int p = sample_pixel(a, s);
  host_map[0] = (unsigned long long)(excl[s] + ((p >= 0 && a.depth[p] != 0) ? 1 : 0));
  __threadfence_system();
  host_map[2] = seq;
}

// ---- keyframe branch -------------------------------------------------------------------------------------------------
struct KeyframeArgs {
  int n;
  float R[9], T[3];  // as mp_Tracker forms them from inv(pose): R = inv(pose)[:3,:3]^T, T = inv(pose)[:3,3]
  float q[4];        // scipy Rotation.from_matrix(R).as_quat(): x y z w
};

__global__ void __launch_bounds__(256)
keyframe_kernel(KeyframeArgs a, const float* __restrict__ pts_cam, const float* __restrict__ rots, float* __restrict__ pts_world,
                float* __restrict__ rots_world) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const float x = pts_cam[3 * (size_t)i], y = pts_cam[3 * (size_t)i + 1], z = pts_cam[3 * (size_t)i + 2];
  // points = (R p) - (R T)   (mp_Tracker.py:229)
#pragma unroll
  for (int r = 0; r < 3; r++) {
    const float rp = a.R[3 * r] * x + a.R[3 * r + 1] * y + a.R[3 * r + 2] * z;
    const float rt = a.R[3 * r] * a.T[0] + a.R[3 * r + 1] * a.T[1] + a.R[3 * r + 2] * a.T[2];
    pts_world[3 * (size_t)i + r] = rp - rt;
  }
  if (rots) {  // q1 * Q2, both (x, y, z, w) (mp_Tracker.py:385-392)
    const float4 Q = reinterpret_cast<const float4*>(rots)[i];
    const float x0 = a.q[0], y0 = a.q[1], z0 = a.q[2], w0 = a.q[3];
    float4 o;
    o.x = w0 * Q.x + x0 * Q.w + y0 * Q.z - z0 * Q.y;
    o.y = w0 * Q.y + y0 * Q.w + z0 * Q.x - x0 * Q.z;
    o.z = w0 * Q.z + z0 * Q.w + x0 * Q.y - y0 * Q.x;
    o.w = w0 * Q.w - x0 * Q.x - y0 * Q.y - z0 * Q.z;
    reinterpret_cast<float4*>(rots_world)[i] = o;
  }
}

struct FarFlag {
  const float* d2;
  float th;
  __host__ __device__ int operator()(int i) const { return d2[i] > th ? 1 : 0; }
};

__global__ void __launch_bounds__(256)
keep_far_kernel(int n_trk, FarFlag f, const int* __restrict__ excl, const int32_t* __restrict__ trackable, int32_t* __restrict__ out,
                unsigned long long* host_map, unsigned long long seq) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_trk) return;
  const int on = f(j);
  if (on) out[excl[j]] = trackable[j];  // trackable_filter[not_overlapped] (mp_Tracker.py:268-269)
  if (j == n_trk - 1 && host_map) {
    host_map[0] = (unsigned long long)(excl[j] + on);
    __threadfence_system();
    host_map[2] = seq;
  }
}

struct FrontScratch {
  std::mutex mu;
  Scratch excl, cub_tmp;
  HostMailbox box;  // [0] point / kept count, [1] trackable count, [2] and [3] their sequence words
};
static FrontScratch g_front;

}  // namespace gsicp

using namespace gsicp;

extern "C" int gsicp_frontend_max_points(int W, int H, int step) {
  if (W <= 0 || H <= 0 || step <= 0) return GSICP_EINVAL;
  return (H / step + 1) * ((W + step - 1) / step);
}

extern "C" int gsicp_frontend_cloud(const uint16_t* d_depth, const uint8_t* d_rgb, int W, int H, int step, float fx, float fy,
                                    float cx, float cy, float depth_scale, float depth_trunc, float* d_points,
                                    float* d_colors, float* d_z, int32_t* d_filter, int32_t* d_trackable, int* n_points,
                                    int* n_trackable, void* stream_v) {
  if (!d_depth || !d_rgb || !d_points || !d_colors || !d_z || !d_filter || !d_trackable || !n_points || !n_trackable || W <= 0 ||
      H <= 0 || step <= 0) {
    set_error("gsicp_frontend_cloud: bad arguments");
    return GSICP_EINVAL;
  }
  cudaStream_t stream = (cudaStream_t)stream_v;
  std::lock_guard<std::mutex> lock(g_front.mu);
  HostMailbox& box = g_front.box;
  if (int e = box.ensure(4 * sizeof(unsigned long long))) return e;
  CloudArgs a;
  a.W = W; a.H = H; a.step = step; a.rows = H / step + 1; a.cols = (W + step - 1) / step;
  a.fx = fx; a.fy = fy; a.cx = cx; a.cy = cy; a.depth_scale = depth_scale; a.depth_trunc = depth_trunc;
  a.depth = d_depth; a.rgb = d_rgb;
  const int ns = a.rows * a.cols;
  if (int e = flag_exclusive_scan<int>(ns, NonZeroDepth{a}, g_front.excl, g_front.cub_tmp, stream)) return e;
  const unsigned long long seq = ++box.seq;
  GSICP_LAUNCH(cloud_kernel, (ns + 255) / 256, 256, 0, stream, a, ns, g_front.excl.as<int>(), d_points, d_colors, d_z, d_filter,
               (unsigned int*)nullptr);
  GSICP_LAUNCH(publish_count_kernel, 1, 1, 0, stream, ns, g_front.excl.as<int>(), a, box.dev, seq);
  GSICP_CUDA(cudaGetLastError());
  if (int e = box.wait(2, seq, stream, "front-end point count")) return e;
  const int n = (int)box.host[0];
  *n_points = n;
  *n_trackable = 0;
  if (n == 0) return GSICP_OK;
  if (int e = flag_exclusive_scan<int>(n, FlagAt{d_filter}, g_front.excl, g_front.cub_tmp, stream)) return e;
  GSICP_LAUNCH(slots_kernel, (n + 255) / 256, 256, 0, stream, n, g_front.excl.as<int>(), d_filter, d_trackable, box.dev, seq, 1);
  GSICP_CUDA(cudaGetLastError());
  if (int e = box.wait(3, seq, stream, "front-end trackable count")) return e;
  *n_trackable = (int)box.host[1];
  return GSICP_OK;
}

extern "C" int gsicp_frontend_keyframe(int n, const float* d_points_cam, const float* d_rots, const float R[9], const float T[3],
                                       const float q_xyzw[4], float* d_points_world, float* d_rots_world, void* stream_v) {
  if (n < 0 || (n > 0 && (!d_points_cam || !d_points_world || !R || !T)) || (d_rots && (!q_xyzw || !d_rots_world))) {
    set_error("gsicp_frontend_keyframe: bad arguments");
    return GSICP_EINVAL;
  }
  if (n == 0) return GSICP_OK;
  KeyframeArgs a;
  a.n = n;
  for (int i = 0; i < 9; i++) a.R[i] = R[i];
  for (int i = 0; i < 3; i++) a.T[i] = T[i];
  for (int i = 0; i < 4; i++) a.q[i] = q_xyzw ? q_xyzw[i] : 0.f;
  GSICP_LAUNCH(keyframe_kernel, (n + 255) / 256, 256, 0, (cudaStream_t)stream_v, a, d_points_cam, d_rots, d_points_world, d_rots_world);
  GSICP_CUDA(cudaGetLastError());
  return GSICP_OK;
}

extern "C" int gsicp_frontend_not_overlapped(int n_trackable, const float* d_sq_dist, float threshold, const int32_t* d_trackable,
                                             int32_t* d_out, int* n_out, void* stream_v) {
  if (n_trackable < 0 || !n_out || (n_trackable > 0 && (!d_sq_dist || !d_trackable || !d_out))) {
    set_error("gsicp_frontend_not_overlapped: bad arguments");
    return GSICP_EINVAL;
  }
  *n_out = 0;
  if (n_trackable == 0) return GSICP_OK;
  cudaStream_t stream = (cudaStream_t)stream_v;
  std::lock_guard<std::mutex> lock(g_front.mu);
  HostMailbox& box = g_front.box;
  if (int e = box.ensure(4 * sizeof(unsigned long long))) return e;
  const FarFlag f{d_sq_dist, threshold};
  if (int e = flag_exclusive_scan<int>(n_trackable, f, g_front.excl, g_front.cub_tmp, stream)) return e;
  const unsigned long long seq = ++box.seq;
  GSICP_LAUNCH(keep_far_kernel, (n_trackable + 255) / 256, 256, 0, stream, n_trackable, f, g_front.excl.as<int>(), d_trackable, d_out,
               box.dev, seq);
  GSICP_CUDA(cudaGetLastError());
  if (int e = box.wait(2, seq, stream, "front-end kept count")) return e;
  *n_out = (int)box.host[0];
  return GSICP_OK;
}
