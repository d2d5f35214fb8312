// map_table.cu — the mapper's Gaussian-table bookkeeping on the device (SURVEY.md §8f row N3).
//
// Replaces, for the six parameter groups of scene/gaussian_model.py (xyz, f_dc, f_rest, opacity, scaling, rotation):
//   gsicp_adam_step        torch.optim.Adam(l, lr=0.0, eps=1e-15).step() (gaussian_model.py:214-225, mp_Mapper.py:248):
//                          ONE launch updates every group (the foreach implementation issues ~10 launches per step, the
//                          per-tensor one ~10 per GROUP), same arithmetic: exp_avg.lerp_(g, 1-b1); exp_avg_sq = b2 v + (1-b2) g g;
//                          p -= (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps)
//   gsicp_table_compact    prune_points / _prune_optimizer (gaussian_model.py:409-446): boolean-mask row selection of any number
//                          of row-major arrays (parameters, both Adam moments, gradient accumulators, masks) that share the mask:
//                          one scan + one scatter launch instead of one index kernel per tensor (~25 tensors)
//   gsicp_trackable_target get_trackable_gaussians_tensor (gaussian_model.py:205-215): opacity filter AND trackable mask ->
//                          compacted (xyz, normalised rotation, exp(scaling)) written straight into device buffers that
//                          FastGICP.set_input_target / set_target_covariances_fromqs take without leaving the GPU (the
//                          reference goes GPU -> CPU -> shared memory -> numpy -> pybind -> kd-tree at every tracking keyframe)
#include <mutex>
#include "host_common.h"
#include "scan.cuh"

namespace gsicp {

constexpr int kAdamMaxTensors = 8;
struct AdamTensors {
  int n;
  float* p[kAdamMaxTensors];
  const float* g[kAdamMaxTensors];
  float* m[kAdamMaxTensors];
  float* v[kAdamMaxTensors];
  unsigned long long end[kAdamMaxTensors];  // cumulative element counts
  float step_size[kAdamMaxTensors];         // lr / (1 - beta1^step)
};

__global__ void __launch_bounds__(256)
adam_kernel(AdamTensors t, unsigned long long total, float w1, float beta2, float w2, float bc2_sqrt_inv, float eps) {
  for (unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (unsigned long long)gridDim.x * blockDim.x) {
    int k = 0;
#pragma unroll
    for (int j = 0; j < kAdamMaxTensors - 1; j++)
      if (j < t.n - 1 && idx >= t.end[j]) k = j + 1;
    const unsigned long long i = idx - (k > 0 ? t.end[k - 1] : 0ull);
    const float g = t.g[k][i];
    float m = t.m[k][i], v = t.v[k][i];
    // w1 = float(1 - beta1), w2 = float(1 - beta2) are formed in double on the host and rounded once, as PyTorch passes them
    m = m + w1 * (g - m);                          // exp_avg.lerp_(grad, 1 - beta1)
    v = v * beta2 + w2 * g * g;                    // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
    const float denom = sqrtf(v) * bc2_sqrt_inv + eps;
    t.p[k][i] = t.p[k][i] - t.step_size[k] * (m / denom);
    t.m[k][i] = m;
    t.v[k][i] = v;
  }
}

// ---- row compaction -------------------------------------------------------------------------------------------------
constexpr int kCompactMaxArrays = 40;
struct CompactArrays {
  int n;
  const char* src[kCompactMaxArrays];
  char* dst[kCompactMaxArrays];
  int row_bytes[kCompactMaxArrays];  // multiples of 4 except byte-sized rows (masks)
};
struct KeepFlag {
  const uint8_t* keep;
  __host__ __device__ int operator()(int i) const { return keep[i] ? 1 : 0; }
};

__global__ void __launch_bounds__(256)
compact_rows_kernel(int rows, const uint8_t* __restrict__ keep, const int* __restrict__ excl, CompactArrays a,
                    unsigned long long* host_count, unsigned long long seq) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == rows - 1 && host_count) {
    host_count[0] = (unsigned long long)(excl[i] + (keep[i] ? 1 : 0));
    __threadfence_system();
    host_count[1] = seq;
  }
  if (i >= rows || !keep[i]) return;
  const size_t d = (size_t)excl[i];
  for (int k = 0; k < a.n; k++) {
    const int rb = a.row_bytes[k];
    const char* s = a.src[k] + (size_t)i * rb;
    char* o = a.dst[k] + d * rb;
    if ((rb & 3) == 0) {
      for (int b = 0; b < rb; b += 4) *reinterpret_cast<uint32_t*>(o + b) = *reinterpret_cast<const uint32_t*>(s + b);
    } else {
      for (int b = 0; b < rb; b++) o[b] = s[b];
    }
  }
}

// ---- trackable target -------------------------------------------------------------------------------------------------
struct TrackFlag {
  const float* opacity_raw;
  const uint8_t* trackable;
  float th;
  __host__ __device__ int operator()(int i) const {
    const float o = 1.0f / (1.0f + expf(-opacity_raw[i]));  // torch.sigmoid
    return (trackable[i] && o > th) ? 1 : 0;
  }
};

__global__ void __launch_bounds__(256)
trackable_target_kernel(int P, TrackFlag f, const int* __restrict__ excl, const float* __restrict__ xyz,
                        const float* __restrict__ rot_raw, const float* __restrict__ scale_raw, float* __restrict__ out_xyz,
                        float* __restrict__ out_rot, float* __restrict__ out_scale, unsigned long long* host_count,
                        unsigned long long seq) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  const int keep = f(i);
  if (i == P - 1 && host_count) {
    host_count[0] = (unsigned long long)(excl[i] + keep);
    __threadfence_system();
    host_count[1] = seq;
  }
  if (!keep) return;
  const size_t d = (size_t)excl[i];
  out_xyz[3 * d + 0] = xyz[3 * (size_t)i];
  out_xyz[3 * d + 1] = xyz[3 * (size_t)i + 1];
  out_xyz[3 * d + 2] = xyz[3 * (size_t)i + 2];
  const float4 q = reinterpret_cast<const float4*>(rot_raw)[i];
  const float nrm = fmaxf(sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w), 1e-12f);  // torch.nn.functional.normalize
  reinterpret_cast<float4*>(out_rot)[d] = make_float4(q.x / nrm, q.y / nrm, q.z / nrm, q.w / nrm);
  out_scale[3 * d + 0] = expf(scale_raw[3 * (size_t)i]);  // scaling_activation = torch.exp
  out_scale[3 * d + 1] = expf(scale_raw[3 * (size_t)i + 1]);
  out_scale[3 * d + 2] = expf(scale_raw[3 * (size_t)i + 2]);
}

struct TableScratch {
  std::mutex mu;
  Scratch excl, cub_tmp;
  HostMailbox box;  // [0] row count, [1] sequence word
};
static TableScratch g_tab;

}  // namespace gsicp

using namespace gsicp;

extern "C" int gsicp_adam_step(int n_tensors, float* const* d_params, const float* const* d_grads, float* const* d_exp_avg,
                               float* const* d_exp_avg_sq, const size_t* counts, const float* lrs, int step, double beta1,
                               double beta2, double eps, void* stream_v) {
  if (n_tensors < 0 || n_tensors > kAdamMaxTensors || step < 1) {
    set_error("gsicp_adam_step: %d tensors (max %d), step %d", n_tensors, kAdamMaxTensors, step);
    return GSICP_EINVAL;
  }
  AdamTensors t;
  t.n = 0;
  unsigned long long total = 0;
  const double bc1 = 1.0 - std::pow(beta1, (double)step);
  const double bc2_sqrt = std::sqrt(1.0 - std::pow(beta2, (double)step));
  for (int k = 0; k < n_tensors; k++) {
    if (counts[k] == 0) continue;
    if (!d_params[k] || !d_grads[k] || !d_exp_avg[k] || !d_exp_avg_sq[k]) {
      set_error("gsicp_adam_step: null buffer in tensor %d", k);
      return GSICP_EINVAL;
    }
    const int j = t.n++;
    t.p[j] = d_params[k]; t.g[j] = d_grads[k]; t.m[j] = d_exp_avg[k]; t.v[j] = d_exp_avg_sq[k];
    total += counts[k];
    t.end[j] = total;
    t.step_size[j] = (float)((double)lrs[k] / bc1);
  }
  if (total == 0) return GSICP_OK;
  const int blocks = (int)std::min<unsigned long long>((total + 255) / 256, 148ull * 16);
  GSICP_LAUNCH(adam_kernel, blocks, 256, 0, (cudaStream_t)stream_v, t, total, (float)(1.0 - beta1), (float)beta2,
               (float)(1.0 - beta2), (float)(1.0 / bc2_sqrt), (float)eps);
  GSICP_CUDA(cudaGetLastError());
  return GSICP_OK;
}

extern "C" long long gsicp_table_compact(int rows, const uint8_t* d_keep, int n_arrays, const void* const* d_src,
                                         void* const* d_dst, const int* row_bytes, void* stream_v) {
  if (rows < 0 || n_arrays < 0 || n_arrays > kCompactMaxArrays || (rows > 0 && !d_keep)) {
    set_error("gsicp_table_compact: bad arguments (%d rows, %d arrays, max %d)", rows, n_arrays, kCompactMaxArrays);
    return GSICP_EINVAL;
  }
  if (rows == 0) return 0;
  cudaStream_t stream = (cudaStream_t)stream_v;
  std::lock_guard<std::mutex> lock(g_tab.mu);
  HostMailbox& box = g_tab.box;
  if (int e = box.ensure(2 * sizeof(unsigned long long))) return e;
  if (int e = flag_exclusive_scan<int>(rows, KeepFlag{d_keep}, g_tab.excl, g_tab.cub_tmp, stream)) return e;
  CompactArrays a;
  a.n = n_arrays;
  for (int k = 0; k < n_arrays; k++) {
    if (!d_src[k] || !d_dst[k] || row_bytes[k] <= 0) {
      set_error("gsicp_table_compact: bad array %d", k);
      return GSICP_EINVAL;
    }
    a.src[k] = (const char*)d_src[k];
    a.dst[k] = (char*)d_dst[k];
    a.row_bytes[k] = row_bytes[k];
  }
  const unsigned long long seq = ++box.seq;
  GSICP_LAUNCH(compact_rows_kernel, (rows + 255) / 256, 256, 0, stream, rows, d_keep, g_tab.excl.as<int>(), a, box.dev, seq);
  GSICP_CUDA(cudaGetLastError());
  if (int e = box.wait(1, seq, stream, "compacted row count")) return e;
  return (long long)box.host[0];
}

extern "C" long long gsicp_trackable_target(int P, const float* d_xyz, const float* d_rotation_raw, const float* d_scaling_raw,
                                            const float* d_opacity_raw, const uint8_t* d_trackable, float opacity_th,
                                            float* d_out_xyz, float* d_out_rot, float* d_out_scale, void* stream_v) {
  if (P < 0) return GSICP_EINVAL;
  if (P == 0) return 0;
  if (!d_xyz || !d_rotation_raw || !d_scaling_raw || !d_opacity_raw || !d_trackable || !d_out_xyz || !d_out_rot || !d_out_scale) {
    set_error("gsicp_trackable_target: null buffer");
    return GSICP_EINVAL;
  }
  cudaStream_t stream = (cudaStream_t)stream_v;
  std::lock_guard<std::mutex> lock(g_tab.mu);
  HostMailbox& box = g_tab.box;
  if (int e = box.ensure(2 * sizeof(unsigned long long))) return e;
  const TrackFlag f{d_opacity_raw, d_trackable, opacity_th};
  if (int e = flag_exclusive_scan<int>(P, f, g_tab.excl, g_tab.cub_tmp, stream)) return e;
  const unsigned long long seq = ++box.seq;
  GSICP_LAUNCH(trackable_target_kernel, (P + 255) / 256, 256, 0, stream, P, f, g_tab.excl.as<int>(), d_xyz, d_rotation_raw,
               d_scaling_raw, d_out_xyz, d_out_rot, d_out_scale, box.dev, seq);
  GSICP_CUDA(cudaGetLastError());
  if (int e = box.wait(1, seq, stream, "trackable target count")) return e;
  return (long long)box.host[0];
}
