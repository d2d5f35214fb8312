// gicp.cu — Generalized-ICP tracker on the GPU behind the pygicp.FastGICP interface.
//
// Replaces fast_gicp::FastGICP<PointXYZ,PointXYZ> + LsqRegistration (CPU, OpenMP, PCL kd-tree):
//   FG = submodules/fast_gicp ; fgi = FG/include/fast_gicp/gicp/impl/fast_gicp_impl.hpp ;
//   lsq = FG/include/fast_gicp/gicp/impl/lsq_registration_impl.hpp
//
//   covariance_kernel   fgi:382-479 / 588-706 / 710-825  k-NN (exact, grid) -> mean -> cov/k -> Jacobi SVD
//                       -> quaternion(U), sqrt(sigma) -> NORMALIZED_ELLIPSE covariance (+ filter compaction)
//   cov_from_qs_kernel  fgi:828-902  covariances from (quaternion, scale) incl. the (w,x,y,z) ctor quirk
//   correspond_kernel   fgi:242-272  warp per source point: fp32 transform -> exact 1-NN (coalesced cell-row scans)
//   linearize_kernel    fgi:273-293 + 296-352  thread per source point: Mahalanobis (RCR^-1) -> e, J=[skew(Tp) | -I]
//                       -> 28-double block reduction (21 H + 6 b + err), deterministic last-block finalisation,
//                       result published into mapped pinned host memory
//   error_kernel        fgi:355-378  sum e^T M e with frozen correspondences
//   align()             pcl::Registration::align + fgi:225-240 + lsq:53-173 (LM loop, 6x6 LDLT on the host)
//
// Data layout in HBM (DESIGN.md §3): points fp32 xyz (12 B) + the same points in grid-cell order as
// float4 {x,y,z,index}; covariances as the 6 unique fp64 entries (48 B, the reference stores 128-B
// Matrix4d); Mahalanobis matrices 48 B per source point.  Compiled with -fmad=false (see gicp_math.cuh).
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "gicp_math.cuh"
#include <algorithm>

#include "grid.cuh"
#include "comm.cuh"

namespace gsicp {

constexpr int kRed = 28;       // 21 (upper triangle of H, row-major) + 6 (b) + 1 (error)
constexpr int kLinBlock = 128;

struct PoseD {  // pose in both precisions, passed by value
  double R[3][3], t[3];
  float Rf[3][3], tf[3];
};

// ------------------------------------------------------------------------------------------------
// covariance kernel
// ------------------------------------------------------------------------------------------------
struct CovArgs {
  int n;             // points in the cloud
  int k;             // neighbours requested
  float knn_max;     // compared with SQUARED distances (reference quirk, fgi:620)
  int clamp;         // 1: values = max(values, 1e-3)  (fgi:468-469: calculate_covariances only)
  const int32_t* filter;  // NULL: every point keeps its covariance at its own index
  const float* xyz;
  float* rots;       // [4n] x,y,z,w
  float* scales;     // [3n]
  double* cov;       // [6 * slots]
  float* new_xyz;    // [3 * num_trackable] (only with filter)
  const float* z;    // NULL, or per-point z values: exported scales are divided by max(1, z^1.5 * 2) (fgi:534-538)
  // multi-GPU (SURVEY §8e "GICP covariance: shard query points"): this rank handles point i iff its covariance slot lies
  // in [slot_begin, slot_end) — the source range its LM kernel linearises — or, for a point without a slot (untrackable),
  // iff i lies in [idx_begin, idx_end).  Single GPU: everything.
  int slot_begin, slot_end, idx_begin, idx_end;
  __device__ __forceinline__ bool mine(int i) const {
    if (filter) {
      const int f = filter[i];
      if (f > 0) return (f - 1) >= slot_begin && (f - 1) < slot_end;
      return i >= idx_begin && i < idx_end;
    }
    return i >= slot_begin && i < slot_end;
  }
};

// k-NN of every point of the cloud in itself, one warp per point: ids and squared distances sorted by (d2, id).
// The query point itself is its own nearest neighbour (distance 0), as with the reference's kd-tree search.
template <int K>
__global__ void __launch_bounds__(128)
knn_kernel(GridView g, int n, int k, const float* __restrict__ xyz, uint32_t* __restrict__ nn_id, float* __restrict__ nn_d2,
           CovArgs own) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= n || !own.mine(i)) return;  // warp-uniform
  const int lane = threadIdx.x & 31;
  const int kk = min(k, K);
  float d2;
  uint32_t id;
  grid_knn_warp(g, xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2], kk, 0xffffffffu, d2, id);
  if (lane < kk) {
    nn_id[(size_t)i * K + lane] = id;
    nn_d2[(size_t)i * K + lane] = d2;
  }
}

template <int K>
__global__ void __launch_bounds__(128, 1)
covariance_kernel(CovArgs a, const uint32_t* __restrict__ nn_id, const float* __restrict__ nn_d2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n || !a.mine(i)) return;
  const float qx = a.xyz[3 * (size_t)i], qy = a.xyz[3 * (size_t)i + 1], qz = a.xyz[3 * (size_t)i + 2];
  const int kk = min(a.k, K);
  struct { uint32_t id[K]; float d2[K]; } nn;
#pragma unroll
  for (int j = 0; j < K; j++) {
    nn.id[j] = (j < kk) ? nn_id[(size_t)i * K + j] : 0xffffffffu;
    nn.d2[j] = (j < kk) ? nn_d2[(size_t)i * K + j] : FLT_MAX;
  }

  const int found = min(kk, a.n);
  int reliable = 0;  // neighbours are sorted ascending, so the reliable ones are a prefix
  for (int j = 0; j < K; j++)
    if (j < found && nn.d2[j] < a.knn_max) reliable++;

  double mean[3] = {0, 0, 0};
  for (int j = 0; j < K; j++) {
    if (j < reliable) {
      const uint32_t id = nn.id[j];
      mean[0] += (double)a.xyz[3 * (size_t)id];
      mean[1] += (double)a.xyz[3 * (size_t)id + 1];
      mean[2] += (double)a.xyz[3 * (size_t)id + 2];
    }
  }
  const double inv_n = (double)reliable;
  mean[0] /= inv_n; mean[1] /= inv_n; mean[2] /= inv_n;  // NaN when no neighbour is reliable, like the reference
  double C[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
  for (int j = 0; j < K; j++) {
    if (j < reliable) {
      const uint32_t id = nn.id[j];
      const double dx = (double)a.xyz[3 * (size_t)id] - mean[0];
      const double dy = (double)a.xyz[3 * (size_t)id + 1] - mean[1];
      const double dz = (double)a.xyz[3 * (size_t)id + 2] - mean[2];
      C[0][0] += dx * dx; C[0][1] += dx * dy; C[0][2] += dx * dz;
      C[1][1] += dy * dy; C[1][2] += dy * dz; C[2][2] += dz * dz;
    }
  }
  const double kd = (double)a.k;  // divides by k, not by the neighbour count (fgi:635)
  C[0][0] /= kd; C[0][1] /= kd; C[0][2] /= kd; C[1][1] /= kd; C[1][2] /= kd; C[2][2] /= kd;
  C[1][0] = C[0][1]; C[2][0] = C[0][2]; C[2][1] = C[1][2];

  double U[3][3], S[3], V[3][3];
  svd3_jacobi(C, U, S, V);
  double q[4];
  quat_from_matrix(U, q);
  a.rots[4 * (size_t)i + 0] = (float)q[0];
  a.rots[4 * (size_t)i + 1] = (float)q[1];
  a.rots[4 * (size_t)i + 2] = (float)q[2];
  a.rots[4 * (size_t)i + 3] = (float)q[3];
  a.scales[3 * (size_t)i + 0] = (float)sqrt(S[0]);
  a.scales[3 * (size_t)i + 1] = (float)sqrt(S[1]);
  a.scales[3 * (size_t)i + 2] = (float)sqrt(S[2]);
  if (a.z) {  // calculate_covariances_withz
    const float z = (float)fmax(1.0, pow((double)a.z[i], 1.5) * 2.0);
    a.scales[3 * (size_t)i + 0] = __fdiv_rn((float)sqrt(S[0]), z);
    a.scales[3 * (size_t)i + 1] = __fdiv_rn((float)sqrt(S[1]), z);
    a.scales[3 * (size_t)i + 2] = __fdiv_rn((float)sqrt(S[2]), z);
  }

  int slot = i;
  if (a.filter) {
    const int f = a.filter[i];
    if (f == 0) return;
    slot = f - 1;
  }
  double values[3];
  if (S[1] == 0.0) {  // NORMALIZED_ELLIPSE (fgi:460-469, 681-689): normalised by the MIDDLE singular value
    values[0] = values[1] = values[2] = 1e-9;
  } else {
    values[0] = S[0] / S[1]; values[1] = S[1] / S[1]; values[2] = S[2] / S[1];
    if (a.clamp) {
      values[0] = fmax(values[0], 1e-3); values[1] = fmax(values[1], 1e-3); values[2] = fmax(values[2], 1e-3);
    }
  }
  double Rg[3][3];
  a_diag_bt(U, values, V, Rg);
  double* o = a.cov + 6 * (size_t)slot;
  // the reference keeps the full (numerically almost symmetric) 3x3; we keep its symmetric part's
  // upper triangle taken from the upper entries
  o[0] = Rg[0][0]; o[1] = Rg[0][1]; o[2] = Rg[0][2]; o[3] = Rg[1][1]; o[4] = Rg[1][2]; o[5] = Rg[2][2];
  if (a.filter) {
    a.new_xyz[3 * (size_t)slot + 0] = qx;
    a.new_xyz[3 * (size_t)slot + 1] = qy;
    a.new_xyz[3 * (size_t)slot + 2] = qz;
  }
}

// Sharded runs: every rank keeps the COMPLETE compacted cloud (the k-NN / SVD work is what is sharded, not 12 bytes per point)
__global__ void compact_xyz_kernel(int n, const int32_t* __restrict__ filter, const float* __restrict__ xyz, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int f = filter[i];
  if (f <= 0) return;
  out[3 * (size_t)(f - 1) + 0] = xyz[3 * (size_t)i];
  out[3 * (size_t)(f - 1) + 1] = xyz[3 * (size_t)i + 1];
  out[3 * (size_t)(f - 1) + 2] = xyz[3 * (size_t)i + 2];
}

// covariances from (quaternion, scale) (fgi:828-902)
__global__ void cov_from_qs_kernel(int n, const float* __restrict__ rots, const float* __restrict__ scales,
                                   double* __restrict__ cov) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double sv[3];
  for (int d = 0; d < 3; d++) {
    const double s = (double)scales[3 * (size_t)i + d];
    sv[d] = s * s;
  }
  if (sv[1] < 1e-3) {
    sv[0] = sv[1] = sv[2] = 1e-3;
  } else {
    const double m = sv[1];
    sv[0] = sv[0] / m; sv[1] = sv[1] / m; sv[2] = sv[2] / m;
  }
  // Reference quirk (fgi:890-894): the stored (x,y,z,w) is passed to a (w,x,y,z) constructor.
  double w = (double)rots[4 * (size_t)i + 0], x = (double)rots[4 * (size_t)i + 1];
  double y = (double)rots[4 * (size_t)i + 2], z = (double)rots[4 * (size_t)i + 3];
  const double nrm = sqrt(x * x + y * y + z * z + w * w);
  if (nrm > 0.0) {  // Eigen's normalized() leaves a zero quaternion untouched
    x /= nrm; y /= nrm; z /= nrm; w /= nrm;
  }
  double R[3][3], C[3][3];
  quat_to_matrix(x, y, z, w, R);
  a_diag_bt(R, sv, R, C);
  double* o = cov + 6 * (size_t)i;
  o[0] = C[0][0]; o[1] = C[0][1]; o[2] = C[0][2]; o[3] = C[1][1]; o[4] = C[1][2]; o[5] = C[2][2];
}

// ------------------------------------------------------------------------------------------------
// linearize / error kernels
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// block-level reduction of NV doubles per thread into partial[blockIdx][NV]; the last block to finish
// sums the partials in block order (deterministic) into out[NV].
//
// When `host_out` is non-null (every run but a sharded one with the all-reduce callback) the last block also publishes the
// sums into the handle's HostMailbox (mapped pinned host memory, host_common.h) and then bumps the sequence word the host
// spins on: the result reaches the LM loop without a D2H memcpy or a cudaStreamSynchronize round trip.
template <int NV>
__device__ __forceinline__ void block_reduce_finalize(double* v, double* __restrict__ partial, double* __restrict__ out,
                                                      unsigned int* __restrict__ counter, double* host_out = nullptr,
                                                      volatile unsigned long long* host_seq = nullptr,
                                                      unsigned long long seq = 0, CommView comm = CommView(),
                                                      unsigned long long xseq = 0) {
  __shared__ double s_red[kLinBlock / 32][NV];
  __shared__ double s_tot[NV];
  __shared__ bool s_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < NV; k++) {
    const double r = warp_sum_d(v[k]);
    if (lane == 0) s_red[warp][k] = r;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double r = 0.0;
#pragma unroll
    for (int w = 0; w < kLinBlock / 32; w++) r += s_red[w][threadIdx.x];
    partial[(size_t)blockIdx.x * NV + threadIdx.x] = r;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int done = atomicAdd(counter, 1u);
    s_last = (done == gridDim.x - 1);
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    if (threadIdx.x < NV) {
      double r = 0.0;
      for (unsigned int b = 0; b < gridDim.x; b++) r += partial[(size_t)b * NV + threadIdx.x];
      s_tot[threadIdx.x] = r;
    }
    __syncthreads();
    if (comm.active()) {
      // multi-GPU: the last block exchanges this rank's sums with the peers through their segments (comm.cuh) and adds
      // the world's slots in rank order — the result the host reads is already the global one, bit-identical on all ranks
      comm_lm_publish(comm, xseq, s_tot, NV);
      comm_lm_collect(comm, xseq, s_tot, NV);  // a lost peer leaves the local sums in place after the poll budget
    }
    if (threadIdx.x < NV) {
      out[threadIdx.x] = s_tot[threadIdx.x];
      if (host_out) host_out[threadIdx.x] = s_tot[threadIdx.x];
    }
    if (host_out) {
      __threadfence_system();
      __syncthreads();  // s_last is block-uniform
    }
    if (threadIdx.x == 0) {
      *counter = 0u;  // ready for the next launch
      if (host_seq) {
        *host_seq = seq;
        __threadfence_system();
      }
    }
  }
}

struct LinArgs {
  int begin, end;          // source range of this rank
  double max_corr_sq;      // corr_dist_threshold_^2 in double (fgi:271)
  const float* src_xyz;
  const double* src_cov;
  const float* tgt_xyz;
  const double* tgt_cov;
  int32_t* corr;
  float* sqd;
  double* mahal;           // [6 * n_src]
  double* partial;
  double* out;             // [28]
  unsigned int* counter;
  double* host_out;        // mapped pinned [28] or null
  volatile unsigned long long* host_seq;
  unsigned long long seq;
  CommView comm;             // multi-GPU: exchange inside the last block
  unsigned long long xseq;
};

// Correspondence search (fgi:242-272): one WARP per source point.  fp32 transform of the query, exact 1-NN in the
// target grid, squared distance and thresholded index.
__global__ void __launch_bounds__(128)
correspond_kernel(GridView tgt, PoseD T, int begin, int end, double max_corr_sq, const float* __restrict__ src_xyz,
                  int32_t* __restrict__ corr, float* __restrict__ sqd) {
  const int i = begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (i >= end) return;  // warp-uniform
  const float px = src_xyz[3 * (size_t)i], py = src_xyz[3 * (size_t)i + 1], pz = src_xyz[3 * (size_t)i + 2];
  // fp32 transform without contraction, in the order Eigen's packet product evaluates trans_f * getVector4fMap()
  // (fgi:260): (c0*x + c1*y) + (c2*z + c3*1).  Pinned against the reference build (tests/test_gicp_reference.py): the
  // squared distances below are bit-identical to fast_gicp's.
  const float tx = __fadd_rn(__fadd_rn(__fmul_rn(T.Rf[0][0], px), __fmul_rn(T.Rf[0][1], py)), __fadd_rn(__fmul_rn(T.Rf[0][2], pz), T.tf[0]));
  const float ty = __fadd_rn(__fadd_rn(__fmul_rn(T.Rf[1][0], px), __fmul_rn(T.Rf[1][1], py)), __fadd_rn(__fmul_rn(T.Rf[1][2], pz), T.tf[1]));
  const float tz = __fadd_rn(__fadd_rn(__fmul_rn(T.Rf[2][0], px), __fmul_rn(T.Rf[2][1], py)), __fadd_rn(__fmul_rn(T.Rf[2][2], pz), T.tf[2]));
  float d2;
  uint32_t id;
  grid_nn_warp(tgt, tx, ty, tz, d2, id);
  if ((threadIdx.x & 31) == 0) {
    sqd[i] = d2;
    corr[i] = ((tgt.n > 0) && ((double)d2 < max_corr_sq)) ? (int32_t)id : -1;
  }
}

// pcl::Registration::getFitnessScore: sum and count of the squared NN distances <= max_range (one CTA, deterministic).
__global__ void __launch_bounds__(1024)
fitness_kernel(int n, const float* __restrict__ sqd, double max_range, double* __restrict__ out) {
  __shared__ double s_sum[32], s_cnt[32];
  double sum = 0.0, cnt = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double d = (double)sqd[i];
    if (d <= max_range) {
      sum += d;
      cnt += 1.0;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    sum += __shfl_down_sync(0xffffffffu, sum, o);
    cnt += __shfl_down_sync(0xffffffffu, cnt, o);
  }
  if ((threadIdx.x & 31) == 0) {
    s_sum[threadIdx.x >> 5] = sum;
    s_cnt[threadIdx.x >> 5] = cnt;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, c = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) {
      a += s_sum[w];
      c += s_cnt[w];
    }
    out[0] = a;
    out[1] = c;
  }
}

// Sharded runs: every rank owns the correspondences of its source range only.  When the caller asks for them
// (get_source_correspondence) the ranges are merged through the all-reduce callback: each entry is encoded so that it is
// non-zero on exactly one rank (index + 1, squared distance) and zero elsewhere — the sum is exact.
__global__ void corr_pack_kernel(int n, int begin, int end, const int32_t* __restrict__ corr, const float* __restrict__ sqd,
                                 double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const bool mine = i >= begin && i < end;
  out[i] = mine ? (double)(corr[i] + 1) : 0.0;
  out[(size_t)n + i] = mine ? (double)sqd[i] : 0.0;
}
__global__ void corr_unpack_kernel(int n, const double* __restrict__ in, int32_t* __restrict__ corr, float* __restrict__ sqd) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  corr[i] = (int32_t)in[i] - 1;
  sqd[i] = (float)in[(size_t)n + i];
}

// Mahalanobis + residual/Jacobian of ONE matched source point i <-> target point j (fgi:273-352): adds the point's 21 H
// entries (upper triangle, row-major), 6 b entries and its error term to v[28], stores the Mahalanobis matrix.
__device__ __forceinline__ void linearize_point(const PoseD& T, int i, int j, const float* __restrict__ src_xyz,
                                                const double* __restrict__ src_cov, const float* __restrict__ tgt_xyz,
                                                const double* __restrict__ tgt_cov, double* __restrict__ mahal, double* v) {
  const float px = src_xyz[3 * (size_t)i], py = src_xyz[3 * (size_t)i + 1], pz = src_xyz[3 * (size_t)i + 2];
  const double* ca = src_cov + 6 * (size_t)i;
  const double* cb = tgt_cov + 6 * (size_t)j;
  const double A[3][3] = {{ca[0], ca[1], ca[2]}, {ca[1], ca[3], ca[4]}, {ca[2], ca[4], ca[5]}};
  // RCR = C_B + R C_A R^T  (fgi:280)
  double RA[3][3], RCR[3][3];
#pragma unroll
  for (int r = 0; r < 3; r++)
#pragma unroll
    for (int c = 0; c < 3; c++) RA[r][c] = (T.R[r][0] * A[0][c] + T.R[r][1] * A[1][c]) + T.R[r][2] * A[2][c];
  const double B[3][3] = {{cb[0], cb[1], cb[2]}, {cb[1], cb[3], cb[4]}, {cb[2], cb[4], cb[5]}};
#pragma unroll
  for (int r = 0; r < 3; r++)
#pragma unroll
    for (int c = 0; c < 3; c++) RCR[r][c] = B[r][c] + ((RA[r][0] * T.R[c][0] + RA[r][1] * T.R[c][1]) + RA[r][2] * T.R[c][2]);
  double M[3][3];
  if (!inverse3(RCR, M)) {
    // reference: pseudo-inverse via complete orthogonal decomposition (fgi:283-286); a singular
    // RCR cannot occur with regularised covariances — contribute nothing.
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
      for (int c = 0; c < 3; c++) M[r][c] = 0.0;
  }
  double* mo = mahal + 6 * (size_t)i;
  mo[0] = M[0][0]; mo[1] = M[0][1]; mo[2] = M[0][2]; mo[3] = M[1][1]; mo[4] = M[1][2]; mo[5] = M[2][2];
  // use the stored (symmetric) representation from here on so linearize and compute_error agree
  M[1][0] = M[0][1]; M[2][0] = M[0][2]; M[2][1] = M[1][2];

  const double ax = (double)px, ay = (double)py, az = (double)pz;
  const double qx = ((T.R[0][0] * ax + T.R[0][1] * ay) + T.R[0][2] * az) + T.t[0];
  const double qy = ((T.R[1][0] * ax + T.R[1][1] * ay) + T.R[1][2] * az) + T.t[1];
  const double qz = ((T.R[2][0] * ax + T.R[2][1] * ay) + T.R[2][2] * az) + T.t[2];
  const double e[3] = {(double)tgt_xyz[3 * (size_t)j] - qx, (double)tgt_xyz[3 * (size_t)j + 1] - qy,
                       (double)tgt_xyz[3 * (size_t)j + 2] - qz};
  double Me[3];
#pragma unroll
  for (int r = 0; r < 3; r++) Me[r] = (M[r][0] * e[0] + M[r][1] * e[1]) + M[r][2] * e[2];
  v[27] += (e[0] * Me[0] + e[1] * Me[1]) + e[2] * Me[2];

  // J = [S | -I], S = skew(q):  S = [[0,-qz,qy],[qz,0,-qx],[-qy,qx,0]]
  const double S[3][3] = {{0.0, -qz, qy}, {qz, 0.0, -qx}, {-qy, qx, 0.0}};
  double MS[3][3];  // M * S
#pragma unroll
  for (int r = 0; r < 3; r++)
#pragma unroll
    for (int c = 0; c < 3; c++) MS[r][c] = (M[r][0] * S[0][c] + M[r][1] * S[1][c]) + M[r][2] * S[2][c];
  double H[6][6];
#pragma unroll
  for (int r = 0; r < 3; r++)
#pragma unroll
    for (int c = 0; c < 3; c++) {
      H[r][c] = (S[0][r] * MS[0][c] + S[1][r] * MS[1][c]) + S[2][r] * MS[2][c];  // S^T M S
      H[r][3 + c] = -((S[0][r] * M[0][c] + S[1][r] * M[1][c]) + S[2][r] * M[2][c]);  // -S^T M
      H[3 + r][3 + c] = M[r][c];
    }
  int o = 0;
#pragma unroll
  for (int r = 0; r < 6; r++)
#pragma unroll
    for (int c = r; c < 6; c++) v[o++] += H[r][c];
#pragma unroll
  for (int r = 0; r < 3; r++) {
    v[21 + r] += (S[0][r] * Me[0] + S[1][r] * Me[1]) + S[2][r] * Me[2];  // S^T M e
    v[24 + r] += -Me[r];
  }
}

// e^T M e of one matched pair with the cached Mahalanobis matrix (fgi:355-378)
__device__ __forceinline__ double error_point(const PoseD& T, int i, int j, const float* __restrict__ src_xyz,
                                              const float* __restrict__ tgt_xyz, const double* __restrict__ mahal) {
  const double ax = (double)src_xyz[3 * (size_t)i], ay = (double)src_xyz[3 * (size_t)i + 1], az = (double)src_xyz[3 * (size_t)i + 2];
  const double qx = ((T.R[0][0] * ax + T.R[0][1] * ay) + T.R[0][2] * az) + T.t[0];
  const double qy = ((T.R[1][0] * ax + T.R[1][1] * ay) + T.R[1][2] * az) + T.t[1];
  const double qz = ((T.R[2][0] * ax + T.R[2][1] * ay) + T.R[2][2] * az) + T.t[2];
  const double e[3] = {(double)tgt_xyz[3 * (size_t)j] - qx, (double)tgt_xyz[3 * (size_t)j + 1] - qy,
                       (double)tgt_xyz[3 * (size_t)j + 2] - qz};
  // the Mahalanobis matrices are rewritten by other blocks between the phases of the persistent LM kernel: read them
  // through L2 (ld.global.cg), never from a stale L1 line
  const double* mp = mahal + 6 * (size_t)i;
  const double m[6] = {__ldcg(mp), __ldcg(mp + 1), __ldcg(mp + 2), __ldcg(mp + 3), __ldcg(mp + 4), __ldcg(mp + 5)};
  const double Me0 = (m[0] * e[0] + m[1] * e[1]) + m[2] * e[2];
  const double Me1 = (m[1] * e[0] + m[3] * e[1]) + m[4] * e[2];
  const double Me2 = (m[2] * e[0] + m[4] * e[1]) + m[5] * e[2];
  return (e[0] * Me0 + e[1] * Me1) + e[2] * Me2;
}

// Normal-equation reduction of the host-driven path: one THREAD per source point.
__global__ void __launch_bounds__(kLinBlock, 1)
linearize_kernel(PoseD T, LinArgs a) {
  const int i = a.begin + blockIdx.x * blockDim.x + threadIdx.x;
  double v[kRed];
#pragma unroll
  for (int k = 0; k < kRed; k++) v[k] = 0.0;
  if (i < a.end) {
    const int32_t j = a.corr[i];
    if (j >= 0) linearize_point(T, i, j, a.src_xyz, a.src_cov, a.tgt_xyz, a.tgt_cov, a.mahal, v);
  }
  block_reduce_finalize<kRed>(v, a.partial, a.out, a.counter, a.host_out, a.host_seq, a.seq, a.comm, a.xseq);
}

struct ErrArgs {
  int begin, end;
  const float* src_xyz;
  const float* tgt_xyz;
  const int32_t* corr;
  const double* mahal;
  double* partial;
  double* out;  // [1]
  unsigned int* counter;
  double* host_out;
  volatile unsigned long long* host_seq;
  unsigned long long seq;
  CommView comm;
  unsigned long long xseq;
};

__global__ void __launch_bounds__(kLinBlock)
error_kernel(PoseD T, ErrArgs a) {
  const int i = a.begin + blockIdx.x * blockDim.x + threadIdx.x;
  double v[1] = {0.0};
  if (i < a.end) {
    const int32_t j = a.corr[i];
    if (j >= 0) v[0] = error_point(T, i, j, a.src_xyz, a.tgt_xyz, a.mahal);
  }
  block_reduce_finalize<1>(v, a.partial, a.out, a.counter, a.host_out, a.host_seq, a.seq, a.comm, a.xseq);
}

// ------------------------------------------------------------------------------------------------
// Device-resident Levenberg-Marquardt loop: ONE persistent kernel per align()
// (lsq_registration_impl.hpp:53-78 computeTransformation + :125-173 step_lm, with fgi:242-378 as its phases).
//
//   outer iteration:  phase L  every warp: correspondence search (warp-cooperative exact 1-NN in the target grid) for 4
//                              source points, then lanes 0..3 build Mahalanobis + J^T M J + J^T M e of their point in
//                              fp64; per-thread 28-double accumulators -> block reduction -> partial[block][28]
//                     grid barrier; every block sums the partials in the same fixed order (H, b, y0 identical everywhere)
//                     and its thread 0 takes the LM decision redundantly — no broadcast, no host.
//     up to 10 trials: solve (H + lambda I) d = -b (pivoted LDL^T), delta = (so3_exp, t), xi = delta x0
//                     phase E  sum e^T M e at xi with frozen correspondences / cached Mahalanobis; grid barrier; rho test.
// The host launches it once and spins on one sequence word in mapped pinned memory: zero host round trips inside the loop
// (the host-driven path below costs one launch + one spin-wait per phase).  Sums are deterministic: fixed point -> lane,
// fixed block order.
// Launch shape: one 256-thread block per SM at most (half of each SM's registers), ordinary launch + an atomic-counter
// grid barrier instead of a cooperative launch: the kernel starts on whatever SMs have room while the mapper's kernels
// run on the other stream (a cooperative launch would wait for — and then occupy — the whole GPU).  All blocks are
// co-resident once the other kernels drain (grid <= SM count), so the barrier cannot deadlock; a poll budget turns a
// lost peer into an error status instead of a hang.
// ------------------------------------------------------------------------------------------------
constexpr int kLmBlock = 256;     // threads per block of align_lm_kernel
constexpr int kLmChunk = 4;       // source points per warp visit
constexpr int kLmSeg = 8;         // partial-sum segments per value in the cross-block reduction
constexpr long long kLmPollBudget = 1ll << 27;
constexpr int kLmPersistentMax = 65536;  // source points per rank up to which the persistent LM kernel is used  // barrier polls before giving up (seconds of wall time)

struct LmResult {  // lives in mapped pinned host memory; written by block 0
  double R[9], t[3];      // final pose x0
  double H[36];           // Hessian of the last accepted step (lsq:169)
  double lambda;
  int iterations;         // outer iterations run (= value align() returns)
  int converged;
  int status;             // 0 ok, 1 "lm not converged" (step_lm returned false), 3 grid barrier / peer exchange timed out
  int n_lin, n_err;
  int n_marks;            // phase timestamps recorded (GSICP_LM_MARKS=1; tools/prof_align.py)
  unsigned long long seq;
  unsigned long long marks[48];  // %globaltimer of block 0 at: start, then after L, reduce, trial, E, reduce per phase
};

struct LmArgs {
  GridView tgt;
  int begin, end;            // source range of this rank
  double max_corr_sq;
  const float* src_xyz;
  const double* src_cov;
  const float* tgt_xyz;
  const double* tgt_cov;
  int32_t* corr;
  float* sqd;
  double* mahal;
  double* partL;             // [blocks][28]
  double* partE;             // [2][blocks]
  unsigned int* barrier;     // grid-barrier counter, zero at launch
  CommView comm;             // multi-GPU: the per-rank sums are exchanged through the peers' segments inside the kernel
  unsigned long long xseq;   // first exchange sequence number of this launch
  int max_iterations, lm_max_iterations;
  double rot_eps, trans_eps, init_lambda_factor;
  Iso guess;
  LmResult* result;          // device alias of the mapped host block
  unsigned long long seq;
  int marks;                 // record phase timestamps into result->marks (profiling aid)
};

__device__ __forceinline__ PoseD make_pose_dev(const Iso& x) {
  PoseD p;
#pragma unroll
  for (int i = 0; i < 3; i++) {
#pragma unroll
    for (int j = 0; j < 3; j++) {
      p.R[i][j] = x.R[i][j];
      p.Rf[i][j] = (float)x.R[i][j];
    }
    p.t[i] = x.t[i];
    p.tf[i] = (float)x.t[i];
  }
  return p;
}

// fp32 transform of a source point in the order Eigen's packet product evaluates trans_f * getVector4fMap() (fgi:260)
__device__ __forceinline__ void transform_f32(const PoseD& T, float px, float py, float pz, float& tx, float& ty, float& tz) {
  tx = __fadd_rn(__fadd_rn(__fmul_rn(T.Rf[0][0], px), __fmul_rn(T.Rf[0][1], py)), __fadd_rn(__fmul_rn(T.Rf[0][2], pz), T.tf[0]));
  ty = __fadd_rn(__fadd_rn(__fmul_rn(T.Rf[1][0], px), __fmul_rn(T.Rf[1][1], py)), __fadd_rn(__fmul_rn(T.Rf[1][2], pz), T.tf[1]));
  tz = __fadd_rn(__fadd_rn(__fmul_rn(T.Rf[2][0], px), __fmul_rn(T.Rf[2][1], py)), __fadd_rn(__fmul_rn(T.Rf[2][2], pz), T.tf[2]));
}

// Grid barrier on a monotonically increasing counter (zeroed by the host before the launch): arrival k of every block
// completes when the counter reaches k * gridDim.x.  Returns false when the poll budget ran out.
__device__ __forceinline__ bool grid_barrier(unsigned int* counter, unsigned int& epoch) {
  __shared__ int s_ok;
  __syncthreads();
  if (threadIdx.x == 0) {
    epoch += gridDim.x;
    __threadfence();  // release this block's global writes
    atomicAdd(counter, 1u);
    long long polls = 0;
    int ok = 1;
    while (true) {
      unsigned int v;
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
      if (v >= epoch) break;
      if (++polls > kLmPollBudget) {
        ok = 0;
        break;
      }
    }
    s_ok = ok;
  }
  __syncthreads();
  return s_ok != 0;
}

// Block-level sum of NV doubles per thread -> out[NV] (thread t < NV writes value t); warps in index order.
template <int NV>
__device__ __forceinline__ void block_sum_store(const double* v, double* __restrict__ out) {
  __shared__ double s_red[kLmBlock / 32][NV];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < NV; k++) {
    const double r = warp_sum_d(v[k]);
    if (lane == 0) s_red[warp][k] = r;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double r = 0.0;
#pragma unroll
    for (int w = 0; w < kLmBlock / 32; w++) r += s_red[w][threadIdx.x];
    out[threadIdx.x] = r;
  }
  __syncthreads();
}

// Same result layout as block_sum_store, for values that are produced in several passes: each pass adds its warp sums into
// the warp's row of s_acc (lane 0), block_acc_store then adds the rows in warp order.
template <int NV>
__device__ __forceinline__ void warp_acc_add(const double* v, double (*s_acc)[NV]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < NV; k++) {
    const double r = warp_sum_d(v[k]);
    if (lane == 0) s_acc[warp][k] += r;
  }
}
template <int NV>
__device__ __forceinline__ void block_acc_store(double (*s_acc)[NV], double* __restrict__ out) {
  __syncthreads();
  if (threadIdx.x < NV) {
    double r = 0.0;
#pragma unroll
    for (int w = 0; w < kLmBlock / 32; w++) r += s_acc[w][threadIdx.x];
    out[threadIdx.x] = r;
  }
  __syncthreads();
}

// Sum partial[b][NV] over the blocks in a fixed order, identically in every block: thread (seg, k) adds the blocks
// b = seg, seg + kLmSeg, ...; thread k < NV then adds the kLmSeg segment sums in order.  Result in s_out[NV].
template <int NV>
__device__ __forceinline__ void reduce_partials(const double* __restrict__ partial, int nblocks, double* s_out) {
  __shared__ double s_seg[kLmSeg][NV];
  const int k = threadIdx.x % NV, seg = threadIdx.x / NV;
  if (seg < kLmSeg) {
    double r = 0.0;
    for (int b = seg; b < nblocks; b += kLmSeg) r += __ldcg(partial + (size_t)b * NV + k);
    s_seg[seg][k] = r;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double r = 0.0;
#pragma unroll
    for (int sg = 0; sg < kLmSeg; sg++) r += s_seg[sg][threadIdx.x];
    s_out[threadIdx.x] = r;
  }
  __syncthreads();
}

// (256, 2): caps the kernel at 128 registers so that one block takes half of an SM's register file
__global__ void __launch_bounds__(kLmBlock, 2)
align_lm_kernel(LmArgs a) {
  __shared__ double s_sum[kRed];
  __shared__ double s_accL[kLmBlock / 32][kRed];
  __shared__ Iso s_x0, s_xi, s_delta;
  __shared__ double s_H[6][6], s_b[6], s_d[6];
  __shared__ double s_y0, s_lambda, s_nu;
  __shared__ int s_state;  // 0: run another trial / phase, 1: step accepted or converged inside step_lm, 2: lm failed

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int warps_per_block = kLmBlock / 32;
  const int gwarp = blockIdx.x * warps_per_block + warp, total_warps = gridDim.x * warps_per_block;
  const int gthread = blockIdx.x * kLmBlock + threadIdx.x, total_threads = gridDim.x * kLmBlock;
  const int n = a.end - a.begin;
  const int nchunks = (n + kLmChunk - 1) / kLmChunk;

  if (threadIdx.x == 0) {
    s_x0 = a.guess;
    s_lambda = -1.0;
  }
  __syncthreads();

  GridMeta grid_meta = {};  // loaded once: the search would otherwise start every chunk with this dependent load
  if (a.tgt.n > 0) grid_meta = *a.tgt.meta;
  int n_marks = 0;
  auto mark = [&]() {
    if (a.marks && blockIdx.x == 0 && threadIdx.x == 0 && n_marks < 48) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      a.result->marks[n_marks++] = t;
    }
  };
  mark();
  unsigned int epoch = 0;  // thread 0's barrier target
  unsigned long long xseq = a.xseq;
  int iterations = 0, converged = 0, status = 0, n_lin = 0, n_err = 0;
  for (int it = 0; it < a.max_iterations && !converged; it++) {
    iterations = it + 1;
    // ---------------- phase L: correspondences + linearisation at x0 ----------------
    {
      const PoseD T = make_pose_dev(s_x0);
      for (int k = lane; k < kRed; k += 32) s_accL[warp][k] = 0.0;
      __syncwarp();
      // A warp takes its chunks of kLmChunk points in groups of 32 / kLmChunk: the nearest-neighbour searches of one chunk
      // run in lock step (grid_nn_warp_multi), lane 4 s + k keeps the match of point k of the group's s-th chunk, and ONE
      // linearisation pass then serves the whole group with up to 32 lanes busy.
      constexpr int kGroup = 32 / kLmChunk;
      for (int cg = gwarp; cg < nchunks; cg += kGroup * total_warps) {
        int my_i = -1, my_j = -1;
        for (int sl = 0; sl < kGroup; sl++) {
          const int c = cg + sl * total_warps;
          if (c >= nchunks) break;  // warp-uniform
          const int i0 = a.begin + c * kLmChunk;
          float tx[kLmChunk], ty[kLmChunk], tz[kLmChunk], d2[kLmChunk];
          uint32_t id[kLmChunk];
#pragma unroll
          for (int k = 0; k < kLmChunk; k++) {
            const int i = min(i0 + k, a.end - 1);  // the tail of the last chunk repeats its last point (result unused)
            const float px = a.src_xyz[3 * (size_t)i], py = a.src_xyz[3 * (size_t)i + 1], pz = a.src_xyz[3 * (size_t)i + 2];
            transform_f32(T, px, py, pz, tx[k], ty[k], tz[k]);
          }
          grid_nn_warp_multi<kLmChunk>(a.tgt, grid_meta, tx, ty, tz, d2, id);
#pragma unroll
          for (int k = 0; k < kLmChunk; k++) {
            const int i = i0 + k;
            if (i < a.end) {  // warp-uniform
              const int32_t j = ((a.tgt.n > 0) && ((double)d2[k] < a.max_corr_sq)) ? (int32_t)id[k] : -1;
              if (lane == 0) {
                a.sqd[i] = d2[k];
                a.corr[i] = j;
              }
              if (lane == sl * kLmChunk + k) {
                my_i = i;
                my_j = j;
              }
            }
          }
        }
        // the 28 sums live in registers only for the duration of this pass (the search above needs the registers)
        double v[kRed];
#pragma unroll
        for (int k = 0; k < kRed; k++) v[k] = 0.0;
        if (my_j >= 0) linearize_point(T, my_i, my_j, a.src_xyz, a.src_cov, a.tgt_xyz, a.tgt_cov, a.mahal, v);
        warp_acc_add<kRed>(v, s_accL);
      }
      block_acc_store<kRed>(s_accL, a.partL + (size_t)blockIdx.x * kRed);
    }
    mark();  // L done in block 0
    if (!grid_barrier(a.barrier, epoch)) {
      status = 3;
      break;
    }
    mark();  // barrier passed
    if (a.comm.active()) {
      // this rank's sums go to every peer's segment (block 0), then every block of every rank adds the world's slots in
      // rank order: H, b, y0 are bit-identical on all ranks and the redundant LM decision stays in lock step
      if (blockIdx.x == 0) {
        reduce_partials<kRed>(a.partL, gridDim.x, s_sum);
        comm_lm_publish(a.comm, xseq, s_sum, kRed);
      }
      if (!comm_lm_collect(a.comm, xseq, s_sum, kRed)) {
        status = 3;
        break;
      }
      xseq++;
    } else {
      reduce_partials<kRed>(a.partL, gridDim.x, s_sum);
    }
    n_lin++;
    mark();  // H, b, y0 reduced
    if (threadIdx.x == 0) {
      int o = 0;
      for (int r = 0; r < 6; r++)
        for (int c = r; c < 6; c++) {
          s_H[r][c] = s_sum[o];
          s_H[c][r] = s_sum[o];
          o++;
        }
      for (int r = 0; r < 6; r++) s_b[r] = s_sum[21 + r];
      s_y0 = s_sum[27];
      if (s_lambda < 0.0) {  // lsq:130-132
        double mx = 0.0;
        for (int i = 0; i < 6; i++) mx = fmax(mx, fabs(s_H[i][i]));
        s_lambda = a.init_lambda_factor * mx;
      }
      s_nu = 2.0;
      s_state = 0;
    }
    __syncthreads();
    // ---------------- LM trials (lsq:135-170) ----------------
    int trial = 0;
    for (; trial < a.lm_max_iterations; trial++) {
      if (threadIdx.x == 0) lm_trial(s_H, s_b, s_lambda, s_x0, s_d, s_delta, s_xi);
      __syncthreads();
      mark();  // trial solved
      // phase E: error at xi with frozen correspondences
      {
        const PoseD T = make_pose_dev(s_xi);
        double v[1] = {0.0};
        for (int i = a.begin + gthread; i < a.end; i += total_threads) {
          const int32_t j = __ldcg(a.corr + i);  // written by another block in phase L: through L2
          if (j >= 0) v[0] += error_point(T, i, j, a.src_xyz, a.tgt_xyz, a.mahal);
        }
        block_sum_store<1>(v, a.partE + (size_t)(trial & 1) * gridDim.x + blockIdx.x);
      }
      mark();  // E done in block 0
      if (!grid_barrier(a.barrier, epoch)) {
        status = 3;
        break;
      }
      mark();  // barrier passed
      __shared__ double s_yi[1];
      if (a.comm.active()) {
        if (blockIdx.x == 0) {
          reduce_partials<1>(a.partE + (size_t)(trial & 1) * gridDim.x, gridDim.x, s_yi);
          comm_lm_publish(a.comm, xseq, s_yi, 1);
        }
        if (!comm_lm_collect(a.comm, xseq, s_yi, 1)) {
          status = 3;
          break;
        }
        xseq++;
      } else {
        reduce_partials<1>(a.partE + (size_t)(trial & 1) * gridDim.x, gridDim.x, s_yi);
      }
      n_err++;
      mark();  // error reduced
      if (threadIdx.x == 0) {
        const double yi = s_yi[0];
        double dot = 0.0;
        for (int i = 0; i < 6; i++) dot += s_d[i] * (s_lambda * s_d[i] - s_b[i]);
        const double rho = (s_y0 - yi) / dot;
        if (rho < 0) {
          if (lm_is_converged(a.rot_eps, a.trans_eps, s_delta)) {
            s_state = 1;  // step_lm returns true without moving x0
          } else {
            s_lambda = s_nu * s_lambda;
            s_nu = 2 * s_nu;
            s_state = 0;
          }
        } else {
          s_x0 = s_xi;
          s_lambda = s_lambda * fmax(1.0 / 3.0, 1 - pow(2 * rho - 1, 3));
          if (blockIdx.x == 0)
            for (int r = 0; r < 6; r++)
              for (int c = 0; c < 6; c++) a.result->H[6 * r + c] = s_H[r][c];
          s_state = 1;
        }
      }
      __syncthreads();
      if (s_state == 1) break;
    }
    if (status == 3) break;
    if (s_state != 1) {  // the 10 trials were rejected: "lm not converged!!" (lsq:70-73)
      status = 1;
      break;
    }
    converged = lm_is_converged(a.rot_eps, a.trans_eps, s_delta) ? 1 : 0;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    LmResult* r = a.result;
    for (int i = 0; i < 3; i++) {
      for (int j = 0; j < 3; j++) r->R[3 * i + j] = s_x0.R[i][j];
      r->t[i] = s_x0.t[i];
    }
    r->lambda = s_lambda;
    r->iterations = iterations;
    r->converged = converged;
    r->status = status;
    r->n_lin = n_lin;
    r->n_err = n_err;
    mark();
    r->n_marks = n_marks;
    __threadfence_system();
    *(volatile unsigned long long*)&r->seq = a.seq;
    __threadfence_system();
  }
}

__global__ void f64_to_f32_kernel(size_t n, const double* __restrict__ in, float* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (float)in[i];
}

__global__ void identity_filter_kernel(int n, int32_t* f) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) f[i] = i + 1;
}

// ------------------------------------------------------------------------------------------------
// host side: 6x6 LDLT, SE(3) helpers
// ------------------------------------------------------------------------------------------------
static PoseD make_pose(const Iso& x) {
  PoseD p;
  for (int i = 0; i < 3; i++) {
    for (int j = 0; j < 3; j++) {
      p.R[i][j] = x.R[i][j];
      p.Rf[i][j] = (float)x.R[i][j];
    }
    p.t[i] = x.t[i];
    p.tf[i] = (float)x.t[i];
  }
  return p;
}

struct Cloud {
  int n = 0;           // points currently held (after a *_with_filter call: the trackable subset)
  Scratch xyz;         // float [3n]
  Scratch xyz_alt;     // compaction target
  DeviceGrid grid;
  bool grid_stale = true;  // xyz changed since the grid was built; rebuilt on first use (ensure_grid)
  Scratch cov;         // double [6 * cov_n]
  int cov_n = 0;
  Scratch rots, scales;
  int rots_n = 0, scales_n = 0;  // element counts (4 * N_all, 3 * N_all)
  Scratch filter;      // int32 [filter_n]
  int filter_n = -1, num_trackable = 0;
  Scratch zvals;       // float [z_n]  (set_*_z_values)
  int z_n = -1;
  void clear_cov() { cov_n = 0; rots_n = 0; scales_n = 0; }
};

}  // namespace gsicp

using namespace gsicp;

struct gsicp_gicp {
  Cloud src, tgt;
  double max_corr = (double)std::numeric_limits<float>::max();  // corr_dist_threshold_ (fgi:18)
  float knn_max = 0.5f;
  int k = 10;
  int max_iterations = 64;
  double rot_eps = 2e-3, trans_eps = 5e-4;
  int lm_max_iterations = 10;
  double lm_init_lambda_factor = 1e-9, lm_lambda = -1.0;
  bool converged = false;
  int nr_iterations = 0;
  float final_transformation[16];
  double final_hessian[36];
  cudaStream_t stream = 0;
  Scratch corr, sqd, mahal, partial, red_out, counter, staging_dev, nn_id, nn_d2;
  int corr_n = 0;
  double* h_red = nullptr;     // pinned [28]
  HostMailbox lin_box;         // linearize / error sums: [0, kRed) as doubles, [kRed] sequence word
  HostMailbox lm_box;          // LmResult of align_lm_kernel
  void* h_stage = nullptr;     // pinned staging for H2D conversions
  size_t h_stage_cap = 0;
  int shard_count = 1, shard_index = 0;
  gsicp_comm* comm = nullptr;    // in-library exchange over peer memory (gsicp_gicp_set_comm); replaces the callback
  bool src_partial = false;      // sharded covariances: this rank holds only its own source rotations / scales / covariances
  gsicp_allreduce_fn reduce = nullptr;
  void* reduce_user = nullptr;
  bool host_lm = false;          // gsicp_gicp_set_host_lm: host-driven LM loop (one launch + one spin-wait per phase)
  Scratch lm_partL, lm_partE, lm_barrier;
  int lm_max_blocks = 0;         // co-resident blocks of align_lm_kernel on this device
};

namespace {

int ensure_stage(gsicp_gicp* h, size_t bytes) {
  if (bytes <= h->h_stage_cap) return GSICP_OK;
  if (h->h_stage) cudaFreeHost(h->h_stage);
  h->h_stage = nullptr;
  h->h_stage_cap = 0;
  const size_t want = bytes + bytes / 2 + 4096;
  GSICP_CUDA(cudaMallocHost(&h->h_stage, want));
  h->h_stage_cap = want;
  return GSICP_OK;
}

// Host array -> device through the pinned staging buffer.  Large arrays (the 300k-point target and its 2.1M rotation /
// scale floats arrive as pageable numpy memory at every tracking keyframe) are cut into 1 MB chunks: each is copied (or
// converted double -> float) into the staging buffer and its DMA is issued at once, so the transfer of chunk k overlaps
// the host-side copy of chunk k+1.
struct HostSeg {
  void* dst;         // device
  const void* src;   // host
  size_t count;      // elements (float out)
  bool src_is_f64;
};

int upload_staged(gsicp_gicp* h, const HostSeg* segs, int nseg) {
  size_t total = 0;
  for (int i = 0; i < nseg; i++) total += segs[i].count * sizeof(float);
  if (total == 0) return GSICP_OK;
  if (int e = ensure_stage(h, total)) return e;
  GSICP_CUDA(cudaStreamSynchronize(h->stream));  // the previous transfer out of the staging buffer has finished
  constexpr size_t kChunkElems = (1u << 20) / sizeof(float);
  struct Chunk { int seg; size_t first, count, stage_off; };
  std::vector<Chunk> chunks;
  size_t off = 0;
  for (int i = 0; i < nseg; i++) {
    for (size_t f = 0; f < segs[i].count; f += kChunkElems) {
      const size_t c = std::min(kChunkElems, segs[i].count - f);
      chunks.push_back({i, f, c, off});
      off += c;
    }
  }
  float* stage = (float*)h->h_stage;
  // Copying chunk k+1 overlaps the DMA of chunk k.  A team of 6 copy threads was measured slower end to end (1.98-2.67 ms
  // vs 1.51 ms per keyframe: thread start-up and contention with the two Python threads cost more than the extra copy
  // bandwidth buys).
  for (const Chunk& ch : chunks) {
    const HostSeg& sg = segs[ch.seg];
    float* out = stage + ch.stage_off;
    if (sg.src_is_f64) {
      const double* in = (const double*)sg.src + ch.first;
      for (size_t k = 0; k < ch.count; k++) out[k] = (float)in[k];
    } else {
      std::memcpy(out, (const float*)sg.src + ch.first, ch.count * sizeof(float));
    }
    GSICP_CUDA(cudaMemcpyAsync((float*)sg.dst + ch.first, out, ch.count * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  }
  return GSICP_OK;
}

void shard_range(const gsicp_gicp* h, int n, int& begin, int& end) {
  if (h->shard_count <= 1) {
    begin = 0;
    end = n;
    return;
  }
  const long long per = ((long long)n + h->shard_count - 1) / h->shard_count;
  begin = (int)std::min<long long>(n, per * h->shard_index);
  end = (int)std::min<long long>(n, per * (h->shard_index + 1));
}

int set_cloud(gsicp_gicp* h, Cloud& c, const void* xyz, int n, int is_f32, bool device_src) {
  if (n < 0 || (n > 0 && !xyz)) {
    set_error("set_input: bad arguments");
    return GSICP_EINVAL;
  }
  c.n = n;
  c.grid_stale = true;
  c.clear_cov();
  if (n == 0) return GSICP_OK;
  if (int e = c.xyz.ensure((size_t)n * 3 * sizeof(float))) return e;
  const size_t cnt = (size_t)n * 3;
  if (device_src) {
    GSICP_CUDA(cudaMemcpyAsync(c.xyz.ptr, xyz, cnt * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
  } else if (is_f32 && cnt * sizeof(float) <= (64u << 10)) {
    // small pageable source: the runtime stages it itself — no extra host copy, no stream sync
    GSICP_CUDA(cudaMemcpyAsync(c.xyz.ptr, xyz, cnt * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  } else {
    // large pageable float32 source (a 300k-point map is 3.6 MB), or float64 from numpy (main.cpp:37-45 eigen2pcl casts
    // to float): staged through pinned memory — several times faster than the runtime's own pageable path
    // (measured: 190 vs 580 frames/s end to end)
    HostSeg sg{c.xyz.ptr, xyz, cnt, !is_f32};
    if (int e = upload_staged(h, &sg, 1)) return e;
  }
  c.grid_stale = true;
  return GSICP_OK;
}

// The search grid of a cloud is built when a search first needs it: the tracker's source cloud is searched once (its own
// k-NN), and the compacted cloud a *_with_filter call leaves behind is searched only if it later serves as a target.
int ensure_grid(gsicp_gicp* h, Cloud& c) {
  if (!c.grid_stale) return GSICP_OK;
  ProfScope ps(kProfGridBuild, h->stream);
  if (int e = c.grid.build(c.xyz.as<float>(), c.n, h->stream)) return e;
  c.grid_stale = false;
  return GSICP_OK;
}

int set_filter(gsicp_gicp* h, Cloud& c, int num_trackable, const int32_t* filter, int n, bool device_src = false) {
  if (n < 0 || num_trackable < 0 || (n > 0 && !filter)) {
    set_error("set_filter: bad arguments");
    return GSICP_EINVAL;
  }
  c.num_trackable = num_trackable;
  c.filter_n = n;
  if (n == 0) return GSICP_OK;
  if (int e = c.filter.ensure((size_t)n * 4)) return e;
  // pageable source: the runtime stages it before returning, so no pinned staging buffer (and no sync) is needed
  GSICP_CUDA(cudaMemcpyAsync(c.filter.ptr, filter, (size_t)n * 4, device_src ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                             h->stream));
  return GSICP_OK;
}

// covariances of a cloud; with_filter: keep only trackable points afterwards (fgi:588-706 / 710-825)
int compute_covariances(gsicp_gicp* h, Cloud& c, bool with_filter, bool clamp, bool withz = false) {
  const int n = c.n;
  if (n == 0) {
    fprintf(stderr, "no point cloud\n");
    return GSICP_OK;
  }
  if (withz && c.z_n != n) {  // the reference indexes z_values[i] unchecked (fgi:534)
    set_error("z values (%d) do not match the cloud size %d", c.z_n, n);
    return GSICP_ESTATE;
  }
  if (h->k > 32 || h->k < 1) {
    set_error("correspondence randomness k=%d unsupported (1..32)", h->k);
    return GSICP_EINVAL;
  }
  int slots = n;
  const int32_t* d_filter = nullptr;
  if (with_filter) {
    if (c.filter_n < 0) {  // no filter ever set: every point is trackable (the reference would read out of bounds)
      if (int e = c.filter.ensure((size_t)n * 4)) return e;
      GSICP_LAUNCH(identity_filter_kernel, (n + 255) / 256, 256, 0, h->stream, n, c.filter.as<int32_t>());
      c.num_trackable = n;
    } else if (c.filter_n != n) {
      set_error("filter length %d does not match the cloud size %d", c.filter_n, n);
      return GSICP_ESTATE;
    }
    slots = c.num_trackable;
    d_filter = c.filter.as<int32_t>();
  }
  if (int e = c.cov.ensure((size_t)(slots > 0 ? slots : 1) * 6 * sizeof(double))) return e;
  if (int e = c.rots.ensure((size_t)n * 4 * sizeof(float))) return e;
  if (int e = c.scales.ensure((size_t)n * 3 * sizeof(float))) return e;
  if (with_filter)
    if (int e = c.xyz_alt.ensure((size_t)(slots > 0 ? slots : 1) * 3 * sizeof(float))) return e;
  CovArgs a;
  a.n = n; a.k = h->k; a.knn_max = h->knn_max; a.clamp = clamp ? 1 : 0;
  a.filter = d_filter; a.xyz = c.xyz.as<float>(); a.rots = c.rots.as<float>(); a.scales = c.scales.as<float>();
  a.cov = c.cov.as<double>(); a.new_xyz = with_filter ? c.xyz_alt.as<float>() : nullptr;
  a.z = withz ? c.zvals.as<float>() : nullptr;
  // the k-NN + SVD of the SOURCE cloud is sharded over the ranks of the exchange group (each rank needs only the
  // covariances of the source range it linearises); target covariances are needed everywhere and stay replicated
  const bool sharded = h->comm && h->shard_count > 1 && (&c == &h->src);
  a.slot_begin = 0; a.slot_end = slots; a.idx_begin = 0; a.idx_end = n;
  if (sharded) {
    shard_range(h, slots, a.slot_begin, a.slot_end);
    shard_range(h, n, a.idx_begin, a.idx_end);
    GSICP_CUDA(cudaMemsetAsync(c.rots.ptr, 0, (size_t)n * 4 * sizeof(float), h->stream));  // entries of other ranks: zero (merged on demand)
    GSICP_CUDA(cudaMemsetAsync(c.scales.ptr, 0, (size_t)n * 3 * sizeof(float), h->stream));
    GSICP_CUDA(cudaMemsetAsync(c.cov.ptr, 0, (size_t)(slots > 0 ? slots : 1) * 6 * sizeof(double), h->stream));
  }
  if (&c == &h->src) h->src_partial = sharded;
  const int grid = (n + 127) / 128;
  if (int e = ensure_grid(h, c)) return e;
  {
  ProfScope ps(kProfCovariance, h->stream);
  const int K = h->k <= 10 ? 10 : (h->k <= 20 ? 20 : 32);
  if (int e = h->nn_id.ensure((size_t)n * K * 4)) return e;
  if (int e = h->nn_d2.ensure((size_t)n * K * 4)) return e;
  uint32_t* nid = h->nn_id.as<uint32_t>();
  float* nd2 = h->nn_d2.as<float>();
  const int kgrid = (int)(((size_t)n * 32 + 127) / 128);
  if (K == 10) {
    GSICP_LAUNCH(knn_kernel<10>, kgrid, 128, 0, h->stream, c.grid.view(), n, h->k, c.xyz.as<float>(), nid, nd2, a);
    GSICP_LAUNCH(covariance_kernel<10>, grid, 128, 0, h->stream, a, nid, nd2);
  } else if (K == 20) {
    GSICP_LAUNCH(knn_kernel<20>, kgrid, 128, 0, h->stream, c.grid.view(), n, h->k, c.xyz.as<float>(), nid, nd2, a);
    GSICP_LAUNCH(covariance_kernel<20>, grid, 128, 0, h->stream, a, nid, nd2);
  } else {
    GSICP_LAUNCH(knn_kernel<32>, kgrid, 128, 0, h->stream, c.grid.view(), n, h->k, c.xyz.as<float>(), nid, nd2, a);
    GSICP_LAUNCH(covariance_kernel<32>, grid, 128, 0, h->stream, a, nid, nd2);
  }
  }
  if (sharded && with_filter)  // the compacted cloud itself is complete on every rank
    GSICP_LAUNCH(compact_xyz_kernel, (n + 255) / 256, 256, 0, h->stream, n, d_filter, c.xyz.as<float>(), c.xyz_alt.as<float>());
  GSICP_CUDA(cudaGetLastError());
  c.rots_n = 4 * n;
  c.scales_n = 3 * n;
  c.cov_n = slots;
  if (with_filter) {
    std::swap(c.xyz, c.xyz_alt);
    c.n = slots;
    c.filter_n = -1;  // consumed; a new cloud needs a new filter
    c.grid_stale = true;
  }
  return GSICP_OK;
}

int covs_from_qs(gsicp_gicp* h, Cloud& c, const float* rots, const float* scales, int n, bool device_src = false) {
  if (n < 0 || (n > 0 && (!rots || !scales))) return GSICP_EINVAL;
  if (int e = c.cov.ensure((size_t)(n > 0 ? n : 1) * 6 * sizeof(double))) return e;
  if (int e = c.rots.ensure((size_t)(n > 0 ? n : 1) * 4 * sizeof(float))) return e;
  if (int e = c.scales.ensure((size_t)(n > 0 ? n : 1) * 3 * sizeof(float))) return e;
  if (n > 0 && device_src) {
    GSICP_CUDA(cudaMemcpyAsync(c.rots.ptr, rots, (size_t)n * 4 * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
    GSICP_CUDA(cudaMemcpyAsync(c.scales.ptr, scales, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
    GSICP_LAUNCH(cov_from_qs_kernel, (n + 255) / 256, 256, 0, h->stream, n, c.rots.as<float>(), c.scales.as<float>(),
                 c.cov.as<double>());
    GSICP_CUDA(cudaGetLastError());
  } else if (n > 0) {
    if ((size_t)n * 7 * sizeof(float) <= (64u << 10)) {
      GSICP_CUDA(cudaMemcpyAsync(c.rots.ptr, rots, (size_t)n * 4 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
      GSICP_CUDA(cudaMemcpyAsync(c.scales.ptr, scales, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    } else {  // pinned staging for large arrays (see set_cloud)
      HostSeg sg[2] = {{c.rots.ptr, rots, (size_t)n * 4, false}, {c.scales.ptr, scales, (size_t)n * 3, false}};
      if (int e = upload_staged(h, sg, 2)) return e;
    }
    GSICP_LAUNCH(cov_from_qs_kernel, (n + 255) / 256, 256, 0, h->stream, n, c.rots.as<float>(), c.scales.as<float>(),
                 c.cov.as<double>());
    GSICP_CUDA(cudaGetLastError());
  }
  c.rots_n = 4 * n;
  c.scales_n = 3 * n;
  c.cov_n = n;
  return GSICP_OK;
}

int ensure_lin_buffers(gsicp_gicp* h) {
  const int n = h->src.n;
  const int blocks = (n + kLinBlock - 1) / kLinBlock + 1;
  if (int e = h->corr.ensure((size_t)(n + 1) * 4)) return e;
  if (int e = h->sqd.ensure((size_t)(n + 1) * 4)) return e;
  if (int e = h->mahal.ensure((size_t)(n + 1) * 6 * sizeof(double))) return e;
  if (int e = h->partial.ensure((size_t)blocks * kRed * sizeof(double))) return e;
  if (int e = h->red_out.ensure(kRed * sizeof(double))) return e;
  if (!h->counter.ptr) {
    if (int e = h->counter.ensure(sizeof(unsigned int))) return e;
    GSICP_CUDA(cudaMemsetAsync(h->counter.ptr, 0, sizeof(unsigned int), h->stream));
  }
  if (!h->h_red) GSICP_CUDA(cudaMallocHost(&h->h_red, kRed * sizeof(double)));
  return h->lin_box.ensure((kRed + 1) * sizeof(unsigned long long));
}

// ---- sum-merge of a sharded array over the exchange group (getters of sharded runs; not on the LM path) ----
// Every rank stages its copy (entries it does not own are zero) in the upper half of its exchange heap; after a barrier
// each rank adds the world's copies in rank order.  Exact: every entry is non-zero on at most one rank.
template <typename T>
__global__ void comm_stage_kernel(size_t count, const T* __restrict__ in, T* __restrict__ stage) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) stage[i] = in[i];
}
// correspondences: owned range [begin, end) as index + 1 (so that "unmatched" -1 becomes 0), others 0
__global__ void comm_stage_corr_kernel(int n, int begin, int end, const int32_t* __restrict__ corr, int32_t* __restrict__ stage) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) stage[i] = (i >= begin && i < end) ? corr[i] + 1 : 0;
}
template <typename T>
__global__ void comm_sum_kernel(CommView c, size_t heap_off, size_t count, T* __restrict__ out, T bias) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  T r = 0;
  for (int k = 0; k < c.world; k++) {
    const volatile T* src = reinterpret_cast<const volatile T*>(c.seg[k] + kCommHeapOff + heap_off);
    r += src[i];
  }
  out[i] = r + bias;
}

template <typename T>
int comm_sum_merge(gsicp_gicp* h, T* d_buf, size_t count, T bias = 0, const int32_t* corr_src = nullptr, int cb = 0, int ce = 0) {
  gsicp_comm* c = h->comm;
  const size_t half = (c->heap_bytes() / 2) & ~size_t(255);
  if (count * sizeof(T) > half) {
    set_error("exchange heap too small for a merge of %zu bytes (half heap = %zu)", count * sizeof(T), half);
    return GSICP_ENOMEM;
  }
  T* stage = reinterpret_cast<T*>(c->local + kCommHeapOff + half);
  const int blocks = (int)((count + 255) / 256);
  if (corr_src)
    GSICP_LAUNCH(comm_stage_corr_kernel, blocks, 256, 0, h->stream, (int)count, cb, ce, corr_src, reinterpret_cast<int32_t*>(stage));
  else
    GSICP_LAUNCH(comm_stage_kernel<T>, blocks, 256, 0, h->stream, count, d_buf, stage);
  if (int e = comm_stream_barrier(c, h->stream)) return e;
  GSICP_LAUNCH(comm_sum_kernel<T>, blocks, 256, 0, h->stream, c->view(), half, count, d_buf, bias);
  if (int e = comm_stream_barrier(c, h->stream)) return e;  // the staging area may be reused
  GSICP_CUDA(cudaGetLastError());
  return GSICP_OK;
}

// Sharded covariances leave every rank with its own rotations / scales / covariances only: complete them on demand.
int complete_source_exports(gsicp_gicp* h) {
  if (!h->src_partial || !h->comm) return GSICP_OK;
  if (h->src.rots_n > 0)
    if (int e = comm_sum_merge<float>(h, h->src.rots.as<float>(), (size_t)h->src.rots_n)) return e;
  if (h->src.scales_n > 0)
    if (int e = comm_sum_merge<float>(h, h->src.scales.as<float>(), (size_t)h->src.scales_n)) return e;
  if (h->src.cov_n > 0)
    if (int e = comm_sum_merge<double>(h, h->src.cov.as<double>(), (size_t)h->src.cov_n * 6)) return e;
  h->src_partial = false;
  return GSICP_OK;
}

// Exchange sequence numbers (comm.cuh): consecutive exchanges must alternate the parity slot.  A host-driven kernel
// consumes exactly one number; the persistent LM kernel consumes a data-dependent count from a reserved range, so a
// stream barrier re-aligns the ranks before and after it (every rank has finished reading the slots of the previous
// launch before any rank writes them again).
int comm_take_seq(gsicp_gicp* h, unsigned long long reserve, unsigned long long* first) {
  gsicp_comm* c = h->comm;
  if (c->lm_resync || reserve > 1) {
    if (int e = comm_stream_barrier(c, h->stream)) return e;
    c->lm_resync = false;
  }
  *first = c->lm_seq + 1;
  c->lm_seq += reserve;
  if (reserve > 1) c->lm_resync = true;
  return GSICP_OK;
}

// The n sums of a linearize / error launch into h->h_red.  Single-GPU and in-kernel-exchange runs read them from the mailbox
// the kernel published into; a sharded run with the all-reduce callback sums red_out over the ranks and copies it back.
int collect_sums(gsicp_gicp* h, int n, bool direct, unsigned long long seq) {
  if (h->shard_count > 1 && h->reduce) {
    const int rc = h->reduce(h->reduce_user, h->red_out.as<double>(), n, (void*)h->stream);
    if (rc != 0) {
      set_error("all-reduce callback failed (%d)", rc);
      return GSICP_ECUDA;
    }
  }
  if (direct) {
    GSICP_CUDA(cudaGetLastError());
    if (int e = h->lin_box.wait(kRed, seq, h->stream, "GICP reduction")) return e;
    std::memcpy(h->h_red, h->lin_box.host, n * sizeof(double));
  } else {
    GSICP_CUDA(cudaMemcpyAsync(h->h_red, h->red_out.ptr, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    GSICP_CUDA(cudaStreamSynchronize(h->stream));
  }
  return GSICP_OK;
}

// fgi:296-352.  H may be null (error only).
int run_linearize(gsicp_gicp* h, const Iso& x, double H[6][6], double b[6], double* err) {
  if (int e = ensure_lin_buffers(h)) return e;
  if (h->corr_n != h->src.n) {
    // sharded runs leave the other ranks' entries untouched: start from "unmatched"
    GSICP_CUDA(cudaMemsetAsync(h->corr.ptr, 0xff, (size_t)(h->src.n + 1) * 4, h->stream));
    GSICP_CUDA(cudaMemsetAsync(h->sqd.ptr, 0, (size_t)(h->src.n + 1) * 4, h->stream));
    h->corr_n = h->src.n;
  }
  int begin, end;
  shard_range(h, h->src.n, begin, end);
  LinArgs a;
  a.begin = begin; a.end = end;
  a.max_corr_sq = h->max_corr * h->max_corr;
  a.src_xyz = h->src.xyz.as<float>(); a.src_cov = h->src.cov.as<double>();
  a.tgt_xyz = h->tgt.xyz.as<float>(); a.tgt_cov = h->tgt.cov.as<double>();
  a.corr = h->corr.as<int32_t>(); a.sqd = h->sqd.as<float>(); a.mahal = h->mahal.as<double>();
  a.partial = h->partial.as<double>(); a.out = h->red_out.as<double>(); a.counter = h->counter.as<unsigned int>();
  const bool xchg = h->shard_count > 1 && h->comm;  // in-kernel exchange: the published sums are already global
  const bool direct = h->shard_count <= 1 || xchg;   // publish straight into mapped host memory
  a.host_out = direct ? (double*)h->lin_box.dev : nullptr;
  a.host_seq = direct ? (volatile unsigned long long*)(h->lin_box.dev + kRed) : nullptr;
  a.seq = ++h->lin_box.seq;
  a.comm = CommView();
  a.xseq = 0;
  if (xchg) {
    a.comm = h->comm->view();
    if (int e = comm_take_seq(h, 1, &a.xseq)) return e;
  }
  int blocks = (end - begin + kLinBlock - 1) / kLinBlock;
  if (blocks < 1) blocks = 1;
  if (end > begin)
    if (int e = ensure_grid(h, h->tgt)) return e;
  { ProfScope ps(kProfLinearize, h->stream);
  if (end > begin) {
    const int nn_blocks = (int)(((size_t)(end - begin) * 32 + 127) / 128);
    GSICP_LAUNCH(correspond_kernel, nn_blocks, 128, 0, h->stream, h->tgt.grid.view(), make_pose(x), begin, end, a.max_corr_sq,
                 a.src_xyz, a.corr, a.sqd);
  }
  GSICP_LAUNCH(linearize_kernel, blocks, kLinBlock, 0, h->stream, make_pose(x), a); }
  if (int e = collect_sums(h, kRed, direct, a.seq)) return e;
  if (H && b) {
    int o = 0;
    for (int r = 0; r < 6; r++)
      for (int c = r; c < 6; c++) {
        H[r][c] = h->h_red[o];
        H[c][r] = h->h_red[o];
        o++;
      }
    for (int r = 0; r < 6; r++) b[r] = h->h_red[21 + r];
  }
  *err = h->h_red[27];
  return GSICP_OK;
}

int run_error(gsicp_gicp* h, const Iso& x, double* err) {  // fgi:355-378
  if (int e = ensure_lin_buffers(h)) return e;
  int begin, end;
  shard_range(h, h->src.n, begin, end);
  ErrArgs a;
  a.begin = begin; a.end = end;
  a.src_xyz = h->src.xyz.as<float>(); a.tgt_xyz = h->tgt.xyz.as<float>();
  a.corr = h->corr.as<int32_t>(); a.mahal = h->mahal.as<double>();
  a.partial = h->partial.as<double>(); a.out = h->red_out.as<double>(); a.counter = h->counter.as<unsigned int>();
  const bool xchg = h->shard_count > 1 && h->comm;
  const bool direct = h->shard_count <= 1 || xchg;
  a.host_out = direct ? (double*)h->lin_box.dev : nullptr;
  a.host_seq = direct ? (volatile unsigned long long*)(h->lin_box.dev + kRed) : nullptr;
  a.seq = ++h->lin_box.seq;
  a.comm = CommView();
  a.xseq = 0;
  if (xchg) {
    a.comm = h->comm->view();
    if (int e = comm_take_seq(h, 1, &a.xseq)) return e;
  }
  int blocks = (end - begin + kLinBlock - 1) / kLinBlock;
  if (blocks < 1) blocks = 1;
  { ProfScope ps(kProfError, h->stream);
  GSICP_LAUNCH(error_kernel, blocks, kLinBlock, 0, h->stream, make_pose(x), a); }
  if (int e = collect_sums(h, 1, direct, a.seq)) return e;
  *err = h->h_red[0];
  return GSICP_OK;
}

bool is_converged(const gsicp_gicp* h, const Iso& delta) { return lm_is_converged(h->rot_eps, h->trans_eps, delta); }

// lsq:125-173.  Returns 1 = step taken / converged, 0 = failed ("lm not converged"), <0 = error.
int step_lm(gsicp_gicp* h, Iso& x0, Iso& delta) {
  double H[6][6], b[6], y0;
  if (int e = run_linearize(h, x0, H, b, &y0)) return e;
  if (h->lm_lambda < 0.0) {
    double mx = 0.0;
    for (int i = 0; i < 6; i++) mx = std::max(mx, std::fabs(H[i][i]));
    h->lm_lambda = h->lm_init_lambda_factor * mx;
  }
  double nu = 2.0;
  for (int it = 0; it < h->lm_max_iterations; it++) {
    double d[6];
    Iso xi;
    lm_trial(H, b, h->lm_lambda, x0, d, delta, xi);
    double yi;
    if (int e = run_error(h, xi, &yi)) return e;
    double dot = 0.0;
    for (int i = 0; i < 6; i++) dot += d[i] * (h->lm_lambda * d[i] - b[i]);
    const double rho = (y0 - yi) / dot;
    if (rho < 0) {
      if (is_converged(h, delta)) return 1;
      h->lm_lambda = nu * h->lm_lambda;
      nu = 2 * nu;
      continue;
    }
    x0 = xi;
    h->lm_lambda = h->lm_lambda * std::max(1.0 / 3.0, 1 - std::pow(2 * rho - 1, 3));
    for (int i = 0; i < 6; i++)
      for (int j = 0; j < 6; j++) h->final_hessian[6 * i + j] = H[i][j];
    return 1;
  }
  return 0;
}

// The whole LM loop of one align() on the device (align_lm_kernel): one launch, one spin-wait.
// Returns the number of outer iterations (>= 1) or a negative error.
int run_align_device(gsicp_gicp* h, Iso& x0) {
  if (int e = ensure_lin_buffers(h)) return e;
  if (h->corr_n != h->src.n) {
    GSICP_CUDA(cudaMemsetAsync(h->corr.ptr, 0xff, (size_t)(h->src.n + 1) * 4, h->stream));
    GSICP_CUDA(cudaMemsetAsync(h->sqd.ptr, 0, (size_t)(h->src.n + 1) * 4, h->stream));
    h->corr_n = h->src.n;
  }
  if (int e = h->lm_box.ensure(sizeof(LmResult))) return e;
  if (h->lm_max_blocks == 0) {
    int dev = 0, sms = 0;
    GSICP_CUDA(cudaGetDevice(&dev));
    GSICP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    h->lm_max_blocks = sms > 0 ? sms : 1;  // one block per SM: always co-resident on an otherwise idle device
  }
  int begin, end;
  shard_range(h, h->src.n, begin, end);
  const int nchunks = (end - begin + kLmChunk - 1) / kLmChunk;
  int blocks = (nchunks + (kLmBlock / 32) - 1) / (kLmBlock / 32);
  blocks = std::max(1, std::min(blocks, h->lm_max_blocks));
  if (int e = h->lm_partL.ensure((size_t)h->lm_max_blocks * kRed * sizeof(double))) return e;
  if (int e = h->lm_partE.ensure((size_t)h->lm_max_blocks * 2 * sizeof(double))) return e;
  if (int e = h->lm_barrier.ensure(sizeof(unsigned int))) return e;
  GSICP_CUDA(cudaMemsetAsync(h->lm_barrier.ptr, 0, sizeof(unsigned int), h->stream));
  if (end > begin)
    if (int e = ensure_grid(h, h->tgt)) return e;
  LmArgs a = {};
  a.tgt = h->tgt.grid.view();
  a.begin = begin; a.end = end;
  a.max_corr_sq = h->max_corr * h->max_corr;
  a.src_xyz = h->src.xyz.as<float>(); a.src_cov = h->src.cov.as<double>();
  a.tgt_xyz = h->tgt.xyz.as<float>(); a.tgt_cov = h->tgt.cov.as<double>();
  a.corr = h->corr.as<int32_t>(); a.sqd = h->sqd.as<float>(); a.mahal = h->mahal.as<double>();
  a.partL = h->lm_partL.as<double>(); a.partE = h->lm_partE.as<double>();
  a.barrier = h->lm_barrier.as<unsigned int>();
  a.comm = CommView();
  a.xseq = 0;
  if (h->comm && h->shard_count > 1) {
    a.comm = h->comm->view();
    // an align runs at most max_iterations * (1 + lm_max_iterations) exchanges: reserve that many sequence numbers
    const unsigned long long bound = (unsigned long long)std::max(1, h->max_iterations) * (unsigned long long)(1 + std::max(1, h->lm_max_iterations));
    if (int e = comm_take_seq(h, bound + 1, &a.xseq)) return e;
  }
  a.max_iterations = h->max_iterations; a.lm_max_iterations = h->lm_max_iterations;
  a.rot_eps = h->rot_eps; a.trans_eps = h->trans_eps; a.init_lambda_factor = h->lm_init_lambda_factor;
  a.guess = x0;
  a.result = reinterpret_cast<LmResult*>(h->lm_box.dev);
  a.seq = ++h->lm_box.seq;
  static const int s_marks = [] { const char* e = getenv("GSICP_LM_MARKS"); return e ? atoi(e) : 0; }();
  a.marks = s_marks;
  {
    ProfScope ps(kProfLinearize, h->stream);  // slot "gicp_linearize": the whole device-resident LM loop
    GSICP_LAUNCH(align_lm_kernel, blocks, kLmBlock, 0, h->stream, a);
  }
  GSICP_CUDA(cudaGetLastError());
  static_assert(offsetof(LmResult, seq) % sizeof(unsigned long long) == 0, "LmResult::seq must be a mailbox word");
  if (int e = h->lm_box.wait(offsetof(LmResult, seq) / sizeof(unsigned long long), a.seq, h->stream, "align result")) return e;
  const LmResult r = *reinterpret_cast<const LmResult*>(h->lm_box.host);
  if (s_marks && r.n_marks > 1) {
    fprintf(stderr, "[lm marks] total %.1f us:", (double)(r.marks[r.n_marks - 1] - r.marks[0]) * 1e-3);
    for (int i = 1; i < r.n_marks; i++) fprintf(stderr, " %.1f", (double)(r.marks[i] - r.marks[i - 1]) * 1e-3);
    fprintf(stderr, "\n");
  }
  for (int i = 0; i < 3; i++) {
    for (int j = 0; j < 3; j++) x0.R[i][j] = r.R[3 * i + j];
    x0.t[i] = r.t[i];
  }
  h->lm_lambda = r.lambda;
  h->converged = r.converged != 0;
  h->nr_iterations = r.iterations - 1;
  // final_hessian_ is only assigned by an accepted step (lsq:169); it keeps its previous value otherwise
  if (r.n_err > 0) {
    bool any = false;
    for (int i = 0; i < 36; i++) any = any || (r.H[i] != 0.0);
    if (any) std::memcpy(h->final_hessian, r.H, sizeof(double) * 36);
  }
  if (r.status == 1) fprintf(stderr, "lm not converged!!\n");
  if (r.status == 3) {
    set_error("align: the device-side grid barrier timed out");
    return GSICP_ECUDA;
  }
  return r.iterations;
}

int copy_out(gsicp_gicp* h, const Scratch& s, size_t bytes, void* out) {
  if (bytes == 0) return GSICP_OK;
  if (!out) return GSICP_EINVAL;
  GSICP_CUDA(cudaMemcpyAsync(out, s.ptr, bytes, cudaMemcpyDeviceToHost, h->stream));
  GSICP_CUDA(cudaStreamSynchronize(h->stream));
  return GSICP_OK;
}

int copy_cov_out(gsicp_gicp* h, const Cloud& c, double* out) {
  if (c.cov_n == 0) return GSICP_OK;
  std::vector<double> tmp((size_t)c.cov_n * 6);
  if (int e = copy_out(h, c.cov, tmp.size() * sizeof(double), tmp.data())) return e;
  for (int i = 0; i < c.cov_n; i++) {
    const double* s = &tmp[(size_t)i * 6];
    double* o = out + (size_t)i * 9;
    o[0] = s[0]; o[1] = s[1]; o[2] = s[2]; o[3] = s[1]; o[4] = s[3]; o[5] = s[4]; o[6] = s[2]; o[7] = s[4]; o[8] = s[5];
  }
  return GSICP_OK;
}

}  // namespace

extern "C" {

gsicp_gicp* gsicp_gicp_create(void) {
  gsicp_gicp* h = new gsicp_gicp();
  for (int i = 0; i < 16; i++) h->final_transformation[i] = (i % 5 == 0) ? 1.f : 0.f;
  for (int i = 0; i < 36; i++) h->final_hessian[i] = (i % 7 == 0) ? 1.0 : 0.0;
  if (cudaFree(nullptr) != cudaSuccess) {  // initialises the context
    set_error("gsicp_gicp_create: no usable CUDA device (%s)", cudaGetErrorString(cudaGetLastError()));
    delete h;
    return nullptr;
  }
  return h;
}

void gsicp_gicp_destroy(gsicp_gicp* h) {
  if (!h) return;
  auto fr = [](Scratch& s) {
    if (s.ptr) cudaFree(s.ptr);
    s.ptr = nullptr;
  };
  for (Cloud* c : {&h->src, &h->tgt}) {
    fr(c->xyz); fr(c->xyz_alt); fr(c->cov); fr(c->rots); fr(c->scales); fr(c->filter); fr(c->zvals);
    fr(c->grid.meta_buf); fr(c->grid.bbox_buf); fr(c->grid.cell_start); fr(c->grid.cursor); fr(c->grid.cell_of_pt);
    fr(c->grid.pts); fr(c->grid.cub_tmp);
  }
  fr(h->corr); fr(h->sqd); fr(h->mahal); fr(h->partial); fr(h->red_out); fr(h->counter); fr(h->staging_dev); fr(h->nn_id); fr(h->nn_d2);
  fr(h->lm_partL); fr(h->lm_partE); fr(h->lm_barrier);
  h->lm_box.release();
  h->lin_box.release();
  if (h->h_red) cudaFreeHost(h->h_red);
  if (h->h_stage) cudaFreeHost(h->h_stage);
  delete h;
}

#define H_CHECK(h) \
  if (!(h)) { set_error("null handle"); return GSICP_EINVAL; }

int gsicp_gicp_set_max_correspondence_distance(gsicp_gicp* h, double d) { H_CHECK(h); h->max_corr = d; return GSICP_OK; }
int gsicp_gicp_set_max_knn_distance(gsicp_gicp* h, double d) { H_CHECK(h); h->knn_max = (float)d; return GSICP_OK; }
int gsicp_gicp_set_correspondence_randomness(gsicp_gicp* h, int k) { H_CHECK(h); h->k = k; return GSICP_OK; }
int gsicp_gicp_set_max_iterations(gsicp_gicp* h, int n) { H_CHECK(h); h->max_iterations = n; return GSICP_OK; }
int gsicp_gicp_set_stream(gsicp_gicp* h, void* s) { H_CHECK(h); h->stream = (cudaStream_t)s; return GSICP_OK; }
int gsicp_gicp_set_host_lm(gsicp_gicp* h, int on) { H_CHECK(h); h->host_lm = on != 0; return GSICP_OK; }

int gsicp_gicp_set_input_source(gsicp_gicp* h, const void* xyz, int n, int is_f32) {
  H_CHECK(h);
  h->corr_n = -1;
  return set_cloud(h, h->src, xyz, n, is_f32, false);
}
int gsicp_gicp_set_input_target(gsicp_gicp* h, const void* xyz, int n, int is_f32) {
  H_CHECK(h);
  return set_cloud(h, h->tgt, xyz, n, is_f32, false);
}
int gsicp_gicp_set_input_source_device(gsicp_gicp* h, const float* d_xyz, int n) {
  H_CHECK(h);
  h->corr_n = -1;
  return set_cloud(h, h->src, d_xyz, n, 1, true);
}
int gsicp_gicp_set_input_target_device(gsicp_gicp* h, const float* d_xyz, int n) {
  H_CHECK(h);
  return set_cloud(h, h->tgt, d_xyz, n, 1, true);
}
int gsicp_gicp_set_source_filter(gsicp_gicp* h, int nt, const int32_t* f, int n) { H_CHECK(h); return set_filter(h, h->src, nt, f, n); }
int gsicp_gicp_set_target_filter(gsicp_gicp* h, int nt, const int32_t* f, int n) { H_CHECK(h); return set_filter(h, h->tgt, nt, f, n); }
int gsicp_gicp_set_source_filter_device(gsicp_gicp* h, int nt, const int32_t* f, int n) { H_CHECK(h); return set_filter(h, h->src, nt, f, n, true); }
int gsicp_gicp_set_target_filter_device(gsicp_gicp* h, int nt, const int32_t* f, int n) { H_CHECK(h); return set_filter(h, h->tgt, nt, f, n, true); }

int gsicp_gicp_calculate_target_covariance_with_filter(gsicp_gicp* h) { H_CHECK(h); return compute_covariances(h, h->tgt, true, false); }
int gsicp_gicp_calculate_source_covariance(gsicp_gicp* h) { H_CHECK(h); return compute_covariances(h, h->src, false, true); }
int gsicp_gicp_calculate_target_covariance(gsicp_gicp* h) { H_CHECK(h); return compute_covariances(h, h->tgt, false, true); }
int gsicp_gicp_calculate_target_covariance_withz(gsicp_gicp* h) { H_CHECK(h); return compute_covariances(h, h->tgt, false, true, true); }

static int set_z_values(gsicp_gicp* h, Cloud& c, const float* z, int n) {
  if (n < 0 || (n > 0 && !z)) return GSICP_EINVAL;
  if (int e = c.zvals.ensure((size_t)(n > 0 ? n : 1) * sizeof(float))) return e;
  if (n > 0) GSICP_CUDA(cudaMemcpyAsync(c.zvals.ptr, z, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  c.z_n = n;
  return GSICP_OK;
}
int gsicp_gicp_set_source_z_values(gsicp_gicp* h, const float* z, int n) { H_CHECK(h); return set_z_values(h, h->src, z, n); }
int gsicp_gicp_set_target_z_values(gsicp_gicp* h, const float* z, int n) { H_CHECK(h); return set_z_values(h, h->tgt, z, n); }

int gsicp_gicp_swap_source_and_target(gsicp_gicp* h) {
  H_CHECK(h);
  std::swap(h->src, h->tgt);  // clouds, grids, covariances, rotations, scales (fgi:66-76)
  std::swap(h->src.filter, h->tgt.filter);  // filters and z values are not swapped by the reference
  std::swap(h->src.filter_n, h->tgt.filter_n);
  std::swap(h->src.num_trackable, h->tgt.num_trackable);
  std::swap(h->src.zvals, h->tgt.zvals);
  std::swap(h->src.z_n, h->tgt.z_n);
  h->corr_n = -1;
  return GSICP_OK;
}

int gsicp_gicp_set_source_covariances_fromqs(gsicp_gicp* h, const float* r, const float* s, int n) { H_CHECK(h); return covs_from_qs(h, h->src, r, s, n); }
int gsicp_gicp_set_target_covariances_fromqs(gsicp_gicp* h, const float* r, const float* s, int n) { H_CHECK(h); return covs_from_qs(h, h->tgt, r, s, n); }
int gsicp_gicp_set_source_covariances_fromqs_device(gsicp_gicp* h, const float* r, const float* s, int n) { H_CHECK(h); return covs_from_qs(h, h->src, r, s, n, true); }
int gsicp_gicp_set_target_covariances_fromqs_device(gsicp_gicp* h, const float* r, const float* s, int n) { H_CHECK(h); return covs_from_qs(h, h->tgt, r, s, n, true); }

int gsicp_gicp_align(gsicp_gicp* h, const float guess[16], float out[16]) {
  H_CHECK(h);
  if (!guess || !out) return GSICP_EINVAL;
  // pcl::Registration::align: initCompute fails without a target
  if (h->tgt.n == 0 || h->src.n == 0) {
    set_error("align: %s cloud is empty", h->tgt.n == 0 ? "target" : "source");
    return GSICP_ESTATE;
  }
  h->converged = false;
  // fgi:225-240: lazily compute missing covariances
  if (h->src.cov_n != h->src.n) {
    if (int e = compute_covariances(h, h->src, true, false)) return e;
    h->corr_n = -1;
  }
  if (h->tgt.cov_n != h->tgt.n) {
    if (int e = compute_covariances(h, h->tgt, false, true)) return e;
  }
  if (h->src.n == 0) {
    set_error("align: no trackable source points");
    return GSICP_ESTATE;
  }
  Iso x0;
  for (int i = 0; i < 3; i++) {
    for (int j = 0; j < 3; j++) x0.R[i][j] = (double)guess[4 * i + j];
    x0.t[i] = (double)guess[4 * i + 3];
  }
  h->lm_lambda = -1.0;
  int iters = 0;
  int lb, le;
  shard_range(h, h->src.n, lb, le);
  // The persistent kernel (one block per SM) wins where launch / wait latency dominates; above kLmPersistentMax points per
  // rank the phases are throughput-bound and the full-occupancy kernels of the host-driven loop are faster
  // (in a sharded run their last block exchanges through the peers' segments as well: no host-side collective either way).
  if (!h->host_lm && (h->shard_count <= 1 || h->comm) && (le - lb) <= kLmPersistentMax) {
    // device-resident LM loop: one persistent kernel, zero host round trips inside the loop
    if (h->lm_box.host) std::memset(reinterpret_cast<LmResult*>(h->lm_box.host)->H, 0, sizeof(LmResult::H));
    iters = run_align_device(h, x0);
    if (iters < 0) return iters;
  } else {
    for (int i = 0; i < h->max_iterations && !h->converged; i++) {
      h->nr_iterations = i;
      iters = i + 1;
      Iso delta;
      const int rc = step_lm(h, x0, delta);
      if (rc < 0) return rc;
      if (rc == 0) {
        fprintf(stderr, "lm not converged!!\n");
        break;
      }
      h->converged = is_converged(h, delta);
    }
  }
  for (int i = 0; i < 3; i++) {
    for (int j = 0; j < 3; j++) h->final_transformation[4 * i + j] = (float)x0.R[i][j];
    h->final_transformation[4 * i + 3] = (float)x0.t[i];
  }
  h->final_transformation[12] = 0.f; h->final_transformation[13] = 0.f; h->final_transformation[14] = 0.f;
  h->final_transformation[15] = 1.f;
  std::memcpy(out, h->final_transformation, sizeof(float) * 16);
  return iters;
}

int gsicp_gicp_has_converged(gsicp_gicp* h) { H_CHECK(h); return h->converged ? 1 : 0; }
int gsicp_gicp_get_final_hessian(gsicp_gicp* h, double out[36]) { H_CHECK(h); std::memcpy(out, h->final_hessian, sizeof(double) * 36); return GSICP_OK; }

int gsicp_gicp_source_size(gsicp_gicp* h) { H_CHECK(h); return h->src.n; }
int gsicp_gicp_target_size(gsicp_gicp* h) { H_CHECK(h); return h->tgt.n; }
int gsicp_gicp_source_rotationsq_size(gsicp_gicp* h) { H_CHECK(h); return h->src.rots_n; }
int gsicp_gicp_target_rotationsq_size(gsicp_gicp* h) { H_CHECK(h); return h->tgt.rots_n; }
int gsicp_gicp_source_scales_size(gsicp_gicp* h) { H_CHECK(h); return h->src.scales_n; }
int gsicp_gicp_target_scales_size(gsicp_gicp* h) { H_CHECK(h); return h->tgt.scales_n; }
int gsicp_gicp_get_source_rotationsq(gsicp_gicp* h, float* o) { H_CHECK(h); if (int e = complete_source_exports(h)) return e; return copy_out(h, h->src.rots, (size_t)h->src.rots_n * 4, o); }
int gsicp_gicp_get_target_rotationsq(gsicp_gicp* h, float* o) { H_CHECK(h); return copy_out(h, h->tgt.rots, (size_t)h->tgt.rots_n * 4, o); }
int gsicp_gicp_get_source_scales(gsicp_gicp* h, float* o) { H_CHECK(h); if (int e = complete_source_exports(h)) return e; return copy_out(h, h->src.scales, (size_t)h->src.scales_n * 4, o); }
int gsicp_gicp_get_target_scales(gsicp_gicp* h, float* o) { H_CHECK(h); return copy_out(h, h->tgt.scales, (size_t)h->tgt.scales_n * 4, o); }
int gsicp_gicp_get_source_covariances(gsicp_gicp* h, double* o) { H_CHECK(h); if (int e = complete_source_exports(h)) return e; return copy_cov_out(h, h->src, o); }
int gsicp_gicp_get_target_covariances(gsicp_gicp* h, double* o) { H_CHECK(h); return copy_cov_out(h, h->tgt, o); }

int gsicp_gicp_get_source_correspondence(gsicp_gicp* h, int32_t* corr, float* sq_dist) {
  H_CHECK(h);
  if (h->corr_n != h->src.n) {
    // reference prints "source and correspondence size mismatch" and returns stale vectors (fast_gicp.hpp:82-87)
    fprintf(stderr, "source and correspondence size mismatch. Did you change src after align()?\n");
    set_error("no correspondences for the current source cloud");
    return GSICP_ESTATE;
  }
  if (h->src.n == 0) return GSICP_OK;
  if (!corr || !sq_dist) return GSICP_EINVAL;
  if (h->shard_count > 1 && h->comm) {  // merge the ranks' ranges through the exchange heap (SURVEY §8e: only when asked for)
    int begin, end;
    shard_range(h, h->src.n, begin, end);
    if (int e = comm_sum_merge<int32_t>(h, h->corr.as<int32_t>(), (size_t)h->src.n, -1, h->corr.as<int32_t>(), begin, end)) return e;
    // squared distances: zero outside the own range, then summed
    GSICP_CUDA(cudaMemsetAsync(h->sqd.as<float>(), 0, (size_t)begin * 4, h->stream));
    if (end < h->src.n) GSICP_CUDA(cudaMemsetAsync(h->sqd.as<float>() + end, 0, (size_t)(h->src.n - end) * 4, h->stream));
    if (int e = comm_sum_merge<float>(h, h->sqd.as<float>(), (size_t)h->src.n)) return e;
  } else if (h->shard_count > 1 && h->reduce) {  // merge the ranks' ranges (SURVEY §8e: gathered only when asked for)
    const int n = h->src.n;
    int begin, end;
    shard_range(h, n, begin, end);
    if (int e = h->staging_dev.ensure((size_t)n * 2 * sizeof(double))) return e;
    double* buf = h->staging_dev.as<double>();
    GSICP_LAUNCH(corr_pack_kernel, (n + 255) / 256, 256, 0, h->stream, n, begin, end, h->corr.as<int32_t>(), h->sqd.as<float>(), buf);
    if (h->reduce(h->reduce_user, buf, 2 * n, (void*)h->stream) != 0) {
      set_error("all-reduce callback failed");
      return GSICP_ECUDA;
    }
    GSICP_LAUNCH(corr_unpack_kernel, (n + 255) / 256, 256, 0, h->stream, n, buf, h->corr.as<int32_t>(), h->sqd.as<float>());
    GSICP_CUDA(cudaGetLastError());
  }
  GSICP_CUDA(cudaMemcpyAsync(corr, h->corr.ptr, (size_t)h->src.n * 4, cudaMemcpyDeviceToHost, h->stream));
  GSICP_CUDA(cudaMemcpyAsync(sq_dist, h->sqd.ptr, (size_t)h->src.n * 4, cudaMemcpyDeviceToHost, h->stream));
  GSICP_CUDA(cudaStreamSynchronize(h->stream));
  return GSICP_OK;
}

int gsicp_gicp_get_fitness_score(gsicp_gicp* h, double max_range, double* out) {
  H_CHECK(h);
  if (!out) return GSICP_EINVAL;
  *out = std::numeric_limits<double>::max();
  const int n = h->src.n;
  if (n == 0 || h->tgt.n == 0) return GSICP_OK;
  if (int e = ensure_grid(h, h->tgt)) return e;
  if (int e = h->nn_id.ensure((size_t)n * 4)) return e;
  if (int e = h->nn_d2.ensure((size_t)n * 4)) return e;
  if (int e = h->red_out.ensure(kRed * sizeof(double))) return e;
  Iso x;
  for (int i = 0; i < 3; i++) {
    for (int j = 0; j < 3; j++) x.R[i][j] = (double)h->final_transformation[4 * i + j];
    x.t[i] = (double)h->final_transformation[4 * i + 3];
  }
  const int nn_blocks = (int)(((size_t)n * 32 + 127) / 128);
  GSICP_LAUNCH(correspond_kernel, nn_blocks, 128, 0, h->stream, h->tgt.grid.view(), make_pose(x), 0, n,
               std::numeric_limits<double>::infinity(), h->src.xyz.as<float>(), h->nn_id.as<int32_t>(), h->nn_d2.as<float>());
  GSICP_LAUNCH(fitness_kernel, 1, 1024, 0, h->stream, n, h->nn_d2.as<float>(), max_range, h->red_out.as<double>());
  double r[2] = {0, 0};
  GSICP_CUDA(cudaMemcpyAsync(r, h->red_out.ptr, sizeof(r), cudaMemcpyDeviceToHost, h->stream));
  GSICP_CUDA(cudaStreamSynchronize(h->stream));
  if (r[1] > 0.0) *out = r[0] / r[1];
  return GSICP_OK;
}

static int pose_from16(const double p[16], Iso& x) {
  if (!p) return GSICP_EINVAL;
  for (int i = 0; i < 3; i++) {
    for (int j = 0; j < 3; j++) x.R[i][j] = p[4 * i + j];
    x.t[i] = p[4 * i + 3];
  }
  return GSICP_OK;
}

static int ready_for_linearize(gsicp_gicp* h) {
  if (h->src.n == 0 || h->tgt.n == 0 || h->src.cov_n != h->src.n || h->tgt.cov_n != h->tgt.n) {
    set_error("linearize: clouds or covariances missing (src %d/%d, tgt %d/%d)", h->src.cov_n, h->src.n, h->tgt.cov_n,
              h->tgt.n);
    return GSICP_ESTATE;
  }
  return GSICP_OK;
}

int gsicp_gicp_linearize(gsicp_gicp* h, const double pose[16], double Hout[36], double b[6], double* err) {
  H_CHECK(h);
  Iso x;
  if (int e = pose_from16(pose, x)) return e;
  if (int e = ready_for_linearize(h)) return e;
  double H[6][6], bb[6], er;
  if (int e = run_linearize(h, x, H, bb, &er)) return e;
  if (Hout) std::memcpy(Hout, H, sizeof(H));
  if (b) std::memcpy(b, bb, sizeof(bb));
  if (err) *err = er;
  return GSICP_OK;
}

int gsicp_gicp_compute_error(gsicp_gicp* h, const double pose[16], double* err) {
  H_CHECK(h);
  Iso x;
  if (int e = pose_from16(pose, x)) return e;
  if (int e = ready_for_linearize(h)) return e;
  if (h->corr_n != h->src.n) {
    set_error("compute_error: run linearize first");
    return GSICP_ESTATE;
  }
  return run_error(h, x, err);
}

int gsicp_gicp_set_shard(gsicp_gicp* h, int count, int index, gsicp_allreduce_fn reduce, void* user) {
  H_CHECK(h);
  if (count < 1 || index < 0 || index >= count) return GSICP_EINVAL;
  h->shard_count = count; h->shard_index = index; h->reduce = reduce; h->reduce_user = user;
  h->corr_n = -1;
  return GSICP_OK;
}

int gsicp_gicp_set_comm(gsicp_gicp* h, gsicp_comm* comm) {
  H_CHECK(h);
  if (comm && !comm->connected) {
    set_error("gsicp_gicp_set_comm: the exchange group is not connected");
    return GSICP_ESTATE;
  }
  h->comm = comm;
  h->shard_count = comm ? comm->world : 1;
  h->shard_index = comm ? comm->rank : 0;
  h->reduce = nullptr;
  h->reduce_user = nullptr;
  h->corr_n = -1;
  h->src.clear_cov();
  return GSICP_OK;
}

}  // extern "C"

// Test hook (tests/test_exchange_gpu.py): load every kernel of this translation unit and of comm.cu now.  With CUDA's
// default lazy module loading the FIRST launch of a kernel may synchronise the context; two exchange ranks emulated inside
// one process / one context would then deadlock on a peer that spins on a flag.  One process per GPU (the real layout) never
// needs this.
namespace gsicp { int comm_preload_kernels(); }
extern "C" int gsicp_test_preload_kernels(void) {
  cudaFuncAttributes fa;
  const void* fns[] = {(const void*)knn_kernel<10>, (const void*)knn_kernel<20>, (const void*)knn_kernel<32>,
                       (const void*)covariance_kernel<10>, (const void*)covariance_kernel<20>, (const void*)covariance_kernel<32>,
                       (const void*)compact_xyz_kernel, (const void*)cov_from_qs_kernel, (const void*)correspond_kernel,
                       (const void*)fitness_kernel, (const void*)corr_pack_kernel, (const void*)corr_unpack_kernel,
                       (const void*)linearize_kernel, (const void*)error_kernel, (const void*)align_lm_kernel,
                       (const void*)f64_to_f32_kernel, (const void*)identity_filter_kernel,
                       (const void*)comm_stage_kernel<int32_t>, (const void*)comm_stage_kernel<float>, (const void*)comm_stage_kernel<double>,
                       (const void*)comm_stage_corr_kernel,
                       (const void*)comm_sum_kernel<int32_t>, (const void*)comm_sum_kernel<float>, (const void*)comm_sum_kernel<double>};
  for (const void* f : fns) GSICP_CUDA(cudaFuncGetAttributes(&fa, f));
  return gsicp::comm_preload_kernels();
}
