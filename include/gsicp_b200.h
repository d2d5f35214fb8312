/*
 * gsicp_b200.h — C ABI of libgsicp_b200.so (sm_100a).
 *
 * Drop-in boundary for the two data-parallel hot paths of GS-ICP-SLAM
 * (SURVEY.md §8b).  Every entry point cites the reference interface it
 * replaces (paths relative to the reference checkout):
 *
 *   DGR = submodules/diff-gaussian-rasterization
 *   FG  = submodules/fast_gicp
 *   SK  = submodules/simple-knn
 *
 * Conventions: plain pointers and sizes only (no torch / Eigen / pybind types);
 * all `const float*` / `float*` arguments named d_* are DEVICE pointers on the
 * current CUDA device; `stream` is a cudaStream_t passed as void*; functions
 * return >= 0 on success and a negative GSICP_E* code on failure (no exceptions
 * cross the ABI); gsicp_last_error() returns a thread-local message.
 */
#ifndef GSICP_B200_H
#define GSICP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSICP_OK 0
#define GSICP_EINVAL (-1)   /* bad argument (reference: AT_ERROR / std::invalid_argument) */
#define GSICP_ECUDA (-2)    /* CUDA runtime error */
#define GSICP_ENOMEM (-3)   /* workspace callback returned NULL */
#define GSICP_ESTATE (-4)   /* call sequence error (e.g. align() without target) */

const char* gsicp_last_error(void);
/* "sm_100a" + build flags; lets host code verify the native library is the one loaded. */
const char* gsicp_build_info(void);
/* Number of kernel launches issued by this library since process start (bench.py: gpu_launches). */
uint64_t gsicp_launch_count(void);

/* Per-kernel device timing for the roofline leg of bench.py: when enabled, the hot kernels are bracketed by
 * CUDA events on their launching stream.  Kernels are indexed 0..gsicp_prof_count()-1 (gsicp_prof_name). */
void gsicp_prof_enable(int on);
void gsicp_prof_reset(void);
int gsicp_prof_count(void);
const char* gsicp_prof_name(int k);
int gsicp_prof_read(int k, double* total_ms, long* count);

/* ------------------------------------------------------------------------------------------
 * Rasterizer (mapper hot path)
 * ------------------------------------------------------------------------------------------ */

/* Resizable-buffer callback: must return a device pointer to at least `bytes` bytes (128-B
 * aligned) that stays valid until the matching backward call.  Mirrors the reference's
 * std::function<char*(size_t)> resize functors (DGR/rasterize_points.cu:27-33). */
typedef void* (*gsicp_alloc_fn)(size_t bytes, void* user);

/* Inputs of one rasterization — the argument list of CudaRasterizer::Rasterizer::forward
 * (DGR/cuda_rasterizer/rasterizer.h:35-60, rasterizer_impl.cu:201-227). */
typedef struct gsicp_raster_args {
  int P;                 /* number of Gaussians */
  int D;                 /* active SH degree (0..3) */
  int M;                 /* SH coefficients stored per Gaussian (0 if colours precomputed) */
  int width, height;
  float tan_fovx, tan_fovy;
  float scale_modifier;
  int prefiltered;       /* reference: trap if a "prefiltered" point is culled (auxiliary.h:161-165) */
  int debug;             /* synchronise + check after every stage (auxiliary.h:171-178) */
  const float* d_background;     /* [3] */
  const float* d_means3D;        /* [P,3] */
  const float* d_shs;            /* [P,M,3] or NULL */
  const float* d_colors_precomp; /* [P,3]  or NULL */
  const float* d_opacities;      /* [P] */
  const float* d_scales;         /* [P,3] or NULL */
  const float* d_rotations;      /* [P,4] (x,y,z,w), used UN-normalised (forward.cu:134-138) */
  const float* d_cov3D_precomp;  /* [P,6] or NULL */
  const float* d_viewmatrix;     /* [16] row-major storage of the transposed world->view */
  const float* d_projmatrix;     /* [16] likewise, full projection */
  const float* d_campos;         /* [3] */
  /* Tile sharding for multi-GPU (SURVEY §8e): this rank renders tiles t with
   * t % tile_shard_count == tile_shard_index.  (1, 0) = all tiles. */
  int tile_shard_count, tile_shard_index;
} gsicp_raster_args;

/* Forward.  Replaces RasterizeGaussiansCUDA -> Rasterizer::forward
 * (DGR/rasterize_points.cu:35-121, rasterizer_impl.cu:201-347).
 * Outputs (device, caller-allocated, zero-initialised like torch::full(...,0)):
 *   d_out_color [3,H,W], d_out_depth [1,H,W], d_radii int32[P], d_is_used uint8[P].
 * The three callbacks size the state kept for backward (private layout, see DESIGN.md).
 * Returns num_rendered (tile instances, >= 0) or a negative error. */
int gsicp_raster_forward(const gsicp_raster_args* args,
                         float* d_out_color, float* d_out_depth,
                         int32_t* d_radii, uint8_t* d_is_used,
                         gsicp_alloc_fn geom_alloc, gsicp_alloc_fn binning_alloc,
                         gsicp_alloc_fn image_alloc, void* user, void* stream);

/* Backward.  Replaces RasterizeGaussiansBackwardCUDA -> Rasterizer::backward
 * (DGR/rasterize_points.cu:123-206, rasterizer_impl.cu:351-454).
 * Gradient outputs are caller-allocated device buffers which need NOT be initialised — every element is written,
 * zeros for Gaussians outside the view (the reference zero-fills ten P-sized tensors first, rasterize_points.cu:158-167):
 * dL_dmeans2D[P,3], dL_dcolors[P,3], dL_dopacity[P], dL_dmeans3D[P,3], dL_dcov3D[P,6], dL_dsh[P,M,3], dL_dscales[P,3],
 * dL_drotations[P,4].  The per-Gaussian scratch of the reference (dL_dconic[P,6] + dL_ddepths[P]) lives in the geometry
 * buffer of the forward pass: d_work is ignored (may be NULL) and gsicp_raster_backward_work_bytes() returns 0; both
 * are kept so that round-1 callers keep linking. */
size_t gsicp_raster_backward_work_bytes(int P);
/* Multi-GPU (tile-sharded rendering, SURVEY §8e): with an exchange group set (gsicp_raster_set_comm) and
 * tile_shard_count > 1, the 12 render moments of the visible Gaussians are summed over the ranks between the
 * render-backward and the per-Gaussian-backward kernels; every rank then returns the FULL parameter gradients. */
int gsicp_raster_backward(const gsicp_raster_args* args, int num_rendered,
                          const int32_t* d_radii,
                          const void* d_geom, const void* d_binning, const void* d_image,
                          const float* d_dL_dout_color, const float* d_dL_dout_depth,
                          float* d_dL_dmeans2D, float* d_dL_dcolors, float* d_dL_dopacity,
                          float* d_dL_dmeans3D, float* d_dL_dcov3D, float* d_dL_dsh,
                          float* d_dL_dscales, float* d_dL_drotations,
                          void* d_work, void* stream);

/* Introspection of the saved state for the parity tests (point_list bit-exactness):
 * copies the sorted tile-instance list (uint32[num_rendered]) and the per-tile ranges
 * (uint32[2*tiles]) out of the binning / image buffers.  Device -> device. */
int gsicp_raster_export_binning(const gsicp_raster_args* args, int num_rendered,
                                const void* d_binning, const void* d_image,
                                uint32_t* d_point_list, uint32_t* d_ranges, void* stream);

/* Replaces markVisible / checkFrustum (DGR/rasterize_points.cu:208-227,
 * rasterizer_impl.cu:54-66): present[i] = view-space z > 0.2. */
int gsicp_mark_visible(int P, const float* d_means3D, const float* d_viewmatrix,
                       const float* d_projmatrix, uint8_t* d_present, void* stream);

/* ------------------------------------------------------------------------------------------
 * simple-knn
 * ------------------------------------------------------------------------------------------ */

/* Replaces distCUDA2 -> SimpleKNN::knn (SK/spatial.cu:15-25, SK/simple_knn.cu:185-221):
 * d_out[i] = mean of the 3 smallest squared distances from point i to the other points. */
int gsicp_dist2(int P, const float* d_points, float* d_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * GICP tracker (pygicp.FastGICP).  Host pointers unless named d_*.
 * ------------------------------------------------------------------------------------------ */

typedef struct gsicp_gicp gsicp_gicp;

/* FastGICP::FastGICP() defaults (FG/include/fast_gicp/gicp/impl/fast_gicp_impl.hpp:9-33,
 * lsq_registration_impl.hpp:9-22): k=10, knn_max=0.5, NORMALIZED_ELLIPSE, LM, 64 iters. */
gsicp_gicp* gsicp_gicp_create(void);
void gsicp_gicp_destroy(gsicp_gicp*);

int gsicp_gicp_set_max_correspondence_distance(gsicp_gicp*, double d);  /* main.cpp:204 */
int gsicp_gicp_set_max_knn_distance(gsicp_gicp*, double d);             /* main.cpp:205, fgi:51-53 */
int gsicp_gicp_set_correspondence_randomness(gsicp_gicp*, int k);       /* main.cpp:203 */
int gsicp_gicp_set_max_iterations(gsicp_gicp*, int n);                  /* pcl::Registration::setMaximumIterations */

/* set_input_source / set_input_target (main.cpp:167-168 + eigen2pcl :37-45, fgi:94-105,120-130):
 * xyz is row-major (N,3) float64 on the host (is_f32 != 0: float32); stored as fp32; covariances
 * and rotations/scales of that cloud are cleared; the NN grid over the cloud is rebuilt. */
int gsicp_gicp_set_input_source(gsicp_gicp*, const void* xyz, int n, int is_f32);
int gsicp_gicp_set_input_target(gsicp_gicp*, const void* xyz, int n, int is_f32);
/* Zero-copy variants ("next" row N1): device fp32 (N,3). */
int gsicp_gicp_set_input_source_device(gsicp_gicp*, const float* d_xyz, int n);
int gsicp_gicp_set_input_target_device(gsicp_gicp*, const float* d_xyz, int n);

/* set_source_filter / set_target_filter (main.cpp:254-261, fgi:189-202). */
int gsicp_gicp_set_source_filter(gsicp_gicp*, int num_trackable, const int32_t* filter, int n);
int gsicp_gicp_set_target_filter(gsicp_gicp*, int num_trackable, const int32_t* filter, int n);

/* calculate_target_covariance_with_filter (fgi:157-166,710-825),
 * calculate_source_covariance / calculate_target_covariance (fgi:107-117,132-142,382-479). */
int gsicp_gicp_calculate_target_covariance_with_filter(gsicp_gicp*);
int gsicp_gicp_calculate_source_covariance(gsicp_gicp*);
int gsicp_gicp_calculate_target_covariance(gsicp_gicp*);
/* main.cpp:228 / fgi:145-154,481-583: as calculate_target_covariance, exported scales divided by max(1, z^1.5 * 2);
 * GSICP_ESTATE unless set_target_z_values supplied one z per target point. */
int gsicp_gicp_calculate_target_covariance_withz(gsicp_gicp*);
int gsicp_gicp_set_source_z_values(gsicp_gicp*, const float* z, int n);     /* main.cpp:246-249, fgi:182-186 */
int gsicp_gicp_set_target_z_values(gsicp_gicp*, const float* z, int n);     /* main.cpp:250-253, fgi:205-209 */
/* main.cpp:169 / fgi:66-76: exchanges clouds, search structures, covariances, rotations and scales (filters and z values
 * stay where they are, as in the reference) and drops the correspondences. */
int gsicp_gicp_swap_source_and_target(gsicp_gicp*);

/* set_source/target_covariances_fromqs (main.cpp:234-245, fgi:828-902). n = number of points. */
int gsicp_gicp_set_source_covariances_fromqs(gsicp_gicp*, const float* rots_xyzw, const float* scales, int n);
int gsicp_gicp_set_target_covariances_fromqs(gsicp_gicp*, const float* rots_xyzw, const float* scales, int n);
/* Zero-copy variants ("next" row N3): device fp32 arrays. */
int gsicp_gicp_set_source_covariances_fromqs_device(gsicp_gicp*, const float* d_rots_xyzw, const float* d_scales, int n);
int gsicp_gicp_set_target_covariances_fromqs_device(gsicp_gicp*, const float* d_rots_xyzw, const float* d_scales, int n);

/* align (main.cpp:173-179; pcl::Registration::align -> fgi:225-240 -> lsq:53-78).
 * guess/out: row-major 4x4 float32.  Returns the number of LM outer iterations run. */
int gsicp_gicp_align(gsicp_gicp*, const float guess[16], float out[16]);
int gsicp_gicp_has_converged(gsicp_gicp*);
int gsicp_gicp_get_final_hessian(gsicp_gicp*, double out[36]);          /* lsq:44-46 */
/* main.cpp:172 -> pcl::Registration::getFitnessScore(max_range): mean squared NN distance of the source points, moved by
 * the final transformation, over those with squared distance <= max_range; DBL_MAX if there is none. */
int gsicp_gicp_get_fitness_score(gsicp_gicp*, double max_range, double* out);

/* Getters (main.cpp:206-233, fast_gicp.hpp:82-110). *_size return element counts. */
int gsicp_gicp_source_size(gsicp_gicp*);          /* input_->size() (after filtering: trackable) */
int gsicp_gicp_target_size(gsicp_gicp*);
int gsicp_gicp_source_rotationsq_size(gsicp_gicp*);
int gsicp_gicp_target_rotationsq_size(gsicp_gicp*);
int gsicp_gicp_source_scales_size(gsicp_gicp*);
int gsicp_gicp_target_scales_size(gsicp_gicp*);
int gsicp_gicp_get_source_rotationsq(gsicp_gicp*, float* out);
int gsicp_gicp_get_target_rotationsq(gsicp_gicp*, float* out);
int gsicp_gicp_get_source_scales(gsicp_gicp*, float* out);
int gsicp_gicp_get_target_scales(gsicp_gicp*, float* out);
/* main.cpp:230-233.  Sharded handles merge the ranks' ranges through the exchange group first (collective call). */
int gsicp_gicp_get_source_correspondence(gsicp_gicp*, int32_t* corr, float* sq_dist);
/* Test/diagnostic access: regularised 3x3 covariances as 9 doubles per point (row-major). */
int gsicp_gicp_get_source_covariances(gsicp_gicp*, double* out);
int gsicp_gicp_get_target_covariances(gsicp_gicp*, double* out);

/* One linearize at a given pose (LsqRegistration::evaluateCost, lsq:48-51): H row-major 6x6,
 * b[6]; returns error through *err.  Used by the parity tests and by bench.py's roofline leg. */
int gsicp_gicp_linearize(gsicp_gicp*, const double pose[16], double H[36], double b[6], double* err);
int gsicp_gicp_compute_error(gsicp_gicp*, const double pose[16], double* err);

/* ---- Multi-GPU exchange group (one process per GPU; replaces the survey sketch's gsicp_gicp_comm_init(ncclComm_t)) ----
 * Each rank allocates a symmetric device segment and exports it as a 64-byte CUDA IPC handle; after the application
 * has exchanged the handles (any channel: torch.distributed.all_gather_object in the Python host code), every rank
 * maps its peers' segments (NVLink peer access).  The kernels then exchange their partial sums by writing straight into
 * the peers' segments and polling sequence flags: no host hop and no second kernel per exchange.
 *   GICP:        source points (LM linearisation AND k-NN covariances) are sharded over the ranks; the 28-double normal
 *                equations / the 1-double error are exchanged inside the persistent LM kernel (fgi:296-378).
 *   rasterizer:  screen tiles are sharded; the per-Gaussian render moments accumulate in the segment and are all-reduced
 *                inside gsicp_raster_backward as a reduce-scatter + all-gather of P2P loads (rank r sums the world's rows of
 *                its slice of the table in rank order, every rank then copies each row from its owner).
 * heap_bytes: per-rank exchange heap (>= 96 bytes per Gaussian for the rasterizer: accumulators in the lower half, the reduced
 * slice / the staging of sharded getters in the upper half).  Every rank must issue the same exchanging calls in the same
 * order.  A barrier whose peer never arrives gives up after its poll budget; the next exchanging call then returns GSICP_ECUDA
 * ("a peer did not arrive") instead of continuing with partial sums. */
typedef struct gsicp_comm gsicp_comm;
int gsicp_comm_alloc(size_t heap_bytes, gsicp_comm** out, void* handle64);
int gsicp_comm_connect(gsicp_comm*, int world, int rank, const void* handles /* world x 64 bytes, rank order */);
void gsicp_comm_destroy(gsicp_comm*);
/* Test hook: all ranks of the group live in this process on one device (plain device pointers instead of IPC handles). */
int gsicp_comm_connect_local(gsicp_comm*, int world, int rank, gsicp_comm* const* group);
int gsicp_comm_world(const gsicp_comm*);
int gsicp_comm_rank(const gsicp_comm*);
int gsicp_comm_barrier(gsicp_comm*, void* stream);   /* stream-ordered barrier over the group */
/* The handle shards its source points over the group: shard count and index are the group's world and rank.
 * NULL: back to single-GPU. */
int gsicp_gicp_set_comm(gsicp_gicp*, gsicp_comm*);
/* Stores the group only; the tile shard still comes from gsicp_raster_args (tile_shard_count, tile_shard_index).
 * NULL: back to single-GPU. */
int gsicp_raster_set_comm(gsicp_comm*);

/* Stream on which the handle's kernels run (default: legacy default stream 0). */
int gsicp_gicp_set_stream(gsicp_gicp*, void* stream);
/* Test / A-B hook: 1 = drive the LM loop from the host (one launch + one wait per linearize / compute_error), 0 (default) =
 * the device-resident loop (one persistent kernel per align, lsq_registration_impl.hpp:53-173 on the GPU).  Same results.
 * In a sharded run the setting must be the same on every rank of the group: the two loops exchange differently. */
int gsicp_gicp_set_host_lm(gsicp_gicp* h, int on);

/* ---- fused mapping loss (SURVEY.md §8f row N2; the caller side of the rasterizer) ----------------------------------
 * Replaces utils/loss_utils.py:17-20 (l1_loss), :38-69 (ssim/_ssim) and their combination in mp_Mapper.py:225-242:
 *   loss = (1-lambda) * mean(|image - gt| where gt != 0) + lambda * (1 - mean(ssim(where(gt != 0, image, 0), gt)))
 *          + depth_weight * mean(|depth/d_max - gt_depth/d_max| where gt_depth != 0)
 * image, gt_image: [3,H,W] fp32; depth, gt_depth: [1,H,W] fp32 (device).  mask_by_depth != 0 applies
 * gt_image *= (gt_depth > 0) first (mp_Mapper.py:225-228).  d_loss receives the scalar, d_parts3 (optional) {L1, SSIM,
 * L1_depth}; d_ssim_map
 * (optional, [3,H,W]) receives the SSIM map.  d_work: gsicp_mapping_loss_work_bytes(H, W) bytes, kept for backward. */
size_t gsicp_mapping_loss_work_bytes(int H, int W);
int gsicp_mapping_loss_forward(int H, int W, const float* d_image, const float* d_depth, const float* d_gt_image,
                               const float* d_gt_depth, float lambda_dssim, float depth_weight, float d_max,
                               int mask_by_depth, float* d_loss, float* d_parts3, float* d_ssim_map, void* d_work,
                               void* stream);
/* d_grad_loss: device scalar dL/dloss (NULL = 1).  Writes d_grad_image [3,H,W] and d_grad_depth [1,H,W]. */
int gsicp_mapping_loss_backward(int H, int W, const float* d_image, const float* d_depth, const float* d_gt_image,
                                const float* d_gt_depth, float lambda_dssim, float depth_weight, float d_max,
                                int mask_by_depth, const float* d_grad_loss, const void* d_work, float* d_grad_image,
                                float* d_grad_depth, void* stream);

/* ---- Mapper bookkeeping on the device (SURVEY.md §8f row N3; scene/gaussian_model.py) ----
 * gsicp_adam_step: torch.optim.Adam(..., eps=1e-15).step() for up to 8 parameter tensors in ONE launch
 *   (gaussian_model.py:214-225 builds six groups with their own lr; mp_Mapper.py:248 steps them).  Host arrays of device
 *   pointers; counts in elements; `step` is the 1-based step number after the increment, like Adam's state["step"].
 *   The hyper-parameters are doubles: (1 - beta) is formed in double and rounded to float once, as PyTorch does.
 * gsicp_table_compact: boolean-mask row selection (prune_points / _prune_optimizer, gaussian_model.py:409-446) of n_arrays
 *   row-major arrays sharing one mask: dst[k][j] = src[k][i] for the j-th kept row i.  Returns the kept-row count (>= 0) or
 *   a negative error; dst buffers must hold `rows` rows.
 * gsicp_trackable_target: get_trackable_gaussians_tensor (gaussian_model.py:205-215): rows with sigmoid(opacity) > th and
 *   trackable != 0, compacted as (xyz, normalised rotation xyzw, exp(scaling)) into device buffers of P rows; returns the
 *   count.  The outputs go to gsicp_gicp_set_input_target_device / set_target_covariances_fromqs_device without a D2H copy. */
int gsicp_adam_step(int n_tensors, float* const* d_params, const float* const* d_grads, float* const* d_exp_avg,
                    float* const* d_exp_avg_sq, const size_t* counts, const float* lrs, int step, double beta1, double beta2,
                    double eps, void* stream);
long long gsicp_table_compact(int rows, const uint8_t* d_keep, int n_arrays, const void* const* d_src, void* const* d_dst,
                              const int* row_bytes, void* stream);
long long gsicp_trackable_target(int P, const float* d_xyz, const float* d_rotation_raw, const float* d_scaling_raw,
                                 const float* d_opacity_raw, const uint8_t* d_trackable, float opacity_th, float* d_out_xyz,
                                 float* d_out_rot, float* d_out_scale, void* stream);

/* ---- Tracker front-end on the device (SURVEY.md §8f row N1; mp_Tracker.py:394-431, 229, 256-274, 374-392) ----
 * gsicp_frontend_cloud: set_downsample_filter + downsample_and_make_pointcloud2: depth uint16 [H,W] and rgb uint8 [H,W,3]
 *   (device) -> camera-frame points [n,3], colours [n,3] (/255), z [n] of the sampled pixels with depth != 0 in raster
 *   order, the 1-based trackable filter [n] pygicp's set_source_filter takes (0 = z > depth_trunc) and the indices of the
 *   trackable points [n_trackable].  Output buffers hold gsicp_frontend_max_points(W, H, step) rows.
 * gsicp_frontend_keyframe: points to the world frame (R p - R T with R, T as mp_Tracker.py:224-229 forms them) and
 *   q_cam (x) rots (quaternion_multiply, xyzw); d_rots may be NULL.
 * gsicp_frontend_not_overlapped: eliminate_overlapped2 + the filter update (mp_Tracker.py:267-269): trackable indices whose
 *   squared NN distance exceeds the threshold, compacted. */
int gsicp_frontend_max_points(int W, int H, int step);
int gsicp_frontend_cloud(const uint16_t* d_depth, const uint8_t* d_rgb, int W, int H, int step, float fx, float fy, float cx,
                         float cy, float depth_scale, float depth_trunc, float* d_points, float* d_colors, float* d_z,
                         int32_t* d_filter, int32_t* d_trackable, int* n_points, int* n_trackable, void* stream);
int gsicp_frontend_keyframe(int n, const float* d_points_cam, const float* d_rots, const float R[9], const float T[3],
                            const float q_xyzw[4], float* d_points_world, float* d_rots_world, void* stream);
int gsicp_frontend_not_overlapped(int n_trackable, const float* d_sq_dist, float threshold, const int32_t* d_trackable,
                                  int32_t* d_out, int* n_out, void* stream);
/* Device-resident filters for the zero-copy tracker path (N1): like gsicp_gicp_set_source/target_filter with device pointers. */
int gsicp_gicp_set_source_filter_device(gsicp_gicp*, int num_trackable, const int32_t* d_filter, int n);
int gsicp_gicp_set_target_filter_device(gsicp_gicp*, int num_trackable, const int32_t* d_filter, int n);

#ifdef __cplusplus
}
#endif
#endif /* GSICP_B200_H */
