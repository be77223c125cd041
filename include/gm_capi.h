/* gm_capi.h — C-ABI of the B200-native geometric_mapping per-scan hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / PCL / Eigen / ROS types.
 * Each entry point replaces one reference seam (file:line relative to the reference repo
 * wangqiaoli/geometric_mapping); INTEGRATION.md shows the binding the reference's
 * src/geometric_mapping.cpp:cloud_cb would add.
 *
 * Conventions
 *   - Every call returns gm_status (0 = ok).  Nothing throws across the ABI.
 *   - A gm_ctx owns all device buffers for scans of up to max_points; no allocation per scan.
 *     A ctx is not thread-safe and is bound to the CUDA device current at gm_create().
 *   - Points are pcl::PointXYZ-compatible: 4 floats {x,y,z,pad}, 16-byte stride.
 *     Normals are pcl::Normal-compatible: 8 floats {nx,ny,nz,0, curvature,0,0,0}, 32-byte stride.
 *   - Calls are asynchronous on the ctx stream; gm_download_* / gm_get_* synchronise that stream.
 *   - There is NO CPU fallback: without a CUDA device gm_create() fails with GM_ERR_NO_DEVICE.
 */
#ifndef GM_CAPI_H
#define GM_CAPI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define GM_API __attribute__((visibility("default")))
#else
#define GM_API
#endif

typedef int32_t gm_status;
enum {
  GM_OK = 0,
  GM_ERR_INVALID_ARG = 1,
  GM_ERR_NO_DEVICE = 2,       /* no CUDA device / driver: the product has no CPU path            */
  GM_ERR_CUDA = 3,            /* a CUDA call failed; gm_last_error() has the text                */
  GM_ERR_CAPACITY = 4,        /* n > max_points or H > max_hypotheses                            */
  GM_ERR_STAGE_ORDER = 5,     /* a stage was called before the stage that produces its input     */
  GM_WARN_VOXEL_OVERFLOW = 6, /* pcl::VoxelGrid overflow rule: output = input, unchanged (A.5)   */
  GM_ERR_NN_INDEX_RANGE = 7,  /* reference quirk B.3: nn index >= compacted size (normals->at()
                                 would throw at src/tunnel_processing.cpp:247)                   */
  GM_ERR_INTERNAL = 8,        /* device-side consistency check failed (look-back spin bound)     */
  GM_ERR_NO_MODEL = 9         /* every RANSAC hypothesis was degenerate                          */
};

/* Mirror of class Parameters (include/geometric_mapping/paramHandler.hpp:26-36; ROS keys at
 * src/paramHandler.cpp:13,19,25,31,37,43,49,61) plus the builder-defined RANSAC / polyline
 * fields for the stages the reference only stubs (src/tunnel_processing.cpp:149-154). */
typedef struct gm_params {
  double boxFilterBound;    /* "boxFilterBound"     default 5.0  */
  double voxelGridLeafSize; /* "voxelGridLeafSize"  default 0.1  (field leafSize) */
  double neighborRadius;    /* "neighborRadius"     default 0.03 */
  double weightingFactor;   /* "weightingFactor"    default 0.2  */
  int32_t displayCloud;     /* default 1 */
  int32_t displayNormals;   /* default 1 */
  int32_t displayCenterAxis;/* default 1 */
  int32_t usePCLViz;        /* default 0; accepted and ignored (GUI, out of scope) */
  /* --- input semantics --- */
  int32_t is_dense;         /* default 1: pcl::CropBox keeps NaN points of a dense cloud (A.1) */
  int32_t nn_index_mode;    /* 0 = reference-faithful (1-NN indexes the PRE-compaction cloud,
                               quirk B.3), 1 = fixed (post-compaction index) */
  /* --- builder-defined RANSAC --- */
  double ransacThreshold;   /* tau, default 0.05 m */
  double cylinderRadiusMin; /* default 0.5  */
  double cylinderRadiusMax; /* default 10.0 */
  int32_t refitIterations;  /* Gauss-Newton steps of the cylinder refit, default 5 */
  int32_t maxSlices;        /* polyline capacity, default 256 */
  double sliceLength;       /* polyline slice length along the center axis, default 1.0 m */
  /* --- reference quirks as switches (SURVEY App. B / 8f.2): 0 = reference-faithful (default), 1 = "fixed" --- */
  int32_t weight_mode;      /* getLocalFrame weights: 0 = exp((curv + 0.001/wf)^2), grows with curvature (B.2,
                               src/tunnel_processing.cpp:106); 1 = exp(-(curv/wf)^2) (builder-defined) */
  int32_t arrow_mode;       /* normal arrows: 0 = end point is the normal vector itself (B.4, :247-249);
                               1 = end = centroid + normal.  Read by the host shims; see gm_markers_normals_mode */
} gm_params;

typedef struct gm_ctx gm_ctx;

/* Sizes produced by the stages (all int32; -1 = stage not run). */
typedef struct gm_counts {
  int32_t n_input;   /* points uploaded                                   */
  int32_t n_cropped; /* M  after chopCloud                                */
  int32_t n_valid;   /* M' after NaN-normal compaction                    */
  int32_t n_voxels;  /* V                                                 */
  int32_t n_cells;   /* occupied neighbour-grid cells (diagnostic)        */
  int32_t voxel_overflow; /* 1 if the VoxelGrid overflow rule fired       */
  int32_t nn_out_of_range;/* count of 1-NN indices >= n_valid (quirk B.3) */
  int32_t device_error;   /* non-zero = internal device-side check failed */
} gm_counts;

/* Eigen frame of getLocalFrame: vals ascending; vecs[r*3+k] = component r of eigenvector k,
 * so the center axis (src/geometric_mapping.cpp:91-92, eigenVecs.col(0)) is vecs[0],vecs[3],vecs[6]. */
typedef struct gm_frame {
  float vals[3];
  float vecs[9];
  float scatter[9]; /* the 3x3 "normal intensity" matrix, row-major */
} gm_frame;

/* One ARROW marker's numeric payload (rvizArrow, src/tunnel_processing.cpp:161-205). */
typedef struct gm_arrow {
  float start[3];
  float end[3];
  float scale[3];
  float color_argb[4]; /* pushed as (a,r,g,b): src/tunnel_processing.cpp:199-202 */
  int32_t id;
} gm_arrow;

typedef enum { GM_MODEL_PLANE = 0, GM_MODEL_CYLINDER = 1 } gm_model_kind;

/* Result of one RANSAC + refit (builder-defined stage a8). */
typedef struct gm_model {
  int32_t kind;        /* gm_model_kind */
  int32_t best_id;     /* winning hypothesis id, -1 if none */
  int32_t best_count;  /* its inlier count */
  int32_t refit_count; /* inliers used by the refit */
  float hyp[8];        /* winning hypothesis: plane {a,b,c,d}; cylinder {q(3),dir(3),r} */
  float coef[8];       /* refined model, same layout */
  float rms;           /* RMS residual of the refit inliers against the refined model */
  float pad_;
} gm_model;

/* One cross-section of the center-axis polyline (builder-defined, SURVEY A.10). */
typedef struct gm_slice {
  float center[3];
  float dir[3];
  float radius;
  float rms;
  float t_mid;
  int32_t count;
} gm_slice;

/* Result of the builder-defined compression stage (SURVEY A.10): the segmented cloud represented
 * by its refined primitives, the polyline and the voxel-downsampled residual (label 0) points. */
typedef struct gm_compression {
  int32_t n_points, n_plane, n_cylinder, n_residual, n_residual_voxels, n_slices;
  float plane_coef[4];    /* refined plane                                              */
  float plane_u[3], plane_v[3]; /* orthonormal in-plane basis (canonical, from the normal)   */
  float plane_bounds[4];  /* umin, umax, vmin, vmax of the plane inliers in that basis  */
  float plane_rms;
  float cyl_coef[7];      /* refined cylinder {q, dir, r}                               */
  float cyl_t_range[2];   /* extent of the cylinder inliers along dir, from q           */
  float cyl_rms;
  float residual_rms;     /* RMS distance of a residual point to its voxel centroid     */
  float total_rms;        /* reconstruction RMS over all n_points                        */
  float leaf;             /* residual voxel size (voxelGridLeafSize)                    */
  float ratio;            /* bytes_in / bytes_out                                       */
  uint64_t bytes_in;      /* 16 * n_points                                              */
  uint64_t bytes_out;     /* size of the blob gm_download_compressed writes             */
} gm_compression;

/* ---- lifecycle ------------------------------------------------------------------------- */
GM_API void gm_params_default(gm_params* p);
GM_API gm_status gm_create(const gm_params* p, size_t max_points, int32_t max_hypotheses, gm_ctx** out);
GM_API void gm_destroy(gm_ctx* ctx);
GM_API gm_status gm_set_params(gm_ctx* ctx, const gm_params* p);
GM_API gm_status gm_get_params(const gm_ctx* ctx, gm_params* out);
/* Use an existing cudaStream_t (e.g. torch's current stream).  NULL = the ctx's own (non-blocking)
 * stream; to run on CUDA's legacy default stream pass cudaStreamLegacy ((cudaStream_t)0x1). */
GM_API gm_status gm_set_stream(gm_ctx* ctx, void* cuda_stream);
/* Inlier-counting strategy of gm_ransac: 0 (default) = tile-culled over the cell-sorted cloud of the
 * scan whenever gm_normals produced one (identical counts, hypotheses whose inlier band provably
 * misses a 32-point tile are skipped for it); 1 = always the brute-force FP32 kernels. */
GM_API gm_status gm_set_count_mode(gm_ctx* ctx, int32_t mode);
/* Summation order of the neighbourhood sums of gm_normals (pcl::computeMeanAndCovarianceMatrix at
 * src/tunnel_processing.cpp:70).  0 (default) = neighbours are added in the order the grid search finds them: the
 * neighbour SET and count are exact, the float sums differ from PCL's by rounding.  1 = neighbours are added in
 * FLANN's result order (ascending squared distance, ties by index), the order pcl::NormalEstimation sums them in:
 * normals and curvatures are then bit-identical to the CPU oracle's and every later stage can be checked end to
 * end from the raw points.  A verification mode: ~40x slower than mode 0. */
GM_API gm_status gm_set_normals_mode(gm_ctx* ctx, int32_t mode);
/* k-nearest-neighbour normals: pcl::NormalEstimation::setKSearch(k) instead of setRadiusSearch(r) at
 * src/tunnel_processing.cpp:69 (the reference uses the radius; the k mode is what the north-star calls "grid-hashed k-NN").
 * k = 0 (default) = radius mode; 1 <= k <= 64: every point takes its k nearest points (itself included, ties by index).
 * neighborRadius then only sizes the search grid (pick it near the expected distance of the k-th neighbour); the search
 * is exact whatever its value.  Neighbours are summed in FLANN's result order: normals are bit-identical to the oracle's.
 * keep_indices = 1 also stores the neighbour lists (M x k, -1 padded) for gm_download_knn_indices. */
GM_API gm_status gm_set_knn(gm_ctx* ctx, int32_t k, int32_t keep_indices);
GM_API gm_status gm_download_knn_indices(gm_ctx* ctx, int32_t* out_m_x_k, size_t capacity_points);
/* Optional radius cap of the k mode: only points with d^2 < float(r*r) count as neighbours (FLANN's radiusSearch with max_nn = k:
 * the k nearest within r).  0 (default) = plain k-NN as pcl::NormalEstimation::setKSearch.  An isolated point (a lidar
 * outlier metres away from any surface) otherwise drags the exact search through every grid block between it and its k-th
 * neighbour; with a cap it ends with fewer than 3 neighbours, gets a NaN normal and leaves with the compaction, as in radius mode. */
GM_API gm_status gm_set_knn_max_radius(gm_ctx* ctx, double max_radius);
/* VoxelGrid strategy of gm_voxel / gm_compress: 0 (default) = sort-free dense tables whenever the number of lattice
 * cells of the crop box (or of the box given with gm_set_voxel_bbox) is at most 2^23, else sort-based; 1 = always
 * sort-based.  Same voxels, order, counts and centroids either way. */
GM_API gm_status gm_set_voxel_mode(gm_ctx* ctx, int32_t mode);
/* ---- map slabs (SURVEY 8e: one large map split along an axis over several contexts / GPUs) ----
 * gm_set_grid_box: build the neighbour grid over this box instead of the whole crop cube (the region
 *   the slab occupies, halo included; points outside it stay correct, only slower).  NULL,NULL = cube.
 * gm_set_owned_range: the context was given the slab lo <= coord[axis] < hi PLUS a halo (>= neighborRadius)
 *   of its neighbours.  Halo points take part in the neighbour search, then leave with the NaN normals:
 *   every later stage (voxels, frame, RANSAC, labels, compression) sees owned points only, with the same
 *   normals a single context would compute for them.  axis = -1: everything is owned.
 * gm_get_voxel_bbox / gm_set_voxel_bbox: pcl::getMinMax3D of the compacted cloud, and its override before
 *   gm_voxel: with the all-reduced (min/max) box of all slabs every slab uses ONE VoxelGrid lattice, so voxel
 *   keys are those of the whole map; slabs cut at multiples of the leaf own disjoint voxels.  NULL,NULL = own box. */
GM_API gm_status gm_set_grid_box(gm_ctx* ctx, const float* min3, const float* max3);
GM_API gm_status gm_set_owned_range(gm_ctx* ctx, int32_t axis, float lo, float hi);
GM_API gm_status gm_get_voxel_bbox(gm_ctx* ctx, float* min3, float* max3);
GM_API gm_status gm_set_voxel_bbox(gm_ctx* ctx, const float* min3, const float* max3);
/* Same box used only as a BOUND: the VoxelGrid box is still computed from the cloud (and all-reduced over the ranks by
 * gm_allreduce_voxel_bbox) on the device, but the promise that it lies inside [min3, max3] lets the sort-free dense
 * tables be sized without a host round trip.  A point outside the promised box raises device_error. */
GM_API gm_status gm_set_voxel_bbox_hint(gm_ctx* ctx, const float* min3, const float* max3);
GM_API const char* gm_last_error(const gm_ctx* ctx);
GM_API const char* gm_status_string(gm_status s);
GM_API int32_t gm_version(void);
/* Kernels launched by this ctx since creation (or since gm_reset_launch_count). */
GM_API int64_t gm_launch_count(const gm_ctx* ctx);
GM_API void gm_reset_launch_count(gm_ctx* ctx);
GM_API gm_status gm_synchronize(gm_ctx* ctx);

/* ---- input: replaces pcl::fromROSMsg(*input, *cloud), src/geometric_mapping.cpp:55 -------- */
/* Host buffer -> device (async H2D on the ctx stream).  stride_bytes >= 12; 16 for PointXYZ. */
GM_API gm_status gm_upload_scan(gm_ctx* ctx, const float* xyz_host, size_t n, size_t stride_bytes);
/* sensor_msgs/PointCloud2 payload as pcl::fromROSMsg reads it (src/geometric_mapping.cpp:55): n points of
 * point_step bytes, float32 x/y/z fields at the given byte offsets (any other fields are ignored),
 * little endian.  The raw bytes are copied to the device and gathered there. */
GM_API gm_status gm_upload_pointcloud2(gm_ctx* ctx, const void* data_host, size_t n, size_t point_step,
                                       size_t offset_x, size_t offset_y, size_t offset_z);
/* Scan already resident in HBM as n x float4 (not copied; must outlive the processing calls). */
GM_API gm_status gm_set_scan_device(gm_ctx* ctx, const float* xyzw_device, size_t n);

/* ---- per-point times and deskew (builder-defined: the reference treats every scan as a snapshot) -------------------
 * A spinning lidar takes a sweep over a scan period (typically 0.1 s) while it moves: at 1.5 m/s a point at the end of a
 * 10 Hz sweep is 15 cm from where a snapshot would put it.
 * gm_upload_pointcloud2_timed is gm_upload_pointcloud2 plus the float32 field at byte offset offset_t (offset_t + 4 <=
 *   point_step): each point's time in seconds, as velodyne_pointcloud publishes it (PointXYZIRT::time).  The times are
 *   decoded on the device from the same staged bytes; the first timed upload allocates their buffer (4 bytes a point).
 *   Every other upload (gm_upload_scan, gm_upload_pointcloud2, gm_set_scan_device, gm_inject_compacted) gives an untimed
 *   scan.  gm_download_point_times copies the n decoded times of a timed scan (GM_ERR_STAGE_ORDER for an untimed one) and
 *   synchronises the ctx stream like the other downloads.
 * gm_deskew rewrites the uploaded scan in place, before gm_crop: every point is expressed in the sensor frame at time t_ref,
 *   the sensor moving by delta34 over period seconds at constant velocity.  delta34 (row-major [R | t]) is the motion from
 *   the previous scan's frame to this scan's frame, in the previous scan's frame (gm_odometry_step's delta34).
 *   Constants, in double from D = double(delta34):
 *     v = (R21 - R12, R02 - R20, R10 - R01),  theta = atan2(|v| / 2, (R00 + R11 + R22 - 1) / 2),  u = v / |v|,
 *     td = (D[3], D[7], D[11]);  |v| = 0 gives theta = 0 and u = 0 (the identity rotation).
 *   Per point i, in double:
 *     a = ((double)t_i - t_ref) / period,  phi = a * theta,
 *     R(a) = cos(phi) I + sin(phi) [u]x + (1 - cos(phi)) u u^T,
 *     p' = R(a) p + a td,  stored as float(p') with w = 1.
 *   The rotation is interpolated along the geodesic and the translation linearly (the decoupled form); a = 1 gives delta34
 *   itself.  A motion near 180 degrees within one period is not supported (theta is taken from the trace and |v|).
 *   Exact cases: an identity delta34, or a point with t_i == t_ref, leaves the point's coordinates unchanged (a zero
 *   coordinate may change its sign); a point with a non-finite coordinate or time becomes (NaN, NaN, NaN, 1), which the
 *   stages then treat as any NaN input point (gm_crop's is_dense rule).
 *   One launch (k_deskew), no host synchronisation: each block derives the constants, the point count is read on the
 *   device.  gm_process_scan and its CUDA graphs read the deskewed scan as any uploaded one.
 *   Rules: GM_ERR_INVALID_ARG, with nothing launched, for a NULL or non-finite delta34, a non-finite t_ref, or period <= 0
 *   or non-finite; GM_ERR_STAGE_ORDER for an untimed scan, after gm_crop (or gm_process_scan) of this upload, and for a
 *   second gm_deskew / gm_odometry_deskew of the same upload (deskewing twice is almost always a bug). */
GM_API gm_status gm_upload_pointcloud2_timed(gm_ctx* ctx, const void* data_host, size_t n, size_t point_step,
                                             size_t offset_x, size_t offset_y, size_t offset_z, size_t offset_t);
GM_API gm_status gm_download_point_times(gm_ctx* ctx, float* out, size_t capacity_points);
GM_API gm_status gm_deskew(gm_ctx* ctx, const float* delta34, double t_ref, double period);

/* ---- stages ---------------------------------------------------------------------------- */
/* chopCloud(bound, cloud): src/tunnel_processing.cpp:39-49, called src/geometric_mapping.cpp:57 */
GM_API gm_status gm_crop(gm_ctx* ctx);
/* getNormals(neighborRadius, cloud, kdtree): src/tunnel_processing.cpp:52-89 — radius-search
 * normals + curvature (pcl::NormalEstimation), then NaN-normal removal compacting cloud and
 * normals.  The kd-tree out-param is replaced by the device neighbour grid kept in ctx. */
GM_API gm_status gm_normals(gm_ctx* ctx);
/* compute part of rvizNormals(leaf, cloud, kdtree, normals): src/tunnel_processing.cpp:215-220
 * (pcl::VoxelGrid) and :233-249 (1-NN of each centroid -> normal). */
GM_API gm_status gm_voxel(gm_ctx* ctx);
/* getLocalFrame(n, weightingFactor, normals, vals, vecs): src/tunnel_processing.cpp:92-148 */
GM_API gm_status gm_local_frame(gm_ctx* ctx);

/* Builder-defined stages the reference stubs as getCylinder (src/tunnel_processing.cpp:149-154,
 * include/geometric_mapping/tunnel_processing.hpp:56-59).
 * gm_ransac: generate H hypotheses from injected sample indices (host array, H x 3 for planes,
 * H x 2 for cylinders; indices into the compacted cloud), count inliers of ids [h_begin,h_end)
 * over the compacted cloud, and reduce the local best into a packed key
 *   key = (uint64(count + 1) << 32) | (0xFFFFFFFF - id)       (max = best, ties -> lowest id).
 * Multi-GPU: each rank passes its own [h_begin,h_end); all-reduce(max) the keys between
 * gm_ransac and gm_ransac_select. */
GM_API gm_status gm_ransac(gm_ctx* ctx, int32_t kind, const int32_t* samples_host, int32_t H,
                           int32_t h_begin, int32_t h_end);
/* Device address of the 8-byte packed best key of `kind` (for an NCCL all-reduce in place). */
GM_API gm_status gm_ransac_key_device_ptr(gm_ctx* ctx, int32_t kind, void** key_dev);
/* Copy the 8-byte key to / from a caller-owned device buffer (e.g. the int64 tensor handed to the
 * collective), asynchronously on the ctx stream: export -> all-reduce(MAX) -> import -> select. */
GM_API gm_status gm_ransac_export_key(gm_ctx* ctx, int32_t kind, void* dst_device);
GM_API gm_status gm_ransac_import_key(gm_ctx* ctx, int32_t kind, const void* src_device);
/* Decode the (possibly all-reduced) key on device, refit the winning primitive (plane: PCA of
 * inliers; cylinder: refitIterations Gauss-Newton steps) and keep the result in ctx. */
GM_API gm_status gm_ransac_select(gm_ctx* ctx, int32_t kind);
/* One RANSAC step for both primitives with the plane and cylinder work side by side on two streams of the ctx
 * (same results as the four separate calls).  Multi-GPU: gm_ransac_pair -> gm_ransac_export_keys -> ONE
 * all-reduce(MAX) of 2 x int64 -> gm_ransac_import_keys -> gm_ransac_select_pair. */
GM_API gm_status gm_ransac_pair(gm_ctx* ctx, const int32_t* plane_samples_host, int32_t Hp, int32_t p_begin, int32_t p_end,
                                const int32_t* cyl_samples_host, int32_t Hc, int32_t c_begin, int32_t c_end);
GM_API gm_status gm_ransac_select_pair(gm_ctx* ctx);
GM_API gm_status gm_ransac_export_keys(gm_ctx* ctx, void* dst_device_16_bytes);
GM_API gm_status gm_ransac_import_keys(gm_ctx* ctx, const void* src_device_16_bytes);
/* Per-point labels from the refined models: 1 plane, 2 cylinder, 0 neither. */
GM_API gm_status gm_label(gm_ctx* ctx);
/* Center-axis polyline + cross-sections along the getLocalFrame axis over points with label 2. */
GM_API gm_status gm_axis_polyline(gm_ctx* ctx);

/* Geometric approximation (compression) of the segmented cloud; needs labels and the polyline.
 * The name the north-star gives this stage has no counterpart in the reference sources. */
GM_API gm_status gm_compress(gm_ctx* ctx);
GM_API gm_status gm_get_compression(gm_ctx* ctx, gm_compression* out);
/* Packed little-endian blob: 'GMC1' header (gm_compression) | n_slices x gm_slice | n_residual_voxels
 * x {x,y,z} float.  Pass buf = NULL to query the size. */
GM_API gm_status gm_download_compressed(gm_ctx* ctx, void* buf, size_t capacity, size_t* bytes);

/* ---- sequential multi-primitive extraction (builder-defined, SURVEY A.9: "repeat after removing inliers") --------
 * Up to max_primitives rounds over the compacted cloud (M' points).  Round r (0-based):
 *   1. R_r = the ascending compacted indices no earlier round claimed, n_r = |R_r|.
 *   2. Sampling: the caller's uint32 draws (max_primitives x Hp x 3 for planes, max_primitives x Hc x 2 for cylinders, one
 *      block per round) map to sample indices R_r[(uint64(u) * n_r) >> 32], or -1 when n_r = 0.
 *   3. Plane / cylinder hypotheses are generated from those indices exactly as gm_ransac generates them (same
 *      coefficients for the same indices); inliers are counted over R_r only; the best of each kind is the packed-key
 *      argmax of gm_ransac (ties -> lowest id).
 *   4. The kind with the larger best count wins (tie -> plane).  The round is accepted iff
 *      best_count >= max(min_inliers, 1); otherwise extraction stops and this and every later round add nothing.
 *   5. The winner is refitted on its inliers within R_r as gm_ransac_select does (plane PCA; cylinder Gauss-Newton).
 *   6. Exactly the points of R_r the WINNING HYPOTHESIS counted as inliers get primitive id r + 1 (so the number claimed
 *      equals best_count).  The refined coefficients are reported and used by gm_compress_primitives only.
 * Every compacted point gets one uint8 id: 0 = residual, k = the k-th extracted primitive.  The rounds run without host
 * synchronisation: the launch sequence depends only on (max_primitives, Hp > 0, Hc > 0).  Needs the compacted cloud
 * (cylinders read its normals, as gm_ransac does).  Extraction has buffers of its own (allocated by the first call):
 * gm_ransac's hypotheses, models, labels and compression are untouched. */
#define GM_MAX_PRIMITIVES 64
typedef struct gm_primitive {
  gm_model model;       /* kind, best_id (within its round), best_count (= points claimed), refit_count, hyp, coef, rms */
  int32_t n_remaining;  /* unclaimed points at the start of its round */
  int32_t pad_;
} gm_primitive;
GM_API gm_status gm_extract_primitives(gm_ctx* ctx, int32_t max_primitives, int32_t min_inliers,
                                       const uint32_t* plane_draws_host, int32_t Hp,
                                       const uint32_t* cyl_draws_host, int32_t Hc);
/* *n = number of primitives extracted; GM_ERR_CAPACITY if it exceeds capacity (out may be NULL to query it). */
GM_API gm_status gm_get_primitives(gm_ctx* ctx, gm_primitive* out, int32_t capacity, int32_t* n);
/* M' primitive ids, in compacted order. */
GM_API gm_status gm_download_primitive_ids(gm_ctx* ctx, uint8_t* out, size_t capacity_points);

/* Compression of the extracted primitives, the counterpart of gm_compress: every primitive as its refined surface and
 * extents, the residual (id 0) points voxel-downsampled at voxelGridLeafSize.  Needs gm_extract_primitives. */
typedef struct gm_primitive_compression {
  int32_t n_points, n_primitives, n_residual, n_residual_voxels;
  float leaf;          /* residual voxel size                                                   */
  float residual_rms;  /* RMS distance of a residual point to its voxel centroid                */
  float total_rms;     /* reconstruction RMS over all n_points (claimed points: to their surface) */
  float ratio;         /* bytes_in / bytes_out                                                  */
  uint64_t bytes_in;   /* 16 * n_points                                                         */
  uint64_t bytes_out;  /* size of the blob gm_download_compressed_primitives writes             */
} gm_primitive_compression;
typedef struct gm_primitive_record {
  int32_t kind;        /* gm_model_kind */
  int32_t count;       /* points claimed */
  float coef[7];       /* refined plane {a,b,c,d} or cylinder {q, dir, r} */
  float extents[4];    /* plane: umin, umax, vmin, vmax in gm_compress's canonical in-plane basis; cylinder: tmin, tmax along dir from q, 0, 0 */
  float rms;           /* RMS distance of its claimed points to the refined surface */
} gm_primitive_record;
GM_API gm_status gm_compress_primitives(gm_ctx* ctx);
/* Packed little-endian blob: 'GMP1' | version u32 | gm_primitive_compression | n_primitives x gm_primitive_record |
 * n_residual_voxels x {x,y,z} float.  Pass buf = NULL to query the size. */
GM_API gm_status gm_download_compressed_primitives(gm_ctx* ctx, void* buf, size_t capacity, size_t* bytes);

/* ---- scan-to-scan registration (builder-defined: the reference computes no pose) -----------------------------------
 * Point-to-plane ICP of the SOURCE context's VoxelGrid centroids (V points, after gm_voxel; under the VoxelGrid overflow
 * rule its cloud as it is) against the TARGET context's compacted cloud and normals (after gm_normals, which builds the
 * neighbour grid the search walks: an injected compacted cloud has none and gives GM_ERR_STAGE_ORDER).  target == source
 * is allowed; both must be on the same device.  The pose T_i is held in double on the device, T_0 = init_pose34.
 * Iteration i (0-based):
 *   1. Tf = float(T_i) element-wise; every centroid c is transformed as p = Tf c with the fmaf chains of gm_map_insert.
 *   2. Correspondence: the compacted target point q nearest to p (FLANN ((dx^2)+dy^2)+dz^2 in float, ties -> lowest
 *      compacted index), accepted iff d^2 < float(d_max * d_max) (product in double, as the radius search takes it).
 *      This is the exact nearest point, not an approximation.
 *   3. With the compacted normal n of q, in double: r = n.(p - q), J = [p x n, n] (derivative with respect to a
 *      left-applied twist (w, v)).
 *   4. A = sum J J^T, g = sum J r, sum r^2 and the count m over the accepted points, in fixed-order double partials:
 *      bitwise reproducible run to run.
 *   5. A = V L V^T by cyclic Jacobi in double (eigenvalues ascending, each eigenvector's largest-|component| positive);
 *      xi = -sum over k with lambda_k > degeneracy_ratio * lambda_max of (v_k.g / lambda_k) v_k; the other directions
 *      are not updated (n_degenerate of them): they stay at the initial guess.  Then T_{i+1} = [R(w) | v] o T_i, i.e.
 *      R <- R(w) R, t <- R(w) t + v, R(w) by Rodrigues in double.
 *   6. Stop after the update with converged = 1 when |w| < min_rotation_step and |v| < min_translation_step; stop
 *      without an update (converged = 0) when m < 6 or lambda_max <= 0.  Later iterations are no-ops.
 * The launch sequence depends only on max_iterations: gm_launch_count(source) grows by max_iterations + 1, and there is
 * no host synchronisation between iterations.  The reported pose is the pose after the last update; correspondences,
 * residuals, rmse, fitness, the spectrum and n_degenerate belong to the last executed iteration, evaluated at its input
 * pose.  V = 0 gives n_correspondences = 0, converged = 0 and the initial pose.
 * The work runs on the source stream after the target stream's pending work, and the target stream waits for it before
 * any later work (a new scan on the target cannot overwrite the grid under the search).  The results live in the source
 * context until a new scan or neighbour grid there; they have buffers of their own (allocated by the first call). */
#define GM_MAX_ICP_ITERATIONS 64
typedef struct gm_icp_params {
  float init_pose34[12];               /* source -> target guess, row-major [R|t] (the layout gm_map_insert takes)        */
  double max_correspondence_distance;  /* d_max, metres, > 0                                         default 0.5          */
  int32_t max_iterations;              /* 1 .. GM_MAX_ICP_ITERATIONS                                 default 30           */
  int32_t pad_;
  double min_rotation_step;            /* rad: converged when |w| < this ...                         default 1e-5         */
  double min_translation_step;         /* m:   ... and |v| < this                                    default 1e-5         */
  double degeneracy_ratio;             /* [0, 1): directions with lambda_k <= ratio * lambda_max are not updated; default 0
                                          (only lambda_k <= 0 is dropped: plain Gauss-Newton)                             */
} gm_icp_params;
typedef struct gm_registration {
  float pose34[12];          /* refined source -> target                                                     */
  int32_t iterations;        /* iterations executed (including one that stopped without an update)           */
  int32_t converged;         /* 1 = stopped on the step thresholds                                           */
  int32_t n_source;          /* source points (the source's voxel centroids, V)                              */
  int32_t n_correspondences; /* of the last executed iteration                                               */
  float rmse;                /* sqrt(sum r^2 / n_correspondences) over those (0 without correspondences)     */
  float fitness;             /* n_correspondences / n_source (0 when V = 0)                                  */
  int32_t n_degenerate;      /* eigen-directions not updated in the last executed iteration                  */
  int32_t pad_;
  double eigenvalues[6];     /* of that iteration's J^T J, ascending                                         */
  double eigenvectors[36];   /* row-major, column k = eigenvector k, parameters (wx, wy, wz, vx, vy, vz)     */
} gm_registration;
GM_API void gm_icp_params_default(gm_icp_params* p);  /* identity guess and the defaults above */
GM_API gm_status gm_register(gm_ctx* source, gm_ctx* target, const gm_icp_params* p);
GM_API gm_status gm_get_registration(gm_ctx* source, gm_registration* out);  /* synchronises the source stream */
/* V entries of the last executed iteration: compacted target index or -1, float(r) or NaN; residual may be NULL */
GM_API gm_status gm_download_correspondences(gm_ctx* source, int32_t* target_index, float* residual, size_t capacity_points);

/* Fused per-scan path = the body of cloud_cb (src/geometric_mapping.cpp:48-125) plus the
 * builder-defined segmentation: crop -> normals -> voxel -> local frame -> RANSAC plane(Hp)
 * + cylinder(Hc) -> select/refit -> labels -> polyline.  samples may be NULL when H == 0. */
GM_API gm_status gm_process_scan(gm_ctx* ctx, const int32_t* plane_samples_host, int32_t Hp,
                                 const int32_t* cyl_samples_host, int32_t Hc);

/* gm_process_scan replays a CUDA graph: the first scan of a given (size bucket of 32768 points, Hp, Hc, parameters)
 * runs as plain stream launches, the second is captured, every later one is ONE cudaGraphLaunch (33 kernels on three
 * streams).  mode 0 = always plain launches, 1 = always graphs, 2 = auto (default; env GM_GRAPH overrides): graphs for scans of up
 * to 524288 points, where launch overhead dominates, plain launches above, where the GPU is the limit and host copies
 * pipeline better without (measured: DESIGN.md section 4).  If the stream cannot be captured the library keeps working with plain
 * launches; gm_get_graph_stats tells which happened. */
GM_API gm_status gm_set_graph_mode(gm_ctx* ctx, int32_t mode);
GM_API gm_status gm_get_graph_stats(const gm_ctx* ctx, int64_t* captures, int64_t* replays);

/* ---- results (synchronise the ctx stream) ---------------------------------------------- */
GM_API gm_status gm_get_counts(gm_ctx* ctx, gm_counts* out);
/* cloud: which = 0 cropped (pre-compaction, M), 1 compacted (M'), written as n x float4 */
GM_API gm_status gm_download_cloud(gm_ctx* ctx, int32_t which, float* out_xyzw, size_t capacity_points);
/* normals: which = 0 pre-compaction (M, NaN rows included), 1 compacted (M'); n x 8 floats */
GM_API gm_status gm_download_normals(gm_ctx* ctx, int32_t which, float* out8, size_t capacity_points);
/* work of the radius search of the last gm_normals: distance tests executed (population of the 27-cell stencil
 * summed over the points) and how many of them were within the radius (diagnostic; feeds bench.py's roofline) */
GM_API gm_status gm_get_search_stats(gm_ctx* ctx, int64_t* candidates, int64_t* neighbors);
/* neighbour counts of the radius search per cropped point (M int32) */
GM_API gm_status gm_download_neighbor_counts(gm_ctx* ctx, int32_t* out, size_t capacity_points);
/* pre-compaction index -> compacted index or -1 (M int32) */
GM_API gm_status gm_download_valid_map(gm_ctx* ctx, int32_t* out, size_t capacity_points);
/* voxel keys and voxel rank of every compacted point (M' int32 each); either may be NULL */
GM_API gm_status gm_download_voxel_assignment(gm_ctx* ctx, int32_t* keys, int32_t* assign, size_t capacity_points);
/* per voxel: centroid (V x float4), key, member count, 1-NN index, 1-NN normal (V x 8 floats); any may be NULL */
GM_API gm_status gm_download_voxels(gm_ctx* ctx, float* centroids_xyzw, int32_t* keys, int32_t* counts,
                                    int32_t* nn_index, float* nn_normal8, size_t capacity_voxels);
/* VoxelGrid lattice: min_b[3], div_b[3] */
GM_API gm_status gm_get_voxel_grid(gm_ctx* ctx, int32_t grid6[6]);
GM_API gm_status gm_get_frame(gm_ctx* ctx, gm_frame* out);
/* hypothesis table of the last gm_ransac(kind): coef (plane H x 4, cylinder H x 7), inlier test
 * parameters (cylinder only, H x 12, may be NULL), counts (H int32, -1 = degenerate or not in
 * this rank's range) */
GM_API gm_status gm_download_hypotheses(gm_ctx* ctx, int32_t kind, float* coef, float* test12, int32_t* counts, int32_t capacity_h);
GM_API gm_status gm_get_model(gm_ctx* ctx, int32_t kind, gm_model* out);
GM_API gm_status gm_download_labels(gm_ctx* ctx, uint8_t* out, size_t capacity_points);
GM_API gm_status gm_download_polyline(gm_ctx* ctx, gm_slice* out, int32_t capacity, int32_t* n_slices);

/* ---- pipelined end-to-end use: enqueue all result copies, synchronise once ---------------- */
/* Fixed-size summary of one scan (filled by gm_fetch_async). */
typedef struct gm_scan_summary {
  gm_counts counts;
  gm_frame frame;
  gm_model plane;
  gm_model cylinder;
  int32_t n_slices;
  int32_t pad_;
} gm_scan_summary;

/* Caller-provided (ideally pinned) host destinations; NULL = skip.  Copies are enqueued on the ctx
 * stream without a host round trip, so variable-size outputs are copied up to the number of
 * INPUT points (an upper bound of every later size); read the true sizes from summary->counts
 * after gm_synchronize().  cloud_xyzw is the cloud that cloud_cb publishes on cloudOutput
 * (src/geometric_mapping.cpp:100-107): cropped and NaN-normal-compacted. */
typedef struct gm_host_outputs {
  gm_scan_summary* summary;
  float* cloud_xyzw;      size_t cloud_capacity;    /* points */
  float* normals8;        size_t normals_capacity;  /* points */
  uint8_t* labels;        size_t labels_capacity;   /* points */
  gm_slice* slices;       int32_t slices_capacity;
  float* centroids_xyzw;  float* nn_normal8; size_t voxel_capacity; /* voxels */
} gm_host_outputs;
GM_API gm_status gm_fetch_async(gm_ctx* ctx, const gm_host_outputs* out);

/* ---- per-stage device timing (CUDA events on the ctx stream) -------------------------------- */
GM_API gm_status gm_profile_enable(gm_ctx* ctx, int32_t on);
GM_API int32_t gm_profile_num_segments(void);
GM_API const char* gm_profile_segment_name(int32_t i);
/* Synchronises; adds the elapsed ms and call counts since the last reset into ms_sum/calls
 * (arrays of gm_profile_num_segments()), then resets. */
GM_API gm_status gm_profile_read(gm_ctx* ctx, float* ms_sum, int32_t* calls);

/* ---- test hooks: inject a stage's input so stages can be parity-checked in isolation ---- */
/* Replace the compacted cloud (and normals, may be NULL) held in ctx: n x float4 / n x 8 floats. */
GM_API gm_status gm_inject_compacted(gm_ctx* ctx, const float* xyzw_host, const float* normals8_host, size_t n);

/* ---- host-side formatting of the published numbers (a6) --------------------------------- */
/* rvizEigens(vals, vecs): src/tunnel_processing.cpp:260-300 -> 3 arrows */
GM_API void gm_markers_eigen(const gm_frame* frame, gm_arrow out[3]);
/* rvizNormals marker payload: src/tunnel_processing.cpp:228-252 -> V arrows from the voxel results */
GM_API void gm_markers_normals(const float* centroids_xyzw, const float* nn_normal8, int32_t V, gm_arrow* out);
/* same with the arrow-end switch of gm_params.arrow_mode (0 = reference quirk B.4, 1 = end = start + normal) */
GM_API void gm_markers_normals_mode(const float* centroids_xyzw, const float* nn_normal8, int32_t V, int32_t arrow_mode, gm_arrow* out);

/* ---- on-disk store of the per-scan compressed primitives (SURVEY 8f.3; builder-defined: the reference keeps nothing between
 * callbacks, src/geometric_mapping.cpp:48-125).  Append-only file of the GMC1 blobs of gm_download_compressed, one record per
 * scan with its id, stamp and pose [R|t] (row-major 3x4, NULL = identity), each protected by a CRC-32; the index is rebuilt
 * when the file is opened and a torn last record is dropped.  Host-side I/O only. */
typedef struct gm_store gm_store;
GM_API gm_status gm_store_open(const char* path, int32_t create_if_missing, gm_store** out);
GM_API void gm_store_close(gm_store* store);
GM_API gm_status gm_store_append(gm_store* store, gm_ctx* ctx /* after gm_compress */, uint64_t scan_id, uint64_t stamp_ns, const float* pose34);
GM_API gm_status gm_store_append_blob(gm_store* store, uint64_t scan_id, uint64_t stamp_ns, const float* pose34, const void* blob, size_t bytes);
GM_API int64_t gm_store_count(const gm_store* store);
GM_API gm_status gm_store_info(const gm_store* store, int64_t index, uint64_t* scan_id, uint64_t* stamp_ns, float* pose34, uint64_t* blob_bytes);
/* buf = NULL queries the size */
GM_API gm_status gm_store_read(gm_store* store, int64_t index, void* buf, size_t capacity, size_t* bytes);

/* ---- ROS-free encoders of the published messages (SURVEY 8f.1): the byte payloads a ROS 1 publisher would put on the
 * wire for what cloud_cb publishes (src/geometric_mapping.cpp:100-117), so a transport that is not roscpp can ship them
 * and a subscriber deserialises them as the stock message types.
 *   cloudOutput       sensor_msgs/PointCloud2 as pcl::toROSMsg(PointCloud<PointXYZ>) lays it out (:102-103): height 1, fields
 *                     x,y,z FLOAT32 @ 0,4,8, point_step 16
 *   normalsOutput /   visualization_msgs/MarkerArray of ARROW markers as rvizArrow fills them (src/tunnel_processing.cpp:
 *   eigenBasisOutput  171-203; frame "/velodyne", include/geometric_mapping/tunnel_processing.hpp:72-73), from the gm_arrow
 *                     payloads of gm_markers_eigen / gm_markers_normals (ns "eigenBasis" / "normals")
 * The *_size functions give the exact byte count; GM_ERR_CAPACITY if the buffer is smaller. */
GM_API size_t gm_pointcloud2_size(size_t n_points, const char* frame_id);
GM_API gm_status gm_encode_pointcloud2(const float* xyzw, size_t n, const char* frame_id, uint32_t seq, uint64_t stamp_ns, int32_t is_dense,
                                       void* buf, size_t capacity, size_t* bytes);
GM_API size_t gm_marker_array_size(int32_t n_markers, const char* frame_id, const char* ns);
GM_API gm_status gm_encode_marker_array(const gm_arrow* arrows, int32_t n, const char* frame_id, const char* ns, uint64_t stamp_ns, void* buf,
                                        size_t capacity, size_t* bytes);

/* ---- aggregated voxel map across scans (SURVEY 8f.3; builder-defined, the reference keeps nothing between
 * callbacks, src/geometric_mapping.cpp:48-125) --------------------------------------------------------
 * A device hash table keyed by the GLOBAL VoxelGrid cell floor(p * inv_leaf) of every inserted point, holding the
 * point count and the coordinate sums in 2^-20 m fixed point: insertion order (scans, contexts, streams) does
 * not change the result.  gm_map_insert adds the compacted cloud of `ctx` (after gm_normals; asynchronous on
 * the ctx stream), optionally only the points with label == label_filter (after gm_label; -1 = all), after the
 * rigid transform pose34 = row-major [R|t] (NULL = identity; p' = R p + t as fmaf chains).  gm_map_download
 * returns the voxels sorted by (z, y, x) index: integer cell, count, centroid = sum / count.  gm_map_save / load:
 * little-endian file 'GMM1' | leaf f64 | V u64 | keys u64[V] | counts i32[V] | sums i64[3V] (exact state).
 * A map lives on the device current at gm_map_create / gm_map_load.  The gm_map_* and gm_odometry_* calls that take no
 * context work on that device whichever device is current, and leave the caller's current device as it was; one that
 * synchronises the device synchronises the caller's current device and then, if that is another one, the map's. */
typedef struct gm_map gm_map;
GM_API gm_status gm_map_create(double leaf, size_t capacity_voxels, gm_map** out);
GM_API void gm_map_destroy(gm_map* map);
GM_API gm_status gm_map_clear(gm_map* map);
GM_API gm_status gm_map_insert(gm_map* map, gm_ctx* ctx, const float* pose34, int32_t label_filter);
/* GM_ERR_CAPACITY if an insert found the table full (those points were dropped) */
GM_API gm_status gm_map_stats(gm_map* map, int64_t* n_voxels, int64_t* n_points, int64_t* n_out_of_range);
GM_API gm_status gm_map_download(gm_map* map, int32_t* ijk, int32_t* counts, float* centroids_xyzw, size_t capacity, size_t* n);
GM_API gm_status gm_map_save(gm_map* map, const char* path);
GM_API gm_status gm_map_load(const char* path, size_t min_capacity_voxels, gm_map** out);
GM_API double gm_map_leaf(const gm_map* map);
/* ---- a window on a map: eviction into an archive, and the exact way back ---------------------------------------------
 * gm_map_evict keeps the voxels of `map` inside a cube of cells around center3 and moves the others into `archive`
 * (NULL = drops them), so that a long run can work in a local map sized to what the sensor sees.
 *   Centre cell.  c[a] = (int)floorf(center3[a] * inv_leaf), the float product of gm_map_insert's cell (inv_leaf = 1 / (float)leaf).
 *   Kept.  A voxel of cell (i, j, k) is kept iff max(|i - c0|, |j - c1|, |k - c2|) <= half_cells, in 64-bit integers: a
 *     Chebyshev cube of 2 half_cells + 1 cells a side, with no float test.
 *   After the call the map holds exactly the kept voxels with their counts and sums unchanged (no tombstones); n_voxels and
 *     n_points of gm_map_stats describe them, and overflow and out_of_range (records of earlier inserts) stay as they were
 *     until gm_map_clear.  Each evicted voxel's count and sums are added as integers to the archive's entry of the same key,
 *     created if absent (gm_map_load's add).  An archive that is full drops the voxels that do not fit, and its gm_map_stats
 *     then gives GM_ERR_CAPACITY.  Counts and sums are integers, so the adds are exact: gm_map_merge(archive, map) after
 *     any number of evictions gives back, bit for bit, the map that was never evicted.
 *   Ordering.  Asynchronous on ctx's stream; ctx only supplies the stream and the launch count.  It is a map operation on
 *     both maps: it waits for the previous gm_map_insert / gm_register_map / gm_odometry_step / gm_map_evict on the map and on
 *     the archive, and the next operation on either waits for it.
 *   Launches.  GM_MAP_EVICT_LAUNCHES kernels, always: the split (each voxel to the archive or to the map's scratch), then
 *     the clear of the table and the re-insertion of the kept voxels, which return at once, reading it from device memory,
 *     when nothing was evicted.  No host synchronisation; the first call allocates the map's scratch (36 bytes a slot).
 *     The slot layout afterwards is not that of the original insertion, which changes no output: every read of a map is in
 *     key order.
 *   Errors.  GM_ERR_INVALID_ARG, with nothing launched, for half_cells < 0, a non-finite centre or a centre cell outside
 *     the key range [-2^20, 2^20), archive == map, an archive whose leaf is not bitwise the map's, and a context or archive
 *     on another device than the map.
 * gm_map_merge adds every voxel of src into dst (dst += src by the same integer add; src is unchanged), in one kernel on
 * the device, and synchronises the device as gm_map_clear and gm_map_load do.  The leaf and device rules are those of
 * gm_map_evict, and dst != src.  GM_ERR_CAPACITY if dst overflowed (a voxel found it full and was dropped).  The whole map
 * of a windowed run is gm_map_merge(archive, local) then gm_map_save(archive); an archive saved and cleared every so often
 * gives GMM1 segment files whose key-wise sum is the same map. */
#define GM_MAP_EVICT_LAUNCHES 3
GM_API gm_status gm_map_evict(gm_map* map, gm_ctx* ctx, gm_map* archive, const float* center3, int32_t half_cells);
GM_API gm_status gm_map_merge(gm_map* dst, const gm_map* src);  /* dst += src, src unchanged */

/* ---- scan-to-map registration (builder-defined: the reference keeps no map) -------------------------------------------
 * gm_register with the aggregated voxel map as the target: localises a scan in the map being built, or in one reloaded
 * with gm_map_load, without chaining scan-to-scan poses.  Map planes, for every occupied voxel v:
 *   - its centroid c_v is exactly what gm_map_download reports, float((double)sum / 2^20 / count);
 *   - N(v) = the occupied voxels among the 27 at offsets (dx, dy, dz) in {-1, 0, 1}^3, v included, visited in ascending
 *     (dz, dy, dx) order.  With |N(v)| < GM_MAP_PLANE_MIN_VOXELS, v has no plane.  Otherwise mu = the sequential double
 *     mean of their centroids, C = the sequential double sum of (c - mu)(c - mu)^T over N(v) divided by |N(v)|, and
 *     cyclic Jacobi (the sign rule of gm_register's spectrum) gives lambda0 <= lambda1 <= lambda2; v has a plane iff
 *     lambda0 <= max_planarity * lambda1 and lambda1 > 0, and its normal is float(eigenvector 0).
 *   The neighbourhood uses the voxel centroids only, so the map's state and its file format are those of any map, saved
 *   by any version.  How flat a voxel neighbourhood looks depends on the scan noise relative to the leaf: 0.1 suits
 *   centimetre noise at a 10 cm leaf; 0.01 keeps only the flattest surfaces.
 * gm_register_map runs steps 1-6 of gm_register above with the source context's VoxelGrid centroids and this search:
 *   2'. Correspondence: among the voxels that have a plane, the one whose centroid q is nearest to p (FLANN
 *       ((dx^2)+dy^2)+dz^2 in float, ties -> lowest map key, i.e. first in gm_map_download order), accepted iff
 *       d^2 < float(d_max * d_max).  This is the exact nearest candidate, not an approximation.  The search walks cube
 *       shells of voxels around p's voxel, clipped to the bounding box of the voxels with a plane: its work per point is
 *       bounded by that box (and by d_max), and a map without planes or a point far from the box costs no search.
 *   3'. n = that voxel's normal: r = n.(p - q), J = [p x n, n] as in step 3.
 * Arguments are checked as by gm_register, plus 0 < max_planarity <= 1 and source and map on the same device (the one
 * current at gm_map_create / gm_map_load).  The result is the source's registration: gm_get_registration reads it,
 * gm_download_map_correspondences gives the matched voxels (gm_download_correspondences gives GM_ERR_STAGE_ORDER after a
 * map registration, and gm_download_map_correspondences after a context one).  The launches are the planes of the map
 * (k_map_planes, once per call), then those of gm_register: gm_launch_count(source) grows by max_iterations + 2, with no
 * host synchronisation.  An empty map, or one without planes, gives 0 correspondences, converged = 0 and the initial pose.
 * Ordering: gm_map_insert and gm_register_map wait on their context's stream for the previous of these two calls on the
 * same map, whichever context issued it, so map operations from several contexts of the map's device run in call order
 * without a host synchronisation. */
#define GM_MAP_PLANE_MIN_VOXELS 5
GM_API gm_status gm_register_map(gm_ctx* source, gm_map* map, const gm_icp_params* p, double max_planarity);
/* V entries of the last executed iteration: the matched voxel's integer cell (the ijk of gm_map_download) or INT32_MIN x 3,
 * float(r) or NaN; residual may be NULL */
GM_API gm_status gm_download_map_correspondences(gm_ctx* source, int32_t* ijk /* V x 3 */, float* residual, size_t capacity_points);
/* the plane of every voxel in gm_map_download's order and count: {nx, ny, nz, 1}, or {NaN, NaN, NaN, 0} without a plane
 * (what gm_register_map searches with the same max_planarity); synchronises the device.  normals_xyzw = NULL: *n only */
GM_API gm_status gm_map_download_planes(gm_map* map, double max_planarity, float* normals_xyzw, size_t capacity, size_t* n);

/* ---- map odometry (builder-defined: the reference computes no pose) ---------------------------------------------------
 * Builds a map from the scans alone without a host round trip: each gm_odometry_step predicts the scan's pose, registers
 * the scan to the map from it (gm_register_map), accepts or rejects the result and inserts the scan at the accepted pose
 * (gm_map_insert), all on the context's stream.  The trajectory, one gm_odometry_record per step, lives in device memory.
 * Step k (k = gm_odometry_steps() when it is called) needs ctx after gm_voxel: its VoxelGrid centroids are the
 * registration source and its compacted cloud is what the insert takes.  ctx must be on the map's device; any number of
 * contexts may take turns (e.g. two, so that the next scan is processed while a step runs).
 *   Guess G_k.  P_j = the float pose34 of step j's record.  Poses compose rigidly in double from the float inputs, unfused:
 *     (A o B): R[i][j] = (A[i][0]*B[0][j] + A[i][1]*B[1][j]) + A[i][2]*B[2][j],
 *              t[i]    = ((A[i][0]*B[0][3] + A[i][1]*B[1][3]) + A[i][2]*B[2][3]) + A[i][3]   (gm_register's update order);
 *     the inverse of a float pose is [R^T | -(R^T t)], (R^T t)[i] = (R[0][i]*t[0] + R[1][i]*t[1]) + R[2][i]*t[2].
 *     k = 0:                 G = icp.init_pose34; delta34 must be NULL (else GM_ERR_INVALID_ARG).
 *     k >= 1, delta34 given: G = P_{k-1} o delta, delta = the sensor's motion since the previous scan in the previous
 *                            scan's frame (wheel odometry, an IMU; the identity gives "constant pose").
 *     k >= 1, delta34 NULL:  constant velocity, G = P_{k-1} o (P_{k-2}^-1 o P_{k-1}), the inner product kept in double;
 *                            at k = 1 delta = the identity.
 *     G is rounded to float element by element and the registration starts from T_0 = double(G).
 *   Registration.  Exactly gm_register_map(ctx, map, icp with init_pose34 = G, max_planarity): the same launches and the
 *     same results, which gm_get_registration and gm_download_map_correspondences on ctx then report.  Step 0 with
 *     register_first = 0 does not register (a new map) and clears ctx's registration.
 *   Gate.  A registered step is accepted iff (double)fitness >= min_fitness and n_correspondences >= 6, with fitness and
 *     rmse the floats gm_get_registration computes.  An unregistered step 0 is always accepted.
 *   Insert.  An accepted step inserts all of ctx's compacted points at pose34 = float(T) element by element (what
 *     gm_get_registration returns): the map gm_map_insert(map, ctx, pose34, -1) would give.  A rejected step inserts nothing
 *     and records the guess as its pose, so the next guesses dead-reckon across it; its ICP result stays readable through
 *     gm_get_registration.  The gate is what keeps a failed registration out of the map: nothing removes what was inserted
 *     (a window, below, moves voxels to the archive but never drops a point unless its archive is NULL or full).
 *   Ordering.  A step is a map operation: it waits for the previous gm_map_insert / gm_register_map / gm_odometry_step on
 *     the map, whichever context issued it, and the next one waits for its insert.  There is no host synchronisation
 *     (the first registration of a context allocates its buffers once, as gm_register_map does).
 *   Launches.  A registered step launches k_odom_begin (the guess and the registration's start), k_map_planes,
 *     icp.max_iterations x k_regmap_iter, k_odom_gate and the insert: gm_launch_count(ctx) grows by max_iterations + 4.
 *     An unregistered step 0 launches k_odom_begin, k_odom_gate and the insert: + 3.  The insert is launched even for an
 *     empty scan (its kernel reads the point count on the device).  With a window, add GM_MAP_EVICT_LAUNCHES to each:
 *     max_iterations + 4 + GM_MAP_EVICT_LAUNCHES and 3 + GM_MAP_EVICT_LAUNCHES.
 *   Window (gm_odometry_set_window; off by default).  With half_cells > 0, each step ends, after its insert, with exactly the
 *     launches of gm_map_evict(map, ctx, archive, t, half_cells), t = (pose34[3], pose34[7], pose34[11]) of the step's own
 *     record, read from device memory: still no host round trip.  A rejected step evicts around its guess (its recorded
 *     pose); a centre gm_map_evict would refuse evicts nothing.  The step then also waits for and orders the archive as
 *     gm_map_evict does.  The window may be set or changed between steps; half_cells = 0 turns it off.  Rules: half_cells
 *     >= 0, and an archive (NULL = evicted voxels are dropped) must be another map of the same leaf on the map's device, or
 *     GM_ERR_INVALID_ARG.  The archive must outlive the odometry.
 *     Sizing.  With crop bound B (boxFilterBound), d_max = icp.max_correspondence_distance, and every ICP iterate of step
 *     k + 1 within s metres of step k's pose,
 *         half_cells >= floor((sqrt(3) * B + s + d_max) / leaf) + 2
 *     keeps every voxel the next registration can match (a scan point lies within sqrt(3) B of its sensor, one cell for
 *     the centre's rounding) and every neighbour its plane reads (one more cell), so the trajectory is the one without a
 *     window.  The local map then needs capacity for the voxels of a cube of 2 half_cells + 1 cells around the sensor,
 *     not for the run.
 *   Errors.  gm_odometry_create checks icp by gm_register_map's rules and 0 <= min_fitness <= 1, register_first in {0, 1},
 *     max_steps >= 1.  A step k >= max_steps gives GM_ERR_CAPACITY, a missing stage GM_ERR_STAGE_ORDER, a context on
 *     another device GM_ERR_INVALID_ARG: then nothing is launched and gm_odometry_steps does not move.
 * Destroy the odometry before its map. */
typedef struct gm_odometry gm_odometry;
typedef struct gm_odometry_params {
  gm_icp_params icp;        /* d_max, iterations, step thresholds, degeneracy_ratio as for gm_register_map; init_pose34 = the
                               first scan's pose in the map frame (register_first = 0) or the guess of it (1)                */
  double max_planarity;     /* as gm_register_map                                                 default 0.1  */
  double min_fitness;       /* the gate, see above                                                default 0.5  */
  int32_t register_first;   /* 0: step 0 inserts at init_pose34 without registering (a new map);
                               1: step 0 registers from init_pose34 (a map from gm_map_load, or one another odometry fills)
                                                                                                  default 0    */
  int32_t max_steps;        /* trajectory capacity, >= 1                                          default 4096 */
} gm_odometry_params;
typedef struct gm_odometry_record {
  float pose34[12];         /* the scan's pose in the map frame: the registered pose if accepted, else the guess */
  float guess34[12];        /* the prediction the step started from */
  int32_t accepted;         /* 1 = the scan was inserted into the map */
  int32_t registered;       /* 0 only for an unregistered step 0 */
  int32_t iterations, converged, n_source, n_correspondences, n_degenerate;
  float rmse, fitness;      /* as gm_get_registration reports them (0 for an unregistered step) */
  int32_t pad_;
} gm_odometry_record;
GM_API void gm_odometry_params_default(gm_odometry_params* p);
GM_API gm_status gm_odometry_create(gm_map* map, const gm_odometry_params* p, gm_odometry** out);
GM_API void gm_odometry_destroy(gm_odometry* odo);
GM_API gm_status gm_odometry_step(gm_odometry* odo, gm_ctx* ctx, const float* delta34 /* NULL = constant velocity */);
GM_API gm_status gm_odometry_set_window(gm_odometry* odo, int32_t half_cells /* 0 = off, the default */, gm_map* archive /* may be NULL */);
/* gm_odometry_deskew: gm_deskew of ctx's timed scan, the one the next gm_odometry_step (step k = gm_odometry_steps()) will
 * take, with the constant-velocity increment of the trajectory in device memory as the delta:
 *     delta = float(P_{k-2}^-1 o P_{k-1}) element by element (the guess's composition and order, above); the identity
 *     for k < 2, which leaves the points unchanged.
 * Launches: k_odom_delta (one thread, writes the 12 floats to ctx's delta slot), then gm_deskew's k_deskew reading them:
 *   gm_launch_count(ctx) grows by 2, with no host synchronisation.  The results are those of gm_deskew with that delta.
 * Ordering: it waits on ctx's stream for the map's last operation, i.e. for step k - 1 from whichever context issued it
 *   (the records it reads).  The cost: with two contexts taking turns, scan k's crop, normals and voxel stages can no
 *   longer overlap step k - 1's registration.  A caller with an IMU or wheel odometry calls gm_deskew with that delta
 *   instead and keeps the overlap.
 * Rules: those of gm_deskew for ctx, t_ref and period; GM_ERR_INVALID_ARG for a context on another device than the map;
 *   GM_ERR_CAPACITY when k >= max_steps.  Nothing is launched when a call is refused. */
#define GM_ODOMETRY_DESKEW_LAUNCHES 2
GM_API gm_status gm_odometry_deskew(gm_odometry* odo, gm_ctx* ctx, double t_ref, double period);
GM_API int32_t gm_odometry_steps(const gm_odometry* odo);  /* steps issued so far (host counter, no synchronisation) */
/* the records of every step issued so far, in step order; *n = their number.  Waits for the last of them.  out = NULL: *n only */
GM_API gm_status gm_odometry_get(gm_odometry* odo, gm_odometry_record* out, int32_t capacity, int32_t* n);

/* ---- multi-GPU data-path collectives over NVLink peer memory (SURVEY 8e; builder-defined: the reference is one process,
 * src/geometric_mapping.cpp:128-170) -------------------------------------------------------------------------------
 * One process per GPU.  Every rank creates a gm_comm (a mailbox in its own HBM), publishes its 64-byte handle
 * (cudaIpcMemHandle_t) to the others by any means (bench.py: one torch.distributed all_gather at start-up) and connects
 * with the table of all handles (world x 64 bytes, entry r = rank r).  After that the collectives of the data path are
 * kernels storing into the peers' mailboxes over NVLink and polling their own: no library call, no host round trip.
 *   gm_ransac_sharded        hypotheses [0,H) split over the ranks (every rank holds the same scan): count own share,
 *                            (count,id) MAX with the winner's coefficients through the mailboxes, refit -> same models
 *                            on every rank.  Replaces gm_ransac_pair + export/all-reduce/import + gm_ransac_select_pair.
 *   gm_allreduce_voxel_bbox  map slabs: MIN/MAX of the compacted clouds' bounding boxes (one VoxelGrid lattice)
 *   gm_allreduce_frame       map slabs: SUM of the scatter matrices, re-solved: getLocalFrame of the whole map
 * All ranks must issue the same sequence of these calls.  world = 1 works without peers (used by the tests). */
typedef struct gm_comm gm_comm;
GM_API gm_status gm_comm_create(int32_t rank, int32_t world, gm_comm** out);
GM_API gm_status gm_comm_handle(gm_comm* comm, void* handle_64_bytes);
GM_API gm_status gm_comm_connect(gm_comm* comm, const void* handles_world_x_64_bytes);
/* peers inside one process (several devices driven by one process): mailbox addresses instead of IPC handles */
GM_API gm_status gm_comm_mailbox(gm_comm* comm, void** mailbox_device_ptr);
GM_API gm_status gm_comm_connect_local(gm_comm* comm, void* const* mailboxes_world);
GM_API void gm_comm_destroy(gm_comm* comm);
GM_API int32_t gm_comm_rank(const gm_comm* comm);
GM_API int32_t gm_comm_world(const gm_comm* comm);
GM_API const char* gm_comm_last_error(const gm_comm* comm);
GM_API gm_status gm_set_comm(gm_ctx* ctx, gm_comm* comm);
GM_API gm_status gm_ransac_sharded(gm_ctx* ctx, const int32_t* plane_samples_host, int32_t Hp, const int32_t* cyl_samples_host, int32_t Hc);
GM_API gm_status gm_allreduce_voxel_bbox(gm_ctx* ctx);
GM_API gm_status gm_allreduce_frame(gm_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* GM_CAPI_H */
