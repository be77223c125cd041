// gm_capi.cu — context + C-ABI (include/gm_capi.h) of the B200-native per-scan hot path.
// There is no CPU fallback anywhere in this file: every stage is a sequence of CUDA kernel
// launches on the ctx stream, and gm_create() fails without a device.
#include "../../include/gm_capi.h"
#include "gm_sort.cuh"
#include "gm_ransac.cuh"
#include "gm_polyline.cuh"
#include "gm_compress.cuh"
#include "gm_primitives.cuh"
#include "gm_map.cuh"
#include "gm_comm.cuh"
#include "gm_register.cuh"
#include "gm_odometry.cuh"
#include "gm_deskew.cuh"
#include <new>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>

using namespace gm;

#include <vector>

namespace {
constexpr int GM_VERSION = 1;
constexpr int FRAME_BLOCKS = 296;
constexpr int REFIT_BLOCKS = 296;
constexpr size_t kPartialsRegion = (size_t)296 * 32;  // doubles per concurrent reduction

// profiling segments (gm_profile_*): one CUDA-event pair per segment per call
enum Seg {
  SEG_CROP, SEG_GRID_KEYS, SEG_GRID_SORT, SEG_GRID_BUILD, SEG_NORMALS, SEG_COMPACT, SEG_VOX_KEYS, SEG_VOX_SORT,
  SEG_VOX_REDUCE, SEG_VOX_NN, SEG_FRAME, SEG_PLANE_HYP, SEG_PLANE_COUNT, SEG_PLANE_ARGMAX, SEG_PLANE_REFIT,
  SEG_CYL_HYP, SEG_CYL_COUNT, SEG_CYL_ARGMAX, SEG_CYL_REFIT, SEG_LABEL, SEG_POLYLINE, SEG_COUNT
};
const char* kSegNames[SEG_COUNT] = {
  "crop", "grid_keys", "grid_sort", "grid_build", "normals", "compact", "voxel_keys", "voxel_sort",
  "voxel_reduce", "voxel_nn", "frame", "plane_hyp", "plane_count", "plane_argmax", "plane_refit",
  "cyl_hyp", "cyl_count", "cyl_argmax", "cyl_refit", "label", "polyline"};

struct SummaryDev {  // same layout as gm_scan_summary
  gm_counts counts;
  gm_frame frame;
  gm_model plane, cylinder;
  int32_t n_slices, pad_;
};
static_assert(sizeof(SummaryDev) == sizeof(gm_scan_summary), "summary layout");

__global__ void k_pack_summary(const DevState* st, const FrameOut* fr, const ModelState* ms, const PolyState* ps,
                               int held_mask, SummaryDev* out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  out->counts.n_input = st->n_input; out->counts.n_cropped = st->n_crop; out->counts.n_valid = st->n_valid;
  out->counts.n_voxels = st->vox.n_voxels; out->counts.n_cells = st->n_cells; out->counts.voxel_overflow = st->vox.overflow;
  out->counts.nn_out_of_range = st->nn_oor; out->counts.device_error = st->error;
  for (int k = 0; k < 3; ++k) out->frame.vals[k] = fr->vals[k];
  for (int k = 0; k < 9; ++k) { out->frame.vecs[k] = fr->vecs[k]; out->frame.scatter[k] = fr->scatter[k]; }
  for (int m = 0; m < 2; ++m) {
    gm_model* o = m == 0 ? &out->plane : &out->cylinder;
    const ModelState* i = ms + m;
    const bool have = (held_mask >> m) & 1;
    o->kind = m; o->best_id = have ? i->best_id : -1; o->best_count = have ? i->best_count : -1;
    o->refit_count = have ? i->refit_count : 0;
    for (int k = 0; k < 8; ++k) { o->hyp[k] = have ? i->hyp[k] : 0.f; o->coef[k] = have ? i->coef[k] : 0.f; }
    o->rms = have ? i->rms : 0.f; o->pad_ = 0.f;
  }
  out->n_slices = ((held_mask >> 2) & 1) ? ps->S : 0;
  out->pad_ = 0;
}

// One cudaMalloc'd array of `count` elements (at least one is allocated), freed with its owner.  Captured CUDA graphs
// hold the raw address: alloc() may only run where a new graph generation starts or before the first capture.
template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t count = 0;
  DevBuf() = default;
  DevBuf(DevBuf&& o) noexcept : p(o.p), count(o.count) { o.p = nullptr; o.count = 0; }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { reset(); }
  void reset() {
    if (p) cudaFree(p);
    p = nullptr;
    count = 0;
  }
  cudaError_t alloc(size_t n) {
    reset();
    cudaError_t e = cudaMalloc((void**)&p, std::max<size_t>(n, 1) * sizeof(T));
    if (e == cudaSuccess) count = n;
    return e;
  }
  operator T*() const { return p; }
  T* operator->() const { return p; }
};

// The RANSAC tables of one set of H hypotheses per kind (index = kind): sample indices, hypotheses, counts, the
// winner's key and its refitted model.
struct HypSet {
  DevBuf<int> samples[2];  // [3H] plane, [2H] cylinder
  DevBuf<float4> plane_coef;
  DevBuf<float> model7, test12;
  DevBuf<int> hvalid[2], counts[2];
  DevBuf<unsigned long long> key;  // [2]
  DevBuf<ModelState> model;        // [2]
  cudaError_t alloc(size_t H) {  // stops at the first failure and returns it
    cudaError_t e;
    (void)((e = samples[0].alloc(3 * H)) || (e = samples[1].alloc(2 * H)) || (e = plane_coef.alloc(H)) || (e = model7.alloc(7 * H)) ||
           (e = test12.alloc(12 * H)) || (e = hvalid[0].alloc(H)) || (e = hvalid[1].alloc(H)) || (e = counts[0].alloc(H)) ||
           (e = counts[1].alloc(H)) || (e = key.alloc(2)) || (e = model.alloc(2)));
    return e;
  }
};
}  // namespace

struct gm_ctx {
  gm_params prm;
  size_t cap = 0;   // max points
  int hcap = 0;     // max hypotheses
  int device = 0;
  int num_sms = 148;
  int gn_blocks = 148;  // cooperative grid of the cylinder refit
  cudaStream_t own_stream = nullptr, stream = nullptr;
  // gm_process_scan forks the independent stages of one scan onto these (joined before labels)
  cudaStream_t branch[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join[3] = {nullptr, nullptr, nullptr};
  bool concurrent = true;
  std::string err;
  int64_t launches = 0;

  // scan + valid stages
  size_t n_input = 0;
  const float4* d_scan = nullptr;  // points to d_in or to the caller's device buffer
  unsigned stages = 0;             // bit set over Stage
  bool injected = false;           // the compacted cloud came from gm_inject_compacted, not from this scan's normals
  int ransac_H[2] = {0, 0};
  GridSpec grid{};
  bool grid_box_set = false;
  double grid_box_min[3] = {0, 0, 0}, grid_box_max[3] = {0, 0, 0};
  OwnedRange own{-1, 0.f, 0.f};
  bool vox_bbox_set = false;
  bool vox_bbox_is_hint = false;  // the box only bounds the lattice (dense-table sizing); the real box is computed / all-reduced on the device
  float vox_bbox[6] = {0, 0, 0, 0, 0, 0};

  // device buffers
  DevBuf<unsigned char> d_raw;  // PointCloud2 staging (grown on demand)
  // per-point times of a timed PointCloud2 upload, and the delta gm_odometry_deskew hands k_deskew (12 floats); both
  // allocated by the first timed upload
  DevBuf<float> d_time, d_delta;
  bool scan_timed = false;   // the scan came from gm_upload_pointcloud2_timed: d_time holds its times
  bool deskew_open = false;  // gm_deskew may still run on it: timed, not deskewed, no gm_crop since the upload
  DevBuf<float4> d_in, d_crop, d_sorted, d_cloud_c;
  DevBuf<float4> d_sorted_valid, d_leaf_bounds;  // inputs of the tile-culled counting (written by k_normals)
  int count_mode = 0;  // 0 = tile-culled when the cell-sorted cloud exists, 1 = always brute force
  DevBuf<float4> d_normals, d_normals_c, d_centroid, d_nn_normal;
  DevBuf<unsigned> d_keys[2], d_vals[2];
  DevBuf<unsigned> d_ucell_key;
  DevBuf<int> d_cell_id, d_ucell_start, d_nbr, d_valid_map;
  DevBuf<int2> d_runs;
  DevBuf<int2> d_cell_nruns;  // per occupied cell: {number of runs, number of candidates}
  // dense VoxelGrid tables (sort-free path): count, voxel id and 3 fixed-point sums per key; the count of d_dense_cnt
  // is the number of keys the tables hold
  DevBuf<int> d_dense_cnt, d_dense_id;
  DevBuf<long long> d_dense_sum;
  DevBuf<unsigned long long> d_dense_state;  // look-back tile states of the scan over the tables
  int voxel_mode = 0;  // 0 = dense tables when the key range fits, 1 = always sort
  bool vox_assign_on_demand = false;  // the scan's VoxelGrid took the dense path, which leaves d_vkey_pt / d_assign unwritten
  int normals_mode = 0;  // 0 = neighbours summed in cell-run order (fast), 1 = in FLANN's (d2, index) order (bit-identical to the oracle)
  int knn_k = 0;         // > 0: k-nearest-neighbour normals (setKSearch) instead of the radius search
  double knn_max_radius = 0.0;  // > 0: only neighbours nearer than this count (FLANN's radius + max_nn form); 0 = plain k-NN
  DevBuf<int> d_knn_idx;  // optional M x k neighbour indices of the last gm_normals (gm_set_knn(.., keep_indices = 1))
  bool knn_keep = false;
  DevBuf<BlockEntry> d_tab;  // dense block table of the neighbour grid (1 << (key_bits - 6) entries)
  DevBuf<int> d_vkey_pt, d_assign, d_vox_start, d_vox_key, d_vox_count, d_nn_idx;
  DevBuf<unsigned char> d_labels;
  DevBuf<unsigned long long> d_state64;
  DevBuf<unsigned long long> d_state64_b;  // tile states of the cylinder-refit compaction (may run concurrently with the voxel branch)
  DevBuf<unsigned> d_rs_hist;              // segment histograms [segments][256]
  DevBuf<Rs2Aux> d_rs_aux;                 // group sums / totals / completion counter of one pass; zero between passes
  DevBuf<TileCtl> d_ctl;         // [3] launch control of the look-back kernels: d_state64 | d_state64_b | d_dense_state
  size_t n_grid = 0;             // n_input rounded up to a bucket: what grids are sized by (kernels read the true n on the device)
  DevBuf<DevState> d_st;
  DevBuf<double> d_partials;
  DevBuf<FrameOut> d_frame;
  // ransac (index = kind): the scan's hypothesis set, its samples staged from the host through h_samples
  HypSet hyp;
  int* h_samples[2] = {nullptr, nullptr};
  cudaEvent_t ev_samples[2] = {nullptr, nullptr};
  // polyline
  DevBuf<PolyState> d_poly;
  DevBuf<long long> d_poly_acc;
  DevBuf<unsigned long long> d_poly_part;  // per-block (min,max) of the polyline range pass
  DevBuf<float4> d_poly_list;  // the cylinder points the polyline passes walk (k_poly_range), count in d_counters[10]
  DevBuf<gm_slice> d_slices;
  DevBuf<SummaryDev> d_summary;
  // compression stage: residual (label 0) cloud and its voxel grid
  DevBuf<VoxState> d_res_vs;
  DevBuf<CompStats> d_comp;
  DevBuf<float4> d_res_pts, d_res_centroid;
  DevBuf<int> d_res_key_pt, d_res_assign, d_res_vox_start, d_res_vox_key, d_res_vox_count;
  DevBuf<double> d_comp_part;
  DevBuf<unsigned long long> d_comp_mm;
  DevBuf<unsigned> d_counters;  // last-block tickets: [0] frame, [1] plane refit, [2] cylinder GN
  DevBuf<float4> d_inl;         // compacted cylinder inliers
  // sequential multi-primitive extraction (gm_primitives.cuh), allocated by the first gm_extract_primitives.  Its
  // tickets, partials, look-back states and d_inl are the scratch gm_ransac uses (same stream order, never concurrent).
  DevBuf<float4> d_pr_sv, d_pr_cc, d_pr_lb;  // working copies with the claimed points blanked: cell-sorted cloud, compacted cloud, leaf bounds
  DevBuf<int> d_pr_rem;                      // R_r
  DevBuf<unsigned char> d_pr_ids;            // primitive id per compacted point
  DevBuf<unsigned> d_pr_draws[2];
  HypSet pr_hyp;                             // the hypothesis set of one extraction round
  DevBuf<PrimState> d_pr_state;
  // compression of the extracted primitives: the residual cloud goes to d_pr_sv, its centroids to d_pr_cc
  DevBuf<int> d_pr_assign, d_pr_vox_start, d_pr_vox_key, d_pr_vox_count;
  DevBuf<VoxState> d_pr_vs;
  DevBuf<PrimComp> d_pr_comp;
  DevBuf<CompStats> d_pr_stats;
  // CUDA-graph replay of gm_process_scan: the launch sequence of one scan depends only on (bucketed size, hypothesis
  // counts, parameters / modes), never on per-scan host values (tile epochs, barrier parities and the scan pointer
  // live in device memory), so it is captured once per key and replayed with ONE cudaGraphLaunch
  struct ScanGraph { int kind; size_t n_grid; int Hp, Hc; unsigned long long gen; int uses; cudaGraphExec_t exec; long long launches; unsigned long long stamp; };
  std::vector<ScanGraph> graphs;
  unsigned long long graph_gen = 0;   // bumped by every setter that changes what a scan launches
  unsigned long long graph_clock = 0;
  int graph_mode = 2;                 // 2 = auto (default): graphs for scans up to kGraphAutoPoints, plain launches above; 1 = always; 0 = never (GM_GRAPH / gm_set_graph_mode)
  bool samples_staged = false;        // the sample indices of the current call are already on their way to the device
  long long graph_replays = 0, graph_captures = 0;
  std::string graph_note;
  // peer-memory collectives (gm_comm.cuh); `sharded` marks a RANSAC round whose keys travel through the mailboxes
  struct gm_comm* comm = nullptr;
  bool sharded = false;
  DevBuf<double> d_frame_sums;  // [8] the 6 scatter sums of the last gm_local_frame, kept for gm_allreduce_frame
  // registration of this context's voxel centroids (gm_register with this context as the source), allocated by the first
  // call: block partials, last-block ticket, pose / result state, per-centroid correspondence and residual
  DevBuf<double> d_reg_part;
  DevBuf<unsigned> d_reg_ticket;
  DevBuf<RegState> d_reg_state;
  DevBuf<int> d_reg_idx;
  DevBuf<float> d_reg_res;
  cudaEvent_t ev_reg[2] = {nullptr, nullptr};  // target stream -> source stream, and back
  // gm_register_map: the matched map key per centroid (allocated by the first call), and which kind of target the last
  // registration had (0 = a context, whose correspondences are in d_reg_idx; 1 = a map, in d_reg_key)
  DevBuf<unsigned long long> d_reg_key;
  int reg_target = 0;
  // profiling
  bool profiling = false;
  std::vector<cudaEvent_t> ev_pool;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> seg_events[SEG_COUNT];
};

static const CommDev* comm_dev(const gm_ctx* ctx);  // device copy of the peer table of the attached gm_comm (or null)

namespace {
struct SegTimer {
  gm_ctx* ctx; cudaEvent_t e1 = nullptr; int seg;
  static cudaEvent_t get(gm_ctx* c) {
    if (!c->ev_pool.empty()) { cudaEvent_t e = c->ev_pool.back(); c->ev_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr; cudaEventCreate(&e); return e;
  }
  SegTimer(gm_ctx* c, int s) : ctx(c), seg(s) {  // s < 0: not timed
    if (!c->profiling || s < 0) return;
    cudaEvent_t e0 = get(c); e1 = get(c);
    cudaEventRecord(e0, c->stream);
    c->seg_events[s].push_back({e0, e1});
  }
  ~SegTimer() { if (e1) cudaEventRecord(e1, ctx->stream); }
};

// The results a context holds, in pipeline order.  A stage's entry point fails with GM_ERR_STAGE_ORDER unless the
// stages it reads are held, and marks its own stage.  Running a stage again does not drop the later ones.  A change
// of input drops a stage and everything after it: a new scan from CROP on, a new crop box or is_dense from CROP on, a
// new neighbour grid from NORMALS on (the compacted cloud too, even an injected one).  A new extraction drops the
// compression of the previous one (PRIMS_COMP), whose buffers it reuses.  REGISTRATION is the result of gm_register
// with this context as the source; only a new scan or grid here drops it.
enum Stage {
  SCAN, CROP, NORMALS, COMPACTED, VOXEL, FRAME, RANSAC_PLANE, RANSAC_CYL, MODEL_PLANE, MODEL_CYL, LABELS, POLY, COMP,
  PRIMS, PRIMS_COMP, REGISTRATION
};
inline Stage ransac_stage(int kind) { return Stage(RANSAC_PLANE + kind); }
inline Stage model_stage(int kind) { return Stage(MODEL_PLANE + kind); }

inline bool has(const gm_ctx* ctx, Stage s) { return (ctx->stages >> s) & 1u; }
template <class... S>
gm_status require(const gm_ctx* ctx, S... s) { return (has(ctx, s) && ...) ? GM_OK : GM_ERR_STAGE_ORDER; }
template <class... S>
void mark(gm_ctx* ctx, S... s) { ((ctx->stages |= 1u << s), ...); }
inline void invalidate_from(gm_ctx* ctx, Stage s) { ctx->stages &= (1u << s) - 1u; }

// Every setter that changes what a scan launches calls this: captured graphs of older generations are no longer used.
inline void new_graph_generation(gm_ctx* ctx) { ++ctx->graph_gen; }
}  // namespace

#define GM_CUDA(call)                                                                            \
  do {                                                                                           \
    cudaError_t e_ = (call);                                                                     \
    if (e_ != cudaSuccess) {                                                                     \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                             \
      return GM_ERR_CUDA;                                                                        \
    }                                                                                            \
  } while (0)

#define GM_LAUNCH(ctx, kernel, grid, block, ...)                                                 \
  do {                                                                                           \
    kernel<<<(grid), (block), 0, (ctx)->stream>>>(__VA_ARGS__);                                  \
    ++(ctx)->launches;                                                                           \
  } while (0)

#define GM_CHECK_LAUNCHES(ctx)                                                                   \
  do {                                                                                           \
    cudaError_t e_ = cudaGetLastError();                                                         \
    if (e_ != cudaSuccess) {                                                                     \
      (ctx)->err = std::string("kernel launch: ") + cudaGetErrorString(e_);                      \
      return GM_ERR_CUDA;                                                                        \
    }                                                                                            \
  } while (0)

namespace {

inline int div_up(long long a, long long b) { return (int)((a + b - 1) / b); }

// src/tunnel_processing.cpp:106: exp((curv + .001/weightingFactor)^2) -- note the precedence (mode 0); mode 1: exp(-(curv/wf)^2)
inline WeightLaw weight_law(const gm_params& p) {
  WeightLaw w;
  if (p.weight_mode == 1) { w.scale = 1.0 / p.weightingFactor; w.shift = 0.0; w.sgn = -1.0; }
  else { w.scale = 1.0; w.shift = .001 / p.weightingFactor; w.sgn = 1.0; }
  return w;
}

int bits_for(unsigned long long max_value) {
  int b = 0;
  while (b < 64 && (max_value >> b) != 0ull) ++b;
  return std::max(b, 1);
}

// Neighbour grid over a box (default: the crop cube; gm_set_grid_box narrows it to the region a map
// slab actually occupies): cell slightly larger than the search radius so that, with float rounding of
// the cell coordinate, every d < r neighbour lies in the 27-cell neighbourhood.  The cell grows when
// the box would need more than 2^24 blocks (dense block table) or 4092 cells on an axis.
GridSpec make_grid(const gm_params& p, const double* box_min, const double* box_max) {
  GridSpec g{};
  float rf = (float)p.neighborRadius;
  double bound = std::fabs(p.boxFilterBound);
  double lo[3], span[3];
  for (int a = 0; a < 3; ++a) {
    double mn = box_min ? std::max(box_min[a], -bound) : -bound, mx = box_max ? std::min(box_max[a], bound) : bound;
    if (!(mx > mn)) { mn = -bound; mx = bound; }
    lo[a] = mn; span[a] = mx - mn;
  }
  double cell = (double)rf * (1.0 + 1.0 / 256.0);
  if (!(cell > 0.0)) cell = 1e-3;
  const int kMaxDim = 4092;  // 1023 blocks of 4 cells: at most 10 block bits per axis (the sum is capped at 24 below)
  for (;;) {
    int total_bits = 0;
    bool ok = true;
    for (int a = 0; a < 3; ++a) {
      int dim = (int)std::floor(span[a] / cell) + 1;
      if (dim > kMaxDim) { ok = false; break; }
      dim = std::max(dim, 1);
      const int nb = (dim + 3) / 4;
      int bits = 1;
      while ((1 << bits) <= nb) ++bits;  // (1 << bits) > nb: block coordinate 2^bits - 1 is never used
      g.dim[a] = dim; g.bits[a] = bits;
      total_bits += bits;
    }
    if (ok && total_bits <= 24) break;
    cell *= 1.25;
  }
  g.bmin = std::min(g.bits[0], std::min(g.bits[1], g.bits[2]));
  for (int a = 0; a < 3; ++a) g.origin[a] = (float)lo[a];
  g.cell = (float)cell;
  g.inv_cell = (float)(1.0 / cell);
  g.key_bits = g.bits[0] + g.bits[1] + g.bits[2] + 6;
  g.sentinel = g.key_bits >= 32 ? 0xFFFFFFFFu : ((1u << g.key_bits) - 1u);
  return g;
}

bool same_grid(const GridSpec& a, const GridSpec& b) { return std::memcmp(&a, &b, sizeof(GridSpec)) == 0; }

gm_status ensure_block_table(gm_ctx* ctx);

// Recompute the neighbour grid from the params / grid box; a different grid invalidates the block
// table of the old one (rare path, synchronous).
gm_status regrid(gm_ctx* ctx) {
  const GridSpec old = ctx->grid;
  ctx->grid = make_grid(ctx->prm, ctx->grid_box_set ? ctx->grid_box_min : nullptr, ctx->grid_box_set ? ctx->grid_box_max : nullptr);
  if (!same_grid(old, ctx->grid)) {
    GM_CUDA(cudaStreamSynchronize(ctx->stream));
    // everything built on the old grid (runs, block table, normals, and whatever consumed them) is stale: the next stage
    // after gm_crop must be gm_normals again (GM_ERR_STAGE_ORDER otherwise), not a search over an empty table
    invalidate_from(ctx, NORMALS);
    ctx->d_tab.reset();  // forces reallocation + clear
    return ensure_block_table(ctx);
  }
  return GM_OK;
}

// (Re)allocate and zero the dense block table for the current grid.
gm_status ensure_block_table(gm_ctx* ctx) {
  const size_t need = (size_t)1 << (ctx->grid.key_bits - 6);
  if (need != ctx->d_tab.count) GM_CUDA(ctx->d_tab.alloc(need));
  GM_CUDA(cudaMemset(ctx->d_tab, 0, need * sizeof(BlockEntry)));
  GM_CUDA(cudaMemset(&ctx->d_st->tab_cells, 0, sizeof(int)));
  // cudaMemset runs on the legacy default stream, which does NOT order with this ctx's non-blocking streams:
  // without this the first kernels of the next call could run before (or while) the tables are cleared
  GM_CUDA(cudaDeviceSynchronize());
  return GM_OK;
}

// Grids are sized by the input size rounded up to a bucket (kernels read the true size from device state), so that
// scans of slightly different sizes -- a lidar never returns the same number of points twice -- share one CUDA graph.
constexpr size_t kGridBucket = 32768;
inline size_t grid_bucket(size_t n, size_t cap) { return n == 0 ? 0 : std::min(cap, (n + kGridBucket - 1) / kGridBucket * kGridBucket); }

// LSD radix sort of (d_keys[0], d_vals[0]) -> returns the buffer index holding the result: the segment form of gm_sort.cuh
// (byte-counter histograms, <= 592 segments, balanced digits of <= 8 bits, 2 launches per pass, no memsets).  Round 1's tile
// form (3 launches per pass) is kept as a baseline in tools/microbench/sort_v1.cuh.
gm_status radix_sort(gm_ctx* ctx, const int* n_ptr, size_t n_cap, int key_bits, int* result_buf) {
  const Rs2Plan plan = rs2_plan(n_cap, key_bits);
  if ((size_t)plan.segments * 256 > ctx->d_rs_hist.count) { ctx->err = "radix histogram capacity"; return GM_ERR_CAPACITY; }
  unsigned* const keys[2] = {ctx->d_keys[0], ctx->d_keys[1]};
  unsigned* const vals[2] = {ctx->d_vals[0], ctx->d_vals[1]};
  *result_buf = rs2_sort(ctx->stream, keys, vals, n_ptr, n_cap, key_bits, ctx->d_rs_hist, ctx->d_rs_aux, nullptr);
  ctx->launches += 2 * plan.passes;
  GM_CHECK_LAUNCHES(ctx);
  return GM_OK;
}

gm_status sync_state(gm_ctx* ctx, DevState* host) {
  GM_CUDA(cudaMemcpyAsync(host, ctx->d_st, sizeof(DevState), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  return GM_OK;
}

int n_crop(const DevState& h) { return h.n_crop; }
int n_valid(const DevState& h) { return h.n_valid; }
int n_voxels(const DevState& h) { return h.vox.n_voxels; }

struct Copy { void* dst; const void* src; size_t item_bytes; };

// Device -> host download of per-point or per-voxel arrays: reads the device counts into *h, fails with
// GM_ERR_CAPACITY unless count(*h) items fit `capacity`, then copies that many items to every non-null destination
// and waits for the copies unless `wait` is false.
gm_status download(gm_ctx* ctx, DevState* h, int (*count)(const DevState&), size_t capacity, std::initializer_list<Copy> copies,
                   bool wait = true) {
  gm_status s = sync_state(ctx, h);
  if (s != GM_OK) return s;
  const size_t n = (size_t)count(*h);
  if (n > capacity) return GM_ERR_CAPACITY;
  for (const Copy& c : copies)
    if (c.dst && n * c.item_bytes > 0) GM_CUDA(cudaMemcpyAsync(c.dst, c.src, n * c.item_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (wait) GM_CUDA(cudaStreamSynchronize(ctx->stream));
  return GM_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------
extern "C" {

void gm_params_default(gm_params* p) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  p->boxFilterBound = 5.0;     // include/geometric_mapping/paramHandler.hpp:26
  p->voxelGridLeafSize = .1;   // :27
  p->neighborRadius = .03;     // :28
  p->weightingFactor = .2;     // :29
  p->displayCloud = 1;         // :31
  p->displayNormals = 1;       // :32
  p->displayCenterAxis = 1;    // :33
  p->usePCLViz = 0;            // :36
  p->is_dense = 1;
  p->nn_index_mode = 0;
  p->ransacThreshold = 0.05;
  p->cylinderRadiusMin = 0.5;
  p->cylinderRadiusMax = 10.0;
  p->refitIterations = 5;
  p->maxSlices = 256;
  p->sliceLength = 1.0;
  p->weight_mode = 0;
  p->arrow_mode = 0;
}

const char* gm_status_string(gm_status s) {
  switch (s) {
    case GM_OK: return "ok";
    case GM_ERR_INVALID_ARG: return "invalid argument";
    case GM_ERR_NO_DEVICE: return "no CUDA device (this library has no CPU path)";
    case GM_ERR_CUDA: return "CUDA error";
    case GM_ERR_CAPACITY: return "capacity exceeded";
    case GM_ERR_STAGE_ORDER: return "stage called before its input was produced";
    case GM_WARN_VOXEL_OVERFLOW: return "VoxelGrid overflow rule: leaf too small, cloud returned unchanged";
    case GM_ERR_NN_INDEX_RANGE: return "1-NN index beyond the compacted normals (reference quirk B.3)";
    case GM_ERR_INTERNAL: return "device-side consistency check failed";
    case GM_ERR_NO_MODEL: return "no valid RANSAC hypothesis";
    default: return "unknown status";
  }
}

int32_t gm_version(void) { return GM_VERSION; }

static gm_status validate_params(const gm_params* p) {
  if (!p) return GM_ERR_INVALID_ARG;
  if (!(p->boxFilterBound > 0.0) || !(p->voxelGridLeafSize > 0.0) || !(p->neighborRadius > 0.0)) return GM_ERR_INVALID_ARG;
  if (p->weightingFactor == 0.0) return GM_ERR_INVALID_ARG;
  if (!(p->ransacThreshold > 0.0) || p->refitIterations < 0 || p->maxSlices < 1 || !(p->sliceLength > 0.0)) return GM_ERR_INVALID_ARG;
  if (p->weight_mode < 0 || p->weight_mode > 1 || p->arrow_mode < 0 || p->arrow_mode > 1) return GM_ERR_INVALID_ARG;
  return GM_OK;
}

gm_status gm_create(const gm_params* p, size_t max_points, int32_t max_hypotheses, gm_ctx** out) {
  if (!out) return GM_ERR_INVALID_ARG;
  *out = nullptr;
  if (validate_params(p) != GM_OK || max_points == 0 || max_points >= (1ull << 30) || max_hypotheses < 0) return GM_ERR_INVALID_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return GM_ERR_NO_DEVICE; }
  gm_ctx* ctx = new (std::nothrow) gm_ctx();
  if (!ctx) return GM_ERR_INTERNAL;
  ctx->prm = *p;
  ctx->cap = max_points;
  ctx->hcap = std::max(max_hypotheses, 1);
  const size_t N = max_points;
  const size_t H = (size_t)ctx->hcap;
  auto fail = [&](cudaError_t e, const char* what) {
    std::fprintf(stderr, "gm_create: %s: %s\n", what, cudaGetErrorString(e));
    gm_destroy(ctx);
    return GM_ERR_CUDA;
  };
  cudaError_t e;
  if ((e = cudaGetDevice(&ctx->device)) != cudaSuccess) return fail(e, "cudaGetDevice");
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, ctx->device)) != cudaSuccess) return fail(e, "cudaGetDeviceProperties");
  ctx->num_sms = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) return fail(e, "cudaStreamCreate");
  ctx->stream = ctx->own_stream;
#define A(buf, count) if ((e = ctx->buf.alloc(count)) != cudaSuccess) return fail(e, #buf)
  A(d_in, N); A(d_crop, N); A(d_sorted, N + 1); A(d_cloud_c, N);  // d_walk_runs reads candidates in pairs: one element of slack
  A(d_sorted_valid, N); A(d_leaf_bounds, 2 * ((N + 31) / 32));
  A(d_normals, 2 * N); A(d_normals_c, 2 * N); A(d_centroid, N); A(d_nn_normal, 2 * N);
  A(d_keys[0], N); A(d_keys[1], N); A(d_vals[0], N); A(d_vals[1], N);
  A(d_ucell_key, N + 1); A(d_cell_id, N); A(d_ucell_start, N + 1); A(d_nbr, N); A(d_valid_map, N);
  A(d_runs, GRID_RUNS * N); A(d_cell_nruns, N);
  A(d_vkey_pt, N); A(d_assign, N); A(d_vox_start, N + 1); A(d_vox_key, N); A(d_vox_count, N); A(d_nn_idx, N);
  A(d_labels, N);
  A(d_state64, (size_t)div_up((long long)N, CP_TILE) + 2); A(d_state64_b, (size_t)div_up((long long)N, CP_TILE) + 2);
  A(d_rs_hist, RS2_HIST_WORDS); A(d_rs_aux, 1);
  A(d_st, 1); A(d_ctl, 3); A(d_frame_sums, 8);
  A(d_partials, 3 * kPartialsRegion);  // 3 regions: frame | plane refit | cylinder GN (may run concurrently)
  A(d_frame, 1); A(hyp, H);
  A(d_poly, 1); A(d_summary, 1); A(d_res_vs, 1); A(d_comp, 1); A(d_res_pts, N); A(d_res_centroid, N); A(d_res_key_pt, N); A(d_res_assign, N);
  A(d_res_vox_start, N + 1); A(d_res_vox_key, N); A(d_res_vox_count, N); A(d_comp_part, (size_t)CS_NV * (div_up((long long)N, CP_TILE) + 1) + 1024); A(d_comp_mm, (size_t)6 * (div_up((long long)N, CP_TILE) + 1)); A(d_counters, 16); A(d_poly_part, 2 * 4096); A(d_poly_list, 2 * N); A(d_inl, N); A(d_poly_acc, (size_t)POLY_NACC * (size_t)std::max(p->maxSlices, 1)); A(d_slices, (size_t)std::max(p->maxSlices, 1));
#undef A
  if ((e = cudaMallocHost((void**)&ctx->h_samples[0], 3 * H * sizeof(int))) != cudaSuccess) return fail(e, "h_samples0");
  if ((e = cudaMallocHost((void**)&ctx->h_samples[1], 2 * H * sizeof(int))) != cudaSuccess) return fail(e, "h_samples1");
  for (int k = 0; k < 2; ++k)
    if ((e = cudaEventCreateWithFlags(&ctx->ev_samples[k], cudaEventDisableTiming)) != cudaSuccess) return fail(e, "event");
  if ((e = cudaMemset(ctx->d_st, 0, sizeof(DevState))) != cudaSuccess) return fail(e, "memset");
  if ((e = cudaMemset(ctx->d_rs_aux, 0, sizeof(Rs2Aux))) != cudaSuccess) return fail(e, "memset");
  if ((e = cudaMemset(ctx->d_ctl, 0, 3 * sizeof(TileCtl))) != cudaSuccess) return fail(e, "memset");
  if ((e = cudaMemset(ctx->d_state64, 0, ((size_t)div_up((long long)N, CP_TILE) + 2) * sizeof(unsigned long long))) != cudaSuccess) return fail(e, "memset");
  if ((e = cudaMemset(ctx->d_state64_b, 0, ((size_t)div_up((long long)N, CP_TILE) + 2) * sizeof(unsigned long long))) != cudaSuccess) return fail(e, "memset");
  for (int b = 0; b < 3; ++b) {
    if ((e = cudaStreamCreateWithFlags(&ctx->branch[b], cudaStreamNonBlocking)) != cudaSuccess) return fail(e, "branch stream");
    if ((e = cudaEventCreateWithFlags(&ctx->ev_join[b], cudaEventDisableTiming)) != cudaSuccess) return fail(e, "event");
  }
  if ((e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)) != cudaSuccess) return fail(e, "event");
  { const char* env = std::getenv("GM_SERIAL"); ctx->concurrent = !(env && env[0] == '1'); }
  { const char* env = std::getenv("GM_COUNT_MODE"); ctx->count_mode = (env && env[0] == '1') ? 1 : 0; }
  { const char* env = std::getenv("GM_VOXEL_MODE"); ctx->voxel_mode = (env && env[0] == '1') ? 1 : 0; }
  { const char* env = std::getenv("GM_GRAPH"); ctx->graph_mode = env ? std::max(0, std::min(2, std::atoi(env))) : 2; }
  { const char* env = std::getenv("GM_NORMALS_MODE"); ctx->normals_mode = (env && env[0] == '1') ? 1 : 0; }

  if ((e = cudaMemset(ctx->hyp.key, 0, 2 * sizeof(unsigned long long))) != cudaSuccess) return fail(e, "memset");
  if ((e = cudaMemset(ctx->d_counters, 0, 16 * sizeof(unsigned))) != cudaSuccess) return fail(e, "memset");
  if ((e = cudaMemset(ctx->hyp.model, 0, 2 * sizeof(ModelState))) != cudaSuccess) return fail(e, "memset");
  {
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_cyl_gn_all, RF_BLOCK, 0)) != cudaSuccess) return fail(e, "occupancy");
    ctx->gn_blocks = std::max(1, std::min(ctx->num_sms, per_sm * ctx->num_sms));
    if ((size_t)ctx->gn_blocks * 2 * GN_NV > kPartialsRegion) return fail(cudaErrorInvalidValue, "partials capacity");
  }
  if ((e = cudaDeviceSynchronize()) != cudaSuccess) return fail(e, "sync");  // the memsets above ran on the legacy stream
  ctx->grid = make_grid(ctx->prm, nullptr, nullptr);
  if (ensure_block_table(ctx) != GM_OK) { std::fprintf(stderr, "gm_create: %s\n", ctx->err.c_str()); gm_destroy(ctx); return GM_ERR_CUDA; }
  *out = ctx;
  return GM_OK;
}

void gm_destroy(gm_ctx* ctx) {
  if (!ctx) return;
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  for (int k = 0; k < 2; ++k) {
    if (ctx->h_samples[k]) cudaFreeHost(ctx->h_samples[k]);
    if (ctx->ev_samples[k]) cudaEventDestroy(ctx->ev_samples[k]);
  }
  for (auto& g : ctx->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  for (auto& v : ctx->seg_events) for (auto& pr : v) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
  for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
  for (int b = 0; b < 3; ++b) { if (ctx->branch[b]) cudaStreamDestroy(ctx->branch[b]); if (ctx->ev_join[b]) cudaEventDestroy(ctx->ev_join[b]); }
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  for (cudaEvent_t e : ctx->ev_reg) if (e) cudaEventDestroy(e);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  delete ctx;  // frees the device buffers
}

gm_status gm_set_params(gm_ctx* ctx, const gm_params* p) {
  if (!ctx || validate_params(p) != GM_OK) return GM_ERR_INVALID_ARG;
  new_graph_generation(ctx);
  if (p->maxSlices > ctx->prm.maxSlices) { ctx->err = "maxSlices cannot grow after gm_create"; return GM_ERR_CAPACITY; }
  if (p->boxFilterBound != ctx->prm.boxFilterBound || p->is_dense != ctx->prm.is_dense) invalidate_from(ctx, CROP);  // the crop itself is stale
  ctx->prm = *p;
  return regrid(ctx);
}

gm_status gm_get_params(const gm_ctx* ctx, gm_params* out) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  *out = ctx->prm;
  return GM_OK;
}

gm_status gm_set_grid_box(gm_ctx* ctx, const float* min3, const float* max3) {
  if (!ctx || ((min3 == nullptr) != (max3 == nullptr))) return GM_ERR_INVALID_ARG;
  new_graph_generation(ctx);
  if (min3 && ctx->knn_k > 0) { ctx->err = "k-NN normals need the default neighbour grid"; return GM_ERR_INVALID_ARG; }
  ctx->grid_box_set = min3 != nullptr;
  if (min3) {
    for (int a = 0; a < 3; ++a) {
      if (!(max3[a] >= min3[a])) return GM_ERR_INVALID_ARG;
      ctx->grid_box_min[a] = min3[a]; ctx->grid_box_max[a] = max3[a];
    }
  }
  return regrid(ctx);
}

gm_status gm_set_owned_range(gm_ctx* ctx, int32_t axis, float lo, float hi) {
  if (!ctx || axis > 2 || (axis >= 0 && !(hi >= lo))) return GM_ERR_INVALID_ARG;
  new_graph_generation(ctx);
  ctx->own.axis = axis < 0 ? -1 : axis;
  ctx->own.lo = lo; ctx->own.hi = hi;
  return GM_OK;
}

gm_status gm_set_voxel_bbox(gm_ctx* ctx, const float* min3, const float* max3) {
  if (!ctx || ((min3 == nullptr) != (max3 == nullptr))) return GM_ERR_INVALID_ARG;
  new_graph_generation(ctx);
  ctx->vox_bbox_set = min3 != nullptr;
  ctx->vox_bbox_is_hint = false;
  if (min3) for (int a = 0; a < 3; ++a) { ctx->vox_bbox[a] = min3[a]; ctx->vox_bbox[3 + a] = max3[a]; }
  return GM_OK;
}

gm_status gm_set_voxel_bbox_hint(gm_ctx* ctx, const float* min3, const float* max3) {
  gm_status s = gm_set_voxel_bbox(ctx, min3, max3);
  if (s == GM_OK) ctx->vox_bbox_is_hint = min3 != nullptr;
  return s;
}

gm_status gm_get_search_stats(gm_ctx* ctx, int64_t* candidates, int64_t* neighbors) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, NORMALS)) return s;
  DevState h;
  gm_status s = sync_state(ctx, &h);
  if (s != GM_OK) return s;
  if (candidates) *candidates = (int64_t)h.n_candidates;
  if (neighbors) *neighbors = (int64_t)h.n_neighbors;
  return GM_OK;
}

gm_status gm_get_voxel_bbox(gm_ctx* ctx, float* min3, float* max3) {
  if (!ctx || !min3 || !max3) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, COMPACTED)) return s;
  DevState h;
  gm_status s = sync_state(ctx, &h);
  if (s != GM_OK) return s;
  auto dec = [](int i) { int b = (i >= 0) ? i : (i ^ 0x7FFFFFFF); float f; std::memcpy(&f, &b, 4); return f; };
  for (int a = 0; a < 3; ++a) { min3[a] = dec(h.vox.bbox_min[a]); max3[a] = dec(h.vox.bbox_max[a]); }
  return GM_OK;
}

gm_status gm_set_stream(gm_ctx* ctx, void* cuda_stream) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  new_graph_generation(ctx);
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
  return GM_OK;
}

gm_status gm_set_voxel_mode(gm_ctx* ctx, int32_t mode) {
  if (!ctx || (mode != 0 && mode != 1)) return GM_ERR_INVALID_ARG;
  new_graph_generation(ctx);
  ctx->voxel_mode = mode;
  return GM_OK;
}

gm_status gm_set_normals_mode(gm_ctx* ctx, int32_t mode) {
  if (!ctx || (mode != 0 && mode != 1)) return GM_ERR_INVALID_ARG;
  new_graph_generation(ctx);
  ctx->normals_mode = mode;
  return GM_OK;
}

gm_status gm_set_knn(gm_ctx* ctx, int32_t k, int32_t keep_indices) {
  if (!ctx || k < 0 || k > KNN_MAX) return GM_ERR_INVALID_ARG;
  new_graph_generation(ctx);
  if (k > 0 && ctx->grid_box_set) { ctx->err = "k-NN normals need the default neighbour grid (the crop cube): clear gm_set_grid_box first"; return GM_ERR_INVALID_ARG; }
  ctx->knn_k = k;
  ctx->knn_keep = k > 0 && keep_indices != 0;
  return GM_OK;
}

gm_status gm_set_knn_max_radius(gm_ctx* ctx, double max_radius) {
  if (!ctx || !(max_radius >= 0.0)) return GM_ERR_INVALID_ARG;
  new_graph_generation(ctx);
  ctx->knn_max_radius = max_radius;
  return GM_OK;
}

gm_status gm_download_knn_indices(gm_ctx* ctx, int32_t* out, size_t capacity_points) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, NORMALS)) return s;
  if (ctx->knn_k <= 0 || !ctx->knn_keep || !ctx->d_knn_idx) return GM_ERR_STAGE_ORDER;
  DevState h;
  return download(ctx, &h, n_crop, capacity_points, {{out, ctx->d_knn_idx, ctx->knn_k * sizeof(int)}});
}

gm_status gm_set_count_mode(gm_ctx* ctx, int32_t mode) {
  if (!ctx || (mode != 0 && mode != 1)) return GM_ERR_INVALID_ARG;
  new_graph_generation(ctx);
  ctx->count_mode = mode;
  return GM_OK;
}

const char* gm_last_error(const gm_ctx* ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }
int64_t gm_launch_count(const gm_ctx* ctx) { return ctx ? ctx->launches : 0; }
void gm_reset_launch_count(gm_ctx* ctx) { if (ctx) ctx->launches = 0; }
gm_status gm_synchronize(gm_ctx* ctx) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  return GM_OK;
}

// A new input cloud: nothing computed from the previous one is valid any more.
static void new_scan(gm_ctx* ctx, size_t n) {
  ctx->n_input = n;
  ctx->n_grid = grid_bucket(n, ctx->cap);
  invalidate_from(ctx, CROP);
  mark(ctx, SCAN);
  ctx->injected = false;
  ctx->scan_timed = ctx->deskew_open = false;
}

static gm_status begin_scan(gm_ctx* ctx, size_t n) {
  new_scan(ctx, n);
  GM_LAUNCH(ctx, k_begin_scan, 1, 32, ctx->d_st, (int)n, ctx->d_scan);
  GM_CHECK_LAUNCHES(ctx);
  return GM_OK;
}

gm_status gm_upload_scan(gm_ctx* ctx, const float* xyz_host, size_t n, size_t stride_bytes) {
  if (!ctx || (n && !xyz_host) || stride_bytes < 12) return GM_ERR_INVALID_ARG;
  if (n > ctx->cap) { ctx->err = "scan larger than max_points"; return GM_ERR_CAPACITY; }
  if (n) {
    if (stride_bytes == 16) {
      GM_CUDA(cudaMemcpyAsync(ctx->d_in, xyz_host, n * 16, cudaMemcpyHostToDevice, ctx->stream));
    } else {
      size_t width = std::min<size_t>(stride_bytes, 16);
      GM_CUDA(cudaMemcpy2DAsync(ctx->d_in, 16, xyz_host, stride_bytes, width, n, cudaMemcpyHostToDevice, ctx->stream));
      GM_LAUNCH(ctx, k_set_w_one, div_up((long long)n, 256), 256, ctx->d_in, (int)n);
    }
  }
  ctx->d_scan = ctx->d_in;
  return begin_scan(ctx, n);
}

// ot < 0: untimed (gm_upload_pointcloud2); else the float32 time at byte offset ot goes to d_time
static gm_status upload_pointcloud2(gm_ctx* ctx, const void* data_host, size_t n, size_t point_step, size_t ox, size_t oy, size_t oz, long long ot) {
  if (!ctx || (n && !data_host) || point_step < 4 || ox + 4 > point_step || oy + 4 > point_step || oz + 4 > point_step ||
      (ot >= 0 && (size_t)ot + 4 > point_step))
    return GM_ERR_INVALID_ARG;
  if (n > ctx->cap) { ctx->err = "scan larger than max_points"; return GM_ERR_CAPACITY; }
  const bool timed = ot >= 0;
  if (timed && !ctx->d_time) {  // not on the per-scan fast path: only the first timed upload
    GM_CUDA(cudaStreamSynchronize(ctx->stream));
    GM_CUDA(ctx->d_time.alloc(ctx->cap));
    GM_CUDA(ctx->d_delta.alloc(12));
  }
  if (n) {
    const size_t bytes = n * point_step;
    if (bytes > ctx->d_raw.count) {  // not on the per-scan fast path: only when a larger message arrives
      GM_CUDA(cudaStreamSynchronize(ctx->stream));
      GM_CUDA(ctx->d_raw.alloc(ctx->cap * point_step));
    }
    GM_CUDA(cudaMemcpyAsync(ctx->d_raw, data_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (timed)
      GM_LAUNCH(ctx, k_decode_pointcloud2<true>, div_up((long long)n, 256), 256, ctx->d_raw, (int)n, (int)point_step, (int)ox, (int)oy, (int)oz, ctx->d_in,
                (int)ot, ctx->d_time);
    else
      GM_LAUNCH(ctx, k_decode_pointcloud2<false>, div_up((long long)n, 256), 256, ctx->d_raw, (int)n, (int)point_step, (int)ox, (int)oy, (int)oz, ctx->d_in,
                0, nullptr);
  }
  ctx->d_scan = ctx->d_in;
  gm_status s = begin_scan(ctx, n);
  if (s == GM_OK) ctx->scan_timed = ctx->deskew_open = timed;
  return s;
}

gm_status gm_upload_pointcloud2(gm_ctx* ctx, const void* data_host, size_t n, size_t point_step, size_t ox, size_t oy, size_t oz) {
  return upload_pointcloud2(ctx, data_host, n, point_step, ox, oy, oz, -1);
}

gm_status gm_upload_pointcloud2_timed(gm_ctx* ctx, const void* data_host, size_t n, size_t point_step, size_t ox, size_t oy, size_t oz, size_t ot) {
  if (ot > (size_t)INT32_MAX) return GM_ERR_INVALID_ARG;
  return upload_pointcloud2(ctx, data_host, n, point_step, ox, oy, oz, (long long)ot);
}

gm_status gm_download_point_times(gm_ctx* ctx, float* out, size_t capacity_points) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  if (!ctx->scan_timed) return GM_ERR_STAGE_ORDER;
  if (ctx->n_input > capacity_points) return GM_ERR_CAPACITY;
  if (ctx->n_input) GM_CUDA(cudaMemcpyAsync(out, ctx->d_time, ctx->n_input * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  return GM_OK;
}

// gm_deskew's rules (the caller checks the delta): GM_ERR_INVALID_ARG for t_ref or period, GM_ERR_STAGE_ORDER unless
// the scan may still be deskewed
static gm_status deskew_check(gm_ctx* ctx, double t_ref, double period) {
  if (!std::isfinite(t_ref) || !std::isfinite(period) || !(period > 0.0)) return GM_ERR_INVALID_ARG;
  if (!has(ctx, SCAN) || !ctx->deskew_open) return GM_ERR_STAGE_ORDER;
  return GM_OK;
}

// The one launch of k_deskew over the scan, with the delta from the host (delta_dev null) or from device memory.
static gm_status deskew_launch(gm_ctx* ctx, const Pose34& delta, const float* delta_dev, double t_ref, double period) {
  const int blocks = std::max(1, std::min(div_up((long long)ctx->n_input, DSK_BLOCK), ctx->num_sms * 16));
  GM_LAUNCH(ctx, k_deskew, blocks, DSK_BLOCK, ctx->d_st, ctx->d_in, ctx->d_time, delta, delta_dev, t_ref, period);
  GM_CHECK_LAUNCHES(ctx);
  ctx->deskew_open = false;
  return GM_OK;
}

gm_status gm_deskew(gm_ctx* ctx, const float* delta34, double t_ref, double period) {
  if (!ctx || !delta34) return GM_ERR_INVALID_ARG;
  for (int e = 0; e < 12; ++e)
    if (!std::isfinite(delta34[e])) return GM_ERR_INVALID_ARG;
  if (gm_status s = deskew_check(ctx, t_ref, period)) return s;
  Pose34 delta;
  std::memcpy(delta.r, delta34, sizeof(delta.r));
  return deskew_launch(ctx, delta, nullptr, t_ref, period);
}

gm_status gm_set_scan_device(gm_ctx* ctx, const float* xyzw_device, size_t n) {
  if (!ctx || (n && !xyzw_device)) return GM_ERR_INVALID_ARG;
  if (n > ctx->cap) { ctx->err = "scan larger than max_points"; return GM_ERR_CAPACITY; }
  ctx->d_scan = (const float4*)xyzw_device;
  return begin_scan(ctx, n);
}

// ---- a1 --------------------------------------------------------------------------------------
gm_status gm_crop(gm_ctx* ctx) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, SCAN)) return s;
  const size_t n = ctx->n_grid;
  if (n) {
    float hi = (float)ctx->prm.boxFilterBound, lo = (float)(-ctx->prm.boxFilterBound);
    SegTimer seg_(ctx, SEG_CROP);
    GM_LAUNCH(ctx, k_crop, div_up((long long)n, CPL_TILE), CP_BLOCK, ctx->d_st, lo, hi, ctx->prm.is_dense,
              ctx->d_crop, ctx->d_state64, ctx->d_ctl + 0, ctx->d_st);
    GM_CHECK_LAUNCHES(ctx);
  }
  mark(ctx, CROP);
  ctx->deskew_open = false;
  return GM_OK;
}


// ---- a2 + a3 ---------------------------------------------------------------------------------
gm_status gm_normals(gm_ctx* ctx) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, CROP)) return s;
  const size_t n = ctx->n_grid;  // upper bound of M (bucketed)
  if (n) {
    const int* n_ptr = &ctx->d_st->n_crop;
    const GridSpec g = ctx->grid;
    int blocks = std::min(div_up((long long)n, 256), ctx->num_sms * 16);
    { SegTimer seg_(ctx, SEG_GRID_KEYS);
      GM_LAUNCH(ctx, k_cell_keys, blocks, 256, ctx->d_crop, n_ptr, g, ctx->d_keys[0], ctx->d_vals[0]); }
    int buf = 0;
    gm_status s;
    { SegTimer seg_(ctx, SEG_GRID_SORT);
      s = radix_sort(ctx, n_ptr, n, g.key_bits, &buf); }
    if (s != GM_OK) return s;
    { SegTimer seg_(ctx, SEG_GRID_BUILD);
    GM_LAUNCH(ctx, k_clear_blocks, std::min(div_up((long long)n, 256), ctx->num_sms * 8), 256, ctx->d_ucell_key, ctx->d_st, g.sentinel, ctx->d_tab);
    GM_LAUNCH(ctx, k_cell_heads, div_up((long long)n, CPL_TILE), CP_BLOCK, ctx->d_keys[buf], ctx->d_vals[buf], ctx->d_crop, n_ptr,
              g.sentinel, ctx->d_sorted, ctx->d_cell_id, ctx->d_ucell_key, ctx->d_ucell_start, ctx->d_tab, ctx->d_state64, ctx->d_ctl + 0, ctx->d_st);
    GM_LAUNCH(ctx, k_cell_runs, std::min(div_up((long long)n, 128), ctx->num_sms * 16), 128, ctx->d_ucell_key,
              ctx->d_ucell_start, ctx->d_tab, ctx->d_st, g, ctx->d_runs, ctx->d_cell_nruns); }
    // pcl::KdTreeFLANN::radiusSearch hands FLANN static_cast<float>(radius * radius), the product taken in double
    const float r2 = (float)(ctx->prm.neighborRadius * ctx->prm.neighborRadius);
    { SegTimer seg_(ctx, SEG_NORMALS);
      if (ctx->knn_k > 0) {
        const int K = ctx->knn_k;
        int* idx_out = nullptr;
        if (ctx->knn_keep) {
          const size_t need = ctx->cap * (size_t)K;
          if (need > ctx->d_knn_idx.count) {  // rare path (first use / larger k)
            GM_CUDA(cudaStreamSynchronize(ctx->stream));
            GM_CUDA(ctx->d_knn_idx.alloc(need));
          }
          idx_out = ctx->d_knn_idx;
        }
        k_normals_knn<<<div_up((long long)n, KNN_BLOCK), KNN_BLOCK, (size_t)(K + KNN_AUX) * KNN_BLOCK * sizeof(unsigned long long), ctx->stream>>>(
            ctx->d_sorted, ctx->d_crop, ctx->d_cell_id, ctx->d_runs, ctx->d_cell_nruns, ctx->d_tab, ctx->d_ucell_start, n_ptr, g, K,
            ctx->knn_max_radius > 0.0 ? (float)(ctx->knn_max_radius * ctx->knn_max_radius) : HUGE_VALF, ctx->d_normals,
            ctx->d_nbr, ctx->d_sorted_valid, ctx->d_leaf_bounds, ctx->own, ctx->d_st, idx_out);
        ++ctx->launches;
      } else if (ctx->normals_mode == 1) {
        GM_LAUNCH(ctx, k_normals<1>, div_up((long long)n, NRM_BLOCK), NRM_BLOCK, ctx->d_sorted, ctx->d_cell_id, ctx->d_runs, ctx->d_cell_nruns, n_ptr, r2,
                  ctx->d_normals, ctx->d_nbr, ctx->d_sorted_valid, ctx->d_leaf_bounds, ctx->own, ctx->d_st);
      } else {
        GM_LAUNCH(ctx, k_normals<0>, div_up((long long)n, NRM_BLOCK), NRM_BLOCK, ctx->d_sorted, ctx->d_cell_id, ctx->d_runs, ctx->d_cell_nruns, n_ptr, r2,
                  ctx->d_normals, ctx->d_nbr, ctx->d_sorted_valid, ctx->d_leaf_bounds, ctx->own, ctx->d_st);
      } }
    { SegTimer seg_(ctx, SEG_COMPACT);
      GM_LAUNCH(ctx, k_compact_valid, div_up((long long)n, CP_TILE), CP_BLOCK, ctx->d_crop, ctx->d_normals, n_ptr, ctx->d_cloud_c,
                ctx->d_normals_c, ctx->d_valid_map, ctx->d_state64, ctx->d_ctl + 0, ctx->d_st, ctx->own); }
    GM_CHECK_LAUNCHES(ctx);
  }
  mark(ctx, NORMALS, COMPACTED);
  ctx->injected = false;
  return GM_OK;
}

// ---- a4 --------------------------------------------------------------------------------------
namespace {
struct VoxBuffers { int *key_pt, *assign, *vox_start, *vox_key, *vox_count; float4* centroid; };

constexpr size_t kDenseMaxKeys = (size_t)1 << 23;  // 8M keys x 32 B = 256 MB of tables at most

// Make the dense tables hold `range` keys (zero-initialised; they clean themselves afterwards).  Rare path.
gm_status ensure_dense(gm_ctx* ctx, size_t range) {
  if (range <= ctx->d_dense_cnt.count) return GM_OK;
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int b = 0; b < 3; ++b) if (ctx->branch[b]) GM_CUDA(cudaStreamSynchronize(ctx->branch[b]));
  ctx->d_dense_cnt.reset();  // holds the capacity: allocated last, so that a failure below leaves it 0
  const size_t ntiles = (size_t)div_up((long long)range, CPL_TILE) + 2;
  GM_CUDA(ctx->d_dense_state.alloc(ntiles));
  GM_CUDA(cudaMemset(ctx->d_dense_state, 0, ntiles * sizeof(unsigned long long)));
  GM_CUDA(ctx->d_dense_id.alloc(range));
  GM_CUDA(ctx->d_dense_sum.alloc(3 * range));
  GM_CUDA(ctx->d_dense_cnt.alloc(range));
  GM_CUDA(cudaMemset(ctx->d_dense_cnt, 0, range * sizeof(int)));
  GM_CUDA(cudaMemset(ctx->d_dense_id, 0, range * sizeof(int)));
  GM_CUDA(cudaMemset(ctx->d_dense_sum, 0, 3 * range * sizeof(long long)));
  GM_CUDA(cudaDeviceSynchronize());  // legacy-stream memsets do not order with the ctx's non-blocking streams (this raced: zero centroids)
  return GM_OK;
}

bool dense_voxel_path(const gm_ctx* ctx, size_t key_range) { return ctx->voxel_mode == 0 && key_range > 0 && key_range <= kDenseMaxKeys; }

// pcl::VoxelGrid of `pts` (vs->n points, bbox already in vs).  `key_range` = host-side upper bound of the number
// of lattice cells (0 = unknown).  Small enough: dense tables, no sort (2 launches, a 3rd for the per-point key and
// voxel id in o.key_pt / o.assign unless `assign` is false); else keys -> sort -> heads -> centroids, which always
// writes them.  Both give the same voxels in the same order with the same fixed-point centroids.
gm_status voxel_downsample(gm_ctx* ctx, const float4* pts, VoxState* vs, size_t n_cap, int key_bits, size_t key_range, const VoxBuffers& o,
                           int* sorted_buf, bool assign = true) {
  const float leaf_f = (float)ctx->prm.voxelGridLeafSize;
  const float inv = 1.0f / leaf_f;
  int blocks = std::min(div_up((long long)n_cap, 256), ctx->num_sms * 16);
  gm_status s;
  if (dense_voxel_path(ctx, key_range)) {
    if ((s = ensure_dense(ctx, key_range)) != GM_OK) return s;
    { SegTimer seg_(ctx, SEG_VOX_KEYS);
      if (pts == ctx->d_cloud_c && has(ctx, NORMALS) && !ctx->injected) {
        // the scan's own compacted cloud: accumulate over its cell-sorted copy with warp-combined atomics
        GM_LAUNCH(ctx, k_voxel_accumulate_sorted, blocks, 256, ctx->d_sorted_valid, &ctx->d_st->n_crop, vs, inv,
                  ctx->d_dense_cnt, (unsigned long long*)ctx->d_dense_sum.p, (int)key_range, &ctx->d_st->error);
      } else {
        GM_LAUNCH(ctx, k_voxel_accumulate, blocks, 256, pts, vs, inv, ctx->d_dense_cnt, (unsigned long long*)ctx->d_dense_sum.p,
                  (int)key_range, &ctx->d_st->error);
      } }
    { SegTimer seg_(ctx, SEG_VOX_REDUCE);
      GM_LAUNCH(ctx, k_voxel_dense_scan, div_up((long long)key_range, CPL_TILE), CP_BLOCK, ctx->d_dense_cnt, ctx->d_dense_sum, ctx->d_dense_id,
                (int)key_range, o.vox_key, o.vox_count, o.centroid, ctx->d_dense_state, ctx->d_ctl + 2, vs, &ctx->d_st->error);
      if (assign) GM_LAUNCH(ctx, k_voxel_assign, blocks, 256, pts, vs, inv, ctx->d_dense_id, (int)key_range, o.key_pt, o.assign); }
    *sorted_buf = 0;
    GM_CHECK_LAUNCHES(ctx);
    return GM_OK;
  }
  { SegTimer seg_(ctx, SEG_VOX_KEYS);
    GM_LAUNCH(ctx, k_voxel_keys, blocks, 256, pts, vs, inv, ctx->d_keys[0], ctx->d_vals[0], o.key_pt); }
  int buf = 0;
  { SegTimer seg_(ctx, SEG_VOX_SORT);
    s = radix_sort(ctx, &vs->n, n_cap, key_bits, &buf); }
  if (s != GM_OK) return s;
  { SegTimer seg_(ctx, SEG_VOX_REDUCE);
    GM_LAUNCH(ctx, k_voxel_heads, div_up((long long)n_cap, CPL_TILE), CP_BLOCK, ctx->d_keys[buf], ctx->d_vals[buf], o.assign, o.vox_start, o.vox_key,
              ctx->d_state64, ctx->d_ctl + 0, vs, &ctx->d_st->error);
    GM_LAUNCH(ctx, k_voxel_centroids, std::min(div_up((long long)n_cap * 32, VC_BLOCK), ctx->num_sms * 16), VC_BLOCK, ctx->d_vals[buf], pts,
              o.vox_start, vs, o.centroid, o.vox_count); }
  *sorted_buf = buf;
  GM_CHECK_LAUNCHES(ctx);
  return GM_OK;
}

// static upper bound of the voxel key range from the crop box (no host round trip for the bbox)
int voxel_key_bits(const gm_ctx* ctx, size_t n, size_t* key_range) {
  *key_range = 0;
  if (ctx->injected) return 32;
  const float inv = 1.0f / (float)ctx->prm.voxelGridLeafSize;
  double b = std::fabs(ctx->prm.boxFilterBound) * (double)inv;
  double div = std::floor(b) - std::floor(-b) + 2.0;
  double total = div * div * div;
  int bits = 32;
  if (total < 2147483647.0 && (double)n < 2147483647.0) { *key_range = (size_t)total; bits = bits_for((unsigned long long)total); }
  if (ctx->vox_bbox_set) {
    // a caller-supplied box (gm_set_voxel_bbox) holds the whole cloud, hence every sub-cloud: its lattice bounds the key range
    // (same float expressions as k_voxel_keys)
    const float* b = ctx->vox_bbox;
    double t2 = 1.0;
    for (int a = 0; a < 3; ++a) t2 *= (double)((long long)std::floor(b[3 + a] * inv) - (long long)std::floor(b[a] * inv) + 1);
    if (t2 >= 1.0 && t2 < 2147483647.0 && (*key_range == 0 || t2 < (double)*key_range)) { *key_range = (size_t)t2; bits = std::min(bits, bits_for((unsigned long long)t2)); }
  }
  return bits;
}
}  // namespace

gm_status gm_voxel(gm_ctx* ctx) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, COMPACTED)) return s;
  const size_t n = ctx->n_grid;
  if (n) {
    VoxBuffers o{ctx->d_vkey_pt, ctx->d_assign, ctx->d_vox_start, ctx->d_vox_key, ctx->d_vox_count, ctx->d_centroid};
    int buf = 0;
    size_t key_range = 0;
    int key_bits = voxel_key_bits(ctx, n, &key_range);
    if (ctx->vox_bbox_set && !ctx->vox_bbox_is_hint) {
      const float* b = ctx->vox_bbox;
      GM_LAUNCH(ctx, k_set_bbox, 1, 32, &ctx->d_st->vox, b[0], b[1], b[2], b[3], b[4], b[5]);
    }
    // nothing in a scan reads the per-point assignment: on the dense path gm_download_voxel_assignment computes it
    gm_status s = voxel_downsample(ctx, ctx->d_cloud_c, &ctx->d_st->vox, n, key_bits, key_range, o, &buf, false);
    if (s != GM_OK) return s;
    ctx->vox_assign_on_demand = dense_voxel_path(ctx, key_range);
    if (has(ctx, NORMALS)) {
      SegTimer seg_(ctx, SEG_VOX_NN);
      GM_LAUNCH(ctx, k_voxel_nn, std::min(div_up((long long)n * NN_GROUP, NN_BLOCK), ctx->num_sms * 16), NN_BLOCK, ctx->d_centroid, ctx->d_sorted,
                ctx->d_tab, ctx->d_ucell_start, ctx->d_runs, ctx->d_cell_nruns, ctx->d_valid_map, ctx->d_normals_c, ctx->grid, ctx->prm.nn_index_mode,
                ctx->d_st, ctx->d_nn_idx, ctx->d_nn_normal);
    }
    GM_CHECK_LAUNCHES(ctx);
  }
  mark(ctx, VOXEL);
  return GM_OK;
}

// ---- a5 --------------------------------------------------------------------------------------
gm_status gm_local_frame(gm_ctx* ctx) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, COMPACTED)) return s;
  const WeightLaw law = weight_law(ctx->prm);
  SegTimer seg_(ctx, SEG_FRAME);
  GM_LAUNCH(ctx, k_frame, FRAME_BLOCKS, FR_BLOCK, ctx->d_normals_c, &ctx->d_st->n_valid, law, ctx->d_partials + 0 * kPartialsRegion, ctx->d_counters + 0,
            ctx->d_frame, ctx->d_frame_sums);
  GM_CHECK_LAUNCHES(ctx);
  mark(ctx, FRAME);
  return GM_OK;
}

// ---- a8 --------------------------------------------------------------------------------------
// injected sample indices: host -> pinned staging -> device (the staging buffer is free again once the copy has run)
// Only the ids [h_begin, h_end) this call evaluates are copied (a rank of a sharded round never touches the rest).
static gm_status stage_samples(gm_ctx* ctx, int kind, const int32_t* samples_host, int h_begin, int h_end, int per) {
  if (h_end <= h_begin) return GM_OK;
  const size_t off = (size_t)h_begin * per, cnt = (size_t)(h_end - h_begin) * per;
  GM_CUDA(cudaEventSynchronize(ctx->ev_samples[kind]));
  std::memcpy(ctx->h_samples[kind] + off, samples_host + off, cnt * sizeof(int));
  GM_CUDA(cudaMemcpyAsync(ctx->hyp.samples[kind] + off, ctx->h_samples[kind] + off, cnt * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  GM_CUDA(cudaEventRecord(ctx->ev_samples[kind], ctx->stream));
  return GM_OK;
}

// The cloud an inlier count reads: the compacted points and their device count, and optionally the cell-sorted copy
// with its leaf bounds and device count, which selects tile-culled counting (same counts, see gm_ransac.cuh).
struct CountView {
  const float4* pts;
  const int* n;
  const float4* sorted = nullptr;
  const float4* leaf_bounds = nullptr;
  const int* n_sorted = nullptr;
};

// co-resident 64-thread blocks per SM (register limited to 14) of the brute-force count
constexpr int kCountBlocksPerSm = 8;

// Hypotheses [h_begin, h_end) of `kind` into `hs` (all H when gen_all) from the scan's compacted cloud, then, unless
// `cloud` is null, their inlier counts over `cloud` with the argmax folded into the counting kernel's last block.
// `comm` is the peer table of a sharded round (or null); `timed` records the *_hyp and *_count profile segments.
static gm_status launch_hyp_count(gm_ctx* ctx, HypSet& hs, int kind, int H, int h_begin, int h_end, int gen_all, const CommDev* comm,
                                  const CountView* cloud, bool timed) {
  const int* n_valid = &ctx->d_st->n_valid;
  const float tau = (float)ctx->prm.ransacThreshold;
  const int hb = div_up(H, 128);
  { SegTimer seg_(ctx, !timed ? -1 : kind == 0 ? SEG_PLANE_HYP : SEG_CYL_HYP);
  if (kind == 0) {
    GM_LAUNCH(ctx, k_plane_hypotheses, hb, 128, ctx->d_cloud_c, n_valid, hs.samples[0], H, hs.plane_coef, hs.hvalid[0], hs.counts[0],
              h_begin, h_end, gen_all);
  } else {
    GM_LAUNCH(ctx, k_cyl_hypotheses, hb, 128, ctx->d_cloud_c, ctx->d_normals_c, n_valid, hs.samples[1], H, (float)ctx->prm.cylinderRadiusMin,
              (float)ctx->prm.cylinderRadiusMax, tau, hs.model7, hs.test12, hs.hvalid[1], hs.counts[1], h_begin, h_end, gen_all);
  } }
  if (cloud) {
    SegTimer seg_(ctx, !timed ? -1 : kind == 0 ? SEG_PLANE_COUNT : SEG_CYL_COUNT);
    unsigned* ticket = ctx->d_counters + 3 + kind;
    if (cloud->sorted) {
      const int blocks = std::max(1, div_up((long long)ctx->n_grid, TC_SUPER));
      const auto count_tiles = kind == 0 ? k_count_tiles<0> : k_count_tiles<1>;
      GM_LAUNCH(ctx, count_tiles, blocks, TC_BLOCK, cloud->sorted, cloud->leaf_bounds, cloud->n_sorted, hs.plane_coef, hs.test12,
                hs.hvalid[kind], h_begin, h_end, tau, hs.counts[kind], H, hs.key + kind, ticket, comm, hs.model7);
    } else {
      const int K = kind == 0 ? RC_KP : RC_KC;
      const int groups = div_up(h_end - h_begin, RC_BLOCK * K);
      // every slice at least half a tile
      const int slices = std::max(1, std::min(div_up((long long)ctx->n_grid, RC_TILE / 2), div_up(ctx->num_sms * kCountBlocksPerSm, groups)));
      const dim3 grid(slices, groups);
      if (kind == 0) {
        GM_LAUNCH(ctx, k_count_plane<RC_KP>, grid, RC_BLOCK, cloud->pts, cloud->n, hs.plane_coef, hs.hvalid[0], h_begin, h_end, tau,
                  hs.counts[0], H, hs.key + 0, ticket, comm);
      } else {
        GM_LAUNCH(ctx, k_count_cyl<RC_KC>, grid, RC_BLOCK, cloud->pts, cloud->n, hs.test12, h_begin, h_end, hs.counts[1], H, hs.key + 1,
                  ticket, comm, hs.model7);
      }
    }
  }
  GM_CHECK_LAUNCHES(ctx);
  return GM_OK;
}

// Refit of the winner of `kind` in `hs` over `pts` and its device count `n`: the plane refit, or the cylinder's inlier
// compaction and all its Gauss-Newton passes in one cooperative launch (grid barrier between passes).
static gm_status launch_refit(gm_ctx* ctx, HypSet& hs, int kind, int H, const float4* pts, const int* n) {
  ModelState* ms = hs.model + kind;
  const float tau = (float)ctx->prm.ransacThreshold;
  if (kind == 0) {
    GM_LAUNCH(ctx, k_plane_refit, REFIT_BLOCKS, RF_BLOCK, pts, n, hs.key + 0, H, hs.plane_coef, ms, tau, ctx->d_partials + 1 * kPartialsRegion,
              ctx->d_counters + 1);
  } else {
    GM_LAUNCH(ctx, k_cyl_inlier_compact, std::max(1, div_up((long long)ctx->n_grid, CPL_TILE)), CP_BLOCK, pts, n, hs.key + 1, H, hs.model7,
              hs.test12, ms, ctx->d_inl, ctx->d_state64_b, ctx->d_ctl + 1, &ctx->d_st->error);
    const float4* inl = ctx->d_inl;
    int iters = ctx->prm.refitIterations;
    double* partials = ctx->d_partials + 2 * kPartialsRegion;
    unsigned* bars = ctx->d_counters + 5;  // counters [5],[6]: the two barrier counters, [7]: which one the next launch uses
    int* err = &ctx->d_st->error;
    void* args[] = {(void*)&inl, (void*)&ms, (void*)&iters, (void*)&tau, (void*)&partials, (void*)&bars, (void*)&err};
    GM_CUDA(cudaLaunchCooperativeKernel((const void*)k_cyl_gn_all, dim3(ctx->gn_blocks), dim3(RF_BLOCK), args, 0, ctx->stream));
    ++ctx->launches;
  }
  GM_CHECK_LAUNCHES(ctx);
  return GM_OK;
}

gm_status gm_ransac(gm_ctx* ctx, int32_t kind, const int32_t* samples_host, int32_t H, int32_t h_begin, int32_t h_end) {
  if (!ctx || (kind != 0 && kind != 1) || H < 0 || (H > 0 && !samples_host)) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, COMPACTED)) return s;
  if (H > ctx->hcap) { ctx->err = "H larger than max_hypotheses"; return GM_ERR_CAPACITY; }
  h_begin = std::max(h_begin, 0);
  h_end = std::min(h_end, H);
  const int per = kind == 0 ? 3 : 2;
  if (H > 0) {
    // a peer-memory sharded round ships the winner's coefficients with its key, so only this rank's share is uploaded and
    // generated; otherwise (single GPU, or keys all-reduced by the caller) every rank generates all H to be able to refit any winner
    const int gen_all = ctx->sharded ? 0 : 1;
    if (!ctx->samples_staged) { gm_status st_ = stage_samples(ctx, kind, samples_host, gen_all ? 0 : h_begin, gen_all ? H : h_end, per); if (st_ != GM_OK) return st_; }
    const CommDev* commdev = ctx->sharded ? comm_dev(ctx) : nullptr;
    CountView cloud{ctx->d_cloud_c, &ctx->d_st->n_valid};
    if (ctx->count_mode == 0 && has(ctx, NORMALS) && !ctx->injected) {  // the cell-sorted cloud of this scan
      cloud.sorted = ctx->d_sorted_valid; cloud.leaf_bounds = ctx->d_leaf_bounds; cloud.n_sorted = &ctx->d_st->n_crop;
    }
    const bool count = h_end > h_begin && ctx->n_input > 0;
    if (gm_status s = launch_hyp_count(ctx, ctx->hyp, kind, H, h_begin, h_end, gen_all, commdev, count ? &cloud : nullptr, true)) return s;
    if (!count) {
      SegTimer seg_(ctx, kind == 0 ? SEG_PLANE_ARGMAX : SEG_CYL_ARGMAX);
      GM_LAUNCH(ctx, k_argmax, 1, AM_BLOCK, ctx->hyp.counts[kind], H, ctx->hyp.key + kind, commdev, kind, ctx->hyp.plane_coef, ctx->hyp.model7,
                ctx->hyp.test12);
    }
  } else {
    GM_CUDA(cudaMemsetAsync(ctx->hyp.key + kind, 0, sizeof(unsigned long long), ctx->stream));
  }
  GM_CHECK_LAUNCHES(ctx);
  mark(ctx, ransac_stage(kind));
  ctx->ransac_H[kind] = H;
  ctx->stages &= ~(1u << model_stage(kind));  // the model of the previous round is stale until gm_ransac_select
  return GM_OK;
}

gm_status gm_ransac_key_device_ptr(gm_ctx* ctx, int32_t kind, void** key_dev) {
  if (!ctx || !key_dev || (kind != 0 && kind != 1)) return GM_ERR_INVALID_ARG;
  *key_dev = (void*)(ctx->hyp.key + kind);
  return GM_OK;
}

gm_status gm_ransac_export_key(gm_ctx* ctx, int32_t kind, void* dst_device) {
  if (!ctx || !dst_device || (kind != 0 && kind != 1)) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, ransac_stage(kind))) return s;
  GM_CUDA(cudaMemcpyAsync(dst_device, ctx->hyp.key + kind, sizeof(unsigned long long), cudaMemcpyDeviceToDevice, ctx->stream));
  return GM_OK;
}

gm_status gm_ransac_import_key(gm_ctx* ctx, int32_t kind, const void* src_device) {
  if (!ctx || !src_device || (kind != 0 && kind != 1)) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, ransac_stage(kind))) return s;
  GM_CUDA(cudaMemcpyAsync(ctx->hyp.key + kind, src_device, sizeof(unsigned long long), cudaMemcpyDeviceToDevice, ctx->stream));
  return GM_OK;
}

gm_status gm_ransac_select(gm_ctx* ctx, int32_t kind) {
  if (!ctx || (kind != 0 && kind != 1)) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, ransac_stage(kind))) return s;
  SegTimer seg_(ctx, kind == 0 ? SEG_PLANE_REFIT : SEG_CYL_REFIT);
  if (gm_status s = launch_refit(ctx, ctx->hyp, kind, ctx->ransac_H[kind], ctx->d_cloud_c, &ctx->d_st->n_valid)) return s;
  mark(ctx, model_stage(kind));
  return GM_OK;
}

gm_status gm_label(gm_ctx* ctx) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, COMPACTED)) return s;
  if (ctx->n_input) {
    int blocks = std::min(div_up((long long)ctx->n_grid, 256), ctx->num_sms * 16);
    SegTimer seg_(ctx, SEG_LABEL);
    GM_LAUNCH(ctx, k_label, blocks, 256, ctx->d_cloud_c, &ctx->d_st->n_valid, ctx->hyp.model + 0, ctx->hyp.model + 1,
              has(ctx, MODEL_PLANE) ? 1 : 0, has(ctx, MODEL_CYL) ? 1 : 0, (float)ctx->prm.ransacThreshold, ctx->d_labels);
    GM_CHECK_LAUNCHES(ctx);
  }
  mark(ctx, LABELS);
  return GM_OK;
}

gm_status gm_axis_polyline(gm_ctx* ctx) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, FRAME, LABELS)) return s;
  const int S = ctx->prm.maxSlices;
  const int* n_ptr = &ctx->d_st->n_valid;
  const WeightLaw shift = weight_law(ctx->prm);
  SegTimer seg_(ctx, SEG_POLYLINE);
  {
    // 3 launches: range (+basis, +zeroing, +slice layout, +the list of cylinder points) and two accumulation passes over
    // that list (moments -> means + circle fit; residuals -> output), each with the per-slice step that consumes it
    // folded into its last block
    int blocks = std::max(1, std::min(div_up((long long)std::max<size_t>(ctx->n_grid, 1), POLY_BLOCK), ctx->num_sms * 4));
    const int cap = (int)ctx->cap;
    unsigned* n_list = ctx->d_counters + 10;
    GM_LAUNCH(ctx, k_poly_range, blocks, POLY_BLOCK, ctx->d_cloud_c, ctx->d_normals_c, ctx->d_labels, n_ptr, ctx->d_frame, shift, ctx->d_poly,
              ctx->d_poly_acc, POLY_NACC * S, ctx->d_poly_part, ctx->d_counters + 8, ctx->d_poly_list, cap, n_list, ctx->prm.sliceLength, S);
    const ModelState* cylm = has(ctx, MODEL_CYL) ? ctx->hyp.model + 1 : nullptr;
    GM_LAUNCH(ctx, k_poly_pass<0>, blocks, POLY_BLOCK, ctx->d_poly_list, cap, n_list, ctx->d_poly, ctx->d_poly_acc, ctx->d_slices,
              ctx->d_counters + 9, cylm);
    GM_LAUNCH(ctx, k_poly_pass<2>, blocks, POLY_BLOCK, ctx->d_poly_list, cap, n_list, ctx->d_poly, ctx->d_poly_acc, ctx->d_slices,
              ctx->d_counters + 11, cylm);
  }
  GM_CHECK_LAUNCHES(ctx);
  mark(ctx, POLY);
  return GM_OK;
}

gm_status gm_compress(gm_ctx* ctx) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, LABELS, POLY)) return s;
  const size_t n = std::max<size_t>(ctx->n_grid, 1);
  gm_status s;
  GM_LAUNCH(ctx, k_vox_reset, 1, 32, ctx->d_res_vs);
  const int tiles = div_up((long long)n, CP_TILE);
  GM_LAUNCH(ctx, k_comp_split, tiles, CP_BLOCK, ctx->d_cloud_c, ctx->d_labels, &ctx->d_st->n_valid, ctx->hyp.model + 0, ctx->hyp.model + 1,
            has(ctx, MODEL_PLANE) ? 1 : 0, has(ctx, MODEL_CYL) ? 1 : 0, ctx->d_res_pts, ctx->d_res_vs, ctx->d_state64, ctx->d_ctl + 0, &ctx->d_st->error,
            ctx->d_comp_part, ctx->d_comp_mm, ctx->d_counters + 12, ctx->d_comp);
  VoxBuffers o{ctx->d_res_key_pt, ctx->d_res_assign, ctx->d_res_vox_start, ctx->d_res_vox_key, ctx->d_res_vox_count, ctx->d_res_centroid};
  int buf = 0;
  size_t res_range = 0;
  const int res_bits = voxel_key_bits(ctx, n, &res_range);
  if ((s = voxel_downsample(ctx, ctx->d_res_pts, ctx->d_res_vs, n, res_bits, res_range, o, &buf)) != GM_OK) return s;
  GM_LAUNCH(ctx, k_comp_residual_error, ctx->num_sms * 2, CR_BLOCK, ctx->d_res_pts, ctx->d_res_assign, ctx->d_res_centroid, ctx->d_res_vs,
            ctx->d_comp_part, ctx->d_counters + 13, ctx->d_comp);
  GM_CHECK_LAUNCHES(ctx);
  mark(ctx, COMP);
  return GM_OK;
}

namespace {
// A compressed blob (GMC1, GMP1) starts with its 4-byte magic, a 4-byte version 1 and its header; returns where the
// body starts.
unsigned char* put_blob_header(void* buf, uint32_t magic, const void* header, size_t header_bytes) {
  unsigned char* p = (unsigned char*)buf;
  const uint32_t version = 1;
  std::memcpy(p, &magic, 4); std::memcpy(p + 4, &version, 4);
  std::memcpy(p + 8, header, header_bytes);
  return p + 8 + header_bytes;
}

// ... and ends with the `n` residual voxel centroids as packed xyz; waits for every copy of the blob.
gm_status put_blob_centroids(gm_ctx* ctx, unsigned char* p, const float4* centroids, int n) {
  if (n > 0)  // strided copy: float4 centroids -> packed xyz
    GM_CUDA(cudaMemcpy2DAsync(p, 12, centroids, 16, 12, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  return GM_OK;
}

gm_status fetch_compression(gm_ctx* ctx, gm_compression* out, VoxState* vs_host) {
  CompStats c;
  PolyState ps;
  GM_CUDA(cudaMemcpyAsync(&c, ctx->d_comp, sizeof(c), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaMemcpyAsync(vs_host, ctx->d_res_vs, sizeof(VoxState), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaMemcpyAsync(&ps, ctx->d_poly, sizeof(ps), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  std::memset(out, 0, sizeof(*out));
  out->n_points = c.n_points; out->n_plane = c.n_plane; out->n_cylinder = c.n_cyl; out->n_residual = c.n_residual;
  out->n_residual_voxels = vs_host->n_voxels; out->n_slices = ps.S;
  std::memcpy(out->plane_coef, c.plane_coef, sizeof(out->plane_coef));
  std::memcpy(out->plane_u, c.plane_u, sizeof(out->plane_u));
  std::memcpy(out->plane_v, c.plane_v, sizeof(out->plane_v));
  std::memcpy(out->plane_bounds, c.plane_bounds, sizeof(out->plane_bounds));
  out->plane_rms = c.plane_rms;
  std::memcpy(out->cyl_coef, c.cyl_coef, sizeof(out->cyl_coef));
  std::memcpy(out->cyl_t_range, c.cyl_t_range, sizeof(out->cyl_t_range));
  out->cyl_rms = c.cyl_rms; out->residual_rms = c.residual_rms; out->total_rms = c.total_rms;
  out->leaf = (float)ctx->prm.voxelGridLeafSize;
  out->bytes_in = 16ull * (uint64_t)std::max(c.n_points, 0);
  out->bytes_out = 8 + sizeof(gm_compression) + (uint64_t)std::max(ps.S, 0) * sizeof(gm_slice) + 12ull * (uint64_t)std::max(vs_host->n_voxels, 0);
  out->ratio = out->bytes_out ? (float)((double)out->bytes_in / (double)out->bytes_out) : 0.f;
  return GM_OK;
}
}  // namespace

gm_status gm_get_compression(gm_ctx* ctx, gm_compression* out) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, COMP)) return s;
  VoxState vs;
  return fetch_compression(ctx, out, &vs);
}

gm_status gm_download_compressed(gm_ctx* ctx, void* buf, size_t capacity, size_t* bytes) {
  if (!ctx || !bytes) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, COMP)) return s;
  gm_compression h;
  VoxState vs;
  gm_status s = fetch_compression(ctx, &h, &vs);
  if (s != GM_OK) return s;
  *bytes = (size_t)h.bytes_out;
  if (!buf) return GM_OK;
  if (capacity < h.bytes_out) return GM_ERR_CAPACITY;
  unsigned char* p = put_blob_header(buf, 0x31434D47u /* 'GMC1' */, &h, sizeof(h));
  if (h.n_slices > 0) { GM_CUDA(cudaMemcpyAsync(p, ctx->d_slices, (size_t)h.n_slices * sizeof(gm_slice), cudaMemcpyDeviceToHost, ctx->stream)); p += (size_t)h.n_slices * sizeof(gm_slice); }
  return put_blob_centroids(ctx, p, ctx->d_res_centroid, h.n_residual_voxels);
}

}  // extern "C" (templates need C++ linkage)

// Runs `body` with ctx->stream temporarily replaced by branch stream `b` (which first waits for
// the fork event), then records the branch's join event.
template <class F>
static gm_status run_branch(gm_ctx* ctx, int b, F&& body) {
  cudaStream_t main_stream = ctx->stream;
  cudaError_t e = cudaStreamWaitEvent(ctx->branch[b], ctx->ev_fork, 0);
  if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return GM_ERR_CUDA; }
  ctx->stream = ctx->branch[b];
  gm_status s = body();
  ctx->stream = main_stream;
  if (s != GM_OK) return s;
  e = cudaEventRecord(ctx->ev_join[b], ctx->branch[b]);
  if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return GM_ERR_CUDA; }
  return GM_OK;
}

// The plane step on branch stream 1 and the cylinder step on the main stream, side by side, then the main stream waits
// for the branch.  They run one after the other unless the context is concurrent, not profiling, and `may_fork`.
template <class P, class C>
static gm_status plane_and_cylinder(gm_ctx* ctx, P&& plane, C&& cylinder, bool may_fork = true) {
  gm_status s;
  if (ctx->concurrent && !ctx->profiling && may_fork) {
    GM_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
    if ((s = run_branch(ctx, 1, plane)) != GM_OK) return s;
    if ((s = cylinder()) != GM_OK) return s;
    GM_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[1], 0));
    return GM_OK;
  }
  if ((s = plane()) != GM_OK) return s;
  return cylinder();
}

static gm_status process_scan_body(gm_ctx* ctx, const int32_t* plane_samples_host, int32_t Hp, const int32_t* cyl_samples_host, int32_t Hc) {
  gm_status s;
  if ((s = gm_crop(ctx)) != GM_OK) return s;
  if ((s = gm_normals(ctx)) != GM_OK) return s;
  // After the NaN compaction four stages only READ the compacted cloud / normals and write disjoint
  // outputs: voxel grid + 1-NN, local frame, plane RANSAC + refit, cylinder RANSAC + refit.  They are
  // forked onto separate streams so the latency-bound small kernels overlap the FP32-bound inlier
  // counting (which runs at ~20 % warp occupancy); labels and the polyline need all of them.
  auto plane = [&]() -> gm_status {
    if (Hp <= 0) return GM_OK;
    gm_status r = gm_ransac(ctx, GM_MODEL_PLANE, plane_samples_host, Hp, 0, Hp);
    return r != GM_OK ? r : gm_ransac_select(ctx, GM_MODEL_PLANE);
  };
  auto cylinder = [&]() -> gm_status {
    if (Hc <= 0) return GM_OK;
    gm_status r = gm_ransac(ctx, GM_MODEL_CYLINDER, cyl_samples_host, Hc, 0, Hc);
    return r != GM_OK ? r : gm_ransac_select(ctx, GM_MODEL_CYLINDER);
  };
  if (ctx->concurrent && !ctx->profiling) {
    GM_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
    if ((s = run_branch(ctx, 0, [&] { return gm_voxel(ctx); })) != GM_OK) return s;
    if ((s = run_branch(ctx, 1, [&]() -> gm_status { gm_status r = gm_local_frame(ctx); return r != GM_OK ? r : plane(); })) != GM_OK) return s;
    if ((s = cylinder()) != GM_OK) return s;  // the longest branch stays on the main stream
    for (int b = 0; b < 2; ++b) GM_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[b], 0));
  } else {
    if ((s = gm_voxel(ctx)) != GM_OK) return s;
    if ((s = gm_local_frame(ctx)) != GM_OK) return s;
    if ((s = plane()) != GM_OK) return s;
    if ((s = cylinder()) != GM_OK) return s;
  }
  if ((s = gm_label(ctx)) != GM_OK) return s;
  if ((s = gm_axis_polyline(ctx)) != GM_OK) return s;
  return GM_OK;
}

// the stages a whole scan holds afterwards (what process_scan_body marks when it runs as plain launches)
static void mark_processed(gm_ctx* ctx, int Hp, int Hc) {
  mark(ctx, CROP, NORMALS, COMPACTED, VOXEL, FRAME, LABELS, POLY);
  ctx->injected = false;
  ctx->deskew_open = false;
  size_t key_range = 0;  // the VoxelGrid path the replayed gm_voxel took
  voxel_key_bits(ctx, ctx->n_grid, &key_range);
  ctx->vox_assign_on_demand = dense_voxel_path(ctx, key_range);
  const int H[2] = {Hp, Hc};
  for (int k = 0; k < 2; ++k)
    if (H[k] > 0) { mark(ctx, ransac_stage(k), model_stage(k)); ctx->ransac_H[k] = H[k]; }
}

static void drop_graph(gm_ctx::ScanGraph& g) {
  if (g.exec) cudaGraphExecDestroy(g.exec);
  g.exec = nullptr;
}

// Graph policy of gm_process_scan.  Measured on B200 (bench.py, GM_GRAPH=0/1): replaying the captured graph removes ~100 us
// of launch calls per scan -- 200k-point frames go from 7.8e3 to 1.37e4 frames/s, single-scan latency at 1M points from
// 0.68 to 0.65 ms -- while the saturated throughput at 1M points is the same either way (the GPU is the limit), and the
// end-to-end pipeline with 35 MB of host copies per scan in flight on four streams runs 6-13 % FASTER with plain launches
// (their pacing interleaves the contexts' kernels and copies better than four resident graphs do).  Hence "auto".
constexpr size_t kGraphAutoPoints = 524288;
static bool use_graph(const gm_ctx* ctx) { return ctx->graph_mode == 1 || (ctx->graph_mode == 2 && ctx->n_grid <= kGraphAutoPoints); }

// Run `body` (a fixed sequence of launches on the ctx streams) as a CUDA graph keyed by (kind, bucketed size, Hp, Hc,
// parameter generation): the first call of a key runs `body` as plain launches (buffers that grow on demand are allocated
// there, outside any capture), the second captures it (nothing executes during capture) and launches the graph, every
// later one is ONE cudaGraphLaunch.  `stage` copies the per-call host inputs (sample indices) before the graph runs.
template <class Stage, class Body>
static gm_status run_graphed(gm_ctx* ctx, int kind, int Hp, int Hc, Stage&& stage, Body&& body) {
  gm_ctx::ScanGraph* g = nullptr;
  for (auto& e : ctx->graphs)
    if (e.kind == kind && e.n_grid == ctx->n_grid && e.Hp == Hp && e.Hc == Hc && e.gen == ctx->graph_gen) { g = &e; break; }
  if (!g) {
    if (ctx->graphs.size() >= 8) {  // evict the least recently used entry
      size_t v = 0;
      for (size_t i = 1; i < ctx->graphs.size(); ++i) if (ctx->graphs[i].stamp < ctx->graphs[v].stamp) v = i;
      drop_graph(ctx->graphs[v]);
      ctx->graphs.erase(ctx->graphs.begin() + (long)v);
    }
    ctx->graphs.push_back(gm_ctx::ScanGraph{kind, ctx->n_grid, Hp, Hc, ctx->graph_gen, 0, nullptr, 0, 0});
    g = &ctx->graphs.back();
  }
  g->stamp = ++ctx->graph_clock;
  ++g->uses;
  if (!g->exec && g->uses == 1) return body();
  gm_status s = stage();
  if (s != GM_OK) return s;
  if (!g->exec) {
    cudaGraph_t graph = nullptr;
    cudaError_t e = cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal);
    if (e == cudaSuccess) {
      const long long l0 = ctx->launches;
      ctx->samples_staged = true;
      s = body();
      ctx->samples_staged = false;
      g->launches = ctx->launches - l0;
      e = cudaStreamEndCapture(ctx->stream, &graph);
      if (s != GM_OK && e == cudaSuccess) e = cudaErrorUnknown;
      if (e == cudaSuccess) e = cudaGraphInstantiate(&g->exec, graph, 0);
      if (graph) cudaGraphDestroy(graph);
    }
    if (e != cudaSuccess) {  // cannot capture on this stream / driver: keep working with plain launches, and say so
      cudaGetLastError();
      ctx->graph_note = std::string("graph capture failed, using stream launches: ") + cudaGetErrorString(e);
      ctx->graph_mode = 0;
      g->exec = nullptr;
      ctx->samples_staged = true;  // already staged above
      s = body();
      ctx->samples_staged = false;
      return s;
    }
    ++ctx->graph_captures;
  } else {
    ctx->launches += g->launches;
  }
  GM_CUDA(cudaGraphLaunch(g->exec, ctx->stream));
  ++ctx->graph_replays;
  return GM_OK;
}

extern "C" {

gm_status gm_process_scan(gm_ctx* ctx, const int32_t* plane_samples_host, int32_t Hp, const int32_t* cyl_samples_host, int32_t Hc) {
  if (!ctx || Hp < 0 || Hc < 0 || (Hp > 0 && !plane_samples_host) || (Hc > 0 && !cyl_samples_host)) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, SCAN)) return s;
  if (Hp > ctx->hcap || Hc > ctx->hcap) { ctx->err = "H larger than max_hypotheses"; return GM_ERR_CAPACITY; }
  auto body = [&] { return process_scan_body(ctx, plane_samples_host, Hp, cyl_samples_host, Hc); };
  const bool graphable = use_graph(ctx) && ctx->concurrent && !ctx->profiling && ctx->n_grid > 0;
  if (!graphable) return body();
  auto stage = [&]() -> gm_status {
    gm_status s;
    if (Hp > 0 && (s = stage_samples(ctx, 0, plane_samples_host, 0, Hp, 3)) != GM_OK) return s;
    if (Hc > 0 && (s = stage_samples(ctx, 1, cyl_samples_host, 0, Hc, 2)) != GM_OK) return s;
    return GM_OK;
  };
  gm_status s = run_graphed(ctx, 0, Hp, Hc, stage, body);
  if (s == GM_OK) mark_processed(ctx, Hp, Hc);
  return s;
}

gm_status gm_set_graph_mode(gm_ctx* ctx, int32_t mode) {
  if (!ctx || mode < 0 || mode > 2) return GM_ERR_INVALID_ARG;
  ctx->graph_mode = mode;
  return GM_OK;
}

gm_status gm_get_graph_stats(const gm_ctx* ctx, int64_t* captures, int64_t* replays) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (captures) *captures = ctx->graph_captures;
  if (replays) *replays = ctx->graph_replays;
  return GM_OK;
}

// Plane and cylinder rounds of one RANSAC step side by side (they only read the compacted / cell-sorted cloud and
// write disjoint outputs): the multi-GPU hand-off runs gm_ransac_pair -> ONE all-reduce of both keys ->
// gm_ransac_select_pair, so a sharded round costs one collective and the longer of the two refits.
gm_status gm_ransac_pair(gm_ctx* ctx, const int32_t* plane_samples_host, int32_t Hp, int32_t p_begin, int32_t p_end,
                         const int32_t* cyl_samples_host, int32_t Hc, int32_t c_begin, int32_t c_end) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, COMPACTED)) return s;
  return plane_and_cylinder(ctx, [&] { return gm_ransac(ctx, GM_MODEL_PLANE, plane_samples_host, Hp, p_begin, p_end); },
                            [&] { return gm_ransac(ctx, GM_MODEL_CYLINDER, cyl_samples_host, Hc, c_begin, c_end); });
}

gm_status gm_ransac_select_pair(gm_ctx* ctx) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, RANSAC_PLANE, RANSAC_CYL)) return s;
  return plane_and_cylinder(ctx, [&] { return gm_ransac_select(ctx, GM_MODEL_PLANE); }, [&] { return gm_ransac_select(ctx, GM_MODEL_CYLINDER); });
}

/* both keys (plane, cylinder) as 16 contiguous bytes */
gm_status gm_ransac_export_keys(gm_ctx* ctx, void* dst_device) {
  if (!ctx || !dst_device) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, RANSAC_PLANE, RANSAC_CYL)) return s;
  GM_CUDA(cudaMemcpyAsync(dst_device, ctx->hyp.key, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, ctx->stream));
  return GM_OK;
}
gm_status gm_ransac_import_keys(gm_ctx* ctx, const void* src_device) {
  if (!ctx || !src_device) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, RANSAC_PLANE, RANSAC_CYL)) return s;
  GM_CUDA(cudaMemcpyAsync(ctx->hyp.key, src_device, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, ctx->stream));
  return GM_OK;
}

}  // extern "C"

// ---- sequential multi-primitive extraction (gm_primitives.cuh) -------------------------------------------------------
namespace {
static_assert(sizeof(PrimRec) == sizeof(gm_primitive), "primitive layout");
static_assert(sizeof(PrimCompRec) == sizeof(gm_primitive_record), "primitive record layout");

// The first call allocates the working copies and hypothesis tables; the draw buffers grow to the largest call.  Rare
// path (synchronous): a context that never extracts keeps its footprint.
gm_status ensure_prim_buffers(gm_ctx* ctx, size_t plane_draws, size_t cyl_draws) {
  const bool first = ctx->d_pr_state.count == 0;
  if (!first && plane_draws <= ctx->d_pr_draws[0].count && cyl_draws <= ctx->d_pr_draws[1].count) return GM_OK;
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  if (first || plane_draws > ctx->d_pr_draws[0].count) GM_CUDA(ctx->d_pr_draws[0].alloc(plane_draws));
  if (first || cyl_draws > ctx->d_pr_draws[1].count) GM_CUDA(ctx->d_pr_draws[1].alloc(cyl_draws));
  if (!first) return GM_OK;
  const size_t N = ctx->cap, H = (size_t)ctx->hcap;
  GM_CUDA(ctx->d_pr_sv.alloc(N)); GM_CUDA(ctx->d_pr_cc.alloc(N)); GM_CUDA(ctx->d_pr_lb.alloc(2 * ((N + 31) / 32)));
  GM_CUDA(ctx->d_pr_rem.alloc(N)); GM_CUDA(ctx->d_pr_ids.alloc(N));
  GM_CUDA(ctx->pr_hyp.alloc(H));
  GM_CUDA(ctx->d_pr_state.alloc(1));  // last: a failure above leaves the set unallocated
  return GM_OK;
}

gm_status extract_rounds(gm_ctx* ctx, int K, int min_inliers, int Hp, int Hc) {
  const size_t n = ctx->n_grid;
  PrimState* ps = ctx->d_pr_state;
  HypSet& hs = ctx->pr_hyp;
  // the scan's cell-sorted copy exists: claims walk it and keep its leaf bounds current; counting uses it unless count_mode = 1
  const bool sorted = has(ctx, NORMALS) && !ctx->injected;
  // Hypotheses read the original compacted cloud (R_r indices are never blanked); counts and refits read the blanked
  // working copies through the live sizes, which are 0 once extraction stopped.
  CountView cloud{ctx->d_pr_cc, &ps->n_valid_live};
  if (sorted && ctx->count_mode == 0) { cloud.sorted = ctx->d_pr_sv; cloud.leaf_bounds = ctx->d_pr_lb; cloud.n_sorted = &ps->n_crop_live; }
  GM_CUDA(cudaMemsetAsync(ctx->d_pr_ids, 0, n, ctx->stream));
  GM_CUDA(cudaMemcpyAsync(ctx->d_pr_cc, ctx->d_cloud_c, n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream));
  if (sorted) {
    GM_CUDA(cudaMemcpyAsync(ctx->d_pr_sv, ctx->d_sorted_valid, n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream));
    GM_CUDA(cudaMemcpyAsync(ctx->d_pr_lb, ctx->d_leaf_bounds, 2 * ((n + 31) / 32) * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream));
  }
  const int H[2] = {Hp, Hc};
  gm_status s;
  // the step of each kind that has hypotheses; side by side as in gm_ransac_pair when both have
  auto both = [&](auto&& step) -> gm_status {
    return plane_and_cylinder(ctx, [&]() -> gm_status { return Hp > 0 ? step(0) : GM_OK; },
                              [&]() -> gm_status { return Hc > 0 ? step(1) : GM_OK; }, Hp > 0 && Hc > 0);
  };
  const int draws = Hp * 3 + Hc * 2;
  const int point_blocks = std::min(div_up((long long)n, 256), ctx->num_sms * 8);
  for (int r = 0; r < K; ++r) {
    GM_LAUNCH(ctx, k_prim_remaining, std::max(1, div_up((long long)n, CPL_TILE)), CP_BLOCK, ctx->d_pr_ids, ctx->d_pr_state, ctx->d_pr_rem,
              ctx->d_state64, ctx->d_ctl + 0, &ctx->d_st->error);
    GM_LAUNCH(ctx, k_prim_draws, std::max(1, std::min(div_up(draws, 256), ctx->num_sms * 4)), 256, ctx->d_pr_draws[0] + (size_t)r * Hp * 3, Hp * 3,
              ctx->d_pr_draws[1] + (size_t)r * Hc * 2, Hc * 2, ctx->d_pr_rem, ctx->d_pr_state, hs.samples[0], hs.samples[1]);
    if ((s = both([&](int k) { return launch_hyp_count(ctx, hs, k, H[k], 0, H[k], 1, nullptr, &cloud, false); })) != GM_OK) return s;
    GM_LAUNCH(ctx, k_prim_decide, 1, 32, hs.key, Hp > 0 ? 1 : 0, Hc > 0 ? 1 : 0, min_inliers, Hp, Hc, hs.plane_coef, hs.test12, ctx->d_pr_state);
    // the key of a kind that did not win the round is 0, so its refit finds no model
    if ((s = both([&](int k) { return launch_refit(ctx, hs, k, H[k], ctx->d_pr_cc, &ps->n_valid_live); })) != GM_OK) return s;
    const float tau = (float)ctx->prm.ransacThreshold;
    if (sorted) {
      GM_LAUNCH(ctx, k_prim_claim_sorted, point_blocks, 256, ctx->d_pr_sv, ctx->d_pr_lb, ctx->d_valid_map, ctx->d_pr_cc, ctx->d_pr_ids,
                ctx->d_pr_state, hs.model, tau, r);
    } else {
      GM_LAUNCH(ctx, k_prim_claim_compact, point_blocks, 256, ctx->d_pr_cc, ctx->d_pr_ids, ctx->d_pr_state, hs.model, tau, r);
    }
    GM_CHECK_LAUNCHES(ctx);
  }
  return GM_OK;
}

// Compression buffers of the extracted primitives (first gm_compress_primitives; rare path, synchronous)
gm_status ensure_prim_comp_buffers(gm_ctx* ctx) {
  if (ctx->d_pr_stats.count) return GM_OK;
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  const size_t N = ctx->cap;
  GM_CUDA(ctx->d_pr_assign.alloc(N)); GM_CUDA(ctx->d_pr_vox_start.alloc(N + 1)); GM_CUDA(ctx->d_pr_vox_key.alloc(N));
  GM_CUDA(ctx->d_pr_vox_count.alloc(N)); GM_CUDA(ctx->d_pr_vs.alloc(1)); GM_CUDA(ctx->d_pr_comp.alloc(1));
  GM_CUDA(ctx->d_pr_stats.alloc(1));  // last: a failure above leaves the set unallocated
  return GM_OK;
}
}  // namespace

extern "C" {

gm_status gm_extract_primitives(gm_ctx* ctx, int32_t max_primitives, int32_t min_inliers, const uint32_t* plane_draws_host, int32_t Hp,
                                const uint32_t* cyl_draws_host, int32_t Hc) {
  if (!ctx || max_primitives < 0 || max_primitives > GM_MAX_PRIMITIVES || Hp < 0 || Hc < 0 || (Hp > 0 && !plane_draws_host) ||
      (Hc > 0 && !cyl_draws_host))
    return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, COMPACTED)) return s;
  if (Hp > ctx->hcap || Hc > ctx->hcap) { ctx->err = "H larger than max_hypotheses"; return GM_ERR_CAPACITY; }
  const size_t np = (size_t)max_primitives * Hp * 3, nc = (size_t)max_primitives * Hc * 2;
  gm_status s = ensure_prim_buffers(ctx, np, nc);
  if (s != GM_OK) return s;
  ctx->stages &= ~((1u << PRIMS) | (1u << PRIMS_COMP));
  if (np) GM_CUDA(cudaMemcpyAsync(ctx->d_pr_draws[0], plane_draws_host, np * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  if (nc) GM_CUDA(cudaMemcpyAsync(ctx->d_pr_draws[1], cyl_draws_host, nc * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  GM_LAUNCH(ctx, k_prim_begin, 1, 32, ctx->d_pr_state, ctx->d_st);
  GM_CHECK_LAUNCHES(ctx);
  if (ctx->n_grid && (s = extract_rounds(ctx, max_primitives, min_inliers, Hp, Hc)) != GM_OK) return s;
  mark(ctx, PRIMS);
  return GM_OK;
}

gm_status gm_get_primitives(gm_ctx* ctx, gm_primitive* out, int32_t capacity, int32_t* n) {
  if (!ctx || !n) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, PRIMS)) return s;
  int np = 0;
  GM_CUDA(cudaMemcpyAsync(&np, &ctx->d_pr_state->n_prims, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  *n = np;
  if (!out) return GM_OK;
  if (np > capacity) return GM_ERR_CAPACITY;
  GM_CUDA(cudaMemcpyAsync(out, ctx->d_pr_state->prim, (size_t)np * sizeof(gm_primitive), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  return GM_OK;
}

gm_status gm_download_primitive_ids(gm_ctx* ctx, uint8_t* out, size_t capacity_points) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, PRIMS)) return s;
  DevState h;
  return download(ctx, &h, n_valid, capacity_points, {{out, ctx->d_pr_ids, 1}});
}

gm_status gm_compress_primitives(gm_ctx* ctx) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, PRIMS)) return s;
  gm_status s = ensure_prim_comp_buffers(ctx);
  if (s != GM_OK) return s;
  const size_t n = std::max<size_t>(ctx->n_grid, 1);
  GM_LAUNCH(ctx, k_prim_comp_reset, 1, 64, ctx->d_pr_comp, ctx->d_pr_vs);
  GM_LAUNCH(ctx, k_prim_comp_split, div_up((long long)n, CP_TILE), CP_BLOCK, ctx->d_cloud_c, ctx->d_pr_ids, &ctx->d_st->n_valid, ctx->d_pr_state,
            ctx->d_pr_sv, ctx->d_pr_vs, ctx->d_state64, ctx->d_ctl + 0, &ctx->d_st->error, ctx->d_counters + 12, ctx->d_pr_comp, ctx->d_pr_stats);
  // the residual cloud is in d_pr_sv, its voxel centroids go to d_pr_cc (extraction scratch until the next extraction)
  VoxBuffers o{ctx->d_pr_rem, ctx->d_pr_assign, ctx->d_pr_vox_start, ctx->d_pr_vox_key, ctx->d_pr_vox_count, ctx->d_pr_cc};
  int buf = 0;
  size_t res_range = 0;
  const int res_bits = voxel_key_bits(ctx, n, &res_range);
  if ((s = voxel_downsample(ctx, ctx->d_pr_sv, ctx->d_pr_vs, n, res_bits, res_range, o, &buf)) != GM_OK) return s;
  GM_LAUNCH(ctx, k_comp_residual_error, ctx->num_sms * 2, CR_BLOCK, ctx->d_pr_sv, ctx->d_pr_assign, ctx->d_pr_cc, ctx->d_pr_vs, ctx->d_comp_part,
            ctx->d_counters + 13, ctx->d_pr_stats);
  GM_CHECK_LAUNCHES(ctx);
  mark(ctx, PRIMS_COMP);
  return GM_OK;
}

gm_status gm_download_compressed_primitives(gm_ctx* ctx, void* buf, size_t capacity, size_t* bytes) {
  if (!ctx || !bytes) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, PRIMS_COMP)) return s;
  std::vector<PrimComp> pc(1);  // ~7 KB
  CompStats cs;
  VoxState vs;
  GM_CUDA(cudaMemcpyAsync(pc.data(), ctx->d_pr_comp, sizeof(PrimComp), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaMemcpyAsync(&cs, ctx->d_pr_stats, sizeof(CompStats), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaMemcpyAsync(&vs, ctx->d_pr_vs, sizeof(VoxState), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  const PrimComp& c = pc[0];
  gm_primitive_compression h;
  std::memset(&h, 0, sizeof(h));
  h.n_points = c.n_points; h.n_primitives = c.n_prims; h.n_residual = c.n_residual; h.n_residual_voxels = vs.n_voxels;
  h.leaf = (float)ctx->prm.voxelGridLeafSize;
  h.residual_rms = cs.residual_rms; h.total_rms = cs.total_rms;
  h.bytes_in = 16ull * (uint64_t)std::max(c.n_points, 0);
  h.bytes_out = 8 + sizeof(h) + (uint64_t)std::max(c.n_prims, 0) * sizeof(gm_primitive_record) + 12ull * (uint64_t)std::max(vs.n_voxels, 0);
  h.ratio = (float)((double)h.bytes_in / (double)h.bytes_out);
  *bytes = (size_t)h.bytes_out;
  if (!buf) return GM_OK;
  if (capacity < h.bytes_out) return GM_ERR_CAPACITY;
  unsigned char* p = put_blob_header(buf, 0x31504D47u /* 'GMP1' */, &h, sizeof(h));
  std::memcpy(p, c.rec, (size_t)h.n_primitives * sizeof(gm_primitive_record)); p += (size_t)h.n_primitives * sizeof(gm_primitive_record);
  return put_blob_centroids(ctx, p, ctx->d_pr_cc, h.n_residual_voxels);
}

}  // extern "C"

// ---- scan-to-scan registration (gm_register.cuh) -------------------------------------------------
namespace {
static_assert(sizeof(gm_icp_params) == 88 && sizeof(gm_registration) == 416, "registration layouts");

int reg_blocks(const gm_ctx* ctx) { return ctx->num_sms * 8; }

// First call: the source's registration buffers and events (rare path, synchronous).
gm_status ensure_reg_buffers(gm_ctx* ctx) {
  if (ctx->d_reg_state.count) return GM_OK;
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  for (cudaEvent_t& e : ctx->ev_reg)
    if (!e) GM_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  GM_CUDA(ctx->d_reg_part.alloc((size_t)reg_blocks(ctx) * REG_NV));
  GM_CUDA(ctx->d_reg_idx.alloc(ctx->cap));
  GM_CUDA(ctx->d_reg_res.alloc(ctx->cap));
  GM_CUDA(ctx->d_reg_ticket.alloc(1));
  GM_CUDA(cudaMemsetAsync(ctx->d_reg_ticket, 0, sizeof(unsigned), ctx->stream));
  GM_CUDA(ctx->d_reg_state.alloc(1));  // last: a failure above leaves the set unallocated
  GM_CUDA(cudaMemsetAsync(ctx->d_reg_state, 0, sizeof(RegState), ctx->stream));
  return GM_OK;
}

bool finite_pose(const float* t) {
  for (int k = 0; k < 12; ++k) if (!std::isfinite(t[k])) return false;
  return true;
}

// gm_register's argument rules (gm_register_map adds its max_planarity's)
bool valid_icp_args(const gm_icp_params* p) {
  const double dmax = p->max_correspondence_distance;
  return dmax > 0.0 && std::isfinite(dmax) && p->max_iterations >= 1 && p->max_iterations <= GM_MAX_ICP_ITERATIONS &&
         p->min_rotation_step >= 0.0 && p->min_translation_step >= 0.0 && p->degeneracy_ratio >= 0.0 && p->degeneracy_ratio < 1.0 &&
         finite_pose(p->init_pose34);
}

// The kernel parameters of an ICP of `source`, and the grid of its iterations: a warp per source voxel, at most
// reg_blocks, at least one block (the kernels read the voxel count on the device).
RegParams icp_setup(const gm_ctx* source, const gm_icp_params* p, int* blocks) {
  *blocks = std::max(1, std::min(div_up((long long)source->n_grid * 32, REG_BLOCK), reg_blocks(source)));
  const double dmax = p->max_correspondence_distance;
  return RegParams{dmax, (float)(dmax * dmax), p->min_rotation_step, p->min_translation_step, p->degeneracy_ratio};
}

// The per-point outputs of ctx's last registration, whose target was a context (target 0) or a map (1): n_source of them,
// GM_ERR_CAPACITY above capacity_points, else d_idx copied into *idx and, if not null, the residuals into residual.
template <class T>
gm_status download_reg_points(gm_ctx* ctx, int target, const T* d_idx, std::vector<T>* idx, float* residual, size_t capacity_points) {
  if (gm_status s = require(ctx, REGISTRATION)) return s;
  if (ctx->reg_target != target) return GM_ERR_STAGE_ORDER;  // the other of gm_download_correspondences / _map_correspondences
  int V = 0;
  GM_CUDA(cudaMemcpyAsync(&V, &ctx->d_reg_state->n_source, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  if ((size_t)V > capacity_points) return GM_ERR_CAPACITY;
  if (V <= 0) return GM_OK;
  idx->resize((size_t)V);
  GM_CUDA(cudaMemcpyAsync(idx->data(), d_idx, (size_t)V * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
  if (residual) GM_CUDA(cudaMemcpyAsync(residual, ctx->d_reg_res, (size_t)V * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  return GM_OK;
}
}  // namespace

extern "C" {

void gm_icp_params_default(gm_icp_params* p) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  p->init_pose34[0] = p->init_pose34[5] = p->init_pose34[10] = 1.0f;
  p->max_correspondence_distance = 0.5;
  p->max_iterations = 30;
  p->min_rotation_step = 1e-5;
  p->min_translation_step = 1e-5;
  p->degeneracy_ratio = 0.0;
}

gm_status gm_register(gm_ctx* source, gm_ctx* target, const gm_icp_params* p) {
  if (!source || !target || !p) return GM_ERR_INVALID_ARG;
  gm_ctx* ctx = source;  // GM_CUDA / GM_LAUNCH report on the source
  if (source->device != target->device) { ctx->err = "gm_register: source and target on different devices"; return GM_ERR_INVALID_ARG; }
  if (!valid_icp_args(p)) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(target, NORMALS)) return s;
  if (target->injected) return GM_ERR_STAGE_ORDER;
  if (gm_status s = require(source, VOXEL)) return s;
  if (gm_status s = ensure_reg_buffers(source)) return s;
  ctx->stages &= ~(1u << REGISTRATION);
  if (target != source) {
    GM_CUDA(cudaEventRecord(source->ev_reg[0], target->stream));
    GM_CUDA(cudaStreamWaitEvent(source->stream, source->ev_reg[0], 0));
  }
  Pose34 init;
  std::memcpy(init.r, p->init_pose34, sizeof(init.r));
  GM_LAUNCH(ctx, k_reg_begin, 1, 32, source->d_reg_state, init, &source->d_st->vox.n_voxels);
  int blocks;
  const RegParams rp = icp_setup(source, p, &blocks);
  // an empty target built no grid this scan: its block table may still describe an earlier one
  const int search = target->n_grid > 0 ? 1 : 0;
  for (int it = 0; it < p->max_iterations; ++it)
    GM_LAUNCH(ctx, k_reg_iter, blocks, REG_BLOCK, source->d_centroid, &source->d_st->vox.n_voxels, target->d_sorted, target->d_tab,
              target->d_ucell_start, target->d_runs, target->d_cell_nruns, target->d_valid_map, target->d_cloud_c, target->d_normals_c,
              target->grid, target->d_st, search, rp, source->d_reg_state, source->d_reg_part, source->d_reg_ticket, source->d_reg_idx,
              source->d_reg_res);
  GM_CHECK_LAUNCHES(ctx);
  if (target != source) {
    GM_CUDA(cudaEventRecord(source->ev_reg[1], source->stream));
    GM_CUDA(cudaStreamWaitEvent(target->stream, source->ev_reg[1], 0));
  }
  source->reg_target = 0;
  mark(source, REGISTRATION);
  return GM_OK;
}

gm_status gm_get_registration(gm_ctx* ctx, gm_registration* out) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, REGISTRATION)) return s;
  RegState h;
  GM_CUDA(cudaMemcpyAsync(&h, ctx->d_reg_state, sizeof(RegState), cudaMemcpyDeviceToHost, ctx->stream));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  std::memset(out, 0, sizeof(*out));
  for (int k = 0; k < 12; ++k) out->pose34[k] = (float)h.T[k];
  out->iterations = h.iterations;
  out->converged = h.converged;
  out->n_source = h.n_source;
  out->n_correspondences = h.n_corr;
  out->rmse = h.n_corr > 0 ? (float)std::sqrt(h.sum_r2 / (double)h.n_corr) : 0.0f;
  out->fitness = h.n_source > 0 ? (float)((double)h.n_corr / (double)h.n_source) : 0.0f;
  out->n_degenerate = h.n_degenerate;
  std::memcpy(out->eigenvalues, h.eig, sizeof(h.eig));
  std::memcpy(out->eigenvectors, h.vecs, sizeof(h.vecs));
  return GM_OK;
}

gm_status gm_download_correspondences(gm_ctx* ctx, int32_t* target_index, float* residual, size_t capacity_points) {
  if (!ctx || !target_index) return GM_ERR_INVALID_ARG;
  std::vector<int> idx;
  if (gm_status s = download_reg_points(ctx, 0, ctx->d_reg_idx.p, &idx, residual, capacity_points)) return s;
  std::copy(idx.begin(), idx.end(), target_index);
  return GM_OK;
}

// ---- results ---------------------------------------------------------------------------------
gm_status gm_get_counts(gm_ctx* ctx, gm_counts* out) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  DevState h;
  gm_status s = sync_state(ctx, &h);
  if (s != GM_OK) return s;
  out->n_input = has(ctx, SCAN) ? h.n_input : -1;
  out->n_cropped = has(ctx, CROP) ? h.n_crop : -1;
  out->n_valid = has(ctx, COMPACTED) ? h.n_valid : -1;
  out->n_voxels = has(ctx, VOXEL) ? h.vox.n_voxels : -1;
  out->n_cells = has(ctx, NORMALS) ? h.n_cells : -1;
  out->voxel_overflow = h.vox.overflow;
  out->nn_out_of_range = h.nn_oor;
  out->device_error = h.error;
  if (h.error) { ctx->err = "device-side look-back spin bound hit"; return GM_ERR_INTERNAL; }
  return GM_OK;
}

#define GM_D2H(dst, src, bytes)                                                                  \
  do {                                                                                           \
    if ((bytes) > 0) GM_CUDA(cudaMemcpyAsync((dst), (src), (bytes), cudaMemcpyDeviceToHost, ctx->stream)); \
  } while (0)

gm_status gm_download_cloud(gm_ctx* ctx, int32_t which, float* out, size_t capacity_points) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  if (which < 0 || which > 1) return GM_ERR_STAGE_ORDER;
  if (gm_status s = require(ctx, which == 0 ? CROP : COMPACTED)) return s;
  DevState h;
  return download(ctx, &h, which == 0 ? n_crop : n_valid, capacity_points, {{out, which == 0 ? ctx->d_crop : ctx->d_cloud_c, 16}});
}

gm_status gm_download_normals(gm_ctx* ctx, int32_t which, float* out8, size_t capacity_points) {
  if (!ctx || !out8) return GM_ERR_INVALID_ARG;
  if (which < 0 || which > 1) return GM_ERR_STAGE_ORDER;
  if (gm_status s = require(ctx, which == 0 ? NORMALS : COMPACTED)) return s;
  DevState h;
  return download(ctx, &h, which == 0 ? n_crop : n_valid, capacity_points, {{out8, which == 0 ? ctx->d_normals : ctx->d_normals_c, 32}});
}

gm_status gm_download_neighbor_counts(gm_ctx* ctx, int32_t* out, size_t capacity_points) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, NORMALS)) return s;
  DevState h;
  return download(ctx, &h, n_crop, capacity_points, {{out, ctx->d_nbr, 4}});
}

gm_status gm_download_valid_map(gm_ctx* ctx, int32_t* out, size_t capacity_points) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, NORMALS)) return s;
  DevState h;
  return download(ctx, &h, n_crop, capacity_points, {{out, ctx->d_valid_map, 4}});
}

gm_status gm_download_voxel_assignment(gm_ctx* ctx, int32_t* keys, int32_t* assign, size_t capacity_points) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, VOXEL)) return s;
  if (ctx->vox_assign_on_demand && ctx->n_grid > 0) {
    GM_LAUNCH(ctx, k_voxel_lookup, std::min(div_up((long long)ctx->n_grid, 256), ctx->num_sms * 16), 256, ctx->d_cloud_c, &ctx->d_st->vox,
              ctx->d_vox_key, ctx->d_vkey_pt, ctx->d_assign);
    GM_CHECK_LAUNCHES(ctx);
  }
  DevState h;
  gm_status s = download(ctx, &h, n_valid, capacity_points, {{keys, ctx->d_vkey_pt, 4}, {assign, ctx->d_assign, 4}});
  if (s != GM_OK) return s;
  return h.vox.overflow ? GM_WARN_VOXEL_OVERFLOW : GM_OK;
}

gm_status gm_download_voxels(gm_ctx* ctx, float* centroids, int32_t* keys, int32_t* counts, int32_t* nn_index, float* nn_normal8,
                             size_t capacity_voxels) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, VOXEL)) return s;
  // asking for the 1-NN outputs without normals fails after the other copies are queued, without waiting for them
  const bool nn_missing = (nn_index || nn_normal8) && !has(ctx, NORMALS);
  DevState h;
  gm_status s = download(ctx, &h, n_voxels, capacity_voxels,
                         {{centroids, ctx->d_centroid, 16}, {keys, ctx->d_vox_key, 4}, {counts, ctx->d_vox_count, 4},
                          {nn_missing ? nullptr : nn_index, ctx->d_nn_idx, 4}, {nn_missing ? nullptr : nn_normal8, ctx->d_nn_normal, 32}},
                         !nn_missing);
  if (s != GM_OK) return s;
  if (nn_missing) return GM_ERR_STAGE_ORDER;
  if (h.vox.overflow) return GM_WARN_VOXEL_OVERFLOW;
  if (h.nn_oor && has(ctx, NORMALS)) return GM_ERR_NN_INDEX_RANGE;
  return GM_OK;
}

gm_status gm_get_voxel_grid(gm_ctx* ctx, int32_t grid6[6]) {
  if (!ctx || !grid6) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, VOXEL)) return s;
  DevState h;
  gm_status s = sync_state(ctx, &h);
  if (s != GM_OK) return s;
  for (int a = 0; a < 3; ++a) { grid6[a] = h.vox.min_b[a]; grid6[3 + a] = h.vox.div_b[a]; }
  return GM_OK;
}

gm_status gm_get_frame(gm_ctx* ctx, gm_frame* out) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, FRAME)) return s;
  static_assert(sizeof(FrameOut) == sizeof(gm_frame), "frame layout");
  GM_D2H(out, ctx->d_frame, sizeof(gm_frame));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  return GM_OK;
}

gm_status gm_download_hypotheses(gm_ctx* ctx, int32_t kind, float* coef, float* test12, int32_t* counts, int32_t capacity_h) {
  if (!ctx || (kind != 0 && kind != 1)) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, ransac_stage(kind))) return s;
  size_t H = (size_t)ctx->ransac_H[kind];
  if ((int)H > capacity_h) return GM_ERR_CAPACITY;
  if (coef) {
    if (kind == 0) GM_D2H(coef, ctx->hyp.plane_coef, H * 16);
    else GM_D2H(coef, ctx->hyp.model7, H * 28);
  }
  if (test12 && kind == 1) GM_D2H(test12, ctx->hyp.test12, H * 48);
  if (counts) GM_D2H(counts, ctx->hyp.counts[kind], H * 4);
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  return GM_OK;
}

gm_status gm_get_model(gm_ctx* ctx, int32_t kind, gm_model* out) {
  if (!ctx || !out || (kind != 0 && kind != 1)) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, model_stage(kind))) return s;
  ModelState h;
  GM_D2H(&h, ctx->hyp.model + kind, sizeof(ModelState));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  out->kind = h.kind; out->best_id = h.best_id; out->best_count = h.best_count; out->refit_count = h.refit_count;
  std::memcpy(out->hyp, h.hyp, sizeof(out->hyp));
  std::memcpy(out->coef, h.coef, sizeof(out->coef));
  out->rms = h.rms; out->pad_ = 0.f;
  return h.best_id < 0 ? GM_ERR_NO_MODEL : GM_OK;
}

gm_status gm_download_labels(gm_ctx* ctx, uint8_t* out, size_t capacity_points) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, LABELS)) return s;
  DevState h;
  return download(ctx, &h, n_valid, capacity_points, {{out, ctx->d_labels, 1}});
}

gm_status gm_download_polyline(gm_ctx* ctx, gm_slice* out, int32_t capacity, int32_t* n_slices) {
  if (!ctx || !n_slices) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, POLY)) return s;
  PolyState h;
  GM_D2H(&h, ctx->d_poly, sizeof(PolyState));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  *n_slices = h.S;
  if (h.S > capacity) return GM_ERR_CAPACITY;
  if (out && h.S > 0) {
    GM_D2H(out, ctx->d_slices, (size_t)h.S * sizeof(gm_slice));
    GM_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return GM_OK;
}

// ---- pipelined fetch + profiling ---------------------------------------------------------------
gm_status gm_fetch_async(gm_ctx* ctx, const gm_host_outputs* out) {
  if (!ctx || !out) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, SCAN)) return s;
  const size_t n = ctx->n_input;
  if (out->summary) {
    int mask = (has(ctx, MODEL_PLANE) ? 1 : 0) | (has(ctx, MODEL_CYL) ? 2 : 0) | (has(ctx, POLY) ? 4 : 0);
    GM_LAUNCH(ctx, k_pack_summary, 1, 32, ctx->d_st, ctx->d_frame, ctx->hyp.model, ctx->d_poly, mask, ctx->d_summary);
    GM_CHECK_LAUNCHES(ctx);
    GM_CUDA(cudaMemcpyAsync(out->summary, ctx->d_summary, sizeof(SummaryDev), cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (out->cloud_xyzw && has(ctx, COMPACTED)) GM_D2H(out->cloud_xyzw, ctx->d_cloud_c, std::min(n, out->cloud_capacity) * 16);
  if (out->normals8 && has(ctx, COMPACTED)) GM_D2H(out->normals8, ctx->d_normals_c, std::min(n, out->normals_capacity) * 32);
  if (out->labels && has(ctx, LABELS)) GM_D2H(out->labels, ctx->d_labels, std::min(n, out->labels_capacity));
  if (out->slices && has(ctx, POLY))
    GM_D2H(out->slices, ctx->d_slices, (size_t)std::min(ctx->prm.maxSlices, out->slices_capacity) * sizeof(gm_slice));
  if (has(ctx, VOXEL)) {
    if (out->centroids_xyzw) GM_D2H(out->centroids_xyzw, ctx->d_centroid, std::min(n, out->voxel_capacity) * 16);
    if (out->nn_normal8 && has(ctx, NORMALS)) GM_D2H(out->nn_normal8, ctx->d_nn_normal, std::min(n, out->voxel_capacity) * 32);
  }
  return GM_OK;
}

gm_status gm_profile_enable(gm_ctx* ctx, int32_t on) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  ctx->profiling = on != 0;
  return GM_OK;
}
int32_t gm_profile_num_segments(void) { return SEG_COUNT; }
const char* gm_profile_segment_name(int32_t i) { return (i >= 0 && i < SEG_COUNT) ? kSegNames[i] : ""; }
gm_status gm_profile_read(gm_ctx* ctx, float* ms_sum, int32_t* calls) {
  if (!ctx || !ms_sum || !calls) return GM_ERR_INVALID_ARG;
  GM_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int s = 0; s < SEG_COUNT; ++s) {
    for (auto& pr : ctx->seg_events[s]) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) { ms_sum[s] += ms; calls[s] += 1; }
      ctx->ev_pool.push_back(pr.first);
      ctx->ev_pool.push_back(pr.second);
    }
    ctx->seg_events[s].clear();
  }
  cudaGetLastError();
  return GM_OK;
}

// ---- test hook -------------------------------------------------------------------------------
gm_status gm_inject_compacted(gm_ctx* ctx, const float* xyzw_host, const float* normals8_host, size_t n) {
  if (!ctx || (n && !xyzw_host)) return GM_ERR_INVALID_ARG;
  if (n > ctx->cap) return GM_ERR_CAPACITY;
  new_scan(ctx, n);
  GM_LAUNCH(ctx, k_begin_scan, 1, 32, ctx->d_st, (int)n, (const float4*)nullptr);
  if (n) {
    GM_CUDA(cudaMemcpyAsync(ctx->d_cloud_c, xyzw_host, n * 16, cudaMemcpyHostToDevice, ctx->stream));
    if (normals8_host) GM_CUDA(cudaMemcpyAsync(ctx->d_normals_c, normals8_host, n * 32, cudaMemcpyHostToDevice, ctx->stream));
    else GM_CUDA(cudaMemsetAsync(ctx->d_normals_c, 0, n * 32, ctx->stream));
  }
  int nn = (int)n;
  GM_CUDA(cudaMemcpyAsync(&ctx->d_st->n_valid, &nn, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  GM_CUDA(cudaMemcpyAsync(&ctx->d_st->n_crop, &nn, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  GM_CUDA(cudaMemcpyAsync(&ctx->d_st->vox.n, &nn, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  GM_CUDA(cudaStreamSynchronize(ctx->stream));  // nn is a stack variable
  if (n) GM_LAUNCH(ctx, k_bbox, std::min(div_up((long long)n, 256), ctx->num_sms * 8), 256, ctx->d_cloud_c, &ctx->d_st->vox);
  GM_CHECK_LAUNCHES(ctx);
  mark(ctx, COMPACTED);
  ctx->injected = true;
  return GM_OK;
}

// ---- a6: host-side formatting of the published numbers ------------------------------------------
void gm_markers_eigen(const gm_frame* frame, gm_arrow out[3]) {
  // src/tunnel_processing.cpp:265: eigenValNorms = (1/eigenVals.norm()) * eigenVals.cwiseAbs()
  const float* v = frame->vals;
  float nrm = std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
  float inv = 1.0f / nrm;
  for (int i = 0; i < 3; ++i) {
    float e = inv * std::fabs(v[i]);
    gm_arrow& a = out[i];
    a.start[0] = a.start[1] = a.start[2] = 0.0f;
    a.end[0] = frame->vecs[0 * 3 + i]; a.end[1] = frame->vecs[1 * 3 + i]; a.end[2] = frame->vecs[2 * 3 + i];
    a.scale[0] = (float)(0.1 - (0.05 * e));     // :275
    a.scale[1] = (float)(0.3 - (0.15 * e));     // :276
    a.scale[2] = (float)(0.25 - (0.125 * e));   // :277
    a.color_argb[0] = 1.0f;                     // :280-287, pushed as (a,r,g,b)
    a.color_argb[1] = (i == 0) ? 1.0f : 0.0f;
    a.color_argb[2] = (i == 1) ? 1.0f : 0.0f;
    a.color_argb[3] = (i == 2) ? 1.0f : 0.0f;
    a.id = i;
  }
}

void gm_markers_normals(const float* centroids, const float* nn_normal8, int32_t V, gm_arrow* out) {
  gm_markers_normals_mode(centroids, nn_normal8, V, 0, out);
}

void gm_markers_normals_mode(const float* centroids, const float* nn_normal8, int32_t V, int32_t arrow_mode, gm_arrow* out) {
  for (int32_t i = 0; i < V; ++i) {
    gm_arrow& a = out[i];
    for (int k = 0; k < 3; ++k) {
      a.start[k] = centroids[(size_t)i * 4 + k];        // src/tunnel_processing.cpp:242-244
      a.end[k] = nn_normal8[(size_t)i * 8 + k];         // :247-249: end = the normal itself (quirk B.4)
      if (arrow_mode == 1) a.end[k] = a.start[k] + a.end[k];  // "fixed": the arrow points along the normal from the centroid
    }
    a.scale[0] = 0.025f; a.scale[1] = 0.075f; a.scale[2] = 0.0625f;  // :230
    a.color_argb[0] = 1.0f; a.color_argb[1] = 0.0f; a.color_argb[2] = 0.0f; a.color_argb[3] = 1.0f;  // :231 -> a=1,b=1 (quirk B.5)
    a.id = i;
  }
}

}  // extern "C"


// ---- on-disk store of the per-scan compressed primitives (SURVEY 8f.3; builder-defined) --------------------------------
// Append-only file: 'GMS1' | version u32, then one record per scan:
//   'GMSR' u32 | scan_id u64 | stamp_ns u64 | pose [R|t] 12 x f32 | blob_bytes u64 | blob (the GMC1 blob of
//   gm_download_compressed) | crc32(blob) u32
// The index (offset of every record) is rebuilt by scanning the file when it is opened; a torn last record (crash during an
// append) fails its length / CRC check, is ignored, and the next append overwrites it.
struct gm_store {
  FILE* f = nullptr;
  std::string path, err;
  struct Rec { uint64_t scan_id, stamp_ns, blob_bytes; long blob_off; float pose[12]; };
  std::vector<Rec> recs;
  long end = 8;  // where the next record goes
};

namespace {
uint32_t crc32_of(const unsigned char* p, size_t n) {
  static uint32_t table[256];
  static bool init = false;
  if (!init) {
    for (uint32_t i = 0; i < 256; ++i) { uint32_t c = i; for (int k = 0; k < 8; ++k) c = (c & 1u) ? 0xEDB88320u ^ (c >> 1) : c >> 1; table[i] = c; }
    init = true;
  }
  uint32_t c = 0xFFFFFFFFu;
  for (size_t i = 0; i < n; ++i) c = table[(c ^ p[i]) & 0xFFu] ^ (c >> 8);
  return c ^ 0xFFFFFFFFu;
}
constexpr uint32_t kStoreMagic = 0x31534D47u /* 'GMS1' */, kRecMagic = 0x52534D47u /* 'GMSR' */;
constexpr size_t kRecHead = 4 + 8 + 8 + 48 + 8;
}  // namespace

extern "C" {

gm_status gm_store_open(const char* path, int32_t create, gm_store** out) {
  if (!path || !out) return GM_ERR_INVALID_ARG;
  *out = nullptr;
  gm_store* st = new (std::nothrow) gm_store();
  if (!st) return GM_ERR_INTERNAL;
  try {
    st->path = path;
    st->f = std::fopen(path, "r+b");
    if (!st->f && create) {
      st->f = std::fopen(path, "w+b");
      const uint32_t hdr[2] = {kStoreMagic, 1u};
      if (!st->f || std::fwrite(hdr, 4, 2, st->f) != 2 || std::fflush(st->f) != 0) { if (st->f) std::fclose(st->f); delete st; return GM_ERR_INVALID_ARG; }
    }
    if (!st->f) { delete st; return GM_ERR_INVALID_ARG; }
    uint32_t hdr[2] = {0, 0};
    std::fseek(st->f, 0, SEEK_SET);
    if (std::fread(hdr, 4, 2, st->f) != 2 || hdr[0] != kStoreMagic || hdr[1] != 1u) { std::fclose(st->f); delete st; return GM_ERR_INVALID_ARG; }
    std::fseek(st->f, 0, SEEK_END);
    const long fsize = std::ftell(st->f);
    long off = 8;
    std::vector<unsigned char> blob;
    while (off + (long)kRecHead + 4 <= fsize) {  // rebuild the index; stop at the first record that does not check out
      unsigned char h[kRecHead];
      std::fseek(st->f, off, SEEK_SET);
      if (std::fread(h, 1, kRecHead, st->f) != kRecHead) break;
      uint32_t magic; gm_store::Rec r;
      std::memcpy(&magic, h, 4); std::memcpy(&r.scan_id, h + 4, 8); std::memcpy(&r.stamp_ns, h + 12, 8);
      std::memcpy(r.pose, h + 20, 48); std::memcpy(&r.blob_bytes, h + 68, 8);
      if (magic != kRecMagic || r.blob_bytes > (uint64_t)(fsize - off - (long)kRecHead - 4)) break;
      blob.resize((size_t)r.blob_bytes);
      uint32_t crc = 0;
      if ((r.blob_bytes && std::fread(blob.data(), 1, blob.size(), st->f) != blob.size()) || std::fread(&crc, 4, 1, st->f) != 1) break;
      if (crc != crc32_of(blob.data(), blob.size())) break;
      r.blob_off = off + (long)kRecHead;
      st->recs.push_back(r);
      off += (long)kRecHead + (long)r.blob_bytes + 4;
    }
    st->end = off;
  } catch (...) { if (st->f) std::fclose(st->f); delete st; return GM_ERR_INTERNAL; }
  *out = st;
  return GM_OK;
}

void gm_store_close(gm_store* st) {
  if (!st) return;
  if (st->f) std::fclose(st->f);
  delete st;
}

gm_status gm_store_append_blob(gm_store* st, uint64_t scan_id, uint64_t stamp_ns, const float* pose34, const void* blob, size_t bytes) {
  if (!st || !st->f || (bytes && !blob)) return GM_ERR_INVALID_ARG;
  try {
    gm_store::Rec r{};
    r.scan_id = scan_id; r.stamp_ns = stamp_ns; r.blob_bytes = bytes; r.blob_off = st->end + (long)kRecHead;
    const float ident[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
    std::memcpy(r.pose, pose34 ? pose34 : ident, 48);
    unsigned char h[kRecHead];
    std::memcpy(h, &kRecMagic, 4); std::memcpy(h + 4, &r.scan_id, 8); std::memcpy(h + 12, &r.stamp_ns, 8);
    std::memcpy(h + 20, r.pose, 48); std::memcpy(h + 68, &r.blob_bytes, 8);
    const uint32_t crc = crc32_of((const unsigned char*)blob, bytes);
    if (std::fseek(st->f, st->end, SEEK_SET) != 0 || std::fwrite(h, 1, kRecHead, st->f) != kRecHead ||
        (bytes && std::fwrite(blob, 1, bytes, st->f) != bytes) || std::fwrite(&crc, 4, 1, st->f) != 1 || std::fflush(st->f) != 0) {
      st->err = "write failed";
      return GM_ERR_INVALID_ARG;
    }
    st->recs.push_back(r);
    st->end += (long)kRecHead + (long)bytes + 4;
  } catch (...) { return GM_ERR_INTERNAL; }
  return GM_OK;
}

/* compress output of `ctx` (after gm_compress) -> one record */
gm_status gm_store_append(gm_store* st, gm_ctx* ctx, uint64_t scan_id, uint64_t stamp_ns, const float* pose34) {
  if (!st || !ctx) return GM_ERR_INVALID_ARG;
  size_t bytes = 0;
  gm_status s = gm_download_compressed(ctx, nullptr, 0, &bytes);
  if (s != GM_OK) return s;
  try {
    std::vector<unsigned char> blob(bytes);
    if ((s = gm_download_compressed(ctx, blob.data(), blob.size(), &bytes)) != GM_OK) return s;
    return gm_store_append_blob(st, scan_id, stamp_ns, pose34, blob.data(), bytes);
  } catch (...) { return GM_ERR_INTERNAL; }
}

int64_t gm_store_count(const gm_store* st) { return st ? (int64_t)st->recs.size() : -1; }

gm_status gm_store_info(const gm_store* st, int64_t i, uint64_t* scan_id, uint64_t* stamp_ns, float* pose34, uint64_t* blob_bytes) {
  if (!st || i < 0 || i >= (int64_t)st->recs.size()) return GM_ERR_INVALID_ARG;
  const gm_store::Rec& r = st->recs[(size_t)i];
  if (scan_id) *scan_id = r.scan_id;
  if (stamp_ns) *stamp_ns = r.stamp_ns;
  if (pose34) std::memcpy(pose34, r.pose, 48);
  if (blob_bytes) *blob_bytes = r.blob_bytes;
  return GM_OK;
}

gm_status gm_store_read(gm_store* st, int64_t i, void* buf, size_t capacity, size_t* bytes) {
  if (!st || !st->f || i < 0 || i >= (int64_t)st->recs.size() || !bytes) return GM_ERR_INVALID_ARG;
  const gm_store::Rec& r = st->recs[(size_t)i];
  *bytes = (size_t)r.blob_bytes;
  if (!buf) return GM_OK;
  if (capacity < r.blob_bytes) return GM_ERR_CAPACITY;
  if (std::fseek(st->f, r.blob_off, SEEK_SET) != 0 || (r.blob_bytes && std::fread(buf, 1, (size_t)r.blob_bytes, st->f) != r.blob_bytes)) return GM_ERR_INVALID_ARG;
  return GM_OK;
}

}  // extern "C"


// ---- ROS-free encoders of what cloud_cb publishes (SURVEY 8f.1) ------------------------------------------------------
// ROS 1 wire format (little endian; string / array = uint32 length + payload), written field by field in message order.
namespace {
struct Wr {
  unsigned char* p; size_t cap, n = 0; bool ok = true;
  Wr(void* b, size_t c) : p((unsigned char*)b), cap(c) {}
  void raw(const void* src, size_t k) { if (p && n + k <= cap) std::memcpy(p + n, src, k); else if (p) ok = false; n += k; }
  void u8(uint8_t v) { raw(&v, 1); }
  void u32(uint32_t v) { raw(&v, 4); }
  void i32(int32_t v) { raw(&v, 4); }
  void f32(float v) { raw(&v, 4); }
  void f64(double v) { raw(&v, 8); }
  void str(const char* s) { const uint32_t l = s ? (uint32_t)std::strlen(s) : 0u; u32(l); if (l) raw(s, l); }
  void header(uint32_t seq, uint64_t stamp_ns, const char* frame) { u32(seq); u32((uint32_t)(stamp_ns / 1000000000ull)); u32((uint32_t)(stamp_ns % 1000000000ull)); str(frame); }
};

// sensor_msgs/PointCloud2 exactly as pcl::toROSMsg(pcl::PointCloud<pcl::PointXYZ>) builds it (src/geometric_mapping.cpp:102-103):
// unorganised (height 1), fields x,y,z FLOAT32 at offsets 0,4,8, point_step 16 (the PointXYZ padding word travels), is_dense as given
size_t write_pointcloud2(Wr& w, const float* xyzw, size_t n, const char* frame, uint32_t seq, uint64_t stamp_ns, int is_dense) {
  w.header(seq, stamp_ns, frame);
  w.u32(1); w.u32((uint32_t)n);
  w.u32(3);
  const char* names[3] = {"x", "y", "z"};
  for (uint32_t k = 0; k < 3; ++k) { w.str(names[k]); w.u32(4 * k); w.u8(7 /* FLOAT32 */); w.u32(1); }
  w.u8(0); w.u32(16); w.u32((uint32_t)(16 * n));
  w.u32((uint32_t)(16 * n));
  if (n) w.raw(xyzw, 16 * n);
  w.u8(is_dense ? 1 : 0);
  return w.n;
}

// visualization_msgs/Marker as rvizArrow fills it (src/tunnel_processing.cpp:171-203): ARROW (0), ADD (0), two points,
// default pose / lifetime / frame_locked, colour serialised r,g,b,a from the (a,r,g,b) payload
void write_marker(Wr& w, const gm_arrow& a, const char* frame, const char* ns, uint64_t stamp_ns) {
  w.header(0, stamp_ns, frame);
  w.str(ns); w.i32(a.id); w.i32(0); w.i32(0);
  for (int k = 0; k < 7; ++k) w.f64(0.0);                       // pose: position + orientation, value-initialised
  for (int k = 0; k < 3; ++k) w.f64((double)a.scale[k]);
  w.f32(a.color_argb[1]); w.f32(a.color_argb[2]); w.f32(a.color_argb[3]); w.f32(a.color_argb[0]);
  w.i32(0); w.i32(0);                                          // lifetime
  w.u8(0);                                                     // frame_locked
  w.u32(2);
  for (int k = 0; k < 3; ++k) w.f64((double)a.start[k]);
  for (int k = 0; k < 3; ++k) w.f64((double)a.end[k]);
  w.u32(0);                                                    // colors[]
  w.str(""); w.str("");                                        // text, mesh_resource
  w.u8(0);                                                     // mesh_use_embedded_materials
}
}  // namespace

extern "C" {

size_t gm_pointcloud2_size(size_t n_points, const char* frame_id) {
  Wr w(nullptr, 0);
  return write_pointcloud2(w, nullptr, n_points, frame_id, 0, 0, 1);
}

gm_status gm_encode_pointcloud2(const float* xyzw, size_t n, const char* frame_id, uint32_t seq, uint64_t stamp_ns, int32_t is_dense, void* buf,
                                size_t capacity, size_t* bytes) {
  if ((n && !xyzw) || !buf || n > 0x0FFFFFFFu) return GM_ERR_INVALID_ARG;
  Wr w(buf, capacity);
  write_pointcloud2(w, xyzw, n, frame_id, seq, stamp_ns, is_dense);
  if (bytes) *bytes = w.n;
  return w.ok ? GM_OK : GM_ERR_CAPACITY;
}

size_t gm_marker_array_size(int32_t n_markers, const char* frame_id, const char* ns) {
  Wr w(nullptr, 0);
  gm_arrow a{};
  write_marker(w, a, frame_id, ns, 0);
  return 4 + (size_t)std::max(n_markers, 0) * w.n;
}

gm_status gm_encode_marker_array(const gm_arrow* arrows, int32_t n, const char* frame_id, const char* ns, uint64_t stamp_ns, void* buf,
                                 size_t capacity, size_t* bytes) {
  if (n < 0 || (n && !arrows) || !buf) return GM_ERR_INVALID_ARG;
  Wr w(buf, capacity);
  w.u32((uint32_t)n);
  for (int32_t i = 0; i < n; ++i) write_marker(w, arrows[i], frame_id, ns, stamp_ns);
  if (bytes) *bytes = w.n;
  return w.ok ? GM_OK : GM_ERR_CAPACITY;
}

}  // extern "C"


// ---- peer-memory collectives (gm_comm.cuh) -----------------------------------------------------------------------
struct gm_comm {
  int rank = 0, world = 1, device = 0;
  DevBuf<CommBox> d_box;  // this rank's mailbox
  DevBuf<CommDev> d_dev;  // device copy of the peer table
  CommDev h_dev{};
  bool connected = false;
  void* opened[COMM_MAX_RANKS] = {};
  std::string err;
};

static const CommDev* comm_dev(const gm_ctx* ctx) { return ctx->comm ? ctx->comm->d_dev.p : nullptr; }

extern "C" {

gm_status gm_comm_create(int32_t rank, int32_t world, gm_comm** out) {
  if (!out) return GM_ERR_INVALID_ARG;
  *out = nullptr;
  if (world < 1 || world > COMM_MAX_RANKS || rank < 0 || rank >= world) return GM_ERR_INVALID_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return GM_ERR_NO_DEVICE; }
  gm_comm* c = new (std::nothrow) gm_comm();
  if (!c) return GM_ERR_INTERNAL;
  c->rank = rank; c->world = world;
  cudaGetDevice(&c->device);
  if (c->d_box.alloc(1) != cudaSuccess || c->d_dev.alloc(1) != cudaSuccess ||
      cudaMemset(c->d_box, 0, sizeof(CommBox)) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) {
    cudaGetLastError();
    gm_comm_destroy(c);
    return GM_ERR_CUDA;
  }
  c->h_dev.local = c->d_box; c->h_dev.rank = rank; c->h_dev.world = world;
  c->h_dev.peer[rank] = c->d_box;
  if (world == 1) {
    if (cudaMemcpy(c->d_dev, &c->h_dev, sizeof(CommDev), cudaMemcpyHostToDevice) != cudaSuccess) { gm_comm_destroy(c); return GM_ERR_CUDA; }
    c->connected = true;
  }
  *out = c;
  return GM_OK;
}

gm_status gm_comm_handle(gm_comm* c, void* handle64) {
  if (!c || !handle64) return GM_ERR_INVALID_ARG;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t h;
  if (cudaIpcGetMemHandle(&h, c->d_box) != cudaSuccess) { c->err = cudaGetErrorString(cudaGetLastError()); return GM_ERR_CUDA; }
  std::memcpy(handle64, &h, 64);
  return GM_OK;
}

gm_status gm_comm_connect(gm_comm* c, const void* handles) {
  if (!c || !handles) return GM_ERR_INVALID_ARG;
  if (c->connected) return GM_OK;
  for (int r = 0; r < c->world; ++r) {
    if (r == c->rank) continue;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, (const unsigned char*)handles + (size_t)r * 64, 64);
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { c->err = std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e); cudaGetLastError(); return GM_ERR_CUDA; }
    c->opened[r] = p;
    c->h_dev.peer[r] = (CommBox*)p;
  }
  if (cudaMemcpy(c->d_dev, &c->h_dev, sizeof(CommDev), cudaMemcpyHostToDevice) != cudaSuccess) return GM_ERR_CUDA;
  c->connected = true;
  return GM_OK;
}

/* same-process peers (several contexts / devices driven by one process): mailbox addresses instead of IPC handles */
gm_status gm_comm_mailbox(gm_comm* c, void** box) {
  if (!c || !box) return GM_ERR_INVALID_ARG;
  *box = c->d_box;
  return GM_OK;
}
gm_status gm_comm_connect_local(gm_comm* c, void* const* boxes) {
  if (!c || !boxes) return GM_ERR_INVALID_ARG;
  for (int r = 0; r < c->world; ++r) {
    if (r == c->rank) continue;
    if (!boxes[r]) return GM_ERR_INVALID_ARG;
    c->h_dev.peer[r] = (CommBox*)boxes[r];
  }
  if (cudaMemcpy(c->d_dev, &c->h_dev, sizeof(CommDev), cudaMemcpyHostToDevice) != cudaSuccess) return GM_ERR_CUDA;
  c->connected = true;
  return GM_OK;
}

void gm_comm_destroy(gm_comm* c) {
  if (!c) return;
  cudaDeviceSynchronize();
  for (int r = 0; r < COMM_MAX_RANKS; ++r) if (c->opened[r]) cudaIpcCloseMemHandle(c->opened[r]);
  delete c;
  cudaGetLastError();
}

int32_t gm_comm_rank(const gm_comm* c) { return c ? c->rank : -1; }
int32_t gm_comm_world(const gm_comm* c) { return c ? c->world : 0; }
const char* gm_comm_last_error(const gm_comm* c) { return c ? c->err.c_str() : "null comm"; }

gm_status gm_set_comm(gm_ctx* ctx, gm_comm* comm) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (comm && !comm->connected) { ctx->err = "gm_comm is not connected"; return GM_ERR_STAGE_ORDER; }
  new_graph_generation(ctx);
  ctx->comm = comm;
  return GM_OK;
}

// One hypothesis-sharded RANSAC round for both primitives: this rank generates, counts and arg-maxes its share of the
// ids [0, H); the last block of each counting kernel stores (key, winner coefficients) into every peer's mailbox; a
// one-warp kernel per primitive picks the global winner out of this rank's own mailbox; both winners are refitted
// (every rank holds the same scan, so every rank ends with the same models).  No host synchronisation, no library
// collective, no copies: 2 x (hypotheses + count/argmax/send + receive) + refits.
gm_status gm_ransac_sharded(gm_ctx* ctx, const int32_t* plane_samples_host, int32_t Hp, const int32_t* cyl_samples_host, int32_t Hc) {
  if (!ctx || Hp <= 0 || Hc <= 0 || !plane_samples_host || !cyl_samples_host) return GM_ERR_INVALID_ARG;
  if (!ctx->comm) { ctx->err = "gm_ransac_sharded needs gm_set_comm"; return GM_ERR_STAGE_ORDER; }
  if (gm_status s = require(ctx, COMPACTED)) return s;
  const int W = ctx->comm->world, R = ctx->comm->rank;
  auto range = [&](int H, int& b, int& e) { const int per = (H + W - 1) / W; b = std::min(R * per, H); e = std::min((R + 1) * per, H); };
  int pb, pe, cb, ce;
  range(Hp, pb, pe); range(Hc, cb, ce);
  auto recv = [&](int kind, int H) -> gm_status {
    GM_LAUNCH(ctx, k_comm_recv_model, 1, 32, ctx->comm->h_dev, kind, H, ctx->hyp.key + kind, ctx->hyp.plane_coef, ctx->hyp.model7, ctx->hyp.test12,
              ctx->hyp.counts[kind], &ctx->d_st->error);
    GM_CHECK_LAUNCHES(ctx);
    return GM_OK;
  };
  auto plane = [&]() -> gm_status {
    gm_status r = gm_ransac(ctx, GM_MODEL_PLANE, plane_samples_host, Hp, pb, pe);
    if (r == GM_OK) r = recv(0, Hp);
    return r != GM_OK ? r : gm_ransac_select(ctx, GM_MODEL_PLANE);
  };
  auto cylinder = [&]() -> gm_status {
    gm_status r = gm_ransac(ctx, GM_MODEL_CYLINDER, cyl_samples_host, Hc, cb, ce);
    if (r == GM_OK) r = recv(1, Hc);
    return r != GM_OK ? r : gm_ransac_select(ctx, GM_MODEL_CYLINDER);
  };
  auto body = [&]() -> gm_status {
    ctx->sharded = true;
    const gm_status s = plane_and_cylinder(ctx, plane, cylinder);
    ctx->sharded = false;
    return s;
  };
  const bool graphable = ctx->graph_mode != 0 && ctx->concurrent && !ctx->profiling && ctx->n_grid > 0;  // a round is ~10 short launches: always worth it
  if (!graphable) return body();
  auto stage = [&]() -> gm_status {
    gm_status s = stage_samples(ctx, 0, plane_samples_host, pb, pe, 3);
    return s != GM_OK ? s : stage_samples(ctx, 1, cyl_samples_host, cb, ce, 2);
  };
  // (world, rank) are part of what is launched: the comm is attached with gm_set_comm, which starts a new graph generation
  gm_status s = run_graphed(ctx, 1, Hp, Hc, stage, body);
  if (s == GM_OK) {
    mark(ctx, RANSAC_PLANE, RANSAC_CYL, MODEL_PLANE, MODEL_CYL);
    ctx->ransac_H[0] = Hp; ctx->ransac_H[1] = Hc;
  }
  return s;
}

// map slabs: MIN/MAX of the bounding boxes of the compacted clouds of all ranks, in place in device state (after
// gm_normals, before gm_voxel): every slab then builds its voxels on ONE lattice.  One kernel, no host round trip.
gm_status gm_allreduce_voxel_bbox(gm_ctx* ctx) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (!ctx->comm) { ctx->err = "needs gm_set_comm"; return GM_ERR_STAGE_ORDER; }
  if (gm_status s = require(ctx, COMPACTED)) return s;
  GM_LAUNCH(ctx, k_comm_bbox, 1, 32, ctx->comm->h_dev, ctx->d_st->vox.bbox_min, ctx->d_st->vox.bbox_max, &ctx->d_st->error);
  GM_CHECK_LAUNCHES(ctx);
  return GM_OK;
}

// map slabs: the local frame of the WHOLE map = eigen-decomposition of the sum of the slabs' scatter matrices
// (getLocalFrame, src/tunnel_processing.cpp:92-148, applied to all normals of all ranks).  After gm_local_frame.
gm_status gm_allreduce_frame(gm_ctx* ctx) {
  if (!ctx) return GM_ERR_INVALID_ARG;
  if (!ctx->comm) { ctx->err = "needs gm_set_comm"; return GM_ERR_STAGE_ORDER; }
  if (gm_status s = require(ctx, FRAME)) return s;
  GM_LAUNCH(ctx, k_comm_sum, 1, 32, ctx->comm->h_dev, ctx->d_frame_sums, 6, &ctx->d_st->error);
  GM_LAUNCH(ctx, k_frame_solve, 1, 32, ctx->d_frame_sums, ctx->d_frame);
  GM_CHECK_LAUNCHES(ctx);
  return GM_OK;
}

}  // extern "C"

// ---- aggregated voxel map across scans (SURVEY 8f.3) -------------------------------------------------
struct gm_map {
  double leaf = 0.1;
  float inv_leaf = 10.f;
  unsigned long long n_slots = 0;
  DevBuf<unsigned long long> d_keys;
  DevBuf<int> d_cnt;
  DevBuf<long long> d_sums;
  DevBuf<MapState> d_st;
  DevBuf<int> d_cursor;
  int num_sms = 148;
  int device = 0;
  // the last map operation issued on a context stream (gm_map_insert, gm_register_map): the next one waits for it
  cudaEvent_t ev_last = nullptr;
  // per-slot plane tables of k_map_planes (allocated by the first use): centroid + has-plane flag, normal
  DevBuf<float4> d_plane_cent, d_plane_nrm;
  DevBuf<int> d_plane_box;  // [8] cells of the voxels with a plane: min x, y, z, -, -max x, y, z, - (k_map_planes)
  // gm_map_evict's scratch (allocated by the first eviction): the kept voxels, n_slots entries, and the split's counters
  DevBuf<unsigned long long> d_kept_keys;
  DevBuf<int> d_kept_cnt;
  DevBuf<long long> d_kept_sums;
  DevBuf<MapEvictState> d_evict_st;
  ~gm_map() { if (ev_last) cudaEventDestroy(ev_last); }
};

// GM_CUDA of the map calls that take no context
#define GM_MAP_CUDA(call) do { if ((call) != cudaSuccess) return GM_ERR_CUDA; } while (0)

namespace {
// The device scope of a map call that takes no context: the map's device is current until the scope ends, then the
// caller's again.  With sync, the caller's device is synchronised first (an insert from a context there is then complete)
// and then, if it is another one, the map's.
struct MapDeviceScope {
  int caller = -1, device;
  cudaError_t status;
  MapDeviceScope(int map_device, bool sync) : device(map_device) {
    status = cudaGetDevice(&caller);
    if (status == cudaSuccess && sync) status = cudaDeviceSynchronize();
    if (status == cudaSuccess && caller != device) status = cudaSetDevice(device);
    if (status == cudaSuccess && sync && caller != device) status = cudaDeviceSynchronize();
    if (status != cudaSuccess) cudaGetLastError();
  }
  ~MapDeviceScope() { if (caller >= 0 && caller != device) cudaSetDevice(caller); }
};

gm_status map_clear_device(gm_map* m) {
  if (cudaMemset(m->d_keys, 0xFF, m->n_slots * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMemset(m->d_cnt, 0, m->n_slots * sizeof(int)) != cudaSuccess ||
      cudaMemset(m->d_sums, 0, 3 * m->n_slots * sizeof(long long)) != cudaSuccess ||
      cudaMemset(m->d_st, 0, sizeof(MapState)) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) return GM_ERR_CUDA;
  return GM_OK;
}

int map_blocks(const gm_map* m) { return (int)std::min<unsigned long long>((m->n_slots + 255) / 256, (unsigned long long)m->num_sms * 16); }

cudaError_t ensure_plane_tables(gm_map* m) {
  if (m->d_plane_cent.count) return cudaSuccess;
  cudaError_t e = m->d_plane_nrm.alloc(m->n_slots);
  if (e == cudaSuccess) e = m->d_plane_box.alloc(8);
  if (e == cudaSuccess) e = m->d_plane_cent.alloc(m->n_slots);  // last: a failure above leaves the pair unallocated
  return e;
}

// What map_export gathers of every voxel besides the map's state: nothing, key + count + sums, or key + plane normal.
enum MapExportKind { MAP_STATE, MAP_VOXELS, MAP_PLANES };
struct MapExport {
  MapState st{};
  std::vector<unsigned long long> keys;
  std::vector<int> cnt;         // MAP_VOXELS
  std::vector<long long> sums;  // MAP_VOXELS, 3 a voxel
  std::vector<float4> nrm;      // MAP_PLANES
};

// The gathered values d, w per voxel, copied back into *out in key order: out's voxel i = d's voxel order[i].
template <class T>
cudaError_t copy_in_order(const DevBuf<T>& d, size_t w, const std::vector<size_t>& order, std::vector<T>* out) {
  std::vector<T> h(w * order.size());
  const cudaError_t e = cudaMemcpy(h.data(), d, h.size() * sizeof(T), cudaMemcpyDeviceToHost);
  out->resize(h.size());
  for (size_t i = 0; i < order.size(); ++i) std::copy_n(&h[w * order[i]], w, &(*out)[w * i]);
  return e;
}

// In the map's device scope: synchronise, read the state, then gather `what` of the occupied slots into temporary V-sized
// buffers (MAP_PLANES: k_map_planes at max_planarity first), copy them back and sort them by key (z-major, then y, then
// x): a deterministic order whatever the insertion history.  An empty map, or one of more than `capacity` voxels, gathers
// nothing.
gm_status map_export(gm_map* m, MapExportKind what, MapExport* x, double max_planarity = 0.0, size_t capacity = SIZE_MAX) {
  MapDeviceScope scope(m->device, true);
  GM_MAP_CUDA(scope.status);
  GM_MAP_CUDA(cudaMemcpy(&x->st, m->d_st, sizeof(MapState), cudaMemcpyDeviceToHost));
  const size_t V = (size_t)std::max(x->st.n_voxels, 0);
  if (what == MAP_STATE || V == 0 || V > capacity) return GM_OK;
  const bool planes = what == MAP_PLANES;
  DevBuf<unsigned long long> dk; DevBuf<int> dc; DevBuf<long long> ds; DevBuf<float4> dn;
  GM_MAP_CUDA(dk.alloc(V));
  if (planes) {
    GM_MAP_CUDA(ensure_plane_tables(m));
    GM_MAP_CUDA(dn.alloc(V));
    GM_MAP_CUDA(cudaMemset(m->d_plane_box, 0x7F, 8 * sizeof(int)));
    k_map_planes<<<map_blocks(m), 256>>>(m->d_keys, m->d_cnt, m->d_sums, m->n_slots - 1ull, max_planarity, m->d_plane_cent, m->d_plane_nrm,
                                         m->d_plane_box);
  } else {
    GM_MAP_CUDA(dc.alloc(V));
    GM_MAP_CUDA(ds.alloc(3 * V));
  }
  GM_MAP_CUDA(cudaMemset(m->d_cursor, 0, sizeof(int)));
  k_map_export<<<map_blocks(m), 256>>>(m->d_keys, m->d_cnt, m->d_sums, m->d_plane_nrm, m->n_slots, dk, dc, ds, dn, (int)V, m->d_cursor);
  GM_MAP_CUDA(cudaGetLastError());
  std::vector<unsigned long long> k(V);
  GM_MAP_CUDA(cudaMemcpy(k.data(), dk, V * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  std::vector<size_t> order(V);
  std::iota(order.begin(), order.end(), size_t(0));
  std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return k[a] < k[b]; });
  for (size_t j : order) x->keys.push_back(k[j]);
  cudaError_t e = planes ? copy_in_order(dn, 1, order, &x->nrm) : copy_in_order(dc, 1, order, &x->cnt);
  if (e == cudaSuccess && !planes) e = copy_in_order(ds, 3, order, &x->sums);
  return e == cudaSuccess ? GM_OK : GM_ERR_CUDA;
}

// the leaf and device rules of gm_map_evict / gm_map_merge / gm_odometry_set_window: the same lattice, the same device
bool same_lattice(const gm_map* a, const gm_map* b) {
  return a->device == b->device && std::memcmp(&a->leaf, &b->leaf, sizeof(double)) == 0;
}

cudaError_t ensure_evict_buffers(gm_map* m) {
  if (m->d_evict_st.count) return cudaSuccess;
  cudaError_t e = m->d_kept_keys.alloc(m->n_slots);
  if (e == cudaSuccess) e = m->d_kept_cnt.alloc(m->n_slots);
  if (e == cudaSuccess) e = m->d_kept_sums.alloc(3 * m->n_slots);
  if (e == cudaSuccess) e = m->d_evict_st.alloc(1);  // last: a failure above leaves the set unallocated
  return e;
}

// The launches of gm_map_evict on ctx's stream, after its checks and waits (buffers allocated): the counters' reset, then
// k_map_evict_split, k_map_evict_clear and k_map_restore.  Centre = c3 (host), or the translation of the device pose
// pose34_dev.  Shared by gm_map_evict and gm_odometry_step.
gm_status map_evict_launch(gm_map* m, gm_ctx* ctx, gm_map* archive, const float* c3, const float* pose34_dev, int half_cells) {
  GM_CUDA(cudaMemsetAsync(m->d_evict_st, 0, sizeof(MapEvictState), ctx->stream));
  const float cx = c3 ? c3[0] : 0.f, cy = c3 ? c3[1] : 0.f, cz = c3 ? c3[2] : 0.f;
  GM_LAUNCH(ctx, k_map_evict_split, map_blocks(m), 256, m->d_keys, m->d_cnt, m->d_sums, m->n_slots - 1ull, m->inv_leaf, cx, cy, cz, pose34_dev,
            half_cells, archive ? (unsigned long long*)archive->d_keys : nullptr, archive ? (int*)archive->d_cnt : nullptr,
            archive ? (long long*)archive->d_sums : nullptr, archive ? archive->n_slots - 1ull : 0ull, archive ? (MapState*)archive->d_st : nullptr,
            m->d_kept_keys, m->d_kept_cnt, m->d_kept_sums, m->d_evict_st);
  GM_LAUNCH(ctx, k_map_evict_clear, map_blocks(m), 256, m->d_keys, m->d_cnt, m->d_sums, m->n_slots, m->d_evict_st, m->d_st);
  GM_LAUNCH(ctx, k_map_restore, map_blocks(m), 256, m->d_kept_keys, m->d_kept_cnt, m->d_kept_sums, 0, m->d_evict_st, m->d_keys, m->d_cnt,
            m->d_sums, m->n_slots - 1ull, m->d_st);
  GM_CHECK_LAUNCHES(ctx);
  return GM_OK;
}
}  // namespace

extern "C" {

gm_status gm_map_create(double leaf, size_t capacity_voxels, gm_map** out) {
  if (!out) return GM_ERR_INVALID_ARG;
  *out = nullptr;
  if (!(leaf > 0.0) || capacity_voxels == 0 || capacity_voxels > (1ull << 31)) return GM_ERR_INVALID_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return GM_ERR_NO_DEVICE; }
  gm_map* m = new gm_map();
  m->leaf = leaf;
  m->inv_leaf = 1.0f / (float)leaf;  // as pcl::VoxelGrid: inverse_leaf_size = 1 / leaf_size (float)
  unsigned long long slots = 64;
  while (slots < 2ull * capacity_voxels) slots <<= 1;  // load factor <= 0.5
  m->n_slots = slots;
  int dev = 0; cudaGetDevice(&dev);
  m->device = dev;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) m->num_sms = prop.multiProcessorCount;
  if (cudaEventCreateWithFlags(&m->ev_last, cudaEventDisableTiming) != cudaSuccess || m->d_keys.alloc(slots) != cudaSuccess || m->d_cnt.alloc(slots) != cudaSuccess || m->d_sums.alloc(3 * slots) != cudaSuccess ||
      m->d_st.alloc(1) != cudaSuccess || m->d_cursor.alloc(1) != cudaSuccess || map_clear_device(m) != GM_OK) {
    gm_map_destroy(m);
    return GM_ERR_CUDA;
  }
  *out = m;
  return GM_OK;
}

void gm_map_destroy(gm_map* m) {
  if (!m) return;
  MapDeviceScope scope(m->device, true);
  delete m;
}

gm_status gm_map_clear(gm_map* m) {
  if (!m) return GM_ERR_INVALID_ARG;
  MapDeviceScope scope(m->device, true);
  GM_MAP_CUDA(scope.status);
  return map_clear_device(m);
}

gm_status gm_map_insert(gm_map* m, gm_ctx* ctx, const float* pose34, int32_t label_filter) {
  if (!m || !ctx || label_filter > 255) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(ctx, COMPACTED)) return s;
  if (label_filter >= 0 && !has(ctx, LABELS)) return GM_ERR_STAGE_ORDER;
  if (ctx->n_input == 0) return GM_OK;
  Pose34 T{};
  if (pose34) std::memcpy(T.r, pose34, sizeof(T.r));
  int blocks = std::min(div_up((long long)ctx->n_input, 256), ctx->num_sms * 16);
  const bool ordered = ctx->device == m->device;  // map operations issued on streams of the map's device run in call order
  if (ordered) GM_CUDA(cudaStreamWaitEvent(ctx->stream, m->ev_last, 0));
  GM_LAUNCH(ctx, k_map_insert, blocks, 256, ctx->d_cloud_c, ctx->d_labels, &ctx->d_st->n_valid, label_filter < 0 ? -1 : label_filter, T,
            pose34 ? 1 : 0, m->inv_leaf, m->d_keys, m->d_cnt, m->d_sums, m->n_slots - 1ull, m->d_st);
  GM_CHECK_LAUNCHES(ctx);
  if (ordered) GM_CUDA(cudaEventRecord(m->ev_last, ctx->stream));
  return GM_OK;
}

gm_status gm_map_stats(gm_map* m, int64_t* n_voxels, int64_t* n_points, int64_t* n_out_of_range) {
  if (!m) return GM_ERR_INVALID_ARG;
  MapExport x;
  if (gm_status s = map_export(m, MAP_STATE, &x)) return s;
  if (n_voxels) *n_voxels = x.st.n_voxels;
  if (n_points) *n_points = (int64_t)x.st.n_points;
  if (n_out_of_range) *n_out_of_range = x.st.out_of_range;
  return x.st.overflow ? GM_ERR_CAPACITY : GM_OK;
}

gm_status gm_map_download(gm_map* m, int32_t* ijk, int32_t* counts, float* centroids_xyzw, size_t capacity, size_t* n) {
  if (!m || !n) return GM_ERR_INVALID_ARG;
  MapExport d;
  if (gm_status s = map_export(m, MAP_VOXELS, &d)) return s;
  *n = d.keys.size();
  if (!ijk && !counts && !centroids_xyzw) return d.st.overflow ? GM_ERR_CAPACITY : GM_OK;
  if (capacity < d.keys.size()) return GM_ERR_CAPACITY;
  for (size_t i = 0; i < d.keys.size(); ++i) {
    if (ijk) { int x, y, z; map_unpack(d.keys[i], x, y, z); ijk[3 * i] = x; ijk[3 * i + 1] = y; ijk[3 * i + 2] = z; }
    if (counts) counts[i] = d.cnt[i];
    if (centroids_xyzw) {
      const double c = (double)d.cnt[i];
      for (int a = 0; a < 3; ++a) centroids_xyzw[4 * i + a] = (float)((double)d.sums[3 * i + a] / 1048576.0 / c);
      centroids_xyzw[4 * i + 3] = 1.0f;
    }
  }
  return d.st.overflow ? GM_ERR_CAPACITY : GM_OK;
}

gm_status gm_map_save(gm_map* m, const char* path) {
  if (!m || !path) return GM_ERR_INVALID_ARG;
  MapExport d;
  if (gm_status s = map_export(m, MAP_VOXELS, &d)) return s;
  FILE* f = std::fopen(path, "wb");
  if (!f) return GM_ERR_INVALID_ARG;
  const uint32_t magic = 0x314D4D47u /* 'GMM1' */, version = 1;
  const uint64_t V = d.keys.size();
  bool ok = std::fwrite(&magic, 4, 1, f) == 1 && std::fwrite(&version, 4, 1, f) == 1 && std::fwrite(&m->leaf, 8, 1, f) == 1 &&
            std::fwrite(&V, 8, 1, f) == 1;
  if (ok && V) ok = std::fwrite(d.keys.data(), 8, V, f) == V && std::fwrite(d.cnt.data(), 4, V, f) == V && std::fwrite(d.sums.data(), 8, 3 * V, f) == 3 * V;
  ok = (std::fclose(f) == 0) && ok;
  return ok ? GM_OK : GM_ERR_INVALID_ARG;
}

gm_status gm_map_load(const char* path, size_t min_capacity_voxels, gm_map** out) {
  if (!path || !out) return GM_ERR_INVALID_ARG;
  *out = nullptr;
  FILE* f = std::fopen(path, "rb");
  if (!f) return GM_ERR_INVALID_ARG;
  uint32_t magic = 0, version = 0; double leaf = 0; uint64_t V = 0;
  bool ok = std::fread(&magic, 4, 1, f) == 1 && std::fread(&version, 4, 1, f) == 1 && std::fread(&leaf, 8, 1, f) == 1 && std::fread(&V, 8, 1, f) == 1 &&
            magic == 0x314D4D47u && version == 1 && leaf > 0.0 && V < (1ull << 31);
  if (ok) {  // the header is not trusted: V must match what the file actually holds before anything is allocated
    const long here = std::ftell(f);
    ok = here >= 0 && std::fseek(f, 0, SEEK_END) == 0;
    const long end = ok ? std::ftell(f) : -1;
    ok = ok && end >= here && (uint64_t)(end - here) == V * 36ull && std::fseek(f, here, SEEK_SET) == 0;
  }
  std::vector<unsigned long long> k; std::vector<int> c; std::vector<long long> su;
  try {
    if (ok && V) {
      k.resize(V); c.resize(V); su.resize(3 * V);
      ok = std::fread(k.data(), 8, V, f) == V && std::fread(c.data(), 4, V, f) == V && std::fread(su.data(), 8, 3 * V, f) == 3 * V;
    }
  } catch (...) { ok = false; }
  std::fclose(f);
  for (uint64_t i = 0; ok && i < V; ++i) ok = c[i] > 0 && k[i] != MAP_EMPTY && (i == 0 || k[i] > k[i - 1]);  // sorted, unique, real voxels
  if (!ok) return GM_ERR_INVALID_ARG;
  gm_map* m = nullptr;
  gm_status s = gm_map_create(leaf, std::max<size_t>(std::max<size_t>(min_capacity_voxels, (size_t)V), 1), &m);
  if (s != GM_OK) return s;
  if (V) {
    DevBuf<unsigned long long> dk; DevBuf<int> dc; DevBuf<long long> ds;
    cudaError_t e = dk.alloc((size_t)V);
    if (e == cudaSuccess) e = dc.alloc((size_t)V);
    if (e == cudaSuccess) e = ds.alloc(3 * (size_t)V);
    if (e == cudaSuccess) e = cudaMemcpy(dk, k.data(), V * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dc, c.data(), V * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(ds, su.data(), 3 * V * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
      k_map_restore<<<std::min<unsigned long long>((V + 255) / 256, (unsigned long long)m->num_sms * 16), 256>>>(dk, dc, ds, (int)V, nullptr, m->d_keys,
                                                                                                     m->d_cnt, m->d_sums, m->n_slots - 1ull, m->d_st);
      e = cudaDeviceSynchronize();
    }
    if (e != cudaSuccess) { gm_map_destroy(m); return GM_ERR_CUDA; }
  }
  *out = m;
  return GM_OK;
}

double gm_map_leaf(const gm_map* m) { return m ? m->leaf : 0.0; }

gm_status gm_map_evict(gm_map* m, gm_ctx* ctx, gm_map* archive, const float* center3, int32_t half_cells) {
  if (!m || !ctx || !center3 || half_cells < 0 || archive == m) return GM_ERR_INVALID_ARG;
  if (ctx->device != m->device) { ctx->err = "gm_map_evict: context and map on different devices"; return GM_ERR_INVALID_ARG; }
  if (archive && !same_lattice(m, archive)) { ctx->err = "gm_map_evict: archive on another device or with another leaf"; return GM_ERR_INVALID_ARG; }
  long long cell[3];
  if (!map_center_cell(center3, m->inv_leaf, cell)) { ctx->err = "gm_map_evict: centre not finite or outside the key range"; return GM_ERR_INVALID_ARG; }
  GM_CUDA(ensure_evict_buffers(m));
  GM_CUDA(cudaStreamWaitEvent(ctx->stream, m->ev_last, 0));
  if (archive) GM_CUDA(cudaStreamWaitEvent(ctx->stream, archive->ev_last, 0));
  if (gm_status s = map_evict_launch(m, ctx, archive, center3, nullptr, half_cells)) return s;
  GM_CUDA(cudaEventRecord(m->ev_last, ctx->stream));
  if (archive) GM_CUDA(cudaEventRecord(archive->ev_last, ctx->stream));
  return GM_OK;
}

gm_status gm_map_merge(gm_map* dst, const gm_map* src) {
  if (!dst || !src || dst == src || !same_lattice(dst, src)) return GM_ERR_INVALID_ARG;
  MapDeviceScope scope(dst->device, true);
  GM_MAP_CUDA(scope.status);
  k_map_merge<<<map_blocks(src), 256>>>(src->d_keys, src->d_cnt, src->d_sums, src->n_slots, dst->d_keys, dst->d_cnt, dst->d_sums,
                                        dst->n_slots - 1ull, dst->d_st);
  GM_MAP_CUDA(cudaGetLastError());
  MapExport x;
  if (gm_status s = map_export(dst, MAP_STATE, &x)) return s;  // synchronises: the state after the merge
  return x.st.overflow ? GM_ERR_CAPACITY : GM_OK;
}

}  // extern "C"

// ---- scan-to-map registration (gm_register.cuh, k_map_planes in gm_map.cuh) ------------------------------------------
namespace {
inline bool valid_planarity(double r) { return r > 0.0 && r <= 1.0; }

// gm_register_map's argument rules (gm_odometry_create checks its icp by them too)
bool valid_regmap_args(const gm_icp_params* p, double max_planarity) { return valid_icp_args(p) && valid_planarity(max_planarity); }

// The buffers a scan-to-map registration of `source` uses (allocated by the first call).
gm_status regmap_buffers(gm_ctx* source, gm_map* map) {
  gm_ctx* ctx = source;
  if (gm_status s = ensure_reg_buffers(source)) return s;
  if (!source->d_reg_key.count) GM_CUDA(source->d_reg_key.alloc(source->cap));
  GM_CUDA(ensure_plane_tables(map));
  return GM_OK;
}

// The launches of gm_register_map on the source stream, after its checks and the wait for the map's last operation:
// the map's planes, begin() (the kernel that sets the registration's start), then max_iterations x k_regmap_iter.
// Shared by gm_register_map and gm_odometry_step so that a step registers exactly as the call does.
template <class Begin>
gm_status regmap_launch(gm_ctx* source, gm_map* map, const gm_icp_params* p, double max_planarity, Begin begin) {
  gm_ctx* ctx = source;  // GM_CUDA / GM_LAUNCH report on the source
  ctx->stages &= ~(1u << REGISTRATION);
  const unsigned long long mask = map->n_slots - 1ull;
  GM_CUDA(cudaMemsetAsync(map->d_plane_box, 0x7F, 8 * sizeof(int), source->stream));
  GM_LAUNCH(ctx, k_map_planes, map_blocks(map), 256, map->d_keys, map->d_cnt, map->d_sums, mask, max_planarity, map->d_plane_cent,
            map->d_plane_nrm, map->d_plane_box);
  begin();
  int blocks;
  const RegParams rp = icp_setup(source, p, &blocks);
  for (int it = 0; it < p->max_iterations; ++it)
    GM_LAUNCH(ctx, k_regmap_iter, blocks, REG_BLOCK, source->d_centroid, &source->d_st->vox.n_voxels, map->d_keys, map->d_plane_cent,
              map->d_plane_nrm, map->d_plane_box, mask, map->inv_leaf, map->leaf, rp, source->d_reg_state, source->d_reg_part, source->d_reg_ticket,
              source->d_reg_key, source->d_reg_res);
  GM_CHECK_LAUNCHES(ctx);
  source->reg_target = 1;
  mark(source, REGISTRATION);
  return GM_OK;
}
}  // namespace

extern "C" {

gm_status gm_register_map(gm_ctx* source, gm_map* map, const gm_icp_params* p, double max_planarity) {
  if (!source || !map || !p) return GM_ERR_INVALID_ARG;
  gm_ctx* ctx = source;  // GM_CUDA / GM_LAUNCH report on the source
  if (source->device != map->device) { ctx->err = "gm_register_map: source and map on different devices"; return GM_ERR_INVALID_ARG; }
  if (!valid_regmap_args(p, max_planarity)) return GM_ERR_INVALID_ARG;
  if (gm_status s = require(source, VOXEL)) return s;
  if (gm_status s = regmap_buffers(source, map)) return s;
  GM_CUDA(cudaStreamWaitEvent(source->stream, map->ev_last, 0));
  Pose34 init;
  std::memcpy(init.r, p->init_pose34, sizeof(init.r));
  gm_status s = regmap_launch(source, map, p, max_planarity, [&] {
    GM_LAUNCH(ctx, k_reg_begin, 1, 32, source->d_reg_state, init, &source->d_st->vox.n_voxels);
  });
  if (s != GM_OK) return s;
  GM_CUDA(cudaEventRecord(map->ev_last, source->stream));
  return GM_OK;
}

gm_status gm_download_map_correspondences(gm_ctx* ctx, int32_t* ijk, float* residual, size_t capacity_points) {
  if (!ctx || !ijk) return GM_ERR_INVALID_ARG;
  std::vector<unsigned long long> keys;
  if (gm_status s = download_reg_points(ctx, 1, ctx->d_reg_key.p, &keys, residual, capacity_points)) return s;
  for (size_t i = 0; i < keys.size(); ++i) {
    int x = INT32_MIN, y = INT32_MIN, z = INT32_MIN;
    if (keys[i] != MAP_EMPTY) map_unpack(keys[i], x, y, z);
    ijk[3 * i] = x; ijk[3 * i + 1] = y; ijk[3 * i + 2] = z;
  }
  return GM_OK;
}

gm_status gm_map_download_planes(gm_map* m, double max_planarity, float* normals_xyzw, size_t capacity, size_t* n) {
  if (!m || !n || !valid_planarity(max_planarity)) return GM_ERR_INVALID_ARG;
  MapExport x;
  if (gm_status s = map_export(m, normals_xyzw ? MAP_PLANES : MAP_STATE, &x, max_planarity, capacity)) return s;
  *n = (size_t)std::max(x.st.n_voxels, 0);
  if (normals_xyzw && capacity < *n) return GM_ERR_CAPACITY;
  for (size_t i = 0; i < x.nrm.size(); ++i) std::memcpy(normals_xyzw + 4 * i, &x.nrm[i], sizeof(float4));
  return x.st.overflow ? GM_ERR_CAPACITY : GM_OK;  // as gm_map_download: an insert found the table full
}

}  // extern "C"

// ---- map odometry (gm_odometry.cuh) -----------------------------------------------------------------------------------
static_assert(sizeof(gm_odometry_params) == 112 && sizeof(gm_odometry_record) == 136 && sizeof(OdomRecord) == sizeof(gm_odometry_record) &&
              offsetof(OdomRecord, accepted) == offsetof(gm_odometry_record, accepted) &&
              offsetof(OdomRecord, fitness) == offsetof(gm_odometry_record, fitness), "odometry layouts");

struct gm_odometry {
  gm_map* map = nullptr;
  gm_odometry_params p{};
  int32_t steps = 0;                 // steps issued
  DevBuf<OdomRecord> d_rec;          // the trajectory, max_steps records
  DevBuf<OdomInsert> d_ins;          // pose and flag of the current step's insert
  cudaStream_t stream = nullptr;     // the trajectory download
  int32_t window = 0;                // gm_odometry_set_window: half_cells of the local map's window, 0 = off
  gm_map* archive = nullptr;         // where the window evicts to (null: dropped)
  ~gm_odometry() { if (stream) cudaStreamDestroy(stream); }
};

extern "C" {

void gm_odometry_params_default(gm_odometry_params* p) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  gm_icp_params_default(&p->icp);
  p->max_planarity = 0.1;
  p->min_fitness = 0.5;
  p->register_first = 0;
  p->max_steps = 4096;
}

gm_status gm_odometry_create(gm_map* map, const gm_odometry_params* p, gm_odometry** out) {
  if (!out) return GM_ERR_INVALID_ARG;
  *out = nullptr;
  if (!map || !p || !valid_regmap_args(&p->icp, p->max_planarity) || !(p->min_fitness >= 0.0 && p->min_fitness <= 1.0) ||
      (p->register_first != 0 && p->register_first != 1) || p->max_steps < 1)
    return GM_ERR_INVALID_ARG;
  MapDeviceScope scope(map->device, false);
  GM_MAP_CUDA(scope.status);
  gm_odometry* o = new gm_odometry();
  o->map = map;
  o->p = *p;
  cudaError_t e = o->d_rec.alloc((size_t)p->max_steps);
  if (e == cudaSuccess) e = o->d_ins.alloc(1);
  if (e == cudaSuccess) e = cudaMemset(o->d_rec, 0, (size_t)p->max_steps * sizeof(OdomRecord));
  if (e == cudaSuccess) e = cudaMemset(o->d_ins, 0, sizeof(OdomInsert));
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&o->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { delete o; return GM_ERR_CUDA; }
  *out = o;
  return GM_OK;
}

void gm_odometry_destroy(gm_odometry* odo) {
  if (!odo) return;
  MapDeviceScope scope(odo->map->device, true);  // as gm_map_destroy: the steps in flight read the trajectory
  delete odo;
}

gm_status gm_odometry_step(gm_odometry* odo, gm_ctx* ctx, const float* delta34) {
  if (!odo || !ctx) return GM_ERR_INVALID_ARG;
  gm_map* map = odo->map;
  const int k = odo->steps;
  if (k >= odo->p.max_steps) return GM_ERR_CAPACITY;
  if (delta34 && (k == 0 || !finite_pose(delta34))) return GM_ERR_INVALID_ARG;
  if (ctx->device != map->device) { ctx->err = "gm_odometry_step: context and map on different devices"; return GM_ERR_INVALID_ARG; }
  if (gm_status s = require(ctx, COMPACTED, VOXEL)) return s;
  const bool registered = k > 0 || odo->p.register_first;
  if (registered)
    if (gm_status s = regmap_buffers(ctx, map)) return s;
  gm_map* archive = odo->window > 0 ? odo->archive : nullptr;
  if (odo->window > 0) GM_CUDA(ensure_evict_buffers(map));
  GM_CUDA(cudaStreamWaitEvent(ctx->stream, map->ev_last, 0));
  if (archive) GM_CUDA(cudaStreamWaitEvent(ctx->stream, archive->ev_last, 0));
  Pose34 init{}, delta{};
  int mode = ODOM_INIT;
  if (k == 0) {
    std::memcpy(init.r, odo->p.icp.init_pose34, sizeof(init.r));
  } else if (delta34 || k == 1) {  // constant velocity at k = 1: delta = identity
    mode = ODOM_DELTA;
    if (delta34) std::memcpy(delta.r, delta34, sizeof(delta.r));
    else delta.r[0] = delta.r[5] = delta.r[10] = 1.0f;
  } else {
    mode = ODOM_VELOCITY;
  }
  RegState* st = registered ? (RegState*)ctx->d_reg_state : nullptr;
  auto begin = [&] { GM_LAUNCH(ctx, k_odom_begin, 1, 32, odo->d_rec, k, mode, init, delta, st, &ctx->d_st->vox.n_voxels); };
  if (registered) {
    if (gm_status s = regmap_launch(ctx, map, &odo->p.icp, odo->p.max_planarity, begin)) return s;
  } else {
    ctx->stages &= ~(1u << REGISTRATION);
    begin();
  }
  GM_LAUNCH(ctx, k_odom_gate, 1, 32, odo->d_rec, k, st, odo->p.min_fitness, odo->d_ins);
  // gm_map_insert's grid, at least one block: the kernel reads the point count on the device
  const int blocks = std::max(1, std::min(div_up((long long)ctx->n_input, 256), ctx->num_sms * 16));
  GM_LAUNCH(ctx, k_map_insert_gated, blocks, 256, ctx->d_cloud_c, &ctx->d_st->n_valid, &odo->d_ins->pose, &odo->d_ins->accept, map->inv_leaf,
            map->d_keys, map->d_cnt, map->d_sums, map->n_slots - 1ull, map->d_st);
  GM_CHECK_LAUNCHES(ctx);
  // the window: gm_map_evict's launches, centred on the translation of the pose record k holds
  if (odo->window > 0)
    if (gm_status s = map_evict_launch(map, ctx, archive, nullptr, odo->d_rec[k].pose34, odo->window)) return s;
  GM_CUDA(cudaEventRecord(map->ev_last, ctx->stream));
  if (archive) GM_CUDA(cudaEventRecord(archive->ev_last, ctx->stream));
  odo->steps = k + 1;
  return GM_OK;
}

gm_status gm_odometry_deskew(gm_odometry* odo, gm_ctx* ctx, double t_ref, double period) {
  if (!odo || !ctx) return GM_ERR_INVALID_ARG;
  gm_map* map = odo->map;
  const int k = odo->steps;
  if (k >= odo->p.max_steps) return GM_ERR_CAPACITY;
  if (ctx->device != map->device) { ctx->err = "gm_odometry_deskew: context and map on different devices"; return GM_ERR_INVALID_ARG; }
  if (gm_status s = deskew_check(ctx, t_ref, period)) return s;
  GM_CUDA(cudaStreamWaitEvent(ctx->stream, map->ev_last, 0));  // step k - 1 has written the records k_odom_delta reads
  GM_LAUNCH(ctx, k_odom_delta, 1, 32, odo->d_rec, k, ctx->d_delta);
  return deskew_launch(ctx, Pose34{}, ctx->d_delta, t_ref, period);
}

gm_status gm_odometry_set_window(gm_odometry* odo, int32_t half_cells, gm_map* archive) {
  if (!odo || half_cells < 0) return GM_ERR_INVALID_ARG;
  if (archive && (archive == odo->map || !same_lattice(odo->map, archive))) return GM_ERR_INVALID_ARG;
  odo->window = half_cells;
  odo->archive = archive;
  return GM_OK;
}

int32_t gm_odometry_steps(const gm_odometry* odo) { return odo ? odo->steps : 0; }

gm_status gm_odometry_get(gm_odometry* odo, gm_odometry_record* out, int32_t capacity, int32_t* n) {
  if (!odo || !n) return GM_ERR_INVALID_ARG;
  *n = odo->steps;
  if (!out) return GM_OK;
  if (capacity < odo->steps) return GM_ERR_CAPACITY;
  cudaError_t e = cudaStreamWaitEvent(odo->stream, odo->map->ev_last, 0);  // after every step issued so far
  if (e == cudaSuccess && odo->steps > 0)
    e = cudaMemcpyAsync(out, odo->d_rec, (size_t)odo->steps * sizeof(OdomRecord), cudaMemcpyDeviceToHost, odo->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(odo->stream);
  return e == cudaSuccess ? GM_OK : GM_ERR_CUDA;
}

}  // extern "C"
