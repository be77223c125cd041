// gm_stages.cuh — kernels of the reference-pinned stages a1..a5 (SURVEY.md section 8a).
// Compiled with -fmad=false: a*b+c is never contracted, so plain expressions reproduce the
// unfused PCL/FLANN arithmetic that integer decisions depend on (neighbour sets, voxel keys);
// fused multiply-adds appear only where fmaf() is written explicitly.
#pragma once
#include "gm_device.cuh"
#include <math_constants.h>

namespace gm {

// Device-resident per-scan state: sizes flow from stage to stage without host round trips.
// State of one VoxelGrid run (the compacted cloud, or the residual cloud of the compression stage).
struct VoxState {
  int n, n_voxels, overflow, pad_;
  int bbox_min[3], bbox_max[3];  // ordered-int encoded floats
  int min_b[3], div_b[3], mul[3];
  float v_inv;
};
__device__ __forceinline__ void d_vox_reset(VoxState* v) {
  v->n = 0; v->n_voxels = 0; v->overflow = 0; v->pad_ = 0; v->v_inv = 0.f;
  for (int a = 0; a < 3; ++a) {
    v->bbox_min[a] = float_to_ordered(CUDART_INF_F);
    v->bbox_max[a] = float_to_ordered(-CUDART_INF_F);
    v->min_b[a] = 0; v->div_b[a] = 0; v->mul[a] = 0;
  }
}

struct DevState {
  const float4* scan;   // the input scan of this context (set by k_begin_scan; read by k_crop)
  int n_input, n_crop, n_valid, n_cells, nn_oor, error;
  int n_sorted_finite;  // cropped points with finite coordinates (sorted before the NaN tail)
  int tab_cells;        // occupied cells currently recorded in the block table (cleared by the next build)
  unsigned long long n_candidates;  // distance tests of the radius search (sum over points of their stencil population)
  unsigned long long n_neighbors;   // of which within the radius
  VoxState vox;         // VoxelGrid of the compacted cloud (vox.n mirrors n_valid)
};

struct GridSpec {
  float origin[3];   // lower corner of the grid box (default: -bound on every axis)
  float inv_cell;    // 1/cell
  float cell;
  int dim[3];        // cells per axis (points outside the box are clamped into the border cells)
  int bits[3];       // bits of the BLOCK coordinate per axis (blocks are 4x4x4 cells)
  int bmin;          // min(bits): the low bmin bits of the three block coordinates are Morton-interleaved
  int key_bits;      // bits of a cell key (bits[0]+bits[1]+bits[2] + 6); the block table has 1 << (key_bits - 6) entries
  unsigned sentinel; // key of non-finite points: all ones in key_bits, never a real cell
};

// Cell key = code of the 4x4x4-cell BLOCK the cell lies in, then the cell's row-major position inside
// the block (x fastest).  Block code = Morton interleave of the low bmin bits of the block coordinates
// with the remaining high bits of the longer axes stacked on top (a plain Morton code when the grid is
// a cube).  Sorting by it keeps two properties at once:
//   * cells adjacent in x inside a block are adjacent keys, so the 3-cell x-neighbourhood of a cell
//     is one contiguous run of the sorted cloud, or two when it crosses a block face;
//   * consecutive points are spatially compact in all three axes (a 512-point tile of the C1 scan is
//     a ~0.3 m blob instead of a 6 m long row), which is what makes the tile-culled inlier counting
//     (gm_ransac.cuh) effective.
constexpr int GRID_RUNS = 18;  // per occupied cell: 9 (dy,dz) rows x up to 2 x-segments

// Dense table over the blocks (index = block code): which of the 64 cells of the block are
// occupied and the rank of its first occupied cell in the sorted cell list.  The rank of any cell is
// then first + popc(mask below its local code): neighbour lookups need no search at all.  Only the
// entries of occupied blocks are ever written, and the next build clears exactly those (O(cells)).
struct __align__(16) BlockEntry { unsigned long long mask; int first; int pad_; };

__host__ __device__ __forceinline__ unsigned gm_spread3(unsigned x) {  // 10 bits -> every third bit
  x &= 0x3FFu;
  x = (x | (x << 16)) & 0x030000FFu;
  x = (x | (x << 8)) & 0x0300F00Fu;
  x = (x | (x << 4)) & 0x030C30C3u;
  x = (x | (x << 2)) & 0x09249249u;
  return x;
}
__host__ __device__ __forceinline__ unsigned gm_compact3(unsigned x) {
  x &= 0x09249249u;
  x = (x | (x >> 2)) & 0x030C30C3u;
  x = (x | (x >> 4)) & 0x0300F00Fu;
  x = (x | (x >> 8)) & 0x030000FFu;
  x = (x | (x >> 16)) & 0x3FFu;
  return x;
}
__host__ __device__ __forceinline__ unsigned gm_cell_key(const GridSpec& g, int cx, int cy, int cz) {
  const unsigned bx = (unsigned)cx >> 2, by = (unsigned)cy >> 2, bz = (unsigned)cz >> 2;
  const unsigned lowmask = (1u << g.bmin) - 1u;
  const unsigned m = gm_spread3(bx & lowmask) | (gm_spread3(by & lowmask) << 1) | (gm_spread3(bz & lowmask) << 2);
  const int hx = g.bits[0] - g.bmin, hy = g.bits[1] - g.bmin;
  const unsigned hi = ((bz >> g.bmin) << (hx + hy)) | ((by >> g.bmin) << hx) | (bx >> g.bmin);
  const unsigned code = (hi << (3 * g.bmin)) | m;
  return (code << 6) | (((unsigned)cz & 3u) << 4) | (((unsigned)cy & 3u) << 2) | ((unsigned)cx & 3u);
}
__host__ __device__ __forceinline__ void gm_cell_coords(const GridSpec& g, unsigned key, int& cx, int& cy, int& cz) {
  const unsigned code = key >> 6;
  const unsigned m = code & ((1u << (3 * g.bmin)) - 1u), hi = code >> (3 * g.bmin);
  const int hx = g.bits[0] - g.bmin, hy = g.bits[1] - g.bmin;
  const unsigned bx = gm_compact3(m) | ((hi & ((1u << hx) - 1u)) << g.bmin);
  const unsigned by = gm_compact3(m >> 1) | (((hi >> hx) & ((1u << hy) - 1u)) << g.bmin);
  const unsigned bz = gm_compact3(m >> 2) | ((hi >> (hx + hy)) << g.bmin);
  cx = (int)((bx << 2) | (key & 3u));
  cy = (int)((by << 2) | ((key >> 2) & 3u));
  cz = (int)((bz << 2) | ((key >> 4) & 3u));
}
__device__ __forceinline__ void gm_cell_of(const GridSpec& g, float x, float y, float z, int& cx, int& cy, int& cz) {
  cx = min(max((int)floorf((x - g.origin[0]) * g.inv_cell), 0), g.dim[0] - 1);
  cy = min(max((int)floorf((y - g.origin[1]) * g.inv_cell), 0), g.dim[1] - 1);
  cz = min(max((int)floorf((z - g.origin[2]) * g.inv_cell), 0), g.dim[2] - 1);
}

// Points of a map slab that this context does not own (halo points given to it for the neighbour
// search only): dropped together with the NaN normals.  axis < 0: everything is owned.
struct OwnedRange { int axis; float lo, hi; };
__device__ __forceinline__ bool d_owned(const OwnedRange& o, const float4 p) {
  if (o.axis < 0) return true;
  const float v = (o.axis == 0) ? p.x : ((o.axis == 1) ? p.y : p.z);
  return v >= o.lo && v < o.hi;
}

// Coordinate sums of a voxel are kept in 2^-20 m fixed point (x * 2^20 is exact in float, llrint rounds it to
// an integer): integer addition is associative, so a centroid does not depend on the order in which its
// members arrive -- bitwise reproducible with atomics, across map slabs, and in the aggregated map.
// centroid = float(double(sum) / 2^20 / count).  (pcl::VoxelGrid accumulates in float in the unspecified
// order of an unstable std::sort; this form is within 1e-6 m of any such order.)
constexpr float GM_FX20 = 1048576.0f;
__device__ __forceinline__ long long d_fx20(float v) { return __float2ll_rn(v * GM_FX20); }
__device__ __forceinline__ float d_centroid_of(long long sum, int count) { return (float)((double)sum / 1048576.0 / (double)count); }

constexpr int CP_BLOCK = 256;
constexpr int CP_IPT = 4;                      // items per thread where each item is register heavy
constexpr int CP_TILE = CP_BLOCK * CP_IPT;
constexpr int CPL_IPT = 8;                     // light items: fewer, larger tiles -> shorter look-back walks
constexpr int CPL_TILE = CP_BLOCK * CPL_IPT;

__device__ __forceinline__ bool finite3(float x, float y, float z) { return isfinite(x) && isfinite(y) && isfinite(z); }

// ---------------------------------------------------------------------------------------------
__global__ void k_begin_scan(DevState* st, int n_input, const float4* scan) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    st->scan = scan;
    st->n_input = n_input; st->n_crop = 0; st->n_valid = 0; st->n_cells = 0;
    st->nn_oor = 0; st->error = 0; st->n_sorted_finite = 0;  // tab_cells survives: it describes the block table
    st->n_candidates = 0ull; st->n_neighbors = 0ull;
    d_vox_reset(&st->vox);
  }
}

// PointCloud2 decode: gather the float32 x,y,z fields (byte offsets, arbitrary point_step) into PointXYZ; TIMED also
// gathers the float32 field at byte offset ot (the point's time, gm_upload_pointcloud2_timed) into times.  The untimed
// instantiation ignores the two trailing arguments.
template <bool TIMED>
__global__ void k_decode_pointcloud2(const unsigned char* __restrict__ raw, int n, int point_step, int ox, int oy, int oz,
                                     float4* __restrict__ out, int ot, float* __restrict__ times) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned char* p = raw + (size_t)i * point_step;
  constexpr int F = TIMED ? 4 : 3;
  float v[F];
  int off[F] = {ox, oy, oz};
  int align = point_step | ox | oy | oz;
  if constexpr (TIMED) { off[3] = ot; align |= ot; }
  if ((align & 3) == 0) {  // aligned records (the usual case: x,y,z,(intensity,ring) float32 fields)
    const float* f = reinterpret_cast<const float*>(p);
    out[i] = make_float4(f[ox >> 2], f[oy >> 2], f[oz >> 2], 1.0f);
    if constexpr (TIMED) times[i] = f[ot >> 2];
    return;
  }
#pragma unroll
  for (int k = 0; k < F; ++k) {  // byte-wise: fields need not be 4-byte aligned inside the record
    unsigned u = (unsigned)p[off[k]] | ((unsigned)p[off[k] + 1] << 8) | ((unsigned)p[off[k] + 2] << 16) | ((unsigned)p[off[k] + 3] << 24);
    v[k] = __uint_as_float(u);
  }
  out[i] = make_float4(v[0], v[1], v[2], 1.0f);
  if constexpr (TIMED) times[i] = v[3];
}

__global__ void k_set_w_one(float4* p, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i].w = 1.0f;
}

// a1 chopCloud / pcl::CropBox (src/tunnel_processing.cpp:39-49, SURVEY A.1): stable compaction of
// the points with every coordinate in [lo,hi]; NaN handling per is_dense.
__global__ void __launch_bounds__(CP_BLOCK, 4)
k_crop(const DevState* __restrict__ scan, float lo, float hi, int is_dense, float4* __restrict__ out,
       unsigned long long* state, TileCtl* ctl, DevState* st) {
  __shared__ CompactSmem<CP_BLOCK, CPL_IPT> sm;
  unsigned epoch;
  const int tile = tile_begin(ctl, epoch), base = tile * CPL_TILE;
  const int n = scan->n_input;                      // written by k_begin_scan: the launch itself carries no per-scan argument
  const float4* __restrict__ in = scan->scan;
  if (base >= n) { tile_end(ctl); return; }
  float4 p[CPL_IPT];
  bool f[CPL_IPT];
#pragma unroll
  for (int j = 0; j < CPL_IPT; ++j) {
    int i = base + j * CP_BLOCK + threadIdx.x;
    f[j] = false;
    if (i < n) {
      p[j] = in[i];
      bool drop = (p[j].x < lo) || (p[j].y < lo) || (p[j].z < lo) || (p[j].x > hi) || (p[j].y > hi) || (p[j].z > hi);
      if (!is_dense && !finite3(p[j].x, p[j].y, p[j].z)) drop = true;
      f[j] = !drop;
    }
  }
  unsigned ranks[CPL_IPT], total;
  tile_compact_ranks<CP_BLOCK, CPL_IPT>(f, ranks, total, state, epoch, tile, &st->error, sm);
#pragma unroll
  for (int j = 0; j < CPL_IPT; ++j)
    if (f[j]) out[ranks[j]] = p[j];
  if (base + CPL_TILE >= n && threadIdx.x == 0) st->n_crop = (int)total;
  tile_end(ctl);
}

// Neighbour-grid cell key of every cropped point (sentinel ncells for non-finite points, which
// are never anyone's neighbour).
__global__ void k_cell_keys(const float4* __restrict__ pts, const int* __restrict__ n_ptr, GridSpec g,
                            unsigned* __restrict__ keys, unsigned* __restrict__ idx) {
  const int n = *n_ptr;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float4 p = pts[i];
    unsigned key = g.sentinel;
    if (finite3(p.x, p.y, p.z)) {
      int cx, cy, cz;
      gm_cell_of(g, p.x, p.y, p.z, cx, cy, cz);
      key = gm_cell_key(g, cx, cy, cz);
    }
    keys[i] = key;
    idx[i] = (unsigned)i;
  }
}

// After the sort: gather points into cell order (w := original index), number the occupied cells
// and record each cell's key and first sorted position (stable compaction of the "head" flags).
__global__ void __launch_bounds__(CP_BLOCK)
k_cell_heads(const unsigned* __restrict__ skeys, const unsigned* __restrict__ sidx, const float4* __restrict__ pts,
             const int* __restrict__ n_ptr, unsigned sentinel, float4* __restrict__ sorted_pts, int* __restrict__ cell_id,
             unsigned* __restrict__ ucell_key, int* __restrict__ ucell_start, BlockEntry* __restrict__ tab,
             unsigned long long* state, TileCtl* ctl, DevState* st) {
  __shared__ CompactSmem<CP_BLOCK, CPL_IPT> sm;
  const int n = *n_ptr;
  unsigned epoch;
  const int tile = tile_begin(ctl, epoch), base = tile * CPL_TILE;
  if (base >= n) { tile_end(ctl); return; }
  bool f[CPL_IPT], bh[CPL_IPT];
  unsigned key[CPL_IPT];
  int nfinite_local = 0;
#pragma unroll
  for (int j = 0; j < CPL_IPT; ++j) {
    int i = base + j * CP_BLOCK + threadIdx.x;
    f[j] = false;
    key[j] = 0;
    if (i < n) {
      key[j] = skeys[i];
      unsigned prev = (i > 0) ? skeys[i - 1] : 0xFFFFFFFFu;
      f[j] = (i == 0) || (key[j] != prev);
      bh[j] = (i == 0) || ((key[j] >> 6) != (prev >> 6));  // first cell of its block
      unsigned src = sidx[i];
      float4 p = pts[src];
      p.w = __int_as_float((int)src);
      sorted_pts[i] = p;
      if (key[j] != sentinel) {
        // last finite position + 1 == number of finite points (sentinel keys sort last)
        if (i + 1 == n || skeys[i + 1] == sentinel) nfinite_local = i + 1;
      }
    }
  }
  if (nfinite_local) st->n_sorted_finite = nfinite_local;
  unsigned ranks[CPL_IPT], total;
  tile_compact_ranks<CP_BLOCK, CPL_IPT>(f, ranks, total, state, epoch, tile, &st->error, sm);
#pragma unroll
  for (int j = 0; j < CPL_IPT; ++j) {
    int i = base + j * CP_BLOCK + threadIdx.x;
    if (i < n) {
      int id = f[j] ? (int)ranks[j] : (int)ranks[j] - 1;
      cell_id[i] = id;
      if (f[j]) {
        ucell_key[id] = key[j]; ucell_start[id] = i;
        if (key[j] != sentinel) {
          BlockEntry* e = tab + (key[j] >> 6);
          atomicOr(&e->mask, 1ull << (key[j] & 63u));
          if (bh[j]) e->first = id;
        }
      }
    }
  }
  if (base + CPL_TILE >= n && threadIdx.x == 0) { st->n_cells = (int)total; st->tab_cells = (int)total; }
  tile_end(ctl);
}

// Clear the block-table entries of the previous build (its sorted cell list is still in ucell_key).
__global__ void k_clear_blocks(const unsigned* __restrict__ ucell_key, DevState* st, unsigned sentinel, BlockEntry* __restrict__ tab) {
  const int U = st->tab_cells;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < U; j += gridDim.x * blockDim.x) {
    const unsigned key = ucell_key[j];
    if (key != sentinel) { BlockEntry z; z.mask = 0ull; z.first = 0; z.pad_ = 0; tab[key >> 6] = z; }
  }
}

__device__ __forceinline__ int lower_bound_u32(const unsigned* __restrict__ a, int n, unsigned key) {
  int lo = 0, hi = n;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// Sorted-position range [start,end) of the cells x0..x1 of row (cy,cz), all inside ONE 4-cell x-block
// (consecutive local codes): two popcounts on the block's occupancy mask, no search.
__device__ __forceinline__ int2 cell_segment(const GridSpec& g, const BlockEntry* __restrict__ tab, const int* __restrict__ ucell_start,
                                             int U, int n_finite, int x0, int x1, int cy, int cz) {
  const unsigned key = gm_cell_key(g, x0, cy, cz);
  const BlockEntry e = tab[key >> 6];
  const unsigned c0 = key & 63u, c1 = c0 + (unsigned)(x1 - x0);
  const int a = e.first + __popcll(e.mask & ((1ull << c0) - 1ull));
  const int b = e.first + __popcll(e.mask & ((2ull << c1) - 1ull));
  if (a == b) return make_int2(0, 0);
  const int s = min(ucell_start[a], n_finite);
  const int t = (b < U) ? min(ucell_start[b], n_finite) : n_finite;
  return make_int2(s, t);
}

// For every occupied cell: the non-empty sorted-position runs that cover its 27-cell neighbourhood
// (per (dy,dz) row the part of x-1..x+1 in the first x-block it touches and the part in the next one),
// runs that happen to be adjacent in the sorted cloud merged; at most GRID_RUNS of them.
__global__ void k_cell_runs(const unsigned* __restrict__ ucell_key, const int* __restrict__ ucell_start, const BlockEntry* __restrict__ tab,
                            const DevState* __restrict__ st, GridSpec g, int2* __restrict__ runs, int2* __restrict__ cell_info) {
  const int U = st->n_cells, nf = st->n_sorted_finite;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < U; j += gridDim.x * blockDim.x) {
    const unsigned key = ucell_key[j];
    int2* out = runs + (size_t)j * GRID_RUNS;
    int m = 0;
    int2 cur = make_int2(0, 0);
    if (key != g.sentinel) {
      int cx, cy0, cz0;
      gm_cell_coords(g, key, cx, cy0, cz0);
      const int x0 = max(cx - 1, 0), x1 = min(cx + 1, g.dim[0] - 1);
      const int split = x0 | 3;  // last cell of x0's block
      // all 18 segment lookups first (independent loads in flight together), then the in-order merge
      int2 seg[GRID_RUNS];
#pragma unroll
      for (int k = 0; k < 9; ++k) {
        const int cy = cy0 + (k % 3) - 1, cz = cz0 + (k / 3) - 1;
        const bool in = cy >= 0 && cz >= 0 && cy < g.dim[1] && cz < g.dim[2];
        seg[2 * k] = in ? cell_segment(g, tab, ucell_start, U, nf, x0, min(x1, split), cy, cz) : make_int2(0, 0);
        seg[2 * k + 1] = (in && x1 > split) ? cell_segment(g, tab, ucell_start, U, nf, split + 1, x1, cy, cz) : make_int2(0, 0);
      }
#pragma unroll
      for (int q = 0; q < GRID_RUNS; ++q) {
        const int2 r = seg[q];
        if (r.y <= r.x) continue;
        if (cur.y == r.x && cur.y > cur.x) { cur.y = r.y; continue; }  // contiguous with the pending run
        if (cur.y > cur.x) out[m++] = cur;
        cur = r;
      }
      if (cur.y > cur.x) out[m++] = cur;
    }
    int total = 0;
    for (int i = 0; i < m; ++i) total += out[i].y - out[i].x;
    cell_info[j] = make_int2(m, total);  // number of runs, number of candidates
  }
}

// ---- libm-independent atan2 / sin / cos for pcl::computeRoots ---------------------------------------
// pcl::computeRoots calls std::atan2 / std::cos / std::sin on floats; their last bit depends on the libm.
// Here they are evaluated in double with only + - * / sqrt in a fixed order (no contraction: -fmad=false) and
// rounded to float once: accurate to ~1e-16 before rounding, hence the correctly rounded float value, on any
// IEEE-754 machine.  The CPU oracle evaluates the same operation sequence, so given bit-identical covariance
// matrices the normals are bit-identical (gm_set_normals_mode(1) provides that accumulation order).
__device__ __forceinline__ double d_atan_unit(double t) {  // t in [0,1]
  const double t1 = t / (1.0 + sqrt(1.0 + t * t));
  const double t2 = t1 / (1.0 + sqrt(1.0 + t1 * t1));
  const double z2 = t2 * t2;
  double p = 1.0 / 27.0;
  p = p * z2 - 1.0 / 25.0; p = p * z2 + 1.0 / 23.0; p = p * z2 - 1.0 / 21.0; p = p * z2 + 1.0 / 19.0;
  p = p * z2 - 1.0 / 17.0; p = p * z2 + 1.0 / 15.0; p = p * z2 - 1.0 / 13.0; p = p * z2 + 1.0 / 11.0;
  p = p * z2 - 1.0 / 9.0;  p = p * z2 + 1.0 / 7.0;  p = p * z2 - 1.0 / 5.0;  p = p * z2 + 1.0 / 3.0;
  p = 1.0 - p * z2;
  return 4.0 * (t2 * p);
}
__device__ __forceinline__ float d_atan2f_pos(float yf, float xf) {  // y >= +0
  const double PI = 3.14159265358979323846, HALF_PI = 1.57079632679489661923;
  if (isnan(yf) || isnan(xf)) return CUDART_NAN_F;
  const double y = yf, x = fabs((double)xf);
  const bool neg = signbit(xf);
  double a;
  if (y == 0.0 && x == 0.0) a = 0.0;
  else if (x >= y) a = d_atan_unit(y / x);
  else a = HALF_PI - d_atan_unit(x / y);
  if (neg) a = PI - a;
  return (float)a;
}
__device__ __forceinline__ float d_sinf_small(float xf) {  // x in [0, pi/3]
  const double x = xf, x2 = x * x;
  double p = -1.0 / 25852016738884976640000.0;
  p = p * x2 + 1.0 / 51090942171709440000.0;
  p = p * x2 - 1.0 / 121645100408832000.0;
  p = p * x2 + 1.0 / 355687428096000.0;
  p = p * x2 - 1.0 / 1307674368000.0;
  p = p * x2 + 1.0 / 6227020800.0;
  p = p * x2 - 1.0 / 39916800.0;
  p = p * x2 + 1.0 / 362880.0;
  p = p * x2 - 1.0 / 5040.0;
  p = p * x2 + 1.0 / 120.0;
  p = p * x2 - 1.0 / 6.0;
  p = p * x2 + 1.0;
  return (float)(x * p);
}
__device__ __forceinline__ float d_cosf_small(float xf) {
  const double x = xf, x2 = x * x;
  double p = 1.0 / 620448401733239439360000.0;
  p = p * x2 - 1.0 / 1124000727777607680000.0;
  p = p * x2 + 1.0 / 2432902008176640000.0;
  p = p * x2 - 1.0 / 6402373705728000.0;
  p = p * x2 + 1.0 / 20922789888000.0;
  p = p * x2 - 1.0 / 87178291200.0;
  p = p * x2 + 1.0 / 479001600.0;
  p = p * x2 - 1.0 / 3628800.0;
  p = p * x2 + 1.0 / 40320.0;
  p = p * x2 - 1.0 / 720.0;
  p = p * x2 + 1.0 / 24.0;
  p = p * x2 - 1.0 / 2.0;
  p = p * x2 + 1.0;
  return (float)p;
}

// ---- pcl::eigen33 smallest eigenpair, float (common/impl/eigen.hpp; SURVEY A.4) -------------
__device__ __forceinline__ void d_compute_roots2(float b, float c, float roots[3]) {
  roots[0] = 0.0f;
  float d = b * b - 4.0f * c;
  if (d < 0.0f) d = 0.0f;
  float sd = sqrtf(d);
  roots[2] = 0.5f * (b + sd);
  roots[1] = 0.5f * (b - sd);
}

__device__ __forceinline__ void d_swapf(float& a, float& b) { float t = a; a = b; b = t; }

__device__ void d_compute_roots(float m00, float m01, float m02, float m11, float m12, float m22, float roots[3]) {
  float c0 = m00 * m11 * m22 + 2.0f * m01 * m02 * m12 - m00 * m12 * m12 - m11 * m02 * m02 - m22 * m01 * m01;
  float c1 = m00 * m11 - m01 * m01 + m00 * m22 - m02 * m02 + m11 * m22 - m12 * m12;
  float c2 = m00 + m11 + m22;
  if (fabsf(c0) < 1.1920928955078125e-07f) {
    d_compute_roots2(c2, c1, roots);
  } else {
    const float s_inv3 = 1.0f / 3.0f;
    const float s_sqrt3 = 1.7320508075688772f;
    float c2_over_3 = c2 * s_inv3;
    float a_over_3 = (c1 - c2 * c2_over_3) * s_inv3;
    if (a_over_3 > 0.0f) a_over_3 = 0.0f;
    float half_b = 0.5f * (c0 + c2_over_3 * (2.0f * c2_over_3 * c2_over_3 - c1));
    float q = half_b * half_b + a_over_3 * a_over_3 * a_over_3;
    if (q > 0.0f) q = 0.0f;
    float rho = sqrtf(-a_over_3);
    const float theta = d_atan2f_pos(sqrtf(-q), half_b) * s_inv3;
    const float cos_theta = d_cosf_small(theta), sin_theta = d_sinf_small(theta);
    roots[0] = c2_over_3 + 2.0f * rho * cos_theta;
    roots[1] = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
    roots[2] = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
    if (roots[0] >= roots[1]) d_swapf(roots[0], roots[1]);
    if (roots[1] >= roots[2]) {
      d_swapf(roots[1], roots[2]);
      if (roots[0] >= roots[1]) d_swapf(roots[0], roots[1]);
    }
    if (roots[0] <= 0.0f) d_compute_roots2(c2, c1, roots);
  }
}

__device__ void d_eigen33_smallest(float c00, float c01, float c02, float c11, float c12, float c22,
                                   float& eigenvalue, float& ex, float& ey, float& ez) {
  float scale = fmaxf(fmaxf(fmaxf(fabsf(c00), fabsf(c01)), fmaxf(fabsf(c02), fabsf(c11))), fmaxf(fabsf(c12), fabsf(c22)));
  if (scale <= 1.17549435e-38f) scale = 1.0f;
  float m00 = c00 / scale, m01 = c01 / scale, m02 = c02 / scale, m11 = c11 / scale, m12 = c12 / scale, m22 = c22 / scale;
  float roots[3];
  d_compute_roots(m00, m01, m02, m11, m12, m22, roots);
  eigenvalue = roots[0] * scale;
  m00 -= roots[0]; m11 -= roots[0]; m22 -= roots[0];
  // rows r0=(m00,m01,m02) r1=(m01,m11,m12) r2=(m02,m12,m22)
  float v1x = m01 * m12 - m02 * m11, v1y = m02 * m01 - m00 * m12, v1z = m00 * m11 - m01 * m01;
  float v2x = m01 * m22 - m02 * m12, v2y = m02 * m02 - m00 * m22, v2z = m00 * m12 - m01 * m02;
  float v3x = m11 * m22 - m12 * m12, v3y = m12 * m02 - m01 * m22, v3z = m01 * m12 - m11 * m02;
  float l1 = v1x * v1x + v1y * v1y + v1z * v1z;
  float l2 = v2x * v2x + v2y * v2y + v2z * v2z;
  float l3 = v3x * v3x + v3y * v3y + v3z * v3z;
  float vx, vy, vz, l;
  if (l1 >= l2 && l1 >= l3) { vx = v1x; vy = v1y; vz = v1z; l = l1; }
  else if (l2 >= l1 && l2 >= l3) { vx = v2x; vy = v2y; vz = v2z; l = l2; }
  else { vx = v3x; vy = v3y; vz = v3z; l = l3; }
  float s = sqrtf(l);
  ex = vx / s; ey = vy / s; ez = vz / s;
}

// a2 pcl::NormalEstimation::compute, radius mode (src/tunnel_processing.cpp:58-70; SURVEY A.2-A.4).
// One thread per point in cell-sorted order: neighbouring lanes sit in the same or adjacent cells,
// so their candidate runs coincide and the candidate loads are warp-coherent L1 hits.
// The neighbour predicate is the exact FLANN L2_Simple form (unfused, strict <).
// (A variant testing candidate pairs with the packed sub/mul/add.f32x2 ops was measured 22 % SLOWER:
// packed ops hold the FP32 pipe two cycles, so only issue slots are saved, and ptxas 12.9 contracts
// mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even under -fmad=false, which breaks the exact predicate.)
// Side outputs for the tile-culled inlier counting (gm_ransac.cuh): the cloud in cell-sorted order
// with the points that the NaN compaction will drop blanked to NaN (`sorted_valid`), and the bounding
// box of the surviving points of every 32-point leaf (= one warp here): leaf_bounds[2*leaf] = min,
// [2*leaf+1] = max; an empty leaf has min = +inf, max = -inf.
constexpr int NRM_BLOCK = 128;

// single-pass mean + covariance from the 9 sums (pcl::computeMeanAndCovarianceMatrix, SURVEY A.3), eigen33, curvature and
// flipNormalTowardsViewpoint(0,0,0) (A.4): the operation order of the oracle, op for op
__device__ __forceinline__ void d_normal_from_sums(float a0, float a1, float a2, float a3, float a4, float a5, float a6, float a7, float a8,
                                                   int cnt, const float4 p, float4& o0, float4& o1) {
  const float c = (float)cnt;
  a0 /= c; a1 /= c; a2 /= c; a3 /= c; a4 /= c; a5 /= c; a6 /= c; a7 /= c; a8 /= c;
  const float c00 = a0 - a6 * a6, c01 = a1 - a6 * a7, c02 = a2 - a6 * a8;
  const float c11 = a3 - a7 * a7, c12 = a4 - a7 * a8, c22 = a5 - a8 * a8;
  float ev, nx, ny, nz;
  d_eigen33_smallest(c00, c01, c02, c11, c12, c22, ev, nx, ny, nz);
  const float eig_sum = c00 + c11 + c22;
  const float curv = (eig_sum != 0.0f) ? fabsf(ev / eig_sum) : 0.0f;
  const float vx = 0.0f - p.x, vy = 0.0f - p.y, vz = 0.0f - p.z;
  const float cos_theta = vx * nx + vy * ny + vz * nz;
  if (cos_theta < 0.0f) { nx *= -1.0f; ny *= -1.0f; nz *= -1.0f; }
  o0 = make_float4(nx, ny, nz, 0.f);
  o1 = make_float4(curv, 0.f, 0.f, 0.f);
}

// common tail of the normals kernels (whole warp): outputs in ORIGINAL (cropped) order, the cell-sorted copy with the points
// the NaN compaction will drop blanked, the bounding box of the warp's surviving points, search statistics
__device__ __forceinline__ void d_normals_epilogue(int i, bool active, const float4 p, const float4 o0, const float4 o1, int cnt, int ncand,
                                                   float4* __restrict__ normals, int* __restrict__ nbr_count, float4* __restrict__ sorted_valid,
                                                   float4* __restrict__ leaf_bounds, const OwnedRange& own, DevState* st) {
  const float qnan = CUDART_NAN_F;
  const int orig = __float_as_int(p.w);
  const bool keep = active && finite3(o0.x, o0.y, o0.z) && d_owned(own, p);  // the predicate of k_compact_valid
  if (active) {
    normals[2 * (size_t)orig] = o0;
    normals[2 * (size_t)orig + 1] = o1;
    nbr_count[orig] = cnt;
    sorted_valid[i] = keep ? p : make_float4(qnan, qnan, qnan, p.w);
  }
  const float lx = warp_min(keep ? p.x : CUDART_INF_F), ly = warp_min(keep ? p.y : CUDART_INF_F), lz = warp_min(keep ? p.z : CUDART_INF_F);
  const float hx = warp_max(keep ? p.x : -CUDART_INF_F), hy = warp_max(keep ? p.y : -CUDART_INF_F), hz = warp_max(keep ? p.z : -CUDART_INF_F);
  const int wc = __reduce_add_sync(FULL, ncand), wn = __reduce_add_sync(FULL, cnt);  // search statistics (diagnostic)
  if (lane_id() == 0) {
    atomicAdd(&st->n_candidates, (unsigned long long)wc);
    atomicAdd(&st->n_neighbors, (unsigned long long)wn);
    leaf_bounds[2 * (size_t)(i >> 5)] = make_float4(lx, ly, lz, 0.f);
    leaf_bounds[2 * (size_t)(i >> 5) + 1] = make_float4(hx, hy, hz, 0.f);
  }
}

// ONE flat walk over the candidates of all runs of a cell (not a loop over runs with a loop over candidates inside): lanes of
// a warp are points of neighbouring cells whose run lists differ, and the warp pays max-over-lanes of the TOTAL candidate
// count instead of the sum of per-run maxima.  The next run is fetched one switch ahead so the switch itself does not wait
// on memory.  Two candidates of the current run per trip (the second masked off when the run has one left): the run
// bookkeeping is paid once per pair and the two loads are in flight together.  f(candidate as two 64-bit halves, valid).
// (Issuing the loads of the NEXT pair before processing the current one was measured: k_normals<0> 0.204 -> 0.222 ms, no
// change for k_normals_knn.)
template <class F>
__device__ __forceinline__ void d_walk_runs(const float4* __restrict__ sp, const int2* __restrict__ rr, int nr, F&& f) {
  const ulonglong2* __restrict__ sp2 = reinterpret_cast<const ulonglong2*>(sp);
  int k = 0, t = 0, end = 0;
  int2 nxt = (nr > 0) ? rr[0] : make_int2(0, 0);
  for (;;) {
    const bool sw = t >= end;  // runs are non-empty by construction
    if (sw && k >= nr) break;
    // the switch itself without a branch (lanes switch at different trips: a branch here ran in 42 % of the trips with 9
    // of 32 lanes active)
    t = sw ? nxt.x : t;
    end = sw ? nxt.y : end;
    k += sw ? 1 : 0;
    if (sw && k < nr) nxt = __ldg(rr + k);
    // an odd run end reads one element past the run (masked off by `valid`): `sp` has one element of slack past the last
    // point, and f must not let the contents of an invalid candidate reach its sums (it may be a non-finite point)
    const ulonglong2 q0 = __ldg(sp2 + t), q1 = __ldg(sp2 + t + 1);
    const bool two = t + 1 < end;
    t += 2;
    f(q0, true);
    f(q1, two);
  }
}

// One candidate of the radius search: exact FLANN distance ((dx*dx + dy*dy) + dz*dz, every product and sum rounded on its
// own: fma(d,d,+0) IS the rounded product), then the nine sums and the count with masked operands: a hit adds the candidate,
// a miss adds +0 (no branch; same sums as a skipped add).  ptxas turns PREDICATED packed instructions into the packed
// instruction plus two SELs, so masking three operands is the cheaper form.
__device__ __forceinline__ void d_normals_accumulate(u64 pxy, float pz, const ulonglong2 q, float r2, bool valid, u64& a01, u64& a24, u64& a67,
                                                     u64& a8c, float& a3, float& a5) {
  float qx, qy, qz, qw, sx, sy;
  d_unpack2(q.x, qx, qy); d_unpack2(q.y, qz, qw);
  const u64 d = d_sub2(pxy, q.x);
  d_unpack2(d_fma2(d, d, 0ull), sx, sy);
  const float dz = pz - qz;
  const float d2 = (sx + sy) + dz * dz;
  const bool hit = valid && d2 < r2;
  // BOTH factors of every product are the masked values (equal to the candidate's on a hit): whatever an invalid slot
  // holds -- a non-finite point past the end of a run -- never reaches an accumulator (0 * NaN would poison it)
  const float mx = hit ? qx : 0.f, my = hit ? qy : 0.f, mz = hit ? qz : 0.f, m1 = hit ? 1.0f : 0.f;
  const u64 mxy = d_pack2(mx, my);
  a01 = d_fma2(d_pack2(mx, mx), mxy, a01);  // xx, xy
  a24 = d_fma2(d_pack2(mz, mz), mxy, a24);  // xz, yz
  a3 = fmaf(my, my, a3);
  a5 = fmaf(mz, mz, a5);
  a67 = d_add2(a67, mxy);
  a8c = d_add2(a8c, d_pack2(mz, m1));
}

// MODE 0 (default): neighbours are accumulated in cell-run order as they are found (fast; the sums differ from the
//   oracle's by float rounding only -- the neighbour SET and count are exact).
// MODE 1 (gm_set_normals_mode(1), verification): neighbours are accumulated in FLANN's result order, ascending
//   (d2, index) -- the order pcl::NormalEstimation sums them in -- by repeated selection of the next smallest pair
//   over the same candidate runs (O(neighbours x candidates): ~40x slower, no scratch memory).  With the
//   libm-independent eigen33 above the normals are then bit-identical to the CPU oracle's.
template <int MODE>
__global__ void __launch_bounds__(NRM_BLOCK)
k_normals(const float4* __restrict__ sp, const int* __restrict__ cell_id, const int2* __restrict__ runs, const int2* __restrict__ cell_info,
          const int* __restrict__ n_ptr, float r2, float4* __restrict__ normals, int* __restrict__ nbr_count,
          float4* __restrict__ sorted_valid, float4* __restrict__ leaf_bounds, OwnedRange own, DevState* st) {
  const int n = *n_ptr;
  const int i = blockIdx.x * NRM_BLOCK + threadIdx.x;
  if ((i & ~31) >= n) return;  // warp-uniform: the whole leaf is past the end
  const bool active = i < n;
  const float qnan = CUDART_NAN_F;
  const float4 p = active ? sp[i] : make_float4(qnan, qnan, qnan, 0.f);
  const int orig = __float_as_int(p.w);
  float4 o0 = make_float4(qnan, qnan, qnan, 0.f), o1 = make_float4(qnan, 0.f, 0.f, 0.f);
  int cnt = 0, ncand = 0;
  if (active && finite3(p.x, p.y, p.z)) {
    const int cid = cell_id[i];
    const int2* rr = runs + (size_t)cid * GRID_RUNS;
    const int2 info = cell_info[cid];
    const int nr = info.x, total = info.y;
    ncand = total;
    if (MODE == 0) {
      // accumulators as f32x2 pairs: (xx,xy) (xz,yz) (x,y) (z,count); yy and zz stay scalar.  The count is
      // carried as a float (exact below 2^24 neighbours) so that it shares an instruction with the z sum.
      u64 a01 = 0ull, a24 = 0ull, a67 = 0ull, a8c = 0ull;
      float a3 = 0.f, a5 = 0.f;
      const u64 pxy = d_pack2(p.x, p.y);
      d_walk_runs(sp, rr, nr, [&](const ulonglong2 q, const bool valid) {
        d_normals_accumulate(pxy, p.z, q, r2, valid, a01, a24, a67, a8c, a3, a5);
      });
      float a0, a1, a2, a4, a6, a7, a8, cntf;
      d_unpack2(a01, a0, a1); d_unpack2(a24, a2, a4); d_unpack2(a67, a6, a7); d_unpack2(a8c, a8, cntf);
      cnt = (int)cntf;
      if (cnt >= 3) d_normal_from_sums(a0, a1, a2, a3, a4, a5, a6, a7, a8, cnt, p, o0, o1);
    } else {
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, a4 = 0.f, a5 = 0.f, a6 = 0.f, a7 = 0.f, a8 = 0.f;
      float last_d2 = -1.0f;  // every real d2 is >= 0
      int last_id = -1;
      for (;;) {
        float best_d2 = CUDART_INF_F;
        int best_id = 0x7FFFFFFF;
        float4 bq = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int k = 0; k < nr; ++k) {
          const int2 run = rr[k];
          for (int t = run.x; t < run.y; ++t) {
            const float4 q = sp[t];
            const int id = __float_as_int(q.w);
            const float dx = p.x - q.x, dy = p.y - q.y, dz = p.z - q.z;
            const float d2 = (dx * dx + dy * dy) + dz * dz;
            const bool after = d2 > last_d2 || (d2 == last_d2 && id > last_id);
            const bool better = d2 < best_d2 || (d2 == best_d2 && id < best_id);
            if (d2 < r2 && after && better) { best_d2 = d2; best_id = id; bq = q; }
          }
        }
        if (best_id == 0x7FFFFFFF) break;
        a0 += bq.x * bq.x; a1 += bq.x * bq.y; a2 += bq.x * bq.z;
        a3 += bq.y * bq.y; a4 += bq.y * bq.z; a5 += bq.z * bq.z;
        a6 += bq.x; a7 += bq.y; a8 += bq.z;
        ++cnt;
        last_d2 = best_d2; last_id = best_id;
      }
      if (cnt >= 3) d_normal_from_sums(a0, a1, a2, a3, a4, a5, a6, a7, a8, cnt, p, o0, o1);
    }
  }
  d_normals_epilogue(i, active, p, o0, o1, cnt, ncand, normals, nbr_count, sorted_valid, leaf_bounds, own, st);
}



// ---- a2, k mode: pcl::NormalEstimation with setKSearch(k) (the north-star's "grid-hashed k-NN") ---------------------------
// The k nearest points (FLANN L2_Simple distance, the query included, ties by ascending index) instead of the points
// within a radius; the rest of the pipeline (single-pass covariance, eigen33, curvature, flip) is the same.
// One thread per query keeps its k best (d2, index) pairs as 64-bit keys in a max-heap in shared memory: a candidate is
// offered only if it beats the current k-th key (the root); the finished heap is sorted into FLANN's result order, so
// the neighbours are summed in exactly the order pcl::NormalEstimation sums them and the normals are bit-identical to
// the CPU oracle's in this mode.
//   pass A   the 27-cell stencil (the runs of the radius mode), only candidates nearer than one cell.  Complete iff k keys
//            were found: nothing outside the stencil can be nearer.  (Size the grid -- neighborRadius -- near the expected
//            distance of the k-th neighbour and almost every point ends here.)
//   pass B1  (sparser neighbourhoods) the rest of the stencil, then rings 2, 3, .. of cells through the block table (as far as
//            the radius cap, if there is one); complete when the k-th distance is below the ring's distance.
//   pass B2  (isolated points) restart over whole 4x4x4-cell blocks in growing Chebyshev shells around the query's block
//            -- a block is ONE contiguous run of the sorted cloud and an empty block costs one table read.
constexpr int KNN_BLOCK = 32;  // ONE warp per block: a warp held up by a sparse query (pass B) keeps only its own shared memory
                               // (64: 3.1 ms, 128 / 256: 3.6 / 4.1 ms; smaller carve-outs for more L1: slower, profiles/r02_knn.md)
constexpr int KNN_MAX = 64;
constexpr int KNN_WIDE = 4;  // 8: same time
constexpr int KNN_BINS = 32;  // histogram bins of pass A (u32 each) ...
constexpr int KNN_BND = 16;   // ... overlaid by the boundary buffer (u64 each): the same KNN_BINS * 4 bytes per thread
constexpr int KNN_AUX = KNN_BND + 1;  // + one word that takes what is not wanted (bin KNN_BINS / slot KNN_BND): no branch in the walks

// the FLANN L2_Simple distance of the radius kernel: ((dx*dx + dy*dy) + dz*dz), every product and sum rounded on its own
__device__ __forceinline__ float d_flann_d2(u64 pxy, float pz, const ulonglong2 q) {
  float sx, sy, qz, qw;
  const u64 d = d_sub2(pxy, q.x);
  d_unpack2(d_fma2(d, d, 0ull), sx, sy);
  d_unpack2(q.y, qz, qw);
  const float dz = pz - qz;
  return (sx + sy) + dz * dz;
}
// The k best (d2, index) keys of one query as a binary MAX-HEAP in shared memory (element j of this thread's heap is
// slot[j * KNN_BLOCK]): the root is the current k-th key, an accepted candidate costs one sift of <= log2(k) steps (the
// sparse-neighbourhood passes B1/B2 insert this way; pass A selects without inserting, see the kernel).  sort() heap-sorts
// in place at the end: the list is then in FLANN's result order (ascending distance, ties by index).
struct KnnList {
  unsigned long long* slot;
  int K, cnt;
  unsigned long long worst;  // the root once the heap is full, else "infinity"
  __device__ __forceinline__ void reset() { cnt = 0; worst = ~0ull; }
  __device__ __forceinline__ static unsigned long long make_key(float d2, int id) {
    return ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned)id;  // d2 >= +0: the float bits order like the value
  }
  __device__ __forceinline__ void offer(float d2, int id) { offer_key(make_key(d2, id)); }
  // sift `key` down from the root of the heap of the first n elements
  __device__ __forceinline__ void sift_down(const unsigned long long key, int n, int j = 0) {
    for (;;) {
      int c = 2 * j + 1;
      if (c >= n) break;
      unsigned long long vc = slot[c * KNN_BLOCK];
      if (c + 1 < n) {
        const unsigned long long v2 = slot[(c + 1) * KNN_BLOCK];
        if (v2 > vc) { vc = v2; ++c; }
      }
      if (vc <= key) break;
      slot[j * KNN_BLOCK] = vc;
      j = c;
    }
    slot[j * KNN_BLOCK] = key;
  }
  __device__ __forceinline__ void offer_key(const unsigned long long key) {
    if (!(key < worst)) return;  // (NaN distances have the largest bit patterns: never accepted once the heap is full)
    if (cnt < K) {               // grow: sift up
      int j = cnt++;
      while (j > 0) {
        const int par = (j - 1) >> 1;
        const unsigned long long v = slot[par * KNN_BLOCK];
        if (v >= key) break;
        slot[j * KNN_BLOCK] = v;
        j = par;
      }
      slot[j * KNN_BLOCK] = key;
      if (cnt == K) worst = slot[0];
    } else {                     // replace the root (the k-th key so far)
      sift_down(key, K);
      worst = slot[0];
    }
  }
  __device__ __forceinline__ void heapify() {  // make the first cnt slots (any order) a heap
    for (int j = (cnt >> 1) - 1; j >= 0; --j) sift_down(slot[j * KNN_BLOCK], cnt, j);
    worst = (cnt == K) ? slot[0] : ~0ull;
  }
  __device__ __forceinline__ void sort() {  // in-place heap sort: ascending keys
    for (int n = cnt - 1; n > 0; --n) {
      const unsigned long long last = slot[n * KNN_BLOCK];
      slot[n * KNN_BLOCK] = slot[0];
      sift_down(last, n);
    }
  }
};

__global__ void __launch_bounds__(KNN_BLOCK)
k_normals_knn(const float4* __restrict__ sp, const float4* __restrict__ crop, const int* __restrict__ cell_id, const int2* __restrict__ runs,
              const int2* __restrict__ cell_info, const BlockEntry* __restrict__ tab, const int* __restrict__ ucell_start, const int* __restrict__ n_ptr,
              GridSpec g, int K, float max_r2 /* neighbours must be nearer than this (+inf = plain k-NN) */, float4* __restrict__ normals,
              int* __restrict__ nbr_count, float4* __restrict__ sorted_valid, float4* __restrict__ leaf_bounds, OwnedRange own, DevState* st,
              int* __restrict__ knn_idx) {
  extern __shared__ unsigned long long knn_smem[];  // [K][KNN_BLOCK]
  const int n = *n_ptr;
  const int i = blockIdx.x * KNN_BLOCK + threadIdx.x;
  if ((i & ~31) >= n) return;
  const bool active = i < n;
  const float qnan = CUDART_NAN_F;
  const float4 p = active ? sp[i] : make_float4(qnan, qnan, qnan, 0.f);
  const int orig = __float_as_int(p.w);
  float4 o0 = make_float4(qnan, qnan, qnan, 0.f), o1 = make_float4(qnan, 0.f, 0.f, 0.f);
  int cnt = 0, ncand = 0;
  const bool work = active && finite3(p.x, p.y, p.z);
  KnnList L;
  L.slot = knn_smem + threadIdx.x;
  L.K = K;
  L.reset();
  const int cid = work ? cell_id[i] : 0;
  const int2* rr = runs + (size_t)cid * GRID_RUNS;
  const int2 info = work ? cell_info[cid] : make_int2(0, 0);
  const int nr = info.x, total = info.y;
  // ---- pass A: the 27-cell stencil; only candidates nearer than one cell can matter if this pass is to be complete.
  // Keeping the k best in a heap WHILE walking costs a data-dependent sift per accepted candidate, and the lanes of a warp
  // accept at different moments: even with per-lane pending buffers the warp ran those loops a few lanes at a time
  // (profiles/r02_knn.md).  So pass A SELECTS instead, with two uniform walks over the same candidates:
  //   walk 1  histogram of d2 in KNN_BINS equal bins over [0, one cell]^2 (bin index is monotone in d2, equal d2 -> equal bin);
  //           the bin b* in which the running count reaches k holds the k-th neighbour: everything in a lower bin is in.
  //   walk 2  keys of the lower bins go straight into the list, keys of bin b* into a small boundary buffer (it overlays
  //           the histogram); the k - |lower| smallest boundary keys complete the list.
  // No walk contains a data-dependent loop.  The list is then made a heap for the later passes / the final sort.
  // Neither walk branches on the candidate: a candidate that does not count increments a spare bin, a key that is not kept is
  // stored to a spare word (divergent branches in a flat walk cost k_normals<0> 10 %).
  // (More than KNN_BND keys in the boundary bin -- coincident points -- : that lane falls back to heap insertion.)
  const float lim1 = (g.cell * 0.999f) * (g.cell * 0.999f);
  {
    unsigned long long* bnd = knn_smem + (size_t)K * KNN_BLOCK + threadIdx.x;  // [KNN_AUX][KNN_BLOCK] u64: this thread's words ...
    unsigned* hist32 = reinterpret_cast<unsigned*>(bnd);                       // ... and the same words as 2 x u32 bins each
    auto hist_at = [&](int bq) -> unsigned& { return hist32[(((bq >> 1) * KNN_BLOCK) << 1) | (bq & 1)]; };
#pragma unroll
    for (int j = 0; j < KNN_AUX; ++j) bnd[j * KNN_BLOCK] = 0ull;
    const float binscale = (float)KNN_BINS / lim1;
    const u64 pxy = d_pack2(p.x, p.y);
    d_walk_runs(sp, rr, nr, [&](const ulonglong2 q, const bool valid) {
      const float d2 = d_flann_d2(pxy, p.z, q);
      const bool elig = valid && d2 <= lim1 && d2 < max_r2;
      hist_at(elig ? min((int)(d2 * binscale), KNN_BINS - 1) : KNN_BINS) += 1u;
    });
    int bstar = KNN_BINS, below = 0, cum = 0;
#pragma unroll 4
    for (int bq = 0; bq < KNN_BINS; ++bq) {
      const int c = (int)hist_at(bq);
      if (bstar == KNN_BINS && cum + c >= K) { bstar = bq; below = cum; }
      cum += c;
    }
    // fewer than k candidates within one cell: all of them are in (bstar stays KNN_BINS), the later passes go on
    int c = 0, m = 0;
    bool ovf = false;
    d_walk_runs(sp, rr, nr, [&](const ulonglong2 q, const bool valid) {
      const float d2 = d_flann_d2(pxy, p.z, q);
      const bool elig = valid && d2 <= lim1 && d2 < max_r2;
      const int bq = min((int)(d2 * binscale), KNN_BINS - 1);
      const bool lower = elig && bq < bstar, isb = elig && bq == bstar, fits = isb && m < KNN_BND;
      L.slot[(lower ? c : K + (fits ? m : KNN_BND)) * KNN_BLOCK] = KnnList::make_key(d2, (int)(unsigned)(q.y >> 32));
      c += lower ? 1 : 0;
      m += fits ? 1 : 0;
      ovf = ovf || (isb && !fits);
    });
    if (!ovf) {
      const int need = (bstar < KNN_BINS) ? K - below : 0;  // 1 <= need <= m
      for (int s = 0; s < need; ++s) {                        // the `need` smallest boundary keys, by selection
        int best = s;
        unsigned long long bk = bnd[s * KNN_BLOCK];
        for (int j = s + 1; j < m; ++j) {
          const unsigned long long v = bnd[j * KNN_BLOCK];
          if (v < bk) { bk = v; best = j; }
        }
        bnd[best * KNN_BLOCK] = bnd[s * KNN_BLOCK];
        L.slot[(c + s) * KNN_BLOCK] = bk;
      }
      L.cnt = c + need;
      L.heapify();
    } else {
      L.reset();
      for (int k = 0; k < nr; ++k) {
        const int2 run = rr[k];
        for (int t = run.x; t < run.y; ++t) {
          const float4 q = sp[t];
          const float dx = p.x - q.x, dy = p.y - q.y, dz = p.z - q.z;
          const float d2 = (dx * dx + dy * dy) + dz * dz;
          if (d2 <= lim1 && d2 < max_r2) L.offer(d2, __float_as_int(q.w));
        }
      }
    }
  }
  if (work) {
    const int U = st->n_cells, nf = st->n_sorted_finite;
    // The candidates of a sorted-position range, KNN_WIDE loads in flight at a time: a sparse query runs these loops with the
    // rest of its warp waiting, and one dependent load per candidate was most of what it cost.
    auto offer_range = [&](int t0, int t1) {
      for (int t = t0; t < t1; t += 4) {
        float4 q4[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) q4[u] = sp[min(t + u, t1 - 1)];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float ex = p.x - q4[u].x, ey = p.y - q4[u].y, ez = p.z - q4[u].z;
          const float e2 = (ex * ex + ey * ey) + ez * ez;
          if (t + u < t1 && e2 < max_r2) L.offer(e2, __float_as_int(q4[u].w));
        }
      }
    };
    ncand = total;
    // k keys, all within one cell of the query (the filter above) -- or the radius cap lies inside the stencil's reach
    bool complete = L.cnt == K || max_r2 <= lim1;
    if (!complete && nf > L.cnt) {
      // ---- pass B1: growing rings of CELLS around the query's cell.  The list was never full in pass A, so it holds EVERY
      // stencil candidate nearer than one cell; the stencil is walked once more for the farther ones (d2 > lim1), then ring k >= 2 = its rows through the block table.  After ring k every
      // unexamined point is at least k cells away.  Sparse surface points end here (the k-th neighbour is within 2-3 cells).
      int cx, cy, cz;
      gm_cell_of(g, p.x, p.y, p.z, cx, cy, cz);
      {
        const u64 pxy = d_pack2(p.x, p.y);
        d_walk_runs(sp, rr, nr, [&](const ulonglong2 q, const bool valid) {
          const float d2 = d_flann_d2(pxy, p.z, q);
          if (valid && d2 > lim1 && d2 < max_r2) L.offer(d2, (int)(unsigned)(q.y >> 32));
        });
      }
      auto done_at = [&](int ring) {  // the k-th neighbour, or the radius cap, lies inside what has been examined
        const float lim = (float)ring * g.cell * 0.999f;
        return (L.cnt == K && __uint_as_float((unsigned)(L.worst >> 32)) <= lim * lim) || max_r2 <= lim * lim;
      };
      complete = done_at(1);
      // with a radius cap the rings go as far as the cap (and pass B2 is never needed); without one, 3 rings, then blocks
      const int max_ring = (max_r2 < CUDART_INF_F) ? (int)ceilf(sqrtf(max_r2) / (g.cell * 0.999f)) + 1 : 3;
      for (int ring = 2; !complete && ring <= max_ring; ++ring) {
        const int inner = 2 * ring - 1, T = 8 * ring + 2 * inner * inner;  // perimeter rows (full x span) + inner rows (two end cells)
        for (int t = 0; t < T; ++t) {
          int dy, dz, x0, x1;
          if (t < 8 * ring) {
            if (t < 2 * ring + 1) { dz = -ring; dy = t - ring; }
            else if (t < 4 * ring + 2) { dz = ring; dy = t - (2 * ring + 1) - ring; }
            else if (t < 6 * ring + 1) { dy = -ring; dz = t - (4 * ring + 2) - (ring - 1); }
            else { dy = ring; dz = t - (6 * ring + 1) - (ring - 1); }
            x0 = cx - ring; x1 = cx + ring;
          } else {
            const int u2 = t - 8 * ring, cell = u2 >> 1;
            dy = cell % inner - (ring - 1); dz = cell / inner - (ring - 1);
            x0 = x1 = (u2 & 1) ? cx + ring : cx - ring;
          }
          const int yy = cy + dy, zz = cz + dz;
          if (yy < 0 || zz < 0 || yy >= g.dim[1] || zz >= g.dim[2]) continue;
          x0 = max(x0, 0); x1 = min(x1, g.dim[0] - 1);
          for (int xs = x0; xs <= x1;) {
            const int xe = min(x1, xs | 3);
            const int2 seg = cell_segment(g, tab, ucell_start, U, nf, xs, xe, yy, zz);
            ncand += seg.y - seg.x;
            offer_range(seg.x, seg.y);
            xs = xe + 1;
          }
        }
        complete = done_at(ring);
      }
    }
    if (!complete && nf > L.cnt && !(max_r2 < CUDART_INF_F)) {
      // ---- pass B2 (isolated points, no radius cap): whole blocks in growing shells, from scratch
      L.reset();
      int cx, cy, cz;
      gm_cell_of(g, p.x, p.y, p.z, cx, cy, cz);
      const int bx = cx >> 2, by = cy >> 2, bz = cz >> 2;
      const int nbx = (g.dim[0] + 3) >> 2, nby = (g.dim[1] + 3) >> 2, nbz = (g.dim[2] + 3) >> 2;
      const int bmax = max(max(max(bx, nbx - 1 - bx), max(by, nby - 1 - by)), max(bz, nbz - 1 - bz));
      for (int b = 0; b <= bmax; ++b) {
        for (int dz = -b; dz <= b; ++dz) {
          const int z = bz + dz;
          if (z < 0 || z >= nbz) continue;
          for (int dy = -b; dy <= b; ++dy) {
            const int y = by + dy;
            if (y < 0 || y >= nby) continue;
            const bool face = (dz == -b || dz == b || dy == -b || dy == b);
            for (int dx = -b; dx <= b; dx += (face || b == 0) ? 1 : 2 * b) {  // inner rows: only the two end blocks
              const int x = bx + dx;
              if (x < 0 || x >= nbx) continue;
              const BlockEntry e = tab[gm_cell_key(g, x << 2, y << 2, z << 2) >> 6];
              if (e.mask == 0ull) continue;
              // prune by geometry once the list is full: a block, then each of its occupied cells, whose box lies farther
              // from the query than the current k-th neighbour cannot contribute (boxes grown by 0.1 % for the float
              // rounding of the cell coordinate)
              const float wd2 = (L.cnt == K) ? __uint_as_float((unsigned)(L.worst >> 32)) : CUDART_INF_F;
              const float bs = 4.0f * g.cell, slack = 0.001f * g.cell;
              const float bx0 = g.origin[0] + (float)x * bs, by0 = g.origin[1] + (float)y * bs, bz0 = g.origin[2] + (float)z * bs;
              {
                const float ddx = fmaxf(fmaxf(bx0 - slack - p.x, p.x - (bx0 + bs + slack)), 0.f);
                const float ddy = fmaxf(fmaxf(by0 - slack - p.y, p.y - (by0 + bs + slack)), 0.f);
                const float ddz = fmaxf(fmaxf(bz0 - slack - p.z, p.z - (bz0 + bs + slack)), 0.f);
                if ((ddx * ddx + ddy * ddy) + ddz * ddz > wd2) continue;
              }
              unsigned long long m = e.mask;
              int rank = e.first;
              while (m) {
                const int lc = __ffsll((long long)m) - 1;  // local cell code: x fastest, then y, then z (2 bits each)
                m &= m - 1ull;
                const int c_id = rank++;
                const float cx0 = bx0 + (float)(lc & 3) * g.cell, cy0 = by0 + (float)((lc >> 2) & 3) * g.cell, cz0 = bz0 + (float)(lc >> 4) * g.cell;
                const float ddx = fmaxf(fmaxf(cx0 - slack - p.x, p.x - (cx0 + g.cell + slack)), 0.f);
                const float ddy = fmaxf(fmaxf(cy0 - slack - p.y, p.y - (cy0 + g.cell + slack)), 0.f);
                const float ddz = fmaxf(fmaxf(cz0 - slack - p.z, p.z - (cz0 + g.cell + slack)), 0.f);
                const float cur = (L.cnt == K) ? __uint_as_float((unsigned)(L.worst >> 32)) : CUDART_INF_F;
                if ((ddx * ddx + ddy * ddy) + ddz * ddz > cur) continue;
                const int t0 = min(ucell_start[c_id], nf), t1 = (c_id + 1 < U) ? min(ucell_start[c_id + 1], nf) : nf;
                ncand += t1 - t0;
                offer_range(t0, t1);
              }
            }
          }
        }
        // every unexamined point lies b whole blocks (4 cells each) or more beyond the query's block
        const float lim = 4.0f * (float)b * g.cell * 0.999f;
        if (L.cnt == K && __uint_as_float((unsigned)(L.worst >> 32)) <= lim * lim) break;
      }
    }
    L.sort();
    cnt = L.cnt;
    if (knn_idx != nullptr)
      for (int j = 0; j < K; ++j) knn_idx[(size_t)orig * K + j] = j < cnt ? (int)(unsigned)L.slot[j * KNN_BLOCK] : -1;
    if (cnt >= 3) {
      // the list is in FLANN's result order: sum in that order, plain float operations (the oracle's, op for op)
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, a4 = 0.f, a5 = 0.f, a6 = 0.f, a7 = 0.f, a8 = 0.f;
      for (int j = 0; j < cnt; ++j) {
        const float4 q = crop[(int)(unsigned)L.slot[j * KNN_BLOCK]];
        a0 += q.x * q.x; a1 += q.x * q.y; a2 += q.x * q.z;
        a3 += q.y * q.y; a4 += q.y * q.z; a5 += q.z * q.z;
        a6 += q.x; a7 += q.y; a8 += q.z;
      }
      d_normal_from_sums(a0, a1, a2, a3, a4, a5, a6, a7, a8, cnt, p, o0, o1);
    }
  }
  d_normals_epilogue(i, active, p, o0, o1, cnt, ncand, normals, nbr_count, sorted_valid, leaf_bounds, own, st);
}

// a3 removeNaNNormalsFromPointCloud + ExtractIndices (src/tunnel_processing.cpp:74-85): stable
// compaction of cloud and normals by isfinite(nx,ny,nz); also the bounding box of the survivors
// (pcl::getMinMax3D of the VoxelGrid that follows).
__global__ void __launch_bounds__(CP_BLOCK)
k_compact_valid(const float4* __restrict__ pts, const float4* __restrict__ normals, const int* __restrict__ n_ptr,
                float4* __restrict__ pts_c, float4* __restrict__ normals_c, int* __restrict__ valid_map,
                unsigned long long* state, TileCtl* ctl, DevState* st, OwnedRange own) {
  __shared__ CompactSmem<CP_BLOCK, CP_IPT> sm;
  __shared__ float s_red[6][CP_BLOCK / 32];
  const int n = *n_ptr;
  unsigned epoch;
  const int tile = tile_begin(ctl, epoch), base = tile * CP_TILE;
  if (base >= n) { tile_end(ctl); return; }
  bool f[CP_IPT];
  float4 p[CP_IPT], n0[CP_IPT], n1[CP_IPT];
  float mn[3] = {CUDART_INF_F, CUDART_INF_F, CUDART_INF_F}, mx[3] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
#pragma unroll
  for (int j = 0; j < CP_IPT; ++j) {
    int i = base + j * CP_BLOCK + threadIdx.x;
    f[j] = false;
    if (i < n) {
      p[j] = pts[i];
      n0[j] = normals[2 * (size_t)i];
      n1[j] = normals[2 * (size_t)i + 1];
      f[j] = finite3(n0[j].x, n0[j].y, n0[j].z) && d_owned(own, p[j]);
      if (f[j]) {
        mn[0] = fminf(mn[0], p[j].x); mn[1] = fminf(mn[1], p[j].y); mn[2] = fminf(mn[2], p[j].z);
        mx[0] = fmaxf(mx[0], p[j].x); mx[1] = fmaxf(mx[1], p[j].y); mx[2] = fmaxf(mx[2], p[j].z);
      }
    }
  }
  unsigned ranks[CP_IPT], total;
  tile_compact_ranks<CP_BLOCK, CP_IPT>(f, ranks, total, state, epoch, tile, &st->error, sm);
#pragma unroll
  for (int j = 0; j < CP_IPT; ++j) {
    int i = base + j * CP_BLOCK + threadIdx.x;
    if (i < n) {
      valid_map[i] = f[j] ? (int)ranks[j] : -1;
      if (f[j]) {
        pts_c[ranks[j]] = p[j];
        normals_c[2 * (size_t)ranks[j]] = n0[j];
        normals_c[2 * (size_t)ranks[j] + 1] = n1[j];
      }
    }
  }
  if (base + CP_TILE >= n && threadIdx.x == 0) { st->n_valid = (int)total; st->vox.n = (int)total; }
  // block bbox -> global (min/max are order independent: deterministic)
  const int w = threadIdx.x >> 5;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float lo = warp_min(mn[a]), hi = warp_max(mx[a]);
    if (lane_id() == 0) { s_red[a][w] = lo; s_red[3 + a][w] = hi; }
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    float lo = CUDART_INF_F, hi = -CUDART_INF_F;
    for (int ww = 0; ww < CP_BLOCK / 32; ++ww) { lo = fminf(lo, s_red[threadIdx.x][ww]); hi = fmaxf(hi, s_red[3 + threadIdx.x][ww]); }
    if (lo <= hi) {
      atomicMin(&st->vox.bbox_min[threadIdx.x], float_to_ordered(lo));
      atomicMax(&st->vox.bbox_max[threadIdx.x], float_to_ordered(hi));
    }
  }
  tile_end(ctl);
}

// Replace the bounding box of the compacted cloud (all-reduced box of all map slabs -> one global lattice).
__global__ void k_set_bbox(VoxState* vs, float x0, float y0, float z0, float x1, float y1, float z1) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    vs->bbox_min[0] = float_to_ordered(x0); vs->bbox_min[1] = float_to_ordered(y0); vs->bbox_min[2] = float_to_ordered(z0);
    vs->bbox_max[0] = float_to_ordered(x1); vs->bbox_max[1] = float_to_ordered(y1); vs->bbox_max[2] = float_to_ordered(z1);
  }
}

// Bounding box only (used when the compacted cloud was injected).
__global__ void k_bbox(const float4* __restrict__ pts, VoxState* vs) {
  const int n = vs->n;
  float mn[3] = {CUDART_INF_F, CUDART_INF_F, CUDART_INF_F}, mx[3] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float4 p = pts[i];
    mn[0] = fminf(mn[0], p.x); mn[1] = fminf(mn[1], p.y); mn[2] = fminf(mn[2], p.z);
    mx[0] = fmaxf(mx[0], p.x); mx[1] = fmaxf(mx[1], p.y); mx[2] = fmaxf(mx[2], p.z);
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float lo = warp_min(mn[a]), hi = warp_max(mx[a]);
    if (lane_id() == 0 && lo <= hi) {
      atomicMin(&vs->bbox_min[a], float_to_ordered(lo));
      atomicMax(&vs->bbox_max[a], float_to_ordered(hi));
    }
  }
}

// a4 pcl::VoxelGrid lattice (SURVEY A.5): min_b, div_b, divb_mul and the overflow rule, derived
// from the bounding box by every block (cheap, avoids a 1-thread kernel); block 0 publishes it.
// Voxel key per compacted point: ijk = int(floor(p*inv) - float(min_b)); key = ijk . divb_mul
struct VoxLattice { int minb[3]; int mul[3]; int overflow; };
// thread 0 of every block derives the lattice from the bounding box (cheap, avoids a 1-thread kernel); block 0 publishes it
__device__ __forceinline__ void d_vox_lattice(VoxState* st, float inv, VoxLattice* out /* shared */) {
  if (threadIdx.x == 0) {
    const int n = st->n;
    float mn[3], mx[3];
    for (int a = 0; a < 3; ++a) { mn[a] = ordered_to_float(st->bbox_min[a]); mx[a] = ordered_to_float(st->bbox_max[a]); }
    int div[3] = {0, 0, 0}, minb[3] = {0, 0, 0}, overflow = 0;
    if (n > 0) {
      long long dx = (long long)((mx[0] - mn[0]) * inv) + 1;
      long long dy = (long long)((mx[1] - mn[1]) * inv) + 1;
      long long dz = (long long)((mx[2] - mn[2]) * inv) + 1;
      if (dx * dy * dz > 2147483647LL) overflow = 1;
      for (int a = 0; a < 3; ++a) {
        int lo = (int)floorf(mn[a] * inv), hi = (int)floorf(mx[a] * inv);
        minb[a] = lo; div[a] = hi - lo + 1;
      }
    }
    for (int a = 0; a < 3; ++a) out->minb[a] = minb[a];
    out->mul[0] = 1; out->mul[1] = div[0]; out->mul[2] = div[0] * div[1];
    out->overflow = overflow;
    if (blockIdx.x == 0) {
      st->v_inv = inv;
      st->overflow = overflow;
      for (int a = 0; a < 3; ++a) { st->min_b[a] = minb[a]; st->div_b[a] = div[a]; st->mul[a] = out->mul[a]; }
    }
  }
  __syncthreads();
}
__device__ __forceinline__ int d_vox_key(const VoxLattice& L, float inv, const float4 p) {
  int ijk0 = (int)(floorf(p.x * inv) - (float)L.minb[0]);
  int ijk1 = (int)(floorf(p.y * inv) - (float)L.minb[1]);
  int ijk2 = (int)(floorf(p.z * inv) - (float)L.minb[2]);
  return ijk0 + ijk1 * L.mul[1] + ijk2 * L.mul[2];
}

__global__ void k_voxel_keys(const float4* __restrict__ pts, VoxState* st, float inv,
                             unsigned* __restrict__ keys, unsigned* __restrict__ idx, int* __restrict__ key_of_point) {
  __shared__ VoxLattice L;
  d_vox_lattice(st, inv, &L);
  const int n = st->n;
  const bool overflow = L.overflow != 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float4 p = pts[i];
    int key = overflow ? i : d_vox_key(L, inv, p);
    keys[i] = (unsigned)key;
    idx[i] = (unsigned)i;
    key_of_point[i] = key;
  }
}

// ---- VoxelGrid without a sort ---------------------------------------------------------------------
// When the key range is known (on the host) to fit the dense tables, a voxel is just the table entry of its
// key: one pass adds every point to its entry (count + fixed-point sums, integer atomics), one look-back
// compaction over the table numbers the occupied keys in ascending order (= the voxel order of
// pcl::VoxelGrid), emits key / count / centroid, remembers the voxel id per key and zeroes the entries it
// consumed (the tables clean themselves), and one pass maps every point to its voxel id.  3 launches and
// ~60 B of traffic per point instead of the 12 launches / 132 B of the sort-based path below.
__global__ void k_voxel_accumulate(const float4* __restrict__ pts, VoxState* st, float inv,
                                   int* __restrict__ dcnt, unsigned long long* __restrict__ dsum, int capacity, int* err) {
  __shared__ VoxLattice L;
  d_vox_lattice(st, inv, &L);
  const int n = st->n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    const int key = d_vox_key(L, inv, p);
    if ((unsigned)key >= (unsigned)capacity) { atomicExch(err, 4); continue; }  // cannot happen: the host bound covers the crop box
    atomicAdd(&dcnt[key], 1);
    atomicAdd(&dsum[3 * (size_t)key + 0], (unsigned long long)d_fx20(p.x));
    atomicAdd(&dsum[3 * (size_t)key + 1], (unsigned long long)d_fx20(p.y));
    atomicAdd(&dsum[3 * (size_t)key + 2], (unsigned long long)d_fx20(p.z));
  }
}

// The same accumulation over the CELL-SORTED copy of the cloud (dropped points blanked to NaN, .w = cropped
// index): the sums do not depend on the order, and in this order neighbouring lanes of a warp mostly fall into
// the same voxel.  Runs of equal keys in consecutive lanes are combined with a segmented warp scan (head flags
// from one ballot, 5 shuffle steps) and only the last lane of a run issues the atomics: ~5x fewer than one set
// per point.  (A match.any + redux.sync grouping of ALL equal keys of the warp was measured no faster than plain
// per-point atomics: 42 us, 425 instructions per warp iteration — the per-group redux loops diverge.)
__global__ void __launch_bounds__(256)
k_voxel_accumulate_sorted(const float4* __restrict__ sv, const int* __restrict__ n_ptr, VoxState* st,
                          float inv, int* __restrict__ dcnt, unsigned long long* __restrict__ dsum, int capacity, int* err) {
  __shared__ VoxLattice L;
  d_vox_lattice(st, inv, &L);
  const int n = *n_ptr;
  const int lane = threadIdx.x & 31;
  for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {  // block-uniform trip count
    const int i = base + threadIdx.x;
    int key = -1, c = 0;
    long long fx = 0, fy = 0, fz = 0;
    if (i < n) {
      const float4 p = sv[i];
      if (p.x == p.x) {  // not blanked
        key = d_vox_key(L, inv, p);
        if ((unsigned)key >= (unsigned)capacity) { atomicExch(err, 4); key = -1; }
        else { c = 1; fx = d_fx20(p.x); fy = d_fx20(p.y); fz = d_fx20(p.z); }
      }
    }
    const int prev = __shfl_up_sync(FULL, key, 1);
    const unsigned heads = __ballot_sync(FULL, lane == 0 || key != prev);
    const int start = 31 - __clz(heads & (0xFFFFFFFFu >> (31 - lane)));  // first lane of this lane's run
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int tc = __shfl_up_sync(FULL, c, d);
      const long long tx = __shfl_up_sync(FULL, fx, d), ty = __shfl_up_sync(FULL, fy, d), tz = __shfl_up_sync(FULL, fz, d);
      if (lane - d >= start) { c += tc; fx += tx; fy += ty; fz += tz; }
    }
    const bool last = lane == 31 || ((heads >> (lane + 1)) & 1u);
    if (last && key >= 0) {
      atomicAdd(&dcnt[key], c);
      atomicAdd(&dsum[3 * (size_t)key + 0], (unsigned long long)fx);
      atomicAdd(&dsum[3 * (size_t)key + 1], (unsigned long long)fy);
      atomicAdd(&dsum[3 * (size_t)key + 2], (unsigned long long)fz);
    }
  }
}

__global__ void __launch_bounds__(CP_BLOCK)
k_voxel_dense_scan(int* __restrict__ dcnt, long long* __restrict__ dsum, int* __restrict__ did, int range,
                   int* __restrict__ vox_key, int* __restrict__ vox_count, float4* __restrict__ centroids,
                   unsigned long long* state, TileCtl* ctl, VoxState* st, int* err) {
  __shared__ CompactSmem<CP_BLOCK, CPL_IPT> sm;
  unsigned epoch;
  const int tile = tile_begin(ctl, epoch), base = tile * CPL_TILE;
  bool f[CPL_IPT];
  int c[CPL_IPT];
#pragma unroll
  for (int j = 0; j < CPL_IPT; ++j) {
    const int k = base + j * CP_BLOCK + threadIdx.x;
    c[j] = (k < range) ? dcnt[k] : 0;
    f[j] = c[j] > 0;
  }
  unsigned ranks[CPL_IPT], total;
  tile_compact_ranks<CP_BLOCK, CPL_IPT>(f, ranks, total, state, epoch, tile, err, sm);
#pragma unroll
  for (int j = 0; j < CPL_IPT; ++j) {
    if (!f[j]) continue;
    const int k = base + j * CP_BLOCK + threadIdx.x;
    const int v = (int)ranks[j];
    long long* sp = dsum + 3 * (size_t)k;
    const long long sx = sp[0], sy = sp[1], sz = sp[2];
    vox_key[v] = k; vox_count[v] = c[j];
    centroids[v] = make_float4(d_centroid_of(sx, c[j]), d_centroid_of(sy, c[j]), d_centroid_of(sz, c[j]), 1.0f);
    did[k] = v;
    dcnt[k] = 0; sp[0] = 0; sp[1] = 0; sp[2] = 0;  // self-cleaning
  }
  if (tile == (int)gridDim.x - 1 && threadIdx.x == 0) st->n_voxels = (int)total;
  tile_end(ctl);
}

// point -> voxel id (and its key, recomputed from the point: cheaper than carrying it through the sorted pass)
__global__ void k_voxel_assign(const float4* __restrict__ pts, VoxState* st, float inv, const int* __restrict__ did, int capacity,
                               int* __restrict__ key_of_point, int* __restrict__ assign) {
  __shared__ VoxLattice L;
  d_vox_lattice(st, inv, &L);
  const int n = st->n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int key = d_vox_key(L, inv, pts[i]);
    key_of_point[i] = key;
    assign[i] = ((unsigned)key < (unsigned)capacity) ? did[key] : -1;
  }
}

// The same point -> (key, voxel id) on demand, for the dense path run without k_voxel_assign: the key from the lattice
// block 0 of k_voxel_accumulate(_sorted) published in *st, the id by a binary search in the ascending voxel keys (not
// from the per-key id table: a later VoxelGrid on the same context, e.g. the compression residual, reuses it).
__global__ void k_voxel_lookup(const float4* __restrict__ pts, const VoxState* __restrict__ st, const int* __restrict__ vox_key,
                               int* __restrict__ key_of_point, int* __restrict__ assign) {
  const int n = st->n, V = st->n_voxels;
  VoxLattice L;
  for (int a = 0; a < 3; ++a) { L.minb[a] = st->min_b[a]; L.mul[a] = st->mul[a]; }
  L.overflow = st->overflow;
  const float inv = st->v_inv;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int key = L.overflow ? i : d_vox_key(L, inv, pts[i]);
    const int v = lower_bound_u32(reinterpret_cast<const unsigned*>(vox_key), V, (unsigned)key);
    key_of_point[i] = key;
    assign[i] = (v < V && vox_key[v] == key) ? v : -1;
  }
}

// After the voxel sort: number the voxels (ascending key), record their first sorted position and
// the voxel rank of every point.
__global__ void __launch_bounds__(CP_BLOCK)
k_voxel_heads(const unsigned* __restrict__ skeys, const unsigned* __restrict__ sidx, int* __restrict__ assign,
              int* __restrict__ vox_start, int* __restrict__ vox_key, unsigned long long* state, TileCtl* ctl, VoxState* st,
              int* err) {
  __shared__ CompactSmem<CP_BLOCK, CPL_IPT> sm;
  const int n = st->n;
  unsigned epoch;
  const int tile = tile_begin(ctl, epoch), base = tile * CPL_TILE;
  if (base >= n) { tile_end(ctl); return; }
  bool f[CPL_IPT];
  unsigned key[CPL_IPT];
#pragma unroll
  for (int j = 0; j < CPL_IPT; ++j) {
    int i = base + j * CP_BLOCK + threadIdx.x;
    f[j] = false; key[j] = 0;
    if (i < n) {
      key[j] = skeys[i];
      f[j] = (i == 0) || (key[j] != skeys[i - 1]);
    }
  }
  unsigned ranks[CPL_IPT], total;
  tile_compact_ranks<CP_BLOCK, CPL_IPT>(f, ranks, total, state, epoch, tile, err, sm);
#pragma unroll
  for (int j = 0; j < CPL_IPT; ++j) {
    int i = base + j * CP_BLOCK + threadIdx.x;
    if (i < n) {
      int id = f[j] ? (int)ranks[j] : (int)ranks[j] - 1;
      assign[sidx[i]] = id;
      if (f[j]) { vox_start[id] = i; vox_key[id] = (int)key[j]; }
    }
  }
  if (base + CPL_TILE >= n && threadIdx.x == 0) st->n_voxels = (int)total;
  tile_end(ctl);
}

// Centroid per voxel (sort-based path): fixed-point sums of the members (same order-independent definition as
// the dense path above), one warp per voxel, lanes stride over the members, shuffle tree for the totals.
constexpr int VC_BLOCK = 128;
__global__ void __launch_bounds__(VC_BLOCK)
k_voxel_centroids(const unsigned* __restrict__ sidx, const float4* __restrict__ pts,
                  const int* __restrict__ vox_start, const VoxState* __restrict__ st,
                  float4* __restrict__ centroids, int* __restrict__ vox_count) {
  const int V = st->n_voxels, n = st->n;
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * VC_BLOCK) >> 5;
  for (int j = (blockIdx.x * VC_BLOCK + threadIdx.x) >> 5; j < V; j += warps_total) {
    const int s = vox_start[j], e = (j + 1 < V) ? vox_start[j + 1] : n;
    long long sx = 0, sy = 0, sz = 0;
    for (int t = s + lane; t < e; t += 32) {
      const float4 q = pts[sidx[t]];
      sx += d_fx20(q.x); sy += d_fx20(q.y); sz += d_fx20(q.z);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sx += __shfl_down_sync(FULL, sx, o); sy += __shfl_down_sync(FULL, sy, o); sz += __shfl_down_sync(FULL, sz, o);
    }
    if (lane == 0) {
      const int c = e - s;
      // overflow rule (A.5): the output is the input cloud unchanged, not a rounded copy of it
      centroids[j] = st->overflow ? pts[sidx[s]] : make_float4(d_centroid_of(sx, c), d_centroid_of(sy, c), d_centroid_of(sz, c), 1.0f);
      vox_count[j] = c;
    }
  }
}

// a4 second half: kdtree->nearestKSearch(centroid, 1) (src/tunnel_processing.cpp:239) as an exact
// expanding search over the neighbour grid of the PRE-compaction cloud (quirk B.3), FLANN
// L2_Simple distance, ties -> lowest original index.  Then normals->at(index) (:247-249).
// mode 0 (reference-faithful): index = pre-compaction index, looked up in the COMPACTED normals;
// index >= n_valid is counted in nn_oor (the reference would throw).  mode 1 (fixed): only points
// that survived compaction are candidates and the index is the compacted one.
// Ring 1 of most voxels by a group of lanes (k_voxel_nn), the rest by a warp: lanes take the x-runs of the cube
// shells as tasks (two popcount lookups + a short scan each), then a lexicographic (d2, index) warp minimum.
constexpr int NN_BLOCK = 128;

__device__ __forceinline__ void d_nn_scan(const float4* __restrict__ sp, const int* __restrict__ valid_map, int mode,
                                          int2 r, const float4 c, float& best, int& bi) {
  for (int t = r.x; t < r.y; ++t) {
    const float4 q = sp[t];
    int id = __float_as_int(q.w);
    if (mode == 1) { id = valid_map[id]; if (id < 0) continue; }
    float dx = c.x - q.x, dy = c.y - q.y, dz = c.z - q.z;
    float d2 = (dx * dx + dy * dy) + dz * dz;
    if (d2 < best || (d2 == best && id < bi)) { best = d2; bi = id; }
  }
}

// scan the cells x0..x1 of row (cy,cz): one segment per 4-cell x-block the span touches
__device__ __forceinline__ void d_nn_scan_row(const float4* __restrict__ sp, const int* __restrict__ valid_map, int mode,
                                              const GridSpec& g, const BlockEntry* __restrict__ tab, const int* __restrict__ ucell_start,
                                              int U, int nf, int x0, int x1, int cy, int cz, const float4 c, float& best, int& bi) {
  if (cy < 0 || cz < 0 || cy >= g.dim[1] || cz >= g.dim[2]) return;
  x0 = max(x0, 0); x1 = min(x1, g.dim[0] - 1);
  for (int xs = x0; xs <= x1;) {
    const int xe = min(x1, xs | 3);
    d_nn_scan(sp, valid_map, mode, cell_segment(g, tab, ucell_start, U, nf, xs, xe, cy, cz), c, best, bi);
    xs = xe + 1;
  }
}

// Rings k0.. of the expanding cube-shell search of one centroid by the whole warp (best / bi: what the rings before k0
// gave, the same on every lane): ring 1 as the 9 rows of the 27-cell cube, ring k >= 2 as 8k perimeter rows with the
// full x span + (2k-1)^2 inner rows with two end cells; after each ring a lexicographic (d2, index) warp minimum.
__device__ __forceinline__ void d_nn_rings(const float4* __restrict__ sp, const int* __restrict__ valid_map, int mode, const GridSpec& g,
                                           const BlockEntry* __restrict__ tab, const int* __restrict__ ucell_start, int U, int nf,
                                           const float4 c, int cx, int cy, int cz, int k0, int kmax, float& best, int& bi) {
  const int lane = threadIdx.x & 31;
  for (int k = k0; k <= kmax; ++k) {
    if (k == 1) {
      if (lane < 9)
        d_nn_scan_row(sp, valid_map, mode, g, tab, ucell_start, U, nf, cx - 1, cx + 1, cy + (lane % 3) - 1, cz + (lane / 3) - 1, c, best, bi);
    } else {
      const int inner = 2 * k - 1, T = 8 * k + 2 * inner * inner;
      for (int t = lane; t < T; t += 32) {
        int dy, dz, x0, x1;
        if (t < 8 * k) {
          if (t < 2 * k + 1) { dz = -k; dy = t - k; }
          else if (t < 4 * k + 2) { dz = k; dy = t - (2 * k + 1) - k; }
          else if (t < 6 * k + 1) { dy = -k; dz = t - (4 * k + 2) - (k - 1); }
          else { dy = k; dz = t - (6 * k + 1) - (k - 1); }
          x0 = cx - k; x1 = cx + k;
        } else {
          int u2 = t - 8 * k, cell = u2 >> 1;
          dy = cell % inner - (k - 1); dz = cell / inner - (k - 1);
          x0 = x1 = (u2 & 1) ? cx + k : cx - k;
        }
        d_nn_scan_row(sp, valid_map, mode, g, tab, ucell_start, U, nf, x0, x1, cy + dy, cz + dz, c, best, bi);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      float ob = __shfl_xor_sync(FULL, best, o);
      int oi = __shfl_xor_sync(FULL, bi, o);
      if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
    }
    // every unexplored cell is at Chebyshev distance >= k+1 from the query cell, hence every
    // point in it is at least k*cell away from the query
    double lim = (double)k * (double)g.cell * 0.999;
    if (bi != 0x7FFFFFFF && (double)best <= lim * lim) break;
  }
}

// Ring 1 of a centroid whose own cell is occupied (nearly all of them) reuses that cell's runs from the normals stage.  A
// group of NN_GROUP lanes takes one centroid (32 / NN_GROUP in flight per warp): the runs' lengths are turned into
// offsets of one flat candidate range by a group scan, lane l takes the candidates l, l + NN_GROUP, ... of it (slices
// cross run boundaries freely: the (d2, index) minimum does not depend on how the candidates are split), NN_BATCH of
// them loaded together, then a group minimum.  Centroids in an empty cell, and those whose ring-1 best is not provably
// the nearest, go on one at a time with the whole warp (d_nn_rings).
constexpr int NN_GROUP = 8;
constexpr int NN_BATCH = 4;

__global__ void __launch_bounds__(NN_BLOCK)
k_voxel_nn(const float4* __restrict__ centroids, const float4* __restrict__ sp,
           const BlockEntry* __restrict__ tab, const int* __restrict__ ucell_start, const int2* __restrict__ runs, const int2* __restrict__ cell_info,
           const int* __restrict__ valid_map, const float4* __restrict__ normals_c, GridSpec g,
           int mode, DevState* st, int* __restrict__ nn_idx, float4* __restrict__ nn_normal) {
  constexpr int G = NN_GROUP, PER_WARP = 32 / G;
  __shared__ int2 s_run[NN_BLOCK / G][GRID_RUNS];  // per group and run of the cell: {run start - flat offset, flat end}
  const int V = st->vox.n_voxels, U = st->n_cells, nf = st->n_sorted_finite, nvalid = st->n_valid;
  const int lane = threadIdx.x & 31, gl = lane & (G - 1);
  const unsigned gmask = ((1u << G) - 1u) << (lane & ~(G - 1));
  int2* const sr = s_run[threadIdx.x / G];
  const int kmax = max(g.dim[0], max(g.dim[1], g.dim[2]));
  const double lim1 = (double)g.cell * 0.999;  // the ring-1 stop of d_nn_rings
  const int warps_total = (gridDim.x * NN_BLOCK) >> 5;
  for (int j0 = ((blockIdx.x * NN_BLOCK + threadIdx.x) >> 5) * PER_WARP; j0 < V; j0 += warps_total * PER_WARP) {  // warp-uniform
    const int j = j0 + lane / G;
    const bool live = j < V;
    float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
    int cx = 0, cy = 0, cz = 0, k0 = kmax + 1;  // k0: the first ring the warp still has to search
    float best = CUDART_INF_F;
    int bi = 0x7FFFFFFF;
    if (live) {
      c = centroids[j];
      gm_cell_of(g, c.x, c.y, c.z, cx, cy, cz);
      const unsigned ckey = gm_cell_key(g, cx, cy, cz);
      const BlockEntry e = tab[ckey >> 6];
      if ((e.mask >> (ckey & 63u)) & 1ull) {
        const int jc = e.first + __popcll(e.mask & ((1ull << (ckey & 63u)) - 1ull));
        // the cell's run slots are loaded together with its run count (slots past the count hold stale values and are
        // masked off): one dependent load less on the way to the candidates
        constexpr int SLOTS = (GRID_RUNS + G - 1) / G;
        const int2* const rp = runs + (size_t)jc * GRID_RUNS;
        int2 run[SLOTS];
#pragma unroll
        for (int i = 0; i < SLOTS; ++i) run[i] = (i * G + gl < GRID_RUNS) ? __ldg(rp + i * G + gl) : make_int2(0, 0);
        const int2 info = cell_info[jc];  // number of runs, number of candidates
        int carry = 0;
#pragma unroll
        for (int i = 0; i < SLOTS; ++i) {
          const int r = i * G + gl;
          const int len = (r < info.x) ? run[i].y - run[i].x : 0;
          int incl = len;
#pragma unroll
          for (int o = 1; o < G; o <<= 1) {
            const int t = __shfl_up_sync(gmask, incl, o, G);
            if (gl >= o) incl += t;
          }
          if (r < info.x) sr[r] = make_int2(run[i].x - (carry + incl - len), carry + incl);
          carry += __shfl_sync(gmask, incl, G - 1, G);
        }
        __syncwarp(gmask);
        int k = 0;
        int2 cur = sr[0];
        for (int f0 = 0; f0 < info.y; f0 += G * NN_BATCH) {
          int pos[NN_BATCH];
#pragma unroll
          for (int u = 0; u < NN_BATCH; ++u) {
            const int f = f0 + u * G + gl;
            pos[u] = -1;
            if (f < info.y) {
              while (f >= cur.y) cur = sr[++k];
              pos[u] = f + cur.x;
            }
          }
          float4 q[NN_BATCH];
          int id[NN_BATCH];
#pragma unroll
          for (int u = 0; u < NN_BATCH; ++u) {
            q[u] = (pos[u] >= 0) ? __ldg(sp + pos[u]) : make_float4(0.f, 0.f, 0.f, 0.f);
            id[u] = __float_as_int(q[u].w);
          }
          if (mode == 1) {
#pragma unroll
            for (int u = 0; u < NN_BATCH; ++u) id[u] = (pos[u] >= 0) ? __ldg(valid_map + id[u]) : -1;
          }
#pragma unroll
          for (int u = 0; u < NN_BATCH; ++u) {
            if (pos[u] < 0 || id[u] < 0) continue;
            float dx = c.x - q[u].x, dy = c.y - q[u].y, dz = c.z - q[u].z;
            float d2 = (dx * dx + dy * dy) + dz * dz;
            if (d2 < best || (d2 == best && id[u] < bi)) { best = d2; bi = id[u]; }
          }
        }
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) {
          float ob = __shfl_xor_sync(gmask, best, o, G);
          int oi = __shfl_xor_sync(gmask, bi, o, G);
          if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
        }
        if (!(bi != 0x7FFFFFFF && (double)best <= lim1 * lim1)) k0 = 2;
        __syncwarp(gmask);  // s_run is rewritten by the group's next centroid
      } else {
        k0 = 1;
      }
    }
    unsigned todo = __ballot_sync(FULL, gl == 0 && k0 <= kmax);
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const float4 cc = make_float4(__shfl_sync(FULL, c.x, src), __shfl_sync(FULL, c.y, src), __shfl_sync(FULL, c.z, src), 0.f);
      float b = __shfl_sync(FULL, best, src);
      int bb = __shfl_sync(FULL, bi, src);
      d_nn_rings(sp, valid_map, mode, g, tab, ucell_start, U, nf, cc, __shfl_sync(FULL, cx, src), __shfl_sync(FULL, cy, src),
                 __shfl_sync(FULL, cz, src), __shfl_sync(FULL, k0, src), kmax, b, bb);
      if (lane == src) { best = b; bi = bb; }
    }
    if (live && gl == 0) {
      if (bi == 0x7FFFFFFF) bi = -1;
      nn_idx[j] = bi;
      const float qnan = CUDART_NAN_F;
      float4 o0 = make_float4(qnan, qnan, qnan, 0.f), o1 = make_float4(qnan, 0.f, 0.f, 0.f);
      if (bi >= 0 && bi < nvalid) { o0 = normals_c[2 * (size_t)bi]; o1 = normals_c[2 * (size_t)bi + 1]; }
      else atomicAdd(&st->nn_oor, 1);
      nn_normal[2 * (size_t)j] = o0;
      nn_normal[2 * (size_t)j + 1] = o1;
    }
  }
}

// ---- cyclic Jacobi, double, symmetric 3x3 -> ascending eigenvalues / column eigenvectors ------
// Stand-in for Eigen::SelfAdjointEigenSolver (src/tunnel_processing.cpp:129; SURVEY A.6).
// Sign convention: largest-|component| of each eigenvector positive.
__device__ void d_jacobi3(const double Ain[9], double vals[3], double vecs[9]) {
  double A[3][3], V[3][3];
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { A[i][j] = Ain[i * 3 + j]; V[i][j] = (i == j) ? 1.0 : 0.0; }
  for (int sweep = 0; sweep < 64; ++sweep) {
    double off = A[0][1] * A[0][1] + A[0][2] * A[0][2] + A[1][2] * A[1][2];
    double diag = A[0][0] * A[0][0] + A[1][1] * A[1][1] + A[2][2] * A[2][2];
    if (off <= 1e-300 || off <= 1e-34 * diag) break;
    for (int p = 0; p < 2; ++p) for (int q = p + 1; q < 3; ++q) {
      if (A[p][q] == 0.0) continue;
      double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
      double t = ((theta >= 0.0) ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
      double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
      for (int k = 0; k < 3; ++k) { double akp = A[k][p], akq = A[k][q]; A[k][p] = c * akp - s * akq; A[k][q] = s * akp + c * akq; }
      for (int k = 0; k < 3; ++k) { double apk = A[p][k], aqk = A[q][k]; A[p][k] = c * apk - s * aqk; A[q][k] = s * apk + c * aqk; }
      for (int k = 0; k < 3; ++k) { double vkp = V[k][p], vkq = V[k][q]; V[k][p] = c * vkp - s * vkq; V[k][q] = s * vkp + c * vkq; }
    }
  }
  int order[3] = {0, 1, 2};
  double d[3] = {A[0][0], A[1][1], A[2][2]};
  // stable insertion sort by eigenvalue
  for (int i = 1; i < 3; ++i) {
    int o = order[i], j = i - 1;
    while (j >= 0 && d[order[j]] > d[o]) { order[j + 1] = order[j]; --j; }
    order[j + 1] = o;
  }
  for (int k = 0; k < 3; ++k) {
    int c = order[k];
    vals[k] = d[c];
    double v[3] = {V[0][c], V[1][c], V[2][c]};
    double n = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
    int big = 0;
    if (fabs(v[1]) > fabs(v[big])) big = 1;
    if (fabs(v[2]) > fabs(v[big])) big = 2;
    double sgn = (v[big] < 0.0) ? -1.0 : 1.0;
    for (int r = 0; r < 3; ++r) vecs[r * 3 + k] = sgn * v[r] / n;
  }
}

// Weight law of getLocalFrame as w = float(exp(sgn * t^2)), t = curv * scale + shift.  Reference (mode 0,
// src/tunnel_processing.cpp:106): scale 1, shift 0.001/wf, sgn +1 -- the weight GROWS with curvature (quirk B.2).
// "Fixed" law (mode 1, builder-defined, SURVEY 8f.2): scale 1/wf, shift 0, sgn -1.
struct WeightLaw { double scale, shift, sgn; };
__device__ __forceinline__ float d_weight(const WeightLaw& w, float curv) {
  const double t = (double)curv * w.scale + w.shift;
  return (float)exp(w.sgn * t * t);
}

// a5 getLocalFrame (src/tunnel_processing.cpp:92-148), diagonal form of the dense weights*normals
// product.  w_i = float(exp((double(curv_i) + 0.001/wf)^2)); Wn = w_i*n_i in float; the 3x3
// scatter sum is accumulated in double (fixed grid, fixed tree -> reproducible); the last block to
// finish sums the per-block partials in block order and runs the eigen solve.
constexpr int FR_BLOCK = 256;
struct FrameOut { float vals[3]; float vecs[9]; float scatter[9]; };

// 6 double sums (xx xy xz yy yz zz) -> float scatter matrix (the reference's is float), eigen-decomposition
__device__ __forceinline__ void d_frame_solve(const double* fin, FrameOut* out) {
  float Sf[9] = {(float)fin[0], (float)fin[1], (float)fin[2], (float)fin[1], (float)fin[3], (float)fin[4], (float)fin[2], (float)fin[4], (float)fin[5]};
  double Sd[9], vals[3], vecs[9];
  for (int k = 0; k < 9; ++k) { Sd[k] = Sf[k]; out->scatter[k] = Sf[k]; }
  d_jacobi3(Sd, vals, vecs);
  for (int k = 0; k < 3; ++k) out->vals[k] = (float)vals[k];
  for (int k = 0; k < 9; ++k) out->vecs[k] = (float)vecs[k];
}

__global__ void __launch_bounds__(FR_BLOCK)
k_frame(const float4* __restrict__ normals_c, const int* __restrict__ n_ptr, WeightLaw law, double* __restrict__ partials,
        unsigned* counter, FrameOut* out, double* __restrict__ sums_out /* [6] the double sums, for gm_allreduce_frame */) {
  __shared__ double sm[6 * (FR_BLOCK / 32)];
  __shared__ double fin[6];
  const int n = *n_ptr;
  double s[6] = {0, 0, 0, 0, 0, 0};
  for (int i = blockIdx.x * FR_BLOCK + threadIdx.x; i < n; i += gridDim.x * FR_BLOCK) {
    float4 n0 = normals_c[2 * (size_t)i];
    float curv = normals_c[2 * (size_t)i + 1].x;
    float w = d_weight(law, curv);
    float a = w * n0.x, b = w * n0.y, c = w * n0.z;
    s[0] += (double)a * (double)a; s[1] += (double)a * (double)b; s[2] += (double)a * (double)c;
    s[3] += (double)b * (double)b; s[4] += (double)b * (double)c; s[5] += (double)c * (double)c;
  }
  block_sum_store<6, FR_BLOCK>(s, sm, partials + (size_t)blockIdx.x * 6);
  if (!d_last_block(counter, gridDim.x)) return;
  d_reduce_partials<6>(partials, gridDim.x, fin);
  if (threadIdx.x != 0) return;
  for (int k = 0; k < 6; ++k) sums_out[k] = fin[k];
  d_frame_solve(fin, out);
}

// the frame of the SUM of the scatter matrices of several contexts / ranks (map slabs): same solve, other sums
__global__ void k_frame_solve(const double* __restrict__ sums6, FrameOut* out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) d_frame_solve(sums6, out);
}

}  // namespace gm
