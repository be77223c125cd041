// gm_map.cuh — aggregated voxel map across scans (SURVEY.md section 8f.3, builder-defined: the reference
// processes every scan on its own, src/geometric_mapping.cpp:48-125, and keeps nothing).
// An open-addressing hash table keyed by the GLOBAL voxel index floor(p * inv_leaf) (the VoxelGrid
// cell of pcl::VoxelGrid, independent of any bounding box), holding per voxel the point count and the
// coordinate sums in 2^-20 m fixed point.  Integer atomics are associative, so the map does not depend
// on the order in which scans, blocks or threads arrive: bitwise reproducible, and two maps built from
// the same scans in a different order are identical.
#pragma once
#include "gm_stages.cuh"

namespace gm {

constexpr unsigned long long MAP_EMPTY = 0xFFFFFFFFFFFFFFFFull;
constexpr int MAP_COORD_BITS = 21;                 // +-2^20 voxels per axis
constexpr int MAP_COORD_OFF = 1 << 20;
constexpr float MAP_FX = GM_FX20;                  // 2^20: exact scaling of a float (same fixed point as the VoxelGrid centroids)

struct MapState { unsigned long long n_points; int n_voxels; int overflow; int out_of_range; int pad_; };

__host__ __device__ __forceinline__ unsigned long long map_hash(unsigned long long k) {  // splitmix64 finaliser
  k ^= k >> 30; k *= 0xBF58476D1CE4E5B9ull;
  k ^= k >> 27; k *= 0x94D049BB133111EBull;
  k ^= k >> 31;
  return k;
}
__host__ __device__ __forceinline__ bool map_pack(int ix, int iy, int iz, unsigned long long& key) {
  const int lim = MAP_COORD_OFF;
  if (ix < -lim || ix >= lim || iy < -lim || iy >= lim || iz < -lim || iz >= lim) return false;
  key = (unsigned long long)(unsigned)(ix + lim) | ((unsigned long long)(unsigned)(iy + lim) << MAP_COORD_BITS) |
        ((unsigned long long)(unsigned)(iz + lim) << (2 * MAP_COORD_BITS));
  return true;
}
__host__ __device__ __forceinline__ void map_unpack(unsigned long long key, int& ix, int& iy, int& iz) {
  const unsigned long long m = (1ull << MAP_COORD_BITS) - 1ull;
  ix = (int)(key & m) - MAP_COORD_OFF;
  iy = (int)((key >> MAP_COORD_BITS) & m) - MAP_COORD_OFF;
  iz = (int)((key >> (2 * MAP_COORD_BITS)) & m) - MAP_COORD_OFF;
}

struct Pose34 { float r[12]; };  // row-major [R | t]

// Insert the points pts[0..n) (optionally only those with labels[i] == label_filter) after the rigid
// transform p' = R p + t, evaluated as fmaf chains (bit-identical to the oracle's std::fmaf).
__device__ __forceinline__ void d_map_insert(const float4* __restrict__ pts, const unsigned char* __restrict__ labels, const int n,
                                             int label_filter, const Pose34& T, int use_pose, float inv_leaf,
                                             unsigned long long* __restrict__ keys, int* __restrict__ cnt, long long* __restrict__ sums,
                                             unsigned long long slot_mask, MapState* st) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (label_filter >= 0 && labels[i] != (unsigned char)label_filter) continue;
    const float4 p = pts[i];
    float x = p.x, y = p.y, z = p.z;
    if (use_pose) {
      x = fmaf(T.r[0], p.x, fmaf(T.r[1], p.y, fmaf(T.r[2], p.z, T.r[3])));
      y = fmaf(T.r[4], p.x, fmaf(T.r[5], p.y, fmaf(T.r[6], p.z, T.r[7])));
      z = fmaf(T.r[8], p.x, fmaf(T.r[9], p.y, fmaf(T.r[10], p.z, T.r[11])));
    }
    if (!finite3(x, y, z)) { atomicAdd(&st->out_of_range, 1); continue; }
    const float fx = floorf(x * inv_leaf), fy = floorf(y * inv_leaf), fz = floorf(z * inv_leaf);
    unsigned long long key;
    if (!(fabsf(fx) < 2.0e6f && fabsf(fy) < 2.0e6f && fabsf(fz) < 2.0e6f) || !map_pack((int)fx, (int)fy, (int)fz, key)) {
      atomicAdd(&st->out_of_range, 1);
      continue;
    }
    unsigned long long slot = map_hash(key) & slot_mask;
    bool placed = false;
    for (unsigned long long probe = 0; probe <= slot_mask; ++probe) {
      unsigned long long prev = keys[slot];
      if (prev == MAP_EMPTY) {
        prev = atomicCAS(&keys[slot], MAP_EMPTY, key);
        if (prev == MAP_EMPTY) { atomicAdd(&st->n_voxels, 1); prev = key; }
      }
      if (prev == key) { placed = true; break; }
      slot = (slot + 1) & slot_mask;
    }
    if (!placed) { atomicExch(&st->overflow, 1); continue; }
    atomicAdd(&cnt[slot], 1);
    // x * 2^20 is exact in float (power-of-two scaling); llrintf rounds it to the nearest integer
    atomicAdd(reinterpret_cast<unsigned long long*>(sums) + 3 * slot + 0, (unsigned long long)__float2ll_rn(x * MAP_FX));
    atomicAdd(reinterpret_cast<unsigned long long*>(sums) + 3 * slot + 1, (unsigned long long)__float2ll_rn(y * MAP_FX));
    atomicAdd(reinterpret_cast<unsigned long long*>(sums) + 3 * slot + 2, (unsigned long long)__float2ll_rn(z * MAP_FX));
    atomicAdd(&st->n_points, 1ull);
  }
}

__global__ void k_map_insert(const float4* __restrict__ pts, const unsigned char* __restrict__ labels, const int* __restrict__ n_ptr,
                             int label_filter, Pose34 T, int use_pose, float inv_leaf, unsigned long long* __restrict__ keys,
                             int* __restrict__ cnt, long long* __restrict__ sums /* 3 per slot */, unsigned long long slot_mask,
                             MapState* st) {
  d_map_insert(pts, labels, *n_ptr, label_filter, T, use_pose, inv_leaf, keys, cnt, sums, slot_mask, st);
}

// k_map_insert of every point at a pose the device decided (gm_odometry_step): pose and go/no-go flag are read from
// device memory, and a flag of 0 inserts nothing.
__global__ void k_map_insert_gated(const float4* __restrict__ pts, const int* __restrict__ n_ptr, const Pose34* __restrict__ pose,
                                   const int* __restrict__ accept, float inv_leaf, unsigned long long* __restrict__ keys,
                                   int* __restrict__ cnt, long long* __restrict__ sums, unsigned long long slot_mask, MapState* st) {
  if (!*accept) return;
  const Pose34 T = *pose;
  d_map_insert(pts, nullptr, *n_ptr, -1, T, 1, inv_leaf, keys, cnt, sums, slot_mask, st);
}

// Add one voxel (key, count, fixed-point sums s3[0..3)) to the table: the entry of `key`, created if absent, gets the
// count and the sums added as integers.  A full table drops the voxel and raises overflow.  Shared by gm_map_load,
// gm_map_evict (the archive, and the kept voxels' re-insertion) and gm_map_merge, so all of them add alike.
__device__ __forceinline__ void d_map_add(unsigned long long key, int c, const long long* __restrict__ s3, unsigned long long* __restrict__ keys,
                                          int* __restrict__ cnt, long long* __restrict__ sums, unsigned long long slot_mask, MapState* st) {
  unsigned long long slot = map_hash(key) & slot_mask;
  bool placed = false;
  for (unsigned long long probe = 0; probe <= slot_mask; ++probe) {
    unsigned long long prev = atomicCAS(&keys[slot], MAP_EMPTY, key);
    if (prev == MAP_EMPTY) { atomicAdd(&st->n_voxels, 1); prev = key; }
    if (prev == key) { placed = true; break; }
    slot = (slot + 1) & slot_mask;
  }
  if (!placed) { atomicExch(&st->overflow, 1); return; }
  atomicAdd(&cnt[slot], c);
  for (int a = 0; a < 3; ++a) atomicAdd(reinterpret_cast<unsigned long long*>(sums) + 3 * slot + a, (unsigned long long)s3[a]);
  atomicAdd(&st->n_points, (unsigned long long)c);
}

// ---- window eviction (gm_map_evict) and merge (gm_map_merge) ----------------------------------------------------------
// Linear probing has no parallel delete, so an eviction rebuilds the table: k_map_evict_split adds the evicted voxels to
// the archive and compacts the kept ones into the map's scratch arrays, k_map_evict_clear empties the table and
// k_map_restore re-adds the kept voxels.  The last two return at once when nothing was evicted.

struct MapEvictState { int n_kept; int evicted; };  // zeroed before every eviction

// Add n dense voxels (key, count and fixed-point sums as stored) to the table: the saved voxels of gm_map_load (es null),
// or the kept voxels of an eviction (n = es->n_kept) if es->evicted, which re-adds them to the emptied table and so
// recounts n_voxels and n_points.  Kept voxels are at most the voxels the table held, so they all fit.
__global__ void k_map_restore(const unsigned long long* __restrict__ in_keys, const int* __restrict__ in_cnt,
                              const long long* __restrict__ in_sums, int n, const MapEvictState* __restrict__ es,
                              unsigned long long* __restrict__ keys, int* __restrict__ cnt, long long* __restrict__ sums,
                              unsigned long long slot_mask, MapState* st) {
  if (es) {
    if (!es->evicted) return;
    n = es->n_kept;
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    d_map_add(in_keys[i], in_cnt[i], in_sums + 3 * (size_t)i, keys, cnt, sums, slot_mask, st);
}

// The window's centre cell, c[a] = (int)floorf(center[a] * inv_leaf) as d_map_insert computes a point's cell.  false for a
// non-finite centre or a cell outside the key range.  Host and device evaluate the same float product and floorf.
__host__ __device__ __forceinline__ bool map_center_cell(const float c3[3], float inv_leaf, long long cell[3]) {
  for (int a = 0; a < 3; ++a) {
    const float f = floorf(c3[a] * inv_leaf);
    if (!(fabsf(f) < 2.0e6f)) return false;  // NaN and infinities too
    cell[a] = (long long)(int)f;
    if (cell[a] < -MAP_COORD_OFF || cell[a] >= MAP_COORD_OFF) return false;
  }
  return true;
}

// One thread per slot.  Centre = (cx, cy, cz), or the translation (pose34[3], pose34[7], pose34[11]) of a device pose when
// pose34 is not null (gm_odometry_step: the step's recorded pose); a centre map_center_cell refuses evicts nothing.  A voxel
// is kept iff max_a |cell_a - c_a| <= half_cells (64-bit integers).  Kept voxels go to out_* in any order (warp-aggregated
// cursor es->n_kept); evicted ones are added to the archive (a_keys null: dropped) and set es->evicted.  Every lane of a warp
// runs the same number of iterations (n_slots and the stride are multiples of 32), so the ballots see full warps.
__global__ void k_map_evict_split(const unsigned long long* __restrict__ keys, const int* __restrict__ cnt, const long long* __restrict__ sums,
                                  unsigned long long slot_mask, float inv_leaf, float cx, float cy, float cz, const float* __restrict__ pose34,
                                  int half_cells, unsigned long long* __restrict__ a_keys, int* __restrict__ a_cnt, long long* __restrict__ a_sums,
                                  unsigned long long a_mask, MapState* a_st, unsigned long long* __restrict__ out_keys, int* __restrict__ out_cnt,
                                  long long* __restrict__ out_sums, MapEvictState* es) {
  float c3[3] = {cx, cy, cz};
  if (pose34) { c3[0] = pose34[3]; c3[1] = pose34[7]; c3[2] = pose34[11]; }
  long long c[3];
  if (!map_center_cell(c3, inv_leaf, c)) return;
  const int lane = threadIdx.x & 31;
  bool gone_any = false;
  for (unsigned long long s = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; s <= slot_mask;
       s += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long key = keys[s];
    bool kept = false, gone = false;
    if (key != MAP_EMPTY) {
      int ix, iy, iz;
      map_unpack(key, ix, iy, iz);
      const long long d = max(llabs((long long)ix - c[0]), max(llabs((long long)iy - c[1]), llabs((long long)iz - c[2])));
      kept = d <= (long long)half_cells;
      gone = !kept;
    }
    const unsigned m = __ballot_sync(0xFFFFFFFFu, kept);
    int base = 0;
    if (lane == 0 && m) base = atomicAdd(&es->n_kept, __popc(m));
    base = __shfl_sync(0xFFFFFFFFu, base, 0);
    if (kept) {
      const int o = base + __popc(m & ((1u << lane) - 1u));
      out_keys[o] = key;
      out_cnt[o] = cnt[s];
      for (int a = 0; a < 3; ++a) out_sums[3 * (size_t)o + a] = sums[3 * s + a];
    }
    if (gone) {
      gone_any = true;
      if (a_keys) d_map_add(key, cnt[s], sums + 3 * s, a_keys, a_cnt, a_sums, a_mask, a_st);
    }
  }
  if (__any_sync(0xFFFFFFFFu, gone_any) && lane == 0) es->evicted = 1;
}

// Empty every slot and zero n_voxels and n_points (overflow and out_of_range stay), if anything was evicted.
__global__ void k_map_evict_clear(unsigned long long* __restrict__ keys, int* __restrict__ cnt, long long* __restrict__ sums,
                                  unsigned long long n_slots, const MapEvictState* __restrict__ es, MapState* st) {
  if (!es->evicted) return;
  if (blockIdx.x == 0 && threadIdx.x == 0) { st->n_voxels = 0; st->n_points = 0ull; }
  for (unsigned long long s = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; s < n_slots; s += (unsigned long long)gridDim.x * blockDim.x) {
    keys[s] = MAP_EMPTY;
    cnt[s] = 0;
  }
  for (unsigned long long s = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; s < 3 * n_slots; s += (unsigned long long)gridDim.x * blockDim.x)
    sums[s] = 0;
}

// dst += src: every occupied slot of src added to dst (gm_map_merge).
__global__ void k_map_merge(const unsigned long long* __restrict__ s_keys, const int* __restrict__ s_cnt, const long long* __restrict__ s_sums,
                            unsigned long long s_slots, unsigned long long* __restrict__ keys, int* __restrict__ cnt, long long* __restrict__ sums,
                            unsigned long long slot_mask, MapState* st) {
  for (unsigned long long s = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; s < s_slots; s += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long key = s_keys[s];
    if (key != MAP_EMPTY) d_map_add(key, s_cnt[s], s_sums + 3 * s, keys, cnt, sums, slot_mask, st);
  }
}

// Slot of `key`, or -1.  Keys are never removed, so the probe sequence of an absent key ends at an empty slot (or after
// n_slots probes in a full table).
__device__ __forceinline__ long long d_map_find(const unsigned long long* __restrict__ keys, unsigned long long key,
                                                unsigned long long slot_mask) {
  unsigned long long slot = map_hash(key) & slot_mask;
  for (unsigned long long probe = 0; probe <= slot_mask; ++probe) {
    const unsigned long long k = keys[slot];
    if (k == key) return (long long)slot;
    if (k == MAP_EMPTY) return -1;
    slot = (slot + 1) & slot_mask;
  }
  return -1;
}

constexpr int MAP_PLANE_MIN_VOXELS = 5;  // GM_MAP_PLANE_MIN_VOXELS

// centroid of an occupied slot exactly as gm_map_download reports it: float(sum / 2^20 / count) in double
__device__ __forceinline__ void d_map_centroid(const int* __restrict__ cnt, const long long* __restrict__ sums, long long s, float c[3]) {
  const double n = (double)cnt[s];
#pragma unroll
  for (int a = 0; a < 3; ++a) c[a] = (float)((double)sums[3 * s + a] / 1048576.0 / n);
}

// Plane of every occupied voxel v (include/gm_capi.h, gm_register_map): the centroids of the occupied voxels among the
// 27 around v, v included, in ascending (dz, dy, dx) order; their sequential double mean and covariance; d_jacobi3.
// One thread per slot.  cent[s] = {centroid, 1 if v has a plane else 0}, nrm[s] = {normal, 1} or {NaN x3, 0}; empty slots
// are not written (the search only reads slots d_map_find returns).  box = the cells of the voxels with a plane, as
// atomicMin of {min x, y, z, -, -max x, y, z, -}: the caller sets its 8 ints to 0x7F7F7F7F (larger than any cell) first.
__global__ void k_map_planes(const unsigned long long* __restrict__ keys, const int* __restrict__ cnt, const long long* __restrict__ sums,
                             unsigned long long slot_mask, double max_planarity, float4* __restrict__ cent, float4* __restrict__ nrm,
                             int* __restrict__ box) {
  int bmin[3] = {INT_MAX, INT_MAX, INT_MAX}, bneg[3] = {INT_MAX, INT_MAX, INT_MAX};
  for (unsigned long long s = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; s <= slot_mask;
       s += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long key = keys[s];
    if (key == MAP_EMPTY) continue;
    int ix, iy, iz;
    map_unpack(key, ix, iy, iz);
    float nb[27][3];
    int m = 0;
#pragma unroll 1
    for (int o = 0; o < 27; ++o) {
      unsigned long long k2;
      if (!map_pack(ix + o % 3 - 1, iy + (o / 3) % 3 - 1, iz + o / 9 - 1, k2)) continue;
      const long long s2 = (k2 == key) ? (long long)s : d_map_find(keys, k2, slot_mask);
      if (s2 < 0) continue;
      d_map_centroid(cnt, sums, s2, nb[m]);
      ++m;
    }
    float self[3];
    d_map_centroid(cnt, sums, (long long)s, self);
    float4 n4 = make_float4(CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, 0.f);
    if (m >= MAP_PLANE_MIN_VOXELS) {
      double mu[3] = {0.0, 0.0, 0.0};
#pragma unroll 1
      for (int i = 0; i < m; ++i)
        for (int a = 0; a < 3; ++a) mu[a] += (double)nb[i][a];
      for (int a = 0; a < 3; ++a) mu[a] /= (double)m;
      double c6[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};  // xx xy xz yy yz zz
#pragma unroll 1
      for (int i = 0; i < m; ++i) {
        const double dx = (double)nb[i][0] - mu[0], dy = (double)nb[i][1] - mu[1], dz = (double)nb[i][2] - mu[2];
        c6[0] += dx * dx; c6[1] += dx * dy; c6[2] += dx * dz;
        c6[3] += dy * dy; c6[4] += dy * dz; c6[5] += dz * dz;
      }
      for (int k = 0; k < 6; ++k) c6[k] /= (double)m;
      const double C[9] = {c6[0], c6[1], c6[2], c6[1], c6[3], c6[4], c6[2], c6[4], c6[5]};
      double vals[3], vecs[9];
      d_jacobi3(C, vals, vecs);
      if (vals[0] <= max_planarity * vals[1] && vals[1] > 0.0) n4 = make_float4((float)vecs[0], (float)vecs[3], (float)vecs[6], 1.f);
    }
    cent[s] = make_float4(self[0], self[1], self[2], n4.w);
    nrm[s] = n4;
    if (n4.w != 0.f) {
      bmin[0] = min(bmin[0], ix); bmin[1] = min(bmin[1], iy); bmin[2] = min(bmin[2], iz);
      bneg[0] = min(bneg[0], -ix); bneg[1] = min(bneg[1], -iy); bneg[2] = min(bneg[2], -iz);
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    bmin[a] = __reduce_min_sync(0xFFFFFFFFu, bmin[a]);
    bneg[a] = __reduce_min_sync(0xFFFFFFFFu, bneg[a]);
  }
  if ((threadIdx.x & 31) == 0 && bmin[0] != INT_MAX) {
#pragma unroll
    for (int a = 0; a < 3; ++a) { atomicMin(box + a, bmin[a]); atomicMin(box + 4 + a, bneg[a]); }
  }
}

// Gather the occupied slots into dense arrays (order = slot order; the host sorts by key): the key, and the count, the
// sums and the plane normal of k_map_planes into those of out_cnt, out_sums and out_nrm that are not null.
__global__ void k_map_export(const unsigned long long* __restrict__ keys, const int* __restrict__ cnt, const long long* __restrict__ sums,
                             const float4* __restrict__ nrm, unsigned long long n_slots, unsigned long long* __restrict__ out_keys,
                             int* __restrict__ out_cnt, long long* __restrict__ out_sums, float4* __restrict__ out_nrm, int capacity, int* cursor) {
  for (unsigned long long s = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; s < n_slots; s += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long k = keys[s];
    if (k == MAP_EMPTY) continue;
    const int o = atomicAdd(cursor, 1);
    if (o >= capacity) continue;
    out_keys[o] = k;
    if (out_cnt) out_cnt[o] = cnt[s];
    if (out_sums)
      for (int a = 0; a < 3; ++a) out_sums[3 * (size_t)o + a] = sums[3 * s + a];
    if (out_nrm) out_nrm[o] = nrm[s];
  }
}

}  // namespace gm
