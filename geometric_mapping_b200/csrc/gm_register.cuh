// gm_register.cuh — scan-to-scan registration (builder-defined: the reference computes no pose, every scan is
// processed in its own sensor frame, src/geometric_mapping.cpp:48-125).  Point-to-plane ICP of a source context's
// VoxelGrid centroids against a target context's compacted cloud and normals, the correspondences searched over the
// target's neighbour grid.  One launch per iteration and no host synchronisation between them: the pose lives on the
// device in double, and the last block of every iteration reduces, solves, updates it and decides whether to stop.
// Scan-to-map registration (k_regmap_iter) shares all of it but the search: the nearest plane of the aggregated voxel map
// (k_map_planes, gm_map.cuh) through the map's hash table.
// Semantics: include/gm_capi.h (gm_register, gm_register_map).
#pragma once
#include "gm_stages.cuh"
#include "gm_map.cuh"

namespace gm {

constexpr int REG_BLOCK = 128;
// per-block double partials: A = sum J J^T (21, upper triangle row-major), g = sum J r (6), sum r^2, m
constexpr int REG_NV = 29;

struct RegState {
  double T[12];                  // current pose source -> target, row-major [R|t]
  double eig[6], vecs[36];       // spectrum of the last executed iteration (ascending; column k = eigenvector k)
  double sum_r2;                 // sum of r^2 of the last executed iteration
  int done;                      // later iterations are no-ops
  int iterations, converged, n_corr, n_source, n_degenerate;
};

struct RegParams {
  double d_max;
  float r2max;                   // float(d_max * d_max), the product in double (radius-search convention)
  double min_rot, min_trans, ratio;
};

// T_0 = double(init) and a cleared result: the start of every registration (k_reg_begin, k_odom_begin).  One thread.
__device__ __forceinline__ void d_reg_start(RegState* st, const float init[12], const int* __restrict__ n_source) {
  for (int k = 0; k < 12; ++k) st->T[k] = (double)init[k];
  for (int k = 0; k < 6; ++k) st->eig[k] = 0.0;
  for (int k = 0; k < 36; ++k) st->vecs[k] = 0.0;
  st->sum_r2 = 0.0;
  st->done = 0; st->iterations = 0; st->converged = 0; st->n_corr = 0; st->n_degenerate = 0;
  st->n_source = *n_source;
}

__global__ void k_reg_begin(RegState* st, Pose34 init, const int* __restrict__ n_source) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  d_reg_start(st, init.r, n_source);
}

// Exact nearest compacted target point of c (FLANN L2_Simple, ties -> lowest compacted index), or none when it is not
// nearer than d_max: the expanding cube-shell search of k_voxel_nn (mode 1), one warp per query, with one more stop.
// After shell k every unexplored cell is at Chebyshev distance >= k+1 from the query cell.  On an axis where neither
// the query nor the point was clamped into a border cell that puts the point at least k*cell away; where one of them
// was clamped it lies beyond that border, on the far side from the other, so the gap only grows.  The bound therefore
// also holds for queries far outside the grid box: once k*cell*0.999 >= d_max nothing unexplored can be accepted.
__device__ __forceinline__ void d_reg_nn(const float4 c, const float4* __restrict__ sp, const BlockEntry* __restrict__ tab,
                                         const int* __restrict__ ucell_start, const int2* __restrict__ runs,
                                         const int2* __restrict__ cell_info, const int* __restrict__ valid_map, const GridSpec& g,
                                         int U, int nf, double d_max, float& best, int& bi) {
  const int lane = threadIdx.x & 31;
  int cx, cy, cz;
  gm_cell_of(g, c.x, c.y, c.z, cx, cy, cz);
  best = CUDART_INF_F;
  bi = 0x7FFFFFFF;
  const int kmax = max(g.dim[0], max(g.dim[1], g.dim[2]));
  for (int k = 1; k <= kmax; ++k) {
    if (k == 1) {
      const unsigned ckey = gm_cell_key(g, cx, cy, cz);
      const BlockEntry e = tab[ckey >> 6];
      if ((e.mask >> (ckey & 63u)) & 1ull) {
        const int jc = e.first + __popcll(e.mask & ((1ull << (ckey & 63u)) - 1ull));
        const int nr = cell_info[jc].x;
        for (int r0 = 0; r0 < nr; r0 += 16) {
          const int r = r0 + (lane & 15);
          if (r < nr) {
            const int2 run = runs[(size_t)jc * GRID_RUNS + r];
            const int mid = run.x + ((run.y - run.x + 1) >> 1);
            d_nn_scan(sp, valid_map, 1, (lane < 16) ? make_int2(run.x, mid) : make_int2(mid, run.y), c, best, bi);
          }
        }
      } else if (lane < 9) {
        d_nn_scan_row(sp, valid_map, 1, g, tab, ucell_start, U, nf, cx - 1, cx + 1, cy + (lane % 3) - 1, cz + (lane / 3) - 1, c, best, bi);
      }
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
        d_nn_scan_row(sp, valid_map, 1, g, tab, ucell_start, U, nf, x0, x1, cy + dy, cz + dz, c, best, bi);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      float ob = __shfl_xor_sync(FULL, best, o);
      int oi = __shfl_xor_sync(FULL, bi, o);
      if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
    }
    const double lim = (double)k * (double)g.cell * 0.999;
    if (bi != 0x7FFFFFFF && (double)best <= lim * lim) break;
    if (lim >= d_max) break;
  }
}

// ---- cyclic Jacobi, double, symmetric 6x6: d_jacobi3 generalised (same rotation formulas, stop test, ascending stable
// order, unit columns with their largest-|component| positive).  One thread; the loops stay rolled so that the arrays
// live in the (L1-cached) stack frame instead of inflating the register count of the search.
__device__ __forceinline__ void d_jacobi6(const double Ain[36], double vals[6], double vecs[36]) {
  double A[6][6], V[6][6];
#pragma unroll 1
  for (int i = 0; i < 6; ++i)
#pragma unroll 1
    for (int j = 0; j < 6; ++j) { A[i][j] = Ain[i * 6 + j]; V[i][j] = (i == j) ? 1.0 : 0.0; }
#pragma unroll 1
  for (int sweep = 0; sweep < 64; ++sweep) {
    double off = 0.0, diag = 0.0;
#pragma unroll 1
    for (int p = 0; p < 5; ++p)
#pragma unroll 1
      for (int q = p + 1; q < 6; ++q) off += A[p][q] * A[p][q];
#pragma unroll 1
    for (int i = 0; i < 6; ++i) diag += A[i][i] * A[i][i];
    if (off <= 1e-300 || off <= 1e-34 * diag) break;
#pragma unroll 1
    for (int p = 0; p < 5; ++p)
#pragma unroll 1
      for (int q = p + 1; q < 6; ++q) {
        if (A[p][q] == 0.0) continue;
        double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
        double t = ((theta >= 0.0) ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll 1
        for (int k = 0; k < 6; ++k) { double akp = A[k][p], akq = A[k][q]; A[k][p] = c * akp - s * akq; A[k][q] = s * akp + c * akq; }
#pragma unroll 1
        for (int k = 0; k < 6; ++k) { double apk = A[p][k], aqk = A[q][k]; A[p][k] = c * apk - s * aqk; A[q][k] = s * apk + c * aqk; }
#pragma unroll 1
        for (int k = 0; k < 6; ++k) { double vkp = V[k][p], vkq = V[k][q]; V[k][p] = c * vkp - s * vkq; V[k][q] = s * vkp + c * vkq; }
      }
  }
  int order[6] = {0, 1, 2, 3, 4, 5};
  double d[6];
#pragma unroll 1
  for (int i = 0; i < 6; ++i) d[i] = A[i][i];
#pragma unroll 1
  for (int i = 1; i < 6; ++i) {
    int o = order[i], j = i - 1;
    while (j >= 0 && d[order[j]] > d[o]) { order[j + 1] = order[j]; --j; }
    order[j + 1] = o;
  }
#pragma unroll 1
  for (int k = 0; k < 6; ++k) {
    const int c = order[k];
    vals[k] = d[c];
    double n2 = 0.0;
    int big = 0;
#pragma unroll 1
    for (int r = 0; r < 6; ++r) {
      n2 += V[r][c] * V[r][c];
      if (fabs(V[r][c]) > fabs(V[big][c])) big = r;
    }
    const double n = sqrt(n2), sgn = (V[big][c] < 0.0) ? -1.0 : 1.0;
#pragma unroll 1
    for (int r = 0; r < 6; ++r) vecs[r * 6 + k] = sgn * V[r][c] / n;
  }
}

// R(w) = I + a [w]x + b [w]x^2, a = sin(th)/th, b = (1 - cos th)/th^2 = 2 sin^2(th/2)/th^2 (series below 1e-6 rad)
__device__ __forceinline__ void d_rodrigues(const double w[3], double R[9]) {
  const double th2 = (w[0] * w[0] + w[1] * w[1]) + w[2] * w[2];
  const double th = sqrt(th2);
  double a, b;
  if (th < 1e-6) { a = 1.0 - th2 / 6.0; b = 0.5 - th2 / 24.0; }
  else { const double s = sin(0.5 * th); a = sin(th) / th; b = 2.0 * s * s / th2; }
  const double K[9] = {0.0, -w[2], w[1], w[2], 0.0, -w[0], -w[1], w[0], 0.0};
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) R[i * 3 + j] = ((i == j) ? 1.0 : 0.0) + a * K[i * 3 + j] + b * (w[i] * w[j] - ((i == j) ? th2 : 0.0));
}

// Last block, one thread: spectrum, truncated Gauss-Newton step, pose update, stop decision.
__device__ __forceinline__ void d_reg_solve(const double* fin, const RegParams& prm, RegState* st) {
  double A[36], g[6];
  for (int a = 0, k = 0; a < 6; ++a)
    for (int b = a; b < 6; ++b, ++k) { A[a * 6 + b] = fin[k]; A[b * 6 + a] = fin[k]; }
  for (int a = 0; a < 6; ++a) g[a] = fin[21 + a];
  const int m = (int)fin[28];
  double vals[6], vecs[36];
  d_jacobi6(A, vals, vecs);
  const double lmax = vals[5];
  double xi[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  int ndeg = 0;
  for (int k = 0; k < 6; ++k) {
    if (!(vals[k] > prm.ratio * lmax)) { ++ndeg; continue; }
    double dot = 0.0;
    for (int i = 0; i < 6; ++i) dot += vecs[i * 6 + k] * g[i];
    const double coef = dot / vals[k];
    for (int i = 0; i < 6; ++i) xi[i] -= coef * vecs[i * 6 + k];
  }
  for (int k = 0; k < 6; ++k) st->eig[k] = vals[k];
  for (int k = 0; k < 36; ++k) st->vecs[k] = vecs[k];
  st->sum_r2 = fin[27];
  st->n_corr = m;
  st->n_degenerate = ndeg;
  st->iterations += 1;
  if (m < 6 || !(lmax > 0.0)) { st->converged = 0; st->done = 1; return; }
  double R[9];
  d_rodrigues(xi, R);
  double T[12];
  for (int k = 0; k < 12; ++k) T[k] = st->T[k];
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) st->T[i * 4 + j] = (R[i * 3 + 0] * T[j] + R[i * 3 + 1] * T[4 + j]) + R[i * 3 + 2] * T[8 + j];
    st->T[i * 4 + 3] = ((R[i * 3 + 0] * T[3] + R[i * 3 + 1] * T[7]) + R[i * 3 + 2] * T[11]) + xi[3 + i];
  }
  const double wn = sqrt((xi[0] * xi[0] + xi[1] * xi[1]) + xi[2] * xi[2]);
  const double vn = sqrt((xi[3] * xi[3] + xi[4] * xi[4]) + xi[5] * xi[5]);
  if (wn < prm.min_rot && vn < prm.min_trans) { st->converged = 1; st->done = 1; }
}

// p = float(T)·c as the fmaf chains of k_map_insert
__device__ __forceinline__ float4 d_reg_transform(const float Tf[12], const float4 c) {
  float4 p;
  p.x = fmaf(Tf[0], c.x, fmaf(Tf[1], c.y, fmaf(Tf[2], c.z, Tf[3])));
  p.y = fmaf(Tf[4], c.x, fmaf(Tf[5], c.y, fmaf(Tf[6], c.z, Tf[7])));
  p.z = fmaf(Tf[8], c.x, fmaf(Tf[9], c.y, fmaf(Tf[10], c.z, Tf[11])));
  p.w = 1.0f;
  return p;
}

// One accepted correspondence (lane 0 of its warp): r = n·(p - q) and J = [p x n, n] in double (unfused: -fmad=false),
// added to the warp's slot s of REG_NV sums.  -> float(r)
__device__ __forceinline__ float d_reg_accumulate(double* s, const float4 p, const float4 q, const float4 n) {
  const double px = p.x, py = p.y, pz = p.z, nx = n.x, ny = n.y, nz = n.z;
  const double dx = px - (double)q.x, dy = py - (double)q.y, dz = pz - (double)q.z;
  const double r = (nx * dx + ny * dy) + nz * dz;
  const double J[6] = {py * nz - pz * ny, pz * nx - px * nz, px * ny - py * nx, nx, ny, nz};
#pragma unroll
  for (int a = 0, k = 0; a < 6; ++a)
#pragma unroll
    for (int b = a; b < 6; ++b, ++k) s[k] += J[a] * J[b];
#pragma unroll
  for (int a = 0; a < 6; ++a) s[21 + a] += J[a] * r;
  s[27] += r * r;
  s[28] += 1.0;
  return (float)r;
}

// End of an iteration, every thread of the block: the block total is the warp slots in warp order, the last block
// reduces the block partials in block order, solves and updates (the k_frame pattern): bitwise reproducible.
template <int W>
__device__ __forceinline__ void d_reg_finish(double (*wsum)[REG_NV], double* fin, const RegParams& prm, RegState* st,
                                             double* __restrict__ partials, unsigned* ticket) {
  __syncthreads();
  if (threadIdx.x < REG_NV) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < W; ++w) t += wsum[w][threadIdx.x];
    partials[(size_t)blockIdx.x * REG_NV + threadIdx.x] = t;
    __threadfence();
  }
  if (!d_last_block(ticket, gridDim.x)) return;
  d_reduce_partials<REG_NV>(partials, gridDim.x, fin);
  if (threadIdx.x != 0) return;
  d_reg_solve(fin, prm, st);
}

// One ICP iteration.  Warp per source point: p = float(T)·c as the fmaf chains of k_map_insert, exact nearest compacted
// target point q within d_max, r = n·(p - q) and J = [p x n, n] in double (unfused: -fmad=false).  Lane 0 of each warp
// adds its points to the warp's slot in shared memory (in registers the 29 sums would stay live across the search and
// spill), then d_reg_finish.  Launched with REG_BLOCK threads; the register budget is explicit because ptxas' own
// choice (72) spills around the search (96: no spills, 5 blocks per SM).
__global__ void __maxnreg__(96)
k_reg_iter(const float4* __restrict__ src, const int* __restrict__ n_src_ptr, const float4* __restrict__ sp,
           const BlockEntry* __restrict__ tab, const int* __restrict__ ucell_start, const int2* __restrict__ runs,
           const int2* __restrict__ cell_info, const int* __restrict__ valid_map, const float4* __restrict__ cloud_c,
           const float4* __restrict__ normals_c, GridSpec g, const DevState* __restrict__ tst, int search, RegParams prm,
           RegState* st, double* __restrict__ partials, unsigned* ticket, int* __restrict__ corr, float* __restrict__ resid) {
  constexpr int W = REG_BLOCK / 32;
  __shared__ double wsum[W][REG_NV];
  __shared__ double fin[REG_NV];
  if (*(volatile int*)&st->done) return;  // written by an earlier launch only: every block takes the same branch
  float Tf[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) Tf[k] = (float)st->T[k];
  const int V = *n_src_ptr;
  const int U = search ? tst->n_cells : 0, nf = search ? tst->n_sorted_finite : 0;
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * REG_BLOCK) >> 5;
  double* s = wsum[threadIdx.x >> 5];
  for (int k = lane; k < REG_NV; k += 32) s[k] = 0.0;
  __syncwarp();
  for (int j = (blockIdx.x * REG_BLOCK + threadIdx.x) >> 5; j < V; j += warps_total) {
    const float4 p = d_reg_transform(Tf, src[j]);
    float best = CUDART_INF_F;
    int bi = 0x7FFFFFFF;
    if (search && finite3(p.x, p.y, p.z)) d_reg_nn(p, sp, tab, ucell_start, runs, cell_info, valid_map, g, U, nf, prm.d_max, best, bi);
    if (lane == 0) {
      int id = -1;
      float rf = CUDART_NAN_F;
      if (bi != 0x7FFFFFFF && best < prm.r2max) {
        rf = d_reg_accumulate(s, p, cloud_c[bi], normals_c[2 * (size_t)bi]);
        id = bi;
      }
      corr[j] = id;
      resid[j] = rf;
    }
  }
  d_reg_finish<W>(wsum, fin, prm, st, partials, ticket);
}

// ---- scan-to-map registration (gm_register_map) ----------------------------------------------------------------------
// Face f of cube shell k around (cx, cy, cz), clipped to the plane box [lo, hi] (inclusive cells): f 0/1 = the z faces,
// 2/3 the y faces without their z edges, 4/5 the x faces without their y and z edges, 6 the centre (shell 1 only).
// The faces partition the shell.  -> number of cells (0 when the clipped face is empty).
struct MapFace { int x0, x1, y0, y1, z0, z1; };
__device__ __forceinline__ long long d_shell_face(int f, int k, int cx, int cy, int cz, const int* lo, const int* hi, MapFace& r) {
  switch (f) {
    case 0: case 1: r.x0 = cx - k; r.x1 = cx + k; r.y0 = cy - k; r.y1 = cy + k; r.z0 = r.z1 = cz + (f == 0 ? -k : k); break;
    case 2: case 3: r.x0 = cx - k; r.x1 = cx + k; r.y0 = r.y1 = cy + (f == 2 ? -k : k); r.z0 = cz - k + 1; r.z1 = cz + k - 1; break;
    case 4: case 5: r.x0 = r.x1 = cx + (f == 4 ? -k : k); r.y0 = cy - k + 1; r.y1 = cy + k - 1; r.z0 = cz - k + 1; r.z1 = cz + k - 1; break;
    default: r.x0 = r.x1 = cx; r.y0 = r.y1 = cy; r.z0 = r.z1 = cz; if (k != 1) r.x1 = r.x0 - 1; break;
  }
  r.x0 = max(r.x0, lo[0]); r.x1 = min(r.x1, hi[0]);
  r.y0 = max(r.y0, lo[1]); r.y1 = min(r.y1, hi[1]);
  r.z0 = max(r.z0, lo[2]); r.z1 = min(r.z1, hi[2]);
  if (r.x1 < r.x0 || r.y1 < r.y0 || r.z1 < r.z0) return 0;
  return (long long)(r.x1 - r.x0 + 1) * (r.y1 - r.y0 + 1) * (r.z1 - r.z0 + 1);
}

// Exact nearest map voxel of p among those with a plane (cent[s].w != 0): FLANN ((dx^2)+dy^2)+dz^2 from p to the voxel
// centroid in float, ties -> lowest map key, or none when it is not nearer than d_max.  One warp per query over cube
// shells of voxels around p's voxel floor(p * inv_leaf) (k_map_insert's cell), the lanes sharing each shell: shell 1 is
// the 27 voxels around it, shell k >= 2 the voxels at Chebyshev distance k, each a hash lookup.  Only the part of a shell
// inside `box` (the cells of the voxels with a plane: box[0..2] = min, box[4..6] = -max, k_map_planes) is visited, shells
// that miss the box are skipped, and the search ends once no cell of the box is left unexplored, so the work per query
// is bounded by the plane voxels' extent whatever d_max is; an empty box ends it at once.
// The stop rules are d_reg_nn's with the leaf as the cell.  A centroid is the mean of points that all fall in its voxel,
// so it lies in that voxel up to the 2^-20 m fixed-point rounding of the sums (and the float rounding of the centroid
// and of p * inv_leaf): after shell k every unexplored voxel is at Chebyshev distance >= k + 1 from p's voxel, so its
// centroid is at least k * leaf from p on some axis, less those roundings, which the 0.1 % margin covers for leaves of a
// millimetre and more at mapping coordinates.  A query beyond +-2^22 voxels on an axis is clamped there: every map voxel
// lies within +-2^20 (map_pack), so on that axis the true gap is larger than the clamped one and the bound still holds.
__device__ __forceinline__ void d_regmap_nn(const float4 p, const unsigned long long* __restrict__ keys, const float4* __restrict__ cent,
                                            const int* __restrict__ box, unsigned long long slot_mask, float inv_leaf, double leaf,
                                            double d_max, float& best, unsigned long long& bkey, long long& bslot) {
  const int lane = threadIdx.x & 31;
  best = CUDART_INF_F;
  bkey = MAP_EMPTY;
  bslot = -1;
  const int lo[3] = {box[0], box[1], box[2]}, hi[3] = {-box[4], -box[5], -box[6]};
  if (lo[0] > hi[0]) return;  // no voxel has a plane
  constexpr float CL = 4194304.0f;  // 2^22
  const int cx = (int)fminf(fmaxf(floorf(p.x * inv_leaf), -CL), CL);
  const int cy = (int)fminf(fmaxf(floorf(p.y * inv_leaf), -CL), CL);
  const int cz = (int)fminf(fmaxf(floorf(p.z * inv_leaf), -CL), CL);
  // Chebyshev distance from p's voxel to the nearest (D) and the farthest (R) cell of the box
  const int D = max(max(max(0, max(lo[0] - cx, cx - hi[0])), max(lo[1] - cy, cy - hi[1])), max(lo[2] - cz, cz - hi[2]));
  const int R = max(max(max(cx - lo[0], hi[0] - cx), max(cy - lo[1], hi[1] - cy)), max(cz - lo[2], hi[2] - cz));
  const int k0 = max(1, D);
  // shells 1 .. k0-1 hold no candidate: the state after them is "nothing found", so d_max may already end the search
  if (k0 >= 2 && (double)(k0 - 1) * leaf * 0.999 >= d_max) return;
  for (int k = k0;; ++k) {
    long long T = 0;
    MapFace fc;
#pragma unroll 1
    for (int f = 0; f < 7; ++f) T += d_shell_face(f, k, cx, cy, cz, lo, hi, fc);
    int f = 0;
    long long base = 0, area = d_shell_face(0, k, cx, cy, cz, lo, hi, fc);
    for (long long t = lane; t < T; t += 32) {
      while (t >= base + area) { base += area; ++f; area = d_shell_face(f, k, cx, cy, cz, lo, hi, fc); }
      const long long u = t - base;
      const int nx = fc.x1 - fc.x0 + 1, ny = fc.y1 - fc.y0 + 1;
      const long long r = u / nx;
      unsigned long long key;
      if (!map_pack(fc.x0 + (int)(u - r * nx), fc.y0 + (int)(r % ny), fc.z0 + (int)(r / ny), key)) continue;
      const long long s = d_map_find(keys, key, slot_mask);
      if (s < 0) continue;
      const float4 c = cent[s];
      if (c.w == 0.f) continue;
      const float ex = p.x - c.x, ey = p.y - c.y, ez = p.z - c.z;
      const float d2 = (ex * ex + ey * ey) + ez * ez;
      if (d2 < best || (d2 == best && key < bkey)) { best = d2; bkey = key; bslot = s; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(FULL, best, o);
      const unsigned long long ok = __shfl_xor_sync(FULL, bkey, o);
      const long long os = __shfl_xor_sync(FULL, bslot, o);
      if (ob < best || (ob == best && ok < bkey)) { best = ob; bkey = ok; bslot = os; }
    }
    const double lim = (double)k * leaf * 0.999;
    if (bkey != MAP_EMPTY && (double)best <= lim * lim) break;
    if (lim >= d_max) break;
    if (k >= R) break;  // every cell of the box has been visited
  }
}

// One ICP iteration against the map: k_reg_iter with d_regmap_nn as the search and the matched voxel's centroid and
// plane normal (k_map_planes) as q and n.  corr_key[j] = the matched map key or MAP_EMPTY.
__global__ void __maxnreg__(96)
k_regmap_iter(const float4* __restrict__ src, const int* __restrict__ n_src_ptr, const unsigned long long* __restrict__ keys,
              const float4* __restrict__ cent, const float4* __restrict__ nrm, const int* __restrict__ box, unsigned long long slot_mask,
              float inv_leaf, double leaf, RegParams prm, RegState* st, double* __restrict__ partials, unsigned* ticket, unsigned long long* __restrict__ corr_key,
              float* __restrict__ resid) {
  constexpr int W = REG_BLOCK / 32;
  __shared__ double wsum[W][REG_NV];
  __shared__ double fin[REG_NV];
  if (*(volatile int*)&st->done) return;  // written by an earlier launch only: every block takes the same branch
  float Tf[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) Tf[k] = (float)st->T[k];
  const int V = *n_src_ptr;
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * REG_BLOCK) >> 5;
  double* s = wsum[threadIdx.x >> 5];
  for (int k = lane; k < REG_NV; k += 32) s[k] = 0.0;
  __syncwarp();
  for (int j = (blockIdx.x * REG_BLOCK + threadIdx.x) >> 5; j < V; j += warps_total) {
    const float4 p = d_reg_transform(Tf, src[j]);
    float best = CUDART_INF_F;
    unsigned long long bkey = MAP_EMPTY;
    long long bslot = -1;
    if (finite3(p.x, p.y, p.z)) d_regmap_nn(p, keys, cent, box, slot_mask, inv_leaf, leaf, prm.d_max, best, bkey, bslot);
    if (lane == 0) {
      unsigned long long key = MAP_EMPTY;
      float rf = CUDART_NAN_F;
      if (bkey != MAP_EMPTY && best < prm.r2max) {
        rf = d_reg_accumulate(s, p, cent[bslot], nrm[bslot]);
        key = bkey;
      }
      corr_key[j] = key;
      resid[j] = rf;
    }
  }
  d_reg_finish<W>(wsum, fin, prm, st, partials, ticket);
}

}  // namespace gm
