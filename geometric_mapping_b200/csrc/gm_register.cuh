// gm_register.cuh — scan-to-scan registration (builder-defined: the reference computes no pose, every scan is
// processed in its own sensor frame, src/geometric_mapping.cpp:48-125).  Point-to-plane ICP of a source context's
// VoxelGrid centroids against a target context's compacted cloud and normals, the correspondences searched over the
// target's neighbour grid.  One launch per iteration and no host synchronisation between them: the pose lives on the
// device in double, and the last block of every iteration reduces, solves, updates it and decides whether to stop.
// Semantics: include/gm_capi.h (gm_register).
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

__global__ void k_reg_begin(RegState* st, Pose34 init, const int* __restrict__ n_source) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  for (int k = 0; k < 12; ++k) st->T[k] = (double)init.r[k];
  for (int k = 0; k < 6; ++k) st->eig[k] = 0.0;
  for (int k = 0; k < 36; ++k) st->vecs[k] = 0.0;
  st->sum_r2 = 0.0;
  st->done = 0; st->iterations = 0; st->converged = 0; st->n_corr = 0; st->n_degenerate = 0;
  st->n_source = *n_source;
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

// One ICP iteration.  Warp per source point: p = float(T)·c as the fmaf chains of k_map_insert, exact nearest compacted
// target point q within d_max, r = n·(p - q) and J = [p x n, n] in double (unfused: -fmad=false).  Lane 0 of each warp
// adds its points to the warp's slot in shared memory (in registers the 29 sums would stay live across the search and
// spill), the block total is the warp slots in warp order, and the last block reduces the block partials in block
// order, solves and updates (the k_frame pattern): bitwise reproducible.  Launched with REG_BLOCK threads; the register
// budget is explicit because ptxas' own choice (72) spills around the search (96: no spills, 5 blocks per SM).
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
    const float4 c = src[j];
    float4 p;
    p.x = fmaf(Tf[0], c.x, fmaf(Tf[1], c.y, fmaf(Tf[2], c.z, Tf[3])));
    p.y = fmaf(Tf[4], c.x, fmaf(Tf[5], c.y, fmaf(Tf[6], c.z, Tf[7])));
    p.z = fmaf(Tf[8], c.x, fmaf(Tf[9], c.y, fmaf(Tf[10], c.z, Tf[11])));
    p.w = 1.0f;
    float best = CUDART_INF_F;
    int bi = 0x7FFFFFFF;
    if (search && finite3(p.x, p.y, p.z)) d_reg_nn(p, sp, tab, ucell_start, runs, cell_info, valid_map, g, U, nf, prm.d_max, best, bi);
    if (lane == 0) {
      int id = -1;
      float rf = CUDART_NAN_F;
      if (bi != 0x7FFFFFFF && best < prm.r2max) {
        const float4 q = cloud_c[bi], n = normals_c[2 * (size_t)bi];
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
        id = bi;
        rf = (float)r;
      }
      corr[j] = id;
      resid[j] = rf;
    }
  }
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

}  // namespace gm
