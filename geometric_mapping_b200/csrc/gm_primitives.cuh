// gm_primitives.cuh — builder-defined sequential multi-primitive extraction (SURVEY A.9: "repeat after removing
// inliers (stable compaction)") and the compression of its result.
//
// Round r of gm_extract_primitives works on R_r, the ascending list of compacted indices that no earlier round claimed:
//   k_prim_remaining   R_r and n_r (stable look-back compaction of the unclaimed indices)
//   k_prim_draws       caller draw u -> sample index R_r[(uint64(u) * n_r) >> 32]  (-1 when n_r = 0 or after a stop)
//   hypotheses + counts: the kernels of gm_ransac.cuh, unchanged, over working copies of the cloud in which the claimed
//                      points are blanked to NaN (NaN is never an inlier)
//   k_prim_decide      plane vs cylinder (ties -> plane), stop rule, clears the loser's key (both on a stop)
//   refits            k_plane_refit / k_cyl_inlier_compact + k_cyl_gn_all, unchanged, on the blanked compacted copy
//   k_prim_claim_*     the inliers of the winning HYPOTHESIS get id r + 1 and are blanked; the primitive is recorded
// The claim uses the hypothesis, not the refined model: it is the set the integer count was taken over, so every round is
// an integer function of bit-exact quantities and the cascade is reproducible against the oracle.
#pragma once
#include "gm_compress.cuh"

namespace gm {

constexpr int PR_MAX = 64;  // GM_MAX_PRIMITIVES: ids are uint8

struct PrimRec {  // same layout as gm_primitive
  int kind, best_id, best_count, refit_count;
  float hyp[8], coef[8];
  float rms, pad_;
  int n_remaining, pad2_;
};

struct PrimState {
  int n_rem;                 // n_r of the current round
  int n_valid_live, n_crop_live;  // the cloud sizes the counting / refit / claim kernels see: 0 once extraction stopped
  int stopped;               // a round failed the stop rule: this and every later round add nothing
  int n_prims;
  int win;                   // kind of the current round's winner, -1 = none
  int pad_[2];
  float4 plane;              // winning plane hypothesis
  float test[12];            // winning cylinder hypothesis (inlier test)
  PrimRec prim[PR_MAX];
};

__global__ void k_prim_begin(PrimState* ps, const DevState* st) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  ps->n_rem = 0;
  ps->n_valid_live = st->n_valid;
  ps->n_crop_live = st->n_crop;
  ps->stopped = 0;
  ps->n_prims = 0;
  ps->win = -1;
}

// R_r: the compacted indices with id 0, ascending
__global__ void __launch_bounds__(CP_BLOCK)
k_prim_remaining(const unsigned char* __restrict__ ids, PrimState* ps, int* __restrict__ rem, unsigned long long* state, TileCtl* ctl,
                 int* err) {
  __shared__ CompactSmem<CP_BLOCK, CPL_IPT> sm;
  const int n = ps->n_valid_live;
  unsigned epoch;
  const int tile = tile_begin(ctl, epoch), base = tile * CPL_TILE;
  if (base >= n) {
    if (tile == 0 && threadIdx.x == 0) ps->n_rem = 0;
    tile_end(ctl);
    return;
  }
  bool f[CPL_IPT];
#pragma unroll
  for (int j = 0; j < CPL_IPT; ++j) {
    const int i = base + j * CP_BLOCK + threadIdx.x;
    f[j] = i < n && ids[i] == 0;
  }
  unsigned ranks[CPL_IPT], total;
  tile_compact_ranks<CP_BLOCK, CPL_IPT>(f, ranks, total, state, epoch, tile, err, sm);
#pragma unroll
  for (int j = 0; j < CPL_IPT; ++j)
    if (f[j]) rem[ranks[j]] = base + j * CP_BLOCK + threadIdx.x;
  if (base + CPL_TILE >= n && threadIdx.x == 0) ps->n_rem = (int)total;
  tile_end(ctl);
}

__device__ __forceinline__ int d_map_draw(unsigned u, const int* rem, int n) {
  return n > 0 ? rem[((unsigned long long)u * (unsigned long long)n) >> 32] : -1;
}

// draws of this round (Hp x 3 plane, Hc x 2 cylinder) -> sample indices into the compacted cloud
__global__ void k_prim_draws(const unsigned* __restrict__ dp, int np, const unsigned* __restrict__ dc, int nc, const int* __restrict__ rem,
                             const PrimState* __restrict__ ps, int* __restrict__ sp, int* __restrict__ sc) {
  const int n = ps->stopped ? 0 : ps->n_rem;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < np + nc; i += gridDim.x * blockDim.x) {
    if (i < np) sp[i] = d_map_draw(dp[i], rem, n);
    else sc[i - np] = d_map_draw(dc[i - np], rem, n);
  }
}

// One thread: the winner of the round and the stop rule.  The loser's key (both keys on a stop) is cleared, so that the
// refit kernels that follow find no model for it and do no work.
__global__ void k_prim_decide(unsigned long long* key /* [2] */, int hp_on, int hc_on, int min_inliers, int Hp, int Hc,
                              const float4* __restrict__ plane_coef, const float* __restrict__ test12, PrimState* ps) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const unsigned long long kp = hp_on ? key[0] : 0ull, kc = hc_on ? key[1] : 0ull;
  const int cp = (int)(unsigned)(kp >> 32) - 1, cc = (int)(unsigned)(kc >> 32) - 1;
  const int win = cp >= cc ? 0 : 1;  // tie -> plane
  const unsigned long long kw = win == 0 ? kp : kc;
  const int best = win == 0 ? cp : cc;
  const int id = (int)(0xFFFFFFFFu - (unsigned)(kw & 0xFFFFFFFFull));
  const bool accept = !ps->stopped && best >= max(min_inliers, 1) && id >= 0 && id < (win == 0 ? Hp : Hc);
  if (!accept) {
    ps->stopped = 1;
    ps->win = -1;
    ps->n_valid_live = 0;
    ps->n_crop_live = 0;
    key[0] = 0ull; key[1] = 0ull;
    return;
  }
  ps->win = win;
  key[win ^ 1] = 0ull;
  if (win == 0) ps->plane = plane_coef[id];
  else for (int k = 0; k < 12; ++k) ps->test[k] = test12[(size_t)id * 12 + k];
}

__device__ __forceinline__ bool d_prim_inlier(const float4 plane, const CylTest& ct, int win, const float4 p, float tau) {
  return win == 0 ? d_plane_inlier(plane, p, tau) : d_cyl_inlier(ct, p);
}

// block 0 / thread 0 of the claim: the refined model of the winner -> primitive table entry `round`
__device__ __forceinline__ void d_prim_commit(const ModelState* __restrict__ ms, PrimState* ps, int round) {
  const ModelState& m = ms[ps->win];
  PrimRec& o = ps->prim[round];
  o.kind = m.kind; o.best_id = m.best_id; o.best_count = m.best_count; o.refit_count = m.refit_count;
  for (int k = 0; k < 8; ++k) { o.hyp[k] = m.hyp[k]; o.coef[k] = m.coef[k]; }
  o.rms = m.rms; o.pad_ = 0.f;
  o.n_remaining = ps->n_rem; o.pad2_ = 0;
  ps->n_prims = round + 1;
}

// Claim over the cell-sorted working copy, one warp per 32-point leaf: the inliers of the winning hypothesis get id
// round + 1 (sorted .w = cropped index -> valid_map -> compacted index) and are blanked in both working copies; the leaf's
// bounds are rewritten from the points it has left, so later rounds cull tighter (still a superset: counts stay exact).
__global__ void k_prim_claim_sorted(float4* __restrict__ sv, float4* __restrict__ leaf_bounds, const int* __restrict__ valid_map,
                                    float4* __restrict__ cc, unsigned char* __restrict__ ids, PrimState* ps, const ModelState* __restrict__ ms,
                                    float tau, int round) {
  const int win = ps->win;
  if (win < 0) return;
  if (blockIdx.x == 0 && threadIdx.x == 0) d_prim_commit(ms, ps, round);
  const int n = ps->n_crop_live;
  const float4 plane = ps->plane;
  const CylTest ct = d_load_cyl_test(ps->test);
  const float qnan = CUDART_NAN_F;
  const int warps = gridDim.x * (blockDim.x >> 5);
  for (int leaf = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); leaf * 32 < n; leaf += warps) {
    const int i = leaf * 32 + lane_id();
    float4 p = make_float4(qnan, qnan, qnan, 0.f);
    if (i < n) p = sv[i];
    const bool claim = i < n && d_prim_inlier(plane, ct, win, p, tau);
    if (claim) {
      const int ci = valid_map[__float_as_int(p.w)];
      ids[ci] = (unsigned char)(round + 1);
      cc[ci] = make_float4(qnan, qnan, qnan, cc[ci].w);
      sv[i] = make_float4(qnan, qnan, qnan, p.w);
    }
    const bool keep = !claim && p.x == p.x;  // the points still unclaimed (blanked / dropped points are NaN)
    const float lx = warp_min(keep ? p.x : CUDART_INF_F), ly = warp_min(keep ? p.y : CUDART_INF_F), lz = warp_min(keep ? p.z : CUDART_INF_F);
    const float hx = warp_max(keep ? p.x : -CUDART_INF_F), hy = warp_max(keep ? p.y : -CUDART_INF_F), hz = warp_max(keep ? p.z : -CUDART_INF_F);
    if (lane_id() == 0) {
      leaf_bounds[2 * (size_t)leaf] = make_float4(lx, ly, lz, 0.f);
      leaf_bounds[2 * (size_t)leaf + 1] = make_float4(hx, hy, hz, 0.f);
    }
  }
}

// Claim over the compacted working copy (an injected cloud has no cell-sorted copy)
__global__ void k_prim_claim_compact(float4* __restrict__ cc, unsigned char* __restrict__ ids, PrimState* ps, const ModelState* __restrict__ ms,
                                     float tau, int round) {
  const int win = ps->win;
  if (win < 0) return;
  if (blockIdx.x == 0 && threadIdx.x == 0) d_prim_commit(ms, ps, round);
  const int n = ps->n_valid_live;
  const float4 plane = ps->plane;
  const CylTest ct = d_load_cyl_test(ps->test);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = cc[i];
    if (d_prim_inlier(plane, ct, win, p, tau)) {
      ids[i] = (unsigned char)(round + 1);
      cc[i] = make_float4(CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, p.w);
    }
  }
}

// ---- compression of the extracted primitives ---------------------------------------------------------------------
// Per primitive: claimed points, the extents of their projections (plane: u / v in the canonical in-plane basis of the
// refined normal, as gm_compress; cylinder: t along the refined axis from q) and the squared distances to the refined
// surface.  The sums are taken in 2^-32 m^2 fixed point: integer adds are exact in any order, so one shared-memory
// atomic per point gives a reproducible total without per-primitive block reductions.
constexpr double PC_FX = 4294967296.0;  // 2^32

struct PrimCompRec {  // same layout as gm_primitive_record
  int kind, count;
  float coef[7];
  float extents[4];  // plane: umin, umax, vmin, vmax; cylinder: tmin, tmax, 0, 0
  float rms;
};

struct PrimComp {
  int n_points, n_prims, n_residual, pad_;
  unsigned long long cnt[PR_MAX], sq[PR_MAX];
  unsigned long long mm[PR_MAX][4];  // ordered doubles: min, max, min, max
  PrimCompRec rec[PR_MAX];
};

__global__ void k_prim_comp_reset(PrimComp* pc, VoxState* vs) {
  for (int k = threadIdx.x; k < PR_MAX; k += blockDim.x) {
    pc->cnt[k] = 0ull; pc->sq[k] = 0ull;
    pc->mm[k][0] = ~0ull; pc->mm[k][1] = 0ull; pc->mm[k][2] = ~0ull; pc->mm[k][3] = 0ull;
  }
  if (threadIdx.x == 0) d_vox_reset(vs);
}

__global__ void __launch_bounds__(CP_BLOCK, 2)
k_prim_comp_split(const float4* __restrict__ pts, const unsigned char* __restrict__ ids, const int* __restrict__ n_ptr, const PrimState* __restrict__ ps,
                  float4* __restrict__ res_pts, VoxState* res_vs, unsigned long long* state, TileCtl* ctl, int* err, unsigned* ticket,
                  PrimComp* out, CompStats* stats) {
  __shared__ CompactSmem<CP_BLOCK, CP_IPT> sm;
  // per primitive, plane: 0..2 normal, 3..5 u, 6..8 v, 12 d; cylinder: 0..2 axis, 3..5 q, 6..8 u, 9..11 w, 12 r
  __shared__ double s_f[PR_MAX][13];
  __shared__ unsigned long long s_cnt[PR_MAX], s_sq[PR_MAX], s_mm[PR_MAX][4];
  __shared__ float s_red[6][CP_BLOCK / 32];
  const int n = *n_ptr;
  const int np = ps->n_prims;
  unsigned epoch;
  const int tile = tile_begin(ctl, epoch), base = tile * CP_TILE;
  for (int k = threadIdx.x; k < np; k += CP_BLOCK) {
    const PrimRec& r = ps->prim[k];
    double* f = s_f[k];
    for (int a = 0; a < 13; ++a) f[a] = 0.0;
    const int o = r.kind == 0 ? 0 : 3;  // normal / axis
    const double dir[3] = {(double)r.coef[o], (double)r.coef[o + 1], (double)r.coef[o + 2]};
    double u[3], v[3];
    d_perp_basis_d(dir, u, v);
    for (int a = 0; a < 3; ++a) {
      f[a] = dir[a];
      if (r.kind == 0) { f[3 + a] = u[a]; f[6 + a] = v[a]; }
      else { f[3 + a] = (double)r.coef[a]; f[6 + a] = u[a]; f[9 + a] = v[a]; }
    }
    f[12] = (double)r.coef[r.kind == 0 ? 3 : 6];
    s_cnt[k] = 0ull; s_sq[k] = 0ull;
    s_mm[k][0] = ~0ull; s_mm[k][1] = 0ull; s_mm[k][2] = ~0ull; s_mm[k][3] = 0ull;
  }
  __syncthreads();
  bool f[CP_IPT];
  float4 p[CP_IPT];
  float mn[3] = {CUDART_INF_F, CUDART_INF_F, CUDART_INF_F}, mx[3] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
#pragma unroll
  for (int j = 0; j < CP_IPT; ++j) {
    const int i = base + j * CP_BLOCK + threadIdx.x;
    f[j] = false;
    if (i >= n) continue;
    p[j] = pts[i];
    const int id = ids[i];
    if (id == 0) {
      f[j] = true;
      mn[0] = fminf(mn[0], p[j].x); mn[1] = fminf(mn[1], p[j].y); mn[2] = fminf(mn[2], p[j].z);
      mx[0] = fmaxf(mx[0], p[j].x); mx[1] = fmaxf(mx[1], p[j].y); mx[2] = fmaxf(mx[2], p[j].z);
      continue;
    }
    const int k = id - 1;
    const double* F = s_f[k];
    const double x = p[j].x, y = p[j].y, z = p[j].z;
    double e, s0, s1 = 0.0;
    if (ps->prim[k].kind == 0) {
      e = F[0] * x + F[1] * y + F[2] * z + F[12];
      s0 = F[3] * x + F[4] * y + F[5] * z;
      s1 = F[6] * x + F[7] * y + F[8] * z;
    } else {
      const double vx = x - F[3], vy = y - F[4], vz = z - F[5];
      const double A = F[6] * vx + F[7] * vy + F[8] * vz, B = F[9] * vx + F[10] * vy + F[11] * vz;
      e = sqrt(A * A + B * B) - F[12];
      s0 = F[0] * vx + F[1] * vy + F[2] * vz;
    }
    atomicAdd(&s_cnt[k], 1ull);
    atomicAdd(&s_sq[k], (unsigned long long)__double2ull_rn(e * e * PC_FX));
    atomicMin(&s_mm[k][0], d_double_to_ordered(s0)); atomicMax(&s_mm[k][1], d_double_to_ordered(s0));
    if (ps->prim[k].kind == 0) { atomicMin(&s_mm[k][2], d_double_to_ordered(s1)); atomicMax(&s_mm[k][3], d_double_to_ordered(s1)); }
  }
  if (base < n) {
    unsigned ranks[CP_IPT], total;
    tile_compact_ranks<CP_BLOCK, CP_IPT>(f, ranks, total, state, epoch, tile, err, sm);
#pragma unroll
    for (int j = 0; j < CP_IPT; ++j)
      if (f[j]) res_pts[ranks[j]] = p[j];
    if (base + CP_TILE >= n && threadIdx.x == 0) res_vs->n = (int)total;
  }
  tile_end(ctl);
  // residual bounding box (order independent)
  const int w = threadIdx.x >> 5;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float lo = warp_min(mn[a]), hi = warp_max(mx[a]);
    if (lane_id() == 0) { s_red[a][w] = lo; s_red[3 + a][w] = hi; }
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    float lo = CUDART_INF_F, hi = -CUDART_INF_F;
    for (int ww = 0; ww < CP_BLOCK / 32; ++ww) { lo = fminf(lo, s_red[threadIdx.x][ww]); hi = fmaxf(hi, s_red[3 + threadIdx.x][ww]); }
    if (lo <= hi) { atomicMin(&res_vs->bbox_min[threadIdx.x], float_to_ordered(lo)); atomicMax(&res_vs->bbox_max[threadIdx.x], float_to_ordered(hi)); }
  }
  for (int k = threadIdx.x; k < np; k += CP_BLOCK) {
    if (!s_cnt[k]) continue;
    atomicAdd(&out->cnt[k], s_cnt[k]);
    atomicAdd(&out->sq[k], s_sq[k]);
    for (int c = 0; c < 4; c += 2) { atomicMin(&out->mm[k][c], s_mm[k][c]); atomicMax(&out->mm[k][c + 1], s_mm[k][c + 1]); }
  }
  if (!d_last_block(ticket, gridDim.x)) return;
  if (threadIdx.x != 0) return;
  unsigned long long claimed = 0ull, sq = 0ull;
  for (int k = 0; k < np; ++k) {
    const PrimRec& r = ps->prim[k];
    PrimCompRec& o = out->rec[k];
    const unsigned long long c = *(volatile unsigned long long*)&out->cnt[k];
    const unsigned long long s = *(volatile unsigned long long*)&out->sq[k];
    o.kind = r.kind;
    o.count = (int)c;
    for (int a = 0; a < 7; ++a) o.coef[a] = r.coef[a];
    for (int a = 0; a < 4; ++a) o.extents[a] = 0.f;
    if (c) {
      const int ne = r.kind == 0 ? 4 : 2;
      for (int a = 0; a < ne; ++a) o.extents[a] = (float)d_ordered_to_double(*(volatile unsigned long long*)&out->mm[k][a]);
    }
    o.rms = c ? (float)sqrt((double)s / PC_FX / (double)c) : 0.f;
    claimed += c;
    sq += s;
  }
  out->n_points = n;
  out->n_prims = np;
  out->n_residual = n - (int)claimed;
  // the totals k_comp_residual_error completes (residual_rms, total_rms)
  stats->n_points = n;
  stats->n_plane = (int)claimed; stats->n_cyl = 0;
  stats->n_residual = n - (int)claimed;
  stats->sq_plane = (double)sq / PC_FX; stats->sq_cyl = 0.0; stats->sq_res = 0.0;
  stats->residual_rms = 0.f; stats->total_rms = 0.f;
  __threadfence();
}

}  // namespace gm
