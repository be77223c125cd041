// gm_polyline.cuh — builder-defined center-axis polyline + cross-sections (SURVEY A.10).
// The reference produces one global axis direction (src/geometric_mapping.cpp:91-92); this stage
// slices the cylinder-labelled points along that axis and fits, per slice, a circle in the
// plane perpendicular to the axis (centre, radius) and a local axis direction (the a5 scatter
// matrix restricted to the slice).
//
// Per-slice sums are accumulated as 64-bit fixed point (2^-32 resolution) with integer atomics:
// integer addition is associative, so the result is bitwise reproducible regardless of the
// order in which threads arrive (float/double atomics would not be).
#pragma once
#include "gm_ransac.cuh"
#include "../../include/gm_capi.h"

namespace gm {

constexpr int POLY_BLOCK = 256;
constexpr int POLY_NACC = 24;       // 8-byte slots per slice: 0..15 fixed-point sums, 16..21 doubles
constexpr int POLY_SMEM_SLICES = 256;
constexpr double POLY_FX = 4294967296.0;  // 2^32

struct PolyState {
  double axis[3], u[3], w[3];
  unsigned long long tmin_ord, tmax_ord;
  double t0, L;
  int S, pad_;
};

__device__ __forceinline__ unsigned long long d_double_to_ordered(double d) {
  unsigned long long b = (unsigned long long)__double_as_longlong(d);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double d_ordered_to_double(unsigned long long o) {
  unsigned long long b = (o & 0x8000000000000000ull) ? (o & 0x7FFFFFFFFFFFFFFFull) : ~o;
  return __longlong_as_double((long long)b);
}
__device__ __forceinline__ long long d_to_fx(double v) { return __double2ll_rn(v * POLY_FX); }
__device__ __forceinline__ double d_from_fx(long long v) { return (double)v / POLY_FX; }

// Per-slice epilogues, run by the last block of the pass that produced their inputs.
__device__ __forceinline__ void d_poly_finish(const PolyState* ps, const long long* acc, gm_slice* out) {
  const double* aux = reinterpret_cast<const double*>(acc);
  for (int s = threadIdx.x; s < ps->S; s += blockDim.x) {
    const long long* a = acc + (size_t)s * POLY_NACC;
    long long cnt = __ldcg(a + 0);
    double n = (double)cnt;
    gm_slice o;
    for (int k = 0; k < 3; ++k) { o.center[k] = 0.f; o.dir[k] = 0.f; }
    o.radius = 0.f; o.rms = 0.f;
    double tm = ps->t0 + ((double)s + 0.5) * ps->L;
    o.t_mid = (float)tm;
    o.count = (int)cnt;
    if (n >= 3 && aux[(size_t)s * POLY_NACC + 21] != 0.0) {
      double ma = aux[(size_t)s * POLY_NACC + 16], mb = aux[(size_t)s * POLY_NACC + 17];
      double ca = aux[(size_t)s * POLY_NACC + 18], cb = aux[(size_t)s * POLY_NACC + 19], rad = aux[(size_t)s * POLY_NACC + 20];
      double ctr_a = ma + ca, ctr_b = mb + cb;
      for (int k = 0; k < 3; ++k) o.center[k] = (float)(ctr_a * ps->u[k] + ctr_b * ps->w[k] + tm * ps->axis[k]);
      double N[9] = {d_from_fx(__ldcg(a + 3)), d_from_fx(__ldcg(a + 4)), d_from_fx(__ldcg(a + 5)), 0, d_from_fx(__ldcg(a + 6)),
                     d_from_fx(__ldcg(a + 7)), 0, 0, d_from_fx(__ldcg(a + 8))};
      N[3] = N[1]; N[6] = N[2]; N[7] = N[5];
      double vals[3], vecs[9];
      d_jacobi3(N, vals, vecs);
      double d[3] = {vecs[0], vecs[3], vecs[6]};
      if (d[0] * ps->axis[0] + d[1] * ps->axis[1] + d[2] * ps->axis[2] < 0) { d[0] = -d[0]; d[1] = -d[1]; d[2] = -d[2]; }
      for (int k = 0; k < 3; ++k) o.dir[k] = (float)d[k];
      o.radius = (float)rad;
      o.rms = (float)sqrt(d_from_fx(__ldcg(a + 15)) / n);
    }
    out[s] = o;
  }
}

// Launch 1 of 3: axis basis from the local frame, zero the accumulators, range of t = axis.p over
// the cylinder-labelled points (per-block min/max, reduced by the last block, which also lays out
// the slices), and the dense list the two passes walk.  The passes read only the cylinder points:
// walking the labels there instead leaves most lanes idle, because the compacted cloud is in input
// order and its labels are mixed in every warp.
//   list[k]       = x, y, z, w     w = d_weight(law, curvature), the float the passes widen to double
//   list[cap + k] = n.x, n.y, n.z, 0
// Exact copies of the inputs: the passes compute every product from them as they would from the cloud.
// The order of the list depends on block scheduling, which no output sees: every per-slice sum is an
// integer.  *n_list counts the records; the last block of k_poly_pass<2> sets it back to 0.
constexpr int POLY_RANGE_IPT = 4;  // labels per thread and tile: IPT x (POLY_BLOCK / 32) = 32 warp counts, one per lane of warp 0
__global__ void __launch_bounds__(POLY_BLOCK)
k_poly_range(const float4* __restrict__ pts, const float4* __restrict__ normals, const unsigned char* __restrict__ labels,
             const int* __restrict__ n_ptr, const FrameOut* __restrict__ frame, WeightLaw law, PolyState* ps, long long* acc,
             int n_acc, unsigned long long* part /* 2 x gridDim */, unsigned* ticket, float4* __restrict__ list, int cap,
             unsigned* n_list, double L, int max_slices) {
  constexpr int W = POLY_BLOCK / 32, TILE = POLY_RANGE_IPT * POLY_BLOCK;
  static_assert(POLY_RANGE_IPT * W == 32, "warp 0 scans the tile's warp counts with one lane each");
  __shared__ unsigned long long s_lo[W], s_hi[W];
  __shared__ unsigned s_cnt[32], s_off[32];
  const int n = *n_ptr;
  const int warp = threadIdx.x >> 5;
  const double a0 = (double)frame->vecs[0], a1 = (double)frame->vecs[3], a2 = (double)frame->vecs[6];
  for (int i = blockIdx.x * POLY_BLOCK + threadIdx.x; i < n_acc; i += gridDim.x * POLY_BLOCK) acc[i] = 0;
  unsigned long long lo = 0xFFFFFFFFFFFFFFFFull, hi = 0ull;
  for (int tile = blockIdx.x * TILE; tile < n; tile += gridDim.x * TILE) {
    bool cyl[POLY_RANGE_IPT];
    unsigned ball[POLY_RANGE_IPT];
#pragma unroll
    for (int j = 0; j < POLY_RANGE_IPT; ++j) {
      const int i = tile + j * POLY_BLOCK + threadIdx.x;
      cyl[j] = i < n && labels[i] == 2;
    }
#pragma unroll
    for (int j = 0; j < POLY_RANGE_IPT; ++j) {
      ball[j] = __ballot_sync(FULL, cyl[j]);
      if (lane_id() == 0) s_cnt[j * W + warp] = __popc(ball[j]);
    }
    __syncthreads();
    if (warp == 0) {  // list offsets of the tile's warps: one atomic per tile
      const unsigned c = s_cnt[lane_id()];
      unsigned inc = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned v = __shfl_up_sync(FULL, inc, o);
        if (lane_id() >= o) inc += v;
      }
      unsigned base = 0;
      if (lane_id() == 31 && inc > 0) base = atomicAdd(n_list, inc);
      s_off[lane_id()] = __shfl_sync(FULL, base, 31) + inc - c;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < POLY_RANGE_IPT; ++j) {
      if (!cyl[j]) continue;
      const size_t i = (size_t)(tile + j * POLY_BLOCK + threadIdx.x);
      const float4 p = pts[i];
      const double t = a0 * (double)p.x + a1 * (double)p.y + a2 * (double)p.z;
      const unsigned long long o = d_double_to_ordered(t);
      lo = o < lo ? o : lo;
      hi = o > hi ? o : hi;
      const unsigned k = s_off[j * W + warp] + __popc(ball[j] & lanemask_lt());
      if (k < (unsigned)cap) {
        const float4 n0 = normals[2 * i];
        list[k] = make_float4(p.x, p.y, p.z, d_weight(law, normals[2 * i + 1].x));
        list[(size_t)cap + k] = make_float4(n0.x, n0.y, n0.z, 0.f);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    unsigned long long l2 = __shfl_xor_sync(FULL, lo, o), h2 = __shfl_xor_sync(FULL, hi, o);
    lo = l2 < lo ? l2 : lo;
    hi = h2 > hi ? h2 : hi;
  }
  if (lane_id() == 0) { s_lo[warp] = lo; s_hi[warp] = hi; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < W; ++w) { lo = s_lo[w] < lo ? s_lo[w] : lo; hi = s_hi[w] > hi ? s_hi[w] : hi; }
    part[2 * blockIdx.x] = lo;
    part[2 * blockIdx.x + 1] = hi;
    __threadfence();
  }
  if (!d_last_block(ticket, gridDim.x)) return;
  lo = 0xFFFFFFFFFFFFFFFFull; hi = 0ull;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += POLY_BLOCK) {
    unsigned long long l2 = __ldcg(part + 2 * b), h2 = __ldcg(part + 2 * b + 1);
    lo = l2 < lo ? l2 : lo;
    hi = h2 > hi ? h2 : hi;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    unsigned long long l2 = __shfl_xor_sync(FULL, lo, o), h2 = __shfl_xor_sync(FULL, hi, o);
    lo = l2 < lo ? l2 : lo;
    hi = h2 > hi ? h2 : hi;
  }
  if (lane_id() == 0) { s_lo[warp] = lo; s_hi[warp] = hi; }
  __syncthreads();
  if (threadIdx.x != 0) return;
  for (int w = 1; w < W; ++w) { lo = s_lo[w] < lo ? s_lo[w] : lo; hi = s_hi[w] > hi ? s_hi[w] : hi; }
  double ax[3] = {a0, a1, a2}, u[3], w[3];
  d_perp_basis_d(ax, u, w);
  for (int k = 0; k < 3; ++k) { ps->axis[k] = ax[k]; ps->u[k] = u[k]; ps->w[k] = w[k]; }
  ps->tmin_ord = lo; ps->tmax_ord = hi;
  ps->L = L; ps->t0 = 0.0; ps->S = 0; ps->pad_ = 0;
  if (lo <= hi) {
    double tmin = d_ordered_to_double(lo), tmax = d_ordered_to_double(hi);
    double t0 = floor(tmin / L) * L;
    int S = (int)floor((tmax - t0) / L) + 1;
    ps->t0 = t0;
    ps->S = S > max_slices ? max_slices : S;
  }
}

// Means AND circle fit from ONE pass: the moments are taken about a fixed point near every slice's mean -- the axis of
// the refined cylinder, (ca0, cb0) in the (u, w) plane -- and moved to the slice mean algebraically afterwards (offsets
// of a few decimetres against a 2.5 m section: no cancellation to speak of, and the sums themselves are exact integers).
__device__ __forceinline__ void d_poly_means_and_fit(const PolyState* ps, long long* acc, double ca0, double cb0) {
  double* aux = reinterpret_cast<double*>(acc);
  for (int s = threadIdx.x; s < ps->S; s += blockDim.x) {
    const long long* a = acc + (size_t)s * POLY_NACC;
    const double n = (double)__ldcg(a + 0);
    double ma = 0.0, mb = 0.0, ca = 0.0, cb = 0.0, rad = 0.0, ok = 0.0;
    if (n > 0) {
      const double Sa = d_from_fx(__ldcg(a + 1)), Sb = d_from_fx(__ldcg(a + 2));
      ma = Sa / n; mb = Sb / n;
      if (n >= 3) {
        const double Raa = d_from_fx(__ldcg(a + 9)), Rab = d_from_fx(__ldcg(a + 10)), Rbb = d_from_fx(__ldcg(a + 11));
        const double Raz = d_from_fx(__ldcg(a + 12)), Rbz = d_from_fx(__ldcg(a + 13)), Rz = d_from_fx(__ldcg(a + 14));
        const double m2 = ma * ma + mb * mb;
        const double Saa = Raa - n * ma * ma, Sab = Rab - n * ma * mb, Sbb = Rbb - n * mb * mb;
        const double Sz = Rz - n * m2;
        const double Saz = Raz - 2.0 * ma * Raa - 2.0 * mb * Rab + m2 * Sa - ma * Rz + 2.0 * ma * ma * Sa + 2.0 * ma * mb * Sb - n * ma * m2;
        const double Sbz = Rbz - 2.0 * ma * Rab - 2.0 * mb * Rbb + m2 * Sb - mb * Rz + 2.0 * ma * mb * Sa + 2.0 * mb * mb * Sb - n * mb * m2;
        const double det = Saa * Sbb - Sab * Sab;
        if (fabs(det) > 1e-300) {
          const double Ac = (Saz * Sbb - Sbz * Sab) / det, Bc = (Sbz * Saa - Saz * Sab) / det;
          ca = 0.5 * Ac; cb = 0.5 * Bc;
          rad = sqrt(Sz / n + ca * ca + cb * cb);
          ok = 1.0;
        }
      }
    }
    aux[(size_t)s * POLY_NACC + 16] = ca0 + ma;   // slice mean in absolute (u, w) coordinates
    aux[(size_t)s * POLY_NACC + 17] = cb0 + mb;
    aux[(size_t)s * POLY_NACC + 18] = ca;
    aux[(size_t)s * POLY_NACC + 19] = cb;
    aux[(size_t)s * POLY_NACC + 20] = rad;
    aux[(size_t)s * POLY_NACC + 21] = ok;
  }
}

// Adds each lane's NS values to slot[s * stride + k] of its slice s (s < 0: nothing to add).  The lanes of one slice
// sum their values first, so that one lane per slice issues the NS atomics: a 64-bit shared-memory add is a
// compare-and-swap loop, and lanes of one warp that add to the same word make each other retry.  Integer sums: the
// result is the same in any order.
template <int NS>
__device__ __forceinline__ void d_poly_warp_add(int s, unsigned long long (&v)[NS], unsigned long long* slot, int stride) {
  const unsigned grp = __match_any_sync(FULL, s);
  const unsigned later = grp & (0xFFFFFFFEu << lane_id());
  int next = later ? __ffs(later) - 1 : 32;  // next lane of the same slice, 32: none
  const int size = __reduce_max_sync(FULL, s >= 0 ? __popc(grp) : 0);
  // pointer jumping: after the step of distance d every lane holds the sum of its group's lanes from itself up to
  // 2d - 1 places further, so the first lane of the group ends with the whole group
  for (int d = 1; d < size; d <<= 1) {
#pragma unroll
    for (int k = 0; k < NS; ++k) {
      const unsigned long long o = __shfl_sync(FULL, v[k], next & 31);
      if (next < 32) v[k] += o;
    }
    const int n2 = __shfl_sync(FULL, next, next & 31);
    next = next < 32 ? n2 : 32;
  }
  if (s >= 0 && (grp & lanemask_lt()) == 0) {
#pragma unroll
    for (int k = 0; k < NS; ++k) atomicAdd(slot + (size_t)s * stride + k, v[k]);
  }
}

// Accumulation passes over the dense list of cylinder points, each followed (in the last block to finish) by the
// per-slice step that consumes it.
// PASS 0: n, sum a', sum b', weighted normal scatter (slots 0..8) AND the second/third moments of (a', b') for the
//         algebraic circle fit (9..14), a' = a - ca0, b' = b - cb0                         -> slice means + circle fit
// PASS 2: squared residuals against the fitted circle (slot 15)                            -> output slices
// (PASS 1, the separate centred-moment pass of round 1, is gone.)
template <int PASS>
__global__ void __launch_bounds__(POLY_BLOCK)
k_poly_pass(const float4* __restrict__ list, int cap, unsigned* n_list, const PolyState* __restrict__ ps,
            long long* __restrict__ acc, gm_slice* __restrict__ out, unsigned* ticket, const ModelState* __restrict__ cyl) {
  constexpr int NS = PASS == 0 ? 15 : 1;
  constexpr int SLOT0 = PASS == 0 ? 0 : 15;
  constexpr int SMEM_WORDS = POLY_SMEM_SLICES * (PASS == 0 ? 9 : 1);
  __shared__ unsigned long long s_acc[SMEM_WORDS];
  const int n = (int)min(*n_list, (unsigned)cap);
  const int S = ps->S;
  const bool use_smem = S * NS <= SMEM_WORDS;
  // fixed centring point of pass 0: where the refined cylinder's axis meets the (u, w) plane (0 without a model)
  double ca0 = 0.0, cb0 = 0.0;
  if (PASS == 0 && cyl != nullptr && cyl->best_id >= 0) {
    ca0 = ps->u[0] * (double)cyl->coef[0] + ps->u[1] * (double)cyl->coef[1] + ps->u[2] * (double)cyl->coef[2];
    cb0 = ps->w[0] * (double)cyl->coef[0] + ps->w[1] * (double)cyl->coef[1] + ps->w[2] * (double)cyl->coef[2];
  }
  // up to one copy of the accumulators per warp, so that warps do not make each other's compare-and-swap retry
  int copies = 1;
  while (copies < POLY_BLOCK / 32 && 2 * copies * S * NS <= SMEM_WORDS) copies *= 2;
  const int my_copy = (threadIdx.x >> 5) & (copies - 1);
  if (S > 0) {
    if (use_smem) {
      for (int i = threadIdx.x; i < copies * S * NS; i += POLY_BLOCK) s_acc[i] = 0ull;
      __syncthreads();
    }
    const double a0 = ps->axis[0], a1 = ps->axis[1], a2 = ps->axis[2];
    const double u0 = ps->u[0], u1 = ps->u[1], u2 = ps->u[2];
    const double w0 = ps->w[0], w1 = ps->w[1], w2 = ps->w[2];
    const double t0 = ps->t0, L = ps->L;
    const double* aux = reinterpret_cast<const double*>(acc);
    // whole warps step through the list together: the warp sums need every lane
    for (int base = blockIdx.x * POLY_BLOCK + (threadIdx.x & ~31); base < n; base += gridDim.x * POLY_BLOCK) {
      const int i = base + lane_id();
      int s = -1;
      unsigned long long v[NS];
#pragma unroll
      for (int k = 0; k < NS; ++k) v[k] = 0ull;
      if (i < n) {
        const float4 p = list[i];
        const double x = p.x, y = p.y, z = p.z;
        const double t = a0 * x + a1 * y + a2 * z;
        s = (int)floor((t - t0) / L);
        if (s < 0 || s >= S) {
          s = -1;
        } else if (PASS == 0) {
          const double a = u0 * x + u1 * y + u2 * z - ca0, b = w0 * x + w1 * y + w2 * z - cb0;
          const float4 n0 = list[(size_t)cap + i];
          const double wt = (double)p.w;
          const double na = wt * (double)n0.x, nb = wt * (double)n0.y, nc = wt * (double)n0.z;
          const double zz = a * a + b * b;
          v[0] = 1; v[1] = d_to_fx(a); v[2] = d_to_fx(b);
          v[3] = d_to_fx(na * na); v[4] = d_to_fx(na * nb); v[5] = d_to_fx(na * nc);
          v[6] = d_to_fx(nb * nb); v[7] = d_to_fx(nb * nc); v[8] = d_to_fx(nc * nc);
          v[9] = d_to_fx(a * a); v[10] = d_to_fx(a * b); v[11] = d_to_fx(b * b);
          v[12] = d_to_fx(a * zz); v[13] = d_to_fx(b * zz); v[14] = d_to_fx(zz);
        } else {
          const double ma = aux[(size_t)s * POLY_NACC + 16], mb = aux[(size_t)s * POLY_NACC + 17];
          const double ca = aux[(size_t)s * POLY_NACC + 18], cb = aux[(size_t)s * POLY_NACC + 19], rad = aux[(size_t)s * POLY_NACC + 20];
          const double a = u0 * x + u1 * y + u2 * z - ma - ca, b = w0 * x + w1 * y + w2 * z - mb - cb;
          const double e = sqrt(a * a + b * b) - rad;
          v[0] = d_to_fx(e * e);
        }
      }
      if (use_smem) d_poly_warp_add<NS>(s, v, s_acc + (size_t)my_copy * S * NS, NS);
      else d_poly_warp_add<NS>(s, v, reinterpret_cast<unsigned long long*>(acc) + SLOT0, POLY_NACC);
    }
    if (use_smem) {
      __syncthreads();
      for (int i = threadIdx.x; i < S * NS; i += POLY_BLOCK) {
        unsigned long long v = 0ull;
        for (int c = 0; c < copies; ++c) v += s_acc[c * S * NS + i];  // integer sums: any order, same result
        if (v) atomicAdd(reinterpret_cast<unsigned long long*>(acc) + (size_t)(i / NS) * POLY_NACC + SLOT0 + (i % NS), v);
      }
    }
  }
  __threadfence();
  if (!d_last_block(ticket, gridDim.x)) return;
  if (PASS == 0) {
    d_poly_means_and_fit(ps, acc, ca0, cb0);
  } else {
    d_poly_finish(ps, acc, out);
    if (threadIdx.x == 0) *n_list = 0u;  // every block has read it: the next range pass appends from 0
  }
}

}  // namespace gm
