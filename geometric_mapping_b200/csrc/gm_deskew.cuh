// gm_deskew.cuh — motion compensation of a swept scan (builder-defined: the reference treats a scan as a snapshot).
// Each point, taken at its own time t_i during the sweep, is expressed in the sensor frame at t_ref, the sensor moving by
// delta over one period at constant velocity: rotation along the geodesic, translation linearly.
// Semantics (the formula, the exact cases and the rules): include/gm_capi.h (gm_deskew).
#pragma once
#include "gm_map.cuh"

namespace gm {

constexpr int DSK_BLOCK = 256;

// The constants of a delta (row-major [R | t], float), in double: theta, the axis u and the translation td.
struct DeskewConst { double theta, u[3], td[3]; };

__device__ __forceinline__ void d_deskew_constants(const float delta[12], DeskewConst* c) {
  double D[12];
  for (int k = 0; k < 12; ++k) D[k] = (double)delta[k];
  const double vx = D[9] - D[6], vy = D[2] - D[8], vz = D[4] - D[1];
  const double nv = sqrt((vx * vx + vy * vy) + vz * vz);
  const bool rot = nv > 0.0;  // |v| = 0: theta = 0 and u = 0, so that no 0 * NaN enters R(a)
  c->theta = rot ? atan2(nv / 2.0, (((D[0] + D[5]) + D[10]) - 1.0) / 2.0) : 0.0;
  c->u[0] = rot ? vx / nv : 0.0;
  c->u[1] = rot ? vy / nv : 0.0;
  c->u[2] = rot ? vz / nv : 0.0;
  c->td[0] = D[3]; c->td[1] = D[7]; c->td[2] = D[11];
}

// In place over pts[0, n), n = st->n_input.  The delta is delta_dev (12 floats in device memory, written by an earlier
// kernel on the stream) when it is not null, else the launch argument delta.  Each block derives the constants once.
// p' = R(a) p + a td, a = (t_i - t_ref) / period, R(a) p = cos(phi) p + sin(phi) (u x p) + (1 - cos(phi)) (u . p) u,
// phi = a theta; a non-finite coordinate or time gives (NaN, NaN, NaN, 1).
__global__ void __launch_bounds__(DSK_BLOCK)
k_deskew(const DevState* __restrict__ st, float4* __restrict__ pts, const float* __restrict__ times, Pose34 delta,
         const float* __restrict__ delta_dev, double t_ref, double period) {
  __shared__ DeskewConst sc;
  if (threadIdx.x == 0) d_deskew_constants(delta_dev ? delta_dev : delta.r, &sc);
  __syncthreads();
  const DeskewConst c = sc;
  const int n = st->n_input;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    const float t = times[i];
    float4 o;
    if (!finite3(p.x, p.y, p.z) || !isfinite(t)) {
      o = make_float4(CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, 1.0f);
    } else {
      const double a = ((double)t - t_ref) / period;
      double s, co;
      sincos(a * c.theta, &s, &co);
      const double x = p.x, y = p.y, z = p.z;
      const double cx = c.u[1] * z - c.u[2] * y, cy = c.u[2] * x - c.u[0] * z, cz = c.u[0] * y - c.u[1] * x;
      const double k = (1.0 - co) * ((c.u[0] * x + c.u[1] * y) + c.u[2] * z);
      o.x = (float)(((co * x + s * cx) + k * c.u[0]) + a * c.td[0]);
      o.y = (float)(((co * y + s * cy) + k * c.u[1]) + a * c.td[1]);
      o.z = (float)(((co * z + s * cz) + k * c.u[2]) + a * c.td[2]);
      o.w = 1.0f;
    }
    pts[i] = o;
  }
}

}  // namespace gm
