// gm_odometry.cuh — map odometry on the device (builder-defined: the reference computes no pose).  One step predicts
// the scan's pose from the trajectory (k_odom_begin), runs gm_register_map's ICP from it (gm_register.cuh), gates the
// result and records it (k_odom_gate), and inserts the scan at the recorded pose (k_map_insert_gated, gm_map.cuh), all
// on the context's stream: the pose never travels to the host.  k_odom_delta gives gm_odometry_deskew the
// constant-velocity increment for k_deskew (gm_deskew.cuh).
// Semantics: include/gm_capi.h (gm_odometry_*).
#pragma once
#include "gm_register.cuh"

namespace gm {

// = gm_odometry_record (static_assert in gm_capi.cu)
struct OdomRecord {
  float pose34[12], guess34[12];
  int accepted, registered, iterations, converged, n_source, n_correspondences, n_degenerate;
  float rmse, fitness;
  int pad_;
};

// what the insert of the current step reads: the pose and the go/no-go flag
struct OdomInsert {
  Pose34 pose;
  int accept;
};

// C = A o B of two rigid [R | t] in double, unfused (-fmad=false), in the order d_reg_solve updates the pose in
__device__ __forceinline__ void d_pose_compose(const double A[12], const double B[12], double C[12]) {
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) C[i * 4 + j] = (A[i * 4 + 0] * B[j] + A[i * 4 + 1] * B[4 + j]) + A[i * 4 + 2] * B[8 + j];
    C[i * 4 + 3] = ((A[i * 4 + 0] * B[3] + A[i * 4 + 1] * B[7]) + A[i * 4 + 2] * B[11]) + A[i * 4 + 3];
  }
}

// C = [R^T | -(R^T t)], each entry of R^T t summed in the same order
__device__ __forceinline__ void d_pose_inverse(const double A[12], double C[12]) {
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) C[i * 4 + j] = A[j * 4 + i];
    C[i * 4 + 3] = -((A[i] * A[3] + A[4 + i] * A[7]) + A[8 + i] * A[11]);
  }
}

__device__ __forceinline__ void d_pose_load(const float P[12], double D[12]) {
  for (int k = 0; k < 12; ++k) D[k] = (double)P[k];
}

enum OdomGuess { ODOM_INIT = 0, ODOM_DELTA = 1, ODOM_VELOCITY = 2 };

// Step k, one thread: the guess G (ODOM_INIT: init; ODOM_DELTA: P_{k-1} o delta; ODOM_VELOCITY: P_{k-1} o (P_{k-2}^-1 o
// P_{k-1})) rounded to float into record k, and, for a registered step (st != null), the registration's start from it.
__global__ void k_odom_begin(OdomRecord* __restrict__ rec, int k, int mode, Pose34 init, Pose34 delta, RegState* st,
                             const int* __restrict__ n_source) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float G[12];
  if (mode == ODOM_INIT) {
    for (int e = 0; e < 12; ++e) G[e] = init.r[e];
  } else {
    double P1[12], D[12], Gd[12];
    d_pose_load(rec[k - 1].pose34, P1);
    if (mode == ODOM_DELTA) {
      d_pose_load(delta.r, D);
    } else {
      double P2[12], P2i[12];
      d_pose_load(rec[k - 2].pose34, P2);
      d_pose_inverse(P2, P2i);
      d_pose_compose(P2i, P1, D);
    }
    d_pose_compose(P1, D, Gd);
    for (int e = 0; e < 12; ++e) G[e] = (float)Gd[e];
  }
  for (int e = 0; e < 12; ++e) rec[k].guess34[e] = G[e];
  if (st) d_reg_start(st, G, n_source);
}

// gm_odometry_deskew for step k, one thread: the constant-velocity increment float(P_{k-2}^-1 o P_{k-1}) of
// k_odom_begin's ODOM_VELOCITY guess, element by element (the identity for k < 2), into delta[12] for k_deskew.
__global__ void k_odom_delta(const OdomRecord* __restrict__ rec, int k, float* __restrict__ delta) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (k < 2) {
    for (int e = 0; e < 12; ++e) delta[e] = (e == 0 || e == 5 || e == 10) ? 1.0f : 0.0f;
    return;
  }
  double P1[12], P2[12], P2i[12], D[12];
  d_pose_load(rec[k - 1].pose34, P1);
  d_pose_load(rec[k - 2].pose34, P2);
  d_pose_inverse(P2, P2i);
  d_pose_compose(P2i, P1, D);
  for (int e = 0; e < 12; ++e) delta[e] = (float)D[e];
}

// Step k, one thread: the gate and record k, and the insert's pose and flag.  st = null: an unregistered step (always
// accepted at the guess).  rmse and fitness are computed as gm_get_registration computes them.
__global__ void k_odom_gate(OdomRecord* __restrict__ rec, int k, const RegState* __restrict__ st, double min_fitness,
                            OdomInsert* __restrict__ ins) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  OdomRecord& r = rec[k];
  float pose[12];
  int accept = 1;
  if (st) {
    const int m = st->n_corr, V = st->n_source;
    const float rmse = m > 0 ? (float)sqrt(st->sum_r2 / (double)m) : 0.0f;
    const float fitness = V > 0 ? (float)((double)m / (double)V) : 0.0f;
    accept = ((double)fitness >= min_fitness && m >= 6) ? 1 : 0;
    for (int e = 0; e < 12; ++e) pose[e] = accept ? (float)st->T[e] : r.guess34[e];
    r.registered = 1;
    r.iterations = st->iterations;
    r.converged = st->converged;
    r.n_source = V;
    r.n_correspondences = m;
    r.n_degenerate = st->n_degenerate;
    r.rmse = rmse;
    r.fitness = fitness;
  } else {
    for (int e = 0; e < 12; ++e) pose[e] = r.guess34[e];
    r.registered = 0;
    r.iterations = r.converged = r.n_source = r.n_correspondences = r.n_degenerate = 0;
    r.rmse = r.fitness = 0.0f;
  }
  r.pad_ = 0;
  r.accepted = accept;
  for (int e = 0; e < 12; ++e) { r.pose34[e] = pose[e]; ins->pose.r[e] = pose[e]; }
  ins->accept = accept;
}

}  // namespace gm
