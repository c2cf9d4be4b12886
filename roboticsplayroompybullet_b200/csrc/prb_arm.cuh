// prb_arm.cuh — the arm's Jacobians, mass matrix and inverse dynamics in every env (sm_100a, fp32, CUDA cores);
// prb_arm_dynamics.
//
// prb_arm_kernel: ONE WARP PER ENV, ARM_ENVS envs per block, everything in an ArmMem in shared memory.
//   * load     lane j < nd reads q_j, qd_j (the caller's arrays or the env's state row, read only) and qdd_j (0 without
//              the caller's array); the free-body quaternions and slide coordinates are read too, so that phase_fk's
//              lanes past the arm work on defined values (nothing of theirs is used);
//   * fk       phase_fk (lane = link; dynamics only when M or tau is asked for) gives the link frames, axes, COMs and
//              bias wrenches;
//   * crba     crba_joint (lane = joint j), the step's own arithmetic: mass-matrix row j and h_j into W.Q;
//   * points   lane p < P places point p in the world (link frame or site_pose) and notes its link;
//   * stores   position [P,3], J [P,6,nd], J qd [P,6] and M [nd,nd] of the env are contiguous runs, written one
//              element per lane and pass so that a warp's stores coalesce; lane j writes tau_j = sum_k M_jk qdd_k + h_j.
// The kernel reads the state and the caller's arrays and writes only the outputs it is given.
#pragma once
#include <stdint.h>

#include <string>

#include "../../include/prb.h"
#include "prb_kernels.cuh"

#define ARM_ENVS 4              // envs (warps) per block
#define ARM_MAX_POINTS 16

struct ArmParams {
  int N, P;
  int link[ARM_MAX_POINTS];     // model link of point p (sites resolved to their link)
  int site[ARM_MAX_POINTS];     // -1: local_position in the link frame; 0..3: in that site's frame
  float local[ARM_MAX_POINTS][3];
};

// the fields phase_fk and crba_joint read and write, the qdd row and the points
struct ArmMem {
  float q[PRB_MAXD], qd[PRB_MAXD], qdd[PRB_MAXD];
  float lR[PRB_MAXD][9], lp[PRB_MAXD][3], la[PRB_MAXD][3], lw[PRB_MAXD][3], lv[PRB_MAXD][3], lc[PRB_MAXD][3];
  float lIw[PRB_MAXD][6], lf[PRB_MAXD][3], ln[PRB_MAXD][3];
  float fquat[PRB_MAXFREE][4], fR[PRB_MAXFREE][9], fIinv[PRB_MAXFREE][6];
  float sq[PRB_MAXSLIDE], sR[PRB_MAXSLIDE][9], sp[PRB_MAXSLIDE][3];
  float Mm[PRB_MAXD][PRB_MAXD + 1];
  float Q[PRB_MAXD];            // h_j: crba_joint's bias torque (the step keeps -h_j - jdamp_j qd_j here instead)
  float x[ARM_MAX_POINTS][3];   // world position of point p
};

// row r of column j of the Jacobian of the point x on model link l: 0 unless j is an ancestor-or-self of l; revolute
// (a_j x (x - p_j), a_j), prismatic (a_j, 0)
PRB_D float arm_jac(const DevModel& M, const ArmMem& W, int l, v3 x, int r, int j) {
  if (!((M.anc_mask[l] >> j) & 1u)) return 0.f;
  const v3 a = ld3(W.la[j]);
  if (M.jtype[j] != 0) return r < 3 ? comp(a, r) : 0.f;
  return r < 3 ? comp(cross(a, x - ld3(W.lp[j])), r) : comp(a, r - 3);
}

// q, qd, qdd [N,nd] (NULL: the state's q and qd, qdd = 0); jac [N,P,6,nd], pos [N,P,3], vel [N,P,6], mm [N,nd,nd],
// tau [N,nd], each optional
__global__ void __launch_bounds__(32 * ARM_ENVS) prb_arm_kernel(const DevModel* __restrict__ Mp, const float* __restrict__ state,
                                                               const __grid_constant__ ArmParams P, const float* __restrict__ q_in,
                                                               const float* __restrict__ qd_in, const float* __restrict__ qdd_in,
                                                               float* __restrict__ jac, float* __restrict__ pos,
                                                               float* __restrict__ vel, float* __restrict__ mm, float* __restrict__ tau) {
  __shared__ ArmMem SM[ARM_ENVS];
  const DevModel& M = *Mp;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t e = (int64_t)blockIdx.x * ARM_ENVS + warp;
  if (e >= P.N) return;                  // whole warps of the last block
  ArmMem& W = SM[warp];
  const int nd = M.nd;
  const float* st = state + e * M.state_stride;
  if (lane < nd) {
    W.q[lane] = q_in ? q_in[e * nd + lane] : st[lane];
    W.qd[lane] = qd_in ? qd_in[e * nd + lane] : st[nd + lane];
    W.qdd[lane] = qdd_in ? qdd_in[e * nd + lane] : 0.f;
  }
  if (lane < M.n_free) for (int k = 0; k < 4; k++) W.fquat[lane][k] = st[5 * nd + 13 * lane + 3 + k];
  if (lane < M.n_slide) W.sq[lane] = st[5 * nd + 13 * M.n_free + 2 * lane];
  __syncwarp();
  const bool dyn = mm || tau;
  phase_fk(M, W, lane, dyn);
  if (dyn) {
    if (lane < nd) crba_joint(M, W, lane, [&](float h) { W.Q[lane] = h; });
    __syncwarp();
  }
  if (lane < P.P) {
    const int l = P.link[lane], s = P.site[lane];
    const v3 o = ld3(P.local[lane]);
    v3 x;
    if (s >= 0) {
      v3 ps; m3 Rs;
      site_pose(M, W, s, ps, Rs);
      x = ps + mul(Rs, o);
    } else {
      x = ld3(W.lp[l]) + mul(ldm(W.lR[l]), o);
    }
    st3(W.x[lane], x);
  }
  __syncwarp();

  const int np = P.P;
  if (pos) {
    float* out = pos + e * (3 * np);
    for (int i = lane; i < 3 * np; i += 32) out[i] = W.x[i / 3][i % 3];
  }
  if (jac) {
    float* out = jac + e * (6 * nd * np);
    for (int i = lane; i < 6 * nd * np; i += 32) {
      const int p = i / (6 * nd), r = (i / nd) % 6, j = i % nd;
      out[i] = arm_jac(M, W, P.link[p], ld3(W.x[p]), r, j);
    }
  }
  if (vel) {
    float* out = vel + e * (6 * np);
    for (int i = lane; i < 6 * np; i += 32) {
      const int p = i / 6, r = i % 6, l = P.link[p];
      const v3 x = ld3(W.x[p]);
      float s = 0.f;
      for (int j = 0; j < nd; j++) s += arm_jac(M, W, l, x, r, j) * W.qd[j];
      out[i] = s;
    }
  }
  if (mm) {
    float* out = mm + e * (nd * nd);
    for (int i = lane; i < nd * nd; i += 32) out[i] = W.Mm[i / nd][i % nd];
  }
  if (tau && lane < nd) {
    float s = W.Q[lane];
    if (qdd_in) {
      float mq = 0.f;
      for (int k = 0; k < nd; k++) mq += W.Mm[lane][k] * W.qdd[k];
      s = mq + s;
    }
    tau[e * nd + lane] = s;
  }
}

// prb_arm_query, the points and the arrays -> kernel parameters; returns why the call is rejected, or "" if it is valid
static inline std::string arm_params(const prb_arm_query& a, const prb_arm_point* points, const void* jac, const void* pos,
                                     const void* vel, const void* mm, const void* tau, int N, int nd, const int* site_link,
                                     ArmParams* P) {
  if (a.num_points < 0 || a.num_points > ARM_MAX_POINTS) return "num_points must be in 0..16";
  if (a.reserved != 0) return "reserved must be 0";
  if (!jac && !pos && !vel && !mm && !tau) return "at least one output is required";
  const bool point_out = jac || pos || vel;
  if (a.num_points > 0 && !point_out) return "points need jacobian_dev, point_position_dev or point_velocity_dev";
  if (a.num_points == 0 && point_out) return "jacobian_dev, point_position_dev and point_velocity_dev need num_points >= 1";
  if (a.num_points > 0 && !points) return "points_host is required when num_points > 0";
  P->N = N; P->P = a.num_points;
  for (int p = 0; p < ARM_MAX_POINTS; p++) {
    P->link[p] = 0; P->site[p] = -1;
    P->local[p][0] = P->local[p][1] = P->local[p][2] = 0.f;
    if (p >= a.num_points) continue;
    const prb_arm_point& t = points[p];
    if (t.reserved != 0) return "point " + std::to_string(p) + ": reserved must be 0";
    if (t.site < -1 || t.site > 3) return "point " + std::to_string(p) + ": site must be -1 (a link) or a site 0..3";
    if (t.site >= 0 && t.link != -1) return "point " + std::to_string(p) + ": a site point must have link -1";
    if (t.site < 0 && (t.link < 0 || t.link >= nd)) return "point " + std::to_string(p) + ": link must be in 0..nd-1";
    P->site[p] = t.site;
    P->link[p] = t.site >= 0 ? site_link[t.site] : t.link;
    for (int k = 0; k < 3; k++) P->local[p][k] = t.local_position[k];
  }
  return "";
}

static inline unsigned arm_blocks(int N) { return (unsigned)((N + ARM_ENVS - 1) / ARM_ENVS); }
