// prb_kernels.cuh — the batched simulator's device code (sm_100a, fp32, CUDA cores).
//
// Execution model
//   * prb_ik_kernel      one THREAD per env: action clip -> rpy->quat -> chained damped-least-
//                        squares IK on the serial arm chain (registers only) -> joint-limit and
//                        per-step clipping -> motor targets.  Reference path:
//                        environments.py:206-208, 955-961, 984-1034, 1037-1073; inverseKinematics.py:44-50.
//   * prb_step_kernel    (fused variant; the default step path is the split pipeline of
//                        prb_stream.cuh, which reuses every phase below except the solver)
//                        one WARP per env, all 12 physics substeps of an env step fused in one
//                        launch with the env's state, kinematics, mass matrix, contact manifold
//                        and constraint rows resident in shared memory; lanes are links /
//                        colliders / collider pairs / contacts in the set-up phases and velocity
//                        DoF in the projected-Gauss-Seidel sweeps (J.dv by warp-shuffle
//                        reduction).  Ends with the fused observation/reward write.  Reference
//                        path: environments.py:209-214 (runSimulation, calc_state, reward).
//   * reset              rounds of {seat objects, settle on the masked step pipeline, finish}: prb_reset.cuh
//                        (environments.py:173-187, 492-603).
//   * prb_reward_kernel  stateless batched compute_reward (relabelling): environments.py:278-304,
//                        playRewardFunc.py:66-77.
//
// Dynamics formulation (differs from the oracle's articulated-body algorithm on purpose):
// world-frame recursive Newton-Euler for the bias forces, composite-rigid-body mass matrix,
// dense Cholesky -> M^-1 kept in shared memory; every constraint row stores J and M^-1 J^T.
//
// All warp-collective operations (__shfl*, __ballot, __syncwarp) are executed in warp-uniform
// control flow with the full mask.
#pragma once
#include "prb_device.h"

#define FULL 0xffffffffu

// Per-env on-chip capacities of the FUSED kernel (prb_step_kernel / prb_reset_kernel): worst-case
// sizes, ~44 KB of shared memory per env.  If even these overflow, contacts are dropped (counted in
// DevOut::overflow).  The step path proper uses the split pipeline of prb_stream.cuh, whose
// constraint rows live in HBM and cannot overflow; the fused kernel remains for reset (100 settle
// substeps inside one launch) and as an A/B reference (PRB_PIPELINE=fused).
struct CfgL {
  static constexpr int MAXJROW = 40;       // limit + motor + gear rows
  static constexpr int MAXCONTACT = 32;    // contact points per substep after manifold reduction (one per lane)
  static constexpr int MAXOVL = 32;        // overlapping collider pairs handed to the narrow phase (one per lane)
  static constexpr int MAXCAND = 128;      // narrow-phase candidates (4 per overlapping pair) before reduction
  static constexpr int POOL = 3072;        // floats of packed contact-row Jacobians (J and M^-1 J^T segments)
  static constexpr int ACAP = 5888;        // floats of island-blocked Delassus matrix J M^-1 J^T (full R_i x R_i blocks)
  static constexpr int APAD = 160;         // slack read (and multiplied by 0) by lanes outside the sender's island
  static constexpr int MAXSLOT = 4;        // sweep units per lane
  static constexpr bool ABORT = false;
  static constexpr int WPB = 5;            // warps (envs) per thread block; the block's warps are re-aligned every substep
  static constexpr int MINBLOCKS = 1;      // resident blocks per SM the register allocation targets
};

struct Contact {
  float pbx, pby, pbz, nx, ny, nz, dist;
  int cols;   // ca | cb << 8
};

template <class CFG>
struct WarpMemT {
  typedef CFG Cfg;
  // ---- simulation state of this env (loaded once per launch, written back at the end)
  float q[PRB_MAXD], qd[PRB_MAXD], mtarget[PRB_MAXD], mkp[PRB_MAXD], mmaximp[PRB_MAXD];
  float fpos[PRB_MAXFREE][3], fquat[PRB_MAXFREE][4], fvel[PRB_MAXFREE][3], fang[PRB_MAXFREE][3];
  float sq[PRB_MAXSLIDE], sqd[PRB_MAXSLIDE];
  float goal[12], lastq[8], last_valid, reset_count;
  // ---- kinematics / dynamics of the current substep
  float lp[PRB_MAXD][3], la[PRB_MAXD][3], lc[PRB_MAXD][3], lw[PRB_MAXD][3], lv[PRB_MAXD][3];
  float fR[PRB_MAXFREE][9], fIinv[PRB_MAXFREE][6];
  float sp[PRB_MAXSLIDE][3], sR[PRB_MAXSLIDE][9];
  float Minv[PRB_MAXD][PRB_MAXD + 1], Q[PRB_MAXD];
  float vs[32];
  // ---- collision
  unsigned short ovl[CFG::MAXOVL];
  int n_ovl, n_contact, n_jrow, pool_used, overflow;
  int dbg_a, dbg_c, dbg_p, dbg_u;
  Contact ct[CFG::MAXCONTACT];
  // Everything in the first member is dead by the time the Delassus matrix is built (link
  // rotations/inertias/bias wrenches, the Cholesky workspace, collider AABBs, narrow-phase
  // candidates), so A overlays it.
  union {
    struct {
      float lR[PRB_MAXD][9], lIw[PRB_MAXD][6], lf[PRB_MAXD][3], ln[PRB_MAXD][3];
      float Mm[PRB_MAXD][PRB_MAXD + 1];
      float2 aabb[PRB_MAXCOL][3];   // per axis (lo, hi): 8-byte loads in the broad phase
      Contact cand[CFG::MAXCAND];
    };
    float A[CFG::ACAP + CFG::APAD];
  };
  // ---- constraint rows
  signed char jr_dof[CFG::MAXJROW], jr_dof2[CFG::MAXJROW];
  float jr_sign[CFG::MAXJROW], jr_rhs[CFG::MAXJROW], jr_invD[CFG::MAXJROW], jr_lo[CFG::MAXJROW], jr_hi[CFG::MAXJROW], jr_lam[CFG::MAXJROW];
  unsigned jr_meta[CFG::MAXJROW];     // island block base (16 bits) | local row id (8) | island (8)
  unsigned char jr_R[CFG::MAXJROW], ct_R[CFG::MAXCONTACT];   // rows in the unit's island block
  int unit_meta[32 * CFG::MAXSLOT + 2];         // per sweep unit g (at index g + 1): island << 16 | island-local row id
  // per contact: rows 0 normal, 1 spin, 2 friction-1, 3 friction-2
  float cr_rhs[CFG::MAXCONTACT][4], cr_invD[CFG::MAXCONTACT][4], cr_lam[CFG::MAXCONTACT][4];
  float cr_cfm[CFG::MAXCONTACT], cr_mu[CFG::MAXCONTACT], cr_spin[CFG::MAXCONTACT];
  signed char cr_bodyA[CFG::MAXCONTACT], cr_bodyB[CFG::MAXCONTACT];
  unsigned short cr_offA[CFG::MAXCONTACT], cr_offB[CFG::MAXCONTACT];
  unsigned ct_meta[CFG::MAXCONTACT];  // address base of the island block (16) | local id of the normal row (8) | island (8)
  float pool[CFG::POOL];
};

PRB_D float warp_sum(float v) {
  v += __shfl_xor_sync(FULL, v, 16);
  v += __shfl_xor_sync(FULL, v, 8);
  v += __shfl_xor_sync(FULL, v, 4);
  v += __shfl_xor_sync(FULL, v, 2);
  v += __shfl_xor_sync(FULL, v, 1);
  return v;
}
PRB_D int warp_excl_scan(int v, int lane, int* total) {
  int s = v;
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(FULL, s, o);
    if (lane >= o) s += t;
  }
  *total = __shfl_sync(FULL, s, 31);
  return s - v;
}

PRB_D unsigned warp_or(unsigned v) {
  v |= __shfl_xor_sync(FULL, v, 16);
  v |= __shfl_xor_sync(FULL, v, 8);
  v |= __shfl_xor_sync(FULL, v, 4);
  v |= __shfl_xor_sync(FULL, v, 2);
  v |= __shfl_xor_sync(FULL, v, 1);
  return v;
}

// body index of a velocity DoF and geometry helpers -------------------------------------------
// bodies: 0 arm, 1..n_free free bodies, n_free+1.. slide bodies, -1 static
PRB_D int dof_body(const DevModel& M, int d, int* li, int* n) {
  if (d < M.nd) { *li = d; *n = M.nd; return 0; }
  int r = d - M.nd;
  if (r < 6 * M.n_free) { *li = r % 6; *n = 6; return 1 + r / 6; }
  r -= 6 * M.n_free;
  if (r < M.n_slide) { *li = 0; *n = 1; return 1 + M.n_free + r; }
  *li = 0; *n = 0; return -2;
}
PRB_D int body_size(const DevModel& M, int body) { return body == 0 ? M.nd : (body <= M.n_free ? 6 : 1); }
PRB_D int body_dof0(const DevModel& M, int body) {
  return body == 0 ? 0 : (body <= M.n_free ? M.nd + 6 * (body - 1) : M.nd + 6 * M.n_free + (body - 1 - M.n_free));
}

// ============================================================================ IK (thread per env)
// One calculateInverseKinematics call restated for a serial revolute chain of NJ joints whose
// last link carries the end-effector site; base frame coordinates; q updated in place.
template <int NJ>
PRB_D void ik_call(const DevModel& M, float* q, v3 tp, const float* tq, int max_iters) {
  const float lambda = M.params[P_IK_DAMPING], thresh = M.params[P_IK_THRESHOLD];
  float diff = 1e30f;
  for (int it = 0; it < max_iters && diff > thresh; it++) {
    v3 a[NJ], pj[NJ];
    m3 R = ident3();
    v3 p = V3(0, 0, 0);
#pragma unroll
    for (int j = 0; j < NJ; j++) {
      p = p + mul(R, ld3(M.jpos[j]));
      m3 R0 = mul(R, ldm(M.jrot[j]));
      v3 ax = ld3(M.axis[j]);
      a[j] = mul(R0, ax);
      pj[j] = p;
      R = mul(R0, axis_angle(ax, q[j]));
    }
    v3 ep = p + mul(R, ld3(M.site_pos[0]));
    m3 eR = mul(R, ldm(M.site_rot[0]));
    float eq[4];
    mat_to_quat(eR, eq);
    v3 dp = tp - ep;
    diff = norm(dp);
    float e[6];
    e[0] = dp.x; e[1] = dp.y; e[2] = dp.z;
    {  // rotation error = angle * axis of (target * current^-1); atan2 form is fp32-safe near 0
      float inv[4] = {-eq[0], -eq[1], -eq[2], eq[3]}, dq[4];
      quat_mul(tq, inv, dq);
      float s = sqrtf(dq[0] * dq[0] + dq[1] * dq[1] + dq[2] * dq[2]);
      float angle = 2.0f * atan2f(s, dq[3]);
      if (angle > PRB_PI_F) angle -= 2.0f * PRB_PI_F;
      float k = s > 1e-12f ? angle / s : 0.f;
      if (s <= 1e-12f) { e[3] = angle; e[4] = 0; e[5] = 0; }   // Bullet's getAxis() fallback (1,0,0)
      else { e[3] = dq[0] * k; e[4] = dq[1] * k; e[5] = dq[2] * k; }
    }
    float J[6][NJ];
#pragma unroll
    for (int j = 0; j < NJ; j++) {
      v3 jl = cross(a[j], ep - pj[j]);
      J[0][j] = jl.x; J[1][j] = jl.y; J[2][j] = jl.z; J[3][j] = a[j].x; J[4][j] = a[j].y; J[5][j] = a[j].z;
    }
    // (J^T J + lambda I) x = J^T e, Cholesky in registers
    float A[NJ][NJ], b[NJ];
#pragma unroll
    for (int i = 0; i < NJ; i++) {
#pragma unroll
      for (int j = 0; j <= i; j++) {
        float s = 0;
#pragma unroll
        for (int k = 0; k < 6; k++) s += J[k][i] * J[k][j];
        A[i][j] = s + (i == j ? lambda : 0.f);
      }
      float s = 0;
#pragma unroll
      for (int k = 0; k < 6; k++) s += J[k][i] * e[k];
      b[i] = s;
    }
#pragma unroll
    for (int k = 0; k < NJ; k++) {
      float d = A[k][k];
#pragma unroll
      for (int m = 0; m < k; m++) d -= A[k][m] * A[k][m];
      d = sqrtf(d);
      A[k][k] = d;
      float inv = 1.0f / d;
#pragma unroll
      for (int r = k + 1; r < NJ; r++) {
        float s = A[r][k];
#pragma unroll
        for (int m = 0; m < k; m++) s -= A[r][m] * A[k][m];
        A[r][k] = s * inv;
      }
    }
#pragma unroll
    for (int r = 0; r < NJ; r++) {
      float s = b[r];
#pragma unroll
      for (int m = 0; m < r; m++) s -= A[r][m] * b[m];
      b[r] = s / A[r][r];
    }
#pragma unroll
    for (int r = NJ - 1; r >= 0; r--) {
      float s = b[r];
#pragma unroll
      for (int m = r + 1; m < NJ; m++) s -= A[m][r] * b[m];
      b[r] = s / A[r][r];
    }
    float mx = 0;
#pragma unroll
    for (int i = 0; i < NJ; i++) mx = fmaxf(mx, fabsf(b[i]));
    const float maxang = 45.0f * PRB_PI_F / 180.0f;
    float sc = mx > maxang ? maxang / mx : 1.0f;
#pragma unroll
    for (int i = 0; i < NJ; i++) q[i] += b[i] * sc;
  }
}
// world target -> base coordinates, then `calls` chained solves (inverseKinematics.py:44-50)
template <int NJ>
PRB_D void ik_world(const DevModel& M, float* q, const float* tpos_w, const float* tquat_w, int calls, int iters) {
  m3 bR = ldm(M.base_rot);
  v3 tp = tmul(bR, ld3(tpos_w) - ld3(M.base_pos));
  float bqi[4] = {-M.base_quat[0], -M.base_quat[1], -M.base_quat[2], M.base_quat[3]}, tq[4];
  quat_mul(bqi, tquat_w, tq);
  for (int c = 0; c < calls; c++) ik_call<NJ>(M, q, tp, tq, iters);
}

// world pose of the end-effector site for joint angles q (the pose calc_actor_state reports,
// environments.py:746-764): serial chain of NJ joints, site 0 on the last link
template <int NJ>
PRB_D void ee_world(const DevModel& M, const float* q, v3& pos, float* quat) {
  m3 R = ldm(M.base_rot);
  v3 p = ld3(M.base_pos);
#pragma unroll
  for (int j = 0; j < NJ; j++) {
    p = p + mul(R, ld3(M.jpos[j]));
    R = mul(mul(R, ldm(M.jrot[j])), axis_angle(ld3(M.axis[j]), q[j]));
  }
  pos = p + mul(R, ld3(M.site_pos[0]));
  mat_to_quat(mul(R, ldm(M.site_rot[0])), quat);
}
// xyz + quaternion + gripper = 8; joint decoders: one entry per IK joint + gripper (7 UR5, 8 Panda); rpy decoders 7 (environments.py:88-112)
PRB_HD int action_dim_of(int action_type, int n_ik) { return (action_type == 2 || action_type == 3) ? 8 : (action_type >= 4 ? n_ik + 1 : 7); }

// perform_action (environments.py:915-981) -> goto / goto_joint_poses (:984-1034) -> close_gripper (:1037-1073).
// action_type: 0 absolute_rpy, 1 relative_rpy, 2 absolute_quat, 3 relative_quat, 4 absolute_joints, 5 relative_joints
template <int NJ>
PRB_D void ik_action_env(const DevModel& M, float* st /* this env's state */, const float* act, float* target_out) {
  const int nd = M.nd;
  const int atype = (int)(M.params[P_ACTION_TYPE] + 0.5f), adim = action_dim_of(atype, NJ);
  float a[8];
#pragma unroll
  for (int k = 0; k < 8; k++) {
    a[k] = 0.f;
    if (k < adim - 1) a[k] = clampf(act[k], -M.params[P_ACTION_HIGH_XYZ], M.params[P_ACTION_HIGH_XYZ]);
  }
  const float grip = clampf(act[adim - 1], -M.params[P_ACTION_HIGH_GRIP], M.params[P_ACTION_HIGH_GRIP]);
  float q[NJ], q0[NJ];
#pragma unroll
  for (int i = 0; i < NJ; i++) { q0[i] = st[i]; q[i] = q0[i]; }
  if (atype >= 4) {                            // joint space: no IK (:973-981)
#pragma unroll
    for (int i = 0; i < NJ; i++) q[i] = (atype == 5 ? q0[i] : 0.f) + a[i];
  } else {
    float tp[3] = {a[0], a[1], a[2]}, tq[4];
    if (atype == 0) quat_from_euler(a + 3, tq);
    else if (atype == 2) { tq[0] = a[3]; tq[1] = a[4]; tq[2] = a[5]; tq[3] = a[6]; }
    else {                                     // relative to the current end-effector pose (:945-953, 962-970)
      v3 cp; float cq[4];
      ee_world<NJ>(M, q0, cp, cq);
      tp[0] += cp.x; tp[1] += cp.y; tp[2] += cp.z;
      if (atype == 1) {
        float rpy[3];
        euler_from_quat(cq, rpy);
        rpy[0] += a[3]; rpy[1] += a[4]; rpy[2] += a[5];
        quat_from_euler(rpy, tq);
      } else { tq[0] = cq[0] + a[3]; tq[1] = cq[1] + a[4]; tq[2] = cq[2] + a[5]; tq[3] = cq[3] + a[6]; }
    }
    if (atype >= 2) {                          // commanded quaternions are used normalised
      const float nrm = sqrtf(tq[0] * tq[0] + tq[1] * tq[1] + tq[2] * tq[2] + tq[3] * tq[3]);
      const float inv = nrm > 1e-12f ? 1.0f / nrm : 0.f;
      if (nrm > 1e-12f) { tq[0] *= inv; tq[1] *= inv; tq[2] *= inv; tq[3] *= inv; } else { tq[0] = tq[1] = tq[2] = 0.f; tq[3] = 1.f; }
    }
    ik_world<NJ>(M, q, tp, tq, M.ik_calls, M.ik_iters);
  }
  const float dt = M.params[P_DT];
#pragma unroll
  for (int i = 0; i < NJ; i++) {
    float t = clampf(q[i], M.ctrl_ll[i], M.ctrl_ul[i]);
    t = clampf(t, q0[i] - M.ctrl_inc[i], q0[i] + M.ctrl_inc[i]);
    st[2 * nd + i] = t;
    st[3 * nd + i] = M.params[P_MOTOR_KP];
    st[4 * nd + i] = M.params[P_ARM_FORCE] * dt;
    target_out[i] = t;
  }
  for (int k = 0; k < M.n_grip; k++) {
    int d = M.grip_dof[k];
    float t = M.grip_mimic[k] >= 0 ? st[M.grip_mimic[k]] : M.grip_scale[k] * grip + M.grip_offset[k];
    st[2 * nd + d] = t;
    st[3 * nd + d] = M.params[P_MOTOR_KP];
    st[4 * nd + d] = M.grip_force[k] * dt;
  }
}

__global__ void __launch_bounds__(128) prb_ik_kernel(const DevModel* __restrict__ Mp, float* __restrict__ state,
                                                      const float* __restrict__ action, float* __restrict__ target_poses, int N) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  const DevModel& M = *Mp;
  float* st = state + (size_t)e * M.state_stride;
  const int adim = action_dim_of((int)(M.params[P_ACTION_TYPE] + 0.5f), M.n_ik);
  if (M.n_ik == 6) ik_action_env<6>(M, st, action + (size_t)e * adim, target_poses + (size_t)e * 6);
  else ik_action_env<7>(M, st, action + (size_t)e * adim, target_poses + (size_t)e * 7);
}

// ============================================================================ state <-> shared memory
template <class WM>
PRB_D void load_state(const DevModel& M, WM& W, const float* st, int lane) {
  const int nd = M.nd;
  for (int i = lane; i < M.state_dim; i += 32) {
    float v = st[i];
    int k = i;
    if (k < nd) { W.q[k] = v; continue; } k -= nd;
    if (k < nd) { W.qd[k] = v; continue; } k -= nd;
    if (k < nd) { W.mtarget[k] = v; continue; } k -= nd;
    if (k < nd) { W.mkp[k] = v; continue; } k -= nd;
    if (k < nd) { W.mmaximp[k] = v; continue; } k -= nd;
    if (k < 13 * M.n_free) {
      int b = k / 13, r = k % 13;
      if (r < 3) W.fpos[b][r] = v; else if (r < 7) W.fquat[b][r - 3] = v; else if (r < 10) W.fvel[b][r - 7] = v; else W.fang[b][r - 10] = v;
      continue;
    }
    k -= 13 * M.n_free;
    if (k < 2 * M.n_slide) { if (k & 1) W.sqd[k >> 1] = v; else W.sq[k >> 1] = v; continue; }
    k -= 2 * M.n_slide;
    if (k < M.goal_dim) { W.goal[k] = v; continue; } k -= M.goal_dim;
    if (k < 8) { W.lastq[k] = v; continue; } k -= 8;
    if (k == 0) W.last_valid = v; else W.reset_count = v;
  }
  __syncwarp();
}
template <class WM>
PRB_D void store_state(const DevModel& M, const WM& W, float* st, int lane) {
  const int nd = M.nd;
  __syncwarp();
  for (int i = lane; i < M.state_dim; i += 32) {
    float v;
    int k = i;
    if (k < nd) v = W.q[k];
    else if ((k -= nd) < nd) v = W.qd[k];
    else if ((k -= nd) < nd) v = W.mtarget[k];
    else if ((k -= nd) < nd) v = W.mkp[k];
    else if ((k -= nd) < nd) v = W.mmaximp[k];
    else if ((k -= nd) < 13 * M.n_free) {
      int b = k / 13, r = k % 13;
      v = r < 3 ? W.fpos[b][r] : (r < 7 ? W.fquat[b][r - 3] : (r < 10 ? W.fvel[b][r - 7] : W.fang[b][r - 10]));
    } else if ((k -= 13 * M.n_free) < 2 * M.n_slide) v = (k & 1) ? W.sqd[k >> 1] : W.sq[k >> 1];
    else if ((k -= 2 * M.n_slide) < M.goal_dim) v = W.goal[k];
    else if ((k -= M.goal_dim) < 8) v = W.lastq[k];
    else v = (k - 8 == 0) ? W.last_valid : W.reset_count;
    st[i] = v;
  }
}

// Free-body constants of one env, fd[FD_N * b + FD_*] (the split pipeline's setup kernel stages them per env; phase_fk
// and phase_vstar read the model's own when fd is NULL)
enum { FD_MASS = 0, FD_INERTIA = 1, FD_LD = 4, FD_AD = 5, FD_N = 6 };

// ============================================================================ kinematics + bias (lane = arm link)
// Each lane walks its own root->link path, accumulating the frame, the velocity and the
// velocity-product acceleration (recursive Newton-Euler forward pass with qdd = 0 and gravity
// folded in as base acceleration); no inter-lane communication.
template <class WM>
PRB_D void phase_fk(const DevModel& M, WM& W, int lane, bool dynamics, const float* fd = nullptr) {
  if (lane < M.nd) {
    m3 R = ldm(M.base_rot);
    v3 p = ld3(M.base_pos);
    v3 w = V3(0, 0, 0), v = V3(0, 0, 0), al = V3(0, 0, 0), ac = V3(0, 0, -M.params[P_GRAVITY_Z]);
    v3 aw = V3(0, 0, 0);
    const int depth = M.depth[lane];
#pragma unroll 1
    for (int k = 0; k < depth; k++) {
      const int j = M.path[lane][k];
      const float qj = W.q[j], qdj = W.qd[j];
      v3 r = mul(R, ld3(M.jpos[j]));
      v3 vo = v + cross(w, r);
      v3 ao = ac + cross(al, r) + cross(w, cross(w, r));
      p = p + r;
      m3 R0 = mul(R, ldm(M.jrot[j]));
      v3 ax = ld3(M.axis[j]);
      aw = mul(R0, ax);
      if (M.jtype[j] == 0) {
        R = mul(R0, axis_angle(ax, qj));
        v3 wj = aw * qdj;
        al = al + cross(w, wj);
        w = w + wj;
        v = vo; ac = ao;
      } else {
        R = R0;
        v3 d = aw * qj, dd = aw * qdj;
        p = p + d;
        v = vo + cross(w, d) + dd;
        ac = ao + cross(al, d) + cross(w, cross(w, d)) + cross(w, dd) * 2.0f;
      }
    }
    stm(W.lR[lane], R); st3(W.lp[lane], p); st3(W.la[lane], aw); st3(W.lw[lane], w); st3(W.lv[lane], v);
    v3 rc = mul(R, ld3(M.com[lane]));
    st3(W.lc[lane], p + rc);
    if (dynamics) {
      float Iw[6];
      rot_sym(R, M.inertia[lane], Iw);
      for (int k = 0; k < 6; k++) W.lIw[lane][k] = Iw[k];
      v3 acom = ac + cross(al, rc) + cross(w, cross(w, rc));
      st3(W.lf[lane], acom * M.mass[lane]);
      st3(W.ln[lane], symmul(Iw, al) + cross(w, symmul(Iw, w)));
    }
  }
  // free / slide body frames (lanes past the arm)
  int b = lane - M.nd;
  if (b >= 0 && b < M.n_free) {
    m3 R; quat_to_mat(W.fquat[b], R); stm(W.fR[b], R);
    if (dynamics) {
      const float* I = fd ? fd + FD_N * b + FD_INERTIA : M.free_inertia[b];
      float Dg[6] = {1.0f / I[0], 0, 0, 1.0f / I[1], 0, 1.0f / I[2]}, o[6];
      rot_sym(R, Dg, o);
      for (int k = 0; k < 6; k++) W.fIinv[b][k] = o[k];
    }
  }
  int s = lane - M.nd - M.n_free;
  if (s >= 0 && s < M.n_slide) {
    m3 R0 = ldm(M.slide_rot[s]);
    v3 ax = ld3(M.slide_axis[s]), p0 = ld3(M.slide_pos[s]);
    if (M.slide_jtype[s] == 0) { stm(W.sR[s], mul(R0, axis_angle(ax, W.sq[s]))); st3(W.sp[s], p0); }
    else { stm(W.sR[s], R0); st3(W.sp[s], p0 + ld3(M.slide_axis_w[s]) * W.sq[s]); }
  }
  __syncwarp();
}

// Joint j's bias torque tau_j (the velocity-product and gravity term h_j of tau = M qdd + h) and mass-matrix row j
// (W.Mm[j][k] and W.Mm[k][j], k <= j), by direct sums over subtree(j).  put(tau_j) runs where the step stores its
// generalized force, so that phase_crba and prb_arm_kernel share this arithmetic and its order.
template <class WM, class PUT>
PRB_D void crba_joint(const DevModel& M, WM& W, int j, PUT put) {
  const int nd = M.nd;
  const bool rev = M.jtype[j] == 0;
  const v3 aj = ld3(W.la[j]), pj = ld3(W.lp[j]);
  float tau = 0;
  v3 P = V3(0, 0, 0), L = V3(0, 0, 0);
  unsigned mask = M.sub_mask[j];
#pragma unroll 1
  for (int i = j; i < nd; i++) {
    if (!((mask >> i) & 1u)) continue;
    v3 ci = ld3(W.lc[i]), fi = ld3(W.lf[i]), ni = ld3(W.ln[i]);
    v3 rc = ci - pj;
    tau += rev ? dot(aj, ni + cross(rc, fi)) : dot(aj, fi);
    float mi = M.mass[i];
    v3 ui = rev ? cross(aj, rc) : aj;
    v3 pm = ui * mi;
    P = P + pm;
    L = L + cross(rc, pm);
    if (rev) L = L + symmul(W.lIw[i], aj);
  }
  put(tau);
  unsigned anc = M.anc_mask[j];
#pragma unroll 1
  for (int k = 0; k <= j; k++) {
    float val = 0.f;
    if ((anc >> k) & 1u) {
      v3 ak = ld3(W.la[k]);
      val = M.jtype[k] == 0 ? dot(ak, L + cross(pj - ld3(W.lp[k]), P)) : dot(ak, P);
    }
    W.Mm[j][k] = val;
    W.Mm[k][j] = val;
  }
}

// generalized bias forces W.Q = -tau - jdamp qd and the mass matrix W.Mm (lane = joint j)
template <class WM>
PRB_D void phase_crba(const DevModel& M, WM& W, int lane) {
  if (lane < M.nd) crba_joint(M, W, lane, [&](float tau) { W.Q[lane] = -tau - M.jdamp[lane] * W.qd[lane]; });
  __syncwarp();
}

// Cholesky M = L L^T (lane = row: the row lives in registers, the pivot column travels by shuffle; same operations in
// the same order as the textbook in-place loop), then lane c solves for column c of M^-1
template <int ND, class WM>
PRB_D void phase_minv(WM& W, int lane) {
  {
    float Lr[ND];
    const int row = lane < ND ? lane : ND - 1;        // idle lanes shadow the last row; nothing of theirs is stored
#pragma unroll
    for (int c = 0; c < ND; c++) Lr[c] = W.Mm[row][c];
#pragma unroll
    for (int k = 0; k < ND; k++) {
      const float d = sqrtf(__shfl_sync(FULL, Lr[k], k));
      if (lane == k) Lr[k] = d;
      else if (lane > k) Lr[k] = Lr[k] / d;
#pragma unroll
      for (int c = k + 1; c < ND; c++) {
        const float lck = __shfl_sync(FULL, Lr[k], c);
        if (lane > k && c <= lane) Lr[c] -= Lr[k] * lck;
      }
    }
    __syncwarp();
    if (lane < ND) {
#pragma unroll
      for (int c = 0; c < ND; c++) if (c <= lane) W.Mm[lane][c] = Lr[c];
    }
    __syncwarp();
  }
  if (lane < ND) {
    float x[ND];
#pragma unroll
    for (int r = 0; r < ND; r++) {
      float s = (r == lane) ? 1.0f : 0.0f;
#pragma unroll
      for (int m = 0; m < r; m++) s -= W.Mm[r][m] * x[m];
      x[r] = s / W.Mm[r][r];
    }
#pragma unroll
    for (int r = ND - 1; r >= 0; r--) {
      float s = x[r];
#pragma unroll
      for (int m = r + 1; m < ND; m++) s -= W.Mm[m][r] * x[m];
      x[r] = s / W.Mm[r][r];
    }
#pragma unroll
    for (int r = 0; r < ND; r++) W.Minv[r][lane] = x[r];
  }
  __syncwarp();
}

// unconstrained velocity update v* = v + dt * a  (lane = velocity DoF); result in W.vs and returned
template <class WM>
PRB_D float phase_vstar(const DevModel& M, WM& W, int lane, const float* fd = nullptr) {
  const float dt = M.params[P_DT], g = M.params[P_GRAVITY_Z], vmax = M.params[P_MAX_COORD_VEL];
  const int nd = M.nd;
  // free bodies: one lane per body does the coupled 3-vector algebra
  int b = lane - nd;
  if (b >= 0 && b < M.n_free) {
    m3 R = ldm(W.fR[b]);
    float kl = fd ? fd[FD_N * b + FD_LD] : M.free_ld[b], ka = fd ? fd[FD_N * b + FD_AD] : M.free_ad[b];
    v3 vl = ld3(W.fvel[b]), w = ld3(W.fang[b]);
    v3 acc = V3(0, 0, g) + vl * (-(kl + kl * norm(vl)));
    v3 wb = tmul(R, w);
    v3 Id = ld3(fd ? fd + FD_N * b + FD_INERTIA : M.free_inertia[b]);
    v3 gy = cross(wb, V3(Id.x * wb.x, Id.y * wb.y, Id.z * wb.z));
    v3 wdb = V3(-gy.x / Id.x, -gy.y / Id.y, -gy.z / Id.z) + wb * (-(ka + ka * norm(wb)));
    v3 wd = mul(R, wdb);
    int o = nd + 6 * b;
    W.vs[o] = clampf(vl.x + dt * acc.x, -vmax, vmax); W.vs[o + 1] = clampf(vl.y + dt * acc.y, -vmax, vmax);
    W.vs[o + 2] = clampf(vl.z + dt * acc.z, -vmax, vmax); W.vs[o + 3] = clampf(w.x + dt * wd.x, -vmax, vmax);
    W.vs[o + 4] = clampf(w.y + dt * wd.y, -vmax, vmax); W.vs[o + 5] = clampf(w.z + dt * wd.z, -vmax, vmax);
  }
  float v = 0.f;
  if (lane < nd) {
    float acc = 0;
    for (int j = 0; j < nd; j++) acc += W.Minv[lane][j] * W.Q[j];
    v = clampf(W.qd[lane] + dt * acc, -vmax, vmax);
    W.vs[lane] = v;
  }
  int s = lane - nd - 6 * M.n_free;
  if (s >= 0 && s < M.n_slide) {
    float a;
    if (M.slide_jtype[s] == 1) a = g * M.slide_axis_w[s][2];
    else { float ka = M.slide_ad[s], w = W.sqd[s]; a = -w * (ka + ka * fabsf(w)); }
    v = clampf(W.sqd[s] + dt * a, -vmax, vmax);
    W.vs[lane] = v;
  }
  __syncwarp();
  if (lane < M.nv) v = W.vs[lane];
  return v;
}

// ============================================================================ collision
template <class WM>
PRB_D void body_frame(const DevModel& M, const WM& W, int body, int link, m3& R, v3& p) {
  if (body < 0) { R = ident3(); p = V3(0, 0, 0); }
  else if (body == 0) {
    if (link < 0) { R = ldm(M.base_rot); p = ld3(M.base_pos); }
    else { R = ldm(W.lR[link]); p = ld3(W.lp[link]); }
  } else if (body <= M.n_free) { R = ldm(W.fR[body - 1]); p = ld3(W.fpos[body - 1]); }
  else { R = ldm(W.sR[body - 1 - M.n_free]); p = ld3(W.sp[body - 1 - M.n_free]); }
}
template <class WM>
PRB_D void collider_frame(const DevModel& M, const WM& W, int c, m3& R, v3& p) {
  m3 Rb; v3 pb;
  body_frame(M, W, M.col_body[c], M.col_link[c], Rb, pb);
  R = mul(Rb, ldm(M.col_rot[c]));
  p = pb + mul(Rb, ld3(M.col_pos[c]));
}

struct CPoint { v3 pos, n; float depth; };

// clip the quad p (4 2-D points) against the rectangle +-h; returns the number of points in ret
PRB_DN int clip_quad(const float h[2], const float p_in[8], float ret[16]) {
  int nq = 4, nr = 0;
  float buffer[16];
  const float* q = p_in;
  float* r = ret;
  for (int dir = 0; dir <= 1; dir++) {
    for (int sign = -1; sign <= 1; sign += 2) {
      const float* pq = q;
      float* pr = r;
      nr = 0;
      bool full = false;
      for (int i = nq; i > 0 && !full; i--) {
        if (sign * pq[dir] < h[dir]) {
          pr[0] = pq[0]; pr[1] = pq[1]; pr += 2; nr++;
          if (nr & 8) { full = true; break; }
        }
        const float* nextq = (i > 1) ? pq + 2 : q;
        if ((sign * pq[dir] < h[dir]) ^ (sign * nextq[dir] < h[dir])) {
          pr[1 - dir] = pq[1 - dir] + (nextq[1 - dir] - pq[1 - dir]) / (nextq[dir] - pq[dir]) * (sign * h[dir] - pq[dir]);
          pr[dir] = sign * h[dir];
          pr += 2; nr++;
          if (nr & 8) { full = true; break; }
        }
        pq += 2;
      }
      q = r;
      if (full) goto done;
      r = (q == ret) ? buffer : ret;
      nq = nr;
    }
  }
done:
  if (q != ret) for (int i = 0; i < nr * 2; i++) ret[i] = q[i];
  return nr;
}
PRB_DN void cull_points(int n, const float p[], int m, int i0, int iret[]) {
  float a, cx, cy, q;
  if (n == 1) { cx = p[0]; cy = p[1]; }
  else if (n == 2) { cx = 0.5f * (p[0] + p[2]); cy = 0.5f * (p[1] + p[3]); }
  else {
    a = 0; cx = 0; cy = 0;
    for (int i = 0; i < n - 1; i++) {
      q = p[i * 2] * p[i * 2 + 3] - p[i * 2 + 2] * p[i * 2 + 1];
      a += q; cx += q * (p[i * 2] + p[i * 2 + 2]); cy += q * (p[i * 2 + 1] + p[i * 2 + 3]);
    }
    q = p[n * 2 - 2] * p[1] - p[0] * p[n * 2 - 1];
    if (fabsf(a + q) > 1.1920929e-7f) a = 1.0f / (3.0f * (a + q)); else a = 1e18f;
    cx = a * (cx + q * (p[n * 2 - 2] + p[0])); cy = a * (cy + q * (p[n * 2 - 1] + p[1]));
  }
  float A[8]; int avail[8];
  for (int i = 0; i < n; i++) { A[i] = atan2f(p[i * 2 + 1] - cy, p[i * 2] - cx); avail[i] = 1; }
  avail[i0] = 0; iret[0] = i0; iret++;
  for (int j = 1; j < m; j++) {
    a = j * (2 * PRB_PI_F / m) + A[i0];
    if (a > PRB_PI_F) a -= 2 * PRB_PI_F;
    float maxdiff = 1e9f, diff; *iret = i0;
    for (int i = 0; i < n; i++) if (avail[i]) {
      diff = fabsf(A[i] - a); if (diff > PRB_PI_F) diff = 2 * PRB_PI_F - diff;
      if (diff < maxdiff - 1e-5f) { maxdiff = diff; *iret = i; }                               // ties: the first point wins
    }
    avail[*iret] = 0; iret++;
  }
}
// box-box: separating-axis search + face clipping / edge-edge closest points; normal from box 2
// (B) to box 1 (A), points on B, depth >= 0; at most 4 points.
PRB_DN int box_box(v3 p1, const m3& R1, v3 h1, v3 p2, const m3& R2, v3 h2, CPoint* out) {
  // TIE: a later axis replaces the current best only if it separates by 1 um more.  Resting boxes tie structurally (the
  // table's top face and the block's bottom face are the same axis); with Bullet's plain `>` the winner - and with it the
  // ORDER of the clipped points, which a 50-sweep Gauss-Seidel is sensitive to - is decided by the last rounding error,
  // differently in fp32 and fp64.  The oracle applies the same rule.
  const float fudge = 1.05f, EPS = 1.1920929e-7f, TIE = 1e-6f;
  float A[3] = {h1.x, h1.y, h1.z}, B[3] = {h2.x, h2.y, h2.z};
  v3 p = p2 - p1, ppv3 = tmul(R1, p);
  float pp[3] = {ppv3.x, ppv3.y, ppv3.z};
  float Rm[3][3], Q[3][3];
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) { Rm[i][j] = dot(col(R1, i), col(R2, j)); Q[i][j] = fabsf(Rm[i][j]); }
  float s = -1e30f, s2, l;
  int invert = 0, code = 0, nrm_box = 0, nrm_col = 0;
  v3 normalC = V3(0, 0, 0);
#define PRB_TST(e1, e2, bx, cl, cc) { float E1 = (e1); s2 = fabsf(E1) - (e2); if (s2 > 0) return 0; \
    if (s2 > s + TIE) { s = s2; nrm_box = bx; nrm_col = cl; invert = (E1 < 0); code = (cc); } }
  PRB_TST(pp[0], (A[0] + B[0] * Q[0][0] + B[1] * Q[0][1] + B[2] * Q[0][2]), 1, 0, 1);
  PRB_TST(pp[1], (A[1] + B[0] * Q[1][0] + B[1] * Q[1][1] + B[2] * Q[1][2]), 1, 1, 2);
  PRB_TST(pp[2], (A[2] + B[0] * Q[2][0] + B[1] * Q[2][1] + B[2] * Q[2][2]), 1, 2, 3);
  PRB_TST(dot(col(R2, 0), p), (A[0] * Q[0][0] + A[1] * Q[1][0] + A[2] * Q[2][0] + B[0]), 2, 0, 4);
  PRB_TST(dot(col(R2, 1), p), (A[0] * Q[0][1] + A[1] * Q[1][1] + A[2] * Q[2][1] + B[1]), 2, 1, 5);
  PRB_TST(dot(col(R2, 2), p), (A[0] * Q[0][2] + A[1] * Q[1][2] + A[2] * Q[2][2] + B[2]), 2, 2, 6);
#undef PRB_TST
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) Q[i][j] += 1.0e-5f;
#define PRB_TST(e1, e2, n1, n2, n3, cc) { float E1 = (e1); s2 = fabsf(E1) - (e2); if (s2 > EPS) return 0; \
    l = sqrtf((n1) * (n1) + (n2) * (n2) + (n3) * (n3)); \
    if (l > EPS) { s2 /= l; if (s2 * fudge > s + TIE) { s = s2; nrm_box = 0; normalC = V3((n1) / l, (n2) / l, (n3) / l); invert = (E1 < 0); code = (cc); } } }
  PRB_TST(pp[2] * Rm[1][0] - pp[1] * Rm[2][0], (A[1] * Q[2][0] + A[2] * Q[1][0] + B[1] * Q[0][2] + B[2] * Q[0][1]), 0, -Rm[2][0], Rm[1][0], 7);
  PRB_TST(pp[2] * Rm[1][1] - pp[1] * Rm[2][1], (A[1] * Q[2][1] + A[2] * Q[1][1] + B[0] * Q[0][2] + B[2] * Q[0][0]), 0, -Rm[2][1], Rm[1][1], 8);
  PRB_TST(pp[2] * Rm[1][2] - pp[1] * Rm[2][2], (A[1] * Q[2][2] + A[2] * Q[1][2] + B[0] * Q[0][1] + B[1] * Q[0][0]), 0, -Rm[2][2], Rm[1][2], 9);
  PRB_TST(pp[0] * Rm[2][0] - pp[2] * Rm[0][0], (A[0] * Q[2][0] + A[2] * Q[0][0] + B[1] * Q[1][2] + B[2] * Q[1][1]), Rm[2][0], 0, -Rm[0][0], 10);
  PRB_TST(pp[0] * Rm[2][1] - pp[2] * Rm[0][1], (A[0] * Q[2][1] + A[2] * Q[0][1] + B[0] * Q[1][2] + B[2] * Q[1][0]), Rm[2][1], 0, -Rm[0][1], 11);
  PRB_TST(pp[0] * Rm[2][2] - pp[2] * Rm[0][2], (A[0] * Q[2][2] + A[2] * Q[0][2] + B[0] * Q[1][1] + B[1] * Q[1][0]), Rm[2][2], 0, -Rm[0][2], 12);
  PRB_TST(pp[1] * Rm[0][0] - pp[0] * Rm[1][0], (A[0] * Q[1][0] + A[1] * Q[0][0] + B[1] * Q[2][2] + B[2] * Q[2][1]), -Rm[1][0], Rm[0][0], 0, 13);
  PRB_TST(pp[1] * Rm[0][1] - pp[0] * Rm[1][1], (A[0] * Q[1][1] + A[1] * Q[0][1] + B[0] * Q[2][2] + B[2] * Q[2][0]), -Rm[1][1], Rm[0][1], 0, 14);
  PRB_TST(pp[1] * Rm[0][2] - pp[0] * Rm[1][2], (A[0] * Q[1][2] + A[1] * Q[0][2] + B[0] * Q[2][1] + B[1] * Q[2][0]), -Rm[1][2], Rm[0][2], 0, 15);
#undef PRB_TST
  if (!code) return 0;
  v3 normal = nrm_box == 1 ? col(R1, nrm_col) : (nrm_box == 2 ? col(R2, nrm_col) : mul(R1, normalC));
  if (invert) normal = normal * -1.0f;
  float depth = -s;
  if (code > 6) {
    v3 pa = p1, pb = p2;
    for (int j = 0; j < 3; j++) { float sg = dot(normal, col(R1, j)) > 0 ? 1.0f : -1.0f; pa = pa + col(R1, j) * (sg * A[j]); }
    for (int j = 0; j < 3; j++) { float sg = dot(normal, col(R2, j)) > 0 ? -1.0f : 1.0f; pb = pb + col(R2, j) * (sg * B[j]); }
    v3 ua = col(R1, (code - 7) / 3), ub = col(R2, (code - 7) % 3);
    v3 dpp = pb - pa;
    float uaub = dot(ua, ub), q1 = dot(ua, dpp), q2 = -dot(ub, dpp), d = 1 - uaub * uaub;
    float beta = d <= 0.0001f ? 0.f : (uaub * q1 + q2) / d;
    out[0].pos = pb + ub * beta; out[0].n = normal * -1.0f; out[0].depth = depth;
    return 1;
  }
  const bool first = code <= 3;
  const m3& Ra = first ? R1 : R2;
  const m3& Rb = first ? R2 : R1;
  v3 pa = first ? p1 : p2, pb = first ? p2 : p1;
  const float* Sa = first ? A : B;
  const float* Sb = first ? B : A;
  v3 normal2 = first ? normal : normal * -1.0f;
  v3 nr = tmul(Rb, normal2);
  float anr[3] = {fabsf(nr.x), fabsf(nr.y), fabsf(nr.z)};
  int lanr, a1, a2;
  if (anr[1] > anr[0]) { if (anr[1] > anr[2]) { a1 = 0; lanr = 1; a2 = 2; } else { a1 = 0; a2 = 1; lanr = 2; } }
  else { if (anr[0] > anr[2]) { lanr = 0; a1 = 1; a2 = 2; } else { a1 = 0; a2 = 1; lanr = 2; } }
  v3 center = comp(nr, lanr) < 0 ? (pb - pa) + col(Rb, lanr) * Sb[lanr] : (pb - pa) - col(Rb, lanr) * Sb[lanr];
  int codeN = first ? code - 1 : code - 4, code1, code2;
  if (codeN == 0) { code1 = 1; code2 = 2; } else if (codeN == 1) { code1 = 0; code2 = 2; } else { code1 = 0; code2 = 1; }
  float quad[8], c1 = dot(center, col(Ra, code1)), c2 = dot(center, col(Ra, code2));
  float m11 = dot(col(Ra, code1), col(Rb, a1)), m12 = dot(col(Ra, code1), col(Rb, a2));
  float m21 = dot(col(Ra, code2), col(Rb, a1)), m22 = dot(col(Ra, code2), col(Rb, a2));
  {
    float k1 = m11 * Sb[a1], k2 = m21 * Sb[a1], k3 = m12 * Sb[a2], k4 = m22 * Sb[a2];
    quad[0] = c1 - k1 - k3; quad[1] = c2 - k2 - k4; quad[2] = c1 - k1 + k3; quad[3] = c2 - k2 + k4;
    quad[4] = c1 + k1 + k3; quad[5] = c2 + k2 + k4; quad[6] = c1 + k1 - k3; quad[7] = c2 + k2 - k4;
  }
  float rect[2] = {Sa[code1], Sa[code2]}, ret[16];
  int n = clip_quad(rect, quad, ret);
  if (n < 1) return 0;
  float point[24], dep[8], det1 = 1.0f / (m11 * m22 - m12 * m21);
  m11 *= det1; m12 *= det1; m21 *= det1; m22 *= det1;
  int cnum = 0;
  for (int j = 0; j < n; j++) {
    float k1 = m22 * (ret[j * 2] - c1) - m12 * (ret[j * 2 + 1] - c2);
    float k2 = -m21 * (ret[j * 2] - c1) + m11 * (ret[j * 2 + 1] - c2);
    v3 pt = center + col(Rb, a1) * k1 + col(Rb, a2) * k2;
    float d = Sa[codeN] - dot(normal2, pt);
    if (d >= 0) {
      point[cnum * 3] = pt.x; point[cnum * 3 + 1] = pt.y; point[cnum * 3 + 2] = pt.z;
      dep[cnum] = d; ret[cnum * 2] = ret[j * 2]; ret[cnum * 2 + 1] = ret[j * 2 + 1]; cnum++;
    }
  }
  if (cnum < 1) return 0;
  int idx[8], m = cnum;
  if (cnum > 4) {
    int i1 = 0; float maxd = dep[0];
    for (int i = 1; i < cnum; i++) if (dep[i] > maxd + 1e-7f) { maxd = dep[i]; i1 = i; }      // ties: the first point wins (as in the oracle)
    cull_points(cnum, ret, 4, i1, idx); m = 4;
  } else for (int i = 0; i < cnum; i++) idx[i] = i;
  for (int j = 0; j < m; j++) {
    int i = idx[j];
    v3 pw = V3(point[i * 3], point[i * 3 + 1], point[i * 3 + 2]) + pa;
    if (code >= 4) pw = pw - normal * dep[i];
    out[j].pos = pw; out[j].n = normal * -1.0f; out[j].depth = dep[i];
  }
  return m;
}

// collider AABBs -> broad phase over the static pair list -> narrow phase (lane = pair) ->
// contacts compacted in pair order (deterministic: the PGS sweep order depends on it)
// Manifold reduction ties: candidates closer than 2 um in depth / distance / height over the longest edge count as
// equal and the first one (pair order) wins (DESIGN.md, tie rules: the parity checker applies the same rule in fp64).
constexpr float MTIE = 2e-6f;
template <class WM>
PRB_D void phase_collide_broad(const DevModel& M, WM& W, int lane) {
#pragma unroll 1
  for (int c = lane; c < M.n_col; c += 32) {
    m3 R; v3 p;
    collider_frame(M, W, c, R, p);
    v3 h = ld3(M.col_half[c]);
    v3 e = V3(fabsf(R.m[0]) * h.x + fabsf(R.m[1]) * h.y + fabsf(R.m[2]) * h.z,
              fabsf(R.m[3]) * h.x + fabsf(R.m[4]) * h.y + fabsf(R.m[5]) * h.z,
              fabsf(R.m[6]) * h.x + fabsf(R.m[7]) * h.y + fabsf(R.m[8]) * h.z);
    W.aabb[c][0] = make_float2(p.x - e.x, p.x + e.x); W.aabb[c][1] = make_float2(p.y - e.y, p.y + e.y); W.aabb[c][2] = make_float2(p.z - e.z, p.z + e.z);
  }
  __syncwarp();
  int n_ovl = 0;
  // lane = pair, four groups of 32 pairs per trip: the eight index loads of a trip are issued together, ahead of the tests
#pragma unroll 1
  for (int base = 0; base < M.n_pair; base += 128) {
    int ia[4], ib[4];
#pragma unroll
    for (int g = 0; g < 4; g++) {
      const int k = base + 32 * g + lane;
      const bool in = k < M.n_pair;
      ia[g] = in ? (int)M.pair_a[k] : 0; ib[g] = in ? (int)M.pair_b[k] : 0;
    }
#pragma unroll
    for (int g = 0; g < 4; g++) {
      if (base + 32 * g < M.n_pair) {                  // warp-uniform
        const int k = base + 32 * g + lane;
        const float2 ax = W.aabb[ia[g]][0], ay = W.aabb[ia[g]][1], az = W.aabb[ia[g]][2];
        const float2 bx = W.aabb[ib[g]][0], by = W.aabb[ib[g]][1], bz = W.aabb[ib[g]][2];
        const bool hit = k < M.n_pair && !(ax.x > bx.y || ax.y < bx.x || ay.x > by.y || ay.y < by.x || az.x > bz.y || az.y < bz.x);
        const unsigned bal = __ballot_sync(FULL, hit);
        if (hit) {
          const int slot = n_ovl + __popc(bal & ((1u << lane) - 1u));
          if (slot < WM::Cfg::MAXOVL) W.ovl[slot] = (unsigned short)k; else W.overflow |= 1;      // bit 0: overlapping pairs
        }
        n_ovl += __popc(bal);
      }
    }
  }
  if (n_ovl > WM::Cfg::MAXOVL) n_ovl = WM::Cfg::MAXOVL;
  if (lane == 0) W.n_ovl = n_ovl;
  __syncwarp();
}

// second half of the collision phase (its own function: the setup kernel re-aligns the warps of a block between the halves)
template <class WM>
PRB_D void phase_collide_narrow(const DevModel& M, WM& W, int lane) {
  const int n_ovl = W.n_ovl;
  // narrow phase: lane = overlapping pair, in passes of 32 pairs (a second pass only when more than 32 pairs overlap;
  // ONE loop body: this kernel is instruction-fetch sensitive, unrolled copies of rarely taken passes cost time).
  // Candidates are appended in pair order.  The same pass marks where the runs of equal object pair begin (the pair
  // list is sorted by object pair, so runs are contiguous) and writes the run table over the consumed part of W.ovl.
  int total = 0, n_runs = 0, carry_key = -2;
#pragma unroll 1
  for (int h = 0; h * 32 < n_ovl; h++) {
    const int idx = h * 32 + lane;
    CPoint cp[4];
    int n = 0, ca = 0, cb = 0, key = -1;
    if (idx < n_ovl) {
      int k = W.ovl[idx];
      ca = M.pair_a[k]; cb = M.pair_b[k];
      m3 Ra, Rb; v3 pa, pb;
      collider_frame(M, W, ca, Ra, pa);
      collider_frame(M, W, cb, Rb, pb);
      n = box_box(pa, Ra, ld3(M.col_half[ca]), pb, Rb, ld3(M.col_half[cb]), cp);
      key = (int)M.col_obj[ca] << 8 | (int)M.col_obj[cb];
    }
    int tot;
    const int off = total + warp_excl_scan(n, lane, &tot);
    total += tot;
    for (int i = 0; i < n; i++) {
      if (off + i >= WM::Cfg::MAXCAND) { W.overflow |= 1; break; }     // (only reachable with 64 pairs: 4 x 32 candidates always fit)
      Contact& c = W.cand[off + i];
      c.pbx = cp[i].pos.x; c.pby = cp[i].pos.y; c.pbz = cp[i].pos.z;
      c.nx = cp[i].n.x; c.ny = cp[i].n.y; c.nz = cp[i].n.z; c.dist = -cp[i].depth; c.cols = ca | (cb << 8);
    }
    int prev_key = __shfl_up_sync(FULL, key, 1);
    if (lane == 0) prev_key = carry_key;
    carry_key = __shfl_sync(FULL, key, 31);
    const bool run_start = idx < n_ovl && key != prev_key;
    const unsigned startmask = __ballot_sync(FULL, run_start);
    __syncwarp();                                  // every lane has read its pair index: entries <= idx of W.ovl are free
    if (run_start) W.ovl[n_runs + __popc(startmask & ((1u << lane) - 1u))] = (unsigned short)(off < WM::Cfg::MAXCAND ? off : WM::Cfg::MAXCAND);
    n_runs += __popc(startmask);                   // (run index <= pair index: the table never overtakes the unread pairs)
  }
  const int ncand = total < WM::Cfg::MAXCAND ? total : WM::Cfg::MAXCAND;
  __syncwarp();
  // ---- manifold reduction: <= 4 points per pair of collision objects; lane = run reduces it, then an ordered
  //      compaction into ct[]
  int total2 = 0;
#pragma unroll 1
  for (int h = 0; h * 32 < n_runs; h++) {
    const int r = h * 32 + lane;
    int keep[4] = {0, 0, 0, 0}, m = 0;
    if (r < n_runs) {
      int b0 = W.ovl[r], b1 = (r + 1 < n_runs) ? (int)W.ovl[r + 1] : ncand;
      if (b0 > ncand) b0 = ncand;
      if (b1 > ncand) b1 = ncand;
      int nn = b1 - b0;
      const Contact* c = &W.cand[b0];
      if (nn <= 4) { m = nn; for (int i = 0; i < nn; i++) keep[i] = b0 + i; }
      else {
        int i0 = 0;
        for (int i = 1; i < nn; i++) if (c[i].dist < c[i0].dist - MTIE) i0 = i;     // ties: the first candidate wins
        v3 p0 = V3(c[i0].pbx, c[i0].pby, c[i0].pbz);
        int i1 = -1; float best = -1.f;
        for (int i = 0; i < nn; i++) if (i != i0) { v3 d = V3(c[i].pbx, c[i].pby, c[i].pbz) - p0; float v = norm(d); if (v > best + MTIE) { best = v; i1 = i; } }
        v3 p1 = V3(c[i1].pbx, c[i1].pby, c[i1].pbz), e01 = p1 - p0;
        const float atol = norm(e01) * MTIE;   // an area tolerance: MTIE of height over the longest edge
        int i2 = -1; best = -1.f;
        for (int i = 0; i < nn; i++) if (i != i0 && i != i1) { v3 x = cross(V3(c[i].pbx, c[i].pby, c[i].pbz) - p0, e01); float v = norm(x); if (v > best + atol) { best = v; i2 = i; } }
        v3 p2 = V3(c[i2].pbx, c[i2].pby, c[i2].pbz);
        int i3 = -1; best = -1.f;
        for (int i = 0; i < nn; i++) if (i != i0 && i != i1 && i != i2) {
          v3 pi = V3(c[i].pbx, c[i].pby, c[i].pbz), a = pi - p0, b = pi - p1, d = pi - p2;
          float v = norm(cross(a, b)) + norm(cross(b, d)) + norm(cross(d, a));
          if (v > best + 4.f * atol) { best = v; i3 = i; }
        }
        for (int i = 0; i < nn; i++) if (i == i0 || i == i1 || i == i2 || i == i3) keep[m++] = b0 + i;
      }
    }
    int t2;
    const int first = warp_excl_scan(m, lane, &t2);     // this run's first output, relative to the pass
    // Copy in order of destination, 32 destinations per trip: lane = destination, its source from the run that owns it
    // (the last lane whose first output is <= it).  ct may be the head of cand (SetupMemT): a contact's source is never
    // before its destination, so a trip's writes land only on sources of this or an earlier trip (read before the
    // __syncwarp) and never on those of later trips or passes.  (Lanes that each wrote their own run's contacts could
    // overwrite one that another lane of the pass has still to read.)
#pragma unroll 1
    for (int base = 0; base < t2 && total2 + base < WM::Cfg::MAXCONTACT; base += 32) {
      const int rel = base + lane;
      int own = 0;
#pragma unroll
      for (int s = 16; s > 0; s >>= 1) if (__shfl_sync(FULL, first, own + s) <= rel) own += s;
      const int i = rel - __shfl_sync(FULL, first, own);
      const int k0 = __shfl_sync(FULL, keep[0], own), k1 = __shfl_sync(FULL, keep[1], own);
      const int k2 = __shfl_sync(FULL, keep[2], own), k3 = __shfl_sync(FULL, keep[3], own);
      const int dst = total2 + rel, src = i == 0 ? k0 : (i == 1 ? k1 : (i == 2 ? k2 : k3));
      Contact kc;
      if (rel < t2 && dst < WM::Cfg::MAXCONTACT) kc = W.cand[src];
      __syncwarp();
      if (rel < t2 && dst < WM::Cfg::MAXCONTACT) W.ct[dst] = kc;
    }
    total2 += t2;
  }
  if (lane == 0) {
    W.n_contact = total2 < WM::Cfg::MAXCONTACT ? total2 : WM::Cfg::MAXCONTACT;
    if (total2 > WM::Cfg::MAXCONTACT) W.overflow |= 2;                                           // bit 1: contacts
  }
  __syncwarp();
}

template <class WM>
PRB_D void phase_collide(const DevModel& M, WM& W, int lane) {
  phase_collide_broad(M, W, lane);
  phase_collide_narrow(M, W, lane);
}

// ============================================================================ constraint rows
// Jacobian of a unit force `dir` at world point pt (or unit torque when angular) on the body of
// collider `col`, written as (J, B = M^-1 J^T) segment; returns J.B and accumulates J.v*
template <class WM>
PRB_DN float fill_segment(const DevModel& M, const WM& W, int col, v3 pt, v3 dir, float sign, bool angular,
                         float* seg, float* rel) {
  const int body = M.col_body[col];
  float d = 0.f;
  if (body == 0) {
    const int link = M.col_link[col], nd = M.nd;
    float* J = seg; float* B = seg + nd;
    unsigned anc = M.anc_mask[link];
    for (int j = 0; j < nd; j++) {
      float g = 0.f;
      if ((anc >> j) & 1u) {
        v3 aj = ld3(W.la[j]);
        if (M.jtype[j] == 0) g = angular ? dot(aj, dir) : dot(aj, cross(pt - ld3(W.lp[j]), dir));
        else g = angular ? 0.f : dot(aj, dir);
      }
      J[j] = sign * g;
    }
    for (int i = 0; i < nd; i++) {
      float s = 0.f;
      for (int j = 0; j < nd; j++) s += W.Minv[i][j] * J[j];
      B[i] = s;
    }
    for (int j = 0; j < nd; j++) { d += J[j] * B[j]; *rel += J[j] * W.vs[j]; }
  } else if (body <= M.n_free) {
    const int b = body - 1, o = M.nd + 6 * b;
    float* J = seg; float* B = seg + 6;
    v3 t = angular ? dir : cross(pt - ld3(W.fpos[b]), dir);
    v3 jl = angular ? V3(0, 0, 0) : dir * sign, ja = t * sign;
    float im = 1.0f / M.free_mass[b];
    v3 bl = jl * im, ba = symmul(W.fIinv[b], ja);
    J[0] = jl.x; J[1] = jl.y; J[2] = jl.z; J[3] = ja.x; J[4] = ja.y; J[5] = ja.z;
    B[0] = bl.x; B[1] = bl.y; B[2] = bl.z; B[3] = ba.x; B[4] = ba.y; B[5] = ba.z;
    for (int k = 0; k < 6; k++) { d += J[k] * B[k]; *rel += J[k] * W.vs[o + k]; }
  } else {
    const int s = body - 1 - M.n_free, o = M.nd + 6 * M.n_free + s;
    v3 a = ld3(M.slide_axis_w[s]);
    float g;
    if (M.slide_jtype[s] == 0) g = angular ? dot(a, dir) : dot(a, cross(pt - ld3(W.sp[s]), dir));
    else g = angular ? 0.f : dot(a, dir);
    seg[0] = sign * g; seg[1] = sign * g * M.slide_minv[s];
    d = seg[0] * seg[1]; *rel += seg[0] * W.vs[o];
  }
  return d;
}
PRB_D int col_dyn_body(const DevModel& M, int col) {  // -1 when the collider cannot move
  int b = M.col_body[col];
  if (b < 0 || (b == 0 && M.col_link[col] < 0)) return -1;
  return b;
}
PRB_D void plane_space(v3 n, v3& p, v3& q) {
  if (fabsf(n.z) > 0.70710678f) {
    float a = n.y * n.y + n.z * n.z, k = 1.0f / sqrtf(a);
    p = V3(0, -n.z * k, n.y * k);
    q = V3(a * k, -n.x * p.z, n.x * p.y);
  } else {
    float a = n.x * n.x + n.y * n.y, k = 1.0f / sqrtf(a);
    p = V3(-n.y * k, n.x * k, 0);
    q = V3(-n.z * p.y, n.z * p.x, a * k);
  }
}

template <class WM>
PRB_D void phase_rows(const DevModel& M, WM& W, int lane) {
  const float dt = M.params[P_DT], erp = M.params[P_ERP_JOINT], erp2 = M.params[P_ERP_CONTACT];
  const int nd = M.nd;
  // ---- joint rows, built serially by lane 0 (<= 40 rows of a few flops each): limits, motors, gear
  if (lane == 0) {
    int nr = 0;
    for (int i = 0; i < nd; i++) {
      if (M.lo[i] > M.hi[i]) continue;
      for (int side = 0; side < 2; side++) {
        float pen = side == 0 ? W.q[i] - M.lo[i] : M.hi[i] - W.q[i];
        if (pen > 0.f) continue;
        float sg = side == 0 ? 1.0f : -1.0f;
        float invD = 1.0f / W.Minv[i][i];
        float rel = sg * W.vs[i];
        float e = pen > -0.04f ? erp : erp2;
        if (nr >= WM::Cfg::MAXJROW) { W.overflow = 1; break; }
        W.jr_dof[nr] = (signed char)i; W.jr_dof2[nr] = -1; W.jr_sign[nr] = sg;
        W.jr_rhs[nr] = (-pen * e / dt - rel) * invD; W.jr_invD[nr] = invD;
        W.jr_lo[nr] = 0.f; W.jr_hi[nr] = M.params[P_LIMIT_MAX_IMPULSE]; W.jr_lam[nr] = 0.f;
        nr++;
      }
    }
    for (int i = 0; i < nd; i++) {
      if (W.mmaximp[i] <= 0.f) continue;
      float invD = 1.0f / W.Minv[i][i];
      float v = W.vs[i];
      float target_v = W.mkp[i] * (W.mtarget[i] - W.q[i]) / dt + v + M.params[P_MOTOR_KD] * (0.f - v);
      if (nr >= WM::Cfg::MAXJROW) { W.overflow = 1; break; }
      W.jr_dof[nr] = (signed char)i; W.jr_dof2[nr] = -1; W.jr_sign[nr] = 1.0f;
      W.jr_rhs[nr] = (target_v - v) * invD; W.jr_invD[nr] = invD;
      W.jr_lo[nr] = -W.mmaximp[i]; W.jr_hi[nr] = W.mmaximp[i]; W.jr_lam[nr] = 0.f;
      nr++;
    }
    for (int s = 0; s < M.n_slide; s++) {
      int o = nd + 6 * M.n_free + s;
      float maximp = M.slide_motor[s][3] < 0 ? M.params[P_DEFAULT_MOTOR_IMPULSE] : M.slide_motor[s][3];
      if (maximp <= 0.f) continue;
      float invD = 1.0f / M.slide_minv[s];
      float v = W.vs[o];
      float target_v = M.slide_motor[s][1] * (M.slide_motor[s][0] - W.sq[s]) / dt + v + M.slide_motor[s][2] * (0.f - v);
      if (nr >= WM::Cfg::MAXJROW) { W.overflow = 1; break; }
      W.jr_dof[nr] = (signed char)o; W.jr_dof2[nr] = -1; W.jr_sign[nr] = 1.0f;
      W.jr_rhs[nr] = (target_v - v) * invD; W.jr_invD[nr] = invD;
      W.jr_lo[nr] = -maximp; W.jr_hi[nr] = maximp; W.jr_lam[nr] = 0.f;
      nr++;
    }
    if (M.gear_a >= 0 && nr < WM::Cfg::MAXJROW) {
      int a = M.gear_a, b = M.gear_b;
      float r = M.params[P_GEAR_RATIO];
      float D = W.Minv[a][a] + 2.f * r * W.Minv[a][b] + r * r * W.Minv[b][b];
      float invD = 1.0f / D;
      float rel = W.vs[a] + r * W.vs[b];
      W.jr_dof[nr] = (signed char)a; W.jr_dof2[nr] = (signed char)b; W.jr_sign[nr] = 1.0f;
      W.jr_rhs[nr] = (-rel * M.params[P_GEAR_ERP]) * invD; W.jr_invD[nr] = invD;
      W.jr_lo[nr] = -M.params[P_GEAR_MAX_IMPULSE]; W.jr_hi[nr] = M.params[P_GEAR_MAX_IMPULSE]; W.jr_lam[nr] = 0.f;
      nr++;
    }
    W.n_jrow = nr;
  }
  // ---- contact rows: lane = contact.  Pool space by exclusive scan of the segment sizes.
  int nc = W.n_contact;
  int bodyA = -1, bodyB = -1, need = 0, ca = 0, cb = 0;
  if (lane < nc) {
    int cols = W.ct[lane].cols;
    ca = cols & 0xff; cb = (cols >> 8) & 0xff;
    bodyA = col_dyn_body(M, ca); bodyB = col_dyn_body(M, cb);
    int nA = bodyA >= 0 ? body_size(M, bodyA) : 0, nB = bodyB >= 0 ? body_size(M, bodyB) : 0;
    need = 4 * 2 * (nA + nB);
  }
  int total;
  int off = warp_excl_scan(need, lane, &total);
  // contacts that do not fit in the pool are dropped (deepest-first ordering is not attempted)
  if (lane == 0 && total > W.dbg_p) W.dbg_p = total;
  bool fits = (lane < nc) && (off + need <= WM::Cfg::POOL);
  unsigned fitmask = __ballot_sync(FULL, fits);
  int nfit = __popc(fitmask & ((nc >= 32) ? FULL : ((1u << nc) - 1u)));
  // since sizes are scanned in order, the fitting contacts are a prefix
  if (lane == 0) { if (nfit < nc) W.overflow = 1; W.n_contact = nfit; }
  nc = nfit;
  if (lane < nc) {
    const Contact c = W.ct[lane];
    v3 n = V3(c.nx, c.ny, c.nz), pb = V3(c.pbx, c.pby, c.pbz), pa = pb + n * c.dist;
    int nA = bodyA >= 0 ? body_size(M, bodyA) : 0, nB = bodyB >= 0 ? body_size(M, bodyB) : 0;
    int offA = off, offB = off + 8 * nA;
    W.cr_bodyA[lane] = (signed char)bodyA; W.cr_bodyB[lane] = (signed char)bodyB;
    W.cr_offA[lane] = (unsigned short)offA; W.cr_offB[lane] = (unsigned short)offB;
    // contact softness (URDF <contact> stiffness/damping on the gripper links)
    float cfm = 0.f, e = erp2;
    float sa = M.col_stiff[ca], sb = M.col_stiff[cb];
    if (sa >= 0.f || sb >= 0.f) {
      float ka = sa >= 0.f ? sa : 1e18f, kb = sb >= 0.f ? sb : 1e18f;
      float da = sa >= 0.f ? M.col_damp[ca] : 0.1f, db = sb >= 0.f ? M.col_damp[cb] : 0.1f;
      float kk = 1.0f / (1.0f / ka + 1.0f / kb), dd = da + db;
      float denom = fmaxf(dt * kk + dd, 1.1920929e-7f);
      cfm = 1.0f / denom; e = dt * kk / denom;
    }
    cfm /= dt;
    float spin = M.col_spin[ca] * M.col_fric[ca] + M.col_spin[cb] * M.col_fric[cb];
    float mu = clampf(M.col_fric[ca] * M.col_fric[cb], -10.f, 10.f);
    v3 t1, t2;
    plane_space(n, t1, t2);
#pragma unroll 1
    for (int k = 0; k < 4; k++) {
      v3 dir = k == 0 ? n : (k == 1 ? n : (k == 2 ? t1 : t2));
      bool ang = (k == 1);
      if (k == 1 && !(spin > 0.f)) {   // no torsional row: keep its segment zeroed (it is still summed with lambda = 0)
        for (int i = 0; i < 2 * nA; i++) W.pool[offA + 2 * nA + i] = 0.f;
        for (int i = 0; i < 2 * nB; i++) W.pool[offB + 2 * nB + i] = 0.f;
        W.cr_invD[lane][1] = 0.f; W.cr_rhs[lane][1] = 0.f; W.cr_lam[lane][1] = 0.f;
        continue;
      }
      float rel = 0.f, D = 0.f;
      if (bodyA >= 0) D += fill_segment(M, W, ca, pa, dir, 1.0f, ang, &W.pool[offA + k * 2 * nA], &rel);
      if (bodyB >= 0) D += fill_segment(M, W, cb, pb, dir, -1.0f, ang, &W.pool[offB + k * 2 * nB], &rel);
      if (k == 0) D += cfm;
      float invD = D > 1.1920929e-7f ? 1.0f / D : 0.f;
      float rhs;
      if (k == 0) {
        float pen = c.dist + M.params[P_LINEAR_SLOP];
        float poserr = 0.f, velerr = -rel;
        if (pen > 0.f) velerr -= pen / dt; else poserr = -pen * e / dt;
        rhs = (poserr + velerr) * invD;
        W.cr_cfm[lane] = cfm * invD;
      } else rhs = -rel * invD;
      W.cr_rhs[lane][k] = rhs; W.cr_invD[lane][k] = invD; W.cr_lam[lane][k] = 0.f;
    }
    W.cr_mu[lane] = mu; W.cr_spin[lane] = spin > 0.f ? spin : 0.f;
  }
  __syncwarp();
}

// ============================================================================ islands + Delassus matrix
// The PGS sweeps run in impulse space: u_r = (J M^-1 J^T lambda)_r is kept per row by the lane that
// owns the row, and a row update only broadcasts its impulse change.  A = J M^-1 J^T is stored in
// shared memory, symmetric-packed and blocked by simulation island (rows of different islands do
// not couple), so memory is sum_i R_i (R_i + 1) / 2 instead of R^2.
//
// Row ownership: joint row j -> lane j & 31, slot j >> 5; contact c -> lane c (rows normal, spin,
// friction 1, friction 2).  Local row ids inside an island: its joint rows first (in row order),
// then its contacts in order, each contributing [normal, (spin), friction 1, friction 2].
struct LaneMap { int body, li, n; float self_minv; };

// Constraint "units" in sweep order: joint rows, contact normals, spinning-friction rows, lateral
// friction PAIRS (two rows solved together by the implicit cone).  Unit g is owned by lane g & 31
// in slot g >> 5, so a lane holds at most RR::MS units and every sweep step has a uniform slot.
template <int MAXSLOT_>
struct RowRegsT {
  static constexpr int MS = MAXSLOT_;
  float ua[MAXSLOT_], ub[MAXSLOT_];        // J M^-1 J^T lambda of the unit's row(s)
  float la[MAXSLOT_], lb[MAXSLOT_];        // accumulated impulses
  float rhsa[MAXSLOT_], rhsb[MAXSLOT_], ida[MAXSLOT_], idb[MAXSLOT_];
  float p0[MAXSLOT_], p1[MAXSLOT_];        // joint: lo, hi | normal: cfm | spin: coefficient | pair: mu
  int meta[MAXSLOT_];                         // island << 16 | island-local row id of row a (-1: empty slot)
  int pa[MAXSLOT_];                           // index in A of this unit's row a (row b follows at + R_island)
  int pbo[MAXSLOT_];                          // R_island for pair units (offset from row a to row b), else 0
  int cidx[MAXSLOT_];                         // contact index of the unit (contact units)
  int nslots;
};

PRB_D int tri(int r) { return (r * (r + 1)) >> 1; }

// B = M^-1 J^T of contact row (c,k) at velocity DoF `dof`
template <class WM>
PRB_DN float contact_B_at(const DevModel& M, const WM& W, int c, int k, int dof) {
  int li, n;
  int body = dof_body(M, dof, &li, &n);
  int base = -1;
  if (body == W.cr_bodyA[c]) base = W.cr_offA[c];
  else if (body == W.cr_bodyB[c]) base = W.cr_offB[c];
  if (base < 0 || body < 0) return 0.f;
  return W.pool[base + k * 2 * n + n + li];
}
// J_(c,k) . B_(c2,k2) over the bodies the two contacts share
template <class WM>
PRB_DN float contact_dot(const DevModel& M, const WM& W, int c, int k, int c2, int k2) {
  float s = 0.f;
  const int bA = W.cr_bodyA[c], bB = W.cr_bodyB[c], b2A = W.cr_bodyA[c2], b2B = W.cr_bodyB[c2];
#pragma unroll 1
  for (int x = 0; x < 2; x++) {
    const int bx = x == 0 ? bA : bB;
    if (bx < 0) continue;
    const int n = body_size(M, bx);
    const float* J = &W.pool[(x == 0 ? W.cr_offA[c] : W.cr_offB[c]) + k * 2 * n];
#pragma unroll 1
    for (int y = 0; y < 2; y++) {
      const int by = y == 0 ? b2A : b2B;
      if (by != bx) continue;
      const float* B = &W.pool[(y == 0 ? W.cr_offA[c2] : W.cr_offB[c2]) + k2 * 2 * n + n];
      for (int i = 0; i < n; i++) s += J[i] * B[i];
    }
  }
  return s;
}
// inverse-mass coupling between two joint-row DoFs
template <class WM>
PRB_D float dof_minv(const DevModel& M, const WM& W, int d, int d2) {
  if (d < M.nd && d2 < M.nd) return W.Minv[d][d2];
  if (d == d2) { int s = d - M.nd - 6 * M.n_free; return (s >= 0 && s < M.n_slide) ? M.slide_minv[s] : 0.f; }
  return 0.f;
}
template <class WM>
PRB_D float jrow_jrow(const DevModel& M, const WM& W, int j, int j2) {
  const float r = M.params[P_GEAR_RATIO];
  int a = W.jr_dof[j], a2 = W.jr_dof2[j], b = W.jr_dof[j2], b2 = W.jr_dof2[j2];
  float v = dof_minv(M, W, a, b);
  if (a2 >= 0) v += r * dof_minv(M, W, a2, b);
  if (b2 >= 0) { v += r * dof_minv(M, W, a, b2); if (a2 >= 0) v += r * r * dof_minv(M, W, a2, b2); }
  return v * W.jr_sign[j] * W.jr_sign[j2];
}
template <class WM>
PRB_D float jrow_contact(const DevModel& M, const WM& W, int j, int c, int k) {
  float v = contact_B_at(M, W, c, k, W.jr_dof[j]);
  if (W.jr_dof2[j] >= 0) v += M.params[P_GEAR_RATIO] * contact_B_at(M, W, c, k, W.jr_dof2[j]);
  return v * W.jr_sign[j];
}

// islands, local row ids, A; fills the per-lane row registers
template <class WM, class RR>
PRB_D void phase_delassus(const DevModel& M, WM& W, int lane, RR& R) {
  const int nb = 1 + M.n_free + M.n_slide;
  int nc = W.n_contact;
  const int njr = W.n_jrow;
  // ---- connected components over the (<= 6) dynamic bodies, from the contact list
  int bA = -1, bB = -1;
  if (lane < nc) { bA = W.cr_bodyA[lane]; bB = W.cr_bodyB[lane]; }
  unsigned reach[8];
  for (int x = 0; x < 8; x++) {
    unsigned mine = 0;
    if (x < nb && bA >= 0 && bB >= 0 && (bA == x || bB == x)) mine = (1u << bA) | (1u << bB);
    reach[x] = warp_or(mine) | (1u << x);
  }
  for (int it = 0; it < 3; it++)
    for (int x = 0; x < 8; x++) {
      unsigned r = reach[x];
      for (int y = 0; y < 8; y++) if ((r >> y) & 1u) r |= reach[y];
      reach[x] = r;
    }
  // island label of a body = lowest body index it reaches
  int my_islC = -1, my_islJ[2] = {-1, -1};
  if (lane < nc) { int bb = bA >= 0 ? bA : bB; my_islC = __ffs((int)reach[bb & 7]) - 1; }
  for (int sl = 0; sl < 2; sl++) {
    int j = sl * 32 + lane;
    if (j < njr) { int li, n; int body = dof_body(M, W.jr_dof[j], &li, &n); my_islJ[sl] = __ffs((int)reach[body & 7]) - 1; }
  }
  bool spin_on = lane < nc && W.cr_spin[lane] > 0.f;
  // ---- local ids per island by one packed scan per island; block bases by running sum.
  //      If the packed blocks do not fit, the last contact is dropped and the layout redone
  //      (flagged in W.overflow; needs > ~89 coupled rows in one island).
  int locJ[2] = {0, 0}, locC = 0, baseJ[2] = {0, 0}, baseC = 0, RJ[2] = {1, 1}, RC = 1;
  int used = 0;
  bool dead = false;      // contact dropped because its island block does not fit
  for (;;) {
    used = 0;
    int Lmax = -1, Rmax = 0;
    const int my_rows = (lane < nc && !dead) ? (spin_on ? 4 : 3) : 0;
#pragma unroll 1
    for (int L = 0; L < nb; L++) {
      int cnt = (my_islJ[0] == L ? 1 : 0) | (my_islJ[1] == L ? 1 << 8 : 0) | ((my_rows && my_islC == L) ? my_rows << 16 : 0);
      int tot;
      int pre = warp_excl_scan(cnt, lane, &tot);
      int nJ0 = tot & 0xff, nJ1 = (tot >> 8) & 0xff, nC = tot >> 16;
      int RL = nJ0 + nJ1 + nC;
      if (RL == 0) continue;                        // uniform
      if (my_islJ[0] == L) { locJ[0] = pre & 0xff; baseJ[0] = used; RJ[0] = RL; }
      if (my_islJ[1] == L) { locJ[1] = nJ0 + ((pre >> 8) & 0xff); baseJ[1] = used; RJ[1] = RL; }
      if (my_islC == L) { locC = nJ0 + nJ1 + (pre >> 16); baseC = used; RC = RL; }
      used += RL * RL;
      if (RL > Rmax) { Rmax = RL; Lmax = L; }
    }
    if (used <= WM::Cfg::ACAP) break;                    // uniform
    // drop the last contact of the largest island (flagged) and lay out again
    unsigned mk = __ballot_sync(FULL, my_rows > 0 && my_islC == Lmax);
    if (mk == 0u) break;
    if (lane == 31 - __clz((int)mk)) dead = true;
    if (lane == 0) W.overflow = 1;
  }
  if (lane >= nc || dead) my_islC = -1;
  spin_on = spin_on && !dead;
  if (dead) { for (int k = 0; k < 4; k++) { W.cr_rhs[lane][k] = 0.f; W.cr_invD[lane][k] = 0.f; } W.cr_spin[lane] = 0.f; }
  __syncwarp();
  if (lane == 0) { if (used > W.dbg_a) W.dbg_a = used; if (nc > W.dbg_c) W.dbg_c = nc; }
  // lanes outside a sender's island read up to 2 R + 1 floats past their own row: keep that finite
  for (int i = used + lane; i < used + WM::Cfg::APAD && i < WM::Cfg::ACAP + WM::Cfg::APAD; i += 32) W.A[i] = 0.f;
  // ---- per-row metadata: block base (16 bits) | island-local row id (8) | island (8); block size R
  for (int sl = 0; sl < 2; sl++) {
    int j = sl * 32 + lane;
    if (j < njr) { W.jr_meta[j] = (unsigned)baseJ[sl] | ((unsigned)locJ[sl] << 16) | ((unsigned)my_islJ[sl] << 24); W.jr_R[j] = (unsigned char)RJ[sl]; }
  }
  if (lane < nc) { W.ct_meta[lane] = (unsigned)baseC | ((unsigned)locC << 16) | ((unsigned)(my_islC & 0xff) << 24); W.ct_R[lane] = (unsigned char)RC; }
  __syncwarp();
  // ---- fill A: full R x R block per island, A[base + r * R + s].  The lane owning receiving row r
  //      computes the entries against every sender row s <= r and mirrors them.
  for (int sl = 0; sl < 2; sl++) {
    int j = sl * 32 + lane;
    if (j >= njr) continue;
    const int r = locJ[sl], Rn = RJ[sl], base = baseJ[sl];
#pragma unroll 1
    for (int j2 = 0; j2 <= j; j2++) {
      unsigned m2 = W.jr_meta[j2];
      if ((int)(m2 >> 24) != my_islJ[sl]) continue;
      const int r2 = (int)((m2 >> 16) & 0xff);
      const float v = jrow_jrow(M, W, j, j2);
      W.A[base + r * Rn + r2] = v; W.A[base + r2 * Rn + r] = v;
    }
  }
  if (lane < nc && !dead) {
    const int c = lane, Rn = RC, base = baseC;
    int k_of[4], nk = 0;
    k_of[nk++] = 0; if (spin_on) k_of[nk++] = 1; k_of[nk++] = 2; k_of[nk++] = 3;
#pragma unroll 1
    for (int kk = 0; kk < nk; kk++) {
      const int k = k_of[kk], r = locC + kk;
#pragma unroll 1
      for (int j2 = 0; j2 < njr; j2++) {
        unsigned m2 = W.jr_meta[j2];
        if ((int)(m2 >> 24) != my_islC) continue;
        const int r2 = (int)((m2 >> 16) & 0xff);
        const float v = jrow_contact(M, W, j2, c, k);
        W.A[base + r * Rn + r2] = v; W.A[base + r2 * Rn + r] = v;
      }
#pragma unroll 1
      for (int c2 = 0; c2 <= c; c2++) {
        unsigned m2 = W.ct_meta[c2];
        if ((int)(m2 >> 24) != my_islC) continue;
        const int loc2 = (int)((m2 >> 16) & 0xff);
        const bool sp2 = W.cr_spin[c2] > 0.f;
        int kk2 = 0;
#pragma unroll 1
        for (int k2 = 0; k2 < 4; k2++) {
          if (k2 == 1 && !sp2) continue;
          const int r2 = loc2 + kk2; kk2++;
          if (r2 > r) break;
          const float v = contact_dot(M, W, c, k, c2, k2);
          W.A[base + r * Rn + r2] = v; W.A[base + r2 * Rn + r] = v;
        }
      }
    }
  }
  // ---- unit registers (sweep order: joint rows | normals | spin rows | friction pairs)
  const unsigned spinmask = __ballot_sync(FULL, spin_on);
  const int nspin = __popc(spinmask);
  const int g_n = njr, g_s = njr + nc, g_f = njr + nc + nspin, g_end = g_f + nc;
  if (lane == 0 && g_end > W.dbg_u) W.dbg_u = g_end;
  R.nslots = (g_end + 31) >> 5;          // <= (40 + 96 + 31) / 32 = 5 in theory; capped below
  if (R.nslots > RR::MS) { R.nslots = RR::MS; if (lane == 0) W.overflow = 1; }
  __syncwarp();
#pragma unroll
  for (int k = 0; k < RR::MS; k++) {
    const int g = 32 * k + lane;
    R.ua[k] = 0.f; R.ub[k] = 0.f; R.la[k] = 0.f; R.lb[k] = 0.f;
    R.rhsa[k] = 0.f; R.rhsb[k] = 0.f; R.ida[k] = 0.f; R.idb[k] = 0.f; R.p0[k] = 0.f; R.p1[k] = 0.f;
    R.meta[k] = 0x7fff0000; R.pa[k] = 0; R.pbo[k] = 0; R.cidx[k] = 0;      // empty slot: island no sender has
    if (g < g_n) {
      const unsigned m = W.jr_meta[g];
      const int base = (int)(m & 0xffff), loc = (int)((m >> 16) & 0xff), isl = (int)(m >> 24);
      R.rhsa[k] = W.jr_rhs[g]; R.ida[k] = W.jr_invD[g]; R.p0[k] = W.jr_lo[g]; R.p1[k] = W.jr_hi[g];
      R.meta[k] = (isl << 16) | loc; R.pa[k] = base + loc * (int)W.jr_R[g];
    } else if (g < g_end) {
      int c, row;
      if (g < g_s) { c = g - g_n; row = 0; }
      else if (g < g_f) {           // (g - g_s)-th contact with a spin row
        unsigned mm = spinmask; for (int i = 0; i < g - g_s; i++) mm &= mm - 1;
        c = __ffs((int)mm) - 1; row = 1;
      } else { c = g - g_f; row = 2; }
      const unsigned m = W.ct_meta[c];
      const int base = (int)(m & 0xffff), loc = (int)((m >> 16) & 0xff), isl = (int)(m >> 24), Rn = (int)W.ct_R[c];
      const bool sp = (spinmask >> c) & 1u;
      const int r = loc + (row == 0 ? 0 : (row == 1 ? 1 : (sp ? 2 : 1)));
      R.cidx[k] = c;
      if (isl != 255) {          // 255: contact dropped on overflow -> inert unit (rhs = invD = 0, couples with nothing)
        R.meta[k] = (isl << 16) | r; R.pa[k] = base + r * Rn;
        R.rhsa[k] = W.cr_rhs[c][row]; R.ida[k] = W.cr_invD[c][row];
        if (row == 0) R.p0[k] = W.cr_cfm[c];
        else if (row == 1) R.p0[k] = W.cr_spin[c];
        else { R.p0[k] = W.cr_mu[c]; R.rhsb[k] = W.cr_rhs[c][3]; R.idb[k] = W.cr_invD[c][3]; R.pbo[k] = Rn; }
      }
    }
    W.unit_meta[1 + g] = R.meta[k];
  }
  if (lane == 0) { W.unit_meta[0] = 0x7fff0000; W.unit_meta[1 + 32 * RR::MS] = 0x7fff0000; }
  __syncwarp();
}

// ============================================================================ PGS (lane = unit owner)
// Each unit keeps the index of its own row(s) of the island block, so the coupling to sender row s
// is A[pa + s] (A is symmetric).  Lanes whose unit is in another island read a finite in-range
// value and multiply it by zero.  The sender's row id comes from a per-unit table (it is known
// before the sweep starts), so the A loads of the NEXT step are issued before the current step's
// impulse change is broadcast: the dependent chain per step is candidate -> shuffle -> FMA.
enum { U_JOINT = 0, U_NORMAL = 1, U_SPIN = 2, U_PAIR = 3 };

template <int NS, bool PAIR>
struct ACoef { float a[NS], b[NS], a2[PAIR ? NS : 1], b2[PAIR ? NS : 1]; };

template <int NS, bool PAIR, class WM, class RR>
PRB_D void pgs_load(const WM& W, const RR& R, int smeta, ACoef<NS, PAIR>& C) {
  const int sloc = smeta & 0xffff;
#pragma unroll
  for (int k = 0; k < NS; k++) {
    const float* row = &W.A[R.pa[k] + sloc];
    C.a[k] = row[0];
    C.b[k] = row[R.pbo[k]];                  // pair units: second row; single units: pbo = 0, ub unused
    if (PAIR) { C.a2[k] = row[1]; C.b2[k] = row[R.pbo[k] + 1]; }
  }
}
template <int NS, bool PAIR, class RR>
PRB_D void pgs_apply(RR& R, int smeta, const ACoef<NS, PAIR>& C, float d1, float d2) {
  const int sisl = smeta >> 16;
#pragma unroll
  for (int k = 0; k < NS; k++) {
    const bool on = (R.meta[k] >> 16) == sisl;
    const float m1 = on ? d1 : 0.f;
    R.ua[k] = fmaf(C.a[k], m1, R.ua[k]);
    R.ub[k] = fmaf(C.b[k], m1, R.ub[k]);
    if (PAIR) {
      const float m2 = on ? d2 : 0.f;
      R.ua[k] = fmaf(C.a2[k], m2, R.ua[k]);
      R.ub[k] = fmaf(C.b2[k], m2, R.ub[k]);
    }
  }
}

// solve the unit in slot K of lane src; returns the impulse change(s) as seen by the owner
template <int K, int TYPE, class WM, class RR>
PRB_D void pgs_candidate(WM& W, RR& R, int lane, int src, float& d1, float& d2) {
  d2 = 0.f;
  if (TYPE == U_JOINT) {
    const float delta = R.rhsa[K] - R.ua[K] * R.ida[K];
    const float nl = clampf(R.la[K] + delta, R.p0[K], R.p1[K]);
    d1 = nl - R.la[K];
    if (lane == src) R.la[K] = nl;
  } else if (TYPE == U_NORMAL) {
    const float delta = R.rhsa[K] - R.la[K] * R.p0[K] - R.ua[K] * R.ida[K];
    const float nl = fmaxf(R.la[K] + delta, 0.f);
    d1 = nl - R.la[K];
    if (lane == src) { R.la[K] = nl; W.cr_lam[R.cidx[K]][0] = nl; }     // read by the friction units of this contact
  } else if (TYPE == U_SPIN) {
    const float tot = W.cr_lam[R.cidx[K]][0];
    const float lim = R.p0[K] * tot;
    const float delta = R.rhsa[K] - R.ua[K] * R.ida[K];
    const float nl = clampf(R.la[K] + delta, -lim, lim);
    d1 = tot > 0.f ? nl - R.la[K] : 0.f;                              // Bullet skips the row while the normal impulse is 0
    if (lane == src && tot > 0.f) R.la[K] = nl;
  } else {
    const float lim = R.p0[K] * W.cr_lam[R.cidx[K]][0];
    const float sumA = R.la[K] + (R.rhsa[K] - R.ua[K] * R.ida[K]);
    const float sumB = R.lb[K] + (R.rhsb[K] - R.ub[K] * R.idb[K]);
    float na = sumA, nb = sumB;
    if (sumA < -lim || sumA > lim || sumB < -lim || sumB > lim) {
      // |lim sin(atan2(A,B))| and |lim cos(atan2(A,B))| as |lim A| / r and |lim B| / r
      const float ss = sumA * sumA + sumB * sumB;
      const float inv = ss > 0.f ? rsqrtf(ss) : 0.f;
      const float ca_ = fabsf(lim * sumA) * inv, cb_ = ss > 0.f ? fabsf(lim * sumB) * inv : fabsf(lim);
      na = clampf(sumA, -ca_, ca_); nb = clampf(sumB, -cb_, cb_);
    }
    d1 = na - R.la[K]; d2 = nb - R.lb[K];
    if (lane == src) { R.la[K] = na; R.lb[K] = nb; }
  }
}

// units g in [ga, gb), all living in slot K, swept upwards (dir = +1) or downwards (dir = -1)
template <int NS, int K, int TYPE, class WM, class RR>
PRB_D void pgs_range(WM& W, RR& R, int lane, int ga, int gb, int dir) {
  constexpr bool PAIR = (TYPE == U_PAIR);
  const int n = gb - ga;
  if (n <= 0) return;
  int g = dir > 0 ? ga : gb - 1;
  int smeta = W.unit_meta[1 + g];
  ACoef<NS, PAIR> C;
  pgs_load<NS, PAIR>(W, R, smeta, C);
#pragma unroll 1
  for (int i = 0; i < n; i++) {
    const int smeta_n = W.unit_meta[1 + g + dir];          // table is padded on both ends
    ACoef<NS, PAIR> Cn;
    pgs_load<NS, PAIR>(W, R, smeta_n, Cn);                 // next step's coefficients, independent of this step
    float d1, d2;
    const int src = g & 31;
    pgs_candidate<K, TYPE>(W, R, lane, src, d1, d2);
    d1 = __shfl_sync(FULL, d1, src);
    if (PAIR) d2 = __shfl_sync(FULL, d2, src);
    pgs_apply<NS, PAIR>(R, smeta, C, d1, d2);
    C = Cn; smeta = smeta_n; g += dir;
  }
}
// a phase's units [g0, g1) split by the slot they live in
template <int NS, int TYPE, class WM, class RR>
PRB_D void pgs_phase(WM& W, RR& R, int lane, int g0, int g1, int dir) {
  if (dir > 0) {
    pgs_range<NS, 0, TYPE>(W, R, lane, max(g0, 0), min(g1, 32), 1);
    if (NS > 1) pgs_range<NS, (NS > 1 ? 1 : 0), TYPE>(W, R, lane, max(g0, 32), min(g1, 64), 1);
    if (NS > 2) pgs_range<NS, (NS > 2 ? 2 : 0), TYPE>(W, R, lane, max(g0, 64), min(g1, 96), 1);
    if (NS > 3) pgs_range<NS, (NS > 3 ? 3 : 0), TYPE>(W, R, lane, max(g0, 96), min(g1, 128), 1);
  } else {
    if (NS > 3) pgs_range<NS, (NS > 3 ? 3 : 0), TYPE>(W, R, lane, max(g0, 96), min(g1, 128), -1);
    if (NS > 2) pgs_range<NS, (NS > 2 ? 2 : 0), TYPE>(W, R, lane, max(g0, 64), min(g1, 96), -1);
    if (NS > 1) pgs_range<NS, (NS > 1 ? 1 : 0), TYPE>(W, R, lane, max(g0, 32), min(g1, 64), -1);
    pgs_range<NS, 0, TYPE>(W, R, lane, max(g0, 0), min(g1, 32), -1);
  }
}
template <int NS, class WM, class RR>
PRB_D void pgs_sweeps(const DevModel& M, WM& W, RR& R, int lane, int g_n, int g_s, int g_f, int g_end) {
#pragma unroll 1
  for (int it = 0; it < M.solver_iters; it++) {
    pgs_phase<NS, U_JOINT>(W, R, lane, 0, g_n, (it & 1) ? 1 : -1);
    pgs_phase<NS, U_NORMAL>(W, R, lane, g_n, min(g_s, g_end), 1);
    __syncwarp();                                      // normal impulses visible to the friction units
    pgs_phase<NS, U_SPIN>(W, R, lane, g_s, min(g_f, g_end), 1);
    pgs_phase<NS, U_PAIR>(W, R, lane, g_f, g_end, 1);
    __syncwarp();
  }
}

// 50 projected-Gauss-Seidel sweeps in btMultiBodyConstraintSolver::solveSingleIteration order:
// non-contact rows (direction alternating per iteration), normals, spinning friction, lateral
// friction as an implicit cone over the row pair.  Returns dv = M^-1 J^T lambda for this lane's DoF.
template <class WM, class RR>
PRB_D float phase_pgs(const DevModel& M, WM& W, int lane, const LaneMap& lm, RR& R) {
  const int njr = W.n_jrow, nc = W.n_contact, nd = M.nd;
  const unsigned spinmask = __ballot_sync(FULL, lane < nc && W.cr_spin[lane < nc ? lane : 0] > 0.f);
  const int nspin = __popc(spinmask);
  const int g_n = njr, g_s = njr + nc, g_f = g_s + nspin;
  const int g_end = min(g_f + nc, 32 * RR::MS);
  if (RR::MS <= 2 || R.nslots <= 2) pgs_sweeps<2>(M, W, R, lane, g_n, g_s, g_f, g_end);
  else pgs_sweeps<RR::MS>(M, W, R, lane, g_n, g_s, g_f, g_end);
  // ---- publish the impulses and rebuild dv = M^-1 J^T lambda with lane = velocity DoF
  __syncwarp();
  if (lane < nc) { W.cr_lam[lane][1] = 0.f; W.cr_lam[lane][2] = 0.f; W.cr_lam[lane][3] = 0.f; }
  __syncwarp();
#pragma unroll
  for (int k = 0; k < RR::MS; k++) {
    const int g = 32 * k + lane;
    if (g < g_n) W.jr_lam[g] = R.la[k];
    else if (g < g_s) W.cr_lam[R.cidx[k]][0] = R.la[k];
    else if (g < g_f) W.cr_lam[R.cidx[k]][1] = R.la[k];
    else if (g < g_end) { W.cr_lam[R.cidx[k]][2] = R.la[k]; W.cr_lam[R.cidx[k]][3] = R.lb[k]; }
  }
  __syncwarp();
  float dv = 0.f;
  const float ratio = M.params[P_GEAR_RATIO];
#pragma unroll 1
  for (int j = 0; j < njr; j++) {
    const int d = W.jr_dof[j], d2 = W.jr_dof2[j];
    float b = 0.f;
    if (d < nd) { if (lane < nd) b = W.Minv[lane][d]; }
    else if (lane == d) b = lm.self_minv;
    if (d2 >= 0 && lane < nd) b += ratio * W.Minv[lane][d2];
    dv += b * W.jr_sign[j] * W.jr_lam[j];
  }
  if (lm.body >= 0) {
#pragma unroll 1
    for (int c = 0; c < nc; c++) {
      int base = -1;
      if (lm.body == W.cr_bodyA[c]) base = W.cr_offA[c];
      else if (lm.body == W.cr_bodyB[c]) base = W.cr_offB[c];
      if (base < 0) continue;
      const float* seg = &W.pool[base + lm.n + lm.li];
      dv += seg[0] * W.cr_lam[c][0] + seg[2 * lm.n] * W.cr_lam[c][1] + seg[4 * lm.n] * W.cr_lam[c][2] + seg[6 * lm.n] * W.cr_lam[c][3];
    }
  }
  return dv;
}

// ============================================================================ integrate (lane = DoF)
template <class WM>
PRB_D void phase_integrate(const DevModel& M, WM& W, int lane, float vstar, float dv) {
  const float dt = M.params[P_DT], vmax = M.params[P_MAX_COORD_VEL];
  const int nd = M.nd;
  float v = clampf(vstar + dv, -vmax, vmax);
  if (lane < M.nv) W.vs[lane] = v;
  __syncwarp();
  if (lane < nd) { W.qd[lane] = v; W.q[lane] += dt * v; }
  int b = lane - nd;
  if (b >= 0 && b < M.n_free) {
    int o = nd + 6 * b;
    v3 vl = ld3(&W.vs[o]), w = ld3(&W.vs[o + 3]);
    st3(W.fvel[b], vl); st3(W.fang[b], w);
    st3(W.fpos[b], ld3(W.fpos[b]) + vl * dt);
    float ang = norm(w);
    if (ang * dt > 0.78539816f) ang = 0.5f * 1.57079633f / dt;
    v3 ax;
    if (ang < 0.001f) ax = w * (0.5f * dt - dt * dt * dt * 0.020833333333f * ang * ang);
    else ax = w * (sinf(0.5f * ang * dt) / ang);
    float dq[4] = {ax.x, ax.y, ax.z, cosf(ang * dt * 0.5f)}, nq[4];
    quat_mul(dq, W.fquat[b], nq);
    float inv = 1.0f / sqrtf(nq[0] * nq[0] + nq[1] * nq[1] + nq[2] * nq[2] + nq[3] * nq[3]);
    for (int k = 0; k < 4; k++) W.fquat[b][k] = nq[k] * inv;
  }
  int s = lane - nd - 6 * M.n_free;
  if (s >= 0 && s < M.n_slide) { W.sqd[s] = v; W.sq[s] += dt * v; }
  __syncwarp();
}

// one stepSimulation()
template <int ND, class WM>
PRB_D void substep(const DevModel& M, WM& W, int lane, const LaneMap& lm) {
  phase_fk(M, W, lane, true);
  phase_collide(M, W, lane);
  phase_crba(M, W, lane);
  phase_minv<ND>(W, lane);
  float vstar = phase_vstar(M, W, lane);
  phase_rows(M, W, lane);
  RowRegsT<WM::Cfg::MAXSLOT> R;
  phase_delassus(M, W, lane, R);
  float dv = phase_pgs(M, W, lane, lm, R);
  phase_integrate(M, W, lane, vstar, dv);
}

PRB_D LaneMap make_lanemap(const DevModel& M, int lane) {
  LaneMap lm;
  lm.body = dof_body(M, lane, &lm.li, &lm.n);
  lm.self_minv = 0.f;
  int s = lane - M.nd - 6 * M.n_free;
  if (s >= 0 && s < M.n_slide) lm.self_minv = M.slide_minv[s];
  return lm;
}

// ============================================================================ observation / reward
PRB_D float py_mod2(float a) { float r = fmodf(a, 2.0f); if (r != 0.f && r < 0.f) r += 2.0f; return r; }
PRB_D float reward_of(const DevModel& M, const float* ag, const float* dg) {
  if (M.play) {  // playRewardFunc.py:66-77
    for (int k = 0; k < 3; k++) if (fabsf(dg[k] - ag[k]) > 0.05f) return -1.f;
    float eg[3], ea[3];
    euler_from_quat(dg + 3, eg); euler_from_quat(ag + 3, ea);
    for (int k = 0; k < 3; k++) if (fabsf(eg[k] - ea[k]) > PRB_PI_F / 4) return -1.f;
    if (fabsf(dg[7] - ag[7]) > 0.025f) return -1.f;
    if (fabsf(dg[8] - ag[8]) > 0.04f) return -1.f;
    if (fabsf(dg[9] - ag[9]) > 0.01f) return -1.f;
    if (fabsf(dg[10] - ag[10]) > 0.3f) return -1.f;
    return 0.f;
  }
  float dx = ag[0] - dg[0], dy = ag[1] - dg[1], dz = ag[2] - dg[2];
  float d = sqrtf(dx * dx + dy * dy + dz * dz);
  return d > M.params[P_SPARSE_THRESH] ? -1.0f : -d;
}
template <class WM>
PRB_D void site_pose(const DevModel& M, const WM& W, int site, v3& pos, m3& R) {
  int l = M.site_link[site];
  m3 lR = ldm(W.lR[l]);
  pos = ld3(W.lp[l]) + mul(lR, ld3(M.site_pos[site]));
  R = mul(lR, ldm(M.site_rot[site]));
}

// calc_state (environments.py:799-864) fused with compute_reward; every lane assembles the small
// vectors redundantly (a few hundred flops), the ray test is spread over lanes; returns reward.
template <class WM>
PRB_D float phase_observe(const DevModel& M, WM& W, int lane, const DevOut& O, size_t e, bool write) {
  phase_fk(M, W, lane, false);
  v3 ep; m3 eR;
  site_pose(M, W, 0, ep, eR);
  float eq[4];
  mat_to_quat(eR, eq);
  const int el = M.site_link[0];
  v3 w = ld3(W.lw[el]), vl = ld3(W.lv[el]) + cross(w, ep - ld3(W.lp[el]));
  float grip = M.arm_kind == 0 ? W.q[M.grip_obs_dof] * 23.0f : W.q[M.grip_obs_dof];
  // gripper_proprioception: ray from above the palm to between the pads, nearest box hit
  float prop = -1.f;
  if (M.arm_kind == 0) {
    v3 g1, g2, wr; m3 t;
    site_pose(M, W, 2, g1, t); site_pose(M, W, 3, g2, t); site_pose(M, W, 1, wr, t);
    v3 avg = (g1 + g2) * 0.5f, ew = ep - wr;
    v3 from = ep - ew * 0.5f, to = avg + ew * 0.2f, d = to - from;
    float best = 1.0f; int hit = -1;
    for (int c = lane; c < M.n_col; c += 32) {
      m3 R; v3 p;
      collider_frame(M, W, c, R, p);
      v3 o = tmul(R, from - p), dl = tmul(R, d), h = ld3(M.col_half[c]);
      float t0 = 0.f, t1 = 1.f; bool ok = true;
      for (int k = 0; k < 3; k++) {
        float ok_ = comp(o, k), dk = comp(dl, k), hk = comp(h, k);
        if (fabsf(dk) < 1e-12f) { if (ok_ < -hk || ok_ > hk) ok = false; }
        else {
          float ta = (-hk - ok_) / dk, tb = (hk - ok_) / dk;
          if (ta > tb) { float tt = ta; ta = tb; tb = tt; }
          t0 = fmaxf(t0, ta); t1 = fminf(t1, tb);
          if (t0 > t1) ok = false;
        }
      }
      if (ok && t0 < best) { best = t0; hit = c; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      float ob = __shfl_xor_sync(FULL, best, o); int oh = __shfl_xor_sync(FULL, hit, o);
      if (ob < best || (ob == best && oh >= 0 && (hit < 0 || oh < hit))) { best = ob; hit = oh; }
    }
    int li = hit >= 0 ? M.col_urdf[hit] : -1;
    prop = (hit < 0 || best == 1.0f || li == 18 || li == 20) ? 0.f : 1.f;
  }
  float st[24], ag[12];
  int n = 0, na = 0;
  st[n++] = ep.x; st[n++] = ep.y; st[n++] = ep.z;
  if (M.return_velocity) { st[n++] = vl.x; st[n++] = vl.y; st[n++] = vl.z; }
  if (M.use_orientation) for (int k = 0; k < 4; k++) st[n++] = eq[k];
  st[n++] = grip;
  if (M.n_free > 0) {
    for (int k = 0; k < 3; k++) st[n++] = W.fpos[0][k];
    if (M.use_orientation) for (int k = 0; k < 4; k++) st[n++] = W.fquat[0][k];
    if (M.return_velocity) for (int k = 0; k < 3; k++) st[n++] = W.fvel[0][k];
    for (int k = 0; k < 3; k++) ag[na++] = W.fpos[0][k];
    if (M.use_orientation) for (int k = 0; k < 4; k++) ag[na++] = W.fquat[0][k];
    if (M.play) {
      float ex[4] = {W.fpos[1][1], W.sq[0], W.sq[1], (py_mod2(W.sq[2]) * PRB_PI_F) / (2.2f * PRB_PI_F)};
      for (int k = 0; k < 4; k++) { st[n++] = ex[k]; ag[na++] = ex[k]; }
    }
  } else { ag[0] = ep.x; ag[1] = ep.y; ag[2] = ep.z; na = 3; }
  if (M.play) {  // quaternion_safe_the_obs
    if (W.last_valid > 0.5f) {
      bool fe = true, fo = true;
      for (int k = 0; k < 4; k++) {
        float a = st[3 + k], l = W.lastq[k];
        int sa = (a > 0.f) - (a < 0.f), sl = (l > 0.f) - (l < 0.f);
        if (sa != -sl) fe = false;
        a = st[11 + k]; l = W.lastq[4 + k]; sa = (a > 0.f) - (a < 0.f); sl = (l > 0.f) - (l < 0.f);
        if (sa != -sl) fo = false;
      }
      if (fe) for (int k = 0; k < 4; k++) st[3 + k] = -st[3 + k];
      if (fo) for (int k = 0; k < 4; k++) { st[11 + k] = -st[11 + k]; ag[3 + k] = -ag[3 + k]; }
    }
    __syncwarp();
    if (lane < 4) W.lastq[lane] = st[3 + lane];
    else if (lane < 8) W.lastq[lane] = st[11 + lane - 4];
    if (lane == 8) W.last_valid = 1.0f;
    __syncwarp();
  }
  float dg[12];
  for (int k = 0; k < M.goal_dim; k++) dg[k] = W.goal[k];
  float r = reward_of(M, ag, dg);
  if (write) {
    for (int k = lane; k < M.obs_dim; k += 32) O.obs_quat[e * M.obs_dim + k] = st[k];
    if (lane < M.goal_dim) { O.achieved_goal[e * M.goal_dim + lane] = ag[lane]; O.desired_goal[e * M.goal_dim + lane] = dg[lane]; }
    if (lane < 4) O.cag[e * 4 + lane] = lane < 3 ? comp(ep, lane) : grip;
    {  // full_positional_state
      float f[24]; int k = 0;
      f[k++] = ep.x; f[k++] = ep.y; f[k++] = ep.z;
      if (M.use_orientation) for (int j = 0; j < 4; j++) f[k++] = st[3 + j];
      f[k++] = grip;
      if (M.n_free > 0) for (int j = 0; j < na; j++) f[k++] = ag[j];
      if (lane < M.fps_dim) O.fps[e * M.fps_dim + lane] = f[lane];
    }
    if (lane < 8) O.joints[e * 8 + lane] = M.joints_obs_dof[lane] >= 0 ? W.q[M.joints_obs_dof[lane]] : 0.f;
    if (lane < 6) O.velocity[e * 6 + lane] = lane < 3 ? comp(vl, lane) : comp(w, lane - 3);
    {  // 'observation' = state[0:3] + euler(state[3:7]) + state[7:]  (environments.py:859)
      float eu[3], o[24]; int k = 0;
      euler_from_quat(st + 3, eu);
      o[k++] = st[0]; o[k++] = st[1]; o[k++] = st[2]; o[k++] = eu[0]; o[k++] = eu[1]; o[k++] = eu[2];
      for (int j = 7; j < n; j++) o[k++] = st[j];
      if (lane < M.observation_dim) O.observation[e * M.observation_dim + lane] = o[lane];
    }
    if (lane == 0) { O.proprio[e] = prop; O.reward[e] = r; O.success[e] = r < 0.f ? 0.f : 1.f; }
  }
  return r;
}

#ifdef PRB_EMU
static char g_emu_smem[8 * sizeof(WarpMemT<CfgL>) + 256];
#define PRB_SMEM_DECL WM* wm = (WM*)g_emu_smem
#else
#define PRB_SMEM_DECL extern __shared__ __align__(16) unsigned char prb_dyn_smem[]; WM* wm = (WM*)prb_dyn_smem
#endif

// ============================================================================ step kernel (warp per env)
// Small tier (CfgS): warp w of the grid steps env w.  An env that outgrows the small capacities is
// appended to `redo_list` and left untouched.  Large tier (CfgL): warp w steps env redo_list[w].
// The warps of a block are re-aligned with a block barrier at every substep: the substep's set-up
// code is far larger than the instruction cache, so warps drifting apart would each stream it
// from L2 separately (measured: 3 stall cycles per issue on instruction fetch without this).
template <int ND, class CFG>
__global__ void __launch_bounds__(32 * CFG::WPB, CFG::MINBLOCKS) prb_step_kernel(const DevModel* __restrict__ Mp, float* __restrict__ state,
                                                                              DevOut O, const int* __restrict__ in_list, const int* __restrict__ in_count,
                                                                              int* __restrict__ redo_list, int* __restrict__ redo_count,
                                                                              int N, int n_substeps, int observe) {
  typedef WarpMemT<CFG> WM;
  PRB_SMEM_DECL;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int slot = blockIdx.x * CFG::WPB + wib;
  int e = slot;
  bool active = slot < N;
  if (in_list != nullptr) {                        // this tier only runs what the previous one handed over
    const int cnt = *in_count;
    if (blockIdx.x * CFG::WPB >= cnt) return;      // whole block idle
    active = slot < cnt;
    e = active ? in_list[slot] : 0;
  }
  const DevModel& M = *Mp;
  WM& W = wm[wib];
  float* st = state + (size_t)e * M.state_stride;
  if (active) {
    load_state(M, W, st, lane);
    if (lane == 0) { W.overflow = 0; W.dbg_a = 0; W.dbg_c = 0; W.dbg_p = 0; W.dbg_u = 0; }
    __syncwarp();
  }
  const LaneMap lm = make_lanemap(M, lane);
#pragma unroll 1
  for (int s = 0; s < n_substeps; s++) {
    __syncthreads();
    if (active) {
      substep<ND>(M, W, lane, lm);
      if (CFG::ABORT && W.overflow) {            // uniform per warp: shared flag read after the substep's final __syncwarp
        if (lane == 0) redo_list[atomicAdd(redo_count, 1)] = e;
        active = false;
      }
    }
  }
  if (!active) return;
  __syncwarp();
  if (lane == 0 && O.dbg) { O.dbg[4 * e] = W.dbg_a; O.dbg[4 * e + 1] = W.dbg_c; O.dbg[4 * e + 2] = W.dbg_p; O.dbg[4 * e + 3] = W.dbg_u; }
  if (observe) phase_observe(M, W, lane, O, (size_t)e, true);
  __syncwarp();
  if (lane == 0 && W.overflow && O.overflow) atomicAdd(O.overflow, 1ull);
  store_state(M, W, st, lane);
}

// ============================================================================ stateless reward (relabelling)
__global__ void prb_reward_kernel(const DevModel* __restrict__ Mp, const float* __restrict__ ag, const float* __restrict__ dg,
                                  long long B, float* __restrict__ out) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const DevModel& M = *Mp;
  float a[12], d[12];
  for (int k = 0; k < M.goal_dim; k++) { a[k] = ag[i * M.goal_dim + k]; d[k] = dg[i * M.goal_dim + k]; }
  out[i] = reward_of(M, a, d);
}

// initial state: arm at q = 0 with the default velocity motors, bodies at their load poses
__global__ void prb_init_kernel(const DevModel* __restrict__ Mp, float* __restrict__ state, int N) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  const DevModel& M = *Mp;
  float* st = state + (size_t)e * M.state_stride;
  const int nd = M.nd;
  for (int i = 0; i < M.state_stride; i++) st[i] = 0.f;
  for (int i = 0; i < nd; i++) st[4 * nd + i] = M.params[P_DEFAULT_MOTOR_IMPULSE];
  for (int b = 0; b < M.n_free; b++) {
    for (int k = 0; k < 3; k++) st[5 * nd + 13 * b + k] = M.free_pos0[b][k];
    for (int k = 0; k < 4; k++) st[5 * nd + 13 * b + 3 + k] = M.free_quat0[b][k];
  }
}
