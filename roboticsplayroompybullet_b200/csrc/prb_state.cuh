// prb_state.cuh — read, write, save and restore the link and joint states of every env (sm_100a, fp32, CUDA cores);
// prb_body_states, prb_write_state, prb_restore_state.
//
// prb_body_state_kernel: ONE WARP PER ENV, STATE_ENVS envs per block, a StateMem in shared memory.
//   * joints   lane j < nd + n_slide copies q_j and qd_j (arm DoF, then the slide joints) from the state row into
//              one run of nd + n_slide floats per output;
//   * load     lane j < nd reads q_j, qd_j; lane b < n_free the free-body quaternion, lane s < n_slide the slide
//              coordinate (the rows phase_fk reads);
//   * fk       the step's phase_fk without dynamics (lane = link) gives lR, lp, lw, lv and lc;
//   * rows     lane r < K = nd + n_free + n_slide builds row r (pos | quat xyzw | linear velocity | angular velocity)
//              in shared memory: arm link r in its link frame (lp, lv) or COM frame (lc, lv + lw x (lc - lp)), free
//              body r - nd as its 13 state floats, slide body r - nd - n_free from sR / sp and sqd along or about its
//              world axis;
//   * stores   the env's [K,13] block is one contiguous run, written one element per lane and pass.
// The kernel reads the state and writes only the outputs it is given.
//
// prb_write_state_kernel: ONE WARP PER ENV.  Lane j < nd + n_slide reads the selected joint position and velocity of
// column j, lane 13 b + k < 13 n_free the selected word k of free body b (a quaternion word divided by the quaternion's
// norm); a ballot accepts the env only if every selected value is finite and every selected quaternion has a norm
// >= 1e-6.  Accepted envs get exactly the selected state words; `written` flags them for the contact-report clear and
// the masked observe that follow in prb_capi.cu.
//
// prb_restore_state_kernel: thread per state word, the masked row copy of a snapshot.
#pragma once
#include <stdint.h>

#include <string>

#include "../../include/prb.h"
#include "prb_render.cuh"       // RenderFkMem: the fields phase_fk reads and writes

#define STATE_ENVS 4            // envs (warps) per block
#define STATE_MAXK (PRB_MAXD + PRB_MAXFREE + PRB_MAXSLIDE)

struct StateMem {
  RenderFkMem F;
  float row[STATE_MAXK][13];
};

// prb_state_write's bit masks, checked
struct StateWrite {
  unsigned jq, jqd, fpose, fvel;
};

// body [N,K,13], jq and jqd [N,nd+n_slide]; each optional
__global__ void __launch_bounds__(32 * STATE_ENVS) prb_body_state_kernel(const DevModel* __restrict__ Mp, const float* __restrict__ state,
                                                                          int N, int frame, float* __restrict__ body,
                                                                          float* __restrict__ jq, float* __restrict__ jqd) {
  __shared__ StateMem SM[STATE_ENVS];
  const DevModel& M = *Mp;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t e = (int64_t)blockIdx.x * STATE_ENVS + warp;
  if (e >= N) return;                    // whole warps of the last block
  const int nd = M.nd, nf = M.n_free, ns = M.n_slide, nj = nd + ns, K = nd + nf + ns;
  const int so = 5 * nd + 13 * nf;       // slide (q, qd) pairs in the state row
  const float* st = state + e * M.state_stride;
  if (lane < nj) {
    const int iq = lane < nd ? lane : so + 2 * (lane - nd);
    const int iqd = lane < nd ? nd + lane : iq + 1;
    if (jq) jq[e * nj + lane] = st[iq];
    if (jqd) jqd[e * nj + lane] = st[iqd];
  }
  if (!body) return;
  StateMem& W = SM[warp];
  RenderFkMem& F = W.F;
  if (lane < nd) { F.q[lane] = st[lane]; F.qd[lane] = st[nd + lane]; }
  if (lane < nf) for (int k = 0; k < 4; k++) F.fquat[lane][k] = st[5 * nd + 13 * lane + 3 + k];
  if (lane < ns) F.sq[lane] = st[so + 2 * lane];
  __syncwarp();
  phase_fk(M, F, lane, false);
  if (lane < nd) {
    float* r = W.row[lane];
    const v3 p = ld3(F.lp[lane]), w = ld3(F.lw[lane]), v = ld3(F.lv[lane]);
    const v3 o = frame ? ld3(F.lc[lane]) : p;
    st3(r, o);
    mat_to_quat(ldm(F.lR[lane]), r + 3);
    st3(r + 7, frame ? v + cross(w, o - p) : v);
    st3(r + 10, w);
  } else if (lane < nd + nf) {
    float* r = W.row[lane];
    const float* src = st + 5 * nd + 13 * (lane - nd);
    for (int k = 0; k < 13; k++) r[k] = src[k];
  } else if (lane < K) {
    float* r = W.row[lane];
    const int s = lane - nd - nf;
    const v3 d = ld3(M.slide_axis_w[s]) * st[so + 2 * s + 1], z = V3(0.f, 0.f, 0.f);
    const bool rev = M.slide_jtype[s] == 0;
    st3(r, ld3(F.sp[s]));
    mat_to_quat(ldm(F.sR[s]), r + 3);
    st3(r + 7, rev ? z : d);
    st3(r + 10, rev ? d : z);
  }
  __syncwarp();
  float* out = body + e * (13 * K);
  const float* rows = &W.row[0][0];
  for (int i = lane; i < 13 * K; i += 32) out[i] = rows[i];
}

// jq, jqd [N,nd+n_slide] and body [N,K,13] in the read layouts (only the selected words are read); mask [N] (NULL: all);
// status [N] optional (0 not masked, 1 written, 2 rejected); written [N] always (1: written, else 0)
__global__ void __launch_bounds__(32 * STATE_ENVS) prb_write_state_kernel(const DevModel* __restrict__ Mp, float* __restrict__ state, int N,
                                                                           StateWrite P, const float* __restrict__ jq,
                                                                           const float* __restrict__ jqd, const float* __restrict__ body,
                                                                           const uint8_t* __restrict__ mask, uint8_t* __restrict__ status,
                                                                           uint8_t* __restrict__ written) {
  const DevModel& M = *Mp;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t e = (int64_t)blockIdx.x * STATE_ENVS + warp;
  if (e >= N) return;
  if (mask && mask[e] == 0) {
    if (lane == 0) { written[e] = 0; if (status) status[e] = 0; }
    return;
  }
  const int nd = M.nd, nf = M.n_free, ns = M.n_slide, nj = nd + ns, K = nd + nf + ns;
  const int so = 5 * nd + 13 * nf;
  bool ok = true;
  const bool sq = lane < nj && ((P.jq >> lane) & 1u), sqd = lane < nj && ((P.jqd >> lane) & 1u);
  float vq = 0.f, vqd = 0.f;
  if (sq) { vq = jq[e * nj + lane]; ok = ok && isfinite(vq); }
  if (sqd) { vqd = jqd[e * nj + lane]; ok = ok && isfinite(vqd); }
  const int b = lane / 13, k = lane % 13;
  const bool sf = lane < 13 * nf && (((k < 7 ? P.fpose : P.fvel) >> b) & 1u);
  float vf = 0.f;
  if (sf) {
    const float* src = body + (e * K + nd + b) * 13;
    vf = src[k];
    ok = ok && isfinite(vf);
    if (k >= 3 && k < 7) {
      // unfused, correctly rounded fp32: the same bits as ((x x + y y) + z z) + w w, sqrt and divide on any fp32 host
      const float x = src[3], y = src[4], z = src[5], w = src[6];
      const float n2 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z)), __fmul_rn(w, w));
      const float n = __fsqrt_rn(n2);
      ok = ok && n >= 1e-6f && isfinite(n);
      vf = __fdiv_rn(vf, n);
    }
  }
  const bool accept = __ballot_sync(0xffffffffu, !ok) == 0u;
  if (lane == 0) { written[e] = accept ? 1 : 0; if (status) status[e] = accept ? 1 : 2; }
  if (!accept) return;
  float* st = state + e * M.state_stride;
  if (sq) st[lane < nd ? lane : so + 2 * (lane - nd)] = vq;
  if (sqd) st[lane < nd ? nd + lane : so + 2 * (lane - nd) + 1] = vqd;
  if (sf) st[5 * nd + 13 * b + k] = vf;
}

// state row e = snapshot row e for the masked envs (mask NULL: all), every word of the [N, stride] rows
__global__ void prb_restore_state_kernel(float* __restrict__ state, const float* __restrict__ src, const uint8_t* __restrict__ mask,
                                         int64_t words, int stride) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= words) return;
  if (mask && mask[i / stride] == 0) return;
  state[i] = src[i];
}

// returns why a prb_body_states call is rejected, or "" if it is valid
static inline std::string body_query_check(const prb_body_query& q, const void* body, const void* jq, const void* jqd) {
  if (q.frame != 0 && q.frame != 1) return "frame must be 0 (link frame) or 1 (centre-of-mass frame)";
  if (q.reserved != 0) return "reserved must be 0";
  if (!body && !jq && !jqd) return "at least one output is required";
  return "";
}

// prb_state_write and its inputs -> kernel parameters; returns why the call is rejected, or "" if it is valid
static inline std::string state_write_params(const prb_state_write& w, const void* jq, const void* jqd, const void* body,
                                             int nd, int n_free, int n_slide, StateWrite* P) {
  const unsigned nj_mask = (1u << (nd + n_slide)) - 1u, nf_mask = (1u << n_free) - 1u;
  if (w.reserved != 0) return "reserved must be 0";
  if ((w.joint_positions | w.joint_velocities) & ~nj_mask)
    return "joint bits must be below nd + n_slide = " + std::to_string(nd + n_slide);
  if ((w.free_poses | w.free_velocities) & ~nf_mask) return "free-body bits must be below n_free = " + std::to_string(n_free);
  if (!(w.joint_positions | w.joint_velocities | w.free_poses | w.free_velocities)) return "no bit is set: nothing to write";
  if (w.joint_positions && !jq) return "joint_positions needs joint_q_dev";
  if (w.joint_velocities && !jqd) return "joint_velocities needs joint_qd_dev";
  if ((w.free_poses | w.free_velocities) && !body) return "free_poses and free_velocities need body_dev";
  P->jq = w.joint_positions; P->jqd = w.joint_velocities; P->fpose = w.free_poses; P->fvel = w.free_velocities;
  return "";
}

static inline unsigned state_blocks(int N) { return (unsigned)((N + STATE_ENVS - 1) / STATE_ENVS); }
