// prb_dynamics.cuh — per-env dynamics (prb_enable_dynamics / prb_randomize_dynamics, include/prb.h).
//
// The table (layout: prb_stream.cuh, "per-env dynamics table") overrides the model's collider friction and free-body
// mass, inertia and damping for each env.  The setup kernel is its only reader: it stages an env's free-body constants
// at the start of each launch and reads the env's friction row in place (stage_dynamics); the solver kernels only see
// what the setup kernel derives from them (inverse masses and inertias, row bounds).
//
// prb_randomize_dynamics_kernel (thread per env) draws scale factors s ~ U[lo, hi] and writes value = model value * s
// (fp32), so a draw never compounds.  One draw per body for each friction field (PyBullet keeps friction per link or
// base; all colliders of a body share it), one per free body for mass, linear and angular damping; the inertia diagonal
// takes its mass's draw.  Keying rng4(seed, env_offset + e, reset counter of the env, DYN_RNG_BLOCK + k): the draws
// depend on the seed, the global env id and the episode only, never on sharding, batch size or which envs are drawn
// together.  The reset uses blocks 0-5.
#pragma once
#include "prb_stream.cuh"

#define DYN_RNG_BLOCK 16u
#define DYN_MAXBODY 8          // static scene + arm + free bodies + slide bodies (<= 1 + 1 + PRB_MAXFREE + PRB_MAXSLIDE)

// [lo, hi] per field, the scale of the model's value (include/prb.h prb_dynamics_ranges)
struct DynRanges { float lateral_friction[2], spinning_friction[2], mass[2], linear_damping[2], angular_damping[2]; };

PRB_D float dyn_scale(const float* r, float u) { return clampf(r[0] + (r[1] - r[0]) * u, r[0], r[1]); }

// Uniform draws of one env: u[d] for lateral friction of body d - 1 (d < DYN_MAXBODY), spinning friction of body
// d - DYN_MAXBODY - 1, then mass, linear damping, angular damping of free body b at 2 DYN_MAXBODY + {0, 1, 2} PRB_MAXFREE + b.
#define DYN_NDRAW (2 * DYN_MAXBODY + 3 * PRB_MAXFREE)

__global__ void __launch_bounds__(128) prb_randomize_dynamics_kernel(const DevModel* __restrict__ Mp, const float* __restrict__ state,
                                                                     float* __restrict__ dyn, const unsigned char* __restrict__ mask,
                                                                     int N, unsigned long long seed, unsigned env_offset, DynRanges r) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  if (mask != nullptr && mask[e] == 0) return;
  const DevModel& M = *Mp;
  const int nc = M.n_col, nf = M.n_free;
  // the env's lifetime reset counter: the attempt id of the reset that follows (prb_reset_place_kernel)
  const int o_cnt = 5 * M.nd + 13 * nf + 2 * M.n_slide + M.goal_dim + 8 + 1;
  const uint32_t episode = (uint32_t)state[(size_t)e * M.state_stride + o_cnt];
  float u[(DYN_NDRAW + 3) / 4 * 4];
  for (int k = 0; k < (DYN_NDRAW + 3) / 4; k++) rng4(seed, env_offset + (uint32_t)e, episode, DYN_RNG_BLOCK + (uint32_t)k, u + 4 * k);
  float* fric = dyn + dyn_offset(N, nc, nf, DYN_FRIC) + (size_t)e * nc;
  float* spin = dyn + dyn_offset(N, nc, nf, DYN_SPIN) + (size_t)e * nc;
  for (int c = 0; c < nc; c++) {
    const int body = M.col_body[c] + 1;
    fric[c] = M.col_fric[c] * dyn_scale(r.lateral_friction, u[body]);
    spin[c] = M.col_spin[c] * dyn_scale(r.spinning_friction, u[DYN_MAXBODY + body]);
  }
  for (int b = 0; b < nf; b++) {
    const size_t i = (size_t)e * nf + b;
    const float sm = dyn_scale(r.mass, u[2 * DYN_MAXBODY + b]);
    dyn[dyn_offset(N, nc, nf, DYN_MASS) + i] = M.free_mass[b] * sm;
    for (int k = 0; k < 3; k++) dyn[dyn_offset(N, nc, nf, DYN_INERTIA) + 3 * i + k] = M.free_inertia[b][k] * sm;
    dyn[dyn_offset(N, nc, nf, DYN_LD) + i] = M.free_ld[b] * dyn_scale(r.linear_damping, u[2 * DYN_MAXBODY + PRB_MAXFREE + b]);
    dyn[dyn_offset(N, nc, nf, DYN_AD) + i] = M.free_ad[b] * dyn_scale(r.angular_damping, u[2 * DYN_MAXBODY + 2 * PRB_MAXFREE + b]);
  }
}
