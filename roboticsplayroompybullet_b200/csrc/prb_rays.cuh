// prb_rays.cuh — ray casts against every env's collision boxes (sm_100a, fp32, CUDA cores); prb_ray_test.
//
// prb_ray_kernel<ENVS>: every env is served by one group of threads that
//   * set-up   with its first warp reads the env's state row (read only) and runs phase_fk without dynamics
//              (render_load_fk, shared with prb_render_kernel) and places the ray frame (a site of the arm); then one
//              thread per collider writes the world -> box transform: the rows of R_box^T with -(R_box^T p_box) and the
//              half extents;
//   * rays     one thread per ray tests every collider of the mask in index order (slab rule below) and writes the
//              nearest hit.
// The launch shape follows R, the rays per env: ENVS = RAY_ENVS_SMALL envs per block of one warp each when R <= 32
// (a warp's set-up serves all its rays); ENVS = 1 above that: one block of up to 8 warps per env and blockIdx.y
// chunks of RAY_CHUNK rays, so that a block's set-up is spread over up to RAY_CHUNK rays.
// The kernel reads the state and writes only the result arrays it is given.
#pragma once
#include <math.h>

#include <string>

#include "../../include/prb.h"
#include "prb_render.cuh"

#define RAY_ENVS_SMALL 4      // envs (warps) per block of the warp-per-env shape
#define RAY_MAX_WARPS 8       // warps per block of the block-per-env shape
#define RAY_CHUNK 1024        // rays per block of the block-per-env shape
#define RAY_MAX_RAYS 16384

struct RayParams {
  int N, R, per_env, frame;
  unsigned long long mask;   // colliders to test, bits >= n_col cleared
};

struct RayMem {
  float4 g[PRB_MAXCOL][3];   // row k of R_box^T, with -(R_box^T p_box)_k in .w: o_k = g_k . (x, 1)
  float4 h[PRB_MAXCOL];      // half extents
  float Rs[9], ps[3];        // ray frame -> world
  RenderFkMem F;
};

// per-collider set-up (thread c)
PRB_D void ray_collider(const DevModel& M, RayMem& S, int c) {
  m3 R; v3 p;
  collider_frame(M, S.F, c, R, p);
  const v3 q = tmul(R, p);
  S.g[c][0] = make_float4(R.m[0], R.m[3], R.m[6], -q.x);
  S.g[c][1] = make_float4(R.m[1], R.m[4], R.m[7], -q.y);
  S.g[c][2] = make_float4(R.m[2], R.m[5], R.m[8], -q.z);
  const v3 h = ld3(M.col_half[c]);
  S.h[c] = make_float4(h.x, h.y, h.z, 0.f);
}

// Entry fraction of the segment a + t d, t in [0, 1], into box c, or +inf for a miss; *axis: the slab whose entry set
// it (-1: none > 0, the start is inside).  This is phase_observe's slab rule (prb_kernels.cuh, gripper_proprioception)
// restated on the precomputed transform: parallel below |dl_k| < 1e-12, t0 from 0 and t1 from 1 clipped per axis, hit
// when t0 <= t1, the caller keeping t0 < 1.  phase_observe is step-pipeline code and stays as it is, so the rule is
// duplicated here; tests/test_cpu_rays.py checks the two agree on the gripper ray.
PRB_D float ray_slab(const RayMem& S, int c, const v3& a, const v3& d, int* axis) {
  const float4 hh = S.h[c];
  float t0 = 0.f, t1 = 1.f;
  int ax = -1;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const float4 g = S.g[c][k];
    const float hk = k == 0 ? hh.x : (k == 1 ? hh.y : hh.z);
    const float ok = fmaf(g.x, a.x, fmaf(g.y, a.y, fmaf(g.z, a.z, g.w)));
    const float dk = fmaf(g.x, d.x, fmaf(g.y, d.y, g.z * d.z));
    if (fabsf(dk) < 1e-12f) {
      if (ok < -hk || ok > hk) return INFINITY;
    } else {
      float ta = (-hk - ok) / dk, tb = (hk - ok) / dk;
      if (ta > tb) { const float tt = ta; ta = tb; tb = tt; }
      if (ta > t0) { t0 = ta; ax = k; }
      t1 = fminf(t1, tb);
    }
  }
  *axis = ax;
  return t0 <= t1 ? t0 : INFINITY;
}

// from / to: [R,3] (per_env 0) or [N,R,3]; col, frac [N,R] (required), pos, nrm [N,R,3] (optional)
template <int ENVS>
__global__ void __launch_bounds__(32 * RAY_MAX_WARPS) prb_ray_kernel(const DevModel* __restrict__ Mp, const float* __restrict__ state,
                                                                    const __grid_constant__ RayParams P, const float* __restrict__ from,
                                                                    const float* __restrict__ to, int* __restrict__ col,
                                                                    float* __restrict__ frac, float* __restrict__ pos, float* __restrict__ nrm) {
  __shared__ RayMem SM[ENVS];
  const DevModel& M = *Mp;
  const int grp = ENVS > 1 ? (int)(threadIdx.x >> 5) : 0;
  const int t = ENVS > 1 ? (int)(threadIdx.x & 31) : (int)threadIdx.x;     // thread of the env's group
  const int gsize = ENVS > 1 ? 32 : (int)blockDim.x;
  const int64_t e = (int64_t)blockIdx.x * ENVS + grp;
  if (e >= P.N) return;                  // whole warps of the last block (ENVS > 1, which syncs per warp only)
  RayMem& S = SM[grp];
  if (t < 32) {
    render_load_fk(M, S.F, state + e * M.state_stride, t);
    if (t == 0 && P.frame >= 0) {
      v3 p; m3 R;
      site_pose(M, S.F, P.frame, p, R);
      stm(S.Rs, R); st3(S.ps, p);
    }
  }
  if (ENVS > 1) __syncwarp(); else __syncthreads();
  for (int c = t; c < M.n_col; c += gsize) ray_collider(M, S, c);
  if (ENVS > 1) __syncwarp(); else __syncthreads();

  const int64_t R = P.R, r0 = (int64_t)blockIdx.y * RAY_CHUNK, r1 = r0 + RAY_CHUNK < R ? r0 + RAY_CHUNK : R;
#pragma unroll 1
  for (int64_t r = r0 + t; r < r1; r += gsize) {
    const int64_t i = e * R + r;                                   // result index; N R 3 may exceed 2^31
    const int64_t src = 3 * (P.per_env ? i : r);
    v3 a = V3(from[src], from[src + 1], from[src + 2]), b = V3(to[src], to[src + 1], to[src + 2]);
    if (P.frame >= 0) {
      const m3 Rs = ldm(S.Rs);
      const v3 ps = ld3(S.ps);
      a = ps + mul(Rs, a); b = ps + mul(Rs, b);
    }
    const v3 d = b - a;
    // explicit: fmaxf / fminf drop NaNs, so the slab arithmetic alone would report hits for a NaN endpoint
    const bool finite = isfinite(a.x) && isfinite(a.y) && isfinite(a.z) && isfinite(d.x) && isfinite(d.y) && isfinite(d.z);
    float best = 1.0f;
    int hit = -1, ax = -1;
    unsigned long long m = finite ? P.mask : 0ull;
    while (m) {
      const int c = __ffsll((long long)m) - 1;
      m &= m - 1;
      const float t0 = ray_slab(S, c, a, d, &ax);
      if (t0 < best) { best = t0; hit = c; }
    }
    col[i] = hit;
    frac[i] = best;
    if (pos) {
      const v3 x = hit >= 0 ? a + d * best : V3(0.f, 0.f, 0.f);
      pos[3 * i] = x.x; pos[3 * i + 1] = x.y; pos[3 * i + 2] = x.z;
    }
    if (nrm) {
      v3 n = V3(0.f, 0.f, 0.f);
      if (hit >= 0) {
        ray_slab(S, hit, a, d, &ax);
        if (ax >= 0) {
          const float4 g = S.g[hit][ax];
          const float dk = fmaf(g.x, d.x, fmaf(g.y, d.y, g.z * d.z));
          n = dk > 0.f ? V3(-g.x, -g.y, -g.z) : V3(g.x, g.y, g.z);
        } else {
          const float L = norm(d);
          if (L > 0.f) n = d * (-1.0f / L);
        }
      }
      nrm[3 * i] = n.x; nrm[3 * i + 1] = n.y; nrm[3 * i + 2] = n.z;
    }
  }
}

// prb_rays and the arrays -> kernel parameters; returns why the call is rejected, or "" if it is valid
static inline std::string ray_params(const prb_rays& r, const void* from, const void* to, const void* col, const void* frac,
                                     int N, int n_col, RayParams* P) {
  if (r.num_rays < 1 || r.num_rays > RAY_MAX_RAYS) return "num_rays must be in 1..16384";
  if (r.per_env != 0 && r.per_env != 1) return "per_env must be 0 (shared [R,3] rays) or 1 ([N,R,3])";
  if (r.frame < -1 || r.frame > 3) return "frame must be -1 (world) or a site 0..3";
  if (r.reserved != 0) return "reserved must be 0";
  if (!from || !to || !col || !frac) return "from_dev, to_dev, hit_collider_dev and hit_fraction_dev are required";
  P->N = N; P->R = r.num_rays; P->per_env = r.per_env; P->frame = r.frame;
  P->mask = r.collider_mask & (n_col >= 64 ? ~0ull : (1ull << n_col) - 1);
  return "";
}

// launch shape of R rays per env: envs per block (template), grid, threads per block
struct RayLaunch { bool small; unsigned gx, gy, threads; };
static inline RayLaunch ray_launch(int N, int R) {
  RayLaunch L;
  L.small = R <= 32;
  if (L.small) { L.gx = (N + RAY_ENVS_SMALL - 1) / RAY_ENVS_SMALL; L.gy = 1; L.threads = 32 * RAY_ENVS_SMALL; }
  else {
    const int warps = (R + 31) / 32 < RAY_MAX_WARPS ? (R + 31) / 32 : RAY_MAX_WARPS;
    L.gx = N; L.gy = (R + RAY_CHUNK - 1) / RAY_CHUNK; L.threads = 32 * warps;
  }
  return L;
}
