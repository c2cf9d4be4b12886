// prb_render.cuh — camera images of the batched worlds (sm_100a, fp32, CUDA cores).
//
// prb_render_kernel: ONE BLOCK PER ENV (RENDER_WARPS warps).  Every collider is an oriented box, so a frame is a
// ray cast against at most PRB_MAXCOL boxes per pixel:
//   * set-up   warp 0 reads the env's state row (read only), runs phase_fk without dynamics and places the camera
//              (composed with the end-effector site 0 for an attached camera); then one thread per collider writes
//              the box's rotation from camera to box coordinates, the slab offsets of the eye (the eye is the same
//              for every pixel), the box axes dotted with the light and the box's conservative screen rectangle;
//   * pixels   each warp takes 8x8 tiles in turn, builds the 64-bit mask of the boxes whose rectangle meets the
//              tile (two ballots: PRB_MAXCOL = 64 is one word) and tests two pixels per lane against those boxes
//              only: slab test with phase_observe's parallel-ray rule, nearest entry in [near, far), the lower
//              collider index on a tie; then shading of the face that was hit.
// The kernel reads the state and writes only the image buffers it is given (and the box-test counter).
#pragma once
#include <math.h>
#include <string.h>

#include <cmath>
#include <string>

#include "../../include/prb.h"
#include "prb_kernels.cuh"

#define RENDER_WARPS 8
#define RENDER_TILE 8

// Everything a frame needs besides the model and the state, passed by value (__grid_constant__): no copy per call.
struct RenderParams {
  int W, H, attach, tiles_x, n_tiles;
  // eye-space ray of the pixel at NDC (x, y): h = inverse(proj) (x, y, 1, 1) = (ray[0] x + ray[1] y + ray[2],
  // ray[3] x + ray[4] y + ray[5], ray[6] x + ray[7] y + ray[8], .); the direction scaled to unit eye depth is
  // (-h.x / h.z, -h.y / h.z, -1), so the ray parameter of a hit is its eye-space depth
  float ray[9];
  float proj[8];        // rows 0 and 1 of the projection (culling); clip w = -z_eye
  float near_d, far_d;  // eye depth of the near and far planes
  float cam[12];        // camera frame -> reference frame (world, or site 0 when attached): R (row-major), t
  float light[3], ambient, diffuse, background[3];
  float rgb[PRB_MAXCOL][3];
};

// the fields phase_fk / body_frame / site_pose read and write
struct RenderFkMem {
  float q[PRB_MAXD], qd[PRB_MAXD];
  float lR[PRB_MAXD][9], lp[PRB_MAXD][3], la[PRB_MAXD][3], lw[PRB_MAXD][3], lv[PRB_MAXD][3], lc[PRB_MAXD][3];
  float lIw[PRB_MAXD][6], lf[PRB_MAXD][3], ln[PRB_MAXD][3];
  float fpos[PRB_MAXFREE][3], fquat[PRB_MAXFREE][4], fR[PRB_MAXFREE][9], fIinv[PRB_MAXFREE][6];
  float sq[PRB_MAXSLIDE], sR[PRB_MAXSLIDE][9], sp[PRB_MAXSLIDE][3];
};

struct RenderMem {
  float4 geo[PRB_MAXCOL][4];   // rows k of B = R_box^T R_cam with a_k = -h_k - o_k in .w, then (b_k = h_k - o_k, -)
  float4 rect[PRB_MAXCOL];     // pixel-index rectangle (j_lo, i_lo, j_hi, i_hi) with one pixel of margin
  float ndl[PRB_MAXCOL][3];    // box axis k (world) . light
  float Rc[9], eye[3];         // camera frame -> world
  RenderFkMem F;
};

// reciprocal of a ray component; |d| < 1e-12 is a ray parallel to the slab (phase_observe's rule), where a huge
// finite value keeps that rule's inside / outside decision without a branch
PRB_D float render_rcp(float d) { return fabsf(d) < 1e-12f ? copysignf(1e30f, d) : __fdividef(1.0f, d); }

// Entry depth of the ray t (dx, dy, -1) (camera coordinates, from the eye) into box g, or +inf for a miss.
PRB_D float render_slab(const float4& g0, const float4& g1, const float4& g2, const float4& g3, float dx, float dy,
                        float nearv, float farv) {
  const float i0 = render_rcp(fmaf(g0.x, dx, fmaf(g0.y, dy, -g0.z)));
  const float i1 = render_rcp(fmaf(g1.x, dx, fmaf(g1.y, dy, -g1.z)));
  const float i2 = render_rcp(fmaf(g2.x, dx, fmaf(g2.y, dy, -g2.z)));
  const float a0 = g0.w * i0, b0 = g3.x * i0, a1 = g1.w * i1, b1 = g3.y * i1, a2 = g2.w * i2, b2 = g3.z * i2;
  const float t0 = fmaxf(fmaxf(nearv, fminf(a0, b0)), fmaxf(fminf(a1, b1), fminf(a2, b2)));
  const float t1 = fminf(fminf(farv, fmaxf(a0, b0)), fminf(fmaxf(a1, b1), fmaxf(a2, b2)));
  return t0 <= t1 ? t0 : INFINITY;
}

// n . light for the face through which the ray enters box c; where the near plane cuts the box, n = -ray direction
PRB_D float render_ndl(const RenderMem& S, const RenderParams& P, int c, float dx, float dy) {
  float best = -INFINITY, ndl = 0.f;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const float4 g = S.geo[c][k];
    const float bk = k == 0 ? S.geo[c][3].x : (k == 1 ? S.geo[c][3].y : S.geo[c][3].z);
    const float d = fmaf(g.x, dx, fmaf(g.y, dy, -g.z));
    const float inv = render_rcp(d);
    const float lo = fminf(g.w * inv, bk * inv);
    if (lo > best) { best = lo; ndl = d > 0.f ? -S.ndl[c][k] : S.ndl[c][k]; }
  }
  if (best < P.near_d) {
    const v3 dw = mul(ldm(S.Rc), V3(dx, dy, -1.0f));
    ndl = -dot(dw, ld3(P.light)) / norm(dw);
  }
  return ndl;
}

// lanes of one warp: the env's state row st (read only) -> F, positions with zero velocities, then phase_fk without
// dynamics; prb_render_kernel and prb_ray_kernel (prb_rays.cuh) place the colliders and sites from F
PRB_D void render_load_fk(const DevModel& M, RenderFkMem& F, const float* st, int lane) {
  if (lane < M.nd) { F.q[lane] = st[lane]; F.qd[lane] = 0.f; }
  if (lane < M.n_free) {
    for (int k = 0; k < 3; k++) F.fpos[lane][k] = st[5 * M.nd + 13 * lane + k];
    for (int k = 0; k < 4; k++) F.fquat[lane][k] = st[5 * M.nd + 13 * lane + 3 + k];
  }
  if (lane < M.n_slide) F.sq[lane] = st[5 * M.nd + 13 * M.n_free + 2 * lane];
  __syncwarp();
  phase_fk(M, F, lane, false);
}

PRB_D unsigned char render_byte(float x) { return (unsigned char)floorf(255.0f * clampf(x, 0.f, 1.f) + 0.5f); }

// per-collider set-up (thread c): camera -> box rotation, slab offsets of the eye, axes . light, screen rectangle
PRB_D void render_collider(const DevModel& M, RenderMem& S, const RenderParams& P, int c) {
  m3 R; v3 p;
  collider_frame(M, S.F, c, R, p);
  const m3 Rc = ldm(S.Rc);
  const v3 eye = ld3(S.eye), h = ld3(M.col_half[c]);
  m3 RT;
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) RT.m[3 * i + j] = R.m[3 * j + i];
  const m3 B = mul(RT, Rc);
  const v3 o = tmul(R, eye - p);
  S.geo[c][0] = make_float4(B.m[0], B.m[1], B.m[2], -h.x - o.x);
  S.geo[c][1] = make_float4(B.m[3], B.m[4], B.m[5], -h.y - o.y);
  S.geo[c][2] = make_float4(B.m[6], B.m[7], B.m[8], -h.z - o.z);
  S.geo[c][3] = make_float4(h.x - o.x, h.y - o.y, h.z - o.z, 0.f);
  const v3 l = ld3(P.light);
  for (int k = 0; k < 3; k++) S.ndl[c][k] = dot(col(R, k), l);
  // corners in camera coordinates: centre Rc^T (p - eye) + (R_c^T R) (+-h) = ce + B^T (+-h)
  const v3 ce = tmul(Rc, p - eye);
  float jlo = INFINITY, jhi = -INFINITY, ilo = INFINITY, ihi = -INFINITY;
  bool full = false, all_far = true;
  for (int k = 0; k < 8; k++) {
    const v3 s = V3((k & 1) ? h.x : -h.x, (k & 2) ? h.y : -h.y, (k & 4) ? h.z : -h.z);
    const v3 e = ce + tmul(B, s);
    const float w = -e.z;
    if (w < P.near_d) full = true;
    if (w <= P.far_d) all_far = false;
    const float xc = P.proj[0] * e.x + P.proj[1] * e.y + P.proj[2] * e.z + P.proj[3];
    const float yc = P.proj[4] * e.x + P.proj[5] * e.y + P.proj[6] * e.z + P.proj[7];
    const float j = (xc / w + 1.0f) * 0.5f * P.W - 0.5f, i = (1.0f - yc / w) * 0.5f * P.H - 0.5f;
    jlo = fminf(jlo, j); jhi = fmaxf(jhi, j); ilo = fminf(ilo, i); ihi = fmaxf(ihi, i);
  }
  float4 r = make_float4(jlo - 1.0f, ilo - 1.0f, jhi + 1.0f, ihi + 1.0f);
  if (full) r = make_float4(-1e30f, -1e30f, 1e30f, 1e30f);
  if (all_far) r = make_float4(1e30f, 1e30f, -1e30f, -1e30f);    // wholly beyond the far plane
  S.rect[c] = r;
}

// rgb [N,H,W,3] (required), depth [N,H,W] and seg [N,H,W] (optional); tests: pixel-box tests summed (optional)
__global__ void __launch_bounds__(32 * RENDER_WARPS) prb_render_kernel(const DevModel* __restrict__ Mp, const float* __restrict__ state,
                                                                      const __grid_constant__ RenderParams P, unsigned char* __restrict__ rgb,
                                                                      float* __restrict__ depth, int* __restrict__ seg,
                                                                      unsigned long long* __restrict__ tests) {
  __shared__ RenderMem S;
  const DevModel& M = *Mp;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t e = blockIdx.x;
  if (warp == 0) {
    RenderFkMem& F = S.F;
    render_load_fk(M, F, state + e * M.state_stride, lane);
    if (lane == 0) {
      m3 Rc = ldm(P.cam);
      v3 eye = ld3(P.cam + 9);
      if (P.attach) {
        v3 ps; m3 Rs;
        site_pose(M, F, 0, ps, Rs);
        eye = ps + mul(Rs, eye);
        Rc = mul(Rs, Rc);
      }
      stm(S.Rc, Rc); st3(S.eye, eye);
    }
  }
  __syncthreads();
  if ((int)threadIdx.x < M.n_col) render_collider(M, S, P, threadIdx.x);
  __syncthreads();

  const int W = P.W, H = P.H, ncol = M.n_col;
  const size_t img0 = e * (size_t)W * H;
  unsigned count = 0;                 // pixel-box tests of this lane
  const unsigned char bg[3] = {render_byte(P.background[0]), render_byte(P.background[1]), render_byte(P.background[2])};
#pragma unroll 1
  for (int t = warp; t < P.n_tiles; t += RENDER_WARPS) {
    const int x0 = (t % P.tiles_x) * RENDER_TILE, y0 = (t / P.tiles_x) * RENDER_TILE;
    const float fx0 = (float)x0, fy0 = (float)y0, fx1 = (float)(x0 + RENDER_TILE - 1), fy1 = (float)(y0 + RENDER_TILE - 1);
    bool in0 = false, in1 = false;
    if (lane < ncol) { const float4 r = S.rect[lane]; in0 = r.x <= fx1 && r.z >= fx0 && r.y <= fy1 && r.w >= fy0; }
    if (lane + 32 < ncol) { const float4 r = S.rect[lane + 32]; in1 = r.x <= fx1 && r.z >= fx0 && r.y <= fy1 && r.w >= fy0; }
    const unsigned long long mask = (unsigned long long)__ballot_sync(FULL, in0) | ((unsigned long long)__ballot_sync(FULL, in1) << 32);
    // lane's two pixels: rows lane / 8 and 4 + lane / 8 of the tile, column lane % 8
    const int j = x0 + (lane & 7), i0 = y0 + (lane >> 3), i1 = i0 + 4;
    const float xn = 2.0f * (j + 0.5f) / W - 1.0f;
    const float yn0 = 1.0f - 2.0f * (i0 + 0.5f) / H, yn1 = 1.0f - 2.0f * (i1 + 0.5f) / H;
    float dx[2], dy[2];
    {
      const float yn[2] = {yn0, yn1};
#pragma unroll
      for (int q = 0; q < 2; q++) {
        const float hx = fmaf(P.ray[0], xn, fmaf(P.ray[1], yn[q], P.ray[2]));
        const float hy = fmaf(P.ray[3], xn, fmaf(P.ray[4], yn[q], P.ray[5]));
        const float hz = fmaf(P.ray[6], xn, fmaf(P.ray[7], yn[q], P.ray[8]));
        const float s = -1.0f / hz;
        dx[q] = hx * s; dy[q] = hy * s;
      }
    }
    float best0 = P.far_d, best1 = P.far_d;
    int hit0 = -1, hit1 = -1;
    unsigned long long m = mask;
    while (m) {
      const int c = __ffsll((long long)m) - 1;
      m &= m - 1;
      const float4 g0 = S.geo[c][0], g1 = S.geo[c][1], g2 = S.geo[c][2], g3 = S.geo[c][3];
      const float t0 = render_slab(g0, g1, g2, g3, dx[0], dy[0], P.near_d, P.far_d);
      const float t1 = render_slab(g0, g1, g2, g3, dx[1], dy[1], P.near_d, P.far_d);
      if (t0 < best0) { best0 = t0; hit0 = c; }
      if (t1 < best1) { best1 = t1; hit1 = c; }
    }
    const bool v0 = j < W && i0 < H, v1 = j < W && i1 < H;
    count += (unsigned)__popcll(mask) * ((v0 ? 1u : 0u) + (v1 ? 1u : 0u));
#pragma unroll
    for (int q = 0; q < 2; q++) {
      const bool v = q == 0 ? v0 : v1;
      if (!v) continue;
      const int hit = q == 0 ? hit0 : hit1;
      const size_t px = img0 + (size_t)(q == 0 ? i0 : i1) * W + j;
      unsigned char* o = rgb + 3 * px;
      if (hit >= 0) {
        const float ndl = render_ndl(S, P, hit, dx[q], dy[q]);
        const float shade = P.ambient + P.diffuse * fmaxf(0.f, ndl);
        o[0] = render_byte(P.rgb[hit][0] * shade); o[1] = render_byte(P.rgb[hit][1] * shade); o[2] = render_byte(P.rgb[hit][2] * shade);
      } else {
        o[0] = bg[0]; o[1] = bg[1]; o[2] = bg[2];
      }
      if (depth) depth[px] = q == 0 ? best0 : best1;
      if (seg) seg[px] = hit;
    }
  }
  if (tests) {
    for (int o = 16; o > 0; o >>= 1) count += __shfl_xor_sync(FULL, count, o);
    if (lane == 0 && count) atomicAdd(tests, (unsigned long long)count);
  }
}

// ---------------------------------------------------------------------------- camera set-up (host, fp64)
// Gauss-Jordan inverse with partial pivoting; false when a is singular (relative to its largest entry).
static inline bool inv4(const double a_in[4][4], double out[4][4]) {
  double a[4][8], amax = 0;
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 8; j++) { a[i][j] = j < 4 ? a_in[i][j] : (j - 4 == i ? 1.0 : 0.0); if (j < 4) amax = fmax(amax, fabs(a[i][j])); }
  if (!(amax > 0) || !std::isfinite(amax)) return false;
  for (int c = 0; c < 4; c++) {
    int p = c;
    for (int r = c + 1; r < 4; r++) if (fabs(a[r][c]) > fabs(a[p][c])) p = r;
    if (!(fabs(a[p][c]) > 1e-9 * amax)) return false;
    for (int j = 0; j < 8; j++) { double t = a[c][j]; a[c][j] = a[p][j]; a[p][j] = t; }
    const double d = a[c][c];
    for (int j = 0; j < 8; j++) a[c][j] /= d;
    for (int r = 0; r < 4; r++) {
      if (r == c) continue;
      const double f = a[r][c];
      for (int j = 0; j < 8; j++) a[r][j] -= f * a[c][j];
    }
  }
  for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) out[i][j] = a[i][4 + j];
  return true;
}

// prb_camera -> kernel parameters; returns why the camera is rejected, or "" if it is valid
static inline std::string render_params(const prb_camera& c, const float* rgb, int n_col, RenderParams* P) {
  if (c.width < 1 || c.width > 1024 || c.height < 1 || c.height > 1024) return "width and height must be in 1..1024";
  if (c.attach != 0 && c.attach != 1) return "attach must be 0 (world camera) or 1 (end-effector site frame)";
  double V[4][4], Pm[4][4], PV[4][4], tmp[4][4];
  for (int r = 0; r < 4; r++)
    for (int k = 0; k < 4; k++) { V[r][k] = c.view[4 * k + r]; Pm[r][k] = c.proj[4 * k + r]; }   // column-major
  for (int r = 0; r < 4; r++)
    for (int k = 0; k < 4; k++) {
      double s = 0;
      for (int m = 0; m < 4; m++) s += Pm[r][m] * V[m][k];
      PV[r][k] = s;
    }
  if (!inv4(PV, tmp)) return "proj * view is singular";
  double Pinv[4][4];
  if (!inv4(Pm, Pinv)) return "proj is singular";
  if (fabs(Pm[3][0]) > 1e-6 || fabs(Pm[3][1]) > 1e-6 || fabs(Pm[3][3]) > 1e-6 || fabs(Pm[3][2] + 1.0) > 1e-6)
    return "proj must be a perspective projection with clip w = -z_eye (computeProjectionMatrixFOV layout)";
  if (fabs(V[3][0]) > 1e-6 || fabs(V[3][1]) > 1e-6 || fabs(V[3][2]) > 1e-6 || fabs(V[3][3] - 1.0) > 1e-6) return "view must be a rigid transform";
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      double s = 0;
      for (int m = 0; m < 3; m++) s += V[i][m] * V[j][m];
      if (fabs(s - (i == j ? 1.0 : 0.0)) > 1e-4) return "view must be a rigid transform (orthonormal rotation)";
    }
  const double A = Pm[2][2], B = Pm[2][3];
  const double nearv = B / (A - 1.0), farv = B / (A + 1.0);
  if (!(nearv > 0 && farv > nearv && std::isfinite(farv))) return "proj must have 0 < near < far";
  double L = 0;
  for (int k = 0; k < 3; k++) L += (double)c.light_dir[k] * c.light_dir[k];
  L = sqrt(L);
  if (!(L > 0) || !std::isfinite(L)) return "light_dir must be a non-zero finite vector";
  if (!std::isfinite(c.ambient) || !std::isfinite(c.diffuse)) return "ambient and diffuse must be finite";
  memset(P, 0, sizeof(*P));
  P->W = c.width; P->H = c.height; P->attach = c.attach;
  P->tiles_x = (c.width + RENDER_TILE - 1) / RENDER_TILE;
  P->n_tiles = P->tiles_x * ((c.height + RENDER_TILE - 1) / RENDER_TILE);
  for (int r = 0; r < 3; r++) {
    P->ray[3 * r] = (float)Pinv[r][0]; P->ray[3 * r + 1] = (float)Pinv[r][1]; P->ray[3 * r + 2] = (float)(Pinv[r][2] + Pinv[r][3]);
  }
  for (int r = 0; r < 2; r++) for (int k = 0; k < 4; k++) P->proj[4 * r + k] = (float)Pm[r][k];
  P->near_d = (float)nearv; P->far_d = (float)farv;
  // inverse of the rigid view: R^T, -R^T t
  for (int i = 0; i < 3; i++) {
    for (int j = 0; j < 3; j++) P->cam[3 * i + j] = (float)V[j][i];
    P->cam[9 + i] = (float)(-(V[0][i] * V[0][3] + V[1][i] * V[1][3] + V[2][i] * V[2][3]));
  }
  for (int k = 0; k < 3; k++) {
    P->light[k] = (float)(c.light_dir[k] / L);
    if (!std::isfinite(c.background[k])) return "background must be finite";
    P->background[k] = c.background[k];
  }
  P->ambient = c.ambient; P->diffuse = c.diffuse;
  for (int i = 0; i < n_col; i++)
    for (int k = 0; k < 3; k++) {
      if (!std::isfinite(rgb[3 * i + k])) return "colours must be finite";
      P->rgb[i][k] = rgb[3 * i + k];
    }
  return "";
}
