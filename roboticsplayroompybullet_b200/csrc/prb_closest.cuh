// prb_closest.cuh — closest points between the collision boxes of every env (sm_100a, fp32, CUDA cores);
// prb_closest_points.
//
// prb_closest_kernel<CULL>: ONE WARP PER ENV, CLOSEST_ENVS envs per block.
//   * set-up   the warp reads the env's state row (read only) and runs phase_fk without dynamics (render_load_fk, shared
//              with prb_render_kernel and prb_ray_kernel); then one lane per collider writes the world rotation, centre,
//              half extents and bounding radius |h| to shared memory;
//   * query    the lanes list the colliders of both masks and walk the (a, b) pairs, a != b, in (a, b) order.  Culling
//              (CULL): every pair has an upper bound U and a lower bound L of its signed distance from the two
//              centre-in-box distances (closest_bounds); the warp takes min(U + margin) and keeps, compacted by ballot, the
//              pairs whose L - margin is below it and below max_distance.  Then one lane per kept pair computes the exact
//              signed distance and witness (closest_pair) and keeps its best; the warp takes the arg-min on (d, a, b)
//              and the lane that holds it writes the result.
// CULL = false keeps every pair (a test checks that the results are the same bits).  The kernel reads the state and
// writes only the result arrays it is given.
#pragma once
#include <math.h>

#include <cmath>
#include <string>

#include "../../include/prb.h"
#include "prb_render.cuh"

#define CLOSEST_ENVS 4            // envs (warps) per block
#define CLOSEST_MAX_QUERIES 64
#define CLOSEST_EDGE_EPS2 1e-10f  // an edge cross a_i x b_j with |a_i x b_j|^2 below this is not a SAT axis
#define CLOSEST_FREE_EPS 1e-4f    // a box axis with |n.a_k| below this spans the support feature along n (witness only)

struct ClosestParams {
  int N, Q;
  float max_distance;
  int pad;
  unsigned long long ma[CLOSEST_MAX_QUERIES], mb[CLOSEST_MAX_QUERIES];   // bits >= n_col cleared
};

struct ClosestMem {
  float R[PRB_MAXCOL][9];        // world rotation of collider c (row-major; column k is box axis k)
  float4 c[PRB_MAXCOL];          // world centre, bounding radius |h| in .w
  float4 h[PRB_MAXCOL];          // half extents
  unsigned char la[PRB_MAXCOL], lb[PRB_MAXCOL];   // colliders of the query's masks, ascending
  unsigned short buf[64];        // kept pair indices waiting for a full warp
  RenderFkMem F;
};

// per-collider set-up (lane c)
PRB_D void closest_collider(const DevModel& M, ClosestMem& S, int c) {
  m3 R; v3 p;
  collider_frame(M, S.F, c, R, p);
  stm(S.R[c], R);
  const v3 h = ld3(M.col_half[c]);
  S.c[c] = make_float4(p.x, p.y, p.z, norm(h));
  S.h[c] = make_float4(h.x, h.y, h.z, 0.f);
}

PRB_D v3 cl_v3(float4 a) { return V3(a.x, a.y, a.z); }
PRB_D v3 cl_abs(v3 a) { return V3(fabsf(a.x), fabsf(a.y), fabsf(a.z)); }
// column j of B by selects: a runtime index into m3 would put B in local memory
PRB_D v3 cl_col(const m3& B, int j) { return j == 0 ? col(B, 0) : (j == 1 ? col(B, 1) : col(B, 2)); }

// x moved into the support feature of the box |x_k| <= h_k along direction u: an axis with |u_k| < CLOSEST_FREE_EPS is
// free (clamped), the others sit at sign(u_k) h_k (sign(0) = +)
PRB_D v3 cl_feature(v3 x, v3 u, v3 h) {
  return V3(fabsf(u.x) < CLOSEST_FREE_EPS ? clampf(x.x, -h.x, h.x) : (u.x >= 0.f ? h.x : -h.x),
            fabsf(u.y) < CLOSEST_FREE_EPS ? clampf(x.y, -h.y, h.y) : (u.y >= 0.f ? h.y : -h.y),
            fabsf(u.z) < CLOSEST_FREE_EPS ? clampf(x.z, -h.z, h.z) : (u.z >= 0.f ? h.z : -h.z));
}

// signed distance of point p to box (R, c, h): > 0 outside (Euclidean), <= 0 inside (minus the distance to the surface)
PRB_D float closest_point_box(const m3& R, v3 c, v3 h, v3 p) {
  const v3 q = cl_abs(tmul(R, p - c));
  const float dx = q.x - h.x, dy = q.y - h.y, dz = q.z - h.z;
  const float ox = fmaxf(dx, 0.f), oy = fmaxf(dy, 0.f), oz = fmaxf(dz, 0.f);
  return sqrtf(ox * ox + oy * oy + oz * oz) + fminf(fmaxf(dx, fmaxf(dy, dz)), 0.f);
}

// Bounds of the signed distance d of boxes a and b: L <= d <= U, up to the margin *m.  With s_b = point_box(c_b, A):
// d <= max(s_b, 0) (c_b is in B), and d >= s_b - r_b, since every point of B lies within r_b of c_b and moving B by
// r_b - s_b away from A's nearest surface point separates them; likewise with a and b swapped.  *m covers fp32
// rounding of these bounds and of closest_pair, and SAT axes that closest_pair skips (near-parallel edges).
PRB_D void closest_bounds(const ClosestMem& S, int a, int b, float* L, float* U, float* m) {
  const m3 Ra = ldm(S.R[a]), Rb = ldm(S.R[b]);
  const float4 ca = S.c[a], cb = S.c[b];
  const v3 pa = cl_v3(ca), pb = cl_v3(cb);
  const float sb = closest_point_box(Ra, pa, cl_v3(S.h[a]), pb);
  const float sa = closest_point_box(Rb, pb, cl_v3(S.h[b]), pa);
  *L = fmaxf(sb - cb.w, sa - ca.w);
  *U = fminf(fmaxf(sb, 0.f), fmaxf(sa, 0.f));
  *m = 1e-4f + 1e-4f * (norm(pb - pa) + ca.w + cb.w);
}

// Closest points of the segments p + s u, s in [-hp, hp], and q + t v, t in [-hq, hq] (u, v unit): *s, *t.
PRB_D void closest_segments(v3 p, v3 u, float hp, v3 q, v3 v, float hq, float* s_out, float* t_out) {
  const v3 r = p - q;
  const float b = dot(u, v), c = dot(u, r), f = dot(v, r);
  const float den = 1.0f - b * b;
  float s = den > 1e-12f ? clampf((b * f - c) / den, -hp, hp) : 0.f;
  float t = b * s + f;
  if (t < -hq) { t = -hq; s = clampf(b * t - c, -hp, hp); }
  else if (t > hq) { t = hq; s = clampf(b * t - c, -hp, hp); }
  *s_out = s; *t_out = t;
}

// Signed distance of boxes a and b, the witness points on A and B and the normal from B to A (world).
// In A's frame: A is the box |x_k| <= ha_k, B has centre t and axes the columns of Bm.
//   * SAT over 15 axes: A's 3 faces, B's 3 faces, the 9 edge crosses a_i x b_j (skipped when |a_i x b_j|^2 < 1e-10);
//     the overlap along n is ha.|n| + hb.|Bm^T n| - |t.n|; the minimum overlap wins, the lowest axis on a tie.
//   * no axis separates (min overlap >= 0): d = -min overlap; the normal is that axis turned towards A (n.(c_a - c_b) >= 0,
//     the axis as it is on 0).  The witness is one deepest point, chosen among candidates (below) by how far its pair of
//     points lies outside the two boxes and off their support planes: the support vertices alone fail when a small box
//     B rests on a large box A, when two faces overlap in part with no vertex of either over the other, or when a face
//     rests on an edge.
//   * separated: d is the minimum over A's 8 vertices against box B, B's 8 vertices against box A and the 12 x 12
//     edge-edge segment distances (exact for disjoint boxes); the witness is that minimum's pair of points and the normal
//     (pa - pb) / d from the vector whose length gave d (pa and pb are rebuilt in A's frame, which near contact costs
//     pa - pb its relative precision), or the best separating axis when rounding makes d 0.
PRB_D float closest_pair(const ClosestMem& S, int a, int b, v3* pa_w, v3* pb_w, v3* n_w) {
  const m3 Ra = ldm(S.R[a]), Rbw = ldm(S.R[b]);
  const v3 ha = cl_v3(S.h[a]), hb = cl_v3(S.h[b]);
  m3 Bm;                                                       // Ra^T Rb: column j is b_j in A's frame
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) Bm.m[3 * i + j] = Ra.m[i] * Rbw.m[j] + Ra.m[3 + i] * Rbw.m[3 + j] + Ra.m[6 + i] * Rbw.m[6 + j];
  const v3 t = tmul(Ra, cl_v3(S.c[b]) - cl_v3(S.c[a]));

  float best = INFINITY;
  int kbest = 0;
  v3 nbest = V3(1.f, 0.f, 0.f);
#pragma unroll 1
  for (int k = 0; k < 15; k++) {
    v3 n;
    if (k < 3) n = V3(k == 0 ? 1.f : 0.f, k == 1 ? 1.f : 0.f, k == 2 ? 1.f : 0.f);
    else if (k < 6) n = cl_col(Bm, k - 3);
    else {
      const int i = (k - 6) / 3, j = (k - 6) % 3;
      const v3 ei = V3(i == 0 ? 1.f : 0.f, i == 1 ? 1.f : 0.f, i == 2 ? 1.f : 0.f);
      n = cross(ei, cl_col(Bm, j));
      const float l2 = dot(n, n);
      if (l2 < CLOSEST_EDGE_EPS2) continue;
      n = n * (1.0f / sqrtf(l2));
    }
    const float ov = dot(ha, cl_abs(n)) + dot(hb, cl_abs(tmul(Bm, n))) - fabsf(dot(t, n));
    if (ov < best) { best = ov; kbest = k; nbest = n; }
  }
  if (dot(nbest, t) > 0.f) nbest = nbest * -1.0f;             // towards A: n.(c_a - c_b) = -n.t >= 0

  float d;
  v3 pa = V3(0.f, 0.f, 0.f), pb = pa, n = nbest;
  if (best >= 0.f) {                                           // touching or overlapping
    d = -best;
    // candidates (pa = pb + d n in each): for an edge cross the point of A's support edge nearest B's support edge;
    // A's support vertex along -n; B's support vertex along n; two rounds of alternate projection between A's support
    // feature along -n and B's along n shifted by d n (cl_feature: the vertex, edge or face spanned by the axes
    // perpendicular to n), from B's or from A's feature centre.  The first with the least L1 distance outside the two
    // boxes and off the two support planes wins.
    const v3 nb = tmul(Bm, n);
    const v3 va = V3(n.x <= 0.f ? ha.x : -ha.x, n.y <= 0.f ? ha.y : -ha.y, n.z <= 0.f ? ha.z : -ha.z);
    const v3 sb = V3(nb.x >= 0.f ? hb.x : -hb.x, nb.y >= 0.f ? hb.y : -hb.y, nb.z >= 0.f ? hb.z : -hb.z);
    const v3 vb = t + mul(Bm, sb);
    const float lo_a = dot(n, va), hi_b = dot(n, vb);            // min over A and max over B of n.x
    float err = INFINITY;
#pragma unroll 1
    for (int cand = kbest >= 6 ? 0 : 1; cand < 5; cand++) {
      v3 xa, xb;
      if (cand == 0) {
        const int i = (kbest - 6) / 3, j = (kbest - 6) % 3;
        const v3 ei = V3(i == 0 ? 1.f : 0.f, i == 1 ? 1.f : 0.f, i == 2 ? 1.f : 0.f);
        const v3 bj = cl_col(Bm, j);
        const v3 qa = va - ei * comp(va, i), qb = vb - bj * comp(sb, j);
        float s, u;
        closest_segments(qa, ei, comp(ha, i), qb, bj, comp(hb, j), &s, &u);
        xa = qa + ei * s;
        xb = xa - n * d;
      } else if (cand == 1) { xa = va; xb = va - n * d; }
      else if (cand == 2) { xb = vb; xa = vb + n * d; }
      else {                             // alternate between the two support features, from B's (3) or A's (4) centre
        const v3 mn = n * -1.0f;
        xa = cand == 3 ? cl_feature(t + mul(Bm, cl_feature(V3(0.f, 0.f, 0.f), nb, hb)) + n * d, mn, ha)
                       : cl_feature(V3(0.f, 0.f, 0.f), mn, ha);
#pragma unroll 1
        for (int it = 0; it < 2; it++) {
          xb = t + mul(Bm, cl_feature(tmul(Bm, xa - n * d - t), nb, hb));
          xa = cl_feature(xb + n * d, mn, ha);
        }
        xb = xa - n * d;
      }
      const v3 oa = cl_abs(xa) - ha, ob = cl_abs(tmul(Bm, xb - t)) - hb;
      const float e = fmaxf(oa.x, 0.f) + fmaxf(oa.y, 0.f) + fmaxf(oa.z, 0.f) + fmaxf(ob.x, 0.f) + fmaxf(ob.y, 0.f) +
                      fmaxf(ob.z, 0.f) + fabsf(dot(n, xa) - lo_a) + fabsf(dot(n, xb) - hi_b);
      if (e < err) { err = e; pa = xa; pb = xb; }
    }
  } else {                                                     // separated: feature enumeration
    float d2 = INFINITY;
    v3 sv = n;                                                 // pa - pb of the best feature, as its distance sees it
#pragma unroll 1
    for (int v = 0; v < 8; v++) {
      const v3 sg = V3(v & 1 ? -1.f : 1.f, v & 2 ? -1.f : 1.f, v & 4 ? -1.f : 1.f);
      // vertex of A against B
      const v3 x = V3(sg.x * ha.x, sg.y * ha.y, sg.z * ha.z);
      const v3 q = tmul(Bm, x - t);
      const v3 qc = V3(clampf(q.x, -hb.x, hb.x), clampf(q.y, -hb.y, hb.y), clampf(q.z, -hb.z, hb.z));
      const v3 dq = q - qc;
      const float e2 = dot(dq, dq);
      if (e2 < d2) { d2 = e2; pa = x; pb = t + mul(Bm, qc); sv = mul(Bm, dq); }
      // vertex of B against A
      const v3 y = t + mul(Bm, V3(sg.x * hb.x, sg.y * hb.y, sg.z * hb.z));
      const v3 yc = V3(clampf(y.x, -ha.x, ha.x), clampf(y.y, -ha.y, ha.y), clampf(y.z, -ha.z, ha.z));
      const v3 dy = y - yc;
      const float f2 = dot(dy, dy);
      if (f2 < d2) { d2 = f2; pa = yc; pb = y; sv = dy * -1.0f; }
    }
#pragma unroll 1
    for (int ea = 0; ea < 12; ea++) {
      const int i = ea >> 2;                                   // edge of A along axis i, the others at +-h
      const int i1 = i == 0 ? 1 : 0, i2 = i == 2 ? 1 : 2;
      const float s1 = ea & 1 ? -1.f : 1.f, s2 = ea & 2 ? -1.f : 1.f;
      const v3 p = V3(i1 == 0 ? s1 * ha.x : 0.f, i1 == 1 ? s1 * ha.y : (i2 == 1 ? s2 * ha.y : 0.f), i2 == 2 ? s2 * ha.z : 0.f);
      const v3 u = V3(i == 0 ? 1.f : 0.f, i == 1 ? 1.f : 0.f, i == 2 ? 1.f : 0.f);
#pragma unroll 1
      for (int eb = 0; eb < 12; eb++) {
        const int j = eb >> 2;
        const int j1 = j == 0 ? 1 : 0, j2 = j == 2 ? 1 : 2;
        const float r1 = eb & 1 ? -1.f : 1.f, r2 = eb & 2 ? -1.f : 1.f;
        const v3 lq = V3(j1 == 0 ? r1 * hb.x : 0.f, j1 == 1 ? r1 * hb.y : (j2 == 1 ? r2 * hb.y : 0.f), j2 == 2 ? r2 * hb.z : 0.f);
        const v3 q = t + mul(Bm, lq), v = cl_col(Bm, j);
        float s, w;
        closest_segments(p, u, comp(ha, i), q, v, comp(hb, j), &s, &w);
        const v3 xa = p + u * s, xb = q + v * w, dd = xa - xb;
        const float e2 = dot(dd, dd);
        if (e2 < d2) { d2 = e2; pa = xa; pb = xb; sv = dd; }
      }
    }
    d = sqrtf(d2);
    if (d > 0.f) n = sv * (1.0f / d);
  }
  const v3 ca = cl_v3(S.c[a]);
  *pa_w = ca + mul(Ra, pa);
  *pb_w = ca + mul(Ra, pb);
  *n_w = mul(Ra, n);
  return d;
}

// col_a, col_b, dist [N,Q] (required), pos_a, pos_b, nrm [N,Q,3] (optional)
// __maxnreg__: with __launch_bounds__(128) ptxas stops at 80 registers and spills; 96 leaves it at 84 with no stack
template <bool CULL>
__global__ void __maxnreg__(96) prb_closest_kernel(const DevModel* __restrict__ Mp, const float* __restrict__ state,
                                                   const __grid_constant__ ClosestParams P, int* __restrict__ col_a,
                                                   int* __restrict__ col_b, float* __restrict__ dist, float* __restrict__ pos_a,
                                                   float* __restrict__ pos_b, float* __restrict__ nrm) {
  __shared__ ClosestMem SM[CLOSEST_ENVS];
  const DevModel& M = *Mp;
  const int w = (int)(threadIdx.x >> 5), lane = (int)(threadIdx.x & 31);
  const int64_t e = (int64_t)blockIdx.x * CLOSEST_ENVS + w;
  if (e >= P.N) return;                  // whole warps of the last block; every sync below is per warp
  ClosestMem& S = SM[w];
  render_load_fk(M, S.F, state + e * M.state_stride, lane);
  __syncwarp();
  for (int c = lane; c < M.n_col; c += 32) closest_collider(M, S, c);
  const unsigned lt = (1u << lane) - 1u;

#pragma unroll 1
  for (int q = 0; q < P.Q; q++) {
    __syncwarp();                        // the previous query's lists and buffer are no longer read
    const unsigned long long ma = P.ma[q], mb = P.mb[q];
    for (int c = lane; c < PRB_MAXCOL; c += 32) {
      const unsigned long long below = (1ull << c) - 1ull;
      if ((ma >> c) & 1ull) S.la[__popcll(ma & below)] = (unsigned char)c;
      if ((mb >> c) & 1ull) S.lb[__popcll(mb & below)] = (unsigned char)c;
    }
    __syncwarp();
    const int nb = __popcll(mb), np = __popcll(ma) * nb;
    float thr = P.max_distance;
    if (CULL) {
      float u = INFINITY;
      for (int p = lane; p < np; p += 32) {
        const int a = S.la[p / nb], b = S.lb[p % nb];
        if (a == b) continue;
        float L, U, m;
        closest_bounds(S, a, b, &L, &U, &m);
        u = fminf(u, U + m);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) u = fminf(u, __shfl_xor_sync(0xffffffffu, u, o));
      thr = fminf(thr, u);
    }
    float bd = INFINITY;                 // this lane's best pair and its witness (world)
    int bp = 0x7fffffff;
    v3 ba = V3(0.f, 0.f, 0.f), bb = ba, bn = ba;
    int cnt = 0;
    for (int base = 0; base < np; base += 32) {
      const int p = base + lane;
      bool keep = false;
      if (p < np) {
        const int a = S.la[p / nb], b = S.lb[p % nb];
        keep = a != b;
        if (CULL && keep) {
          float L, U, m;
          closest_bounds(S, a, b, &L, &U, &m);
          keep = L - m <= thr;
        }
      }
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      if (keep) S.buf[cnt + __popc(bal & lt)] = (unsigned short)p;
      cnt += __popc(bal);
      __syncwarp();
      if (cnt >= 32) {                   // a full warp of kept pairs
        const int pp = S.buf[lane];
        v3 xa, xb, xn;
        const float d = closest_pair(S, S.la[pp / nb], S.lb[pp % nb], &xa, &xb, &xn);
        if (d <= P.max_distance && (d < bd || (d == bd && pp < bp))) { bd = d; bp = pp; ba = xa; bb = xb; bn = xn; }
        __syncwarp();
        if (lane < cnt - 32) S.buf[lane] = S.buf[32 + lane];
        cnt -= 32;
        __syncwarp();
      }
    }
    if (lane < cnt) {
      const int pp = S.buf[lane];
      v3 xa, xb, xn;
      const float d = closest_pair(S, S.la[pp / nb], S.lb[pp % nb], &xa, &xb, &xn);
      if (d <= P.max_distance && (d < bd || (d == bd && pp < bp))) { bd = d; bp = pp; ba = xa; bb = xb; bn = xn; }
    }
    float wd = bd;                       // warp arg-min on (d, p); the lane holding it writes (lane 0 a miss)
    int wp = bp;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float od = __shfl_xor_sync(0xffffffffu, wd, o);
      const int op = __shfl_xor_sync(0xffffffffu, wp, o);
      if (od < wd || (od == wd && op < wp)) { wd = od; wp = op; }
    }
    if (wp == 0x7fffffff ? lane == 0 : bp == wp) {
      const int64_t i = e * P.Q + q;     // result index
      const bool hit = wp != 0x7fffffff;
      if (!hit) { ba = V3(0.f, 0.f, 0.f); bb = ba; bn = ba; }
      col_a[i] = hit ? (int)S.la[wp / nb] : -1; col_b[i] = hit ? (int)S.lb[wp % nb] : -1; dist[i] = wd;
      if (pos_a) { pos_a[3 * i] = ba.x; pos_a[3 * i + 1] = ba.y; pos_a[3 * i + 2] = ba.z; }
      if (pos_b) { pos_b[3 * i] = bb.x; pos_b[3 * i + 1] = bb.y; pos_b[3 * i + 2] = bb.z; }
      if (nrm) { nrm[3 * i] = bn.x; nrm[3 * i + 1] = bn.y; nrm[3 * i + 2] = bn.z; }
    }
  }
}

// prb_closest, the queries and the arrays -> kernel parameters; returns why the call is rejected, or "" if it is valid
static inline std::string closest_params(const prb_closest& c, const prb_closest_query* queries, const void* col_a,
                                         const void* col_b, const void* dist, int N, int n_col, ClosestParams* P) {
  if (c.num_queries < 1 || c.num_queries > CLOSEST_MAX_QUERIES) return "num_queries must be in 1..64";
  if (c.reserved != 0 || c.reserved2 != 0) return "reserved fields must be 0";
  if (!std::isfinite(c.max_distance) || c.max_distance < 0.f) return "max_distance must be finite and >= 0";
  if (!queries || !col_a || !col_b || !dist) return "queries_host, collider_a_dev, collider_b_dev and distance_dev are required";
  const unsigned long long valid = n_col >= 64 ? ~0ull : (1ull << n_col) - 1;
  P->N = N; P->Q = c.num_queries; P->max_distance = c.max_distance; P->pad = 0;
  for (int q = 0; q < CLOSEST_MAX_QUERIES; q++) {
    P->ma[q] = q < c.num_queries ? queries[q].mask_a & valid : 0ull;
    P->mb[q] = q < c.num_queries ? queries[q].mask_b & valid : 0ull;
  }
  return "";
}

static inline unsigned closest_blocks(int N) { return (unsigned)((N + CLOSEST_ENVS - 1) / CLOSEST_ENVS); }
