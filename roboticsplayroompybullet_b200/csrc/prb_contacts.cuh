// prb_contacts.cuh — the contact report (prb_enable_contacts / prb_get_contacts, include/prb.h).
//
// With the report enabled, a step's last build launch of the setup kernel writes every contact's colliders, geometry and
// the locator of its solver record into the report (phase_rows_stream), the solver kernels of that substep copy their
// staged impulses back to the records (their writeback flag), and prb_contact_report_kernel, launched once after the
// step's final setup launch (which integrates and observes but builds no rows, so the records survive it), turns the
// impulses into forces and writes the padding.  Layout of the report: prb_stream.cuh, "contact report".
#pragma once
#include "prb_stream.cuh"

#define CREP_WPB 8      // envs (one warp each) per block

enum { CREP_REPORT = 0, CREP_CLEAR = 1 };

// CREP_REPORT: forces of the contacts the last substep solved (impulse / dt), padding after them.
// CREP_CLEAR: count 0 and padding everywhere for the envs of `mask` (every env when mask is NULL).
__global__ void __launch_bounds__(32 * CREP_WPB) prb_contact_report_kernel(float* __restrict__ crep, const float* __restrict__ sbuf,
                                                                          const float4* __restrict__ hbuf, int N, float dt, int mode,
                                                                          const unsigned char* __restrict__ mask) {
  const int lane = threadIdx.x & 31;
  const int e = blockIdx.x * CREP_WPB + (threadIdx.x >> 5);
  if (e >= N) return;
  if (mode == CREP_CLEAR && mask != nullptr && mask[e] == 0) return;
  int* cnt = crep_count(crep, N);
  const int n = mode == CREP_REPORT ? cnt[e] : 0;
  if (mode == CREP_CLEAR && lane == 0) cnt[e] = 0;
  const size_t NS = (size_t)N * SB_MAXCONTACT, s0 = (size_t)e * SB_MAXCONTACT;
  const float4* col = reinterpret_cast<const float4*>(sbuf) + (size_t)(e >> 5) * (SB_Q * 32) + (e & 31);
#pragma unroll
  for (int h = 0; h < 2; h++) {
    const int i = h * 32 + lane;
    const size_t s = s0 + i;
    if (i < n) {
      const long long loc = (long long)(unsigned)__float_as_int(crep[CREP_F1 * NS + s]) |
                            ((long long)__float_as_int(crep[CREP_F2 * NS + s]) << 32);
      float ln, l1, l2;
      if (loc & 1) {                                   // compact record (slots 1, 2): lambda0 at +1 .w, lambda2, 3 at +5 .xy
        const float4* r = col + (size_t)(loc >> 1) * 32;
        const float4 q5 = r[5 * 32];
        ln = r[32].w; l1 = q5.x; l2 = q5.y;
      } else {                                         // slot-0 record: quad +3 = {lambda n, lambda spin, lambda t1, lambda t2}
        const float4 L = hbuf[loc >> 1];
        ln = L.x; l1 = L.z; l2 = L.w;
      }
      crep[CREP_FN * NS + s] = ln / dt;
      crep[CREP_F1 * NS + s] = l1 / dt;
      crep[CREP_F2 * NS + s] = l2 / dt;
    } else {
      crep[CREP_COL_A * NS + s] = __int_as_float(-1);
      crep[CREP_COL_B * NS + s] = __int_as_float(-1);
      crep[CREP_DIST * NS + s] = 0.f;
      crep[CREP_FN * NS + s] = 0.f;
      crep[CREP_F1 * NS + s] = 0.f;
      crep[CREP_F2 * NS + s] = 0.f;
    }
  }
  // the 3-vector fields: the padding of an env is one contiguous run of each [N, 64, 3] array
  const int vf[5] = {CREP_POS_A, CREP_POS_B, CREP_NORMAL, CREP_DIR1, CREP_DIR2};
#pragma unroll
  for (int k = 0; k < 5; k++) {
    float* v = crep + vf[k] * NS + 3 * s0;
    for (int w = 3 * n + lane; w < 3 * SB_MAXCONTACT; w += 32) v[w] = 0.f;
  }
}
