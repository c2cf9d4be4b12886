// closest_emu.cpp — prb_closest_points' kernel source (prb_closest.cuh) under the CPU SIMT emulator (tests only).
#include "cuda_emu.h"

// what prb_closest.cuh uses beyond the step kernels
#define __grid_constant__
#define __maxnreg__(n)
static inline int __popcll(unsigned long long x) { return __builtin_popcountll(x); }
static inline int __ffsll(long long x) { return __builtin_ffsll(x); }

#include "../../roboticsplayroompybullet_b200/csrc/prb_closest.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_convert.h"

static DevModel g_M;
static std::string g_err;

extern "C" {
int cemu_set_model(const prb_model* m) { g_err = prb_convert_model(m, &g_M); return g_err.empty() ? 0 : -1; }
const char* cemu_error() { return g_err.c_str(); }
int cemu_state_stride() { return g_M.state_stride; }
int cemu_state_dim() { return g_M.state_dim; }
// prb_closest_points (prb_capi.cu) on the emulator, with the same checks and launch shape; cull 0: every pair is tested
// exactly.  Returns 0, or -1 with cemu_error() for a rejected call.
int cemu_closest_points(const float* state, int N, const prb_closest* c, const prb_closest_query* queries, int* col_a,
                        int* col_b, float* dist, float* pos_a, float* pos_b, float* nrm, int cull) {
  ClosestParams P;
  g_err = closest_params(*c, queries, col_a, col_b, dist, N, g_M.n_col, &P);
  if (!g_err.empty()) return -1;
  emu_dim3 g, b; g.x = closest_blocks(N); b.x = 32 * CLOSEST_ENVS;
  if (cull)
    emu::launch(g, b, [&]() { prb_closest_kernel<true>(&g_M, state, P, col_a, col_b, dist, pos_a, pos_b, nrm); });
  else
    emu::launch(g, b, [&]() { prb_closest_kernel<false>(&g_M, state, P, col_a, col_b, dist, pos_a, pos_b, nrm); });
  return 0;
}
}
