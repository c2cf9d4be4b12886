// rays_emu.cpp — prb_ray_test's kernel source (prb_rays.cuh) under the CPU SIMT emulator (tests only).
#include "cuda_emu.h"

// what prb_rays.cuh uses beyond the step kernels
#define __grid_constant__
static inline int __popcll(unsigned long long x) { return __builtin_popcountll(x); }
static inline int __ffsll(long long x) { return __builtin_ffsll(x); }

#include "../../roboticsplayroompybullet_b200/csrc/prb_rays.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_convert.h"

static DevModel g_M;
static std::string g_err;

extern "C" {
int yemu_set_model(const prb_model* m) { g_err = prb_convert_model(m, &g_M); return g_err.empty() ? 0 : -1; }
const char* yemu_error() { return g_err.c_str(); }
int yemu_state_stride() { return g_M.state_stride; }
int yemu_state_dim() { return g_M.state_dim; }
int yemu_ray_max() { return RAY_MAX_RAYS; }
// prb_ray_test (prb_capi.cu) on the emulator, with the same checks and launch shape; force_large: the block-per-env
// shape whatever R is.  Returns 0, or -1 with yemu_error() for a rejected call.
int yemu_ray_test(const float* state, int N, const prb_rays* r, const float* from, const float* to, int* col, float* frac,
                  float* pos, float* nrm, int force_large) {
  RayParams P;
  g_err = ray_params(*r, from, to, col, frac, N, g_M.n_col, &P);
  if (!g_err.empty()) return -1;
  RayLaunch L = ray_launch(N, P.R);
  if (force_large && L.small) { L.small = false; L.gx = N; L.gy = 1; L.threads = 32; }
  emu_dim3 g, b; g.x = L.gx; b.x = L.threads;
  for (unsigned y = 0; y < L.gy; y++) {
    if (L.small)
      emu::launch_y(g, b, y, [&]() { prb_ray_kernel<RAY_ENVS_SMALL>(&g_M, state, P, from, to, col, frac, pos, nrm); });
    else
      emu::launch_y(g, b, y, [&]() { prb_ray_kernel<1>(&g_M, state, P, from, to, col, frac, pos, nrm); });
  }
  return 0;
}
}
