// render_emu.cpp — prb_render's kernel source (prb_render.cuh) under the CPU SIMT emulator (tests only).
#include "cuda_emu.h"

// what prb_render.cuh uses beyond the step kernels
#define __grid_constant__
static inline int __popcll(unsigned long long x) { return __builtin_popcountll(x); }
static inline int __ffsll(long long x) { return __builtin_ffsll(x); }

#include "../../roboticsplayroompybullet_b200/csrc/prb_render.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_convert.h"

static DevModel g_M;
static std::string g_err;

extern "C" {
int remu_set_model(const prb_model* m) { g_err = prb_convert_model(m, &g_M); return g_err.empty() ? 0 : -1; }
const char* remu_error() { return g_err.c_str(); }
int remu_state_stride() { return g_M.state_stride; }
int remu_state_dim() { return g_M.state_dim; }
// prb_render (prb_capi.cu) on the emulator: one block per env; returns 0, or -1 with remu_error() for a bad camera
int remu_render(const float* state, int N, const prb_camera* cam, const float* col_rgb, unsigned char* rgb, float* depth, int* seg,
                unsigned long long* tests) {
  RenderParams P;
  g_err = render_params(*cam, col_rgb, g_M.n_col, &P);
  if (!g_err.empty()) return -1;
  emu_dim3 g, b; g.x = N; b.x = 32 * RENDER_WARPS;
  emu::launch(g, b, [&]() { prb_render_kernel(&g_M, state, P, rgb, depth, seg, tests); });
  return 0;
}
}
