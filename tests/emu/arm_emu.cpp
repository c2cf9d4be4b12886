// arm_emu.cpp — prb_arm_dynamics' kernel source (prb_arm.cuh) under the CPU SIMT emulator (tests only).
#include "cuda_emu.h"

// what prb_arm.cuh uses beyond the step kernels
#define __grid_constant__

#include "../../roboticsplayroompybullet_b200/csrc/prb_arm.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_convert.h"

static DevModel g_M;
static std::string g_err;

extern "C" {
int cemu_set_model(const prb_model* m) { g_err = prb_convert_model(m, &g_M); return g_err.empty() ? 0 : -1; }
const char* cemu_error() { return g_err.c_str(); }
int cemu_state_stride() { return g_M.state_stride; }
int cemu_state_dim() { return g_M.state_dim; }
// prb_arm_dynamics (prb_capi.cu) on the emulator, with the same checks and launch shape.  Returns 0, or -1 with
// cemu_error() for a rejected call.
int cemu_arm_dynamics(const float* state, int N, const prb_arm_query* q, const prb_arm_point* points, const float* q_in,
                      const float* qd_in, const float* qdd_in, float* jac, float* pos, float* vel, float* mm, float* tau) {
  ArmParams P;
  g_err = arm_params(*q, points, jac, pos, vel, mm, tau, N, g_M.nd, g_M.site_link, &P);
  if (!g_err.empty()) return -1;
  emu_dim3 g, b; g.x = arm_blocks(N); b.x = 32 * ARM_ENVS;
  emu::launch(g, b, [&]() { prb_arm_kernel(&g_M, state, P, q_in, qd_in, qdd_in, jac, pos, vel, mm, tau); });
  return 0;
}
}
