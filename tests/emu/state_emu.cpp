// state_emu.cpp — the kernel source of prb_body_states, prb_write_state and prb_restore_state (prb_state.cuh) under the
// CPU SIMT emulator (tests only).  The step harness prb_emu.cpp is compiled in too, so that the masked observe after a
// write or restore runs the split pipeline's setup kernel exactly as prb_capi.cu launches it, and so that EmuSim can
// drive this library.
#include "cuda_emu.h"

// what prb_state.cuh (and prb_render.cuh, which it includes) uses beyond the step kernels
#define __grid_constant__
static inline int __popcll(unsigned long long x) { return __builtin_popcountll(x); }
static inline int __ffsll(long long x) { return __builtin_ffsll(x); }
static inline float __fmul_rn(float a, float b) { return a * b; }
static inline float __fadd_rn(float a, float b) { return a + b; }
static inline float __fsqrt_rn(float a) { return sqrtf(a); }
static inline float __fdiv_rn(float a, float b) { return a / b; }

#include "prb_emu.cpp"
#include "../../roboticsplayroompybullet_b200/csrc/prb_state.cuh"

// the masked observe of prb_write_state / prb_restore_state (prb_capi.cu: run_step(h, 0, 1, s, mask))
static void observe_masked(float* state, DevOut* O, int N, const unsigned char* mask) {
  O->overflow = &g_overflow; O->dbg = nullptr; O->ovf_env = nullptr;
  if (g_M.nd == 12) run_step_nd<12>(state, *O, N, 0, 1, mask); else run_step_nd<9>(state, *O, N, 0, 1, mask);
}

extern "C" {
int semu_max_bodies() { return STATE_MAXK; }
// prb_body_states on the emulator, with the same checks and launch shape.  Returns 0, or -1 with emu_error().
int semu_body_states(const float* state, int N, const prb_body_query* q, float* body, float* jq, float* jqd) {
  g_err = body_query_check(*q, body, jq, jqd);
  if (!g_err.empty()) return -1;
  emu_dim3 g, b; g.x = state_blocks(N); b.x = 32 * STATE_ENVS;
  emu::launch(g, b, [&]() { prb_body_state_kernel(&g_M, state, N, q->frame, body, jq, jqd); });
  return 0;
}
// prb_write_state: the write kernel, then the masked observe of the written envs (the emulator has no contact report)
int semu_write_state(float* state, DevOut* O, int N, const prb_state_write* w, const float* jq, const float* jqd,
                     const float* body, const unsigned char* mask, unsigned char* status) {
  StateWrite P;
  g_err = state_write_params(*w, jq, jqd, body, g_M.nd, g_M.n_free, g_M.n_slide, &P);
  if (!g_err.empty()) return -1;
  std::vector<unsigned char> written(N, 0xcd);
  emu_dim3 g, b; g.x = state_blocks(N); b.x = 32 * STATE_ENVS;
  emu::launch(g, b, [&]() { prb_write_state_kernel(&g_M, state, N, P, jq, jqd, body, mask, status, written.data()); });
  observe_masked(state, O, N, written.data());
  return 0;
}
// prb_restore_state: the masked row copy, then the masked observe (mask NULL: every env, prb_observe)
void semu_restore_state(float* state, DevOut* O, int N, const float* src, const unsigned char* mask) {
  const int64_t words = (int64_t)N * g_M.state_stride;
  emu_dim3 g, b; g.x = (unsigned)((words + 255) / 256); b.x = 256;
  emu::launch(g, b, [&]() { prb_restore_state_kernel(state, src, mask, words, g_M.state_stride); });
  if (mask) observe_masked(state, O, N, mask);
  else emu_observe(state, O, N);
}
}
