// dynamics_emu.cpp — the split step pipeline with the per-env dynamics table (prb_capi.cu launch_step: the table goes to
// every setup launch; optionally the contact report too) and prb_randomize_dynamics_kernel, under the CPU SIMT emulator
// (tests only).
#include "cuda_emu.h"
#include "../../roboticsplayroompybullet_b200/csrc/prb_contacts.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_dynamics.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_convert.h"

static DevModel g_M;
static std::string g_err;
static std::vector<float> g_sbuf;
static std::vector<float4> g_hbuf;
static unsigned long long g_overflow = 0;

// dyn NULL: the model's dynamics; crep NULL: no contact report
template <int ND>
static void run_step_nd(float* state, DevOut O, int N, int nsub, int observe, const float* dyn, float* crep) {
  g_sbuf.assign(sbuf_bytes(N) / sizeof(float), 0.f);
  g_hbuf.assign(hbuf_bytes(N) / sizeof(float4), make_float4(0.f, 0.f, 0.f, 0.f));
  int heavy_cnt[4 * ARM_NCLASS] = {0};
  emu_dim3 gs, bs, gp, bp;
  bs.x = 32 * SetupCfg::WPB; gs.x = (N + SetupCfg::WPB - 1) / SetupCfg::WPB;
  bp.x = PGS_BLOCK; gp.x = (N + PGS_BLOCK - 1) / PGS_BLOCK;
  const bool report = crep != nullptr && nsub > 0;
  for (int i = 0; i <= nsub; i++) {
    int flags = (i > 0 ? SETUP_INTEGRATE : 0) | (i < nsub ? SETUP_BUILD : 0) | ((i == nsub && observe) ? SETUP_OBSERVE : 0);
    if (flags == 0) break;
    const int wb = (report && i == nsub - 1) ? 1 : 0;
    memset(heavy_cnt, 0, sizeof(heavy_cnt));
    emu::launch(gs, bs, [&]() { prb_setup_kernel<ND>(&g_M, state, g_sbuf.data(), O, N, flags, g_hbuf.data(), heavy_cnt, nullptr, nullptr, 0,
                                                     wb ? crep : nullptr, dyn); });
    if (i < nsub) {
      emu::launch(gp, bp, [&]() { prb_pgs_joint_kernel<ND>(&g_M, g_sbuf.data(), N, nullptr); });
      for (int y = 0; y < g_M.n_free; y++) {
        emu_dim3 gy = gp;
        emu::launch_y(gy, bp, y, [&]() { prb_pgs_free_kernel(&g_M, g_sbuf.data(), N, nullptr, nullptr, 0, wb); });
      }
      for (int k = 0; k < ARM_NCLASS; k++) {
        emu_dim3 gh, bq; gh.x = 2; bq.x = 32;
        float4* hc = g_hbuf.data() + arm_class_base(k, N);
        int* wc = heavy_cnt + 4 * k;
        const int cq = arm_capq(k), bq_ = arm_bufq(k);
        switch (k) {
          case 0: emu::launch(gh, bq, [&]() { prb_pgs_arm_kernel<ND, false, arm_lanes(0)>(&g_M, g_sbuf.data(), hc, wc, cq, bq_, wb); }); break;
          case 1: emu::launch(gh, bq, [&]() { prb_pgs_arm_kernel<ND, false, arm_lanes(1)>(&g_M, g_sbuf.data(), hc, wc, cq, bq_, wb); }); break;
          case 2: emu::launch(gh, bq, [&]() { prb_pgs_arm_kernel<ND, false, arm_lanes(2)>(&g_M, g_sbuf.data(), hc, wc, cq, bq_, wb); }); break;
          case 3: emu::launch(gh, bq, [&]() { prb_pgs_arm_kernel<ND, false, arm_lanes(3)>(&g_M, g_sbuf.data(), hc, wc, cq, bq_, wb); }); break;
          default: emu::launch(gh, bq, [&]() { prb_pgs_arm_kernel<ND, true, arm_lanes(4)>(&g_M, g_sbuf.data(), hc, wc, cq, bq_, wb); }); break;
        }
      }
    }
  }
  if (report) {
    emu_dim3 g, b; b.x = 32 * CREP_WPB; g.x = (N + CREP_WPB - 1) / CREP_WPB;
    emu::launch(g, b, [&]() { prb_contact_report_kernel(crep, g_sbuf.data(), g_hbuf.data(), N, g_M.params[P_DT], CREP_REPORT, nullptr); });
  }
}
static void run_step(float* state, DevOut O, int N, int nsub, int observe, const float* dyn, float* crep) {
  if (g_M.nd == 12) run_step_nd<12>(state, O, N, nsub, observe, dyn, crep); else run_step_nd<9>(state, O, N, nsub, observe, dyn, crep);
}

extern "C" {
int demu_set_model(const prb_model* m) { g_err = prb_convert_model(m, &g_M); return g_err.empty() ? 0 : -1; }
const char* demu_error() { return g_err.c_str(); }
int demu_state_stride() { return g_M.state_stride; }
long long demu_table_words(int N) { return (long long)dyn_words(N, g_M.n_col, g_M.n_free); }
long long demu_field_offset(int N, int f) { return (long long)dyn_offset(N, g_M.n_col, g_M.n_free, f); }
long long demu_report_words(int N) { return (long long)crep_words(N); }
void demu_substeps(float* state, int N, int nsub, const float* dyn, float* crep) {
  DevOut O; memset(&O, 0, sizeof(O)); O.overflow = &g_overflow;
  run_step(state, O, N, nsub, 0, dyn, crep);
}
void demu_step(float* state, const float* action, DevOut* O, int N, const float* dyn, float* crep) {
  O->overflow = &g_overflow; O->dbg = nullptr; O->ovf_env = nullptr;
  emu_dim3 g, b; b.x = 128; g.x = (N + 127) / 128;
  emu::launch(g, b, [&]() { prb_ik_kernel(&g_M, state, action, O->target_poses, N); });
  run_step(state, *O, N, g_M.n_substeps, 1, dyn, crep);
}
// r: the ten bounds of prb_dynamics_ranges in struct order
void demu_randomize(const float* state, float* dyn, const unsigned char* mask, int N, unsigned long long seed, unsigned env_offset, const float* r) {
  DynRanges d;
  memcpy(&d, r, sizeof(d));
  emu_dim3 g, b; b.x = 128; g.x = (N + 127) / 128;
  emu::launch(g, b, [&]() { prb_randomize_dynamics_kernel(&g_M, state, dyn, mask, N, seed, env_offset, d); });
}
void demu_clear_report(float* crep, int N) {
  emu_dim3 g, b; b.x = 32 * CREP_WPB; g.x = (N + CREP_WPB - 1) / CREP_WPB;
  emu::launch(g, b, [&]() { prb_contact_report_kernel(crep, nullptr, nullptr, N, g_M.params[P_DT], CREP_CLEAR, nullptr); });
}
}
