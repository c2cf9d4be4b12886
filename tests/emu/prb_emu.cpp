// prb_emu.cpp — runs the product's kernel source under the CPU SIMT emulator (tests only).  One translation unit with
// the kernel headers prb_capi.cu includes, the step launch sequence of its launch_step, and one emu_ entry point per
// C API call the tests exercise.
#include "cuda_emu.h"
#include "../../roboticsplayroompybullet_b200/csrc/prb_reset.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_render.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_rays.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_closest.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_arm.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_state.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_contacts.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_dynamics.cuh"
#include "../../roboticsplayroompybullet_b200/csrc/prb_convert.h"

static DevModel g_M;
static std::string g_err;

static std::vector<float> g_sbuf;
static std::vector<float4> g_hbuf;
static long long g_class_count[ARM_NCLASS] = {0};     // envs solved per arm-island class since the last query
static int g_fused = 0;     // 1: run the fused warp-per-env kernel instead of the split pipeline
static float* g_crep = nullptr;       // contact report (prb_handle::crep with contacts on); NULL: off
static const float* g_dyn = nullptr;  // per-env dynamics table (prb_handle::dyn with dynamics on); NULL: the model's
static unsigned long long g_overflow = 0;

// mirrors launch_step of prb_capi.cu: the report is filled by a step of all envs, the table goes to every setup launch
template <int ND>
static void run_step_nd(float* state, DevOut O, int N, int nsub, int observe, const unsigned char* active = nullptr,
                        const int* elist = nullptr, int n_list = 0) {
  if (g_fused && active == nullptr && elist == nullptr) {
    emu_dim3 g, b; b.x = 32 * CfgL::WPB; g.x = (N + CfgL::WPB - 1) / CfgL::WPB;
    emu::launch(g, b, [&]() { prb_step_kernel<ND, CfgL>(&g_M, state, O, nullptr, nullptr, nullptr, nullptr, N, nsub, observe); });
    return;
  }
  g_sbuf.assign(sbuf_bytes(N) / sizeof(float), 0.f);
  g_hbuf.assign(hbuf_bytes(N) / sizeof(float4), make_float4(0.f, 0.f, 0.f, 0.f));
  int heavy_cnt[4 * ARM_NCLASS] = {0};
  emu_dim3 gs, bs, gp, bp;
  const int n = elist != nullptr ? n_list : N;         // work items (prb_capi.cu launch_step)
  bs.x = 32 * SetupCfg::WPB; gs.x = (n + SetupCfg::WPB - 1) / SetupCfg::WPB;
  bp.x = PGS_BLOCK; gp.x = (n + PGS_BLOCK - 1) / PGS_BLOCK;
  const bool report = g_crep != nullptr && active == nullptr && elist == nullptr && nsub > 0;
  for (int i = 0; i <= nsub; i++) {
    const int wb = (report && i == nsub - 1) ? 1 : 0;
    int flags = (i > 0 ? SETUP_INTEGRATE : 0) | (i < nsub ? SETUP_BUILD : 0) | ((i == nsub && observe) ? SETUP_OBSERVE : 0);
    if (flags == 0) break;
    memset(heavy_cnt, 0, sizeof(heavy_cnt));
    emu::launch(gs, bs, [&]() { prb_setup_kernel<ND>(&g_M, state, g_sbuf.data(), O, N, flags, g_hbuf.data(), heavy_cnt, active, elist, n_list,
                                                     wb ? g_crep : nullptr, g_dyn); });
    if (i < nsub) {
      emu::launch(gp, bp, [&]() { prb_pgs_joint_kernel<ND>(&g_M, g_sbuf.data(), N, active, elist, n_list); });
      for (int y = 0; y < g_M.n_free; y++) {
        emu_dim3 gy = gp;
        emu::launch_y(gy, bp, y, [&]() { prb_pgs_free_kernel(&g_M, g_sbuf.data(), N, active, elist, n_list, wb); });
      }
      for (int k = 0; k < ARM_NCLASS; k++) {
        g_class_count[k] += heavy_cnt[4 * k];
        emu_dim3 gh, bq; gh.x = 2; bq.x = 32;             // two persistent blocks share the class's work counter
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
    emu::launch(g, b, [&]() { prb_contact_report_kernel(g_crep, g_sbuf.data(), g_hbuf.data(), N, g_M.params[P_DT], CREP_REPORT, nullptr); });
  }
}
static void run_step(float* state, DevOut* O, int N, int nsub, int observe, const unsigned char* active = nullptr) {
  O->overflow = &g_overflow; O->dbg = nullptr; O->ovf_env = nullptr;
  if (g_M.nd == 12) run_step_nd<12>(state, *O, N, nsub, observe, active); else run_step_nd<9>(state, *O, N, nsub, observe, active);
}

static int g_reset_rounds = 0;
// mirrors reset_rounds() of prb_capi.cu
template <int ND>
static void emu_reset_nd(float* state, DevOut o, const unsigned char* mask, int N, unsigned long long seed, unsigned env_offset) {
  std::vector<unsigned char> pending(N, 0), ovf(N, 0);
  std::vector<int> ctl(2 * N, 0), elist[2];
  elist[0].assign(N, 0); elist[1].assign(N, 0);
  int n_prev = 0;
  o.ovf_env = ovf.data();
  emu_dim3 gp, bp, gf, bf;
  bp.x = 128; gp.x = (N + 127) / 128;
  bf.x = 32 * SetupCfg::WPB; gf.x = (N + SetupCfg::WPB - 1) / SetupCfg::WPB;
  g_reset_rounds = 0;
  for (int round = 0; round < RESET_MAX_ATTEMPTS * RESET_MAX_TRIES; round++) {
    const bool list0 = round == 0 && mask != nullptr;
    int n0 = 0;
    emu::launch(gp, bp, [&]() { prb_reset_place_kernel(&g_M, state, ctl.data(), mask, pending.data(), N, seed, env_offset, round == 0,
                                                       list0 ? elist[1].data() : nullptr, list0 ? &n0 : nullptr); });
    if (list0) { n_prev = n0; if (n0 == 0) return; }
    if (round == 0 && !list0) run_step_nd<ND>(state, o, N, g_M.settle_steps, 0, pending.data());
    else run_step_nd<ND>(state, o, N, g_M.settle_steps, 0, nullptr, elist[(round - 1) & 1].data(), n_prev);
    int n_pending = 0;
    int* lout = elist[round & 1].data();
    emu::launch(gf, bf, [&]() { prb_reset_finish_kernel<ND>(&g_M, state, o, ctl.data(), pending.data(), &n_pending, N, seed, env_offset, lout); });
    g_reset_rounds = round + 1;
    n_prev = n_pending;
    if (n_pending == 0) break;
  }
}
extern "C" {
int emu_reset_rounds() { return g_reset_rounds; }
int emu_set_model(const prb_model* m) { g_err = prb_convert_model(m, &g_M); return g_err.empty() ? 0 : -1; }
const char* emu_error() { return g_err.c_str(); }
int emu_state_stride() { return g_M.state_stride; }
int emu_state_dim() { return g_M.state_dim; }
int emu_warpmem_bytes() { return (int)sizeof(SetupMemT<SetupCfg>); }
int emu_warpmem_large_bytes() { return (int)sizeof(WarpMemT<CfgL>); }
int emu_devmodel_bytes() { return (int)sizeof(DevModel); }
int emu_max_contacts() { return SB_MAXCONTACT; }
int emu_ray_max() { return RAY_MAX_RAYS; }
int emu_max_bodies() { return STATE_MAXK; }

// the step's contact report and dynamics table (NULL: off), as prb_enable_contacts / prb_enable_dynamics set them
void emu_set_report(float* crep) { g_crep = crep; }
void emu_set_dynamics(const float* dyn) { g_dyn = dyn; }
long long emu_report_words(int N) { return (long long)crep_words(N); }
long long emu_dyn_table_words(int N) { return (long long)dyn_words(N, g_M.n_col, g_M.n_free); }
long long emu_dyn_field_offset(int N, int f) { return (long long)dyn_offset(N, g_M.n_col, g_M.n_free, f); }
// clear_contacts of prb_capi.cu: with the report on, the masked envs' report becomes empty (mask NULL: every env)
void emu_clear_contacts(int N, const unsigned char* mask) {
  if (g_crep == nullptr) return;
  emu_dim3 g, b; b.x = 32 * CREP_WPB; g.x = (N + CREP_WPB - 1) / CREP_WPB;
  emu::launch(g, b, [&]() { prb_contact_report_kernel(g_crep, nullptr, nullptr, N, g_M.params[P_DT], CREP_CLEAR, mask); });
}

void emu_init(float* state, int N) {
  emu_dim3 g, b; b.x = 128; g.x = (N + 127) / 128;
  emu::launch(g, b, [&]() { prb_init_kernel(&g_M, state, N); });
}
void emu_ik(float* state, const float* action, float* target, int N) {
  emu_dim3 g, b; b.x = 128; g.x = (N + 127) / 128;
  emu::launch(g, b, [&]() { prb_ik_kernel(&g_M, state, action, target, N); });
}
void emu_set_fused(int f) { g_fused = f; }
float* emu_sbuf() { return g_sbuf.data(); }
int emu_sbuf_q() { return SB_Q; }
void emu_class_counts(long long* out, int clear) { for (int k = 0; k < ARM_NCLASS; k++) { out[k] = g_class_count[k]; if (clear) g_class_count[k] = 0; } }
int emu_arm_nclass() { return ARM_NCLASS; }
// narrow-phase candidates (before manifold reduction) left in the scratch of warp `w` of the last launched block
int emu_last_candidates(int w, int n, float* out) {
  const SetupMemT<SetupCfg>& W = ((const SetupMemT<SetupCfg>*)g_emu_smem2)[w];
  for (int i = 0; i < n; i++) {
    const Contact& c = W.cand[i];
    float* o = out + 9 * i;
    o[0] = c.pbx; o[1] = c.pby; o[2] = c.pbz; o[3] = c.nx; o[4] = c.ny; o[5] = c.nz; o[6] = c.dist; o[7] = (float)(c.cols & 0xff); o[8] = (float)((c.cols >> 8) & 0xff);
  }
  return n;
}
// contacts the setup kernel generated for the env of warp `w` of the last launched block: {pb, n, dist, ca, cb} each (tests)
int emu_last_contacts(int w, float* out) {
  const SetupMemT<SetupCfg>& W = ((const SetupMemT<SetupCfg>*)g_emu_smem2)[w];
  for (int i = 0; i < W.n_contact; i++) {
    const Contact& c = W.ct[i];
    float* o = out + 9 * i;
    o[0] = c.pbx; o[1] = c.pby; o[2] = c.pbz; o[3] = c.nx; o[4] = c.ny; o[5] = c.nz; o[6] = c.dist; o[7] = (float)(c.cols & 0xff); o[8] = (float)((c.cols >> 8) & 0xff);
  }
  return W.n_contact;
}
int emu_arm_capq(int k) { return arm_capq(k); }
unsigned long long emu_overflow() { return g_overflow; }
void emu_substeps(float* state, int N, int nsub) { DevOut O; memset(&O, 0, sizeof(O)); run_step(state, &O, N, nsub, 0); }
void emu_step(float* state, const float* action, DevOut* O, int N) {
  emu_ik(state, action, O->target_poses, N);
  run_step(state, O, N, g_M.n_substeps, 1);
}
void emu_observe(float* state, DevOut* O, int N) { run_step(state, O, N, 0, 1); }
void emu_reset(float* state, DevOut* O, const unsigned char* mask, int N, unsigned long long seed, unsigned env_offset) {
  emu_clear_contacts(N, mask);
  DevOut o = *O;
  o.overflow = &g_overflow; o.dbg = nullptr;
  if (g_M.nd == 12) emu_reset_nd<12>(state, o, mask, N, seed, env_offset);
  else emu_reset_nd<9>(state, o, mask, N, seed, env_offset);
}
void emu_reset_to(float* state, DevOut* O, const float* obs, const unsigned char* mask, int N, unsigned long long seed, unsigned env_offset, int restore_env) {
  emu_clear_contacts(N, mask);
  DevOut o = *O;
  o.overflow = &g_overflow; o.dbg = nullptr; o.ovf_env = nullptr;
  emu_dim3 g, b; b.x = 32 * SetupCfg::WPB; g.x = (N + SetupCfg::WPB - 1) / SetupCfg::WPB;
  if (g_M.nd == 12) emu::launch(g, b, [&]() { prb_reset_to_kernel<12>(&g_M, state, o, obs, mask, N, seed, env_offset, restore_env); });
  else emu::launch(g, b, [&]() { prb_reset_to_kernel<9>(&g_M, state, o, obs, mask, N, seed, env_offset, restore_env); });
}
void emu_reward(const float* ag, const float* dg, long long B, float* out) {
  emu_dim3 g, b; b.x = 128; g.x = (unsigned)((B + 127) / 128);
  emu::launch(g, b, [&]() { prb_reward_kernel(&g_M, ag, dg, B, out); });
}
int emu_box_box(const float* p1, const float* R1, const float* h1, const float* p2, const float* R2, const float* h2, float* out) {
  CPoint c[4];
  int n = box_box(ld3(p1), ldm(R1), ld3(h1), ld3(p2), ldm(R2), ld3(h2), c);
  for (int i = 0; i < n; i++) { st3(out + 7 * i, c[i].pos); st3(out + 7 * i + 3, c[i].n); out[7 * i + 6] = c[i].depth; }
  return n;
}

// r: the ten bounds of prb_dynamics_ranges in struct order
void emu_randomize_dynamics(const float* state, float* dyn, const unsigned char* mask, int N, unsigned long long seed, unsigned env_offset,
                            const float* r) {
  DynRanges d;
  memcpy(&d, r, sizeof(d));
  emu_dim3 g, b; b.x = 128; g.x = (N + 127) / 128;
  emu::launch(g, b, [&]() { prb_randomize_dynamics_kernel(&g_M, state, dyn, mask, N, seed, env_offset, d); });
}

// The batched queries below run with prb_capi.cu's checks and launch shapes; each returns 0, or -1 with emu_error() for
// a rejected call.
// prb_render: one block per env
int emu_render(const float* state, int N, const prb_camera* cam, const float* col_rgb, unsigned char* rgb, float* depth, int* seg,
               unsigned long long* tests) {
  RenderParams P;
  g_err = render_params(*cam, col_rgb, g_M.n_col, &P);
  if (!g_err.empty()) return -1;
  emu_dim3 g, b; g.x = N; b.x = 32 * RENDER_WARPS;
  emu::launch(g, b, [&]() { prb_render_kernel(&g_M, state, P, rgb, depth, seg, tests); });
  return 0;
}
// prb_ray_test; force_large: the block-per-env shape whatever R is
int emu_ray_test(const float* state, int N, const prb_rays* r, const float* from, const float* to, int* col, float* frac,
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
// prb_closest_points; cull 0: every pair is tested exactly
int emu_closest_points(const float* state, int N, const prb_closest* c, const prb_closest_query* queries, int* col_a,
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
// prb_arm_dynamics
int emu_arm_dynamics(const float* state, int N, const prb_arm_query* q, const prb_arm_point* points, const float* q_in,
                     const float* qd_in, const float* qdd_in, float* jac, float* pos, float* vel, float* mm, float* tau) {
  ArmParams P;
  g_err = arm_params(*q, points, jac, pos, vel, mm, tau, N, g_M.nd, g_M.site_link, &P);
  if (!g_err.empty()) return -1;
  emu_dim3 g, b; g.x = arm_blocks(N); b.x = 32 * ARM_ENVS;
  emu::launch(g, b, [&]() { prb_arm_kernel(&g_M, state, P, q_in, qd_in, qdd_in, jac, pos, vel, mm, tau); });
  return 0;
}
// prb_body_states
int emu_body_states(const float* state, int N, const prb_body_query* q, float* body, float* jq, float* jqd) {
  g_err = body_query_check(*q, body, jq, jqd);
  if (!g_err.empty()) return -1;
  emu_dim3 g, b; g.x = state_blocks(N); b.x = 32 * STATE_ENVS;
  emu::launch(g, b, [&]() { prb_body_state_kernel(&g_M, state, N, q->frame, body, jq, jqd); });
  return 0;
}
// prb_write_state: the write kernel, then the written envs' report cleared and their masked observe
int emu_write_state(float* state, DevOut* O, int N, const prb_state_write* w, const float* jq, const float* jqd,
                    const float* body, const unsigned char* mask, unsigned char* status) {
  StateWrite P;
  g_err = state_write_params(*w, jq, jqd, body, g_M.nd, g_M.n_free, g_M.n_slide, &P);
  if (!g_err.empty()) return -1;
  std::vector<unsigned char> written(N, 0xcd);
  emu_dim3 g, b; g.x = state_blocks(N); b.x = 32 * STATE_ENVS;
  emu::launch(g, b, [&]() { prb_write_state_kernel(&g_M, state, N, P, jq, jqd, body, mask, status, written.data()); });
  emu_clear_contacts(N, written.data());
  run_step(state, O, N, 0, 1, written.data());
  return 0;
}
// prb_restore_state: the masked row copy, then the masked envs' report cleared and their observe (mask NULL: every env)
void emu_restore_state(float* state, DevOut* O, int N, const float* src, const unsigned char* mask) {
  const int64_t words = (int64_t)N * g_M.state_stride;
  emu_dim3 g, b; g.x = (unsigned)((words + 255) / 256); b.x = 256;
  emu::launch(g, b, [&]() { prb_restore_state_kernel(state, src, mask, words, g_M.state_stride); });
  emu_clear_contacts(N, mask);
  run_step(state, O, N, 0, 1, mask);
}
}
