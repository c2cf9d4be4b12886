// prb_capi.cu — the C-ABI shared library (include/prb.h) around the sm_100a kernels.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include <cuda_runtime.h>
#include <stdio.h>

#include <string>

#include "../../include/prb.h"
#include "prb_convert.h"
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <thread>
#include <vector>
#include "prb_reset.cuh"
#include "prb_render.cuh"
#include "prb_rays.cuh"
#include "prb_closest.cuh"
#include "prb_arm.cuh"
#include "prb_state.cuh"
#include "prb_contacts.cuh"
#include "prb_dynamics.cuh"

struct prb_handle {
  DevModel hm;
  DevModel* dm = nullptr;
  int N = 0, device = 0, sms = 148;
  unsigned env_offset = 0;
  unsigned long long seed = 0;
  float* state = nullptr;
  float* out = nullptr;
  float* action_stage = nullptr;   // device staging for prb_step_host
  // prb_step_host into pageable memory: pinned staging block, read back in chunks that worker threads copy out as they land
  float* out_stage = nullptr;
  static constexpr int OUT_CHUNKS = 8;
  cudaEvent_t ev_chunk[OUT_CHUNKS] = {};
  int host_threads = 4;
  int64_t out_floats = 0;
  DevOut O;
  int64_t launches = 0;
  int fused = 0;                   // PRB_PIPELINE=fused: A/B reference path (warp-per-env kernel, 12 substeps in one launch)
  float* sbuf = nullptr;           // record stream of the split pipeline (prb_stream.cuh)
  float4* hbuf = nullptr;          // arm-island ("heavy") class buffers
  int* heavy_cnt = nullptr;        // {bundle-list length, -, work counter, -} per class
  // high-priority side streams: the size classes of the arm-island solver overlap each other and the joint / free-body solvers
  cudaStream_t side[ARM_NCLASS] = {};
  cudaStream_t side_free = nullptr;   // the free-body islands' kernel (independent of the arm's island)
  cudaEvent_t ev_join_free = nullptr;
  int free_side = 0;                  // 1: free-body kernel on its own stream, beside the joint-row kernel
  cudaEvent_t ev_fork = nullptr, ev_join[ARM_NCLASS] = {};
  int dims[12] = {};
  int smem = 0, regs = 0;          // setup kernel (reported)
  int regs_pgs = 0;
  int smem_fused = 0;
  // reset rounds (prb_reset.cuh)
  unsigned char* pending = nullptr;
  int* reset_ctl = nullptr;
  int* n_pending = nullptr;        // device counter
  int* elist[2] = {nullptr, nullptr};   // pending envs of the previous / this reset round (compacted, unordered)
  int* n_pending_host = nullptr;   // pinned
  int reset_rounds = 0;            // rounds of the most recent prb_reset
  int timing = 0;
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t evk[64];             // per-launch events of the most recent step (timing mode)
  int n_evk = 0;
  unsigned long long* render_tests = nullptr;   // pixel-box tests of prb_render (allocated by the first render)
  float* crep = nullptr;           // contact report (prb_stream.cuh layout; allocated when first enabled)
  int contacts = 0;                // 1: prb_step / prb_substeps refresh the contact report
  float* dyn = nullptr;            // per-env dynamics table (prb_stream.cuh layout; allocated when first enabled)
  int dynamics = 0;                // 1: every setup launch reads the table instead of the model
  unsigned char* written = nullptr;   // [N] envs the last prb_write_state wrote (its clear and observe mask)
  std::string err;
};

static std::string g_err;  // errors before a handle exists

// Every entry point runs on the handle's device and leaves the caller's current device untouched
// (several handles on different GPUs may live in one process).
struct DevGuard {
  int prev = -1;
  explicit DevGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

#define CK(h, call)                                                              \
  do {                                                                           \
    cudaError_t e_ = (call);                                                     \
    if (e_ != cudaSuccess) {                                                     \
      (h)->err = std::string(#call) + ": " + cudaGetErrorString(e_);             \
      return PRB_ERR_CUDA;                                                       \
    }                                                                            \
  } while (0)

// One env step (or n raw substeps).  Split pipeline: per substep one warp-per-env setup launch
// (integrate previous solution + build rows) and the thread-per-env solver launches; a final setup
// launch integrates the last solution and writes the observation.  No host synchronisation.
// With the contact report enabled, a step of all envs (not a reset's masked settle steps) also fills the report from
// its last substep: that substep's setup launch writes the contacts, its solvers write their impulses back, and one
// prb_contact_report_kernel launch after the final setup launch writes the forces.
// With the per-env dynamics table enabled, every setup launch (masked and listed ones too, so that a reset's settle
// substeps run with the env's own masses and frictions) reads it.
template <int ND>
static int launch_step(prb_handle* h, int nsub, int observe, cudaStream_t s, const unsigned char* active = nullptr,
                       const int* elist = nullptr, int n_list = 0) {
  if (h->fused && active == nullptr) {
    dim3 gl((h->N + CfgL::WPB - 1) / CfgL::WPB), bl(32 * CfgL::WPB);
    prb_step_kernel<ND, CfgL><<<gl, bl, h->smem_fused, s>>>(h->dm, h->state, h->O, nullptr, nullptr, nullptr, nullptr, h->N, nsub, observe);
    h->launches++;
    CK(h, cudaGetLastError());
    return PRB_OK;
  }
  h->n_evk = 0;
  const int N = h->N;
  const int n = elist != nullptr ? n_list : N;                  // work items: the listed envs (later reset rounds) or all of them
  dim3 gs((n + SetupCfg::WPB - 1) / SetupCfg::WPB), bs(32 * SetupCfg::WPB);
  // persistent solver blocks: resident blocks per SM (shared-memory limited) x SMs
  const int ng = (n + PGS_BLOCK - 1) / PGS_BLOCK;
  const int pj = 6 * h->sms, pf = 3 * h->sms;
  dim3 gp(ng < pj ? ng : pj), gf(ng < pf ? ng : pf, h->hm.n_free), bp(PGS_BLOCK);
  int gcls[ARM_NCLASS], smcls[ARM_NCLASS];
  for (int k = 0; k < ARM_NCLASS; k++) {
    smcls[k] = PGS_SMEM_ARM(k);
    const int per_sm = (227 * 1024) / (smcls[k] + 1024);
    const int want = (n + arm_lanes(k) - 1) / arm_lanes(k);       // bundles if every env were in this class
    gcls[k] = (per_sm > 0 ? per_sm : 1) * h->sms;
    if (gcls[k] > want) gcls[k] = want;
  }
  const bool timed = h->timing != 0;
  const bool report = h->contacts && active == nullptr && elist == nullptr && nsub > 0;
  for (int i = 0; i <= nsub; i++) {
    const int wb = (report && i == nsub - 1) ? 1 : 0;
    int flags = (i > 0 ? SETUP_INTEGRATE : 0) | (i < nsub ? SETUP_BUILD : 0) | ((i == nsub && observe) ? SETUP_OBSERVE : 0);
    if (flags == 0) break;
    if (timed && h->n_evk < 62) CK(h, cudaEventRecord(h->evk[h->n_evk++], s));
    if (i < nsub) CK(h, cudaMemsetAsync(h->heavy_cnt, 0, 4 * ARM_NCLASS * sizeof(int), s));
    prb_setup_kernel<ND><<<gs, bs, h->smem, s>>>(h->dm, h->state, h->sbuf, h->O, N, flags, h->hbuf, h->heavy_cnt, active, elist, n_list,
                                                    wb ? h->crep : nullptr, h->dynamics ? h->dyn : nullptr);
    h->launches++;
    if (i < nsub) {
      if (timed && h->n_evk < 62) CK(h, cudaEventRecord(h->evk[h->n_evk++], s));
      // the islands of a substep are independent: the arm-island solver (few envs, long dependent
      // chains) goes first on high-priority side streams, the two light kernels fill the
      // machine behind it; the streams join before the next setup launch
      CK(h, cudaEventRecord(h->ev_fork, s));
      for (int k = ARM_NCLASS - 1; k >= 0; k--) {        // largest islands first
        CK(h, cudaStreamWaitEvent(h->side[k], h->ev_fork, 0));
        float4* hc = h->hbuf + arm_class_base(k, N);
        int* wc = h->heavy_cnt + 4 * k;
        switch (k) {                                      // envs per block = the record stride, a template constant
          case 0: prb_pgs_arm_kernel<ND, false, arm_lanes(0)><<<gcls[k], 32, smcls[k], h->side[k]>>>(h->dm, h->sbuf, hc, wc, arm_capq(k), arm_bufq(k), wb); break;
          case 1: prb_pgs_arm_kernel<ND, false, arm_lanes(1)><<<gcls[k], 32, smcls[k], h->side[k]>>>(h->dm, h->sbuf, hc, wc, arm_capq(k), arm_bufq(k), wb); break;
          case 2: prb_pgs_arm_kernel<ND, false, arm_lanes(2)><<<gcls[k], 32, smcls[k], h->side[k]>>>(h->dm, h->sbuf, hc, wc, arm_capq(k), arm_bufq(k), wb); break;
          case 3: prb_pgs_arm_kernel<ND, false, arm_lanes(3)><<<gcls[k], 32, smcls[k], h->side[k]>>>(h->dm, h->sbuf, hc, wc, arm_capq(k), arm_bufq(k), wb); break;
          default: prb_pgs_arm_kernel<ND, true, arm_lanes(4)><<<gcls[k], 32, smcls[k], h->side[k]>>>(h->dm, h->sbuf, hc, wc, arm_capq(k), arm_bufq(k), wb); break;
        }
        CK(h, cudaEventRecord(h->ev_join[k], h->side[k]));
      }
      prb_pgs_joint_kernel<ND><<<gp, bp, PGS_SMEM_J, s>>>(h->dm, h->sbuf, N, active, elist, n_list);
      if (h->hm.n_free > 0) {
        if (h->free_side) {
          CK(h, cudaStreamWaitEvent(h->side_free, h->ev_fork, 0));
          prb_pgs_free_kernel<<<gf, bp, PGS_SMEM_F, h->side_free>>>(h->dm, h->sbuf, N, active, elist, n_list, wb);
          CK(h, cudaEventRecord(h->ev_join_free, h->side_free));
          CK(h, cudaStreamWaitEvent(s, h->ev_join_free, 0));
        } else {
          prb_pgs_free_kernel<<<gf, bp, PGS_SMEM_F, s>>>(h->dm, h->sbuf, N, active, elist, n_list, wb);
        }
      }
      for (int k = 0; k < ARM_NCLASS; k++) CK(h, cudaStreamWaitEvent(s, h->ev_join[k], 0));
      h->launches += (h->hm.n_free > 0 ? 2 : 1) + ARM_NCLASS;
    }
  }
  if (timed && h->n_evk < 64) CK(h, cudaEventRecord(h->evk[h->n_evk++], s));
  if (report) {
    prb_contact_report_kernel<<<(N + CREP_WPB - 1) / CREP_WPB, 32 * CREP_WPB, 0, s>>>(h->crep, h->sbuf, h->hbuf, N, h->hm.params[P_DT],
                                                                                    CREP_REPORT, nullptr);
    h->launches++;
  }
  CK(h, cudaGetLastError());
  return PRB_OK;
}

// prb_reset / prb_reset_to / prb_set_state: the report of the envs they change becomes empty (mask NULL: all envs)
static int clear_contacts(prb_handle* h, const uint8_t* mask_dev, cudaStream_t s) {
  if (!h->contacts) return PRB_OK;
  prb_contact_report_kernel<<<(h->N + CREP_WPB - 1) / CREP_WPB, 32 * CREP_WPB, 0, s>>>(h->crep, h->sbuf, h->hbuf, h->N, h->hm.params[P_DT],
                                                                                     CREP_CLEAR, mask_dev);
  h->launches++;
  CK(h, cudaGetLastError());
  return PRB_OK;
}
static int run_step(prb_handle* h, int nsub, int observe, cudaStream_t s, const unsigned char* active = nullptr) {
  return h->hm.nd == 12 ? launch_step<12>(h, nsub, observe, s, active) : launch_step<9>(h, nsub, observe, s, active);
}

template <int ND, bool INPLACE, int LANES>
static int arm_attrs(prb_handle* h, int smax) {
  CK(h, cudaFuncSetAttribute(prb_pgs_arm_kernel<ND, INPLACE, LANES>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax));
  CK(h, cudaFuncSetAttribute(prb_pgs_arm_kernel<ND, INPLACE, LANES>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  return PRB_OK;
}

template <int ND>
static int setup_kernels(prb_handle* h) {
  h->smem = SetupCfg::WPB * (int)sizeof(SetupMemT<SetupCfg>);
  h->smem_fused = CfgL::WPB * (int)sizeof(WarpMemT<CfgL>);
  CK(h, cudaFuncSetAttribute(prb_setup_kernel<ND>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem));
  CK(h, cudaFuncSetAttribute(prb_step_kernel<ND, CfgL>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem_fused));
  CK(h, cudaFuncSetAttribute(prb_reset_finish_kernel<ND>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem));
  CK(h, cudaFuncSetAttribute(prb_reset_to_kernel<ND>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem));
  cudaFuncAttributes fa;
  CK(h, cudaFuncGetAttributes(&fa, prb_setup_kernel<ND>));
  h->regs = fa.numRegs;
  int smax = 0;
  for (int k = 0; k < ARM_NCLASS; k++) smax = PGS_SMEM_ARM(k) > smax ? PGS_SMEM_ARM(k) : smax;
  {
    int rc = arm_attrs<ND, false, arm_lanes(0)>(h, smax);
    if (rc == PRB_OK) rc = arm_attrs<ND, false, arm_lanes(1)>(h, smax);
    if (rc == PRB_OK) rc = arm_attrs<ND, false, arm_lanes(2)>(h, smax);
    if (rc == PRB_OK) rc = arm_attrs<ND, false, arm_lanes(3)>(h, smax);
    if (rc == PRB_OK) rc = arm_attrs<ND, true, arm_lanes(4)>(h, smax);
    if (rc != PRB_OK) return rc;
  }
  CK(h, cudaFuncSetAttribute(prb_pgs_joint_kernel<ND>, cudaFuncAttributeMaxDynamicSharedMemorySize, PGS_SMEM_J));
  CK(h, cudaFuncSetAttribute(prb_pgs_joint_kernel<ND>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CK(h, cudaFuncSetAttribute(prb_pgs_free_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PGS_SMEM_F));
  CK(h, cudaFuncSetAttribute(prb_pgs_free_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CK(h, cudaFuncGetAttributes(&fa, prb_pgs_arm_kernel<ND, false, arm_lanes(2)>));
  h->regs_pgs = fa.numRegs;
  return PRB_OK;
}

// Rounds of {seat objects, settle on the masked step pipeline, finish} until no env is pending (prb_reset.cuh).
// Synchronises the stream once per round (one 4-byte read), like the reference's reset, which is synchronous.
template <int ND>
static int reset_rounds(prb_handle* h, const uint8_t* mask_dev, cudaStream_t s) {
  const int N = h->N;
  const int max_rounds = RESET_MAX_ATTEMPTS * RESET_MAX_TRIES;
  dim3 gf((N + SetupCfg::WPB - 1) / SetupCfg::WPB), bf(32 * SetupCfg::WPB);
  h->reset_rounds = 0;
  const bool trace = getenv("PRB_TRACE_RESET") != nullptr;      // per-round wall time and pending count on stderr
  for (int round = 0; round < max_rounds; round++) {
    struct timespec t0, t1;
    if (trace) clock_gettime(CLOCK_MONOTONIC, &t0);
    // a masked reset compacts the masked envs into a list first (one more 4-byte read): its rounds cost what those envs cost
    const bool list0 = round == 0 && mask_dev != nullptr;
    if (list0) CK(h, cudaMemsetAsync(h->n_pending, 0, sizeof(int), s));
    prb_reset_place_kernel<<<(N + 127) / 128, 128, 0, s>>>(h->dm, h->state, h->reset_ctl, mask_dev, h->pending, N, h->seed, h->env_offset, round == 0,
                                                          list0 ? h->elist[1] : nullptr, list0 ? h->n_pending : nullptr);
    h->launches++;
    CK(h, cudaGetLastError());
    if (list0) {
      CK(h, cudaMemcpyAsync(h->n_pending_host, h->n_pending, sizeof(int), cudaMemcpyDeviceToHost, s));
      CK(h, cudaStreamSynchronize(s));
      if (*h->n_pending_host == 0) { h->reset_rounds = 0; return PRB_OK; }       // empty mask
    }
    // round 0 steps the masked batch; later rounds step the list of pending envs the previous round's finish kernel wrote
    int rc = (round == 0 && !list0) ? launch_step<ND>(h, h->hm.settle_steps, 0, s, h->pending)
                                    : launch_step<ND>(h, h->hm.settle_steps, 0, s, nullptr, h->elist[(round - 1) & 1], *h->n_pending_host);
    if (rc != PRB_OK) return rc;
    CK(h, cudaMemsetAsync(h->n_pending, 0, sizeof(int), s));
    prb_reset_finish_kernel<ND><<<gf, bf, h->smem, s>>>(h->dm, h->state, h->O, h->reset_ctl, h->pending, h->n_pending, N, h->seed, h->env_offset, h->elist[round & 1]);
    h->launches++;
    CK(h, cudaGetLastError());
    CK(h, cudaMemcpyAsync(h->n_pending_host, h->n_pending, sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(h, cudaStreamSynchronize(s));
    h->reset_rounds = round + 1;
    if (trace) {
      clock_gettime(CLOCK_MONOTONIC, &t1);
      fprintf(stderr, "[prb_reset] round %d: %.1f ms, %d envs still pending\n", round, 1e3 * (t1.tv_sec - t0.tv_sec) + 1e-6 * (t1.tv_nsec - t0.tv_nsec), *h->n_pending_host);
    }
    if (*h->n_pending_host == 0) break;
  }
  return PRB_OK;
}

extern "C" {

const char* prb_version(void) { return "prb_b200 0.1 (sm_100a)"; }

const char* prb_last_error(prb_handle* h) { return h ? h->err.c_str() : g_err.c_str(); }

int prb_create(const prb_model* model, const prb_config* cfg, prb_handle** out) {
  if (!model || !cfg || !out || cfg->num_envs <= 0) { g_err = "prb_create: bad arguments"; return PRB_ERR_INVALID; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    g_err = "prb_create: no CUDA device (this library has no CPU fallback)";
    return PRB_ERR_NO_DEVICE;
  }
  prb_handle* h = new prb_handle();
  std::string why = prb_convert_model(model, &h->hm);
  if (!why.empty()) { g_err = "prb_create: " + why; delete h; return PRB_ERR_INVALID; }
  if (h->hm.nd != 12 && h->hm.nd != 9) { g_err = "prb_create: arm must have 12 (UR5+Robotiq) or 9 (Panda) DoF"; delete h; return PRB_ERR_INVALID; }
  h->N = cfg->num_envs; h->device = cfg->device; h->env_offset = (unsigned)cfg->env_offset; h->seed = cfg->seed;
  *out = h;
  if (h->device < 0 || h->device >= ndev) { h->err = "prb_create: device ordinal out of range"; return PRB_ERR_INVALID; }
  DevGuard guard(h->device);
  CK(h, cudaDeviceGetAttribute(&h->sms, cudaDevAttrMultiProcessorCount, h->device));
  CK(h, cudaMalloc(&h->dm, sizeof(DevModel)));
  CK(h, cudaMemcpy(h->dm, &h->hm, sizeof(DevModel), cudaMemcpyHostToDevice));
  const DevModel& M = h->hm;
  const int64_t N = h->N;
  CK(h, cudaMalloc(&h->state, sizeof(float) * N * M.state_stride));
  const int dims[12] = {M.obs_dim, M.goal_dim, M.goal_dim, 4, M.fps_dim, 8, 6, M.observation_dim, 1, 1, 1, M.n_ik};
  int64_t tot = 0;
  for (int i = 0; i < 12; i++) { tot += N * dims[i]; h->dims[i] = dims[i]; }
  h->out_floats = tot;
  CK(h, cudaMalloc(&h->out, sizeof(float) * tot));
  CK(h, cudaMemset(h->out, 0, sizeof(float) * tot));
  CK(h, cudaMalloc(&h->action_stage, sizeof(float) * N * 8));   // <= 8 entries per action
  CK(h, cudaMalloc(&h->O.overflow, sizeof(unsigned long long)));
  CK(h, cudaMemset(h->O.overflow, 0, sizeof(unsigned long long)));
  CK(h, cudaMalloc(&h->O.dbg, sizeof(int) * 4 * N));
  CK(h, cudaMemset(h->O.dbg, 0, sizeof(int) * 4 * N));
  CK(h, cudaMalloc(&h->O.ovf_env, N));
  CK(h, cudaMemset(h->O.ovf_env, 0, N));
  CK(h, cudaMalloc(&h->pending, N));
  CK(h, cudaMemset(h->pending, 0, N));
  CK(h, cudaMalloc(&h->written, N));
  CK(h, cudaMemset(h->written, 0, N));
  CK(h, cudaMalloc(&h->reset_ctl, sizeof(int) * 2 * N));
  CK(h, cudaMemset(h->reset_ctl, 0, sizeof(int) * 2 * N));
  CK(h, cudaMalloc(&h->n_pending, sizeof(int)));
  for (int k = 0; k < 2; k++) CK(h, cudaMalloc(&h->elist[k], sizeof(int) * N));
  CK(h, cudaMallocHost(&h->n_pending_host, sizeof(int)));
  float** slots[12] = {&h->O.obs_quat, &h->O.achieved_goal, &h->O.desired_goal, &h->O.cag, &h->O.fps, &h->O.joints,
                       &h->O.velocity, &h->O.observation, &h->O.proprio, &h->O.reward, &h->O.success, &h->O.target_poses};
  int64_t off = 0;
  for (int i = 0; i < 12; i++) { *slots[i] = h->out + off; off += N * dims[i]; }
  {
    const char* p = getenv("PRB_PIPELINE");
    h->fused = (p && strcmp(p, "fused") == 0) ? 1 : 0;

  }
  {                                            // the split pipeline's buffers are always needed (reset runs on it)
    const size_t sb_bytes = sbuf_bytes(N);   // whole 32-env groups + prefetch slack
    CK(h, cudaMalloc(&h->sbuf, sb_bytes));
    CK(h, cudaMemset(h->sbuf, 0, sb_bytes));
    CK(h, cudaMalloc(&h->hbuf, hbuf_bytes(N)));
    CK(h, cudaMemset(h->hbuf, 0, hbuf_bytes(N)));
    CK(h, cudaMalloc(&h->heavy_cnt, 4 * ARM_NCLASS * sizeof(int)));
    int lo_pri = 0, hi_pri = 0;
    CK(h, cudaDeviceGetStreamPriorityRange(&lo_pri, &hi_pri));
    CK(h, cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    CK(h, cudaStreamCreateWithFlags(&h->side_free, cudaStreamNonBlocking));
    CK(h, cudaEventCreateWithFlags(&h->ev_join_free, cudaEventDisableTiming));
    { const char* v = getenv("PRB_FREE_SIDE"); h->free_side = v ? atoi(v) : 1; }
    for (int k = 0; k < ARM_NCLASS; k++) {
      CK(h, cudaStreamCreateWithPriority(&h->side[k], cudaStreamNonBlocking, hi_pri));
      CK(h, cudaEventCreateWithFlags(&h->ev_join[k], cudaEventDisableTiming));
    }
  }
  {
    int rc = M.nd == 12 ? setup_kernels<12>(h) : setup_kernels<9>(h);
    if (rc != PRB_OK) return rc;
  }
  prb_init_kernel<<<(h->N + 127) / 128, 128>>>(h->dm, h->state, h->N);
  h->launches++;
  CK(h, cudaGetLastError());
  CK(h, cudaDeviceSynchronize());
  return PRB_OK;
}

int prb_destroy(prb_handle* h) {
  if (!h) return PRB_ERR_INVALID;
  {
  DevGuard guard(h->device);
  cudaDeviceSynchronize();
  cudaFree(h->dm); cudaFree(h->state); cudaFree(h->out); cudaFree(h->action_stage); cudaFree(h->O.overflow); cudaFree(h->O.dbg); cudaFree(h->sbuf);
  cudaFree(h->O.ovf_env); cudaFree(h->pending); cudaFree(h->written); cudaFree(h->reset_ctl); cudaFree(h->n_pending); cudaFree(h->elist[0]); cudaFree(h->elist[1]);
  if (h->n_pending_host) cudaFreeHost(h->n_pending_host);
  if (h->out_stage) { cudaFreeHost(h->out_stage); for (int c = 0; c < prb_handle::OUT_CHUNKS; c++) cudaEventDestroy(h->ev_chunk[c]); }
  for (int k = 0; k < ARM_NCLASS; k++) {
    if (h->side[k]) cudaStreamDestroy(h->side[k]);
    if (h->ev_join[k]) cudaEventDestroy(h->ev_join[k]);
  }
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->side_free) cudaStreamDestroy(h->side_free);
  if (h->ev_join_free) cudaEventDestroy(h->ev_join_free);
  cudaFree(h->hbuf); cudaFree(h->heavy_cnt);
  if (h->render_tests) cudaFree(h->render_tests);
  if (h->crep) cudaFree(h->crep);
  if (h->dyn) cudaFree(h->dyn);
  for (int i = 0; i < 3; i++) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  if (h->ev[0]) for (int i = 0; i < 64; i++) cudaEventDestroy(h->evk[i]);
  }
  delete h;
  return PRB_OK;
}

int prb_get_buffers(prb_handle* h, prb_buffers* b) {
  if (!h || !b) return PRB_ERR_INVALID;
  const DevModel& M = h->hm;
  b->state = h->state; b->out_base = h->out;
  b->obs_quat = h->O.obs_quat; b->achieved_goal = h->O.achieved_goal; b->desired_goal = h->O.desired_goal;
  b->controllable_achieved_goal = h->O.cag; b->full_positional_state = h->O.fps; b->joints = h->O.joints;
  b->velocity = h->O.velocity; b->observation = h->O.observation; b->gripper_proprioception = h->O.proprio;
  b->reward = h->O.reward; b->is_success = h->O.success; b->target_poses = h->O.target_poses;
  b->out_floats = h->out_floats; b->num_envs = h->N; b->state_dim = M.state_dim; b->state_stride = M.state_stride;
  b->obs_dim = M.obs_dim; b->goal_dim = M.goal_dim; b->fps_dim = M.fps_dim; b->observation_dim = M.observation_dim; b->n_ik = M.n_ik;
  return PRB_OK;
}

int prb_step(prb_handle* h, const float* action_dev, void* stream) {
  if (!h || !action_dev) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if (h->timing) CK(h, cudaEventRecord(h->ev[0], s));
  prb_ik_kernel<<<(h->N + 127) / 128, 128, 0, s>>>(h->dm, h->state, action_dev, h->O.target_poses, h->N);
  h->launches++;
  CK(h, cudaGetLastError());
  if (h->timing) CK(h, cudaEventRecord(h->ev[1], s));
  int rc = run_step(h, h->hm.n_substeps, 1, s);
  if (h->timing) CK(h, cudaEventRecord(h->ev[2], s));
  return rc;
}

int prb_enable_kernel_timing(prb_handle* h, int32_t enable) {
  if (!h) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  if (enable && !h->ev[0]) {
    for (int i = 0; i < 3; i++) CK(h, cudaEventCreate(&h->ev[i]));
    for (int i = 0; i < 64; i++) CK(h, cudaEventCreate(&h->evk[i]));
  }
  h->timing = enable ? 1 : 0;
  return PRB_OK;
}

int prb_last_kernel_ms(prb_handle* h, float* ik_ms, float* step_ms) {
  if (!h || !h->ev[0]) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  CK(h, cudaEventSynchronize(h->ev[2]));
  if (ik_ms) CK(h, cudaEventElapsedTime(ik_ms, h->ev[0], h->ev[1]));
  if (step_ms) CK(h, cudaEventElapsedTime(step_ms, h->ev[1], h->ev[2]));
  return PRB_OK;
}

int prb_last_tier_ms(prb_handle* h, float* setup_ms, float* pgs_ms) {
  if (!h || !h->ev[0]) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  CK(h, cudaEventSynchronize(h->ev[2]));
  float a = 0.f, b = 0.f;
  // per-launch events alternate setup, solver, setup, solver, ..., setup, end
  for (int i = 0; i + 1 < h->n_evk; i++) {
    float ms = 0.f;
    CK(h, cudaEventElapsedTime(&ms, h->evk[i], h->evk[i + 1]));
    if (i & 1) b += ms; else a += ms;
  }
  if (setup_ms) *setup_ms = a;
  if (pgs_ms) *pgs_ms = b;
  return PRB_OK;
}

int prb_observe(prb_handle* h, void* stream) {
  if (!h) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  return run_step(h, 0, 1, (cudaStream_t)stream);
}

int prb_substeps(prb_handle* h, int32_t n, void* stream) {
  if (!h || n < 0) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  return run_step(h, n, 0, (cudaStream_t)stream);
}

int prb_reset(prb_handle* h, const uint8_t* mask_dev, void* stream) {
  if (!h) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const int rc = clear_contacts(h, mask_dev, s);
  if (rc != PRB_OK) return rc;
  return h->hm.nd == 12 ? reset_rounds<12>(h, mask_dev, s) : reset_rounds<9>(h, mask_dev, s);
}

int prb_reset_rounds(prb_handle* h) { return h ? h->reset_rounds : -1; }

int prb_reset_to(prb_handle* h, const float* obs_dev, const uint8_t* mask_dev, int32_t restore_env, void* stream) {
  if (!h || !obs_dev) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const int rc = clear_contacts(h, mask_dev, s);
  if (rc != PRB_OK) return rc;
  dim3 g((h->N + SetupCfg::WPB - 1) / SetupCfg::WPB), b(32 * SetupCfg::WPB);
  if (h->hm.nd == 12) prb_reset_to_kernel<12><<<g, b, h->smem, s>>>(h->dm, h->state, h->O, obs_dev, mask_dev, h->N, h->seed, h->env_offset, restore_env);
  else prb_reset_to_kernel<9><<<g, b, h->smem, s>>>(h->dm, h->state, h->O, obs_dev, mask_dev, h->N, h->seed, h->env_offset, restore_env);
  h->launches++;
  CK(h, cudaGetLastError());
  return PRB_OK;
}

__global__ void prb_set_goal_kernel(const DevModel* __restrict__ Mp, float* __restrict__ state, const float* __restrict__ goal,
                                    const unsigned char* __restrict__ mask, int N) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  const DevModel& M = *Mp;
  if (i >= N * M.goal_dim) return;
  int e = i / M.goal_dim, k = i % M.goal_dim;
  if (mask && !mask[e]) return;
  state[(size_t)e * M.state_stride + 5 * M.nd + 13 * M.n_free + 2 * M.n_slide + k] = goal[i];
}

int prb_set_goal(prb_handle* h, const float* goal_dev, const uint8_t* mask_dev, void* stream) {
  if (!h || !goal_dev) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  int n = h->N * h->hm.goal_dim;
  prb_set_goal_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->dm, h->state, goal_dev, mask_dev, h->N);
  h->launches++;
  CK(h, cudaGetLastError());
  return PRB_OK;
}

int prb_compute_reward(prb_handle* h, const float* ag_dev, const float* dg_dev, int64_t B, float* out_dev, void* stream) {
  if (!h || !ag_dev || !dg_dev || !out_dev || B < 0) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  if (B == 0) return PRB_OK;
  prb_reward_kernel<<<(unsigned)((B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->dm, ag_dev, dg_dev, (long long)B, out_dev);
  h->launches++;
  CK(h, cudaGetLastError());
  return PRB_OK;
}

int prb_get_state(prb_handle* h, float* host_out) {
  if (!h || !host_out) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  const DevModel& M = h->hm;
  CK(h, cudaDeviceSynchronize());
  CK(h, cudaMemcpy2D(host_out, sizeof(float) * M.state_dim, h->state, sizeof(float) * M.state_stride,
                     sizeof(float) * M.state_dim, h->N, cudaMemcpyDeviceToHost));
  return PRB_OK;
}

int prb_set_state(prb_handle* h, const float* host_in) {
  if (!h || !host_in) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  const DevModel& M = h->hm;
  CK(h, cudaDeviceSynchronize());
  CK(h, cudaMemcpy2D(h->state, sizeof(float) * M.state_stride, host_in, sizeof(float) * M.state_dim,
                     sizeof(float) * M.state_dim, h->N, cudaMemcpyHostToDevice));
  return clear_contacts(h, nullptr, nullptr);
}

int prb_step_host(prb_handle* h, const float* action_host, float* out_host, void* stream) {
  if (!h || !action_host || !out_host) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const int adim = action_dim_of((int)(h->hm.params[P_ACTION_TYPE] + 0.5f), h->hm.n_ik);
  CK(h, cudaMemcpyAsync(h->action_stage, action_host, sizeof(float) * h->N * adim, cudaMemcpyHostToDevice, s));
  int rc = prb_step(h, h->action_stage, stream);
  if (rc != PRB_OK) return rc;
  cudaPointerAttributes at;
  const bool pinned = cudaPointerGetAttributes(&at, out_host) == cudaSuccess && (at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged);
  cudaGetLastError();                                  // an unregistered pointer may leave an error behind on older drivers
  if (pinned) {
    CK(h, cudaMemcpyAsync(out_host, h->out, sizeof(float) * h->out_floats, cudaMemcpyDeviceToHost, s));
    CK(h, cudaStreamSynchronize(s));
    return PRB_OK;
  }
  // Pageable destination (a fresh numpy array per step, as the reference returns): read the block back into pinned
  // staging in chunks; worker threads copy chunk c out while chunk c + 1 is still on the bus.
  if (!h->out_stage) {
    CK(h, cudaMallocHost(&h->out_stage, sizeof(float) * h->out_floats));
    for (int c = 0; c < prb_handle::OUT_CHUNKS; c++) CK(h, cudaEventCreateWithFlags(&h->ev_chunk[c], cudaEventDisableTiming));
    const char* v = getenv("PRB_HOST_THREADS");
    int hw = (int)std::thread::hardware_concurrency();
    h->host_threads = v ? atoi(v) : (hw >= 16 ? 8 : (hw >= 8 ? 4 : (hw >= 2 ? 2 : 1)));
    if (h->host_threads < 1) h->host_threads = 1;
  }
  const int NC = prb_handle::OUT_CHUNKS;
  const int64_t per = ((h->out_floats + NC - 1) / NC + 1023) / 1024 * 1024;       // floats per chunk (4 KB multiples)
  for (int c = 0; c < NC; c++) {
    const int64_t a = c * per, b = a + per < h->out_floats ? a + per : h->out_floats;
    if (a < b) CK(h, cudaMemcpyAsync(h->out_stage + a, h->out + a, sizeof(float) * (b - a), cudaMemcpyDeviceToHost, s));
    CK(h, cudaEventRecord(h->ev_chunk[c], s));
  }
  const int T = h->host_threads < 16 ? h->host_threads : 16;
  cudaError_t werr[16] = {};
  auto worker = [&](int t) {
    if (t > 0) cudaSetDevice(h->device);
    for (int c = 0; c < NC; c++) {
      cudaError_t e = cudaEventSynchronize(h->ev_chunk[c]);
      if (e != cudaSuccess) { werr[t] = e; return; }
      const int64_t a = c * per, b = a + per < h->out_floats ? a + per : h->out_floats;
      if (a >= b) continue;
      const int64_t n = b - a, lo = a + n * t / T, hi = a + n * (t + 1) / T;
      memcpy(out_host + lo, h->out_stage + lo, sizeof(float) * (hi - lo));
    }
  };
  {
    std::vector<std::thread> th;
    for (int t = 1; t < T; t++) th.emplace_back(worker, t);
    worker(0);
    for (auto& x : th) x.join();
  }
  for (int t = 0; t < T; t++) CK(h, werr[t]);
  CK(h, cudaStreamSynchronize(s));
  return PRB_OK;
}

int prb_render(prb_handle* h, const prb_camera* cam, const float* col_rgb_host, uint8_t* rgb_dev, float* depth_dev,
               int32_t* seg_dev, void* stream) {
  if (!h) return PRB_ERR_INVALID;
  if (!cam || !col_rgb_host || !rgb_dev) { h->err = "prb_render: camera, colours and rgb_dev are required"; return PRB_ERR_INVALID; }
  RenderParams P;
  const std::string why = render_params(*cam, col_rgb_host, h->hm.n_col, &P);
  if (!why.empty()) { h->err = "prb_render: " + why; return PRB_ERR_INVALID; }
  DevGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if (!h->render_tests) {
    CK(h, cudaMalloc(&h->render_tests, sizeof(unsigned long long)));
    CK(h, cudaMemsetAsync(h->render_tests, 0, sizeof(unsigned long long), s));
  }
  // one block per env; the kernel indexes pixels in 64 bits (65 536 envs x 1024 x 1024 x 3 bytes exceeds 2^32)
  prb_render_kernel<<<h->N, 32 * RENDER_WARPS, 0, s>>>(h->dm, h->state, P, rgb_dev, depth_dev, seg_dev, h->render_tests);
  h->launches++;
  CK(h, cudaGetLastError());
  return PRB_OK;
}

int64_t prb_render_box_tests(prb_handle* h) {
  if (!h) return -1;
  if (!h->render_tests) return 0;
  DevGuard guard(h->device);
  unsigned long long v = 0;
  if (cudaDeviceSynchronize() != cudaSuccess) return -1;
  if (cudaMemcpy(&v, h->render_tests, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return (int64_t)v;
}

int prb_ray_test(prb_handle* h, const prb_rays* r, const float* from_dev, const float* to_dev, int32_t* hit_collider_dev,
                 float* hit_fraction_dev, float* hit_position_dev, float* hit_normal_dev, void* stream) {
  if (!h) return PRB_ERR_INVALID;
  if (!r) { h->err = "prb_ray_test: rays are required"; return PRB_ERR_INVALID; }
  RayParams P;
  const std::string why = ray_params(*r, from_dev, to_dev, hit_collider_dev, hit_fraction_dev, h->N, h->hm.n_col, &P);
  if (!why.empty()) { h->err = "prb_ray_test: " + why; return PRB_ERR_INVALID; }
  DevGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const RayLaunch L = ray_launch(h->N, P.R);
  if (L.small)
    prb_ray_kernel<RAY_ENVS_SMALL><<<L.gx, L.threads, 0, s>>>(h->dm, h->state, P, from_dev, to_dev, hit_collider_dev, hit_fraction_dev,
                                                              hit_position_dev, hit_normal_dev);
  else
    prb_ray_kernel<1><<<dim3(L.gx, L.gy), L.threads, 0, s>>>(h->dm, h->state, P, from_dev, to_dev, hit_collider_dev, hit_fraction_dev,
                                                             hit_position_dev, hit_normal_dev);
  h->launches++;
  CK(h, cudaGetLastError());
  return PRB_OK;
}

int prb_closest_points(prb_handle* h, const prb_closest* q, const prb_closest_query* queries_host, int32_t* collider_a_dev,
                       int32_t* collider_b_dev, float* distance_dev, float* position_on_a_dev, float* position_on_b_dev,
                       float* normal_on_b_dev, void* stream) {
  if (!h) return PRB_ERR_INVALID;
  if (!q) { h->err = "prb_closest_points: the call struct is required"; return PRB_ERR_INVALID; }
  ClosestParams P;
  const std::string why = closest_params(*q, queries_host, collider_a_dev, collider_b_dev, distance_dev, h->N, h->hm.n_col, &P);
  if (!why.empty()) { h->err = "prb_closest_points: " + why; return PRB_ERR_INVALID; }
  DevGuard guard(h->device);
  prb_closest_kernel<true><<<closest_blocks(h->N), 32 * CLOSEST_ENVS, 0, (cudaStream_t)stream>>>(
      h->dm, h->state, P, collider_a_dev, collider_b_dev, distance_dev, position_on_a_dev, position_on_b_dev, normal_on_b_dev);
  h->launches++;
  CK(h, cudaGetLastError());
  return PRB_OK;
}

int prb_arm_dynamics(prb_handle* h, const prb_arm_query* q, const prb_arm_point* points_host, const float* q_dev,
                     const float* qd_dev, const float* qdd_dev, float* jacobian_dev, float* point_position_dev,
                     float* point_velocity_dev, float* mass_matrix_dev, float* tau_dev, void* stream) {
  if (!h) return PRB_ERR_INVALID;
  if (!q) { h->err = "prb_arm_dynamics: the call struct is required"; return PRB_ERR_INVALID; }
  ArmParams P;
  const std::string why = arm_params(*q, points_host, jacobian_dev, point_position_dev, point_velocity_dev, mass_matrix_dev,
                                     tau_dev, h->N, h->hm.nd, h->hm.site_link, &P);
  if (!why.empty()) { h->err = "prb_arm_dynamics: " + why; return PRB_ERR_INVALID; }
  DevGuard guard(h->device);
  prb_arm_kernel<<<arm_blocks(h->N), 32 * ARM_ENVS, 0, (cudaStream_t)stream>>>(
      h->dm, h->state, P, q_dev, qd_dev, qdd_dev, jacobian_dev, point_position_dev, point_velocity_dev, mass_matrix_dev, tau_dev);
  h->launches++;
  CK(h, cudaGetLastError());
  return PRB_OK;
}

int prb_body_states(prb_handle* h, const prb_body_query* q, float* body_dev, float* joint_q_dev, float* joint_qd_dev,
                    void* stream) {
  if (!h) return PRB_ERR_INVALID;
  if (!q) { h->err = "prb_body_states: the call struct is required"; return PRB_ERR_INVALID; }
  const std::string why = body_query_check(*q, body_dev, joint_q_dev, joint_qd_dev);
  if (!why.empty()) { h->err = "prb_body_states: " + why; return PRB_ERR_INVALID; }
  DevGuard guard(h->device);
  prb_body_state_kernel<<<state_blocks(h->N), 32 * STATE_ENVS, 0, (cudaStream_t)stream>>>(h->dm, h->state, h->N, q->frame, body_dev,
                                                                                        joint_q_dev, joint_qd_dev);
  h->launches++;
  CK(h, cudaGetLastError());
  return PRB_OK;
}

int prb_write_state(prb_handle* h, const prb_state_write* w, const float* joint_q_dev, const float* joint_qd_dev,
                    const float* body_dev, const uint8_t* mask_dev, uint8_t* status_dev, void* stream) {
  if (!h) return PRB_ERR_INVALID;
  if (!w) { h->err = "prb_write_state: the call struct is required"; return PRB_ERR_INVALID; }
  StateWrite P;
  const std::string why = state_write_params(*w, joint_q_dev, joint_qd_dev, body_dev, h->hm.nd, h->hm.n_free, h->hm.n_slide, &P);
  if (!why.empty()) { h->err = "prb_write_state: " + why; return PRB_ERR_INVALID; }
  DevGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  prb_write_state_kernel<<<state_blocks(h->N), 32 * STATE_ENVS, 0, s>>>(h->dm, h->state, h->N, P, joint_q_dev, joint_qd_dev, body_dev,
                                                                       mask_dev, status_dev, h->written);
  h->launches++;
  CK(h, cudaGetLastError());
  const int rc = clear_contacts(h, h->written, s);
  if (rc != PRB_OK) return rc;
  return run_step(h, 0, 1, s, h->written);
}

int prb_save_state(prb_handle* h, float* dst_dev, void* stream) {
  if (!h) return PRB_ERR_INVALID;
  if (!dst_dev) { h->err = "prb_save_state: dst_dev is required"; return PRB_ERR_INVALID; }
  DevGuard guard(h->device);
  CK(h, cudaMemcpyAsync(dst_dev, h->state, sizeof(float) * (size_t)h->N * h->hm.state_stride, cudaMemcpyDeviceToDevice,
                        (cudaStream_t)stream));
  return PRB_OK;
}

int prb_restore_state(prb_handle* h, const float* src_dev, const uint8_t* mask_dev, void* stream) {
  if (!h) return PRB_ERR_INVALID;
  if (!src_dev) { h->err = "prb_restore_state: src_dev is required"; return PRB_ERR_INVALID; }
  DevGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t words = (int64_t)h->N * h->hm.state_stride;
  prb_restore_state_kernel<<<(unsigned)((words + 255) / 256), 256, 0, s>>>(h->state, src_dev, mask_dev, words, h->hm.state_stride);
  h->launches++;
  CK(h, cudaGetLastError());
  const int rc = clear_contacts(h, mask_dev, s);
  if (rc != PRB_OK) return rc;
  return run_step(h, 0, 1, s, mask_dev);
}

int prb_enable_contacts(prb_handle* h, int32_t enable) {
  if (!h) return PRB_ERR_INVALID;
  if (enable && h->fused) {
    h->err = "prb_enable_contacts: PRB_PIPELINE=fused has no record stream to report contacts from";
    return PRB_ERR_INVALID;
  }
  DevGuard guard(h->device);
  if (enable && !h->contacts) {                    // off -> on: the report starts empty
    const int64_t N = h->N;
    if (!h->crep) CK(h, cudaMalloc(&h->crep, crep_words(N) * sizeof(float)));
    CK(h, cudaDeviceSynchronize());
    CK(h, cudaMemset(h->crep, 0, crep_words(N) * sizeof(float)));
    CK(h, cudaMemset(crep_field(h->crep, N, CREP_COL_A), 0xff, 2 * N * SB_MAXCONTACT * sizeof(float)));    // collider ids -1
    CK(h, cudaDeviceSynchronize());
  }
  h->contacts = enable ? 1 : 0;
  return PRB_OK;
}

int prb_get_contacts(prb_handle* h, prb_contacts* out) {
  if (!h || !out) return PRB_ERR_INVALID;
  if (!h->crep) { h->err = "prb_get_contacts: the contact report was never enabled (prb_enable_contacts)"; return PRB_ERR_INVALID; }
  float* c = h->crep;
  const int64_t N = h->N;
  out->count = crep_count(c, N);
  out->collider_a = reinterpret_cast<int32_t*>(crep_field(c, N, CREP_COL_A));
  out->collider_b = reinterpret_cast<int32_t*>(crep_field(c, N, CREP_COL_B));
  out->position_on_a = crep_field(c, N, CREP_POS_A);
  out->position_on_b = crep_field(c, N, CREP_POS_B);
  out->normal_on_b = crep_field(c, N, CREP_NORMAL);
  out->distance = crep_field(c, N, CREP_DIST);
  out->normal_force = crep_field(c, N, CREP_FN);
  out->lateral_friction_1 = crep_field(c, N, CREP_F1);
  out->lateral_friction_2 = crep_field(c, N, CREP_F2);
  out->lateral_friction_dir_1 = crep_field(c, N, CREP_DIR1);
  out->lateral_friction_dir_2 = crep_field(c, N, CREP_DIR2);
  out->num_envs = h->N;
  out->max_contacts = SB_MAXCONTACT;
  return PRB_OK;
}

static bool range_ok(const float* r) {   // finite 0 <= lo <= hi
  return isfinite(r[0]) && isfinite(r[1]) && r[0] >= 0.f && r[0] <= r[1];
}

// draws (and, from enable, the model's values: every range (1, 1)) for the envs of mask_dev
static int draw_dynamics(prb_handle* h, const DynRanges& r, const uint8_t* mask_dev, cudaStream_t s) {
  prb_randomize_dynamics_kernel<<<(h->N + 127) / 128, 128, 0, s>>>(h->dm, h->state, h->dyn, mask_dev, h->N, h->seed, h->env_offset, r);
  h->launches++;
  CK(h, cudaGetLastError());
  return PRB_OK;
}

int prb_enable_dynamics(prb_handle* h, int32_t enable) {
  if (!h) return PRB_ERR_INVALID;
  if (enable && h->fused) {
    h->err = "prb_enable_dynamics: PRB_PIPELINE=fused reads the model's dynamics only";
    return PRB_ERR_INVALID;
  }
  DevGuard guard(h->device);
  if (enable && !h->dynamics) {                    // off -> on: every env starts from the model's values
    const DevModel& M = h->hm;
    if (!h->dyn) CK(h, cudaMalloc(&h->dyn, dyn_words(h->N, M.n_col, M.n_free) * sizeof(float)));
    CK(h, cudaDeviceSynchronize());
    const DynRanges unit = {{1.f, 1.f}, {1.f, 1.f}, {1.f, 1.f}, {1.f, 1.f}, {1.f, 1.f}};
    const int rc = draw_dynamics(h, unit, nullptr, nullptr);
    if (rc != PRB_OK) return rc;
    CK(h, cudaDeviceSynchronize());
  }
  h->dynamics = enable ? 1 : 0;
  return PRB_OK;
}

int prb_get_dynamics(prb_handle* h, prb_dynamics* out) {
  if (!h || !out) return PRB_ERR_INVALID;
  if (!h->dyn) { h->err = "prb_get_dynamics: the dynamics table was never enabled (prb_enable_dynamics)"; return PRB_ERR_INVALID; }
  const DevModel& M = h->hm;
  const int64_t N = h->N;
  out->lateral_friction = h->dyn + dyn_offset(N, M.n_col, M.n_free, DYN_FRIC);
  out->spinning_friction = h->dyn + dyn_offset(N, M.n_col, M.n_free, DYN_SPIN);
  out->mass = h->dyn + dyn_offset(N, M.n_col, M.n_free, DYN_MASS);
  out->local_inertia_diagonal = h->dyn + dyn_offset(N, M.n_col, M.n_free, DYN_INERTIA);
  out->linear_damping = h->dyn + dyn_offset(N, M.n_col, M.n_free, DYN_LD);
  out->angular_damping = h->dyn + dyn_offset(N, M.n_col, M.n_free, DYN_AD);
  out->num_envs = h->N;
  out->n_col = M.n_col;
  out->n_free = M.n_free;
  return PRB_OK;
}

int prb_randomize_dynamics(prb_handle* h, const prb_dynamics_ranges* r, const uint8_t* mask_dev, void* stream) {
  if (!h || !r) return PRB_ERR_INVALID;
  if (!h->dynamics) { h->err = "prb_randomize_dynamics: the dynamics table is not enabled (prb_enable_dynamics)"; return PRB_ERR_INVALID; }
  if (!range_ok(r->lateral_friction) || !range_ok(r->spinning_friction) || !range_ok(r->linear_damping) ||
      !range_ok(r->angular_damping) || !range_ok(r->mass) || !(r->mass[0] > 0.f)) {
    h->err = "prb_randomize_dynamics: every range needs finite 0 <= lo <= hi (mass: 0 < lo)";
    return PRB_ERR_INVALID;
  }
  DevGuard guard(h->device);
  DynRanges d;
  for (int k = 0; k < 2; k++) {
    d.lateral_friction[k] = r->lateral_friction[k]; d.spinning_friction[k] = r->spinning_friction[k]; d.mass[k] = r->mass[k];
    d.linear_damping[k] = r->linear_damping[k]; d.angular_damping[k] = r->angular_damping[k];
  }
  return draw_dynamics(h, d, mask_dev, (cudaStream_t)stream);
}

int64_t prb_launch_count(prb_handle* h) { return h ? h->launches : 0; }

int prb_debug_usage(prb_handle* h, int32_t* host_out /* [N,4] */) {
  if (!h || !host_out) return PRB_ERR_INVALID;
  DevGuard guard(h->device);
  CK(h, cudaDeviceSynchronize());
  CK(h, cudaMemcpy(host_out, h->O.dbg, sizeof(int) * 4 * h->N, cudaMemcpyDeviceToHost));
  return PRB_OK;
}

int64_t prb_overflow_count(prb_handle* h) {
  if (!h) return -1;
  DevGuard guard(h->device);
  unsigned long long v = 0;
  if (cudaDeviceSynchronize() != cudaSuccess) return -1;      // orders the read against non-blocking user streams
  if (cudaMemcpy(&v, h->O.overflow, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return (int64_t)v;
}

int prb_kernel_info(prb_handle* h, int32_t* smem_bytes_per_block, int32_t* envs_per_block, int32_t* regs_per_thread) {
  if (!h) return PRB_ERR_INVALID;
  if (smem_bytes_per_block) *smem_bytes_per_block = h->smem;
  if (envs_per_block) *envs_per_block = SetupCfg::WPB;
  if (regs_per_thread) *regs_per_thread = h->regs;
  return PRB_OK;
}

}  // extern "C"
