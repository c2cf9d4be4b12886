// prb_stream.cuh — the split ("stream") step pipeline.
//
// One stepSimulation() substep = one setup launch + the constraint solve:
//   prb_setup_kernel   one WARP per env: integrate the previous substep's solution, then kinematics,
//                      collision detection, mass matrix and its inverse, unconstrained velocities and
//                      the constraint rows of this substep, written as records to HBM.  The last launch
//                      of an env step also runs the fused observation / reward write.
//   solver kernels     the 50 projected-Gauss-Seidel sweeps, in velocity space, in
//                      btMultiBodyConstraintSolver::solveSingleIteration order.  All three are ONE THREAD
//                      PER ENV: the island's velocity change lives in registers, the records are staged
//                      once into shared memory (lane-interleaved float4 columns, conflict-free) and swept
//                      there; no shuffles or barriers inside the sweeps.  The constraint islands of an env
//                      are solved by different kernels concurrently (see "Constraint islands").
//
// History (profiles/): r1 v9 re-streamed 4.5 kB of explicit Jacobian rows per env per iteration from HBM;
// r1 v27 staged the records once and gave an arm island four lanes (quad shuffles, ~125 warp instructions per
// row visit for 8 envs: 66 % of the step's kernel time for 28 % of the envs); r2 gives every island one thread
// (~80 instructions per contact visit for up to 32 envs) and hands the arm islands to the solver through
// per-size-class "heavy" buffers that are contiguous per thread block, so a block stages its envs with one
// bulk async copy (cp.async.bulk + mbarrier).
//
// Reference path: environments.py:485-490 (12 x stepSimulation), Bullet btMultiBodyDynamicsWorld.
#pragma once
#include "prb_kernels.cuh"

// ---- Constraint islands.  Rows that share no dynamic body never exchange data in Gauss-Seidel, so the
// sweep order BETWEEN islands is immaterial (bit-identical results) and islands can be solved
// concurrently.  Bodies are grouped as {arm + door/button/dial}, {free body 0}, {free body 1}; a
// contact between two groups merges them.  Each island is solved by the "slot" of its lowest group:
//   slot 0: joint rows (limits, motors, gear) + every contact of the island that contains the arm
//   slot 1, 2: contacts of a free body (block, drawer) that touches only static geometry (or the
//              other free body) — the common case; these records need no arm data at all.
// Within a slot the contacts keep Bullet's order.
//
// ---- Record stream.  Envs are grouped by 32; float4 number q of env (g, l) lives at float4 index
// g * 32 * SB_Q + q * 32 + l.  All offsets are in float4 units ("q").
#define Q_HDR 0          // ints {njr | nc0 << 8 | canon << 24 | (arm class + 1) << 25, -, -, end of region 0}
                         //      {n_contact[1] | n_spin[1] << 8 | slot of free body 0 << 16 | slot of free body 1 << 18, start[1], t_spin[1], -}
                         //      {n_contact[2] | n_spin[2] << 8, start[2], t_spin[2], -}
#define Q_VSTAR 3        // 8 q: unconstrained velocities v* of the substep (word i = DoF i)
#define Q_DV 11          // 8 q: solver output M^-1 J^T lambda (word i = DoF i)
#define Q_ST 19          // region 0 of a LIGHT env (arm island without contacts); a heavy env's region 0 is in its class buffer
// ---- region 0 (same layout in the stream and in the heavy buffers; offsets relative to its start)
#define R0_HQ 0          // ints {env, njr | nc << 8 | canon << 24, slot owners of the free bodies (as Q_HDR+1 .x), end of region}
#define R0_BODY 1        // 2 q per free body: world inverse inertia {xx xy xz yy} {yz zz 1/m -}
#define R0_MINV 5        // 12 rows x 3 q: arm inverse mass matrix (row d at R0_MINV + 3 d, zero padded)
#define R0_JROW 41       // njr x 1 q: {packed, rhs, invD, hi}
                         //   packed: pd | pd2 << 8 | a << 16 | a2 << 20 | neg << 24 | sym << 25
                         //   pd/pd2: dv word of the DoF (arm: d, slide s: DVW_SLIDE(s); pd2 = 0xff: none);
                         //   a/a2: arm row (15: not arm); neg: J = -e_d; sym: lo = -hi (else lo = 0)
                         // rows are ordered [limits][arm motors by DoF][slide motors][gear]; "canon": every arm DoF and
                         // every slide body has a motor row (always, once an action was applied) — the solvers then run
                         // the motor rows fully unrolled with compile-time register indices;
                         // then ceil(njr / 4) q of accumulated impulses (zeroed by the solver), then the contacts
#define SB_MAXJROW 40    // 2 limit rows + 1 motor per arm DoF, 3 slide motors, gear
#define SB_MAXCONTACT 64 // contacts per env after manifold reduction (two per lane in the row writer)
// slot 0 contact record, fixed layout (the solver issues every load of a visit at a fixed offset before it has
// decoded the flags, so nothing depends on a previous load):
//   +0 H0 {flags, rhs n, invD n, cfm * invD n}     +1 H1 {rhs spin, invD spin, spin coefficient, mu}
//   +2 H2 {rhs t1, rhs t2, invD t1, invD t2}        +3 L  {lambda n, lambda spin, lambda t1, lambda t2}
//   +4 G0 {n.xyz, rS.x}  +5 G1 {t1.xyz, rS.y}  +6 G2 {rF.xyz, rS.z}   (free-body side: lever arm rF; second free body: rS)
//   +7 SL {J of the slide side for the rows n, spin, t1, t2}            (B = J * slide_minv)
//   +8 ... arm side, explicit 12-wide J and B = M^-1 J^T, 6 q per row: n, t1, t2, [spin] (fixed offsets 8, 14, 20, 26)
//   flags: 1 arm side | 2 free-body side | 4 its body index | 8 its sign is -1 | 16 second free body (index 1 - first)
//          | 32 slide side | slide index << 6 | 256 spin row | size in q << 16
#define CR_ARM 1
#define CR_FREE 2
#define CR_FB 4
#define CR_FNEG 8
#define CR_TWO 16
#define CR_SLIDE 32
#define CR_SPIN 256
#define CR_BASE_Q 8
#define CR_MAX_Q 32      // 8 + 4 rows x 6 q; also the look-ahead of the solver's fixed-offset loads
// ---- slots 1, 2 (stream, from Q_S12): compact contact record (6 q, +1 q when the second side is the other free body):
//   +0 {packed, cfm * invD0, rhs0, invD0}     +1 {n.xyz, lambda0}        +2 {rP.xyz, mu}
//   +3 {t1.xyz, lambda1 (spin)}               +4 {rhs2, rhs3, invD2, invD3}   +5 {lambda2, lambda3, -, -}
//   +6 {rS.xyz, -} when side S is a free body
//   packed: kS << 2 | iP << 4 | iS << 7 | neg << 10 | spin << 11 | stride << 12
//   (kS: 0 static, 1 free; iX: free body index; neg: sign of P is -1; stride: q to the slot's next
//   record — a record never straddles the stage boundary PGS_STAGE_F)
// spin list entry (1 q): {t of the contact record, spin coefficient, rhs1, invD1}
#define CT_BASE_Q 6
#define R0_LIGHT_END (R0_JROW + SB_MAXJROW + SB_MAXJROW / 4)
#define Q_S12 (Q_ST + R0_LIGHT_END + 1)
#define SB_Q (Q_S12 + SB_MAXCONTACT * 7 + SB_MAXCONTACT + 2 * 8 + 12)
#define SB_PAD_Q 48      // readable slack after the last group (the solvers prefetch one record ahead)
// stage capacities (q of shared memory per env) of the light solver kernels
#ifndef PGS_STAGE_J
#define PGS_STAGE_J 72   // joint-row kernel: region 0 up to the impulses of <= 24 joint rows; 6 blocks per SM
#endif
#ifndef PGS_STAGE_F
#define PGS_STAGE_F 64   // free-body kernel: 10 contact records; 6 blocks per SM
#endif
#define PGS_MAXJROW_J ((PGS_STAGE_J - R0_JROW) * 4 / 5)     // njr + ceil(njr / 4) <= PGS_STAGE_J - R0_JROW
// ---- arm-island ("heavy") size classes: class k gives an env ARM_CAPQ(k) q of shared memory and a thread block
// ARM_LANES(k) envs, so that classes 0-3 keep 3-7 blocks (one warp each; 48-56 envs) resident per SM; class 4 stages the first
// ARM_CAPQ(4) q and reads the records beyond that in place.  Class 4 (the largest islands, ~0.2 % of the envs) runs ONE
// env per warp: its 50-sweep chain is the latency floor of a substep at small batch sizes, and lanes of one warp that
// take different branches of a visit (free / slide side, spin row, zero impulse change) would serialise into it.  The heavy buffer of a class is an array of bundles of
// ARM_LANES(k) envs, lane-interleaved like the stage: a block stages its bundle with ONE bulk copy.
#define ARM_NCLASS 5
#define ARM_BUFQ_MAX (R0_LIGHT_END + SB_MAXCONTACT * CR_MAX_Q + CR_MAX_Q + 4)
#ifndef ARM_CAPQ0         // (overridable: the CPU tests build a variant with tiny stages to exercise the read-in-place path)
#define ARM_CAPQ0 136
#define ARM_CAPQ1 220
#define ARM_CAPQ2 288
#define ARM_CAPQ3 440
#define ARM_CAPQ4 (R0_LIGHT_END + 32 * CR_MAX_Q + CR_MAX_Q + 4)   // 32 arm contacts staged whole; the rest is read in place
#endif

#ifndef ARM_LANES3
#define ARM_LANES3 8
#endif
#ifndef ARM_LANES4
#define ARM_LANES4 1      // measured r2p: 4 / 2 / 1 envs per warp -> 22.4 / 21.0 / 19.6 ms per env step at 8 192 envs (70.6 / 70.2 / 70.6 ms at 65 536)
#endif
#ifndef ARM_LANES12
#define ARM_LANES12 8      // measured r2u at 65 536 envs: 16 / 12 / 8 / 6 / 4 envs per warp in classes 1-2 -> 69.5 / 68.8 / 68.6 / 72.1 / 75.9 ms per env step
#endif
PRB_HD constexpr int arm_lanes(int k) { return k == 0 ? 32 : (k <= 2 ? ARM_LANES12 : (k == 3 ? ARM_LANES3 : ARM_LANES4)); }
PRB_HD int arm_capq(int k) { return k == 0 ? ARM_CAPQ0 : (k == 1 ? ARM_CAPQ1 : (k == 2 ? ARM_CAPQ2 : (k == 3 ? ARM_CAPQ3 : ARM_CAPQ4))); }
PRB_HD int arm_bufq(int k) { return k == ARM_NCLASS - 1 ? ARM_BUFQ_MAX : arm_capq(k); }
// float4 offset of class k's buffer inside the heavy allocation for N envs (every class can take all N)
PRB_HD size_t arm_class_base(int k, int64_t N) {
  size_t o = 0;
  for (int j = 0; j < k; j++) o += (size_t)((N + arm_lanes(j) - 1) / arm_lanes(j)) * arm_lanes(j) * arm_bufq(j);
  return o;
}
PRB_HD size_t hbuf_bytes(int64_t N) { return (arm_class_base(ARM_NCLASS, N) + 64) * sizeof(float4); }
// class of an arm island whose region ends at tEnd (the solver's fixed-offset loads look CR_MAX_Q - CR_BASE_Q q ahead)
PRB_HD int arm_class_of(int tEnd) {
  const int need = tEnd + CR_MAX_Q - CR_BASE_Q;
  for (int k = 0; k < ARM_NCLASS - 1; k++) if (need <= arm_capq(k)) return k;
  return ARM_NCLASS - 1;
}
#define DVW_SLIDE(s) (28 + (s))
enum { K_STATIC = 0, K_FREE = 1, K_SLIDE = 2, K_ARM = 3 };

// ---- contact report (prb_enable_contacts, include/prb.h): one allocation, field-major.  With NS = N * SB_MAXCONTACT and
// s = e * SB_MAXCONTACT + i, scalar field f of contact i of env e is word f * NS + s; a 3-vector field takes three units,
// [N, 64, 3] from word f * NS.  The int32 count [N] follows the 21 fields.  Between the setup launch that writes a
// contact's geometry and prb_contact_report_kernel (prb_contacts.cuh), the words CREP_F1 / CREP_F2 of the contact hold the
// 64-bit locator of its impulses: (float4 offset of the slot-0 record's quad +3 in the heavy allocation) << 1, or (q of the
// compact record in the env's stream column) << 1 | 1.
enum { CREP_COL_A = 0, CREP_COL_B = 1, CREP_POS_A = 2, CREP_POS_B = 5, CREP_NORMAL = 8, CREP_DIST = 11, CREP_FN = 12,
       CREP_F1 = 13, CREP_F2 = 14, CREP_DIR1 = 15, CREP_DIR2 = 18, CREP_WORDS = 21 };
PRB_HD size_t crep_words(int64_t N) { return (size_t)N * (CREP_WORDS * SB_MAXCONTACT + 1); }
PRB_HD float* crep_field(float* crep, int64_t N, int f) { return crep + (size_t)f * N * SB_MAXCONTACT; }
PRB_HD int* crep_count(float* crep, int64_t N) { return reinterpret_cast<int*>(crep_field(crep, N, CREP_WORDS)); }
PRB_D void crep_geometry(float* crep, int N, int e, int i, int ca, int cb, v3 pa, v3 pb, v3 n, float dist, v3 t1, v3 t2,
                         long long loc) {
  const size_t NS = (size_t)N * SB_MAXCONTACT, s = (size_t)e * SB_MAXCONTACT + i;
  crep[CREP_COL_A * NS + s] = __int_as_float(ca);
  crep[CREP_COL_B * NS + s] = __int_as_float(cb);
  st3(crep + CREP_POS_A * NS + 3 * s, pa);
  st3(crep + CREP_POS_B * NS + 3 * s, pb);
  st3(crep + CREP_NORMAL * NS + 3 * s, n);
  crep[CREP_DIST * NS + s] = dist;
  crep[CREP_F1 * NS + s] = __int_as_float((int)(unsigned)(loc & 0xffffffffll));
  crep[CREP_F2 * NS + s] = __int_as_float((int)(loc >> 32));
  st3(crep + CREP_DIR1 * NS + 3 * s, t1);
  st3(crep + CREP_DIR2 * NS + 3 * s, t2);
}

// ---- per-env dynamics table (prb_enable_dynamics, include/prb.h): one allocation, one dense fp32 array per field in the
// order of prb_dynamics: lateral_friction [N, n_col], spinning_friction [N, n_col], mass [N, n_free],
// local_inertia_diagonal [N, n_free, 3], linear_damping [N, n_free], angular_damping [N, n_free].
enum { DYN_FRIC = 0, DYN_SPIN, DYN_MASS, DYN_INERTIA, DYN_LD, DYN_AD };
PRB_HD size_t dyn_offset(int64_t N, int n_col, int n_free, int f) {
  const size_t c = (size_t)N * n_col, b = (size_t)N * n_free;
  return f <= DYN_SPIN ? f * c : 2 * c + (f == DYN_MASS ? 0 : (f == DYN_INERTIA ? b : (f == DYN_LD ? 4 * b : 5 * b)));
}
PRB_HD size_t dyn_words(int64_t N, int n_col, int n_free) { return dyn_offset(N, n_col, n_free, DYN_AD) + (size_t)N * n_free; }

struct SV {              // one env's column: q i at b[i * stride]
  float4* b;
  int stride;
  PRB_D float4& q(int i) const { return b[(size_t)i * stride]; }
  PRB_D float& w(int i) const { return reinterpret_cast<float*>(&b[(size_t)(i >> 2) * stride])[i & 3]; }
};
PRB_D SV sv_of(float* sbuf, int e) {
  SV s;
  s.b = reinterpret_cast<float4*>(sbuf) + (size_t)(e >> 5) * (SB_Q * 32) + (e & 31);
  s.stride = 32;
  return s;
}
// column of list slot i of class k in the heavy allocation
PRB_D SV hv_of(float4* hbuf, int k, int i, int N) {
  const int L = arm_lanes(k);
  SV s;
  s.b = hbuf + arm_class_base(k, N) + (size_t)(i / L) * ((size_t)arm_bufq(k) * L) + (i % L);
  s.stride = L;
  return s;
}
PRB_HD size_t sbuf_bytes(int64_t N) { return ((size_t)((N + 31) / 32) * 32 * SB_Q + 32 * SB_PAD_Q) * sizeof(float4); }

struct SetupCfg {
  static constexpr int MAXJROW = SB_MAXJROW;
  static constexpr int MAXCONTACT = SB_MAXCONTACT;
  static constexpr int MAXOVL = 64;       // overlapping collider pairs into the narrow phase (two per lane beyond 32)
  static constexpr int MAXCAND = 128;     // narrow-phase candidates before manifold reduction (pairs yield 0-4 points each)
#ifndef PRB_SETUP_WPB
#define PRB_SETUP_WPB 8       // measured r2c at 65536 envs: 4 warps 35.6 ms of setup per env step, 8 warps 29.9 ms, 16 warps 31.2 ms
#endif
  static constexpr int WPB = PRB_SETUP_WPB;     // warps (envs) per thread block
};
// PRB_SETUP_SYNC: the warps of a block are re-aligned with a block barrier between the phases of the setup kernel.  Its
// code (~15k SASS instructions, executed once per warp) is far larger than the instruction caches; warps drifting apart
// each stream it on their own (r2b: 3.4 stall cycles per issue waiting for instructions).  Measured r2c (15k instructions):
// no gain over simply running 8 warps per block (29.7 vs 29.9 ms).  Measured r2v (16.8k instructions after the 64-pair /
// 64-contact capacity, instruction-cache hit rate 66 %): 30.7 -> 27.8 ms of setup per env step, so ON by default.
// Level 2 adds barriers inside the dynamics phase (CRBA | M^-1 | v*).
#ifndef PRB_SETUP_SYNC
#define PRB_SETUP_SYNC 1
#endif
#if PRB_SETUP_SYNC && !defined(PRB_EMU)
#define SETUP_ALIGN() __syncthreads()
#else
#define SETUP_ALIGN() ((void)0)
#endif
#if PRB_SETUP_SYNC >= 2 && !defined(PRB_EMU)
#define SETUP_ALIGN2() __syncthreads()
#else
#define SETUP_ALIGN2() ((void)0)
#endif

// shared memory of one env in the setup kernel: state + the substep's kinematics / collision scratch.  2 blocks x 8 envs
// per SM take 120 kB of the SM's 256 kB of L1 / shared memory and leave the rest to L1 (11 784 B per env before the
// phases shared one region: 27.8 -> 23.9 ms of setup per env step, profiles/r3_setup_smem.md).
template <class CFG>
struct SetupMemT {
  typedef CFG Cfg;
  float q[PRB_MAXD], qd[PRB_MAXD], mtarget[PRB_MAXD], mkp[PRB_MAXD], mmaximp[PRB_MAXD];
  float fpos[PRB_MAXFREE][3], fquat[PRB_MAXFREE][4], fvel[PRB_MAXFREE][3], fang[PRB_MAXFREE][3];
  float sq[PRB_MAXSLIDE], sqd[PRB_MAXSLIDE];
  float goal[12], lastq[8], last_valid, reset_count;
  float lp[PRB_MAXD][3], la[PRB_MAXD][3], lc[PRB_MAXD][3], lw[PRB_MAXD][3], lv[PRB_MAXD][3];
  float fR[PRB_MAXFREE][9], fIinv[PRB_MAXFREE][6];
  float sp[PRB_MAXSLIDE][3], sR[PRB_MAXSLIDE][9];
  float Minv[PRB_MAXD][PRB_MAXD + 1];
  float vs[30];                                   // velocity DoF (nv <= 27); 30 keeps sizeof an odd multiple of 8 (below)
  float fdyn[PRB_MAXFREE * FD_N];                 // the env's free-body constants (phase_fk FD_* layout)
  const float* fric;                              // the env's collider friction row: the dynamics table's or the model's
  const float* spin;
  unsigned short ovl[CFG::MAXOVL];
  int n_ovl, n_contact, n_jrow, overflow;
  int dbg_a, dbg_c, dbg_p, dbg_u;
  float lR[PRB_MAXD][9], lIw[PRB_MAXD][6], lf[PRB_MAXD][3], ln[PRB_MAXD][3];   // phase_fk (lR: also collider frames, observe)
  // one region, reused by the phases in turn
  union {
    float2 aabb[PRB_MAXCOL][3];   // broad phase: per axis (lo, hi)
    Contact cand[CFG::MAXCAND];   // narrow phase; manifold reduction compacts the kept contacts into its head: ct
    struct {
      Contact ct[CFG::MAXCONTACT];          // narrow phase -> phase_rows_stream
      float Mm[PRB_MAXD][PRB_MAXD + 1];     // phase_crba -> phase_minv
      float Q[PRB_MAXD];                    // phase_crba -> phase_vstar
    };
  };
};
static_assert(SetupCfg::MAXCONTACT <= SetupCfg::MAXCAND, "ct is the head of cand");
// With a size that is a multiple of 16 every env's W is 16-byte aligned, ptxas merges shared loads into 128-bit ones
// (230 LDS.128 instead of 63 in prb_setup_kernel<12>) and the kernel spills at its 128 registers.
static_assert(sizeof(SetupMemT<SetupCfg>) % 16 == 8, "setup kernel shared memory per env: keep W 8-byte aligned only");

PRB_D int body_kind(const DevModel& M, int body) { return body < 0 ? K_STATIC : (body == 0 ? K_ARM : (body <= M.n_free ? K_FREE : K_SLIDE)); }
PRB_D int kind_rank(int k) { return k == K_ARM ? 3 : (k == K_SLIDE ? 2 : (k == K_FREE ? 1 : 0)); }

// One side of one constraint row: J = unit force `dir` at world point pt (or unit torque when angular)
// on the body of collider col, times sign; B = M^-1 J^T.  Returns J.B and accumulates J.v*.  When gJ is
// given, an arm side writes (accum: adds to) its explicit J and B, 3 q each at `stride`; a slide side
// returns its scalar J in *js; free-body sides store nothing (the solvers rebuild them from the
// contact geometry).
template <int ND, class WM>
PRB_D float side_row(const DevModel& M, const WM& W, int col, v3 pt, v3 dir, float sign, bool angular,
                     float4* gJ, float4* gB, int stride, bool accum, float* js, float* rel) {
  const int body = M.col_body[col];
  float d = 0.f;
  if (body == 0) {
    const int link = M.col_link[col];
    float J[12], B[12];
    const unsigned anc = M.anc_mask[link];
#pragma unroll
    for (int j = 0; j < 12; j++) {
      float g = 0.f;
      if (j < ND && ((anc >> j) & 1u)) {
        v3 aj = ld3(W.la[j]);
        if (M.jtype[j] == 0) g = angular ? dot(aj, dir) : dot(aj, cross(pt - ld3(W.lp[j]), dir));
        else g = angular ? 0.f : dot(aj, dir);
      }
      J[j] = sign * g;
    }
    float r = 0.f;
#pragma unroll
    for (int i = 0; i < 12; i++) {
      float s = 0.f;
      if (i < ND) {
#pragma unroll
        for (int j = 0; j < ND; j++) s = fmaf(W.Minv[i][j], J[j], s);
        d = fmaf(J[i], s, d); r = fmaf(J[i], W.vs[i], r);
      }
      B[i] = s;
    }
    if (gJ) {
#pragma unroll
      for (int k = 0; k < 3; k++) {
        float4 j4 = make_float4(J[4 * k], J[4 * k + 1], J[4 * k + 2], J[4 * k + 3]);
        float4 b4 = make_float4(B[4 * k], B[4 * k + 1], B[4 * k + 2], B[4 * k + 3]);
        if (accum) {                           // second arm side of an arm-arm contact
          const float4 pj = gJ[(size_t)k * stride], pb = gB[(size_t)k * stride];
          j4 = make_float4(j4.x + pj.x, j4.y + pj.y, j4.z + pj.z, j4.w + pj.w);
          b4 = make_float4(b4.x + pb.x, b4.y + pb.y, b4.z + pb.z, b4.w + pb.w);
        }
        gJ[(size_t)k * stride] = j4; gB[(size_t)k * stride] = b4;
      }
    }
    *rel += r;
  } else if (body <= M.n_free) {
    const int b = body - 1, o = M.nd + 6 * b;
    v3 t = angular ? dir : cross(pt - ld3(W.fpos[b]), dir);
    v3 jl = angular ? V3(0, 0, 0) : dir * sign, ja = t * sign;
    float im = 1.0f / W.fdyn[FD_N * b + FD_MASS];
    v3 bl = jl * im, ba = symmul(W.fIinv[b], ja);
    float J[6] = {jl.x, jl.y, jl.z, ja.x, ja.y, ja.z}, B[6] = {bl.x, bl.y, bl.z, ba.x, ba.y, ba.z};
    float r = 0.f;
#pragma unroll
    for (int k = 0; k < 6; k++) { d = fmaf(J[k], B[k], d); r = fmaf(J[k], W.vs[o + k], r); }
    *rel += r;
  } else {
    const int s = body - 1 - M.n_free, o = M.nd + 6 * M.n_free + s;
    v3 a = ld3(M.slide_axis_w[s]);
    float g;
    if (M.slide_jtype[s] == 0) g = angular ? dot(a, dir) : dot(a, cross(pt - ld3(W.sp[s]), dir));
    else g = angular ? 0.f : dot(a, dir);
    const float j = sign * g, bb = j * M.slide_minv[s];
    *js = j;
    d = j * bb; *rel += j * W.vs[o];
  }
  return d;
}

PRB_D int dvw_of(const DevModel& M, int d) {     // velocity DoF -> dv word of a joint row
  if (d < M.nd) return d;
  return DVW_SLIDE(d - M.nd - 6 * M.n_free);
}
PRB_D float4 jrow_q(const DevModel& M, int d, int d2, int neg, int sym, float rhs, float invD, float hi) {
  const int nd = M.nd;
  const int pk = dvw_of(M, d) | ((d2 < 0 ? 0xff : dvw_of(M, d2)) << 8) | ((d < nd ? d : 15) << 16) |
                 (((d2 >= 0 && d2 < nd) ? d2 : 15) << 20) | (neg << 24) | (sym << 25);
  return make_float4(__int_as_float(pk), rhs, invD, hi);
}

// the two sides of a contact ordered by kind (P = the higher-ranked side: arm > slide > free > static), their groups
// (0: arm + slide bodies, 1 + b: free body b, -1: static) and the torsional friction coefficient
struct ContactSides { int colP, colS, kP, kS, grpP, grpS; bool swapped, has_spin; float spin; };
template <class WM>
PRB_D ContactSides contact_sides(const DevModel& M, const WM& W, const Contact& c) {
  ContactSides s;
  const int ca = c.cols & 0xff, cb = (c.cols >> 8) & 0xff;
  const int kA = body_kind(M, col_dyn_body(M, ca)), kB = body_kind(M, col_dyn_body(M, cb));
  s.swapped = kind_rank(kB) > kind_rank(kA);
  s.colP = s.swapped ? cb : ca; s.colS = s.swapped ? ca : cb;
  s.kP = s.swapped ? kB : kA; s.kS = s.swapped ? kA : kB;
  s.grpP = s.kP == K_FREE ? M.col_body[s.colP] : 0;
  s.grpS = s.kS == K_STATIC ? -1 : (s.kS == K_FREE ? M.col_body[s.colS] : 0);
  s.spin = __ldg(W.spin + ca) * __ldg(W.fric + ca) + __ldg(W.spin + cb) * __ldg(W.fric + cb);
  s.has_spin = s.spin > 0.f;
  return s;
}

// constraint rows of the substep -> record stream / heavy buffers (crep: the contact report's geometry and locators too)
template <int ND, class WM>
PRB_D void phase_rows_stream(const DevModel& M, WM& W, int lane, int e, int N, const SV& S, float4* __restrict__ hbuf,
                             int* __restrict__ heavy_cnt, float* __restrict__ crep) {
  const float dt = M.params[P_DT], erp = M.params[P_ERP_JOINT], erp2 = M.params[P_ERP_CONTACT];
  const int nd = M.nd;
  // ---- joint rows, one lane per DoF: limits (lane = arm DoF), motors (lane = arm DoF; lanes 16.. = slide bodies), gear (lane 20).
  // Row order (Bullet's): [limits by DoF, lower side first][arm motors by DoF][slide motors][gear]
  float4 jr_lim[2], jr_mot = make_float4(0.f, 0.f, 0.f, 0.f);
  int n_lim = 0, n_mot = 0, n_sl = 0, n_gear = 0;
  jr_lim[0] = jr_mot; jr_lim[1] = jr_mot;
  if (lane < nd) {
    const int i = lane;
    const float invD = 1.0f / W.Minv[i][i];
    if (!(M.lo[i] > M.hi[i])) {
#pragma unroll
      for (int side = 0; side < 2; side++) {
        const float pen = side == 0 ? W.q[i] - M.lo[i] : M.hi[i] - W.q[i];
        if (pen > 0.f) continue;
        const float sg = side == 0 ? 1.0f : -1.0f;
        const float rel = sg * W.vs[i];
        const float er = pen > -0.04f ? erp : erp2;
        const float4 row = jrow_q(M, i, -1, side, 0, (-pen * er / dt - rel) * invD, invD, M.params[P_LIMIT_MAX_IMPULSE]);
        if (n_lim == 0) jr_lim[0] = row; else jr_lim[1] = row;
        n_lim++;
      }
    }
    if (W.mmaximp[i] > 0.f) {
      const float v = W.vs[i];
      const float target_v = W.mkp[i] * (W.mtarget[i] - W.q[i]) / dt + v + M.params[P_MOTOR_KD] * (0.f - v);
      jr_mot = jrow_q(M, i, -1, 0, 1, (target_v - v) * invD, invD, W.mmaximp[i]);
      n_mot = 1;
    }
  } else if (lane >= 16 && lane - 16 < M.n_slide) {
    const int s = lane - 16, o = nd + 6 * M.n_free + s;
    const float maximp = M.slide_motor[s][3] < 0 ? M.params[P_DEFAULT_MOTOR_IMPULSE] : M.slide_motor[s][3];
    if (maximp > 0.f) {
      const float invD = 1.0f / M.slide_minv[s];
      const float v = W.vs[o];
      const float target_v = M.slide_motor[s][1] * (M.slide_motor[s][0] - W.sq[s]) / dt + v + M.slide_motor[s][2] * (0.f - v);
      jr_mot = jrow_q(M, o, -1, 0, 1, (target_v - v) * invD, invD, maximp);
      n_sl = 1;
    }
  } else if (lane == 20 && M.gear_a >= 0) {
    const int a = M.gear_a, b = M.gear_b;
    const float r = M.params[P_GEAR_RATIO];
    const float D = W.Minv[a][a] + 2.f * r * W.Minv[a][b] + r * r * W.Minv[b][b];
    const float invD = 1.0f / D;
    const float rel = W.vs[a] + r * W.vs[b];
    jr_mot = jrow_q(M, a, b, 0, 1, (-rel * M.params[P_GEAR_ERP]) * invD, invD, M.params[P_GEAR_MAX_IMPULSE]);
    n_gear = 1;
  }
  int jtot;
  const int jpre = warp_excl_scan(n_lim | (n_mot << 8) | (n_sl << 16) | (n_gear << 24), lane, &jtot);
  const int nL = jtot & 0xff, nMo = (jtot >> 8) & 0xff, nSl = (jtot >> 16) & 0xff, nGe = (jtot >> 24) & 0xff;
  const int njr = nL + nMo + nSl + nGe;            // <= 2 nd + nd + n_slide + 1 <= SB_MAXJROW
  const bool canon = nMo == nd && nSl == M.n_slide;
  // ---- contacts: lane = contact, up to TWO per lane (contact h * 32 + lane; the second pass only runs for > 32 contacts)
  const int nc = W.n_contact;
  const int nh = nc > 32 ? 2 : 1;                        // warp-uniform
  int slot_[2] = {-1, -1}, size0_[2] = {0, 0}, off0_[2] = {0, 0};
  int t_[2] = {0, 0}, stride_[2] = {0, 0}, srank_[2] = {0, 0}, region_[2] = {0, 0}, tspin_[2] = {0, 0};
  // islands over the three groups {arm + slide bodies, free body 0, free body 1} -> slot of each free body and of each contact
  int slotf[PRB_MAXFREE];
  {
    bool m01 = false, m02 = false, m12 = false;
#pragma unroll
    for (int h = 0; h < 2; h++) {
      if (h < nh) {
        const int idx = h * 32 + lane;
        int lo_ = 0, hi_ = 0;
        bool two = false;
        if (idx < nc) {
          const ContactSides cs = contact_sides(M, W, W.ct[idx]);
          two = cs.grpS >= 0 && cs.grpS != cs.grpP;
          lo_ = min(cs.grpP, cs.grpS); hi_ = max(cs.grpP, cs.grpS);
        }
        m01 = m01 || __any_sync(FULL, two && lo_ == 0 && hi_ == 1);
        m02 = m02 || __any_sync(FULL, two && lo_ == 0 && hi_ == 2);
        m12 = m12 || __any_sync(FULL, two && lo_ == 1 && hi_ == 2);
      }
    }
    const bool c01 = m01 || (m12 && m02), c02 = m02 || (m12 && m01), c12 = m12 || (m01 && m02);
    slotf[0] = c01 ? 0 : 1;
    slotf[1] = c02 ? 0 : (c12 ? 1 : 2);
  }
  // ---- placement.  Slot 0: one record per contact, in contact order
  int tot0 = 0, nc0 = 0;
  int size12_[2] = {0, 0};
  bool spin_[2] = {false, false};
#pragma unroll
  for (int h = 0; h < 2; h++) {
    if (h < nh) {
      const int idx = h * 32 + lane;
      if (idx < nc) {
        const ContactSides cs = contact_sides(M, W, W.ct[idx]);
        slot_[h] = cs.grpP == 0 ? 0 : slotf[cs.grpP - 1];
        spin_[h] = cs.has_spin;
        if (slot_[h] == 0) size0_[h] = CR_BASE_Q + (cs.kP == K_ARM ? (cs.has_spin ? 24 : 18) : 0);
        else size12_[h] = CT_BASE_Q + (cs.kS == K_FREE ? 1 : 0);
      }
      int tot;
      off0_[h] = tot0 + warp_excl_scan(size0_[h], lane, &tot);
      tot0 += tot;
      nc0 += __popc(__ballot_sync(FULL, slot_[h] == 0));
    }
  }
  const int tC0 = R0_JROW + njr + ((njr + 3) >> 2);
  const int tEnd0 = tC0 + tot0;
  // slots 1, 2: compact records + spin list per region
  int ncs[3] = {nc0, 0, 0}, nss[3] = {0, 0, 0}, tsp[3] = {0, 0, 0}, start[3] = {0, 0, 0};
  {
    int region = 0;                                   // start of the slot's region relative to Q_S12
#pragma unroll
    for (int sidx = 1; sidx < 3; sidx++) {
      unsigned mask[2] = {0u, 0u}, smask[2] = {0u, 0u};
      int ts[2] = {0, 0}, total = 0;
#pragma unroll
      for (int h = 0; h < 2; h++) {
        if (h < nh) {
          const bool mine = slot_[h] == sidx;
          mask[h] = __ballot_sync(FULL, mine);
          smask[h] = __ballot_sync(FULL, mine && spin_[h]);
          int tt;
          ts[h] = total + warp_excl_scan(mine ? size12_[h] : 0, lane, &tt);
          total += tt;
        }
      }
      // a record never straddles the stage boundary of the free-body solver: the first one that would is moved up to it
      int shift = 0;
      {
        const bool st0 = slot_[0] == sidx && ts[0] < PGS_STAGE_F && ts[0] + size12_[0] > PGS_STAGE_F;
        const unsigned sm0 = __ballot_sync(FULL, st0);
        if (sm0) {
          const int sl_ = __ffs((int)sm0) - 1;
          shift = PGS_STAGE_F - __shfl_sync(FULL, ts[0], sl_);
          if (lane >= sl_) ts[0] += shift;
          ts[1] += shift;
        } else if (nh > 1) {
          const bool st1 = slot_[1] == sidx && ts[1] < PGS_STAGE_F && ts[1] + size12_[1] > PGS_STAGE_F;
          const unsigned sm1 = __ballot_sync(FULL, st1);
          if (sm1) {
            const int sl_ = __ffs((int)sm1) - 1;
            shift = PGS_STAGE_F - __shfl_sync(FULL, ts[1], sl_);
            if (lane >= sl_) ts[1] += shift;
          }
        }
      }
      const int tend = total + shift;
      const int t_first1 = __shfl_sync(FULL, ts[1], mask[1] ? __ffs((int)mask[1]) - 1 : 0);    // first record of the second pass
#pragma unroll
      for (int h = 0; h < 2; h++) {
        if (h < nh) {
          const unsigned later = mask[h] & ~((2u << lane) - 1u);        // lanes of this slot after me in my pass (lane 31: none)
          const int nl = later ? __ffs((int)later) - 1 : lane;
          const int tnext = __shfl_sync(FULL, ts[h], nl);
          if (slot_[h] == sidx) {
            t_[h] = ts[h];
            stride_[h] = later ? tnext - ts[h] : ((h == 0 && mask[1]) ? t_first1 - ts[h] : size12_[h]);
            tspin_[h] = tend; region_[h] = region;
            srank_[h] = (h ? __popc(smask[0]) : 0) + __popc(smask[h] & ((1u << lane) - 1u));
          }
        }
      }
      ncs[sidx] = __popc(mask[0]) + __popc(mask[1]); nss[sidx] = __popc(smask[0]) + __popc(smask[1]);
      tsp[sidx] = tend; start[sidx] = region;
      region += tend + nss[sidx];
    }
    if (lane == 0) { W.dbg_p = Q_S12 + region; W.dbg_a = tEnd0; }
  }
  // ---- where region 0 goes: a light env keeps it in its stream column; an arm island with contacts (or more joint
  // rows than the light kernel stages) takes the next slot of its size class's heavy buffer
  const bool heavy = nc0 > 0 || njr > PGS_MAXJROW_J;
  const int cls = arm_class_of(tEnd0);
  int hslot = 0;
  if (heavy && lane == 0) hslot = atomicAdd(heavy_cnt + 4 * cls, 1);       // heavy_cnt: {bundle-list length, -, work counter, -} per class
  hslot = __shfl_sync(FULL, hslot, 0);
  SV R;
  if (heavy) R = hv_of(hbuf, cls, hslot, N);
  else { R.b = &S.q(Q_ST); R.stride = 32; }
  const int info = ncs[1] | (nss[1] << 8) | (slotf[0] << 16) | (slotf[1] << 18);
  // ---- region 0, fixed part: header, free-body table, arm inverse mass matrix (lane = row), joint rows
  if (lane == 31) R.q(R0_HQ) = make_float4(__int_as_float(e), __int_as_float(njr | (nc0 << 8) | ((canon ? 1 : 0) << 24)), __int_as_float(info), __int_as_float(tEnd0));
  if (lane < ND) {
    float r[12];
#pragma unroll
    for (int j = 0; j < 12; j++) r[j] = j < ND ? W.Minv[lane][j] : 0.f;
#pragma unroll
    for (int k = 0; k < 3; k++) R.q(R0_MINV + 3 * lane + k) = make_float4(r[4 * k], r[4 * k + 1], r[4 * k + 2], r[4 * k + 3]);
  }
  if (lane >= 24 && lane - 24 < PRB_MAXFREE) {
    const int b = lane - 24;
    float4 i0 = make_float4(0.f, 0.f, 0.f, 0.f), i1 = i0;
    if (b < M.n_free) {
      i0 = make_float4(W.fIinv[b][0], W.fIinv[b][1], W.fIinv[b][2], W.fIinv[b][3]);
      i1 = make_float4(W.fIinv[b][4], W.fIinv[b][5], 1.0f / W.fdyn[FD_N * b + FD_MASS], 0.f);
    }
    R.q(R0_BODY + 2 * b) = i0; R.q(R0_BODY + 2 * b + 1) = i1;
    if (heavy) { S.q(Q_ST + R0_BODY + 2 * b) = i0; S.q(Q_ST + R0_BODY + 2 * b + 1) = i1; }    // the free-body kernel reads the stream
  }
  {
    const int pL = jpre & 0xff, pMo = (jpre >> 8) & 0xff, pSl = (jpre >> 16) & 0xff;
    if (n_lim > 0) R.q(R0_JROW + pL) = jr_lim[0];
    if (n_lim > 1) R.q(R0_JROW + pL + 1) = jr_lim[1];
    if (n_mot) R.q(R0_JROW + nL + pMo) = jr_mot;
    if (n_sl) R.q(R0_JROW + nL + nMo + pSl) = jr_mot;
    if (n_gear) R.q(R0_JROW + nL + nMo + nSl) = jr_mot;
  }
  if (lane == 0) W.n_jrow = njr;
  // the solver's fixed-offset loads look up to CR_MAX_Q - CR_BASE_Q q past the last record: keep that finite (zeros), so that
  // its unconditional arm-side arithmetic never meets stale NaNs of an env that used this slot before
  if (heavy && lane < CR_MAX_Q - CR_BASE_Q) R.q(tEnd0 + lane) = make_float4(0.f, 0.f, 0.f, 0.f);
  // ---- contact rows
#pragma unroll 1
  for (int h = 0; h < nh; h++) {
    const int idx = h * 32 + lane;
    if (idx >= nc) continue;
    const Contact c = W.ct[idx];
    const ContactSides cs = contact_sides(M, W, c);
    const int colP = cs.colP, colS = cs.colS, kP = cs.kP, kS = cs.kS;
    const bool swapped = cs.swapped, has_spin = cs.has_spin;
    const float spin = cs.spin;
    const bool s0 = (h ? slot_[1] : slot_[0]) == 0;
    const bool armP = s0 && kP == K_ARM;
    const int size0 = h ? size0_[1] : size0_[0], off0 = h ? off0_[1] : off0_[0];
    const int t = h ? t_[1] : t_[0], stride12 = h ? stride_[1] : stride_[0], t_spin_mine = h ? tspin_[1] : tspin_[0];
    const int spin_rank = h ? srank_[1] : srank_[0], region_mine = h ? region_[1] : region_[0];
    const int ca = c.cols & 0xff, cb = (c.cols >> 8) & 0xff;
    v3 n = V3(c.nx, c.ny, c.nz), pb = V3(c.pbx, c.pby, c.pbz), pa = pb + n * c.dist;
    const v3 pP = swapped ? pb : pa, pS = swapped ? pa : pb;
    const float sP = swapped ? -1.0f : 1.0f;
    float cfm = 0.f, er = erp2;
    float sa = M.col_stiff[ca], sb = M.col_stiff[cb];
    if (sa >= 0.f || sb >= 0.f) {       // URDF <contact> stiffness / damping on the gripper links
      float ka = sa >= 0.f ? sa : 1e18f, kb = sb >= 0.f ? sb : 1e18f;
      float da = sa >= 0.f ? M.col_damp[ca] : 0.1f, db = sb >= 0.f ? M.col_damp[cb] : 0.1f;
      float kk = 1.0f / (1.0f / ka + 1.0f / kb), dd = da + db;
      float denom = fmaxf(dt * kk + dd, 1.1920929e-7f);
      cfm = 1.0f / denom; er = dt * kk / denom;
    }
    cfm /= dt;
    const float mu = clampf(__ldg(W.fric + ca) * __ldg(W.fric + cb), -10.f, 10.f);
    v3 t1, t2;
    plane_space(n, t1, t2);
    float cfms = 0.f;
    float rhs[4] = {0.f, 0.f, 0.f, 0.f}, invDs[4] = {0.f, 0.f, 0.f, 0.f}, jsl[4] = {0.f, 0.f, 0.f, 0.f};
    float4* rec = s0 ? &R.q(tC0 + off0) : nullptr;           // slot 0 record
    const int rstride = R.stride;
    if (crep) {                     // a slot-0 contact always makes its env heavy: its record is in the heavy allocation
      const long long loc = s0 ? (long long)((rec + (size_t)3 * rstride) - hbuf) << 1 : ((long long)(Q_S12 + region_mine + t) << 1) | 1;
      crep_geometry(crep, N, e, idx, ca, cb, pa, pb, n, c.dist, t1, t2, loc);
    }
#pragma unroll 1
    for (int k = 0; k < 4; k++) {
      v3 dir = k == 0 ? n : (k == 1 ? n : (k == 2 ? t1 : t2));
      const bool ang = (k == 1);
      if (k == 1 && !has_spin) continue;      // no torsional row: never visited by the solver
      const int ridx = k == 0 ? 0 : (k == 1 ? 3 : k - 1);     // arm rows in memory: n, t1, t2, spin
      float4* rowJ = armP ? rec + (size_t)(CR_BASE_Q + 6 * ridx) * rstride : nullptr;
      float4* rowB = armP ? rowJ + (size_t)3 * rstride : nullptr;
      float js = 0.f;
      float rel = 0.f, D = 0.f;
      D += side_row<ND>(M, W, colP, pP, dir, sP, ang, rowJ, rowB, rstride, false, &js, &rel);
      if (kS != K_STATIC) D += side_row<ND>(M, W, colS, pS, dir, -sP, ang, rowJ, rowB, rstride, true, &js, &rel);
      if (k == 0) D += cfm;
      const float invD = D > 1.1920929e-7f ? 1.0f / D : 0.f;
      if (k == 0) {
        float pen = c.dist + M.params[P_LINEAR_SLOP];
        float poserr = 0.f, velerr = -rel;
        if (pen > 0.f) velerr -= pen / dt; else poserr = -pen * er / dt;
        rhs[0] = (poserr + velerr) * invD;
        cfms = cfm * invD;
      } else rhs[k] = -rel * invD;
      invDs[k] = invD; jsl[k] = js;
    }
    if (s0) {
      // sides by kind: arm (P), slide (P or S), free (P, or S under an arm / slide P; both when P and S are free bodies)
      const bool slideP = kP == K_SLIDE, slideS = kS == K_SLIDE, freeP = kP == K_FREE, freeS = kS == K_FREE;
      if (slideP && slideS) W.overflow |= 4;                       // two slide bodies in one contact: not representable
      const int sld = slideP ? M.col_body[colP] - 1 - M.n_free : (slideS ? M.col_body[colS] - 1 - M.n_free : 0);
      const int fb = freeP ? M.col_body[colP] - 1 : (freeS ? M.col_body[colS] - 1 : 0);
      const float sgnF = freeP ? sP : -sP;
      const bool two = freeP && freeS;
      const int flags = (armP ? CR_ARM : 0) | ((freeP || freeS) ? CR_FREE : 0) | (fb ? CR_FB : 0) | (sgnF < 0.f ? CR_FNEG : 0) |
                        (two ? CR_TWO : 0) | ((slideP || slideS) ? (CR_SLIDE | (sld << 6)) : 0) | (has_spin ? CR_SPIN : 0) | (size0 << 16);
      v3 rF = V3(0, 0, 0), rS2 = V3(0, 0, 0);
      if (freeP) rF = pP - ld3(W.fpos[fb]); else if (freeS) rF = pS - ld3(W.fpos[fb]);
      if (two) rS2 = pS - ld3(W.fpos[M.col_body[colS] - 1]);
      rec[0] = make_float4(__int_as_float(flags), rhs[0], invDs[0], cfms);
      rec[(size_t)1 * rstride] = make_float4(rhs[1], invDs[1], spin, mu);
      rec[(size_t)2 * rstride] = make_float4(rhs[2], rhs[3], invDs[2], invDs[3]);
      rec[(size_t)3 * rstride] = make_float4(0.f, 0.f, 0.f, 0.f);
      rec[(size_t)4 * rstride] = make_float4(n.x, n.y, n.z, rS2.x);
      rec[(size_t)5 * rstride] = make_float4(t1.x, t1.y, t1.z, rS2.y);
      rec[(size_t)6 * rstride] = make_float4(rF.x, rF.y, rF.z, rS2.z);
      rec[(size_t)7 * rstride] = make_float4(jsl[0], jsl[1], jsl[2], jsl[3]);
    } else {                                   // slots 1, 2: compact record (both sides are free bodies or static)
      const int iP = M.col_body[colP] - 1, iS = kS == K_FREE ? M.col_body[colS] - 1 : 0;
      const v3 rP = pP - ld3(W.fpos[iP]);
      const int packed = (kS << 2) | (iP << 4) | (iS << 7) | ((swapped ? 1 : 0) << 10) | ((has_spin ? 1 : 0) << 11) | (stride12 << 12);
      float4* r12 = &S.q(Q_S12 + region_mine + t);
      r12[0] = make_float4(__int_as_float(packed), cfms, rhs[0], invDs[0]);
      r12[32] = make_float4(n.x, n.y, n.z, 0.f);
      r12[64] = make_float4(rP.x, rP.y, rP.z, mu);
      r12[96] = make_float4(t1.x, t1.y, t1.z, 0.f);
      r12[128] = make_float4(rhs[2], rhs[3], invDs[2], invDs[3]);
      r12[160] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (kS == K_FREE) { const v3 rS = pS - ld3(W.fpos[iS]); r12[192] = make_float4(rS.x, rS.y, rS.z, 0.f); }
      if (has_spin) S.q(Q_S12 + region_mine + t_spin_mine + spin_rank) = make_float4(__int_as_float(t), spin, rhs[1], invDs[1]);
    }
  }
  __syncwarp();
  if (lane == 0) {
    S.q(Q_HDR) = make_float4(__int_as_float(njr | (nc0 << 8) | ((canon ? 1 : 0) << 24) | ((heavy ? cls + 1 : 0) << 25)), 0.f, 0.f, __int_as_float(tEnd0));
    S.q(Q_HDR + 1) = make_float4(__int_as_float(info), __int_as_float(start[1]), __int_as_float(tsp[1]), 0.f);
    S.q(Q_HDR + 2) = make_float4(__int_as_float(ncs[2] | (nss[2] << 8)), __int_as_float(start[2]), __int_as_float(tsp[2]), 0.f);
    if (nc > W.dbg_c) W.dbg_c = nc;
    W.dbg_u = heavy ? cls + 1 : 0;
  }
  if (lane < M.nv) S.w(4 * Q_VSTAR + lane) = W.vs[lane];
}

// ============================================================================ setup kernel (warp per env)
enum { SETUP_INTEGRATE = 1, SETUP_BUILD = 2, SETUP_OBSERVE = 4 };

#ifdef PRB_EMU
static char g_emu_smem2[8 * sizeof(SetupMemT<SetupCfg>) + 256];
#define PRB_SMEM_DECL2 WM* wm = (WM*)g_emu_smem2
#else
#define PRB_SMEM_DECL2 extern __shared__ __align__(16) unsigned char prb_dyn_smem2[]; WM* wm = (WM*)prb_dyn_smem2
#endif

// Env of work item i.  Normally the identity over [0, N), optionally masked (`active`); the later rounds of a reset
// pass a compacted list of the envs still pending (`elist`, n_list entries) so that their cost follows the count.
PRB_D int env_of(int i, int N, const unsigned char* active, const int* elist, int n_list, bool* on) {
  if (elist != nullptr) { *on = i < n_list; return *on ? elist[i] : 0; }
  *on = i < N && (active == nullptr || active[i] != 0);
  return i;
}

// The env's dynamics constants for this launch: its row of the per-env table (dyn, prb_enable_dynamics), else the model's.
// Free-body constants are copied into W.fdyn; the friction rows are read in place through W.fric / W.spin (L1-resident,
// a few reads per contact).
template <class WM>
PRB_D void stage_dynamics(const DevModel& M, WM& W, int lane, int e, int N, const float* __restrict__ dyn) {
  const int nc = M.n_col, nf = M.n_free;
  if (lane < FD_N * nf) {
    const int b = lane / FD_N, k = lane - FD_N * b;
    float v;
    if (dyn) {
      const size_t f = dyn_offset(N, nc, nf, k == FD_MASS ? DYN_MASS : (k < FD_LD ? DYN_INERTIA : (k == FD_LD ? DYN_LD : DYN_AD)));
      v = dyn[f + (k < FD_LD && k != FD_MASS ? (size_t)3 * (e * nf + b) + (k - FD_INERTIA) : (size_t)e * nf + b)];
    } else {
      v = k == FD_MASS ? M.free_mass[b] : (k < FD_LD ? M.free_inertia[b][k - FD_INERTIA] : (k == FD_LD ? M.free_ld[b] : M.free_ad[b]));
    }
    W.fdyn[lane] = v;
  }
  if (lane == 0) {
    W.fric = dyn ? dyn + dyn_offset(N, nc, nf, DYN_FRIC) + (size_t)e * nc : M.col_fric;
    W.spin = dyn ? dyn + dyn_offset(N, nc, nf, DYN_SPIN) + (size_t)e * nc : M.col_spin;
  }
}

#ifndef PRB_SETUP_MINB
#define PRB_SETUP_MINB 2       // 2 x 8 warps per SM = 128 registers per thread; measured r2l: 1 block (natural register count) 43.9 ms of setup per env step, 2 x 10 warps at 96 registers (spills) 40.2 ms, this 31.8 ms
#endif
template <int ND>
__global__ void __launch_bounds__(32 * SetupCfg::WPB, PRB_SETUP_MINB) prb_setup_kernel(const DevModel* __restrict__ Mp, float* __restrict__ state,
                                                                         float* __restrict__ sbuf, DevOut O, int N, int flags,
                                                                         float4* __restrict__ hbuf, int* __restrict__ heavy_cnt,
                                                                         const unsigned char* __restrict__ active,
                                                                         const int* __restrict__ elist = nullptr, int n_list = 0,
                                                                         float* __restrict__ crep = nullptr,
                                                                         const float* __restrict__ dyn = nullptr) {
  typedef SetupMemT<SetupCfg> WM;
  PRB_SMEM_DECL2;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  // masked / listed stepping (reset: only the envs being reset settle); an idle warp still takes part in the block barriers
  bool on;
  const int e = env_of(blockIdx.x * SetupCfg::WPB + wib, N, active, elist, n_list, &on);
#if !PRB_SETUP_SYNC
  if (!on) return;
#endif
  const DevModel& M = *Mp;
  WM& W = wm[wib];
  float* st = state + (size_t)(on ? e : 0) * M.state_stride;
  const SV S = sv_of(sbuf, on ? e : 0);
  if (on) {
    load_state(M, W, st, lane);
    if (lane == 0) { W.overflow = 0; W.dbg_a = 0; W.dbg_c = 0; W.dbg_p = 0; W.dbg_u = 0; }
    stage_dynamics(M, W, lane, e, N, dyn);
    __syncwarp();
    if (flags & SETUP_INTEGRATE) {
      float vstar = 0.f, dv = 0.f;
      if (lane < M.nv) { vstar = S.w(4 * Q_VSTAR + lane); dv = S.w(4 * Q_DV + lane); }
      phase_integrate(M, W, lane, vstar, dv);
    }
  }
  if (flags & SETUP_BUILD) {
    SETUP_ALIGN();
    if (on) phase_fk(M, W, lane, true, W.fdyn);
    SETUP_ALIGN();
    if (on) phase_collide_broad(M, W, lane);
    SETUP_ALIGN();
    if (on) phase_collide_narrow(M, W, lane);
    SETUP_ALIGN();
    if (on) phase_crba(M, W, lane);
    SETUP_ALIGN2();
    if (on) phase_minv<ND>(W, lane);
    SETUP_ALIGN2();
    if (on) phase_vstar(M, W, lane, W.fdyn);
    SETUP_ALIGN();
    if (on) {
      phase_rows_stream<ND>(M, W, lane, e, N, S, hbuf, heavy_cnt, crep);
      __syncwarp();
      if (crep && lane == 0) crep_count(crep, N)[e] = W.n_contact;
      // a dropped contact marks the env; the mark is counted (once per env step) by the launch that observes
      if (lane == 0 && W.overflow) { if (O.ovf_env) O.ovf_env[e] = 1; else if (O.overflow) atomicAdd(O.overflow, 1ull); }
      if (lane == 0 && O.dbg) { O.dbg[4 * e] = W.dbg_u | (W.dbg_a << 8); O.dbg[4 * e + 1] = W.dbg_c; O.dbg[4 * e + 2] = W.dbg_p; O.dbg[4 * e + 3] = W.n_jrow | (W.overflow << 8); }
    }
  }
  if (!on) return;
  if (flags & SETUP_OBSERVE) {
    phase_observe(M, W, lane, O, (size_t)e, true);
    if (lane == 0 && O.ovf_env && O.ovf_env[e]) { O.ovf_env[e] = 0; if (O.overflow) atomicAdd(O.overflow, 1ull); }
  }
  __syncwarp();
  if (flags & (SETUP_INTEGRATE | SETUP_OBSERVE)) store_state(M, W, st, lane);
}

// ============================================================================ solver kernels (one thread per env)
//   prb_pgs_joint_kernel   slot 0 of the light envs (arm island without contacts): joint rows only, 32 envs / warp
//   prb_pgs_free_kernel    slots 1 and 2 (blockIdx.y): free-body islands, compact records, 32 envs / warp
//   prb_pgs_arm_kernel     slot 0 of the heavy envs, one launch per size class: joint rows + contact records,
//                          ARM_LANES(class) envs / warp, bundle staged by one bulk async copy
#define PGS_BLOCK 32
#define PGS_SMEM_J (PGS_STAGE_J * 32 * 16)
#define PGS_F_SLACKQ 8    // the free-body kernel loads the record after the current one (6 q) ahead of time: readable slack after the stage
#define PGS_SMEM_F ((PGS_STAGE_F + PGS_F_SLACKQ) * 32 * 16)
#define PGS_SMEM_ARM(k) (arm_capq(k) * arm_lanes(k) * 16)

#ifdef PRB_EMU
static float4 g_emu_pgs_smem[ARM_BUFQ_MAX * 32 + (PGS_STAGE_J + PGS_STAGE_F + 16) * 32];
#define PRB_PGS_SMEM_DECL float4* sm = g_emu_pgs_smem
#else
#define PRB_PGS_SMEM_DECL extern __shared__ __align__(128) float4 prb_pgs_smem[]; float4* sm = prb_pgs_smem
#endif

PRB_D float sel3(const float* a, int s) { return s == 0 ? a[0] : (s == 1 ? a[1] : a[2]); }   // register select (constant indices)
PRB_D float dot4(const float4& a, const float4& b, float s) { return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, fmaf(a.w, b.w, s)))); }
PRB_D float4* stream_col(float* sbuf, int e) { return reinterpret_cast<float4*>(sbuf) + (size_t)(e >> 5) * (SB_Q * 32) + (e & 31); }

// velocity change of the arm's island, in registers: arm DoF, slide bodies, free bodies (+ their inverse inertia)
struct IslandV {
  float A[12];
  float sl[PRB_MAXSLIDE];
  v3 fv[PRB_MAXFREE], fw[PRB_MAXFREE];
  float I[PRB_MAXFREE][6], invm[PRB_MAXFREE];
  // register selects (no runtime-indexed arrays: they would live in local memory)
  PRB_D float arm(int a) const {
    float r = A[0];
#pragma unroll
    for (int k = 1; k < 12; k++) r = a == k ? A[k] : r;
    return r;
  }
  PRB_D float slide(int s) const { return s == 0 ? sl[0] : (s == 1 ? sl[1] : sl[2]); }
  PRB_D void slide_add(int s, float v) { sl[0] += s == 0 ? v : 0.f; sl[1] += s == 1 ? v : 0.f; sl[2] += s == 2 ? v : 0.f; }
  PRB_D void arm_axpy(const float4& m0, const float4& m1, const float4& m2, float a) {
    A[0] = fmaf(m0.x, a, A[0]); A[1] = fmaf(m0.y, a, A[1]); A[2] = fmaf(m0.z, a, A[2]); A[3] = fmaf(m0.w, a, A[3]);
    A[4] = fmaf(m1.x, a, A[4]); A[5] = fmaf(m1.y, a, A[5]); A[6] = fmaf(m1.z, a, A[6]); A[7] = fmaf(m1.w, a, A[7]);
    A[8] = fmaf(m2.x, a, A[8]); A[9] = fmaf(m2.y, a, A[9]); A[10] = fmaf(m2.z, a, A[10]); A[11] = fmaf(m2.w, a, A[11]);
  }
  PRB_D float arm_dot(const float4& j0, const float4& j1, const float4& j2) const {
    const float p0 = fmaf(j0.x, A[0], fmaf(j0.y, A[1], fmaf(j0.z, A[2], j0.w * A[3])));
    const float p1 = fmaf(j1.x, A[4], fmaf(j1.y, A[5], fmaf(j1.z, A[6], j1.w * A[7])));
    const float p2 = fmaf(j2.x, A[8], fmaf(j2.y, A[9], fmaf(j2.z, A[10], j2.w * A[11])));
    return (p0 + p1) + p2;
  }
  PRB_D v3 vel(int b) const { return b ? fv[PRB_MAXFREE - 1] : fv[0]; }
  PRB_D v3 ang(int b) const { return b ? fw[PRB_MAXFREE - 1] : fw[0]; }
  // J . dv of a free-body side: unit force d at lever arm r (or unit torque d), times sgn
  PRB_D float jdot(int b, float sgn, v3 r, v3 d, bool angular) const {
    const v3 ww = ang(b);
    return sgn * (angular ? dot(d, ww) : dot(d, vel(b) + cross(ww, r)));
  }
  // dv += B P: P = sum of direction * impulse (linear rows) or the angular impulse (spin row)
  PRB_D void apply(int b, float sgn, v3 r, v3 P, bool angular) {
    const v3 Ps = P * sgn;
    float Ib[6];
#pragma unroll
    for (int k = 0; k < 6; k++) Ib[k] = b ? I[PRB_MAXFREE - 1][k] : I[0][k];
    const float im = b ? invm[PRB_MAXFREE - 1] : invm[0];
    v3 dv = V3(0, 0, 0), dw;
    if (angular) dw = symmul(Ib, Ps);
    else { dv = Ps * im; dw = symmul(Ib, cross(r, Ps)); }
    if (b) { fv[PRB_MAXFREE - 1] = fv[PRB_MAXFREE - 1] + dv; fw[PRB_MAXFREE - 1] = fw[PRB_MAXFREE - 1] + dw; }
    else { fv[0] = fv[0] + dv; fw[0] = fw[0] + dw; }
  }
  PRB_D void clear() {
#pragma unroll
    for (int k = 0; k < 12; k++) A[k] = 0.f;
#pragma unroll
    for (int k = 0; k < PRB_MAXSLIDE; k++) sl[k] = 0.f;
#pragma unroll
    for (int b = 0; b < PRB_MAXFREE; b++) { fv[b] = V3(0, 0, 0); fw[b] = V3(0, 0, 0); }
  }
};

// ---- joint rows of region 0.  col: this env's column of the staged region (q t at col[t * stride])
struct JointRows {
  const float4* col;
  int stride, njr, nL, t_jlam;
  bool canon;
  float ratio;
  float sminv[PRB_MAXSLIDE];
  float lm[12], ls[PRB_MAXSLIDE];       // impulses of the canonical motor rows (registers)
};
// any row: limits, gear, and every row of an env whose motor set is not the canonical one.  Its impulse lives in the
// staged region (word j of the area at t_jlam)
PRB_D bool jrow_generic(JointRows& R, IslandV& V, int j) {
  const float4 r = R.col[(size_t)(R0_JROW + j) * R.stride];
  const int pk = __float_as_int(r.x);
  const int pd = pk & 0xff, a = (pk >> 16) & 15, a2 = (pk >> 20) & 15;
  const int sidx = pd - DVW_SLIDE(0);                            // slide index when a == 15
  const float sg = ((pk >> 24) & 1) ? -1.0f : 1.0f;
  float u = a != 15 ? V.arm(a) : V.slide(sidx);
  if (a2 != 15) u = fmaf(R.ratio, V.arm(a2), u);
  u *= sg;
  float* pl = reinterpret_cast<float*>(const_cast<float4*>(R.col) + (size_t)(R.t_jlam + (j >> 2)) * R.stride) + (j & 3);
  const float l0 = *pl;
  const float hi = r.w, lo = ((pk >> 25) & 1) ? -hi : 0.f;
  const float nl = clampf(l0 + (r.y - u * r.z), lo, hi);
  const float dl = (nl - l0) * sg;
  if (dl != 0.f) {
    *pl = nl;
    if (a != 15) {
      const float4* m = R.col + (size_t)(R0_MINV + 3 * a) * R.stride;
      V.arm_axpy(m[0], m[R.stride], m[2 * R.stride], dl);
      if (a2 != 15) {
        const float4* m2 = R.col + (size_t)(R0_MINV + 3 * a2) * R.stride;
        V.arm_axpy(m2[0], m2[R.stride], m2[2 * R.stride], dl * R.ratio);
      }
    } else V.slide_add(sidx, sel3(R.sminv, sidx) * dl);
  }
  return dl != 0.f;
}
// a joint-limit row of an arm DoF (the rows before the motors of a canonical env): one-sided, single DoF
PRB_D bool jrow_limit(JointRows& R, IslandV& V, int j) {
  const float4 r = R.col[(size_t)(R0_JROW + j) * R.stride];
  const int pk = __float_as_int(r.x);
  const int a = (pk >> 16) & 15;
  const float sg = ((pk >> 24) & 1) ? -1.0f : 1.0f;
  const float4* m = R.col + (size_t)(R0_MINV + 3 * a) * R.stride;
  const float4 m0 = m[0], m1 = m[R.stride], m2 = m[2 * R.stride];
  float* pl = reinterpret_cast<float*>(const_cast<float4*>(R.col) + (size_t)(R.t_jlam + (j >> 2)) * R.stride) + (j & 3);
  const float l0 = *pl;
  const float u = V.arm(a) * sg;
  const float nl = clampf(l0 + (r.y - u * r.z), 0.f, r.w);
  const float dl = (nl - l0) * sg;
  *pl = nl;
  V.arm_axpy(m0, m1, m2, dl);
  return dl != 0.f;
}
// the motor row of arm DoF D / slide body S_ of a canonical env: compile-time register indices, impulse in a register
template <int D>
PRB_D bool jrow_motor(JointRows& R, IslandV& V) {
  const float4 r = R.col[(size_t)(R0_JROW + R.nL + D) * R.stride];
  const float4* m = R.col + (size_t)(R0_MINV + 3 * D) * R.stride;
  const float4 m0 = m[0], m1 = m[R.stride], m2 = m[2 * R.stride];
  const float l0 = R.lm[D];
  const float nl = clampf(l0 + (r.y - V.A[D] * r.z), -r.w, r.w);
  const float dl = nl - l0;
  R.lm[D] = nl;
  V.arm_axpy(m0, m1, m2, dl);
  return dl != 0.f;
}
template <int ND, int S_>
PRB_D bool jrow_slide(JointRows& R, IslandV& V) {
  const float4 r = R.col[(size_t)(R0_JROW + R.nL + ND + S_) * R.stride];
  const float l0 = R.ls[S_];
  const float nl = clampf(l0 + (r.y - V.sl[S_] * r.z), -r.w, r.w);
  const float dl = nl - l0;
  R.ls[S_] = nl;
  V.sl[S_] += R.sminv[S_] * dl;
  return dl != 0.f;
}
template <int ND, int D>
struct MotorUnroll {
  static PRB_D bool up(JointRows& R, IslandV& V) { bool c = MotorUnroll<ND, D - 1>::up(R, V); return jrow_motor<D>(R, V) | c; }
  static PRB_D bool down(JointRows& R, IslandV& V) { bool c = jrow_motor<D>(R, V); return MotorUnroll<ND, D - 1>::down(R, V) | c; }
};
template <int ND>
struct MotorUnroll<ND, -1> {
  static PRB_D bool up(JointRows&, IslandV&) { return false; }
  static PRB_D bool down(JointRows&, IslandV&) { return false; }
};
// one pass over the joint rows; direction alternates per iteration (btMultiBodyConstraintSolver: odd iterations ascend)
template <int ND>
PRB_D bool jrows_pass(JointRows& R, IslandV& V, int n_slide, bool ascending) {
  bool changed = false;
  if (!R.canon) {
#pragma unroll 1
    for (int ii = 0; ii < R.njr; ii++) changed |= jrow_generic(R, V, ascending ? ii : R.njr - 1 - ii);
    return changed;
  }
  const int tail0 = R.nL + ND + n_slide;                       // rows after the motors (gear)
  if (ascending) {
#pragma unroll 1
    for (int j = 0; j < R.nL; j++) changed |= jrow_limit(R, V, j);
    changed |= MotorUnroll<ND, ND - 1>::up(R, V);
    if (n_slide > 0) changed |= jrow_slide<ND, 0>(R, V);
    if (n_slide > 1) changed |= jrow_slide<ND, 1>(R, V);
    if (n_slide > 2) changed |= jrow_slide<ND, 2>(R, V);
#pragma unroll 1
    for (int j = tail0; j < R.njr; j++) changed |= jrow_generic(R, V, j);
  } else {
#pragma unroll 1
    for (int j = R.njr - 1; j >= tail0; j--) changed |= jrow_generic(R, V, j);
    if (n_slide > 2) changed |= jrow_slide<ND, 2>(R, V);
    if (n_slide > 1) changed |= jrow_slide<ND, 1>(R, V);
    if (n_slide > 0) changed |= jrow_slide<ND, 0>(R, V);
    changed |= MotorUnroll<ND, ND - 1>::down(R, V);
#pragma unroll 1
    for (int j = R.nL - 1; j >= 0; j--) changed |= jrow_limit(R, V, j);
  }
  return changed;
}
template <int ND>
PRB_D void jrows_init(JointRows& R, const DevModel& M, const float4* col, int stride, int h1, bool valid) {
  R.col = col; R.stride = stride;
  R.njr = valid ? (h1 & 0xff) : 0; R.canon = (h1 >> 24) & 1;
  R.nL = R.njr - ND - M.n_slide - (M.gear_a >= 0 ? 1 : 0);     // meaningful when canon
  R.t_jlam = R0_JROW + R.njr;
  R.ratio = M.params[P_GEAR_RATIO];
#pragma unroll
  for (int s = 0; s < PRB_MAXSLIDE; s++) { R.sminv[s] = s < M.n_slide ? M.slide_minv[s] : 0.f; R.ls[s] = 0.f; }
#pragma unroll
  for (int d = 0; d < 12; d++) R.lm[d] = 0.f;
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (valid) for (int k = 0; k < ((R.njr + 3) >> 2); k++) const_cast<float4*>(col)[(size_t)(R.t_jlam + k) * stride] = z4;
}
// velocity change -> stream (linear DoF order): arm, slides, and the free bodies this island owns
PRB_D void island_store(const DevModel& M, const IslandV& V, float* sbuf, int e, int info, bool with_free) {
  float* gd = reinterpret_cast<float*>(stream_col(sbuf, e) + Q_DV * 32);
  const int nd = M.nd, nf = M.n_free;
#pragma unroll
  for (int i = 0; i < 12; i++) if (i < nd) gd[(i >> 2) * 128 + (i & 3)] = V.A[i];
#pragma unroll
  for (int s = 0; s < PRB_MAXSLIDE; s++) if (s < M.n_slide) { const int d = nd + 6 * nf + s; gd[(d >> 2) * 128 + (d & 3)] = V.sl[s]; }
  if (with_free) {
#pragma unroll
    for (int b = 0; b < PRB_MAXFREE; b++)
      if (b < nf && ((info >> (16 + 2 * b)) & 3) == 0) {
        const float v6[6] = {V.fv[b].x, V.fv[b].y, V.fv[b].z, V.fw[b].x, V.fw[b].y, V.fw[b].z};
#pragma unroll
        for (int k = 0; k < 6; k++) { const int d = nd + 6 * b + k; gd[(d >> 2) * 128 + (d & 3)] = v6[k]; }
      }
  }
}

// ---- slot 0 of the light envs: joint rows only
template <int ND>
__global__ void __launch_bounds__(PGS_BLOCK) prb_pgs_joint_kernel(const DevModel* __restrict__ Mp, float* __restrict__ sbuf, int N,
                                                                 const unsigned char* __restrict__ active,
                                                                 const int* __restrict__ elist = nullptr, int n_list = 0) {
  PRB_PGS_SMEM_DECL;
  const int lane = threadIdx.x;
  const DevModel& M = *Mp;
  // persistent blocks: a block walks groups of 32 envs (launching one block per group costs more than
  // the solve: each block launch allocates its shared memory); warp-uniform control flow, per-lane predicates
  const int ngroups = ((elist != nullptr ? n_list : N) + PGS_BLOCK - 1) / PGS_BLOCK;
  for (int g = blockIdx.x; g < ngroups; g += gridDim.x) {
    bool valid;
    const int e = env_of(g * PGS_BLOCK + lane, N, active, elist, n_list, &valid);
    float4* G = stream_col(sbuf, valid ? e : 0);
    const int h0 = valid ? __float_as_int(G[Q_HDR * 32].x) : 0;
    if ((h0 >> 25) & 7) valid = false;                     // heavy: prb_pgs_arm_kernel solves it from its class buffer
    if (!__any_sync(FULL, valid)) continue;
    const int njr = valid ? (h0 & 0xff) : 0;
    float4* col = sm + lane;
    const float4* Gr = G + Q_ST * 32;
    {
      const int tq = R0_JROW + njr;
#pragma unroll 8
      for (int q = R0_MINV; q < tq; q++) col[q * 32] = Gr[q * 32];
    }
    IslandV V;
    V.clear();
    JointRows R;
    jrows_init<ND>(R, M, col, 32, h0, valid);
    const int iters = M.solver_iters;
    bool live = valid;
#pragma unroll 1
    for (int it = 0; it < iters; it++) {
      // A sweep that changes no impulse leaves the state untouched, so every later sweep repeats it
      // exactly: retiring the lane there is bit-identical to running all the iterations.
      bool changed = false;
      if (live) changed = jrows_pass<ND>(R, V, M.n_slide, (it & 1) != 0);
      __syncwarp();
      live = live && changed;
      if (!__any_sync(FULL, live)) break;
    }
    if (valid) island_store(M, V, sbuf, e, 0, false);
    __syncwarp();
  }
}

// ---- slots 1 and 2 (blockIdx.y + 1): islands of free bodies against static geometry / each other.  One thread per
// env, the bodies' velocity change in registers, compact records in the stage (records past PGS_STAGE_F are read from
// the stream in place), warp-uniform loops, the next record's loads issued before the current record is solved.
// Almost every island is ONE body against static geometry: that case runs without any body-index selects (OneBody);
// a block resting on the drawer makes a two-body island (IslandV's free-body part, register selects).
struct OneBody {
  v3 v, w;
  float I[6], im;
  PRB_D float jdot(int, float sgn, v3 r, v3 d, bool angular) const { return sgn * (angular ? dot(d, w) : dot(d, v + cross(w, r))); }
  PRB_D void apply(int, float sgn, v3 r, v3 P, bool angular) {
    const v3 Ps = P * sgn;
    if (angular) w = w + symmul(I, Ps);
    else { v = v + Ps * im; w = w + symmul(I, cross(r, Ps)); }
  }
};
struct FreeRec {
  int iP, iS; float sP; bool two; v3 n, rP, rS;
};
PRB_D FreeRec free_rec(int pk, const float4& q1, const float4& q2, const float4* rec) {
  FreeRec f;
  f.iP = (pk >> 4) & 7; f.iS = (pk >> 7) & 7;
  f.sP = ((pk >> 10) & 1) ? -1.0f : 1.0f;
  f.two = ((pk >> 2) & 3) == K_FREE;
  f.n = V3(q1.x, q1.y, q1.z); f.rP = V3(q2.x, q2.y, q2.z); f.rS = V3(0, 0, 0);
  if (f.two) { const float4 g = rec[CT_BASE_Q * 32]; f.rS = V3(g.x, g.y, g.z); }
  return f;
}
struct FreeQ { float4 q0, q1, q2, q3, q4, q5; };
template <class BV>
PRB_D bool free_normal(BV& V, float4* rec, const FreeQ& Q) {
  const FreeRec f = free_rec(__float_as_int(Q.q0.x), Q.q1, Q.q2, rec);
  float u = V.jdot(f.iP, f.sP, f.rP, f.n, false);
  if (f.two) u += V.jdot(f.iS, -f.sP, f.rS, f.n, false);
  const float l0 = Q.q1.w;
  const float nl = fmaxf(l0 + (Q.q0.z - l0 * Q.q0.y - u * Q.q0.w), 0.f);
  const float dl = nl - l0;
  if (dl != 0.f) {
    reinterpret_cast<float*>(rec + 32)[3] = nl;
    V.apply(f.iP, f.sP, f.rP, f.n * dl, false);
    if (f.two) V.apply(f.iS, -f.sP, f.rS, f.n * dl, false);
  }
  return dl != 0.f;
}
template <class BV>
PRB_D bool free_spin(BV& V, float4* rec, const float4& h) {
  const float4 q0 = rec[0], q1 = rec[32], q2 = rec[64];
  const float tot = q1.w;
  if (!(tot > 0.f)) return false;                         // Bullet skips the row while the normal impulse is 0
  const FreeRec f = free_rec(__float_as_int(q0.x), q1, q2, rec);
  float u = V.jdot(f.iP, f.sP, f.rP, f.n, true);
  if (f.two) u += V.jdot(f.iS, -f.sP, f.rS, f.n, true);
  const float lim = h.y * tot;
  float* pl = reinterpret_cast<float*>(rec + 96) + 3;
  const float l0 = *pl;
  const float nl = clampf(l0 + (h.z - u * h.w), -lim, lim);
  const float dl = nl - l0;
  if (dl != 0.f) {
    *pl = nl;
    V.apply(f.iP, f.sP, f.rP, f.n * dl, true);
    if (f.two) V.apply(f.iS, -f.sP, f.rS, f.n * dl, true);
  }
  return dl != 0.f;
}
// lateral friction: the two rows of a contact are solved together (implicit cone)
template <class BV>
PRB_D bool free_friction(BV& V, float4* rec, const FreeQ& Q) {
  const FreeRec f = free_rec(__float_as_int(Q.q0.x), Q.q1, Q.q2, rec);
  const v3 t1 = V3(Q.q3.x, Q.q3.y, Q.q3.z), t2 = cross(f.n, t1);
  float ua = V.jdot(f.iP, f.sP, f.rP, t1, false), ub = V.jdot(f.iP, f.sP, f.rP, t2, false);
  if (f.two) { ua += V.jdot(f.iS, -f.sP, f.rS, t1, false); ub += V.jdot(f.iS, -f.sP, f.rS, t2, false); }
  const float lim = Q.q2.w * Q.q1.w;
  const float la = Q.q5.x, lb = Q.q5.y;
  const float sumA = la + (Q.q4.x - ua * Q.q4.z);
  const float sumB = lb + (Q.q4.y - ub * Q.q4.w);
  float na = sumA, nb = sumB;
  if (sumA < -lim || sumA > lim || sumB < -lim || sumB > lim) {
    const float ss = sumA * sumA + sumB * sumB;
    const float inv = ss > 0.f ? rsqrtf(ss) : 0.f;
    const float ca_ = fabsf(lim * sumA) * inv, cb_ = ss > 0.f ? fabsf(lim * sumB) * inv : fabsf(lim);
    na = clampf(sumA, -ca_, ca_); nb = clampf(sumB, -cb_, cb_);
  }
  const float d1 = na - la, d2 = nb - lb;
  if (d1 != 0.f || d2 != 0.f) {
    rec[160] = make_float4(na, nb, 0.f, 0.f);
    const v3 Pv = t1 * d1 + t2 * d2;
    V.apply(f.iP, f.sP, f.rP, Pv, false);
    if (f.two) V.apply(f.iS, -f.sP, f.rS, Pv, false);
  }
  return d1 != 0.f || d2 != 0.f;
}
// the 50 sweeps of one island; sl: this env's staged column, Gr: its records in the stream
// STAGED: every island of the warp fits the stage -> every record pointer is a shared-memory pointer (LDS / STS); otherwise
// a pointer may be either, and all accesses of the sweep become generic loads.
template <class BV, bool STAGED>
PRB_D void free_sweeps(BV& V, float4* sl, float4* Gr, bool live, int nc, int ns, int ncmax, int nsmax, int t_spin, int iters) {
#define PGS_PTR(t_) ((STAGED || (t_) < PGS_STAGE_F) ? sl + (t_) * 32 : Gr + (t_) * 32)
#pragma unroll 1
  for (int it = 0; it < iters; it++) {
    bool changed = false;
    // ---- contact normals (the next record is loaded while the current one is solved; readable slack after the last)
    {
      int t = 0;
      float4* rec = PGS_PTR(0);
      FreeQ Q;
      Q.q0 = rec[0]; Q.q1 = rec[32]; Q.q2 = rec[64];
#pragma unroll 1
      for (int c = 0; c < ncmax; c++) {
        if (live && c < nc) {
          const int tn = t + ((__float_as_int(Q.q0.x) >> 12) & 255);
          float4* recn = PGS_PTR(tn);
          FreeQ N;
          N.q0 = recn[0]; N.q1 = recn[32]; N.q2 = recn[64];
          changed |= free_normal(V, rec, Q);
          t = tn; rec = recn; Q.q0 = N.q0; Q.q1 = N.q1; Q.q2 = N.q2;
        }
        __syncwarp();
      }
    }
    // ---- spinning friction
#pragma unroll 1
    for (int i = 0; i < nsmax; i++) {
      if (live && i < ns) {
        const float4 h = *PGS_PTR(t_spin + i);
        changed |= free_spin(V, PGS_PTR(__float_as_int(h.x)), h);
      }
      __syncwarp();
    }
    // ---- lateral friction
    {
      int t = 0;
      float4* rec = PGS_PTR(0);
      FreeQ Q;
      Q.q0 = rec[0]; Q.q1 = rec[32]; Q.q2 = rec[64]; Q.q3 = rec[96]; Q.q4 = rec[128]; Q.q5 = rec[160];
#pragma unroll 1
      for (int c = 0; c < ncmax; c++) {
        if (live && c < nc) {
          const int tn = t + ((__float_as_int(Q.q0.x) >> 12) & 255);
          float4* recn = PGS_PTR(tn);
          FreeQ N;
          N.q0 = recn[0]; N.q1 = recn[32]; N.q2 = recn[64]; N.q3 = recn[96]; N.q4 = recn[128]; N.q5 = recn[160];
          changed |= free_friction(V, rec, Q);
          t = tn; rec = recn; Q = N;
        }
        __syncwarp();
      }
    }
    // fixed point reached (a sweep changed no impulse): later sweeps are exact repeats, the lane retires
    live = live && changed;
    if (!__any_sync(FULL, live)) break;
  }
#undef PGS_PTR
}

__global__ void __launch_bounds__(PGS_BLOCK) prb_pgs_free_kernel(const DevModel* __restrict__ Mp, float* __restrict__ sbuf, int N,
                                                                const unsigned char* __restrict__ active,
                                                                const int* __restrict__ elist = nullptr, int n_list = 0,
                                                                int writeback = 0) {
  // writeback: the staged records (with their impulses) are copied back to the stream after the sweeps, for the contact
  // report.  Records beyond the stage were updated in place; the stage never holds part of one.
  PRB_PGS_SMEM_DECL;
  const int lane = threadIdx.x;
  const int slot = blockIdx.y + 1;
  const DevModel& M = *Mp;
  const int ngroups = ((elist != nullptr ? n_list : N) + PGS_BLOCK - 1) / PGS_BLOCK;
  for (int g = blockIdx.x; g < ngroups; g += gridDim.x) {     // persistent blocks, warp-uniform control flow
    bool valid;
    const int e = env_of(g * PGS_BLOCK + lane, N, active, elist, n_list, &valid);
    float4* G = stream_col(sbuf, valid ? e : 0);
    const float4 h1 = G[(Q_HDR + 1) * 32], hs = G[(Q_HDR + slot) * 32];
    const int info = __float_as_int(h1.x);
    const int cnt = __float_as_int(hs.x);
    const int start = __float_as_int(hs.y), t_spin = __float_as_int(hs.z);
    int n_own = 0, b_own = 0;
    for (int b = 0; b < M.n_free; b++) if (((info >> (16 + 2 * b)) & 3) == slot) { n_own++; b_own = b; }
    valid = valid && n_own > 0;                            // no body of this slot: merged into another island
    if (!__any_sync(FULL, valid)) continue;
    const int nc = valid ? (cnt & 0xff) : 0, ns = valid ? ((cnt >> 8) & 0xff) : 0;
    int ncmax = nc, nsmax = ns;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { ncmax = max(ncmax, __shfl_xor_sync(FULL, ncmax, o)); nsmax = max(nsmax, __shfl_xor_sync(FULL, nsmax, o)); }
    float4* sl = sm + lane;
    float4* Gr = G + (Q_S12 + start) * 32;
    if (valid) {
      const int tq = min(t_spin + ns, PGS_STAGE_F);
#pragma unroll 8
      for (int q = 0; q < tq; q++) sl[q * 32] = Gr[q * 32];
    }
    IslandV V;
    V.clear();
#pragma unroll
    for (int fb = 0; fb < PRB_MAXFREE; fb++) {
      const float4 i0 = G[(Q_ST + R0_BODY + 2 * fb) * 32], i1 = G[(Q_ST + R0_BODY + 2 * fb + 1) * 32];
      V.I[fb][0] = i0.x; V.I[fb][1] = i0.y; V.I[fb][2] = i0.z; V.I[fb][3] = i0.w; V.I[fb][4] = i1.x; V.I[fb][5] = i1.y;
      V.invm[fb] = i1.z;
    }
    const int iters = M.solver_iters;
    const bool single = n_own == 1;
    if (__any_sync(FULL, valid && single)) {               // one body against static geometry: no selects
      OneBody B;
      B.v = V3(0, 0, 0); B.w = V3(0, 0, 0);
#pragma unroll
      for (int k = 0; k < 6; k++) B.I[k] = b_own ? V.I[PRB_MAXFREE - 1][k] : V.I[0][k];
      B.im = b_own ? V.invm[PRB_MAXFREE - 1] : V.invm[0];
      const bool on = valid && single;
      // (the solver reads one record ahead: PGS_F_SLACKQ q of slack follow the stage)
      if (__all_sync(FULL, !on || t_spin + ns <= PGS_STAGE_F)) free_sweeps<OneBody, true>(B, sl, Gr, on, on ? nc : 0, on ? ns : 0, ncmax, nsmax, t_spin, iters);
      else free_sweeps<OneBody, false>(B, sl, Gr, on, on ? nc : 0, on ? ns : 0, ncmax, nsmax, t_spin, iters);
      if (on) { if (b_own) { V.fv[PRB_MAXFREE - 1] = B.v; V.fw[PRB_MAXFREE - 1] = B.w; } else { V.fv[0] = B.v; V.fw[0] = B.w; } }
    }
    if (__any_sync(FULL, valid && !single)) {
      const bool on = valid && !single;
      free_sweeps<IslandV, false>(V, sl, Gr, on, on ? nc : 0, on ? ns : 0, ncmax, nsmax, t_spin, iters);
    }
    if (valid) {
      float* gd = reinterpret_cast<float*>(G + Q_DV * 32);
#pragma unroll
      for (int b = 0; b < PRB_MAXFREE; b++)
        if (b < M.n_free && ((info >> (16 + 2 * b)) & 3) == slot) {
          const float v6[6] = {V.fv[b].x, V.fv[b].y, V.fv[b].z, V.fw[b].x, V.fw[b].y, V.fw[b].z};
          const int o = M.nd + 6 * b;
#pragma unroll
          for (int k = 0; k < 6; k++) gd[((o + k) >> 2) * 128 + ((o + k) & 3)] = v6[k];
        }
      if (writeback)
        for (int q = 0; q < min(t_spin + ns, PGS_STAGE_F); q++) Gr[q * 32] = sl[q * 32];
    }
    __syncwarp();
  }
}

// ============================================================================ arm-island solver
// One thread per env.  Every load of a contact visit sits at a fixed offset from the record start and is issued
// before the flags are decoded (a record without an arm / slide / free side just reads the next record's bytes
// or the slack after the region), so a visit is: ~12 independent LDS.128 -> 12-FMA dot + free-body terms ->
// clamp -> 12-FMA update + one STS of the impulse.  No shuffles, no barriers: the env's records and velocities
// are private to the thread.
template <int STRIDE>
struct ArmRec {              // one record: q k at p[k * STRIDE] (shared memory, or the heavy buffer when read in place); the
  float4* p;                 // stride is the class's envs per block, a compile-time constant: every load is base + immediate
  PRB_D float4 ld(int k) const { return p[k * STRIDE]; }
  PRB_D float* lam() const { return reinterpret_cast<float*>(p + 3 * STRIDE); }
};
struct FreeGeom { int fb; float sgn; bool two; v3 n, t1, rF, rS; };
PRB_D FreeGeom free_geom(int flags, const float4& G0, const float4& G1, const float4& G2) {
  FreeGeom g;
  g.fb = (flags & CR_FB) ? 1 : 0; g.sgn = (flags & CR_FNEG) ? -1.0f : 1.0f; g.two = (flags & CR_TWO) != 0;
  g.n = V3(G0.x, G0.y, G0.z); g.t1 = V3(G1.x, G1.y, G1.z); g.rF = V3(G2.x, G2.y, G2.z); g.rS = V3(G0.w, G1.w, G2.w);
  return g;
}
// contact normal: lambda >= 0, soft CFM
template <class REC>
PRB_D bool visit_normal(const REC& r, IslandV& V, const float* sminv, int& size) {
  const float4 H0 = r.ld(0), L = r.ld(3), G0 = r.ld(4), G1 = r.ld(5), G2 = r.ld(6), SL = r.ld(7);
  const float4 J0 = r.ld(8), J1 = r.ld(9), J2 = r.ld(10), B0 = r.ld(11), B1 = r.ld(12), B2 = r.ld(13);
  const int flags = __float_as_int(H0.x);
  size = flags >> 16;
  const int sidx = (flags >> 6) & 3;
  // the arm side is computed unconditionally and masked (a record without one reads finite bytes of its neighbour):
  // straight-line code schedules better than a branch per side in this latency-bound loop
  const bool arm = (flags & CR_ARM) != 0;
  float u = arm ? V.arm_dot(J0, J1, J2) : 0.f;
  if (flags & CR_SLIDE) u = fmaf(SL.x, V.slide(sidx), u);
  FreeGeom g = free_geom(flags, G0, G1, G2);
  if (flags & CR_FREE) {
    u += V.jdot(g.fb, g.sgn, g.rF, g.n, false);
    if (g.two) u += V.jdot(1 - g.fb, -g.sgn, g.rS, g.n, false);
  }
  const float l0 = L.x;
  const float nl = fmaxf(l0 + (H0.y - l0 * H0.w - u * H0.z), 0.f);
  const float dl = nl - l0;
  r.lam()[0] = nl;
  V.arm_axpy(B0, B1, B2, arm ? dl : 0.f);
  if (dl != 0.f) {
    if (flags & CR_SLIDE) V.slide_add(sidx, (SL.x * sel3(sminv, sidx)) * dl);
    if (flags & CR_FREE) {
      V.apply(g.fb, g.sgn, g.rF, g.n * dl, false);
      if (g.two) V.apply(1 - g.fb, -g.sgn, g.rS, g.n * dl, false);
    }
  }
  return dl != 0.f;
}
// spinning friction: |lambda| <= coefficient * normal impulse (Bullet skips the row while the normal impulse is 0)
template <class REC>
PRB_D bool visit_spin(const REC& r, IslandV& V, const float* sminv, int& size) {
  const float4 H0 = r.ld(0), H1 = r.ld(1), L = r.ld(3), G0 = r.ld(4), G1 = r.ld(5), G2 = r.ld(6), SL = r.ld(7);
  const float4 J0 = r.ld(26), J1 = r.ld(27), J2 = r.ld(28), B0 = r.ld(29), B1 = r.ld(30), B2 = r.ld(31);
  const int flags = __float_as_int(H0.x);
  size = flags >> 16;
  const float tot = L.x;
  if (!(flags & CR_SPIN) || !(tot > 0.f)) return false;
  const int sidx = (flags >> 6) & 3;
  const bool arm = (flags & CR_ARM) != 0;
  float u = arm ? V.arm_dot(J0, J1, J2) : 0.f;
  if (flags & CR_SLIDE) u = fmaf(SL.y, V.slide(sidx), u);
  FreeGeom g = free_geom(flags, G0, G1, G2);
  if (flags & CR_FREE) {
    u += V.jdot(g.fb, g.sgn, g.rF, g.n, true);
    if (g.two) u += V.jdot(1 - g.fb, -g.sgn, g.rS, g.n, true);
  }
  const float lim = H1.z * tot;
  const float l0 = L.y;
  const float nl = clampf(l0 + (H1.x - u * H1.y), -lim, lim);
  const float dl = nl - l0;
  r.lam()[1] = nl;
  V.arm_axpy(B0, B1, B2, arm ? dl : 0.f);
  if (dl != 0.f) {
    if (flags & CR_SLIDE) V.slide_add(sidx, (SL.y * sel3(sminv, sidx)) * dl);
    if (flags & CR_FREE) {
      V.apply(g.fb, g.sgn, g.rF, g.n * dl, true);
      if (g.two) V.apply(1 - g.fb, -g.sgn, g.rS, g.n * dl, true);
    }
  }
  return dl != 0.f;
}
// lateral friction: the two rows of a contact are solved together (implicit cone)
template <class REC>
PRB_D bool visit_friction(const REC& r, IslandV& V, const float* sminv, int& size) {
  const float4 H0 = r.ld(0), H1 = r.ld(1), H2 = r.ld(2), L = r.ld(3), G0 = r.ld(4), G1 = r.ld(5), G2 = r.ld(6), SL = r.ld(7);
  const float4 Ja0 = r.ld(14), Ja1 = r.ld(15), Ja2 = r.ld(16), Ba0 = r.ld(17), Ba1 = r.ld(18), Ba2 = r.ld(19);
  const float4 Jb0 = r.ld(20), Jb1 = r.ld(21), Jb2 = r.ld(22), Bb0 = r.ld(23), Bb1 = r.ld(24), Bb2 = r.ld(25);
  const int flags = __float_as_int(H0.x);
  size = flags >> 16;
  const int sidx = (flags >> 6) & 3;
  const bool arm = (flags & CR_ARM) != 0;
  float ua = arm ? V.arm_dot(Ja0, Ja1, Ja2) : 0.f, ub = arm ? V.arm_dot(Jb0, Jb1, Jb2) : 0.f;
  if (flags & CR_SLIDE) { const float vs = V.slide(sidx); ua = fmaf(SL.z, vs, ua); ub = fmaf(SL.w, vs, ub); }
  FreeGeom g = free_geom(flags, G0, G1, G2);
  const v3 t2 = cross(g.n, g.t1);
  if (flags & CR_FREE) {
    ua += V.jdot(g.fb, g.sgn, g.rF, g.t1, false); ub += V.jdot(g.fb, g.sgn, g.rF, t2, false);
    if (g.two) { ua += V.jdot(1 - g.fb, -g.sgn, g.rS, g.t1, false); ub += V.jdot(1 - g.fb, -g.sgn, g.rS, t2, false); }
  }
  const float lim = H1.w * L.x;
  const float la = L.z, lb = L.w;
  const float sumA = la + (H2.x - ua * H2.z);
  const float sumB = lb + (H2.y - ub * H2.w);
  float na = sumA, nb = sumB;
  if (sumA < -lim || sumA > lim || sumB < -lim || sumB > lim) {
    // |lim sin(atan2(A,B))| and |lim cos(atan2(A,B))| as |lim A| / r and |lim B| / r
    const float ss = sumA * sumA + sumB * sumB;
    const float inv = ss > 0.f ? rsqrtf(ss) : 0.f;
    const float ca_ = fabsf(lim * sumA) * inv, cb_ = ss > 0.f ? fabsf(lim * sumB) * inv : fabsf(lim);
    na = clampf(sumA, -ca_, ca_); nb = clampf(sumB, -cb_, cb_);
  }
  const float d1 = na - la, d2 = nb - lb;
  r.lam()[2] = na; r.lam()[3] = nb;
  V.arm_axpy(Ba0, Ba1, Ba2, arm ? d1 : 0.f);
  V.arm_axpy(Bb0, Bb1, Bb2, arm ? d2 : 0.f);
  if (d1 != 0.f || d2 != 0.f) {
    if (flags & CR_SLIDE) { const float mi = sel3(sminv, sidx); V.slide_add(sidx, (SL.z * mi) * d1 + (SL.w * mi) * d2); }
    if (flags & CR_FREE) {
      const v3 Pv = g.t1 * d1 + t2 * d2;
      V.apply(g.fb, g.sgn, g.rF, Pv, false);
      if (g.two) V.apply(1 - g.fb, -g.sgn, g.rS, Pv, false);
    }
  }
  return d1 != 0.f || d2 != 0.f;
}

#ifndef PRB_EMU
// 1-D bulk async copy global -> shared, completion on an mbarrier (the TMA engine of sm_90+/sm_100a)
PRB_D void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
PRB_D void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
PRB_D void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
}
PRB_D void bulk_g2s(void* smem_dst, const void* gmem_src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   (unsigned)__cvta_generic_to_shared(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar))
               : "memory");
}
PRB_D void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
#endif

// LANES: envs per block (<= 32, the other threads of the warp idle; compile time: it is the stride of every record load);
// capq: staged q per env; bufq: q reserved per env in the class buffer (> capq only for the last class, whose islands may
// be read in place beyond the stage)
template <int ND, bool INPLACE, int LANES>
__global__ void __launch_bounds__(32) prb_pgs_arm_kernel(const DevModel* __restrict__ Mp, float* __restrict__ sbuf, float4* __restrict__ hcls,
                                                                int* __restrict__ heavy_cnt, int capq, int bufq, int writeback = 0) {
  // writeback: after the sweeps the impulse quad (+3) of every staged contact record is copied back to the class buffer, for
  // the contact report.  Only staged records: INPLACE records read beyond the stage were updated there, and the stage's
  // stale copy of their first q must not overwrite them.
  constexpr int lanes = LANES;
  PRB_PGS_SMEM_DECL;
  const int lane = threadIdx.x;
  const DevModel& M = *Mp;
  const int cnt = heavy_cnt[0];
  const int nb = (cnt + lanes - 1) / lanes;
#ifndef PRB_EMU
  __shared__ __align__(8) unsigned long long mbar;
  if (lane == 0) mbar_init(&mbar, 1);
  __syncwarp();
  unsigned parity = 0;
#endif
  __shared__ int wb_bundle;           // the bundle being solved (read back by the write-back)
  float sminv[PRB_MAXSLIDE];
#pragma unroll
  for (int s = 0; s < PRB_MAXSLIDE; s++) sminv[s] = s < M.n_slide ? M.slide_minv[s] : 0.f;
  // persistent blocks, dynamic scheduling: the block draws the next bundle of the class from a device counter
  for (;;) {
    int b = 0;
    if (lane == 0) b = atomicAdd(heavy_cnt + 2, 1);
    b = __shfl_sync(FULL, b, 0);
    if (b >= nb) break;
    if (writeback && lane == 0) wb_bundle = b;
    float4* Gb = hcls + (size_t)b * ((size_t)bufq * lanes);
    // ---- stage the bundle: capq x lanes float4, contiguous in the class buffer
#ifndef PRB_EMU
    if (lane == 0) {
      fence_async_smem();                                  // the previous bundle's impulse stores precede the async writes
      const unsigned bytes = (unsigned)(capq * lanes * 16);
      mbar_expect_tx(&mbar, bytes);
      bulk_g2s(sm, Gb, bytes, &mbar);
    }
    mbar_wait(&mbar, parity);
    parity ^= 1;
#else
    for (int q = lane; q < capq * lanes; q += 32) sm[q] = Gb[q];
    __syncwarp();
#endif
    // Control flow is kept WARP-UNIFORM (loop bounds = the bundle's maxima, per-lane predicates inside): lanes that
    // drift apart in data-dependent loops would each fetch and issue the same code on their own (measured in r2b:
    // 4.7 of 16 lanes active per instruction, 2-3 x the warp instructions).
    const int i = b * lanes + lane;
    const bool valid = lane < lanes && i < cnt;
    float4* col = sm + (valid ? lane : 0);
    float4* gcol = Gb + (valid ? lane : 0);
    const float4 hq = col[R0_HQ * lanes];
    const int e = __float_as_int(hq.x), h1 = valid ? __float_as_int(hq.y) : 0, info = __float_as_int(hq.z);
    const int nc = (h1 >> 8) & 0xff;
    int ncmax = nc;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ncmax = max(ncmax, __shfl_xor_sync(FULL, ncmax, o));
    IslandV V;
    V.clear();
#pragma unroll
    for (int fb = 0; fb < PRB_MAXFREE; fb++) {
      const float4 i0 = col[(R0_BODY + 2 * fb) * lanes], i1 = col[(R0_BODY + 2 * fb + 1) * lanes];
      V.I[fb][0] = i0.x; V.I[fb][1] = i0.y; V.I[fb][2] = i0.z; V.I[fb][3] = i0.w; V.I[fb][4] = i1.x; V.I[fb][5] = i1.y;
      V.invm[fb] = i1.z;
    }
    JointRows R;
    jrows_init<ND>(R, M, col, lanes, h1, valid);
    const int tC0 = R.t_jlam + ((R.njr + 3) >> 2);
    const int iters = M.solver_iters;
    bool live = valid;
#define ARM_REC(t_) ArmRec<LANES>{(INPLACE && (t_) + CR_MAX_Q > capq) ? gcol + (t_) * lanes : col + (t_) * lanes}
#pragma unroll 1
    for (int it = 0; it < iters; it++) {
      bool changed = false;
      if (live) changed = jrows_pass<ND>(R, V, M.n_slide, (it & 1) != 0);
      __syncwarp();
      int t = tC0, size;
#pragma unroll 1
      for (int k = 0; k < ncmax; k++) {
        if (live && k < nc) { changed |= visit_normal(ARM_REC(t), V, sminv, size); t += size; }
        __syncwarp();
      }
      t = tC0;
#pragma unroll 1
      for (int k = 0; k < ncmax; k++) {
        if (live && k < nc) { changed |= visit_spin(ARM_REC(t), V, sminv, size); t += size; }
        __syncwarp();
      }
      t = tC0;
#pragma unroll 1
      for (int k = 0; k < ncmax; k++) {
        if (live && k < nc) { changed |= visit_friction(ARM_REC(t), V, sminv, size); t += size; }
        __syncwarp();
      }
      // fixed point reached (a sweep changed no impulse): later sweeps are exact repeats, the lane retires
      live = live && changed;
      if (!__any_sync(FULL, live)) break;
    }
#undef ARM_REC
    if (valid) island_store(M, V, sbuf, e, info, true);
    if (writeback && valid) {
      // the bundle's global column and its records' start are derived again from shared memory: no value of the staging
      // stays live across the sweeps, which keep their registers
      float4* gw = hcls + (size_t)wb_bundle * ((size_t)bufq * lanes) + lane;
      const float4* sw = sm + lane;
      const int hw = __float_as_int(sw[R0_HQ * lanes].y), njw = hw & 0xff, ncw = (hw >> 8) & 0xff;
      int t = R0_JROW + njw + ((njw + 3) >> 2);
      for (int k = 0; k < ncw; k++) {
        const bool staged = !(INPLACE && t + CR_MAX_Q > capq);
        const float4* r = (staged ? sw : gw) + (size_t)t * lanes;
        if (staged) gw[(size_t)(t + 3) * lanes] = r[3 * lanes];
        t += __float_as_int(r[0].x) >> 16;
      }
    }
    __syncwarp();                                          // the stage is re-filled by the next bundle
  }
}
