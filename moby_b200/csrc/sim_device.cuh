// Group-cooperative device code of the stepped path for free rigid bodies with sphere / box / plane geometry:
// narrowphase + conservative advancement, semi-implicit Euler with Newton-Euler forward dynamics, island
// grouping, Delassus / LCP assembly (QP-as-LCP and Anitescu-Potra), solve, impulse write-back, restitution.
//
// Behavioural contract (Moby tree): TimeSteppingSimulator.cpp:52-222,272-331,433-455; ConstraintSimulator.cpp:
// 298-355,450-537; CCD.cpp:122-460,585-607; CCD.inl:3-82,805-886,1165-1259; UnilateralConstraint.cpp:695-747,
// 940-1225,1387-1446; ImpactConstraintHandler.cpp:96-168,298-626,1590-2166; ImpactConstraintHandlerQP.cpp:94-497;
// ImpactConstraintHandlerLCP.cpp:36-370.  One thread group (a warp for small scenes) owns one env; the env's
// bodies, contacts, Delassus blocks, LCP matrix and solver work space all live in shared memory, so an env-step
// touches HBM only for its state (13 doubles per body in and out) and its warm-start vector.
#pragma once
#include "lcp_device.cuh"
#include "rc_device.cuh"

namespace b2m {

enum { SH_NONE = 0, SH_SPHERE = 1, SH_BOX = 2, SH_PLANE = 3,
       SH_WHEEL = 4,
       SH_PIN = 5, SH_PINWORLD = 6 };   // example/contact-constrained-pendulum: a pin joint as six frictionless contacts (its collision-detection plugin); dims of SH_PIN = the anchor point in the body frame   // rimless wheel of example/rimless-wheel/coldet-plugin.cpp: dims = (R, W, N_SPOKES) (params.h:4-6); collides with planes only
enum { CNT_ENV_STEPS = 0, CNT_MINI_STEPS, CNT_LCP_SOLVES, CNT_FAST_CALLS, CNT_LEMKE_CALLS, CNT_PIVOTS, CNT_LCP_FAIL,
       CNT_IMPACT_TOL, CNT_CONTACTS, CNT_MAX_N, CNT_OVERFLOW, CNT_PIVOT_FLOPS, CNT_ASM_FLOPS, CNT_CA_ITERS, CNT_STAB_ITERS, CNT_STAB_SOLVES, CNT_STAB_LSFAIL, CNT_COUNT };
#define B2M_NKMAX 64
#define B2M_WHEEL_NS_MAX 16
#define B2M_WTAB_OFF ((size_t)4 * (B2M_NKMAX + 1) * (B2M_NKMAX / 2))   // spoke directions after the friction tables (friction_table.h)
#define B2M_MAX_CLASSES 12
// queue slots of one round: [0, n_classes) impact classes, then the envs that still have time left in their step, then stragglers
#define B2M_SLOT_CONT B2M_MAX_CLASSES
#define B2M_SLOT_STRAGGLER (B2M_MAX_CLASSES + 1)
#define B2M_SLOT_HARD (B2M_MAX_CLASSES + 2)   /* envs whose previous impact was expensive: solved first, on their own stream */
#define B2M_SLOT_HARD_BACK (B2M_MAX_CLASSES + 3)   /* counter only: the hard queue is filled from both ends, costliest envs at the front */
#define B2M_SLOTS (B2M_MAX_CLASSES + 4)
#define B2M_ROUNDS_MAX 8
#define B2M_MAX_STALL 64
// B2M_LEAN builds drop the articulated-body and box-box code paths (scenes of free spheres / boxes on planes): the
// kernels' instruction footprint, not arithmetic, bounds the stepped path (profiles/: no_instruction is the top stall).
#ifndef B2M_LEAN
#define B2M_LEAN 0
#endif
#define B2M_RC(P) (!B2M_LEAN && (P).rc_links)
#define B2M_NGC(P) (!B2M_LEAN && (P).ngc)
#define B2M_BOXBOX (!B2M_LEAN)

struct V3 {
  double x, y, z;
  B2M_HD V3() : x(0), y(0), z(0) {}
  B2M_HD V3(double a, double b, double c) : x(a), y(b), z(c) {}
};
B2M_HD B2M_INL V3 operator+(const V3& a, const V3& b) { return V3(a.x + b.x, a.y + b.y, a.z + b.z); }
B2M_HD B2M_INL V3 operator-(const V3& a, const V3& b) { return V3(a.x - b.x, a.y - b.y, a.z - b.z); }
B2M_HD B2M_INL V3 operator-(const V3& a) { return V3(-a.x, -a.y, -a.z); }
B2M_HD B2M_INL V3 operator*(const V3& a, double s) { return V3(a.x * s, a.y * s, a.z * s); }
B2M_HD B2M_INL double dot(const V3& a, const V3& b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
B2M_HD B2M_INL V3 cross(const V3& a, const V3& b) { return V3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
B2M_HD B2M_INL double norm(const V3& a) { return sqrt(dot(a, a)); }
B2M_HD B2M_INL V3 normalize(const V3& a) { const double n = norm(a); return V3(a.x / n, a.y / n, a.z / n); }
B2M_HD B2M_INL V3 rot(const double* R, const V3& v) { return V3(R[0] * v.x + R[1] * v.y + R[2] * v.z, R[3] * v.x + R[4] * v.y + R[5] * v.z, R[6] * v.x + R[7] * v.y + R[8] * v.z); }
B2M_HD B2M_INL V3 rotT(const double* R, const V3& v) { return V3(R[0] * v.x + R[3] * v.y + R[6] * v.z, R[1] * v.x + R[4] * v.y + R[7] * v.z, R[2] * v.x + R[5] * v.y + R[8] * v.z); }
B2M_HD B2M_INL V3 ld3(const double* p) { return V3(p[0], p[1], p[2]); }
B2M_HD B2M_INL void st3(double* p, const V3& v) { p[0] = v.x; p[1] = v.y; p[2] = v.z; }

// Scene + state of a batch, device pointers (SoA across envs, see include/b200moby.h)
struct SimParams {
  int n_envs, nb, cmax, nmax, npmax, model;
  const int* shape; const int* enabled; const double* mass; const double* dims; const double* inertia;
  const double* mu_c; const double* mu_v; const double* eps; const double* compliance; const int* NK;
  const double* fr_tab;        // [4][B2M_NKMAX+1][B2M_NKMAX/2]: QP cos, QP sin, AP cos, AP sin (host libm values), then the rimless wheel's spoke directions
  double gx, gy, gz, contact_dist_thresh, min_step_size;
  int stab_max_iterations; double stab_eps;   // ConstraintStabilization::max_iterations (0 off, < 0 unlimited) and eps (stab_device.cuh)
  const double* min_step_env;   // optional [env]
  double* q; double* v; double* time; double* zlast; int* zlast_n;
  double* vlast; int* vlast_n;     // [cmax][env], [env]: solution / warm start of the no-slip LCP (ImpactConstraintHandler::_v)
  unsigned long long* counters;
  // Longest-job-first: cost[env] = solver iterations executed in the env's last impact phase, decaying by a quarter per impact (at least 4 hard_cost after it ran over a budget).  An env
  // at or above hard_cost is queued in B2M_SLOT_HARD instead of its class, and that queue is launched first, so the few
  // envs that set the step time (degenerate contact sets: four failed lcp_fast runs, then the Lemke ladder) run
  // alongside the bulk instead of after it.  The same envs are hard step after step (resting contact persists).
  int* cost; int hard_cost; int cost_shift;   // decay per impact: cost -= cost >> cost_shift
  int thread_lanes;            // envs per warp of the thread-per-env impact kernels (0 / 32: all lanes)
  int pivot_budget;            // > 0: per-env pivot budget of the warp-per-env impact kernels; over-budget envs are re-run by the straggler kernel
  // phased step (advance -> impact per LCP class -> advance ...): per-env progress and work queues
  double* hacc;                // [env] seconds of the current step already simulated
  double* hpend;               // [env] length of the mini-step waiting for its impact solve
  int* queue;                  // queue[(round * B2M_SLOTS + slot) * n_envs + i]
  int* qctl;                   // [2][B2M_ROUNDS_MAX][B2M_SLOTS + 1] counts, then heads (slot B2M_SLOTS: the advance launch's own head)
  int n_classes; int class_nmax[B2M_MAX_CLASSES]; int class_cmax[B2M_MAX_CLASSES];
  int class_budget[B2M_MAX_CLASSES];   // solver-iteration budget of the class's thread-per-env launch (0: none); an env whose cost history reaches it goes to the hard queue instead
  int first_rung_handoff;      // != 0: the thread-per-env classes hand on an env whose first lcp_fast rung does not verify (EnvCtx)
  // debug taps (may be null)
  double* tap_MM; double* tap_qq; double* tap_z; int* tap_n;
  // reduced-coordinate articulated body (null / 0 when the scene has none)
  const RCTree* rc; int rc_links, rc_first;
  int ngc;                     // > 0: dense generalized-coordinate layout of the problem data (scenes with an articulated body); largest island dimension
  double* jq; double* jqd; const double* jtau;   // [dof][env]
  // working sets that do not fit an SM's shared memory (many-body scenes, LCP n in the hundreds) live in global
  // memory instead, one slice per resident thread group: slice g starts at gscratch + g * gstride (doubles)
  double* gscratch; size_t gstride;
  // per-kernel accounting: kstat[3 * kslot + {0,1,2}] += envs processed, algorithmic flops (pivot + assembly), LCP solves
  unsigned long long* kstat; int kslot;
  int* env_stat;               // optional [5][env]: LCP failures, lcp_lemke calls, lcp_fast calls, LCP solves, pivots of each env since the tap was armed (parity tests)
  int tap_times;               // debug: tap_prof rows PH_ISLANDS / PH_STORE hold global-timer start / end of the env's impact (B200MOBY_TAP_TIMES=1)
  long long* tap_prof;         // [4 + PH_COUNT][env]: SM cycles, pivots, executed iterations, LCP n of the env's last impact phase, then cycles per phase
};

// Per-env working set carved out of one contiguous block of doubles + ints (shared memory for warp groups).
struct EnvMem {
  // doubles
  double *bx, *bq, *bR, *bvl, *bva, *bmass, *bdims, *bJ, *xsave, *qsave;
  double *pd_dist, *pd_pa, *pd_pb;
  double *cp, *cnrm, *ct1, *ct2, *cdist, *cmu, *cmuv, *ceps, *ccomp;
  double *Jr, *XJ, *Xb, *D, *Cv, *imp, *acc, *dv;
  double *MM, *qq, *z, *zl, *vl, *work;
  double *Lf, *gv;             // dense layout: Cholesky factor scratch (ngc^2 + ngc), generalized velocity of the island (ngc)
  double *jq, *jqd, *jqsave, *jtau, *rS, *rV;   // articulated body: joint state, motion subspaces and spatial velocities of the links (world)
  // ints
  int *bshape, *ben, *pair_a, *pair_b, *cb1, *cb2, *cNK, *icon, *cisl, *corder, *isl_start, *gcoff, *bisl, *frow_c, *frow_j, *scal, *iwork;
  int *ranc, *gcb, *gcl;       // articulated body: ancestor-joint bitmask per link; island coordinate -> (super body, local index)
  long long* prof; long long prof_stride;   // debug: per-phase cycle accumulators of the env being processed (null: off)
  const double* wtab;                       // SimParams::fr_tab + B2M_WTAB_OFF
  long long dbg[4];                         // debug (timeline taps): worst pick-up delay / run time (us), rungs consumed, rungs that hit the pivot cap
  double cdt;                               // SimParams::contact_dist_thresh (the rimless wheel's contact generator reads the simulator's, whatever TOL its caller passes)
};

// phase ids of the impact profile (rows 4.. of SimParams::tap_prof)
enum { PH_LOAD = 0, PH_CONTACTS, PH_ISLANDS, PH_PROBLEM, PH_BUILD, PH_FAST, PH_LEMKE, PH_APPLY, PH_STORE, PH_COUNT };
#ifdef __CUDA_ARCH__
#define B2M_PROF_T0(m) const long long _pt0 = (m).prof ? clock64() : 0
#define B2M_PROF_ADD(m, g, k) do { if ((m).prof && (g).tid == 0) (m).prof[(k) * (m).prof_stride] += clock64() - _pt0; } while (0)
#else
#define B2M_PROF_T0(m) do {} while (0)
#define B2M_PROF_ADD(m, g, k) do {} while (0)
#endif

// The working set has two segments.  "small": bodies, pair distances and the contact list -- all that the advance
// phase (positions, forward dynamics, narrowphase) touches.  "impact": Jacobian rows, Delassus blocks, the LCP and the
// solver's work space -- only envs with an impacting contact ever need it, and it is sized by the env's own LCP class.
struct EnvDims {
  int nb, cmax, nmax, npmax;
  int rcl;      // links of the articulated body (0: none)
  int ngc;      // dense problem-data layout with this many generalized coordinates (0: two 6-wide blocks per contact)
};
B2M_HD inline EnvDims env_dims(const SimParams& P) { EnvDims d; d.nb = P.nb; d.cmax = P.cmax; d.nmax = P.nmax; d.npmax = P.npmax; d.rcl = P.rc_links; d.ngc = P.ngc; return d; }
B2M_HD inline size_t env_small_doubles(const EnvDims& d) { return (size_t)38 * d.nb + 7 * (size_t)d.npmax + 17 * (size_t)d.cmax + (d.rcl ? (size_t)4 * (d.rcl - 1) + 12 * (size_t)d.rcl : 0); }
B2M_HD inline size_t env_small_ints(const EnvDims& d) { return (size_t)2 * d.nb + 2 * (size_t)d.npmax + 3 * (size_t)d.cmax + 16 + (size_t)d.rcl; }
B2M_HD inline size_t env_impact_doubles(const EnvDims& d) {
  size_t lw = lemke_work_doubles(d.nmax), fw = fast_work_doubles(d.nmax);
  const size_t jac = d.ngc ? (size_t)6 * d.cmax * d.ngc + 2 * (size_t)d.ngc * d.ngc + 3 * (size_t)d.ngc : 72 * (size_t)d.cmax + 36 * (size_t)d.nb + 6 * (size_t)d.nb;
  return jac + 6 * (size_t)d.cmax * d.cmax + 10 * (size_t)d.cmax + (size_t)d.nmax * d.nmax + 3 * (size_t)d.nmax + (lw > fw ? lw : fw);
}
B2M_HD inline size_t env_impact_ints(const EnvDims& d) {
  size_t lw = lemke_work_ints(d.nmax), fw = fast_work_ints(d.nmax);
  return (size_t)3 * d.nb + 1 + 3 * (size_t)d.cmax + 2 * (size_t)d.nmax + 2 * (size_t)d.ngc + (lw > fw ? lw : fw);
}
B2M_HD inline size_t env_doubles(const EnvDims& d) { return env_small_doubles(d) + env_impact_doubles(d); }
B2M_HD inline size_t env_ints(const EnvDims& d) { return env_small_ints(d) + env_impact_ints(d); }

B2M_HD inline void env_carve_small(EnvMem& m, double* d, int* i, const EnvDims& D) {
  const int nb = D.nb, cmax = D.cmax, npmax = D.npmax;
  m.bx = d; d += 3 * nb; m.bq = d; d += 4 * nb; m.bR = d; d += 9 * nb; m.bvl = d; d += 3 * nb; m.bva = d; d += 3 * nb;
  m.bmass = d; d += nb; m.bdims = d; d += 3 * nb; m.bJ = d; d += 3 * nb; m.xsave = d; d += 3 * nb; m.qsave = d; d += 4 * nb;
  m.pd_dist = d; d += npmax; m.pd_pa = d; d += 3 * npmax; m.pd_pb = d; d += 3 * npmax;
  m.cp = d; d += 3 * cmax; m.cnrm = d; d += 3 * cmax; m.ct1 = d; d += 3 * cmax; m.ct2 = d; d += 3 * cmax;
  m.cdist = d; d += cmax; m.cmu = d; d += cmax; m.cmuv = d; d += cmax; m.ceps = d; d += cmax; m.ccomp = d; d += cmax;
  m.jq = m.jqd = m.jqsave = m.jtau = m.rS = m.rV = nullptr;
  if (D.rcl) { const int nd = D.rcl - 1; m.jq = d; d += nd; m.jqd = d; d += nd; m.jqsave = d; d += nd; m.jtau = d; d += nd; m.rS = d; d += 6 * D.rcl; m.rV = d; d += 6 * D.rcl; }
  m.bshape = i; i += nb; m.ben = i; i += nb;
  m.pair_a = i; i += npmax; m.pair_b = i; i += npmax;
  m.cb1 = i; i += cmax; m.cb2 = i; i += cmax; m.cNK = i; i += cmax;
  m.scal = i; i += 16;
  m.ranc = i; i += D.rcl;
  m.Jr = nullptr; m.zl = nullptr; m.vl = nullptr; m.prof = nullptr; m.prof_stride = 0; m.gcb = m.gcl = nullptr; m.cdt = 0.0; m.wtab = nullptr;
}
B2M_HD inline void env_carve_impact(EnvMem& m, double* d, int* i, const EnvDims& D) {
  const int nb = D.nb, cmax = D.cmax, nmax = D.nmax;
  if (D.ngc) { m.Jr = d; d += (size_t)3 * cmax * D.ngc; m.XJ = d; d += (size_t)3 * cmax * D.ngc; m.Xb = d; d += (size_t)D.ngc * D.ngc; m.dv = d; d += D.ngc; m.Lf = d; d += (size_t)D.ngc * D.ngc + D.ngc; m.gv = d; d += D.ngc; }
  else { m.Lf = m.gv = nullptr; m.Jr = d; d += 36 * cmax; m.XJ = d; d += 36 * cmax; m.Xb = d; d += 36 * nb; m.dv = d; d += 6 * nb; }
  m.D = d; d += 6 * (size_t)cmax * cmax;
  m.Cv = d; d += 3 * cmax; m.imp = d; d += 3 * cmax; m.acc = d; d += 3 * cmax;
  m.MM = d; d += (size_t)nmax * nmax; m.qq = d; d += nmax; m.z = d; d += nmax; m.zl = d; d += nmax; m.vl = d; d += cmax; m.work = d;
  m.gcoff = i; i += nb; m.bisl = i; i += nb;
  m.icon = i; i += cmax; m.cisl = i; i += cmax; m.corder = i; i += cmax;
  m.isl_start = i; i += nb + 1;
  m.frow_c = i; i += nmax; m.frow_j = i; i += nmax;
  m.gcb = i; i += D.ngc; m.gcl = i; i += D.ngc;
  m.iwork = i;
}
B2M_HD inline void env_carve(EnvMem& m, double* d, int* i, const EnvDims& D) {
  env_carve_small(m, d, i, D);
  env_carve_impact(m, d + env_small_doubles(D), i + env_small_ints(D), D);
}

// scal[] slots
enum { S_NPAIRS = 0, S_NCON = 1, S_NC = 2, S_NGC = 3, S_N = 4, S_NISL = 5, S_FLAG = 6, S_TMP = 7, S_ZLN = 8, S_ZLDIRTY = 9, S_NTOT = 10, S_VLN = 11, S_VLDIRTY = 12, S_FAILED = 13, S_EXEC = 14 };

// Per-env solver budget: when `limit` is set and an env's pivots in this launch exceed it, the env's step is
// abandoned without touching its stored state and the env is queued for the block-per-env kernel, which redoes the
// step with many more threads per pivot (same arithmetic, same results).  Keeps one hard LCP from holding a whole SM.
// first_rung: a one-thread group under a budget (the thread-per-env classes) also hands its env on as soon as the first
// rung of the lcp_fast ladder does not verify.  Such an env has three more rungs and maybe the Lemke ladder ahead, work
// that holds up the 31 other envs of its warp; the hard-queue launch running next to the classes takes it at once.
struct EnvCtx {
  int budget; bool limit;
  void* ladder = nullptr;      // LadderCtx of an impact_warp_kernel warp (the rungs of the Lemke ladder become tasks other warps take, lcp_device.cuh)
  bool first_rung = true;
};

// per-env solver statistics (SimParams::env_stat): the counters an env added to `lc` since `base` was taken
struct EnvStatBase { unsigned long long fail, lemke, fast, solves, pivots; };
B2M_HD B2M_INL EnvStatBase env_stat_base(const unsigned long long* lc);

B2M_HD B2M_INL EnvStatBase env_stat_base(const unsigned long long* lc) {
  EnvStatBase b; b.fail = lc[CNT_LCP_FAIL] + lc[CNT_OVERFLOW]; b.lemke = lc[CNT_LEMKE_CALLS]; b.fast = lc[CNT_FAST_CALLS]; b.solves = lc[CNT_LCP_SOLVES]; b.pivots = lc[CNT_PIVOTS]; return b;
}
template <class G>
B2M_DEV B2M_INL void env_stat_commit(const G& g, const SimParams& P, int e, const unsigned long long* lc, const EnvStatBase& b) {
  if (!P.env_stat || g.tid != 0) return;
  const size_t ne = P.n_envs;
  P.env_stat[e] += (int)(lc[CNT_LCP_FAIL] + lc[CNT_OVERFLOW] - b.fail);
  P.env_stat[ne + e] += (int)(lc[CNT_LEMKE_CALLS] - b.lemke);
  P.env_stat[2 * ne + e] += (int)(lc[CNT_FAST_CALLS] - b.fast);
  P.env_stat[3 * ne + e] += (int)(lc[CNT_LCP_SOLVES] - b.solves);
  P.env_stat[4 * ne + e] += (int)(lc[CNT_PIVOTS] - b.pivots);
}

// ---------- geometry helpers (same formulas, same order as the CPU checker) ----------
B2M_HD B2M_INL void quat_to_R(const double* qt, double* R) {
  const double x = qt[0], y = qt[1], z = qt[2], w = qt[3];
  R[0] = 1.0 - 2.0 * (y * y + z * z); R[1] = 2.0 * (x * y - w * z);       R[2] = 2.0 * (x * z + w * y);
  R[3] = 2.0 * (x * y + w * z);       R[4] = 1.0 - 2.0 * (x * x + z * z); R[5] = 2.0 * (y * z - w * x);
  R[6] = 2.0 * (x * z - w * y);       R[7] = 2.0 * (y * z + w * x);       R[8] = 1.0 - 2.0 * (x * x + y * y);
}
B2M_HD B2M_INL V3 box_vertex(const double* dims, int i) {   // BoxPrimitive.cpp:358-365 order
  const double X = dims[0] * 0.5, Y = dims[1] * 0.5, Z = dims[2] * 0.5;
  return V3((i & 4) ? -X : X, (i & 2) ? -Y : Y, (i & 1) ? -Z : Z);
}
struct BodyRef {
  const double *x, *R, *vl, *va, *dims; int shape, enabled;
  const double* wtab;   // spoke directions (EnvMem::wtab)
};
B2M_HD B2M_INL BodyRef body_ref(const EnvMem& m, int b) {
  BodyRef r; r.x = m.bx + 3 * b; r.R = m.bR + 9 * b; r.vl = m.bvl + 3 * b; r.va = m.bva + 3 * b; r.dims = m.bdims + 3 * b;
  r.shape = m.bshape[b]; r.enabled = m.ben[b]; r.wtab = m.wtab; return r;
}
B2M_HD B2M_INL V3 to_global(const BodyRef& b, const V3& p) { return ld3(b.x) + rot(b.R, p); }
B2M_HD B2M_INL V3 to_local(const BodyRef& b, const V3& p) { return rotT(b.R, p - ld3(b.x)); }
B2M_HD B2M_INL V3 point_vel(const BodyRef& b, const V3& p) {
  if (!b.enabled) return V3();
  return ld3(b.vl) + cross(ld3(b.va), p - ld3(b.x));
}
B2M_HD B2M_INL V3 lin_vel(const BodyRef& b) { return b.enabled ? ld3(b.vl) : V3(); }
B2M_HD B2M_INL V3 ang_vel(const BodyRef& b) { return b.enabled ? ld3(b.va) : V3(); }

}  // namespace b2m
#include "boxbox_device.cuh"
namespace b2m {

B2M_HD B2M_NOINL inline double box_closest_point(const double* dims, const V3& point, V3& closest) {   // BoxPrimitive.cpp:788-836
  const double ext[3] = {dims[0] * 0.5, dims[1] * 0.5, dims[2] * 0.5};
  const double pt[3] = {point.x, point.y, point.z};
  double cl[3] = {point.x, point.y, point.z};
  bool inside = true;
  double sqrDist = 0.0, intDist = -B2M_INF, delta;
  for (int i = 0; i < 3; i++) {
    if (pt[i] < -ext[i]) { delta = pt[i] + ext[i]; cl[i] = -ext[i]; sqrDist += delta * delta; inside = false; }
    else if (pt[i] > ext[i]) { delta = pt[i] - ext[i]; cl[i] = ext[i]; sqrDist += delta * delta; inside = false; }
    else if (inside) { const double d = -fmin(fabs(ext[i] - pt[i]), fabs(pt[i] + ext[i])); intDist = fmax(intDist, d); }
  }
  closest = V3(cl[0], cl[1], cl[2]);
  return inside ? intDist : sqrt(sqrDist);
}

// signed distance + closest points for an ordered pair (PlanePrimitive.cpp:342-411, SpherePrimitive.cpp:104-135, BoxPrimitive.cpp:257-276)
B2M_HD B2M_NOINL inline bool signed_dist_ordered(const BodyRef& A, const BodyRef& B, double& dist, V3& pA, V3& pB) {
  if (A.shape == SH_PLANE && B.shape == SH_BOX) {
    double min_dist = B2M_INF; V3 pb_best, pthis;
    for (int i = 0; i < 8; i++) {
      const V3 vg = to_global(B, box_vertex(B.dims, i));
      const V3 pv = to_local(A, vg);
      if (pv.y < min_dist) { min_dist = pv.y; pb_best = vg; pthis = pv; }
    }
    pthis.y = 0.0;
    dist = min_dist; pA = to_global(A, pthis); pB = pb_best;
    return true;
  }
  if (A.shape == SH_PLANE && B.shape == SH_SPHERE) {
    const V3 c = to_local(A, ld3(B.x));
    const V3 lowest(c.x, c.y - B.dims[0], c.z);
    const V3 pthis(c.x, 0.0, c.z);
    dist = lowest.y; pA = to_global(A, pthis); pB = to_global(A, lowest);
    return true;
  }
  if (A.shape == SH_SPHERE && B.shape == SH_SPHERE) {
    const V3 d = ld3(B.x) - ld3(A.x);
    const double len = norm(d);
    const double dd = len - A.dims[0] - B.dims[0];
    const V3 u = d * (1.0 / len);
    const double sa = (dd > 0.0) ? A.dims[0] : A.dims[0] + dd, sb = (dd > 0.0) ? B.dims[0] : B.dims[0] + dd;
    dist = dd; pA = ld3(A.x) + u * sa; pB = ld3(B.x) - u * sb;
    return true;
  }
  if (A.shape == SH_BOX && B.shape == SH_SPHERE) {
    const V3 c = to_local(A, ld3(B.x)); V3 pbox;
    dist = box_closest_point(A.dims, c, pbox) - B.dims[0];
    const V3 pbox_g = to_global(A, pbox);
    const V3 v = pbox_g - ld3(B.x);
    const double vnorm = norm(v);
    pA = pbox_g;
    pB = (vnorm == 0.0) ? ld3(B.x) : ld3(B.x) + v * ((B.dims[0] + fmin(dist, 0.0)) / vnorm);
    return true;
  }
  if (B2M_BOXBOX && A.shape == SH_BOX && B.shape == SH_BOX) { boxbox_signed_dist(A, B, dist, pA, pB); return true; }   // rule H5 (boxbox_device.cuh)
  return false;
}
// Spoke tip i of the rimless wheel, side s (+1: y = +W/2, -1: y = -W/2), in the wheel frame (coldet-plugin.cpp:110-115)
B2M_HD B2M_INL V3 wheel_tip(const BodyRef& Wh, int i, int s) {
  const double* cs = Wh.wtab + 2 * ((size_t)(int)Wh.dims[2] * B2M_WHEEL_NS_MAX + i);   // host libm cos / sin of M_PI * i * 2.0 / N_SPOKES
  return V3(cs[0] * Wh.dims[0], s * (Wh.dims[1] * .5), cs[1] * Wh.dims[0]);
}
// BladePlanePlugin::calc_signed_dist_wheel_plane (coldet-plugin.cpp:86-137): lowest spoke tip over the plane
B2M_HD B2M_NOINL inline double wheel_plane_signed_dist(const BodyRef& Wh, const BodyRef& P, V3& pwheel, V3& pground) {
  double min_dist = B2M_INF;
  const int ns = (int)Wh.dims[2];
  for (int i = 0; i < ns; i++)
    for (int s = 1; s >= -1; s -= 2) {                         // p1 then p2; strict test, so p2 never wins when W = 0
      const V3 pg = to_global(Wh, wheel_tip(Wh, i, s));
      V3 pp = to_local(P, pg);
      if (pp.y < min_dist) { min_dist = pp.y; pp.y = 0.0; pground = to_global(P, pp); pwheel = pg; }
    }
  return min_dist;
}
B2M_HD inline bool signed_dist(const BodyRef& A, const BodyRef& B, double& dist, V3& pA, V3& pB) {
  // coldet-plugin.cpp:324-334: both argument orders hand (pA, pB) to (pwheel, pground); with the pair the plugin queues,
  // (ground, wheel) (:70), the point reported for the ground is the wheel's and vice versa.  Literal.
  // contact-constrained-pendulum-coldet-plugin.cpp:60-75,140-150: minus the distance from the link's anchor point to the world body's origin
  if ((A.shape == SH_PIN && B.shape == SH_PINWORLD) || (A.shape == SH_PINWORLD && B.shape == SH_PIN)) {
    const BodyRef& L = (A.shape == SH_PIN) ? A : B; const BodyRef& W = (A.shape == SH_PIN) ? B : A;
    pA = to_global(L, V3(L.dims[0], L.dims[1], L.dims[2])); pB = ld3(W.x);
    dist = -norm(to_local(W, pA));
    return true;
  }
  if (A.shape == SH_WHEEL && B.shape == SH_PLANE) { dist = wheel_plane_signed_dist(A, B, pA, pB); return true; }
  if (A.shape == SH_PLANE && B.shape == SH_WHEEL) { dist = wheel_plane_signed_dist(B, A, pA, pB); return true; }
  if (signed_dist_ordered(A, B, dist, pA, pB)) return true;
  if (signed_dist_ordered(B, A, dist, pB, pA)) return true;
  return false;
}

B2M_HD B2M_NOINL inline void orthonormal_basis(const V3& v1, V3& v2, V3& v3) {   // Ravelin Vector3d::determine_orthonormal_basis
  const double x = fabs(v1.x), y = fabs(v1.y), z = fabs(v1.z);
  V3 a;
  if (x < y) { if (x < z) a = V3(1, 0, 0); else a = V3(0, 0, 1); }
  else       { if (y < z) a = V3(0, 1, 0); else a = V3(0, 0, 1); }
  v2 = normalize(cross(v1, a));
  v3 = normalize(cross(v1, v2));
}

struct ContactOut { V3 p, n; int b1, b2; double dist; };

// Contacts of one pair, at most `cap` (CCD.inl:3-82 dispatch and leaves).  Executed by ONE thread; returns the count found.
B2M_HD B2M_NOINL inline int pair_contacts(const EnvMem& m, int ia, int ib, double TOL, ContactOut* out, int cap) {
  const BodyRef A = body_ref(m, ia), B = body_ref(m, ib);
  int cnt = 0;
  if ((A.shape == SH_PIN && B.shape == SH_PINWORLD) || (A.shape == SH_PINWORLD && B.shape == SH_PIN)) {   // contact-constrained-pendulum-coldet-plugin.cpp:78-110
    const int il = (A.shape == SH_PIN) ? ia : ib, iw = (A.shape == SH_PIN) ? ib : ia;
    const BodyRef L = body_ref(m, il);
    const V3 p = to_global(L, V3(L.dims[0], L.dims[1], L.dims[2]));
    const V3 point = (p + V3(0, 0, 0)) * 0.5;                  // midpoint of the anchor point and the GLOBAL origin
    for (int k = 0; k < 6; k++) {                              // normals +y -y +z -z +x -x; violation min(0, -p_k) for both normals of an axis
      const int ax = k < 2 ? 1 : (k < 4 ? 2 : 0);
      const double sg = (k & 1) ? -1.0 : 1.0, pk = ax == 0 ? p.x : (ax == 1 ? p.y : p.z);
      if (cnt < cap) { out[cnt].p = point; out[cnt].n = V3(ax == 0 ? sg : 0.0, ax == 1 ? sg : 0.0, ax == 2 ? sg : 0.0); out[cnt].b1 = il; out[cnt].b2 = iw; out[cnt].dist = fmin(0.0, -pk); }
      cnt++;
    }
    return cnt;
  }
  if ((A.shape == SH_WHEEL && B.shape == SH_PLANE) || (A.shape == SH_PLANE && B.shape == SH_WHEEL)) {     // coldet-plugin.cpp:222-310
    const int iw = (A.shape == SH_WHEEL) ? ia : ib, ip = (A.shape == SH_WHEEL) ? ib : ia;
    const BodyRef Wh = body_ref(m, iw), P = body_ref(m, ip);
    const V3 n = rot(P.R, V3(0, 1, 0));
    const int ns = (int)Wh.dims[2];
    for (int i = 0; i < ns; i++)
      for (int s = 1; s >= -1; s -= 2) {
        if (s < 0 && !(Wh.dims[1] > 0.0)) continue;            // :283
        const V3 pg = to_global(Wh, wheel_tip(Wh, i, s));
        V3 pp = to_local(P, pg);
        const double h = pp.y;
        if (!(h < m.cdt)) continue;                            // the plugin ignores the caller's TOL: `< sim->contact_dist_thresh` (:225,:270)
        pp.y = 0.0;
        if (cnt < cap) { out[cnt].p = (pg + to_global(P, pp)) * 0.5; out[cnt].n = n; out[cnt].b1 = iw; out[cnt].b2 = ip; out[cnt].dist = h; }
        cnt++;
      }
    return cnt;
  }
  if ((A.shape == SH_SPHERE && B.shape == SH_PLANE) || (A.shape == SH_PLANE && B.shape == SH_SPHERE)) {   // CCD.inl:805-846
    const int is = (A.shape == SH_SPHERE) ? ia : ib, ip = (A.shape == SH_SPHERE) ? ib : ia;
    const BodyRef S = body_ref(m, is), P = body_ref(m, ip);
    const V3 c = to_local(P, ld3(S.x));
    const double dist = c.y - S.dims[0];
    if (dist > TOL) return 0;
    const V3 p(c.x, 0.5 * (c.y - S.dims[0]), c.z);
    if (cnt < cap) { out[cnt].p = to_global(P, p); out[cnt].n = rot(P.R, V3(0, 1, 0)); out[cnt].b1 = is; out[cnt].b2 = ip; out[cnt].dist = dist; }
    return cnt + 1;
  }
  if ((A.shape == SH_BOX && B.shape == SH_PLANE) || (A.shape == SH_PLANE && B.shape == SH_BOX)) {         // CCD.inl:850-886
    const int ix = (A.shape == SH_BOX) ? ia : ib, ip = (A.shape == SH_BOX) ? ib : ia;
    const BodyRef X = body_ref(m, ix), P = body_ref(m, ip);
    const V3 n = rot(P.R, V3(0, 1, 0));
    for (int i = 0; i < 8; i++) {
      const V3 vg = to_global(X, box_vertex(X.dims, i));
      const double dist = to_local(P, vg).y;
      if (dist <= TOL) {
        if (cnt < cap) { out[cnt].p = vg; out[cnt].n = -n; out[cnt].b1 = ip; out[cnt].b2 = ix; out[cnt].dist = dist; }
        cnt++;
      }
    }
    return cnt;
  }
  if (A.shape == SH_SPHERE && B.shape == SH_SPHERE) {                                                      // CCD.inl:1165-1206
    const V3 d = ld3(A.x) - ld3(B.x);
    const double dist = norm(d) - A.dims[0] - B.dims[0];
    if (dist > TOL) return 0;
    const V3 n = normalize(d);
    const V3 closest_A = ld3(A.x) - n * A.dims[0], closest_B = ld3(B.x) + n * B.dims[0];
    if (cnt < cap) { out[cnt].p = (closest_A + closest_B) * 0.5; out[cnt].n = n; out[cnt].b1 = ia; out[cnt].b2 = ib; out[cnt].dist = dist; }
    return cnt + 1;
  }
  if ((A.shape == SH_BOX && B.shape == SH_SPHERE) || (A.shape == SH_SPHERE && B.shape == SH_BOX)) {        // CCD.inl:1210-1259
    const int ix = (A.shape == SH_BOX) ? ia : ib, is = (A.shape == SH_BOX) ? ib : ia;
    const BodyRef X = body_ref(m, ix), S = body_ref(m, is);
    const double HX = X.dims[0] * 0.5, HY = X.dims[1] * 0.5, HZ = X.dims[2] * 0.5, Rr = S.dims[0];
    const V3 c = to_local(X, ld3(S.x));
    const V3 pbox(fmin(fmax(c.x, -HX), HX), fmin(fmax(c.y, -HY), HY), fmin(fmax(c.z, -HZ), HZ));
    const V3 pbox_g = to_global(X, pbox);
    V3 psph = rotT(S.R, pbox_g - ld3(S.x));
    const double psph_nrm = norm(psph);
    double dist;
    if (fabs(pbox.x) < HX || fabs(pbox.y) < HY || fabs(pbox.z) < HZ || psph_nrm < Rr) {
      const double box_dist = fmin(HX - fabs(pbox.x), fmin(HY - fabs(pbox.y), HZ - fabs(pbox.z)));
      dist = -fmin(box_dist, Rr - psph_nrm);
    } else {
      psph = psph * (Rr / psph_nrm);
      dist = norm(to_local(X, to_global(S, psph)) - pbox);
    }
    if (dist > TOL) return 0;
    const V3 psph_g = to_global(S, psph);
    V3 p, normal;
    if (dist > 0.0) {
      p = (psph_g + pbox_g) * 0.5;
      normal = pbox_g - psph_g;
      const double nrm = norm(normal);
      if (nrm > B2M_NEAR_ZERO) normal = normal * (1.0 / nrm);
      else normal = normalize(rot(S.R, psph));
    } else {
      p = psph_g;
      normal = normalize(rot(S.R, psph));
    }
    if (cnt < cap) { out[cnt].p = p; out[cnt].n = normal; out[cnt].b1 = ix; out[cnt].b2 = is; out[cnt].dist = dist; }
    return cnt + 1;
  }
  if (B2M_BOXBOX && A.shape == SH_BOX && B.shape == SH_BOX) {                                                            // CCD.inl:86-494, rule H5
    V3 pts[8], normal; double depth[8];
    const int k = boxbox_contacts(A, B, TOL, pts, depth, normal);
    for (int i = 0; i < k; i++) {
      if (cnt < cap) { out[cnt].p = pts[i]; out[cnt].n = normal; out[cnt].b1 = ia; out[cnt].b2 = ib; out[cnt].dist = depth[i]; }
      cnt++;
    }
    return cnt;
  }
  return 0;
}

B2M_HD B2M_INL double contact_vel(const EnvMem& m, const ContactOut& c) {   // UnilateralConstraint.cpp:695-747
  const V3 ta = point_vel(body_ref(m, c.b1), c.p), tb = point_vel(body_ref(m, c.b2), c.p);
  return dot(c.n, ta - tb);
}

B2M_HD B2M_INL double calc_max_dist(const BodyRef& rb, const V3& n, double rmax) {   // CCD.cpp:585-607 (velocity taken at the GLOBAL origin)
  if (!rb.enabled) return 0.0;
  const V3 xd0 = ld3(rb.vl) - cross(ld3(rb.va), ld3(rb.x));
  return dot(n, xd0) + norm(cross(ld3(rb.va), n)) * rmax;
}
B2M_HD B2M_INL double calc_rmax(const BodyRef& b) {                                  // CCD.cpp:1023-1101
  if (b.shape == SH_SPHERE) return b.dims[0];
  if (b.shape == SH_BOX) return sqrt((b.dims[0] / 2.0) * (b.dims[0] / 2.0) + (b.dims[1] / 2.0) * (b.dims[1] / 2.0) + (b.dims[2] / 2.0) * (b.dims[2] / 2.0));
  return 0.0;   // SH_WHEEL too: the plugin keeps the wheel out of CCD::broad_phase (coldet-plugin.cpp:53-67), so _rmax[wheel_cg] stays the map default
}
B2M_HD B2M_INL bool rel_equal(double x, double y) { return fabs(x - y) <= B2M_NEAR_ZERO * fmax(fabs(x), fmax(fabs(y), 1.0)); }
B2M_HD B2M_INL bool collinear(const V3& a, const V3& b, const V3& c) {               // CompGeom.cpp:1923-1931
  return rel_equal((c.z - a.z) * (b.y - a.y), (b.z - a.z) * (c.y - a.y)) &&
         rel_equal((b.z - a.z) * (c.x - a.x), (b.x - a.x) * (c.z - a.z)) &&
         rel_equal((b.x - a.x) * (c.y - a.y), (b.y - a.y) * (c.x - a.x));
}
B2M_HD B2M_NOINL inline double next_CA_box_plane(const BodyRef& box, const V3& rv_lin, const V3& rv_ang, const V3& normal, double offset0) {   // CCD.cpp:407-460
  double max_step = B2M_INF;
  const V3 nP = rotT(box.R, normal);
  const V3 p0 = normal * offset0;
  const double offset = dot(nP, to_local(box, p0));
  const double av_norm = norm(rv_ang);
  const double lv_dot_n = -dot(nP, rv_lin);
  for (int i = 0; i < 8; i++) {
    const V3 vtx = box_vertex(box.dims, i);
    const double r = norm(vtx);
    const double dist = dot(nP, vtx) - offset;
    if (dist < B2M_NEAR_ZERO) continue;
    const double speed = fmax(0.0, lv_dot_n + av_norm * r);
    max_step = fmin(max_step, dist / speed);
  }
  return max_step;
}

// CCD::calc_CA_Euler_step for one pair (CCD.cpp:122-400).  Executed by ONE thread.
B2M_HD B2M_NOINL inline double pair_CA(const EnvMem& m, int p) {
  const int ia = m.pair_a[p], ib = m.pair_b[p];
  const BodyRef A = body_ref(m, ia), B = body_ref(m, ib);
  const double pdist = m.pd_dist[p];
  if (pdist == B2M_INF) return B2M_INF;
  ContactOut con[8];
  if (A.shape == SH_SPHERE || B.shape == SH_SPHERE) {                       // :138-166
    if (!(pdist > B2M_NEAR_ZERO)) {
      const int nc = pair_contacts(m, ia, ib, B2M_NEAR_ZERO, con, 8);
      if (nc == 1 && fabs(contact_vel(m, con[0])) < B2M_NEAR_ZERO * 10) return B2M_INF;
    }
  }
  if (pdist <= 0.0 && (A.shape == SH_WHEEL || B.shape == SH_WHEEL || A.shape == SH_PIN || B.shape == SH_PIN)) return B2M_INF;   // both plugins override calc_next_CA_Euler_step
  if (pdist <= 0.0) {                                                       // :189-190 -> :238-400
    const int nc = pair_contacts(m, ia, ib, B2M_NEAR_ZERO, con, 8);
    if (nc == 0) return B2M_INF;
    const double d = dot(con[0].n, con[0].p);
    for (int i = 0; i < nc; i++) if (contact_vel(m, con[i]) < -B2M_NEAR_ZERO) return 0.0;
    if (nc >= 3 && !collinear(con[0].p, con[1].p, con[2].p)) return B2M_INF;   // :288-330 (always points 0,1,2)
    const BodyRef gA = body_ref(m, con[0].b1), gB = body_ref(m, con[0].b2);
    if (gA.shape == SH_BOX && gB.shape == SH_PLANE) {
      const V3 rl = rotT(gA.R, lin_vel(gA)) - rotT(gA.R, point_vel(gB, ld3(gA.x)));
      const V3 ra = rotT(gA.R, ang_vel(gA) - ang_vel(gB));
      return next_CA_box_plane(gA, rl, ra, con[0].n, d);
    }
    if (gA.shape == SH_PLANE && gB.shape == SH_BOX) {
      const V3 rl = rotT(gB.R, point_vel(gA, ld3(gB.x))) - rotT(gB.R, lin_vel(gB));
      const V3 ra = rotT(gB.R, ang_vel(gA) - ang_vel(gB));
      return next_CA_box_plane(gB, -rl, -ra, -con[0].n, -d);
    }
    if (B2M_BOXBOX && gA.shape == SH_BOX && gB.shape == SH_BOX) {                          // CCD.cpp:350-364 -> :468-541
      const V3 wrel = ang_vel(gA) - ang_vel(gB);
      const V3 rlA = rotT(gA.R, lin_vel(gA) - point_vel(gB, ld3(gA.x))), rlB = rotT(gB.R, point_vel(gA, ld3(gB.x)) - lin_vel(gB));
      return next_CA_box_box(gA, gB, rlA, rotT(gA.R, wrel), rlB, rotT(gB.R, wrel), con[0].n, d);
    }
    return B2M_INF;
  }
  const V3 d0 = ld3(m.pd_pa + 3 * p) - ld3(m.pd_pb + 3 * p);               // :193-229
  const double d0_norm = norm(d0);
  const V3 n0 = d0 * (1.0 / d0_norm);
  const double tA = calc_max_dist(A, -n0, calc_rmax(A));
  const double tB = calc_max_dist(B, n0, calc_rmax(B));
  double total = tA + tB;
  if (total < 0.0) total = 0.0;
  return fmin(B2M_INF, pdist / total);
}

// ---------- articulated body inside the env working set ----------
// Links are bodies [rc_first, rc_first + rc_links); link 0 (the base) is a disabled body.  All moving links form ONE
// super body whose generalized coordinates are the joint positions (ImpactConstraintHandler.cpp:1905-1916 collects
// super bodies, :1817-1895 maps link wrenches through the link Jacobian); its representative in the island code is
// the first moving link.
B2M_HD B2M_INL bool is_link(const SimParams& P, int b) { return B2M_RC(P) > 0 && b > P.rc_first && b < P.rc_first + P.rc_links; }
B2M_HD B2M_INL int super_of(const SimParams& P, int b) { return is_link(P, b) ? P.rc_first + 1 : b; }

// link poses, motion subspaces, spatial and COM velocities from (jq, jqd): what RCArticulatedBodyd::update_link_poses /
// update_link_velocities do after set_generalized_coordinates / _velocity (RCArticulatedBody.cpp:102,142-143)
template <class G>
B2M_DEV B2M_NOINL void rc_refresh(const G& g, const SimParams& P, EnvMem& m) {
  if (g.tid == 0) {
    const RCTree& T = *P.rc;
    RCState s; s.x = m.bx + 3 * P.rc_first; s.R = m.bR + 9 * P.rc_first; s.S = m.rS; s.v = m.rV;
    rc_kinematics(T, m.jq, m.jqd, s);
    for (int i = 1; i < T.n_links; i++) rc_link_velocity(s, i, m.bvl + 3 * (P.rc_first + i), m.bva + 3 * (P.rc_first + i));
  }
  g.sync();
}

// ---------- env load / store ----------
template <class G>
B2M_DEV B2M_NOINL void env_load(const G& g, const SimParams& P, int e, EnvMem& m) {
  const int nb = P.nb, ne = P.n_envs;
  m.cdt = P.contact_dist_thresh; m.wtab = P.fr_tab + B2M_WTAB_OFF;
  if constexpr (G::size == 1) {
    // one thread per env: all 22 words of a body are requested before the first is stored (the element-wise loops below made
    // every global load wait for the local store before it -- ncu, UR10: 18 % of the thread-per-env impact launch sat here)
    for (int b = 0; b < nb; b++) {
      const size_t o = (size_t)b * ne + e;
      const double* qb = P.q + (size_t)b * 7 * ne + e; const double* vb = P.v + (size_t)b * 6 * ne + e;
      const double* db = P.dims + (size_t)b * 3 * ne + e; const double* jb = P.inertia + (size_t)b * 3 * ne + e;
      const int sh = P.shape[o], en = P.enabled[o];
      const double ms = P.mass[o];
      const double q0 = qb[0], q1 = qb[ne], q2 = qb[2 * (size_t)ne], q3 = qb[3 * (size_t)ne], q4 = qb[4 * (size_t)ne], q5 = qb[5 * (size_t)ne], q6 = qb[6 * (size_t)ne];
      const double v0 = vb[0], v1 = vb[ne], v2 = vb[2 * (size_t)ne], v3 = vb[3 * (size_t)ne], v4 = vb[4 * (size_t)ne], v5 = vb[5 * (size_t)ne];
      const double d0 = db[0], d1 = db[ne], d2 = db[2 * (size_t)ne], j0 = jb[0], j1 = jb[ne], j2 = jb[2 * (size_t)ne];
      m.bshape[b] = sh; m.ben[b] = en; m.bmass[b] = ms;
      m.bdims[3 * b] = d0; m.bdims[3 * b + 1] = d1; m.bdims[3 * b + 2] = d2; m.bJ[3 * b] = j0; m.bJ[3 * b + 1] = j1; m.bJ[3 * b + 2] = j2;
      m.bx[3 * b] = q0; m.bx[3 * b + 1] = q1; m.bx[3 * b + 2] = q2;
      m.bq[4 * b] = q3; m.bq[4 * b + 1] = q4; m.bq[4 * b + 2] = q5; m.bq[4 * b + 3] = q6;
      m.bvl[3 * b] = v0; m.bvl[3 * b + 1] = v1; m.bvl[3 * b + 2] = v2; m.bva[3 * b] = v3; m.bva[3 * b + 1] = v4; m.bva[3 * b + 2] = v5;
    }
  } else {
  for (int b = g.tid; b < nb; b += G::size) {
    m.bshape[b] = P.shape[(size_t)b * ne + e];
    m.ben[b] = P.enabled[(size_t)b * ne + e];
    m.bmass[b] = P.mass[(size_t)b * ne + e];
  }
  for (int k = g.tid; k < 3 * nb; k += G::size) { m.bdims[k] = P.dims[(size_t)k * ne + e]; m.bJ[k] = P.inertia[(size_t)k * ne + e]; }
  for (int k = g.tid; k < 3 * nb; k += G::size) { const int b = k / 3, c = k - 3 * b; m.bx[k] = P.q[((size_t)b * 7 + c) * ne + e]; }
  for (int k = g.tid; k < 4 * nb; k += G::size) { const int b = k / 4, c = k - 4 * b; m.bq[k] = P.q[((size_t)b * 7 + 3 + c) * ne + e]; }
  for (int k = g.tid; k < 3 * nb; k += G::size) { const int b = k / 3, c = k - 3 * b; m.bvl[k] = P.v[((size_t)b * 6 + c) * ne + e]; m.bva[k] = P.v[((size_t)b * 6 + 3 + c) * ne + e]; }
  }
  g.sync();
  // quaternions are stored normalised (b200moby_set_state does what set_generalized_coordinates_euler does)
  for (int b = g.tid; b < nb; b += G::size) quat_to_R(m.bq + 4 * b, m.bR + 9 * b);
  if (g.tid == 0) {                                              // all-pairs table (CollisionDetection.cpp:28-54, ConstraintSimulator.cpp:471-485)
    int np = 0;
    for (int i = 0; i < nb; i++)
      for (int j = i + 1; j < nb; j++) {
        if (!(m.ben[i] || m.ben[j])) continue;
        if (m.bshape[i] == SH_NONE || m.bshape[j] == SH_NONE) continue;
        if (P.NK[((size_t)i * nb + j) * ne + e] == 0) continue;
        m.pair_a[np] = i; m.pair_b[np] = j; np++;
      }
    m.scal[S_NPAIRS] = np;
    m.scal[S_ZLN] = P.zlast_n[e];
    m.scal[S_ZLDIRTY] = 0;
    m.scal[S_VLN] = P.vlast_n ? P.vlast_n[e] : 0;
    m.scal[S_VLDIRTY] = 0;
    if (B2M_RC(P)) { m.ranc[0] = 0; for (int i = 1; i < P.rc_links; i++) m.ranc[i] = m.ranc[P.rc->parent[i]] | (1 << i); }
  }
  if (B2M_RC(P)) {
    if constexpr (G::size == 1) {                                 // three joints (nine words) per batch: loads first
      const int nd = P.rc_links - 1;
      int k = 0;
      for (; k + 3 <= nd; k += 3) {
        const size_t o = (size_t)k * ne + e;
        const double a0 = P.jq[o], a1 = P.jq[o + ne], a2 = P.jq[o + 2 * (size_t)ne], b0 = P.jqd[o], b1 = P.jqd[o + ne], b2 = P.jqd[o + 2 * (size_t)ne];
        const double c0 = P.jtau[o], c1 = P.jtau[o + ne], c2 = P.jtau[o + 2 * (size_t)ne];
        m.jq[k] = a0; m.jq[k + 1] = a1; m.jq[k + 2] = a2; m.jqd[k] = b0; m.jqd[k + 1] = b1; m.jqd[k + 2] = b2; m.jtau[k] = c0; m.jtau[k + 1] = c1; m.jtau[k + 2] = c2;
      }
      for (; k < nd; k++) { m.jq[k] = P.jq[(size_t)k * ne + e]; m.jqd[k] = P.jqd[(size_t)k * ne + e]; m.jtau[k] = P.jtau[(size_t)k * ne + e]; }
    } else
    for (int k = g.tid; k < P.rc_links - 1; k += G::size) { m.jq[k] = P.jq[(size_t)k * ne + e]; m.jqd[k] = P.jqd[(size_t)k * ne + e]; m.jtau[k] = P.jtau[(size_t)k * ne + e]; }
    g.sync();
    rc_refresh(g, P, m);
  }
  g.sync();
  if (m.zl) {                                                   // ImpactConstraintHandler::_zlast, kept on chip for the whole launch
    const int zn = m.scal[S_ZLN];                               // a longer vector than this launch's LCP class can never match (H1: zero fill)
    if (zn <= P.nmax) for (int i = g.tid; i < zn; i += G::size) m.zl[i] = P.zlast[(size_t)i * ne + e];
    const int vn = m.scal[S_VLN];
    if (vn <= P.cmax) for (int i = g.tid; i < vn; i += G::size) m.vl[i] = P.vlast[(size_t)i * ne + e];
    g.sync();
  }
}

// what: 1 positions, 2 velocities, 4 warm start
enum { ST_POS = 1, ST_VEL = 2, ST_ZL = 4 };
template <class G>
B2M_DEV B2M_NOINL void env_store(const G& g, const SimParams& P, int e, const EnvMem& m, int what = ST_POS | ST_VEL | ST_ZL) {
  const int nb = P.nb, ne = P.n_envs;
  if (B2M_RC(P)) {
    if (what & ST_POS) for (int i = 1 + g.tid; i < P.rc_links; i += G::size) R_to_quat(m.bR + 9 * (P.rc_first + i), m.bq + 4 * (P.rc_first + i));
    for (int k = g.tid; k < P.rc_links - 1; k += G::size) {
      if (what & ST_POS) P.jq[(size_t)k * ne + e] = m.jq[k];
      if (what & ST_VEL) P.jqd[(size_t)k * ne + e] = m.jqd[k];
    }
    g.sync();
  }
  if constexpr (G::size == 1) {                                  // per body: read the local words first, then the global stores back to back
    for (int b = 0; b < nb; b++) {
      if (!m.ben[b]) continue;
      double* qb = P.q + (size_t)b * 7 * ne + e; double* vb = P.v + (size_t)b * 6 * ne + e;
      if (what & ST_POS) {
        const double q0 = m.bx[3 * b], q1 = m.bx[3 * b + 1], q2 = m.bx[3 * b + 2], q3 = m.bq[4 * b], q4 = m.bq[4 * b + 1], q5 = m.bq[4 * b + 2], q6 = m.bq[4 * b + 3];
        qb[0] = q0; qb[ne] = q1; qb[2 * (size_t)ne] = q2; qb[3 * (size_t)ne] = q3; qb[4 * (size_t)ne] = q4; qb[5 * (size_t)ne] = q5; qb[6 * (size_t)ne] = q6;
      }
      if (what & ST_VEL) {
        const double v0 = m.bvl[3 * b], v1 = m.bvl[3 * b + 1], v2 = m.bvl[3 * b + 2], v3 = m.bva[3 * b], v4 = m.bva[3 * b + 1], v5 = m.bva[3 * b + 2];
        vb[0] = v0; vb[ne] = v1; vb[2 * (size_t)ne] = v2; vb[3 * (size_t)ne] = v3; vb[4 * (size_t)ne] = v4; vb[5 * (size_t)ne] = v5;
      }
    }
  } else {
  for (int k = g.tid; k < 3 * nb; k += G::size) {
    const int b = k / 3, c = k - 3 * b;
    if (!m.ben[b]) continue;
    if (what & ST_POS) P.q[((size_t)b * 7 + c) * ne + e] = m.bx[k];
    if (what & ST_VEL) { P.v[((size_t)b * 6 + c) * ne + e] = m.bvl[k]; P.v[((size_t)b * 6 + 3 + c) * ne + e] = m.bva[k]; }
  }
  if (what & ST_POS) for (int k = g.tid; k < 4 * nb; k += G::size) { const int b = k / 4, c = k - 4 * b; if (m.ben[b]) P.q[((size_t)b * 7 + 3 + c) * ne + e] = m.bq[k]; }
  }
  if ((what & ST_ZL) && m.zl && m.scal[S_ZLDIRTY]) {
    const int zn = m.scal[S_ZLN];
    for (int i = g.tid; i < zn; i += G::size) P.zlast[(size_t)i * ne + e] = m.zl[i];
    if (g.tid == 0) P.zlast_n[e] = zn;
  }
  if ((what & ST_ZL) && m.vl && m.scal[S_VLDIRTY]) {
    const int vn = m.scal[S_VLN];
    for (int i = g.tid; i < vn; i += G::size) P.vlast[(size_t)i * ne + e] = m.vl[i];
    if (g.tid == 0) P.vlast_n[e] = vn;
  }
}

template <class G>
B2M_DEV B2M_NOINL void calc_pairwise_distances(const G& g, EnvMem& m) {       // ConstraintSimulator.cpp:450-468, one thread per pair
  const int np = m.scal[S_NPAIRS];
  for (int p = g.tid; p < np; p += G::size) {
    double dist; V3 pa, pb;
    if (!signed_dist(body_ref(m, m.pair_a[p]), body_ref(m, m.pair_b[p]), dist, pa, pb)) dist = B2M_INF;
    m.pd_dist[p] = dist; st3(m.pd_pa + 3 * p, pa); st3(m.pd_pb + 3 * p, pb);
  }
  g.sync();
}

// Simulator::precalc_fwd_dyn + calc_fwd_dyn for free bodies + v += h a (Simulator.cpp:319-350,482-602;
// TimeSteppingSimulator.cpp:181-192; GravityForce.cpp:32-48).  One thread per body.
template <class G>
B2M_DEV B2M_NOINL void fwd_dyn_integrate_velocity(const G& g, const SimParams& P, EnvMem& m, double h, double t) {
  if (B2M_RC(P)) {   // Simulator.cpp:339-348 controller, :544-553 RCArticulatedBodyd::calc_fwd_dyn (ABA or CRB), then qd += h qdd
    if (g.tid == 0) {
      const RCTree& T = *P.rc;
      const int nd = T.n_links - 1;
      RCState s; s.x = m.bx + 3 * P.rc_first; s.R = m.bR + 9 * P.rc_first; s.S = m.rS; s.v = m.rV;
      double tau[B2M_MAX_LINKS], qdd[B2M_MAX_LINKS], Hw[(B2M_MAX_LINKS - 1) * (B2M_MAX_LINKS - 1)];
      rc_controller(T, m.jq, m.jqd, t, m.jtau, tau);
      const double gv[3] = {P.gx, P.gy, P.gz};
      rc_fwd_dyn(T, T.fdyn, s, m.bmass + P.rc_first, m.bJ + 3 * P.rc_first, m.jqd, tau, gv, qdd, Hw);
      for (int k = 0; k < nd; k++) m.jqd[k] = m.jqd[k] + qdd[k] * h;
    }
    g.sync();
    rc_refresh(g, P, m);
  }
  for (int b = g.tid; b < P.nb; b += G::size) {
    if (!m.ben[b] || is_link(P, b)) continue;
    const double* R = m.bR + 9 * b; const double* J = m.bJ + 3 * b;
    const double mass = m.bmass[b];
    const V3 f = V3(P.gx, P.gy, P.gz) * mass;
    const V3 va = ld3(m.bva + 3 * b), vl = ld3(m.bvl + 3 * b);
    const V3 wb = rotT(R, va);
    const V3 Jw = rot(R, V3(J[0] * wb.x, J[1] * wb.y, J[2] * wb.z));
    const V3 rhs = V3() - cross(va, Jw);
    const V3 rb = rotT(R, rhs);
    const V3 alpha = rot(R, V3(rb.x / J[0], rb.y / J[1], rb.z / J[2]));
    const V3 a = f * (1.0 / mass);
    st3(m.bvl + 3 * b, vl + a * h);
    st3(m.bva + 3 * b, va + alpha * h);
  }
  g.sync();
}

// position half of the semi-implicit Euler step with conservative advancement (TimeSteppingSimulator.cpp:119-168)
template <class G>
B2M_DEV B2M_NOINL double integrate_positions_CA(const G& g, const SimParams& P, int e, EnvMem& m, double dt, unsigned long long* lc) {
  const int nb = P.nb;
  for (int k = g.tid; k < 3 * nb; k += G::size) m.xsave[k] = m.bx[k];
  for (int k = g.tid; k < 4 * nb; k += G::size) m.qsave[k] = m.bq[k];
  if (B2M_RC(P)) for (int k = g.tid; k < P.rc_links - 1; k += G::size) m.jqsave[k] = m.jq[k];
  g.sync();
  double h = 0.0;
  const double min_step = P.min_step_env ? P.min_step_env[e] : P.min_step_size;
  while (h < dt) {
    if (g.tid == 0) lc[CNT_CA_ITERS]++;
    calc_pairwise_distances(g, m);
    const int np = m.scal[S_NPAIRS];
    double CA = B2M_INF;
    for (int p = g.tid; p < np; p += G::size) CA = fmin(CA, pair_CA(m, p));
    CA = g.min(CA);
    if (CA <= 0.0) break;
    double tc = fmax(min_step, CA);
    tc = fmin(dt - h, tc);
    g.sync();
    if (B2M_RC(P)) {   // joint coordinates are their own Euler coordinates: q = qsave + (h + tc) qd
      for (int k = g.tid; k < P.rc_links - 1; k += G::size) m.jq[k] = m.jqd[k] * (h + tc) + m.jqsave[k];
      g.sync();
      rc_refresh(g, P, m);
    }
    for (int b = g.tid; b < nb; b += G::size) {
      if (!m.ben[b] || is_link(P, b)) continue;
      const double s = h + tc;
      const double qx = m.qsave[4 * b], qy = m.qsave[4 * b + 1], qz = m.qsave[4 * b + 2], qw = m.qsave[4 * b + 3];
      const V3 w = ld3(m.bva + 3 * b), vl = ld3(m.bvl + 3 * b);
      const double dw = 0.5 * (-qx * w.x - qy * w.y - qz * w.z);   // Ravelin Quatd::deriv
      const double dx = 0.5 * (+qw * w.x + qz * w.y - qy * w.z);
      const double dy = 0.5 * (-qz * w.x + qw * w.y + qx * w.z);
      const double dz = 0.5 * (+qy * w.x - qx * w.y + qw * w.z);
      m.bx[3 * b] = vl.x * s + m.xsave[3 * b]; m.bx[3 * b + 1] = vl.y * s + m.xsave[3 * b + 1]; m.bx[3 * b + 2] = vl.z * s + m.xsave[3 * b + 2];
      const double nx = dx * s + qx, ny = dy * s + qy, nz = dz * s + qz, nw = dw * s + qw;
      const double nrm = sqrt(nx * nx + ny * ny + nz * nz + nw * nw);
      double* qt = m.bq + 4 * b;
      qt[0] = nx / nrm; qt[1] = ny / nrm; qt[2] = nz / nrm; qt[3] = nw / nrm;
      quat_to_R(qt, m.bR + 9 * b);
    }
    g.sync();
    h += tc;
  }
  return h;
}

// ConstraintSimulator::find_unilateral_constraints (:488-537) + preprocess_constraint (:390-417): contacts in pair order
template <class G>
B2M_DEV B2M_NOINL void find_unilateral_constraints(const G& g, const SimParams& P, int e, EnvMem& m, unsigned long long* lc) {
  const int np = m.scal[S_NPAIRS], nb = P.nb, ne = P.n_envs;
  if (g.tid == 0) {
    int nc = 0; bool overflow = false;
    ContactOut con[8];
    for (int p = 0; p < np; p++) {
      if (!(m.pd_dist[p] < P.contact_dist_thresh)) continue;
      const int k = pair_contacts(m, m.pair_a[p], m.pair_b[p], P.contact_dist_thresh, con, 8);
      for (int i = 0; i < k && i < 8; i++) {
        if (nc >= P.cmax) { overflow = true; break; }
        st3(m.cp + 3 * nc, con[i].p); st3(m.cnrm + 3 * nc, con[i].n);
        V3 t1, t2; orthonormal_basis(con[i].n, t1, t2);
        st3(m.ct1 + 3 * nc, t1); st3(m.ct2 + 3 * nc, t2);
        m.cb1[nc] = con[i].b1; m.cb2[nc] = con[i].b2; m.cdist[nc] = con[i].dist;
        const int lo = min(con[i].b1, con[i].b2), hi = max(con[i].b1, con[i].b2);
        const size_t o = ((size_t)lo * nb + hi) * ne + e;
        m.cmu[nc] = P.mu_c[o]; m.cmuv[nc] = P.mu_v[o]; m.ceps[nc] = P.eps[o]; m.ccomp[nc] = P.compliance[o]; m.cNK[nc] = P.NK[o];
        nc++;
      }
    }
    m.scal[S_NCON] = nc;
    lc[CNT_CONTACTS] += nc;
    if (overflow) lc[CNT_OVERFLOW]++;
  }
  g.sync();
}

B2M_HD B2M_INL double constraint_vel(const EnvMem& m, int c) {
  ContactOut co; co.p = ld3(m.cp + 3 * c); co.n = ld3(m.cnrm + 3 * c); co.b1 = m.cb1[c]; co.b2 = m.cb2[c];
  return contact_vel(m, co);
}

// 6x6 SPD inverse through Cholesky, same order as the checker's inverse_SPD (ImpactConstraintHandler.cpp:1599-1611)
B2M_HD B2M_NOINL inline void inverse_spd6(double* A) {
  double L[36];
  for (int i = 0; i < 36; i++) L[i] = A[i];
  for (int j = 0; j < 6; j++) {
    double d = L[j * 6 + j];
    for (int k = 0; k < j; k++) d = fma(-L[k * 6 + j], L[k * 6 + j], d);
    d = sqrt(d);
    L[j * 6 + j] = d;
    for (int i = j + 1; i < 6; i++) {
      double s = L[j * 6 + i];
      for (int k = 0; k < j; k++) s = fma(-L[k * 6 + i], L[k * 6 + j], s);
      L[j * 6 + i] = s / d;
    }
  }
  for (int j = 0; j < 6; j++) {
    double e[6];
    for (int i = 0; i < 6; i++) e[i] = (i == j) ? 1.0 : 0.0;
    for (int i = 0; i < 6; i++) { double s = e[i]; for (int k = 0; k < i; k++) s = fma(-L[k * 6 + i], e[k], s); e[i] = s / L[i * 6 + i]; }
    for (int i = 5; i >= 0; i--) { double s = e[i]; for (int k = i + 1; k < 6; k++) s = fma(-L[i * 6 + k], e[k], s); e[i] = s / L[i * 6 + i]; }
    for (int i = 0; i < 6; i++) A[j * 6 + i] = e[i];
  }
}

// index helpers for the island-local arrays
B2M_HD B2M_INL double* jrow(const EnvMem& m, int nc, int d, int i, int blk) { return m.Jr + ((((size_t)d * nc + i) * 2 + blk) * 6); }
B2M_HD B2M_INL double* xjrow(const EnvMem& m, int nc, int d, int i, int blk) { return m.XJ + ((((size_t)d * nc + i) * 2 + blk) * 6); }
// D blocks stored for d1<=d2: index 0:nn 1:ns 2:nt 3:ss 4:st 5:tt
B2M_HD B2M_INL int dblk(int d1, int d2) { return d1 == 0 ? d2 : (d1 == 1 ? 2 + d2 : 5); }
B2M_HD B2M_INL double Dn(const EnvMem& m, int nc, int d1, int d2, int i, int j) {
  return (d1 <= d2) ? m.D[(size_t)dblk(d1, d2) * nc * nc + (size_t)i * nc + j] : m.D[(size_t)dblk(d2, d1) * nc * nc + (size_t)j * nc + i];
}

// Lower Cholesky in place by the whole group (LinAlgd::factor_chol; column-major, ld n); every element is produced by the
// same operation sequence as the checker's factor_chol, so the accept / reject decisions below are identical.
template <class G>
B2M_DEV B2M_NOINL bool chol_factor_group(const G& g, double* A, int n) {
  for (int j = 0; j < n; j++) {
    double d = A[(size_t)j * n + j];
    for (int k = 0; k < j; k++) d = fma(-A[(size_t)k * n + j], A[(size_t)k * n + j], d);
    g.sync();
    if (!(d > 0.0)) return false;
    d = sqrt(d);
    if (g.tid == 0) A[(size_t)j * n + j] = d;
    for (int i = j + 1 + g.tid; i < n; i += G::size) {
      double s = A[(size_t)j * n + i];
      for (int k = 0; k < j; k++) s = fma(-A[(size_t)k * n + i], A[(size_t)k * n + j], s);
      A[(size_t)j * n + i] = s / d;
    }
    g.sync();
  }
  return true;
}
// solve_chol_fast for one right-hand side, one thread
B2M_HD B2M_INL void chol_solve1(const double* L, int n, double* b) {
  for (int i = 0; i < n; i++) { double s = b[i]; for (int k = 0; k < i; k++) s = fma(-L[(size_t)k * n + i], b[k], s); b[i] = s / L[(size_t)i * n + i]; }
  for (int i = n - 1; i >= 0; i--) { double s = b[i]; for (int k = i + 1; k < n; k++) s = fma(-L[(size_t)i * n + k], b[k], s); b[i] = s / L[(size_t)i * n + i]; }
}
// inverse_spd_n by the whole group: the factorisation row-parallel, then one column of the inverse per thread; every
// element goes through the same operation sequence as in inverse_spd_n, so the result is bit-identical.  n <= B2M_MAX_LINKS.
template <class G>
B2M_DEV B2M_NOINL void inverse_spd_group(const G& g, double* A, int n, int lda, double* L) {
  for (int t = g.tid; t < n * n; t += G::size) { const int j = t / n, i = t - j * n; L[t] = A[(size_t)j * lda + i]; }
  g.sync();
  chol_factor_group(g, L, n);
  if constexpr (G::size == 1) {                                  // one thread: three columns of the inverse per pass (three independent substitution chains)
    int j = 0;
    for (; j + 3 <= n; j += 3) {
      double e0[B2M_MAX_LINKS], e1[B2M_MAX_LINKS], e2[B2M_MAX_LINKS];
      for (int i = 0; i < n; i++) { e0[i] = (i == j) ? 1.0 : 0.0; e1[i] = (i == j + 1) ? 1.0 : 0.0; e2[i] = (i == j + 2) ? 1.0 : 0.0; }
      for (int i = 0; i < n; i++) {
        double s0 = e0[i], s1 = e1[i], s2 = e2[i];
        for (int k = 0; k < i; k++) { const double l = L[(size_t)k * n + i]; s0 = fma(-l, e0[k], s0); s1 = fma(-l, e1[k], s1); s2 = fma(-l, e2[k], s2); }
        const double d = L[(size_t)i * n + i];
        e0[i] = s0 / d; e1[i] = s1 / d; e2[i] = s2 / d;
      }
      for (int i = n - 1; i >= 0; i--) {
        double s0 = e0[i], s1 = e1[i], s2 = e2[i];
        for (int k = i + 1; k < n; k++) { const double l = L[(size_t)i * n + k]; s0 = fma(-l, e0[k], s0); s1 = fma(-l, e1[k], s1); s2 = fma(-l, e2[k], s2); }
        const double d = L[(size_t)i * n + i];
        e0[i] = s0 / d; e1[i] = s1 / d; e2[i] = s2 / d;
      }
      for (int i = 0; i < n; i++) { A[(size_t)j * lda + i] = e0[i]; A[(size_t)(j + 1) * lda + i] = e1[i]; A[(size_t)(j + 2) * lda + i] = e2[i]; }
    }
    for (; j < n; j++) {
      double e[B2M_MAX_LINKS];
      for (int i = 0; i < n; i++) e[i] = (i == j) ? 1.0 : 0.0;
      chol_solve1(L, n, e);
      for (int i = 0; i < n; i++) A[(size_t)j * lda + i] = e[i];
    }
    return;
  }
  for (int j = g.tid; j < n; j += G::size) {
    double e[B2M_MAX_LINKS];
    for (int i = 0; i < n; i++) e[i] = (i == j) ? 1.0 : 0.0;
    chol_solve1(L, n, e);
    for (int i = 0; i < n; i++) A[(size_t)j * lda + i] = e[i];
  }
  g.sync();
}

// n x n SPD inverse through Cholesky (LinAlgd::inverse_SPD, ImpactConstraintHandler.cpp:1605-1607): A (column-major,
// leading dimension lda) is replaced by its inverse; L: n*n + n doubles of scratch.  One thread; same operation order as
// the checker.
B2M_HD B2M_NOINL inline void inverse_spd_n(double* A, int n, int lda, double* L) {
  double* e = L + (size_t)n * n;
  for (int j = 0; j < n; j++) for (int i = 0; i < n; i++) L[(size_t)j * n + i] = A[(size_t)j * lda + i];
  for (int j = 0; j < n; j++) {
    double d = L[(size_t)j * n + j];
    for (int k = 0; k < j; k++) d = fma(-L[(size_t)k * n + j], L[(size_t)k * n + j], d);
    d = sqrt(d);
    L[(size_t)j * n + j] = d;
    for (int i = j + 1; i < n; i++) {
      double s = L[(size_t)j * n + i];
      for (int k = 0; k < j; k++) s = fma(-L[(size_t)k * n + i], L[(size_t)k * n + j], s);
      L[(size_t)j * n + i] = s / d;
    }
  }
  for (int j = 0; j < n; j++) {
    for (int i = 0; i < n; i++) e[i] = (i == j) ? 1.0 : 0.0;
    for (int i = 0; i < n; i++) { double s = e[i]; for (int k = 0; k < i; k++) s = fma(-L[(size_t)k * n + i], e[k], s); e[i] = s / L[(size_t)i * n + i]; }
    for (int i = n - 1; i >= 0; i--) { double s = e[i]; for (int k = i + 1; k < n; k++) s = fma(-L[(size_t)i * n + k], e[k], s); e[i] = s / L[(size_t)i * n + i]; }
    for (int i = 0; i < n; i++) A[(size_t)j * lda + i] = e[i];
  }
}

// ImpactConstraintHandler::compute_problem_data (:1898-2166) with an articulated body in the scene: dense rows over the
// island's generalized coordinates [free bodies 6 each ..., joint coordinates], X = blockdiag(M_b^-1, H(q)^-1).
// A contact wrench [d, r x d] on link L maps to joint k (an ancestor of L) as d . S_k(lin) + (p x d) . S_k(ang) with S_k
// the joint's world-frame motion subspace about the world origin -- RCArticulatedBodyd::calc_jacobian (:1875) folded in.
template <class G>
B2M_DEV B2M_NOINL void compute_problem_data_dense(const G& g, const SimParams& P, EnvMem& m) {
  const int nc = m.scal[S_NC], nb = P.nb, ngc = m.scal[S_NGC];
  const int rep = P.rc_first + 1;
  for (int t = g.tid; t < ngc * ngc; t += G::size) m.Xb[t] = 0.0;
  g.sync();
  if (m.gcoff[rep] >= 0) {                               // joint-space inertia by CRB, then inverse_SPD
    const RCTree& T = *P.rc;
    double* H = m.Xb + (size_t)m.gcoff[rep] * ngc + m.gcoff[rep];
    if (g.tid == 0) {
      RCState s; s.x = m.bx + 3 * P.rc_first; s.R = m.bR + 9 * P.rc_first; s.S = m.rS; s.v = m.rV;
      rc_crb(T, s, m.bmass + P.rc_first, m.bJ + 3 * P.rc_first, H, ngc);
    }
    g.sync();
    inverse_spd_group(g, H, T.n_links - 1, ngc, m.Lf);
  }
  for (int b = g.tid; b < nb; b += G::size) {            // free bodies: 6x6 blocks as in the block layout
    if (m.gcoff[b] < 0 || is_link(P, b)) continue;
    double Mg[36];
    for (int i = 0; i < 36; i++) Mg[i] = 0.0;
    const double* R = m.bR + 9 * b; const double* J = m.bJ + 3 * b;
    for (int k = 0; k < 3; k++) Mg[k * 6 + k] = m.bmass[b];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) {
        double s = 0.0;
        for (int k = 0; k < 3; k++) s += R[r * 3 + k] * J[k] * R[c * 3 + k];
        Mg[(3 + c) * 6 + (3 + r)] = s;
      }
    inverse_spd6(Mg);
    const int o = m.gcoff[b];
    for (int c = 0; c < 6; c++) for (int r = 0; r < 6; r++) m.Xb[(size_t)(o + c) * ngc + o + r] = Mg[c * 6 + r];
  }
  // generalized velocity of the island
  for (int k = g.tid; k < ngc; k += G::size) {
    const int b = m.gcb[k], l = m.gcl[k];
    m.gv[k] = (b == rep && B2M_RC(P)) ? m.jqd[l] : (l < 3 ? m.bvl[3 * b + l] : m.bva[3 * b + l - 3]);
  }
  // Jacobian rows, one thread per (dir, contact, coordinate)
  for (int t = g.tid; t < 3 * nc * ngc; t += G::size) {
    const int k = t % ngc, i = (t / ngc) % nc, d = t / (ngc * nc);
    const int c = m.icon[i];
    const int sb = m.gcb[k], l = m.gcl[k];
    const V3 dir0 = d == 0 ? ld3(m.cnrm + 3 * c) : (d == 1 ? ld3(m.ct1 + 3 * c) : ld3(m.ct2 + 3 * c));
    const V3 p = ld3(m.cp + 3 * c);
    double val = 0.0;
    for (int blk = 0; blk < 2; blk++) {
      const int bi = blk == 0 ? m.cb1[c] : m.cb2[c];
      if (!m.ben[bi]) continue;
      const V3 dir = blk == 0 ? dir0 : -dir0;
      if (is_link(P, bi)) {
        if (sb != rep) continue;
        const int j = l + 1;                                      // joint of link j
        if (!((m.ranc[bi - P.rc_first] >> j) & 1)) continue;
        const double* S = m.rS + 6 * j;
        const V3 pxd = cross(p, dir);
        val += (dir.x * S[3] + dir.y * S[4] + dir.z * S[5]) + (pxd.x * S[0] + pxd.y * S[1] + pxd.z * S[2]);
      } else {
        if (sb != bi) continue;
        if (l < 3) val += (l == 0 ? dir.x : (l == 1 ? dir.y : dir.z));
        else { const V3 rxd = cross(p - ld3(m.bx + 3 * bi), dir); val += (l == 3 ? rxd.x : (l == 4 ? rxd.y : rxd.z)); }
      }
    }
    m.Jr[t] = val;
  }
  g.sync();
  // X_CdT = (Cd X)^T, kept as rows: XJ[row][k] = sum_kk Jr[row][kk] X[kk][k]
  if constexpr (G::size == 1) {
    // one thread per env: the same dot products (same order of the terms), four at a time -- four independent fma chains and
    // their loads in flight instead of one (ncu, UR10: these three loops were 19 % of the thread-per-env impact launch)
    for (int row = 0; row < 3 * nc; row++) {
      const double* jr = m.Jr + (size_t)row * ngc;
      double* out = m.XJ + (size_t)row * ngc;
      int k = 0;
      for (; k + 4 <= ngc; k += 4) {
        const double* x0 = m.Xb + (size_t)k * ngc; const double* x1 = x0 + ngc; const double* x2 = x1 + ngc; const double* x3 = x2 + ngc;
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        for (int kk = 0; kk < ngc; kk++) { const double a = jr[kk]; s0 = fma(a, x0[kk], s0); s1 = fma(a, x1[kk], s1); s2 = fma(a, x2[kk], s2); s3 = fma(a, x3[kk], s3); }
        out[k] = s0; out[k + 1] = s1; out[k + 2] = s2; out[k + 3] = s3;
      }
      for (; k < ngc; k++) { double s0 = 0.0; for (int kk = 0; kk < ngc; kk++) s0 = fma(jr[kk], m.Xb[(size_t)k * ngc + kk], s0); out[k] = s0; }
    }
    for (int bk = 0; bk < 6; bk++) {
      const int d1 = bk < 3 ? 0 : (bk < 5 ? 1 : 2), d2 = bk < 3 ? bk : (bk < 5 ? bk - 2 : 2);
      for (int i = 0; i < nc; i++) {
        const double* jr = m.Jr + ((size_t)d1 * nc + i) * ngc;
        double* out = m.D + ((size_t)bk * nc + i) * nc;
        int j = 0;
        for (; j + 4 <= nc; j += 4) {
          const double* x0 = m.XJ + ((size_t)d2 * nc + j) * ngc; const double* x1 = x0 + ngc; const double* x2 = x1 + ngc; const double* x3 = x2 + ngc;
          double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
          for (int k = 0; k < ngc; k++) { const double a = jr[k]; s0 = fma(a, x0[k], s0); s1 = fma(a, x1[k], s1); s2 = fma(a, x2[k], s2); s3 = fma(a, x3[k], s3); }
          out[j] = s0; out[j + 1] = s1; out[j + 2] = s2; out[j + 3] = s3;
        }
        for (; j < nc; j++) { const double* xj = m.XJ + ((size_t)d2 * nc + j) * ngc; double s0 = 0.0; for (int k = 0; k < ngc; k++) s0 = fma(jr[k], xj[k], s0); out[j] = s0; }
      }
    }
    {
      int t = 0;
      for (; t + 3 <= 3 * nc; t += 3) {
        const double* j0 = m.Jr + (size_t)t * ngc; const double* j1 = j0 + ngc; const double* j2 = j1 + ngc;
        double s0 = 0.0, s1 = 0.0, s2 = 0.0;
        for (int k = 0; k < ngc; k++) { const double gk = m.gv[k]; s0 = fma(j0[k], gk, s0); s1 = fma(j1[k], gk, s1); s2 = fma(j2[k], gk, s2); }
        m.Cv[t] = s0; m.Cv[t + 1] = s1; m.Cv[t + 2] = s2; m.imp[t] = 0.0; m.imp[t + 1] = 0.0; m.imp[t + 2] = 0.0;
      }
    }
    return;
  }
  for (int t = g.tid; t < 3 * nc * ngc; t += G::size) {
    const int k = t % ngc, row = t / ngc;
    const double* jr = m.Jr + (size_t)row * ngc;
    double s = 0.0;
    for (int kk = 0; kk < ngc; kk++) s = fma(jr[kk], m.Xb[(size_t)k * ngc + kk], s);
    m.XJ[t] = s;
  }
  g.sync();
  // Delassus blocks Cd1 X Cd2^T
  for (int t = g.tid; t < 6 * nc * nc; t += G::size) {
    const int j = t % nc, i = (t / nc) % nc, bk = t / (nc * nc);
    const int d1 = bk < 3 ? 0 : (bk < 5 ? 1 : 2), d2 = bk < 3 ? bk : (bk < 5 ? bk - 2 : 2);
    const double* jr = m.Jr + ((size_t)d1 * nc + i) * ngc;
    const double* xj = m.XJ + ((size_t)d2 * nc + j) * ngc;
    double s = 0.0;
    for (int k = 0; k < ngc; k++) s = fma(jr[k], xj[k], s);
    m.D[t] = s;
  }
  for (int t = g.tid; t < 3 * nc; t += G::size) {
    const double* jr = m.Jr + (size_t)t * ngc;
    double s = 0.0;
    for (int k = 0; k < ngc; k++) s = fma(jr[k], m.gv[k], s);
    m.Cv[t] = s;
    m.imp[t] = 0.0;
  }
  g.sync();
}

// update_from_stacked (:298-397), dense layout: generalized velocity += X_CnT cn + X_CsT cs + X_CtT ct
template <class G>
B2M_DEV B2M_NOINL void apply_to_bodies_dense(const G& g, const SimParams& P, EnvMem& m, const double* imp) {
  const int nc = m.scal[S_NC], ngc = m.scal[S_NGC];
  const int rep = P.rc_first + 1;
  for (int k = g.tid; k < ngc; k += G::size) {
    double s3[3];
    for (int d = 0; d < 3; d++) {
      double s = 0.0;
      for (int i = 0; i < nc; i++) s = fma(m.XJ[((size_t)d * nc + i) * ngc + k], imp[d * nc + i], s);
      s3[d] = s;
    }
    m.dv[k] = (s3[0] + s3[1]) + s3[2];
  }
  g.sync();
  bool rc_touched = false;
  for (int k = g.tid; k < ngc; k += G::size) {
    const int b = m.gcb[k], l = m.gcl[k];
    if (b == rep && B2M_RC(P)) m.jqd[l] = m.jqd[l] + m.dv[k];
    else if (l < 3) m.bvl[3 * b + l] = m.bvl[3 * b + l] + m.dv[k];
    else m.bva[3 * b + l - 3] = m.bva[3 * b + l - 3] + m.dv[k];
  }
  rc_touched = B2M_RC(P) && m.gcoff[rep] >= 0;
  g.sync();
  if (rc_touched) rc_refresh(g, P, m);
}

// ImpactConstraintHandler::compute_problem_data (:1898-2166) for the island whose contacts are icon[0..nc)
template <class G>
B2M_DEV B2M_NOINL void compute_problem_data(const G& g, const SimParams& P, EnvMem& m) {
  if (B2M_NGC(P)) { compute_problem_data_dense(g, P, m); return; }
  const int nc = m.scal[S_NC], nb = P.nb;
  // X = blockdiag(inverse_SPD(generalized inertia)) (:1590-1611), one thread per island body
  for (int b = g.tid; b < nb; b += G::size) {
    if (m.gcoff[b] < 0) continue;
    double Mg[36];
    for (int i = 0; i < 36; i++) Mg[i] = 0.0;
    const double* R = m.bR + 9 * b; const double* J = m.bJ + 3 * b;
    for (int k = 0; k < 3; k++) Mg[k * 6 + k] = m.bmass[b];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) {
        double s = 0.0;
        for (int k = 0; k < 3; k++) s += R[r * 3 + k] * J[k] * R[c * 3 + k];
        Mg[(3 + c) * 6 + (3 + r)] = s;
      }
    inverse_spd6(Mg);
    for (int i = 0; i < 36; i++) m.Xb[36 * b + i] = Mg[i];       // column-major: X(r,c) = Xb[c*6+r]
  }
  // Jacobian rows [d, r x d] (:1817-1895), one thread per (dir, contact, block)
  for (int t = g.tid; t < 3 * nc * 2; t += G::size) {
    const int blk = t & 1, i = (t >> 1) % nc, d = (t >> 1) / nc;
    const int c = m.icon[i];
    const int bi = blk == 0 ? m.cb1[c] : m.cb2[c];
    double* row = jrow(m, nc, d, i, blk);
    if (!m.ben[bi]) { for (int k = 0; k < 6; k++) row[k] = 0.0; continue; }
    V3 dir = d == 0 ? ld3(m.cnrm + 3 * c) : (d == 1 ? ld3(m.ct1 + 3 * c) : ld3(m.ct2 + 3 * c));
    if (blk == 1) dir = -dir;
    const V3 rxd = cross(ld3(m.cp + 3 * c) - ld3(m.bx + 3 * bi), dir);
    row[0] = dir.x; row[1] = dir.y; row[2] = dir.z; row[3] = rxd.x; row[4] = rxd.y; row[5] = rxd.z;
  }
  g.sync();
  // X_CdT restricted to the block's body: XJ = row * X_body (:2125-2127), one thread per (dir, contact, block, k)
  for (int t = g.tid; t < 3 * nc * 2 * 6; t += G::size) {
    const int k = t % 6, rest = t / 6, blk = rest & 1, i = (rest >> 1) % nc, d = (rest >> 1) / nc;
    const int c = m.icon[i];
    const int bi = blk == 0 ? m.cb1[c] : m.cb2[c];
    double s = 0.0;
    if (m.ben[bi]) {
      const double* row = jrow(m, nc, d, i, blk);
      const double* X = m.Xb + 36 * bi;
      for (int kk = 0; kk < 6; kk++) s = fma(row[kk], X[k * 6 + kk], s);
      s = 0.0 + s;
    }
    xjrow(m, nc, d, i, blk)[k] = s;
  }
  g.sync();
  // Delassus blocks Cd1 X Cd2^T (:2133-2149), one thread per (block, i, j)
  for (int t = g.tid; t < 6 * nc * nc; t += G::size) {
    const int j = t % nc, i = (t / nc) % nc, bk = t / (nc * nc);
    const int d1 = bk < 3 ? 0 : (bk < 5 ? 1 : 2), d2 = bk < 3 ? bk : (bk < 5 ? bk - 2 : 2);
    const int ci = m.icon[i], cj = m.icon[j];
    double s = 0.0;
    for (int blk = 0; blk < 2; blk++) {
      const int bi = blk == 0 ? m.cb1[ci] : m.cb2[ci];
      if (!m.ben[bi]) continue;
      int blk2 = -1;
      if (m.cb1[cj] == bi) blk2 = 0; else if (m.cb2[cj] == bi) blk2 = 1;
      if (blk2 < 0) continue;
      const double* row = jrow(m, nc, d1, i, blk);
      const double* xj = xjrow(m, nc, d2, j, blk2);
      for (int k = 0; k < 6; k++) s = fma(row[k], xj[k], s);
    }
    m.D[t] = s;
  }
  // Cd v (:2157-2159)
  for (int t = g.tid; t < 3 * nc; t += G::size) {
    const int i = t % nc, d = t / nc;
    const int c = m.icon[i];
    double s = 0.0;
    for (int blk = 0; blk < 2; blk++) {
      const int bi = blk == 0 ? m.cb1[c] : m.cb2[c];
      if (!m.ben[bi]) continue;
      const double* row = jrow(m, nc, d, i, blk);
      const double v[6] = {m.bvl[3 * bi], m.bvl[3 * bi + 1], m.bvl[3 * bi + 2], m.bva[3 * bi], m.bva[3 * bi + 1], m.bva[3 * bi + 2]};
      for (int k = 0; k < 6; k++) s = fma(row[k], v[k], s);
    }
    m.Cv[t] = s;
    m.imp[t] = 0.0;
  }
  g.sync();
}

// QP-as-LCP (ImpactConstraintHandlerQP.cpp:129-148,216,271-497), nl = 0.  Returns n.
template <class G>
B2M_DEV B2M_NOINL int build_qp_lcp(const G& g, const SimParams& P, EnvMem& m) {
  const int nc = m.scal[S_NC];
  const int NV = 5 * nc;
  if (g.tid == 0) {
    int row = 0;
    for (int i = 0; i < nc; i++) { const int half = m.cNK[m.icon[i]] / 2; for (int j = 0; j < half; j++) { m.frow_c[row] = i; m.frow_j[row] = j; row++; } }
    m.scal[S_N] = NV + nc + row;
  }
  g.sync();
  const int n = m.scal[S_N];
  if (n > P.nmax) return n;
  const double* qcos = P.fr_tab; const double* qsin = P.fr_tab + (size_t)(B2M_NKMAX + 1) * (B2M_NKMAX / 2);
  if constexpr (G::size == 1) {
    // One thread per env: the same entries as the flat loop below, written block by block -- no integer division or
    // per-entry branching, unit-stride stores, several loads in flight (a lone thread is latency-bound; see lu_solve_serial).
    const int nfr = n - NV - nc;
    for (int c = 0; c < n; c++) {
      double* col = m.MM + (size_t)c * n;
      if (c < NV) {
        const int bc = c / nc, j = c - bc * nc;
        const int dc = bc == 0 ? 0 : (bc == 1 || bc == 3 ? 1 : 2);
        const bool cneg = bc >= 3;
        for (int br = 0; br < 5; br++) {                                  // upper-left: +-D(dr,dc)(i,j)
          const int dr = br == 0 ? 0 : (br == 1 || br == 3 ? 1 : 2);
          const bool neg = (br >= 3) != cneg;
          const double* src; int stride;
          if (dr <= dc) { src = m.D + (size_t)dblk(dr, dc) * nc * nc + j; stride = nc; }
          else { src = m.D + (size_t)dblk(dc, dr) * nc * nc + (size_t)j * nc; stride = 1; }
          double* dst = col + br * nc;
          int i = 0;
          for (; i + 4 <= nc; i += 4) {
            const double v0 = src[(size_t)i * stride], v1 = src[(size_t)(i + 1) * stride], v2 = src[(size_t)(i + 2) * stride], v3 = src[(size_t)(i + 3) * stride];
            dst[i] = neg ? -v0 : v0; dst[i + 1] = neg ? -v1 : v1; dst[i + 2] = neg ? -v2 : v2; dst[i + 3] = neg ? -v3 : v3;
          }
          for (; i < nc; i++) { const double v0 = src[(size_t)i * stride]; dst[i] = neg ? -v0 : v0; }
        }
        if (c < nc) col[c] += m.ccomp[m.icon[c]];
        {                                                                  // lower-left, normal rows: A(a, c) = +-D(0,dc)(a,j) [+ compliance]
          const double* src = m.D + (size_t)dblk(0, dc) * nc * nc + j;
          double* dst = col + NV;
          for (int a = 0; a < nc; a++) {
            const double v = src[(size_t)a * nc];
            double av = cneg ? -v : v;
            if (c == a) av += m.ccomp[m.icon[a]];
            dst[a] = av;
          }
        }
        double* dst = col + NV + nc;                                       // lower-left, friction rows
        for (int fr = 0; fr < nfr; fr++) {
          const int i = m.frow_c[fr], jj = m.frow_j[fr];
          const size_t ti = (size_t)m.cNK[m.icon[i]] * (B2M_NKMAX / 2) + jj;
          double av;
          if (c == i) av = m.cmu[m.icon[i]];
          else if (c == nc + i || c == 3 * nc + i) av = -qcos[ti];
          else if (c == 2 * nc + i || c == 4 * nc + i) av = -qsin[ti];
          else av = 0.0;
          dst[fr] = av;
        }
      } else {
        const int a = c - NV;                                              // upper-right = -A^T, lower-right = 0
        if (a < nc) {
          for (int bc = 0; bc < 5; bc++) {
            const int dc = bc == 0 ? 0 : (bc == 1 || bc == 3 ? 1 : 2);
            const double* src = m.D + (size_t)dblk(0, dc) * nc * nc + (size_t)a * nc;
            double* dst = col + bc * nc;
            for (int j = 0; j < nc; j++) {
              const double v = src[j];
              double av = (bc >= 3) ? -v : v;
              if (bc * nc + j == a) av += m.ccomp[m.icon[a]];
              dst[j] = -av;
            }
          }
        } else {
          const int fr = a - nc, i = m.frow_c[fr], jj = m.frow_j[fr];
          const size_t ti = (size_t)m.cNK[m.icon[i]] * (B2M_NKMAX / 2) + jj;
          const double mu = m.cmu[m.icon[i]], cs = qcos[ti], sn = qsin[ti];
          for (int r = 0; r < NV; r++) col[r] = -0.0;
          col[i] = -mu; col[nc + i] = -(-cs); col[3 * nc + i] = -(-cs); col[2 * nc + i] = -(-sn); col[4 * nc + i] = -(-sn);
        }
        for (int r = NV; r < n; r++) col[r] = 0.0;
      }
    }
  } else
  for (int t = g.tid; t < n * n; t += G::size) {
    const int c = t / n, r = t - c * n;
    // entry of A = [H(0:nc,:) ; friction rows] at (a, col<NV)
    double val = 0.0;
    const bool upper = r < NV, left = c < NV;
    if (upper && left) {
      const int br = r / nc, i = r - br * nc, bc = c / nc, j = c - bc * nc;
      const int dr = br == 0 ? 0 : (br == 1 || br == 3 ? 1 : 2), dc = bc == 0 ? 0 : (bc == 1 || bc == 3 ? 1 : 2);
      const double v = Dn(m, nc, dr, dc, i, j);
      val = ((br >= 3) != (bc >= 3)) ? -v : v;
      if (r == c && r < nc) val += m.ccomp[m.icon[r]];
    } else if (upper != left) {
      const int a = (upper ? c : r) - NV, col = upper ? r : c;       // A(a, col); the upper-right block is -A^T
      double av;
      if (a < nc) {
        const int bc = col / nc, j = col - bc * nc;
        const int dc = bc == 0 ? 0 : (bc == 1 || bc == 3 ? 1 : 2);
        const double v = Dn(m, nc, 0, dc, a, j);
        av = (bc >= 3) ? -v : v;
        if (col == a) av += m.ccomp[m.icon[a]];
      } else {
        const int fr = a - nc, i = m.frow_c[fr], j = m.frow_j[fr];
        const int NKi = m.cNK[m.icon[i]];
        const size_t ti = (size_t)NKi * (B2M_NKMAX / 2) + j;
        if (col == i) av = m.cmu[m.icon[i]];
        else if (col == nc + i || col == 3 * nc + i) av = -qcos[ti];
        else if (col == 2 * nc + i || col == 4 * nc + i) av = -qsin[ti];
        else av = 0.0;
      }
      val = upper ? -av : av;
    }
    m.MM[t] = val;
  }
  for (int r = g.tid; r < n; r += G::size) {
    double v;
    if (r < NV) { const int br = r / nc, i = r - br * nc; const int d = br == 0 ? 0 : (br == 1 || br == 3 ? 1 : 2); v = m.Cv[d * nc + i]; if (br >= 3) v = -v; }
    else if (r < NV + nc) v = m.Cv[r - NV];
    else { const int i = m.frow_c[r - NV - nc]; const double cs = m.Cv[nc + i], ct = m.Cv[2 * nc + i]; v = m.cmuv[m.icon[i]] * sqrt(cs * cs + ct * ct); }
    m.qq[r] = v;
  }
  g.sync();
  return n;
}

// Anitescu-Potra LCP (ImpactConstraintHandlerLCP.cpp:94-310), nl = 0.  Returns n.
template <class G>
B2M_DEV B2M_NOINL int build_ap_lcp(const G& g, const SimParams& P, EnvMem& m) {
  const int NC = m.scal[S_NC];
  const int NCONST = 5 * NC;
  if (g.tid == 0) {
    int row = 0;
    for (int i = 0; i < NC; i++) { const int NKi = m.cNK[m.icon[i]]; const int k4 = NKi > 4 ? (NKi + 4) / 4 : 1; for (int k = 0; k < k4; k++) { m.frow_c[row] = i; m.frow_j[row] = k; row++; } }
    m.scal[S_N] = NCONST + row;
  }
  g.sync();
  const int n = m.scal[S_N];
  if (n > P.nmax) return n;
  const double* acos_ = P.fr_tab + 2 * (size_t)(B2M_NKMAX + 1) * (B2M_NKMAX / 2);
  const double* asin_ = P.fr_tab + 3 * (size_t)(B2M_NKMAX + 1) * (B2M_NKMAX / 2);
  for (int t = g.tid; t < n * n; t += G::size) {
    const int c = t / n, r = t - c * n;
    double val = 0.0;
    const bool upper = r < NCONST, left = c < NCONST;
    if (upper && left) {                                        // UL, block order [n, s+, s-, t+, t-]
      const int br = r / NC, i = r - br * NC, bc = c / NC, j = c - bc * NC;
      const int dr = br == 0 ? 0 : (br <= 2 ? 1 : 2), dc = bc == 0 ? 0 : (bc <= 2 ? 1 : 2);
      const bool nr = (br == 2 || br == 4), ncg = (bc == 2 || bc == 4);
      const double v = Dn(m, NC, dr, dc, i, j);
      val = (nr != ncg) ? -v : v;
    } else if (upper != left) {
      const int fr = (upper ? c : r) - NCONST, col = upper ? r : c;
      const int i = m.frow_c[fr], k = m.frow_j[fr];
      const int NKi = m.cNK[m.icon[i]];
      double e = 0.0;                                           // |LL(fr, col)| pattern for the friction blocks
      const int bc = col / NC, j = col - bc * NC;
      if (j == i && bc >= 1) {
        if (NKi > 4) { const size_t ti = (size_t)NKi * (B2M_NKMAX / 2) + k; e = (bc <= 2) ? acos_[ti] : asin_[ti]; }
        else e = 1.0;
      }
      if (upper) val = e;                                       // UR = +cos/sin (:268-275,288-293)
      else val = (bc == 0 && j == i) ? m.cmu[m.icon[i]] : -e;   // LL = [mu, -cos.., -sin..]
    }
    m.MM[t] = val;
  }
  for (int r = g.tid; r < n; r += G::size) {
    double v = 0.0;
    if (r < NCONST) { const int br = r / NC, i = r - br * NC; const int d = br == 0 ? 0 : (br <= 2 ? 1 : 2); v = m.Cv[d * NC + i]; if (br == 2 || br == 4) v = -v; }
    m.qq[r] = v;
  }
  g.sync();
  return n;
}

// update_from_stacked (:298-397) without bilateral joints: v += X_CnT cn + X_CsT cs + X_CtT ct, impulses from `imp`
template <class G>
B2M_DEV B2M_NOINL void apply_to_bodies(const G& g, const SimParams& P, EnvMem& m, const double* imp) {
  if (B2M_NGC(P)) { apply_to_bodies_dense(g, P, m, imp); return; }
  const int nc = m.scal[S_NC], nb = P.nb;
  for (int t = g.tid; t < 6 * nb; t += G::size) {
    const int b = t / 6, k = t - 6 * b;
    if (m.gcoff[b] < 0) continue;
    double s3[3];
    for (int d = 0; d < 3; d++) {
      double s = 0.0;
      for (int i = 0; i < nc; i++) {
        const int c = m.icon[i];
        int blk = -1;
        if (m.cb1[c] == b) blk = 0; else if (m.cb2[c] == b) blk = 1;
        if (blk < 0) continue;
        s = fma(xjrow(m, nc, d, i, blk)[k], imp[d * nc + i], s);
      }
      s3[d] = s;
    }
    m.dv[t] = (s3[0] + s3[1]) + s3[2];
  }
  g.sync();
  for (int t = g.tid; t < 6 * nb; t += G::size) {
    const int b = t / 6, k = t - 6 * b;
    if (m.gcoff[b] < 0) continue;
    if (k < 3) m.bvl[3 * b + k] = m.bvl[3 * b + k] + m.dv[t]; else m.bva[3 * b + k - 3] = m.bva[3 * b + k - 3] + m.dv[t];
  }
  g.sync();
}

// update_constraint_velocities_from_impulses (:427-464), nl = 0
template <class G>
B2M_DEV B2M_NOINL void update_constraint_velocities(const G& g, EnvMem& m, const double* imp) {
  const int nc = m.scal[S_NC];
  for (int t = g.tid; t < 3 * nc; t += G::size) {
    const int i = t % nc, d = t / nc;
    double acc = m.Cv[t];
    for (int k = 0; k < 3; k++) {
      double s = 0.0;
      for (int j = 0; j < nc; j++) s = fma(Dn(m, nc, d, k, i, j), imp[k * nc + j], s);
      acc += s;
    }
    m.Cv[t] = acc;
  }
  g.sync();
}

template <class G>
B2M_DEV double min_constraint_velocity(const G& g, const EnvMem& m) {            // :413-424
  const int nc = m.scal[S_NC];
  double v = B2M_INF;
  for (int i = g.tid; i < nc; i += G::size) v = fmin(v, m.Cv[i]);
  return g.min(v);
}

// solve_qp_work (ImpactConstraintHandlerQP.cpp:94-263): fills imp = [cn | cs | ct].  Returns false when the env is deferred.
template <class G>
B2M_DEV B2M_NOINL bool solve_qp(const G& g, const SimParams& P, int e, EnvMem& m, unsigned long long* lc, EnvCtx& cx) {
  const int nc = m.scal[S_NC];
  int n;
  { B2M_PROF_T0(m); n = build_qp_lcp(g, P, m); B2M_PROF_ADD(m, g, PH_BUILD); }
  if (n > P.nmax) { if (g.tid == 0) { lc[CNT_OVERFLOW]++; } for (int t = g.tid; t < 3 * nc; t += G::size) m.imp[t] = 0.0; g.sync(); return true; }
  const bool warm = (m.scal[S_ZLN] == n);                                           // :158-162 with rule H1 (zero fill)
  for (int i = g.tid; i < n; i += G::size) m.z[i] = warm ? m.zl[i] : 0.0;
  g.sync();
  long long stats[3] = {0, 0, 0};
  int piv = 0;
  int* bud = cx.limit ? &cx.budget : nullptr;
  int st;
#ifdef __CUDA_ARCH__
#define B2M_STAMP(row) do { if (m.prof && P.tap_times && g.tid == 0) { long long _gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(_gt)); m.prof[(row) * m.prof_stride] = _gt; } } while (0)
#else
#define B2M_STAMP(row) do {} while (0)
#endif
  B2M_STAMP(PH_CONTACTS);                                                            // timeline mode: before the lcp_fast ladder
  { B2M_PROF_T0(m); st = lcp_fast_regularized(g, n, m.MM, n, m.qq, -1.0, true, -20, 4, -8, m.z, m.work, m.iwork, &piv, stats, bud, G::size == 1 && cx.limit && cx.first_rung); B2M_PROF_ADD(m, g, PH_FAST); }   // :219
  B2M_STAMP(PH_PROBLEM);                                                             // after it
  if (st == LCP_DEFER) return false;
  long long fast_calls = stats[0], pivots = stats[1], executed = stats[2], lemke_calls = 0;
  if (st == LCP_UNVERIFIED) {
    g.sync();
    stats[0] = stats[1] = stats[2] = 0;
    { B2M_PROF_T0(m);
#ifdef __CUDACC__
      if constexpr (G::size >= 32) {
        if (cx.ladder) {
          LadderCtx LC = *(const LadderCtx*)cx.ladder;
          if (m.prof && P.tap_times) LC.dbg = m.dbg;
          st = lcp_lemke_regularized_pool(g, LC, n, m.MM, n, m.qq, -1.0, -1.0, -20, 1, 1, m.z, &piv, stats);
        }
        else st = lcp_lemke_regularized(g, n, m.MM, n, m.qq, -1.0, -1.0, -20, 1, 1, m.z, m.work, m.iwork, &piv, stats, bud);
      } else
#endif
      st = lcp_lemke_regularized(g, n, m.MM, n, m.qq, -1.0, -1.0, -20, 1, 1, m.z, m.work, m.iwork, &piv, stats, bud);   // :222-225
      B2M_PROF_ADD(m, g, PH_LEMKE); }
    if (st == LCP_DEFER) return false;
    B2M_STAMP(PH_BUILD);                                                             // after the Lemke ladder
    lemke_calls = stats[0]; pivots += stats[1]; executed += stats[2];
    if (st == LCP_UNVERIFIED) { for (int i = g.tid; i < n; i += G::size) m.z[i] = 0.0; if (g.tid == 0) { lc[CNT_LCP_FAIL]++; m.scal[S_FAILED] = 1; } }
  }
  g.sync();
  if (g.tid == 0) {
    lc[CNT_LCP_SOLVES]++; lc[CNT_FAST_CALLS] += fast_calls; lc[CNT_LEMKE_CALLS] += lemke_calls; lc[CNT_PIVOTS] += pivots;
    lc[CNT_PIVOT_FLOPS] += (unsigned long long)executed * 2ull * n * (n + 1);   // iterations that really ran (cycle detector)
    m.scal[S_EXEC] += (int)executed;
    if ((unsigned long long)n > lc[CNT_MAX_N]) lc[CNT_MAX_N] = n;
    m.scal[S_ZLN] = n; m.scal[S_ZLDIRTY] = 1;
  }
  for (int i = g.tid; i < n; i += G::size) m.zl[i] = m.z[i];                        // :233 _zlast = z
  if (P.tap_n) {
    if (g.tid == 0) P.tap_n[e] = n;
    for (int t = g.tid; t < n * n; t += G::size) P.tap_MM[(size_t)e * P.nmax * P.nmax + t] = m.MM[t];
    for (int i = g.tid; i < n; i += G::size) { P.tap_qq[(size_t)e * P.nmax + i] = m.qq[i]; P.tap_z[(size_t)e * P.nmax + i] = m.z[i]; }
  }
  for (int i = g.tid; i < nc; i += G::size) {                                       // update_from_stacked_qp
    m.imp[i] = m.z[i];
    m.imp[nc + i] = m.z[nc + i] - m.z[3 * nc + i];
    m.imp[2 * nc + i] = m.z[2 * nc + i] - m.z[4 * nc + i];
  }
  g.sync();
  return true;
}

// apply_model_to_connected_constraints (ImpactConstraintHandler.cpp:530-626)
template <class G>
B2M_DEV bool apply_qp_model(const G& g, const SimParams& P, int e, EnvMem& m, unsigned long long* lc, EnvCtx& cx) {
  const int nc = m.scal[S_NC];
  if (!solve_qp(g, P, e, m, lc, cx)) return false;
  B2M_PROF_T0(m);
  apply_to_bodies(g, P, m, m.imp);
  update_constraint_velocities(g, m, m.imp);
  const double minv = min_constraint_velocity(g, m);
  B2M_PROF_ADD(m, g, PH_APPLY);
  bool changed = false;                                           // apply_restitution(epd, z) :470-491 (H3: friction kept)
  for (int i = g.tid; i < nc; i += G::size) {
    const double c = m.imp[i] * m.ceps[m.icon[i]];
    m.imp[i] = c;
    if (c > B2M_NEAR_ZERO) changed = true;
  }
  changed = g.any(changed);
  g.sync();
  if (changed) {
    apply_to_bodies(g, P, m, m.imp);
    update_constraint_velocities(g, m, m.imp);
    const double minv_plus = min_constraint_velocity(g, m);
    if (minv_plus < 0.0 && minv_plus < minv - B2M_NEAR_ZERO) {
      if (!solve_qp(g, P, e, m, lc, cx)) return false;
      apply_to_bodies(g, P, m, m.imp);
    }
  }
  return true;
}

// apply_ap_model (ImpactConstraintHandlerLCP.cpp:94-370): imp = this solve, acc += imp (propagate_impulse_data)
template <class G>
B2M_DEV B2M_NOINL bool solve_ap(const G& g, const SimParams& P, int e, EnvMem& m, unsigned long long* lc, EnvCtx& cx) {
  const int NC = m.scal[S_NC];
  const int n = build_ap_lcp(g, P, m);
  if (n > P.nmax) { if (g.tid == 0) { lc[CNT_OVERFLOW]++; } for (int t = g.tid; t < 3 * NC; t += G::size) m.imp[t] = 0.0; g.sync(); return true; }
  long long stats[3] = {0, 0, 0};
  int piv = 0;
  int st = lcp_lemke_regularized(g, n, m.MM, n, m.qq, -1.0, -1.0, -20, 1, -2, m.z, m.work, m.iwork, &piv, stats, cx.limit ? &cx.budget : nullptr);   // :333
  if (st == LCP_DEFER) return false;
  if (st == LCP_UNVERIFIED) { for (int i = g.tid; i < n; i += G::size) m.z[i] = 0.0; if (g.tid == 0) { lc[CNT_LCP_FAIL]++; m.scal[S_FAILED] = 1; } }
  g.sync();
  if (g.tid == 0) {
    lc[CNT_LCP_SOLVES]++; lc[CNT_LEMKE_CALLS] += stats[0]; lc[CNT_PIVOTS] += stats[1];
    lc[CNT_PIVOT_FLOPS] += (unsigned long long)stats[2] * 2ull * n * (n + 1);
    m.scal[S_EXEC] += (int)stats[2];
    if ((unsigned long long)n > lc[CNT_MAX_N]) lc[CNT_MAX_N] = n;
  }
  if (P.tap_n) {
    if (g.tid == 0) P.tap_n[e] = n;
    for (int t = g.tid; t < n * n; t += G::size) P.tap_MM[(size_t)e * P.nmax * P.nmax + t] = m.MM[t];
    for (int i = g.tid; i < n; i += G::size) { P.tap_qq[(size_t)e * P.nmax + i] = m.qq[i]; P.tap_z[(size_t)e * P.nmax + i] = m.z[i]; }
  }
  for (int i = g.tid; i < NC; i += G::size) {                     // :336-342
    m.imp[i] = m.z[i];
    m.imp[NC + i] = m.z[NC + i] - m.z[2 * NC + i];
    m.imp[2 * NC + i] = m.z[3 * NC + i] - m.z[4 * NC + i];
    for (int d = 0; d < 3; d++) m.acc[d * NC + i] += m.imp[d * NC + i];
  }
  g.sync();
  return true;
}

template <class G>
B2M_DEV bool apply_ap_model(const G& g, const SimParams& P, int e, EnvMem& m, unsigned long long* lc, EnvCtx& cx) {   // ImpactConstraintHandlerLCP.cpp:36-91
  const int nc = m.scal[S_NC];
  for (int t = g.tid; t < 3 * nc; t += G::size) m.acc[t] = 0.0;
  g.sync();
  if (!solve_ap(g, P, e, m, lc, cx)) return false;
  update_constraint_velocities(g, m, m.imp);
  const double minv = min_constraint_velocity(g, m);
  bool changed = false;                                           // apply_restitution(q) :497-524
  for (int i = g.tid; i < nc; i += G::size) {
    const double c = m.imp[i] * m.ceps[m.icon[i]];
    m.imp[i] = c;
    if (c > B2M_NEAR_ZERO) changed = true;
  }
  changed = g.any(changed);
  g.sync();
  if (changed) {
    for (int i = g.tid; i < nc; i += G::size) { m.imp[nc + i] = 0.0; m.imp[2 * nc + i] = 0.0; }
    g.sync();
    update_constraint_velocities(g, m, m.imp);
    const double minv_plus = min_constraint_velocity(g, m);
    if (minv_plus < 0.0 && minv_plus < minv - B2M_NEAR_ZERO) { if (!solve_ap(g, P, e, m, lc, cx)) return false; }
    else { for (int t = g.tid; t < 3 * nc; t += G::size) m.acc[t] += m.imp[t]; g.sync(); }
  }
  apply_to_bodies(g, P, m, m.acc);                                // apply_impulses (:676-748): accumulated contact impulses
  return true;
}

// the "check" matrix [[S X S^T, S X T^T], [T X S^T, T X T^T]] over the chosen tangent indices (:1098-1112)
template <class G>
B2M_DEV void noslip_form_Y(const G& g, const EnvMem& m, int nc, const int* Si, int ns, const int* Ti, int nt, double skew, double* Y) {
  const int mm = ns + nt;
  for (int t = g.tid; t < mm * mm; t += G::size) {
    const int a = t % mm, b = t / mm;
    double v;
    if (a < ns && b < ns) v = Dn(m, nc, 1, 1, Si[a], Si[b]);
    else if (a >= ns && b >= ns) v = Dn(m, nc, 2, 2, Ti[a - ns], Ti[b - ns]);
    else if (a < ns) v = Dn(m, nc, 1, 2, Si[a], Ti[b - ns]);
    else v = Dn(m, nc, 1, 2, Si[b], Ti[a - ns]);
    if (a == b) v -= skew;
    Y[t] = v;
  }
  g.sync();
}

// apply_no_slip_model (ImpactConstraintHandler.cpp:1009-1417), nl = 0, no implicit joints: greedy full-rank tangent set by
// trial Cholesky (:1089-1145), Schur-complement LCP in the normal impulses (:1170-1236), lcp_fast with the
// lcp_lemke_regularized fallback (:1239-1284), back-substituted tangent impulses (:1294-1308), velocity update (:1370-1400).
// The scratch matrices live in the island's (unused) QP LCP buffer: 9 nc^2 + 5 nc doubles <= (8 nc)^2.
template <class G>
B2M_DEV B2M_NOINL void apply_no_slip_model(const G& g, const SimParams& P, int e, EnvMem& m, unsigned long long* lc) {
  const int nc = m.scal[S_NC];
  double* Y = m.MM; double* QXW = Y + (size_t)4 * nc * nc; double* WM = QXW + (size_t)2 * nc * nc; double* LM = WM + (size_t)2 * nc * nc;
  double* YXv = LM + (size_t)nc * nc; double* wv = YXv + 2 * nc;
  int* Si = m.frow_c; int* Ti = m.frow_j;
  int ns = 0, nt = 0;
  for (int i = 0; i < nc; i++) {
    if (g.tid == 0) Si[ns] = i;
    g.sync();
    noslip_form_Y(g, m, nc, Si, ns + 1, Ti, nt, B2M_NEAR_ZERO, Y);
    if (chol_factor_group(g, Y, ns + 1 + nt)) ns++;                       // :1115-1116
    g.sync();
    if (g.tid == 0) Ti[nt] = i;
    g.sync();
    noslip_form_Y(g, m, nc, Si, ns, Ti, nt + 1, B2M_NEAR_ZERO, Y);
    if (chol_factor_group(g, Y, ns + nt + 1)) nt++;                       // :1140-1141
    g.sync();
  }
  const int mm = ns + nt;
  noslip_form_Y(g, m, nc, Si, ns, Ti, nt, 0.0, Y);                        // :1165-1176
  const bool ok = (mm == 0) || chol_factor_group(g, Y, mm);               // :1179
  for (int t = g.tid; t < nc * mm; t += G::size) {                       // Q X W^T (:1195-1204), nc x mm column-major
    const int i = t % nc, a = t / nc;
    QXW[t] = (a < ns) ? Dn(m, nc, 0, 1, i, Si[a]) : Dn(m, nc, 0, 2, i, Ti[a - ns]);
  }
  g.sync();
  for (int i = g.tid; i < nc; i += G::size) {                            // Y (W X Q^T), one column per thread (:1207-1208)
    for (int a = 0; a < mm; a++) WM[(size_t)i * mm + a] = QXW[(size_t)a * nc + i];
    if (ok && mm) chol_solve1(Y, mm, WM + (size_t)i * mm);
  }
  if (g.tid == 0) {
    for (int a = 0; a < ns; a++) YXv[a] = m.Cv[nc + Si[a]];              // :1220-1224
    for (int b = 0; b < nt; b++) YXv[ns + b] = m.Cv[2 * nc + Ti[b]];
    if (ok && mm) chol_solve1(Y, mm, YXv);                               // :1227-1228
  }
  g.sync();
  for (int t = g.tid; t < nc * nc; t += G::size) {
    const int i = t % nc, j = t / nc;
    double s = 0.0;
    for (int a = 0; a < mm; a++) s = fma(QXW[(size_t)a * nc + i], WM[(size_t)j * mm + a], s);   // :1211
    LM[t] = Dn(m, nc, 0, 0, i, j) - s;                                   // :1212
  }
  for (int i = g.tid; i < nc; i += G::size) {
    double s = 0.0;
    for (int a = 0; a < mm; a++) s = fma(QXW[(size_t)a * nc + i], YXv[a], s);   // :1231
    m.qq[i] = m.Cv[i] - s;                                               // :1215-1216,1234
  }
  const bool warm = (m.scal[S_VLN] == nc);                               // the member _v (rule H1 extended)
  for (int i = g.tid; i < nc; i += G::size) m.z[i] = warm ? m.vl[i] : 0.0;
  g.sync();
  int piv = 0, ex = 0;
  long long fast_calls = 0, lemke_calls = 0, pivots = 0, executed = 0;
  bool solved = false;
  if (ok) {
    const int st = lcp_fast_solve(g, nc, LM, nc, m.qq, 0.0, -1.0, warm, m.z, m.work, m.iwork, &piv, nullptr, 0, nullptr, nullptr, &ex);   // :1239
    fast_calls = 1; pivots = piv; executed = ex;
    solved = (st == LCP_OK || st == LCP_TRIVIAL);
    if (!solved) {
      g.sync();
      long long stats[3] = {0, 0, 0};
      const int st2 = lcp_lemke_regularized(g, nc, LM, nc, m.qq, -1.0, -1.0, -20, 1, 1, m.z, m.work, m.iwork, &piv, stats, nullptr);   // :1279
      lemke_calls = stats[0]; pivots += stats[1]; executed += stats[2];
      solved = (st2 != LCP_UNVERIFIED);
    }
  }
  g.sync();
  if (!solved) { for (int i = g.tid; i < nc; i += G::size) m.z[i] = 0.0; g.sync(); }
  if (g.tid == 0) {
    if (!solved) { lc[CNT_LCP_FAIL]++; m.scal[S_FAILED] = 1; }
    lc[CNT_LCP_SOLVES]++; lc[CNT_FAST_CALLS] += fast_calls; lc[CNT_LEMKE_CALLS] += lemke_calls; lc[CNT_PIVOTS] += pivots;
    lc[CNT_PIVOT_FLOPS] += (unsigned long long)executed * 2ull * nc * (nc + 1);
    m.scal[S_EXEC] += (int)executed;
    if ((unsigned long long)nc > lc[CNT_MAX_N]) lc[CNT_MAX_N] = nc;
    m.scal[S_VLN] = nc; m.scal[S_VLDIRTY] = 1;
  }
  for (int i = g.tid; i < nc; i += G::size) m.vl[i] = m.z[i];
  if (P.tap_n) {
    if (g.tid == 0) P.tap_n[e] = nc;
    for (int t = g.tid; t < nc * nc; t += G::size) P.tap_MM[(size_t)e * P.nmax * P.nmax + t] = LM[t];
    for (int i = g.tid; i < nc; i += G::size) { P.tap_qq[(size_t)e * P.nmax + i] = m.qq[i]; P.tap_z[(size_t)e * P.nmax + i] = m.z[i]; }
  }
  // [cs; ct] = -(Y W v + Y W X Q^T cn) (:1294-1299)
  for (int a = g.tid; a < mm; a += G::size) { double s = 0.0; for (int i = 0; i < nc; i++) s = fma(QXW[(size_t)a * nc + i], m.z[i], s); wv[a] = s; }
  for (int i = g.tid; i < nc; i += G::size) { m.imp[i] = m.z[i]; m.imp[nc + i] = 0.0; m.imp[2 * nc + i] = 0.0; }
  g.sync();
  if (g.tid == 0 && solved) {
    if (ok && mm) chol_solve1(Y, mm, wv);
    for (int a = 0; a < ns; a++) m.imp[nc + Si[a]] = -(YXv[a] + wv[a]);
    for (int b = 0; b < nt; b++) m.imp[2 * nc + Ti[b]] = -(YXv[ns + b] + wv[ns + b]);
  }
  g.sync();
  apply_to_bodies(g, P, m, m.imp);                                       // :1370-1400
}

// apply_no_slip_model_to_connected_constraints (ImpactConstraintHandler.cpp:236-293); rule H10: the trailing
// update_from_stacked(_epd, _z) with the QP handler's stale _z (:288) is skipped.
template <class G>
B2M_DEV void apply_no_slip_to_connected(const G& g, const SimParams& P, int e, EnvMem& m, unsigned long long* lc) {
  const int nc = m.scal[S_NC];
  apply_no_slip_model(g, P, e, m, lc);
  update_constraint_velocities(g, m, m.imp);                             // :262
  const double minv = min_constraint_velocity(g, m);
  bool changed = false;                                                  // apply_restitution(q) :497-524
  for (int i = g.tid; i < nc; i += G::size) {
    const double c = m.imp[i] * m.ceps[m.icon[i]];
    m.imp[i] = c;
    if (c > B2M_NEAR_ZERO) changed = true;
  }
  changed = g.any(changed);
  g.sync();
  if (changed) {
    for (int i = g.tid; i < nc; i += G::size) { m.imp[nc + i] = 0.0; m.imp[2 * nc + i] = 0.0; }
    g.sync();
    apply_to_bodies(g, P, m, m.imp);                                     // update_from_stacked(q) :271
    update_constraint_velocities(g, m, m.imp);                           // :274
    const double minv_plus = min_constraint_velocity(g, m);
    if (minv_plus < 0.0 && minv_plus < minv - B2M_NEAR_ZERO) apply_no_slip_model(g, P, e, m, lc);   // :281-285
  }
}

// Islands (UnilateralConstraint.cpp:940-1194) with the canonical order of rule H4: seeds in ascending body index,
// neighbours in contact (edge insertion) order, each visited body picks up its remaining contacts in list order.
// only_active: keep the islands that hold an impacting constraint (remove_inactive_groups :1197-1225); the mask of kept
// islands goes to scal[S_FLAG].  Executed by ONE thread.
B2M_HD B2M_NOINL inline void build_islands(const SimParams& P, EnvMem& m, int ncon, bool only_active) {
  const int nb = P.nb;
  unsigned nodes = 0;
  for (int c = 0; c < ncon; c++) { if (m.ben[m.cb1[c]]) nodes |= 1u << super_of(P, m.cb1[c]); if (m.ben[m.cb2[c]]) nodes |= 1u << super_of(P, m.cb2[c]); }
  for (int b = 0; b < nb; b++) m.bisl[b] = -1;
  for (int c = 0; c < ncon; c++) m.cisl[c] = -1;
  int nisl = 0, nord = 0;
  unsigned active = 0;
  int queue[B200MOBY_MAX_BODIES];
  while (nodes) {
    int node = 0; while (!((nodes >> node) & 1u)) node++;
    int qh = 0, qt = 0; unsigned processed = 0, queued = 1u << node;
    queue[qt++] = node;
    m.isl_start[nisl] = nord;
    while (qh < qt) {
      node = queue[qh++];
      nodes &= ~(1u << node);
      processed |= 1u << node;
      m.bisl[node] = nisl;
      for (int c = 0; c < ncon; c++) {
        if (!(m.ben[m.cb1[c]] && m.ben[m.cb2[c]])) continue;
        const int b1 = super_of(P, m.cb1[c]), b2 = super_of(P, m.cb2[c]);
        const int nbr = (b1 == node) ? b2 : ((b2 == node) ? b1 : -1);
        if (nbr >= 0 && !((queued >> nbr) & 1u)) { queued |= 1u << nbr; queue[qt++] = nbr; }
      }
      for (int c = 0; c < ncon; c++)
        if (m.cisl[c] < 0 && ((m.ben[m.cb1[c]] && super_of(P, m.cb1[c]) == node) || (m.ben[m.cb2[c]] && super_of(P, m.cb2[c]) == node))) { m.cisl[c] = nisl; m.corder[nord++] = c; }
    }
    nisl++;
  }
  m.isl_start[nisl] = nord;
  if (only_active) { for (int c = 0; c < ncon; c++) if (constraint_vel(m, c) < -B2M_NEAR_ZERO) active |= 1u << m.cisl[c]; }
  else active = (nisl >= 32) ? 0xffffffffu : ((1u << nisl) - 1u);
  m.scal[S_NISL] = nisl;
  m.scal[S_FLAG] = (int)active;
}

// contacts, generalized-coordinate offsets and counts of island k (after build_islands).  Executed by ONE thread.
B2M_HD B2M_NOINL inline void select_island(const SimParams& P, EnvMem& m, int k) {
  const int nb = P.nb;
  const int s0 = m.isl_start[k], nc = m.isl_start[k + 1] - s0;
  for (int i = 0; i < nc; i++) m.icon[i] = m.corder[s0 + i];
  int gc = 0;
  for (int b = 0; b < nb; b++) {
    if (is_link(P, b)) {                      // every moving link shares the articulated body's coordinates
      const int rep = P.rc_first + 1;
      if (b == rep) {
        if (m.bisl[rep] == k) { m.gcoff[b] = gc; for (int l = 0; l < P.rc_links - 1; l++) { m.gcb[gc + l] = rep; m.gcl[gc + l] = l; } gc += P.rc_links - 1; }
        else m.gcoff[b] = -1;
      } else m.gcoff[b] = m.gcoff[rep];
    } else if (m.bisl[b] == k && m.ben[b]) {
      m.gcoff[b] = gc;
      if (B2M_NGC(P)) for (int l = 0; l < 6; l++) { m.gcb[gc + l] = b; m.gcl[gc + l] = l; }
      gc += 6;
    } else m.gcoff[b] = -1;
  }
  m.scal[S_NC] = nc; m.scal[S_NGC] = gc;
}

// calc_impacting_unilateral_constraint_forces (ConstraintSimulator.cpp:298-355) -> apply_model (ImpactConstraintHandler.cpp:96-168)
template <class G>
B2M_DEV B2M_NOINL bool process_constraints(const G& g, const SimParams& P, int e, EnvMem& m, unsigned long long* lc, EnvCtx& cx) {
  const int ncon = m.scal[S_NCON], nb = P.nb;
  if (ncon == 0) return true;
  bool impacting = false;
  for (int c = g.tid; c < ncon; c += G::size) if (constraint_vel(m, c) < -B2M_NEAR_ZERO) impacting = true;
  if (!g.any(impacting)) return true;
  B2M_PROF_T0(m);
  if (g.tid == 0) build_islands(P, m, ncon, true);
  g.sync();
  B2M_PROF_ADD(m, g, PH_ISLANDS);
  const int nisl = m.scal[S_NISL];
  const unsigned active = (unsigned)m.scal[S_FLAG];
  for (int k = 0; k < nisl; k++) {
    if (!((active >> k) & 1u)) continue;
    if (g.tid == 0) select_island(P, m, k);
    g.sync();
    { B2M_PROF_T0(m); compute_problem_data(g, P, m); B2M_PROF_ADD(m, g, PH_PROBLEM); }
    if (g.tid == 0) {   // SURVEY.md 8(d): F_delassus = 2 (3nc) 36 b + 2 (3nc)^2 6, F_apply = 2 NGC 3nc
      const unsigned long long nc = m.scal[S_NC], ngc = m.scal[S_NGC];
      unsigned long long blocks = 0;
      for (unsigned i = 0; i < nc; i++) blocks += (m.ben[m.cb1[m.icon[i]]] ? 1 : 0) + (m.ben[m.cb2[m.icon[i]]] ? 1 : 0);
      lc[CNT_ASM_FLOPS] += 2 * 3 * 36 * blocks + 2 * (3 * nc) * (3 * nc) * 6 + 2 * ngc * 3 * nc;
    }
    bool all_inf = true;                                             // ImpactConstraintHandler.cpp:122-135
    for (int i = g.tid; i < m.scal[S_NC]; i += G::size) if (m.cmu[m.icon[i]] < 1e2) all_inf = false;
    all_inf = !g.any(!all_inf);
    if (all_inf) apply_no_slip_to_connected(g, P, e, m, lc);
    else if (!(P.model == 1 ? apply_ap_model(g, P, e, m, lc, cx) : apply_qp_model(g, P, e, m, lc, cx))) return false;
    g.sync();
  }
  // ImpactToleranceException check over the solved islands (:153-167): counted, never fatal
  bool still = false;
  for (int c = g.tid; c < ncon; c += G::size) if (((active >> m.cisl[c]) & 1u) && constraint_vel(m, c) < -B2M_NEAR_ZERO) still = true;
  if (g.any(still) && g.tid == 0) lc[CNT_IMPACT_TOL]++;
  return true;
}

// First half of TimeSteppingSimulator::do_mini_step (:114-209): positions with conservative advancement, forward
// dynamics + velocity update, distances, contacts.  Returns h; `impacting` says whether the constraint handler has
// work to do (ConstraintSimulator.cpp:298-355 / ImpactConstraintHandler.cpp:96-120 early-outs).
template <class G>
B2M_DEV double mini_step_advance(const G& g, const SimParams& P, int e, EnvMem& m, double dt, double t, unsigned long long* lc, bool& impacting) {
  const double h = integrate_positions_CA(g, P, e, m, dt, lc);
  fwd_dyn_integrate_velocity(g, P, m, h, t);
  calc_pairwise_distances(g, m);
  find_unilateral_constraints(g, P, e, m, lc);
  const int ncon = m.scal[S_NCON];
  bool imp = false;
  for (int c = g.tid; c < ncon; c += G::size) if (constraint_vel(m, c) < -B2M_NEAR_ZERO) imp = true;
  impacting = g.any(imp);
  return h;
}

// bookkeeping at the end of a mini-step
template <class G>
B2M_DEV void mini_step_account(const G& g, const SimParams& P, const EnvMem& m, unsigned long long* lc) {
  if (g.tid == 0) {     // F_fd = 60 per free body (Newton-Euler); F_narrow = 8 vertices x 20 (box) or 20 (sphere) per pair and distance pass
    lc[CNT_MINI_STEPS]++;
    unsigned long long f = 0;
    for (int b = 0; b < P.nb; b++) if (m.ben[b] && !is_link(P, b)) f += 60;
    if (B2M_RC(P)) f += 500ull * (P.rc_links - 1);   // ABA, Featherstone's operation count (SURVEY.md 8d)
    for (int p = 0; p < m.scal[S_NPAIRS]; p++) f += 3 * ((m.bshape[m.pair_a[p]] == SH_BOX || m.bshape[m.pair_b[p]] == SH_BOX) ? 160 : 20);
    lc[CNT_ASM_FLOPS] += f;
  }
}

// LCP dimension the env's contacts give if they all fall into one island (upper bound of every island's n): picks the
// shared-memory class of the impact kernel.
B2M_HD B2M_INL int contacts_lcp_dim(const EnvMem& m, int ncon, int model) {
  int n = 0;
  bool all_inf = true;
  for (int c = 0; c < ncon; c++) { const int nk = m.cNK[c]; n += (model == 1) ? 5 + (nk > 4 ? (nk + 4) / 4 : 1) : 6 + nk / 2; if (m.cmu[c] < 1e2) all_inf = false; }
  // every island of the env takes the no-slip model: its LCP is nc x nc and its scratch 9 nc^2 + 5 nc doubles of the LCP
  // buffer, which (3 nc + 2)^2 covers -- a much smaller class than the QP / A-P dimension
  if (all_inf && 3 * ncon + 2 < n) n = 3 * ncon + 2;
  return n;
}

// TimeSteppingSimulator::do_mini_step (:114-222); returns h, or -1 when the env is deferred
template <class G>
B2M_DEV double do_mini_step(const G& g, const SimParams& P, int e, EnvMem& m, double dt, double t, unsigned long long* lc, EnvCtx& cx) {
  bool impacting;
  if (g.tid == 0) m.scal[S_FAILED] = 0;
  const double h = mini_step_advance(g, P, e, m, dt, t, lc, impacting);
  if (impacting && !process_constraints(g, P, e, m, lc, cx)) return -1.0;
  mini_step_account(g, P, m, lc);
  return h;
}

// The rest of one TimeSteppingSimulator::step (:433-455) from `h` seconds into it; the env is loaded.  Returns false when deferred.
template <class G>
B2M_DEV bool env_finish_step(const G& g, const SimParams& P, int e, EnvMem& m, double dt, double h, double& t, unsigned long long* lc, EnvCtx& cx) {
  int stalled = 0;
  while (h < dt) {
    const double hh = do_mini_step(g, P, e, m, dt - h, t, lc, cx);
    if (hh < 0.0) return false;
    h += hh; t += hh;
    // The reference loops here until time advances (TimeSteppingSimulator.cpp:439-441) and leaves through an exception
    // when an impact cannot be resolved (ImpactConstraintHandlerQP.cpp:224).  A batch cannot throw: after
    // B2M_MAX_STALL zero-length mini-steps in a row the env gives up the rest of this step and is counted as failed.
    stalled = (hh > 0.0) ? 0 : stalled + 1;
    if (stalled >= B2M_MAX_STALL) { if (g.tid == 0) lc[CNT_LCP_FAIL]++; break; }
    // An unsolved LCP in a zero-length mini-step is where the reference leaves through LCPSolverException: the env gives
    // up the rest of this step at once (the failure is already counted) instead of repeating the same solve.
    g.sync();
    if (hh == 0.0 && m.scal[S_FAILED]) break;
  }
  if (g.tid == 0) lc[CNT_ENV_STEPS]++;
  return true;
}

// n_steps x TimeSteppingSimulator::step (:52-111, :433-455) for env e; stabilization disabled.
// Returns false (and leaves the env's stored state untouched) when the env ran out of its pivot budget.
template <class G>
B2M_DEV bool env_run(const G& g, const SimParams& P, int e, EnvMem& m, double dt, int n_steps, unsigned long long* lc, EnvCtx& cx) {
  env_load(g, P, e, m);
  double t = P.time[e];
  const EnvStatBase sb = env_stat_base(lc);
  for (int s = 0; s < n_steps; s++)
    if (!env_finish_step(g, P, e, m, dt, 0.0, t, lc, cx)) return false;
  env_stat_commit(g, P, e, lc, sb);
  g.sync();
  env_store(g, P, e, m);
  if (g.tid == 0) P.time[e] = t;
  g.sync();
  return true;
}

// ---------------- phased step: advance -> impact (per LCP class) -> advance ... -> finish ----------------
// Most env-steps never need an LCP (free flight, resting without approach velocity): the advance phase runs them with
// the small working set only, so dozens of envs are resident per SM.  An env whose contacts are impacting is parked
// after the first half of its mini-step and queued by the LCP dimension its contacts give; the impact phase picks it
// up with a working set of exactly that class.  Same functions, same arithmetic and the same order of operations per
// env as the fused loop above -- results are bit-identical.
B2M_HD B2M_INL int* q_count(const SimParams& P, int round, int slot) { return P.qctl + round * (B2M_SLOTS + 1) + slot; }
B2M_HD B2M_INL int* q_head(const SimParams& P, int round, int slot) { return P.qctl + (B2M_ROUNDS_MAX + round) * (B2M_SLOTS + 1) + slot; }
B2M_HD B2M_INL int* q_list(const SimParams& P, int round, int slot) { return P.queue + ((size_t)round * B2M_SLOTS + slot) * P.n_envs; }
B2M_DEV B2M_INL int b2m_atomic_inc(int* p) {
#ifdef __CUDA_ARCH__
  return atomicAdd(p, 1);
#else
  return (*p)++;
#endif
}
B2M_DEV B2M_INL void q_push(const SimParams& P, int round, int slot, int e) { q_list(P, round, slot)[b2m_atomic_inc(q_count(P, round, slot))] = e; }
// hard queue: longest jobs first.  `front` entries grow from index 0, the others from the end of the list.
B2M_DEV B2M_INL void q_push_hard(const SimParams& P, int round, int e, bool front) {
  int* list = q_list(P, round, B2M_SLOT_HARD);
  if (front) list[b2m_atomic_inc(q_count(P, round, B2M_SLOT_HARD))] = e;
  else list[P.n_envs - 1 - b2m_atomic_inc(q_count(P, round, B2M_SLOT_HARD_BACK))] = e;
}
// number of entries of a queue slot and its i-th entry in pull order
B2M_HD B2M_INL int q_size(const SimParams& P, int round, int slot) { return *q_count(P, round, slot) + (slot == B2M_SLOT_HARD ? *q_count(P, round, B2M_SLOT_HARD_BACK) : 0); }
B2M_HD B2M_INL int q_at(const SimParams& P, int round, int slot, int i) {
  const int* list = q_list(P, round, slot);
  if (slot != B2M_SLOT_HARD) return list[i];
  const int nf = *q_count(P, round, B2M_SLOT_HARD);
  return i < nf ? list[i] : list[P.n_envs - 1 - (i - nf)];
}

// Advance env e through its step until it completes or needs an impact solve.  `m` carries the small segment only.
template <class G>
B2M_DEV void env_advance(const G& g, const SimParams& P, int e, EnvMem& m, double dt, int round, unsigned long long* lc) {
  env_load(g, P, e, m);
  double t = P.time[e];
  double h = (round == 0) ? 0.0 : P.hacc[e];
  bool parked = false;
  while (h < dt) {
    bool impacting;
    const double hh = mini_step_advance(g, P, e, m, dt - h, t, lc, impacting);
    if (impacting) {
      if (g.tid == 0) {
        P.hacc[e] = h; P.hpend[e] = hh;
        const int ncon = m.scal[S_NCON];
        const int n = contacts_lcp_dim(m, ncon, P.model);
        int cls = 0;
        while (cls < P.n_classes - 1 && (n > P.class_nmax[cls] || ncon > P.class_cmax[cls])) cls++;
        const int hc = P.class_budget[cls] > P.hard_cost ? P.class_budget[cls] : P.hard_cost;   // small classes afford more iterations per env (an iteration costs ~n^2..n^3)
        if (P.cost && P.hard_cost > 0 && P.cost[e] >= hc) q_push_hard(P, round, e, P.cost[e] >= 8 * P.hard_cost);
        else q_push(P, round, cls, e);
      }
      parked = true;
      break;
    }
    mini_step_account(g, P, m, lc);
    h += hh; t += hh;
  }
  if (!parked && g.tid == 0) lc[CNT_ENV_STEPS]++;
  g.sync();
  env_store(g, P, e, m, ST_POS | ST_VEL);
  if (g.tid == 0) P.time[e] = t;
  g.sync();
}

// Second half of the parked mini-step: contacts again from the stored state (same inputs, same results), islands,
// assembly, solve, impulses.  P.cmax / P.nmax are the class's.  Returns false when the env ran over its pivot budget
// (nothing stored; it is queued for the straggler kernel).
template <class G>
B2M_DEV bool env_impact(const G& g, const SimParams& P, int e, EnvMem& m, double dt, int round, unsigned long long* lc, EnvCtx& cx) {
#ifdef __CUDA_ARCH__
  const long long t0 = P.tap_prof ? clock64() : 0;
  long long gt0 = 0;
  if (P.tap_prof && P.tap_times) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt0));
#endif
  const unsigned long long p0 = lc[CNT_PIVOTS], f0 = lc[CNT_PIVOT_FLOPS];
  const EnvStatBase sb = env_stat_base(lc);
  m.prof = P.tap_prof ? P.tap_prof + (size_t)4 * P.n_envs + e : nullptr; m.prof_stride = P.n_envs;
  { B2M_PROF_T0(m); env_load(g, P, e, m); B2M_PROF_ADD(m, g, PH_LOAD); }
  const unsigned long long c0 = lc[CNT_CONTACTS], o0 = lc[CNT_OVERFLOW];
  if (g.tid == 0) { m.scal[S_FAILED] = 0; m.scal[S_EXEC] = 0; }
  m.dbg[0] = m.dbg[1] = m.dbg[2] = m.dbg[3] = 0;
  { B2M_PROF_T0(m);
  calc_pairwise_distances(g, m);
  find_unilateral_constraints(g, P, e, m, lc);
  B2M_PROF_ADD(m, g, PH_CONTACTS); }
  lc[CNT_CONTACTS] = c0; lc[CNT_OVERFLOW] = o0;                  // counted by the advance phase
  if (!process_constraints(g, P, e, m, lc, cx)) {
    // only an env that ran out of its budget is marked expensive: one handed on after its first lcp_fast rung keeps its cost
    // history (marked, ~1,400 such envs per step of configs[1] would sit in the hard queue for several steps and lengthen it)
    if (g.tid == 0) { const int hc = P.pivot_budget > P.hard_cost ? P.pivot_budget : P.hard_cost; q_push(P, round, B2M_SLOT_STRAGGLER, e); if (P.cost && cx.budget < 0 && P.cost[e] < 4 * hc) P.cost[e] = 4 * hc; }
    g.sync();
    return false;
  }
  mini_step_account(g, P, m, lc);
  env_stat_commit(g, P, e, lc, sb);
  g.sync();
  { B2M_PROF_T0(m); env_store(g, P, e, m, ST_VEL | ST_ZL); B2M_PROF_ADD(m, g, PH_STORE); }
  if (g.tid == 0) {
    const double hh = P.hpend[e];
    const double h = P.hacc[e] + hh;
    P.time[e] = P.time[e] + hh;
    if (h < dt && !(hh == 0.0 && m.scal[S_FAILED])) { P.hacc[e] = h; q_push(P, round, B2M_SLOT_CONT, e); }
    else lc[CNT_ENV_STEPS]++;        // done, or given up after an unsolved LCP in a zero-length mini-step
    if (P.cost) { const int prev = P.cost[e], dec = prev - (prev >> P.cost_shift); P.cost[e] = m.scal[S_EXEC] > dec ? m.scal[S_EXEC] : dec; }   // sticky: a hard env stays in the hard queue for a few steps
#ifdef __CUDA_ARCH__
    if (P.tap_prof) {
      const size_t ne = P.n_envs;
      const long long n = m.scal[S_N];
      P.tap_prof[e] = clock64() - t0; P.tap_prof[ne + e] = (long long)(lc[CNT_PIVOTS] - p0);
      P.tap_prof[2 * ne + e] = n > 0 ? (long long)((lc[CNT_PIVOT_FLOPS] - f0) / (2ull * n * (n + 1))) : 0; P.tap_prof[3 * ne + e] = n + 1000ll * P.kslot;   // LCP dimension + 1000 x the kernel slot that ran the env
      if (P.tap_times) {   // timeline mode: the islands / store rows carry the env's start / end on the global timer (ns) instead
        long long gt1; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt1));
        P.tap_prof[(4 + PH_ISLANDS) * ne + e] = gt0; P.tap_prof[(4 + PH_STORE) * ne + e] = gt1;
        P.tap_prof[(4 + PH_APPLY) * ne + e] = m.dbg[0]; P.tap_prof[(4 + PH_LOAD) * ne + e] = m.dbg[1]; P.tap_prof[(4 + PH_LEMKE) * ne + e] = m.dbg[2] + 1000 * m.dbg[3];
      }
    }
#endif
  }
  g.sync();
  return true;
}

// Whatever is left of env e's step after the last round, with the fused loop (full working set).
template <class G>
B2M_DEV void env_finish(const G& g, const SimParams& P, int e, EnvMem& m, double dt, unsigned long long* lc) {
  env_load(g, P, e, m);
  double t = P.time[e];
  EnvCtx cx; cx.limit = false; cx.budget = 0;
  const EnvStatBase sb = env_stat_base(lc);
  env_finish_step(g, P, e, m, dt, P.hacc[e], t, lc, cx);
  env_stat_commit(g, P, e, lc, sb);
  g.sync();
  env_store(g, P, e, m);
  if (g.tid == 0) P.time[e] = t;
  g.sync();
}

#include "stab_device.cuh"

}  // namespace b2m
