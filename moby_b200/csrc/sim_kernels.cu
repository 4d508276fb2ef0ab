// Simulator handle, the fused env-step kernel and the stage kernels behind the C ABI (include/b200moby.h).
// b200moby_step replaces TimeSteppingSimulator::step (Moby src/TimeSteppingSimulator.cpp:52-111) for a batch of
// independent envs: one warp per env, the whole mini-step loop (narrowphase, conservative advancement, forward
// dynamics, assembly, LCP solve, impulses) runs out of shared memory; HBM sees the state and the warm start only.
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <nvtx3/nvToolsExt.h>   // header-only NVTX v3: ranges are no-ops unless a profiler (nsys / ncu --nvtx) is attached
#include "friction_table.h"
#include "host_util.h"
#include "sim_kernel_util.cuh"
#include "rc_host.h"

using namespace b2m;

#define B2M_SMEM_MAX (227 * 1024 - 1024)   /* dynamic shared memory we ask for at most: the opt-in limit minus the kernels' static reduction scratch */

struct ClassPlan {
  int nmax = 0, cmax = 0;
  int threads = 32;          // 32: warp-per-env kernel (wpb warps per block); > 32: one block per env; 1: thread per env (b2m_k_impact_thread(tvariant))
  int tvariant = -1;
  int wpb = 1, grid = 1;
  size_t shmem = 0;
  double* gscratch = nullptr;   // non-null: the working set exceeds shared memory and lives in this global buffer
  size_t gstride = 0;
};

// live handles per device: the hard-queue launch waits for work from launches on other streams (k_impact_warp.cu), which is only
// safe while no other handle's launches can sit between them in a hardware queue (with more streams than
// CUDA_DEVICE_MAX_CONNECTIONS, streams share queues and a launch can be stuck behind another handle's blocked one)
static std::atomic<int> g_live_handles[64];

struct b200moby_sim {
  int device = 0;
  int n_envs = 0, nb = 0, cmax = 0, nmax = 0, npmax = 0;
  SimParams P;
  std::vector<void*> allocs;
  size_t env_d = 0, env_i = 0;
  int wpb = 1, grid = 1, sms = 148;
  size_t shmem = 0;          // full working set of one env (stage kernels, finish kernel)
  bool taps = false;
  bool stage_attr_set = false;
  // phased step plan
  int rounds = 2;
  int adv_wpb = 4, adv_grid = 1; size_t adv_shmem = 0;
  int thread_budget = 12;    // solver iterations a thread-per-env impact may spend on one env before deferring it
  int adv_thread = -1;       // >= 0: the advance phase runs one thread per env (b2m_k_advance_thread(adv_thread)); -1: warp per env
  std::vector<ClassPlan> classes;
  // one step captured as a CUDA graph (b200moby_step): ~25 launches, memsets and the stream fork / join of a step become
  // one cudaGraphLaunch.  Captured on an internal stream; re-captured when dt or anything in SimParams changes.
  cudaGraphExec_t graph_exec = nullptr; cudaStream_t graph_stream = nullptr;
  SimParams graph_P; double graph_dt = 0.0; bool graph_feed = false; long long graph_launches = 0; bool graph_on = true; int graph_captures = 0;
  int* stab_queue = nullptr; // [n_envs + 1] envs selected for stabilization this step, then their count (k_stabilize.cu)
  int* feed_ctr = nullptr;   // [B2M_ROUNDS_MAX] class launches completed in the round (k_impact_warp.cu: the hard-queue launch takes their stragglers)
  bool all_thread_classes = false, any_subwarp_class = false;
  LadderPool pool;           // task pool of the Lemke ladder (lcp_device.cuh) for the hard-queue / straggler launches; ctl == nullptr: off
  int pool_owners = 0;
  ClassPlan straggler;       // full-size kernel (warp per env while the scene's LCPs fit one, else a 256-thread block) for envs over their pivot budget and for the hard queue
  ClassPlan fullws;          // scratch of the full-working-set warp kernels (finish, fused, stage) when it exceeds shared memory
  int fin_grid = 1;
  ClassPlan finblock;        // nmax > B200MOBY_BIG_N: the finish phase runs one 256-thread block per env (threads == 256 when in use)
  bool any_thread_class = false;
  // constraint stabilization phase (k_stabilize.cu): thread-per-env variant, or -1 = warp per env over `stab_scratch`
  int stab_variant = -1, stab_grid = 1; double* stab_scratch = nullptr; size_t stab_stride = 0, stab_nd_env = 0, stab_nd_all = 0;
  int stab_proc_grid = 1;    // thread-per-env process launch: every block that can be resident at once
  bool fused = false;        // B200MOBY_FUSED=1: the single fused warp-per-env kernel (kept for comparison)
  long long launches = 0;
  // the impact classes of one round touch disjoint envs: they run on side streams so that the tail of one class
  // (a few envs with very long pivot sequences) overlaps the other classes' work
  bool concurrent = true;
  std::vector<cudaStream_t> side;
  std::vector<cudaEvent_t> side_done;
  cudaEvent_t fork = nullptr;
  cudaStream_t hard_stream = nullptr; cudaEvent_t hard_done = nullptr;   // the hard queue's launch
  int rc_links = 0, rc_dof = 0;   // articulated body (0: none)
  // per-kernel profile (b200moby_get_kernel_profile): slot 0 advance, 1..n impact classes, n+1 stragglers, n+2 finish
  bool ktiming = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> kev_free;
  std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> kev_pending;
  std::vector<double> kms; std::vector<long long> klaunches;
};

namespace {

// stage kernels: same device functions, one warp per env, results written out instead of carried on
enum { STAGE_FWD_DYN = 0, STAGE_CONTACTS = 1, STAGE_DELASSUS = 2 };
struct StageOut {
  double dt;
  int cap; int* count; double* point; double* normal; double* tan1; double* tan2; int* pair; double* dist;
  int nmax_out; double* MM; double* qq; int* n;
};

__global__ void __launch_bounds__(256) stage_warp_kernel(SimParams P, int stage, StageOut o, int wpb, size_t env_d, size_t env_i) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int w = threadIdx.x >> 5;
  EnvMem m;
  env_mem_full(P, m, smem, w, wpb);
  WarpGroup g(nullptr);
  unsigned long long lc[CNT_COUNT];
  for (int k = 0; k < CNT_COUNT; k++) lc[k] = 0;
  const int ne = P.n_envs;
  for (int e = blockIdx.x * wpb + w; e < ne; e += gridDim.x * wpb) {
    env_load(g, P, e, m);
    if (stage == STAGE_FWD_DYN) {
      fwd_dyn_integrate_velocity(g, P, m, o.dt, P.time[e]);
      for (int k = g.tid; k < 3 * P.nb; k += 32) { const int b = k / 3, c = k - 3 * b; if (m.ben[b]) { P.v[((size_t)b * 6 + c) * ne + e] = m.bvl[k]; P.v[((size_t)b * 6 + 3 + c) * ne + e] = m.bva[k]; } }
    } else {
      calc_pairwise_distances(g, m);
      find_unilateral_constraints(g, P, e, m, lc);
      const int ncon = m.scal[S_NCON];
      if (stage == STAGE_CONTACTS) {
        if (g.tid == 0) o.count[e] = ncon;
        for (int c = g.tid; c < ncon && c < o.cap; c += 32) {
          for (int k = 0; k < 3; k++) {
            o.point[((size_t)c * 3 + k) * ne + e] = m.cp[3 * c + k]; o.normal[((size_t)c * 3 + k) * ne + e] = m.cnrm[3 * c + k];
            o.tan1[((size_t)c * 3 + k) * ne + e] = m.ct1[3 * c + k]; o.tan2[((size_t)c * 3 + k) * ne + e] = m.ct2[3 * c + k];
          }
          o.pair[(size_t)c * ne + e] = m.cb1[c] * P.nb + m.cb2[c];
          o.dist[(size_t)c * ne + e] = m.cdist[c];
        }
      } else {
        int n = 0;
        if (ncon > 0) {
          if (g.tid == 0) {            // all contacts of the env as one island, generation order (matches the checker's helper)
            for (int c = 0; c < ncon; c++) m.icon[c] = c;
            int gc = 0;
            for (int b = 0; b < P.nb; b++) {
              bool in = false;
              for (int c = 0; c < ncon; c++) if (m.cb1[c] == b || m.cb2[c] == b) in = true;
              if (in && m.ben[b]) { m.gcoff[b] = gc; gc += 6; } else m.gcoff[b] = -1;
            }
            m.scal[S_NC] = ncon; m.scal[S_NGC] = gc;
          }
          g.sync();
          compute_problem_data(g, P, m);
          n = (P.model == 1) ? build_ap_lcp(g, P, m) : build_qp_lcp(g, P, m);
          if (n <= P.nmax && n <= o.nmax_out) {
            for (int t = g.tid; t < n * n; t += 32) o.MM[(size_t)e * o.nmax_out * o.nmax_out + t] = m.MM[t];
            for (int i = g.tid; i < n; i += 32) o.qq[(size_t)e * o.nmax_out + i] = m.qq[i];
          }
        }
        if (g.tid == 0) o.n[e] = n;
      }
    }
    g.sync();
  }
}

// set_generalized_coordinates_euler normalises the quaternion it is given (Ravelin RigidBodyd); done once here so
// the kernels can trust the stored state.
__global__ void normalize_quat_kernel(double* q, int nb, int ne) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nb * ne) return;
  const int b = t / ne, e = t - b * ne;
  double* p = q + ((size_t)b * 7 + 3) * ne + e;
  const double x = p[0], y = p[ne], z = p[2 * (size_t)ne], w = p[3 * (size_t)ne];
  const double nrm = sqrt(x * x + y * y + z * z + w * w);
  p[0] = x / nrm; p[ne] = y / nrm; p[2 * (size_t)ne] = z / nrm; p[3 * (size_t)ne] = w / nrm;
}

template <class T>
b200moby_status dev_copy(b200moby_sim* h, const T* src, size_t count, const T** dst) {
  T* d = nullptr;
  B2M_CUDA(cudaMalloc((void**)&d, std::max<size_t>(count, 1) * sizeof(T)));
  h->allocs.push_back(d);
  if (count) B2M_CUDA(cudaMemcpy(d, src, count * sizeof(T), cudaMemcpyHostToDevice));
  *dst = d;
  return B200MOBY_OK;
}
template <class T>
b200moby_status dev_zero(b200moby_sim* h, size_t count, T** dst) {
  T* d = nullptr;
  B2M_CUDA(cudaMalloc((void**)&d, std::max<size_t>(count, 1) * sizeof(T)));
  h->allocs.push_back(d);
  B2M_CUDA(cudaMemset(d, 0, std::max<size_t>(count, 1) * sizeof(T)));
  *dst = d;
  return B200MOBY_OK;
}

const void* impact_block_ptr(int nt) { return nt == 64 ? b2m_k_impact_block64() : (nt == 128 ? b2m_k_impact_block128() : b2m_k_impact_block256()); }

int env_int(const char* name, int dflt) { const char* s = getenv(name); return s ? atoi(s) : dflt; }

b200moby_status plan_grid(const void* kernel, int threads, size_t shmem, int sms, int work, int* grid) {
  B2M_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B2M_SMEM_MAX));
  int per_sm = 0;
  B2M_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, shmem));
  if (per_sm < 1) return b2m_fail(B200MOBY_ERR_UNSUPPORTED, "kernel does not fit an SM (%d threads, %zu bytes of shared memory)", threads, shmem);
  *grid = std::max(1, std::min(work, sms * per_sm));
  return B200MOBY_OK;
}

// Shared memory a kernel needs for `slots` working sets of `per` bytes, or -- when one working set does not fit an SM --
// a global scratch buffer with one slice per resident group (cp.gscratch / cp.gstride; the launch then asks for no
// dynamic shared memory).
b200moby_status plan_memory(b200moby_sim* h, const void* kernel, ClassPlan& cp, int slots_max, int work) {
  EnvDims D = env_dims(h->P); D.cmax = cp.cmax; D.nmax = cp.nmax;
  const size_t ed = (env_doubles(D) + 1) & ~(size_t)1, ei = (env_ints(D) + 3) & ~(size_t)3;
  const size_t per = ed * sizeof(double) + ei * sizeof(int);
  b200moby_status st;
  if (per <= B2M_SMEM_MAX) {
    cp.wpb = 1;
    if (cp.threads == 32) {   // warps per block that put the most envs on an SM (228 KB per SM, 1 KB reserved per block); ties: the wider block
      size_t best = 0;
      for (int w = 1; w <= slots_max && per * w <= B2M_SMEM_MAX; w++) {
        const size_t blocks = std::min<size_t>(32, (size_t)(228 * 1024) / (per * w + 1024));
        if (blocks * w >= best) { best = blocks * w; cp.wpb = w; }
      }
    }
    cp.shmem = per * cp.wpb;
    return plan_grid(kernel, cp.threads == 32 ? cp.wpb * 32 : cp.threads, cp.shmem, h->sms, (work + cp.wpb - 1) / cp.wpb, &cp.grid);
  }
  cp.wpb = (cp.threads == 32) ? slots_max : 1;
  cp.shmem = 0;
  if ((st = plan_grid(kernel, cp.threads == 32 ? cp.wpb * 32 : cp.threads, 0, h->sms, (work + cp.wpb - 1) / cp.wpb, &cp.grid)) != B200MOBY_OK) return st;
  cp.gstride = ed + (ei + 1) / 2;
  const size_t total = cp.gstride * (size_t)cp.grid * cp.wpb;
  double* buf = nullptr;
  B2M_CUDA(cudaMalloc((void**)&buf, total * sizeof(double)));
  h->allocs.push_back(buf);
  cp.gscratch = buf;
  return B200MOBY_OK;
}

// Launch plan of the phased step: grids are persistent (SMs x resident blocks, capped by the batch) and pull env
// indices from the queues, so empty queues cost one short launch.
b200moby_status plan_launch(b200moby_sim* h) {
  int sms = 0;
  B2M_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
  h->sms = sms;
  const int nb = h->nb, ne = h->n_envs;
  const EnvDims D0 = env_dims(h->P);
  h->env_d = (env_doubles(D0) + 1) & ~(size_t)1;
  h->env_i = (env_ints(D0) + 3) & ~(size_t)3;
  h->fused = env_int("B200MOBY_FUSED", 0) != 0;
  h->rounds = std::max(1, std::min(B2M_ROUNDS_MAX, env_int("B200MOBY_ROUNDS", 2)));
  b200moby_status st;
  // full working set, one env per warp-sized block: finish kernel, fused comparison kernel, stage kernels
  {
    ClassPlan& f = h->fullws;
    f.nmax = h->nmax; f.cmax = h->cmax; f.threads = 32;
    B2M_CUDA(cudaFuncSetAttribute(b2m_k_step_warp(), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B2M_SMEM_MAX));
    if ((st = plan_memory(h, b2m_k_finish(), f, 1, ne)) != B200MOBY_OK) return st;
    h->shmem = f.shmem; h->wpb = 1; h->grid = f.gscratch ? f.grid : ne; h->fin_grid = f.grid;
    h->P.gscratch = f.gscratch; h->P.gstride = f.gstride;
  }
  // advance: warps_per_block envs per block, small segment only
  {
    const size_t sd = (env_small_doubles(D0) + 1) & ~(size_t)1, si = (env_small_ints(D0) + 3) & ~(size_t)3;
    const size_t per = sd * sizeof(double) + si * sizeof(int);
    int wpb = env_int("B200MOBY_ADV_WPB", 4);
    while (wpb > 1 && per * wpb > B2M_SMEM_MAX) wpb--;
    if (per > B2M_SMEM_MAX) return b2m_fail(B200MOBY_ERR_UNSUPPORTED, "advance working set (%zu bytes) exceeds one SM's shared memory", per);
    h->adv_wpb = wpb; h->adv_shmem = per * wpb;
    if ((st = plan_grid(b2m_k_advance(), wpb * 32, h->adv_shmem, sms, (ne + wpb - 1) / wpb, &h->adv_grid)) != B200MOBY_OK) return st;
    // thread per env when the small working set fits one of the compiled local-memory sizes (B200MOBY_ADV_THREAD=0: off)
    h->adv_thread = -1;
    if (env_int("B200MOBY_ADV_THREAD", 1) != 0) {
      const size_t nd = env_small_doubles(D0), ni = env_small_ints(D0);
      if (nd <= 256 && ni <= 64) h->adv_thread = 0;
      else if (nd <= 1024 && ni <= 256) h->adv_thread = 1;
      else if (nd <= 4096 && ni <= 1024) h->adv_thread = 2;
    }
  }
  // impact classes by LCP dimension
  {
    const int warp_nmax = env_int("B200MOBY_WARP_NMAX", 40); // classes up to this n: warp per env; above: block per env
    const int bthreads = env_int("B200MOBY_IMPACT_THREADS", 64);
    const int big_n = env_int("B200MOBY_BIG_N", 96);          // classes above this n always get 256 threads per env
    const int ncls = b2m_class_table(h->nmax, h->cmax, h->P.model, B2M_MAX_CLASSES, h->P.class_nmax, h->P.class_cmax);
    h->classes.clear();
    for (int k = 0; k < ncls; k++) {
      ClassPlan c; c.nmax = h->P.class_nmax[k]; c.cmax = h->P.class_cmax[k];
      {   // thread per env when the class's working set fits a compiled local-memory size (B200MOBY_IMPACT_THREAD=0: off)
        EnvDims Dc = env_dims(h->P); Dc.cmax = c.cmax; Dc.nmax = c.nmax;
        const size_t nd = env_doubles(Dc), ni = env_ints(Dc);
        if (env_int("B200MOBY_IMPACT_THREAD", 1) != 0 && c.nmax <= env_int("B200MOBY_THREAD_NMAX", 40)) {
          if (nd <= B2M_THREAD_ND0 && ni <= B2M_THREAD_NI0) c.tvariant = 0;
          else if (nd <= B2M_THREAD_ND1 && ni <= B2M_THREAD_NI1) c.tvariant = 1;
        }
      }
      if (c.tvariant >= 0 && c.nmax <= env_int("B200MOBY_SUBWARP_NMAX", 0) && !B2M_RC(h->P)) {   // small classes: eight lanes per env, four envs per warp (k_impact_warp.cu)
        EnvDims Dc = env_dims(h->P); Dc.cmax = c.cmax; Dc.nmax = c.nmax;
        const size_t ed = (env_doubles(Dc) + 1) & ~(size_t)1, ei = (env_ints(Dc) + 3) & ~(size_t)3, per = ed * sizeof(double) + ei * sizeof(int);
        c.threads = 8; c.tvariant = -1; c.wpb = 1; c.shmem = per * 4;
        if (c.shmem <= 100 * 1024) {
          if ((st = plan_grid(b2m_k_impact_subwarp8(), 32, c.shmem, sms, (ne + 3) / 4, &c.grid)) != B200MOBY_OK) return st;
          h->any_subwarp_class = true;
          h->classes.push_back(c); continue;
        }
        c.threads = 32; c.tvariant = -1;                          // does not fit: fall through to the warp kernel
      }
      if (c.tvariant >= 0) {
        const int lanes = std::max(1, std::min(32, env_int("B200MOBY_THREAD_LANES", 32)));
        h->P.thread_lanes = lanes;
        c.threads = 1; c.grid = std::max(1, std::min((ne + 4 * lanes - 1) / (4 * lanes), sms * 16 * (32 / lanes)));
        h->classes.push_back(c); continue;
      }
      if (c.nmax <= warp_nmax || bthreads <= 32) c.threads = 32;
      else if (c.nmax > big_n) c.threads = 256;
      else c.threads = bthreads <= 64 ? 64 : (bthreads <= 128 ? 128 : 256);
      const void* kern = c.threads == 32 ? b2m_k_impact_warp() : impact_block_ptr(c.threads);
      if ((st = plan_memory(h, kern, c, 4, ne)) != B200MOBY_OK) return st;
      h->classes.push_back(c);
    }
    h->P.n_classes = (int)h->classes.size();
    for (const ClassPlan& c : h->classes) if (c.threads == 1 || c.threads == 8) h->any_thread_class = true;
    h->all_thread_classes = true;
    for (const ClassPlan& c : h->classes) if (c.threads != 1 && c.threads != 8) h->all_thread_classes = false;   // thread- and sub-warp classes can run beside the hard queue (the latter in the shared memory it is made to leave)
    if (env_int("B200MOBY_FEED", 1) != 0) { b200moby_status s3; if ((s3 = dev_zero(h, (size_t)B2M_ROUNDS_MAX, &h->feed_ctr)) != B200MOBY_OK) return s3; }
    h->thread_budget = env_int("B200MOBY_THREAD_BUDGET", 12);
    {   // per-class budget: base x (40 / n)^p, at most 8 x base (an iteration of a small LCP is cheap, so a small class can keep envs the n <= 40 class must hand on)
      const double pw = env_int("B200MOBY_BUDGET_POW10", 15) / 10.0;   // measured on configs[1]: 0 -> 6.89, 1.0 -> 7.16, 1.5 -> 7.27, 2.5 -> 5.34 M env-steps/s
      for (size_t k = 0; k < h->classes.size(); k++) {
        const double f = h->classes[k].nmax < 40 ? std::pow(40.0 / h->classes[k].nmax, pw) : 1.0;
        h->P.class_budget[k] = (h->classes[k].threads == 1 || h->classes[k].threads == 8) ? (int)std::min(8.0 * h->thread_budget, std::floor(h->thread_budget * f)) : 0;
      }
    }
    ClassPlan& sg = h->straggler;
    // stragglers and the hard queue want the shortest latency per pivot for one env: measured on configs[1] (n <= 40),
    // the worst env's chain takes 16 ms on a lone warp and 6.7 ms on a 256-thread block
    sg.nmax = h->nmax; sg.cmax = h->cmax; sg.threads = env_int("B200MOBY_STRAGGLER_THREADS", h->nmax > big_n ? 256 : (h->nmax <= 64 ? 32 : 128));   // n <= 64: the warp-owned pivot loops (lcp_device.cuh), no block barriers   // n = 320 stack LCPs: 2.0 s (256) against 4.3 s (128) per step of 256 envs
    if (sg.threads != 32 && sg.threads != 64 && sg.threads != 128) sg.threads = 256;
    // block per env with the Lemke ladder's rungs as tasks (n in the hundreds): a full grid even for a small batch, the blocks
    // without an env of their own take rungs
    const int sg_work = (sg.threads != 32 && h->nmax > 64 && h->P.model == 0 && env_int("B200MOBY_LADDER", 1) != 0) ? std::max(ne, sms * 8) : ne;
    if ((st = plan_memory(h, sg.threads == 32 ? b2m_k_impact_warp() : impact_block_ptr(sg.threads), sg, 4, sg_work)) != B200MOBY_OK) return st;
    { const int cap = env_int("B200MOBY_HARD_BLOCKS_PER_SM", h->any_subwarp_class ? 1 : 0);      // experiment knob: fewer resident warps of the hard-queue launch per SM (less contention for the shared-memory pipe)
      if (cap > 0 && sg.grid > sms * cap) sg.grid = sms * cap;
      if (env_int("B200MOBY_PLAN_DEBUG", 0)) fprintf(stderr, "[b200moby] hard/straggler plan: threads %d wpb %d grid %d (%d SMs) shmem %zu\n", sg.threads, sg.wpb, sg.grid, sms, sg.shmem); }
    // the Lemke ladder as a task pool: one job buffer per warp of the hard-queue / straggler launches
    memset(&h->pool, 0, sizeof(h->pool));
    // (warp per env, n <= 64) or one per block (n in the hundreds: 0.9 MB per block at n = 320)
    const bool warp_pool = sg.threads == 32 && !sg.gscratch && h->nmax <= 64, block_pool = sg.threads != 32 && h->nmax > 64;
    if ((warp_pool || block_pool) && h->P.model == 0 && env_int("B200MOBY_LADDER", 1) != 0) {
      LadderPool& L = h->pool;
      h->pool_owners = sg.threads == 32 ? sg.grid * sg.wpb : sg.grid;
      L.nmax = h->nmax; L.cap = h->pool_owners * 64;
      L.job_stride = ladder_job_doubles(h->nmax); L.meta_stride = ladder_job_ints();
      b200moby_status s2;
      if ((s2 = dev_zero(h, (size_t)4, &L.ctl)) != B200MOBY_OK) return s2;
      if ((s2 = dev_zero(h, (size_t)L.cap, &L.tasks)) != B200MOBY_OK) return s2;
      if ((s2 = dev_zero(h, (size_t)L.cap, &L.task_gen)) != B200MOBY_OK) return s2;
      if ((s2 = dev_zero(h, L.job_stride * h->pool_owners, &L.jobs)) != B200MOBY_OK) return s2;
      if ((s2 = dev_zero(h, L.meta_stride * h->pool_owners, &L.meta)) != B200MOBY_OK) return s2;
      if ((s2 = dev_zero(h, (size_t)4 * h->pool_owners, &L.jobd)) != B200MOBY_OK) return s2;
    }
    // Large LCPs (n in the hundreds): a warp would spend seconds per solve, so whatever the rounds leave over is finished
    // by one block per env, and more rounds keep that remainder small (each extra round is a handful of short launches).
    h->finblock.threads = 32;
    if (h->nmax > big_n) {
      ClassPlan& fb = h->finblock;
      fb.nmax = h->nmax; fb.cmax = h->cmax; fb.threads = 256;
      if ((st = plan_memory(h, b2m_k_finish_block256(), fb, 1, ne)) != B200MOBY_OK) return st;
      h->rounds = std::max(1, std::min(B2M_ROUNDS_MAX, env_int("B200MOBY_ROUNDS", 4)));
    }
  }
  if (h->P.stab_max_iterations != 0) {
    SimParams Ps = h->P; Ps.nmax = Ps.cmax;                   // the stabilization LCP has one row per contact
    const EnvDims Ds = env_dims(Ps);
    const size_t nd = env_doubles(Ds), ni = env_ints(Ds), xd = stab_extra_doubles(Ds), xi = stab_extra_ints(Ds);
    h->stab_nd_env = nd; h->stab_nd_all = (nd + xd + 1) & ~(size_t)1;
    const bool thr = env_int("B200MOBY_STAB_THREAD", 1) != 0;
    if (thr && nd + xd <= B2M_STAB_ND0 && ni + xi <= B2M_STAB_NI0) h->stab_variant = 0;
    else if (thr && nd + xd <= B2M_STAB_ND1 && ni + xi <= B2M_STAB_NI1) h->stab_variant = 1;
    else {
      h->stab_variant = -1;
      h->stab_grid = std::max(1, std::min((ne + 3) / 4, sms * 8));
      h->stab_stride = h->stab_nd_all + (ni + xi + 1) / 2;
      B2M_CUDA(cudaMalloc((void**)&h->stab_scratch, h->stab_stride * (size_t)h->stab_grid * 4 * sizeof(double)));
      h->allocs.push_back(h->stab_scratch);
    }
    if (h->stab_variant >= 0) {
      int per_sm = 0;
      B2M_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, b2m_k_stabilize_thread(h->stab_variant), 128, 0));
      if (per_sm < 1) return b2m_fail(B200MOBY_ERR_UNSUPPORTED, "stabilization kernel does not fit an SM");
      h->stab_proc_grid = sms * per_sm;
    }
    if (h->stab_variant >= 0 && env_int("B200MOBY_STAB_SELECT", 1) != 0) {
      b200moby_status s4;
      if ((s4 = dev_zero(h, (size_t)ne + 1, &h->stab_queue)) != B200MOBY_OK) return s4;
      if (env_int("B200MOBY_STAB_PROCESS_WARP", 0) != 0) {
        h->stab_grid = std::max(1, std::min((ne + 3) / 4, sms * 8));
        h->stab_stride = h->stab_nd_all + (ni + xi + 1) / 2;
        B2M_CUDA(cudaMalloc((void**)&h->stab_scratch, h->stab_stride * (size_t)h->stab_grid * 4 * sizeof(double)));
        h->allocs.push_back(h->stab_scratch);
      }
    }
  }
  return B200MOBY_OK;
}

// launch with optional event bracketing on the launch's own stream (per-kernel durations for bench.py's roofline block)
b200moby_status timed_launch(b200moby_sim* h, int kslot, const void* kernel, dim3 grid, dim3 block, void** args, size_t shmem, cudaStream_t s) {
  std::pair<cudaEvent_t, cudaEvent_t> ev(nullptr, nullptr);
  if (h->ktiming) {
    if (h->kev_free.empty()) { B2M_CUDA(cudaEventCreate(&ev.first)); B2M_CUDA(cudaEventCreate(&ev.second)); }
    else { ev = h->kev_free.back(); h->kev_free.pop_back(); }
    B2M_CUDA(cudaEventRecord(ev.first, s));
  }
  B2M_CUDA(cudaLaunchKernel(kernel, grid, block, args, shmem, s));
  if (h->ktiming) { B2M_CUDA(cudaEventRecord(ev.second, s)); h->kev_pending.push_back(std::make_pair(kslot, ev)); }
  h->launches++;
  return B200MOBY_OK;
}

// one launch of an impact kernel (warp per env or block per env, per the plan) over queue `slot`; pool: the launch runs
// the rungs of the Lemke ladder as tasks (lcp_device.cuh) -- its task list is cleared on the launch's stream first
b200moby_status launch_impact(b200moby_sim* h, int kslot, const ClassPlan& cp, SimParams& Pk, double dt, int r, int slot, bool pool, cudaStream_t sc, bool feed = false) {
  Pk.gscratch = cp.gscratch; Pk.gstride = cp.gstride; Pk.kslot = kslot;
  if (cp.threads == 32) {
    LadderPool L; memset(&L, 0, sizeof(L));
    if (pool && h->pool.ctl && cp.grid * cp.wpb <= h->pool_owners) {
      L = h->pool;
      B2M_CUDA(cudaMemsetAsync(L.ctl, 0, sizeof(int) * 4, sc));
      B2M_CUDA(cudaMemsetAsync(L.tasks, 0, sizeof(int) * L.cap, sc));
    }
    int wpb = cp.wpb;
    int feed_slot = feed ? B2M_SLOT_STRAGGLER : -1, feed_expect = (int)h->classes.size();
    int* feed_done = h->feed_ctr ? h->feed_ctr + r : nullptr;
    void* a[] = {&Pk, &dt, &r, &slot, &wpb, &L, &feed_slot, &feed_done, &feed_expect};
    return timed_launch(h, kslot, b2m_k_impact_warp(), dim3(cp.grid), dim3(cp.wpb * 32), a, cp.shmem, sc);
  }
  LadderPool L; memset(&L, 0, sizeof(L));
  if (pool && h->pool.ctl && h->straggler.threads == cp.threads && cp.grid <= h->pool_owners) {
    L = h->pool;
    B2M_CUDA(cudaMemsetAsync(L.ctl, 0, sizeof(int) * 4, sc));
    B2M_CUDA(cudaMemsetAsync(L.tasks, 0, sizeof(int) * L.cap, sc));
  }
  void* a[] = {&Pk, &dt, &r, &slot, &L};
  return timed_launch(h, kslot, impact_block_ptr(cp.threads), dim3(cp.grid), dim3(cp.threads), a, cp.shmem, sc);
}

// ConstraintStabilization::stabilize for every env (TimeSteppingSimulator.cpp:95-98), after the step's last kernel
b200moby_status launch_stabilize(b200moby_sim* h, cudaStream_t s) {
  if (h->P.stab_max_iterations == 0) return B200MOBY_OK;
  const int ncls = (int)h->classes.size();
  SimParams Ps = h->P; Ps.nmax = Ps.cmax; Ps.kslot = 4 + ncls;
  if (h->stab_variant >= 0) {
    const int blocks = std::max(1, std::min((h->n_envs + 127) / 128, h->sms * 16));
    int mode = 1; int* queue = nullptr; int* count = nullptr;
    if (h->stab_queue) {                                     // select, then stabilize the selected envs only (k_stabilize.cu)
      mode = 0; queue = h->stab_queue; count = h->stab_queue + h->n_envs;
      B2M_CUDA(cudaMemsetAsync(count, 0, sizeof(int), s));
      void* a0[] = {&Ps, &mode, &queue, &count};
      b200moby_status st = timed_launch(h, 4 + ncls, b2m_k_stabilize_thread(h->stab_variant), dim3(blocks), dim3(128), a0, 0, s);
      if (st != B200MOBY_OK) return st;
      mode = 1;
    }
    if (queue && h->stab_scratch) {                          // selected envs by warps (B200MOBY_STAB_PROCESS_WARP=1)
      Ps.gscratch = h->stab_scratch; Ps.gstride = h->stab_stride;
      void* aw[] = {&Ps, &h->stab_nd_env, &h->stab_nd_all, &queue, &count};
      return timed_launch(h, 4 + ncls, b2m_k_stabilize_warp(), dim3(h->stab_grid), dim3(128), aw, 0, s);
    }
    void* a[] = {&Ps, &mode, &queue, &count};
    return timed_launch(h, 4 + ncls, b2m_k_stabilize_thread(h->stab_variant), dim3(h->stab_proc_grid), dim3(128), a, 0, s);
  }
  Ps.gscratch = h->stab_scratch; Ps.gstride = h->stab_stride;
  int* queue = nullptr; int* count = nullptr;
  void* a[] = {&Ps, &h->stab_nd_env, &h->stab_nd_all, &queue, &count};
  return timed_launch(h, 4 + ncls, b2m_k_stabilize_warp(), dim3(h->stab_grid), dim3(128), a, 0, s);
}

// NVTX range per phase of a step (the equivalent of the reference's FILE_LOG sections, SURVEY.md section 5), on the enqueuing
// host thread; with graphs the ranges mark the capture, plain launches (B200MOBY_GRAPH=0) mark every step
struct NvtxRange { explicit NvtxRange(const char* name) { nvtxRangePushA(name); } ~NvtxRange() { nvtxRangePop(); } };

bool launch_feeds(const b200moby_sim* h) {
  return h->feed_ctr && h->concurrent && h->classes.size() > 1 && h->all_thread_classes && h->straggler.threads == 32 && h->P.hard_cost > 0 &&
         g_live_handles[h->device & 63].load() == 1;
}

// One TimeSteppingSimulator::step for every env: advance, then per round the impact classes, stragglers and the
// next advance; the finish kernel takes whatever the rounds left over.  All launches are asynchronous on `s`.
b200moby_status launch_step(b200moby_sim* h, double dt, cudaStream_t s) {
  SimParams& P = h->P;
  b200moby_status st;
  const int ncls = (int)h->classes.size();
  B2M_CUDA(cudaMemsetAsync(P.qctl, 0, sizeof(int) * 2 * B2M_ROUNDS_MAX * (B2M_SLOTS + 1), s));
  // the hard-queue launch also takes the stragglers of the classes running next to it (k_impact_warp.cu): only when every
  // class is a thread-per-env launch (no shared memory: they are sure to be resident beside it) on concurrent streams
  const bool feed = launch_feeds(h);
  if (feed) {
    B2M_CUDA(cudaMemsetAsync(h->feed_ctr, 0, sizeof(int) * B2M_ROUNDS_MAX, s));
    for (int r = 0; r < h->rounds; r++) B2M_CUDA(cudaMemsetAsync(q_list(P, r, B2M_SLOT_STRAGGLER), 0xff, sizeof(int) * h->n_envs, s));
  }
  NvtxRange step_range("b200moby step");
  for (int r = 0; r < h->rounds; r++) {
    NvtxRange round_range(r == 0 ? "round 0: advance + impact" : "round n: advance + impact");
    { SimParams Pa = P; Pa.kslot = 0;
      void* a[] = {&Pa, &dt, &r, &h->adv_wpb};
      if (h->adv_thread >= 0) {
        const int blocks = std::max(1, std::min((h->n_envs + 127) / 128, h->sms * 16));
        if ((st = timed_launch(h, 0, b2m_k_advance_thread(h->adv_thread), dim3(blocks), dim3(128), a, 0, s)) != B200MOBY_OK) return st;
      } else if ((st = timed_launch(h, 0, b2m_k_advance(), dim3(h->adv_grid), dim3(h->adv_wpb * 32), a, h->adv_shmem, s)) != B200MOBY_OK) return st; }
    const bool conc = h->concurrent && h->classes.size() > 1;
    if (conc) B2M_CUDA(cudaEventRecord(h->fork, s));
    if (P.hard_cost > 0) {   // the expensive envs first, next to the classes
      SimParams Ph = P; Ph.pivot_budget = 0;
      cudaStream_t sc = conc ? h->hard_stream : s;
      if (conc) B2M_CUDA(cudaStreamWaitEvent(sc, h->fork, 0));
      if ((st = launch_impact(h, 3 + ncls, h->straggler, Ph, dt, r, B2M_SLOT_HARD, true, sc, feed)) != B200MOBY_OK) return st;
      if (conc) { B2M_CUDA(cudaEventRecord(h->hard_done, sc)); B2M_CUDA(cudaStreamWaitEvent(s, h->hard_done, 0)); }
    }
    for (size_t c = 0; c < h->classes.size(); c++) {
      ClassPlan& cp = h->classes[c];
      SimParams Pc = P; Pc.cmax = cp.cmax; Pc.nmax = cp.nmax; Pc.gscratch = cp.gscratch; Pc.gstride = cp.gstride; Pc.kslot = 1 + (int)c;
      int slot = (int)c;
      cudaStream_t sc = conc ? h->side[c] : s;
      if (conc) B2M_CUDA(cudaStreamWaitEvent(sc, h->fork, 0));
      if (cp.threads == 1) {
        Pc.pivot_budget = h->P.class_budget[c] > 0 ? h->P.class_budget[c] : h->thread_budget;
        // the first-rung hand-off pays only while the hard-queue launch takes the envs as they arrive: a straggler launch after
        // every class would run them last (the parts feeder: 4.0 -> 10.9 ms per step)
        if (!feed) Pc.first_rung_handoff = 0;
        void* a[] = {&Pc, &dt, &r, &slot};
        st = timed_launch(h, 1 + (int)c, b2m_k_impact_thread(cp.tvariant), dim3(cp.grid), dim3(128), a, 0, sc);
      } else if (cp.threads == 8) {
        Pc.pivot_budget = h->P.class_budget[c] > 0 ? h->P.class_budget[c] : h->thread_budget;
        int wpb = cp.wpb;
        void* a[] = {&Pc, &dt, &r, &slot, &wpb};
        st = timed_launch(h, 1 + (int)c, b2m_k_impact_subwarp8(), dim3(cp.grid), dim3(cp.wpb * 32), a, cp.shmem, sc);
      } else {
        if (cp.threads != 32) Pc.pivot_budget = 0;
        st = launch_impact(h, 1 + (int)c, cp, Pc, dt, r, slot, false, sc);
      }
      if (st != B200MOBY_OK) return st;
      if (feed) { int* ctr = h->feed_ctr + r; void* sa[] = {&ctr}; B2M_CUDA(cudaLaunchKernel(b2m_k_signal(), dim3(1), dim3(1), sa, 0, sc)); h->launches++; }
      if (conc) { B2M_CUDA(cudaEventRecord(h->side_done[c], sc)); B2M_CUDA(cudaStreamWaitEvent(s, h->side_done[c], 0)); }
    }
    if (P.pivot_budget > 0 || h->any_thread_class) {
      SimParams Ps = P; Ps.pivot_budget = 0;
      if ((st = launch_impact(h, 1 + ncls, h->straggler, Ps, dt, r, B2M_SLOT_STRAGGLER, true, s)) != B200MOBY_OK) return st;
    }
  }
  { int r = h->rounds - 1; SimParams Pf = P; Pf.kslot = 2 + ncls;
    void* a[] = {&Pf, &dt, &r};
    if (h->finblock.threads == 256) {
      Pf.gscratch = h->finblock.gscratch; Pf.gstride = h->finblock.gstride;
      if ((st = timed_launch(h, 2 + ncls, b2m_k_finish_block256(), dim3(h->finblock.grid), dim3(256), a, h->finblock.shmem, s)) != B200MOBY_OK) return st;
    } else if ((st = timed_launch(h, 2 + ncls, b2m_k_finish(), dim3(h->fin_grid), dim3(32), a, h->shmem, s)) != B200MOBY_OK) return st; }
  { NvtxRange stab_range("constraint stabilization");
    if ((st = launch_stabilize(h, s)) != B200MOBY_OK) return st; }
  B2M_CUDA(cudaGetLastError());
  return B200MOBY_OK;
}

}  // namespace

extern "C" {

b200moby_status b200moby_create(const b200moby_scene_desc* d, int device, b200moby_handle* out) {
  if (!d || !out) return b2m_fail(B200MOBY_ERR_INVALID, "null descriptor");
  if (!b2m_have_device()) return b2m_fail(B200MOBY_ERR_NO_DEVICE, "no CUDA device: the hot path has no CPU fallback");
  if (d->n_envs <= 0 || d->n_bodies <= 0 || d->n_bodies > B200MOBY_MAX_BODIES) return b2m_fail(B200MOBY_ERR_INVALID, "n_envs > 0 and 0 < n_bodies <= %d required", B200MOBY_MAX_BODIES);
  B2M_CUDA(cudaSetDevice(device));
  const int ne = d->n_envs, nb = d->n_bodies;
  // validate and size
  int cmax = 0, nmax = 0, npmax = 0;
  if (const char* err = b2m_scene_bounds(d, cmax, nmax, npmax)) return b2m_fail(B200MOBY_ERR_INVALID, "%s", err);
  b200moby_sim* h = new b200moby_sim;
  g_live_handles[device & 63]++;
  h->device = device; h->n_envs = ne; h->nb = nb; h->cmax = std::max(cmax, 1); h->nmax = std::max(nmax, 1); h->npmax = std::max(npmax, 1);
  SimParams& P = h->P;
  memset(&P, 0, sizeof(P));
  P.n_envs = ne; P.nb = nb; P.cmax = h->cmax; P.nmax = h->nmax; P.npmax = h->npmax; P.model = d->impact_model;
  b200moby_status st;
#define TRY(x) if ((st = (x)) != B200MOBY_OK) { b200moby_destroy(h); return st; }
  TRY(dev_copy(h, d->shape, (size_t)nb * ne, &P.shape));
  TRY(dev_copy(h, d->enabled, (size_t)nb * ne, &P.enabled));
  TRY(dev_copy(h, d->mass, (size_t)nb * ne, &P.mass));
  TRY(dev_copy(h, d->dims, (size_t)nb * 3 * ne, &P.dims));
  TRY(dev_copy(h, d->inertia, (size_t)nb * 3 * ne, &P.inertia));
  TRY(dev_copy(h, d->mu_coulomb, (size_t)nb * nb * ne, &P.mu_c));
  TRY(dev_copy(h, d->mu_viscous, (size_t)nb * nb * ne, &P.mu_v));
  TRY(dev_copy(h, d->epsilon, (size_t)nb * nb * ne, &P.eps));
  TRY(dev_copy(h, d->compliance, (size_t)nb * nb * ne, &P.compliance));
  TRY(dev_copy(h, d->NK, (size_t)nb * nb * ne, &P.NK));
  std::vector<double> tab = b2m_friction_table();
  TRY(dev_copy(h, tab.data(), tab.size(), &P.fr_tab));
  P.gx = d->gravity[0]; P.gy = d->gravity[1]; P.gz = d->gravity[2];
  P.contact_dist_thresh = d->contact_dist_thresh; P.min_step_size = d->min_step_size;
  P.stab_max_iterations = d->stabilization_max_iterations; P.stab_eps = B2M_NEAR_ZERO;   // ConstraintStabilization.cpp:53-59 (rule H7)
  if (d->min_step_size_env) TRY(dev_copy(h, d->min_step_size_env, (size_t)ne, &P.min_step_env));
  TRY(dev_zero(h, (size_t)nb * 7 * ne, &P.q));
  TRY(dev_zero(h, (size_t)nb * 6 * ne, &P.v));
  TRY(dev_zero(h, (size_t)ne, &P.time));
  TRY(dev_zero(h, (size_t)h->nmax * ne, &P.zlast));
  TRY(dev_zero(h, (size_t)ne, &P.zlast_n));
  TRY(dev_zero(h, (size_t)h->cmax * ne, &P.vlast));
  TRY(dev_zero(h, (size_t)ne, &P.vlast_n));
  TRY(dev_zero(h, (size_t)CNT_COUNT, &P.counters));
  TRY(dev_zero(h, (size_t)3 * (B2M_MAX_CLASSES + 6), &P.kstat));
  TRY(dev_zero(h, (size_t)ne, &P.cost));
  P.tap_times = env_int("B200MOBY_TAP_TIMES", 0);
  P.hard_cost = env_int("B200MOBY_HARD_COST", 12);
  P.cost_shift = std::max(0, std::min(30, env_int("B200MOBY_COST_DECAY_SHIFT", 2)));
  TRY(dev_zero(h, (size_t)ne, &P.hacc));
  TRY(dev_zero(h, (size_t)ne, &P.hpend));
  TRY(dev_zero(h, (size_t)B2M_ROUNDS_MAX * B2M_SLOTS * ne, &P.queue));
  TRY(dev_zero(h, (size_t)2 * B2M_ROUNDS_MAX * (B2M_SLOTS + 1), &P.qctl));
  P.pivot_budget = env_int("B200MOBY_PIVOT_BUDGET", 96);
  P.first_rung_handoff = env_int("B200MOBY_FIRST_RUNG_HANDOFF", 1) != 0;   // 0: off (comparison runs; results are the same)
  if (d->rc && d->rc->n_links > 0) {
    const b200moby_rc_desc& r = *d->rc;
    RCTree T; bool unsup = false;
    if (const char* err = b2m_rc_tree_from_desc(r, nb, T, &unsup)) { b200moby_destroy(h); return b2m_fail(unsup ? B200MOBY_ERR_UNSUPPORTED : B200MOBY_ERR_INVALID, "%s", err); }
    for (int e = 0; e < ne; e++) {
      if (d->enabled[(size_t)r.first_body * ne + e]) { b200moby_destroy(h); return b2m_fail(B200MOBY_ERR_UNSUPPORTED, "articulated body: floating bases are not on the accelerated path; the base link must be a disabled body"); }
      for (int i = 1; i < r.n_links; i++) if (!d->enabled[(size_t)(r.first_body + i) * ne + e]) { b200moby_destroy(h); return b2m_fail(B200MOBY_ERR_INVALID, "articulated body: link %d is disabled", i); }
    }
    TRY(dev_copy(h, &T, 1, &P.rc));
    P.rc_links = r.n_links; P.rc_first = r.first_body;
    P.ngc = b2m_dense_ngc(d);
    h->rc_links = r.n_links; h->rc_dof = r.n_links - 1;
    TRY(dev_zero(h, (size_t)h->rc_dof * ne, &P.jq));
    TRY(dev_zero(h, (size_t)h->rc_dof * ne, &P.jqd));
    double* tau0 = nullptr;
    TRY(dev_zero(h, (size_t)h->rc_dof * ne, &tau0));
    P.jtau = tau0;
  }
  TRY(plan_launch(h));
  h->concurrent = env_int("B200MOBY_CONCURRENT", 1) != 0;
  // default: graph for the two-round plans (configs[1]: neutral on the device, 13x less host work per step); the four-round
  // plans of scenes with large LCPs are ~50 mostly empty launches per step and ran 10 % slower as graph nodes than as plain
  // stream launches (UR10: 3.5 against 3.2 ms per step, tools/ur10_phases.py)
  h->graph_on = env_int("B200MOBY_GRAPH", h->rounds <= 2 ? 1 : 0) != 0;
  if (h->concurrent) {
    h->side.resize(h->classes.size()); h->side_done.resize(h->classes.size());
    for (size_t c = 0; c < h->classes.size(); c++) { h->side[c] = nullptr; h->side_done[c] = nullptr; }
    for (size_t c = 0; c < h->classes.size(); c++) {
      if (cudaStreamCreateWithFlags(&h->side[c], cudaStreamNonBlocking) != cudaSuccess || cudaEventCreateWithFlags(&h->side_done[c], cudaEventDisableTiming) != cudaSuccess) {
        b200moby_destroy(h); return b2m_fail(B200MOBY_ERR_CUDA, "cannot create the impact-class streams");
      }
    }
    if (cudaStreamCreateWithFlags(&h->hard_stream, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreateWithFlags(&h->hard_done, cudaEventDisableTiming) != cudaSuccess) { b200moby_destroy(h); return b2m_fail(B200MOBY_ERR_CUDA, "cannot create the hard-queue stream"); }
    if (cudaEventCreateWithFlags(&h->fork, cudaEventDisableTiming) != cudaSuccess) { b200moby_destroy(h); return b2m_fail(B200MOBY_ERR_CUDA, "cannot create the fork event"); }
  }
#undef TRY
  *out = h;
  return B200MOBY_OK;
}

b200moby_status b200moby_destroy(b200moby_handle h) {
  if (!h) return B200MOBY_OK;
  cudaSetDevice(h->device);
  for (cudaStream_t st : h->side) if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
  for (cudaEvent_t ev : h->side_done) if (ev) cudaEventDestroy(ev);
  if (h->fork) cudaEventDestroy(h->fork);
  if (h->hard_stream) { cudaStreamSynchronize(h->hard_stream); cudaStreamDestroy(h->hard_stream); }
  if (h->hard_done) cudaEventDestroy(h->hard_done);
  if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
  if (h->graph_stream) cudaStreamDestroy(h->graph_stream);
  for (auto& pe : h->kev_pending) { cudaEventDestroy(pe.second.first); cudaEventDestroy(pe.second.second); }
  for (auto& pe : h->kev_free) { cudaEventDestroy(pe.first); cudaEventDestroy(pe.second); }
  for (void* p : h->allocs) cudaFree(p);
  g_live_handles[h->device & 63]--;
  delete h;
  return B200MOBY_OK;
}

b200moby_status b200moby_set_state(b200moby_handle h, const double* q, const double* v) {
  if (!h || !q || !v) return b2m_fail(B200MOBY_ERR_INVALID, "null argument");
  B2M_CUDA(cudaSetDevice(h->device));
  B2M_CUDA(cudaMemcpy(h->P.q, q, sizeof(double) * h->nb * 7 * h->n_envs, cudaMemcpyHostToDevice));
  B2M_CUDA(cudaMemcpy(h->P.v, v, sizeof(double) * h->nb * 6 * h->n_envs, cudaMemcpyHostToDevice));
  normalize_quat_kernel<<<(h->nb * h->n_envs + 255) / 256, 256>>>(h->P.q, h->nb, h->n_envs);
  B2M_CUDA(cudaGetLastError());
  return B200MOBY_OK;
}
b200moby_status b200moby_get_state(b200moby_handle h, double* q, double* v) {
  if (!h) return b2m_fail(B200MOBY_ERR_INVALID, "null handle");
  B2M_CUDA(cudaSetDevice(h->device));
  if (q) B2M_CUDA(cudaMemcpy(q, h->P.q, sizeof(double) * h->nb * 7 * h->n_envs, cudaMemcpyDeviceToHost));
  if (v) B2M_CUDA(cudaMemcpy(v, h->P.v, sizeof(double) * h->nb * 6 * h->n_envs, cudaMemcpyDeviceToHost));
  return B200MOBY_OK;
}
b200moby_status b200moby_set_state_dev(b200moby_handle h, const double* q, const double* v, void* stream) {
  if (!h || !q || !v) return b2m_fail(B200MOBY_ERR_INVALID, "null argument");
  B2M_CUDA(cudaSetDevice(h->device));
  B2M_CUDA(cudaMemcpyAsync(h->P.q, q, sizeof(double) * h->nb * 7 * h->n_envs, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  B2M_CUDA(cudaMemcpyAsync(h->P.v, v, sizeof(double) * h->nb * 6 * h->n_envs, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  normalize_quat_kernel<<<(h->nb * h->n_envs + 255) / 256, 256, 0, (cudaStream_t)stream>>>(h->P.q, h->nb, h->n_envs);
  B2M_CUDA(cudaGetLastError());
  return B200MOBY_OK;
}
b200moby_status b200moby_get_state_dev(b200moby_handle h, double* q, double* v, void* stream) {
  if (!h) return b2m_fail(B200MOBY_ERR_INVALID, "null handle");
  B2M_CUDA(cudaSetDevice(h->device));
  if (q) B2M_CUDA(cudaMemcpyAsync(q, h->P.q, sizeof(double) * h->nb * 7 * h->n_envs, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (v) B2M_CUDA(cudaMemcpyAsync(v, h->P.v, sizeof(double) * h->nb * 6 * h->n_envs, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return B200MOBY_OK;
}

static b200moby_status rc_refresh(b200moby_handle h, cudaStream_t s) {
  void* a[] = {&h->P};
  B2M_CUDA(cudaSetDevice(h->device));
  B2M_CUDA(cudaLaunchKernel(b2m_k_rc_refresh(), dim3((h->n_envs + 127) / 128), dim3(128), a, 0, s));
  h->launches++;
  return B200MOBY_OK;
}
b200moby_status b200moby_set_joint_state(b200moby_handle h, const double* jq, const double* jqd) {
  if (!h || !jq || !jqd) return b2m_fail(B200MOBY_ERR_INVALID, "null argument");
  if (!h->rc_links) return b2m_fail(B200MOBY_ERR_INVALID, "the scene has no articulated body");
  B2M_CUDA(cudaSetDevice(h->device));
  B2M_CUDA(cudaMemcpy(h->P.jq, jq, sizeof(double) * h->rc_dof * h->n_envs, cudaMemcpyHostToDevice));
  B2M_CUDA(cudaMemcpy(h->P.jqd, jqd, sizeof(double) * h->rc_dof * h->n_envs, cudaMemcpyHostToDevice));
  return rc_refresh(h, 0);
}
b200moby_status b200moby_get_joint_state(b200moby_handle h, double* jq, double* jqd) {
  if (!h) return b2m_fail(B200MOBY_ERR_INVALID, "null handle");
  if (!h->rc_links) return b2m_fail(B200MOBY_ERR_INVALID, "the scene has no articulated body");
  B2M_CUDA(cudaSetDevice(h->device));
  if (jq) B2M_CUDA(cudaMemcpy(jq, h->P.jq, sizeof(double) * h->rc_dof * h->n_envs, cudaMemcpyDeviceToHost));
  if (jqd) B2M_CUDA(cudaMemcpy(jqd, h->P.jqd, sizeof(double) * h->rc_dof * h->n_envs, cudaMemcpyDeviceToHost));
  return B200MOBY_OK;
}
b200moby_status b200moby_set_joint_state_dev(b200moby_handle h, const double* jq, const double* jqd, void* stream) {
  if (!h || !jq || !jqd) return b2m_fail(B200MOBY_ERR_INVALID, "null argument");
  if (!h->rc_links) return b2m_fail(B200MOBY_ERR_INVALID, "the scene has no articulated body");
  B2M_CUDA(cudaSetDevice(h->device));
  B2M_CUDA(cudaMemcpyAsync(h->P.jq, jq, sizeof(double) * h->rc_dof * h->n_envs, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  B2M_CUDA(cudaMemcpyAsync(h->P.jqd, jqd, sizeof(double) * h->rc_dof * h->n_envs, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return rc_refresh(h, (cudaStream_t)stream);
}
b200moby_status b200moby_get_joint_state_dev(b200moby_handle h, double* jq, double* jqd, void* stream) {
  if (!h) return b2m_fail(B200MOBY_ERR_INVALID, "null handle");
  if (!h->rc_links) return b2m_fail(B200MOBY_ERR_INVALID, "the scene has no articulated body");
  B2M_CUDA(cudaSetDevice(h->device));
  if (jq) B2M_CUDA(cudaMemcpyAsync(jq, h->P.jq, sizeof(double) * h->rc_dof * h->n_envs, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (jqd) B2M_CUDA(cudaMemcpyAsync(jqd, h->P.jqd, sizeof(double) * h->rc_dof * h->n_envs, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return B200MOBY_OK;
}
b200moby_status b200moby_set_joint_forces(b200moby_handle h, const double* tau) {
  if (!h) return b2m_fail(B200MOBY_ERR_INVALID, "null handle");
  if (!h->rc_links) return b2m_fail(B200MOBY_ERR_INVALID, "the scene has no articulated body");
  B2M_CUDA(cudaSetDevice(h->device));
  if (tau) B2M_CUDA(cudaMemcpy(const_cast<double*>(h->P.jtau), tau, sizeof(double) * h->rc_dof * h->n_envs, cudaMemcpyHostToDevice));
  else B2M_CUDA(cudaMemset(const_cast<double*>(h->P.jtau), 0, sizeof(double) * h->rc_dof * h->n_envs));
  return B200MOBY_OK;
}
b200moby_status b200moby_rc_fwd_dyn_batched(b200moby_handle h, int algorithm, const double* jq, const double* jqd, const double* tau,
                                            double* qdd, void* stream) {
  if (!h || !jq || !jqd || !qdd) return b2m_fail(B200MOBY_ERR_INVALID, "null argument");
  if (!h->rc_links) return b2m_fail(B200MOBY_ERR_INVALID, "the scene has no articulated body");
  if (algorithm != B200MOBY_FDYN_FSAB && algorithm != B200MOBY_FDYN_CRB) return b2m_fail(B200MOBY_ERR_INVALID, "unknown forward-dynamics algorithm %d", algorithm);
  void* a[] = {&h->P, &algorithm, &jq, &jqd, &tau, &qdd};
  B2M_CUDA(cudaSetDevice(h->device));
  B2M_CUDA(cudaLaunchKernel(b2m_k_rc_fwd_dyn(), dim3((h->n_envs + 127) / 128), dim3(128), a, 0, (cudaStream_t)stream));
  h->launches++;
  return B200MOBY_OK;
}
b200moby_status b200moby_rc_inertia_batched(b200moby_handle h, const double* jq, double* H, void* stream) {
  if (!h || !jq || !H) return b2m_fail(B200MOBY_ERR_INVALID, "null argument");
  if (!h->rc_links) return b2m_fail(B200MOBY_ERR_INVALID, "the scene has no articulated body");
  void* a[] = {&h->P, &jq, &H};
  B2M_CUDA(cudaSetDevice(h->device));
  B2M_CUDA(cudaLaunchKernel(b2m_k_rc_inertia(), dim3((h->n_envs + 127) / 128), dim3(128), a, 0, (cudaStream_t)stream));
  h->launches++;
  return B200MOBY_OK;
}

b200moby_status b200moby_step(b200moby_handle h, double dt, int n_steps, void* stream) {
  if (!h || !(dt > 0.0) || n_steps < 0) return b2m_fail(B200MOBY_ERR_INVALID, "bad step arguments");
  if (n_steps == 0) return B200MOBY_OK;
  B2M_CUDA(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (h->fused) {   // comparison path: the whole mini-step loop of n_steps steps in one launch (one step per launch when stabilization is on)
    const int per = h->P.stab_max_iterations != 0 ? 1 : n_steps;
    for (int k = 0; k < n_steps; k += per) {
      int cnt = per;
      void* a[] = {&h->P, &dt, &cnt, &h->env_d};
      B2M_CUDA(cudaLaunchKernel(b2m_k_step_warp(), dim3(h->grid), dim3(32), a, h->shmem, s));
      h->launches++;
      b200moby_status st = launch_stabilize(h, s);
      if (st != B200MOBY_OK) return st;
    }
    return B200MOBY_OK;
  }
  if (h->graph_on && !h->ktiming) {
    if (!h->graph_exec || h->graph_dt != dt || h->graph_feed != launch_feeds(h) || memcmp(&h->graph_P, &h->P, sizeof(SimParams)) != 0) {
      if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }
      if (!h->graph_stream) B2M_CUDA(cudaStreamCreateWithFlags(&h->graph_stream, cudaStreamNonBlocking));
      const long long l0 = h->launches;
      cudaGraph_t graph = nullptr;
      B2M_CUDA(cudaStreamBeginCapture(h->graph_stream, cudaStreamCaptureModeRelaxed));
      const b200moby_status st = launch_step(h, dt, h->graph_stream);
      const cudaError_t ce = cudaStreamEndCapture(h->graph_stream, &graph);
      h->graph_launches = h->launches - l0; h->launches = l0;
      if (st != B200MOBY_OK) { if (graph) cudaGraphDestroy(graph); return st; }
      if (ce != cudaSuccess || !graph) { cudaGetLastError(); h->graph_on = false; }      // capture not possible here: plain launches from now on
      else {
        const cudaError_t ie = cudaGraphInstantiate(&h->graph_exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { cudaGetLastError(); h->graph_exec = nullptr; h->graph_on = false; }
        else { h->graph_P = h->P; h->graph_dt = dt; h->graph_feed = launch_feeds(h); h->graph_captures++; }
      }
    }
    if (h->graph_exec) {
      for (int k = 0; k < n_steps; k++) { B2M_CUDA(cudaGraphLaunch(h->graph_exec, s)); h->launches += h->graph_launches; }
      return B200MOBY_OK;
    }
  }
  for (int k = 0; k < n_steps; k++) {
    b200moby_status st = launch_step(h, dt, s);
    if (st != B200MOBY_OK) return st;
  }
  return B200MOBY_OK;
}

b200moby_status b200moby_set_pivot_budget(b200moby_handle h, int budget) {
  if (!h) return b2m_fail(B200MOBY_ERR_INVALID, "null handle");
  h->P.pivot_budget = budget;
  return B200MOBY_OK;
}

b200moby_status b200moby_get_counters(b200moby_handle h, b200moby_counters* out) {
  if (!h || !out) return b2m_fail(B200MOBY_ERR_INVALID, "null argument");
  unsigned long long c[CNT_COUNT];
  B2M_CUDA(cudaSetDevice(h->device));
  B2M_CUDA(cudaMemcpy(c, h->P.counters, sizeof(c), cudaMemcpyDeviceToHost));
  out->env_steps = c[CNT_ENV_STEPS]; out->mini_steps = c[CNT_MINI_STEPS]; out->lcp_solves = c[CNT_LCP_SOLVES];
  out->lcp_fast_calls = c[CNT_FAST_CALLS]; out->lemke_calls = c[CNT_LEMKE_CALLS]; out->pivots = c[CNT_PIVOTS];
  out->lcp_failures = c[CNT_LCP_FAIL] + c[CNT_OVERFLOW]; out->impact_tol_events = c[CNT_IMPACT_TOL]; out->contacts = c[CNT_CONTACTS];
  out->max_lcp_n = c[CNT_MAX_N]; out->pivot_flops = c[CNT_PIVOT_FLOPS]; out->assembly_flops = c[CNT_ASM_FLOPS]; out->ca_iterations = c[CNT_CA_ITERS];
  out->stab_iterations = c[CNT_STAB_ITERS]; out->stab_lcp_solves = c[CNT_STAB_SOLVES]; out->stab_line_search_failures = c[CNT_STAB_LSFAIL];
  return B200MOBY_OK;
}
b200moby_status b200moby_get_launch_count(b200moby_handle h, long long* out) {
  if (!h || !out) return b2m_fail(B200MOBY_ERR_INVALID, "null argument");
  *out = h->launches;
  return B200MOBY_OK;
}
b200moby_status b200moby_reset_counters(b200moby_handle h) {
  if (!h) return b2m_fail(B200MOBY_ERR_INVALID, "null handle");
  B2M_CUDA(cudaSetDevice(h->device));
  B2M_CUDA(cudaMemset(h->P.counters, 0, sizeof(unsigned long long) * CNT_COUNT));
  return B200MOBY_OK;
}
b200moby_status b200moby_get_time(b200moby_handle h, double* t) {
  if (!h || !t) return b2m_fail(B200MOBY_ERR_INVALID, "null argument");
  B2M_CUDA(cudaSetDevice(h->device));
  B2M_CUDA(cudaMemcpy(t, h->P.time, sizeof(double) * h->n_envs, cudaMemcpyDeviceToHost));
  return B200MOBY_OK;
}

// Debug tap: after this call every impact solve records its LCP; returns the last one per env.
// n: [env]; z: [env][zcap] (host).  First call only arms the tap (returns zeros).
b200moby_status b200moby_get_last_lcp(b200moby_handle h, int* n, double* z, int zcap) {
  if (!h) return b2m_fail(B200MOBY_ERR_INVALID, "null handle");
  B2M_CUDA(cudaSetDevice(h->device));
  if (!h->taps) {
    b200moby_status st;
    if ((st = dev_zero(h, (size_t)h->n_envs * h->nmax * h->nmax, &h->P.tap_MM)) != B200MOBY_OK) return st;
    if ((st = dev_zero(h, (size_t)h->n_envs * h->nmax, &h->P.tap_qq)) != B200MOBY_OK) return st;
    if ((st = dev_zero(h, (size_t)h->n_envs * h->nmax, &h->P.tap_z)) != B200MOBY_OK) return st;
    if ((st = dev_zero(h, (size_t)h->n_envs, &h->P.tap_n)) != B200MOBY_OK) return st;
    h->taps = true;
  }
  if (n) B2M_CUDA(cudaMemcpy(n, h->P.tap_n, sizeof(int) * h->n_envs, cudaMemcpyDeviceToHost));
  if (z) {
    std::vector<double> tmp((size_t)h->n_envs * h->nmax);
    B2M_CUDA(cudaMemcpy(tmp.data(), h->P.tap_z, sizeof(double) * tmp.size(), cudaMemcpyDeviceToHost));
    for (int e = 0; e < h->n_envs; e++) for (int i = 0; i < zcap; i++) z[(size_t)e * zcap + i] = (i < h->nmax) ? tmp[(size_t)e * h->nmax + i] : 0.0;
  }
  return B200MOBY_OK;
}

// Per-kernel profile of the stepped path since the last call with reset != 0: enabling it brackets every launch with
// events on the launch's own stream.  The call synchronises the device.
b200moby_status b200moby_get_kernel_profile(b200moby_handle h, int enable, int reset, b200moby_kernel_profile* out) {
  if (!h) return b2m_fail(B200MOBY_ERR_INVALID, "null handle");
  B2M_CUDA(cudaSetDevice(h->device));
  B2M_CUDA(cudaDeviceSynchronize());
  const int ncls = (int)h->classes.size(), nk = ncls + 5;
  h->kms.resize(nk, 0.0); h->klaunches.resize(nk, 0);
  for (auto& pe : h->kev_pending) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, pe.second.first, pe.second.second) == cudaSuccess) { h->kms[pe.first] += ms; h->klaunches[pe.first]++; }
    h->kev_free.push_back(pe.second);
  }
  h->kev_pending.clear();
  if (out) {
    memset(out, 0, sizeof(*out));
    unsigned long long ks[3 * (B2M_MAX_CLASSES + 6)];
    B2M_CUDA(cudaMemcpy(ks, h->P.kstat, sizeof(ks), cudaMemcpyDeviceToHost));
    out->n_kernels = nk;
    for (int k = 0; k < nk && k < B200MOBY_MAX_KERNELS; k++) {
      b200moby_kernel_stat& o = out->k[k];
      if (k == 0) snprintf(o.name, sizeof(o.name), "advance_kernel");
      else if (k <= ncls) { const ClassPlan& c = h->classes[k - 1]; if (c.threads == 1) snprintf(o.name, sizeof(o.name), "impact_thread_kernel[n<=%d]", c.nmax); else if (c.threads == 8) snprintf(o.name, sizeof(o.name), "impact_subwarp_kernel<8>[n<=%d]", c.nmax); else if (c.threads == 32) snprintf(o.name, sizeof(o.name), "impact_warp_kernel[n<=%d]", c.nmax); else snprintf(o.name, sizeof(o.name), "impact_block_kernel<%d>[n<=%d]", c.threads, c.nmax); o.lcp_nmax = c.nmax; o.threads_per_env = c.threads; }
      else if (k == ncls + 1 || k == ncls + 3) { if (h->straggler.threads == 32) snprintf(o.name, sizeof(o.name), "impact_warp_kernel[%s]", k == ncls + 1 ? "stragglers" : "hard queue"); else snprintf(o.name, sizeof(o.name), "impact_block_kernel<%d>[%s]", h->straggler.threads, k == ncls + 1 ? "stragglers" : "hard queue"); o.lcp_nmax = h->nmax; o.threads_per_env = h->straggler.threads; }
      else if (k == ncls + 4) { snprintf(o.name, sizeof(o.name), h->stab_variant >= 0 ? "stabilize_thread_kernel" : "stabilize_warp_kernel"); o.threads_per_env = h->stab_variant >= 0 ? 1 : 32; }
      else snprintf(o.name, sizeof(o.name), h->finblock.threads == 256 ? "finish_block_kernel<256>" : "finish_kernel");
      if (k == 0 || k == ncls + 2) o.threads_per_env = 32;
      o.ms = h->kms[k]; o.launches = h->klaunches[k];
      o.envs = (long long)ks[3 * k]; o.flops = (long long)ks[3 * k + 1]; o.lcp_solves = (long long)ks[3 * k + 2];
    }
  }
  if (reset) {
    std::fill(h->kms.begin(), h->kms.end(), 0.0); std::fill(h->klaunches.begin(), h->klaunches.end(), 0);
    B2M_CUDA(cudaMemset(h->P.kstat, 0, sizeof(unsigned long long) * 3 * (B2M_MAX_CLASSES + 6)));
  }
  h->ktiming = enable != 0;
  return B200MOBY_OK;
}

// Debug tap: per-env SM cycles, pivots, executed iterations and LCP dimension of the last impact phase; prof is a host
// buffer [13][env] (4 totals + 9 phases: load, contacts, islands, problem data, LCP build, lcp_fast, Lemke, apply, store).
// The first call arms the tap (and returns zeros).
b200moby_status b200moby_get_impact_profile(b200moby_handle h, long long* prof) {
  if (!h || !prof) return b2m_fail(B200MOBY_ERR_INVALID, "null argument");
  B2M_CUDA(cudaSetDevice(h->device));
  if (!h->P.tap_prof) { b200moby_status st; if ((st = dev_zero(h, (size_t)(4 + PH_COUNT) * h->n_envs, &h->P.tap_prof)) != B200MOBY_OK) return st; }
  B2M_CUDA(cudaMemcpy(prof, h->P.tap_prof, sizeof(long long) * (4 + PH_COUNT) * h->n_envs, cudaMemcpyDeviceToHost));
  B2M_CUDA(cudaMemset(h->P.tap_prof, 0, sizeof(long long) * (4 + PH_COUNT) * h->n_envs));
  return B200MOBY_OK;
}

// Debug tap: per-env solver statistics since the previous call; stat: host buffer [5][env] (LCP failures, lcp_lemke calls,
// lcp_fast calls, LCP solves, pivots as the reference counts them).  The first call arms the tap (and returns zeros); reading clears it.
b200moby_status b200moby_get_env_stats(b200moby_handle h, int* stat) {
  if (!h || !stat) return b2m_fail(B200MOBY_ERR_INVALID, "null argument");
  B2M_CUDA(cudaSetDevice(h->device));
  B2M_CUDA(cudaDeviceSynchronize());
  if (!h->P.env_stat) { b200moby_status st; if ((st = dev_zero(h, (size_t)5 * h->n_envs, &h->P.env_stat)) != B200MOBY_OK) return st; }
  B2M_CUDA(cudaMemcpy(stat, h->P.env_stat, sizeof(int) * 5 * h->n_envs, cudaMemcpyDeviceToHost));
  B2M_CUDA(cudaMemset(h->P.env_stat, 0, sizeof(int) * 5 * h->n_envs));
  return B200MOBY_OK;
}

static b200moby_status run_stage(b200moby_handle h, int stage, const double* q, const double* v, StageOut o, void* stream) {
  if (!h || !q || !v) return b2m_fail(B200MOBY_ERR_INVALID, "null argument");
  if (h->rc_links && stage == STAGE_DELASSUS) return b2m_fail(B200MOBY_ERR_UNSUPPORTED, "the assembly stage kernel handles free-body scenes only");
  B2M_CUDA(cudaSetDevice(h->device));
  if (!h->stage_attr_set) { B2M_CUDA(cudaFuncSetAttribute(stage_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B2M_SMEM_MAX)); h->stage_attr_set = true; }   // function attributes are per device: one flag per handle
  SimParams P = h->P;
  P.q = const_cast<double*>(q); P.v = const_cast<double*>(v);
  stage_warp_kernel<<<h->grid, h->wpb * 32, h->shmem, (cudaStream_t)stream>>>(P, stage, o, h->wpb, h->env_d, h->env_i);
  B2M_CUDA(cudaGetLastError());
  return B200MOBY_OK;
}

b200moby_status b200moby_fwd_dyn_batched(b200moby_handle h, const double* q, double* v, double dt, void* stream) {
  StageOut o; memset(&o, 0, sizeof(o)); o.dt = dt;
  return run_stage(h, STAGE_FWD_DYN, q, v, o, stream);
}
b200moby_status b200moby_find_contacts_batched(b200moby_handle h, const double* q, const double* v, int cap, int* count, double* point,
                                               double* normal, double* tan1, double* tan2, int* pair, double* dist, void* stream) {
  if (!count || !point || !normal || !tan1 || !tan2 || !pair || !dist || cap <= 0) return b2m_fail(B200MOBY_ERR_INVALID, "null output");
  StageOut o; memset(&o, 0, sizeof(o));
  o.cap = cap; o.count = count; o.point = point; o.normal = normal; o.tan1 = tan1; o.tan2 = tan2; o.pair = pair; o.dist = dist;
  return run_stage(h, STAGE_CONTACTS, q, v, o, stream);
}
// Host-buffer form for callers without device memory of their own (the C++ facade's get_rigid_constraints): the contacts of
// the simulator's CURRENT state.  Synchronous; temporary device buffers per call -- a documented slow path.
b200moby_status b200moby_find_contacts_host(b200moby_handle h, int cap, int* count, double* point, double* normal, double* tan1, double* tan2,
                                            int* pair, double* dist) {
  if (!h || !count || !point || !normal || !tan1 || !tan2 || !pair || !dist || cap <= 0) return b2m_fail(B200MOBY_ERR_INVALID, "null output");
  B2M_CUDA(cudaSetDevice(h->device));
  const size_t ne = (size_t)h->n_envs, nv = (size_t)cap * 3 * ne;
  int* d_i = nullptr; double* d_d = nullptr;
  B2M_CUDA(cudaMalloc((void**)&d_i, sizeof(int) * (ne + (size_t)cap * ne)));
  if (cudaMalloc((void**)&d_d, sizeof(double) * (4 * nv + (size_t)cap * ne)) != cudaSuccess) { cudaFree(d_i); return b2m_fail(B200MOBY_ERR_CUDA, "out of device memory"); }
  b200moby_status st = b200moby_find_contacts_batched(h, h->P.q, h->P.v, cap, d_i, d_d, d_d + nv, d_d + 2 * nv, d_d + 3 * nv, d_i + ne, d_d + 4 * nv, nullptr);
  cudaError_t ce = cudaDeviceSynchronize();
  if (st == B200MOBY_OK && ce == cudaSuccess) {
    cudaMemcpy(count, d_i, sizeof(int) * ne, cudaMemcpyDeviceToHost); cudaMemcpy(pair, d_i + ne, sizeof(int) * cap * ne, cudaMemcpyDeviceToHost);
    cudaMemcpy(point, d_d, sizeof(double) * nv, cudaMemcpyDeviceToHost); cudaMemcpy(normal, d_d + nv, sizeof(double) * nv, cudaMemcpyDeviceToHost);
    cudaMemcpy(tan1, d_d + 2 * nv, sizeof(double) * nv, cudaMemcpyDeviceToHost); cudaMemcpy(tan2, d_d + 3 * nv, sizeof(double) * nv, cudaMemcpyDeviceToHost);
    ce = cudaMemcpy(dist, d_d + 4 * nv, sizeof(double) * cap * ne, cudaMemcpyDeviceToHost);
  }
  cudaFree(d_i); cudaFree(d_d);
  if (st != B200MOBY_OK) return st;
  if (ce != cudaSuccess) return b2m_fail(B200MOBY_ERR_CUDA, "%s", cudaGetErrorString(ce));
  return B200MOBY_OK;
}
b200moby_status b200moby_delassus_batched(b200moby_handle h, const double* q, const double* v, int nmax, double* MM, double* qq,
                                          int* n, void* stream) {
  if (!MM || !qq || !n || nmax <= 0) return b2m_fail(B200MOBY_ERR_INVALID, "null output");
  StageOut o; memset(&o, 0, sizeof(o));
  o.nmax_out = nmax; o.MM = MM; o.qq = qq; o.n = n;
  return run_stage(h, STAGE_DELASSUS, q, v, o, stream);
}

}  // extern "C"
