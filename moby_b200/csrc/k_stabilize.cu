// Constraint stabilization phase (stab_device.cuh): runs once per TimeSteppingSimulator::step for every env, after the
// step's last kernel.  Most envs leave after one pass over their pairwise distances (nothing closer than sqrt(eps));
// a resting body needs one frictionless nc x nc LCP and a short line search.  Thread per env while the working set
// (the env's with nmax = cmax, plus the stabilization extras) fits a compiled local-memory size -- the same reasoning as
// k_advance.cu / k_impact_thread.cu: short, branchy, scalar work, SoA state unit-stride across the warp -- otherwise
// warp per env with the working set in an L2-resident global slice.
#include "sim_kernel_util.cuh"
using namespace b2m;

template <class G>
__device__ __forceinline__ void stabilize_env(const G& g, const SimParams& P, int e, EnvMem& m, const StabMem& s, unsigned long long* lc) {
  env_load(g, P, e, m);
  const unsigned long long it0 = lc[CNT_STAB_SOLVES];
  const EnvStatBase sb = env_stat_base(lc);
  env_stabilize(g, P, e, m, s, lc);
  g.sync();
  if (lc[CNT_STAB_SOLVES] != it0 || G::size > 1) {        // positions moved (a group does not share lc: always store)
    env_stat_commit(g, P, e, lc, sb);
    env_store(g, P, e, m, ST_POS);
  }
  g.sync();
}

// P.nmax == P.cmax here (the host passes the stabilization view of the parameters).
// Two launches per step.  mode 0 (select): every env evaluates its pairwise distances once and, if some pair is closer than
// eps, puts itself on `queue`.  mode 1 (process): the queued envs are stabilized, 32 per warp.  With one launch over all
// envs a warp of 32 consecutive envs holds on average five that need the LCP and the line search (17 % of configs[1]) and
// runs as long as the slowest of them: compaction cuts the warps that walk the expensive path sixfold.
// The queue's length is known on the device only (the step is one captured graph), so the process launch is a full
// resident grid (sim_kernels.cu) and deals warp ranks round the blocks first: a short queue (4,400 of 65,536 envs on
// configs[1]) still reaches every SM, about one warp each.  Packed block by block it filled 38 blocks on 38 of 148 SMs
// (1.94 ms per step on a B200).  Measured with that layout and fewer envs per warp: 32 / 16 / 8 / 4 lanes -> 1.46 / 1.51 /
// 1.58 / 1.85 ms.  The pass is bound by the latency of its dependent local-memory chains, and local memory is interleaved
// across a warp's lanes: a partly filled warp moves the same sectors for fewer envs, and more warps per SM share the L1.
template <int ND, int NI>
__global__ void __launch_bounds__(128) stabilize_thread_kernel(SimParams P, int mode, int* queue, int* count) {
  double wd[ND];
  int wi[NI];
  const EnvDims D = env_dims(P);
  EnvMem m; StabMem s;
  env_carve(m, wd, wi, D);
  stab_carve(s, wd + env_doubles(D), wi + env_ints(D), D);
  SerialGroup g(nullptr);
  unsigned long long lc[CNT_COUNT];
  for (int k = 0; k < CNT_COUNT; k++) lc[k] = 0;
  unsigned long long envs = 0;
  if (mode == 0) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < P.n_envs; e += gridDim.x * blockDim.x) {
      env_load(g, P, e, m);
      if (stab_eval(g, m, s.uC) < P.stab_eps) queue[atomicAdd(count, 1)] = e;          // the test env_stabilize starts with (:187-197)
    }
    return;
  }
  const int n = queue ? *count : P.n_envs;
  const int first = (((threadIdx.x >> 5) * gridDim.x + blockIdx.x) << 5) + (threadIdx.x & 31);
  for (int i = first; i < n; i += gridDim.x * blockDim.x) { stabilize_env(g, P, queue ? queue[i] : i, m, s, lc); envs++; }
  for (int k = 0; k < CNT_COUNT; k++) {
    unsigned long long v = lc[k];
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long u = __shfl_xor_sync(0xffffffffu, v, o); v = (k == CNT_MAX_N) ? (u > v ? u : v) : v + u; }
    lc[k] = v;
  }
  for (int o = 16; o > 0; o >>= 1) envs += __shfl_xor_sync(0xffffffffu, envs, o);
  if ((threadIdx.x & 31) == 0) commit_counters(P, lc, envs);
}

// warp per env, working set in the warp's slice of P.gscratch (gstride doubles per warp; ints follow the doubles)
__global__ void __launch_bounds__(128) stabilize_warp_kernel(SimParams P, size_t nd_env, size_t nd_all, int* queue, int* count) {
  const EnvDims D = env_dims(P);
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
  double* base = P.gscratch + (size_t)w * P.gstride;
  int* ibase = (int*)(base + nd_all);
  EnvMem m; StabMem s;
  env_carve(m, base, ibase, D);
  stab_carve(s, base + nd_env, ibase + env_ints(D), D);
  WarpGroup g(nullptr);
  unsigned long long lc[CNT_COUNT];
  for (int k = 0; k < CNT_COUNT; k++) lc[k] = 0;
  unsigned long long envs = 0;
  const int n = queue ? *count : P.n_envs;                       // queue: the envs the select launch found (thread-per-env select, warp-per-env work)
  for (int i = w; i < n; i += nw) { stabilize_env(g, P, queue ? queue[i] : i, m, s, lc); envs++; }
  if (g.tid == 0) commit_counters(P, lc, envs);
}

const void* b2m_k_stabilize_thread(int variant) {
  return variant == 0 ? (const void*)stabilize_thread_kernel<B2M_STAB_ND0, B2M_STAB_NI0> : (const void*)stabilize_thread_kernel<B2M_STAB_ND1, B2M_STAB_NI1>;
}
const void* b2m_k_stabilize_warp() { return (const void*)stabilize_warp_kernel; }
