// Impact phase, one THREAD per env.
//
// The impact path of an env (contacts again, islands, problem data, LCP assembly, principal pivoting, impulses) is tens of
// thousands of mostly scalar, branchy instructions with little lane parallelism at these sizes: with a warp per env the
// ncu captures under profiles/ show 7-15 active lanes per instruction, an instruction-cache hit rate of 56-85 % and
// no_instruction / fixed-latency waits as the top stalls -- every env streams the whole program through the SM on its
// own.  Here a warp runs 32 envs of one LCP class in lock step: the same device functions instantiated for the
// one-thread group, the class's working set in the thread's local memory (interleaved by the hardware, so equal indices
// of neighbouring envs coalesce).  Divergence is bounded by a small per-env budget of solver iterations: an env that
// needs more is abandoned untouched and re-run by the straggler kernel (many threads per env, shortest latency per
// pivot), and from then on its recorded cost sends it to the hard queue directly (SimParams::cost).  An env whose first
// lcp_fast rung does not verify is handed on the same way (EnvCtx::first_rung), without that cost.
// Same arithmetic per env as the warp and block kernels: results are bit-identical.
#include "sim_kernel_util.cuh"
using namespace b2m;

template <int ND, int NI>
__global__ void __launch_bounds__(128) impact_thread_kernel(SimParams P, double dt, int round, int slot) {
  double wd[ND];
  int wi[NI];
  EnvMem m;
  env_carve(m, wd, wi, env_dims(P));
  SerialGroup g(nullptr);
  // counters of ONE env at a time: an env that runs over its budget is abandoned untouched and re-run (and counted) by the
  // straggler kernel, so what it counted here is dropped -- as in k_impact_warp.cu and tests/hostsim
  unsigned long long lc[CNT_COUNT], tot[CNT_COUNT];
  for (int k = 0; k < CNT_COUNT; k++) { lc[k] = 0; tot[k] = 0; }
  const int count = q_size(P, round, slot);
  unsigned long long envs = 0;
  // P.thread_lanes (<= 32) envs per warp: fewer lanes in lock step trade lane utilisation for more warps in flight (this
  // kernel is bound by the latency of its dependent chains through local memory, not by issue slots) and for less
  // divergence (a warp lasts as long as its slowest env)
  const int lanes = P.thread_lanes > 0 && P.thread_lanes < 32 ? P.thread_lanes : 32;
  const int lane = threadIdx.x & 31, warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int i = warp * lanes + lane; lane < lanes && i < count; i += nwarps * lanes) {
    for (int k = 0; k < CNT_COUNT; k++) lc[k] = 0;
    EnvCtx cx; cx.limit = P.pivot_budget > 0; cx.budget = P.pivot_budget; cx.first_rung = P.first_rung_handoff != 0;
    if (env_impact(g, P, q_at(P, round, slot, i), m, dt, round, lc, cx)) add_counters(tot, lc);
    envs++;                                            // envs handed to this launch (deferred ones included), like the warp kernel
  }
  for (int k = 0; k < CNT_COUNT; k++) lc[k] = tot[k];
  for (int k = 0; k < CNT_COUNT; k++) {
    unsigned long long v = lc[k];
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long u = __shfl_xor_sync(0xffffffffu, v, o); v = (k == CNT_MAX_N) ? (u > v ? u : v) : v + u; }
    lc[k] = v;
  }
  for (int o = 16; o > 0; o >>= 1) envs += __shfl_xor_sync(0xffffffffu, envs, o);
  if ((threadIdx.x & 31) == 0) commit_counters(P, lc, envs);
}

const void* b2m_k_impact_thread(int variant) {
  return variant == 0 ? (const void*)impact_thread_kernel<B2M_THREAD_ND0, B2M_THREAD_NI0> : (const void*)impact_thread_kernel<B2M_THREAD_ND1, B2M_THREAD_NI1>;
}
