// Group-cooperative LCP solvers: Lemke complementary pivoting on an on-chip tableau and the
// principal-pivoting `lcp_fast`, each with the reference's regularised wrapper.
//
// Behavioural contract = Moby src/LCP.cpp (lcp_fast :41-196, rand_min :199-209 with the documented
// lowest-index tie rule, wrappers :212-487, lcp_lemke :545-1003): same tolerances, same entering /
// leaving rules, same iteration caps, same failure cascade.  What is different is how the numbers are
// produced: the reference re-factorises the n x n basis with LU for every Lemke pivot (O(n^3) per
// pivot); here the tableau B^-1 [N | q] lives in shared memory and a pivot is one rank-one update
// (2 n (n+2) flops) done by all threads of the group.
#pragma once
#include "common.cuh"

namespace b2m {

enum {
  LCP_OK = 0, LCP_TRIVIAL = 1, LCP_RAY = 2, LCP_MAXITER = 3, LCP_SINGULAR = 4, LCP_EMPTY_RATIO = 5,
  LCP_UNVERIFIED = 6, LCP_DEFER = 7, LCP_REGULARIZED = 16
};

// element (r,c) of M + lambda I
B2M_DEV B2M_INL double m_at(const double* M, int ldm, int r, int c, double lambda) {
  double v = M[(size_t)c * ldm + r];
  return (r == c) ? v + lambda : v;
}

// MatrixNd::norm_inf() of M + lambda I: largest |entry|
template <class G>
B2M_DEV B2M_NOINL double norm_inf(const G& g, int n, const double* M, int ldm, double lambda) {
  double m = 0.0;
  if constexpr (G::size == 1) {                                  // one thread: eight loads in flight (max is exact: any order gives the same value)
    double m1 = 0.0, m2 = 0.0, m3 = 0.0;
    for (int c = 0; c < n; c++) {
      const double* Mc = M + (size_t)c * ldm;
      int r = 0;
      for (; r + 8 <= n; r += 8) {
        double v0 = Mc[r], v1 = Mc[r + 1], v2 = Mc[r + 2], v3 = Mc[r + 3], v4 = Mc[r + 4], v5 = Mc[r + 5], v6 = Mc[r + 6], v7 = Mc[r + 7];
        if ((unsigned)(c - r) < 8u) { const int d = c - r; if (d == 0) v0 += lambda; else if (d == 1) v1 += lambda; else if (d == 2) v2 += lambda; else if (d == 3) v3 += lambda; else if (d == 4) v4 += lambda; else if (d == 5) v5 += lambda; else if (d == 6) v6 += lambda; else v7 += lambda; }
        m = fmax(m, fmax(fabs(v0), fabs(v4))); m1 = fmax(m1, fmax(fabs(v1), fabs(v5))); m2 = fmax(m2, fmax(fabs(v2), fabs(v6))); m3 = fmax(m3, fmax(fabs(v3), fabs(v7)));
      }
      for (; r < n; r++) m = fmax(m, fabs(m_at(M, ldm, r, c, lambda)));
    }
    return fmax(fmax(m, m1), fmax(m2, m3));
  }
  for (int e = g.tid; e < n * n; e += G::size) {
    const int c = e / n, r = e - c * n;
    m = fmax(m, fabs(m_at(M, ldm, r, c, lambda)));
  }
  return g.max(m);
}
// The same value in two parts, so that the regularised wrappers scan the n^2 entries once instead of once per attempt:
// the largest off-diagonal |entry| does not depend on lambda; the diagonal's does (n entries).  max is exact, so
// fmax(off, diag(lambda)) == norm_inf(lambda) bit for bit.
template <class G>
B2M_DEV B2M_NOINL double norm_inf_offdiag(const G& g, int n, const double* M, int ldm) {
  double m = 0.0;
  if constexpr (G::size == 1) {                                  // one thread: eight loads in flight (ncu: this scan, one dependent L2-latency load per entry, was 31 % of the thread-per-env impact kernel)
    double m1 = 0.0, m2 = 0.0, m3 = 0.0;
    for (int c = 0; c < n; c++) {
      const double* Mc = M + (size_t)c * ldm;
      int r = 0;
      for (; r + 8 <= n; r += 8) {
        double v0 = Mc[r], v1 = Mc[r + 1], v2 = Mc[r + 2], v3 = Mc[r + 3], v4 = Mc[r + 4], v5 = Mc[r + 5], v6 = Mc[r + 6], v7 = Mc[r + 7];
        if ((unsigned)(c - r) < 8u) { const int d = c - r; if (d == 0) v0 = 0.0; else if (d == 1) v1 = 0.0; else if (d == 2) v2 = 0.0; else if (d == 3) v3 = 0.0; else if (d == 4) v4 = 0.0; else if (d == 5) v5 = 0.0; else if (d == 6) v6 = 0.0; else v7 = 0.0; }
        m = fmax(m, fmax(fabs(v0), fabs(v4))); m1 = fmax(m1, fmax(fabs(v1), fabs(v5))); m2 = fmax(m2, fmax(fabs(v2), fabs(v6))); m3 = fmax(m3, fmax(fabs(v3), fabs(v7)));
      }
      for (; r < n; r++) if (r != c) m = fmax(m, fabs(Mc[r]));
    }
    return fmax(fmax(m, m1), fmax(m2, m3));
  }
  for (int c = 0; c < n; c++)
    for (int r = g.tid; r < n; r += G::size) if (r != c) m = fmax(m, fabs(M[(size_t)c * ldm + r]));
  return g.max(m);
}
template <class G>
B2M_DEV double norm_inf_with(const G& g, int n, const double* M, int ldm, double lambda, double offdiag) {
  if (offdiag < 0.0) return norm_inf(g, n, M, ldm, lambda);
  double m = offdiag;
  for (int i = g.tid; i < n; i += G::size) m = fmax(m, fabs(m_at(M, ldm, i, i, lambda)));
  return g.max(m);
}

// LCP::rand_min with the lowest-index tie rule: first minimum, then the lowest index i with v[i] < v[min] + tol.
template <class G>
B2M_DEV int rand_min(const G& g, const double* v, int m, double tol) {
  double key = B2M_INF; int idx = 0x7fffffff;
  for (int i = g.tid; i < m; i += G::size) { const double x = v[i]; if (x < key) { key = x; idx = i; } }
  g.min_key_idx(key, idx);
  const double thr = key + tol;
  int cand = 0x7fffffff;
  for (int i = g.tid; i < idx; i += G::size) if (v[i] < thr) { cand = i; break; }
  cand = g.min(cand);
  return cand < idx ? cand : idx;
}

// ------------------------------------------------------------------------------------------------
// Lemke.  Work memory: T  n*(n+2) doubles (column-major, ld n: slots 0..n nonbasic columns, column n+1 = x),
//                      dvec n, rvec n+2 doubles; where 2n+1, bas n ints.
// ------------------------------------------------------------------------------------------------
B2M_HD inline size_t lemke_work_doubles(int n) { return (size_t)n * (n + 2) + n + (n + 2); }
B2M_HD inline size_t lemke_work_ints(int n) { return (size_t)3 * n + 1; }

#ifdef __CUDACC__
// ---- warp-owned pivot loop (n <= 64) ------------------------------------------------------------------------------
// The generic loop below spreads every tableau pass over the group with a flat index: for one warp that is 50+ dependent
// load / fma / store rounds per pivot with index arithmetic in between (ncu, round 1: ~3,000 cycles per pivot at n = 40,
// issue slots 14 % busy).  Here lane l OWNS tableau rows l and l + 32: the entering column and x stay in its registers
// for the ratio test, both quotients of the ratio test are formed at once, the pivot element travels by shuffle, and the
// rank-one update walks the columns in batches of eight as ONE straight-line block -- all 24 loads of a batch first, no
// guard inside (a lone warp issues in order: ncu showed 21 cycles per instruction when every element sat behind its own
// branch), row indices clamped instead of predicated, LDS / STS instead of generic accesses when the working set is in
// shared memory.  No barrier other than __syncwarp, no integer division.  Every tableau entry goes through the same
// operations in the same order as in the generic loop (x / p, fma(-d_i, r_c, t)), so results are bit-identical whichever
// kernel runs an env.
// B columns of the rank-one update for the two rows a lane owns: all loads, then the fmas, then the stores.  The pivot
// row is not stored here (s0 / s1 exclude it): the lanes that formed r_c wrote it already.
template <int B>
static __device__ __forceinline__ void lemke_update_batch(double* q0, double* q1, const double* rvec, int c, int n, double nd0, double nd1, bool s0, bool s1, bool h1) {
  double rv[B], t0[B], t1[B];
  const int cn = c * n;
  // h1: the lane has a second row (n > 32: lanes 0 .. n-33).  The others used to re-read their first row through the clamped
  // index, a second 256-byte wavefront pair per column for nothing: predicated off, the second-row load is one 64-byte
  // wavefront at n = 40 (the shared-memory pipe is what the pivot loop contends for, DESIGN.md 4.3)
#pragma unroll
  for (int k = 0; k < B; k++) { rv[k] = rvec[c + k]; t0[k] = q0[cn + k * n]; t1[k] = h1 ? q1[cn + k * n] : 0.0; }
#pragma unroll
  for (int k = 0; k < B; k++) { t0[k] = fma(nd0, rv[k], t0[k]); t1[k] = fma(nd1, rv[k], t1[k]); }
#pragma unroll
  for (int k = 0; k < B; k++) { if (s0) q0[cn + k * n] = t0[k]; if (s1) q1[cn + k * n] = t1[k]; }
}

// N > 0: the LCP dimension is a compile-time constant (the sizes contact sets give: 8 or 10 rows per contact), so every
// tableau address of the update is base + immediate and the column walk is fully unrolled; N == 0: any n <= 64.
template <bool SH, int N>
static __device__ __noinline__ int lemke_loop_warp(int n_rt, double* T, double* rvec, int* where, int* bas, double PIV_TOL, double zero_tol, int r,
                                                   int* log, int log_cap, int& nlog_io, int& piv_io, int& executed_io, int* budget, const volatile int* cancel) {
  if (SH) { __builtin_assume(__isShared(T)); __builtin_assume(__isShared(rvec)); __builtin_assume(__isShared(where)); __builtin_assume(__isShared(bas)); }
  else { __builtin_assume(__isGlobal(T)); __builtin_assume(__isGlobal(rvec)); }     // global scratch: LDG / STG, scheduled for L2 latency (generic loads are scheduled as if shared)
  const int n = N ? N : n_rt;
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int t = 2 * n, MAXITER = min(1000, 50 * n), NC = n + 2;
  const int i0 = lane, i1 = lane + 32;
  const bool h0 = i0 < n, h1 = i1 < n;
  const int j0 = h0 ? i0 : 0, j1 = h1 ? i1 : j0;      // always-valid row indices: a lane without a row recomputes a valid element and does not store it
  double* const xcol = T + n * (n + 1);
  double* const q0 = T + j0;
  double* const q1 = T + j1;
  int s = n, entering = t, status = LCP_OK;
  int nlog = nlog_io, piv = piv_io, executed = executed_io, bud = budget ? *budget : 0;   // in registers for the loop (the references live on the stack)
  bool first = true;
  for (;;) {
    const double d0 = q0[s * n], d1 = q1[s * n];      // entering column, my rows
    if (!first) {
      executed++;
      const double x0 = xcol[j0], x1 = xcol[j1];
      const bool c0 = h0 && d0 > PIV_TOL, c1 = h1 && d1 > PIV_TOL;
      // the four quotients of the ratio test in lock step (b2m_divn: bit-identical to `/`); rows that are no candidates divide by 1
      const double num[4] = {x0 + zero_tol, x1 + zero_tol, x0, x1}, den[4] = {c0 ? d0 : 1.0, c1 ? d1 : 1.0, c0 ? d0 : 1.0, c1 ? d1 : 1.0};
      double quo[4];
      b2m_divn<4>(num, den, quo);
      const double a0 = c0 ? quo[0] : B2M_INF, a1 = c1 ? quo[1] : B2M_INF;
      const double b0 = c0 ? quo[2] : B2M_INF, b1 = c1 ? quo[3] : B2M_INF;
      const double theta = b2m_warp_min(fmin(a0, a1));
      if (theta == B2M_INF) { status = LCP_RAY; break; }
      const int trow = -(where[t] + 1);
      int lo = 0x7fffffff;
      if (c0 && b0 <= theta) lo = (i0 == trow) ? -1 : i0;
      if (c1 && b1 <= theta) { const int key = (i1 == trow) ? -1 : i1; if (key < lo) lo = key; }
      lo = __reduce_min_sync(FULL, lo);
      if (lo == 0x7fffffff) { status = LCP_EMPTY_RATIO; break; }
      r = (lo < 0) ? trow : lo;
    }
    const int leaving = bas[r];
    const double p = __shfl_sync(FULL, (r < 32) ? d0 : d1, r & 31);
    const bool s0 = h0 && i0 != r, s1 = h1 && i1 != r;      // rows this lane stores in the update: its own, except the pivot row
    __syncwarp();                               // everyone has read bas / where / column s before they change
    // pivot row, scaled: lane c forms r_c and writes it both to rvec and into row r of the tableau (its final value)
    {
      const int ca = lane, cb = lane + 32;                 // NC <= 66: two columns per lane, a third one only for lanes 0 and 1 at n = 63, 64
      const bool ha = ca < NC, hb = cb < NC;
      double* const pa = T + (ha ? ca : 0) * n + r;
      double* const pb = T + (hb ? cb : 0) * n + r;
      const double num[2] = {(ca == s) ? 1.0 : *pa, (cb == s) ? 1.0 : *pb}, den[2] = {p, p};
      double rv[2];
      b2m_divn<2>(num, den, rv);
      if (ha) { rvec[ca] = rv[0]; *pa = rv[0]; }
      if (hb) { rvec[cb] = rv[1]; *pb = rv[1]; }
      for (int c = lane + 64; c < NC; c += 32) { const double v = (c == s) ? 1.0 / p : T[c * n + r] / p; rvec[c] = v; T[c * n + r] = v; }
    }
    if (s0) q0[s * n] = 0.0;                    // the leaving variable's column (a unit vector while basic) replaces slot s: starts from zero
    if (s1) q1[s * n] = 0.0;
    if (lane == 0) {
      if (log && nlog < log_cap) log[nlog] = leaving;
      where[entering] = -(r + 1); where[leaving] = s; bas[r] = entering;
    }
    nlog++;
    __syncwarp();
    const double nd0 = -d0, nd1 = -d1;
    if (N) {
#pragma unroll
      for (int c = 0; c + 8 <= N + 2; c += 8) lemke_update_batch<8>(q0, q1, rvec, c, N, nd0, nd1, s0, s1, h1);
      if ((N + 2) & 4) lemke_update_batch<4>(q0, q1, rvec, (N + 2) & ~7, N, nd0, nd1, s0, s1, h1);
      if ((N + 2) & 2) lemke_update_batch<2>(q0, q1, rvec, (N + 2) & ~3, N, nd0, nd1, s0, s1, h1);
      if ((N + 2) & 1) lemke_update_batch<1>(q0, q1, rvec, (N + 2) & ~1, N, nd0, nd1, s0, s1, h1);
    } else {
      int c = 0;
      for (; c + 8 <= NC; c += 8) lemke_update_batch<8>(q0, q1, rvec, c, n, nd0, nd1, s0, s1, h1);   // straight-line batches
      if (NC & 4) { lemke_update_batch<4>(q0, q1, rvec, c, n, nd0, nd1, s0, s1, h1); c += 4; }
      if (NC & 2) { lemke_update_batch<2>(q0, q1, rvec, c, n, nd0, nd1, s0, s1, h1); c += 2; }
      if (NC & 1) lemke_update_batch<1>(q0, q1, rvec, c, n, nd0, nd1, s0, s1, h1);
    }
    __syncwarp();
    if (!first) piv++;
    if (budget && --bud < 0) { status = LCP_DEFER; break; }
    if (cancel && (piv & 63) == 63 && *cancel) { status = LCP_DEFER; break; }     // a speculative rung nobody needs any more (ladder task pool)
    first = false;
    if (leaving == t) break;
    if (piv >= MAXITER) { status = LCP_MAXITER; break; }
    entering = (leaving < n) ? n + leaving : leaving - n;
    s = where[entering];
  }
  nlog_io = nlog; piv_io = piv; executed_io = executed; if (budget) *budget = bud;
  return status;
}

// ---- register-resident tableau (compile-time n, working set in shared memory) ---------------------------------------
// Measured on the hard queue of configs[1] (profiles/r02_hard_queue_timeline.json): a 1,000-pivot rung takes 1.3 ms on an
// idle SM and 4-5 ms while four other warps of the launch pivot next to it -- the shared-memory pipe, not latency, sets
// the pace once several warps walk their tableaus through LDS / STS (about 400 wavefronts per pivot at n = 40).  Here
// lane l keeps its rows l and l + 32 in REGISTERS for the whole solve (2 x (n + 2) doubles, every index a compile-time
// constant in the unrolled loops); per pivot the shared-memory traffic is the pivot row (written once by the lane that
// owns it, scaled by the lanes in parallel, read back as broadcasts) plus bas / where -- about 90 wavefronts -- and the
// rank-one update is a straight run of register fmas.  The entering column of the NEXT pivot is picked up during the
// update (its slot is known as soon as the leaving variable is), so no dynamic register indexing is ever needed.
// Same operations per entry in the same order as lemke_loop_warp and the generic loop: bit-identical results.
// f(integral_constant<int, c>) for the c in [0, NC) that equals s.  s is warp-uniform, so this is one jump for the whole
// warp: the way to reach "register number s" without a per-element select (an FSEL pair per entry made the first version
// of the loop below three times longer than the shared-memory one).
template <int C> struct b2m_ic { static constexpr int value = C; };
#define B2M_SW_CASE(c) case c: if constexpr (c < NC) { asm volatile(""); f(b2m_ic<c>{}); } break;   /* the empty asm keeps the compiler from turning the jump into NC select pairs */
template <int NC, class F>
static __device__ __forceinline__ void b2m_static_switch(int s, F&& f) {
  static_assert(NC <= 44, "extend the case list");
  switch (s) {
    B2M_SW_CASE(0) B2M_SW_CASE(1) B2M_SW_CASE(2) B2M_SW_CASE(3) B2M_SW_CASE(4) B2M_SW_CASE(5) B2M_SW_CASE(6) B2M_SW_CASE(7) B2M_SW_CASE(8) B2M_SW_CASE(9) B2M_SW_CASE(10)
    B2M_SW_CASE(11) B2M_SW_CASE(12) B2M_SW_CASE(13) B2M_SW_CASE(14) B2M_SW_CASE(15) B2M_SW_CASE(16) B2M_SW_CASE(17) B2M_SW_CASE(18) B2M_SW_CASE(19) B2M_SW_CASE(20) B2M_SW_CASE(21)
    B2M_SW_CASE(22) B2M_SW_CASE(23) B2M_SW_CASE(24) B2M_SW_CASE(25) B2M_SW_CASE(26) B2M_SW_CASE(27) B2M_SW_CASE(28) B2M_SW_CASE(29) B2M_SW_CASE(30) B2M_SW_CASE(31) B2M_SW_CASE(32)
    B2M_SW_CASE(33) B2M_SW_CASE(34) B2M_SW_CASE(35) B2M_SW_CASE(36) B2M_SW_CASE(37) B2M_SW_CASE(38) B2M_SW_CASE(39) B2M_SW_CASE(40) B2M_SW_CASE(41) B2M_SW_CASE(42) B2M_SW_CASE(43)
    default: break;
  }
}
#undef B2M_SW_CASE

template <int N>
static __device__ __noinline__ int lemke_loop_warp_reg(double* T, double* rvec, int* where, int* bas, double PIV_TOL, double zero_tol, int r,
                                                       int* log, int log_cap, int& nlog_io, int& piv_io, int& executed_io, int* budget, const volatile int* cancel) {
  __builtin_assume(__isShared(T)); __builtin_assume(__isShared(rvec)); __builtin_assume(__isShared(where)); __builtin_assume(__isShared(bas));
  constexpr int n = N, NC = N + 2, t = 2 * N;
  constexpr bool TWO = N > 32;
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int MAXITER = min(1000, 50 * n);
  const int i0 = lane, i1 = lane + 32;
  const bool h0 = i0 < n, h1 = TWO && i1 < n;
  const int j0 = h0 ? i0 : 0, j1 = h1 ? i1 : j0;
  double R0[NC], R1[TWO ? NC : 1];
#pragma unroll
  for (int c = 0; c < NC; c++) { R0[c] = T[c * n + j0]; if (TWO) R1[c] = T[c * n + j1]; }
  int s = n, entering = t, status = LCP_OK;
  int nlog = nlog_io, piv = piv_io, executed = executed_io, bud = budget ? *budget : 0;
  bool first = true;
  for (;;) {
    double d0 = 0.0, d1 = 0.0;                                   // entering column, my rows: "register s", reached by one warp-uniform jump
    b2m_static_switch<NC>(s, [&](auto ic) { constexpr int c = decltype(ic)::value; d0 = R0[c]; if (TWO) d1 = R1[c]; });
    if (!first) {
      executed++;
      const double x0 = R0[N + 1], x1 = TWO ? R1[N + 1] : 0.0;
      const bool c0 = h0 && d0 > PIV_TOL, c1 = h1 && d1 > PIV_TOL;
      double a0, a1, b0, b1;
      if (TWO) {
        const double num[4] = {x0 + zero_tol, x1 + zero_tol, x0, x1}, den[4] = {c0 ? d0 : 1.0, c1 ? d1 : 1.0, c0 ? d0 : 1.0, c1 ? d1 : 1.0};
        double quo[4];
        b2m_divn<4>(num, den, quo);
        a0 = c0 ? quo[0] : B2M_INF; a1 = c1 ? quo[1] : B2M_INF; b0 = c0 ? quo[2] : B2M_INF; b1 = c1 ? quo[3] : B2M_INF;
      } else {
        const double num[2] = {x0 + zero_tol, x0}, den[2] = {c0 ? d0 : 1.0, c0 ? d0 : 1.0};
        double quo[2];
        b2m_divn<2>(num, den, quo);
        a0 = c0 ? quo[0] : B2M_INF; b0 = c0 ? quo[1] : B2M_INF; a1 = B2M_INF; b1 = B2M_INF;
      }
      const double theta = b2m_warp_min(fmin(a0, a1));
      if (theta == B2M_INF) { status = LCP_RAY; break; }
      const int trow = -(where[t] + 1);
      int lo = 0x7fffffff;
      if (c0 && b0 <= theta) lo = (i0 == trow) ? -1 : i0;
      if (c1 && b1 <= theta) { const int key = (i1 == trow) ? -1 : i1; if (key < lo) lo = key; }
      lo = __reduce_min_sync(FULL, lo);
      if (lo == 0x7fffffff) { status = LCP_EMPTY_RATIO; break; }
      r = (lo < 0) ? trow : lo;
    }
    const int leaving = bas[r];
    const double p = __shfl_sync(FULL, (r < 32) ? d0 : d1, r & 31);
    const bool is0 = h0 && i0 == r, is1 = h1 && i1 == r;        // this lane owns the pivot row
    __syncwarp();                                               // everyone has read bas / where / rvec before they change
    // The owner hands its row over and clears it to -0.0: with the multiplier 1 below, fma(1, r_c, -0.0) == r_c bit for bit
    // (signed zeros included), so the pivot row needs no special case in the update.
    if (is0) {
#pragma unroll
      for (int c = 0; c < NC; c++) { rvec[c] = R0[c]; R0[c] = -0.0; }
    }
    if (TWO && is1) {
#pragma unroll
      for (int c = 0; c < NC; c++) { rvec[c] = R1[c]; R1[c] = -0.0; }
    }
    // the leaving variable's column (a unit vector while basic) replaces slot s: every other row starts it from zero
    b2m_static_switch<NC>(s, [&](auto ic) { constexpr int c = decltype(ic)::value; if (!is0) R0[c] = 0.0; if (TWO && !is1) R1[c] = 0.0; });
    __syncwarp();
    {   // pivot row, scaled: lane c forms r_c (and r_{c+32})
      const int ca = lane, cb = lane + 32;
      const bool ha = ca < NC, hb = cb < NC;
      const double num[2] = {(ca == s) ? 1.0 : rvec[ha ? ca : 0], (cb == s) ? 1.0 : rvec[hb ? cb : 0]}, den[2] = {p, p};
      double rv[2];
      b2m_divn<2>(num, den, rv);
      if (ha) rvec[ca] = rv[0];
      if (hb) rvec[cb] = rv[1];
    }
    if (lane == 0) {
      if (log && nlog < log_cap) log[nlog] = leaving;
      where[entering] = -(r + 1); where[leaving] = s; bas[r] = entering;
    }
    nlog++;
    __syncwarp();
    const double m0 = is0 ? 1.0 : -d0, m1 = is1 ? 1.0 : -d1;
#pragma unroll
    for (int c = 0; c < NC; c++) {
      const double rc = rvec[c];
      R0[c] = fma(m0, rc, R0[c]);
      if (TWO) R1[c] = fma(m1, rc, R1[c]);
    }
    if (!first) piv++;
    if (budget && --bud < 0) { status = LCP_DEFER; break; }
    if (cancel && (piv & 63) == 63 && *cancel) { status = LCP_DEFER; break; }
    first = false;
    if (leaving == t) break;
    if (piv >= MAXITER) { status = LCP_MAXITER; break; }
    entering = (leaving < n) ? n + leaving : leaving - n;
    s = where[entering];
  }
  __syncwarp();
  if (h0) T[n * (n + 1) + i0] = R0[N + 1];                      // x back to the tableau: the caller reads the solution from it
  if (h1) T[n * (n + 1) + i1] = R1[N + 1];
  __syncwarp();
  nlog_io = nlog; piv_io = piv; executed_io = executed; if (budget) *budget = bud;
  return status;
}
// Measured and NOT used by default (profiles/r02_lemke_register_tableau.json): 16.2 M against 22.9 M solves/s at n = 40 and
// 54.8 M against 95.5 M at n = 20 on the batched solver microbenchmark, 8.0 against 7.0 ms for the hard queue of configs[1].
// Shared-memory wavefronts do drop 3.4x (467 M against 1,601 M per launch), but the 2 x 42 register rows leave the
// compiler no registers to keep the pivot-row loads ahead of the fmas (short-scoreboard stalls on every r_c), and the
// jump into "register s" costs instruction fetches (no_instruction stalls) that the compact shared-memory loop never pays.
#ifndef B2M_LEMKE_REG
#define B2M_LEMKE_REG 0
#endif
template <bool SH>
static __device__ __forceinline__ int lemke_loop_warp_n(int n, double* T, double* rvec, int* where, int* bas, double PIV_TOL, double zero_tol, int r,
                                                        int* log, int log_cap, int& nlog, int& piv, int& executed, int* budget, const volatile int* cancel) {
  if (SH && B2M_LEMKE_REG) {
    switch (n) {
      case 40: return lemke_loop_warp_reg<40>(T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
      case 30: return lemke_loop_warp_reg<30>(T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
      case 20: return lemke_loop_warp_reg<20>(T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
      case 10: return lemke_loop_warp_reg<10>(T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
      case 32: return lemke_loop_warp_reg<32>(T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
      case 24: return lemke_loop_warp_reg<24>(T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
      case 16: return lemke_loop_warp_reg<16>(T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
      default: break;
    }
  }
  switch (n) {
    case 40: return lemke_loop_warp<SH, 40>(n, T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
    case 32: return lemke_loop_warp<SH, 32>(n, T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
    case 30: return lemke_loop_warp<SH, 30>(n, T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
    case 24: return lemke_loop_warp<SH, 24>(n, T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
    case 20: return lemke_loop_warp<SH, 20>(n, T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
    case 16: return lemke_loop_warp<SH, 16>(n, T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
    default: return lemke_loop_warp<SH, 0>(n, T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
  }
}
#endif

// No cycle detection: LCP.cpp has no anti-cycling rule (:926-928) and on degenerate problems the pivoting can circle until
// the iteration cap (:548,789).  Round 1 cut such runs short when an (ordered basis, entering variable) pair recurred.
// That is a proof of periodicity only in exact arithmetic: the reference re-solves the entering column with a fresh LU
// every pivot (:834-838) but updates x incrementally (:983-988), the tableau here is incremental throughout, and on
// 1,024 envs x 300 steps of configs[1] the literal run left such "cycles" through rounding 1,268 pivots before the cap
// (same final states, different pivot counts), while a bit-exact variant (recurrence of the tracked state AND of every
// tableau entry's bits) never fired once.  So the solver is literal: it pivots until the reference would stop.
#ifdef __CUDACC__
// Rank-one update of a block-owned tableau that lives in global memory (L2): eight entries per thread in flight, all 24
// loads of a batch ahead of its first fma / store.  The pointer is declared global to the compiler: with generic loads it
// assumes shared-memory latency and interleaves each entry's fma with the next entry's loads, which serialises a batch into
// eight L2 round trips (profiles/r02_ncu_stacks_block_hotspots.txt).  Same operation per entry: bit-identical.  Returns
// the first entry index left for the caller's tail loop and advances (i, c) with it.
template <int NT>
static __device__ __forceinline__ int lemke_update_block_global(double* T, int n, int r, int e, int& i, int& c) {
  __builtin_assume(__isGlobal(T));
  const double* dvec = T + (size_t)n * (n + 2);
  const double* rvec = dvec + n;
  const int di = NT % n, dc = NT / n;
  const int total = n * (n + 2);
  constexpr int B = 8;
  for (; e + (B - 1) * NT < total; e += B * NT) {
    double tv[B], dv[B], rv[B]; bool pr[B];
#pragma unroll
    for (int k = 0; k < B; k++) {
      tv[k] = T[e + k * NT]; dv[k] = dvec[i]; rv[k] = rvec[c]; pr[k] = (i == r);
      i += di; c += dc;
      if (i >= n) { i -= n; c++; }
    }
#pragma unroll
    for (int k = 0; k < B; k++) T[e + k * NT] = pr[k] ? rv[k] : fma(-dv[k], rv[k], tv[k]);
  }
  return e;
}
#endif

template <class G>
B2M_DEV B2M_NOINL int lemke_solve(const G& g, int n, const double* M, int ldm, const double* q, double lambda,
                           double piv_tol, double zero_tol, double* z, double* wd, int* wi, int* pivots_out,
                           int* log, int log_cap, int* log_len, int* budget = nullptr, int* executed_out = nullptr, double offdiag = -1.0,
                           const volatile int* cancel = nullptr) {      // cancel: ladder task pool; a cancelled run returns LCP_DEFER
  double* T = wd;
  double* dvec = T + (size_t)n * (n + 2);
  double* rvec = dvec + n;
  int* where = wi;            // variable id -> nonbasic slot (>= 0) or -(row+1) when basic
  int* bas = wi + 2 * n + 1;  // row -> variable id
  double* xcol = T + (size_t)n * (n + 1);
  const int t = 2 * n;
  const int MAXITER = min(1000, 50 * n);                                   // LCP.cpp:548
  int nlog = 0, piv = 0, status = LCP_OK;

  const double nrm = norm_inf_with(g, n, M, ldm, lambda, offdiag);
  if (zero_tol <= 0.0) zero_tol = B2M_EPS * nrm * n;                       // :570-571
  const double PIV_TOL = (piv_tol > 0.0) ? piv_tol : B2M_EPS * n * fmax(1.0, nrm);   // :761
  // trivial solution (:578-584)
  double mq = B2M_INF;
  for (int i = g.tid; i < n; i += G::size) mq = fmin(mq, q[i]);
  mq = g.min(mq);
  for (int i = g.tid; i < n; i += G::size) z[i] = 0.0;
  if (mq > -zero_tol) { if (pivots_out) *pivots_out = 0; if (log_len) *log_len = 0; g.sync(); return LCP_TRIVIAL; }
  if (!(mq < 0.0)) { if (pivots_out) *pivots_out = 0; if (log_len) *log_len = 0; g.sync(); return LCP_OK; }   // :737-758

  // initial tableau: B = -I  =>  B^-1 M[:,j] = -M[:,j];  cover column B^-1 u = -u with u_i = [q_i < 0]   (:696-698,776-785)
  if (G::size == 32 && ldm == n) {                                         // a warp walks M linearly (coalesced), keeping (row, column) by increments: no integer division
    int r = g.tid % n, c = g.tid / n;
    const int dr = 32 % n, dc = 32 / n;
    for (int e = g.tid; e < n * n; e += 32) {
      const double v = M[e];
      T[e] = -((r == c) ? v + lambda : v);
      r += dr; c += dc;
      if (r >= n) { r -= n; c++; }
    }
  } else
  for (int e = g.tid; e < n * n; e += G::size) { const int c = e / n, r = e - c * n; T[e] = -m_at(M, ldm, r, c, lambda); }
  for (int i = g.tid; i < n; i += G::size) {
    const double qi = q[i];
    T[(size_t)n * n + i] = (qi < 0.0) ? -1.0 : 0.0;
    xcol[i] = qi;
    where[i] = i; where[n + i] = -(i + 1); bas[i] = n + i;
  }
  if (g.tid == 0) where[t] = n;
  g.sync();

  // first leaving row: first minimum of x (:764-771); entering: the artificial variable
  int r; { double key = B2M_INF; int idx = 0x7fffffff;
    for (int i = g.tid; i < n; i += G::size) { const double x = xcol[i]; if (x < key) { key = x; idx = i; } }
    g.min_key_idx(key, idx); r = idx; }
  int s = n;           // entering slot
  int entering = t;
  bool first = true;   // the first pass pivots the artificial variable in (LCP.cpp:776-785); `piv` counts the pivots after it
  int executed = 0;
  bool handled = false;
#ifdef __CUDACC__
  if constexpr (G::size == 32) {
    if (n <= 64) {
      status = __isShared(T) ? lemke_loop_warp_n<true>(n, T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel)
                             : lemke_loop_warp<false, 0>(n, T, rvec, where, bas, PIV_TOL, zero_tol, r, log, log_cap, nlog, piv, executed, budget, cancel);
      handled = true;
    }
  }
#endif
  while (!handled) {
    // entering column
    for (int i = g.tid; i < n; i += G::size) dvec[i] = T[(size_t)s * n + i];
    g.sync();
    if (!first) {
      executed++;
      // ratio test (:886-975)
      // two group reductions per pivot: a finite ratio exists iff some d_i > PIV_TOL, and the artificial variable's row
      // enters the second one as key -1 so that it wins whenever it passes (LCP.cpp:961-975)
      double theta = B2M_INF;
      for (int i = g.tid; i < n; i += G::size) { const double d = dvec[i]; if (d > PIV_TOL) theta = fmin(theta, (xcol[i] + zero_tol) / d); }
      if (cancel && g.tid == 0 && *cancel) theta = -B2M_INF;               // ladder task pool: the owner has its answer; the flag rides on the reduction so that the whole group leaves together
      theta = g.min(theta);
      if (theta == -B2M_INF) { status = LCP_DEFER; break; }
      if (theta == B2M_INF) { status = LCP_RAY; break; }
      int lo = 0x7fffffff;
      const int trow = -(where[t] + 1);
      for (int i = g.tid; i < n; i += G::size) {
        const double d = dvec[i];
        if (d > PIV_TOL && xcol[i] / d <= theta) { const int key = (i == trow) ? -1 : i; if (key < lo) lo = key; }
      }
      lo = g.min(lo);
      if (lo == 0x7fffffff) { status = LCP_EMPTY_RATIO; break; }
      r = (lo < 0) ? trow : lo;
    }
    const int leaving = bas[r];
    const double p = dvec[r];
    g.sync();                                   // everyone has read bas/where/dvec[r] before they change
    // pivot row, scaled; the leaving variable's column (a unit vector while basic) replaces slot s
    for (int c = g.tid; c < n + 2; c += G::size) rvec[c] = (c == s) ? 1.0 / p : T[(size_t)c * n + r] / p;
    for (int i = g.tid; i < n; i += G::size) T[(size_t)s * n + i] = 0.0;
    if (g.tid == 0) {
      if (log && nlog < log_cap) log[nlog] = leaving;
      where[entering] = -(r + 1); where[leaving] = s; bas[r] = entering;
    }
    nlog++;
    g.sync();
    // rank-one update of the whole tableau (x included)
    {
      int i = g.tid % n, c = g.tid / n;
      const int di = G::size % n, dc = G::size / n;
      const int total = n * (n + 2);
      int e = g.tid;
#ifdef __CUDACC__
      if constexpr (G::size > 32) {
        if (__isGlobal(T)) e = lemke_update_block_global<G::size>(T, n, r, e, i, c);     // n in the hundreds: the tableau is in global scratch (L2)
      }
#endif
      for (; e < total; e += G::size) {
        T[e] = (i == r) ? rvec[c] : fma(-dvec[i], rvec[c], T[e]);
        i += di; c += dc;
        if (i >= n) { i -= n; c++; }
      }
    }
    g.sync();
    if (!first) piv++;
    if (budget && --(*budget) < 0) { status = LCP_DEFER; break; }
    first = false;
    if (leaving == t) break;                                               // :800-822 solved
    if (piv >= MAXITER) { status = LCP_MAXITER; break; }                   // :789
    entering = (leaving < n) ? n + leaving : leaving - n;                  // :823-833 complement
    s = where[entering];
  }
  if (status == LCP_OK) {
    for (int i = g.tid; i < n; i += G::size) { const int b = bas[i]; if (b < n) z[b] = xcol[i]; }
  }
  if (pivots_out) *pivots_out = piv;
  if (executed_out) *executed_out = executed;
  if (log_len) *log_len = nlog;
  g.sync();
  return status;
}

// ------------------------------------------------------------------------------------------------
// lcp_fast.  Work memory: A n*n, zz n, w n doubles; nonbas n, bas n ints (+2 ints of scalars).
// The sub-system solve follows the oracle's LU order operation for operation (partial pivoting on the
// first maximum, reciprocal multipliers, fma updates, column-oriented back substitution) so results are
// bit-identical to the CPU checker.
// ------------------------------------------------------------------------------------------------
B2M_HD inline size_t fast_work_doubles(int n) { return (size_t)n * n + 2 * (size_t)n; }
#define B2M_FAST_HIST 16   /* basis sets remembered by lcp_fast's cycle detector */
B2M_HD inline size_t fast_work_ints(int n) { return (size_t)2 * n + 2 + (size_t)(B2M_FAST_HIST + 1) * ((n + 31) / 32); }

#ifdef __CUDACC__
// Warp-owned LU solve (k <= 64): lane l owns rows l and l + 32 of A and keeps its entries of b in registers; the pivot
// search is one redux, the right-hand side travels by shuffle, the trailing update of a row walks the columns in
// straight-line batches of eight (all loads of a batch before the first fma, no guard inside, clamped indices).  Same
// operations on every element, in the same order, as the generic routine below (and as the oracle's solve_fast):
// bit-identical results.
template <int B>
static __device__ __forceinline__ void lu_update_batch(double* q0, double* q1, const double* pr, int c, int k, double nl0, double nl1, bool u0, bool u1) {
  double rv[B], a0[B], a1[B];
  const int ck = c * k;
#pragma unroll
  for (int q = 0; q < B; q++) { rv[q] = pr[ck + q * k]; a0[q] = q0[ck + q * k]; a1[q] = u1 ? q1[ck + q * k] : 0.0; }   // lanes without a live second row skip its load
#pragma unroll
  for (int q = 0; q < B; q++) { a0[q] = fma(nl0, rv[q], a0[q]); a1[q] = fma(nl1, rv[q], a1[q]); }
#pragma unroll
  for (int q = 0; q < B; q++) { if (u0) q0[ck + q * k] = a0[q]; if (u1) q1[ck + q * k] = a1[q]; }
}
template <bool SH>
static __device__ __noinline__ bool lu_solve_warp(int k, double* A, double* b) {
  if (SH) { __builtin_assume(__isShared(A)); __builtin_assume(__isShared(b)); }
  else { __builtin_assume(__isGlobal(A)); }
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int i0 = lane, i1 = lane + 32;
  const bool h0 = i0 < k, h1 = i1 < k;
  const int j0 = h0 ? i0 : 0, j1 = h1 ? i1 : j0;            // always-valid row indices
  double* const q0 = A + j0;
  double* const q1 = A + j1;
  double b0 = b[j0], b1 = b[j1];
  for (int j = 0; j < k; j++) {
    double key = 1.0; int p = 0x7fffffff;                       // lexicographic min of (-|a|, i) == first maximum
    { const double v0 = -fabs(q0[j * k]), v1 = -fabs(q1[j * k]);
      if (h0 && i0 >= j && v0 < key) { key = v0; p = i0; }
      if (h1 && i1 >= j && v1 < key) { key = v1; p = i1; } }
    b2m_warp_min_key_idx(key, p);
    if (key == 0.0 || p == 0x7fffffff) return false;
    if (p != j) {
      for (int c = lane; c < k; c += 32) { const double tmp = A[c * k + j]; A[c * k + j] = A[c * k + p]; A[c * k + p] = tmp; }
      const double vj = __shfl_sync(FULL, (j < 32) ? b0 : b1, j & 31), vp = __shfl_sync(FULL, (p < 32) ? b0 : b1, p & 31);
      if (i0 == j) b0 = vp; else if (i0 == p) b0 = vj;
      if (i1 == j) b1 = vp; else if (i1 == p) b1 = vj;
    }
    __syncwarp();
    const double rinv = 1.0 / A[j * k + j];
    const double bj = __shfl_sync(FULL, (j < 32) ? b0 : b1, j & 31);
    const bool u0 = h0 && i0 > j, u1 = h1 && i1 > j;
    const double l0 = q0[j * k] * rinv, l1 = q1[j * k] * rinv;
    if (u0) { q0[j * k] = l0; b0 = fma(-l0, bj, b0); }
    if (u1) { q1[j * k] = l1; b1 = fma(-l1, bj, b1); }
    const double nl0 = -l0, nl1 = -l1;
    const double* const pr = A + j;                             // pivot row
    int c = j + 1;
    const int rem = k - c;
    for (; c + 8 <= k; c += 8) lu_update_batch<8>(q0, q1, pr, c, k, nl0, nl1, u0, u1);
    if (rem & 4) { lu_update_batch<4>(q0, q1, pr, c, k, nl0, nl1, u0, u1); c += 4; }
    if (rem & 2) { lu_update_batch<2>(q0, q1, pr, c, k, nl0, nl1, u0, u1); c += 2; }
    if (rem & 1) lu_update_batch<1>(q0, q1, pr, c, k, nl0, nl1, u0, u1);
    __syncwarp();
  }
  // column-oriented back substitution; the diagonal is read once, x_c = b_c / u_cc travels by shuffle
  const double dg0 = q0[j0 * k], dg1 = q1[j1 * k];
  for (int c = k - 1; c >= 0; c--) {
    const double a0 = q0[c * k], a1 = q1[c * k];                // independent of the running x: issued ahead of the shuffle / divide chain
    const double bc = __shfl_sync(FULL, (c < 32) ? b0 : b1, c & 31), dc = __shfl_sync(FULL, (c < 32) ? dg0 : dg1, c & 31);
    const double xc = bc / dc;
    if (i0 == c) b0 = xc; else if (h0 && i0 < c) b0 = fma(-a0, xc, b0);
    if (i1 == c) b1 = xc; else if (h1 && i1 < c) b1 = fma(-a1, xc, b1);
  }
  if (h0) b[i0] = b0;
  if (h1) b[i1] = b1;
  __syncwarp();
  return true;
}
#endif

// solves A x = b (A k x k column-major ld k, destroyed; b <- x).  Returns false on an exactly zero pivot.
// One thread per system (the thread-per-env kernels: A and b in the thread's local memory).  Same pivot rule and the
// same fma per element as the generic loop below, but organised for instruction-level parallelism: a lone thread is bound
// by the latency of its dependent load -> fma -> store chains, so every pass reads a batch of operands before it writes
// any (the compiler cannot reorder the generic loop's loads across its stores: it cannot prove that A[c*k+j] and
// A[c*k+i] differ), and the elimination walks columns in the outer loop so the inner one is unit-stride.
// lda is the column stride: the thread-per-env kernels pass the LCP dimension n, the same for every env of a warp, so
// that equal (row, column) of the 32 systems a warp factors in lock step sit at equal local-memory offsets and the
// hardware coalesces them; with lda = k (each env's own count of nonbasic variables) every access of the warp touched up
// to 32 different lines, and the L1's line-per-cycle pipeline -- not latency -- set the kernel's speed.
B2M_DEV B2M_NOINL inline bool lu_solve_serial(int k, double* A, int lda, double* b) {
  for (int j = 0; j < k; j++) {
    double* Aj = A + (size_t)j * lda;
    double key = 1.0; int p = 0x7fffffff;                       // first maximum of |A(i,j)|, i >= j
    for (int i = j; i < k; i++) { const double v = -fabs(Aj[i]); if (v < key) { key = v; p = i; } }
    if (key == 0.0 || p == 0x7fffffff) return false;
    if (p != j) {
      int c = 0;
      for (; c + 4 <= k; c += 4) {
        double* r0 = A + (size_t)c * lda; double* r1 = r0 + lda; double* r2 = r1 + lda; double* r3 = r2 + lda;
        const double a0 = r0[j], a1 = r1[j], a2 = r2[j], a3 = r3[j], b0 = r0[p], b1 = r1[p], b2 = r2[p], b3 = r3[p];
        r0[j] = b0; r1[j] = b1; r2[j] = b2; r3[j] = b3; r0[p] = a0; r1[p] = a1; r2[p] = a2; r3[p] = a3;
      }
      for (; c < k; c++) { double* r0 = A + (size_t)c * lda; const double a0 = r0[j]; r0[j] = r0[p]; r0[p] = a0; }
      const double tmp = b[j]; b[j] = b[p]; b[p] = tmp;
    }
    const double rinv = 1.0 / Aj[j];
    const double bj = b[j];
    {   // multipliers l_i = A(i,j) / A(j,j) and the right-hand side
      int i = j + 1;
      for (; i + 4 <= k; i += 4) {
        const double l0 = Aj[i] * rinv, l1 = Aj[i + 1] * rinv, l2 = Aj[i + 2] * rinv, l3 = Aj[i + 3] * rinv;
        const double c0 = b[i], c1 = b[i + 1], c2 = b[i + 2], c3 = b[i + 3];
        Aj[i] = l0; Aj[i + 1] = l1; Aj[i + 2] = l2; Aj[i + 3] = l3;
        b[i] = fma(-l0, bj, c0); b[i + 1] = fma(-l1, bj, c1); b[i + 2] = fma(-l2, bj, c2); b[i + 3] = fma(-l3, bj, c3);
      }
      for (; i < k; i++) { const double l0 = Aj[i] * rinv; Aj[i] = l0; b[i] = fma(-l0, bj, b[i]); }
    }
    int c = j + 1;
    for (; c + 2 <= k; c += 2) {                                // two columns at a time, four rows per batch
      double* A0 = A + (size_t)c * lda; double* A1 = A0 + lda;
      const double u0 = A0[j], u1 = A1[j];
      int i = j + 1;
      for (; i + 4 <= k; i += 4) {
        const double l0 = Aj[i], l1 = Aj[i + 1], l2 = Aj[i + 2], l3 = Aj[i + 3];
        const double x0 = A0[i], x1 = A0[i + 1], x2 = A0[i + 2], x3 = A0[i + 3];
        const double y0 = A1[i], y1 = A1[i + 1], y2 = A1[i + 2], y3 = A1[i + 3];
        A0[i] = fma(-l0, u0, x0); A0[i + 1] = fma(-l1, u0, x1); A0[i + 2] = fma(-l2, u0, x2); A0[i + 3] = fma(-l3, u0, x3);
        A1[i] = fma(-l0, u1, y0); A1[i + 1] = fma(-l1, u1, y1); A1[i + 2] = fma(-l2, u1, y2); A1[i + 3] = fma(-l3, u1, y3);
      }
      for (; i < k; i++) { const double l0 = Aj[i], x0 = A0[i], y0 = A1[i]; A0[i] = fma(-l0, u0, x0); A1[i] = fma(-l0, u1, y0); }
    }
    for (; c < k; c++) {
      double* A0 = A + (size_t)c * lda;
      const double u0 = A0[j];
      int i = j + 1;
      for (; i + 4 <= k; i += 4) {
        const double l0 = Aj[i], l1 = Aj[i + 1], l2 = Aj[i + 2], l3 = Aj[i + 3];
        const double x0 = A0[i], x1 = A0[i + 1], x2 = A0[i + 2], x3 = A0[i + 3];
        A0[i] = fma(-l0, u0, x0); A0[i + 1] = fma(-l1, u0, x1); A0[i + 2] = fma(-l2, u0, x2); A0[i + 3] = fma(-l3, u0, x3);
      }
      for (; i < k; i++) { const double l0 = Aj[i], x0 = A0[i]; A0[i] = fma(-l0, u0, x0); }
    }
  }
  for (int c = k - 1; c >= 0; c--) {
    const double* Ac = A + (size_t)c * lda;
    const double xc = b[c] / Ac[c];
    b[c] = xc;
    int i = 0;
    for (; i + 4 <= c; i += 4) {
      const double a0 = Ac[i], a1 = Ac[i + 1], a2 = Ac[i + 2], a3 = Ac[i + 3], c0 = b[i], c1 = b[i + 1], c2 = b[i + 2], c3 = b[i + 3];
      b[i] = fma(-a0, xc, c0); b[i + 1] = fma(-a1, xc, c1); b[i + 2] = fma(-a2, xc, c2); b[i + 3] = fma(-a3, xc, c3);
    }
    for (; i < c; i++) b[i] = fma(-Ac[i], xc, b[i]);
  }
  return true;
}

#ifdef __CUDACC__
// Trailing update of column step j of a block-owned LU in global memory: A[c][i] -= l_i * A[c][j] for i, c > j, the (k - j - 1)^2
// entries spread over all NT threads (column-major walk: coalesced), eight entries per thread in flight.  One row per thread
// with a dependent column loop left most of the block idle and paid one L2 round trip per entry (the lcp_fast phase of the
// n = 320 stacks: profiles/r02_stacks_profile_*).  Same fma per entry: bit-identical.
template <int NT>
static __device__ __forceinline__ void lu_trailing_update_block_global(double* A, int k, int j, int tid) {
  __builtin_assume(__isGlobal(A));
  const int m = k - j - 1;
  if (m <= 0) return;
  double* base = A + (size_t)(j + 1) * k + (j + 1);              // entry (ii, cc) at base[cc * k + ii]
  const double* prow = A + (size_t)(j + 1) * k + j;              // pivot-row entry of column cc at prow[cc * k]
  const double* lcol = A + (size_t)j * k + (j + 1);              // multiplier of row ii
  int ii = tid % m, cc = tid / m;
  const int di = NT % m, dc = NT / m;
  const int total = m * m;
  constexpr int B = 8;
  int e = tid;
  for (; e + (B - 1) * NT < total; e += B * NT) {
    double a[B], l[B], pv[B]; int off[B];
#pragma unroll
    for (int q = 0; q < B; q++) {
      off[q] = cc * k + ii; a[q] = base[off[q]]; l[q] = lcol[ii]; pv[q] = prow[cc * k];
      ii += di; cc += dc;
      if (ii >= m) { ii -= m; cc++; }
    }
#pragma unroll
    for (int q = 0; q < B; q++) base[off[q]] = fma(-l[q], pv[q], a[q]);
  }
  for (; e < total; e += NT) {
    const int o = cc * k + ii;
    base[o] = fma(-lcol[ii], prow[cc * k], base[o]);
    ii += di; cc += dc;
    if (ii >= m) { ii -= m; cc++; }
  }
}
#endif

template <class G>
B2M_DEV B2M_NOINL bool lu_solve(const G& g, int k, double* A, double* b) {
  if constexpr (G::size == 1) return lu_solve_serial(k, A, k, b);
#ifdef __CUDACC__
  if constexpr (G::size == 32) { if (k <= 64) return __isShared(A) ? lu_solve_warp<true>(k, A, b) : lu_solve_warp<false>(k, A, b); }
#endif
  for (int j = 0; j < k; j++) {
    double key = 1.0; int p = 0x7fffffff;                       // lexicographic min of (-|a|, i) == first maximum
    for (int i = j + g.tid; i < k; i += G::size) { const double v = -fabs(A[(size_t)j * k + i]); if (v < key) { key = v; p = i; } }
    g.min_key_idx(key, p);
    if (key == 0.0 || p == 0x7fffffff) return false;
    if (p != j) {
      for (int c = g.tid; c < k; c += G::size) { const double tmp = A[(size_t)c * k + j]; A[(size_t)c * k + j] = A[(size_t)c * k + p]; A[(size_t)c * k + p] = tmp; }
      if (g.tid == 0) { const double tmp = b[j]; b[j] = b[p]; b[p] = tmp; }
    }
    g.sync();
    const double rinv = 1.0 / A[(size_t)j * k + j];
    const double bj = b[j];
#ifdef __CUDACC__
    if constexpr (G::size > 32) {
      if (__isGlobal(A)) {                                      // a block's sub-system in global scratch (n in the hundreds): multipliers first, then the
        for (int i = j + 1 + g.tid; i < k; i += G::size) {      // trailing block entry by entry over all threads instead of one row per thread
          const double l = A[(size_t)j * k + i] * rinv;
          A[(size_t)j * k + i] = l;
          b[i] = fma(-l, bj, b[i]);
        }
        g.sync();
        lu_trailing_update_block_global<G::size>(A, k, j, g.tid);
        g.sync();
        continue;
      }
    }
#endif
    for (int i = j + 1 + g.tid; i < k; i += G::size) {
      const double l = A[(size_t)j * k + i] * rinv;
      A[(size_t)j * k + i] = l;
      for (int c = j + 1; c < k; c++) A[(size_t)c * k + i] = fma(-l, A[(size_t)c * k + j], A[(size_t)c * k + i]);
      b[i] = fma(-l, bj, b[i]);
    }
    g.sync();
  }
  for (int c = k - 1; c >= 0; c--) {
    const double xc = b[c] / A[(size_t)c * k + c];
    g.sync();
    if (g.tid == 0) b[c] = xc;
    for (int i = g.tid; i < c; i += G::size) b[i] = fma(-A[(size_t)c * k + i], xc, b[i]);
    g.sync();
  }
  return true;
}

B2M_DEV inline void list_erase(int* L, int& m, int pos) { for (int i = pos; i + 1 < m; i++) L[i] = L[i + 1]; m--; }
B2M_DEV inline void list_insert_sorted(int* L, int& m, int v) { int i = m; while (i > 0 && L[i - 1] > v) { L[i] = L[i - 1]; i--; } L[i] = v; m++; }

// Cycle detector: one lcp_fast iteration is a pure function of the nonbasic index set (lowest-index tie rule), so a
// set seen before in this call proves the iteration will repeat until the 2n cap (LCP.cpp:107,192-195).  The call then
// returns what the reference returns -- failure, z untouched, pivots = 2n -- without spinning through the remaining
// iterations.  Exact, not heuristic: results and reference-equivalent pivot counts are unchanged; *executed_out says
// how many iterations really ran.
template <class G>
B2M_DEV B2M_NOINL int lcp_fast_solve(const G& g, int n, const double* M, int ldm, const double* q, double lambda, double zero_tol,
                              bool warm, double* z, double* wd, int* wi, int* pivots_out, int* log, int log_cap,
                              int* log_len, int* budget = nullptr, int* executed_out = nullptr, double offdiag = -1.0) {
  double* A = wd;
  double* zz = A + (size_t)n * n;
  double* w = zz + n;
  int* nonbas = wi;
  int* bas = wi + n;
  int* cnt = wi + 2 * n;      // cnt[0] = |nonbas|, cnt[1] = |bas|
  const int W32 = (n + 31) >> 5;
  unsigned* cur = (unsigned*)(wi + 2 * n + 2);   // bit i set <=> i is nonbasic
  unsigned* hist = cur + W32;                    // ring of the last B2M_FAST_HIST sets
  int nlog = 0, nh = 0, executed = 0;
  if (executed_out) *executed_out = 0;
  if (zero_tol < 0.0) zero_tol = n * norm_inf_with(g, n, M, ldm, lambda, offdiag) * B2M_EPS;      // LCP.cpp:57-58
  if (warm) {                                                                        // :65-85
    if (g.tid == 0) {
      int k = 0, nb = 0;
      for (int i = 0; i < W32; i++) cur[i] = 0u;
      for (int i = 0; i < n; i++) { if (fabs(z[i]) < zero_tol) bas[nb++] = i; else { nonbas[k++] = i; cur[i >> 5] |= 1u << (i & 31); } }
      cnt[0] = k; cnt[1] = nb;
    }
  } else {                                                                           // :86-103
    double key = B2M_INF; int idx = 0x7fffffff;
    for (int i = g.tid; i < n; i += G::size) { const double x = q[i]; if (x < key) { key = x; idx = i; } }
    g.min_key_idx(key, idx);
    if (key > -zero_tol) {
      for (int i = g.tid; i < n; i += G::size) z[i] = 0.0;
      if (pivots_out) *pivots_out = 0; if (log_len) *log_len = 0;
      g.sync();
      return LCP_TRIVIAL;
    }
    if (g.tid == 0) {
      nonbas[0] = idx; int nb = 0; for (int i = 0; i < n; i++) if (i != idx) bas[nb++] = i; cnt[0] = 1; cnt[1] = nb;
      for (int i = 0; i < W32; i++) cur[i] = 0u;
      cur[idx >> 5] |= 1u << (idx & 31);
    }
  }
  g.sync();
  const int MAX_PIV = 2 * n;                                                         // :107
  int piv = 0, status = LCP_MAXITER;
  for (piv = 0; piv < MAX_PIV; piv++) {
    if (budget && --(*budget) < 0) { status = LCP_DEFER; break; }
    {   // seen this basis before?  (log == nullptr only: the logged variant is the literal one, used by the pivot-log parity tests)
      bool rep = false;
      if (!log) {
        const int stored = nh < B2M_FAST_HIST ? nh : B2M_FAST_HIST;
        for (int t = g.tid; t < stored; t += G::size) {
          bool eq = true;
          for (int i = 0; i < W32; i++) eq = eq && (hist[t * W32 + i] == cur[i]);
          rep = rep || eq;
        }
      }
      if (g.any(rep)) { piv = MAX_PIV; break; }
      if (!log) { for (int i = g.tid; i < W32; i += G::size) hist[(nh % B2M_FAST_HIST) * W32 + i] = cur[i]; nh++; }
    }
    executed++;
    const int k = cnt[0], nb = cnt[1];
    if (G::size == 32 && k <= 64) {                                                    // a warp fills the rows it owns: no integer division
      const double* __restrict__ Mr = M; const int* __restrict__ nbp = nonbas; double* __restrict__ Ar = A;
      for (int r = g.tid; r < k; r += G::size) {
        const int nr = nbp[r];
#pragma unroll 4
        for (int c = 0; c < k; c++) Ar[c * k + r] = m_at(Mr, ldm, nr, nbp[c], lambda);
      }
    } else if (G::size == 1) {                                                         // one thread: column by column, four loads in flight, no integer division
      for (int c = 0; c < k; c++) {
        const int nc = nonbas[c];
        const double* Mc = M + (size_t)nc * ldm;
        double* Ac = A + (size_t)c * n;                                                 // column stride n, not k: see lu_solve_serial
        int r = 0;
        for (; r + 4 <= k; r += 4) {
          const int r0 = nonbas[r], r1 = nonbas[r + 1], r2 = nonbas[r + 2], r3 = nonbas[r + 3];
          const double v0 = Mc[r0], v1 = Mc[r1], v2 = Mc[r2], v3 = Mc[r3];
          Ac[r] = (r0 == nc) ? v0 + lambda : v0; Ac[r + 1] = (r1 == nc) ? v1 + lambda : v1;
          Ac[r + 2] = (r2 == nc) ? v2 + lambda : v2; Ac[r + 3] = (r3 == nc) ? v3 + lambda : v3;
        }
        for (; r < k; r++) { const int r0 = nonbas[r]; const double v0 = Mc[r0]; Ac[r] = (r0 == nc) ? v0 + lambda : v0; }
      }
    } else
    for (int e = g.tid; e < k * k; e += G::size) { const int c = e / k, r = e - c * k; A[e] = m_at(M, ldm, nonbas[r], nonbas[c], lambda); }   // :111
    for (int i = g.tid; i < k; i += G::size) zz[i] = -q[nonbas[i]];                  // :113-115
    g.sync();
    bool lu_ok;
    if constexpr (G::size == 1) lu_ok = lu_solve_serial(k, A, n, zz); else lu_ok = lu_solve(g, k, A, zz);
    if (!lu_ok) { status = LCP_SINGULAR; break; }                                    // :118-126
    if (G::size == 1) {                                                              // :129, four rows of w per pass: four independent fma chains
      int i = 0;
      for (; i + 4 <= nb; i += 4) {
        const int b0 = bas[i], b1 = bas[i + 1], b2 = bas[i + 2], b3 = bas[i + 3];
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        for (int c = 0; c < k; c++) {
          const double* Mc = M + (size_t)nonbas[c] * ldm;
          const double zc = zz[c];
          const double m0 = Mc[b0], m1 = Mc[b1], m2 = Mc[b2], m3 = Mc[b3];
          s0 = fma(m0, zc, s0); s1 = fma(m1, zc, s1); s2 = fma(m2, zc, s2); s3 = fma(m3, zc, s3);
        }
        const double q0 = q[b0], q1 = q[b1], q2 = q[b2], q3 = q[b3];
        w[i] = s0 + q0; w[i + 1] = s1 + q1; w[i + 2] = s2 + q2; w[i + 3] = s3 + q3;
      }
      for (; i < nb; i++) {
        const int b0 = bas[i];
        double s0 = 0.0;
        for (int c = 0; c < k; c++) s0 = fma(M[(size_t)nonbas[c] * ldm + b0], zz[c], s0);
        w[i] = s0 + q[b0];
      }
    } else
    for (int i = g.tid; i < nb; i += G::size) {                                      // :129
      const int bi = bas[i];
      const double* __restrict__ Mr = M; const int* __restrict__ nbp = nonbas; const double* __restrict__ zr = zz;
      double sacc = 0.0;
#pragma unroll 4
      for (int c = 0; c < k; c++) sacc = fma(Mr[(size_t)nbp[c] * ldm + bi], zr[c], sacc);
      w[i] = sacc + q[bi];
    }
    g.sync();
    const int minw = (nb > 0) ? rand_min(g, w, nb, zero_tol) : -1;                   // :130
    if (minw < 0 || w[minw] > -zero_tol) {                                           // :135
      const int minz = (k > 0) ? rand_min(g, zz, k, zero_tol) : -1;                  // :138
      if (minz >= 0 && zz[minz] < -zero_tol) {                                       // :141-150
        g.sync();
        if (g.tid == 0) {
          int kk = k, nbb = nb; const int idx = nonbas[minz];
          list_erase(nonbas, kk, minz); list_insert_sorted(bas, nbb, idx);
          cur[idx >> 5] &= ~(1u << (idx & 31));
          cnt[0] = kk; cnt[1] = nbb;
          if (log && nlog < log_cap) log[nlog] = idx | 0x40000000;
        }
        nlog++;
      } else {                                                                       // :151-162
        g.sync();
        for (int i = g.tid; i < n; i += G::size) z[i] = 0.0;
        g.sync();
        for (int j = g.tid; j < k; j += G::size) z[nonbas[j]] = zz[j];
        status = LCP_OK;
        break;
      }
    } else {                                                                         // :164-189
      const int minz = (k > 0) ? rand_min(g, zz, k, zero_tol) : -1;                  // :176 (old ordering)
      const bool second = (minz >= 0 && zz[minz] < -zero_tol);
      g.sync();
      if (g.tid == 0) {
        int kk = k, nbb = nb; const int idx = bas[minw];
        list_erase(bas, nbb, minw); list_insert_sorted(nonbas, kk, idx);
        cur[idx >> 5] |= 1u << (idx & 31);
        if (log && nlog < log_cap) log[nlog] = idx;
        if (second) {                                                                // :179-188 (position in the NEW list)
          const int idx2 = nonbas[minz];
          list_erase(nonbas, kk, minz); list_insert_sorted(bas, nbb, idx2);
          cur[idx2 >> 5] &= ~(1u << (idx2 & 31));
          if (log && nlog + 1 < log_cap) log[nlog + 1] = idx2 | 0x40000000;
        }
        cnt[0] = kk; cnt[1] = nbb;
      }
      nlog += second ? 2 : 1;
    }
    g.sync();
  }
  if (pivots_out) *pivots_out = piv;
  if (executed_out) *executed_out = executed;
  if (log_len) *log_len = nlog;
  g.sync();
  return status;
}

// Solution checks of the regularised wrappers (LCP.cpp:240-256 with >=, :303-319 with >); w is scratch (n).
template <class G>
B2M_DEV B2M_NOINL bool lcp_verify(const G& g, int n, const double* M, int ldm, const double* q, double lambda, const double* z,
                           double ZERO_TOL, bool strict, double* w) {
  double mz = B2M_INF, mw = B2M_INF, mn = B2M_INF, mx = -B2M_INF;
  if constexpr (G::size == 1) {                                  // one thread: four rows of w = (M + lambda I) z + q per pass (four independent fma chains, each in column order)
    int i = 0;
    for (; i + 4 <= n; i += 4) {
      double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
      for (int c = 0; c < n; c++) {
        const double* Mc = M + (size_t)c * ldm + i;
        const double zc = z[c];
        double a0 = Mc[0], a1 = Mc[1], a2 = Mc[2], a3 = Mc[3];
        if ((unsigned)(c - i) < 4u) { const int d = c - i; if (d == 0) a0 += lambda; else if (d == 1) a1 += lambda; else if (d == 2) a2 += lambda; else a3 += lambda; }
        s0 = fma(a0, zc, s0); s1 = fma(a1, zc, s1); s2 = fma(a2, zc, s2); s3 = fma(a3, zc, s3);
      }
      const double w4[4] = {s0 + q[i], s1 + q[i + 1], s2 + q[i + 2], s3 + q[i + 3]};
      for (int u = 0; u < 4; u++) { const double zi = z[i + u], pr = zi * w4[u]; mz = fmin(mz, zi); mw = fmin(mw, w4[u]); mn = fmin(mn, pr); mx = fmax(mx, pr); }
    }
    for (; i < n; i++) {
      double sacc = 0.0;
      for (int c = 0; c < n; c++) sacc = fma(m_at(M, ldm, i, c, lambda), z[c], sacc);
      const double wi = sacc + q[i], pr = z[i] * wi;
      mz = fmin(mz, z[i]); mw = fmin(mw, wi); mn = fmin(mn, pr); mx = fmax(mx, pr);
    }
  } else
  for (int i = g.tid; i < n; i += G::size) {
    double sacc = 0.0;
    for (int c = 0; c < n; c++) sacc = fma(m_at(M, ldm, i, c, lambda), z[c], sacc);
    const double wi = sacc + q[i];
    const double pr = z[i] * wi;
    mz = fmin(mz, z[i]); mw = fmin(mw, wi); mn = fmin(mn, pr); mx = fmax(mx, pr);
  }
  mz = g.min(mz); mw = g.min(mw); mn = g.min(mn); mx = g.max(mx);
  const bool lo_ok = strict ? (mz > -ZERO_TOL && mw > -ZERO_TOL && mn > -ZERO_TOL) : (mz >= -ZERO_TOL && mw >= -ZERO_TOL && mn >= -ZERO_TOL);
  return lo_ok && (mx < ZERO_TOL);
}

// 10^e from correctly rounded decimal literals (identical on host and device); std::pow(10, e) in the reference
B2M_DEV inline double pow10i(int e) {
  switch (e) {
    case -24: return 1e-24;
    case -23: return 1e-23;
    case -22: return 1e-22;
    case -21: return 1e-21;
    case -20: return 1e-20;
    case -19: return 1e-19;
    case -18: return 1e-18;
    case -17: return 1e-17;
    case -16: return 1e-16;
    case -15: return 1e-15;
    case -14: return 1e-14;
    case -13: return 1e-13;
    case -12: return 1e-12;
    case -11: return 1e-11;
    case -10: return 1e-10;
    case -9: return 1e-9;
    case -8: return 1e-8;
    case -7: return 1e-7;
    case -6: return 1e-6;
    case -5: return 1e-5;
    case -4: return 1e-4;
    case -3: return 1e-3;
    case -2: return 1e-2;
    case -1: return 1e-1;
    case 0: return 1e0;
    case 1: return 1e1;
    case 2: return 1e2;
    case 3: return 1e3;
    case 4: return 1e4;
    case 5: return 1e5;
    case 6: return 1e6;
    case 7: return 1e7;
    case 8: return 1e8;
    case 9: return 1e9;
    case 10: return 1e10;
    case 11: return 1e11;
    case 12: return 1e12;
    case 13: return 1e13;
    case 14: return 1e14;
    case 15: return 1e15;
    case 16: return 1e16;
    case 17: return 1e17;
    case 18: return 1e18;
    case 19: return 1e19;
    case 20: return 1e20;
    case 21: return 1e21;
    case 22: return 1e22;
    case 23: return 1e23;
    case 24: return 1e24;
    default: return pow(10.0, (double)e);
  }
}

// lcp_fast_regularized (LCP.cpp:212-350).  stats[0] += lcp_fast calls, stats[1] += pivots as the
// reference counts them, stats[2] += iterations actually executed (thread 0 only, may be NULL).
// defer_unverified: return LCP_DEFER instead of climbing the regularisation rungs when the first solve does not verify.
template <class G>
B2M_DEV int lcp_fast_regularized(const G& g, int n, const double* M, int ldm, const double* q, double zero_tol, bool warm,
                                    int min_exp, int step_exp, int max_exp, double* z, double* wd, int* wi,
                                    int* pivots_out, long long* stats, int* budget = nullptr, bool defer_unverified = false) {
  if (n == 0) { if (pivots_out) *pivots_out = 0; return LCP_OK; }
  const double offdiag = norm_inf_offdiag(g, n, M, ldm);
  const double ZERO_TOL = (zero_tol > 0.0) ? zero_tol : n * norm_inf_with(g, n, M, ldm, 0.0, offdiag) * B2M_NEAR_ZERO;   // :228
  double* wv = wd + (size_t)n * n + n;   // the solver's w vector doubles as verification scratch
  int total = 0, piv = 0, ex = 0;
  int st = lcp_fast_solve(g, n, M, ldm, q, 0.0, zero_tol, warm, z, wd, wi, &piv, nullptr, 0, nullptr, budget, &ex, offdiag);
  if (st == LCP_DEFER) return st;
  bool zvalid = warm || st == LCP_OK || st == LCP_TRIVIAL;   // z.size()==n in the reference (LCP.cpp:65): warm start of the retries
  total += piv;
  if (stats && g.tid == 0) { stats[0]++; stats[1] += piv; stats[2] += ex; }
  if ((st == LCP_OK || st == LCP_TRIVIAL) && lcp_verify(g, n, M, ldm, q, 0.0, z, ZERO_TOL, false, wv)) {
    if (pivots_out) *pivots_out = piv;   // reference leaves `pivots` at the last solve's count here (:252-255)
    return st;
  }
  if (defer_unverified) return LCP_DEFER;
  int attempt = 0;
  for (int rf = min_exp; rf < max_exp; rf += step_exp, attempt++) {                 // :281-340
    const double lambda = pow10i(rf);
    g.sync();
    st = lcp_fast_solve(g, n, M, ldm, q, lambda, zero_tol, zvalid, z, wd, wi, &piv, nullptr, 0, nullptr, budget, &ex, offdiag);
    if (st == LCP_DEFER) return st;
    zvalid = zvalid || st == LCP_OK || st == LCP_TRIVIAL;
    total += piv;
    if (stats && g.tid == 0) { stats[0]++; stats[1] += piv; stats[2] += ex; }
    if ((st == LCP_OK || st == LCP_TRIVIAL) && lcp_verify(g, n, M, ldm, q, lambda, z, ZERO_TOL, true, wv)) {
      if (pivots_out) *pivots_out = total;
      return LCP_REGULARIZED + attempt;
    }
  }
  if (pivots_out) *pivots_out = total;
  return LCP_UNVERIFIED;
}

// lcp_lemke_regularized (LCP.cpp:353-487).
template <class G>
B2M_DEV int lcp_lemke_regularized(const G& g, int n, const double* M, int ldm, const double* q, double piv_tol,
                                     double zero_tol, int min_exp, int step_exp, int max_exp, double* z, double* wd,
                                     int* wi, int* pivots_out, long long* stats, int* budget = nullptr) {
  if (n == 0) { if (pivots_out) *pivots_out = 0; return LCP_OK; }
  const double offdiag = norm_inf_offdiag(g, n, M, ldm);
  const double ZERO_TOL = (zero_tol > 0.0) ? zero_tol : n * norm_inf_with(g, n, M, ldm, 0.0, offdiag) * B2M_NEAR_ZERO;   // :369
  double* wv = wd + (size_t)n * (n + 2);   // dvec doubles as verification scratch
  int total = 0, piv = 0, ex = 0;
  int st = lemke_solve(g, n, M, ldm, q, 0.0, piv_tol, zero_tol, z, wd, wi, &piv, nullptr, 0, nullptr, budget, &ex, offdiag);
  if (st == LCP_DEFER) return st;
  total += piv;
  if (stats && g.tid == 0) { stats[0]++; stats[1] += piv; stats[2] += ex; }
  if ((st == LCP_OK || st == LCP_TRIVIAL) && lcp_verify(g, n, M, ldm, q, 0.0, z, ZERO_TOL, false, wv)) {
    if (pivots_out) *pivots_out = piv;
    return st;
  }
  int attempt = 0;
  for (int rf = min_exp; rf < max_exp; rf += step_exp, attempt++) {                 // :419-477
    const double lambda = pow10i(rf);
    g.sync();
    st = lemke_solve(g, n, M, ldm, q, lambda, piv_tol, zero_tol, z, wd, wi, &piv, nullptr, 0, nullptr, budget, &ex, offdiag);
    if (st == LCP_DEFER) return st;
    total += piv;
    if (stats && g.tid == 0) { stats[0]++; stats[1] += piv; stats[2] += ex; }
    if ((st == LCP_OK || st == LCP_TRIVIAL) && lcp_verify(g, n, M, ldm, q, lambda, z, ZERO_TOL, true, wv)) {
      if (pivots_out) *pivots_out = total;
      return LCP_REGULARIZED + attempt;
    }
  }
  if (pivots_out) *pivots_out = total;
  for (int i = g.tid; i < n; i += G::size) z[i] = 0.0;
  g.sync();
  return LCP_UNVERIFIED;
}

#ifdef __CUDACC__
// ---- the regularisation ladder of lcp_lemke_regularized, its rungs solved side by side ------------------------------
// LCP.cpp:353-487 tries lambda = 0, then lambda = 10^rf for rf = min_exp, min_exp + step, ... one after the other and
// returns the first solve that passes its checks.  lcp_lemke ignores the incoming z (rule H9), so the rungs do not
// depend on each other: solving them at once on different warps and taking the FIRST rung that verifies, in ladder
// order, returns exactly what the sequential loop returns -- the same z, the same status and the same counters (calls,
// pivots and executed iterations are summed over the rungs up to the accepted one; what later rungs did is discarded).
// Every step a dozen envs of a 65,536-env batch (different ones each step: profiles/r02_impact_profile_*) run a ladder
// of six to ten rungs that each circle to the 1,000-pivot cap (LCP.cpp:548); the step time used to be the latency of
// that whole ladder on one warp.  With the rungs as stealable tasks it is the latency of two rungs.
//
// Mechanism (impact_warp_kernel): the warp that owns the env solves rung 0 itself; if that fails it copies (M, q) to its
// job buffer in global memory and posts one task per remaining rung to the launch's task list.  Any warp of the launch
// that has run out of envs -- and the owner itself while it waits -- takes tasks in order, solves them with the same
// lemke_solve / lcp_verify in its own shared-memory work area and writes status, pivots and z to the job's result
// slots.  The owner reads the results in rung order and cancels what has not started once it has its answer.  Owners
// execute tasks themselves while waiting, helpers never wait: no deadlock.  A task carries the job's generation so
// that tasks of an earlier request are skipped, and a job buffer is reused only when none of its tasks is running.
struct LadderPool {
  int* ctl;                 // [0] tasks posted, [1] tasks taken, [2] warps of the launch that may still post
  int* tasks;               // task list: (owner + 1) << 6 | rung, 0 = not yet published
  int* task_gen;            // generation of the owner's request the task belongs to
  int cap;                  // capacity of the task list
  double* jobs; size_t job_stride;    // per owner: M (nmax^2, ld n), q (nmax), then z of rung r at nmax^2 + nmax + r * nmax
  int* meta; size_t meta_stride;      // per owner: the words below, then 5 per rung (ready, status, ok, pivots, executed)
  double* jobd;             // per owner 4 doubles: piv_tol, zero_tol, ZERO_TOL, offdiag
  int nmax;
};
enum { LJ_GEN = 0, LJ_CANCEL, LJ_INFLIGHT, LJ_N, LJ_NRUNGS, LJ_MINEXP, LJ_STEPEXP, LJ_HDR = 8 };
#define B2M_LADDER_MAX_RUNGS 24
#define LJ_RW 8            /* ints per rung: ready, status, ok, pivots, executed, then (debug) pick-up and finish time in us */
#define LJ_POST 7          /* header word: (debug) time the job was posted, us */
__device__ __forceinline__ int b2m_now_us() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return (int)((t / 1000) & 0x7fffffff); }
#define B2M_LADDER_PROBE 128
B2M_HD inline size_t ladder_job_doubles(int nmax) { return (size_t)nmax * nmax + nmax + (size_t)B2M_LADDER_MAX_RUNGS * nmax; }
B2M_HD inline size_t ladder_job_ints() { return LJ_HDR + LJ_RW * B2M_LADDER_MAX_RUNGS; }
struct LadderCtx { LadderPool pool; int owner; double* wd; int* wi; long long* dbg = nullptr; };    // wd / wi: this warp's Lemke work area (shared memory)

// takes one task from the list and runs it; false when there was none.  G: the warp (WarpGroup) or the block (BlockGroup)
// that owns the work area wd / wi.
template <class G>
static __device__ __noinline__ bool ladder_help_one(const G& g, const LadderPool& L, double* wd, int* wi) {
  int v = 0, tg = 0, run = 0;
  if (g.tid == 0) {
    volatile int* ctl = L.ctl;
    for (;;) {
      const int h = ctl[1], t = min(ctl[0], L.cap);
      if (h >= t) break;
      if (atomicCAS(L.ctl + 1, h, h + 1) != h) continue;
      volatile int* tk = L.tasks;
      while ((v = tk[h]) == 0) {}
      __threadfence();
      tg = ((volatile int*)L.task_gen)[h];
      int* mo = L.meta + (size_t)((v >> 6) - 1) * L.meta_stride;
      atomicAdd(mo + LJ_INFLIGHT, 1);
      __threadfence();
      if (((volatile int*)mo)[LJ_GEN] == tg && ((volatile int*)mo)[LJ_CANCEL] == 0) { run = 1; mo[LJ_HDR + LJ_RW * (v & 63) + 5] = b2m_now_us(); ((volatile int*)mo)[LJ_HDR + LJ_RW * (v & 63)] = 2; }   // 2: taken, running
      else { atomicSub(mo + LJ_INFLIGHT, 1); run = 2; }      // stale or cancelled: skipped, but a task was consumed
      break;
    }
  }
  v = g.bcast(v); run = g.bcast(run);
  if (run == 0) return false;
  if (run == 2) return true;
  const int owner = (v >> 6) - 1, rung = v & 63;
  int* mo = L.meta + (size_t)owner * L.meta_stride;
  const double* jd = L.jobd + (size_t)owner * 4;
  double* job = L.jobs + (size_t)owner * L.job_stride;
  const int n = mo[LJ_N];
  const double* M = job; const double* q = job + (size_t)L.nmax * L.nmax;
  double* zr = job + (size_t)L.nmax * L.nmax + L.nmax + (size_t)rung * L.nmax;
  const double lambda = (rung == 0) ? 0.0 : pow10i(mo[LJ_MINEXP] + (rung - 1) * mo[LJ_STEPEXP]);
  int piv = 0, ex = 0;
  const int st = lemke_solve(g, n, M, n, q, lambda, jd[0], jd[1], zr, wd, wi, &piv, nullptr, 0, nullptr, nullptr, &ex, jd[3], (const volatile int*)(mo + LJ_CANCEL));
  const bool ok = (st == LCP_OK || st == LCP_TRIVIAL) && lcp_verify(g, n, M, n, q, lambda, zr, jd[2], rung > 0, wd + (size_t)n * (n + 2));
  __threadfence();                                     // every thread's part of z before the ready flag
  g.sync();
  if (g.tid == 0) {
    int* r = mo + LJ_HDR + LJ_RW * rung;
    r[1] = st; r[2] = ok ? 1 : 0; r[3] = piv; r[4] = ex; r[6] = b2m_now_us();
    __threadfence();
    ((volatile int*)r)[0] = 1;
    __threadfence();
    atomicSub(mo + LJ_INFLIGHT, 1);
  }
  g.sync();
  return true;
}

// lcp_lemke_regularized for the warp / block that owns the env (g: its group): same results and statistics as the sequential form
template <class G>
static __device__ __noinline__ int lcp_lemke_regularized_pool(const G& g, const LadderCtx& C, int n, const double* M, int ldm, const double* q, double piv_tol,
                                                              double zero_tol, int min_exp, int step_exp, int max_exp, double* z, int* pivots_out, long long* stats) {
  if (n == 0) { if (pivots_out) *pivots_out = 0; return LCP_OK; }
  const LadderPool& L = C.pool;
  const double offdiag = norm_inf_offdiag(g, n, M, ldm);
  const double ZERO_TOL = (zero_tol > 0.0) ? zero_tol : n * norm_inf_with(g, n, M, ldm, 0.0, offdiag) * B2M_NEAR_ZERO;   // :369
  int total = 0, piv = 0, ex = 0;
  // Rung 0 here, but only for B2M_LADDER_PROBE pivots: a solve that is going to succeed is
  // over long before that (profiles/: < 60 pivots at n = 40); one that is still pivoting is very likely circling towards the
  // cap, and then the whole ladder -- rung 0 included, started afresh -- goes to the task list at once instead of after 1,000 pivots.
  int probe = B2M_LADDER_PROBE;
  int st = lemke_solve(g, n, M, ldm, q, 0.0, piv_tol, zero_tol, z, C.wd, C.wi, &piv, nullptr, 0, nullptr, &probe, &ex, offdiag);
  int first_rung = 1;
  if (st == LCP_DEFER) first_rung = 0;
  else {
    total += piv;
    if (stats && g.tid == 0) { stats[0]++; stats[1] += piv; stats[2] += ex; }
    if ((st == LCP_OK || st == LCP_TRIVIAL) && lcp_verify(g, n, M, ldm, q, 0.0, z, ZERO_TOL, false, C.wd + (size_t)n * (n + 2))) {
      if (pivots_out) *pivots_out = piv;
      return st;
    }
  }
  int n_rungs = 1;
  for (int rf = min_exp; rf < max_exp && n_rungs < B2M_LADDER_MAX_RUNGS; rf += step_exp) n_rungs++;
  if (n_rungs == 1 && first_rung == 1) { if (pivots_out) *pivots_out = total; for (int i = g.tid; i < n; i += G::size) z[i] = 0.0; g.sync(); return LCP_UNVERIFIED; }
  // the job: wait until no task of this owner's previous request is running, then publish (M, q) and the rungs
  int* mo = L.meta + (size_t)C.owner * L.meta_stride;
  double* job = L.jobs + (size_t)C.owner * L.job_stride;
  double* jd = L.jobd + (size_t)C.owner * 4;
  int gen = 0;
  g.sync();
  if (g.tid == 0) {
    while (((volatile int*)mo)[LJ_INFLIGHT] != 0) __nanosleep(100);
    gen = mo[LJ_GEN] + 1;
    mo[LJ_POST] = b2m_now_us();
    mo[LJ_CANCEL] = 0; mo[LJ_N] = n; mo[LJ_NRUNGS] = n_rungs; mo[LJ_MINEXP] = min_exp; mo[LJ_STEPEXP] = step_exp;
    jd[0] = piv_tol; jd[1] = zero_tol; jd[2] = ZERO_TOL; jd[3] = offdiag;
    for (int k = first_rung; k < n_rungs; k++) mo[LJ_HDR + LJ_RW * k] = 0;
  }
  g.sync();
  for (int e = g.tid; e < n * n; e += G::size) { const int c = e / n, r = e - c * n; job[e] = M[(size_t)c * ldm + r]; }
  for (int i = g.tid; i < n; i += G::size) job[(size_t)L.nmax * L.nmax + i] = q[i];
  __threadfence();
  g.sync();
  int posted = 0;
  if (g.tid == 0) {
    ((volatile int*)mo)[LJ_GEN] = gen;
    __threadfence();
    const int cnt = n_rungs - first_rung;
    if (((volatile int*)L.ctl)[0] + cnt <= L.cap) {
      const int base = atomicAdd(L.ctl, cnt);
      if (base + cnt <= L.cap) {
        posted = 1;
        for (int k = first_rung; k < n_rungs; k++) { const int idx = base + k - first_rung; L.task_gen[idx] = gen; __threadfence(); ((volatile int*)L.tasks)[idx] = ((C.owner + 1) << 6) | k; }
      } else {                                            // the list filled up in between: publish skip entries so that takers do not wait on them
        for (int k = first_rung; k < n_rungs; k++) { const int idx = base + k - first_rung; if (idx < L.cap) { L.task_gen[idx] = -1; __threadfence(); ((volatile int*)L.tasks)[idx] = ((C.owner + 1) << 6) | k; } }
      }
    }
  }
  posted = g.bcast(posted);
  int result = LCP_UNVERIFIED;
  if (!posted) {                                          // task list full: the remaining rungs one after the other, as the generic wrapper does
    if (first_rung == 0) {
      g.sync();
      st = lemke_solve(g, n, M, ldm, q, 0.0, piv_tol, zero_tol, z, C.wd, C.wi, &piv, nullptr, 0, nullptr, nullptr, &ex, offdiag);
      total += piv;
      if (stats && g.tid == 0) { stats[0]++; stats[1] += piv; stats[2] += ex; }
      if ((st == LCP_OK || st == LCP_TRIVIAL) && lcp_verify(g, n, M, ldm, q, 0.0, z, ZERO_TOL, false, C.wd + (size_t)n * (n + 2))) { if (pivots_out) *pivots_out = piv; return st; }
    }
    int attempt = 0;
    for (int rf = min_exp; rf < max_exp && result == LCP_UNVERIFIED; rf += step_exp, attempt++) {
      const double lambda = pow10i(rf);
      g.sync();
      st = lemke_solve(g, n, M, ldm, q, lambda, piv_tol, zero_tol, z, C.wd, C.wi, &piv, nullptr, 0, nullptr, nullptr, &ex, offdiag);
      total += piv;
      if (stats && g.tid == 0) { stats[0]++; stats[1] += piv; stats[2] += ex; }
      if ((st == LCP_OK || st == LCP_TRIVIAL) && lcp_verify(g, n, M, ldm, q, lambda, z, ZERO_TOL, true, C.wd + (size_t)n * (n + 2))) result = LCP_REGULARIZED + attempt;
    }
  }
  for (int k = first_rung; posted && k < n_rungs; k++) {
    volatile int* r = mo + LJ_HDR + LJ_RW * k;
    for (;;) {
      int ready = 0;
      if (g.tid == 0) ready = r[0];
      ready = g.bcast(ready);
      if (ready == 1) break;
      if (ready == 2 || !ladder_help_one(g, L, C.wd, C.wi)) __nanosleep(200);      // somebody is on it: wait; not taken yet: take tasks (maybe this one)
    }
    __threadfence();
    const int pk = r[3], ek = r[4], okk = r[2];
    if (C.dbg && g.tid == 0) {                            // timeline taps: worst pick-up delay and run time of the rungs consumed, how many
      const int post = mo[LJ_POST], pick = r[5] - post, run = r[6] - r[5];
      if (pick > C.dbg[0]) C.dbg[0] = pick;
      if (run > C.dbg[1]) C.dbg[1] = run;
      C.dbg[2]++;
      if (pk >= 1000) C.dbg[3]++;
    }
    total += pk;
    if (stats && g.tid == 0) { stats[0]++; stats[1] += pk; stats[2] += ek; }
    if (okk) {
      const double* zr = job + (size_t)L.nmax * L.nmax + L.nmax + (size_t)k * L.nmax;
      for (int i = g.tid; i < n; i += G::size) z[i] = ((const volatile double*)zr)[i];
      result = (k == 0) ? r[1] : LCP_REGULARIZED + (k - 1);
      if (k == 0) total = pk;                           // the wrapper reports the first solve's own count when it is accepted (:252-255)
      break;
    }
  }
  g.sync();
  if (g.tid == 0) { ((volatile int*)mo)[LJ_CANCEL] = 1; __threadfence(); }
  if (pivots_out) *pivots_out = total;
  if (result == LCP_UNVERIFIED) { for (int i = g.tid; i < n; i += G::size) z[i] = 0.0; }
  g.sync();
  return result;
}
#endif

}  // namespace b2m
