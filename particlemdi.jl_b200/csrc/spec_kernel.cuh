// The conditional-SMC sweep over the copy-on-write cluster pool with the evaluations run ONE
// OBSERVATION AHEAD of the proposals: one grid barrier per observation step instead of two.
//
// What the reference does per observation t (src/pmdi.jl:209-342): evaluate every distinct cluster
// against x[t] (:218-220), every particle draws a label for every dataset (:223-265), the chosen
// clusters get x[t] added - in place when all referring particles chose it, as a copy otherwise
// (:275-310) - and the weights decide on a resampling (:317-341).  The evaluation of x[t+1] has
// to wait for the adds of x[t], which wait for the draws of step t: a chain of dependent phases.
//
// Here the add does not wait for the draws.  For every live row v the pool keeps a CHILD row
// c(v): while the particles draw their labels for x[t], the evaluation side writes
// c(v) = v + x[t] for EVERY live row and evaluates both v and c(v) against x[t+1].  A particle that
// chooses v simply points its label at c(v) - whether the reference would have added in place or
// split does not matter to it - and after the step's barrier the evaluation side reads how many
// chose v: nobody (c(v) is recycled), everybody (v is recycled: "in place"), or some (both live:
// the split).  Either way the predictive of every possible survivor for x[t+1] is already there,
// so the next proposals start right after the barrier.
//
// The grid is split by role: P-CTAs own the particle slots (proposals, weights), E-CTAs evaluate
// rows.  Every E-CTA keeps the complete list of live rows and replays the (cheap) bookkeeping of a
// step's outcome for all of them, in the same order, so that all E-CTAs hold the same list without
// talking to each other; the expensive part - the row evaluations - is dealt out task j -> E-CTA
// j mod (number of E-CTAs), and only the CTA that owns an entry performs its side effects.  Each
// role's per-step code is small - the sweep is a chain of `steps` dependent grid phases and is bound
// by latency, instruction fetch included.
//
// Per phase A(t), t = 0..steps-1:
//   P-CTAs  decide(t-1): calc_ESS of step t-1 (src/misc.jl:15-25, :317) by one warp while the others
//           already compute their proposals for x[t] (read-only: gather lp through the row map,
//           softmax-cdf, draw); the proposals are committed (choice counted, label -> child row,
//           weight folded with the Phi coupling, src/misc.jl:50-59) once the decision is known;
//           on a resampling the CTA drops the computed proposals, resamples, recomputes.
//   E-CTAs  fix(t-1): outcome of step t-1 for their rows; then for every surviving row v:
//           c(v) = v + x[t], lp(v, x[t+1]), lp(c(v), x[t+1]), and the ids of the next children.
//   -- B(t) --
// Same results as the two-barrier engine and as the dense form: a row's content and predictive
// do not depend on who computes it or when.
//
// The pool's block operators come from pool_types.cuh; the observation ring, the resampling plan, the trace and the
// cross-rank barrier from sweep_common.cuh; the finish kernels from aux_kernels.cuh.  With PMDI_SPEC_GROUP defined
// this header compiles the group kernels and nothing else (spec_group.cu).
#pragma once
#include "pool_types.cuh"
#include "sweep_common.cuh"

#define SPEC_FC 256      // free-row ids per dataset cached by an E-CTA (shared memory)
#define SPEC_EC 512      // entries of the live-row list kept in shared memory (the rest spills to HBM)
#ifdef PMDI_X_GLOBAL
#define SPEC_RB 512      // blocks of a row whose partials meet in shared memory: 65,536 features in 128-feature blocks
#else
#define SPEC_RB 64       // ... 8,192 features (a wider dataset runs the wide kernels)
#endif

struct SpecSmem {
  unsigned long long obs_bar[PMDI_OBS_RING];
  unsigned long long epoch, xepoch;
  double res_mx;
  double red[2][2][SPEC_RB];
  int res_flag;
  int fail;
  int ev;
  int pdone;
  int lpar;                    // E-CTA: which copy of the entry list is current
  int cnt;                     // E-CTA: entries of the live-row list (all datasets)
  int wsum[PMDI_NW];           // E-CTA: per-warp survivor counts of the running fix
  int b_tt[PMDI_MAX_K], b_c[PMDI_MAX_K], b_cc[PMDI_MAX_K], b_next[PMDI_MAX_K];  // E-CTA: the empty clusters' children
  int kc[PMDI_MAX_K];          // E-CTA 0: entries per dataset
  unsigned kadd[PMDI_MAX_K];   // E-CTA 0: clusters that were chosen (the reference's cluster_add! calls)
  unsigned rows_eval[PMDI_MAX_K], rows_ref[PMDI_MAX_K], rows_spec[PMDI_MAX_K];
  unsigned long long tacc[8];
  int tr_n[PMDI_NW];
};

struct SpecTables {
  // P-CTAs
  double* lf;      // [lf_T]
  double* lp_s;    // [NW][Npad]
  int* ch_s;       // [NW][Npad] child ids of the labels' rows
  double* Pi_s;    // [K][N]
  double* lw_s;    // [MS]
  double* inc_s;   // [MU]
  int* lab_s;      // [MU]
  int* pcount;     // [MS]
  int* u_c;        // [MU] row chosen
  int* u_child;    // [MU] its child
  int* u_occ;      // [MU] occupied labels of the unit
  int* u_c1;       // [MU] row chosen one step ago
  int* u_c2;       // [MU] row chosen two steps ago (its choice counter is cleared now)
  int* u_prow;     // [MU] the row the chosen label pointed at before this step's commit (undo)
  double* lw_prev; // [MS] the particles' log-weights before this step's commit (undo)
  int* u_ks;       // [MU] dataset | local slot << 8
  int* rm_s;       // [MU][N]
  // E-CTAs
  int4* el_s;      // [2][SPEC_EC] entries (dataset << 28 | row, child, cluster size, -) of the live-row list
  int* fc_s;       // [K][SPEC_FC] free ids per dataset
  int* fc_top;     // [K]
};

// bounds checks of the instrumented kernel instantiation (every debug-capture sweep of the parity tests runs them):
// a row id outside its pool, a list longer than its storage or an id handed out twice ends the sweep with error 90+
#define SCHECK(cond_, code_) if constexpr (DBG) { if (!(cond_)) { atomicExch(sp.err, (code_)); sm.fail = 1; } }

// grid barrier over this GPU's CTAs (both roles), all threads
__device__ __noinline__ bool spec_gsync(const SweepParams& sp, SpecSmem& sm, bool sys = false) {
  __syncthreads();
  if (threadIdx.x == 0) {
    sm.epoch += (unsigned long long)sp.G;
    if (sys) __threadfence_system(); else __threadfence();
    atomicAdd((unsigned long long*)sp.bar, 1ull);
    if (ld_acquire_u64((const unsigned long long*)sp.bar) < sm.epoch) {
      const unsigned long long t0 = globaltimer_ns();
      unsigned spins = 0;
      while (ld_acquire_u64((const unsigned long long*)sp.bar) < sm.epoch) {
        if (((++spins) & 0x3ffu) == 0) {
          if (__ldcg(sp.err) != 0) { sm.fail = 1; break; }
          if (globaltimer_ns() - t0 > sp.wd_ns) { atomicExch(sp.err, 77); sm.fail = 1; break; }
        }
      }
    }
  }
  __syncthreads();
  return sm.fail == 0;
}

// barrier over the CTAs of ALL ranks (sweep_xsync)
__device__ __noinline__ bool spec_xsync(const SweepParams& sp, SpecSmem& sm) {
  return sweep_xsync(sp, sm, [&](bool sys) { return spec_gsync(sp, sm, sys); });
}

// This CTA's index within its context's grid.  A group launch (k_sweep_spec_group) runs the grids of several contexts
// side by side in one cooperative grid; its prologue leaves each CTA's index within its own context's grid here.
// (The trace and spec_xsync still read blockIdx.x: a group has no trace and no sharded member.)
static __shared__ int spec_group_cta;
template <bool GRP>
__device__ __forceinline__ int spec_cta() {
  if constexpr (GRP) return spec_group_cta;
  else return (int)blockIdx.x;
}

__device__ __forceinline__ int4 ldcg_info(const RowInfo* p) { return __ldcg((const int4*)p); }
__device__ __forceinline__ double info_lp(const int4& v) { return __hiloint2double(v.y, v.x); }

// ------------------------------------------------------------------------------------------------
// P side
// ------------------------------------------------------------------------------------------------
// Proposal of one unit, read-only part (src/pmdi.jl:223-262): label, chosen row, its child, the
// incremental weight - left in the unit tables.  One warp.
template <bool DBG, bool GRP>
__device__ __noinline__ void spec_propose(const SweepParams& sp, SpecSmem& sm, const SpecTables& T, int u, int step) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int K = sp.K, N = sp.N, P = sp.P, par = step & 1;
  const int ks = T.u_ks[u];
  const int k = ks & 0xff, sl = ks >> 8;
  const PoolDev& pd = sp.pd[k];
  const int p = sp.slot0 + spec_cta<GRP>() + sl * sp.GP;  // logical particle
  const int Npad = (N + 31) & ~31;
  double* lps = T.lp_s + warp * Npad;
  int* chs = T.ch_s + warp * Npad;
  const int* rm = T.rm_s + u * N;
  const int empty = pd.cap - 1;
  const RowInfo* info = pd.info + (size_t)par * pd.cap;
  SWEEP_TRACE(step, 42)
  double mx = -INFINITY;
  int occ = 0;
#pragma unroll 1
  for (int m0 = 0; m0 < N; m0 += 64) {  // two labels per lane go out together
    const int ma = m0 + lane, mb = ma + 32;
    const int ra = ma < N ? rm[ma] : empty, rb = mb < N ? rm[mb] : empty;
    const int4 ia = ldcg_info(info + ra), ib = ldcg_info(info + rb);
    if (ma < N) {
      const double a = info_lp(ia);
      lps[ma] = a; chs[ma] = ia.z;
      mx = fmax(mx, a);
      if (DBG && sp.dbg_lp) sp.dbg_lp[(((size_t)step * K + k) * P + p) * N + ma] = a;
    }
    if (mb < N) {
      const double b = info_lp(ib);
      lps[mb] = b; chs[mb] = ib.z;
      mx = fmax(mx, b);
      if (DBG && sp.dbg_lp) sp.dbg_lp[(((size_t)step * K + k) * P + p) * N + mb] = b;
    }
    occ += __popc(__ballot_sync(FULL, ra != empty)) + __popc(__ballot_sync(FULL, rb != empty));
  }
  double uu = 0.0;
  if (p != 0) uu = sp.tape_alloc ? __ldg(sp.tape_alloc + ((size_t)step * K + k) * P + p)
                                 : pm_uniform(sp.seed, sp.iter, DRAW_ALLOC, step, k, p);
  mx = warp_max(mx);
  __syncwarp();
  SWEEP_TRACE(step, 43)
  // f = exp(lp - max) * Pi ; sequential cumsum over labels (src/pmdi.jl:236-241)
#pragma unroll 1
  for (int m = lane; m < N; m += 32) lps[m] = pm_exp(lps[m] - mx) * T.Pi_s[k * N + m];
  __syncwarp();
  SWEEP_TRACE(step, 44)
  if (lane == 0) {
    double run = 0.0;
    int m = 0;
#pragma unroll 1
    for (; m + 4 <= N; m += 4) {  // loads ahead of the dependent adds
      const double v0 = lps[m], v1 = lps[m + 1], v2 = lps[m + 2], v3 = lps[m + 3];
      run += v0; lps[m] = run;
      run += v1; lps[m + 1] = run;
      run += v2; lps[m + 2] = run;
      run += v3; lps[m + 3] = run;
    }
#pragma unroll 1
    for (; m < N; ++m) { run += lps[m]; lps[m] = run; }
  }
  __syncwarp();
  SWEEP_TRACE(step, 45)
  const double tot = lps[N - 1];
  int label;
  if (p == 0) {
    label = (int)sp.s_in[(size_t)k * sp.n_obs + sp.order[sp.n1 - 1 + step]] - 1;  // reference trajectory (:262)
  } else {
    label = N - 1;
#pragma unroll 1
    for (int m0 = 0; m0 < N - 1; m0 += 32) {
      const int m = m0 + lane;
      const bool hit = (m < N - 1) && (pm_div(lps[m < N ? m : 0], tot) > uu);  // strict '>' (:255)
      const unsigned bb = __ballot_sync(FULL, hit);
      if (bb) { label = m0 + __ffs(bb) - 1; break; }
    }
  }
  SWEEP_TRACE(step, 46)
  const double inc = pm_log(tot) + mx;
  if (lane == 0) {
    T.u_c[u] = rm[label]; T.u_child[u] = chs[label]; T.u_occ[u] = occ;
    T.inc_s[u] = inc; T.lab_s[u] = label;
  }
  __syncwarp();
  SWEEP_TRACE(step, 47)
}

// Commit of one unit's proposal: the choice is counted, the label points at the child row, the
// K-th commit of a particle folds its log-weight.  One warp (lane 0 works).
template <bool DBG, bool GRP>
__device__ __noinline__ void spec_commit(const SweepParams& sp, SpecSmem& sm, const SpecTables& T, int u, int step, int ns) {
  const int lane = threadIdx.x & 31;
  const int K = sp.K, N = sp.N, P = sp.P;
  const int ks = T.u_ks[u];
  const int k = ks & 0xff, sl = ks >> 8;
  const PoolDev& pd = sp.pd[k];
  const int slot = spec_cta<GRP>() + sl * sp.GP, p = sp.slot0 + slot;
  const int b3 = step % 3, z3 = (step + 1) % 3;  // choice counters: [3][cap], this step's and the next step's
  if (lane == 0) {
    const int c = T.u_c[u], label = T.lab_s[u], child = T.u_child[u];
    atomicAdd(pd.chosen + (size_t)b3 * pd.cap + c, 1);  // result unused: fire and forget
    // the counter this unit raised two steps ago has been read by every E-CTA: clear it for the next step
    const int c2 = T.u_c2[u];
    if (c2 >= 0) __stcg(pd.chosen + (size_t)z3 * pd.cap + c2, 0);
    T.u_c2[u] = T.u_c1[u]; T.u_c1[u] = c;
    T.u_prow[u] = c;
    T.rm_s[u * N + label] = child;
    __stcg(pd.rowmap + ((size_t)(sm.ev & 1) * sp.Ps + slot) * N + label, child);
#pragma unroll 1
    for (int r = 0; r < sp.R; ++r)  // every rank back-traces the selected particle's lineage itself
      *on_rank(sp, sp.alloc_log + ((size_t)step * K + k) * P + p, r) = (uint8_t)label;
    if (DBG && sp.dbg_alloc) sp.dbg_alloc[((size_t)step * K + k) * P + p] = label + 1;
    atomicAdd(&sm.rows_ref[k], (unsigned)T.u_occ[u]);
    __threadfence_block();
    if (atomicAdd(&T.pcount[sl], 1) == K - 1) {
      __threadfence_block();
      T.pcount[sl] = 0;
      const volatile double* iv = T.inc_s + (size_t)sl * K;
      const volatile int* lv = T.lab_s + (size_t)sl * K;
      double w = T.lw_s[sl];
      T.lw_prev[sl] = w;
#pragma unroll 1
      for (int kk = 0; kk < K; ++kk) w += iv[kk];  // dataset order, as src/pmdi.jl:210,233
      int idx = 0;
#pragma unroll 1
      for (int k1 = 0; k1 < K - 1; ++k1)
#pragma unroll 1
        for (int k2 = k1 + 1; k2 < K; ++k2) {  // Phi_upweight! (src/misc.jl:50-59)
          w += (lv[k1] == lv[k2]) ? sp.l1phi[idx] : 0.0;
          ++idx;
        }
      T.lw_s[sl] = w;
      __stcg(sp.lw + (size_t)(step & 1) * P + p, w);  // two copies by step parity: the decision on step t is taken
                                                      // while step t+1 is already being committed
      if (DBG && sp.dbg_lw) sp.dbg_lw[(size_t)step * P + p] = w;
    }
  }
  SWEEP_TRACE(step, 48)
}

// calc_ESS of step t (src/misc.jl:15-25, src/pmdi.jl:317) straight from the particles' log-weights (every
// commit of step t stored its particle's before the barrier), by the one CTA that has nothing else to do
// (the last of the grid): warp w takes the w-th sixteenth of the particles, eight loads per lane in flight,
// the sixteen partials are combined in a fixed order.  The decision goes to dec[t]; the other CTAs read it
// when they need it - the proposals only at their commit, the evaluation CTAs before the barrier.
__device__ __noinline__ void spec_decide(const SweepParams& sp, SpecSmem& sm, int t) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, P = sp.P;
  // (with several ranks: this rank's particles; the ranks' partials are exchanged below)
  const int per = (sp.Ps + PMDI_NW - 1) / PMDI_NW, p_lo = sp.slot0 + warp * per, p_hi = min(sp.slot0 + sp.Ps, p_lo + per);
  const double* lw = sp.lw + (size_t)(t & 1) * P;
  double mxv = -INFINITY;
#pragma unroll 1
  for (int p0 = p_lo; p0 < p_hi; p0 += 256) {
    double v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int p = p0 + lane + 32 * i;
      v[i] = p < p_hi ? ldcg_f64(lw + p) : -INFINITY;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) mxv = fmax(mxv, v[i]);
  }
  mxv = warp_max(mxv);
  double num = 0.0, den = 0.0;
#pragma unroll 1
  for (int p0 = p_lo; p0 < p_hi; p0 += 256) {
    double v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int p = p0 + lane + 32 * i;
      v[i] = p < p_hi ? ldcg_f64(lw + p) : -INFINITY;
    }
#pragma unroll 1
    for (int i = 0; i < 8; ++i) {
      if (p0 + lane + 32 * i < p_hi) {
        const double e = pm_exp(v[i] - mxv);
        num += e;
        den += e * e;
      }
    }
  }
  num = warp_sum(num);
  den = warp_sum(den);
  if (lane == 0) { sm.red[0][0][warp] = mxv; sm.red[0][0][16 + warp] = num; sm.red[0][0][32 + warp] = den; }
  __syncthreads();
  if (warp == 0) {
    const double m = lane < PMDI_NW ? sm.red[0][0][lane] : -INFINITY;
    double mx = warp_max(m);
    double a = 0.0, b = 0.0;
    if (lane < PMDI_NW && m > -INFINITY) {
      const double e = pm_exp(m - mx);
      a = sm.red[0][0][16 + lane] * e;
      b = sm.red[0][0][32 + lane] * (e * e);
    }
    a = warp_sum(a);
    b = warp_sum(b);
    double gmx = mx;
    if (sp.R > 1) {
      // One (max, sum w, sum w^2) per rank goes to every rank as six 8-byte words (step tag << 32 | half of a
      // double): each word validates itself, so the stores need no fence and no ordering - one NVLink one-way
      // trip instead of a round trip (the fence) plus a trip (the tag).  Slots by step parity: a peer cannot
      // be two steps ahead, it needs this rank's partial of step t+1 first.
      const int par = t & 1;
      const unsigned tag = sp.tag32 + (unsigned)(t + 1);
      unsigned long long* words = sp.rank_words + (size_t)par * sp.R * 8;
      if (lane < 6) {
        const double val = (lane >> 1) == 0 ? mx : (lane >> 1) == 1 ? a : b;
        const unsigned half = (lane & 1) ? (unsigned)__double2hiint(val) : (unsigned)__double2loint(val);
        const unsigned long long word = ((unsigned long long)tag << 32) | half;
#pragma unroll 1
        for (int r = 0; r < sp.R; ++r)
          asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(on_rank(sp, words + (size_t)sp.rank * 8 + lane, r)), "l"(word) : "memory");
      }
      unsigned* hw = (unsigned*)&sm.red[1][0][0];  // the halves as they arrive: [rank][6]
#pragma unroll 1
      for (int idx = lane; idx < 6 * sp.R; idx += 32) {
        const unsigned long long* f = words + (size_t)(idx / 6) * 8 + (idx % 6);
        const unsigned long long t0 = globaltimer_ns();
        unsigned spins = 0;
        unsigned long long w;
        while ((unsigned)((w = *(volatile const unsigned long long*)f) >> 32) != tag) {
          if (((++spins) & 0x3ffu) == 0 && (__ldcg(sp.err) != 0 || globaltimer_ns() - t0 > sp.wd_ns)) { atomicExch(sp.err, 77); break; }
        }
        hw[idx] = (unsigned)w;
      }
      __syncwarp();
      const double rm = lane < sp.R ? __hiloint2double((int)hw[lane * 6 + 1], (int)hw[lane * 6]) : -INFINITY;
      gmx = warp_max(rm);
      double ra = 0.0, rb = 0.0;
      if (lane < sp.R && rm > -INFINITY) {
        const double e = pm_exp(rm - gmx);
        ra = __hiloint2double((int)hw[lane * 6 + 3], (int)hw[lane * 6 + 2]) * e;
        rb = __hiloint2double((int)hw[lane * 6 + 5], (int)hw[lane * 6 + 4]) * (e * e);
      }
      a = warp_sum(ra);
      b = warp_sum(rb);
    }
    if (lane == 0) {
      const int res = (a * a) / b <= 0.5 * (double)P ? 1 : 0;
      mx = gmx;
      sm.res_mx = mx;
      sm.res_flag = res;
      if (!res) sp.ev_of_step[t] = -1;
      __stcg(sp.dec + t, res ? 2 : 1);
    }
  }
  __syncthreads();
}

// every other CTA: the decision of step t, once the D-CTA has published it (one thread polls)
__device__ __noinline__ bool spec_wait_decision(const SweepParams& sp, SpecSmem& sm, int t) {
  if (threadIdx.x == 0) {
    int d;
    const unsigned long long t0 = globaltimer_ns();
    unsigned spins = 0;
    while ((d = *(volatile unsigned char*)(sp.dec + t)) == 0) {
      if (((++spins) & 0x3ffu) == 0 && (__ldcg(sp.err) != 0 || globaltimer_ns() - t0 > sp.wd_ns)) { sm.fail = 1; break; }
    }
    sm.res_flag = d == 2;
  }
  __syncthreads();
  if (sm.fail) { atomicExch(sp.err, 77); return false; }
  return true;
}

// (re)load the owned units' row maps into shared memory.  All threads of a P-CTA.
template <bool GRP>
__device__ __noinline__ void spec_load_units(const SweepParams& sp, SpecSmem& sm, const SpecTables& T, int ns) {
  const int K = sp.K, N = sp.N, nu = ns * K;
#pragma unroll 1
  for (int i = threadIdx.x; i < nu * N; i += PMDI_NT) {
    const int u = i / N, m = i - u * N;
    const int k = u % K, slot = spec_cta<GRP>() + (u / K) * sp.GP;
    T.rm_s[i] = ldcg_i32(sp.pd[k].rowmap + ((size_t)(sm.ev & 1) * sp.Ps + slot) * N + m);
  }
#pragma unroll 1
  for (int u = threadIdx.x; u < nu; u += PMDI_NT) { T.u_c1[u] = -1; T.u_c2[u] = -1; }  // all choice counters are clear
}

// ------------------------------------------------------------------------------------------------
// E side
// ------------------------------------------------------------------------------------------------
// The live-row list: entries (dataset << 28 | row, child, cluster size of the row, -).  Every E-CTA
// has its own two copies (a fix reads one and writes the other): the first SPEC_EC entries in shared
// memory, the rest in HBM.
#define SPEC_KSHIFT 28
#define SPEC_VMASK ((1 << SPEC_KSHIFT) - 1)
__device__ __forceinline__ int4* spec_spill(const SweepParams& sp, int e, int lp) {
  return sp.elist + ((size_t)lp * (sp.G - sp.GP - 1) + e) * sp.lcap;
}
__device__ __forceinline__ int4 spec_entry(const SweepParams& sp, const SpecTables& T, int e, int lp, int i) {
  if (i < SPEC_EC) return T.el_s[lp * SPEC_EC + i];
  return __ldcg(spec_spill(sp, e, lp) + i);
}
__device__ __forceinline__ void spec_set_entry(const SweepParams& sp, const SpecTables& T, int e, int lp, int i, int4 v) {
  if (i < SPEC_EC) T.el_s[lp * SPEC_EC + i] = v;
  else __stcg(spec_spill(sp, e, lp) + i, v);
}
// Global free stack of a dataset (freelist[], ctr[1] = height): an empty slot holds -1.  Push and pop
// claim a slot through the counter and hand the id over through the slot itself, so a push and a pop
// that meet on a slot cannot lose or duplicate an id.  Rare paths: the CTAs work from their caches.
__device__ __noinline__ void spec_gpush(const PoolDev& pd, int id) {
  const int s = atomicAdd(pd.ctr + 1, 1);
  while (atomicCAS(pd.freelist + s, -1, id) != -1) {}
}
__device__ __noinline__ int spec_gclaim(const PoolDev& pd, int want) {  // first of `want` claimed slots, -1: not enough
  int cur = ldcg_i32(pd.ctr + 1);
  while (cur >= want) {
    const int seen = atomicCAS(pd.ctr + 1, cur, cur - want);
    if (seen == cur) return cur - want;
    cur = seen;
  }
  return -1;
}
__device__ __forceinline__ int spec_gtake(const PoolDev& pd, int slot) {
  int id;
  while ((id = atomicExch(pd.freelist + slot, -1)) == -1) {}
  return id;
}
__device__ __forceinline__ void spec_free_id(const SweepParams& sp, const SpecTables& T, int k, int id) {
  const int t = atomicAdd(&T.fc_top[k], 1);
  if (t < SPEC_FC) T.fc_s[k * SPEC_FC + t] = id;
  else { atomicSub(&T.fc_top[k], 1); spec_gpush(sp.pd[k], id); }  // cache full
}
// a free row id of dataset k: from the CTA's cache, else off the global stack
__device__ __forceinline__ int spec_pop_id(const SweepParams& sp, SpecSmem& sm, const SpecTables& T, int k) {
  const int t = atomicSub(&T.fc_top[k], 1) - 1;
  if (t >= 0) return T.fc_s[k * SPEC_FC + t];
  atomicAdd(&T.fc_top[k], 1);
  const int slot = spec_gclaim(sp.pd[k], 1);
  if (slot < 0) { atomicExch(sp.err, 80); sm.fail = 1; return 0; }
  return spec_gtake(sp.pd[k], slot);
}
// keep the caches around their target height (thread k < K), off the step's dependent chain: the CTA that
// owns an entry frees its ids, the CTA that runs a task takes ids - the two drift apart
__device__ __forceinline__ void spec_refill(const SweepParams& sp, SpecSmem& sm, const SpecTables& T) {
  const int k = threadIdx.x >> 5, lane = threadIdx.x & 31;  // warp k: dataset k, a lane per id (one atomic round trip each)
  if (k >= sp.K) return;
  const PoolDev& pd = sp.pd[k];
  const int top = T.fc_top[k], tgt = sp.fc_target;
  __syncwarp();
  if (top < tgt / 2) {
    const int want = tgt - top;
    int first = lane == 0 ? spec_gclaim(pd, want) : 0;
    first = __shfl_sync(FULL, first, 0);
    if (first < 0) return;  // nearly dry: spec_pop_id reports a real exhaustion
#pragma unroll 1
    for (int i = lane; i < want; i += 32) T.fc_s[k * SPEC_FC + top + i] = spec_gtake(pd, first + i);
    __syncwarp();
    if (lane == 0) T.fc_top[k] = top + want;
  } else if (top > SPEC_FC - 32 || top > 2 * tgt + 16) {
    const int keep = min(SPEC_FC / 2, tgt + 8);
#pragma unroll 1
    for (int i = keep + lane; i < top; i += 32) spec_gpush(pd, T.fc_s[k * SPEC_FC + i]);
    __syncwarp();
    if (lane == 0) T.fc_top[k] = keep;
  }
}

// The empty clusters (one per dataset) are not in the list.  Thread k < K: the child handed out for
// the step with parity `par` (the row that will hold the singleton cluster of that step's observation).
__device__ __forceinline__ void spec_load_empty_next(const SweepParams& sp, SpecSmem& sm, int par) {
  const int k = threadIdx.x;
  if (k < sp.K) sm.b_next[k] = ldcg_info(sp.pd[k].info + (size_t)par * sp.pd[k].cap + sp.pd[k].cap - 1).z;
}

// First step only: the children handed out by E'(0) are known to the CTAs that ran the tasks; every
// CTA reads them back into its copy of the list.  All threads.
__device__ __noinline__ void spec_refresh_children(const SweepParams& sp, SpecSmem& sm, const SpecTables& T, int e) {
  const int lp = sm.lpar;
#pragma unroll 1
  for (int i = threadIdx.x; i < sm.cnt; i += PMDI_NT) {
    int4 en = spec_entry(sp, T, e, lp, i);
    const int k = (unsigned)en.x >> SPEC_KSHIFT, v = en.x & SPEC_VMASK;
    en.y = ldcg_info(sp.pd[k].info + v).z;
    spec_set_entry(sp, T, e, lp, i, en);
  }
  spec_load_empty_next(sp, sm, 0);
  __syncthreads();
}

// Outcome of step t1 (src/pmdi.jl:275-310), replayed by EVERY E-CTA for the whole list, in list
// order: the entry (v, c) becomes (v, c'(v)) when nobody chose v, (c, c'(c)) when every reference did
// ("in place"), or both (the split); a dataset's empty cluster gives birth to its child when somebody
// chose an empty label.  Only the CTA that owns an entry (index mod number of E-CTAs) writes: the
// survivors' reference counts (into the other copy: the current one is still being read by the other
// CTAs) and the row ids that fall free.
template <bool DBG>
__device__ __noinline__ void spec_fix(const SweepParams& sp, SpecSmem& sm, const SpecTables& T, int e, int t1) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int K = sp.K, GE = sp.G - sp.GP - 1;
  const int par1 = t1 & 1, parn = par1 ^ 1, b3 = t1 % 3;
  const int lo = sm.lpar, ln = lo ^ 1, n_old = sm.cnt;
  if (tid < K) {  // the empty clusters' children of step t1 and what they were handed for the next step
    const PoolDev& pd = sp.pd[tid];
    const int empty = pd.cap - 1;
    const int4 i1 = ldcg_info(pd.info + (size_t)par1 * pd.cap + empty);
    const int4 in = ldcg_info(pd.info + (size_t)parn * pd.cap + empty);  // .w: the id handed to the child's child
    sm.b_tt[tid] = ldcg_i32(pd.chosen + (size_t)b3 * pd.cap + empty);
    sm.b_c[tid] = i1.z;
    sm.b_next[tid] = in.z;
    sm.b_cc[tid] = in.w;
  }
  SWEEP_TRACE(t1 + 1, 60)
  int nb = 0;  // entries of the new list so far (the same in every thread)
#pragma unroll 1
  for (int base = 0; base < n_old; base += PMDI_NT) {
    const int i = base + tid;
    int ns = 0;
    int4 s0 = make_int4(0, 0, 0, 0), s1 = s0;
    if (i < n_old) {
      const int4 en = spec_entry(sp, T, e, lo, i);
      const int k = (unsigned)en.x >> SPEC_KSHIFT, v = en.x & SPEC_VMASK, c = en.y, n = en.z;
      SCHECK(k < K && v < sp.pd[k < K ? k : 0].cap - 1 && c >= 0 && c < sp.pd[k < K ? k : 0].cap - 1, 94)
      const PoolDev& pd = sp.pd[k < K ? k : 0];
      const int tot = ldcg_i32(pd.chosen + (size_t)b3 * pd.cap + v);
      const int rf = ldcg_i32(pd.refcnt + (size_t)par1 * pd.cap + v);
      const int cv = ldcg_info(pd.info + (size_t)parn * pd.cap + v).z;
      const int cc = ldcg_info(pd.info + (size_t)parn * pd.cap + c).z;
      const bool own = (i % GE) == e;
      const int kc = (k << SPEC_KSHIFT) | c;
      if (e == 0) { atomicAdd(&sm.kc[k], (tot == 0 || tot == rf) ? 1 : 2); if (tot) atomicAdd(&sm.kadd[k], 1u); }
      if (tot == 0) {  // nobody chose v
        ns = 1; s0 = make_int4(en.x, cv, n, 0);
        if (own) { __stcg(pd.refcnt + (size_t)parn * pd.cap + v, rf); spec_free_id(sp, T, k, c); spec_free_id(sp, T, k, cc); }
      } else if (tot == rf) {  // everybody did: "in place" (src/pmdi.jl:284-286)
        ns = 1; s0 = make_int4(kc, cc, n + 1, 0);
        if (own) { __stcg(pd.refcnt + (size_t)parn * pd.cap + c, tot); spec_free_id(sp, T, k, v); spec_free_id(sp, T, k, cv); }
      } else {  // some did: both live (src/pmdi.jl:288-309)
        ns = 2; s0 = make_int4(en.x, cv, n, 0); s1 = make_int4(kc, cc, n + 1, 0);
        if (own) { __stcg(pd.refcnt + (size_t)parn * pd.cap + v, rf - tot); __stcg(pd.refcnt + (size_t)parn * pd.cap + c, tot); }
      }
    }
    SWEEP_TRACE(t1 + 1, 61)
    // exclusive scan of the survivor counts over the CTA: list order is kept
    int incl = ns;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int up = __shfl_up_sync(FULL, incl, o);
      if (lane >= o) incl += up;
    }
    if (n_old <= 32) {  // the whole list is in the first warp (the usual case of a settled chain): no CTA barrier
      if (warp == 0) {
        const int pos = incl - ns;
        if (ns > 0) spec_set_entry(sp, T, e, ln, pos, s0);
        if (ns > 1) spec_set_entry(sp, T, e, ln, pos + 1, s1);
        nb = __shfl_sync(FULL, incl, 31);
      }
    } else {
      if (lane == 31) sm.wsum[warp] = incl;
      __syncthreads();
      int wpre = 0, tot_all = 0;
#pragma unroll
      for (int w = 0; w < PMDI_NW; ++w) {
        const int x = sm.wsum[w];
        if (w < warp) wpre += x;
        tot_all += x;
      }
      const int pos = nb + wpre + incl - ns;
      if (ns > 0) spec_set_entry(sp, T, e, ln, pos, s0);
      if (ns > 1) spec_set_entry(sp, T, e, ln, pos + 1, s1);
      nb += tot_all;
      __syncthreads();
    }
    SWEEP_TRACE(t1 + 1, 62)
  }
  if (n_old == 0) __syncthreads();  // b_* are complete
  else if (n_old <= 32) __syncwarp();  // ... written and read by the first warp
  // births, in dataset order; their side effects by the E-CTAs in turn
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const int tt = sm.b_tt[k], c = sm.b_c[k], cc = sm.b_cc[k];
    const bool own = tid == 0 && ((t1 + k) % GE) == e;
    if (tt > 0) {
      if (tid == 0) spec_set_entry(sp, T, e, ln, nb, make_int4((k << SPEC_KSHIFT) | c, cc, 1, 0));
      if (own) __stcg(sp.pd[k].refcnt + (size_t)parn * sp.pd[k].cap + c, tt);
      if (e == 0 && tid == 0) { sm.kc[k] += 1; sm.kadd[k] += 1u; }
      ++nb;
    } else if (own) {
      spec_free_id(sp, T, k, c); spec_free_id(sp, T, k, cc);
    }
  }
  __syncthreads();
  SCHECK((long long)nb <= sp.lcap, 93)
  if (tid == 0) { sm.cnt = nb; sm.lpar = ln; }
  __syncthreads();
}

// E'(st): this CTA's share of the tasks (task j -> E-CTA j mod GE; tasks = the list's entries, then
// the K empty clusters).  For an entry (v, c): c = v + x[st-1] (mode 2; at st == 0 nothing is added),
// lp(v, x[st]) and lp(c, x[st]) with the ids of their next children -> info[st & 1].  rpc tasks at a
// time, a row's blocks over jq warps, the block partials meet in shared memory.
template <bool DBG>
__device__ __noinline__ void spec_eval(const SweepParams& sp, SpecSmem& sm, const SpecTables& T, int e, int st,
                                       unsigned char* xring, int& obs_ok, int t_dec) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int K = sp.K, par = st & 1, GE = sp.G - sp.GP - 1;
  const int jq = sp.jq, rpc = PMDI_NW / jq;
  const int sub = warp / jq, wj = warp - sub * jq;
  const int n_list = sm.cnt, total = n_list + K, lp = sm.lpar;
#ifdef PMDI_X_GLOBAL  // x[st] and x[st-1] are read from global memory: their observations
  const int oc = sp.order[sp.n1 - 1 + st], op = st > 0 ? sp.order[sp.n1 - 2 + st] : oc;
#else
  const unsigned xc = (unsigned)__cvta_generic_to_shared(xring + (size_t)(st % sp.obs_ring) * sp.sm_x_bytes);
  const unsigned xp = (unsigned)__cvta_generic_to_shared(xring + (size_t)((st + sp.obs_ring - 1) % sp.obs_ring) * sp.sm_x_bytes);
#endif
  const int mode = st == 0 ? 0 : 2;
  int buf = 0;
#pragma unroll 1
  for (int j0 = e; j0 < total; j0 += GE * rpc, buf ^= 1) {
    const int j = j0 + sub * GE;
    bool active = sub < rpc && j < total;
    int k = 0, v = 0, c = 0, nc = 0, id = 0;
    double rcv = 0.0;
    if (active) {
      if (j < n_list) {
        const int4 en = spec_entry(sp, T, e, lp, j);
        k = (unsigned)en.x >> SPEC_KSHIFT; v = en.x & SPEC_VMASK; c = en.y; nc = en.z;
      } else {  // the empty cluster of dataset j - n_list; its child was handed out one step ago
        k = j - n_list; v = sp.pd[k].cap - 1; c = st == 0 ? v : sm.b_next[k]; nc = 0;
      }
      const DsDev& ds = sp.ds[k];
      const PoolDev& pd = sp.pd[k];
      SCHECK(k >= 0 && k < K && v >= 0 && v < pd.cap && (mode == 0 || (c >= 0 && c < pd.cap - 1 && c != v)) && nc >= 0 && nc <= sp.n_obs, 91)
      if (sm.fail) { active = false; }
      if (active && wj < ds.J) {
#ifdef PMDI_X_GLOBAL
        const size_t xrow = (size_t)ds.Dp * PMDI_XBYTES(ds);  // this dataset's rows are an array of their own
        const unsigned char* const xc = (const unsigned char*)ds.xstage + (size_t)oc * xrow;
        const unsigned char* const xp = (const unsigned char*)ds.xstage + (size_t)op * xrow;
        const unsigned xo = 0u;
#else
        if (obs_ok < st) {  // x[st] has landed in the ring (x[st-1] was waited for one step ago)
          if (lane == 0) {
#pragma unroll 1
            for (int s = max(obs_ok + 1, st - 1); s <= st; ++s)
              while (!mbar_try_wait(&sm.obs_bar[s % sp.obs_ring], (unsigned)(s / sp.obs_ring) & 1u)) {}
          }
          __syncwarp();
          obs_ok = st;
        }
        const unsigned xo = (unsigned)ds.x_off;
#endif
        if (wj == 0 && lane < 2) rcv = __ldg(ds.rc + nc + 1 - lane);  // lane 1: the row's size constant, lane 0: its child's
        SWEEP_TRACE(st - 1, 63)
#pragma unroll 1
        for (int jb = wj; jb < ds.J; jb += jq) {
          const int q0 = jb * ds.FB;
          const int nit = min(ds.FB / PMDI_WF, (ds.Dp - q0) / PMDI_WF);
          const int fo = q0 + 2 * lane;
          double vs = 0.0, vd;
          if (ds.type == T_GAUSSIAN) {
            const long long so = (long long)v * ds.Dp + fo;
            vd = gauss_block(ds.sum + so, ds.beta + so, ds.mu + so, ds.lamn + so, (long long)(c - v) * ds.Dp,
                             ds.aux + (long long)v * ds.J + jb, ds.aux + (long long)c * ds.J + jb, ds.flag + fo, nit,
                             mode, nc, xp + xo + fo * 8u, xc + xo + fo * 8u, &vs);
          } else if (ds.type == T_NEGBINOM) {
            vd = nb_block(ds.S + (long long)v * ds.Dp + fo, (long long)(c - v) * ds.Dp, ds.aux + (long long)v * ds.J + jb,
                          ds.aux + (long long)c * ds.J + jb, nit, mode, nc, xp + xo + fo * 4u, xc + xo + fo * 4u,
                          (unsigned)__cvta_generic_to_shared(T.lf), sp.lf_T, &vs);
#ifdef PMDI_USER_TYPES
          } else if (ds.type == T_USER) {
            const unsigned eb = ds.uW < 0 ? 4u : 8u;
            const long long rw = user_row_words(ds);
            vd = user_block(ds, ds.ust + v * rw + fo, (c - v) * rw, ds.flag + fo, nit, mode, nc, xp + xo + fo * eb,
                            xc + xo + fo * eb, &vs);
#endif
          } else {
            vd = cat_block(pd.cw + ((long long)v * ds.Dp + fo) * pd.wpf, (long long)(c - v) * ds.Dp * pd.wpf, pd.wpf,
                           pd.fpw, nit, mode, xp + xo + fo * 4u, xc + xo + fo * 4u, &vs);
          }
          if (lane == 0) {
            const int ri = ds.J <= jq ? sub * jq + jb : jb;  // rows wider than 16 blocks: one row at a time
            if (mode == 0) { sm.red[buf][1][ri] = vd; sm.red[buf][0][ri] = 0.0; }  // plain: the row itself
            else { sm.red[buf][0][ri] = vd; sm.red[buf][1][ri] = vs; }
          }
        }
      }
    }
    if (active && wj == 0 && lane < 2 && (mode || lane == 1)) id = spec_pop_id(sp, sm, T, k);  // while the other warps finish
    SWEEP_TRACE(st - 1, 64)
    __syncthreads();
    SWEEP_TRACE(st - 1, 65)
    if (active && wj == 0) {  // lane 1: the row, lane 0: its child - blocks in order, the size constant first
      const DsDev& ds = sp.ds[k];
      const PoolDev& pd = sp.pd[k];
      const int r0 = ds.J <= jq ? sub * jq : 0;
      double lv = rcv;
      if (lane < 2 && (mode || lane == 1)) {
#pragma unroll 1
        for (int j0 = 0; j0 < ds.J; j0 += 16) {  // independent loads, then the sum in block order
          double pv[16];
#pragma unroll
          for (int u = 0; u < 16; ++u) pv[u] = j0 + u < ds.J ? sm.red[buf][lane][r0 + j0 + u] : 0.0;
#pragma unroll
          for (int u = 0; u < 16; ++u)
            if (j0 + u < ds.J) lv += pv[u];
        }
        SCHECK(id >= 0 && id < pd.cap - 1 && id != v && id != c, 92)
        __stcg(ds.n + id, nc + 2 - lane);
      }
      // the row of the empty cluster also carries the id handed to its child's child (read by the next fix)
      const int id_c = __shfl_sync(FULL, id, 0);
      if (lane < 2 && (mode || lane == 1)) {
        RowInfo iv; iv.lp = lv; iv.child = id; iv.pad = lane == 1 ? id_c : 0;
        *(int4*)(pd.info + (size_t)par * pd.cap + (lane == 1 ? v : c)) = *(int4*)&iv;
      }
      if (lane == 0) atomicAdd(&sm.rows_spec[k], mode ? 2u : 1u);
    }
    SWEEP_TRACE(st - 1, 66)
  }
  // the decision on the resampling after step t_dec (published by the D-CTA early in this phase) is
  // fetched by a thread that has nothing to finish; the barrier below hands it to the CTA
  if (t_dec >= 0 && threadIdx.x == 32) {
    int d;
    const unsigned long long t0 = globaltimer_ns();
    unsigned spins = 0;
#pragma unroll 1
    while ((d = *(volatile unsigned char*)(sp.dec + t_dec)) == 0) {
      if (((++spins) & 0x3ffu) == 0 && (__ldcg(sp.err) != 0 || globaltimer_ns() - t0 > sp.wd_ns)) {
        atomicCAS(sp.err, 0, 77); sm.fail = 1; break;
      }
    }
    sm.res_flag = d == 2;
  }
  __syncthreads();
}

// One warp copies a slice (1 / SPEC_PULL_PARTS of the features) of a live row of another rank's pool and of that
// row's child of the coming step into local rows; the warp of slice 0 also copies aux, the cluster sizes and the
// predictives already computed for the next two observations, and points the child links at the local ids
// handed to the copy.  (An NVLink round trip is ~2 us: a whole row per warp was 30-60 of them in a row.)
#define SPEC_PULL_PARTS 16
__device__ __noinline__ void spec_row_pull(const SweepParams& sp, int4 j0, int4 j1, int parn, int part) {
  const int k = j0.x & 0xff, ra = j0.x >> 8, rb = j0.y, v2 = j0.z, c2 = j0.w, a2 = j1.x, b2 = j1.y;
  const DsDev& ds = sp.ds[k];
  const PoolDev& pd = sp.pd[k];
  const long long sdelta = sp.peer_delta[ra];
  const int lane = threadIdx.x & 31, Dp = ds.Dp;
#define PMDI_SRC(ptr_) ((decltype(ptr_))((const char*)(ptr_) + sdelta))
  const RowInfo* rinfo = PMDI_SRC(pd.info);
  const int4 i1 = ldcg_info(rinfo + (size_t)parn * pd.cap + rb);           // step st+1: lp, child
  const int rc = i1.z;
  const int4 i2 = ldcg_info(rinfo + (size_t)(parn ^ 1) * pd.cap + rb);     // step st+2: lp of the row
  const int4 i2c = ldcg_info(rinfo + (size_t)(parn ^ 1) * pd.cap + rc);    //            lp of its child
  const int n = ldcg_i32(PMDI_SRC(ds.n) + rb);
  long long W = ds.type == T_CATEGORICAL ? (long long)Dp * pd.wpf : (long long)Dp;  // 8-byte words per array of a row
#ifdef PMDI_USER_TYPES
  if (ds.type == T_USER) W = user_row_words(ds);
#endif
  const long long per = ((W / 64 + SPEC_PULL_PARTS - 1) / SPEC_PULL_PARTS) * 64;
  const long long q_lo = part * per, q_hi = min(W, q_lo + per);
#pragma unroll 1
  for (int h = 0; h < 2; ++h) {
    const long long src = h ? rc : rb, dst = h ? c2 : v2;
    if (ds.type == T_GAUSSIAN) {
#pragma unroll 1
      for (long long q = q_lo + 2 * lane; q < q_hi; q += 64) {
        const double2 a = ldcg_f64x2(PMDI_SRC(ds.mu) + src * Dp + q), b = ldcg_f64x2(PMDI_SRC(ds.lamn) + src * Dp + q);
        const double2 c = ldcg_f64x2(PMDI_SRC(ds.sum) + src * Dp + q), d = ldcg_f64x2(PMDI_SRC(ds.beta) + src * Dp + q);
        *(double2*)(ds.mu + dst * Dp + q) = a; *(double2*)(ds.lamn + dst * Dp + q) = b;
        *(double2*)(ds.sum + dst * Dp + q) = c; *(double2*)(ds.beta + dst * Dp + q) = d;
      }
    } else if (ds.type == T_CATEGORICAL) {
#pragma unroll 1
      for (long long q = q_lo + 2 * lane; q < q_hi; q += 64)
        *(ulonglong2*)(pd.cw + dst * W + q) = ldcg_u64x2(PMDI_SRC(pd.cw) + src * W + q);
#ifdef PMDI_USER_TYPES
    } else if (ds.type == T_USER) {  // ust[row][word][feature]: one contiguous range of |uW| * Dp doubles
#pragma unroll 1
      for (long long q = q_lo + 2 * lane; q < q_hi; q += 64)
        *(double2*)(ds.ust + dst * W + q) = ldcg_f64x2(PMDI_SRC(ds.ust) + src * W + q);
#endif
    } else {
#pragma unroll 1
      for (long long q = q_lo + 2 * lane; q < q_hi; q += 64)
        *(longlong2*)(ds.S + dst * Dp + q) = ldcg_i64x2(PMDI_SRC(ds.S) + src * Dp + q);
    }
    if (part == 0) {
#pragma unroll 1
      for (int jj = lane; jj < ds.J; jj += 32) ds.aux[dst * ds.J + jj] = ldcg_f64(PMDI_SRC(ds.aux) + src * ds.J + jj);
    }
  }
#undef PMDI_SRC
  if (lane == 0 && part == 0) {
    ds.n[v2] = n; ds.n[c2] = n + 1; ds.n[a2] = n + 1; ds.n[b2] = n + 2;
    int4 w = i1; w.z = c2; w.w = 0;
    *(int4*)(pd.info + (size_t)parn * pd.cap + v2) = w;
    w = i2; w.z = a2; w.w = 0;
    *(int4*)(pd.info + (size_t)(parn ^ 1) * pd.cap + v2) = w;
    w = i2c; w.z = b2; w.w = 0;
    *(int4*)(pd.info + (size_t)(parn ^ 1) * pd.cap + c2) = w;
  }
}

// ------------------------------------------------------------------------------------------------
// Resampling after step `st` (src/pmdi.jl:318-341), all CTAs: every particle takes its ancestor's
// row map; references are recounted; rows nobody refers to any more (and that are nobody's current
// or next child) go back to the free lists; the list of live rows is rebuilt.  The children of step
// st+1 were computed before the call and stay valid: a row's content does not depend on who refers
// to it.
// With the particles sharded over several GPUs (sp.R > 1) this is the whole-pool form below: rows of
// another rank's ancestors are pulled, and every rank recounts, marks and rescans its whole pool.  On
// one GPU spec_resample (after it) does the same in proportion to the live rows.
// Only spec_resample calls this, and only with sp.R > 1: the `sp.R > 1` test below and spec_xsync's
// one-GPU branch are always taken / never taken here.  They are left as they were so that the sharded
// event runs the code it ran when it also served one GPU (no multi-GPU machine checked a rewrite).
// ------------------------------------------------------------------------------------------------
template <bool GRP>
__device__ __forceinline__ bool spec_resample_sharded(const SweepParams& sp, SpecSmem& sm, const SpecTables& T, int ns,
                                                   int st, int* s_tmp, bool is_p, int e) {
  const int K = sp.K, N = sp.N, Ps = sp.Ps;
  const int ev = sm.ev;
  const long long gt = (long long)spec_cta<GRP>() * PMDI_NT + threadIdx.x, GT = (long long)sp.G * PMDI_NT;
  const int parn = (st + 1) & 1;  // info of step st+1: lp and child ids of everything that may be live;
                                  // also the copy of the reference counts the fix of step st+1 will read
  const bool has_next = st + 1 < sp.steps;
  // sub-phase timers (instrumented runs): tacc[4] wait for all CTAs + plan, [5] row maps + pulls, [7] recount + rebuild
  const bool tm = sp.phase_ns != nullptr && threadIdx.x == 0;
  unsigned long long t_ = tm ? globaltimer_ns() : 0ull;
#define RS_MARK(i_) if (tm) { const unsigned long long n_ = globaltimer_ns(); sm.tacc[i_] += (n_ - t_) * PMDI_NW; t_ = n_; }
  // every E-CTA (of every rank) has finished E'(st+2), every commit of step st is in
  if (!spec_xsync(sp, sm)) return false;
  if (spec_cta<GRP>() == sp.G - 1) {  // the D-CTA knows the maximum; its dynamic shared memory is free for the plan
    extern __shared__ __align__(16) unsigned char plan_raw[];  // (the dynamic shared memory, from its base)
    PlanScratch sc = {sp.sc_w, sp.sc_pp, sp.sc_u, sp.sc_j, sp.sc_anc0};
    if (sp.plan_smem) {
      sc.w = (double*)plan_raw; sc.pp = sc.w + sp.P; sc.u = sc.pp + sp.P;
      sc.j = (int*)(sc.u + sp.P); sc.a0 = sc.j + sp.P;
    }
    pool_resample_plan(sp, st, ev, sm.res_mx, s_tmp, sp.lw + (size_t)(st & 1) * sp.P, sc);
  }
  if (!spec_gsync(sp, sm)) return false;
  RS_MARK(4)
  const int* anc = sp.anc_log + (size_t)ev * sp.P;
  if (gt == (long long)sp.GP * PMDI_NT && has_next)  // rows counted for step st+1 that this decision may kill
    atomicAdd((unsigned long long*)&sp.counters[4], (unsigned long long)sm.cnt);
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const PoolDev& pd = sp.pd[k];
    const int* rm_old = pd.rowmap + (size_t)(ev & 1) * Ps * N;
    int* rm_new = pd.rowmap + (size_t)((ev + 1) & 1) * Ps * N;
#pragma unroll 1
    for (long long i = gt; i < (long long)Ps * N; i += GT) {
      const int slot = (int)(i / N), m = (int)(i - (long long)slot * N);
      const int a = ldcg_i32(anc + sp.slot0 + slot) - 1;
      const int ra = a / Ps, la = a - ra * Ps;
      if (ra == sp.rank) {
        __stcg(rm_new + i, ldcg_i32(rm_old + (size_t)la * N + m));
      } else if (slot == 0 || ldcg_i32(anc + sp.slot0 + slot - 1) != a + 1) {
        // first local child of an ancestor held by another rank: its occupied rows are pulled into four
        // fresh local rows each (the row, its child of step st+1, the two ids handed out for step st+2)
        // A remote row is pulled ONCE however many ancestors over there refer to it (particles that share a
        // cluster on their rank share its copy here): the first to claim it in pull_map reserves the ids.
        const int rb = ldcg_i32(on_rank(sp, rm_old, ra) + (size_t)la * N + m);
        if (rb != pd.cap - 1) {
          int* pm = sp.pull_map + ((size_t)k * sp.R + ra) * pd.cap + rb;
          if (atomicCAS(pm, -1, -2) == -1) {
            // (nobody pushes to the free stack during a resampling: one atomic claims the four slots)
            const int first = atomicSub(pd.ctr + 1, 4) - 4;
            if (first < 0) { atomicExch(sp.err, 80); sm.fail = 1; }
            else {
              const int v2 = spec_gtake(pd, first), c2 = spec_gtake(pd, first + 1);
              const int a2 = spec_gtake(pd, first + 2), b2 = spec_gtake(pd, first + 3);
              const long long job = atomicAdd((unsigned long long*)&sp.counters[5], 1ull);
              sp.pull_jobs[2 * job] = make_int4(k | (ra << 8), rb, v2, c2);
              sp.pull_jobs[2 * job + 1] = make_int4(a2, b2, 0, 0);
              __stcg(pm, v2);
            }
          }
        }
      }
    }
  }
  if (sp.R > 1) {
    if (!spec_gsync(sp, sm)) return false;
    // every label of a first child of a remote ancestor: the local copy of the row it referred to over there
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
      const PoolDev& pd = sp.pd[k];
      const int* rm_old = pd.rowmap + (size_t)(ev & 1) * Ps * N;
      int* rm_new = pd.rowmap + (size_t)((ev + 1) & 1) * Ps * N;
#pragma unroll 1
      for (long long i = gt; i < (long long)Ps * N; i += GT) {
        const int slot = (int)(i / N), m = (int)(i - (long long)slot * N);
        const int a = ldcg_i32(anc + sp.slot0 + slot) - 1;
        const int ra = a / Ps, la = a - ra * Ps;
        if (ra == sp.rank || !(slot == 0 || ldcg_i32(anc + sp.slot0 + slot - 1) != a + 1)) continue;
        const int rb = ldcg_i32(on_rank(sp, rm_old, ra) + (size_t)la * N + m);
        __stcg(rm_new + i, rb == pd.cap - 1 ? rb : ldcg_i32(sp.pull_map + ((size_t)k * sp.R + ra) * pd.cap + rb));
      }
    }
    if (!spec_gsync(sp, sm)) return false;
    // pull the reserved rows (a warp per row); the other children of a remote ancestor share its first child's map
    const long long njobs = __ldcg(&sp.counters[5]);
    const long long gw = gt >> 5, GWp = GT >> 5;
#pragma unroll 1
    for (long long item = gw; item < njobs * SPEC_PULL_PARTS; item += GWp) {
      const long long job = item / SPEC_PULL_PARTS;
      const int part = (int)(item - job * SPEC_PULL_PARTS);
      const int4 j0 = __ldcg(sp.pull_jobs + 2 * job);
      spec_row_pull(sp, j0, __ldcg(sp.pull_jobs + 2 * job + 1), parn, part);
      if (part == 0 && (threadIdx.x & 31) == 0)  // the map is clear again for the next resampling
        __stcg(sp.pull_map + ((size_t)(j0.x & 0xff) * sp.R + (j0.x >> 8)) * sp.pd[j0.x & 0xff].cap + j0.y, -1);
    }
    if (gt == 0) sp.counters[3] += njobs;
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
      int* rm_new = sp.pd[k].rowmap + (size_t)((ev + 1) & 1) * Ps * N;
#pragma unroll 1
      for (long long i = gt; i < (long long)Ps * N; i += GT) {
        const int slot = (int)(i / N), m = (int)(i - (long long)slot * N);
        const int a1 = ldcg_i32(anc + sp.slot0 + slot);
        if ((a1 - 1) / Ps == sp.rank) continue;
        int f = slot;
        while (f > 0 && ldcg_i32(anc + sp.slot0 + f - 1) == a1) --f;
        if (f != slot) __stcg(rm_new + i, ldcg_i32(rm_new + (size_t)f * N + m));
      }
    }
    if (!spec_gsync(sp, sm)) return false;
    if (gt == 0) sp.counters[5] = 0;
  }
  RS_MARK(5)
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const PoolDev& pd = sp.pd[k];
    int* rc_new = pd.refcnt + (size_t)parn * pd.cap;
#pragma unroll 1
    for (long long r = gt; r < pd.cap; r += GT) {
      __stcg(rc_new + r, 0); __stcg(pd.mark + r, 0); __stcg(pd.freelist + r, -1);
      __stcg(pd.chosen + r, 0); __stcg(pd.chosen + pd.cap + r, 0); __stcg(pd.chosen + 2 * (size_t)pd.cap + r, 0);
    }
  }
  if (is_p)
    for (int sl = threadIdx.x; sl < ns; sl += PMDI_NT) T.lw_s[sl] = 1.0;  // logweight .= 1.0 (src/pmdi.jl:319)
  if (!spec_gsync(sp, sm)) return false;
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const PoolDev& pd = sp.pd[k];
    const int* rm_new = pd.rowmap + (size_t)((ev + 1) & 1) * Ps * N;
    int* rc_new = pd.refcnt + (size_t)parn * pd.cap;
#pragma unroll 1
    for (long long i = gt; i < (long long)Ps * N; i += GT) atomicAdd(rc_new + ldcg_i32(rm_new + i), 1);
  }
  if (gt == 0) {
    *sp.gcnt = 0;
    for (int k = 0; k < K; ++k) __stcg(sp.pd[k].ctr + 1, 0);
  }
  if (!spec_gsync(sp, sm)) return false;
  // live rows keep their child of step st+1 and the two ids handed out for step st+2
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const PoolDev& pd = sp.pd[k];
    const int empty = pd.cap - 1;
    const int* rc_new = pd.refcnt + (size_t)parn * pd.cap;
#pragma unroll 1
    for (long long r = gt; r < pd.cap; r += GT) {
      if (r != empty && ldcg_i32(rc_new + r) == 0) continue;
      if (!has_next) continue;
      const int c = ldcg_info(pd.info + (size_t)parn * pd.cap + r).z;
      __stcg(pd.mark + c, 1);
      __stcg(pd.mark + ldcg_info(pd.info + (size_t)(parn ^ 1) * pd.cap + r).z, 1);
      __stcg(pd.mark + ldcg_info(pd.info + (size_t)(parn ^ 1) * pd.cap + c).z, 1);
    }
  }
  if (!spec_gsync(sp, sm)) return false;
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const PoolDev& pd = sp.pd[k];
    const int* rc_new = pd.refcnt + (size_t)parn * pd.cap;
    // (free rows are the many: one counter update per warp, not per row)
#pragma unroll 1
    for (long long rb = (gt >> 5) << 5; rb < pd.cap - 1; rb += GT) {
      const long long r = rb + (threadIdx.x & 31);
      const bool in = r < pd.cap - 1;
      const int rc = in ? ldcg_i32(rc_new + r) : 1;
      if (in && rc > 0) {
        const int i = atomicAdd(sp.gcnt, 1);
        const int c = has_next ? ldcg_info(pd.info + (size_t)parn * pd.cap + r).z : -1;
        __stcg(sp.glist + i, make_int4((k << SPEC_KSHIFT) | (int)r, c, ldcg_i32(sp.ds[k].n + r), 0));
      }
      const bool fr = in && rc == 0 && !ldcg_i32(pd.mark + r);
      const unsigned m = __ballot_sync(FULL, fr);
      if (m) {
        int base = 0;
        const int leader = __ffs(m) - 1;
        if ((int)(threadIdx.x & 31) == leader) base = atomicAdd(pd.ctr + 1, __popc(m));
        base = __shfl_sync(FULL, base, leader);
        if (fr) pd.freelist[base + __popc(m & ((1u << (threadIdx.x & 31)) - 1u))] = (int)r;
      }
    }
  }
  if (!spec_xsync(sp, sm)) return false;  // no rank recycles a row while a peer may still be pulling it
  RS_MARK(7)
#undef RS_MARK
  if (gt == 0 && has_next) atomicAdd((unsigned long long*)&sp.counters[4], (unsigned long long)(-(long long)ldcg_i32(sp.gcnt)));
  if (threadIdx.x == 0) { sm.ev = ev + 1; sm.res_flag = 0; }
  __syncthreads();
  if (is_p) {
    spec_load_units<GRP>(sp, sm, T, ns);
  } else if (e >= 0) {  // every E-CTA takes the whole new list; the cached free ids went back with the scan
    const int nl = ldcg_i32(sp.gcnt);
#pragma unroll 1
    for (int i = threadIdx.x; i < nl; i += PMDI_NT) spec_set_entry(sp, T, e, 0, i, __ldcg(sp.glist + i));
    if (threadIdx.x < K) { T.fc_top[threadIdx.x] = 0; sm.kc[threadIdx.x] = 0; }
    if (threadIdx.x == 0) { sm.cnt = nl; sm.lpar = 0; }
    if (has_next) spec_load_empty_next(sp, sm, parn);
  }
  __syncthreads();
  return !sm.fail;
}

// The resampling on one GPU.  What may be live afterwards is known without looking at the pool: the particles' new
// row maps are copies of old ones, and an old row map refers only to rows of the live-row list (after the fix of
// step st, the copy every E-CTA holds, in the same order) or to the empty row.  Every other row id of a dataset is
//   - on the free stack or in an E-CTA's free-id cache,
//   - the child of step st+1 of a listed row (the entry's .y, computed by E'(st+2)) or one of the two ids E'(st+2)
//     handed out for step st+2 (info[st&1].child of the row and of that child), or
//   - the empty row or an id handed out for it (its children stay reserved whatever the resampling does).
// So only the listed rows need a recount, and a listed row nobody refers to any more frees exactly itself, its child
// and their two ids of step st+2 (none were handed out when st+2 is past the last step).  The caches and the free
// stack are left as they are: the ids in them were free before and stay free.  The choice counters that can be
// non-zero are those the particles raised at steps st and st+1 (each unit's u_c2, u_c1: a commit clears its unit's
// counter of two steps ago): the units clear them themselves.  The empty row's reference count is read by nobody
// (a birth is decided from its choice counter) and is not counted.
// Three grid barriers: the plan (its inputs are complete since the decision) is drawn before the first one; row
// maps and the reset of the listed rows' counts; the recount; then each E-CTA drops the dead rows from its copy of
// the list, and the CTA that owns a dead entry (index mod GE) frees its four ids into its cache.  At the final
// resampling (st+1 == steps) only the row maps are needed: the next sweep's set-up starts the pool afresh.
template <bool GRP>
__device__ __noinline__ bool spec_resample(const SweepParams& sp, SpecSmem& sm, const SpecTables& T, int ns, int st,
                                           int* s_tmp, bool is_p, int e) {
  if (sp.R > 1) return spec_resample_sharded<GRP>(sp, sm, T, ns, st, s_tmp, is_p, e);
  const int K = sp.K, N = sp.N, P = sp.P, GE = sp.G - sp.GP - 1;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ev = sm.ev;
  const long long gt = (long long)spec_cta<GRP>() * PMDI_NT + tid, GT = (long long)sp.G * PMDI_NT;
  const int parn = (st + 1) & 1;  // the copy of the reference counts the fix of step st+1 reads
  const bool has_next = st + 1 < sp.steps;
  // sub-phase timers (instrumented runs): tacc[4] plan + first barrier, [5] row maps + recount, [7] list rebuild
  const bool tm = sp.phase_ns != nullptr && tid == 0;
  unsigned long long t_ = tm ? globaltimer_ns() : 0ull;
#define RS_MARK(i_) if (tm) { const unsigned long long n_ = globaltimer_ns(); sm.tacc[i_] += (n_ - t_) * PMDI_NW; t_ = n_; }
  if (spec_cta<GRP>() == sp.G - 1) {  // the D-CTA: its dynamic shared memory is free for the plan
    extern __shared__ __align__(16) unsigned char plan_raw[];
    PlanScratch sc = {sp.sc_w, sp.sc_pp, sp.sc_u, sp.sc_j, sp.sc_anc0};
    if (sp.plan_smem) {
      sc.w = (double*)plan_raw; sc.pp = sc.w + P; sc.u = sc.pp + P;
      sc.j = (int*)(sc.u + P); sc.a0 = sc.j + P;
    }
    pool_resample_plan(sp, st, ev, sm.res_mx, s_tmp, sp.lw + (size_t)(st & 1) * P, sc);
  }
  // every E-CTA has finished E'(st+2) and the fix of step st, every commit of step st+1 is in, the plan is drawn
  if (!spec_gsync(sp, sm)) return false;
  RS_MARK(4)
  const int* anc = sp.anc_log + (size_t)ev * P;
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const PoolDev& pd = sp.pd[k];
    const int* rm_old = pd.rowmap + (size_t)(ev & 1) * P * N;
    int* rm_new = pd.rowmap + (size_t)((ev + 1) & 1) * P * N;
#pragma unroll 1
    for (long long i = gt; i < (long long)P * N; i += GT) {
      const int p = (int)(i / N), m = (int)(i - (long long)p * N);
      __stcg(rm_new + i, ldcg_i32(rm_old + (size_t)(ldcg_i32(anc + p) - 1) * N + m));
    }
  }
  if (is_p)
    for (int sl = tid; sl < ns; sl += PMDI_NT) T.lw_s[sl] = 1.0;  // logweight .= 1.0 (src/pmdi.jl:319)
  if (tid == 0) { sm.ev = ev + 1; sm.res_flag = 0; }  // (read after the next CTA barrier: the new row maps)
  if (!has_next) {  // the final resampling: the row maps are all the finish kernel reads
    __syncthreads();
    return !sm.fail;
  }
  const int b3 = st % 3, z3 = (st + 1) % 3;
  if (is_p) {
#pragma unroll 1
    for (int u = tid; u < ns * K; u += PMDI_NT) {
      const PoolDev& pd = sp.pd[T.u_ks[u] & 0xff];
      const int c1 = T.u_c1[u], c2 = T.u_c2[u];
      if (c2 >= 0) __stcg(pd.chosen + (size_t)b3 * pd.cap + c2, 0);
      if (c1 >= 0) __stcg(pd.chosen + (size_t)z3 * pd.cap + c1, 0);
    }
  } else if (e >= 0) {
#pragma unroll 1
    for (int i = e + GE * tid; i < sm.cnt; i += GE * PMDI_NT) {  // the entries this CTA owns
      const int4 en = spec_entry(sp, T, e, sm.lpar, i);
      const PoolDev& pd = sp.pd[(unsigned)en.x >> SPEC_KSHIFT];
      __stcg(pd.refcnt + (size_t)parn * pd.cap + (en.x & SPEC_VMASK), 0);
    }
  }
  if (!spec_gsync(sp, sm)) return false;
  // the recount: labels of one warp that refer to the same row are counted by one atomic
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const PoolDev& pd = sp.pd[k];
    const int empty = pd.cap - 1;
    const int* rm_new = pd.rowmap + (size_t)((ev + 1) & 1) * P * N;
    int* rc_new = pd.refcnt + (size_t)parn * pd.cap;
#pragma unroll 1
    for (long long ib = (gt >> 5) << 5; ib < (long long)P * N; ib += GT) {
      const long long i = ib + lane;
      const int r = i < (long long)P * N ? ldcg_i32(rm_new + i) : empty;
      const unsigned same = __match_any_sync(FULL, r);
      if (r != empty && lane == __ffs(same) - 1) atomicAdd(rc_new + r, __popc(same));
    }
  }
  if (is_p) spec_load_units<GRP>(sp, sm, T, ns);  // the new row maps are complete
  if (!spec_gsync(sp, sm)) return false;
  RS_MARK(5)
  if (!is_p && e >= 0) {
    const int lo = sm.lpar, ln = lo ^ 1, n_old = sm.cnt;
    const bool ids2 = st + 2 < sp.steps;  // E'(st+2) ran: the ids of step st+2 are handed out
    int nb = 0;
#pragma unroll 1
    for (int base = 0; base < n_old; base += PMDI_NT) {
      const int i = base + tid;
      int4 en = make_int4(0, 0, 0, 0);
      int rc = 0;
      if (i < n_old) {
        en = spec_entry(sp, T, e, lo, i);
        const int k = (unsigned)en.x >> SPEC_KSHIFT, v = en.x & SPEC_VMASK, c = en.y;
        const PoolDev& pd = sp.pd[k];
        rc = ldcg_i32(pd.refcnt + (size_t)parn * pd.cap + v);
        if (rc == 0 && (i % GE) == e) {  // dead: the row, its child, their ids of step st+2
          spec_free_id(sp, T, k, v);
          spec_free_id(sp, T, k, c);
          if (ids2) {
            spec_free_id(sp, T, k, ldcg_info(pd.info + (size_t)(parn ^ 1) * pd.cap + v).z);
            spec_free_id(sp, T, k, ldcg_info(pd.info + (size_t)(parn ^ 1) * pd.cap + c).z);
          }
        }
      }
      const unsigned keep = __ballot_sync(FULL, rc > 0);
      if (lane == 0) sm.wsum[warp] = __popc(keep);
      __syncthreads();
      int wpre = 0, tot = 0;
#pragma unroll
      for (int w = 0; w < PMDI_NW; ++w) {
        const int x = sm.wsum[w];
        if (w < warp) wpre += x;
        tot += x;
      }
      if (rc > 0) spec_set_entry(sp, T, e, ln, nb + wpre + __popc(keep & ((1u << lane) - 1u)), en);
      nb += tot;
      __syncthreads();
    }
    // rows evaluated ahead for step st+1 that this resampling killed
    if (e == 0 && tid == 0) atomicAdd((unsigned long long*)&sp.counters[4], (unsigned long long)(n_old - nb));
    if (tid < K) sm.kc[tid] = 0;
    if (tid == 0) { sm.cnt = nb; sm.lpar = ln; }
    spec_load_empty_next(sp, sm, parn);
  }
  RS_MARK(7)
#undef RS_MARK
  __syncthreads();
  return !sm.fail;
}

// Pool accounting at the end of a sweep on one GPU (the instrumented kernel): every row id of a dataset is in exactly
// one place - on the free stack, in one E-CTA's free-id cache, a row of the live-row list or that row's child of the
// last step (the list after the fix of step steps-2: the last step's outcome is never fixed, the final resampling
// leaves the list as it is), the empty row or its child of the last step.  Each place counts its ids into the mark
// array (zero since the set-up: on one GPU nothing else writes it); a row counted twice was handed out or freed twice,
// a row counted never has leaked.  Either ends the sweep with error 97.
template <bool GRP>
__device__ __noinline__ bool spec_check_pool(const SweepParams& sp, SpecSmem& sm, const SpecTables& T, int e) {
  const int K = sp.K, GE = sp.G - sp.GP - 1, tid = threadIdx.x;
  const long long gt = (long long)spec_cta<GRP>() * PMDI_NT + tid, GT = (long long)sp.G * PMDI_NT;
  auto count = [&](const PoolDev& pd, int id) {
    if (id >= 0 && id < pd.cap) atomicAdd(pd.mark + id, 1);
    else { atomicExch(sp.err, 97); sm.fail = 1; }
  };
  if (!spec_gsync(sp, sm)) return false;  // every push and pop of the sweep is done
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const PoolDev& pd = sp.pd[k];
    const int h = ldcg_i32(pd.ctr + 1);
#pragma unroll 1
    for (long long s = gt; s < h; s += GT) count(pd, ldcg_i32(pd.freelist + s));
  }
  if (e >= 0) {
#pragma unroll 1
    for (int k = 0; k < K; ++k)
#pragma unroll 1
      for (int i = tid; i < T.fc_top[k]; i += PMDI_NT) count(sp.pd[k], T.fc_s[k * SPEC_FC + i]);
#pragma unroll 1
    for (int i = e + GE * tid; i < sm.cnt; i += GE * PMDI_NT) {  // the entries this CTA owns
      const int4 en = spec_entry(sp, T, e, sm.lpar, i);
      const PoolDev& pd = sp.pd[(unsigned)en.x >> SPEC_KSHIFT];
      count(pd, en.x & SPEC_VMASK);
      count(pd, en.y);
    }
    if (e == 0 && tid < K) { count(sp.pd[tid], sp.pd[tid].cap - 1); count(sp.pd[tid], sm.b_next[tid]); }
  }
  if (!spec_gsync(sp, sm)) return false;
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const PoolDev& pd = sp.pd[k];
#pragma unroll 1
    for (long long r = gt; r < pd.cap; r += GT)
      if (ldcg_i32(pd.mark + r) != 1) { atomicExch(sp.err, 97); sm.fail = 1; }
  }
  __syncthreads();
  return !sm.fail;
}

template <bool DBG, bool GRP>
__device__ __forceinline__ void spec_sweep_body(const SweepParams& sp, SpecSmem& sm, unsigned char* smem_raw, int* s_tmp) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int NW = PMDI_NW;
  const int cta = spec_cta<GRP>();
  const int K = sp.K, N = sp.N, steps = sp.steps, GP = sp.GP;
  const bool is_p = cta < GP;
  const int e = cta - GP;
  const int Npad = (N + 31) & ~31;
  const int ns = is_p ? (sp.Ps - cta + GP - 1) / GP : 0;  // particle slots cta, cta + GP, ...
  const int nu = ns * K;
  const int MS = (sp.Ps + GP - 1) / GP, MU = MS * K;

  // dynamic shared memory: [observation ring][lf table][role tables]
  unsigned char* xring = smem_raw;
  SpecTables T;
#ifdef PMDI_X_GLOBAL
  T.lf = (double*)smem_raw;  // (no observation ring)
#else
  T.lf = (double*)(smem_raw + (size_t)sp.obs_ring * sp.sm_x_bytes);
#endif
  unsigned char* rt = (unsigned char*)(T.lf + ((sp.lf_T + 1) & ~1));  // 16-byte aligned
  T.lp_s = (double*)rt;
  T.Pi_s = T.lp_s + (size_t)NW * Npad;
  T.lw_s = T.Pi_s + (size_t)K * N;
  T.inc_s = T.lw_s + MS;
  T.lw_prev = T.inc_s + MU;
  T.ch_s = (int*)(T.lw_prev + MS);
  T.lab_s = T.ch_s + (size_t)NW * Npad;
  T.pcount = T.lab_s + MU;
  T.u_c = T.pcount + MS;
  T.u_child = T.u_c + MU;
  T.u_occ = T.u_child + MU;
  T.u_c1 = T.u_occ + MU;
  T.u_c2 = T.u_c1 + MU;
  T.u_prow = T.u_c2 + MU;
  T.u_ks = T.u_prow + MU;
  T.rm_s = T.u_ks + MU;
  T.el_s = (int4*)rt;  // the two roles overlay the same region
  T.fc_s = (int*)(T.el_s + (size_t)2 * SPEC_EC);
  T.fc_top = T.fc_s + (size_t)K * SPEC_FC;
  if (tid < PMDI_MAX_K) { sm.rows_eval[tid] = 0; sm.rows_ref[tid] = 0; sm.rows_spec[tid] = 0; sm.kadd[tid] = 0; }
  if (tid < 8) sm.tacc[tid] = 0;
  if (tid < PMDI_NW) sm.tr_n[tid] = 0;
  if (tid == 0) {
    sm.res_flag = 0; sm.fail = 0; sm.ev = 0; sm.pdone = 0; sm.res_mx = 0.0;
    sm.epoch = __ldcg(sp.bar_state); sm.xepoch = __ldcg(sp.bar_state + 1);  // the counters run on from the previous sweep
    sm.lpar = 0; sm.cnt = 0;
#ifndef PMDI_X_GLOBAL
    for (int b = 0; b < sp.obs_ring; ++b) mbar_init(&sm.obs_bar[b], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#endif
  }
  __syncthreads();
  if (is_p) {
#pragma unroll 1
    for (int i = tid; i < K * N; i += PMDI_NT) T.Pi_s[i] = sp.Pi[i];
#pragma unroll 1
    for (int sl = tid; sl < ns; sl += PMDI_NT) { T.lw_s[sl] = sp.lw_init; T.pcount[sl] = 0; }
#pragma unroll 1
    for (int u = tid; u < nu; u += PMDI_NT) T.u_ks[u] = (u % K) | ((u / K) << 8);
    spec_load_units<GRP>(sp, sm, T, ns);
  } else if (cta != sp.G - 1) {
#ifndef PMDI_X_GLOBAL
    if (tid == 0)
      for (int s = 0; s < sp.obs_ring; ++s) pool_issue_obs(sp, s, xring, sm.obs_bar);
#endif
#pragma unroll 1
    for (int i = tid; i < sp.lf_T; i += PMDI_NT) T.lf[i] = sp.lf_glob[i];
    const int nl = ldcg_i32(sp.gcnt);  // the set-up kernel listed the live prefix rows
#pragma unroll 1
    for (int i = tid; i < nl; i += PMDI_NT) spec_set_entry(sp, T, e, 0, i, __ldcg(sp.glist + i));
    if (tid < K) { T.fc_top[tid] = 0; sm.kc[tid] = 0; }
    if (tid == 0) sm.cnt = nl;
    __syncthreads();
    if (e == 0)
      for (int i = tid; i < nl; i += PMDI_NT) atomicAdd(&sm.kc[(unsigned)spec_entry(sp, T, e, 0, i).x >> SPEC_KSHIFT], 1);
    spec_refill(sp, sm, T);
  }
  __syncthreads();

  const bool timing = DBG && sp.phase_ns != nullptr;
  unsigned long long tw_prev = timing ? globaltimer_ns() : 0ull;
#define PHASE_MARK(i_)                                                 \
  if (DBG && timing && lane == 0) {                                    \
    const unsigned long long now_ = globaltimer_ns();                  \
    atomicAdd(&sm.tacc[i_], now_ - tw_prev);                           \
    tw_prev = now_;                                                    \
  }

  int obs_ok = -1;
  const bool is_d = cta == sp.G - 1;  // the CTA that decides on the resamplings
  // ---- A(-1): the predictive of x[0] for every live row, and the ids of the first children
  if (!is_p && !is_d) spec_eval<DBG>(sp, sm, T, e, 0, xring, obs_ok, -1);
  PHASE_MARK(1)
  if (!spec_gsync(sp, sm)) return;
  PHASE_MARK(0)
#pragma unroll 1
  for (int t = 0; t < steps; ++t) {
    SWEEP_TRACE(t, 40)
    if (is_p) {
      // ---- P(t): proposals (read-only), the decision on the resampling after step t-1, commit
#pragma unroll 1
      for (int u = warp; u < nu; u += NW) spec_propose<DBG, GRP>(sp, sm, T, u, t);
      SWEEP_TRACE(t, 49)
#pragma unroll 1
      for (int u = warp; u < nu; u += NW) spec_commit<DBG, GRP>(sp, sm, T, u, t, ns);
      PHASE_MARK(2)
      if (t > 0) {
        // The step was committed without knowing whether step t-1 ends in a resampling: the decision (an exchange
        // over NVLink when the particles are sharded) had the whole of this phase to arrive.  When it says
        // "resample" (a few steps per sweep) the commit is undone, the particles are resampled, the step is redone.
        __syncthreads();
        if (!spec_wait_decision(sp, sm, t - 1)) return;
        if (sm.res_flag) {
#pragma unroll 1
          for (int u = tid; u < nu; u += PMDI_NT) {  // labels back to the rows they pointed at; weights back
            const int ks = T.u_ks[u], k = ks & 0xff, slot = cta + (ks >> 8) * GP, label = T.lab_s[u];
            T.rm_s[u * N + label] = T.u_prow[u];
            __stcg(sp.pd[k].rowmap + ((size_t)(sm.ev & 1) * sp.Ps + slot) * N + label, T.u_prow[u]);
            atomicSub(&sm.rows_ref[k], (unsigned)T.u_occ[u]);
          }
#pragma unroll 1
          for (int sl = tid; sl < ns; sl += PMDI_NT) T.lw_s[sl] = T.lw_prev[sl];
          if (!spec_resample<GRP>(sp, sm, T, ns, t - 1, s_tmp, true, e)) return;
          PHASE_MARK(6)
#pragma unroll 1
          for (int u = warp; u < nu; u += NW) spec_propose<DBG, GRP>(sp, sm, T, u, t);
#pragma unroll 1
          for (int u = warp; u < nu; u += NW) spec_commit<DBG, GRP>(sp, sm, T, u, t, ns);
        }
      }
    } else if (is_d) {
      if (t > 0) {
        spec_decide(sp, sm, t - 1);
        if (sm.res_flag && !spec_resample<GRP>(sp, sm, T, ns, t - 1, s_tmp, false, -1)) return;
      }
    } else {
      // ---- E side: outcome of step t-1, then the children of step t and the predictive of x[t+1]
#ifndef PMDI_X_GLOBAL
      if (tid == PMDI_NT - 1 && t > 0) pool_issue_obs(sp, t - 1 + sp.obs_ring, xring, sm.obs_bar);  // x[t-1]'s slot refills
#endif
      if (t > 0) spec_fix<DBG>(sp, sm, T, e, t - 1);
      else spec_refresh_children(sp, sm, T, e);
      // the distinct clusters the reference evaluates at step t (src/pmdi.jl:218-220): the list and the empty one.
      // The empty one is counted at every step, as k_empty_lp evaluates it for every step; the reference stops
      // evaluating it once a resampling leaves no particle with an empty label (its pool renumbering,
      // src/pmdi.jl:329-339, then drops it), so from there on this count has one row more per step and dataset.
      if (e == 0 && tid < K) { sm.rows_eval[tid] += (unsigned)sm.kc[tid] + 1u; sm.kc[tid] = 0; }  // the next fix counts afresh
      PHASE_MARK(3)
      SWEEP_TRACE(t, 51)
      if (t + 1 < steps) spec_eval<DBG>(sp, sm, T, e, t + 1, xring, obs_ok, t - 1);
      PHASE_MARK(1)
      SWEEP_TRACE(t, 52)
      spec_refill(sp, sm, T);
      if (t > 0) {  // the decision on the resampling after step t-1: fetched inside the evaluation
        if (t + 1 >= steps) {
          __syncthreads();
          if (!spec_wait_decision(sp, sm, t - 1)) return;
        } else if (sm.fail) return;
        if (sm.res_flag) {
          if (!spec_resample<GRP>(sp, sm, T, ns, t - 1, s_tmp, false, e)) return;
          PHASE_MARK(6)
        }
      }
    }
    SWEEP_TRACE(t, 56)
    if (!spec_gsync(sp, sm)) return;  // B(t)
    PHASE_MARK(0)
  }
  // ---- after the last observation: its ESS test
  if (is_d) spec_decide(sp, sm, steps - 1);
  else { __syncthreads(); if (!spec_wait_decision(sp, sm, steps - 1)) return; }
  const int final_res = sm.res_flag;
  if (final_res && !spec_resample<GRP>(sp, sm, T, ns, steps - 1, s_tmp, is_p, is_d ? -1 : e)) return;
  if constexpr (DBG) {
    if (sp.R == 1 && !spec_check_pool<GRP>(sp, sm, T, (is_p || is_d) ? -1 : e)) return;
  }
  if (tid < K) {
    atomicAdd(sp.rows_eval + tid, (unsigned long long)sm.rows_eval[tid]);
    atomicAdd(sp.rows_ref + tid, (unsigned long long)sm.rows_ref[tid]);
    atomicAdd(sp.rows_spec + tid, (unsigned long long)sm.rows_spec[tid]);
    atomicAdd(sp.rows_add + tid, (unsigned long long)sm.kadd[tid]);
  }
  if (cta == 0)  // after a final resampling all log-weights are 1.0 (src/pmdi.jl:319)
    for (int p = tid; p < sp.P; p += PMDI_NT)
      sp.lw_out[p] = final_res ? 1.0 : __ldcg(on_rank(sp, sp.lw + (size_t)((steps - 1) & 1) * sp.P + p, p / sp.Ps));
  if (timing && tid < 8) sp.phase_ns[(size_t)cta * 8 + tid] = sm.tacc[tid] / NW;
  if (cta == 0 && tid == 0) sp.counters[2] = sm.ev;
  // the peers' stores into this rank's allocation log have landed before the finish kernel reads it
  if (sp.R > 1) spec_xsync(sp, sm);
  if (cta == 0 && tid == 0) { sp.bar_state[0] = sm.epoch; sp.bar_state[1] = sm.xepoch; }  // where the next sweep's counters start
#undef PHASE_MARK
}

#define SPEC_KERNEL_PROLOGUE                                                                              \
  extern __shared__ __align__(16) unsigned char smem_raw[];                                               \
  __shared__ __align__(16) SpecSmem sm;                                                                   \
  __shared__ int s_tmp[4];                                                                                \
  __shared__ __align__(16) SweepParams sp_s;                                                              \
  {                                                                                                       \
    const int4* src = (const int4*)&sp_in;                                                                \
    int4* dst = (int4*)&sp_s;                                                                             \
    _Pragma("unroll 1") for (int i = threadIdx.x; i < (int)(sizeof(SweepParams) / 16); i += PMDI_NT) dst[i] = src[i]; \
  }                                                                                                       \
  __syncthreads();

#if defined(PMDI_X_GLOBAL)  // (the wide module, sweep_wide.cu: the observation is read from global memory)
extern "C" __global__ void __launch_bounds__(PMDI_NT, 1) k_sweep_spec_wide(const __grid_constant__ SweepParams sp_in) {
  SPEC_KERNEL_PROLOGUE
  spec_sweep_body<false, false>(sp_s, sm, smem_raw, s_tmp);
}
extern "C" __global__ void __launch_bounds__(PMDI_NT, 1) k_sweep_spec_wide_dbg(const __grid_constant__ SweepParams sp_in) {
  SPEC_KERNEL_PROLOGUE
  spec_sweep_body<true, false>(sp_s, sm, smem_raw, s_tmp);
}
#elif !defined(PMDI_SPEC_GROUP)  // (the group module, spec_group.cu, carries the group kernels alone)
extern "C" __global__ void __launch_bounds__(PMDI_NT, 1) k_sweep_spec(const __grid_constant__ SweepParams sp_in) {
  SPEC_KERNEL_PROLOGUE
  spec_sweep_body<false, false>(sp_s, sm, smem_raw, s_tmp);
}
extern "C" __global__ void __launch_bounds__(PMDI_NT, 1) k_sweep_spec_dbg(const __grid_constant__ SweepParams sp_in) {
  SPEC_KERNEL_PROLOGUE
  spec_sweep_body<true, false>(sp_s, sm, smem_raw, s_tmp);
}

// Start of a sweep: the rho-prefix clusters (rows 0..N-1) are shared by all particles
// (src/pmdi.jl:197-199); the live ones open the list of live rows; every other row is free.
// One block per dataset.
extern "C" __global__ void k_spec_init(SweepParams sp) {
  const int k = blockIdx.x, t = threadIdx.x, NT = blockDim.x, N = sp.N, Ps = sp.Ps;
  const PoolDev pd = sp.pd[k];
  const DsDev& ds = sp.ds[k];
  __shared__ int s_nf;
  for (int i = t; i < 3 * pd.cap; i += NT) pd.chosen[i] = 0;
  for (int r = t; r < pd.cap; r += NT) {
    pd.refcnt[r] = (r < N && ds.n[r] > 0) ? Ps : 0;  // the copy the fix of step 0 reads
    pd.refcnt[pd.cap + r] = 0;
    pd.mark[r] = 0;
    pd.freelist[r] = -1;
  }
  for (long long i = t; i < (long long)Ps * N; i += NT) {
    const int m = (int)(i % N);
    pd.rowmap[i] = ds.n[m] > 0 ? m : pd.cap - 1;
  }
  __syncthreads();
  if (t == 0) {
    int nf = 0;
    for (int m = 0; m < N; ++m) {
      if (ds.n[m] > 0) sp.glist[atomicAdd(sp.gcnt, 1)] = make_int4((k << SPEC_KSHIFT) | m, -1, ds.n[m], 0);
      else pd.freelist[nf++] = m;
    }
    s_nf = nf;
  }
  __syncthreads();
  const int nf0 = s_nf;
  for (int r = N + t; r < pd.cap - 1; r += NT) pd.freelist[nf0 + (r - N)] = r;
  if (t == 0) {
    pd.ctr[1] = nf0 + (pd.cap - 1 - N);
    ds.n[pd.cap - 1] = 0;
  }
  if (k == 0)
    for (int i = t; i < sp.steps; i += NT) sp.dec[i] = 0;
}
#endif

// Several contexts (chains) in ONE cooperative launch: member m owns CTAs cta0[m] .. cta0[m+1]-1 and runs its own sweep
// on them with a member-local CTA index.  A member's barrier counter, watchdog and error word are its own context's
// memory (reached through its SweepParams), so the members synchronise independently of each other.
#define PMDI_GROUP_MAX 16
struct SpecGroupMap {
  int n;
  int cta0[PMDI_GROUP_MAX + 1];
};
#ifdef PMDI_SPEC_GROUP
#define SPEC_GROUP_PROLOGUE                                                                               \
  extern __shared__ __align__(16) unsigned char smem_raw[];                                               \
  __shared__ __align__(16) SpecSmem sm;                                                                   \
  __shared__ int s_tmp[4];                                                                                \
  __shared__ __align__(16) SweepParams sp_s;                                                              \
  {                                                                                                       \
    int m = 0;                                                                                            \
    _Pragma("unroll 1") while (m + 1 < map.n && (int)blockIdx.x >= map.cta0[m + 1]) ++m;                  \
    if (threadIdx.x == 0) spec_group_cta = (int)blockIdx.x - map.cta0[m];                                 \
    const int4* src = (const int4*)(sps + m);                                                             \
    int4* dst = (int4*)&sp_s;                                                                             \
    _Pragma("unroll 1") for (int i = threadIdx.x; i < (int)(sizeof(SweepParams) / 16); i += PMDI_NT) dst[i] = __ldg(src + i); \
  }                                                                                                       \
  __syncthreads();

extern "C" __global__ void __launch_bounds__(PMDI_NT, 1) k_sweep_spec_group(const SweepParams* __restrict__ sps,
                                                                           const __grid_constant__ SpecGroupMap map) {
  SPEC_GROUP_PROLOGUE
  spec_sweep_body<false, true>(sp_s, sm, smem_raw, s_tmp);
}
extern "C" __global__ void __launch_bounds__(PMDI_NT, 1) k_sweep_spec_group_dbg(const SweepParams* __restrict__ sps,
                                                                               const __grid_constant__ SpecGroupMap map) {
  SPEC_GROUP_PROLOGUE
  spec_sweep_body<true, true>(sp_s, sm, smem_raw, s_tmp);
}
#endif
