// The conditional-SMC sweep over a COPY-ON-WRITE CLUSTER POOL: the per-observation loop of the
// reference (src/pmdi.jl:209-342) as one persistent cooperative kernel in which
//   * a cluster shared by several particles is ONE physical row, evaluated once per observation
//     (the reference's `for id in 1:maximum(particle_k)` loop, src/pmdi.jl:218-220);
//   * cluster_add! is copy-on-write (src/pmdi.jl:275-310): when every particle that refers to a row
//     chose it the row is updated in place, otherwise the choosers get a fresh row (one per source
//     row, shared by all of them) and the others keep the old one;
//   * resampling (src/pmdi.jl:318-341) permutes the particles' row maps and recounts references -
//     no statistics move.
// Same results as the dense form (every particle owning its N clusters): a row's content and its
// predictive do not depend on how many particles share it.
//
// Per observation step t the grid runs two phases separated by grid barriers:
//   E(t)  every live row's predictive of x[t].  A CTA takes rows round-robin; the row's 256-feature
//         blocks go to the CTA's warps, the block partials meet in shared memory and ONE number per
//         row (lp[row]) goes to HBM.  A row that was chosen at step t-1 gets x[t-1] added in the same
//         pass: in place, or - split - source row read once, fresh row written, both evaluated.
//   -- B1 --
//   P(t)  per (dataset, particle) unit, one warp: gather lp of the particle's N labels through its
//         row map, softmax-cdf, draw, weight increment (src/pmdi.jl:223-265); count the choosers of
//         the chosen row; the first chooser reserves a row for a possible split.  The K-th proposal
//         of a particle folds its log-weight with the Phi coupling (src/misc.jl:50-59); the CTA's
//         last particle publishes the CTA's (max, sum w, sum w^2).
//   -- B2 --
//   R(t)  choosers learn the row their label now maps to (tot == refcnt: in place); CTA 0 evaluates
//         calc_ESS (src/misc.jl:15-25) and attaches the decision to its arrival at B1(t+1) - then
//         straight into E(t+1).
// The ESS decision of step t is needed only before P(t+1): evaluations never depend on it (rows
// do not change under resampling), so with several GPUs the cross-rank exchange of the ESS
// partials is off the dependent chain; it has the whole of E(t+1) to arrive.
//
// The sweep is a chain of ~2 x steps dependent grid phases, each a few microseconds: it is bound by
// latency, and on this machine latency means INSTRUCTION FETCH as much as memory (32 KB of L1.5
// instruction cache per SM, a miss is an L2 round trip).  Hence: one block operator per cluster
// type (pool_types.cuh), debug capture / tracing / phase timing compiled into a separate kernel
// instantiation, the parameter block in shared memory, rare paths (resampling) out of line.
//
// The block operators are in pool_types.cuh; the observation ring, the resampling plan, the trace and the cross-rank
// barrier, which the spec engine uses too, in sweep_common.cuh; the finish kernels in aux_kernels.cuh.
#pragma once
#include "pool_types.cuh"
#include "sweep_common.cuh"

#define POOL_BIG_REF (1 << 30)
#define POOL_FLAG_SHIFT 44  // grid counter: arrivals in the low 44 bits, resampling decisions above
#define POOL_ARRIVE_MASK ((1ull << POOL_FLAG_SHIFT) - 1ull)
#ifdef PMDI_X_GLOBAL
#define POOL_RB 256  // blocks of a row whose partials meet in shared memory: 65,536 features in 256-feature blocks
#else
#define POOL_RB 32   // ... 8,192 features (a wider dataset runs the wide kernels)
#endif

struct PoolSmem {
  unsigned long long obs_bar[PMDI_OBS_RING];
  unsigned long long epoch;    // local grid-barrier arrivals expected so far
  unsigned long long xepoch;   // cross-rank barrier arrivals expected so far (one per rank)
  unsigned long long flag_base;  // resampling decisions attached to the counter before this sweep
  double res_mx;
  double red[2][2][POOL_RB];   // [row-iteration parity][updated or plain / split source][block] partials
  int res_flag;                // the last resolved step resamples
  int res_next;                // CTA 0: the decision to attach to the next B1 arrival
  int fail;
  int ev;                      // resampling events so far
  int pdone;                   // particles of this CTA folded this step
  int U[2][PMDI_MAX_K];        // by step parity: live rows of each dataset covered by the E phase
  int rbase[2][PMDI_MAX_K + 1];  // by step parity: first row task of each dataset
  unsigned rows_eval[PMDI_MAX_K], rows_ref[PMDI_MAX_K], rows_add[PMDI_MAX_K];
  unsigned long long tacc[8];
  int tr_n[PMDI_NW];
};

struct PoolTables {
  double* lf;      // [lf_T]
  double* lp_s;    // [NW][Npad]
  double* Pi_s;    // [K][N]
  double* lw_s;    // [MS]
  double* inc_s;   // [MS*K]
  int* lab_s;      // [MS*K]
  int* pcount;     // [MS]
  int* u_c;        // [MU] row chosen by the unit this step
  int* u_lab;      // [MU] label chosen
  int* u_lead;     // [MU] first chooser of the row
  int* u_duty;     // [MU] deferred bookkeeping of a leader: 0 none, 1 in place, 2 split
  int* u_dc;       // [MU] duty: source row
  int* u_dd;       // [MU] duty: destination row
  int* u_dtot;     // [MU] duty: number of choosers
  int* u_spare;    // [MU] row reserved by the unit for the next split it leads
  int* u_ks;       // [MU] dataset | local slot index << 8 of the unit
  int* rm_s;       // [MU][N] the units' row maps (copy of rowmap[ev & 1] rows of the owned slots)
};

// Local grid barrier (this GPU's CTAs), all threads.  b1: the barrier after an E phase - CTA 0 attaches
// its ESS decision to its arrival, everybody reads it off the counter it polls anyway (R == 1).
// sys: this CTA's peer stores are made visible system-wide before it arrives (cross-rank barrier).
__device__ __noinline__ bool pool_gsync(const SweepParams& sp, PoolSmem& sm, int b1 = 0, bool sys = false) {
  __syncthreads();
  if (threadIdx.x == 0) {
    sm.epoch += (unsigned long long)sp.G;
    unsigned long long inc = 1ull;
    if (b1 && blockIdx.x == 0 && sm.res_next) inc += 1ull << POOL_FLAG_SHIFT;
    if (sys) __threadfence_system(); else __threadfence();
    atomicAdd((unsigned long long*)sp.bar, inc);
    unsigned long long v = ld_acquire_u64((const unsigned long long*)sp.bar);
    if ((v & POOL_ARRIVE_MASK) < sm.epoch) {
      const unsigned long long t0 = globaltimer_ns();
      unsigned spins = 0;
#pragma unroll 1
      while (((v = ld_acquire_u64((const unsigned long long*)sp.bar)) & POOL_ARRIVE_MASK) < sm.epoch) {
        if (((++spins) & 0x3ffu) == 0) {
          // a CTA that failed has set sp.err before leaving: the others see it here
          if (__ldcg(sp.err) != 0) { sm.fail = 1; break; }
          if (globaltimer_ns() - t0 > sp.wd_ns) { atomicExch(sp.err, 77); sm.fail = 1; break; }
        }
      }
    }
    if (b1) sm.res_flag = (((v >> POOL_FLAG_SHIFT) - sm.flag_base - (unsigned long long)sm.ev) & 0xFFFFFull) != 0ull;
  }
  __syncthreads();
  return sm.fail == 0;
}

// barrier over the CTAs of ALL ranks (sweep_xsync)
__device__ __noinline__ bool pool_xsync(const SweepParams& sp, PoolSmem& sm) {
  return sweep_xsync(sp, sm, [&](bool sys) { return pool_gsync(sp, sm, 0, sys); });
}

// row tasks of the E phase of the step with parity b: the live rows as they are now (stable during
// the P phase before it).  One warp.
__device__ __forceinline__ void pool_snapshot(const SweepParams& sp, PoolSmem& sm, int b) {
  const int lane = threadIdx.x & 31;
  if (lane < sp.K) sm.U[b][lane] = ldcg_i32(sp.pd[lane].ctr);
  __syncwarp();
  if (lane == 0) {
    int base = 0;
#pragma unroll 1
    for (int k = 0; k < sp.K; ++k) { sm.rbase[b][k] = base; base += sm.U[b][k]; }
    sm.rbase[b][sp.K] = base;
  }
  __syncwarp();
}

// E phase of step `st`: predictive of x[st] for every live row; rows chosen at step st-1 (pending
// parity pp = (st-1)&1, or -1 at the first step) get x[st-1] added on the way.  The CTA takes
// `rpc` rows at a time (rpc = 16 warps / jq, jq = blocks per row rounded up to a power of two):
// warp w works on block w % jq (+ jq, ...) of row task w / jq, the partials meet in shared memory.
__device__ __noinline__ void pool_eval_rows(const SweepParams& sp, PoolSmem& sm, const PoolTables& T, int st, int pp,
                                            unsigned char* xring, int& obs_ok) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = st & 1, K = sp.K;
  const int jq = sp.jq, rpc = PMDI_NW / jq;
  const int sub = warp / jq, wj = warp - sub * jq;
  const int total = sm.rbase[b][K];
#ifdef PMDI_X_GLOBAL  // x[st] and x[st-1] are read from global memory: their observations
  const int oc = sp.order[sp.n1 - 1 + st], op = st > 0 ? sp.order[sp.n1 - 2 + st] : oc;
#else
  const unsigned xc = (unsigned)__cvta_generic_to_shared(xring + (size_t)(st % sp.obs_ring) * sp.sm_x_bytes);
  const unsigned xp = (unsigned)__cvta_generic_to_shared(xring + (size_t)((st + sp.obs_ring - 1) % sp.obs_ring) * sp.sm_x_bytes);
#endif
  int buf = 0;
#pragma unroll 1
  for (int base = (int)blockIdx.x * rpc; base < total; base += sp.G * rpc, buf ^= 1) {
    const int idx = base + sub;
    const bool active = sub < rpc && idx < total;
    int k = 0, c = 0, d = 0, mode = 0, nc = 0;
    if (active) {
#pragma unroll 1
      while (k + 1 < K && idx >= sm.rbase[b][k + 1]) ++k;
      const DsDev& ds = sp.ds[k];
      const PoolDev& pd = sp.pd[k];
      if (wj < ds.J) {
#ifndef PMDI_X_GLOBAL
        if (obs_ok < st) {  // x[st] has landed in the ring (x[st-1] was waited for one step ago)
          if (lane == 0) {
#pragma unroll 1
            for (int s = max(obs_ok + 1, st - 1); s <= st; ++s)
#pragma unroll 1
              while (!mbar_try_wait(&sm.obs_bar[s % sp.obs_ring], (unsigned)(s / sp.obs_ring) & 1u)) {}
          }
          __syncwarp();
          obs_ok = st;
        }
#endif
        c = ldcg_i32(pd.live + (idx - sm.rbase[b][k]));
        int tot = 0;  // the row's bookkeeping words in one round trip
        nc = ldcg_i32(ds.n + c);
        const int rf = ldcg_i32(pd.refcnt + c);
        d = c;
        if (pp >= 0) { tot = ldcg_i32(pd.chosen + (size_t)pp * pd.cap + c); d = ldcg_i32(pd.dst + (size_t)pp * pd.cap + c); }
        // every reference chose it: in place (src/pmdi.jl:284-286); some did: split (:288-309)
        mode = tot == 0 ? 0 : (tot == rf ? 1 : 2);
        if (mode != 2) d = c;
#ifdef PMDI_X_GLOBAL
        const size_t xrow = (size_t)ds.Dp * PMDI_XBYTES(ds);  // this dataset's rows are an array of their own
        const unsigned char* const xc = (const unsigned char*)ds.xstage + (size_t)oc * xrow;
        const unsigned char* const xp = (const unsigned char*)ds.xstage + (size_t)op * xrow;
        const unsigned xo = 0u;
#else
        const unsigned xo = (unsigned)ds.x_off;
#endif
#pragma unroll 1
        for (int j = wj; j < ds.J; j += jq) {
          const int q0 = j * ds.FB;
          const int nit = min(ds.FB / PMDI_WF, (ds.Dp - q0) / PMDI_WF);
          const int fo = q0 + 2 * lane;
          double vs = 0.0, v;
          if (ds.type == T_GAUSSIAN) {
            const long long so = (long long)c * ds.Dp + fo;
            v = gauss_block(ds.sum + so, ds.beta + so, ds.mu + so, ds.lamn + so, (long long)(d - c) * ds.Dp,
                            ds.aux + (long long)c * ds.J + j, ds.aux + (long long)d * ds.J + j, ds.flag + fo, nit,
                            mode, nc, xp + xo + fo * 8u, xc + xo + fo * 8u, &vs);
          } else if (ds.type == T_NEGBINOM) {
            v = nb_block(ds.S + (long long)c * ds.Dp + fo, (long long)(d - c) * ds.Dp, ds.aux + (long long)c * ds.J + j,
                         ds.aux + (long long)d * ds.J + j, nit, mode, nc, xp + xo + fo * 4u, xc + xo + fo * 4u,
                         (unsigned)__cvta_generic_to_shared(T.lf), sp.lf_T, &vs);
#ifdef PMDI_USER_TYPES
          } else if (ds.type == T_USER) {
            const unsigned eb = ds.uW < 0 ? 4u : 8u;
            const long long rw = user_row_words(ds);
            v = user_block(ds, ds.ust + c * rw + fo, (d - c) * rw,
                           ds.flag + fo, nit, mode, nc, xp + xo + fo * eb, xc + xo + fo * eb, &vs);
#endif
          } else {
            v = cat_block(pd.cw + ((long long)c * ds.Dp + fo) * pd.wpf, (long long)(d - c) * ds.Dp * pd.wpf, pd.wpf,
                          pd.fpw, nit, mode, xp + xo + fo * 4u, xc + xo + fo * 4u, &vs);
          }
          if (lane == 0) {
            const int ri = ds.J <= jq ? sub * jq + j : j;  // rows wider than 16 blocks: one row at a time
            sm.red[buf][0][ri] = v;
            sm.red[buf][1][ri] = vs;
          }
        }
      }
    }
    __syncthreads();
    if (active && wj == 0 && lane == 0) {  // the row's blocks in order, the size constant first
      const DsDev& ds = sp.ds[k];
      const int r0 = ds.J <= jq ? sub * jq : 0;
      double v = __ldg(ds.rc + nc + (mode ? 1 : 0));
#pragma unroll 1
      for (int j = 0; j < ds.J; ++j) v += sm.red[buf][0][r0 + j];
      __stcg(sp.pd[k].lp + d, v);
      if (mode == 2) {
        double vs = __ldg(ds.rc + nc);
#pragma unroll 1
        for (int j = 0; j < ds.J; ++j) vs += sm.red[buf][1][r0 + j];
        __stcg(sp.pd[k].lp + c, vs);
      }
      atomicAdd(&sm.rows_eval[k], mode == 2 ? 2u : 1u);
      if (mode) atomicAdd(&sm.rows_add[k], 1u);
    }
  }
}

// Deferred bookkeeping of the rows this CTA's leaders resolved at the previous step: after the
// barrier that follows R, nobody reads the old counts any more.  Thread per unit, from the last
// warp downwards (the first warps propose).
__device__ __forceinline__ void pool_duties(const SweepParams& sp, const PoolTables& T, int nu, int pp) {
#pragma unroll 1
  for (int u = PMDI_NT - 1 - (int)threadIdx.x; u < nu; u += PMDI_NT) {
    const int duty = T.u_duty[u];
    if (!duty) continue;
    const int k = T.u_ks[u] & 0xff;
    const PoolDev& pd = sp.pd[k];
    const int c = T.u_dc[u], d = T.u_dd[u], tot = T.u_dtot[u];
    __stcg(pd.chosen + (size_t)pp * pd.cap + c, 0);
    if (duty == 1) {
      __stcg(sp.ds[k].n + c, ldcg_i32(sp.ds[k].n + c) + 1);
    } else {
      if (c != pd.cap - 1) __stcg(pd.refcnt + c, ldcg_i32(pd.refcnt + c) - tot);
      __stcg(pd.refcnt + d, tot);
    }
    T.u_duty[u] = 0;
  }
}

// R phase for this CTA's units: the row each chooser's label maps to from now on.  Thread per unit.
__device__ __forceinline__ void pool_resolve_units(const SweepParams& sp, PoolSmem& sm, const PoolTables& T, int nu,
                                                   int par) {
  const int N = sp.N, G = sp.G;
#pragma unroll 1
  for (int u = threadIdx.x; u < nu; u += PMDI_NT) {
    const int ks = T.u_ks[u];
    const int k = ks & 0xff, slot = (int)blockIdx.x + (ks >> 8) * G;
    const PoolDev& pd = sp.pd[k];
    const int c = T.u_c[u];
    const int tot = ldcg_i32(pd.chosen + (size_t)par * pd.cap + c);
    const int dd = ldcg_i32(pd.dst + (size_t)par * pd.cap + c);
    const bool inplace = tot == ldcg_i32(pd.refcnt + c);
    const int d = inplace ? c : dd;
    T.rm_s[(size_t)u * N + T.u_lab[u]] = d;
    __stcg(pd.rowmap + ((size_t)(sm.ev & 1) * sp.Ps + slot) * N + T.u_lab[u], d);
    if (T.u_lead[u]) {
      if (!inplace) {  // the unit's reserved row is in use now: list it, reserve another
        pd.live[atomicAdd(pd.ctr, 1)] = d;
        __stcg(sp.ds[k].n + d, ldcg_i32(sp.ds[k].n + c) + 1);
        const int fi = atomicSub(pd.ctr + 1, 1) - 1;
        if (fi < 0) { atomicExch(sp.err, 80); sm.fail = 1; }
        else T.u_spare[u] = ldcg_i32(pd.freelist + fi);
      }
      T.u_duty[u] = inplace ? 1 : 2;
      T.u_dc[u] = c; T.u_dd[u] = d; T.u_dtot[u] = tot;
    }
  }
}

// this CTA's (max, sum w, sum w^2) over its particles' log-weights; one warp
__device__ __noinline__ void pool_cta_partial(const SweepParams& sp, const PoolTables& T, int ns, int par) {
  const int lane = threadIdx.x & 31;
  double m = -INFINITY;
#pragma unroll 1
  for (int sl = lane; sl < ns; sl += 32) m = fmax(m, T.lw_s[sl]);
  m = warp_max(m);
  double s1 = 0.0, s2 = 0.0;
#pragma unroll 1
  for (int sl = lane; sl < ns; sl += 32) {
    const double e = pm_exp(T.lw_s[sl] - m);
    s1 += e;
    s2 += e * e;
  }
  s1 = warp_sum(s1);
  s2 = warp_sum(s2);
  if (lane == 0) {
    double* ep = sp.ess_part + ((size_t)par * sp.G + blockIdx.x) * 3;
    __stcg(ep, m); __stcg(ep + 1, s1); __stcg(ep + 2, s2);
  }
}

// Combine `cnt` partials (max, s1, s2, stride `str` doubles) in a fixed order; one warp; every lane
// returns the same bits.  Loads go out eight per lane at a time (one L2 round trip per 256 partials).
__device__ __noinline__ void pool_combine(const double* ep, int cnt, int str, double& mx, double& num, double& den) {
  const int lane = threadIdx.x & 31;
  mx = -INFINITY;
#pragma unroll 1
  for (int c0 = 0; c0 < cnt; c0 += 256) {
    double v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = c0 + lane + 32 * i;
      v[i] = c < cnt ? ldcg_f64(ep + (size_t)str * c) : -INFINITY;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) mx = fmax(mx, v[i]);
  }
  mx = warp_max(mx);
  num = 0.0; den = 0.0;
#pragma unroll 1
  for (int c0 = 0; c0 < cnt; c0 += 256) {
    double m[8], a[8], b[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = c0 + lane + 32 * i;
      if (c < cnt) {
        m[i] = ldcg_f64(ep + (size_t)str * c);
        a[i] = ldcg_f64(ep + (size_t)str * c + 1);
        b[i] = ldcg_f64(ep + (size_t)str * c + 2);
      } else { m[i] = -INFINITY; a[i] = 0.0; b[i] = 0.0; }
    }
#pragma unroll 1
    for (int i = 0; i < 8; ++i) {
      if (c0 + lane + 32 * i < cnt) {
        const double e = pm_exp(m[i] - mx);
        num += a[i] * e;
        den += b[i] * (e * e);
      }
    }
  }
  num = warp_sum(num);
  den = warp_sum(den);
}

// Proposal of one unit (dataset k of a particle slot) at step `step`, one warp: src/pmdi.jl:223-265.
template <bool DBG>
__device__ __noinline__ void pool_propose(const SweepParams& sp, PoolSmem& sm, const PoolTables& T, int u, int step,
                                          int ns) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int K = sp.K, N = sp.N, P = sp.P, par = step & 1;
  const int ks = T.u_ks[u];
  const int k = ks & 0xff, sl = ks >> 8;
  const PoolDev& pd = sp.pd[k];
  const int p = sp.slot0 + (int)blockIdx.x + sl * sp.G;  // logical particle
  double* lps = T.lp_s + warp * ((N + 31) & ~31);
  const int* rm = T.rm_s + u * N;
  const int empty = pd.cap - 1;
  SWEEP_TRACE(step, 42)
  // lp of the unit's N labels: one number per row (E phase); two labels per lane go out together
  double mx = -INFINITY;
  int occ = 0;
#pragma unroll 1
  for (int m0 = 0; m0 < N; m0 += 64) {
    const int ma = m0 + lane, mb = ma + 32;
    const int ra = ma < N ? rm[ma] : empty, rb = mb < N ? rm[mb] : empty;
    const double a = ldcg_f64(pd.lp + ra), b = ldcg_f64(pd.lp + rb);
    if (ma < N) {
      lps[ma] = a;
      mx = fmax(mx, a);
      if (DBG && sp.dbg_lp) sp.dbg_lp[(((size_t)step * K + k) * P + p) * N + ma] = a;
    }
    if (mb < N) {
      lps[mb] = b;
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
  int rank = 1;
  const int c = rm[label];
  if (lane == 0) rank = atomicAdd(pd.chosen + (size_t)par * pd.cap + c, 1);  // in flight during the log below
  const double inc = pm_log(tot) + mx;
  int last_particle = 0;
  SWEEP_TRACE(step, 47)
  if (lane == 0) {
    if (rank == 0) __stcg(pd.dst + (size_t)par * pd.cap + c, T.u_spare[u]);  // first chooser: the row a split would use
    T.u_c[u] = c; T.u_lab[u] = label; T.u_lead[u] = rank == 0;
#pragma unroll 1
    for (int r = 0; r < sp.R; ++r)  // every rank back-traces the selected particle's lineage itself
      *on_rank(sp, sp.alloc_log + ((size_t)step * K + k) * P + p, r) = (uint8_t)label;
    if (DBG && sp.dbg_alloc) sp.dbg_alloc[((size_t)step * K + k) * P + p] = label + 1;
    atomicAdd(&sm.rows_ref[k], (unsigned)occ);
    // ---- weight increment; the K-th proposal of the particle folds its log-weight
    T.inc_s[sl * K + k] = inc;
    T.lab_s[sl * K + k] = label;
    __threadfence_block();
    if (atomicAdd(&T.pcount[sl], 1) == K - 1) {
      __threadfence_block();
      T.pcount[sl] = 0;
      const volatile double* iv = T.inc_s + (size_t)sl * K;
      const volatile int* lv = T.lab_s + (size_t)sl * K;
      double w = T.lw_s[sl];
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
      __stcg(sp.lw + p, w);
      if (DBG && sp.dbg_lw) sp.dbg_lw[(size_t)step * P + p] = w;
      __threadfence_block();
      last_particle = (atomicAdd(&sm.pdone, 1) == ns - 1) ? 1 : 0;
    }
  }
  last_particle = __shfl_sync(FULL, last_particle, 0);
  if (last_particle) {
    if (lane == 0) sm.pdone = 0;
    __threadfence_block();
    pool_cta_partial(sp, T, ns, par);
  }
  SWEEP_TRACE(step, 48)
}

// (re)load the owned units' row maps into shared memory and reserve one row per unit.  All threads.
__device__ __noinline__ void pool_load_units(const SweepParams& sp, PoolSmem& sm, const PoolTables& T, int ns) {
  const int K = sp.K, N = sp.N, nu = ns * K;
#pragma unroll 1
  for (int i = threadIdx.x; i < nu * N; i += PMDI_NT) {
    const int u = i / N, m = i - u * N;
    const int k = u % K, slot = (int)blockIdx.x + (u / K) * sp.G;
    T.rm_s[i] = ldcg_i32(sp.pd[k].rowmap + ((size_t)(sm.ev & 1) * sp.Ps + slot) * N + m);
  }
#pragma unroll 1
  for (int u = threadIdx.x; u < nu; u += PMDI_NT) {
    const PoolDev& pd = sp.pd[u % K];
    const int fi = atomicSub(pd.ctr + 1, 1) - 1;
    if (fi < 0) { atomicExch(sp.err, 80); sm.fail = 1; }
    else T.u_spare[u] = ldcg_i32(pd.freelist + fi);
  }
}

// One warp copies pool row `src` of the rank whose arena is `sdelta` bytes away into local row `dst`:
// statistics, aux, the row's current predictive, the cluster size.
__device__ __noinline__ void pool_row_pull(const SweepParams& sp, int k, long long sdelta, long long src, long long dst) {
  const DsDev& ds = sp.ds[k];
  const int lane = threadIdx.x & 31, Dp = ds.Dp;
#define PMDI_SRC(ptr_) ((decltype(ptr_))((const char*)(ptr_) + sdelta))
  if (ds.type == T_GAUSSIAN) {
#pragma unroll 1
    for (int q = 2 * lane; q < Dp; q += 64) {
      const double2 a = ldcg_f64x2(PMDI_SRC(ds.mu) + src * Dp + q), b = ldcg_f64x2(PMDI_SRC(ds.lamn) + src * Dp + q);
      const double2 c = ldcg_f64x2(PMDI_SRC(ds.sum) + src * Dp + q), d = ldcg_f64x2(PMDI_SRC(ds.beta) + src * Dp + q);
      *(double2*)(ds.mu + dst * Dp + q) = a; *(double2*)(ds.lamn + dst * Dp + q) = b;
      *(double2*)(ds.sum + dst * Dp + q) = c; *(double2*)(ds.beta + dst * Dp + q) = d;
    }
  } else if (ds.type == T_CATEGORICAL) {
    const PoolDev& pd = sp.pd[k];
    const long long W = (long long)Dp * pd.wpf;
#pragma unroll 1
    for (long long q = 2 * lane; q < W; q += 64)
      *(ulonglong2*)(pd.cw + dst * W + q) = ldcg_u64x2(PMDI_SRC(pd.cw) + src * W + q);
#ifdef PMDI_USER_TYPES
  } else if (ds.type == T_USER) {  // ust[row][word][feature]: one contiguous range of |uW| * Dp doubles
    const long long W = user_row_words(ds);
#pragma unroll 1
    for (long long q = 2 * lane; q < W; q += 64)
      *(double2*)(ds.ust + dst * W + q) = ldcg_f64x2(PMDI_SRC(ds.ust) + src * W + q);
#endif
  } else {
#pragma unroll 1
    for (int q = 2 * lane; q < Dp; q += 64)
      *(longlong2*)(ds.S + dst * Dp + q) = ldcg_i64x2(PMDI_SRC(ds.S) + src * Dp + q);
  }
#pragma unroll 1
  for (int jj = lane; jj < ds.J; jj += 32) ds.aux[dst * ds.J + jj] = ldcg_f64(PMDI_SRC(ds.aux) + src * ds.J + jj);
  if (lane == 0) {
    ds.n[dst] = ldcg_i32(PMDI_SRC(ds.n) + src);
    sp.pd[k].lp[dst] = ldcg_f64(PMDI_SRC(sp.pd[k].lp) + src);
  }
#undef PMDI_SRC
}

// Resampling after step `st` (src/pmdi.jl:318-341): every particle takes its ancestor's row map;
// references are recounted, rows nobody refers to any more go back to the free list.  An ancestor
// held by another rank has its occupied rows pulled into this rank's pool through NVLink peer
// memory (once per ancestor: its children here share the copies).
__device__ __noinline__ bool pool_resample(const SweepParams& sp, PoolSmem& sm, const PoolTables& T, int ns, int st,
                                           int* s_tmp) {
  const int K = sp.K, N = sp.N, Ps = sp.Ps;
  const int ev = sm.ev;
  const long long gt = (long long)blockIdx.x * PMDI_NT + threadIdx.x, GT = (long long)sp.G * PMDI_NT;
  // every CTA of every rank: deferred bookkeeping in, this step's log-weights and evaluations final
  if (!pool_xsync(sp, sm)) return false;
  if (blockIdx.x == 0)
    pool_resample_plan(sp, st, ev, sm.res_mx, s_tmp, nullptr, PlanScratch{sp.sc_w, sp.sc_pp, sp.sc_u, sp.sc_j, sp.sc_anc0});
  if (!pool_gsync(sp, sm)) return false;
  const int* anc = sp.anc_log + (size_t)ev * sp.P;
  if (gt == 0 && st + 1 < sp.steps) {  // rows the E phase evaluated ahead of this decision (live now, dead after it)
    long long u = 0;
#pragma unroll 1
    for (int k = 0; k < K; ++k) u += ldcg_i32(sp.pd[k].ctr);
    sp.counters[4] += u;
  }
  // ---- A1: row maps of children of local ancestors; first local child of a remote ancestor reserves rows
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
        const int rb = ldcg_i32(on_rank(sp, rm_old, ra) + (size_t)la * N + m);
        int d = pd.cap - 1;
        if (rb != pd.cap - 1) {
          const int fi = atomicSub(pd.ctr + 1, 1) - 1;
          if (fi < 0) { atomicExch(sp.err, 80); }
          else {
            d = ldcg_i32(pd.freelist + fi);
            const long long job = atomicAdd((unsigned long long*)&sp.counters[5], 1ull);
            sp.pull_jobs[job] = make_int4(k, ra, rb, d);
          }
        }
        __stcg(rm_new + i, d);
      }
    }
#pragma unroll 1
    for (long long r = gt; r < pd.cap; r += GT) __stcg(pd.refcnt + r, 0);
  }
#pragma unroll 1
  for (int sl = threadIdx.x; sl < ns; sl += PMDI_NT) T.lw_s[sl] = 1.0;  // logweight .= 1.0 (src/pmdi.jl:319)
  if (!pool_gsync(sp, sm)) return false;
  // ---- A2: pull the reserved rows; the other children of a remote ancestor share its first child's map
  if (sp.R > 1) {
    const long long njobs = __ldcg(&sp.counters[5]);
    const long long gw = gt >> 5, GWp = GT >> 5;
#pragma unroll 1
    for (long long job = gw; job < njobs; job += GWp) {
      const int4 jb = __ldcg(sp.pull_jobs + job);
      pool_row_pull(sp, jb.x, sp.peer_delta[jb.y], jb.z, jb.w);
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
#pragma unroll 1
        while (f > 0 && ldcg_i32(anc + sp.slot0 + f - 1) == a1) --f;
        if (f != slot) __stcg(rm_new + i, ldcg_i32(rm_new + (size_t)f * N + m));
      }
    }
  }
  if (gt == 0)
#pragma unroll 1
    for (int k = 0; k < K; ++k) { __stcg(sp.pd[k].ctr, 1); __stcg(sp.pd[k].ctr + 1, 0); }  // the lists are rebuilt below
  if (!pool_gsync(sp, sm)) return false;
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const PoolDev& pd = sp.pd[k];
    const int* rm_new = pd.rowmap + (size_t)((ev + 1) & 1) * Ps * N;
#pragma unroll 1
    for (long long i = gt; i < (long long)Ps * N; i += GT) atomicAdd(pd.refcnt + ldcg_i32(rm_new + i), 1);
  }
  if (!pool_gsync(sp, sm)) return false;
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const PoolDev& pd = sp.pd[k];
#pragma unroll 1
    for (long long r = gt; r < pd.cap - 1; r += GT) {
      if (ldcg_i32(pd.refcnt + r) > 0) pd.live[atomicAdd(pd.ctr, 1)] = (int)r;
      else pd.freelist[atomicAdd(pd.ctr + 1, 1)] = (int)r;
    }
    if (gt == 0) { __stcg(pd.refcnt + pd.cap - 1, POOL_BIG_REF); pd.live[0] = pd.cap - 1; }
  }
  if (gt == 0) sp.counters[5] = 0;
  // no rank may hand out a freed row while a peer is still pulling from it
  if (!pool_xsync(sp, sm)) return false;
  if (gt == 0 && st + 1 < sp.steps) {
    long long u = 0;
#pragma unroll 1
    for (int k = 0; k < K; ++k) u += ldcg_i32(sp.pd[k].ctr);
    sp.counters[4] -= u;
  }
  if (threadIdx.x == 0) { sm.ev = ev + 1; sm.res_flag = 0; }
  __syncthreads();
  pool_load_units(sp, sm, T, ns);  // the new row maps; the units' reserved rows were freed with the dead rows
  __syncthreads();
  return !sm.fail;
}

// ---- cross-rank ESS (R > 1).  After B2(t) one warp of CTA 0 folds this rank's CTA partials into
// one (max, sum w, sum w^2) and pushes it, tagged with the step, to every rank; the ranks combine
// the R rank partials before P(t+1) - a whole evaluation phase later.
__device__ __forceinline__ void pool_push_rank_partial(const SweepParams& sp, int t) {
  const int lane = threadIdx.x & 31, par = t & 1;
  double mxv, num, den;
  pool_combine(sp.ess_part + (size_t)par * sp.G * 3, sp.G, 3, mxv, num, den);
  if (lane == 0) {
    double* mine = sp.rank_part + ((size_t)par * sp.R + sp.rank) * 4;
#pragma unroll 1
    for (int r = 0; r < sp.R; ++r) {
      double* e = on_rank(sp, mine, r);
      __stcg(e, mxv); __stcg(e + 1, num); __stcg(e + 2, den);
    }
    __threadfence_system();
#pragma unroll 1
    for (int r = 0; r < sp.R; ++r) {
      unsigned long long* f = (unsigned long long*)(on_rank(sp, mine, r) + 3);
      asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(f), "l"(sp.tag_base + (unsigned long long)(t + 1)) : "memory");
    }
  }
}
// one warp: wait for every rank's partial of step t, then calc_ESS over them (same bits on every rank)
__device__ __noinline__ void pool_resolve_ranks(const SweepParams& sp, PoolSmem& sm, int t) {
  const int lane = threadIdx.x & 31, par = t & 1;
  const double* base = sp.rank_part + (size_t)par * sp.R * 4;
  if (lane < sp.R) {
    const unsigned long long* f = (const unsigned long long*)(base + (size_t)lane * 4 + 3);
    const unsigned long long t0 = globaltimer_ns();
    unsigned spins = 0;
#pragma unroll 1
    while (ld_acquire_sys_u64(f) < sp.tag_base + (unsigned long long)(t + 1)) {
      if (((++spins) & 0x3ffu) == 0) {
        if (__ldcg(sp.err) != 0) break;
        if (globaltimer_ns() - t0 > sp.wd_ns) { atomicExch(sp.err, 77); break; }
      }
    }
  }
  __syncwarp();
  double mxv, num, den;
  pool_combine(base, sp.R, 4, mxv, num, den);
  if (lane == 0) {
    const bool res = (num * num) / den <= 0.5 * (double)sp.P;  // src/pmdi.jl:317
    sm.res_mx = mxv;
    sm.res_flag = res ? 1 : 0;
    if (!res && blockIdx.x == 0) sp.ev_of_step[t] = -1;
  }
}

template <bool DBG>
__device__ __forceinline__ void pool_sweep_body(const SweepParams& sp, PoolSmem& sm, unsigned char* smem_raw, int* s_tmp) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int NW = PMDI_NW;
  const int cta = blockIdx.x;
  const int K = sp.K, N = sp.N, steps = sp.steps, G = sp.G;
  const int Npad = (N + 31) & ~31;
  const int ns = (sp.Ps - cta + G - 1) / G;  // particle slots cta, cta + G, ...
  const int nu = ns * K;
  const int MS = (sp.Ps + G - 1) / G, MU = MS * K;

  // dynamic shared memory: [observation ring][lf table][lp scratch][Pi][lw][inc][unit tables]
  unsigned char* xring = smem_raw;
  PoolTables T;
#ifdef PMDI_X_GLOBAL
  T.lf = (double*)smem_raw;  // (no observation ring)
#else
  T.lf = (double*)(smem_raw + (size_t)sp.obs_ring * sp.sm_x_bytes);
#endif
  T.lp_s = T.lf + sp.lf_T;
  T.Pi_s = T.lp_s + (size_t)NW * Npad;
  T.lw_s = T.Pi_s + (size_t)K * N;
  T.inc_s = T.lw_s + MS;
  T.lab_s = (int*)(T.inc_s + MU);
  T.pcount = T.lab_s + MU;
  T.u_c = T.pcount + MS;
  T.u_lab = T.u_c + MU;
  T.u_lead = T.u_lab + MU;
  T.u_duty = T.u_lead + MU;
  T.u_dc = T.u_duty + MU;
  T.u_dd = T.u_dc + MU;
  T.u_dtot = T.u_dd + MU;
  T.u_spare = T.u_dtot + MU;
  T.u_ks = T.u_spare + MU;
  T.rm_s = T.u_ks + MU;
#pragma unroll 1
  for (int i = tid; i < sp.lf_T; i += PMDI_NT) T.lf[i] = sp.lf_glob[i];
#pragma unroll 1
  for (int i = tid; i < K * N; i += PMDI_NT) T.Pi_s[i] = sp.Pi[i];
#pragma unroll 1
  for (int sl = tid; sl < ns; sl += PMDI_NT) { T.lw_s[sl] = sp.lw_init; T.pcount[sl] = 0; }
#pragma unroll 1
  for (int u = tid; u < nu; u += PMDI_NT) { T.u_duty[u] = 0; T.u_ks[u] = (u % K) | ((u / K) << 8); }
  if (tid < PMDI_MAX_K) { sm.rows_eval[tid] = 0; sm.rows_ref[tid] = 0; sm.rows_add[tid] = 0; }
  if (tid < 8) sm.tacc[tid] = 0;
  if (tid < PMDI_NW) sm.tr_n[tid] = 0;
  if (tid == 0) {
    sm.res_flag = 0; sm.res_next = 0; sm.fail = 0; sm.ev = 0; sm.pdone = 0; sm.res_mx = 0.0;
    const unsigned long long b0 = __ldcg(sp.bar_state);  // the counters run on from the previous sweep
    sm.epoch = b0 & POOL_ARRIVE_MASK; sm.flag_base = b0 >> POOL_FLAG_SHIFT; sm.xepoch = __ldcg(sp.bar_state + 1);
#ifndef PMDI_X_GLOBAL
#pragma unroll 1
    for (int b = 0; b < sp.obs_ring; ++b) mbar_init(&sm.obs_bar[b], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#endif
  }
  if (warp == NW - 1) pool_snapshot(sp, sm, 0);
  __syncthreads();
#ifndef PMDI_X_GLOBAL
  if (tid == 0)
#pragma unroll 1
    for (int s = 0; s < sp.obs_ring; ++s) pool_issue_obs(sp, s, xring, sm.obs_bar);
#endif
  pool_load_units(sp, sm, T, ns);

  const bool timing = DBG && sp.phase_ns != nullptr;
  unsigned long long tw_prev = timing ? globaltimer_ns() : 0ull;
#define PHASE_MARK(i_)                                                 \
  if (DBG && timing && lane == 0) {                                    \
    const unsigned long long now_ = globaltimer_ns();                  \
    atomicAdd(&sm.tacc[i_], now_ - tw_prev);                           \
    tw_prev = now_;                                                    \
  }

  int obs_ok = -1;
  pool_eval_rows(sp, sm, T, 0, -1, xring, obs_ok);
  PHASE_MARK(1)
  if (!pool_gsync(sp, sm, sp.R == 1)) return;  // B1(0)
  PHASE_MARK(0)
#pragma unroll 1
  for (int t = 0; t < steps; ++t) {
    const int par = t & 1;
    SWEEP_TRACE(t, 40)
    // ---- P(t): the last warp keeps house, the others propose
    if (t > 0) {
#ifndef PMDI_X_GLOBAL
      if (tid == PMDI_NT - 1) pool_issue_obs(sp, t - 1 + sp.obs_ring, xring, sm.obs_bar);  // x[t-1] is dead: its slot refills
#endif
      pool_duties(sp, T, nu, par ^ 1);
      if (sp.R > 1) {  // the ranks' partials of step t-1 have had E(t) to arrive
        if (warp == NW - 1) pool_resolve_ranks(sp, sm, t - 1);
        __syncthreads();
      }
      if (sm.res_flag) {
        if (!pool_resample(sp, sm, T, ns, t - 1, s_tmp)) return;
        PHASE_MARK(6)
      }
    }
    if (warp == NW - 1 && t + 1 < steps) pool_snapshot(sp, sm, par ^ 1);  // row tasks of E(t+1): the rows live now
    SWEEP_TRACE(t, 41)
#pragma unroll 1
    for (int u = warp; u < nu; u += NW) pool_propose<DBG>(sp, sm, T, u, t, ns);
    PHASE_MARK(2)
    SWEEP_TRACE(t, 49)
    if (!pool_gsync(sp, sm)) return;  // B2(t): every choice, reservation and ESS partial is in
    PHASE_MARK(4)
    SWEEP_TRACE(t, 50)
    // ---- R(t)
    pool_resolve_units(sp, sm, T, nu, par);
    SWEEP_TRACE(t, 51)
    if (cta == 0 && warp == NW - 1) {
      if (sp.R > 1) {
        pool_push_rank_partial(sp, t);
      } else {  // calc_ESS (src/misc.jl:15-25); the decision travels with CTA 0's arrival at B1(t+1)
        double mxv, num, den;
        pool_combine(sp.ess_part + (size_t)par * G * 3, G, 3, mxv, num, den);
        if (lane == 0) {
          const bool res = (num * num) / den <= 0.5 * (double)sp.P;  // src/pmdi.jl:317
          sm.res_mx = mxv;
          sm.res_next = res ? 1 : 0;
          if (!res) sp.ev_of_step[t] = -1;
        }
      }
    }
    PHASE_MARK(3)
    SWEEP_TRACE(t, 52)
    // ---- E(t+1)
    if (t + 1 < steps) pool_eval_rows(sp, sm, T, t + 1, par, xring, obs_ok);
    PHASE_MARK(1)
    SWEEP_TRACE(t, 56)
    if (!pool_gsync(sp, sm, sp.R == 1)) return;  // B1(t+1)
    PHASE_MARK(0)
  }
  // ---- after the last observation: its bookkeeping (cluster sizes), and its ESS test
  pool_duties(sp, T, nu, (steps - 1) & 1);
  if (sp.R > 1 && warp == NW - 1) pool_resolve_ranks(sp, sm, steps - 1);
  __syncthreads();
  const int final_res = sm.res_flag;
  if (final_res && !pool_resample(sp, sm, T, ns, steps - 1, s_tmp)) return;
  if (tid < K) {
    atomicAdd(sp.rows_eval + tid, (unsigned long long)sm.rows_eval[tid]);
    atomicAdd(sp.rows_ref + tid, (unsigned long long)sm.rows_ref[tid]);
    atomicAdd(sp.rows_add + tid, (unsigned long long)sm.rows_add[tid]);
  }
  if (cta == 0)  // after a final resampling all log-weights are 1.0 (src/pmdi.jl:319)
#pragma unroll 1
    for (int p = tid; p < sp.P; p += PMDI_NT)
      sp.lw_out[p] = final_res ? 1.0 : __ldcg(on_rank(sp, sp.lw + p, p / sp.Ps));
  if (timing && tid < 8) sp.phase_ns[(size_t)cta * 8 + tid] = sm.tacc[tid] / NW;
  if (cta == 0 && tid == 0) sp.counters[2] = sm.ev;
  // the peers' stores into this rank's allocation log have landed before the finish kernel reads it
  if (sp.R > 1) pool_xsync(sp, sm);
  if (cta == 0 && tid == 0) {  // where the next sweep's counters start
    sp.bar_state[0] = ((sm.flag_base + (unsigned long long)sm.ev) << POOL_FLAG_SHIFT) + sm.epoch;
    sp.bar_state[1] = sm.xepoch;
  }
#undef PHASE_MARK
}

// The parameter block lives in shared memory for the whole sweep: the helpers take it by reference, and a
// reference to the kernel's parameter space turns every field access into a generic load from the
// constant window.
#define POOL_KERNEL_PROLOGUE                                                                              \
  extern __shared__ __align__(16) unsigned char smem_raw[];                                               \
  __shared__ __align__(16) PoolSmem sm;                                                                   \
  __shared__ int s_tmp[4];                                                                                \
  __shared__ __align__(16) SweepParams sp_s;                                                              \
  {                                                                                                       \
    static_assert(sizeof(SweepParams) % 16 == 0, "SweepParams is copied in 16-byte words");              \
    const int4* src = (const int4*)&sp_in;                                                                \
    int4* dst = (int4*)&sp_s;                                                                             \
    _Pragma("unroll 1") for (int i = threadIdx.x; i < (int)(sizeof(SweepParams) / 16); i += PMDI_NT) dst[i] = src[i]; \
  }                                                                                                       \
  __syncthreads();

#ifdef PMDI_X_GLOBAL  // (the wide module, sweep_wide.cu: the observation is read from global memory)
extern "C" __global__ void __launch_bounds__(PMDI_NT, 1) k_sweep_pool_wide(const __grid_constant__ SweepParams sp_in) {
  POOL_KERNEL_PROLOGUE
  pool_sweep_body<false>(sp_s, sm, smem_raw, s_tmp);
}
extern "C" __global__ void __launch_bounds__(PMDI_NT, 1) k_sweep_pool_wide_dbg(const __grid_constant__ SweepParams sp_in) {
  POOL_KERNEL_PROLOGUE
  pool_sweep_body<true>(sp_s, sm, smem_raw, s_tmp);
}
#else
// production kernel: no debug capture, no tracing, no phase timing in the instruction stream
extern "C" __global__ void __launch_bounds__(PMDI_NT, 1) k_sweep_pool(const __grid_constant__ SweepParams sp_in) {
  POOL_KERNEL_PROLOGUE
  pool_sweep_body<false>(sp_s, sm, smem_raw, s_tmp);
}
// PMDI_SWEEP_DEBUG / PMDI_SWEEP_TIME_PHASES / PMDI_TRACE_STEP
extern "C" __global__ void __launch_bounds__(PMDI_NT, 1) k_sweep_pool_dbg(const __grid_constant__ SweepParams sp_in) {
  POOL_KERNEL_PROLOGUE
  pool_sweep_body<true>(sp_s, sm, smem_raw, s_tmp);
}

// ------------------------------------------------------------------------------------------------
// set-up kernel of the pool engine (the finish kernels, which every engine runs: aux_kernels.cuh)
// ------------------------------------------------------------------------------------------------

// Start of a sweep: the rho-prefix clusters (rows 0..N-1, built by k_prefix_build / k_proto_aux) are
// shared by all particles (src/pmdi.jl:197-199: particle[u,:,k] .= id; clusters_counts = particles).
// One block per dataset.
extern "C" __global__ void k_pool_init(SweepParams sp) {
  const int k = blockIdx.x, t = threadIdx.x, NT = blockDim.x, N = sp.N, Ps = sp.Ps;
  const PoolDev pd = sp.pd[k];
  const DsDev& ds = sp.ds[k];
  __shared__ int s_nfree0;
#pragma unroll 1
  for (int i = t; i < 2 * pd.cap; i += NT) { pd.chosen[i] = 0; pd.dst[i] = -1; }
#pragma unroll 1
  for (int r = t; r < pd.cap; r += NT) pd.refcnt[r] = (r < N && ds.n[r] > 0) ? Ps : 0;
#pragma unroll 1
  for (long long i = t; i < (long long)Ps * N; i += NT) {
    const int m = (int)(i % N);
    pd.rowmap[i] = ds.n[m] > 0 ? m : pd.cap - 1;
  }
  if (t == 0) {
    int nl = 0, nf = 0;
    pd.live[nl++] = pd.cap - 1;
#pragma unroll 1
    for (int m = 0; m < N; ++m) {
      if (ds.n[m] > 0) pd.live[nl++] = m;
      else pd.freelist[nf++] = m;
    }
    pd.ctr[0] = nl;
    pd.ctr[1] = nf + (pd.cap - 1 - N);
    s_nfree0 = nf;
  }
  __syncthreads();
  const int nf0 = s_nfree0;
#pragma unroll 1
  for (int r = N + t; r < pd.cap - 1; r += NT) pd.freelist[nf0 + (r - N)] = r;
  __syncthreads();
  if (t == 0) { pd.refcnt[pd.cap - 1] = POOL_BIG_REF; ds.n[pd.cap - 1] = 0; }
}
#endif
