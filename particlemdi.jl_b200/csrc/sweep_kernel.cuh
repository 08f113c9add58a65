// The conditional-SMC sweep as ONE persistent kernel: the per-observation loop of the reference
// (src/pmdi.jl:209-342) runs on the device as a DATAFLOW over (dataset, particle) units, with no
// host involvement and no CTA-wide or grid-wide wait on the common path.
//
// Ownership.  A CTA owns a fixed set of particle SLOTS for the whole sweep - all K datasets of a
// slot, i.e. K units of sufficient statistics - so predictive, proposal, add and the particle's
// weight update are CTA-local.  Per observation step only the ESS test needs the grid, and it
// needs three numbers per CTA.
//
// Work.  A unit cycles  items(t) -> proposal(t) -> items(t+1) -> ...  independently of the other
// units of its CTA.  Items are handed to the CTA's 16 warps through per-step queues in shared
// memory (ticket = atomicAdd):
//   fused item  = one 256-feature block of the row the particle chose in step t-1: cluster_add!
//                 of x[t-1] (src/pmdi.jl:300) and calc_logprob of x[t] in one pass over the row;
//   plain item  = calc_logprob of `qb` blocks of any other occupied row (src/pmdi.jl:218-220).
// The warp that finishes the last item of a unit runs the unit's proposal (src/pmdi.jl:223-265:
// softmax-cdf, draw, weight increment) and at once appends the unit's items for step t+1 to the
// next queue, so other warps stream them while the slower units of step t are still going.  The
// warp whose proposal is the K-th of a particle folds the increments and the Phi coupling
// (src/misc.jl:50-59) into the particle's log-weight; the warp that completes the CTA's last
// particle publishes the CTA's (max, sum w, sum w^2), issues the TMA bulk copy of a later
// observation row into the 4-deep shared-memory ring (mbarrier-tracked) and ARRIVES at the grid
// counter - nobody waits there.
//
// The one gate: proposal(t+1) of any unit needs step t RESOLVED - every CTA has arrived and one
// warp of this CTA has combined the partials into calc_ESS (src/misc.jl:15-25; same bits in
// every CTA, so all CTAs take the same branch).  Units that get there early are parked and picked
// up by idle warps.  On the rare resampling step (ESS <= P/2) the CTA drains the queue (which
// applies the pending adds), all warps meet, CTA 0 runs draw_partstar (src/misc.jl:27-47), all
// CTAs move the duplicated particles' rows (two blocking grid barriers), and the step restarts.
#pragma once
#include "cluster_types.cuh"
#include "sweep_common.cuh"

// exclusive scan of in[0..P) (global scratch, CTA-local use) into out; returns the total.
__device__ int block_excl_scan(const int* in, int* out, int P, int* s_tmp /* PMDI_NT+1 ints */) {
  const int t = threadIdx.x;
  const int seg = (P + PMDI_NT - 1) / PMDI_NT;
  const int b = min(P, t * seg), e = min(P, b + seg);
  int s = 0;
  for (int i = b; i < e; ++i) s += in[i];
  __syncthreads();
  s_tmp[t] = s;
  __syncthreads();
  if (t == 0) {
    int acc = 0;
    for (int i = 0; i < PMDI_NT; ++i) { const int v = s_tmp[i]; s_tmp[i] = acc; acc += v; }
    s_tmp[PMDI_NT] = acc;
  }
  __syncthreads();
  int acc = s_tmp[t];
  for (int i = b; i < e; ++i) { const int v = in[i]; out[i] = acc; acc += v; }
  __syncthreads();
  return s_tmp[PMDI_NT];
}

// draw_partstar (src/misc.jl:27-47) + the slot plan, by CTA 0.  Output: anc_log[ev][P] (1-based),
// slot_of/logical_of[next][P], copies[], plan_out[0] = number of copies.
// The Fisher-Yates shuffle followed by partstar[1]=1 and sort! only decides WHICH element of the
// sorted systematic sample is replaced by the reference particle: the one the shuffle moves to
// position 1.  That index is traced through the swaps without moving anything.
__device__ __noinline__ void resample_plan(const SweepParams& sp, int step, int ev, double mx, const double* lw,
                              int* s_tmp) {
  const int P = sp.P, t = threadIdx.x;
  const int* slot_cur = sp.slot_of + (ev & 1) * P;
  int* slot_nxt = sp.slot_of + ((ev + 1) & 1) * P;
  int* logi_nxt = sp.logical_of + ((ev + 1) & 1) * P;
  for (int p = t; p < P; p += PMDI_NT) {
    sp.sc_w[p] = pm_exp(__ldcg(lw + p) - mx);
    // Fisher-Yates pick for position pos = p+1 (entry index p), pos >= 2
    const double us = sp.tape_shuffle ? sp.tape_shuffle[(size_t)step * P + p]
                                      : pm_uniform(sp.seed, sp.iter, DRAW_SHUFFLE, step, 0, p);
    int jj = 1 + (int)floor(us * (double)(p + 1));
    if (jj > p + 1) jj = p + 1;
    sp.sc_j[p] = jj;
    sp.sc_b[p] = 0;  // has_child
  }
  __syncthreads();
  if (t == 0) {  // pprob = cumsum(exp.(logweight .- max)), sequential (misc.jl:29)
    double acc = 0.0;
    for (int p = 0; p < P; ++p) { acc += sp.sc_w[p]; sp.sc_pp[p] = acc; }
  } else if (t == 32) {  // u, u + 1/P, ... by repeated addition (misc.jl:28,35)
    const double r = sp.tape_resamp ? sp.tape_resamp[step]
                                    : pm_uniform(sp.seed, sp.iter, DRAW_RESAMP, step, 0, 0);
    double u = r / (double)P;
    for (int i = 0; i < P; ++i) { sp.sc_u[i] = u; u += 1.0 / (double)P; }
  } else if (t == 64) {  // index of the pre-shuffle element that ends at position 1
    int tt = 0;
    for (int pos = 2; pos <= P; ++pos)
      if (sp.sc_j[pos - 1] - 1 == tt) tt = pos - 1;
    s_tmp[PMDI_NT + 1] = tt;
  }
  __syncthreads();
  const double tot = sp.sc_pp[P - 1];
  for (int i = t; i < P; i += PMDI_NT) {  // first p with pprob[p]/last >= u_i (misc.jl:33-38)
    const double ui = sp.sc_u[i];
    int lo = 0, hi = P;  // hi == P means none
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (pm_div(sp.sc_pp[mid], tot) >= ui) hi = mid; else lo = mid + 1;
    }
    sp.sc_anc0[i] = (lo < P) ? lo + 1 : P;
  }
  __syncthreads();
  const int drop = s_tmp[PMDI_NT + 1];
  int* anc = sp.anc_log + (size_t)ev * P;
  for (int i = t; i < P; i += PMDI_NT) {
    const int a = (i == 0) ? 1 : ((i - 1 < drop) ? sp.sc_anc0[i - 1] : sp.sc_anc0[i]);
    anc[i] = a;
    if (sp.dbg_anc) sp.dbg_anc[(size_t)step * P + i] = a;
  }
  __syncthreads();
  // first child of every ancestor keeps the ancestor's slot; the others take dead slots
  for (int i = t; i < P; i += PMDI_NT) {
    const int first = (i == 0) || (anc[i] != anc[i - 1]);
    sp.sc_a[i] = first ? 0 : 1;  // extra child
    if (first) sp.sc_b[anc[i] - 1] = 1;
  }
  __syncthreads();
  for (int p = t; p < P; p += PMDI_NT) sp.sc_b[p] = sp.sc_b[p] ? 0 : 1;  // dead
  __syncthreads();
  const int n_extra = block_excl_scan(sp.sc_a, sp.sc_c, P, s_tmp);  // sc_c = extra rank
  block_excl_scan(sp.sc_b, sp.sc_d, P, s_tmp);                      // sc_d = dead rank
  for (int p = t; p < P; p += PMDI_NT)
    if (sp.sc_b[p]) sp.sc_j[sp.sc_d[p]] = ldcg_i32(slot_cur + p);  // dead slot list
  __syncthreads();
  for (int i = t; i < P; i += PMDI_NT) {
    const int src = ldcg_i32(slot_cur + anc[i] - 1);
    int dst = src;
    if (sp.sc_a[i]) {
      dst = sp.sc_j[sp.sc_c[i]];
      sp.copies[sp.sc_c[i]] = make_int2(src, dst);
    }
    slot_nxt[i] = dst;
    logi_nxt[dst] = i;
  }
  if (t == 0) {
    sp.plan_out[0] = n_extra;
    sp.ev_of_step[step] = ev;
  }
  __syncthreads();
}

// optional per-warp event trace of one CTA and one step (PMDI_TRACE_STEP): tag << 48 | clock64
__device__ __noinline__ void trace_mark(const SweepParams& sp, int step, unsigned tag) {
  __shared__ int tr_cnt[PMDI_NT / 32];
  if (sp.trace && (int)blockIdx.x == sp.trace_cta && step == sp.trace_step && (threadIdx.x & 31) == 0) {
    const int w = threadIdx.x >> 5;
    unsigned long long* t = sp.trace + w * 128;
    const int n = (t[0] == 0 ? 0 : tr_cnt[w]) + 1;
    if (n < 128) {
      t[n] = ((unsigned long long)tag << 48) | (clock64() & 0xFFFFFFFFFFFFull);
      t[0] = n;
      tr_cnt[w] = n;
    }
  }
}
#define TRACE(step_, tag_) if (sp.trace) trace_mark(sp, (step_), (tag_));

#define PMDI_ITEM_FUSED 0x80000000u
#define PMDI_ITEM_INVALID 0xFFFFFFFFu

// one per step parity
struct StepQ {
  int head;       // tickets handed out
  int tail;       // item slots reserved
  int units_in;   // units that have appended their items (== nu: the list is closed)
  int part_tail;  // partial-sum slots reserved
  int left;       // warps that are done with this list
  int gen;        // the step this buffer serves
  int pdone;      // particles of this CTA whose weight is folded for this step
  int pad;
  unsigned long long ep;  // grid-counter value that completes this step's barrier
};

struct SweepSmem {
  StepQ q[2];
  unsigned long long obs_bar[PMDI_OBS_RING];  // mbarriers of the observation ring
  unsigned long long epoch;                   // arrivals this CTA has made, times G
  double res_mx;  // max log-weight over all particles at res_step
  int res_step;   // last step whose ESS this CTA knows
  int res_claim;  // step a warp has claimed to resolve
  int res_flag;   // ESS <= P/2 at res_step: resample before going on
  int arrived;    // last step this CTA has arrived for
  int fail;
  int ev;         // resampling events so far
  unsigned rows_eval[PMDI_MAX_K];
  unsigned long long tacc[8];
};

// per-CTA views into dynamic shared memory
struct CtaTables {
  unsigned* urow;   // [max_units][N]   occupied rows of a unit: label | n << 8
  int* ucount;      // [max_units]      number of occupied rows
  int* uinfo;       // [max_units]      k << 24 | slot     (unit u = local slot * K + k)
  int* ulog;        // [max_units]      logical particle of the unit's slot (RNG address, log index)
  int* pend;        // [max_units]      pending add: label | n_after << 8, or -1
  int* pe;          // [max_units]      position of the pending row in urow
  int* ustate;      // [max_units]      0, or 1 + step: all items of that step done, proposal parked
  int* remaining;   // [2][max_units]   items of the unit not yet finished, per step parity
  int* pbase;       // [2][max_units]   first partial-sum slot of the unit, per step parity
  unsigned* items;  // [2][item_cap]    fused << 31 | u << 13 | e << 5 | j0, or INVALID
  double* part;     // [2][item_cap]    predictive partial sums
  double* lp_s;     // [NW][Npad]       per-warp proposal scratch
  double* Pi_s;     // [K][N]
  double* lw_s;     // [max_slots]      log-weight of the owned particles
  double* inc_s;    // [2][max_slots*K] this step's weight increments
  int* lab_s;       // [2][max_slots*K] this step's labels
  int* pcount;      // [2][max_slots]   proposals of the particle done this step
  int MU, cap;
};

// the grid counter as seen by this rank: other GPUs add to it through NVLink when R > 1
__device__ __forceinline__ unsigned long long ld_counter(const SweepParams& sp) {
  const unsigned long long* bar = (const unsigned long long*)sp.bar;
  return sp.R > 1 ? ld_acquire_sys_u64(bar) : ld_acquire_u64(bar);
}
// release everything this thread has observed, then add one arrival to EVERY rank's counter
__device__ __forceinline__ void arrive_all(const SweepParams& sp) {
  if (sp.R > 1) {
    __threadfence_system();
#pragma unroll 1
    for (int r = 0; r < sp.R; ++r) atomicAdd_system(on_rank(sp, (unsigned long long*)sp.bar, r), 1ull);
  } else {
    __threadfence();
    atomicAdd((unsigned long long*)sp.bar, 1ull);
  }
}
__device__ __forceinline__ int ld_vol(const int* p) { return *(const volatile int*)p; }
__device__ __forceinline__ void st_vol(int* p, int v) { *(volatile int*)p = v; }

// one thread: bulk-copy the K rows of the observation swept at `step` into ring slot step % 4
__device__ __noinline__ void issue_obs(const SweepParams& sp, int step, unsigned char* xring, unsigned long long* bars) {
  if (step >= sp.steps) return;
  const int b = step % PMDI_OBS_RING;
  const unsigned bar = (unsigned)__cvta_generic_to_shared(bars + b);
  const int obs = sp.order[sp.n1 - 1 + step];
  unsigned total = 0;
#pragma unroll 1
  for (int k = 0; k < sp.K; ++k) total += (unsigned)sp.ds[k].Dp * (sp.ds[k].type == T_GAUSSIAN ? 8u : 4u);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // earlier generic reads of the slot
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(total) : "memory");
#pragma unroll 1
  for (int k = 0; k < sp.K; ++k) {
    const DsDev& ds = sp.ds[k];
    const unsigned bytes = (unsigned)ds.Dp * (ds.type == T_GAUSSIAN ? 8u : 4u);
    const unsigned char* src = (const unsigned char*)ds.xstage + (size_t)obs * bytes;
    const unsigned dst = (unsigned)__cvta_generic_to_shared(xring + (size_t)b * sp.sm_x_bytes + ds.x_off);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
  }
}

// spin until the arrival counter reaches `target` (one thread); false = watchdog / error
__device__ __noinline__ bool bar_wait(const SweepParams& sp, unsigned long long target) {
  const unsigned long long t0 = globaltimer_ns();
  unsigned spins = 0;
  while (ld_counter(sp) < target) {
    if (((++spins) & 0x3ffu) == 0) {
      if (__ldcg(sp.err) != 0) return false;
      if (globaltimer_ns() - t0 > sp.wd_ns) { atomicExch(sp.err, 77); return false; }
    }
  }
  if (sp.R > 1) __threadfence_system(); else __threadfence();
  return true;
}

// blocking full grid barrier (resampling only), all threads of the CTA
__device__ __noinline__ bool grid_sync(const SweepParams& sp, SweepSmem& sm) {
  __syncthreads();
  if (threadIdx.x == 0) {
    sm.epoch += (unsigned long long)sp.R * sp.G;  // every CTA of every rank
    arrive_all(sp);
    if (!bar_wait(sp, sm.epoch)) sm.fail = 1;
  }
  __syncthreads();
  return sm.fail == 0;
}

// occupied rows (and the logical particle) of every owned unit, from the state in HBM
__device__ __noinline__ void rebuild_rows(const SweepParams& sp, const CtaTables& T, int nu, int ev) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, N = sp.N;
#pragma unroll 1
  for (int u = warp; u < nu; u += PMDI_NT / 32) {
    const int k = T.uinfo[u] >> 24, slot = T.uinfo[u] & 0xFFFFFF;
    int cnt = 0;
#pragma unroll 1
    for (int m0 = 0; m0 < N; m0 += 32) {
      const int m = m0 + lane;
      const int nm = (m < N) ? ldcg_i32(sp.ds[k].n + (long long)slot * N + m) : 0;
      const unsigned b = __ballot_sync(FULL, nm > 0);
      if (nm > 0) T.urow[(size_t)u * N + cnt + __popc(b & ((1u << lane) - 1))] = (unsigned)m | ((unsigned)nm << 8);
      cnt += __popc(b);
    }
    if (lane == 0) {
      T.ucount[u] = cnt;
      T.ulog[u] = ldcg_i32(sp.logical_of + (ev & 1) * sp.P + sp.slot0 + slot);
    }
  }
}

// cluster_add! of the pending row of every unit against observation buffer xb (only after the
// last observation: every other pending add is applied by the next step's fused items).
__device__ __noinline__ void flush_adds(const SweepParams& sp, const CtaTables& T, int nu, const unsigned char* xb,
                                        const double* lf) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NW = PMDI_NT / 32, N = sp.N;
#pragma unroll 1
  for (int it = warp; it < nu * sp.Jmax; it += NW) {
    const int u = it / sp.Jmax, j = it - u * sp.Jmax;
    const int k = T.uinfo[u] >> 24, slot = T.uinfo[u] & 0xFFFFFF;
    const DsDev& ds = sp.ds[k];
    if (j >= ds.J || T.pend[u] < 0) continue;
    const int label = T.pend[u] & 0xFF, n = T.pend[u] >> 8;
    const long long row = (long long)slot * N + label;
    if (ds.type == T_GAUSSIAN) gauss_add_block(ds, row, j, n, (const double*)(xb + ds.x_off), lane);
    else if (ds.type == T_CATEGORICAL) cat_add_block(ds, row, j, (const int*)(xb + ds.x_off), lane);
    else nb_add_block(ds, row, j, n, (const int*)(xb + ds.x_off), lane, lf, sp.lf_T);
  }
  __syncthreads();
}

// number of items / partial-sum slots a unit contributes to a step's list
__device__ __forceinline__ void unit_item_counts(const SweepParams& sp, const CtaTables& T, int u, int& nI, int& nB) {
  const int J = sp.ds[T.uinfo[u] >> 24].J, cnt = T.ucount[u], hp = T.pend[u] >= 0 ? 1 : 0;
  nI = (hp ? J : 0) + (cnt - hp) * ((J + sp.qb - 1) / sp.qb);
  nB = cnt * J;
}
// the unit's items, fused blocks first, written by one warp at items[ib ...]
__device__ __forceinline__ void write_unit_items(const SweepParams& sp, const CtaTables& T, int u, int nI,
                                                 unsigned* items) {
  const int lane = threadIdx.x & 31, qb = sp.qb;
  const int J = sp.ds[T.uinfo[u] >> 24].J, hp = T.pend[u] >= 0 ? 1 : 0, pe = T.pe[u];
  const int nF = hp ? J : 0, JQ = (J + qb - 1) / qb;
#pragma unroll 1
  for (int i = lane; i < nI; i += 32) {
    unsigned code;
    if (i < nF) {
      code = PMDI_ITEM_FUSED | ((unsigned)u << 13) | ((unsigned)pe << 5) | (unsigned)i;
    } else {
      const int r = i - nF;
      int e = r / JQ;
      const int q = r - e * JQ;
      if (hp && e >= pe) ++e;  // skip the fused row
      code = ((unsigned)u << 13) | ((unsigned)e << 5) | (unsigned)(q * qb);
    }
    *(volatile unsigned*)(items + i) = code;
  }
}

// (Re)start the queues at step t with the item lists of ALL units (no pending adds): kernel start
// and after a resampling.  All threads.
__device__ __noinline__ void init_queues(const SweepParams& sp, const CtaTables& T, SweepSmem& sm, int nu, int ns, int t) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, b = t & 1;
  for (int i = tid; i < 2 * T.cap; i += PMDI_NT) T.items[i] = PMDI_ITEM_INVALID;
  for (int u = tid; u < nu; u += PMDI_NT) { T.pend[u] = -1; T.pe[u] = 0; T.ustate[u] = 0; }
  for (int i = tid; i < 2 * ns; i += PMDI_NT) T.pcount[i] = 0;
  __syncthreads();
  if (warp == 0) {
    int runI = 0, runB = 0;
#pragma unroll 1
    for (int ub = 0; ub < nu; ub += 32) {
      const int u = ub + lane;
      int cI = 0, cB = 0;
      if (u < nu) unit_item_counts(sp, T, u, cI, cB);
      int iI = cI, iB = cB;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int vI = __shfl_up_sync(FULL, iI, o), vB = __shfl_up_sync(FULL, iB, o);
        if (lane >= o) { iI += vI; iB += vB; }
      }
      if (u < nu) {
        T.remaining[b * T.MU + u] = cI;
        T.pbase[b * T.MU + u] = runB + iB - cB;
        T.remaining[(b ^ 1) * T.MU + u] = runI + iI - cI;  // scratch: first item of the unit
        if (cI == 0) T.ustate[u] = 1 + t;                   // nothing to evaluate: straight to the proposal
      }
      runI += __shfl_sync(FULL, iI, 31);
      runB += __shfl_sync(FULL, iB, 31);
    }
    if (lane == 0) {
      StepQ& q = sm.q[b];
      q.head = 0; q.tail = runI; q.units_in = nu; q.part_tail = runB; q.left = 0; q.gen = t; q.pdone = 0;
      StepQ& q1 = sm.q[b ^ 1];
      q1.head = 0; q1.tail = 0; q1.units_in = 0; q1.part_tail = 0; q1.left = 0; q1.gen = t + 1; q1.pdone = 0;
      if (runI > T.cap || runB > T.cap) { atomicExch(sp.err, 78); sm.fail = 1; }
    }
  }
  __syncthreads();
  if (sm.fail) return;
#pragma unroll 1
  for (int u = warp; u < nu; u += PMDI_NT / 32) {
    int nI, nB;
    unit_item_counts(sp, T, u, nI, nB);
    write_unit_items(sp, T, u, nI, T.items + (size_t)b * T.cap + T.remaining[(b ^ 1) * T.MU + u]);
  }
  __syncthreads();
}

// One work item by one warp; returns the predictive partial sum (identical in all lanes).
__device__ __noinline__ double run_item(const SweepParams& sp, const CtaTables& T, unsigned code,
                                        const unsigned char* xs_cur, const unsigned char* xs_prev,
                                        const double* lf) {
  const int lane = threadIdx.x & 31, N = sp.N, qb = sp.qb, lfT = sp.lf_T;
  const bool fused = (code & PMDI_ITEM_FUSED) != 0;
  const int u = (code >> 13) & 0x3FFFF, e = (code >> 5) & 0xFF, j0 = code & 31;
  const int k = T.uinfo[u] >> 24, slot = T.uinfo[u] & 0xFFFFFF;
  const DsDev& ds = sp.ds[k];
  const unsigned ent = T.urow[(size_t)u * N + e];
  const int m = ent & 0xFF, n = ent >> 8;  // for the fused row n is the size AFTER the pending add
  const long long row = (long long)slot * N + m;
  const int j1 = fused ? j0 + 1 : min(ds.J, j0 + qb);
  if (ds.type == T_GAUSSIAN) {
    if (fused) return gauss_fused_block(ds, row, j0, n, (const double*)(xs_prev + ds.x_off),
                                        (const double*)(xs_cur + ds.x_off), lane);
    return gauss_eval_item(ds, row, j0, j1, n, (const double*)(xs_cur + ds.x_off), lane);
  }
  if (ds.type == T_CATEGORICAL) {
    if (fused) {
      cat_add_block(ds, row, j0, (const int*)(xs_prev + ds.x_off), lane);
      __syncwarp();
    }
    return cat_eval_item(ds, row, j0, j1, (const int*)(xs_cur + ds.x_off), lane);
  }
  if (fused) {
    nb_add_block(ds, row, j0, n, (const int*)(xs_prev + ds.x_off), lane, lf, lfT);
    __syncwarp();
  }
  return nb_eval_item(ds, row, j0, j1, n, (const int*)(xs_cur + ds.x_off), lane, lf, lfT);
}

// calc_ESS over the whole grid from the per-CTA partials of step `st` (max, sum w, sum w^2 with
// w = exp(l - max_cta)), by ONE warp; fixed shape -> identical bits in every CTA.
// Returns ESS <= P/2 (src/pmdi.jl:317); *mx_out = max log-weight.
__device__ __noinline__ bool resolve_ess(const SweepParams& sp, int st, double* mx_out) {
  const int lane = threadIdx.x & 31, G = sp.R * sp.G;  // CTAs of all ranks
  const double* ep = sp.ess_part + (size_t)(st & 1) * 3 * G;
  // One partial per CTA of every rank (148 on one GPU, 1184 on eight).  The loads go out in batches
  // of 8 per lane so that a batch costs ONE L2 round trip; the accumulation order is fixed, so every
  // CTA of every rank gets the same bits.
  double mx = -INFINITY;
#pragma unroll 1
  for (int base = 0; base < G; base += 256) {
    double m[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = base + lane + 32 * i;
      m[i] = (c < G) ? ldcg_f64(ep + 3 * c) : -INFINITY;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) mx = fmax(mx, m[i]);
  }
  mx = warp_max(mx);
  double num = 0.0, den = 0.0;
#pragma unroll 1
  for (int base = 0; base < G; base += 256) {
    double m[8], s1[8], s2[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = base + lane + 32 * i;
      const bool ok = c < G;
      m[i] = ok ? ldcg_f64(ep + 3 * c) : -INFINITY;  // exp(-inf) = 0 pads
      s1[i] = ok ? ldcg_f64(ep + 3 * c + 1) : 0.0;
      s2[i] = ok ? ldcg_f64(ep + 3 * c + 2) : 0.0;
    }
#pragma unroll 1
    for (int i = 0; i < 8; ++i) {
      const double e = pm_exp(m[i] - mx);
      num += s1[i] * e;
      den += s2[i] * (e * e);
    }
  }
  num = warp_sum(num);
  den = warp_sum(den);
  *mx_out = mx;
  const bool do_res = (num * num) / den <= 0.5 * (double)sp.P;
  if (!do_res && blockIdx.x == 0 && lane == 0) sp.ev_of_step[st] = -1;
  return do_res;
}

// Is step `s` resolved?  Warp-uniform result: 0 not yet, 1 yes (go on), 2 yes and it resamples.
// The first warp to find the step's grid barrier complete evaluates the ESS.
__device__ __noinline__ int check_resolved(const SweepParams& sp, SweepSmem& sm, int s) {
  if (s < 0) return 1;
  const int lane = threadIdx.x & 31;
  int r = 0;
  if (lane == 0) {
    const int rs = ld_vol(&sm.res_step);
    if (rs >= s) r = ld_vol(&sm.res_flag) ? 2 : 1;
    else if (rs == s - 1 && ld_vol(&sm.arrived) >= s &&
             ld_counter(sp) >= *(volatile unsigned long long*)&sm.q[s & 1].ep &&  // after `arrived`: never a stale epoch
             atomicCAS(&sm.res_claim, s - 1, s) == s - 1) r = 3;
  }
  r = __shfl_sync(FULL, r, 0);
  if (r == 3) {
    if (sp.R > 1) __threadfence_system(); else __threadfence();
    TRACE(s + 1, 9)
    double mxv;
    const bool res = resolve_ess(sp, s, &mxv);
    if (lane == 0) {
      sm.res_mx = mxv;
      st_vol(&sm.res_flag, res ? 1 : 0);
      __threadfence_block();
      st_vol(&sm.res_step, s);
    }
    __syncwarp();
    TRACE(s + 1, 10)
    r = res ? 2 : 1;
  }
  return r;
}

// The CTA's last particle of step t is folded: publish the CTA's ESS partial, start the copy of a
// later observation, arrive at the grid counter.  One warp.
__device__ __noinline__ void cta_arrive(const SweepParams& sp, const CtaTables& T, SweepSmem& sm, int ns, int t,
                                        unsigned char* xring) {
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
    double* ep = sp.ess_part + ((size_t)(t & 1) * sp.R * sp.G + (size_t)sp.rank * sp.G + blockIdx.x) * 3;
#pragma unroll 1
    for (int r = 0; r < sp.R; ++r) {  // every rank's copy of the partials (NVLink peer stores)
      double* e = on_rank(sp, ep, r);
      __stcg(e, m); __stcg(e + 1, s1); __stcg(e + 2, s2);
    }
    issue_obs(sp, t + PMDI_OBS_RING - 1, xring, sm.obs_bar);  // its ring slot held x[t-1]: free now
    sm.epoch += (unsigned long long)sp.R * sp.G;
    sm.q[t & 1].ep = sm.epoch;
    arrive_all(sp);
    st_vol(&sm.arrived, t);
  }
  __syncwarp();
}

// Proposal for one unit (dataset k, particle slot) at step `step`, by one warp: src/pmdi.jl:223-265;
// then the unit's items of the next step, the particle's weight fold, and the CTA's arrival.
// Written for a short instruction path (it sits between long streaming items).
__device__ __noinline__ void propose_unit(const SweepParams& sp, const CtaTables& T, SweepSmem& sm, int u, int step,
                                          int nu, int ns, unsigned char* xring) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int K = sp.K, N = sp.N, P = sp.P, par = step & 1;
  const int Npad = (N + 31) & ~31;
  const int k = T.uinfo[u] >> 24, slot = T.uinfo[u] & 0xFFFFFF;
  const DsDev& ds = sp.ds[k];
  const int p = T.ulog[u];
  double* lps = T.lp_s + (size_t)warp * Npad;  // lp[label], then f[label], then cumsum[label]
  const double lpe = __ldg(sp.lp_empty + (size_t)step * K + k);
  const int cnt = T.ucount[u];
  const int fe = T.pend[u] >= 0 ? T.pe[u] : -1;  // the row that ran as fused items: one partial per block
  const double* part = T.part + (size_t)par * T.cap + T.pbase[par * T.MU + u];
  unsigned* urow = T.urow + (size_t)u * N;
  const int J = ds.J, qb = sp.qb;
  double uu = 0.0;
  if (p != 0) uu = sp.tape_alloc ? __ldg(sp.tape_alloc + ((size_t)step * K + k) * P + p)
                                 : pm_uniform(sp.seed, sp.iter, DRAW_ALLOC, step, k, p);
#pragma unroll 1
  for (int m = lane; m < N; m += 32) lps[m] = lpe;
  __syncwarp();
#pragma unroll 1
  for (int e = lane; e < cnt; e += 32) {
    const unsigned ent = urow[e];
    double a = __ldg(ds.rc + (ent >> 8));
    const int stride = (e == fe) ? 1 : qb;
#pragma unroll 1
    for (int j = 0; j < J; j += stride) a += part[e * J + j];
    lps[ent & 0xFF] = a;
  }
  __syncwarp();
  double mx = -INFINITY;
#pragma unroll 1
  for (int m = lane; m < N; m += 32) {
    const double v = lps[m];
    mx = fmax(mx, v);
    if (sp.dbg_lp) sp.dbg_lp[(((size_t)step * K + k) * P + p) * N + m] = v;
  }
  mx = warp_max(mx);
  // f = exp(lp - max) * Pi ; sequential cumsum over labels (src/pmdi.jl:236-241)
#pragma unroll 1
  for (int m = lane; m < N; m += 32) lps[m] = pm_exp(lps[m] - mx) * T.Pi_s[k * N + m];
  __syncwarp();
  if (lane == 0) {
    double run = 0.0;
#pragma unroll 1
    for (int m = 0; m < N; ++m) { run += lps[m]; lps[m] = run; }
  }
  __syncwarp();
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
      const unsigned b = __ballot_sync(FULL, hit);
      if (b) { label = m0 + __ffs(b) - 1; break; }
    }
  }
  // bookkeeping of the chosen row: size, occupied-row list, pending add
  int pos = -1;
#pragma unroll 1
  for (int e0 = 0; e0 < cnt; e0 += 32) {
    const int e = e0 + lane;
    const bool hit = (e < cnt) && ((int)(urow[e] & 0xFF) == label);
    const unsigned b = __ballot_sync(FULL, hit);
    if (b) { pos = e0 + __ffs(b) - 1; break; }
  }
  if (lane == 0) {
    int n_new = 1;
    if (pos >= 0) {
      const unsigned ent = urow[pos] + (1u << 8);
      urow[pos] = ent;
      n_new = (int)(ent >> 8);
    } else {
      urow[cnt] = (unsigned)label | (1u << 8);
      T.ucount[u] = cnt + 1;
    }
    ds.n[(long long)slot * N + label] = n_new;
    T.pend[u] = label | (n_new << 8);
    T.pe[u] = pos >= 0 ? pos : cnt;
#pragma unroll 1
    for (int r = 0; r < sp.R; ++r)  // every rank back-traces the selected particle's lineage itself
      *on_rank(sp, sp.alloc_log + ((size_t)step * K + k) * P + p, r) = (uint8_t)label;
    if (sp.dbg_alloc) sp.dbg_alloc[((size_t)step * K + k) * P + p] = label + 1;
    atomicAdd(&sm.rows_eval[k], (unsigned)cnt);
  }
  __syncwarp();
  // ---- the unit's items of step + 1 go to the other queue right away
  {
    StepQ& qn = sm.q[par ^ 1];
    const int nb = par ^ 1;
    int ib = 0, nI = 0, nB = 0;
    if (lane == 0) {
      while (ld_vol(&qn.gen) != step + 1 && !ld_vol(&sm.fail)) __nanosleep(32);
      if (step + 1 < sp.steps) {
        unit_item_counts(sp, T, u, nI, nB);
        ib = atomicAdd(&qn.tail, nI);
        const int pb = atomicAdd(&qn.part_tail, nB);
        T.remaining[nb * T.MU + u] = nI;
        T.pbase[nb * T.MU + u] = pb;
        if (ib + nI > T.cap || pb + nB > T.cap) { atomicExch(sp.err, 78); st_vol(&sm.fail, 1); nI = 0; }
      }
      __threadfence_block();
    }
    ib = __shfl_sync(FULL, ib, 0);
    nI = __shfl_sync(FULL, nI, 0);
    if (nI > 0) write_unit_items(sp, T, u, nI, T.items + (size_t)nb * T.cap + ib);
    __threadfence_block();
    __syncwarp();
    if (lane == 0) atomicAdd(&qn.units_in, 1);
  }
  // ---- weight increment; the K-th proposal of the particle folds its log-weight
  const double inc = pm_log(tot) + mx;
  int last_particle = 0;
  if (lane == 0) {
    const int sl = u / K;
    T.inc_s[(par * ns + sl) * K + k] = inc;
    T.lab_s[(par * ns + sl) * K + k] = label;
    __threadfence_block();
    if (atomicAdd(&T.pcount[par * ns + sl], 1) == K - 1) {
      __threadfence_block();
      T.pcount[par * ns + sl] = 0;
      const volatile double* iv = T.inc_s + (size_t)(par * ns + sl) * K;
      const volatile int* lv = T.lab_s + (size_t)(par * ns + sl) * K;
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
#pragma unroll 1
      for (int r = 0; r < sp.R; ++r) __stcg(on_rank(sp, sp.lw + p, r), w);  // every rank plans the resampling
      if (sp.dbg_lw) sp.dbg_lw[(size_t)step * P + p] = w;
      __threadfence_block();
      last_particle = (atomicAdd(&sm.q[par].pdone, 1) == ns - 1) ? 1 : 0;
    }
  }
  last_particle = __shfl_sync(FULL, last_particle, 0);
  if (last_particle) {
    if (lane == 0) sm.q[par].pdone = 0;
    __threadfence_block();
    TRACE(step, 7)
    cta_arrive(sp, T, sm, ns, step, xring);
  }
}

// Resampling after step `st` (draw_partstar src/misc.jl:27-47 by CTA 0, then every CTA moves the
// duplicated particles' rows, src/pmdi.jl:318-341 in dense form): two blocking grid barriers.
// All threads of the CTA; every pending add has been applied.
__device__ __noinline__ bool do_resample(const SweepParams& sp, const CtaTables& T, SweepSmem& sm, int nu, int ns,
                                         int st, int* s_tmp) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, NW = PMDI_NT / 32;
  const int cta = blockIdx.x, G = sp.G, K = sp.K, N = sp.N;
  const int ev = sm.ev;
  // every rank runs the plan on its own copy of the log-weights: same inputs, same plan
  if (cta == 0) resample_plan(sp, st, ev, sm.res_mx, sp.lw, s_tmp);
  if (!grid_sync(sp, sm)) return false;
  const int ncopy = ldcg_i32(sp.plan_out);
  const int gw = cta * NW + warp, GW = G * NW;
#pragma unroll 1
  for (int idx = gw; idx < ncopy * K * N; idx += GW) {
    const int c = idx / (K * N), rem = idx - c * (K * N);
    const int k = rem / N, m = rem - k * N;
    const int2 cp = __ldcg(sp.copies + c);  // (source, destination) as GLOBAL slots
    const int dl = cp.y - sp.slot0;
    if (dl < 0 || dl >= sp.Ps) continue;     // the rank that holds the destination pulls the row
    const int sr = cp.x / sp.Ps, sl = cp.x - sr * sp.Ps;
    if (sr != sp.rank && lane == 0) atomicAdd((unsigned long long*)&sp.counters[3], 1ull);  // pulled over NVLink
    row_copy(sp.ds[k], sp.peer_delta[sr], (long long)sl * N + m, (long long)dl * N + m, lane);
  }
  for (int sl = tid; sl < ns; sl += PMDI_NT) T.lw_s[sl] = 1.0;  // logweight .= 1.0 (src/pmdi.jl:319)
  if (cta == 0 && tid == 0) { sp.counters[0] += 1; sp.counters[1] += ncopy; }
  if (!grid_sync(sp, sm)) return false;
  if (tid == 0) sm.ev = ev + 1;
  rebuild_rows(sp, T, nu, ev + 1);
  __syncthreads();
  return true;
}

#ifndef PMDI_USER_TYPES  // the dense engine has no user-type hooks: not part of a run-time compiled program
extern "C" __global__ void __launch_bounds__(PMDI_NT, 1) k_sweep(const __grid_constant__ SweepParams sp) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(16) SweepSmem sm;
  __shared__ int s_tmp[PMDI_NT + 2];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int NW = PMDI_NT / 32;
  const int cta = blockIdx.x;
  const int K = sp.K, N = sp.N, steps = sp.steps;
  const int Npad = (N + 31) & ~31;

  // dynamic shared memory: [4 x observation][lf table][lp scratch][Pi][lw][inc][part x2][items x2][tables]
  unsigned char* xring = smem_raw;
  double* lf = (double*)(smem_raw + (size_t)PMDI_OBS_RING * sp.sm_x_bytes);
  const int u0 = sp.cta_off[cta], nu = sp.cta_off[cta + 1] - u0;
  const int ns = nu / K;  // particle slots owned by this CTA
  const int MU = sp.max_units, MS = MU / K;
  CtaTables T;
  T.MU = MU; T.cap = sp.item_cap;
  T.lp_s = lf + sp.lf_T;
  T.Pi_s = T.lp_s + (size_t)NW * Npad;
  T.lw_s = T.Pi_s + (size_t)K * N;
  T.inc_s = T.lw_s + MS;
  T.part = T.inc_s + 2 * (size_t)MU;
  T.items = (unsigned*)(T.part + 2 * (size_t)T.cap);
  T.urow = T.items + 2 * (size_t)T.cap;
  T.ucount = (int*)(T.urow + (size_t)MU * N);
  T.uinfo = T.ucount + MU;
  T.ulog = T.uinfo + MU;
  T.pend = T.ulog + MU;
  T.pe = T.pend + MU;
  T.ustate = T.pe + MU;
  T.remaining = T.ustate + MU;
  T.pbase = T.remaining + 2 * MU;
  T.lab_s = T.pbase + 2 * MU;
  T.pcount = T.lab_s + 2 * MU;
  const int lfT = sp.lf_T;
  for (int i = tid; i < lfT; i += PMDI_NT) lf[i] = sp.lf_glob[i];
  for (int i = tid; i < K * N; i += PMDI_NT) T.Pi_s[i] = sp.Pi[i];
  for (int sl = tid; sl < ns; sl += PMDI_NT) T.lw_s[sl] = sp.lw_init;
  if (tid < PMDI_MAX_K) sm.rows_eval[tid] = 0;
  if (tid < 8) sm.tacc[tid] = 0;
  for (int u = tid; u < nu; u += PMDI_NT) T.uinfo[u] = sp.cta_units[u0 + u];
  if (tid == 0) {
    sm.res_step = -1; sm.res_claim = -1; sm.res_flag = 0; sm.arrived = -1; sm.fail = 0; sm.ev = 0;
    sm.epoch = 0; sm.res_mx = 0.0;
    for (int b = 0; b < PMDI_OBS_RING; ++b) mbar_init(&sm.obs_bar[b], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid == 0)
    for (int s = 0; s < PMDI_OBS_RING - 1; ++s) issue_obs(sp, s, xring, sm.obs_bar);
  rebuild_rows(sp, T, nu, 0);
  __syncthreads();
  init_queues(sp, T, sm, nu, ns, 0);
  if (sm.fail) return;

  const bool timing = sp.phase_ns != nullptr;
  unsigned long long tw_prev = timing ? globaltimer_ns() : 0ull;
#define PHASE_MARK(i_)                                                 \
  if (timing && lane == 0) {                                           \
    const unsigned long long now_ = globaltimer_ns();                  \
    atomicAdd(&sm.tacc[i_], now_ - tw_prev);                           \
    tw_prev = now_;                                                    \
  }

  int t = 0;        // the step whose list this warp is working on
  int obs_ok = -1;  // observations this warp has seen land
  while (t <= steps) {
    StepQ& q = sm.q[t & 1];
    // ---- get a ticket for step t's list, then wait for the item (or for the list to close)
    unsigned code = PMDI_ITEM_INVALID;
    int what = 0;  // 1 run item, 2 leave the list, 3 resampling rendezvous, 4 abort
    int h = -1;
    unsigned idle_spins = 0;
    unsigned long long idle_t0 = 0;
    for (;;) {
      if (lane == 0) {
        what = 0;
        if (((++idle_spins) & 0xffu) == 0) {  // watchdog: a lost CTA / warp becomes an error, not a hang
          const unsigned long long now = globaltimer_ns();
          if (idle_t0 == 0) idle_t0 = now;
          if (__ldcg(sp.err) != 0) st_vol(&sm.fail, 1);
          else if (now - idle_t0 > sp.wd_ns) { atomicExch(sp.err, 79); st_vol(&sm.fail, 1); }
        }
        if (ld_vol(&sm.fail)) what = 4;
        else if (ld_vol(&sm.res_flag) && t == ld_vol(&sm.res_step) + 2) what = 3;
        else if (ld_vol(&q.gen) == t) {
          if (h < 0) h = atomicAdd(&q.head, 1);
          if (h < T.cap) code = *(volatile unsigned*)(T.items + (size_t)(t & 1) * T.cap + h);
          if (code != PMDI_ITEM_INVALID) {
            *(volatile unsigned*)(T.items + (size_t)(t & 1) * T.cap + h) = PMDI_ITEM_INVALID;
            what = 1;
          } else if (ld_vol(&q.units_in) == nu && h >= ld_vol(&q.tail)) {
            what = 2;
          }
        }
      }
      what = __shfl_sync(FULL, what, 0);
      if (what) break;
      // ---- idle: a parked unit whose gate has opened?
      // the parked unit of the EARLIEST step: parked units can be one step apart (one still waiting
      // to be picked up with its gate open, others already through the next step's items), and
      // only the earlier one can make progress
      int pu = -1, pstep = 0;
      {
        int best = 0x7fffffff, best_u = -1;
#pragma unroll 1
        for (int ub = 0; ub < nu; ub += 32) {
          const int u = ub + lane;
          const int st = (u < nu) ? ld_vol(&T.ustate[u]) : 0;
          if (st != 0 && st < best) { best = st; best_u = u; }
        }
        int mn = best;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(FULL, mn, o));
        if (mn != 0x7fffffff) {
          const unsigned b = __ballot_sync(FULL, best == mn);
          pu = __shfl_sync(FULL, best_u, __ffs(b) - 1);
          pstep = mn - 1;
        }
      }
      if (pu >= 0) {
        const int r = check_resolved(sp, sm, pstep - 1);
        if (r) {
          int won = 0;
          if (lane == 0) won = atomicCAS(&T.ustate[pu], pstep + 1, 0) == pstep + 1;
          won = __shfl_sync(FULL, won, 0);
          if (won && r == 1) {
            PHASE_MARK(0)
            TRACE(pstep, 4)
            propose_unit(sp, T, sm, pu, pstep, nu, ns, xring);
            TRACE(pstep, 5)
            PHASE_MARK(2)
          }
        } else {
          __nanosleep(100);
        }
      } else {
        __nanosleep(40);
      }
    }
    PHASE_MARK(0)
    if (what == 4) {
      if (lane == 0 && sp.wd_state) {  // post-mortem of a watchdog: where every warp was
        int* w = sp.wd_state + ((size_t)cta * NW + warp) * 16;
        w[0] = t; w[1] = h; w[2] = q.gen; w[3] = q.head; w[4] = q.tail; w[5] = q.units_in; w[6] = q.left;
        w[7] = sm.res_step; w[8] = sm.res_flag; w[9] = sm.arrived; w[10] = sm.res_claim; w[11] = nu;
        int parked = 0;
        for (int u = 0; u < nu; ++u) parked += T.ustate[u] != 0;
        w[12] = parked; w[13] = sm.q[(t & 1) ^ 1].gen; w[14] = sm.q[(t & 1) ^ 1].units_in; w[15] = sm.q[t & 1].pdone;
      }
      return;
    }
    if (what == 1) {
      code = __shfl_sync(FULL, code, 0);
      __threadfence_block();  // the item's rows were written by other warps of this CTA
      if (obs_ok < t) {  // x[t] (and x[t-1] before it) have landed in the ring
        if (lane == 0) {
#pragma unroll 1
          for (int s = max(obs_ok + 1, t - 1); s <= t; ++s)
            while (!mbar_try_wait(&sm.obs_bar[s % PMDI_OBS_RING], (unsigned)(s / PMDI_OBS_RING) & 1u)) {}
        }
        __syncwarp();
        obs_ok = t;
      }
      TRACE(t, 0x100 | (code & 31) | (((code >> 5) & 7) << 5) | ((T.uinfo[(code >> 13) & 0x3FFFF] >> 24) << 12) | ((code >> 31) << 11))
      const double v = run_item(sp, T, code, xring + (size_t)(t % PMDI_OBS_RING) * sp.sm_x_bytes,
                                xring + (size_t)((t + PMDI_OBS_RING - 1) % PMDI_OBS_RING) * sp.sm_x_bytes, lf);
      TRACE(t, 3)
      PHASE_MARK(1)
      const int u = (code >> 13) & 0x3FFFF;
      int last = 0;
      if (lane == 0) {
        const int b = t & 1;
        T.part[(size_t)b * T.cap + T.pbase[b * MU + u] + ((code >> 5) & 0xFF) * sp.ds[T.uinfo[u] >> 24].J + (code & 31)] = v;
        __threadfence_block();
        last = atomicSub(&T.remaining[b * MU + u], 1) == 1;
      }
      last = __shfl_sync(FULL, last, 0);
      if (last) {  // this warp finished the unit's items of step t
        __threadfence_block();
        const int r = check_resolved(sp, sm, t - 1);
        if (r == 1) {
          TRACE(t, 4)
          propose_unit(sp, T, sm, u, t, nu, ns, xring);
          TRACE(t, 5)
          PHASE_MARK(2)
        } else if (r == 0) {
          if (lane == 0) st_vol(&T.ustate[u], 1 + t);  // parked until step t-1 is resolved
        }
      }
      continue;
    }
    if (what == 2) {  // done with step t's list
      TRACE(t, 6)
      if (lane == 0) {
        if (atomicAdd(&q.left, 1) == NW - 1) {  // last warp out: the buffer now serves step t + 2
          q.head = 0; q.tail = 0; q.units_in = 0; q.part_tail = 0; q.left = 0;
          __threadfence_block();
          st_vol(&q.gen, t + 2);
        }
      }
      __syncwarp();
      if (!(ld_vol(&sm.res_flag) && t == ld_vol(&sm.res_step) + 1)) { ++t; continue; }
      what = 3;  // this list was the drain pass of a resampling step
    }
    // ---- what == 3: resampling after step sm.res_step; every warp of the CTA comes here
    __syncthreads();
    const int st = sm.res_step;
    if (!do_resample(sp, T, sm, nu, ns, st, s_tmp)) return;
    init_queues(sp, T, sm, nu, ns, st + 1);
    if (tid == 0) sm.res_flag = 0;
    __syncthreads();
    if (sm.fail) return;
    t = st + 1;
    PHASE_MARK(6)
  }
  // ------------------------------------------------------------------ weights of the last step
  __syncthreads();
  {
    const int st = steps - 1;
    if (warp == 0) {
      if (lane == 0 && !bar_wait(sp, sm.q[st & 1].ep)) sm.fail = 1;
      __syncwarp();
      if (sm.res_step < st) {
        double mxv;
        const bool r = resolve_ess(sp, st, &mxv);
        if (lane == 0) { sm.res_mx = mxv; sm.res_flag = r ? 1 : 0; sm.res_step = st; }
      }
    }
    __syncthreads();
    if (sm.fail) return;
    if (sm.res_flag) {
      flush_adds(sp, T, nu, xring + (size_t)(st % PMDI_OBS_RING) * sp.sm_x_bytes, lf);
      if (!do_resample(sp, T, sm, nu, ns, st, s_tmp)) return;
    }
  }
  __syncthreads();
  if (tid < K) atomicAdd(sp.rows_eval + tid, (unsigned long long)sm.rows_eval[tid]);
  if (cta == 0)  // every rank holds all P log-weights; after a final resampling they are all 1.0 (:319)
    for (int p = tid; p < sp.P; p += PMDI_NT) sp.lw_out[p] = sm.res_flag ? 1.0 : __ldcg(sp.lw + p);
  if (timing && tid < 8) sp.phase_ns[(size_t)cta * 8 + tid] = sm.tacc[tid] / NW;
  if (cta == 0 && tid == 0) sp.counters[2] = sm.ev;
}
#endif
#undef PHASE_MARK
#undef TRACE
