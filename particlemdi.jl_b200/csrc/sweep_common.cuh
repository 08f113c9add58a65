// What the three sweep engines share (sweep_kernel.cuh dense, pool_kernel.cuh pool, spec_kernel.cuh spec): acquire
// loads, the peer-arena pointer and the mbarriers of the shared-memory observation ring; for pool and spec also the
// ring's bulk copy, the resampling plan, the event trace and the cross-rank barrier.  The non-inlined functions keep
// the names they had in pool_kernel.cuh: ptxas lays out a kernel's non-inlined callees in an order that follows their
// names, so renaming one changes the code of every kernel that calls it.
#pragma once
#include "device_utils.cuh"

#define PMDI_NW (PMDI_NT / 32)  // warps per CTA of the sweep kernels

__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
// the same object in rank r's shared arena (r == own rank: the pointer itself)
template <class T>
__device__ __forceinline__ T* on_rank(const SweepParams& sp, T* p, int r) {
  return (T*)((char*)p + sp.peer_delta[r]);
}

// ---- mbarrier / TMA bulk copy (observation ring) -----------------------------------------------
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
      : "=r"(ok) : "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
  return ok != 0;
}

#ifndef PMDI_X_GLOBAL  // (the wide kernels read the observation from global memory: no ring)
// pool and spec: one thread bulk-copies the K rows of the observation swept at `step` into its ring slot
__device__ __noinline__ void pool_issue_obs(const SweepParams& sp, int step, unsigned char* xring,
                                            unsigned long long* bars) {
  if (step >= sp.steps) return;
  const int b = step % sp.obs_ring;
  const unsigned bar = (unsigned)__cvta_generic_to_shared(bars + b);
  const int obs = sp.order[sp.n1 - 1 + step];
  unsigned total = 0;
#pragma unroll 1
  for (int k = 0; k < sp.K; ++k) total += (unsigned)sp.ds[k].Dp * PMDI_XBYTES(sp.ds[k]);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // earlier generic reads of the slot
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(total) : "memory");
#pragma unroll 1
  for (int k = 0; k < sp.K; ++k) {
    const DsDev& ds = sp.ds[k];
    const unsigned bytes = (unsigned)ds.Dp * PMDI_XBYTES(ds);
    const unsigned char* src = (const unsigned char*)ds.xstage + (size_t)obs * bytes;
    const unsigned dst = (unsigned)__cvta_generic_to_shared(xring + (size_t)b * sp.sm_x_bytes + ds.x_off);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
  }
}
#endif

// pool and spec: optional per-warp event trace of one CTA and one step (PMDI_TRACE_STEP): tag << 48 | clock64; stores
// only.  Smem: the engine's shared-memory struct (tr_n[PMDI_NW]: events per warp).
template <class Smem>
__device__ __forceinline__ void sweep_trace(const SweepParams& sp, Smem& sm, int step, unsigned tag) {
  if (sp.trace && step == sp.trace_step && (int)blockIdx.x == sp.trace_cta && (threadIdx.x & 31) == 0) {
    const int w = threadIdx.x >> 5;
    const int n = ++sm.tr_n[w];
    if (n < 128) {
      sp.trace[w * 128 + n] = ((unsigned long long)tag << 48) | (clock64() & 0xFFFFFFFFFFFFull);
      sp.trace[w * 128] = n;
    }
  }
}
// the trace in the instrumented kernel instantiations only (template parameter DBG)
#define SWEEP_TRACE(step_, tag_) if constexpr (DBG) sweep_trace(sp, sm, (step_), (tag_));

// pool and spec: barrier over the CTAs of ALL ranks: local barrier (peer stores made visible system-wide), one arrival
// per rank on every rank's counter (NVLink peer atomics), local barrier.  Resampling and the end of the sweep.
// gsync(sys) is the engine's local grid barrier; sys: this CTA's peer stores are made visible system-wide before it
// arrives.  Inlined into a non-inlined function of each engine (pool_xsync, spec_xsync), which keeps its name.
template <class Smem, class Gsync>
__device__ __forceinline__ bool sweep_xsync(const SweepParams& sp, Smem& sm, Gsync gsync) {
  if (!gsync(sp.R > 1)) return false;
  if (sp.R > 1) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      unsigned long long* xbar = (unsigned long long*)sp.bar + 1;
      sm.xepoch += (unsigned long long)sp.R;
      __threadfence_system();
#pragma unroll 1
      for (int r = 0; r < sp.R; ++r) atomicAdd_system(on_rank(sp, xbar, r), 1ull);
      const unsigned long long t0 = globaltimer_ns();
      unsigned spins = 0;
#pragma unroll 1
      while (ld_acquire_sys_u64(xbar) < sm.xepoch) {
        if (((++spins) & 0x3ffu) == 0) {
          if (__ldcg(sp.err) != 0) break;
          if (globaltimer_ns() - t0 > sp.wd_ns) { atomicExch(sp.err, 77); break; }
        }
      }
      __threadfence_system();
    }
    if (!gsync(false)) return false;
  }
  return true;
}

// pool and spec: draw_partstar (src/misc.jl:27-47) by one CTA, all threads: anc_log[ev][P] (1-based, non-decreasing,
// anc[0] == 1).  The Fisher-Yates shuffle followed by partstar[1]=1 and sort! only decides WHICH element of the
// sorted systematic sample the reference particle replaces: the one the shuffle moves to position 1; that index is
// traced through the swaps without moving anything.
// Scratch of the plan (P entries each): global memory, or the calling CTA's shared memory when it has room.
struct PlanScratch { double *w, *pp, *u; int *j, *a0; };
__device__ __noinline__ void pool_resample_plan(const SweepParams& sp, int step, int ev, double mx, int* s_tmp,
                                                const double* lw, const PlanScratch sc) {
  if (!lw) lw = sp.lw;  // (the spec engine keeps two copies of the log-weights, by step parity)
  const int P = sp.P, t = threadIdx.x;
#pragma unroll 1
  for (int p = t; p < P; p += PMDI_NT) {
    sc.w[p] = pm_exp(__ldcg(on_rank(sp, lw + p, p / sp.Ps)) - mx);  // the holder's copy (NVLink when remote)
    const double us = sp.tape_shuffle ? sp.tape_shuffle[(size_t)step * P + p]
                                      : pm_uniform(sp.seed, sp.iter, DRAW_SHUFFLE, step, 0, p);
    int jj = 1 + (int)floor(us * (double)(p + 1));
    if (jj > p + 1) jj = p + 1;
    sc.j[p] = jj;
  }
  __syncthreads();
  if (t == 0) {  // pprob = cumsum(exp.(logweight .- max)), sequential (misc.jl:29); loads sixteen ahead of the adds
    double acc = 0.0;
    int p = 0;
#pragma unroll 1
    for (; p + 16 <= P; p += 16) {
      double v[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = sc.w[p + i];
#pragma unroll
      for (int i = 0; i < 16; ++i) { acc += v[i]; sc.pp[p + i] = acc; }
    }
#pragma unroll 1
    for (; p < P; ++p) { acc += sc.w[p]; sc.pp[p] = acc; }
  } else if (t == 32) {  // u, u + 1/P, ... by repeated addition (misc.jl:28,35)
    const double r = sp.tape_resamp ? sp.tape_resamp[step] : pm_uniform(sp.seed, sp.iter, DRAW_RESAMP, step, 0, 0);
    double u = r / (double)P;
#pragma unroll 1
    for (int i = 0; i < P; ++i) { sc.u[i] = u; u += 1.0 / (double)P; }
  } else if (t == 64) {  // index of the pre-shuffle element that ends at position 1
    int tt = 0, pos = 2;
#pragma unroll 1
    for (; pos + 15 <= P; pos += 16) {
      int v[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = sc.j[pos - 1 + i];
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (v[i] - 1 == tt) tt = pos - 1 + i;
    }
#pragma unroll 1
    for (; pos <= P; ++pos)
      if (sc.j[pos - 1] - 1 == tt) tt = pos - 1;
    s_tmp[0] = tt;
  }
  __syncthreads();
  const double tot = sc.pp[P - 1];
#pragma unroll 1
  for (int i = t; i < P; i += PMDI_NT) {  // first p with pprob[p]/last >= u_i (misc.jl:33-38)
    const double ui = sc.u[i];
    int lo = 0, hi = P;
#pragma unroll 1
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (pm_div(sc.pp[mid], tot) >= ui) hi = mid; else lo = mid + 1;
    }
    sc.a0[i] = (lo < P) ? lo + 1 : P;
  }
  __syncthreads();
  const int drop = s_tmp[0];
  int* anc = sp.anc_log + (size_t)ev * P;
#pragma unroll 1
  for (int i = t; i < P; i += PMDI_NT) {
    const int a = (i == 0) ? 1 : ((i - 1 < drop) ? sc.a0[i - 1] : sc.a0[i]);
    anc[i] = a;
    if (sp.dbg_anc) sp.dbg_anc[(size_t)step * P + i] = a;
  }
  __syncthreads();
  int dup = 0;  // particles that duplicate their predecessor's ancestor (a statistic)
#pragma unroll 1
  for (int i = 1 + t; i < P; i += PMDI_NT) dup += anc[i] == anc[i - 1];
  if (dup) atomicAdd((unsigned long long*)&sp.counters[1], (unsigned long long)dup);
  if (t == 0) {
    sp.ev_of_step[step] = ev;
    sp.counters[0] += 1;
  }
}
