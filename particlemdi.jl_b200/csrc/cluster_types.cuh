// The three built-in cluster types of ParticleMDI as warp-level device operators over one
// 256-feature block of one cluster row.  Each operator is what the reference's plugin contract
// computes (calc_logprob / cluster_add!), restructured for HBM streaming:
//   * everything that does not depend on the observation is hoisted out of the predictive into
//     aux[row][block] (maintained by the add) and rc[n] (host-built table by cluster size);
//   * sums of logs become logs of short products (<= 8 factors per lane, no overflow for any
//     statistic the add can produce), so the FP64 pipe stays far below the HBM time;
//   * lgamma at integer arguments is a shared-memory log-factorial table.
// Lane l of a warp owns features {64*it + 2*l, 64*it + 2*l + 1 : it = 0..3} of the block: one
// 128-bit load per statistic array per iteration, 512 contiguous bytes per warp.
#pragma once
#include "device_utils.cuh"



// ------------------------------------------------------------------------------------------
// Gaussian — reference src/datatypes/gaussian_cluster.jl:37-52 (calc_logprob), :54-66 (cluster_add!)
//   log p = nflag*rc_n + sum_q flag_q [ 0.5 log(lam_q/(n+1)) - (n/2+1) log(1 + (x_q-mu_q)^2 lam_q/(n+1)) ]
// stored: mu, lamn = lam/(n+1); aux = sum_q 0.5 log(lamn_q) per block.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double gauss_eval_block(const DsDev& ds, long long row, int j, int n,
                                                   const double* xs, int lane) {
  const int q0 = j * ds.FB;
  const int nit = min(ds.FB / PMDI_WF, (ds.Dp - q0) / PMDI_WF);
  const double* mu = ds.mu + row * ds.Dp + q0 + 2 * lane;
  const double* lm = ds.lamn + row * ds.Dp + q0 + 2 * lane;
  double2 m[4], l[4];
#pragma unroll
  for (int it = 0; it < 4; ++it)
    if (it < nit) {
      m[it] = ldcg_f64x2(mu + it * PMDI_WF);
      l[it] = ldcg_f64x2(lm + it * PMDI_WF);
    }
  double prod = 1.0;
#pragma unroll
  for (int it = 0; it < 4; ++it)
    if (it < nit) {
      const double2 x = *(const double2*)(xs + q0 + it * PMDI_WF + 2 * lane);
      const double d0 = x.x - m[it].x, d1 = x.y - m[it].y;
      double f0 = fma(d0 * d0, l[it].x, 1.0), f1 = fma(d1 * d1, l[it].y, 1.0);
      if (!ds.all_on) {
        const uchar2 fl = *(const uchar2*)(ds.flag + q0 + it * PMDI_WF + 2 * lane);
        f0 = fl.x ? f0 : 1.0;
        f1 = fl.y ? f1 : 1.0;
      }
      prod *= f0 * f1;
    }
  const double s = warp_sum(log(prod));
  return ldcg_f64(ds.aux + row * ds.J + j) - (0.5 * (double)n + 1.0) * s;
}

// x / c for a row constant c with rc = RN(1/c): quotient, exact FMA residual, one correction
// (Markstein): the correctly rounded quotient without the full division sequence.
__device__ __forceinline__ double div_const(double x, double c, double rc) {
  const double q = x * rc;
  const double r = fma(-q, c, x);
  return fma(r, rc, q);
}

// cluster_add! in the operation order of gaussian_cluster.jl:57-63 (each quotient correctly
// rounded, no FMA contraction across the reference's operations), so the stored statistics follow
// the reference's to the bit; n is the size AFTER the add.  The new aux (sum of 0.5 log lamn over
// the flagged features) is taken as one log of the lane's product of <= 8 factors.
__device__ __noinline__ void gauss_add_block(const DsDev& ds, long long row, int j, int n,
                                                const double* xs, int lane) {
  const int q0 = j * ds.FB;
  const int nit = min(ds.FB / PMDI_WF, (ds.Dp - q0) / PMDI_WF);
  const double nn = (double)n;
  const double c1 = __dadd_rn(__dadd_rn(nn, -1.0), 0.001);      // n - 1 + kappa
  const double c2 = __dmul_rn(2.0, __dadd_rn(nn, 0.001));       // 2 (n + kappa)
  const double c3 = __dadd_rn(nn, 0.001);                       // n + kappa
  const double c4 = __dmul_rn(__dadd_rn(__dmul_rn(0.5, nn), 0.5), c3);  // (n/2 + 1/2)(n + kappa)
  const double c5 = __dadd_rn(nn, 1.001);                       // n + 1 + kappa
  const double c6 = __dadd_rn(nn, 1.0);
  const double r2 = __drcp_rn(c2), r3 = __drcp_rn(c3), r6 = __drcp_rn(c6);
  const long long base = row * ds.Dp + q0 + 2 * lane;
  double2 sm[4], bt[4], mu[4], ln[4];
#pragma unroll
  for (int it = 0; it < 4; ++it)
    if (it < nit) {
      const long long o = base + it * PMDI_WF;
      sm[it] = ldcg_f64x2(ds.sum + o); bt[it] = ldcg_f64x2(ds.beta + o);
      mu[it] = ldcg_f64x2(ds.mu + o); ln[it] = ldcg_f64x2(ds.lamn + o);
    }
  double prod = 1.0;
#pragma unroll
  for (int it = 0; it < 4; ++it)
    if (it < nit) {
      const long long o = base + it * PMDI_WF;
      const double2 x = *(const double2*)(xs + q0 + it * PMDI_WF + 2 * lane);
      // padded features carry flag 0: they must not enter aux
      const uchar2 fl = *(const uchar2*)(ds.flag + q0 + it * PMDI_WF + 2 * lane);
      if (fl.x) {
        sm[it].x = __dadd_rn(sm[it].x, x.x);
        const double dd = __dadd_rn(x.x, -mu[it].x);
        bt[it].x = __dadd_rn(bt[it].x, div_const(__dmul_rn(c1, __dmul_rn(dd, dd)), c2, r2));
        mu[it].x = div_const(sm[it].x, c3, r3);
        ln[it].x = div_const(__ddiv_rn(c4, __dmul_rn(bt[it].x, c5)), c6, r6);
        prod *= ln[it].x;
      }
      if (fl.y) {
        sm[it].y = __dadd_rn(sm[it].y, x.y);
        const double dd = __dadd_rn(x.y, -mu[it].y);
        bt[it].y = __dadd_rn(bt[it].y, div_const(__dmul_rn(c1, __dmul_rn(dd, dd)), c2, r2));
        mu[it].y = div_const(sm[it].y, c3, r3);
        ln[it].y = div_const(__ddiv_rn(c4, __dmul_rn(bt[it].y, c5)), c6, r6);
        prod *= ln[it].y;
      }
      *(double2*)(ds.sum + o) = sm[it];
      *(double2*)(ds.beta + o) = bt[it];
      *(double2*)(ds.mu + o) = mu[it];
      *(double2*)(ds.lamn + o) = ln[it];
    }
  const double acc = warp_sum(0.5 * pm_log(prod));
  if (lane == 0) ds.aux[row * ds.J + j] = acc;
}

// Fused cluster_add!(x_prev) + calc_logprob(x_cur) for the row a particle chose in the previous
// step: the row is read once, updated, written back and evaluated against the next observation
// in the same pass (same arithmetic as gauss_add_block followed by gauss_eval_block).
// (noinline with by-value arguments: its register allocation stays out of the item loop)
__device__ __noinline__ double gauss_fused_raw(double* sum_p, double* beta_p, double* mu_p, double* lamn_p,
                                               double* aux_p, const uint8_t* flag_p, int nit, int n,
                                               const double* xp, const double* xc, int lane) {
  const double nn = (double)n;
  const double c1 = __dadd_rn(__dadd_rn(nn, -1.0), 0.001);
  const double c2 = __dmul_rn(2.0, __dadd_rn(nn, 0.001));
  const double c3 = __dadd_rn(nn, 0.001);
  const double c4 = __dmul_rn(__dadd_rn(__dmul_rn(0.5, nn), 0.5), c3);
  const double c5 = __dadd_rn(nn, 1.001);
  const double c6 = __dadd_rn(nn, 1.0);
  const double r2 = __drcp_rn(c2), r3 = __drcp_rn(c3), r6 = __drcp_rn(c6);
  double prodl = 1.0, prode = 1.0;
#pragma unroll 1
  for (int h = 0; h < 4; h += 2) {
    double2 sm[2], bt[2], mu[2], ln[2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
      if (h + i < nit) {
        const int o = (h + i) * PMDI_WF;
        sm[i] = ldcg_f64x2(sum_p + o); bt[i] = ldcg_f64x2(beta_p + o);
        mu[i] = ldcg_f64x2(mu_p + o); ln[i] = ldcg_f64x2(lamn_p + o);
      }
#pragma unroll
    for (int i = 0; i < 2; ++i)
      if (h + i < nit) {
        const int o = (h + i) * PMDI_WF;
        const double2 x = *(const double2*)(xp + o);
        const double2 y = *(const double2*)(xc + o);
        const uchar2 fl = *(const uchar2*)(flag_p + o);
        if (fl.x) {
          sm[i].x = __dadd_rn(sm[i].x, x.x);
          const double dd = __dadd_rn(x.x, -mu[i].x);
          bt[i].x = __dadd_rn(bt[i].x, div_const(__dmul_rn(c1, __dmul_rn(dd, dd)), c2, r2));
          mu[i].x = div_const(sm[i].x, c3, r3);
          ln[i].x = div_const(__ddiv_rn(c4, __dmul_rn(bt[i].x, c5)), c6, r6);
          prodl *= ln[i].x;
          const double d = y.x - mu[i].x;
          prode *= fma(d * d, ln[i].x, 1.0);
        }
        if (fl.y) {
          sm[i].y = __dadd_rn(sm[i].y, x.y);
          const double dd = __dadd_rn(x.y, -mu[i].y);
          bt[i].y = __dadd_rn(bt[i].y, div_const(__dmul_rn(c1, __dmul_rn(dd, dd)), c2, r2));
          mu[i].y = div_const(sm[i].y, c3, r3);
          ln[i].y = div_const(__ddiv_rn(c4, __dmul_rn(bt[i].y, c5)), c6, r6);
          prodl *= ln[i].y;
          const double d = y.y - mu[i].y;
          prode *= fma(d * d, ln[i].y, 1.0);
        }
        *(double2*)(sum_p + o) = sm[i];
        *(double2*)(beta_p + o) = bt[i];
        *(double2*)(mu_p + o) = mu[i];
        *(double2*)(lamn_p + o) = ln[i];
      }
  }
  double a = 0.5 * pm_log(prodl), e = pm_log(prode);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(FULL, a, o);
    e += __shfl_xor_sync(FULL, e, o);
  }
  if (lane == 0) *aux_p = a;
  return a - (0.5 * nn + 1.0) * e;
}
__device__ __forceinline__ double gauss_fused_block(const DsDev& ds, long long row, int j, int n,
                                                    const double* xp, const double* xc, int lane) {
  const int q0 = j * ds.FB;
  const int nit = min(ds.FB / PMDI_WF, (ds.Dp - q0) / PMDI_WF);
  const long long o = row * ds.Dp + q0 + 2 * lane;
  return gauss_fused_raw(ds.sum + o, ds.beta + o, ds.mu + o, ds.lamn + o, ds.aux + row * ds.J + j,
                         ds.flag + q0 + 2 * lane, nit, n, xp + q0 + 2 * lane, xc + q0 + 2 * lane, lane);
}

// aux of a row from its stored state (used after the prefix build)
__device__ __forceinline__ void gauss_aux_block(const DsDev& ds, long long row, int j, int lane) {
  const int q0 = j * ds.FB;
  const int nit = min(ds.FB / PMDI_WF, (ds.Dp - q0) / PMDI_WF);
  double acc = 0.0;
  for (int it = 0; it < nit; ++it) {
    const int q = q0 + it * PMDI_WF + 2 * lane;
    const double2 ln = *(const double2*)(ds.lamn + row * ds.Dp + q);
    if (ds.flag[q]) acc += 0.5 * log(ln.x);
    if (ds.flag[q + 1]) acc += 0.5 * log(ln.y);
  }
  acc = warp_sum(acc);
  if (lane == 0) ds.aux[row * ds.J + j] = acc;
}

// ------------------------------------------------------------------------------------------
// Categorical — reference src/datatypes/categorical_cluster.jl:29-41, :43-51
//   log p = -sum_q flag_q log(nlevels_q + n)  [rc_n]  + sum_q flag_q log(0.5 + counts[x_q, q])
// The staged observation holds level 0 for unflagged / padded features.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double cat_eval_block(const DsDev& ds, long long row, int j,
                                                 const int* xs, int lane) {
  const int q0 = j * ds.FB;
  const int nit = min(ds.FB / PMDI_WF, (ds.Dp - q0) / PMDI_WF);
  const uint32_t* cnt = ds.cnt + row * (long long)ds.Lmax * ds.Dp;
  unsigned c[8];
  int2 lv[4];
#pragma unroll
  for (int it = 0; it < 4; ++it)
    if (it < nit) {
      const int q = q0 + it * PMDI_WF + 2 * lane;
      lv[it] = *(const int2*)(xs + q);
      c[2 * it] = lv[it].x ? ldcg_u32(cnt + (long long)(lv[it].x - 1) * ds.Dp + q) : 0u;
      c[2 * it + 1] = lv[it].y ? ldcg_u32(cnt + (long long)(lv[it].y - 1) * ds.Dp + q + 1) : 0u;
    }
  double prod = 1.0;
#pragma unroll
  for (int it = 0; it < 4; ++it)
    if (it < nit) {
      const double f0 = lv[it].x ? 0.5 + (double)c[2 * it] : 1.0;
      const double f1 = lv[it].y ? 0.5 + (double)c[2 * it + 1] : 1.0;
      prod *= f0 * f1;
    }
  return warp_sum(log(prod));
}

__device__ __noinline__ void cat_add_block(const DsDev& ds, long long row, int j, const int* xs,
                                              int lane) {
  const int q0 = j * ds.FB;
  const int nit = min(ds.FB / PMDI_WF, (ds.Dp - q0) / PMDI_WF);
  uint32_t* cnt = ds.cnt + row * (long long)ds.Lmax * ds.Dp;
  for (int it = 0; it < nit; ++it) {
    const int q = q0 + it * PMDI_WF + 2 * lane;
    const int2 lv = *(const int2*)(xs + q);
    if (lv.x) { uint32_t* p = cnt + (long long)(lv.x - 1) * ds.Dp + q; *p = ldcg_u32(p) + 1u; }
    if (lv.y) { uint32_t* p = cnt + (long long)(lv.y - 1) * ds.Dp + q + 1; *p = ldcg_u32(p) + 1u; }
  }
}

// ------------------------------------------------------------------------------------------
// NegBinom — reference src/datatypes/negbinom_cluster.jl:22-41, :43-51.  All lgamma arguments
// are integers (lf(k) = lgamma(k+1)):
//   term_q = lf(n+1) - lf(n) + [lf(n+1+S_q) - lf(S_q)] + [lf(x_q+S_q) - lf(n+2+x_q+S_q)]
//            \_ rc_n (nflag log(n+1)) _/ \________ aux ________/ \___ per observation ___/
// The staged observation holds -1 for unflagged / padded features.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double nb_eval_block(const DsDev& ds, long long row, int j, int n,
                                                const int* xs, int lane, const double* lf, int T) {
  const int q0 = j * ds.FB;
  const int nit = min(ds.FB / PMDI_WF, (ds.Dp - q0) / PMDI_WF);
  const long long* S = ds.S + row * ds.Dp + q0 + 2 * lane;
  longlong2 s[4];
#pragma unroll
  for (int it = 0; it < 4; ++it)
    if (it < nit) s[it] = ldcg_i64x2(S + it * PMDI_WF);
  double acc = 0.0;
#pragma unroll
  for (int it = 0; it < 4; ++it)
    if (it < nit) {
      const int2 x = *(const int2*)(xs + q0 + it * PMDI_WF + 2 * lane);
      if (x.x >= 0) { const long long a = s[it].x + x.x; acc += lfact(a, lf, T) - lfact(a + n + 2, lf, T); }
      if (x.y >= 0) { const long long a = s[it].y + x.y; acc += lfact(a, lf, T) - lfact(a + n + 2, lf, T); }
    }
  return ldcg_f64(ds.aux + row * ds.J + j) + warp_sum(acc);
}

// n is the size AFTER the add
__device__ __noinline__ void nb_add_block(const DsDev& ds, long long row, int j, int n,
                                             const int* xs, int lane, const double* lf, int T) {
  const int q0 = j * ds.FB;
  const int nit = min(ds.FB / PMDI_WF, (ds.Dp - q0) / PMDI_WF);
  long long* S = ds.S + row * ds.Dp + q0 + 2 * lane;
  double acc = 0.0;
  for (int it = 0; it < nit; ++it) {
    const int2 x = *(const int2*)(xs + q0 + it * PMDI_WF + 2 * lane);
    longlong2 s = ldcg_i64x2(S + it * PMDI_WF);
    if (x.x >= 0) { s.x += x.x; acc += lfact(s.x + n + 1, lf, T) - lfact(s.x, lf, T); }
    if (x.y >= 0) { s.y += x.y; acc += lfact(s.y + n + 1, lf, T) - lfact(s.y, lf, T); }
    *(longlong2*)(S + it * PMDI_WF) = s;
  }
  acc = warp_sum(acc);
  if (lane == 0) ds.aux[row * ds.J + j] = acc;
}

__device__ __forceinline__ void nb_aux_block(const DsDev& ds, long long row, int j, int n, int lane,
                                             const double* lf, int T) {
  const int q0 = j * ds.FB;
  const int nit = min(ds.FB / PMDI_WF, (ds.Dp - q0) / PMDI_WF);
  double acc = 0.0;
  for (int it = 0; it < nit; ++it) {
    const int q = q0 + it * PMDI_WF + 2 * lane;
    const longlong2 s = *(const longlong2*)(ds.S + row * ds.Dp + q);
    if (ds.flag[q]) acc += lfact(s.x + n + 1, lf, T) - lfact(s.x, lf, T);
    if (ds.flag[q + 1]) acc += lfact(s.y + n + 1, lf, T) - lfact(s.y, lf, T);
  }
  acc = warp_sum(acc);
  if (lane == 0) ds.aux[row * ds.J + j] = acc;
}

// ------------------------------------------------------------------------------------------
// Work items of the sweep: up to PMDI_QB consecutive 256-feature blocks [j0, j1) of one row, by
// one warp.  Loads run as a ROLLING prefetch four 64-feature iterations ahead: four named
// register slots are refilled one by one as they are consumed, so 6-8 128-bit loads per lane stay
// in flight for the whole item.  The x-independent aux terms are fetched by the first lanes at the
// start and the warp reduces once per item.  The evaluators are separate (noinline) functions
// with by-value arguments so that their prefetch registers are allocated independently of the
// persistent kernel's state; the staged observation is read with explicit ld.shared.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double2 lds_f64x2(unsigned a) {
  double2 v;
  asm("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ int2 lds_i32x2(unsigned a) {
  int2 v;
  asm("ld.shared.v2.s32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ double lds_f64(unsigned a) {
  double v;
  asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}

// How the pool and spec block operators (pool_types.cuh, user_type.cuh) address the observation.  By default it is
// staged in shared memory: PMDI_XADDR is a 32-bit shared address and the loads are ld.shared.  With PMDI_X_GLOBAL
// (the wide kernels, sweep_wide.cu: an observation too wide to stage) PMDI_XADDR is a byte pointer into
// DsDev::xstage and the loads are read-only global loads.  Without the macro the names expand to exactly the tokens
// the operators had before, so the staged kernels keep their code.
#ifdef PMDI_X_GLOBAL
#define PMDI_XADDR const unsigned char*
#define PMDI_LDX_F64X2(a_) __ldg((const double2*)(a_))
#define PMDI_LDX_I32X2(a_) __ldg((const int2*)(a_))
#else
#define PMDI_XADDR unsigned
#define PMDI_LDX_F64X2(a_) lds_f64x2(a_)
#define PMDI_LDX_I32X2(a_) lds_i32x2(a_)
#endif

// mu / lm / flag / xs point at this lane's first feature of the item; nits 64-feature iterations.
__device__ __noinline__ double gauss_eval_raw(const double* mu, const double* lm, const double* aux,
                                              const uint8_t* flag /* NULL: all on */, unsigned xs, int nits,
                                              int naux, int n, int lane) {
  double a = (lane < naux) ? ldcg_f64(aux + lane) : 0.0;
  double2 m0, m1, m2, m3, l0, l1, l2, l3;
  m0 = m1 = m2 = m3 = l0 = l1 = l2 = l3 = make_double2(0.0, 0.0);
  if (0 < nits) { m0 = ldcg_f64x2(mu); l0 = ldcg_f64x2(lm); }
  if (1 < nits) { m1 = ldcg_f64x2(mu + PMDI_WF); l1 = ldcg_f64x2(lm + PMDI_WF); }
  if (2 < nits) { m2 = ldcg_f64x2(mu + 2 * PMDI_WF); l2 = ldcg_f64x2(lm + 2 * PMDI_WF); }
  if (3 < nits) { m3 = ldcg_f64x2(mu + 3 * PMDI_WF); l3 = ldcg_f64x2(lm + 3 * PMDI_WF); }
  double acc = 0.0;
#define PMDI_G_STEP(M, L, IT)                                                         \
  if (i0 + IT < nits) {                                                               \
    const double2 x = lds_f64x2(xs + (IT) * PMDI_WF * 8);                             \
    const double d0 = x.x - M.x, d1 = x.y - M.y;                                      \
    double f0 = fma(d0 * d0, L.x, 1.0), f1 = fma(d1 * d1, L.y, 1.0);                  \
    if (flag) {                                                                       \
      const uchar2 fl = *(const uchar2*)(flag + (IT) * PMDI_WF);                      \
      f0 = fl.x ? f0 : 1.0;                                                           \
      f1 = fl.y ? f1 : 1.0;                                                           \
    }                                                                                 \
    prod *= f0 * f1;                                                                  \
    if (i0 + IT + 4 < nits) {                                                         \
      M = ldcg_f64x2(mu + (IT + 4) * PMDI_WF);                                        \
      L = ldcg_f64x2(lm + (IT + 4) * PMDI_WF);                                        \
    }                                                                                 \
  }
  for (int i0 = 0; i0 < nits; i0 += 4) {
    double prod = 1.0;
    PMDI_G_STEP(m0, l0, 0)
    PMDI_G_STEP(m1, l1, 1)
    PMDI_G_STEP(m2, l2, 2)
    PMDI_G_STEP(m3, l3, 3)
    acc += pm_log(prod);
    mu += PMDI_FB; lm += PMDI_FB; xs += PMDI_FB * 8;
    if (flag) flag += PMDI_FB;
  }
#undef PMDI_G_STEP
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(FULL, a, o);
    acc += __shfl_xor_sync(FULL, acc, o);
  }
  return a - (0.5 * (double)n + 1.0) * acc;
}
__device__ __forceinline__ double gauss_eval_item(const DsDev& ds, long long row, int j0, int j1, int n,
                                                  const double* xs, int lane) {
  const int base = j0 * PMDI_FB + 2 * lane;
  const int nits = (min(ds.Dp, j1 * PMDI_FB) - j0 * PMDI_FB) / PMDI_WF;
  return gauss_eval_raw(ds.mu + row * ds.Dp + base, ds.lamn + row * ds.Dp + base, ds.aux + row * ds.J + j0,
                        ds.all_on ? nullptr : ds.flag + base,
                        (unsigned)__cvta_generic_to_shared(xs + base), nits, j1 - j0, n, lane);
}

// log-factorial with the table in shared memory (address lf_s), Stirling beyond T
__device__ __forceinline__ double lfact_s(long long k, unsigned lf_s, int T) {
  if (k < (long long)T) return lds_f64(lf_s + (unsigned)k * 8u);
  return pm_lfact_stirling(k);
}

__device__ __noinline__ double nb_eval_raw(const long long* S, const double* aux, unsigned xs, int nits,
                                           int naux, int n, unsigned lf_s, int T, int lane) {
  double a = (lane < naux) ? ldcg_f64(aux + lane) : 0.0;
  longlong2 s0, s1, s2, s3;
  s0 = s1 = s2 = s3 = make_longlong2(0, 0);
  if (0 < nits) s0 = ldcg_i64x2(S);
  if (1 < nits) s1 = ldcg_i64x2(S + PMDI_WF);
  if (2 < nits) s2 = ldcg_i64x2(S + 2 * PMDI_WF);
  if (3 < nits) s3 = ldcg_i64x2(S + 3 * PMDI_WF);
  double acc = 0.0;
  const long long n2 = n + 2;
#define PMDI_NB_STEP(SS, IT)                                                                            \
  if (i0 + IT < nits) {                                                                                 \
    const int2 x = lds_i32x2(xs + (IT) * PMDI_WF * 4);                                                  \
    if (x.x >= 0) { const long long b = SS.x + x.x; acc += lfact_s(b, lf_s, T) - lfact_s(b + n2, lf_s, T); } \
    if (x.y >= 0) { const long long b = SS.y + x.y; acc += lfact_s(b, lf_s, T) - lfact_s(b + n2, lf_s, T); } \
    if (i0 + IT + 4 < nits) SS = ldcg_i64x2(S + (IT + 4) * PMDI_WF);                                    \
  }
  for (int i0 = 0; i0 < nits; i0 += 4) {
    PMDI_NB_STEP(s0, 0)
    PMDI_NB_STEP(s1, 1)
    PMDI_NB_STEP(s2, 2)
    PMDI_NB_STEP(s3, 3)
    S += PMDI_FB; xs += PMDI_FB * 4;
  }
#undef PMDI_NB_STEP
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(FULL, a, o);
    acc += __shfl_xor_sync(FULL, acc, o);
  }
  return a + acc;
}
__device__ __forceinline__ double nb_eval_item(const DsDev& ds, long long row, int j0, int j1, int n,
                                               const int* xs, int lane, const double* lf, int T) {
  const int base = j0 * PMDI_FB + 2 * lane;
  const int nits = (min(ds.Dp, j1 * PMDI_FB) - j0 * PMDI_FB) / PMDI_WF;
  return nb_eval_raw(ds.S + row * ds.Dp + base, ds.aux + row * ds.J + j0,
                     (unsigned)__cvta_generic_to_shared(xs + base), nits, j1 - j0, n,
                     (unsigned)__cvta_generic_to_shared(lf), T, lane);
}

__device__ __noinline__ double cat_eval_raw(const uint32_t* cnt, long long Dp, unsigned xs, int nits, int lane) {
  unsigned a0 = 0, a1 = 0, a2 = 0, a3 = 0, b0 = 0, b1 = 0, b2 = 0, b3 = 0;
  int2 v0, v1, v2, v3;
  v0 = v1 = v2 = v3 = make_int2(0, 0);
#define PMDI_C_LOAD(V, A, B, IT)                                                            \
  {                                                                                         \
    V = lds_i32x2(xs + (IT) * PMDI_WF * 4);                                                 \
    A = V.x ? ldcg_u32(cnt + (long long)(V.x - 1) * Dp + (IT) * PMDI_WF) : 0u;              \
    B = V.y ? ldcg_u32(cnt + (long long)(V.y - 1) * Dp + (IT) * PMDI_WF + 1) : 0u;          \
  }
  if (0 < nits) PMDI_C_LOAD(v0, a0, b0, 0)
  if (1 < nits) PMDI_C_LOAD(v1, a1, b1, 1)
  if (2 < nits) PMDI_C_LOAD(v2, a2, b2, 2)
  if (3 < nits) PMDI_C_LOAD(v3, a3, b3, 3)
  double acc = 0.0;
#define PMDI_C_STEP(V, A, B, IT)                                                            \
  if (i0 + IT < nits) {                                                                     \
    const double f0 = V.x ? 0.5 + (double)A : 1.0;                                          \
    const double f1 = V.y ? 0.5 + (double)B : 1.0;                                          \
    prod *= f0 * f1;                                                                        \
    if (i0 + IT + 4 < nits) PMDI_C_LOAD(V, A, B, IT + 4)                                    \
  }
  for (int i0 = 0; i0 < nits; i0 += 4) {
    double prod = 1.0;
    PMDI_C_STEP(v0, a0, b0, 0)
    PMDI_C_STEP(v1, a1, b1, 1)
    PMDI_C_STEP(v2, a2, b2, 2)
    PMDI_C_STEP(v3, a3, b3, 3)
    acc += pm_log(prod);
    cnt += PMDI_FB; xs += PMDI_FB * 4;
  }
#undef PMDI_C_STEP
#undef PMDI_C_LOAD
  return warp_sum(acc);
}
__device__ __forceinline__ double cat_eval_item(const DsDev& ds, long long row, int j0, int j1,
                                                const int* xs, int lane) {
  const int base = j0 * PMDI_FB + 2 * lane;
  const int nits = (min(ds.Dp, j1 * PMDI_FB) - j0 * PMDI_FB) / PMDI_WF;
  return cat_eval_raw(ds.cnt + row * (long long)ds.Lmax * ds.Dp + base, (long long)ds.Dp,
                      (unsigned)__cvta_generic_to_shared(xs + base), nits, lane);
}

// ------------------------------------------------------------------------------------------
// Row movement for resampling (src/pmdi.jl:318-341 in dense form): one warp moves one cluster
// row src -> dst, or resets dst to the empty state when the source label is empty.
// ------------------------------------------------------------------------------------------
__device__ __noinline__ void row_copy(const DsDev& ds, long long sdelta, long long src, long long dst, int lane) {
  // sdelta: byte offset from this rank's arena to the arena of the rank that holds the source row
  // (0 when it is local); the source is read through NVLink peer memory then.
#define PMDI_SRC(ptr_) ((decltype(ptr_))((const char*)(ptr_) + sdelta))
  const int ns = ldcg_i32(PMDI_SRC(ds.n) + src), nd = ldcg_i32(ds.n + dst);
  if (ns == 0 && nd == 0) return;
  const int Dp = ds.Dp;
  if (ds.type == T_GAUSSIAN) {
    for (int q = 2 * lane; q < Dp; q += 64) {
      double2 a, b, c, d;
      if (ns) {
        a = ldcg_f64x2(PMDI_SRC(ds.mu) + src * Dp + q); b = ldcg_f64x2(PMDI_SRC(ds.lamn) + src * Dp + q);
        c = ldcg_f64x2(PMDI_SRC(ds.sum) + src * Dp + q); d = ldcg_f64x2(PMDI_SRC(ds.beta) + src * Dp + q);
      } else {
        a = make_double2(0.0, 0.0); b = make_double2(1.0, 1.0);
        c = make_double2(0.0, 0.0); d = make_double2(0.5, 0.5);
      }
      *(double2*)(ds.mu + dst * Dp + q) = a; *(double2*)(ds.lamn + dst * Dp + q) = b;
      *(double2*)(ds.sum + dst * Dp + q) = c; *(double2*)(ds.beta + dst * Dp + q) = d;
    }
  } else if (ds.type == T_CATEGORICAL) {
    const long long W = (long long)ds.Lmax * Dp;
    for (long long q = 4 * lane; q < W; q += 128) {
      uint4 v = make_uint4(0, 0, 0, 0);
      if (ns) v = __ldcg((const uint4*)(PMDI_SRC(ds.cnt) + src * W + q));
      *(uint4*)(ds.cnt + dst * W + q) = v;
    }
  } else {
    for (int q = 2 * lane; q < Dp; q += 64) {
      longlong2 v = make_longlong2(0, 0);
      if (ns) v = ldcg_i64x2(PMDI_SRC(ds.S) + src * Dp + q);
      *(longlong2*)(ds.S + dst * Dp + q) = v;
    }
  }
  for (int j = lane; j < ds.J; j += 32) ds.aux[dst * ds.J + j] = ns ? ldcg_f64(PMDI_SRC(ds.aux) + src * ds.J + j) : 0.0;
  if (lane == 0) ds.n[dst] = ns;
#undef PMDI_SRC
}
