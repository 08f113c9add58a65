// Copy-on-write block operators of the pool engine (pool_kernel.cuh).  ONE operator per cluster type
// covers the three things a 256-feature block of a pool row can need at an observation step:
//   mode 0  calc_logprob of the current observation for the row as it is;
//   mode 1  cluster_add! of the previous observation (source row -> destination row; the same row
//           when every particle that refers to it chose it: in place) and calc_logprob of the
//           current observation for the updated row, in one pass;
//   mode 2  the split of src/pmdi.jl:288-309: as mode 1 into a fresh destination row, plus
//           calc_logprob for the unchanged source row - the source is read once.
// One copy of the code per type keeps the per-step instruction footprint of the persistent kernel
// inside the SM's instruction cache (the kernel is bound by dependent latencies, not by bytes).
// Arithmetic: the reference's operation order for the add (gaussian_cluster.jl:57-63,
// categorical_cluster.jl:43-51, negbinom_cluster.jl:43-51), logs of short products for the
// predictive (same forms as cluster_types.cuh).
#pragma once
#include "cluster_types.cuh"
#include "user_type.cuh"

// ------------------------------------------------------------------------------------------
// Gaussian.  Pointers are at this lane's first feature of the block; n = size of the SOURCE row.
// Returns the block partial of the main result (mode 0: the row; modes 1, 2: the updated row):
// aux - (n/2+1) * sum log(1 + d^2 lamn); *v_src (mode 2) = the source row's block partial.
// ------------------------------------------------------------------------------------------
#define PMDI_GAUSS_FEATURE(C)                                                                        \
  if (fl.C) {                                                                                        \
    if (mode != 1) { const double ds_ = y.C - mu[i].C; ps *= fma(ds_ * ds_, ln[i].C, 1.0); }          \
    if (mode) {                                                                                      \
      sm[i].C = __dadd_rn(sm[i].C, x.C);                                                             \
      const double dd = __dadd_rn(x.C, -mu[i].C);                                                    \
      bt[i].C = __dadd_rn(bt[i].C, div_const(__dmul_rn(c1, __dmul_rn(dd, dd)), c2, r2));             \
      mu[i].C = div_const(sm[i].C, c3, r3);                                                          \
      ln[i].C = div_const(pm_div(c4, __dmul_rn(bt[i].C, c5)), c6, r6);                               \
      pl *= ln[i].C;                                                                                 \
      const double d_ = y.C - mu[i].C;                                                               \
      pd *= fma(d_ * d_, ln[i].C, 1.0);                                                              \
    }                                                                                                \
  }

__device__ __noinline__ double gauss_block(const double* s_sum, const double* s_beta, const double* s_mu,
                                           const double* s_lamn, long long d_off /* dst - src, elements */,
                                           const double* s_aux, double* d_aux, const uint8_t* flag_p, int nit,
                                           int mode, int n, PMDI_XADDR xp, PMDI_XADDR xc, double* v_src) {
  const double nn = (double)(n + 1);  // size after the add
  double c1 = 0, c2 = 0, c3 = 0, c4 = 0, c5 = 0, c6 = 0, r2 = 0, r3 = 0, r6 = 0;
  if (mode) {
    c1 = __dadd_rn(__dadd_rn(nn, -1.0), 0.001);                      // n - 1 + kappa
    c2 = __dmul_rn(2.0, __dadd_rn(nn, 0.001));                       // 2 (n + kappa)
    c3 = __dadd_rn(nn, 0.001);                                       // n + kappa
    c4 = __dmul_rn(__dadd_rn(__dmul_rn(0.5, nn), 0.5), c3);          // (n/2 + 1/2)(n + kappa)
    c5 = __dadd_rn(nn, 1.001);                                       // n + 1 + kappa
    c6 = __dadd_rn(nn, 1.0);
    r2 = __drcp_rn(c2); r3 = __drcp_rn(c3); r6 = __drcp_rn(c6);
  }
  double pl = 1.0, pd = 1.0, ps = 1.0;
#pragma unroll 1
  for (int h = 0; h < nit; h += 2) {
    double2 sm[2], bt[2], mu[2], ln[2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
      if (h + i < nit) {
        const int o = (h + i) * PMDI_WF;
        mu[i] = ldcg_f64x2(s_mu + o); ln[i] = ldcg_f64x2(s_lamn + o);
        if (mode) { sm[i] = ldcg_f64x2(s_sum + o); bt[i] = ldcg_f64x2(s_beta + o); }
      }
#pragma unroll
    for (int i = 0; i < 2; ++i)
      if (h + i < nit) {
        const int o = (h + i) * PMDI_WF;
        const double2 y = PMDI_LDX_F64X2(xc + o * 8);
        double2 x = make_double2(0.0, 0.0);
        if (mode) x = PMDI_LDX_F64X2(xp + o * 8);
        const uchar2 fl = *(const uchar2*)(flag_p + o);
        PMDI_GAUSS_FEATURE(x)
        PMDI_GAUSS_FEATURE(y)
        if (mode) {
          *(double2*)(const_cast<double*>(s_sum) + d_off + o) = sm[i];
          *(double2*)(const_cast<double*>(s_beta) + d_off + o) = bt[i];
          *(double2*)(const_cast<double*>(s_mu) + d_off + o) = mu[i];
          *(double2*)(const_cast<double*>(s_lamn) + d_off + o) = ln[i];
        }
      }
  }
  double a = 0.0, e = 0.0, es = 0.0;
  if (mode) { a = 0.5 * pm_log(pl); e = pm_log(pd); }
  if (mode != 1) es = pm_log(ps);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(FULL, a, o);
    e += __shfl_xor_sync(FULL, e, o);
    es += __shfl_xor_sync(FULL, es, o);
  }
  double vs = 0.0;
  if (mode != 1) vs = ldcg_f64(s_aux) - (0.5 * (double)n + 1.0) * es;
  if (mode == 0) return vs;
  if ((threadIdx.x & 31) == 0) *d_aux = a;
  *v_src = vs;
  return a - (0.5 * nn + 1.0) * e;
}
#undef PMDI_GAUSS_FEATURE

// ------------------------------------------------------------------------------------------
// NegBinom.  S pointers at this lane's first feature; observations by PMDI_XADDR (cluster_types.cuh); n =
// size of the source row.  Partials include the row's aux (the x-independent part).
// ------------------------------------------------------------------------------------------
__device__ __noinline__ double nb_block(const long long* s_S, long long d_off, const double* s_aux, double* d_aux,
                                        int nit, int mode, int n, PMDI_XADDR xp, PMDI_XADDR xc, unsigned lf_s, int T,
                                        double* v_src) {
  double aux = 0.0, ed = 0.0, es = 0.0;
  const long long ns2 = n + 2, nd2 = n + 3, na = n + 2;  // source: n+2; after the add: size n+1
#pragma unroll 1
  for (int it = 0; it < nit; ++it) {
    longlong2 s = ldcg_i64x2(s_S + it * PMDI_WF);
    const int2 y = PMDI_LDX_I32X2(xc + it * PMDI_WF * 4);
    if (mode != 1) {
      if (y.x >= 0) { const long long b = s.x + y.x; es += lfact_s(b, lf_s, T) - lfact_s(b + ns2, lf_s, T); }
      if (y.y >= 0) { const long long b = s.y + y.y; es += lfact_s(b, lf_s, T) - lfact_s(b + ns2, lf_s, T); }
    }
    if (mode) {
      const int2 x = PMDI_LDX_I32X2(xp + it * PMDI_WF * 4);
      if (x.x >= 0) { s.x += x.x; aux += lfact_s(s.x + na, lf_s, T) - lfact_s(s.x, lf_s, T); }
      if (x.y >= 0) { s.y += x.y; aux += lfact_s(s.y + na, lf_s, T) - lfact_s(s.y, lf_s, T); }
      *(longlong2*)(const_cast<long long*>(s_S) + d_off + it * PMDI_WF) = s;
      if (y.x >= 0) { const long long b = s.x + y.x; ed += lfact_s(b, lf_s, T) - lfact_s(b + nd2, lf_s, T); }
      if (y.y >= 0) { const long long b = s.y + y.y; ed += lfact_s(b, lf_s, T) - lfact_s(b + nd2, lf_s, T); }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    aux += __shfl_xor_sync(FULL, aux, o);
    ed += __shfl_xor_sync(FULL, ed, o);
    es += __shfl_xor_sync(FULL, es, o);
  }
  double vs = 0.0;
  if (mode != 1) vs = ldcg_f64(s_aux) + es;
  if (mode == 0) return vs;
  if ((threadIdx.x & 31) == 0) *d_aux = aux;
  *v_src = vs;
  return aux + ed;
}

// ------------------------------------------------------------------------------------------
// Categorical, packed counts: a feature's level counts are `fpw` fields of 64/fpw bits in each of
// `wpf` consecutive 64-bit words (cw[row][q][wpf]); level l (1-based) is field (l-1) % fpw of
// word (l-1) / fpw.  With <= 4 levels and n_obs < 65536 a feature is ONE word: 8 bytes per
// predictive term, the reference's own width (an Int64 count), and one 128-bit load per lane
// serves two features.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long ldcg_u64(const unsigned long long* p) { return __ldcg(p); }
__device__ __forceinline__ ulonglong2 ldcg_u64x2(const unsigned long long* p) { return __ldcg((const ulonglong2*)p); }

__device__ __forceinline__ double cat_field(unsigned long long w, int f, int fpw) {
  const int fw = 64 / fpw;
  const unsigned long long mask = fw == 64 ? ~0ull : ((1ull << fw) - 1ull);
  return 0.5 + (double)((w >> (f * fw)) & mask);
}

__device__ __noinline__ double cat_block(const unsigned long long* s_cw, long long d_off /* words */, int wpf, int fpw,
                                         int nit, int mode, PMDI_XADDR xp, PMDI_XADDR xc, double* v_src) {
  const int fw = 64 / fpw;
  double pd = 1.0, ps = 1.0;
#pragma unroll 1
  for (int it = 0; it < nit; ++it) {
    const int2 y = PMDI_LDX_I32X2(xc + it * PMDI_WF * 4);
    int2 x = make_int2(0, 0);
    if (mode) x = PMDI_LDX_I32X2(xp + it * PMDI_WF * 4);
    if (wpf == 1) {
      ulonglong2 w = ldcg_u64x2(s_cw + (size_t)it * PMDI_WF);
      if (mode != 1) {
        if (y.x) ps *= cat_field(w.x, y.x - 1, fpw);
        if (y.y) ps *= cat_field(w.y, y.y - 1, fpw);
      }
      if (mode) {
        if (x.x) w.x += 1ull << ((x.x - 1) * fw);
        if (x.y) w.y += 1ull << ((x.y - 1) * fw);
        *(ulonglong2*)(const_cast<unsigned long long*>(s_cw) + d_off + (size_t)it * PMDI_WF) = w;
        if (y.x) pd *= cat_field(w.x, y.x - 1, fpw);
        if (y.y) pd *= cat_field(w.y, y.y - 1, fpw);
      }
    } else {
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        const int xv = h ? x.y : x.x, yv = h ? y.y : y.x;
        const unsigned long long* sf = s_cw + ((size_t)it * PMDI_WF + h) * wpf;
#pragma unroll 1
        for (int wd = 0; wd < wpf; ++wd) {
          const bool hit_y = yv && (yv - 1) / fpw == wd, hit_x = mode && xv && (xv - 1) / fpw == wd;
          if (!mode && !hit_y) continue;  // plain evaluation reads the observed level's word only
          unsigned long long w = ldcg_u64(sf + wd);
          if (mode != 1 && hit_y) ps *= cat_field(w, (yv - 1) % fpw, fpw);
          if (mode) {
            if (hit_x) w += 1ull << (((xv - 1) % fpw) * fw);
            const_cast<unsigned long long*>(sf)[d_off + wd] = w;
            if (hit_y) pd *= cat_field(w, (yv - 1) % fpw, fpw);
          }
        }
      }
    }
  }
  double ed = 0.0, es = 0.0;
  if (mode) ed = pm_log(pd);
  if (mode != 1) es = pm_log(ps);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ed += __shfl_xor_sync(FULL, ed, o);
    es += __shfl_xor_sync(FULL, es, o);
  }
  if (mode == 0) return es;
  *v_src = es;
  return ed;
}
