// User-defined cluster types as device functors (the reference's plugin contract, README.md:48-88:
// calc_logprob / cluster_add! / calc_logmarginal for a user's cluster struct).  This header is only
// compiled at run time (NVRTC), together with the users' sources, into a private copy of the kernels
// of one engine: pmdi_register_cluster_type hands over a struct
//
//   struct MyType {
//     static constexpr int WORDS = ...;                                        // doubles of state per feature (<= 8)
//     __device__ static void   init(double* st);                               // the empty cluster
//     __device__ static double logprob(const double* st, int n, double x);     // this feature's term of calc_logprob
//                                                                              //   (n = cluster size, x = the observation)
//     __device__ static void   add(double* st, int n, double x);               // cluster_add!; n = size AFTER the add
//     __device__ static double logmarginal(const double* st, int n);           // this feature's calc_logmarginal
//   };
//
// The cluster types of the reference are all of this form: feature-wise sufficient statistics, the
// observation's log-probability a sum over features.  State lives as ust[row][word][feature].
//
// One program carries every user type of a context.  The host puts each source in a namespace of its
// own (pmdi_u0, pmdi_u1, ...: two users may both call their struct `Cluster`) and defines
//   PMDI_USER_TYPES          the number of types (slots) in the program
//   PMDI_USER_TYPE_LIST(X)   X(slot, namespace-qualified struct) for every slot
// A dataset of a user type carries its slot in DsDev::Lmax (a field only Categorical data uses); the
// operators below dispatch on it with one switch.
#pragma once
#include "cluster_types.cuh"

#ifdef PMDI_USER_TYPES
#define PMDI_USER_SLOT(ds_) ((ds_).Lmax)
#define PMDI_USER_CHECK(s_, U_) \
  static_assert(U_::WORDS >= 1 && U_::WORDS <= 8, "a user cluster type keeps 1..8 doubles per feature");
PMDI_USER_TYPE_LIST(PMDI_USER_CHECK)
#undef PMDI_USER_CHECK

__device__ __forceinline__ double user_x(const DsDev& ds, PMDI_XADDR xs_addr, int f, int x_is_int) {
  // staged observation: doubles, or 32-bit integers for integer-valued data
#ifdef PMDI_X_GLOBAL
  if (x_is_int) return (double)__ldg((const int*)(xs_addr + f * 4u));
  return __ldg((const double*)(xs_addr + f * 8u));
#else
  if (x_is_int) { int v; asm("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(xs_addr + f * 4u)); return (double)v; }
  double v; asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(xs_addr + f * 8u)); return v;
#endif
}

// One block of one row, by one warp: mode 0 plain evaluation, 1 add + evaluation, 2 add into the row
// d_off doubles further on + evaluation of both (pool_types.cuh).  s_st at the row's word 0, this lane's
// first feature; xp / xc: addresses of the block's first feature of this lane in the staged observation (PMDI_XADDR:
// shared memory, or global memory in the wide kernels).
template <class U>
__device__ __forceinline__ double user_block_t(const DsDev& ds, const double* s_st, long long d_off, const uint8_t* flag_p,
                                               int nit, int mode, int n, PMDI_XADDR xp, PMDI_XADDR xc, double* v_src) {
  const int W = U::WORDS, Dp = ds.Dp, xi = ds.uW < 0;
  double ed = 0.0, es = 0.0;
#pragma unroll 1
  for (int it = 0; it < nit; ++it) {
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
      const int f = it * PMDI_WF + h;
      double st[U::WORDS];
#pragma unroll
      for (int w = 0; w < W; ++w) st[w] = ldcg_f64(s_st + (long long)w * Dp + f);
      if (flag_p[f]) {
        const double y = user_x(ds, xc, f, xi);
        if (mode != 1) es += U::logprob(st, n, y);
        if (mode) {
          U::add(st, n + 1, user_x(ds, xp, f, xi));
          ed += U::logprob(st, n + 1, y);
        }
      }
      if (mode) {
#pragma unroll
        for (int w = 0; w < W; ++w) const_cast<double*>(s_st)[d_off + (long long)w * Dp + f] = st[w];
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ed += __shfl_xor_sync(FULL, ed, o);
    es += __shfl_xor_sync(FULL, es, o);
  }
  if (mode == 0) return es;
  *v_src = es;
  return ed;
}

// the block operator of the dataset's type; d_off / the row offset of s_st are in units of the type's row
// (WORDS * Dp doubles), which the caller computes from |ds.uW|
__device__ __noinline__ double user_block(const DsDev& ds, const double* s_st, long long d_off, const uint8_t* flag_p,
                                          int nit, int mode, int n, PMDI_XADDR xp, PMDI_XADDR xc, double* v_src) {
  switch (PMDI_USER_SLOT(ds)) {
#define PMDI_USER_CASE(s_, U_) \
    case s_: return user_block_t<U_>(ds, s_st, d_off, flag_p, nit, mode, n, xp, xc, v_src);
    PMDI_USER_TYPE_LIST(PMDI_USER_CASE)
#undef PMDI_USER_CASE
  }
  return 0.0;
}

// sequential cluster_add! of a member list into one feature of a row (prefix build, single-cluster evaluation)
template <class U>
__device__ __forceinline__ void user_build_feature_t(const DsDev& ds, long long row, int q, const int* mem, int cnt, bool on) {
  double st[U::WORDS];
  U::init(st);
  if (on)
    for (int t = 0; t < cnt; ++t) {
      const double x = ds.uW < 0 ? (double)((const int*)ds.x)[(size_t)mem[t] * ds.Dp + q] : ((const double*)ds.x)[(size_t)mem[t] * ds.Dp + q];
      U::add(st, t + 1, x);
    }
  for (int w = 0; w < U::WORDS; ++w) ds.ust[((long long)row * U::WORDS + w) * ds.Dp + q] = st[w];
}
__device__ __noinline__ void user_build_feature(const DsDev& ds, long long row, int q, const int* mem, int cnt, bool on) {
  switch (PMDI_USER_SLOT(ds)) {
#define PMDI_USER_CASE(s_, U_) \
    case s_: user_build_feature_t<U_>(ds, row, q, mem, cnt, on); return;
    PMDI_USER_TYPE_LIST(PMDI_USER_CASE)
#undef PMDI_USER_CASE
  }
}

// calc_logmarginal of one feature of the cluster of `cnt` members (feature selection, single-cluster evaluation)
template <class U>
__device__ __forceinline__ double user_logmarginal_t(const DsDev& ds, int q, const int* mem, int cnt, bool on) {
  double st[U::WORDS];
  U::init(st);
  if (on)
    for (int t = 0; t < cnt; ++t) {
      const double xv = ds.uW < 0 ? (double)((const int*)ds.x)[(size_t)mem[t] * ds.Dp + q]
                                  : ((const double*)ds.x)[(size_t)mem[t] * ds.Dp + q];
      U::add(st, t + 1, xv);
    }
  return U::logmarginal(st, cnt);
}
__device__ __noinline__ double user_logmarginal(const DsDev& ds, int q, const int* mem, int cnt, bool on) {
  switch (PMDI_USER_SLOT(ds)) {
#define PMDI_USER_CASE(s_, U_) \
    case s_: return user_logmarginal_t<U_>(ds, q, mem, cnt, on);
    PMDI_USER_TYPE_LIST(PMDI_USER_CASE)
#undef PMDI_USER_CASE
  }
  return 0.0;
}

// doubles of state of one row of a user-type dataset
__device__ __forceinline__ long long user_row_words(const DsDev& ds) { return (long long)(ds.uW < 0 ? -ds.uW : ds.uW) * ds.Dp; }
#endif
