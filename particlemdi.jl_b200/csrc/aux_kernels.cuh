// Kernels around the persistent sweep: state initialisation, the rho-prefix build
// (src/pmdi.jl:188-207), particle selection + lineage back-trace (src/pmdi.jl:345-350,373),
// the feature-selection log-marginal reduction (src/pmdi.jl:120-128,354-370) and the
// single-cluster evaluation used by the plugin-contract parity tests.
#pragma once
#include "pool_types.cuh"

#ifndef PMDI_X_GLOBAL  // (the wide module, sweep_wide.cu, carries only k_eval_row_wide from here: at the end)

// all rows of a dataset to the empty-cluster state (constructors gaussian_cluster.jl:17-21,
// categorical_cluster.jl:6-10, negbinom_cluster.jl:9-10)
extern "C" __global__ void k_init_rows(DsDev ds, long long rows) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (ds.type == T_GAUSSIAN) {
    for (long long i = t0; i < rows * ds.Dp; i += stride) {
      ds.mu[i] = 0.0; ds.lamn[i] = 1.0; ds.sum[i] = 0.0; ds.beta[i] = 0.5;
    }
  } else if (ds.type == T_CATEGORICAL) {
    for (long long i = t0; i < rows * ds.Lmax * ds.Dp; i += stride) ds.cnt[i] = 0u;
#ifdef PMDI_USER_TYPES
  } else if (ds.type == T_USER) {
    for (long long i = t0; i < rows * ds.Dp; i += stride) user_build_feature(ds, i / ds.Dp, (int)(i % ds.Dp), nullptr, 0, false);
#endif
  } else {
    for (long long i = t0; i < rows * ds.Dp; i += stride) ds.S[i] = 0;
  }
  for (long long i = t0; i < rows * ds.J; i += stride) { ds.aux[i] = 0.0; if (ds.part) ds.part[i] = 0.0; }
  for (long long i = t0; i < rows; i += stride) ds.n[i] = 0;
}

extern "C" __global__ void k_sweep_init(SweepParams sp) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < sp.P) {
    sp.slot_of[t] = t;
    sp.slot_of[sp.P + t] = t;
    sp.logical_of[t] = t;
    sp.logical_of[sp.P + t] = t;
  }
  if (t == 0) {
    *sp.err = 0;
    for (int i = 0; i < 8; ++i) sp.counters[i] = 0;
    sp.plan_out[0] = 0;
    for (int k = 0; k < PMDI_MAX_K; ++k) { sp.rows_eval[k] = 0ull; sp.rows_ref[k] = 0ull; }
  }
}

// Members of every label among the first n1-1 shuffled observations, in shuffle order
// (src/pmdi.jl:193,200-206).  One block per dataset, thread m = label m+1.
extern "C" __global__ void k_prefix_lists(SweepParams sp, int* members /* [K][n1-1] */, int* off /* [K][N+1] */) {
  const int k = blockIdx.x, m = threadIdx.x, N = sp.N, npre = sp.n1 - 1;
  __shared__ int cnt[PMDI_MAX_N + 1];
  const long long* s = sp.s_in + (size_t)k * sp.n_obs;
  int c = 0;
  if (m < N)
    for (int t = 0; t < npre; ++t) c += ((int)s[sp.order[t]] - 1 == m);
  if (m < N) cnt[m] = c;
  __syncthreads();
  if (m == 0) {
    int acc = 0;
    for (int i = 0; i < N; ++i) { const int v = cnt[i]; cnt[i] = acc; acc += v; }
    cnt[N] = acc;
  }
  __syncthreads();
  if (m <= N) off[k * (N + 1) + m] = cnt[m];
  if (m < N) {
    int w = cnt[m];
    for (int t = 0; t < npre; ++t) {
      const int i = sp.order[t];
      if ((int)s[i] - 1 == m) members[(size_t)k * npre + (w++)] = i;
    }
  }
}

// Sequential cluster_add! of the members of one label into row (slot*N + m), one thread per
// feature (literal arithmetic, same bits as the reference).  use_flags = 0 -> all features on.
__device__ __forceinline__ void build_row_feature(const DsDev& ds, const PoolDev* pd, long long row, int q,
                                                  const int* mem, int cnt, int use_flags) {
  const bool on = use_flags ? (ds.flag[q] != 0) : (q < ds.D);
#ifdef PMDI_USER_TYPES
  if (ds.type == T_USER) { user_build_feature(ds, row, q, mem, cnt, on); return; }
#endif
  if (ds.type == T_GAUSSIAN) {
    double sum = 0.0, beta = 0.5, mu = 0.0, lam = 1.0;
    if (on) {
      const double* x = (const double*)ds.x;
      // the member's value is fetched two members ahead of the dependent arithmetic
      double x1 = cnt > 0 ? x[(size_t)mem[0] * ds.Dp + q] : 0.0;
      double x2 = cnt > 1 ? x[(size_t)mem[1] * ds.Dp + q] : 0.0;
      for (int t = 0; t < cnt; ++t) {
        const double nn = (double)(t + 1);
        const double xv = x1;
        x1 = x2;
        if (t + 2 < cnt) x2 = x[(size_t)mem[t + 2] * ds.Dp + q];
        sum = __dadd_rn(sum, xv);
        const double dd = __dadd_rn(xv, -mu);
        beta = __dadd_rn(beta, __ddiv_rn(__dmul_rn(__dadd_rn(__dadd_rn(nn, -1.0), 0.001), __dmul_rn(dd, dd)),
                                         __dmul_rn(2.0, __dadd_rn(nn, 0.001))));
        mu = __ddiv_rn(sum, __dadd_rn(nn, 0.001));
        lam = __ddiv_rn(__dmul_rn(__dadd_rn(__dmul_rn(0.5, nn), 0.5), __dadd_rn(nn, 0.001)),
                        __dmul_rn(beta, __dadd_rn(nn, 1.001)));
      }
    }
    const long long o = row * ds.Dp + q;
    ds.sum[o] = sum; ds.beta[o] = beta; ds.mu[o] = mu;
    ds.lamn[o] = __ddiv_rn(lam, __dadd_rn((double)cnt, 1.0));
    if (!on || cnt == 0) ds.lamn[o] = 1.0;
  } else if (ds.type == T_CATEGORICAL && pd) {  // pool engine: packed counts cw[row][q][wpf]
    unsigned long long* w = pd->cw + ((size_t)row * ds.Dp + q) * pd->wpf;
    for (int i = 0; i < pd->wpf; ++i) w[i] = 0ull;
    if (on) {
      const int* x = (const int*)ds.x;
      const int fw = 64 / pd->fpw;
      for (int t = 0; t < cnt; ++t) {
        const int lv = x[(size_t)mem[t] * ds.Dp + q] - 1;
        w[lv / pd->fpw] += 1ull << ((lv % pd->fpw) * fw);
      }
    }
  } else if (ds.type == T_CATEGORICAL) {
    uint32_t* c = ds.cnt + row * (long long)ds.Lmax * ds.Dp + q;
    for (int l = 0; l < ds.Lmax; ++l) c[(long long)l * ds.Dp] = 0u;
    if (on) {
      const int* x = (const int*)ds.x;
      for (int t = 0; t < cnt; ++t) {
        const int lv = x[(size_t)mem[t] * ds.Dp + q];
        c[(long long)(lv - 1) * ds.Dp] += 1u;
      }
    }
  } else {
    long long S = 0;
    if (on) {
      const int* x = (const int*)ds.x;
      for (int t = 0; t < cnt; ++t) S += x[(size_t)mem[t] * ds.Dp + q];
    }
    ds.S[row * ds.Dp + q] = S;
  }
}

// grid (ceil(Dp/128), N, K): prototypes of the prefix clusters into slot P
extern "C" __global__ void k_prefix_build(SweepParams sp, const int* members, const int* off) {
  const int k = blockIdx.z, m = blockIdx.y, q = blockIdx.x * blockDim.x + threadIdx.x;
  const DsDev& ds = sp.ds[k];
  if (q >= ds.Dp) return;
  const int b = off[k * (sp.N + 1) + m], e = off[k * (sp.N + 1) + m + 1];
  const long long row = sp.proto_base + m;
  build_row_feature(ds, sp.engine ? &sp.pd[k] : nullptr, row, q, members + (size_t)k * (sp.n1 - 1) + b, e - b, 1);
  if (q == 0) ds.n[row] = e - b;
}

// aux of the prototype rows: grid (N, K), one warp per feature block
extern "C" __global__ void k_proto_aux(SweepParams sp) {
  const int k = blockIdx.y, m = blockIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const DsDev& ds = sp.ds[k];
  const long long row = sp.proto_base + m;
  const int n = ds.n[row];
  for (int j = w; j < ds.J; j += blockDim.x >> 5) {
    if (ds.type == T_GAUSSIAN) gauss_aux_block(ds, row, j, lane);
    else if (ds.type == T_NEGBINOM) nb_aux_block(ds, row, j, n, lane, sp.lf_glob, sp.lf_glob_T);
    else if (lane == 0) ds.aux[row * ds.J + j] = 0.0;
  }
}

// every particle starts the sweep with the prototypes (src/pmdi.jl:197-199: particle[u,:,k] .= id)
extern "C" __global__ void k_broadcast(SweepParams sp) {
  const int lane = threadIdx.x & 31;
  const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long GW = ((long long)gridDim.x * blockDim.x) >> 5;
  const long long total = (long long)sp.K * sp.Ps * sp.N;
  for (long long idx = gw; idx < total; idx += GW) {
    const int k = (int)(idx / ((long long)sp.Ps * sp.N));
    const long long rem = idx - (long long)k * sp.Ps * sp.N;
    const int m = (int)(rem % sp.N);
    row_copy(sp.ds[k], 0, (long long)sp.Ps * sp.N + m, rem, lane);
  }
}

// ------------------------------------------------------------------------------------------
// calc_logmarginal of clusters rebuilt from member lists (src/pmdi.jl:358-366); reference formulas
// gaussian_cluster.jl:68-83, categorical_cluster.jl:53-66, negbinom_cluster.jl:53-60.
// k_logmarginal_part: one thread per (feature, cluster) - the add of a cluster's members is sequential
// (the reference's operation order), clusters are independent: grid (ceil(D/128), clusters).
// k_logmarginal: one thread per feature sums the clusters in list order,
//   out[q] = base[q]*base_scale + sum_c lm[c][q];  flags_out[q] = (1 - 1/exp(out+1)) > u_q
// ------------------------------------------------------------------------------------------
extern "C" __global__ void k_logmarginal_part(DsDev ds, const int* c_off, const int* members,
                                              const double* gauss_cst /* per cluster */, const double* nlevels,
                                              int use_flags, double* lm_out /* [clusters][D] */) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
  if (q >= ds.D) return;
  const bool on = use_flags ? (ds.flag[q] != 0) : true;
  const int* mem = members + c_off[c];
  const int cnt = c_off[c + 1] - c_off[c];
  const double n = (double)cnt;
  double lm;
#ifdef PMDI_USER_TYPES
  if (ds.type == T_USER) {
    lm = user_logmarginal(ds, q, mem, cnt, on);
  } else
#endif
  if (ds.type == T_GAUSSIAN) {
    double sum = 0.0, beta = 0.5, mu = 0.0;
    const double* x = (const double*)ds.x;
    if (on) {
      // the member's value is fetched two members ahead of the dependent arithmetic
      double x1 = cnt > 0 ? x[(size_t)mem[0] * ds.Dp + q] : 0.0;
      double x2 = cnt > 1 ? x[(size_t)mem[1] * ds.Dp + q] : 0.0;
      for (int t = 0; t < cnt; ++t) {
        const double nn = (double)(t + 1);
        const double xv = x1;
        x1 = x2;
        if (t + 2 < cnt) x2 = x[(size_t)mem[t + 2] * ds.Dp + q];
        sum = __dadd_rn(sum, xv);
        const double dd = __dadd_rn(xv, -mu);
        beta = __dadd_rn(beta, __ddiv_rn(__dmul_rn(__dadd_rn(__dadd_rn(nn, -1.0), 0.001), __dmul_rn(dd, dd)),
                                         __dmul_rn(2.0, __dadd_rn(nn, 0.001))));
        mu = __ddiv_rn(sum, __dadd_rn(nn, 0.001));
      }
    }
    lm = -(n / 2 + 0.5) * log(beta) + gauss_cst[c];
  } else if (ds.type == T_CATEGORICAL) {
    const int* x = (const int*)ds.x;
    const double nl = nlevels[q];  // 0.5 * column maximum (categorical_cluster.jl:10)
    const int R = (int)(2.0 * nl);
    lm = lgamma(nl * 2) - lgamma(nl * 2 + n);
    for (int r = 1; r <= R; ++r) {
      int cr = 0;
      if (on)
        for (int t = 0; t < cnt; ++t) cr += (x[(size_t)mem[t] * ds.Dp + q] == r);
      lm += lgamma((double)cr + 0.5);
    }
  } else {
    const int* x = (const int*)ds.x;
    long long S = 0;
    if (on)
      for (int t = 0; t < cnt; ++t) S += x[(size_t)mem[t] * ds.Dp + q];
    lm = lgamma((double)S + 1.0) - lgamma((double)S + (n + 1 + 1)) + lgamma(1.0 + n);
  }
  lm_out[(size_t)c * ds.D + q] = lm;
}

extern "C" __global__ void k_logmarginal(DsDev ds, int n_clusters, const double* lm,
                              const double* base, double base_scale, double out_scale, double* out,
                              uint8_t* flags_out, const double* tape_f, unsigned long long seed,
                              unsigned iter, int k) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= ds.D) return;
  double acc = base ? base[q] * base_scale : 0.0;
  for (int c = 0; c < n_clusters; ++c) acc += lm[(size_t)c * ds.D + q];
  acc *= out_scale;
  out[q] = acc;
  if (flags_out) {
    const double u = tape_f ? tape_f[q] : pmdi_philox_uniform(seed, iter, DRAW_FEATURE, 0, k, q);
    flags_out[q] = ((1.0 - 1.0 / exp(acc + 1.0)) > u) ? 1 : 0;
  }
}

// calc_logprob of observation `obs` against the prototype row (slot P, label 0), through the
// same block operators the sweep uses.  One warp; dynamic smem = staged observation row.
extern "C" __global__ void k_eval_row(SweepParams sp, int k, int obs, double* out) {
  extern __shared__ __align__(16) unsigned char xs_raw[];
  const DsDev& ds = sp.ds[k];
  const int lane = threadIdx.x;
  if (PMDI_XBYTES(ds) == 8u) {
    const double* src = (const double*)ds.x + (size_t)obs * ds.Dp;
    for (int q = lane; q < ds.Dp; q += 32) ((double*)xs_raw)[q] = src[q];
  } else {
    const int* src = (const int*)ds.x + (size_t)obs * ds.Dp;
    const int skip = ds.type == T_CATEGORICAL ? 0 : -1;
    for (int q = lane; q < ds.Dp; q += 32) ((int*)xs_raw)[q] = ds.flag[q] ? src[q] : skip;
  }
  __syncwarp();
  const long long row = sp.proto_base;
  const int n = ds.n[row];
  double acc = ds.rc[n];
  for (int j = 0; j < ds.J; ++j) {
    double v;
#ifdef PMDI_USER_TYPES
    if (ds.type == T_USER) {
      const int fo = j * ds.FB + 2 * lane;
      const int nits = min(ds.FB / PMDI_WF, (ds.Dp - j * ds.FB) / PMDI_WF);
      double unused;
      v = user_block(ds, ds.ust + row * user_row_words(ds) + fo, 0, ds.flag + fo, nits, 0, n, 0u,
                     (unsigned)__cvta_generic_to_shared(xs_raw) + fo * (ds.uW < 0 ? 4u : 8u), &unused);
    } else
#endif
    if (ds.type == T_GAUSSIAN) v = gauss_eval_block(ds, row, j, n, (const double*)xs_raw, lane);
    else if (ds.type == T_CATEGORICAL && sp.engine) {
      const PoolDev& pd = sp.pd[k];
      const int base = j * ds.FB + 2 * lane;
      const int nits = min(ds.FB / PMDI_WF, (ds.Dp - j * ds.FB) / PMDI_WF);
      double unused;
      v = cat_block(pd.cw + ((size_t)row * ds.Dp + base) * pd.wpf, 0, pd.wpf, pd.fpw, nits, 0, 0u,
                    (unsigned)__cvta_generic_to_shared(xs_raw) + base * 4u, &unused);
    }
    else if (ds.type == T_CATEGORICAL) v = cat_eval_block(ds, row, j, (const int*)xs_raw, lane);
    else v = nb_eval_block(ds, row, j, n, (const int*)xs_raw, lane, sp.lf_glob, sp.lf_glob_T);
    acc += v;
  }
  if (lane == 0) *out = acc;
}

// single-label prefix build used by pmdi_cluster_eval: members -> prototype row 0 of slot P
extern "C" __global__ void k_build_one(SweepParams sp, int k, const int* members, int cnt) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  const DsDev& ds = sp.ds[k];
  if (q >= ds.Dp) return;
  const long long row = sp.proto_base;
  build_row_feature(ds, sp.engine ? &sp.pd[k] : nullptr, row, q, members, cnt, 1);
  if (q == 0) ds.n[row] = cnt;
}
extern "C" __global__ void k_aux_one(SweepParams sp, int k) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const DsDev& ds = sp.ds[k];
  const long long row = sp.proto_base;
  const int n = ds.n[row];
  for (int j = w; j < ds.J; j += blockDim.x >> 5) {
    if (ds.type == T_GAUSSIAN) gauss_aux_block(ds, row, j, lane);
    else if (ds.type == T_NEGBINOM) nb_aux_block(ds, row, j, n, lane, sp.lf_glob, sp.lf_glob_T);
    else if (lane == 0) ds.aux[row * ds.J + j] = 0.0;
  }
}

// Predictive of the EMPTY cluster for every swept observation (it depends on the observation
// only): lp_empty[step][k] = calc_logprob(x_step, empty cluster of dataset k).  Every label with
// n == 0 of every particle shares this value.  One block per step; the same block operators as
// the sweep, applied to the shared empty row.
extern "C" __global__ void k_empty_lp(SweepParams sp, double* lp_empty) {
  extern __shared__ __align__(16) unsigned char xs_raw[];
  __shared__ double part[PMDI_MAX_K][32];
  const int step = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, NW = blockDim.x >> 5;
  const int obs = sp.order[sp.n1 - 1 + step];
  for (int k = 0; k < sp.K; ++k) {
    const DsDev& ds = sp.ds[k];
    const int words = ds.Dp * (ds.type == T_GAUSSIAN ? 2 : 1);
    const int* src = (const int*)ds.xstage + (size_t)obs * words;
    int* dst = (int*)(xs_raw + ds.x_off);
    for (int q = tid; q < words; q += blockDim.x) dst[q] = src[q];
  }
  __syncthreads();
  const long long row = (long long)(sp.Ps + 1) * sp.N;
  for (int it = warp; it < sp.K * sp.Jmax; it += NW) {
    const int k = it / sp.Jmax, j = it - k * sp.Jmax;
    const DsDev& ds = sp.ds[k];
    if (j >= ds.J) continue;
    double v;
    if (ds.type == T_GAUSSIAN) v = gauss_eval_block(ds, row, j, 0, (const double*)(xs_raw + ds.x_off), lane);
    else if (ds.type == T_CATEGORICAL) v = cat_eval_block(ds, row, j, (const int*)(xs_raw + ds.x_off), lane);
    else v = nb_eval_block(ds, row, j, 0, (const int*)(xs_raw + ds.x_off), lane, sp.lf_glob, sp.lf_glob_T);
    if (lane == 0) part[k][j] = v;
  }
  __syncthreads();
  if (tid < sp.K) {
    const DsDev& ds = sp.ds[tid];
    double a = ds.rc[0];
    for (int j = 0; j < ds.J; ++j) a += part[tid][j];
    lp_empty[(size_t)step * sp.K + tid] = a;
  }
}

// Observation matrix with the feature flags folded in (the sweep stages rows with plain async
// copies): unflagged / padded features become level 0 (categorical) or -1 (NegBinom).
extern "C" __global__ void k_mark_x(const int* x, const uint8_t* flag, int* xq, long long n, int Dp, int skip) {
  const long long total = n * Dp, stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride)
    xq[i] = flag[i % Dp] ? x[i] : skip;
}

// ------------------------------------------------------------------------------------------
// after the sweep kernel (every engine)
// ------------------------------------------------------------------------------------------

// Particle selection (src/pmdi.jl:345-350), lineage back-trace, s[:] = sstar[p_star,:,:] (:373),
// plus the reductions the host's update_hypers reads (src/update_hypers.jl:72,109-115): label counts
// per (label, dataset) and, per dataset pair, the number of observations with equal labels.
// One block.  The sums over the particles are sequential (same bits as the reference's cumsum), read
// from shared memory; the lineage changes at the resampling events only, so it is walked over the
// event list (a few entries) and every step looks its segment up.
#define FIN_PW 4096
#define FIN_EV 512
extern "C" __global__ void k_finish_pool(SweepParams sp, int compat, long long* s_out, long long* p_star_out,
                              int* cur_at, long long* label_counts, long long* pair_agree,
                              long long* contingency) {
  const int t = threadIdx.x, NT = blockDim.x, P = sp.P, K = sp.K, N = sp.N;
  __shared__ double red[32];
  __shared__ double w_s[FIN_PW];
  __shared__ int ev_step[FIN_EV], ev_cur[FIN_EV + 1];
  __shared__ int n_ev;
  const bool in_smem = P <= FIN_PW;
  double mx = -INFINITY;
#pragma unroll 1
  for (int p = t; p < P; p += NT) mx = fmax(mx, sp.lw_out[p]);
  mx = warp_max(mx);
  if ((t & 31) == 0) red[t >> 5] = mx;
  if (t == 0) n_ev = 0;
  __syncthreads();
  mx = red[0];
#pragma unroll 1
  for (int i = 1; i < (NT >> 5); ++i) mx = fmax(mx, red[i]);
#pragma unroll 1
  for (int p = t; p < P; p += NT) {
    const double w = exp(sp.lw_out[p] - mx);
    if (in_smem) w_s[p] = w; else sp.sc_w[p] = w;
  }
  // steps that ended with a resampling, by event number (events are numbered in step order)
#pragma unroll 1
  for (int st = t; st < sp.steps; st += NT) {
    const int ev = sp.ev_of_step[st];
    if (ev >= 0) { atomicMax(&n_ev, ev + 1); if (ev < FIN_EV) ev_step[ev] = st; }
  }
  __syncthreads();
  const int E = n_ev;
  if (t == 0) {
    const double* w = in_smem ? w_s : sp.sc_w;
    double tot = 0.0;
    for (int p = 0; p < P; ++p) tot += w[p];
    const double u = sp.tape_select ? sp.tape_select[0] : pmdi_philox_uniform(sp.seed, sp.iter, DRAW_SELECT, 0, 0, 0);
    const double thr = u * tot;
    int i = 0;
    double cw = w[0];
    while (cw < thr && i < P - 1) { ++i; cw += w[i]; }
    *p_star_out = i + 1;
    // lineage of p_star through the resampling events, backwards (src/__pmdi.jl:285)
    if (E <= FIN_EV) {
      ev_cur[E] = i;
      for (int e = E - 1; e >= 0; --e)
        ev_cur[e] = compat ? i : sp.anc_log[(size_t)e * P + ev_cur[e + 1]] - 1;
    } else {
      int cur = i;
      for (int st = sp.steps - 1; st >= 0; --st) {
        const int ev = sp.ev_of_step[st];
        if (ev >= 0 && !compat) cur = sp.anc_log[(size_t)ev * P + cur] - 1;
        cur_at[st] = cur;
      }
    }
  }
#pragma unroll 1
  for (size_t i = t; i < (size_t)K * sp.n_obs; i += NT) s_out[i] = sp.s_in[i];
#pragma unroll 1
  for (int i = t; i < N * K; i += NT) label_counts[i] = 0;
#pragma unroll 1
  for (int i = t; i < K * (K - 1) / 2; i += NT) pair_agree[i] = 0;
#pragma unroll 1
  for (int i = t; i < K * (K - 1) / 2 * N * N; i += NT) contingency[i] = 0;
  __syncthreads();
  if (E <= FIN_EV) {
    // the particle a step's allocation is read from: the lineage after undoing every event at or
    // after this step = entry of the first event whose step is >= st
#pragma unroll 1
    for (int st = t; st < sp.steps; st += NT) {
      int lo = 0, hi = E;
#pragma unroll 1
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (ev_step[mid] >= st) hi = mid; else lo = mid + 1; }
      cur_at[st] = ev_cur[lo];
    }
    __syncthreads();
  }
#pragma unroll 1
  for (int idx = t; idx < sp.steps * K; idx += NT) {
    const int st = idx / K, k = idx - st * K;
    const int obs = sp.order[sp.n1 - 1 + st];
    s_out[(size_t)k * sp.n_obs + obs] = 1 + sp.alloc_log[((size_t)st * K + k) * P + cur_at[st]];
  }
  __syncthreads();
#pragma unroll 1
  for (size_t i = t; i < (size_t)K * sp.n_obs; i += NT)
    atomicAdd((unsigned long long*)&label_counts[(i / sp.n_obs) * N + (s_out[i] - 1)], 1ull);
#pragma unroll 1
  for (int i = t; i < sp.n_obs; i += NT) {
    int idx = 0;
#pragma unroll 1
    for (int k1 = 0; k1 < K - 1; ++k1)
#pragma unroll 1
      for (int k2 = k1 + 1; k2 < K; ++k2) {
        const int la = (int)s_out[(size_t)k1 * sp.n_obs + i] - 1, lb = (int)s_out[(size_t)k2 * sp.n_obs + i] - 1;
        if (la == lb) atomicAdd((unsigned long long*)&pair_agree[idx], 1ull);
        atomicAdd((unsigned long long*)&contingency[((size_t)idx * N + lb) * N + la], 1ull);
        ++idx;
      }
  }
}

// Sizes of the final particles' clusters (out.cluster_n): computed when the caller asks for them.
extern "C" __global__ void k_cluster_n(SweepParams sp, long long* cluster_n) {
  const int P = sp.P, K = sp.K, N = sp.N;
  const int ev = (int)sp.counters[2];
  const size_t stride = (size_t)gridDim.x * blockDim.x;
#pragma unroll 1
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < (size_t)K * P * N; idx += stride) {
    const int k = (int)(idx / ((size_t)P * N));
    const size_t rem = idx - (size_t)k * P * N;
    const int p = (int)(rem / N), m = (int)(rem % N);
    long long v = -1;  // clusters of particles held by another rank: -1
    if (sp.engine == 0) {
      const int ls = sp.slot_of[(ev & 1) * P + p] - sp.slot0;
      if (ls >= 0 && ls < sp.Ps) v = sp.ds[k].n[(long long)ls * N + m];
    } else {
      const int ls = p - sp.slot0;
      if (ls >= 0 && ls < sp.Ps) {
        const PoolDev& pd = sp.pd[k];
        v = sp.ds[k].n[pd.rowmap[((size_t)(ev & 1) * sp.Ps + ls) * N + m]];
      }
    }
    cluster_n[idx] = v;
  }
}
#else

// k_eval_row for a dataset whose row does not fit in shared memory: the same operators, with the observation read
// from global memory (DsDev::xstage: the flags of Categorical / NegBinom data are folded in, as k_eval_row folds
// them while it stages).  One warp.
extern "C" __global__ void k_eval_row_wide(SweepParams sp, int k, int obs, double* out) {
  const DsDev& ds = sp.ds[k];
  const int lane = threadIdx.x;
  const unsigned char* xs = (const unsigned char*)ds.xstage + (size_t)obs * ds.Dp * PMDI_XBYTES(ds);
  const long long row = sp.proto_base;
  const int n = ds.n[row];
  double acc = ds.rc[n];
  for (int j = 0; j < ds.J; ++j) {
    double v;
#ifdef PMDI_USER_TYPES
    if (ds.type == T_USER) {
      const int fo = j * ds.FB + 2 * lane;
      const int nits = min(ds.FB / PMDI_WF, (ds.Dp - j * ds.FB) / PMDI_WF);
      double unused;
      v = user_block(ds, ds.ust + row * user_row_words(ds) + fo, 0, ds.flag + fo, nits, 0, n, xs,
                     xs + fo * (ds.uW < 0 ? 4u : 8u), &unused);
    } else
#endif
    if (ds.type == T_GAUSSIAN) v = gauss_eval_block(ds, row, j, n, (const double*)xs, lane);
    else if (ds.type == T_CATEGORICAL && sp.engine) {
      const PoolDev& pd = sp.pd[k];
      const int base = j * ds.FB + 2 * lane;
      const int nits = min(ds.FB / PMDI_WF, (ds.Dp - j * ds.FB) / PMDI_WF);
      double unused;
      v = cat_block(pd.cw + ((size_t)row * ds.Dp + base) * pd.wpf, 0, pd.wpf, pd.fpw, nits, 0, xs, xs + base * 4u,
                    &unused);
    }
    else if (ds.type == T_CATEGORICAL) v = cat_eval_block(ds, row, j, (const int*)xs, lane);
    else v = nb_eval_block(ds, row, j, n, (const int*)xs, lane, sp.lf_glob, sp.lf_glob_T);
    acc += v;
  }
  if (lane == 0) *out = acc;
}
#endif
