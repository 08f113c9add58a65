/*
 * Internal types shared by the host side (pmdi_capi) and the sm_100a kernels of libpmdi_cuda.so.
 *
 * HBM layout (DESIGN.md §3).  Every particle owns N clusters per dataset ("dense" form of the
 * reference's copy-on-write pool, src/pmdi.jl:131-146, SURVEY.md §9).  A cluster of dataset k
 * is a ROW r = slot*N + label of Dp feature-contiguous statistics, structure-of-arrays:
 *   Gaussian     mu[r][q], lamn[r][q] = lambda/(n+1), sum[r][q], beta[r][q]      (f64)
 *   Categorical  cnt[r][level][q]                                                (u32)
 *   NegBinom     S[r][q]                                                         (i64)
 * plus per row: n[r] (cluster size), aux[r][j] (x-independent part of the predictive, per
 * 256-feature block j), part[r][j] (this step's predictive partial sums).
 * Local slots 0..Ps-1 are particles (a logical->slot table over the P GLOBAL slots follows
 * resampling so that survivors are never copied), local slot Ps holds the rho-prefix prototypes,
 * local slot Ps+1 row 0 is the shared empty cluster that stands for every label with n == 0.
 */
#ifndef PMDI_INTERNAL_H
#define PMDI_INTERNAL_H
#ifdef __CUDACC_RTC__  /* compiled at run time for a user-defined cluster type (NVRTC has no host headers) */
typedef unsigned char uint8_t;
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;
#else
#include <stdint.h>
#endif

#define PMDI_MAX_K 8
#define PMDI_MAX_N 256
#define PMDI_FB 256 /* features per work item (one warp, 4 iterations of 64) */
#define PMDI_WF 64  /* features per warp iteration: 32 lanes x one 128-bit load */
#define PMDI_NT 512 /* threads per CTA of the sweep kernel */
#define PMDI_OBS_RING 4 /* observations in the sweep kernel's shared-memory ring (pool and spec: at most, as memory allows) */

enum { T_GAUSSIAN = 0, T_CATEGORICAL = 1, T_NEGBINOM = 2, T_USER = 3 /* registered device functor */ };
enum { DRAW_ALLOC = 0, DRAW_RESAMP = 1, DRAW_SHUFFLE = 2, DRAW_SELECT = 3, DRAW_FEATURE = 4 };

/* bytes per staged observation element: doubles for Gaussian data and for user types on Float64 data */
#define PMDI_XBYTES(ds_) (((ds_).type == T_GAUSSIAN || ((ds_).type == T_USER && (ds_).uW > 0)) ? 8u : 4u)

struct DsDev {
  int type, D, Dp, J;
  int Lmax, all_on, x_off /* byte offset of this dataset's row in the smem staging area */, nflag;
  int FB, uW;           /* features per block (one warp's share of a row; aux and J are per block): 256, spec engine 128;
                           user type: doubles of state per feature                                */
  double* ust;          /* user type: state [row][uW][Dp]                                          */
  const void* x;        /* [n_obs][Dp]: f64 (Gaussian) or i32 (others), row-major        */
  const void* xstage;   /* what the sweep stages: x, or x with the feature flags folded in */
  const uint8_t* flag;  /* [Dp], padded features are 0                                    */
  const double* rc;     /* [n_obs+1] x-independent row constant by cluster size           */
  double *mu, *lamn, *sum, *beta;
  uint32_t* cnt;
  long long* S;
  double* part;
  double* aux;
  int* n;
};

/*
 * Pool engine (pool_kernel.cuh): the reference's copy-on-write cluster pool (src/pmdi.jl:131-146,
 * 275-310) on the device.  A dataset's statistics rows are a POOL of `cap` physical rows; a particle
 * refers to its clusters through rowmap[slot][label] -> row.  Particles that have made the same
 * choices share rows; a row is evaluated once per observation whatever the number of particles that
 * refer to it, and resampling permutes row maps instead of moving statistics.  Row cap-1 is the
 * EMPTY cluster (never written; every unoccupied label of every particle refers to it).
 */
/* spec engine (spec_kernel.cuh): what the proposals read about a row at one observation step */
struct RowInfo {
  double lp;   /* predictive of the step's observation                                         */
  int child;   /* the row that holds (this row + the step's observation)                       */
  int pad;
};

struct PoolDev {
  int cap;           /* physical rows, row cap-1 = the empty cluster                         */
  int wpf, fpw;      /* categorical packing: 64-bit words per feature, count fields per word  */
  int pad;
  int* refcnt;       /* [cap] (particle, label) references of a row ([2][cap] in the spec engine)   */
  int* chosen;       /* [2][cap] by step parity: particles that chose the row this step ([3][cap] by step mod 3
                        in the spec engine)                                                    */
  int* dst;          /* [2][cap] by step parity: row id reserved for the split of the row     */
  int* n_eval;       /* [cap] cluster size the row's current predictive was evaluated with    */
  int* live;         /* [cap] list of live rows (live[0] = the empty cluster)                 */
  int* freelist;     /* [cap] stack of free rows                                              */
  int* rowmap;       /* [2][Ps][N] by resampling-event parity: label -> row of a particle slot */
  int* ctr;          /* [0] live rows, [1] free rows                                          */
  unsigned long long* cw; /* [cap][Dp][wpf] packed categorical counts                          */
  double* lp;        /* [cap] this step's predictive of every live row (E phase -> P phase)       */
  RowInfo* info;     /* spec engine: [2][cap] by step parity                                      */
  int* mark;         /* spec engine: [cap] rows a resampling must keep although nobody refers to them */
};

struct __attribute__((aligned(16))) SweepParams {
  int K, N, P, n_obs, n1, steps;
  int G, flags;
  /* particle sharding: R ranks (one GPU each), this one holds slots [slot0, slot0 + Ps) of the P global
     slots; peer_delta[r] turns a pointer into this rank's shared arena into the same object on rank r */
  int R, rank, Ps, slot0;
  long long peer_delta[8];
  DsDev ds[PMDI_MAX_K];
  PoolDev pd[PMDI_MAX_K];
  int engine;             /* 0 dense (sweep_kernel.cuh), 1 pool (pool_kernel.cuh), 2 spec (spec_kernel.cuh) */
  int GP;                 /* spec engine: CTAs 0..GP-1 propose, GP..G-1 evaluate               */
  unsigned char* dec;     /* spec engine: [steps] resampling decision after each step (0 unknown, 1 no, 2 yes) */
  unsigned long long* rows_spec; /* [K] row evaluations actually performed (live rows and their children) */
  int4* glist;            /* spec engine: [lcap] the live-row list a set-up / resampling leaves for the E-CTAs */
  int* gcnt;              /*              its length                                             */
  int4* elist;            /* spec engine: [2][E-CTAs][lcap] the E-CTAs' copies of the list beyond shared memory */
  long long lcap;
  int fc_target;          /* spec engine: free-row ids an E-CTA keeps cached per dataset        */
  int plan_smem;          /* spec engine: the resampling plan's scratch fits the D-CTA's shared memory */
  int pad1;
  unsigned long long* rows_add;  /* [K] clusters that had an observation added (pool / spec engines) */
  /* pool / spec engines: the barrier counters and the step tags of the rank partials run on from sweep to
     sweep (nothing a peer can reach is reset between sweeps, so the ranks need no host barrier) */
  unsigned long long tag_base;
  unsigned long long* bar_state;  /* [2] where the local / cross-rank counters stand; written at the end of a sweep */
  int obs_ring;           /* depth of the shared-memory observation ring (2..4)              */
  long long proto_base;   /* first row of the rho-prefix prototypes (dense: Ps*N, pool: 0)   */
  unsigned long long wd_ns; /* watchdog of the in-kernel waits                               */
  int4* pull_jobs;        /* resampling: (dataset, source rank, source row, local row) of rows to pull */
  int* pull_map;          /* spec engine, several ranks: [K][R][cap] local copy of a remote row during a resampling (-1: none) */
  double* rank_part;      /* [2][R][4] per step parity and rank: max, sum w, sum w^2, step tag */
  unsigned long long* rank_words; /* spec engine: [2][R][8] the same three doubles as six (tag << 32 | half) words: no fence */
  unsigned tag32;         /* ... tag of step t = tag32 + t + 1 (runs on over the sweeps of a context)          */
  unsigned long long* rows_ref; /* [K] occupied (particle, label) rows referenced by proposals */
  const double* Pi;      /* [K][N]                                          */
  const double* l1phi;   /* [npairs] log(1+phi)                             */
  const long long* s_in; /* [K][n_obs] labels 1..N                          */
  const int* order;      /* [n_obs] 0-based observation per position        */
  double lw_init;
  unsigned long long seed;
  unsigned iter;
  int Jmax;                /* max over datasets of J                          */
  const double *tape_alloc, *tape_resamp, *tape_shuffle, *tape_select;
  /* state */
  double* lw;             /* [P] log-weights by logical particle (each written by the CTA that owns the particle) */
  double* ess_part;       /* [2][G][3] per step parity and CTA: max log-weight, sum w, sum w^2 (w = exp(l - max)) */
  double* lw_out;         /* [P] final log-weights (written by CTA 0)        */
  int* slot_of;           /* [2][P] logical -> slot, double-buffered by resampling event */
  int* logical_of;        /* [2][P] slot -> logical                          */
  uint8_t* lab;           /* [2][K][P] by logical particle: label chosen this step (0-based), double-buffered by step */
  double* inc;            /* [2][K][P] by logical particle: incremental log-weight of this step  */
  const double* lp_empty; /* [steps][K] predictive of the empty cluster for every swept observation */
  uint8_t* alloc_log;     /* [steps][K][P] by logical particle               */
  int* anc_log;           /* [events][P] 1-based ancestors                   */
  int* ev_of_step;        /* [steps] event index or -1                       */
  /* resampling plan scratch (CTA 0) */
  double *sc_w, *sc_pp, *sc_u;
  int *sc_j, *sc_anc0, *sc_a, *sc_b, *sc_c, *sc_d;
  int2* copies;
  int* plan_out;          /* [0] number of copies of the current event       */
  /* static ownership of (dataset, slot) units by CTAs */
  const int* cta_off;
  const int* cta_units;   /* k << 24 | slot                                   */
  int max_units, sm_x_bytes;
  int lf_T, item_cap;   /* log-factorial entries in smem; capacity of the per-step item queue */
  int qb;               /* 256-feature blocks per plain work item (dense engine) */
  int jq;               /* pool engine: warps per row task = blocks per row rounded up to a power of two, <= 16 */
  const double* lf_glob;  /* log-factorial table in HBM [lf_glob_T]; its first lf_T entries are staged in smem */
  int lf_glob_T;
  unsigned* bar;          /* grid barrier arrival counter (64-bit, 16 bytes reserved) */
  int* err;
  unsigned long long* rows_eval; /* [K] rows evaluated                        */
  long long* counters;    /* [0] events, [1] copies                           */
  unsigned long long* phase_ns;  /* [G][8] per-CTA per-phase time (optional)  */
  /* per-warp event trace of one CTA and one step (optional): [NW][128] (tag << 48 | clock) */
  unsigned long long* trace;
  int trace_cta, trace_step;
  int* wd_state;          /* [G][NW][16] where every warp was when a watchdog fired */
  /* debug capture */
  double* dbg_lp;
  double* dbg_lw;
  int* dbg_alloc;
  int* dbg_anc;
};

#endif
