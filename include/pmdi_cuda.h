/*
 * libpmdi_cuda.so — C-ABI of the B200-native conditional-SMC allocation sweep of ParticleMDI.
 *
 * This is the drop-in boundary for the hot path of nathancunn/ParticleMDI.jl: everything
 * `pmdi()` does between `shuffle!(order_obs)` and `align_labels!` in one MCMC iteration
 * (reference src/pmdi.jl:188-370).  The reference is pure Julia with no FFI; these are the
 * entry points a Julia `ccall` binding (INTEGRATION.md) or any other host uses instead of the
 * Julia loops.  Plain pointers and sizes only; array layouts are Julia's (column-major,
 * 1-based labels and indices, Int64 / Float64) so that Julia arrays are passed without copies.
 *
 * Conventions: every function returns 0 on success and a non-zero code on failure, with
 * `pmdi_last_error()` giving the message (the reference's only error convention is Julia
 * exceptions / `@assert`, src/pmdi.jl:50-55).  A context is not thread-safe.  There is no CPU
 * fallback: without a CUDA device every compute entry point fails.
 */
#ifndef PMDI_CUDA_H
#define PMDI_CUDA_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* cluster type tags — replace Julia dispatch on dataTypes[k] (src/pmdi.jl:122,189,219,300) */
#define PMDI_GAUSSIAN    0 /* ParticleMDI.GaussianCluster    src/datatypes/gaussian_cluster.jl:11-83    */
#define PMDI_CATEGORICAL 1 /* ParticleMDI.CategoricalCluster src/datatypes/categorical_cluster.jl:2-66  */
#define PMDI_NEGBINOM    2 /* ParticleMDI.NegBinomCluster    src/datatypes/negbinom_cluster.jl:6-60     */

/* element kinds of a host data matrix */
#define PMDI_F64 0
#define PMDI_I64 1

/* pmdi_sweep_args.flags */
#define PMDI_SWEEP_DEBUG        1u /* capture per-step lp / log-weights / allocations / ancestors */
#define PMDI_SWEEP_SSTAR_COMPAT 2u /* emit allocations without following ancestors, as pmdi() does
                                      (src/pmdi.jl:321-324; the tested twin src/__pmdi.jl:285 follows them) */
#define PMDI_SWEEP_TIME_PHASES  4u /* every CTA accumulates per-phase wall time of the sweep kernel (globaltimer) */

typedef struct pmdi_ctx pmdi_ctx;

const char* pmdi_last_error(void);
int pmdi_version(void);

/* Number of CUDA devices visible (0 when there is none; never fails). */
int pmdi_device_count(void);

/*
 * Create a context for K datasets of n_obs rows, at most N clusters, `particles` particles
 * (the arguments of pmdi(), src/pmdi.jl:36-40; same pre-conditions as its asserts :50-55:
 * 1 < N <= n_obs, particles > 1; additionally N <= 256).  `device` is the CUDA ordinal.
 */
int pmdi_ctx_create(pmdi_ctx** out, int32_t K, int64_t n_obs, int32_t N, int32_t particles,
                    int32_t device);
int pmdi_ctx_destroy(pmdi_ctx* ctx);

/*
 * Particle sharding over the GPUs of one node (SURVEY.md 8(e)): one context per GPU / process.
 * Every rank binds the SAME datasets and is created with the GLOBAL particle count; rank r holds
 * particles' statistics for P / n_ranks slots.  Per observation the ranks exchange their ESS
 * partials, log-weights and allocations with NVLink peer stores from inside the sweep kernel, and
 * resampled ancestors held by another rank are pulled through peer memory - no host round trip.
 *   pmdi_ctx_set_ranks   before the first sweep (after pmdi_ctx_create);
 *   pmdi_ipc_export      after all datasets are bound: the CUDA IPC handle of this rank's arena;
 *   pmdi_ipc_import      all ranks' handles, in rank order (exchange them with any host mechanism).
 * Every rank then calls pmdi_sweep (or upload / run / download) with identical arguments, the same number of
 * times; every rank returns the same allocations.  No host synchronisation between the ranks is needed: the
 * in-kernel counters and step tags run on from sweep to sweep.  (Only the dense engine, PMDI_ENGINE=dense,
 * restarts its counters: there a host barrier over all ranks belongs between upload and run.)
 */
#define PMDI_IPC_HANDLE_BYTES 64
int pmdi_ctx_set_ranks(pmdi_ctx* ctx, int32_t rank, int32_t n_ranks);
int pmdi_ipc_export(pmdi_ctx* ctx, void* handle_out /* PMDI_IPC_HANDLE_BYTES */, int64_t* arena_bytes);
int pmdi_ipc_import(pmdi_ctx* ctx, const void* handles /* n_ranks x PMDI_IPC_HANDLE_BYTES */,
                    const int64_t* arena_bytes /* n_ranks, may be NULL */);

/*
 * The engine of this context, ahead of PMDI_ENGINE and of the default rule (spec for K <= 4, pool above; pool for user
 * types on one GPU).  PMDI_ENGINE_AUTO keeps that rule; the numbering is that of pmdi_sweep_out.engine.  An
 * environment variable is process-wide: this lets one context (a member of a group, say) run the spec engine without
 * changing the engine of every other context.  The dense engine is not offered here (PMDI_ENGINE=dense).  Valid only
 * before the context is first prepared (its first upload, sweep, feature, cluster-eval or IPC export call): the
 * memory layout depends on the engine, and a later call fails.
 */
#define PMDI_ENGINE_AUTO (-1)
#define PMDI_ENGINE_POOL 1
#define PMDI_ENGINE_SPEC 2
int pmdi_ctx_set_engine(pmdi_ctx* ctx, int32_t engine);

/*
 * Whether the context sweeps with the wide kernels (*wide = 1) or the staged ones (0); valid once the context is
 * prepared (its first upload, sweep, feature, cluster-eval or IPC export call).  The pool and spec sweeps stage each
 * observation over all datasets in shared memory, two deep, beside their tables.  A context is wide when that does
 * not fit with its N and particle count, or when a dataset has more than 8,192 features; its sweeps then read the
 * observation from global memory instead, with the same results.  The choice is automatic.  PMDI_ENGINE=dense on a
 * wide context runs the pool engine (pmdi_sweep_out.engine says so).  Wide contexts are not yet supported in groups
 * (pmdi_group_create refuses such a member, naming it) or with their particles sharded over GPUs (refused when the
 * context is prepared).
 */
int pmdi_ctx_is_wide(const pmdi_ctx* ctx, int32_t* wide);

/* Use an externally owned cudaStream_t (e.g. the host framework's current stream). */
int pmdi_ctx_set_stream(pmdi_ctx* ctx, void* cuda_stream);
void* pmdi_ctx_get_stream(pmdi_ctx* ctx);

/*
 * Bind dataset k (replaces `dataTypes[k](dataFiles[k])`, src/pmdi.jl:122,189,194).
 * `data` is a HOST column-major n_obs x D matrix with leading dimension `ld` (Julia
 * Matrix{Float64} for PMDI_GAUSSIAN, Matrix{Int64} for the others: levels 1..L for
 * categorical, counts >= 0 for negative-binomial).  It is copied to the device; the caller
 * keeps ownership.  All feature flags are reset to true.  1 <= D <= 65,536 features per dataset; the total width
 * over the datasets is limited by device memory alone (the context's arena grows linearly with every D: the
 * preparing call fails with the bytes it needs and the bytes free when they do not fit).
 */
int pmdi_set_dataset(pmdi_ctx* ctx, int32_t k, int32_t type_tag, int32_t elem_kind,
                     const void* data, int64_t n_obs, int64_t D, int64_t ld);

/* featureFlag[k] (src/pmdi.jl:106-110,367): D bytes, non-zero = feature used by the sweep. */
int pmdi_set_feature_flags(pmdi_ctx* ctx, int32_t k, const uint8_t* flags);

typedef struct pmdi_sweep_args {
  uint32_t flags;
  uint32_t iter;             /* MCMC iteration number, part of the RNG address               */
  uint64_t seed;             /* RNG seed (Philox4x32-10 keyed per draw)                       */
  const int64_t* s;          /* n_obs x K column-major current allocations, labels 1..N       */
  const int64_t* order_obs;  /* n_obs, 1-based permutation (src/pmdi.jl:172)                  */
  int64_t n1;                /* floor(rho * n_obs) >= 1 (src/pmdi.jl:161)                     */
  const double* Pi;          /* N x K column-major normalised weights (src/pmdi.jl:179)       */
  const double* phi;         /* K(K-1)/2 values, pair order (1,2),(1,3).. (src/misc.jl:1-13); may be NULL when K==1 */
  double logweight_init;     /* 0.0 first iteration, 1.0 afterwards (src/pmdi.jl:99,372)      */
  /* optional tapes of uniforms (deterministic mode: "the reference's draws are fed in");
     NULL -> the draw comes from Philox(seed, iter, kind, step, k, index) */
  const double* tape_alloc;   /* [steps][K][P], entry p used for particle p >= 2 (src/pmdi.jl:253) */
  const double* tape_resamp;  /* [steps]    rand() of draw_partstar (src/misc.jl:28)          */
  const double* tape_shuffle; /* [steps][P] entry i-1 drives the shuffle! pick for position i (src/misc.jl:43) */
  const double* tape_select;  /* [1]        p_star draw (src/pmdi.jl:350)                     */
} pmdi_sweep_args;

typedef struct pmdi_sweep_out {
  int64_t* s;             /* n_obs x K column-major new allocations (src/pmdi.jl:373)         */
  int64_t* p_star;        /* 1-based selected particle (src/pmdi.jl:350)                      */
  double*  logweight;     /* P log-weights before the final reset (src/pmdi.jl:345), may be NULL */
  int64_t  n_resamples;   /* resampling events in this sweep                                  */
  int64_t  n_copies;      /* particle stat blocks moved by resampling (all ranks)             */
  int64_t  n_remote_rows; /* cluster rows this rank pulled from another rank's GPU (NVLink)   */
  int64_t  n_evals;       /* cluster*feature predictive terms actually evaluated: every distinct cluster
                             once per observation (the reference's calc_logprob calls, src/__pmdi.jl:187,
                             times D_k); all empty labels share one evaluation per step        */
  int64_t  n_evals_dense; /* steps * P * N * sum_k D_k: the dense count of SURVEY.md 8(d)      */
  int64_t  rows_evaluated[8]; /* per dataset: cluster rows evaluated over the sweep           */
  double   device_ms;     /* device time of the whole sweep (prefix .. selection), CUDA events */
  double   sweep_kernel_ms;  /* device time of the persistent per-observation kernel alone    */
  double   phase_ms[8];   /* with PMDI_SWEEP_TIME_PHASES: per-warp time by phase, mean over CTAs.
                             engine 2 (spec): 0 waiting at the grid barrier, 1 row evaluations (E-CTAs),
                               2 proposals + commits (P-CTAs), 3 outcome bookkeeping (E-CTAs), 6 resampling,
                               4 / 5 / 7 sub-phases of the resampling (all CTAs in + plan; row maps + pulls; rebuild)
                             engine 1 (pool): 0 wait at B1, 1 evaluations, 2 proposals, 3 resolve, 4 wait at B2, 6 resampling
                             engine 0 (dense): 0 idle / waiting, 1 work items, 2 proposals, 6 resampling   */
  double   phase_ms_max[8]; /* same phases, maximum over CTAs                                  */
  /* debug capture, used when PMDI_SWEEP_DEBUG is set; each may be NULL */
  double*  dbg_lp;        /* [steps][K][P][N]                                                 */
  double*  dbg_lw;        /* [steps][P] after coupling, before resampling                     */
  int32_t* dbg_alloc;     /* [steps][K][P] 1-based                                            */
  int32_t* dbg_anc;       /* [steps][P] 1-based ancestors, 0 when the step did not resample   */
  int64_t* cluster_n;     /* [K][P][N] occupancy of every particle's clusters after the sweep
                             (-1 for particles held by another rank) */
  /* device reductions over the NEW allocations for the host's update_hypers (may be NULL):      */
  int64_t* label_counts;  /* N x K column-major: observations per (label, dataset) = countn(s[:,k], N),
                             src/update_hypers.jl:72                                            */
  int64_t* pair_agree;    /* K(K-1)/2, pair order (1,2),(1,3)..: observations with equal labels in
                             both datasets, src/update_hypers.jl:109-115                        */
  int64_t  rows_referenced[8]; /* per dataset: occupied (particle, label) clusters the proposals read;
                             rows_evaluated counts each physical row once per observation       */
  int32_t  engine;        /* 2 copy-on-write pool, evaluations one observation ahead (one grid barrier per step);
                             1 copy-on-write pool, two barriers per step; 0 dense                 */
  int64_t  rows_evaluated_ahead; /* pool engine: rows evaluated for observation t+1 before the resampling
                             decision of step t removed them (evaluation runs ahead of the ESS test);
                             rows_evaluated - rows_evaluated_ahead = the reference's calc_logprob calls */
  int64_t  rows_computed[8]; /* per dataset: row evaluations the device performed.  Engine 2 evaluates every
                             live row AND its child (the row plus the previous observation) one step ahead,
                             so this is about twice rows_evaluated; engines 0/1: equal to rows_evaluated  */
  int64_t  rows_added[8]; /* per dataset: clusters that had an observation added (the reference's cluster_add!
                             calls, src/pmdi.jl:275-310: one per DISTINCT chosen cluster and step; dense: one per
                             particle and step)                                                    */
  int64_t* contingency;   /* K(K-1)/2 tables of N x N (column-major, pair order as pair_agree): entry (la, lb) of
                             pair (a, b), a < b = observations with label la in dataset a and lb in dataset b under
                             the NEW allocations - everything align_labels! (src/misc.jl:61-108) counts; may be NULL */
} pmdi_sweep_out;

/*
 * One conditional-SMC sweep = src/pmdi.jl:188-350 + :373 (prefix build, per-observation
 * predictive / allocation / weight / resampling loop, particle selection, allocations out).
 * Host pointers in, host pointers out; the observation loop runs entirely on the device.
 * pmdi_sweep == pmdi_sweep_upload + pmdi_sweep_run + pmdi_sweep_download.
 */
int pmdi_sweep(pmdi_ctx* ctx, const pmdi_sweep_args* args, pmdi_sweep_out* out);
/* upload: validates the arguments, copies them into a pinned block of the context and queues ONE host -> device
   copy on the context's stream; returns without waiting for the device (the arguments may be reused at once;
   a second upload waits until the first one's copy has left the pinned block).  download: queues ONE
   device -> host copy of the result block, synchronises the stream, hands the results out. */
int pmdi_sweep_upload(pmdi_ctx* ctx, const pmdi_sweep_args* args);   /* host -> device inputs   */
int pmdi_sweep_run(pmdi_ctx* ctx);                                   /* asynchronous, on stream */
int pmdi_sweep_download(pmdi_ctx* ctx, pmdi_sweep_out* out);         /* sync + device -> host   */

/*
 * Groups: several independent contexts (chains) swept in ONE cooperative launch of the spec engine on one GPU.  A
 * chain of the spec engine is bound by the latency of its per-observation steps and leaves most of the GPU idle; a
 * group runs the members' grids side by side, each with its own barrier counter, so that several chains (other seeds,
 * other N, other data) share the GPU instead of taking turns on it.  Results are those of each member swept alone.
 *   pmdi_group_create  1..16 contexts, all on the same device, each on one GPU (not sharded) and on the spec engine
 *                      (built-in types: K <= 4 and PMDI_ENGINE not pool / dense, or pmdi_ctx_set_engine; user types:
 *                      pmdi_ctx_set_engine(ctx, PMDI_ENGINE_SPEC) or PMDI_ENGINE=spec, since their one-GPU default
 *                      is pool); a context is in at most one group.  Members with user-defined cluster types must all
 *                      have the same types in the same slot order (the types of their own compiled programs); members
 *                      with built-in types only may join them.  Such a group runs the group kernels compiled at run time
 *                      with those types (NVRTC, see pmdi_group_type_check); a group of built-in members runs the ones
 *                      built into this library.  Every member's datasets must be bound.  Each member gets a share of the SMs:
 *                      the grid it has alone when the grids fit side by side, otherwise a share of the SM count in
 *                      proportion to those grids (two 117-CTA members: 74 CTAs each).  Its role split and shared
 *                      memory follow the share; a member whose share is too small for it (at least one proposal, one
 *                      evaluation and the deciding CTA, and its tables in shared memory), or that would be wide at its
 *                      share (pmdi_ctx_is_wide), makes the create fail with a message that names it, and nothing changes.
 *   pmdi_group_run     after pmdi_sweep_upload on every member: each member's set-up kernels, one launch of the
 *                      group kernel, each member's finish, all on the group's own stream (it waits for the members'
 *                      uploads); then pmdi_sweep_download on each member as after pmdi_sweep_run.  A member's
 *                      sweep_kernel_ms is the group kernel's time.  With PMDI_SWEEP_DEBUG on any member the
 *                      instrumented twin runs; only the members that asked capture.  PMDI_TRACE_STEP is refused.
 *   pmdi_group_destroy gives every member the whole GPU back (and unloads the group's compiled kernels).
 * A member can still be swept alone (pmdi_sweep), on its share of the SMs; its barrier counters and step tags run on
 * from sweep to sweep whether a sweep ran alone or in the group.  Creating or destroying a group re-sizes the members'
 * grids: upload again before the next run.  pmdi_ctx_destroy of a member detaches it from its group (after any group
 * launch in flight has finished); pmdi_group_run then fails until the group is destroyed.
 */
typedef struct pmdi_group pmdi_group;
#define PMDI_GROUP_MAX_MEMBERS 16
int pmdi_group_create(pmdi_group** out, pmdi_ctx* const* members, int32_t n_members);
int pmdi_group_destroy(pmdi_group* group);
int pmdi_group_run(pmdi_group* group);
/* Compiles the group kernels for these user types (tags of pmdi_register_cluster_type, 1..8, in slot order) now, with
 * no GPU, into the cache pmdi_group_create compiles through; the log is in pmdi_last_error(). */
int pmdi_group_type_check(const int32_t* tags, int32_t n);

/*
 * Feature selection (src/pmdi.jl:120-128 and :354-370).
 * pmdi_feature_null: out[q] = -calc_logmarginal(all n_obs rows in one cluster)[q].
 * pmdi_feature_select: prob[q] = feature_null[q] + sum over occupied labels of
 *   calc_logmarginal(cluster rebuilt from the rows with that label, all features on);
 *   flags[q] = (1 - 1/exp(prob[q]+1)) > u_q, u_q from tape_f (may be NULL -> Philox).
 * `labels` = n_obs labels 1..N of dataset k (a column of s).  Does not change the flags bound
 * to the context; call pmdi_set_feature_flags with the result as pmdi() does.
 */
int pmdi_feature_null(pmdi_ctx* ctx, int32_t k, double* out_D);
int pmdi_feature_select(pmdi_ctx* ctx, int32_t k, const int64_t* labels,
                        const double* feature_null, uint64_t seed, uint32_t iter,
                        const double* tape_f, double* out_prob_D, uint8_t* out_flags_D);

/*
 * Plugin contract, one call each (used by the parity tests and by hosts that want single
 * evaluations): build a cluster of dataset k from `m` rows (1-based indices, in the order
 * given) under the context's feature flags, then
 *   out_logprob  = calc_logprob(row `obs`, cluster, flags)   (may be NULL)
 *   out_logmarg  = calc_logmarginal(cluster)  [D values]     (may be NULL)
 */
int pmdi_cluster_eval(pmdi_ctx* ctx, int32_t k, const int64_t* rows, int64_t m, int64_t obs,
                      double* out_logprob, double* out_logmarg_D);

/*
 * User-defined cluster types as device functors (the reference's plugin contract, README.md:48-88 and the
 * dispatch sites src/pmdi.jl:122,189,219,300,365: a user struct with calc_logprob / cluster_add! /
 * calc_logmarginal).  `cuda_src` is CUDA C++ source that defines a struct named `struct_name` with
 *
 *   static constexpr int WORDS;                                         doubles of state per feature (1..8)
 *   __device__ static void   init(double* st);                          the empty cluster
 *   __device__ static double logprob(const double* st, int n, double x);   this feature's term of calc_logprob
 *                                                                       (n = cluster size, x = the observation)
 *   __device__ static void   add(double* st, int n, double x);          cluster_add!; n = size AFTER the add
 *   __device__ static double logmarginal(const double* st, int n);      this feature's calc_logmarginal
 *
 * (every cluster type of the reference has this form: feature-wise sufficient statistics, log-probability a sum
 * over features).  elem_kind: PMDI_F64 or PMDI_I64, the element type of the data the type is bound to.
 * Returns the type tag (>= 16) for pmdi_set_dataset; registering a name again replaces its source and keeps the tag.
 *
 * A context may bind a different user type to each of its K datasets (up to K <= 8 distinct types).  When it is
 * first prepared, its user types are compiled (NVRTC, sm_100a) into ONE program together with a private copy of
 * this library's set-up kernels and the sweep kernel of the context's engine; each source goes into a namespace of
 * its own, so two types may both name their struct `Cluster`.  A compile error is reported then, with the
 * compiler's log in pmdi_last_error().  WORDS sizes the type's statistics before anything is compiled: it is read
 * from the source text (the number after the first "WORDS ... =") and the compiler checks it against the struct's
 * constant; a source whose text says otherwise (a comment `// WORDS = 2` above the declaration) fails to compile
 * with a message that names the type.
 *   Engines: on one GPU a context with user types runs the pool engine unless PMDI_ENGINE=spec or
 *   pmdi_ctx_set_engine asks for the speculative one; with the particles sharded the rule of the built-in types applies
 *   (spec for K <= 4, pool above).  PMDI_ENGINE=pool / spec are honoured; the dense engine has no user hooks,
 *   PMDI_ENGINE=dense runs pool.  Contexts with user types on the spec engine can be swept together in a group
 *   (pmdi_group_create): the group compiles a program of its own, the "spec-group" program, with the group kernels.
 *   Compile time: about 10-20 s of CPU per program (the spec engine's is the larger).  Programs are cached per
 *   process by kind (pool, spec, spec-group) and (struct name, element kind, source) of every type in slot order: another context with
 *   the same types loads the cached one.  A type registered again with another source is recompiled for contexts
 *   prepared afterwards; a context keeps the program it has.  PMDI_JIT_LOG set: one line per compile (with its
 *   wall time) or cache hit on stderr.
 *   Sharded particles: every rank registers its types in its own process (pmdi() does); pmdi_ipc_import rejects
 *   ranks whose arena layouts - WORDS of the types included - disagree.
 */
int pmdi_register_cluster_type(const char* name, const char* cuda_src, const char* struct_name, int32_t elem_kind,
                               int32_t* out_tag);
/* Compiles a registered type now, alone in its program (no GPU needed), and reports the compiler's verdict; the log
 * is in pmdi_last_error().  tag = PMDI_ALL_USER_TYPES: every type registered in this process, in registration order,
 * in one program (at most 8).  The program is the pool engine's, or the spec engine's when PMDI_ENGINE=spec; it
 * goes into the cache a context compiles through. */
#define PMDI_ALL_USER_TYPES (-1)
int pmdi_cluster_type_check(int32_t tag);

/*
 * Posterior similarity matrices on the device (src/output_analysis/consensus_map.jl:31-65: for every
 * retained iteration and dataset, psm[i, j] += (s[i] == s[j])).
 *   pmdi_psm_begin  zeroes K accumulators of n_obs x n_obs counts on the context's device
 *   pmdi_psm_add    adds one allocation matrix (n_obs x K column-major, labels 1..N)
 *   pmdi_psm_get    out[k][i][j] = count / samples as doubles (K * n_obs * n_obs values)
 */
int pmdi_psm_begin(pmdi_ctx* ctx);
int pmdi_psm_add(pmdi_ctx* ctx, const int64_t* s);
int pmdi_psm_get(pmdi_ctx* ctx, double* out);

/*
 * Posterior summaries of retained allocations, for one chain or several, with no sweep context: the reference's
 * generate_psm (src/output_analysis/consensus_map.jl:31-65, per dataset and "Overall"), the least-squares consensus
 * partition of Dahl (2006), and how far the chains' PSMs are apart.  The added samples stay on the device (n_obs * K
 * bytes each), and the pair counts are kept as exact uint32 (about 2 * n_obs^2 * K * chains bytes).  DESIGN.md §14.
 *   pmdi_summary_create     K datasets (1..8) of n_obs observations (1..65,535), labels 1..N (N <= 256), `chains`
 *                           chains (1..64), on `device`.  Refuses, before allocating, a footprint that does not fit in
 *                           the free device memory (counts, one chunk of samples per chain, one n_obs^2 read-out); the
 *                           message states the bytes needed.
 *   pmdi_summary_add        adds `rows` allocation matrices to chain `chain` (0-based), each n_obs x K column-major int64
 *                           as pmdi_sweep takes them, one after another.  Every label must be in 1..N (checked first:
 *                           a refused call adds nothing).  Copies through pinned staging on the summary's own stream and
 *                           returns without waiting for the device; `s` may be reused at once.  Every 256 samples of a
 *                           chain, and before any result below, the counts are brought up to date.  At most 2^24 rows in all.
 *   pmdi_summary_rows       rows added to chain `chain` (-1 with the error in pmdi_last_error()).
 *   pmdi_summary_psm        the full n_obs x n_obs PSM, row-major: count / rows (a true division of exact values, so it
 *                           equals the same division done in f64 on the host bit for bit).  chain = -1 pools the chains
 *                           (counts summed, divided by all rows); k = -1 is "Overall", (sum over k in order of PSM_k) / K.
 *                           out is double, or float (the double result rounded) when as_f32 != 0.
 *   pmdi_summary_ls         least-squares consensus of dataset k against the pooled PSM pi: for every sample r, in add
 *                           order chain by chain, loss_out[r] = sum_{i<j} (delta_r(i,j) - pi_ij)^2 (computed exactly in
 *                           integers, then rounded twice: to double, and in the division by rows^2).  best_chain / best_row: the lowest loss, the earliest sample
 *                           on ties; partition_out: its n_obs labels 1..N.  Any output may be NULL.
 *   pmdi_summary_agreement  chains >= 2: for every pair of chains a < b (row-major) and dataset k, out[pair * K + k] =
 *                           max (max_out) and mean (mean_out) over i < j of |PSM_a(i,j) - PSM_b(i,j)|.
 *   pmdi_summary_destroy    waits for the summary's work and frees everything.
 */
typedef struct pmdi_summary pmdi_summary;
int pmdi_summary_create(pmdi_summary** out, int32_t device, int32_t K, int64_t n_obs, int32_t N, int32_t chains);
int pmdi_summary_add(pmdi_summary* summary, int32_t chain, const int64_t* s, int64_t rows);
int64_t pmdi_summary_rows(const pmdi_summary* summary, int32_t chain);
int pmdi_summary_psm(pmdi_summary* summary, int32_t chain, int32_t k, void* out, int32_t as_f32);
int pmdi_summary_ls(pmdi_summary* summary, int32_t k, double* loss_out, int32_t* best_chain, int64_t* best_row,
                    int64_t* partition_out);
int pmdi_summary_agreement(pmdi_summary* summary, double* max_out, double* mean_out);
int pmdi_summary_destroy(pmdi_summary* summary);
/* Host only (no device needed): the allocation columns of `rows` CSV rows of pmdi()'s output (header excluded), one
 * row per line.  Each row's first `skip` columns are skipped, then `count` labels are read, written as integers
 * ("12" or "12.0"), into out[row * count + column].  Anything else (a fractional label, too few or too many columns or
 * rows) fails with the row and byte in pmdi_last_error(). */
int pmdi_parse_allocations(const char* text, int64_t len, int64_t rows, int32_t skip, int64_t count, int64_t* out);

/* The uniform the sweep uses for (kind, step, k, index); kinds as in the sweep:
   0 allocation, 1 resampling offset, 2 shuffle pick, 3 selection, 4 feature flag. */
double pmdi_uniform(uint64_t seed, uint32_t iter, uint32_t kind, uint32_t step, uint32_t k,
                    uint32_t index);

#ifdef __cplusplus
}
#endif
#endif /* PMDI_CUDA_H */
