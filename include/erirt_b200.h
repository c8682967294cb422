/*
 * erirt_b200.h -- C ABI of the B200-native Gibbs sweep engine for ExtendedRtIrtModeling.jl.
 *
 * Drop-in boundary (SURVEY.md 8b): the reference has no FFI; its boundary is the Julia method table
 *   sample!(MCMC::T; intercept, itemtype, cov2one)
 * for T in GibbsMlIrt (/root/reference/src/GibbsRtIrt.pl.jl:210), GibbsRtIrt (:278), GibbsRtIrtNull (:367),
 * GibbsRtIrtCross (src/GibbsRtIrtCross.pl.jl:176), GibbsRtIrtCrossQr (:265),
 * GibbsRtIrtLatent (src/GibbsRtIrtLatent.pl.jl:168), GibbsRtIrtLatentQr (:271; README's GibbsRtIrtQuantile).
 * A Julia `sample!` shim (julia/ErirtB200.jl, INTEGRATION.md) calls the functions below through `ccall`:
 *   erirt_create      <- MCMC.Cond::SimConditions            (src/Base.pl.jl:45-62) + sample! kwargs
 *   erirt_set_data    <- MCMC.Data::InputData Y, logT, X      (src/Base.pl.jl:67-78)
 *   erirt_set_state   <- MCMC.Para::InputPara initial values  (setInitialValues, src/GibbsRtIrt.pl.jl:84-133)
 *   erirt_sample      <- the `for m in 1:nIter, l in 1:nChain` loop body (src/GibbsRtIrt.pl.jl:289-324)
 *   erirt_get_trace   -> Post.ra / Post.rt / Post.qr / Post.logLike, Julia layout [nIter, P, nChain] (:319-323)
 *   erirt_get_moments -> Post.mean.θ / ζ / ν (and SDs) when the person trace is not kept (SURVEY 0.10)
 *
 * Conventions: every function returns 0 on success or a negative ERIRT_E_* code; the message is available
 * from erirt_last_error() (thread-local).  No C++ exception crosses this boundary.  Host buffers are owned
 * by the caller and are not retained after a call returns.  One caller thread per handle.  There is NO CPU
 * fallback: without a usable sm_100 CUDA device erirt_create fails with ERIRT_E_CUDA.
 */
#ifndef ERIRT_B200_H
#define ERIRT_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define ERIRT_ABI_VERSION 1

enum erirt_model {
  ERIRT_MLIRT = 0, ERIRT_RTIRT = 1, ERIRT_RTIRT_NULL = 2, ERIRT_RTIRT_CROSS = 3, ERIRT_RTIRT_CROSSQR = 4,
  ERIRT_RTIRT_LATENT = 5, ERIRT_RTIRT_LATENTQR = 6 /* == GibbsRtIrtQuantile */
};
enum erirt_dtype { ERIRT_F32 = 0, ERIRT_F64 = 1 };
enum erirt_error {
  ERIRT_OK = 0, ERIRT_E_ARG = -1, ERIRT_E_CUDA = -2, ERIRT_E_STATE = -3, ERIRT_E_NCCL = -4, ERIRT_E_UNSUPPORTED = -5,
  ERIRT_E_NUMERIC = -6
};
/* compat flags; 0 reproduces the reference source as written (SURVEY quirk register) */
enum erirt_compat { ERIRT_COMPAT_BETA_PRIOR_DIAG = 1, ERIRT_COMPAT_LATENTQR_SCALE_ELEMENTWISE = 2 };

/* state / trace selectors */
enum erirt_field {
  ERIRT_THETA = 0, ERIRT_ZETA = 1, ERIRT_A = 2, ERIRT_B = 3, ERIRT_LAMBDA = 4, ERIRT_SIGMA2 = 5, ERIRT_BETA = 6,
  ERIRT_RHO = 7, ERIRT_SIGMA_P = 8, ERIRT_NU = 9, ERIRT_OMEGA = 10
};
enum erirt_trace { ERIRT_TRACE_RA = 0, ERIRT_TRACE_RT = 1, ERIRT_TRACE_QR = 2, ERIRT_TRACE_LOGLIKE = 3 };

typedef struct erirt_handle erirt_handle;

typedef struct erirt_config {
  int32_t abi_version;    /* ERIRT_ABI_VERSION */
  int32_t model;          /* enum erirt_model */
  int64_t n_subj;         /* persons held by THIS handle (a shard of one chain, or all of them) */
  int64_t n_subj_total;   /* persons of the whole chain (== n_subj when not sharded) */
  int64_t subj_offset;    /* global id of this handle's first person (RNG counters use global ids) */
  int32_t n_item, n_feat;
  int32_t n_iter, n_chain; /* Cond.nIter, Cond.nChain: trace capacity is n_iter*n_chain sweeps, sweep s is
                              (m,l) = ((s-1) / n_chain + 1, (s-1) % n_chain + 1) as in src/GibbsRtIrt.pl.jl:289 */
  int32_t n_burnin;       /* Cond.nBurnin (the reference always passes round(nIter/2), src/Base.pl.jl:60) */
  double q_rt;            /* Cond.qRt (Cond.qRa is never read by the reference) */
  int32_t intercept, itemtype_1pl, cov2one; /* sample! keyword arguments */
  int32_t dtype;          /* enum erirt_dtype: storage and per-cell arithmetic; statistics are always f64 */
  uint64_t seed;
  uint32_t chain;         /* independent-chain id mixed into the Philox key */
  int32_t compat;         /* enum erirt_compat bits */
  int32_t person_trace;   /* 1: keep theta/zeta(/nu) of every sweep on the device (small problems) */
  int32_t device;         /* CUDA device ordinal */
  int32_t use_graph;      /* 1: replay sweeps from a captured CUDA graph */
  int32_t time_kernels;   /* 1: bracket every person-sweep launch with CUDA events (forces plain launches) */
  int32_t nu_cell_moments; /* CrossQr only, 1: keep the post-burn-in running sum / sum of squares of the N x J weights nu on the
                              device (16 bytes per cell, +32 bytes of HBM traffic per cell and sweep): Post.mean.nu of
                              src/GibbsRtIrtCross.pl.jl:310 without the reference's nIter x N*J trace; read with erirt_get_moments(ERIRT_NU) */
  int32_t reserved[6];
} erirt_config;

typedef struct erirt_stats {
  int64_t sweeps_done;
  double last_sample_ms;      /* device time of the last erirt_sample call (CUDA events) */
  double person_kernel_ms;    /* mean duration of the person-sweep kernel in that call (0 under graph replay) */
  int64_t bytes_per_sweep;    /* algorithmic HBM bytes of one sweep for this shard (DESIGN.md) */
  double pg_deferred_frac;    /* fraction of PG cells that needed the exact/retry path in the last sweep */
  int32_t launches_per_sweep; /* kernels this library launches per sweep */
  int32_t sm_count;
} erirt_stats;

int erirt_version(void);
const char* erirt_last_error(void);

int erirt_create(const erirt_config* cfg, erirt_handle** out);
/* Replica batch (DESIGN.md 6.6): one handle holding n_batch (1..65535, else ERIRT_E_ARG) independent problems of the SAME
 * configuration -- model, dimensions, dtype, n_iter, n_chain, n_burnin, q_rt and keyword options -- each with its own data, initial
 * state, parameters, statistics, running moments and traces.  erirt_sample advances all of them with one person launch and one global
 * launch per sweep.  Replica r is the chain of a standalone handle created from *cfg with seed = cfg->seed + r (Philox key
 * make_key(cfg->seed + r, cfg->chain)) and given replica r's data and initial state: same draws, traces, state and moments, up to the
 * summation order of the f64 statistics atomics.  erirt_create(cfg, out) is erirt_create_batch(cfg, 1, out).
 * The other entry points keep their signatures and stack the replicas:
 *   person-indexed arrays (Y, logT, X, theta, zeta, nu, omega, moments) have n_batch * n_subj rows, replica r in rows
 *   [r n_subj, (r+1) n_subj) (leading dimensions >= n_batch * n_subj); every other array (a, b, lambda, sigma2, rho, beta, Sigma_p,
 *   the item vectors of erirt_generate_data) is n_batch consecutive blocks of its standalone length;
 *   erirt_generate_data uses data seed `seed + r` for replica r; the ingest constants are computed per replica;
 *   erirt_get_trace: out[m + n_iter*(c + n_cols*(l + n_chain*r))], Julia's [nIter, P, nChain, nBatch];
 *   erirt_trace_width: the width of one replica;  erirt_trace_ess_rhat: n_batch * n_cols results, replica-major;
 *   erirt_loglik_current: n_batch values;  erirt_get_stats: totals over the batch;
 *   erirt_sample: ERIRT_E_NUMERIC when any replica met a non-positive-definite covariance (the message names the first; each
 *   replica's status is sticky).
 * With n_batch > 1, ERIRT_E_UNSUPPORTED (before any CUDA call) for RtIrtCross / RtIrtCrossQr and person_trace = 1 at create, and
 * from erirt_checkpoint_*, erirt_comm_init and erirt_peer_*. */
int erirt_create_batch(const erirt_config* cfg, int32_t n_batch, erirt_handle** out);
int erirt_destroy(erirt_handle* h);
/* The full-size device buffers of a handle and the ingest staging come from the device's stream-ordered memory pool, which keeps up to
 * ERIRT_POOL_KEEP_MB (environment, default 4096) of freed memory for the next handle of the process.  erirt_trim_pool returns all of
 * it to the driver (call it after erirt_destroy when the GPU memory is needed elsewhere). */
int erirt_trim_pool(int32_t device);

/* Host, column-major float64 as Julia stores them: Y[i + ldY*j] in {0,1}, logT[i + ldT*j] = log(T),
 * X[i + ldX*k].  i runs over this handle's n_subj persons, so a shard passes a pointer offset into the
 * full matrix with the full leading dimension.  logT may be NULL for GibbsMlIrt; X may be NULL if n_feat=0. */
int erirt_set_data(erirt_handle* h, const double* Y, int64_t ldY, const double* logT, int64_t ldT,
                   const double* X, int64_t ldX);
/* Same contract with Y as one byte per response (0/1): a Julia Matrix{Bool} -- what `rand.(BernoulliLogit...)` in
 * src/SimTools.jl:165 produces and InputData stores -- is passed as it lies in memory, without widening it to Float64 first
 * (an eighth of the host->device bytes of Y). */
int erirt_set_data_y8(erirt_handle* h, const uint8_t* Y, int64_t ldY, const double* logT, int64_t ldT,
                      const double* X, int64_t ldX);
/* Same contract with the buffers already on this handle's device (cudaMalloc'ed by the caller). */
int erirt_set_data_device(erirt_handle* h, const double* dY, int64_t ldY, const double* dlogT, int64_t ldT,
                          const double* dX, int64_t ldX);

/* Data generated on the device instead of ingested (SURVEY 8f-1): the N x J part of the reference's simulators,
 *   Y_ij ~ Bernoulli(logistic(a_j (theta_i - b_j))),   logT_ij = lambda_j - zeta_i - theta_i rho_j + e_ij,
 * written straight into the handle's packed layout (replaces erirt_set_data; nothing of size N x J crosses PCIe).  The person-level
 * part of setData* (theta, zeta, X: O(N) values) stays with the caller and is passed in.  error_type selects e_ij:
 *   0  N(0, sigma2_j), logT truncated to (0, inf)   setDataRtIrtNull / setDataRtIrt      src/SimTools.jl:117-178
 *   1  N(0, 1)                                       setDataRtIrtLatent                   src/SimTools.jl:300-343
 *   2  N(0, 0.3)   3  t(5)   4  Gamma(0.5, 1) - 1    setDataRtIrtCross "norm"/"tail"/"skew" src/SimTools.jl:220-255
 * GibbsMlIrt (setDataMlIrt, :349-368): zeta, lambda, sigma2, rho are ignored.  sigma2 == NULL means 1, rho == NULL means 0.
 * The variates come from a Philox stream keyed by `seed` and counted by GLOBAL person id and item, so a sharded chain generates
 * exactly the shards of the one data set.  erirt_get_data copies the data set held by the handle back to the host (column-major
 * Float64; either pointer may be NULL). */
int erirt_generate_data(erirt_handle* h, const double* theta, const double* zeta, const double* a, const double* b,
                        const double* lambda, const double* sigma2, const double* rho, const double* X, int64_t ldX,
                        int32_t error_type, uint64_t seed);
int erirt_get_data(erirt_handle* h, double* Y, int64_t ldY, double* logT, int64_t ldT);

/* Initial / current values of one InputPara field (float64, Julia layout: beta is vec(β) column-major,
 * SIGMA_P is vec(Σp), NU is n_subj (LatentQr) or n_subj x n_item column-major (CrossQr), OMEGA n_subj x n_item).
 * CrossQr draws NU before reading it, so setting it only matters for erirt_loglik_current.
 * One-sweep lookahead: the engine pipelines the person draws of sweep n with the item / structural draws of sweep n+1, so
 * after erirt_sample has run n sweeps erirt_get_state returns theta_n, zeta_n together with a, b, lambda, sigma2, beta,
 * Sigma_p (rho) of sweep n+1 and the auxiliaries omega_{n+1}, nu_{n+1} (the state the next sweep continues from).  The
 * parameters of sweep n itself are the last trace row (erirt_get_trace). */
int erirt_set_state(erirt_handle* h, int32_t field, const double* v, int64_t n);
int erirt_get_state(erirt_handle* h, int32_t field, double* out, int64_t n);

/* Run n_sweeps more sweeps (blocking).  The first call also draws the sweep-1 auxiliaries from the initial state. */
int erirt_sample(erirt_handle* h, int64_t n_sweeps);

/* Copy columns [first_col, first_col+n_cols) of Post.<which> for all sweeps done so far into `out`,
 * laid out like the Julia array restricted to those columns: out[m + n_iter*(c + n_cols*l)].
 * Column order is the reference's: ra = [θ; a; b], rt = [ζ; λ; σ²t], qr per model (SURVEY 8a a4).
 * Person columns (θ, ζ, ν) need person_trace = 1. Entries of sweeps not yet run are NaN. */
int erirt_get_trace(erirt_handle* h, int32_t which, int64_t first_col, int64_t n_cols, double* out);
int64_t erirt_trace_width(erirt_handle* h, int32_t which);

/* Post-burn-in running mean and SD (over sweeps with m > n_burnin) of THETA, ZETA or NU (n = n_subj values; CrossQr's NU is
 * n_subj x n_item column-major and needs erirt_config.nu_cell_moments). */
int erirt_get_moments(erirt_handle* h, int32_t field, double* mean, double* sd, int64_t n);

/* Convergence diagnostics on the device: rank-normalised split-chain bulk ESS and R-hat (Vehtari et al. 2021) of every requested
 * column, the estimator behind `Chains(...) |> ess_rhat` in checkConvergence (src/SimTools.jl:419-443; gate ESS > 400, R-hat < 1.1).
 * One CTA per column (csrc/diagnostics.cuh); ess / rhat are host arrays of n_cols values, NaN for constant or non-finite columns
 * and for fewer than 8 draws per chain.
 *   erirt_trace_ess_rhat: columns [first_col, first_col + n_cols) of Post.<which> as erirt_get_trace orders them, iterations
 *                         skip+1 ... of the completed ones (skip = nBurnin in the reference's use); the traces never leave the device.
 *   erirt_ess_rhat:       any host array in Julia's layout x[m + n_iter*(c + n_cols*l)] (nIter x P x nChain), first `skip`
 *                         iterations of every chain discarded. */
int erirt_trace_ess_rhat(erirt_handle* h, int32_t which, int64_t first_col, int64_t n_cols, int64_t skip, double* ess, double* rhat);
int erirt_ess_rhat(const double* x, int64_t n_iter, int64_t n_cols, int64_t n_chain, int64_t skip, int32_t device, double* ess,
                   double* rhat);

/* getLogLikelihood*(Cond, Data; P) of the state currently held by the handle (every InputPara field as last set
 * with erirt_set_state, or as left by erirt_sample -- with the one-sweep lookahead described at erirt_set_state): used for
 * DIC's D-hat at Post.mean,
 * src/GibbsRtIrt.pl.jl:432-472.  No draw is made and nothing is modified.  CrossQr (getLogLikelihoodRtIrtCrossQr,
 * src/GibbsRtIrtCross.pl.jl:240-258) reads the N x J weights last set with erirt_set_state(ERIRT_NU) or left by erirt_sample. */
int erirt_loglik_current(erirt_handle* h, double* out);

int erirt_get_stats(erirt_handle* h, erirt_stats* out);
/* Debugging aid (compute-sanitizer is not available everywhere): a handle created with ERIRT_GUARDS=1 in the environment places a
 * 256-byte guard zone after every device buffer; this returns how many guard bytes have been overwritten since (0 = clean), or -1
 * when the handle has no guard zones.  A buffer of a replica batch holds the copies of all replicas, so its guard zone catches
 * writes past the last replica, not writes between two replicas.  No counterpart in the reference. */
int64_t erirt_debug_check_guards(erirt_handle* h);

/* ---- checkpoint / resume (SURVEY 8f-4): state, auxiliaries, Philox sweep counter, running moments and traces of the chain ----
 * erirt_checkpoint_save writes erirt_checkpoint_size(h) bytes into the caller's buffer (the caller persists them).
 * erirt_checkpoint_load restores them into a handle created with the SAME erirt_config (model, dimensions, dtype, n_iter,
 * n_chain, n_burnin, person_trace, shard, seed, chain, q_rt, intercept, itemtype_1pl, cov2one, compat, nu_cell_moments -- all
 * checked, ERIRT_E_ARG otherwise) after erirt_set_data; the data is not
 * part of the checkpoint.  The resumed chain continues bit for bit as if it had never stopped.  Sharded chains: every rank
 * saves and loads its own shard. */
int64_t erirt_checkpoint_size(erirt_handle* h);
int erirt_checkpoint_save(erirt_handle* h, void* buf, int64_t size);
int erirt_checkpoint_load(erirt_handle* h, const void* buf, int64_t size);

/* ---- person-sharded chains: one handle per GPU/process, item statistics all-reduced with NCCL ---- */
int erirt_nccl_unique_id(void* id128);                 /* rank 0 creates 128 bytes, caller broadcasts them */
int erirt_comm_init(erirt_handle* h, int32_t rank, int32_t world, const void* id128);  /* id128 == NULL: no NCCL communicator,
                                                                the peer exchange below must be attached before erirt_sample */
/* One-shot exchange over NVLink peer memory, fused into the global draw kernel (replaces the per-sweep ncclAllReduce):
 * every GPU stores its statistics vector into a slot of every peer's exchange buffer as self-validating 8-byte words
 * {32 data bits, sequence number} (no fence, no separate flag), polls its own buffer until the words of this exchange have
 * arrived and sums the slots in rank order (bitwise identical on every GPU).  One process per GPU on one
 * node: erirt_peer_export allocates this GPU's exchange buffer and returns its 64-byte CUDA IPC handle; the caller
 * all-gathers the handles (any transport) and passes the world*64 bytes, in rank order, to erirt_peer_attach.
 * erirt_comm_init must have been called first (it fixes rank/world; with a NULL id no NCCL communicator is created and the
 * one-time ingest constants go through the same exchange). */
int erirt_peer_export(erirt_handle* h, void* ipc_handle64);
int erirt_peer_attach(erirt_handle* h, const void* ipc_handles /* world x 64 bytes */);
/* Unmap the peers' buffers.  Call it on every rank, then synchronise the ranks (host barrier), then erirt_destroy: an
 * exchange buffer must not be freed by its owner while a peer still has it mapped. */
int erirt_peer_detach(erirt_handle* h);

/* ---- parity entry points: one conditional kernel at a time on explicit inputs (tests only) ---- */
/* PG(1, z) on a rows x cols row-major grid; cell (i,j) uses the sampler's counters for person row0+i, item j. */
int erirt_k_pg(const double* z, int64_t rows, int32_t cols, int64_t row0, uint64_t seed, uint32_t chain,
               uint32_t sweep, int32_t dtype, int32_t device, double* out);
/* nu_i = clamp(1/IG(mu_i, lam), 1e-10, 1e10) at the person-level quantile-weight site. */
int erirt_k_nu_person(const double* mu, double lam, int64_t n, int64_t row0, uint64_t seed, uint32_t chain,
                      uint32_t sweep, int32_t dtype, int32_t device, double* out);
/* Raw Philox4x32-10 block (known-answer tests). */
int erirt_k_philox(const uint32_t ctr[4], const uint32_t key[2], int32_t device, uint32_t out[4]);

#ifdef __cplusplus
}
#endif
#endif
