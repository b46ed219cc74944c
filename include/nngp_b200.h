/*
 * include/nngp_b200.h -- C ABI of libnngp_b200.so, the B200-native replacement for the inner loop of the reference's
 * NNGP sampler (reference = R scripts under /root/reference/Scripts; citations below are relative to that tree).
 *
 * The reference has no FFI of its own: its hot path is the body of mcmc_nngp_update_Gaussian and the GpGp / Matrix
 * calls it makes.  Each entry point below names the reference call site(s) it replaces.
 *
 * Calling convention: every function is extern "C", returns void, and takes ONLY pointers, so that it can be bound with
 * R's .C() (dyn.load + .C, no R headers needed), with ctypes, or with any other FFI.  The last argument is always
 * `int *status`: 0 = ok, otherwise one of NNGP_ERR_*; the message is retrievable with nngp_last_error().
 *
 * Data conventions at the boundary are R's: column-major matrices, FP64 (`double`), `int` = int32, indices 1-based,
 * NA_integer_ = INT_MIN.  `field` always includes beta_0 (state$params$field, Scripts/mcmc_nngp_initialize.R:208).
 * Any internal re-numbering of sites (colour-major / Morton) is invisible here.
 *
 * The library needs a CUDA device (sm_100a); there is no CPU fallback: every compute entry point fails with
 * NNGP_ERR_CUDA when no device is usable.  The nngp_host_* functions are set-up utilities that run on the host by design
 * (they replace GpGp::find_ordered_nn / Coloring.R, which are init-time code in the reference as well).
 */
#ifndef NNGP_B200_H
#define NNGP_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define NNGP_OK 0
#define NNGP_ERR_ARG 1      /* bad argument / unknown context */
#define NNGP_ERR_CUDA 2     /* CUDA runtime error or no device */
#define NNGP_ERR_NCCL 3     /* communicator error */
#define NNGP_ERR_STATE 4    /* call order (e.g. sweep before a factor was built) */
#define NNGP_ERR_ALLOC 5

#define NNGP_NA_INT (-2147483647 - 1)

/* covfun_id: the reference's stationary_covfun strings (Scripts/mcmc_nngp_initialize.R:62-69) */
#define NNGP_EXPONENTIAL_ISOTROPIC 0
#define NNGP_EXPONENTIAL_SPHERE 1
#define NNGP_EXPONENTIAL_SCALEDIM 2
#define NNGP_EXPONENTIAL_SPACETIME 3
#define NNGP_MATERN_ISOTROPIC 4
#define NNGP_MATERN_SPHERE 5
#define NNGP_MATERN_SCALEDIM 6
#define NNGP_MATERN_SPACETIME 7

/* factor slots: the sampler keeps a current factor and a proposal (compressed_sparse_chol / new_compressed_sparse_chol,
 * Scripts/mcmc_nngp_update_Gaussian.R:72,123,179) */
#define NNGP_SLOT_CURRENT 0
#define NNGP_SLOT_PROPOSAL 1

/* rng_mode for the field draws of the chromatic sweep */
#define NNGP_RNG_SUPPLIED 0 /* caller passes the normals (R's rnorm stream): bit-comparable with the reference order */
#define NNGP_RNG_PHILOX 1   /* counter-based Philox4x32-10 keyed by (seed, sweep counter, global site id) */
/* The Philox stream.  The normal of site g (0-based reference index; global on a sharded field) in the sweep at counter k under
 * seed s is Philox4x32-10 with counter (g, k & 0xffffffff, k >> 32, 0x4e4e4750) and key (s & 0xffffffff, (s >> 32) ^ 0x5eed5eed),
 * s = (uint64_t)(int64_t)seed; from its output words a = (x << 32) | y, b = (z << 32) | w, u1 = ((a >> 11) + 0.5) 2^-53, u2 likewise
 * from b, and the normal is sqrt(-2 log u1) cospi(2 u2).  Each context keeps a sweep counter that starts at 0 when the context is
 * created and advances by one for every sweep run on it, whatever the rng_mode: nngp_gibbs_sweep and nngp_sweep_loglik_host by
 * n_sweeps, nngp_chain_run* by n_iter * n_chromatic, nngp_time_op ops 2 and 6 by one per repetition, nngp_time_op_group by
 * reps + 1 on each context, the shard colour-stepping entry points by one per sweep.  nngp_chain_run* take
 * seed = (iter_start << 20) ^ chain_index, so nngp_gibbs_sweep with seed s draws under the same key as nngp_chain_run with
 * iter_start = 0 and chain_index = s.  tests/philox_reference.py restates all of this. */

/* internal site layout (performance knob; results are layout-independent up to FP64 summation order) */
#define NNGP_LAYOUT_COLOR 1        /* vectors stored colour-major, reference order inside a colour */
#define NNGP_LAYOUT_COLOR_MORTON 2 /* vectors stored colour-major, Morton (Z-curve) order inside a colour */
#define NNGP_LAYOUT_MORTON 3       /* vectors stored in pure Z-curve order; the sweep walks them colour by colour (default) */

/* ------------------------------------------------------------------------------------------------------------------
 * library / device
 * ------------------------------------------------------------------------------------------------------------------ */
void nngp_version(int *major, int *minor);
void nngp_device_count(int *count, int *status);
/* copies the last error message (NUL-terminated, truncated to *len bytes) */
void nngp_last_error(char *buf, const int *len);
/* the same for R's .C(), which passes a character vector as char **: the message is written into buf[0] (a string of at least
 * *len bytes, e.g. strrep(" ", 1024)) */
void nngp_last_error_r(char **buf, const int *len);

/* ------------------------------------------------------------------------------------------------------------------
 * host-side set-up utilities (init-time in the reference too)
 * ------------------------------------------------------------------------------------------------------------------ */
/* replaces GpGp::find_ordered_nn(locs, m)  (Scripts/mcmc_nngp_initialize.R:93, Scripts/mcmc_nngp_predict.R:5).
 * Exact m nearest PREVIOUS sites by Euclidean distance on the raw coordinates, ties by lower index; column 1 = self;
 * NA padding.  locs n x d column-major; NNarray n x (m+1) column-major out. */
void nngp_host_find_ordered_nn(const double *locs, const int *n, const int *d, const int *m, int *NNarray, int *status);
/* replaces the crossprod() moral graph + naive_greedy_coloring (Scripts/mcmc_nngp_initialize.R:103-110,
 * Scripts/Coloring.R:2-20) without the dense (n+1) x maxdeg scratch: identical first-fit colours 1..K. */
void nngp_host_greedy_coloring(const int *NNarray, const int *n, const int *m, int *coloring, int *n_colors, int *status);
/* drop-in for naive_greedy_coloring(M) itself (Scripts/Coloring.R:2-20): M's compressed-column slots M@p (n + 1) and M@i (0-based),
 * i.e. the MRF adjacency matrix of Scripts/mcmc_nngp_initialize.R:103-109; same colours, no dense (n+1) x maxdeg scratch */
void nngp_host_greedy_coloring_adj(const int *adj_p, const int *adj_i, const int *n, int *coloring, int *n_colors, int *status);
/* OpenMP threads used by the nngp_host_* utilities; n <= 0 = all processors (launchers such as torchrun export OMP_NUM_THREADS=1) */
void nngp_host_set_num_threads(const int *n, int *status);
/* exact max-min (farthest-point) ordering, 1-based permutation (an alternative to GpGp::order_maxmin,
 * Scripts/mcmc_nngp_initialize.R:29, which is a randomised approximation -- see nngp_host_order_maxmin_gpgp) */
void nngp_host_order_maxmin(const double *locs, const int *n, const int *d, int *order, int *status);

/* ------------------------------------------------------------------------------------------------------------------
 * R-compatible random stream and the reference's own ordering / neighbour search on it, for hosts that are not R
 * (the Python mirror): with these, mcmc_nngp_initialize(seed) yields the SAME ordering, NNarray, colouring and initial
 * states as the reference does in R -- checked against the values the reference's vignette prints
 * (tests/test_abi_cpu.py, tests/test_gpu_vignette.py).  A host written in R needs none of this (it has R's RNG and GpGp).
 * rstate: 625 ints, caller-owned: rstate[0] = position (mti), rstate[1..624] = the Mersenne-Twister words, i.e. R's
 * .Random.seed[2:626] for RNGkind("Mersenne-Twister", "Inversion", "Rejection") (the defaults since R 3.6).
 * ------------------------------------------------------------------------------------------------------------------ */
/* set.seed(seed)  (Scripts/mcmc_nngp_initialize.R:17, Scripts/mcmc_nngp_update_Gaussian.R:36) */
void nngp_rng_set_seed(const int *seed, int *rstate, int *status);
/* runif(n), rnorm(n) (inversion), sample.int(n, size) without replacement (rejection sampling), rbeta(n, shape1, shape2)
 * (Cheng's BB; shape1, shape2 > 1 only: initialize.R:193-194 draws rbeta(1, 10, 10)) */
void nngp_rng_runif(int *rstate, const int *n, double *out, int *status);
void nngp_rng_rnorm(int *rstate, const int *n, double *out, int *status);
void nngp_rng_sample_int(int *rstate, const int *n, const int *size, int *out, int *status);
void nngp_rng_rbeta(int *rstate, const int *n, const double *shape1, const double *shape2, double *out, int *status);
/* GpGp::order_maxmin(locs, lonlat)  (Scripts/mcmc_nngp_initialize.R:29), bit-exact on R's stream: coordinate jitter
 * 1e-4 * min column sd * rnorm(n*d), start permutation sample(n), one pass that moves an index to the end of the list when
 * one of its round(min(round(sqrt(n)), n/(j - nmoved + 1))) nearest neighbours precedes it.  order: n, 1-based.  *lonlat != 0:
 * columns 1-2 are longitude / latitude in degrees, mapped to the unit sphere after the jitter (as published; unpinned). */
void nngp_host_order_maxmin_gpgp(const double *locs, const int *n, const int *d, const int *lonlat, int *rstate, int *order, int *status);
/* GpGp::find_ordered_nn(locs, m)  (Scripts/mcmc_nngp_initialize.R:93) bit-exact on R's stream: the same jitter (n*d fresh
 * normals), then nngp_host_find_ordered_nn on the jittered coordinates */
void nngp_host_find_ordered_nn_gpgp(const double *locs, const int *n, const int *d, const int *m, int *rstate, int *NNarray, int *status);

/* ------------------------------------------------------------------------------------------------------------------
 * context: graph structure uploaded once (vecchia_approx, Scripts/mcmc_nngp_initialize.R:80-110)
 * ------------------------------------------------------------------------------------------------------------------ */
/* locs n x d; NNarray n x (m+1); coloring n (1..K, verified to be proper for the moral graph; ALL ZERO = no colouring:
 * a context that never sweeps, e.g. the joint observed ++ predicted site set of mcmc_nngp_predict_field, predict.R:4-8 --
 * its sweep entry points return NNGP_ERR_STATE); locs_match n_obs (1-based site of each observation);
 * device: CUDA ordinal; layout: NNGP_LAYOUT_*.  Returns a context id.
 * Limits: 1 <= d <= 4, 1 <= m <= 31, n * (m + 1) < 2^31 (entry positions are int32; n <= 195M at m = 10, 102M at m = 20). */
void nngp_ctx_create(const int *n, const int *d, const int *m, const double *locs, const int *NNarray,
                     const int *coloring, const int *n_obs, const int *locs_match, const int *covfun_id,
                     const int *device, const int *layout, int *ctx_id, int *status);
void nngp_ctx_destroy(const int *ctx_id, int *status);

/* ---- one latent field sharded over the GPUs of a box by spatial blocks (SURVEY.md 8e; BASELINE.json config 4) ----
 * One process per GPU.  Rank 0 obtains a communicator id (128 bytes) and hands it to its peers by any means (the Python
 * mirror uses torch.distributed, R would use its own sockets); every rank then creates its context at the same time.
 * The context covers the rank's LOCAL site set (owned sites + ghost sites, numbered in the field's order; see
 * <package>/partition.py for how it is derived from NNarray and the block owner of every site):
 *   owned[n]        1 = this rank updates the site, 0 = ghost copy kept current by the halo exchange
 *   global_id[n]    0-based id of the site in the whole field (Philox key, so that results do not depend on the sharding)
 *   global_zpos[n]  position of the site in the whole field's rnorm() hand-out order (NNGP_RNG_SUPPLIED mode)
 *   global_level[n] depth of the site's row in the WHOLE field's solve DAG (0 = no parents); every rank orders its owned rows
 *                   by it in the sharded triangular solve.  NULL = not given: the solve-based entry points are then unavailable
 *   send_site / send_ptr   owned boundary sites per (colour, peer): segment [send_ptr[c*world+h], send_ptr[c*world+h+1])
 *   recv_site / recv_ptr   ghost sites per (colour, peer), in the same order as the owner sends them
 * On such a context nngp_gibbs_sweep exchanges the boundary values of every colour (peer-to-peer transport below: fused into
 * the sweep kernel; NCCL: ncclSend/ncclRecv after it) and nngp_loglik / nngp_ssr / nngp_beta0_moments all-reduce their partial
 * sums; observations are those of the owned sites.  Limits: at most 8 ranks per field.
 * With the peer-to-peer transport nngp_sptrsv / nngp_field_init / nngp_ancillary_propose and nngp_chain_run (no-regressor model) work
 * on the block too: every rank solves its owned rows with the synchronisation-free kernel and stores boundary values straight into
 * the peers' solution vectors; every rank runs the chain loop with the same scalar state (all decisions are taken on all-reduced
 * scalars).  Vectors are the rank's LOCAL vectors (owned + ghost sites); var_y is the whole field's.  Prediction is not sharded. */
void nngp_comm_unique_id(char *id128, int *status);
void nngp_ctx_create_sharded(const int *n, const int *d, const int *m, const double *locs, const int *NNarray,
                             const int *coloring, const int *n_colors, const int *owned, const int *global_id,
                             const int *global_zpos, const int *global_level, const double *n_global, const int *n_obs, const int *locs_match,
                             const int *covfun_id, const int *device, const int *layout, const int *world, const int *rank,
                             const int *send_site, const int *send_ptr, const int *recv_site, const int *recv_ptr,
                             const char *comm_id128, int *ctx_id, int *status);
/* Peer-to-peer transport for the halo and the scalar all-reduces (preferred inside one NVLink box): every rank exports the
 * CUDA IPC handle (64 bytes) of its receive area, the handles are gathered by the caller, and every rank connects with the
 * table of all handles (world * 64 bytes, rank order) plus peer_recv_base[c*world + h] = offset of this rank's colour-c
 * segment inside peer h's receive area (= peer h's recv_ptr[c*world + this rank]).  Afterwards the sweep kernel of a colour
 * stores the new values of its boundary sites (their tiles run first) directly into the peers' ghost slots over NVLink; the
 * value itself is the message (an empty slot holds a reserved NaN payload), so there is no fence and no flag: trailing CTAs of
 * the same launch apply each ghost value as soon as it has landed.  Scalar all-reduces use the same mapped areas. */
void nngp_shard_p2p_export(const int *ctx_id, char *handle64, int *status);
void nngp_shard_p2p_connect(const int *ctx_id, const char *all_handles, const int *peer_recv_base, int *status);
/* Colour-stepping form of one sharded sweep for callers that move the halo themselves (any transport; also how the sharded
 * arithmetic is tested on a single GPU).  Create the contexts with an empty comm_id (first byte 0) to skip NCCL.
 * begin -> for colour in 1..K: sweep_colour; halo_get (packed send buffer of that colour, all peers, send_ptr order);
 * [caller routes the segments]; halo_put (packed receive buffer, recv_ptr order) -> end. */
void nngp_shard_sweep_begin(const int *ctx_id, const double *beta_0, const double *log_scale, const double *log_noise_variance,
                            const int *rng_mode, const double *z, const double *seed, int *status);
void nngp_shard_sweep_colour(const int *ctx_id, const int *colour, int *status);
void nngp_shard_halo_get(const int *ctx_id, const int *colour, double *out, int *status);
void nngp_shard_halo_put(const int *ctx_id, const int *colour, const double *in, int *status);
void nngp_shard_sweep_end(const int *ctx_id, int *status);
/* single-process form of the same transport: the W contexts of the field live in this process (one per GPU -- what an R
 * session on a multi-GPU box has -- or several on one GPU); ctx_ids[h] must be rank h.  Their receive areas are addressed
 * directly (peer access is enabled between distinct devices), no IPC handles are needed. */
void nngp_shard_connect_local(const int *ctx_ids, const int *world, int *status);
/* n_sweeps sweeps of a locally connected field: enqueued on every member, then all are waited for (the members exchange their
 * halos among themselves while they run).  z (NNGP_RNG_SUPPLIED): n_sweeps * n_global normals in the whole field's hand-out order */
void nngp_shard_group_sweep(const int *ctx_ids, const int *world, const int *n_sweeps, const double *beta_0, const double *log_scale,
                            const double *log_noise_variance, const int *rng_mode, const double *z, const double *seed, int *status);
/* Vecchia log-likelihood of a locally connected field (partial sums all-reduced between the members): ll[h] for every member h,
 * all equal */
void nngp_shard_group_loglik(const int *ctx_ids, const int *world, const int *slot, const double *beta_0, const double *log_scale,
                             double *ll, int *status);
/* one chain (reference loop, no-regressor model) on a locally connected field: every member runs the loop on its block on its own
 * host thread with the same scalar state; params_io is the one parameter vector (as nngp_chain_run); records_out / accept_out are the
 * scalar records (identical on every member); field_records_out holds member h's round(n_iter * thin) x n_local(h) block after member
 * h - 1's, or is NULL */
void nngp_shard_group_chain_run(const int *ctx_ids, const int *world, const int *n_shape, double *params_io, const int *n_iter,
                                const double *thin, const int *n_chromatic, const int *iter_start, const int *chain_index, const int *rng_mode,
                                const double *var_y, double *records_out, double *field_records_out, int *accept_out, int *status);
/* host-side set-up of a sharded field (replaces nothing in the reference, which has no multi-GPU path; SURVEY.md 8e):
 * owner[n] = spatial block (0..n_parts-1) of every site by recursive coordinate bisection into equal counts */
void nngp_host_spatial_blocks(const double *locs, const int *n, const int *d, const int *n_parts, int *owner, int *status);
/* everything rank `rank` needs for nngp_ctx_create_sharded, derived from the whole field's structure in O(n (m+1)):
 * build returns a plan id and sizes6 = [n_local, n_obs_local, n_send, n_recv, n_colors, n_owned]; get copies the arrays into
 * caller-allocated buffers (locs n_local x d; NNarray n_local x (m+1); coloring / owned / global_id / global_zpos / global_level n_local;
 * obs_index (0-based index into the field's observations) / locs_match n_obs_local; send_site n_send; recv_site n_recv;
 * send_ptr / recv_ptr n_colors * world + 1) and frees the plan.  At most 8 ranks. */
void nngp_host_shard_plan_build(const double *locs, const int *NNarray, const int *coloring, const int *n, const int *d, const int *m,
                                const int *n_obs, const int *locs_match, const int *owner, const int *rank, const int *world,
                                int *plan_id, int *sizes6, int *status);
void nngp_host_shard_plan_get(const int *plan_id, double *locs, int *NNarray, int *coloring, int *owned, int *global_id, int *global_zpos,
                              int *global_level, int *obs_index, int *locs_match, int *send_site, int *send_ptr, int *recv_site, int *recv_ptr, int *status);
/* performance knobs (results are identical up to FP64 summation order):
 *   NNGP_OPT_SWEEP_VARIANT 0 = one launch per colour, tiles of <= 128 sites / 1024 factor entries per CTA, blocked segmented
 *                          reduction, chained with programmatic dependent launch (the r-independent prologue of colour c+1
 *                          overlaps colour c), replayed from a CUDA graph; colours that would spill into a second wave at
 *                          5 CTAs/SM run a 6-CTAs/SM build (default); 1 = the same chain with 5 CTAs/SM everywhere;
 *                          2 = the same tiles as plain launches; 3 = thread per site (unsharded contexts); 4 = as 0, but a colour
 *                          triggers its dependent launch only after its own wait (at most two colours resident per stream: for
 *                          several chains sharing one GPU)
 *   NNGP_OPT_SOLVE_VARIANT 0 = synchronisation-free single-launch triangular solve; 1 = one launch per DAG level
 *   NNGP_OPT_USE_GRAPH     1 = the colour launches of a sweep are replayed from a captured CUDA graph (default) */
#define NNGP_OPT_SWEEP_VARIANT 1
#define NNGP_OPT_SOLVE_VARIANT 2
#define NNGP_OPT_USE_GRAPH 3
#define NNGP_OPT_SOLVE_CTAS_PER_SM 4 /* window of the sync-free solve: n_sm * value * 256 rows in flight (default 1) */
#define NNGP_OPT_SOLVE_SLEEP_NS 5    /* back-off between dependency polls (default 0) */
#define NNGP_OPT_SOLVE_WINDOW_CTAS 7  /* absolute window of the sync-free solve in CTAs of 256 rows (0 = use per-SM setting) */
#define NNGP_OPT_SOLVE_LEVEL_COPY 6  /* 1 = the factor build also writes the factor in the triangular solve's row order, so that the solve reads coalesced (default); 0 = off (comparison; factors must be rebuilt after switching) */
#define NNGP_OPT_COMMIT_VARIANT 8     /* accept-branch transposition: 0 = tiled, blocked reduction (default), 1 = thread per column */
#define NNGP_OPT_MATERN_TABLE 9       /* Matern families: 1 = per-build interpolation table of the kernel (default), 0 = K_nu per pair */
#define NNGP_OPT_SHARD_GHOST_CTAS 11  /* sharded sweep (peer-to-peer): at most this many ghost CTAs per colour launch, 4 ghost sites in flight each (default 296) */
#define NNGP_OPT_SHARD_GHOST_FIRST 12 /* ... 0 = at the end of the grid (default); 1 = at its head, resident before the peers' values land; 2 = per colour: head iff tiles and ghost CTAs are co-resident; default 0 (measured: 167 / 180 / 168 us on 2 GPUs x 1M sites) */
#define NNGP_OPT_FACTOR_VARIANT 14    /* factor build at m = 20: 0 = one thread per row, as for m <= 10 (default); 1 = one warp per row (measured slower for the exponential family, equal for Matern) */
#define NNGP_OPT_LOGLIK_VARIANT 10    /* log-lik pass: 1 = plain coalesced loads (default, faster); 0 = TMA-staged shared-memory ring (cp.async.bulk + mbarrier) */
#define NNGP_OPT_LOGLIK_FROM_RESIDUAL 15 /* 1 = nngp_loglik (current factor, device field) right after nngp_gibbs_sweep with the same beta_0, and
                                          * nngp_sweep_loglik_host, sum the residual linv (field - beta_0) the sweep keeps instead of the full pass
                                          * (default; equal up to the rounding of the sweep's updates of it); 0 = always the full pass */
void nngp_ctx_set_option(const int *ctx_id, const int *key, const int *value, int *status);
/* development aid: one sweep of a connected sharded field with six time stamps per colour (first tile past its wait, last boundary
 * push, first / last ghost value seen, last ghost site patched, last tile done); out_ns[n_colors][6], ns, -1 = not set.  Every rank
 * of the field must call it at the same time. */
void nngp_shard_timeline(const int *ctx_id, const double *beta_0, const double *log_scale, const double *log_noise_variance,
                         double *out_ns, int *status);

/* development aid: completion time (ns, %globaltimer) of every 256-row chunk of one triangular solve and the DAG level each chunk
 * starts in; *n_chunks: capacity in, count out */
void nngp_solve_timeline(const int *ctx_id, double *out_ns, int *level_of_chunk, int *n_chunks, int *status);

/* info[0]=n, [1]=m, [2]=n_colors, [3]=n_levels (depth of the solve DAG), [4]=nnz, [5]=max column length,
 * [6]=device, [7]=layout */
void nngp_ctx_info(const int *ctx_id, int *info8, int *status);

/* ------------------------------------------------------------------------------------------------------------------
 * Vecchia factor  (GpGp::vecchia_Linv + Matrix::sparseMatrix assembly)
 * ------------------------------------------------------------------------------------------------------------------ */
/* replaces GpGp::vecchia_Linv(covparms, covfun_name, locs, NNarray) followed by Matrix::sparseMatrix(...)
 * (Scripts/mcmc_nngp_update_Gaussian.R:72-73,123-124,179-180; initialize.R:201-207; predict.R:39-40).
 * covparms = c(variance, shape..., nugget) exactly as the reference passes them (c(1, shape, 0)).
 * n_not_pd = number of rows whose neighbour block was not positive definite (the proposal must then be rejected). */
void nngp_factor_build(const int *ctx_id, const int *slot, const double *covparms, const int *n_covparms,
                       int *n_not_pd, int *status);
/* copies the compressed factor (n x (m+1), column-major, unused slots 0) to the host */
void nngp_factor_get(const int *ctx_id, const int *slot, double *Linv, int *status);
/* the accept branch (Scripts/mcmc_nngp_update_Gaussian.R:139-142,194-197): proposal becomes current and
 * precision_diag is recomputed */
void nngp_factor_accept(const int *ctx_id, int *status);
/* makes `slot` the sweep's factor without swapping (used after the initial build, update_Gaussian.R:72-74) */
void nngp_factor_commit(const int *ctx_id, const int *slot, int *status);
/* precision_diag (Scripts/mcmc_nngp_update_Gaussian.R:74,142,197) of the current factor */
void nngp_precision_diag(const int *ctx_id, double *out, int *status);

/* ------------------------------------------------------------------------------------------------------------------
 * device-resident chain state
 * ------------------------------------------------------------------------------------------------------------------ */
void nngp_field_set(const int *ctx_id, const double *field, int *status);
void nngp_field_get(const int *ctx_id, double *field, int *status);
/* y_minus_xb[o] = observed_field[o] - (mu[o] - beta_0), i.e. the response minus the non-intercept fixed effects
 * (equal to observed_field when there are no regressors).  Everything the sampler needs from the observations
 * (residuals_sum update_Gaussian.R:260, the dnorm ratio :129-131, the SSR :281) is derived from it on the device. */
void nngp_obs_set(const int *ctx_id, const double *y_minus_xb, int *status);

/* ------------------------------------------------------------------------------------------------------------------
 * Vecchia log-likelihood and sparse products
 * ------------------------------------------------------------------------------------------------------------------ */
/* replaces ll_compressed_sparse_chol(Linv, field - beta_0, NNarray, log_scale)
 * (Scripts/mcmc_nngp_update_Gaussian.R:8-12, called :185-186) on the device-resident field */
void nngp_loglik(const int *ctx_id, const int *slot, const double *beta_0, const double *log_scale, double *ll,
                 int *status);
/* same, with the (already centred) field passed from the host: the end-to-end form of one log-lik evaluation */
void nngp_loglik_host(const int *ctx_id, const int *slot, const double *z, const double *log_scale, double *ll,
                      int *status);
/* sparse_chol %*% v   (GpGp::Linv_mult; Scripts/mcmc_nngp_update_Gaussian.R:10,127,221-222,241) */
void nngp_spmv(const int *ctx_id, const int *slot, const double *v, double *out, int *status);
/* crossprod(sparse_chol, u) = t(sparse_chol) %*% u  (Scripts/mcmc_nngp_update_Gaussian.R:269) */
void nngp_sptmv(const int *ctx_id, const int *slot, const double *u, double *out, int *status);
/* Matrix::solve(sparse_chol, b)  (initialize.R:208; update_Gaussian.R:127; predict.R:46) */
void nngp_sptrsv(const int *ctx_id, const int *slot, const double *b, double *x, int *status);

/* ------------------------------------------------------------------------------------------------------------------
 * sampler steps on the device-resident state
 * ------------------------------------------------------------------------------------------------------------------ */
/* n_sweeps chromatic Gibbs sweeps of the latent field (Scripts/mcmc_nngp_update_Gaussian.R:257-275) with the current
 * factor.  rng_mode NNGP_RNG_SUPPLIED: z holds n_sweeps * n normals, sweep-major, each sweep in the order in which the
 * reference's rnorm(length(selected_locs)) calls hand them out (colour 1..K, sites ascending inside a colour).
 * NNGP_RNG_PHILOX: z is ignored (may be NULL); seed picks the Philox key, and sweep j of the call (j = 0 .. n_sweeps - 1) draws at
 * the context's sweep counter + j (see NNGP_RNG_PHILOX).  Either mode advances the counter by n_sweeps. */
void nngp_gibbs_sweep(const int *ctx_id, const int *n_sweeps, const double *beta_0, const double *log_scale,
                      const double *log_noise_variance, const int *rng_mode, const double *z, const double *seed,
                      int *status);
/* One step for a caller that keeps state$params$field on the host: field_io (n values, reference order) is uploaded, n_sweeps sweeps
 * run as in nngp_gibbs_sweep, ll receives ll_compressed_sparse_chol of the NEW field (current factor, update_Gaussian.R:8-12) and
 * field_io the new field.  One host->device and one device->host pass over the field per call. */
void nngp_sweep_loglik_host(const int *ctx_id, const int *n_sweeps, const double *beta_0, const double *log_scale,
                            const double *log_noise_variance, const int *rng_mode, const double *z, const double *seed,
                            double *field_io, double *ll, int *status);
/* ancillary proposal (Scripts/mcmc_nngp_update_Gaussian.R:127-131): new_field = beta_0 + exp(.5 dls) *
 * solve(proposal, current %*% (field - beta_0)) is formed on the device and the Gaussian observation log-density
 * difference field_response_ratio is returned.  nngp_ancillary_accept() makes new_field the field. */
void nngp_ancillary_propose(const int *ctx_id, const double *beta_0, const double *delta_log_scale,
                            const double *log_noise_variance, double *field_response_ratio, int *status);
void nngp_ancillary_accept(const int *ctx_id, int *status);
/* beta_0 | field without regressors (Scripts/mcmc_nngp_update_Gaussian.R:219-224): returns mean and variance */
void nngp_beta0_moments(const int *ctx_id, const double *log_scale, double *mean, double *var, int *status);
/* sum_squared_residuals (Scripts/mcmc_nngp_update_Gaussian.R:281) */
void nngp_ssr(const int *ctx_id, double *ssr, int *status);
/* initial field draw (Scripts/mcmc_nngp_initialize.R:201-208): field = beta_0 + exp(.5 log_scale) * solve(slot, z) */
void nngp_field_init(const int *ctx_id, const int *slot, const double *beta_0, const double *log_scale,
                     const double *z, int *status);

/* one chain, n_iter iterations of the reference loop for the no-regressor model (Scripts/mcmc_nngp_update_Gaussian.R:
 * 101-314) entirely behind the ABI: scalars only cross PCIe, plus the thinned field rows.
 * params_io: [beta_0, log_scale, log_noise_variance, logvar_sufficient, logvar_ancillary, shape_1..shape_k]
 * records_out: n_iter x (3 + k) column-major [beta_0, log_scale, log_noise_variance, shape...]
 * field_records_out: round(n_iter * thin) x n column-major, or NULL
 * rng_mode NNGP_RNG_SUPPLIED reproduces R's stream (set.seed(iter_start + chain_index), Mersenne-Twister + inversion)
 * for every draw including the field normals; NNGP_RNG_PHILOX uses R's stream for the scalar draws (skipping the field's rnorm()
 * calls, update_Gaussian.R:75 included) and Philox for the field: seed (iter_start << 20) ^ chain_index, iteration i's sweeps at
 * counters c0 + (i - 1) n_chromatic .. c0 + i n_chromatic - 1, c0 = the context's sweep counter when the call starts (see
 * NNGP_RNG_PHILOX). */
void nngp_chain_run(const int *ctx_id, const int *n_shape, double *params_io, const int *n_iter, const double *thin,
                    const int *n_chromatic, const int *iter_start, const int *chain_index, const int *rng_mode,
                    const double *var_y, double *records_out, double *field_records_out, int *accept_out, int *status);

/* Regressors of the Gaussian model, kept resident in HBM for nngp_chain_run_regressors (X$X, X$locs of
 * Scripts/mcmc_nngp_initialize.R:116-137).  X: n_obs x p column-major, the centred model-matrix columns without the
 * intercept (X$X); observed_field: n_obs; xlocs: the n_xlocs 1-based columns of X that vary with the site only (X$locs;
 * n_xlocs = 0 and NULL when X_locs was not given); first_obs: vecchia_approx$hctam_scol_1 (n, 1-based; used only when
 * n_xlocs > 0: X$X[hctam_scol_1, X$locs], update_Gaussian.R:78). */
void nngp_regressors_set(const int *ctx_id, const int *p, const double *X, const double *observed_field, const int *n_xlocs,
                         const int *xlocs, const int *first_obs, int *status);
/* nngp_chain_run for the model with regressors: additionally the block update of (beta_0, beta) given the field
 * (update_Gaussian.R:226-235) and, with location-level regressors, the interweaved centred update (:237-246) with
 * sparse_chol_X_locs / beta_interweaved_covmat refreshed after every accepted covariance proposal (:77-83,145-151,200-206).
 * X, its products and the field stay on the device; per iteration only (p+1)- and (n_xlocs+1)-vectors cross PCIe.
 * beta_io: p (state$params$beta); solve_1XT1X, chol_solve_1XT1X: (p+1) x (p+1) column-major as stored in X by
 * mcmc_nngp_initialize (:135-136; chol() = upper factor); beta_records_out: n_iter x p column-major or NULL.
 * The R stream is consumed exactly as the reference does: ... rnorm(p+1) (:231), rnorm(n_xlocs+1) (:242) ... */
void nngp_chain_run_regressors(const int *ctx_id, const int *n_shape, double *params_io, double *beta_io,
                               const double *solve_1XT1X, const double *chol_solve_1XT1X, const int *n_iter, const double *thin,
                               const int *n_chromatic, const int *iter_start, const int *chain_index, const int *rng_mode,
                               const double *var_y, double *records_out, double *beta_records_out, double *field_records_out,
                               int *accept_out, int *status);

/* Several chains at once -- the reference advances its chains concurrently (parallel::mclapply over chains,
 * Scripts/mcmc_nngp_update_Gaussian.R:22-26, n_cores of mcmc_nngp_run.R).  One blocking call, so that it also works through
 * R's .C(): chain k runs on context ctx_ids[k] (its own device, stream and device-resident state; the contexts must be distinct)
 * driven by its own host thread, at most max_concurrent (= n_cores) in flight.  Chains on different GPUs run in parallel, chains
 * sharing a GPU overlap on it.  Every chain's result is bit-identical to what nngp_chain_run gives for it alone.
 * Scalars (n_shape, n_iter, thin, n_chromatic, iter_start, rng_mode, var_y) are common to all chains; per-chain blocks are
 * laid out chain after chain: params_io n_chains x (5 + n_shape); chain_index n_chains; records_out n_chains x [n_iter x
 * (3 + n_shape)]; field_records_out n_chains x [round(n_iter * thin) x n] or NULL; accept_out n_chains x [2 n_iter] or NULL;
 * beta_io n_chains x p; beta_records_out n_chains x [n_iter x p] or NULL. */
void nngp_chains_run(const int *n_chains, const int *ctx_ids, const int *n_shape, double *params_io, const int *n_iter, const double *thin,
                     const int *n_chromatic, const int *iter_start, const int *chain_index, const int *rng_mode, const double *var_y,
                     const int *max_concurrent, double *records_out, double *field_records_out, int *accept_out, int *status);
void nngp_chains_run_regressors(const int *n_chains, const int *ctx_ids, const int *n_shape, double *params_io, double *beta_io,
                                const double *solve_1XT1X, const double *chol_solve_1XT1X, const int *n_iter, const double *thin,
                                const int *n_chromatic, const int *iter_start, const int *chain_index, const int *rng_mode,
                                const double *var_y, const int *max_concurrent, double *records_out, double *beta_records_out,
                                double *field_records_out, int *accept_out, int *status);

/* Posterior summary of the field samples stored by the last nngp_chain_run, computed on the device from the record store
 * that stays in HBM (SURVEY.md 8f rank 3): get_summary (Scripts/mcmc_nngp_estimate.R:1-6) of rows first_row .. first_row +
 * n_rows - 1 (1-based) of records$field minus offsets[k] (beta_0 of the same iteration, estimate.R:90-92; NULL = none).
 * out: n x 5 column-major (mean, q0.025, median, q0.975, sd), sites in reference order. */
void nngp_records_summary(const int *ctx_id, const int *first_row, const int *n_rows, const double *offsets, double *out,
                          int *status);

/* ------------------------------------------------------------------------------------------------------------------
 * prediction  (mcmc_nngp_predict_field, Scripts/mcmc_nngp_predict.R:25-54)
 * ------------------------------------------------------------------------------------------------------------------ */
/* The context must have been created over the joint (observed ++ predicted) site set (predict.R:4-5), n_obs_sites =
 * number of observed sites (the first rows).  For one stored sample: builds nothing (uses factor `slot`), forms
 * x_obs = (field - beta_0)/sd and conditionally simulates the n_pred new rows; out = sd * x_pred (predict.R:43-53). */
void nngp_predict_sample(const int *ctx_id, const int *slot, const int *n_obs_sites, const double *field,
                         const double *beta_0, const double *log_scale, const double *z_pred, double *out, int *status);

/* ------------------------------------------------------------------------------------------------------------------
 * measurement
 * ------------------------------------------------------------------------------------------------------------------ */
/* Times `reps` back-to-back launches of one device op with CUDA events on the library's own stream (inputs resident in
 * HBM). op: 0 factor_build(proposal slot, last covparms) 1 loglik 2 one Gibbs sweep (Philox) 3 spmv 4 sptrsv
 * 5 precision_diag/transposition 6 sweep + loglik.  ms_out[reps] per-launch milliseconds; launches_out = kernels launched
 * per repetition. flush_l2 != 0 writes a 256 MB scratch buffer between repetitions (outside the timed events). */
void nngp_time_op(const int *ctx_id, const int *op, const int *reps, const int *flush_l2, double *ms_out,
                  int *launches_out, int *status);
/* `reps` repetitions of op 2 (one Gibbs sweep) or 6 (sweep + log-lik) enqueued on several contexts of ONE device at once (their
 * streams overlap on the device): ms_out[0] = time until the last context finished, CUDA events with a common origin. */
void nngp_time_op_group(const int *ctx_ids, const int *n_ctx, const int *op, const int *reps, double *ms_out, int *status);
/* measured FP64 FMA throughput of the device in GFLOP/s (dependent-free DFMA chains on every SM, 2 flops per DFMA): the
 * denominator of the factor kernel's roofline fraction (SURVEY.md 8d) */
void nngp_fp64_peak(const int *device, double *gflops, int *status);
/* Page-locked host buffers.  Vectors handed to the library from such a buffer are DMA-ed directly (no staging copy); any other
 * host pointer is staged through an internal pinned buffer with a multi-threaded copy.  n_bytes is a double so that .C() can
 * pass sizes beyond 2^31. */
void nngp_host_alloc(const double *n_bytes, void **ptr, int *status);
void nngp_host_free(void **ptr, int *status);
/* cumulative number of kernels this library has launched in this process (for bench.py's gpu_launches) */
void nngp_launch_count(double *count);

#ifdef __cplusplus
}
#endif
#endif /* NNGP_B200_H */
