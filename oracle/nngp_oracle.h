/*
 * oracle/nngp_oracle.h -- TEST INFRASTRUCTURE ONLY.
 *
 * CPU restatement of the reference's NNGP hot path (R scripts under /root/reference/Scripts plus the semantics of the
 * un-vendored CRAN packages GpGp / Matrix they call).  Only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may load this library.  The product (libnngp_b200.so) never links or calls it.
 *
 * PARITY PINNED against reference-held values (round 2): the reference has no tests and R / GpGp / Matrix cannot run in
 * this image (SURVEY.md 8c), but its rendered vignette prints a complete seeded session -- the initial states (100 field
 * values to 8 decimals), 46 Gelman-Rubin-Brooks blocks over 4600 + 1000 iterations of three chains, posterior summaries --
 * and this oracle, driven by R's random stream (r_rng.c, gpgp_order.c, reference_driver.py), reproduces every one of those
 * numbers to the last printed digit (tests/test_vignette_pin.py).  The covariance families the vignette does not use
 * (Matern, sphere, scaledim, spacetime) remain defended by dense-GP identities only (tests/test_oracle_golden.py).
 *
 * Conventions (identical to what R hands over): column-major matrices, FP64, int32 indices, 1-based, NA = INT_MIN.
 */
#ifndef NNGP_ORACLE_H
#define NNGP_ORACLE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define ORACLE_NA_INT (-2147483647 - 1)

enum oracle_covfun {
    ORACLE_EXPONENTIAL_ISOTROPIC = 0,
    ORACLE_EXPONENTIAL_SPHERE = 1,
    ORACLE_EXPONENTIAL_SCALEDIM = 2,
    ORACLE_EXPONENTIAL_SPACETIME = 3,
    ORACLE_MATERN_ISOTROPIC = 4,
    ORACLE_MATERN_SPHERE = 5,
    ORACLE_MATERN_SCALEDIM = 6,
    ORACLE_MATERN_SPACETIME = 7
};

/* ---- GpGp's randomised ordering and jittered neighbour search, on R's stream (gpgp_order.c) ---- */
void oracle_order_maxmin_gpgp(const double *locs, int n, int d, int *order_out);
void oracle_find_ordered_nn_gpgp(const double *locs, int n, int d, int m, int *NNarray);

/* ---- R random numbers (r_rng.c) ---- */
void r_set_seed(uint32_t seed);
double r_unif_rand(void);
double r_norm_rand(void);
double r_qnorm(double p);
void r_runif(int n, double *out);
void r_rnorm(int n, double mean, double sd, double *out);
double r_unif_index(double dn);
void r_sample_perm(int n, int *out);
void r_sample_int(int n, int size, int *out);
double r_rbeta(double aa, double bb);
void r_rng_get_state(uint32_t *state625);
void r_rng_set_state(const uint32_t *state625);

/* modified Bessel function of the second kind, real order (bessel_shim.cpp: std::cyl_bessel_k) */
double oracle_bessel_k(double nu, double x);

/* ---- graph structure ---- */
/* GpGp::find_ordered_nn semantics (exact, no jitter): col 0 = self, then <= m previous sites by increasing distance,
 * ties by lower index.  Scripts/mcmc_nngp_initialize.R:93, golden Vignette.md:221-227. */
void oracle_find_ordered_nn(const double *locs, int n, int d, int m, int *NNarray);
/* pattern(A^T A) incl. diagonal (initialize.R:103-109) as CSC (adj_p[n+1], adj_i, 0-based, sorted). Returns nnz; call
 * with adj_i == NULL to size. */
int64_t oracle_moral_graph(const int *NNarray, int n, int m, int64_t *adj_p, int *adj_i);
/* Coloring.R:2-20, first-fit greedy with the dense incompatibility scratch.  cols are 1..K. Returns K. */
int oracle_naive_greedy_coloring(const int64_t *adj_p, const int *adj_i, int n, int *cols);

/* ---- Vecchia factor and products ---- */
/* GpGp::vecchia_Linv(covparms, covfun_name, locs, NNarray) -> Linv n x (m+1); returns #rows whose block was not PD */
int oracle_vecchia_linv(const double *covparms, int ncovparms, int covfun, const double *locs, int n, int d,
                        const int *NNarray, int m, double *Linv);
/* GpGp::Linv_mult(Linv, z, NNarray) == sparse_chol %*% z */
void oracle_linv_mult(const double *Linv, const double *z, const int *NNarray, int n, int m, double *out);
/* ll_compressed_sparse_chol (update_Gaussian.R:8-12) */
double oracle_ll_compressed_sparse_chol(const double *Linv, const double *field, const int *NNarray, int n, int m,
                                        double log_scale);
/* precision_diag (update_Gaussian.R:74) */
void oracle_precision_diag(const double *Linv, const int *NNarray, int n, int m, double *out);
/* Matrix::solve(sparse_chol, b) (initialize.R:208, update_Gaussian.R:127, predict.R:46) */
void oracle_sparse_chol_solve(const double *Linv, const int *NNarray, int n, int m, const double *b, double *x);
/* crossprod(sparse_chol, u) = t(sparse_chol) %*% u */
void oracle_sparse_chol_tmult(const double *Linv, const int *NNarray, int n, int m, const double *u, double *out);

/* ---- sampler pieces ---- */
/* chromatic sweep exactly as written at update_Gaussian.R:257-275 (one full sparse mat-vec per colour).
 * z: n normals per sweep, consumed colour by colour (colours 1..K), sites ascending within a colour, i.e. the order in
 * which rnorm(length(selected_locs)) would hand them out.  field includes beta_0 and is updated in place. */
void oracle_chromatic_sweep_reference(const double *Linv, const int *NNarray, int n, int m, const int *coloring,
                                      int n_colors, const double *precision_diag, const double *obs_per_loc,
                                      const double *residuals_sum, double beta_0, double log_scale,
                                      double log_noise_variance, const double *z, double *field);
/* the same update written in the O(n m) residual-maintained form (SURVEY.md 8a H6); CPU-baseline variant (b) */
void oracle_chromatic_sweep_residual(const double *Linv, const int *NNarray, int n, int m, const int *coloring,
                                     int n_colors, const double *precision_diag, const double *obs_per_loc,
                                     const double *residuals_sum, double beta_0, double log_scale,
                                     double log_noise_variance, const double *z, double *field);
/* residuals_sum = residuals_sum_matrix %*% (observed_field - mu)   (update_Gaussian.R:90,260) */
void oracle_residuals_sum(const int *locs_match, int n_obs, int n, const double *observed_field, const double *mu,
                          double *out);
/* sum(dnorm(y, mean = field[locs_match] + mu - beta_0, sd = exp(.5 lnv), log = T))  (update_Gaussian.R:129-131) */
double oracle_obs_loglik(const int *locs_match, int n_obs, const double *observed_field, const double *field,
                         const double *mu, double beta_0, double log_noise_variance);
/* sum((y - field[locs_match] - mu + beta_0)^2)   (update_Gaussian.R:281) */
double oracle_ssr(const int *locs_match, int n_obs, const double *observed_field, const double *field,
                  const double *mu, double beta_0);
/* beta_0 | field, no-regressor case (update_Gaussian.R:219-224): returns mean and variance of the Gaussian draw */
void oracle_beta0_moments(const double *Linv, const int *NNarray, int n, int m, const double *field, double log_scale,
                          double *mean, double *var);
/* one stored sample of mcmc_nngp_predict_field (predict.R:43-53). Linv/NNarray cover n + n_pred rows. */
void oracle_predict_field_sample(const double *Linv, const int *NNarray, int n, int n_pred, int m, const double *field,
                                 double beta_0, double log_scale, const double *z_pred, double *out);

/* ---- one chain of mcmc_nngp_update_Gaussian, no-regressor case (update_Gaussian.R:34-315) driven by R's RNG ---- */
typedef struct {
    double shape[4];
    int n_shape;
    double beta_0;
    double log_scale;
    double log_noise_variance;
    double logvar_sufficient;
    double logvar_ancillary;
} oracle_chain_params;

/* Runs n_iterations_update iterations.  field (n) is state$params$field, updated in place.  records: column-major
 * n_iter x (3 + n_shape): beta_0, log_scale, log_noise_variance, shape...; field_records: round(n_iter*thin) x n
 * (row k = iteration k/thin) or NULL.  sweep_form: 0 = as written in R, 1 = residual form. seed = iter_start + chain i.
 * Returns 0 on success. */
int oracle_update_gaussian_chain(const double *locs, int n, int d, const int *NNarray, int m, const int *coloring,
                                 int n_colors, const int *locs_match, int n_obs, const double *obs_per_loc,
                                 const double *observed_field, int covfun, oracle_chain_params *p, double *field,
                                 int n_iterations_update, double field_thinning, int n_chromatic, int iter_start,
                                 int chain_index, int sweep_form, double *records, double *field_records,
                                 int *accept_records);

/* ---- the same chain with regressors (update_Gaussian.R:226-250; X as prepared by mcmc_nngp_initialize.R:116-137) ---- */
typedef struct {
    int p;                          /* ncol(X$X) */
    const double *X;                /* X$X: n_obs x p column-major, centred, no intercept column */
    int n_xlocs;                    /* length(X$locs); 0 = no location-level regressors */
    const int *xlocs;               /* X$locs, 1-based columns of X$X */
    const int *first_obs;           /* vecchia_approx$hctam_scol_1: n, 1-based (used when n_xlocs > 0) */
    const double *solve_1XT1X;      /* (p+1) x (p+1), initialize.R:135 */
    const double *chol_solve_1XT1X; /* (p+1) x (p+1) upper factor, initialize.R:136 */
    double *beta;                   /* p: state$params$beta, in/out */
    double *beta_records;           /* n_iter x p column-major, or NULL */
} oracle_regressors;

/* reg == NULL: identical to oracle_update_gaussian_chain. Returns non-zero if an interweaving matrix is singular. */
int oracle_update_gaussian_chain_x(const double *locs, int n, int d, const int *NNarray, int m, const int *coloring,
                                   int n_colors, const int *locs_match, int n_obs, const double *obs_per_loc,
                                   const double *observed_field, int covfun, oracle_chain_params *p, double *field,
                                   int n_iterations_update, double field_thinning, int n_chromatic, int iter_start,
                                   int chain_index, int sweep_form, double *records, double *field_records,
                                   int *accept_records, const oracle_regressors *reg);

/* ---- the product's on-device Philox normals (device_math.cuh philox_normal, nngp_b200.cu set_sweep_params) ---- */
/* Philox4x32-10 (Salmon et al. 2011) */
void oracle_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
/* key of a seed: s = (uint64)(int64)seed, key = (s & 0xffffffff, (s >> 32) ^ 0x5eed5eed) */
void oracle_philox_key(int64_t seed, uint32_t key[2]);
/* normal of 0-based site `site` at sweep counter `counter`: counter words (site, counter lo, counter hi, 0x4e4e4750); Box-Muller
 * with cos(2 pi u2) (the device takes cospi(2 u2), which glibc lacks) */
double oracle_philox_normal(uint32_t site, uint64_t counter, uint32_t k0, uint32_t k1);
/* the n normals of one sweep in hand-out order: colour 1..n_colors, ascending site index inside a colour */
void oracle_philox_handout(const int *coloring, int n, int n_colors, uint64_t counter, uint32_t k0, uint32_t k1, double *z);

#define ORACLE_RNG_R 0
#define ORACLE_RNG_PHILOX 1
/* oracle_update_gaussian_chain_x with a choice of the field normals.  ORACLE_RNG_R: R's stream, as above (philox_seed and
 * sweep_counter unused).  ORACLE_RNG_PHILOX: as nngp_chain_run* in NNGP_RNG_PHILOX mode -- the scalar draws stay on R's stream
 * (set.seed(iter_start + chain_index)), the dead rnorm(n) of update_Gaussian.R:75 and the rnorm of every sweep are skipped, and
 * sweep j of the call (j = 0, 1, ...) draws the Philox normals of counter sweep_counter + j under philox_seed. */
int oracle_update_gaussian_chain_rng(const double *locs, int n, int d, const int *NNarray, int m, const int *coloring,
                                     int n_colors, const int *locs_match, int n_obs, const double *obs_per_loc,
                                     const double *observed_field, int covfun, oracle_chain_params *p, double *field,
                                     int n_iterations_update, double field_thinning, int n_chromatic, int iter_start,
                                     int chain_index, int sweep_form, double *records, double *field_records,
                                     int *accept_records, const oracle_regressors *reg, int rng_mode, int64_t philox_seed,
                                     uint64_t sweep_counter);

#ifdef __cplusplus
}
#endif
#endif
