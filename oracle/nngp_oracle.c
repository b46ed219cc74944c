/*
 * oracle/nngp_oracle.c -- TEST INFRASTRUCTURE ONLY (never linked into, or called by, the product library).
 *
 * Plain-C, single-threaded, FP64 restatement of the reference's NNGP hot path.  Every function cites the reference
 * lines it follows (paths relative to /root/reference).  The arithmetic of GpGp::vecchia_Linv / GpGp::Linv_mult and
 * Matrix's sparse products/solves lives in CRAN packages that are NOT under /root/reference and are not installed
 * here (GpGp, Matrix: versions unpinned by the reference, circa mid-2021); their published algorithms are restated
 * (SURVEY.md Appendix D) and anchored by the reference's own call sites and by dense-GP identities.
 * PARITY UNPINNED by any reference test (there are none); see oracle/README.md for what is pinned.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include "nngp_oracle.h"

#define NA ORACLE_NA_INT
#define NNAT(i, j) NNarray[(size_t)(i) + (size_t)n * (size_t)(j)]
#define LAT(i, j) Linv[(size_t)(i) + (size_t)n * (size_t)(j)]

/* ------------------------------------------------------------------------------------------------------------- */
/* graph structure                                                                                                 */
/* ------------------------------------------------------------------------------------------------------------- */

typedef struct { double d2; int idx; } cand_t;
static int cand_cmp(const void *a, const void *b)
{
    const cand_t *x = (const cand_t *)a, *y = (const cand_t *)b;
    if (x->d2 < y->d2) return -1;
    if (x->d2 > y->d2) return 1;
    return (x->idx > y->idx) - (x->idx < y->idx);
}

/* Scripts/mcmc_nngp_initialize.R:93 (GpGp::find_ordered_nn); layout pinned by Vignette.md:221-227.
 * Brute force O(n^2 log n): only for test sizes. */
void oracle_find_ordered_nn(const double *locs, int n, int d, int m, int *NNarray)
{
    cand_t *c = (cand_t *)malloc(sizeof(cand_t) * (size_t)(n > 0 ? n : 1));
    for (int i = 0; i < n; i++) {
        for (int p = 0; p < i; p++) {
            double s = 0.0;
            for (int k = 0; k < d; k++) {
                double t = locs[i + (size_t)n * k] - locs[p + (size_t)n * k];
                s += t * t;
            }
            c[p].d2 = s;
            c[p].idx = p;
        }
        qsort(c, (size_t)i, sizeof(cand_t), cand_cmp);
        NNAT(i, 0) = i + 1;
        for (int j = 1; j <= m; j++) NNAT(i, j) = (j <= i) ? c[j - 1].idx + 1 : NA;
    }
    free(c);
}

static int int_cmp(const void *a, const void *b)
{
    int x = *(const int *)a, y = *(const int *)b;
    return (x > y) - (x < y);
}

/* Scripts/mcmc_nngp_initialize.R:103-109: crossprod(sparseMatrix(i=row,j=col,x=1)) = pattern(A^T A): two sites are
 * adjacent iff they appear together in some row of NNarray; the diagonal is present. Golden: Vignette.md:275-306. */
int64_t oracle_moral_graph(const int *NNarray, int n, int m, int64_t *adj_p, int *adj_i)
{
    /* pass 1: count (with duplicates), pass 2: fill, then sort+unique each column */
    int64_t *cnt = (int64_t *)calloc((size_t)n + 1, sizeof(int64_t));
    for (int i = 0; i < n; i++) {
        int b = 0;
        for (int j = 0; j <= m; j++) if (NNAT(i, j) != NA) b++;
        for (int j = 0; j <= m; j++) if (NNAT(i, j) != NA) cnt[NNAT(i, j) - 1 + 1] += b;
    }
    for (int s = 0; s < n; s++) cnt[s + 1] += cnt[s];
    int64_t tot = cnt[n];
    int *buf = (int *)malloc(sizeof(int) * (size_t)(tot > 0 ? tot : 1));
    int64_t *pos = (int64_t *)malloc(sizeof(int64_t) * ((size_t)n + 1));
    memcpy(pos, cnt, sizeof(int64_t) * ((size_t)n + 1));
    for (int i = 0; i < n; i++) {
        for (int j = 0; j <= m; j++) {
            if (NNAT(i, j) == NA) continue;
            int s = NNAT(i, j) - 1;
            for (int k = 0; k <= m; k++) if (NNAT(i, k) != NA) buf[pos[s]++] = NNAT(i, k) - 1;
        }
    }
    int64_t nnz = 0;
    if (adj_p) adj_p[0] = 0;
    for (int s = 0; s < n; s++) {
        int64_t a = cnt[s], b = cnt[s + 1];
        qsort(buf + a, (size_t)(b - a), sizeof(int), int_cmp);
        int last = -1;
        for (int64_t k = a; k < b; k++) {
            if (buf[k] != last) {
                if (adj_i) adj_i[nnz] = buf[k];
                nnz++;
                last = buf[k];
            }
        }
        if (adj_p) adj_p[s + 1] = nnz;
    }
    free(buf); free(pos); free(cnt);
    return nnz;
}

/* Scripts/Coloring.R:2-20.  incompatibilities is the (n+1) x max(degrees) scratch (bytes here instead of doubles);
 * cols[i] = match(0, incompatibilities[i,]) ; incompatibilities[idx[[i]], cols[i]] = 1 (idx includes i itself). */
int oracle_naive_greedy_coloring(const int64_t *adj_p, const int *adj_i, int n, int *cols)
{
    int64_t maxdeg = 0;
    for (int s = 0; s < n; s++) if (adj_p[s + 1] - adj_p[s] > maxdeg) maxdeg = adj_p[s + 1] - adj_p[s];
    unsigned char *inc = (unsigned char *)calloc((size_t)(n + 1) * (size_t)(maxdeg > 0 ? maxdeg : 1), 1);
    int K = 0;
    for (int i = 0; i < n; i++) {
        int c = 0;
        while (inc[(size_t)i * maxdeg + c]) c++; /* match(0, row): first zero; always exists since deg <= maxdeg */
        cols[i] = c + 1;
        if (c + 1 > K) K = c + 1;
        for (int64_t k = adj_p[i]; k < adj_p[i + 1]; k++) inc[(size_t)adj_i[k] * maxdeg + c] = 1;
    }
    free(inc);
    return K;
}

/* ------------------------------------------------------------------------------------------------------------- */
/* covariance functions (GpGp; SURVEY.md Appendix D), zero-nugget / unit-variance as the reference calls them      */
/* ------------------------------------------------------------------------------------------------------------- */

static int covfun_is_matern(int covfun) { return covfun >= ORACLE_MATERN_ISOTROPIC; }

/* coordinates after the family's transformation: scaled by the range(s); lon/lat -> unit sphere for *_sphere */
static int transformed_dim(int covfun, int d)
{
    return (covfun == ORACLE_EXPONENTIAL_SPHERE || covfun == ORACLE_MATERN_SPHERE) ? 3 : d;
}

static void transform_locs(const double *covparms, int covfun, const double *locs, int n, int d, double *tl /* n x dt row-major */)
{
    int dt = transformed_dim(covfun, d);
    for (int i = 0; i < n; i++) {
        double *o = tl + (size_t)i * dt;
        switch (covfun) {
        case ORACLE_EXPONENTIAL_ISOTROPIC:
        case ORACLE_MATERN_ISOTROPIC:
            for (int k = 0; k < d; k++) o[k] = locs[i + (size_t)n * k] / covparms[1];
            break;
        case ORACLE_EXPONENTIAL_SPHERE:
        case ORACLE_MATERN_SPHERE: {
            double lon = locs[i] * M_PI / 180.0, lat = locs[i + (size_t)n] * M_PI / 180.0;
            o[0] = cos(lat) * cos(lon) / covparms[1];
            o[1] = cos(lat) * sin(lon) / covparms[1];
            o[2] = sin(lat) / covparms[1];
            break;
        }
        case ORACLE_EXPONENTIAL_SCALEDIM:
        case ORACLE_MATERN_SCALEDIM:
            for (int k = 0; k < d; k++) o[k] = locs[i + (size_t)n * k] / covparms[1 + k];
            break;
        case ORACLE_EXPONENTIAL_SPACETIME:
        case ORACLE_MATERN_SPACETIME:
            for (int k = 0; k < d - 1; k++) o[k] = locs[i + (size_t)n * k] / covparms[1];
            o[d - 1] = locs[i + (size_t)n * (d - 1)] / covparms[2];
            break;
        }
    }
}

static double kernel_value(int covfun, double variance, double smooth, double normcon, double dist)
{
    if (!covfun_is_matern(covfun)) return variance * exp(-dist);
    if (dist == 0.0) return variance;
    return normcon * pow(dist, smooth) * oracle_bessel_k(smooth, dist);
}

/* GpGp::vecchia_Linv (Scripts/mcmc_nngp_update_Gaussian.R:72,123,179; initialize.R:201; predict.R:39).
 * Per row: neighbours in reverse slot order (farthest first, self last), covariance block, lower Cholesky, solve
 * L^T x = e_last, write x reversed.  Slot 0 = 1/sqrt(F_i); slots >= 1 = -B_ij / sqrt(F_i). */
int oracle_vecchia_linv(const double *covparms, int ncovparms, int covfun, const double *locs, int n, int d,
                        const int *NNarray, int m, double *Linv)
{
    int dt = transformed_dim(covfun, d);
    double *tl = (double *)malloc(sizeof(double) * (size_t)n * dt);
    transform_locs(covparms, covfun, locs, n, d, tl);
    double variance = covparms[0];
    double nugget = covparms[ncovparms - 1] * variance;
    double smooth = covfun_is_matern(covfun) ? covparms[ncovparms - 2] : 0.0;
    double normcon = covfun_is_matern(covfun) ? variance / (pow(2.0, smooth - 1.0) * tgamma(smooth)) : 0.0;
    int M = m + 1, bad = 0;
    double *S = (double *)malloc(sizeof(double) * M * M);
    double *x = (double *)malloc(sizeof(double) * M);
    int *sub = (int *)malloc(sizeof(int) * M);
    for (int i = 0; i < n; i++) {
        int bsize = 0;
        for (int j = 0; j < M; j++) if (NNAT(i, j) != NA) bsize++;
        for (int k = 0; k < bsize; k++) sub[k] = NNAT(i, bsize - 1 - k) - 1;
        for (int a = 0; a < bsize; a++)
            for (int b = 0; b <= a; b++) {
                double s = 0.0;
                for (int k = 0; k < dt; k++) {
                    double t = tl[(size_t)sub[a] * dt + k] - tl[(size_t)sub[b] * dt + k];
                    s += t * t;
                }
                double v = kernel_value(covfun, variance, smooth, normcon, sqrt(s));
                if (a == b) v += nugget;
                S[a * M + b] = v;
            }
        /* lower Cholesky, row by row (Cholesky-Banachiewicz) */
        int ok = 1;
        for (int a = 0; a < bsize; a++) {
            for (int b = 0; b <= a; b++) {
                double s = S[a * M + b];
                for (int k = 0; k < b; k++) s -= S[a * M + k] * S[b * M + k];
                if (a == b) {
                    if (!(s > 0.0)) ok = 0;
                    S[a * M + a] = sqrt(s);
                } else {
                    S[a * M + b] = s / S[b * M + b];
                }
            }
        }
        if (!ok) bad++;
        /* solve L^T x = e_last by back substitution */
        for (int a = bsize - 1; a >= 0; a--) {
            double s = (a == bsize - 1) ? 1.0 : 0.0;
            for (int k = a + 1; k < bsize; k++) s -= S[k * M + a] * x[k];
            x[a] = s / S[a * M + a];
        }
        for (int j = 0; j < M; j++) LAT(i, j) = (j < bsize) ? x[bsize - 1 - j] : 0.0;
    }
    free(sub); free(x); free(S); free(tl);
    return bad;
}

/* GpGp::Linv_mult (update_Gaussian.R:10): out[i] = sum_j Linv[i,j] * z[NNarray[i,j]] */
void oracle_linv_mult(const double *Linv, const double *z, const int *NNarray, int n, int m, double *out)
{
    for (int i = 0; i < n; i++) {
        double s = 0.0;
        for (int j = 0; j <= m; j++)
            if (NNAT(i, j) != NA) s += LAT(i, j) * z[NNAT(i, j) - 1];
        out[i] = s;
    }
}

/* update_Gaussian.R:8-12 */
double oracle_ll_compressed_sparse_chol(const double *Linv, const double *field, const int *NNarray, int n, int m,
                                        double log_scale)
{
    double *chol_field = (double *)malloc(sizeof(double) * (size_t)n);
    oracle_linv_mult(Linv, field, NNarray, n, m, chol_field);
    double sum_log = 0.0, sum_sq = 0.0;
    for (int i = 0; i < n; i++) sum_log += log(LAT(NNAT(i, 0) - 1, 0));
    for (int i = 0; i < n; i++) sum_sq += chol_field[i] * chol_field[i];
    free(chol_field);
    return sum_log - n * 0.5 * log_scale - 0.5 * sum_sq / exp(log_scale);
}

/* update_Gaussian.R:74: (x^2) %*% indicator(k -> column_idx[k]); entries visited in column-major scan of NNarray */
void oracle_precision_diag(const double *Linv, const int *NNarray, int n, int m, double *out)
{
    for (int s = 0; s < n; s++) out[s] = 0.0;
    for (int j = 0; j <= m; j++)
        for (int i = 0; i < n; i++)
            if (NNAT(i, j) != NA) out[NNAT(i, j) - 1] += LAT(i, j) * LAT(i, j);
}

/* Matrix::solve(dtCMatrix, b): forward substitution.  Row i of sparse_chol holds Linv[i,0] on the diagonal and
 * Linv[i,j>=1] at columns NNarray[i,j] < i. */
void oracle_sparse_chol_solve(const double *Linv, const int *NNarray, int n, int m, const double *b, double *x)
{
    for (int i = 0; i < n; i++) {
        double s = b[i];
        for (int j = 1; j <= m; j++)
            if (NNAT(i, j) != NA) s -= LAT(i, j) * x[NNAT(i, j) - 1];
        x[i] = s / LAT(i, 0);
    }
}

/* Matrix::crossprod(sparse_chol, u) */
void oracle_sparse_chol_tmult(const double *Linv, const int *NNarray, int n, int m, const double *u, double *out)
{
    for (int s = 0; s < n; s++) out[s] = 0.0;
    for (int i = 0; i < n; i++)
        for (int j = 0; j <= m; j++)
            if (NNAT(i, j) != NA) out[NNAT(i, j) - 1] += LAT(i, j) * u[i];
}

/* ------------------------------------------------------------------------------------------------------------- */
/* sampler pieces                                                                                                  */
/* ------------------------------------------------------------------------------------------------------------- */

/* transpose structure: for site s the list of (row i, slot j) with NNarray[i,j] == s, rows ascending */
typedef struct { int64_t *p; int *row; int *slot; } csc_t;

static void csc_build(const int *NNarray, int n, int m, csc_t *c)
{
    c->p = (int64_t *)calloc((size_t)n + 1, sizeof(int64_t));
    for (int i = 0; i < n; i++)
        for (int j = 0; j <= m; j++)
            if (NNAT(i, j) != NA) c->p[NNAT(i, j)]++;
    for (int s = 0; s < n; s++) c->p[s + 1] += c->p[s];
    int64_t nnz = c->p[n];
    c->row = (int *)malloc(sizeof(int) * (size_t)(nnz > 0 ? nnz : 1));
    c->slot = (int *)malloc(sizeof(int) * (size_t)(nnz > 0 ? nnz : 1));
    int64_t *pos = (int64_t *)malloc(sizeof(int64_t) * ((size_t)n + 1));
    memcpy(pos, c->p, sizeof(int64_t) * ((size_t)n + 1));
    for (int i = 0; i < n; i++)
        for (int j = 0; j <= m; j++)
            if (NNAT(i, j) != NA) {
                int s = NNAT(i, j) - 1;
                c->row[pos[s]] = i;
                c->slot[pos[s]] = j;
                pos[s]++;
            }
    free(pos);
}
static void csc_free(csc_t *c) { free(c->p); free(c->row); free(c->slot); }

/* update_Gaussian.R:257-275, body of the colour loop for one sweep, in the reference's algorithmic form */
static void sweep_reference(const double *Linv, const int *NNarray, int n, int m, const csc_t *csc, const int *coloring,
                            int n_colors, const double *precision_diag, const double *obs_per_loc,
                            const double *residuals_sum, double beta_0, double log_scale, double log_noise_variance,
                            const double *z, double *field, double *v, double *u)
{
    size_t zi = 0;
    double e_ls = exp(-log_scale), e_ln = exp(-log_noise_variance);
    for (int c = 1; c <= n_colors; c++) {
        for (int s = 0; s < n; s++) v[s] = (field[s] - beta_0) * (coloring[s] != c ? 1.0 : 0.0);   /* :269 */
        oracle_linv_mult(Linv, v, NNarray, n, m, u);                                              /* sparse_chol %*% . */
        for (int s = 0; s < n; s++) {
            if (coloring[s] != c) continue;
            double posterior_precision = e_ls * precision_diag[s] + e_ln * obs_per_loc[s];          /* :264 */
            double t = 0.0;                                                                         /* crossprod(sparse_chol[,sel], u) */
            for (int64_t k = csc->p[s]; k < csc->p[s + 1]; k++)
                t += Linv[(size_t)csc->row[k] + (size_t)n * csc->slot[k]] * u[csc->row[k]];
            double cond_mean = beta_0 - (1.0 / posterior_precision) * (t * e_ls - e_ln * residuals_sum[s]); /* :266-271 */
            field[s] = cond_mean + z[zi++] / sqrt(posterior_precision);                             /* :273 */
        }
    }
}

/* same conditional, O(n m): keep r = sparse_chol %*% (field - beta_0) and patch it after every site */
static void sweep_residual(const double *Linv, int n, const csc_t *csc, const int *coloring, int n_colors,
                           const int *color_order /* sites sorted by (colour, index) */, const int64_t *color_ptr,
                           const double *precision_diag, const double *obs_per_loc, const double *residuals_sum,
                           double beta_0, double log_scale, double log_noise_variance, const double *z, double *field,
                           double *r)
{
    (void)coloring;
    size_t zi = 0;
    double e_ls = exp(-log_scale), e_ln = exp(-log_noise_variance);
    for (int c = 1; c <= n_colors; c++) {
        for (int64_t q = color_ptr[c - 1]; q < color_ptr[c]; q++) {
            int s = color_order[q];
            double posterior_precision = e_ls * precision_diag[s] + e_ln * obs_per_loc[s];
            double w_old = field[s] - beta_0;
            double t = 0.0;
            for (int64_t k = csc->p[s]; k < csc->p[s + 1]; k++)
                t += Linv[(size_t)csc->row[k] + (size_t)n * csc->slot[k]] * r[csc->row[k]];
            t -= precision_diag[s] * w_old;
            double cond_mean = beta_0 - (1.0 / posterior_precision) * (t * e_ls - e_ln * residuals_sum[s]);
            double f_new = cond_mean + z[zi++] / sqrt(posterior_precision);
            double delta = (f_new - beta_0) - w_old;
            for (int64_t k = csc->p[s]; k < csc->p[s + 1]; k++)
                r[csc->row[k]] += Linv[(size_t)csc->row[k] + (size_t)n * csc->slot[k]] * delta;
            field[s] = f_new;
        }
    }
}

static void color_buckets(const int *coloring, int n, int n_colors, int **order, int64_t **ptr)
{
    *ptr = (int64_t *)calloc((size_t)n_colors + 1, sizeof(int64_t));
    *order = (int *)malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
    for (int s = 0; s < n; s++) (*ptr)[coloring[s]]++;
    for (int c = 0; c < n_colors; c++) (*ptr)[c + 1] += (*ptr)[c];
    int64_t *pos = (int64_t *)malloc(sizeof(int64_t) * ((size_t)n_colors + 1));
    memcpy(pos, *ptr, sizeof(int64_t) * ((size_t)n_colors + 1));
    for (int s = 0; s < n; s++) (*order)[pos[coloring[s] - 1]++] = s;
    free(pos);
}

void oracle_chromatic_sweep_reference(const double *Linv, const int *NNarray, int n, int m, const int *coloring,
                                      int n_colors, const double *precision_diag, const double *obs_per_loc,
                                      const double *residuals_sum, double beta_0, double log_scale,
                                      double log_noise_variance, const double *z, double *field)
{
    csc_t csc;
    csc_build(NNarray, n, m, &csc);
    double *v = (double *)malloc(sizeof(double) * (size_t)n), *u = (double *)malloc(sizeof(double) * (size_t)n);
    sweep_reference(Linv, NNarray, n, m, &csc, coloring, n_colors, precision_diag, obs_per_loc, residuals_sum, beta_0,
                    log_scale, log_noise_variance, z, field, v, u);
    free(v); free(u);
    csc_free(&csc);
}

void oracle_chromatic_sweep_residual(const double *Linv, const int *NNarray, int n, int m, const int *coloring,
                                     int n_colors, const double *precision_diag, const double *obs_per_loc,
                                     const double *residuals_sum, double beta_0, double log_scale,
                                     double log_noise_variance, const double *z, double *field)
{
    csc_t csc;
    csc_build(NNarray, n, m, &csc);
    int *order; int64_t *ptr;
    color_buckets(coloring, n, n_colors, &order, &ptr);
    double *w = (double *)malloc(sizeof(double) * (size_t)n), *r = (double *)malloc(sizeof(double) * (size_t)n);
    for (int s = 0; s < n; s++) w[s] = field[s] - beta_0;
    oracle_linv_mult(Linv, w, NNarray, n, m, r);
    sweep_residual(Linv, n, &csc, coloring, n_colors, order, ptr, precision_diag, obs_per_loc, residuals_sum, beta_0,
                   log_scale, log_noise_variance, z, field, r);
    free(w); free(r); free(order); free(ptr);
    csc_free(&csc);
}

/* update_Gaussian.R:90,260 */
void oracle_residuals_sum(const int *locs_match, int n_obs, int n, const double *observed_field, const double *mu,
                          double *out)
{
    for (int s = 0; s < n; s++) out[s] = 0.0;
    for (int o = 0; o < n_obs; o++) out[locs_match[o] - 1] += observed_field[o] - mu[o];
}

/* update_Gaussian.R:129-131, dnorm(..., log = T) = -(log(sqrt(2 pi)) + 0.5 z^2 + log(sd)) */
double oracle_obs_loglik(const int *locs_match, int n_obs, const double *observed_field, const double *field,
                         const double *mu, double beta_0, double log_noise_variance)
{
    double sd = exp(0.5 * log_noise_variance), s = 0.0;
    for (int o = 0; o < n_obs; o++) {
        double zz = (observed_field[o] - (field[locs_match[o] - 1] + mu[o] - beta_0)) / sd;
        s += -(0.918938533204672741780329736406 + 0.5 * zz * zz + log(sd));
    }
    return s;
}

/* update_Gaussian.R:281 */
double oracle_ssr(const int *locs_match, int n_obs, const double *observed_field, const double *field,
                  const double *mu, double beta_0)
{
    double s = 0.0;
    for (int o = 0; o < n_obs; o++) {
        double e = observed_field[o] - field[locs_match[o] - 1] - mu[o] + beta_0;
        s += e * e;
    }
    return s;
}

/* update_Gaussian.R:219-224 */
void oracle_beta0_moments(const double *Linv, const int *NNarray, int n, int m, const double *field, double log_scale,
                          double *mean, double *var)
{
    double *ones = (double *)calloc((size_t)(n > 0 ? n : 1), sizeof(double)), *v = (double *)malloc(sizeof(double) * (size_t)n),
           *u = (double *)malloc(sizeof(double) * (size_t)n);
    for (int i = 0; i < n; i++) ones[i] = 1.0;
    oracle_linv_mult(Linv, ones, NNarray, n, m, v);
    oracle_linv_mult(Linv, field, NNarray, n, m, u);
    double vv = 0.0, uv = 0.0;
    for (int i = 0; i < n; i++) { vv += v[i] * v[i]; uv += u[i] * v[i]; }
    double beta_covmat = (1.0 / vv) * exp(log_scale);
    *var = beta_covmat;
    *mean = exp(-log_scale) * uv * beta_covmat;
    free(ones); free(v); free(u);
}

/* predict.R:43-53: spat_sd * solve(sparse_chol, c((1/spat_sd) * sparse_chol[1:n,1:n] %*% (field - beta_0), z))[-(1:n)] */
void oracle_predict_field_sample(const double *Linv_all, const int *NN_all, int n, int n_pred, int m,
                                 const double *field, double beta_0, double log_scale, const double *z_pred, double *out)
{
    int nt = n + n_pred;
    double spat_sd = exp(0.5 * log_scale);
    double *rhs = (double *)malloc(sizeof(double) * (size_t)nt), *x = (double *)malloc(sizeof(double) * (size_t)nt);
    for (int i = 0; i < n; i++) {
        double s = 0.0;
        for (int j = 0; j <= m; j++) {
            int p = NN_all[(size_t)i + (size_t)nt * j];
            if (p != NA) s += Linv_all[(size_t)i + (size_t)nt * j] * (field[p - 1] - beta_0);
        }
        rhs[i] = (1.0 / spat_sd) * s;
    }
    for (int i = 0; i < n_pred; i++) rhs[n + i] = z_pred[i];
    oracle_sparse_chol_solve(Linv_all, NN_all, nt, m, rhs, x);
    for (int i = 0; i < n_pred; i++) out[i] = spat_sd * x[n + i];
    free(rhs); free(x);
}

/* ------------------------------------------------------------------------------------------------------------- */
/* one chain, no regressors: update_Gaussian.R:34-315                                                              */
/* ------------------------------------------------------------------------------------------------------------- */

static void shape_to_covparms(int covfun, const double *shape, int n_shape, double *cp, int *ncp)
{
    /* update_Gaussian.R:67-71: "log*" -> exp, "qlogis*" -> .5 + .5 plogis; the matern families' last shape is qlogis */
    cp[0] = 1.0;
    for (int j = 0; j < n_shape; j++) {
        int is_qlogis = covfun_is_matern(covfun) && (j == n_shape - 1);
        cp[1 + j] = is_qlogis ? 0.5 + 0.5 * (1.0 / (1.0 + exp(-shape[j]))) : exp(shape[j]);
    }
    cp[1 + n_shape] = 0.0;
    *ncp = n_shape + 2;
}

static double sample_var(const double *x, int n)
{
    double mean = 0.0;
    for (int i = 0; i < n; i++) mean += x[i];
    mean /= n;
    double s = 0.0;
    for (int i = 0; i < n; i++) s += (x[i] - mean) * (x[i] - mean);
    return s / (n - 1);
}

/* ---- small dense helpers for the regression block (R: solve(), chol(); column-major q x q) ---- */
static int dense_chol_lower(double *A, int q)
{
    for (int j = 0; j < q; j++) {
        double dj = A[j + (size_t)q * j];
        for (int k = 0; k < j; k++) dj -= A[j + (size_t)q * k] * A[j + (size_t)q * k];
        if (!(dj > 0.0)) return 1;
        dj = sqrt(dj);
        A[j + (size_t)q * j] = dj;
        for (int i = j + 1; i < q; i++) {
            double v = A[i + (size_t)q * j];
            for (int k = 0; k < j; k++) v -= A[i + (size_t)q * k] * A[j + (size_t)q * k];
            A[i + (size_t)q * j] = v / dj;
        }
        for (int i = 0; i < j; i++) A[i + (size_t)q * j] = 0.0;
    }
    return 0;
}

/* inv = P^-1 for symmetric positive definite P, by Gauss-Jordan elimination with partial pivoting (what solve() does
 * up to the order of operations) */
static int dense_inverse(const double *P, int q, double *inv)
{
    double *A = (double *)malloc(sizeof(double) * (size_t)q * q);
    memcpy(A, P, sizeof(double) * (size_t)q * q);
    for (int i = 0; i < q; i++) for (int j = 0; j < q; j++) inv[i + (size_t)q * j] = (i == j) ? 1.0 : 0.0;
    for (int c = 0; c < q; c++) {
        int piv = c;
        for (int r = c + 1; r < q; r++) if (fabs(A[r + (size_t)q * c]) > fabs(A[piv + (size_t)q * c])) piv = r;
        if (A[piv + (size_t)q * c] == 0.0) { free(A); return 1; }
        if (piv != c)
            for (int j = 0; j < q; j++) {
                double t = A[c + (size_t)q * j]; A[c + (size_t)q * j] = A[piv + (size_t)q * j]; A[piv + (size_t)q * j] = t;
                t = inv[c + (size_t)q * j]; inv[c + (size_t)q * j] = inv[piv + (size_t)q * j]; inv[piv + (size_t)q * j] = t;
            }
        double dinv = 1.0 / A[c + (size_t)q * c];
        for (int j = 0; j < q; j++) { A[c + (size_t)q * j] *= dinv; inv[c + (size_t)q * j] *= dinv; }
        for (int r = 0; r < q; r++) {
            if (r == c) continue;
            double f = A[r + (size_t)q * c];
            if (f == 0.0) continue;
            for (int j = 0; j < q; j++) { A[r + (size_t)q * j] -= f * A[c + (size_t)q * j]; inv[r + (size_t)q * j] -= f * inv[c + (size_t)q * j]; }
        }
    }
    free(A);
    return 0;
}

/* update_Gaussian.R:77-83: sparse_chol_X_locs = sparse_chol %*% cbind(1, X$X[hctam_scol_1, X$locs]) (n x q),
 * beta_interweaved_covmat = solve(crossprod(.)), chol_lower = t(chol(covmat)) */
static int interweave_matrices(const double *Linv, const int *NNarray, int n, int m, const double *Xl, int q,
                               double *scXl, double *cov, double *chol_lower)
{
    for (int l = 0; l < q; l++) oracle_linv_mult(Linv, Xl + (size_t)l * n, NNarray, n, m, scXl + (size_t)l * n);
    double *prec = (double *)malloc(sizeof(double) * (size_t)q * q);
    for (int a = 0; a < q; a++)
        for (int b = 0; b < q; b++) {
            double v = 0.0;
            for (int s = 0; s < n; s++) v += scXl[(size_t)a * n + s] * scXl[(size_t)b * n + s];
            prec[a + (size_t)q * b] = v;
        }
    int bad = dense_inverse(prec, q, cov);
    free(prec);
    if (bad) return 1;
    for (int a = 0; a < q; a++)                               /* symmetrise the rounding of the elimination */
        for (int b = 0; b < a; b++) { double v = 0.5 * (cov[a + (size_t)q * b] + cov[b + (size_t)q * a]); cov[a + (size_t)q * b] = v; cov[b + (size_t)q * a] = v; }
    memcpy(chol_lower, cov, sizeof(double) * (size_t)q * q);
    return dense_chol_lower(chol_lower, q);
}

int oracle_update_gaussian_chain(const double *locs, int n, int d, const int *NNarray, int m, const int *coloring,
                                 int n_colors, const int *locs_match, int n_obs, const double *obs_per_loc,
                                 const double *observed_field, int covfun, oracle_chain_params *p, double *field,
                                 int n_iterations_update, double field_thinning, int n_chromatic, int iter_start,
                                 int chain_index, int sweep_form, double *records, double *field_records,
                                 int *accept_records)
{
    return oracle_update_gaussian_chain_x(locs, n, d, NNarray, m, coloring, n_colors, locs_match, n_obs, obs_per_loc,
                                          observed_field, covfun, p, field, n_iterations_update, field_thinning, n_chromatic,
                                          iter_start, chain_index, sweep_form, records, field_records, accept_records, NULL);
}

/* the same loop with the regression block update_Gaussian.R:226-250 when reg != NULL */
int oracle_update_gaussian_chain_x(const double *locs, int n, int d, const int *NNarray, int m, const int *coloring,
                                   int n_colors, const int *locs_match, int n_obs, const double *obs_per_loc,
                                   const double *observed_field, int covfun, oracle_chain_params *p, double *field,
                                   int n_iterations_update, double field_thinning, int n_chromatic, int iter_start,
                                   int chain_index, int sweep_form, double *records, double *field_records,
                                   int *accept_records, const oracle_regressors *reg)
{
    return oracle_update_gaussian_chain_rng(locs, n, d, NNarray, m, coloring, n_colors, locs_match, n_obs, obs_per_loc,
                                            observed_field, covfun, p, field, n_iterations_update, field_thinning, n_chromatic,
                                            iter_start, chain_index, sweep_form, records, field_records, accept_records, reg,
                                            ORACLE_RNG_R, 0, 0);
}

/* ------------------------------------------------------------------------------------------------------------- */
/* the product's Philox normals                                                                                    */
/* ------------------------------------------------------------------------------------------------------------- */

void oracle_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t x = ctr[0], y = ctr[1], z = ctr[2], w = ctr[3], k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * x, p1 = (uint64_t)0xCD9E8D57u * z;
        uint32_t nx = (uint32_t)(p1 >> 32) ^ y ^ k0, ny = (uint32_t)p1, nz = (uint32_t)(p0 >> 32) ^ w ^ k1, nw = (uint32_t)p0;
        x = nx; y = ny; z = nz; w = nw;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = x; out[1] = y; out[2] = z; out[3] = w;
}

void oracle_philox_key(int64_t seed, uint32_t key[2])
{
    uint64_t s = (uint64_t)seed;
    key[0] = (uint32_t)(s & 0xffffffffu);
    key[1] = (uint32_t)(s >> 32) ^ 0x5eed5eedu;
}

double oracle_philox_normal(uint32_t site, uint64_t counter, uint32_t k0, uint32_t k1)
{
    uint32_t c[4] = {site, (uint32_t)counter, (uint32_t)(counter >> 32), 0x4e4e4750u}, k[2] = {k0, k1}, r[4];
    oracle_philox4x32_10(c, k, r);
    uint64_t a = ((uint64_t)r[0] << 32) | r[1], b = ((uint64_t)r[2] << 32) | r[3];
    double u1 = ((double)(a >> 11) + 0.5) * 1.1102230246251565e-16;   /* 2^-53 */
    double u2 = ((double)(b >> 11) + 0.5) * 1.1102230246251565e-16;
    return sqrt(-2.0 * log(u1)) * cos(2.0 * M_PI * u2);
}

/* sites listed in hand-out order (color_buckets) */
static void philox_fill(const int *order, int n, uint64_t counter, uint32_t k0, uint32_t k1, double *z)
{
    for (int q = 0; q < n; q++) z[q] = oracle_philox_normal((uint32_t)order[q], counter, k0, k1);
}

void oracle_philox_handout(const int *coloring, int n, int n_colors, uint64_t counter, uint32_t k0, uint32_t k1, double *z)
{
    int *order; int64_t *ptr;
    color_buckets(coloring, n, n_colors, &order, &ptr);
    philox_fill(order, n, counter, k0, k1, z);
    free(order); free(ptr);
}

int oracle_update_gaussian_chain_rng(const double *locs, int n, int d, const int *NNarray, int m, const int *coloring,
                                     int n_colors, const int *locs_match, int n_obs, const double *obs_per_loc,
                                     const double *observed_field, int covfun, oracle_chain_params *p, double *field,
                                     int n_iterations_update, double field_thinning, int n_chromatic, int iter_start,
                                     int chain_index, int sweep_form, double *records, double *field_records,
                                     int *accept_records, const oracle_regressors *reg, int rng_mode, int64_t philox_seed,
                                     uint64_t sweep_counter)
{
    const int M = m + 1, n_iter = n_iterations_update, ns = p->n_shape;
    size_t lsz = (size_t)n * M;
    double *Linv = (double *)malloc(sizeof(double) * lsz), *new_Linv = (double *)malloc(sizeof(double) * lsz);
    double *precision_diag = (double *)malloc(sizeof(double) * (size_t)n);
    double *tmp = (double *)malloc(sizeof(double) * (size_t)n), *tmp2 = (double *)malloc(sizeof(double) * (size_t)n);
    double *new_field = (double *)malloc(sizeof(double) * (size_t)n);
    double *mu = (double *)malloc(sizeof(double) * (size_t)n_obs);
    double *residuals_sum = (double *)malloc(sizeof(double) * (size_t)n);
    double *z = (double *)malloc(sizeof(double) * (size_t)n);
    int *acc_suf = (int *)calloc((size_t)n_iter + 1, sizeof(int)), *acc_anc = (int *)calloc((size_t)n_iter + 1, sizeof(int));
    int n_field_rec = (int)nearbyint(n_iter * field_thinning);
    csc_t csc; csc_build(NNarray, n, m, &csc);
    int *order; int64_t *cptr; color_buckets(coloring, n, n_colors, &order, &cptr);
    double cp[8]; int ncp;
    double var_y = sample_var(observed_field, n_obs);
    double innovation[5], new_shape[4];

    r_set_seed((uint32_t)(iter_start + chain_index));                                            /* :36 */
    shape_to_covparms(covfun, p->shape, ns, cp, &ncp);                                           /* :67-71 */
    oracle_vecchia_linv(cp, ncp, covfun, locs, n, d, NNarray, m, Linv);                          /* :72 */
    oracle_precision_diag(Linv, NNarray, n, m, precision_diag);                                  /* :74 */
    const int philox = rng_mode == ORACLE_RNG_PHILOX;
    uint32_t key[2];
    oracle_philox_key(philox_seed, key);
    if (!philox)
        for (int i = 0; i < n; i++) (void)r_norm_rand();                                         /* :75 current_p (dead, but consumes the stream) */
    /* regression state: X$X (n_obs x P), site-level design Xl = cbind(1, X$X[hctam_scol_1, X$locs]) (n x q) */
    const int P = reg ? reg->p : 0, P1 = P + 1, q = (reg && reg->n_xlocs > 0) ? reg->n_xlocs + 1 : 0;
    const int wlen = P1 > q ? P1 : q;
    double *Xl = NULL, *scXl = NULL, *iw_cov = NULL, *iw_chol = NULL, *other = NULL;
    double *gvec = (double *)malloc(sizeof(double) * (size_t)wlen), *bmean = (double *)malloc(sizeof(double) * (size_t)wlen),
           *zz = (double *)malloc(sizeof(double) * (size_t)wlen), *innov = (double *)malloc(sizeof(double) * (size_t)wlen);
    int status = 0;
    if (q > 0) {
        Xl = (double *)malloc(sizeof(double) * (size_t)n * q);
        scXl = (double *)malloc(sizeof(double) * (size_t)n * q);
        iw_cov = (double *)malloc(sizeof(double) * (size_t)q * q);
        iw_chol = (double *)malloc(sizeof(double) * (size_t)q * q);
        other = (double *)malloc(sizeof(double) * (size_t)n);
        for (int s = 0; s < n; s++) {
            Xl[s] = 1.0;
            for (int l = 1; l < q; l++)
                Xl[(size_t)l * n + s] = reg->X[(size_t)(reg->first_obs[s] - 1) + (size_t)n_obs * (reg->xlocs[l - 1] - 1)];
        }
        status = interweave_matrices(Linv, NNarray, n, m, Xl, q, scXl, iw_cov, iw_chol);         /* :77-83 */
    }
#define ORACLE_SET_MU()                                                                            \
    for (int o = 0; o < n_obs; o++) {                                                              \
        double xb = 0.0;                                                                           \
        for (int k = 0; k < P; k++) xb += reg->X[(size_t)o + (size_t)n_obs * k] * reg->beta[k];    \
        mu[o] = p->beta_0 + xb;                                                                    \
    }
    if (reg) { ORACLE_SET_MU() }                                                                 /* :85 */
    else for (int o = 0; o < n_obs; o++) mu[o] = p->beta_0;                                      /* :86 */

    for (int iter = 1; iter <= n_iter && status == 0; iter++) {
        /* ---- ancillary step :113-157 ---- */
        double sd_anc = exp(.5 * p->logvar_ancillary);
        for (int k = 0; k < ns + 1; k++) innovation[k] = 0.0 + sd_anc * r_norm_rand();
        double new_log_scale = p->log_scale + innovation[0];
        for (int k = 0; k < ns; k++) new_shape[k] = p->shape[k] + innovation[1 + k];
        shape_to_covparms(covfun, new_shape, ns, cp, &ncp);
        oracle_vecchia_linv(cp, ncp, covfun, locs, n, d, NNarray, m, new_Linv);                  /* :123 */
        for (int s = 0; s < n; s++) tmp[s] = field[s] - p->beta_0;
        oracle_linv_mult(Linv, tmp, NNarray, n, m, tmp2);
        oracle_sparse_chol_solve(new_Linv, NNarray, n, m, tmp2, tmp);
        double sc = exp(.5 * (new_log_scale - p->log_scale));
        for (int s = 0; s < n; s++) new_field[s] = p->beta_0 + sc * tmp[s];                      /* :127 */
        double sd = exp(0.5 * p->log_noise_variance), ratio = 0.0;
        for (int o = 0; o < n_obs; o++) {                                                        /* :129-131 */
            int s = locs_match[o] - 1;
            double zn = (observed_field[o] - (new_field[s] + mu[o] - p->beta_0)) / sd;
            double zo = (observed_field[o] - (field[s] + mu[o] - p->beta_0)) / sd;
            ratio += -(0.918938533204672741780329736406 + 0.5 * zn * zn + log(sd)) -
                     -(0.918938533204672741780329736406 + 0.5 * zo * zo + log(sd));
        }
        if (ratio + 0.0 > log(r_unif_rand())) {                                                  /* :133 */
            memcpy(p->shape, new_shape, sizeof(double) * ns);
            p->log_scale = new_log_scale;
            memcpy(field, new_field, sizeof(double) * (size_t)n);
            memcpy(Linv, new_Linv, sizeof(double) * lsz);
            oracle_precision_diag(Linv, NNarray, n, m, precision_diag);
            acc_anc[iter] = 1;
            if (q > 0) status |= interweave_matrices(Linv, NNarray, n, m, Xl, q, scXl, iw_cov, iw_chol);   /* :145-151 */
        }
        if (iter_start >= 0 && iter_start <= 2000 && iter % 25 == 0) {                           /* :153-157 */
            int a = 0;
            for (int k = iter - 24; k <= iter; k++) a += acc_anc[k];
            double mean_acc = a / 25.0;
            if (mean_acc < .05) p->logvar_ancillary -= (.4 + .05 * r_norm_rand());
            if (mean_acc > .15) p->logvar_ancillary += (.4 + .05 * r_norm_rand());
        }
        /* ---- sufficient step :165-213 ---- */
        double sd_suf = exp(.5 * p->logvar_sufficient);
        for (int k = 0; k < ns + 1; k++) innovation[k] = 0.0 + sd_suf * r_norm_rand();
        new_log_scale = p->log_scale + innovation[0];
        if (exp(new_log_scale) < var_y) {                                                        /* :167 */
            for (int k = 0; k < ns; k++) new_shape[k] = p->shape[k] + innovation[1 + k];
            shape_to_covparms(covfun, new_shape, ns, cp, &ncp);
            oracle_vecchia_linv(cp, ncp, covfun, locs, n, d, NNarray, m, new_Linv);              /* :179 */
            for (int s = 0; s < n; s++) tmp[s] = field[s] - p->beta_0;
            double GP_ratio = oracle_ll_compressed_sparse_chol(new_Linv, tmp, NNarray, n, m, new_log_scale) -
                              oracle_ll_compressed_sparse_chol(Linv, tmp, NNarray, n, m, p->log_scale); /* :184-186 */
            if (GP_ratio > log(r_unif_rand())) {                                                 /* :189 */
                memcpy(p->shape, new_shape, sizeof(double) * ns);
                p->log_scale = new_log_scale;
                memcpy(Linv, new_Linv, sizeof(double) * lsz);
                oracle_precision_diag(Linv, NNarray, n, m, precision_diag);
                acc_suf[iter] = 1;
                if (q > 0) status |= interweave_matrices(Linv, NNarray, n, m, Xl, q, scXl, iw_cov, iw_chol);   /* :200-206 */
            }
        }
        if (iter_start >= 0 && iter_start <= 2000 && iter % 25 == 0) {                           /* :209-213 */
            int a = 0;
            for (int k = iter - 24; k <= iter; k++) a += acc_suf[k];
            double mean_acc = a / 25.0;
            if (mean_acc < .05) p->logvar_sufficient -= (.2 + .05 * r_norm_rand());
            if (mean_acc > .15) p->logvar_sufficient += (.2 + .05 * r_norm_rand());
        }
        /* ---- beta_0 :219-224: if(length(X$locs) == 0 | is.null(X$X)) ---- */
        if (q == 0) {
            double b0mean, bvar;
            oracle_beta0_moments(Linv, NNarray, n, m, field, p->log_scale, &b0mean, &bvar);
            p->beta_0 = b0mean + sqrt(bvar) * r_norm_rand();
        }
        /* ---- regression coefficients :226-247 ---- */
        if (reg) {
            for (int k = 0; k < P1; k++) gvec[k] = 0.0;                                          /* :229 crossprod(resid, cbind(1, X$X)) */
            for (int o = 0; o < n_obs; o++) {
                double e = observed_field[o] - field[locs_match[o] - 1] + p->beta_0;
                gvec[0] += e;
                for (int k = 0; k < P; k++) gvec[1 + k] += e * reg->X[(size_t)o + (size_t)n_obs * k];
            }
            for (int j = 0; j < P1; j++) {                                                       /* ... %*% X$solve_1XT1X */
                double v = 0.0;
                for (int k = 0; k < P1; k++) v += gvec[k] * reg->solve_1XT1X[k + (size_t)P1 * j];
                bmean[j] = v;
            }
            for (int k = 0; k < P1; k++) zz[k] = r_norm_rand();                                  /* :231 */
            double sd_noise = exp(.5 * p->log_noise_variance);
            for (int j = 0; j < P1; j++) {                                                       /* t(X$chol_solve_1XT1X) %*% z */
                double v = 0.0;
                for (int k = 0; k < P1; k++) v += reg->chol_solve_1XT1X[k + (size_t)P1 * j] * zz[k];
                innov[j] = bmean[j] + sd_noise * v;
            }
            for (int s = 0; s < n; s++) field[s] = field[s] - p->beta_0 + innov[0];              /* :232 */
            p->beta_0 = innov[0];                                                                /* :233 */
            for (int k = 0; k < P; k++) reg->beta[k] = innov[1 + k];                             /* :234 */
            if (q > 0) {                                                                         /* :237-246 interweaving */
                for (int s = 0; s < n; s++) {                                                    /* :240 other_field */
                    double xb = 0.0;
                    for (int l = 1; l < q; l++) xb += Xl[(size_t)l * n + s] * reg->beta[reg->xlocs[l - 1] - 1];
                    other[s] = field[s] + xb;
                }
                oracle_linv_mult(Linv, other, NNarray, n, m, tmp);                               /* sparse_chol %*% other_field */
                for (int j = 0; j < q; j++) {
                    double v = 0.0;
                    for (int s = 0; s < n; s++) v += tmp[s] * scXl[(size_t)j * n + s];
                    gvec[j] = v;
                }
                for (int j = 0; j < q; j++) {                                                    /* :241 */
                    double v = 0.0;
                    for (int k = 0; k < q; k++) v += iw_cov[j + (size_t)q * k] * gvec[k];
                    bmean[j] = v;
                }
                for (int k = 0; k < q; k++) zz[k] = r_norm_rand();                               /* :242 */
                double sd_scale = exp(.5 * p->log_scale);
                for (int j = 0; j < q; j++) {
                    double v = 0.0;
                    for (int k = 0; k < q; k++) v += iw_chol[j + (size_t)q * k] * zz[k];
                    innov[j] = bmean[j] + sd_scale * v;
                }
                p->beta_0 = innov[0];                                                            /* :243 */
                for (int l = 1; l < q; l++) reg->beta[reg->xlocs[l - 1] - 1] = innov[l];         /* :244 */
                for (int s = 0; s < n; s++) {                                                    /* :245 */
                    double xb = 0.0;
                    for (int l = 1; l < q; l++) xb += Xl[(size_t)l * n + s] * reg->beta[reg->xlocs[l - 1] - 1];
                    field[s] = other[s] - xb;
                }
            }
            ORACLE_SET_MU()                                                                      /* :249 */
        } else {
            for (int o = 0; o < n_obs; o++) mu[o] = p->beta_0;                                    /* :250 */
        }
        /* ---- chromatic sweeps :257-275 ---- */
        for (int ic = 0; ic < n_chromatic; ic++) {
            oracle_residuals_sum(locs_match, n_obs, n, observed_field, mu, residuals_sum);       /* :260 */
            if (philox) philox_fill(order, n, sweep_counter++, key[0], key[1], z);
            else for (int q = 0; q < n; q++) z[q] = r_norm_rand(); /* rnorm(length(sel)) colour by colour = one stream */
            if (sweep_form == 0) {
                sweep_reference(Linv, NNarray, n, m, &csc, coloring, n_colors, precision_diag, obs_per_loc,
                                residuals_sum, p->beta_0, p->log_scale, p->log_noise_variance, z, field, tmp, tmp2);
            } else {
                for (int s = 0; s < n; s++) tmp[s] = field[s] - p->beta_0;
                oracle_linv_mult(Linv, tmp, NNarray, n, m, tmp2);
                sweep_residual(Linv, n, &csc, coloring, n_colors, order, cptr, precision_diag, obs_per_loc,
                               residuals_sum, p->beta_0, p->log_scale, p->log_noise_variance, z, field, tmp2);
            }
        }
        /* ---- noise variance :281-293 ---- */
        double ssr = oracle_ssr(locs_match, n_obs, observed_field, field, mu, p->beta_0);
        for (int k = 0; k < 10; k++) {
            double inn = 0.0 + .01 * r_norm_rand();
            if (exp(p->log_noise_variance + inn) < var_y) {
                if (-.5 * n_obs * inn - .5 * ssr * (exp(-p->log_noise_variance - inn) - exp(-p->log_noise_variance)) >
                    log(r_unif_rand()))
                    p->log_noise_variance += inn;
            }
        }
        /* ---- records :305-311 ---- */
        if (records) {
            records[(size_t)(iter - 1)] = p->beta_0;
            records[(size_t)(iter - 1) + (size_t)n_iter] = p->log_scale;
            records[(size_t)(iter - 1) + (size_t)n_iter * 2] = p->log_noise_variance;
            for (int k = 0; k < ns; k++) records[(size_t)(iter - 1) + (size_t)n_iter * (3 + k)] = p->shape[k];
        }
        if (reg && reg->beta_records)                                                            /* :305 */
            for (int k = 0; k < P; k++) reg->beta_records[(size_t)(iter - 1) + (size_t)n_iter * k] = reg->beta[k];
        if (field_records) {
            double t = iter * field_thinning;
            if (nearbyint(t) == t) {
                int row = (int)t - 1;
                if (row >= 0 && row < n_field_rec)
                    for (int s = 0; s < n; s++) field_records[(size_t)row + (size_t)n_field_rec * s] = field[s];
            }
        }
        if (accept_records) { accept_records[iter - 1] = acc_anc[iter]; accept_records[n_iter + iter - 1] = acc_suf[iter]; }
    }
    free(Linv); free(new_Linv); free(precision_diag); free(tmp); free(tmp2); free(new_field); free(mu);
    free(residuals_sum); free(z); free(acc_suf); free(acc_anc); free(order); free(cptr);
    free(Xl); free(scXl); free(iw_cov); free(iw_chol); free(other); free(gvec); free(bmean); free(zz); free(innov);
    csc_free(&csc);
#undef ORACLE_SET_MU
    return status;
}
