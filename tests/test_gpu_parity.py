"""GPU parity tests: every call goes through the C ABI (libnngp_b200.so via ctypes) and is compared with the CPU oracle on
the same seeded inputs.  Tolerances (FP64): deterministic kernels <= 1e-10 relative (BASELINE.json north_star)."""
import numpy as np
import pytest

import nngp_b200 as nb
from oracle import oracle as O
from problems import make_problem, make_regression_problem

pytestmark = pytest.mark.gpu

TOL = 1e-10


def rel_rows(a, b):
    """max over rows of ||a_i - b_i|| / ||b_i||  (SURVEY.md 7.3: tolerance stated on the factor row)"""
    num = np.linalg.norm(a - b, axis=1)
    den = np.linalg.norm(b, axis=1)
    return float(np.max(num / den))


def rel_vec(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


CASES = [
    ("exponential_isotropic", 2, 10, [1.0, 0.07, 0.0]),
    ("exponential_isotropic", 2, 5, [1.0, 0.05, 0.0]),
    ("exponential_isotropic", 3, 10, [1.0, 0.3, 0.0]),
    ("exponential_isotropic", 2, 7, [1.0, 0.1, 0.0]),       # generic (non-specialised) M
    ("exponential_isotropic", 2, 20, [1.0, 0.1, 0.0]),
    ("exponential_scaledim", 2, 10, [1.0, 0.05, 0.11, 0.0]),
    ("exponential_spacetime", 3, 10, [1.0, 0.2, 0.5, 0.0]),
    ("matern_isotropic", 2, 10, [1.0, 0.07, 0.75, 0.0]),
    ("matern_isotropic", 2, 20, [1.0, 0.1, 0.6, 0.0]),
    ("matern_scaledim", 2, 5, [1.0, 0.05, 0.11, 0.9, 0.0]),
    ("matern_spacetime", 3, 5, [1.0, 0.2, 0.5, 0.55, 0.0]),
    # generic<16> (M = 9..16), generic<24> (M = 17..24, and m = 20 at d = 3), generic<32> (M = 25..32); the row kernels at MT = 0
    ("exponential_isotropic", 2, 8, [1.0, 0.1, 0.0]),
    ("matern_isotropic", 3, 12, [1.0, 0.25, 0.8, 0.0]),
    ("exponential_spacetime", 3, 15, [1.0, 0.2, 0.4, 0.0]),
    ("matern_isotropic", 2, 16, [1.0, 0.02, 1.2, 0.0]),     # range 0.05: conditioning alone puts precision_diag at 1.4e-10
    ("exponential_isotropic", 3, 20, [1.0, 0.3, 0.0]),
    ("matern_scaledim", 2, 21, [1.0, 0.05, 0.08, 0.6, 0.0]),
    ("exponential_isotropic", 2, 24, [1.0, 0.1, 0.0]),
    ("matern_isotropic", 3, 24, [1.0, 0.25, 0.9, 0.0]),
    ("exponential_scaledim", 3, 31, [1.0, 0.2, 0.3, 0.25, 0.0]),
    ("matern_isotropic", 2, 31, [1.0, 0.05, 0.7, 0.0]),
    # d = 1 and d = 4 (transformed dimensions 1 and 4: generic kernels only)
    ("exponential_isotropic", 1, 10, [1.0, 0.001, 0.0]),
    ("matern_isotropic", 1, 5, [1.0, 0.001, 0.4, 0.0]),
    ("exponential_isotropic", 4, 10, [1.0, 0.4, 0.0]),
    ("exponential_scaledim", 4, 10, [1.0, 0.3, 0.4, 0.5, 0.6, 0.0]),
    ("matern_spacetime", 4, 10, [1.0, 0.4, 0.5, 0.85, 0.0]),
    ("matern_scaledim", 4, 20, [1.0, 0.5, 0.4, 0.6, 0.3, 0.45, 0.0]),
    # a nugget (diagonal s2 (1 + tau)) and variances other than 1 (the Matern table carries the variance in its coefficients)
    ("matern_isotropic", 2, 10, [1.0, 0.07, 0.75, 0.3]),
    ("exponential_isotropic", 2, 10, [0.4, 0.07, 0.2]),
    ("matern_isotropic", 2, 20, [2.5, 0.1, 0.6, 0.0]),
    ("matern_isotropic", 3, 5, [3.7, 0.3, 1.45, 0.1]),
]


@pytest.mark.parametrize("covfun,d,m,cp", CASES)
@pytest.mark.parametrize("layout", [nb.LAYOUT_COLOR, nb.LAYOUT_COLOR_MORTON, nb.LAYOUT_MORTON])
def test_factor_and_products(covfun, d, m, cp, layout):
    P = make_problem(4000, m, d=d, seed=11)
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], covfun, layout=layout) as ctx:
        assert ctx.factor_build(cp) == 0
        Lg = ctx.factor_get()
        Lo = O.vecchia_Linv(cp, covfun, P["locs"], P["NNarray"])
        assert rel_rows(Lg, Lo) < TOL
        assert np.all(Lg[P["NNarray"] == nb.NA_INT] == 0.0)
        # precision_diag
        assert rel_vec(ctx.precision_diag(), O.precision_diag(Lo, P["NNarray"])) < TOL
        # log-likelihood, both entry points
        z = P["field"] - 0.3
        ll_o = O.ll_compressed_sparse_chol(Lo, z, P["NNarray"], 0.4)
        ctx.field_set(P["field"])
        assert abs(ctx.loglik(0.3, 0.4) - ll_o) < TOL * abs(ll_o)
        assert abs(ctx.loglik_host(z, 0.4) - ll_o) < TOL * abs(ll_o)
        # products and the triangular solve
        v = P["rng"].standard_normal(P["n"])
        assert rel_vec(ctx.spmv(v), O.Linv_mult(Lo, v, P["NNarray"])) < TOL
        assert rel_vec(ctx.sptmv(v), O.sparse_chol_tmult(Lo, P["NNarray"], v)) < TOL
        assert rel_vec(ctx.sptrsv(v), O.sparse_chol_solve(Lo, P["NNarray"], v)) < 1e-9   # conditioning of the solve


def test_sphere_factor():
    """*_sphere: transformed dimension 3 -- reg<6,3>, reg<11,3>, and at m = 20 generic<24> (thread per row) or warp<21,3>"""
    rng = np.random.default_rng(3)
    n = 3000
    lonlat = np.column_stack([rng.uniform(-120, -70, n), rng.uniform(25, 50, n)])
    for m in (5, 10, 20):
        P = make_problem(n, m, locs=lonlat, seed=3)
        for covfun, cp in (("exponential_sphere", [1.0, 0.05, 0.0]), ("matern_sphere", [1.0, 0.05, 0.8, 0.0])):
            Lo = O.vecchia_Linv(cp, covfun, lonlat, P["NNarray"])
            with nb.NNGPContext(lonlat, P["NNarray"], P["coloring"], P["locs_match"], covfun) as ctx:
                for fv in ((0, 1) if m == 20 else (0,)):
                    ctx.set_option("factor_variant", fv)
                    assert ctx.factor_build(cp) == 0, (m, covfun, fv)
                    assert rel_rows(ctx.factor_get(), Lo) < 1e-9, (m, covfun, fv)


@pytest.mark.parametrize("n", [4001, 20000])
@pytest.mark.parametrize("covfun,d,cp", [("exponential_isotropic", 2, [1.0, 0.1, 0.0]), ("exponential_spacetime", 3, [1.0, 0.2, 0.4, 0.0]),
                                         ("matern_isotropic", 2, [1.0, 0.1, 0.6, 0.0]), ("matern_isotropic", 3, [1.3, 0.25, 1.1, 0.2])])
def test_warp_per_row_factor_build(n, covfun, d, cp):
    """factor_variant = 1 (vecchia_factor_warp_kernel<21, dt>, m = 20) against the oracle: the first m (partial) rows go through
    factor_row_generic on lane 0; n = 4001 ends in a ragged 32-row round and n = 20000 makes the grid-stride loop run more than one
    round per block (the grid is min(ceil(n / 32), 2 n_SM) blocks); both slots; the triangular solve reads the level-ordered copy of
    the factor that this kernel writes itself; a negative variance fails every pivot."""
    m = 20
    P = make_problem(n, m, d=d, seed=n + d)
    cp2 = [cp[0] * 0.8, cp[1] * 1.3] + cp[2:]
    Lo = O.vecchia_Linv(cp, covfun, P["locs"], P["NNarray"])
    Lo2 = O.vecchia_Linv(cp2, covfun, P["locs"], P["NNarray"])
    v = P["rng"].standard_normal(n)
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], covfun) as ctx:
        ctx.set_option("factor_variant", 1)
        assert ctx.factor_build(cp) == 0
        assert ctx.factor_build(cp2, slot=nb.SLOT_PROPOSAL) == 0
        Lg, Lg2 = ctx.factor_get(), ctx.factor_get(nb.SLOT_PROPOSAL)
        assert rel_rows(Lg, Lo) < TOL and rel_rows(Lg2, Lo2) < TOL
        assert rel_rows(Lg[:m], Lo[:m]) < TOL and np.all(Lg[P["NNarray"] == nb.NA_INT] == 0.0)
        assert rel_vec(ctx.sptrsv(v), O.sparse_chol_solve(Lo, P["NNarray"], v)) < 1e-9
        assert rel_vec(ctx.sptrsv(v, slot=nb.SLOT_PROPOSAL), O.sparse_chol_solve(Lo2, P["NNarray"], v)) < 1e-9
        ctx.field_set(P["field"])
        ll_o = O.ll_compressed_sparse_chol(Lo, P["field"] - 0.3, P["NNarray"], 0.4)
        assert abs(ctx.loglik(0.3, 0.4) - ll_o) < TOL * abs(ll_o)
        assert ctx.factor_build([-cp[0]] + cp[1:]) == n


@pytest.mark.parametrize("n,m", [(1, 3), (5, 10), (12, 10), (40, 1), (1000, 10)])
def test_small_and_ragged(n, m):
    """n <= m: every row is partial (NA-padded)."""
    P = make_problem(n, m, seed=n)
    cp = [1.0, 0.2, 0.0]
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        assert ctx.factor_build(cp) == 0
        Lo = O.vecchia_Linv(cp, "exponential_isotropic", P["locs"], P["NNarray"])
        assert rel_rows(ctx.factor_get(), Lo) < TOL
        v = P["rng"].standard_normal(n)
        assert rel_vec(ctx.sptrsv(v), O.sparse_chol_solve(Lo, P["NNarray"], v)) < 1e-9
        ctx.field_set(P["field"])
        ll_o = O.ll_compressed_sparse_chol(Lo, P["field"] - 0.1, P["NNarray"], -0.2)
        assert abs(ctx.loglik(0.1, -0.2) - ll_o) < TOL * max(1.0, abs(ll_o))


def test_not_positive_definite_is_flagged_not_fatal():
    """A block that fails the Cholesky pivot test (pivot <= 0 or NaN, LAPACK's criterion) is counted, not fatal: the caller
    rejects the proposal (SURVEY.md 8b error convention).  Every kernel family: reg<6,2>, generic<16>, reg<21,2,MINB=1>, warp<21,2>,
    generic<32>, and d = 4."""
    for m, d, fv in ((5, 2, 0), (12, 2, 0), (20, 2, 0), (20, 2, 1), (31, 2, 0), (10, 4, 0)):
        case = dict(m=m, d=d, factor_variant=fv)
        P = make_problem(500, m, d=d, seed=5)
        with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
            ctx.set_option("factor_variant", fv)
            assert ctx.factor_build([-1.0, 0.2, 0.0]) == 500, case          # negative variance: every pivot fails
            assert ctx.factor_build([1.0, 0.2, 0.0]) == 0, case             # and the context is still usable
            _, bad = O.vecchia_Linv([-1.0, 0.2, 0.0], "exponential_isotropic", P["locs"], P["NNarray"], return_bad=True)
            assert bad == 500
        locs = P["locs"].copy()
        twin = P["NNarray"][300, 1]
        locs[300] = locs[twin - 1]                          # exact duplicate of a neighbour: pivot is 0 up to rounding
        # every row whose block holds both copies is singular: each is flagged or a huge-but-finite row, never a crash
        # (m = 5: 2 such rows); every other row is the oracle's
        singular = np.any(P["NNarray"] == 301, axis=1) & np.any(P["NNarray"] == twin, axis=1)
        with nb.NNGPContext(locs, P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
            ctx.set_option("factor_variant", fv)
            assert 0 <= ctx.factor_build([1.0, 0.2, 0.0]) <= int(singular.sum()), case
            Lo = O.vecchia_Linv([1.0, 0.2, 0.0], "exponential_isotropic", locs, P["NNarray"])
            assert rel_rows(ctx.factor_get()[~singular], Lo[~singular]) < TOL, case


@pytest.mark.parametrize("layout", [nb.LAYOUT_COLOR, nb.LAYOUT_COLOR_MORTON, nb.LAYOUT_MORTON])
@pytest.mark.parametrize("m,n_extra,drop", [(10, 0, 0.0), (5, 300, 0.0), (10, 200, 0.3), (31, 100, 0.0), (12, 0, 0.2)])
def test_chromatic_sweep_supplied_normals(layout, m, n_extra, drop):
    """Same normals in the reference's hand-out order => same field as update_Gaussian.R:257-275 written literally; generic neighbour
    counts included (m = 31 at d = 2, m = 12 at d = 4)."""
    d = 4 if m == 12 else 2
    P = make_problem(3000, m, d=d, seed=21, n_extra_obs=n_extra, drop_obs_frac=drop)
    cp = [1.0, 0.08 if d == 2 else 0.3, 0.0]
    beta_0, ls, lnv = 0.3, 0.2, -1.1
    Lo = O.vecchia_Linv(cp, "exponential_isotropic", P["locs"], P["NNarray"])
    pd = O.precision_diag(Lo, P["NNarray"])
    mu = np.full(P["n_obs"], beta_0)
    n_sweeps = 3
    z = P["rng"].standard_normal(n_sweeps * P["n"])
    f = P["field"].copy()
    for s in range(n_sweeps):
        rs = O.residuals_sum(P["locs_match"], P["n"], P["y"], mu)
        f = O.chromatic_sweep(Lo, P["NNarray"], P["coloring"], pd, P["obs_per_loc"], rs, beta_0, ls, lnv,
                              z[s * P["n"]:(s + 1) * P["n"]], f, form="reference")
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], layout=layout) as ctx:
        ctx.factor_build(cp)
        ctx.factor_commit()
        ctx.field_set(P["field"])
        ctx.obs_set(P["y"])
        ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=n_sweeps, z=z)
        assert rel_vec(ctx.field_get(), f) < TOL
        assert abs(ctx.ssr() - O.ssr(P["locs_match"], P["y"], f, mu, beta_0)) < TOL * P["n_obs"]


def test_philox_sweep_is_stationary_for_the_exact_conditional():
    """SURVEY.md 8c(7): many Philox sweeps on a tiny model reproduce the posterior mean and covariance
    (Q/s2 + D/t2)^-1 -- a distributional check of the on-device generator and of the sweep."""
    n, m = 30, 4
    P = make_problem(n, m, seed=2)
    cp = [1.0, 0.5, 0.0]
    beta_0, ls, lnv = 0.0, 0.1, -0.5
    Lo = O.vecchia_Linv(cp, "exponential_isotropic", P["locs"], P["NNarray"])
    A = np.zeros((n, n))
    for i in range(n):
        for j in range(m + 1):
            if P["NNarray"][i, j] != nb.NA_INT:
                A[i, P["NNarray"][i, j] - 1] = Lo[i, j]
    prec = A.T @ A * np.exp(-ls) + np.diag(P["obs_per_loc"]) * np.exp(-lnv)
    cov = np.linalg.inv(prec)
    mean = cov @ (np.exp(-lnv) * np.bincount(P["locs_match"] - 1, weights=P["y"], minlength=n))
    n_samp = 20000
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        ctx.factor_build(cp)
        ctx.factor_commit()
        ctx.field_set(np.zeros(n))
        ctx.obs_set(P["y"])
        ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=200, seed=7)
        S = np.empty((n_samp, n))
        for k in range(n_samp):
            ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=1, seed=7)
            S[k] = ctx.field_get()
    sd = np.sqrt(np.diag(cov))
    assert np.max(np.abs(S.mean(0) - mean) / sd) < 0.08
    emp = np.cov(S.T)
    assert np.max(np.abs(emp - cov)) / np.max(np.abs(cov)) < 0.08


def test_ancillary_beta0_and_field_init():
    P = make_problem(3000, 10, seed=31, n_extra_obs=100)
    cp_cur, cp_new = [1.0, 0.08, 0.0], [1.0, 0.09, 0.0]
    beta_0, ls, dls, lnv = 0.3, 0.2, 0.05, -1.0
    Lc = O.vecchia_Linv(cp_cur, "exponential_isotropic", P["locs"], P["NNarray"])
    Ln = O.vecchia_Linv(cp_new, "exponential_isotropic", P["locs"], P["NNarray"])
    mu = np.full(P["n_obs"], beta_0)
    new_field = beta_0 + np.exp(0.5 * dls) * O.sparse_chol_solve(Ln, P["NNarray"], O.Linv_mult(Lc, P["field"] - beta_0, P["NNarray"]))
    ratio_o = (O.obs_loglik(P["locs_match"], P["y"], new_field, mu, beta_0, lnv)
               - O.obs_loglik(P["locs_match"], P["y"], P["field"], mu, beta_0, lnv))
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        ctx.factor_build(cp_cur, nb.SLOT_CURRENT)
        ctx.factor_build(cp_new, nb.SLOT_PROPOSAL)
        ctx.field_set(P["field"])
        ctx.obs_set(P["y"])
        ratio = ctx.ancillary_propose(beta_0, dls, lnv)
        assert abs(ratio - ratio_o) < 1e-9 * max(1.0, abs(ratio_o))
        bm, bv = ctx.beta0_moments(ls)
        bm_o, bv_o = O.beta0_moments(Lc, P["NNarray"], P["field"], ls)
        assert abs(bm - bm_o) < TOL * max(1, abs(bm_o)) and abs(bv - bv_o) < TOL * bv_o
        ctx.ancillary_accept()
        assert rel_vec(ctx.field_get(), new_field) < 1e-9
        assert rel_rows(ctx.factor_get(nb.SLOT_CURRENT), Ln) < TOL          # proposal became current
        assert rel_vec(ctx.precision_diag(), O.precision_diag(Ln, P["NNarray"])) < TOL
        z = P["rng"].standard_normal(P["n"])
        ctx.field_init(0.7, 0.3, z)
        want = 0.7 + np.sqrt(np.exp(0.3)) * O.sparse_chol_solve(Ln, P["NNarray"], z)
        assert rel_vec(ctx.field_get(), want) < 1e-9


def test_predict_sample():
    """predict.R:43-53 on the device: exponential and Matern with nu <= 1/2 (reachable through predict.R:37's 1.5 plogis) and near
    3/2 at a generic neighbour count, every storage layout, new sites after the observed ones, every site new, and none new"""
    n, n_pred = 1500, 700
    rng = np.random.default_rng(8)
    locs = rng.random((n + n_pred, 2))
    field = 0.3 + rng.standard_normal(n + n_pred)
    z = rng.standard_normal(n + n_pred)
    for covfun, m, cp in (("exponential_isotropic", 10, [1.0, 0.2, 0.0]), ("matern_isotropic", 10, [1.0, 0.1, 0.3, 0.0]),
                          ("matern_isotropic", 15, [1.0, 0.1, 1.45, 0.0])):
        nn = nb.find_ordered_nn(locs, m)
        Lo = O.vecchia_Linv(cp, covfun, locs, nn)
        for layout in (nb.LAYOUT_COLOR, nb.LAYOUT_COLOR_MORTON, nb.LAYOUT_MORTON):
            with nb.NNGPContext(locs, nn, np.zeros(n + n_pred, dtype=np.int32), np.zeros(0, dtype=np.int32), covfun, layout=layout) as ctx:   # all-zero colouring = no sweeps
                assert ctx.factor_build(cp) == 0
                for n0 in (n, 0, n + n_pred):
                    case = dict(covfun=covfun, m=m, layout=layout, n_obs_sites=n0)
                    got = ctx.predict_sample(n0, field[:n0], 0.3, 0.5, z[:n + n_pred - n0])
                    want = O.predict_field_sample(Lo, nn, n0, field[:n0], 0.3, 0.5, z[:n + n_pred - n0])
                    assert got.shape == (n + n_pred - n0,), case
                    if n0 < n + n_pred:
                        assert rel_vec(got, want) < 1e-9, case
                with pytest.raises(nb.NNGPError) as e:                  # a context without a colouring refuses to sweep
                    ctx.gibbs_sweep(0.0, 0.0, 0.0, n_sweeps=1, seed=1)
                assert e.value.status == 4


@pytest.mark.parametrize("covfun,shape", [("exponential_isotropic", [np.log(0.1)]), ("matern_isotropic", [np.log(0.1), 0.3])])
def test_chain_run_matches_oracle_chain_with_r_stream(covfun, shape):
    """nngp_chain_run in NNGP_RNG_SUPPLIED mode consumes R's stream (set.seed(iter_start + i)) exactly like
    update_Gaussian.R:34-315; the oracle chain does the same on the CPU."""
    n, m = 1200, 5
    P = make_problem(n, m, seed=41)
    cp = [1.0, 0.1, 0.0] if covfun.startswith("exp") else [1.0, 0.1, 0.7, 0.0]
    L0 = O.vecchia_Linv(cp, covfun, P["locs"], P["NNarray"])
    w = O.sparse_chol_solve(L0, P["NNarray"], P["rng"].standard_normal(n))
    y = 1.0 + w + np.sqrt(0.1) * P["rng"].standard_normal(n)
    lm = np.arange(1, n + 1, dtype=np.int32)
    p0 = dict(shape=shape, beta_0=0.9, log_scale=0.1, log_noise_variance=np.log(0.2))
    n_iter = 50
    po, fo, reco, freco, acco = O.update_gaussian_chain(P["locs"], P["NNarray"], P["coloring"], lm, np.ones(n), y, covfun,
                                                        p0, 0.9 + w, n_iter, 0.5, 2, 0, 1, 0)
    var_y = np.var(y, ddof=1)
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], lm, covfun) as ctx:
        ctx.field_set(0.9 + w)
        ctx.obs_set(y)
        pg, recg, frecg, accg = ctx.chain_run(p0, n_iter, var_y, thin=0.5, n_chromatic=2, iter_start=0, chain_index=1,
                                              rng_mode=nb.RNG_SUPPLIED)
        fg = ctx.field_get()
    assert np.array_equal(accg, acco)                         # same accept/reject decisions
    assert np.max(np.abs(recg - reco)) < 1e-8
    assert np.max(np.abs(fg - fo)) < 1e-7
    assert np.max(np.abs(frecg - freco)) < 1e-7
    assert abs(pg["logvar_ancillary"] - po["logvar_ancillary"]) < 1e-12


REGRESSOR_CHAIN_CASES = [   # n sites, p_locs, p_obs, extra observations, covfun, shape, X$locs (None: 1..p_locs)
    (1500, 2, 1, 300, "exponential_isotropic", [np.log(0.1)], None),
    (1500, 0, 3, 0, "exponential_isotropic", [np.log(0.1)], None),
    (1500, 3, 0, 100, "matern_isotropic", [np.log(0.1), 0.3], None),
    (1500, 20, 4, 50, "exponential_isotropic", [np.log(0.1)], None),
    # around op_atb's row chunks (kAtbRowsPerChunk = 4096 rows, nngp_b200.cu): one full chunk of observations with p + 1 = 17 (one
    # column past a 16-wide tile); 4097 observations and 4097 sites with q = 17, so both products get a second chunk of one row;
    # 13 000 observations over 10 000 sites with 80 columns (4 and 3 chunks, 6 x 2 tiles of the interweaving product)
    (4000, 4, 12, 96, "exponential_isotropic", [np.log(0.1)], None),
    (4097, 16, 2, 0, "matern_isotropic", [np.log(0.1), 0.3], None),
    (10000, 20, 60, 3000, "exponential_isotropic", [np.log(0.1)], None),
    (10000, 20, 60, 3000, "matern_isotropic", [np.log(0.05), -0.5], None),
    # X$locs not a prefix of X's columns: the interweaving step reads and writes beta through the X$locs map
    (1500, 2, 2, 100, "exponential_isotropic", [np.log(0.1)], [3, 1]),
]


def _regressor_case_id(i, case):
    """pytest's id of (p_locs, p_obs, extra, covfun, shape), with n and X$locs appended where they are not 1500 and a prefix"""
    n, p_locs, p_obs, extra, covfun, _, xlocs = case
    s = f"{p_locs}-{p_obs}-{extra}-{covfun}-shape{i}"
    return s + (f"-n{n}" if n != 1500 else "") + (f"-xlocs{'_'.join(map(str, xlocs))}" if xlocs else "")


@pytest.mark.parametrize("n,p_locs,p_obs,extra,covfun,shape,xlocs", REGRESSOR_CHAIN_CASES,
                         ids=[_regressor_case_id(i, c) for i, c in enumerate(REGRESSOR_CHAIN_CASES)])
def test_chain_run_regressors_matches_oracle_chain_with_r_stream(n, p_locs, p_obs, extra, covfun, shape, xlocs):
    """nngp_chain_run_regressors (update_Gaussian.R:101-314 with the regression block :226-250 on the device: X resident in
    HBM, crossprod()s as streaming A^T B kernels, interweaving matrices refreshed on every accept) against the oracle chain
    (itself checked against the dense transcription of the R loop, tests/test_oracle_golden.py), both driven by R's stream."""
    from problems import assert_regression_chain_matches
    m, n_iter = 5, 50
    P = make_regression_problem(n, m, seed=23, n_extra_obs=extra, p_locs=p_locs, p_obs=p_obs, xlocs=xlocs)
    K, chunks = 4096, lambda rows: -(-rows // 4096)    # kAtbRowsPerChunk (nngp_b200.cu): op_atb sums partials over chunks of K rows
    if n == 4000:      # exactly one full chunk of observations, p + 1 = 17
        assert P["n_obs"] == K and P["X"].shape[1] + 1 == 17
    elif n == 4097:    # a second chunk of one row for the observations and for the sites, q = 17
        assert P["n_obs"] == K + 1 and n == K + 1 and p_locs + 1 == 17
    elif n == 10000:   # 4 chunks of observations, 3 of sites
        assert chunks(P["n_obs"]) == 4 and chunks(n) == 3
    p0 =dict(shape=shape, beta_0=0.5, log_scale=-0.2, log_noise_variance=np.log(0.15), logvar_sufficient=-2.0, logvar_ancillary=-2.0)
    beta0 = 0.1 * np.ones(P["X"].shape[1])
    field0 = 0.5 + P["w"]
    reg = dict(X=P["X"], xlocs=P["xlocs"], first_obs=P["first_obs"], solve_1XT1X=P["solve_1XT1X"],
               chol_solve_1XT1X=P["chol_solve_1XT1X"], beta=beta0)
    ora = O.update_gaussian_chain(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], P["obs_per_loc"],
                                  P["y"], covfun, p0, field0, n_iter, 0.5, 2, 0, 3, 1, regressors=reg)
    var_y = float(np.var(P["y"], ddof=1))
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], covfun) as ctx:
        ctx.regressors_set(P["X"], P["y"], xlocs=P["xlocs"], first_obs=P["first_obs"])
        ctx.field_set(field0)
        dev = ctx.chain_run_regressors(p0, beta0, P["solve_1XT1X"], P["chol_solve_1XT1X"], n_iter, var_y, thin=0.5,
                                       n_chromatic=2, iter_start=0, chain_index=3, rng_mode=nb.RNG_SUPPLIED)
        dev = dev + (ctx.field_get(), ctx.ssr())               # the context's y - X beta corresponds to the final beta
    assert_regression_chain_matches(dev, ora, P["X"], P["y"], P["locs_match"], f"n={n} p_locs={p_locs} p_obs={p_obs} {covfun}")


def test_regressor_error_paths():
    from problems import make_regression_problem
    P = make_regression_problem(300, 5, seed=2, p_locs=1, p_obs=1)
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        ctx.field_set(P["field"])
        with pytest.raises(nb.NNGPError) as e:                  # no regressors on the device yet
            ctx._reg_p = 2
            ctx.chain_run_regressors(dict(shape=[0.0], beta_0=0.0, log_scale=0.0, log_noise_variance=0.0), np.zeros(2), P["solve_1XT1X"],
                                     P["chol_solve_1XT1X"], 1, 1.0)
        assert e.value.status == 4
        with pytest.raises(nb.NNGPError) as e:                  # X$locs names a column that does not exist
            ctx.regressors_set(P["X"], P["y"], xlocs=[3], first_obs=P["first_obs"])
        assert e.value.status == 1
        # collinear location-level regressors: the interweaving precision is singular -> an error, not garbage
        Xc = np.column_stack([P["X"][:, 0], P["X"][:, 0]])
        ctx.regressors_set(Xc, P["y"], xlocs=[1, 2], first_obs=P["first_obs"])
        with pytest.raises(nb.NNGPError):
            ctx.chain_run_regressors(dict(shape=[np.log(0.1)], beta_0=0.0, log_scale=0.0, log_noise_variance=0.0), np.zeros(2), np.eye(3),
                                     np.eye(3), 1, 1.0)


def test_error_paths():
    P = make_problem(200, 5, seed=1)
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        with pytest.raises(nb.NNGPError) as e:
            ctx.loglik(0.0, 0.0)                                # no factor yet
        assert e.value.status == 4
        with pytest.raises(nb.NNGPError) as e:
            ctx.factor_build([1.0, 0.1, 0.2, 0.0])              # wrong covparms length
        assert e.value.status == 1
    bad = P["NNarray"].copy()
    bad[10, 1] = 50                                              # a "neighbour" that is not a previous site
    with pytest.raises(nb.NNGPError):
        nb.NNGPContext(P["locs"], bad, P["coloring"], P["locs_match"])
    improper = P["coloring"].copy()
    improper[P["NNarray"][150, 1] - 1] = improper[150]           # a site and one of its parents share a colour: racy sweep
    with pytest.raises(nb.NNGPError) as e:
        nb.NNGPContext(P["locs"], P["NNarray"], improper, P["locs_match"])
    assert "not proper" in str(e.value)


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("n,m", [(20000, 10), (3000, 5)])
def test_every_sweep_variant_matches_the_reference_loop(variant, n, m):
    """All kernel variants of the sweep (PDL chain of tiles with and without the 6-CTAs/SM build, dependents triggered after the wait,
    plain tiled launches, thread-per-site) are the same map given the same normals; multi-sweep launches included (n = 20000 gives
    several CTAs per colour); the captured graph's replay and direct launches give the same field bit for bit."""
    P = make_problem(n, m, seed=77, n_extra_obs=n // 20)
    cp = [1.0, 0.05, 0.0]
    beta_0, ls, lnv = -0.2, 0.3, -0.9
    Lo = O.vecchia_Linv(cp, "exponential_isotropic", P["locs"], P["NNarray"])
    pd = O.precision_diag(Lo, P["NNarray"])
    mu = np.full(P["n_obs"], beta_0)
    n_sweeps = 3
    z = P["rng"].standard_normal(n_sweeps * n)
    f = P["field"].copy()
    rs = O.residuals_sum(P["locs_match"], n, P["y"], mu)
    for s in range(n_sweeps):
        f = O.chromatic_sweep(Lo, P["NNarray"], P["coloring"], pd, P["obs_per_loc"], rs, beta_0, ls, lnv,
                              z[s * n:(s + 1) * n], f, form="residual")
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        ctx.set_option("sweep_variant", variant)
        ctx.factor_build(cp)
        ctx.factor_commit()
        ctx.field_set(P["field"])
        ctx.obs_set(P["y"])
        ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=n_sweeps, z=z)
        fz = ctx.field_get()
        assert rel_vec(fz, f) < TOL
        # Philox draws are keyed by (seed, sweep counter, site): identical across variants
        ctx.field_set(P["field"])
        ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=2, seed=5)
        a = ctx.field_get()
        ctx.set_option("use_graph", 0)
        ctx.field_set(P["field"])
        ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=n_sweeps, z=z)
        assert np.array_equal(ctx.field_get(), fz)
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], layout=nb.LAYOUT_COLOR) as ctx:
        ctx.set_option("sweep_variant", 3)
        ctx.factor_build(cp)
        ctx.factor_commit()
        ctx.field_set(P["field"])
        ctx.obs_set(P["y"])
        ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=n_sweeps, z=z)     # same per-context sweep counter as above
        ctx.field_set(P["field"])
        ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=2, seed=5)
        assert rel_vec(ctx.field_get(), a) < TOL


@pytest.mark.parametrize("solve_variant,level_copy,m", [(0, 1, 10), (0, 0, 10), (1, 1, 10), (0, 1, 7), (0, 1, 20)])
def test_both_solve_variants(solve_variant, level_copy, m):
    """sync-free solve reading the level-ordered copy of the factor (default) or the storage-ordered tables, and the level-scheduled
    launches; both factor slots (the ancillary step solves with the PROPOSAL factor)"""
    P = make_problem(30000, m, seed=13)
    cp, cp2 = [1.0, 0.05, 0.0], [1.0, 0.08, 0.0]
    Lo = O.vecchia_Linv(cp, "exponential_isotropic", P["locs"], P["NNarray"])
    Lo2 = O.vecchia_Linv(cp2, "exponential_isotropic", P["locs"], P["NNarray"])
    v = P["rng"].standard_normal(P["n"])
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        ctx.set_option("solve_variant", solve_variant)
        ctx.set_option("solve_level_copy", level_copy)
        ctx.factor_build(cp)
        ctx.factor_build(cp2, slot=nb.SLOT_PROPOSAL)
        assert rel_vec(ctx.sptrsv(v), O.sparse_chol_solve(Lo, P["NNarray"], v)) < 1e-9
        assert rel_vec(ctx.sptrsv(v, slot=nb.SLOT_PROPOSAL), O.sparse_chol_solve(Lo2, P["NNarray"], v)) < 1e-9
        ctx.factor_accept()                                    # the proposal becomes the current factor: the copies swap with it
        x0 = ctx.sptrsv(v)
        assert rel_vec(x0, O.sparse_chol_solve(Lo2, P["NNarray"], v)) < 1e-9
        assert rel_vec(ctx.sptrsv(v, slot=nb.SLOT_PROPOSAL), O.sparse_chol_solve(Lo, P["NNarray"], v)) < 1e-9
        # the schedule knobs change which CTA takes which rows and when, never the arithmetic of a row (fixed association): the
        # same solution bit for bit -- one CTA walking the whole DAG, 8 CTAs per SM, a back-off between polls, no graph replay
        for opt, val, default in (("solve_window_ctas", 1, 0), ("solve_ctas_per_sm", 8, 1), ("solve_sleep_ns", 200, 0), ("use_graph", 0, 1)):
            ctx.set_option(opt, val)
            assert np.array_equal(ctx.sptrsv(v), x0), (opt, val)
            ctx.set_option(opt, default)


@pytest.mark.parametrize("commit_variant", [0, 1])
def test_both_transposition_variants(commit_variant):
    P = make_problem(20000, 10, seed=14)
    cp = [1.0, 0.05, 0.0]
    Lo = O.vecchia_Linv(cp, "exponential_isotropic", P["locs"], P["NNarray"])
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        ctx.set_option("commit_variant", commit_variant)
        ctx.factor_build(cp)
        ctx.factor_commit()
        assert rel_vec(ctx.precision_diag(), O.precision_diag(Lo, P["NNarray"])) < TOL


@pytest.mark.parametrize("nu,m", [(0.51, 10), (0.75, 10), (0.99, 10), (1.3, 5)])
def test_matern_table_matches_direct_bessel_and_oracle(nu, m):
    """The per-build interpolation table of the Matern kernel agrees with the direct K_nu evaluation and with the oracle
    (std::cyl_bessel_k) on factor rows; distances span coincident-scale to far-field (early sites of the ordering)."""
    P = make_problem(6000, m, seed=19)
    cp = [1.0, 0.03, nu, 0.0]
    Lo = O.vecchia_Linv(cp, "matern_isotropic", P["locs"], P["NNarray"])
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], "matern_isotropic") as ctx:
        assert ctx.factor_build(cp) == 0
        Lt = ctx.factor_get()
        ctx.set_option("matern_table", 0)
        assert ctx.factor_build(cp) == 0
        Ld = ctx.factor_get()
    assert rel_rows(Lt, Lo) < TOL
    assert rel_rows(Ld, Lo) < TOL
    assert rel_rows(Lt, Ld) < TOL      # smoother kernels have worse-conditioned blocks: 1e-15 kernel differences show up at 1e-11


@pytest.mark.parametrize("m", [5, 10, 20])
@pytest.mark.parametrize("variant", [0, 1])
def test_both_loglik_variants(variant, m):
    """plain coalesced loads vs the TMA-staged ring (cp.async.bulk + mbarrier): same partial sums, ragged last tile included"""
    P = make_problem(10007, m, seed=23)
    cp = [1.0, 0.05, 0.0]
    Lo = O.vecchia_Linv(cp, "exponential_isotropic", P["locs"], P["NNarray"])
    ll_o = O.ll_compressed_sparse_chol(Lo, P["field"] - 0.3, P["NNarray"], 0.2)
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        ctx.set_option("loglik_variant", variant)
        ctx.factor_build(cp)
        ctx.field_set(P["field"])
        assert abs(ctx.loglik(0.3, 0.2) - ll_o) < TOL * abs(ll_o)


def test_device_record_store_and_summary():
    """Field records come back in R's layout from the device-side store, and nngp_records_summary reproduces get_summary
    (estimate.R:1-6: mean, type-7 quantiles, sd with n-1) of records$field minus beta_0."""
    n, m = 3000, 5
    P = make_problem(n, m, seed=51)
    lm = np.arange(1, n + 1, dtype=np.int32)
    y = 0.5 + P["rng"].standard_normal(n)
    p0 = dict(shape=[np.log(0.1)], beta_0=0.4, log_scale=0.0, log_noise_variance=-0.5)
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], lm) as ctx:
        ctx.field_set(P["field"])
        ctx.obs_set(y)
        _, rec, frec, _ = ctx.chain_run(p0, 40, float(np.var(y, ddof=1)), thin=0.5, n_chromatic=2, iter_start=0, chain_index=1)
        assert frec.shape == (20, n) and np.all(np.isfinite(frec))
        assert np.max(np.abs(frec[-1] - ctx.field_get())) == 0.0          # iteration 40 is stored in the last row
        b0 = rec[1::2, 0][10:]                                            # beta_0 of iterations 22, 24, ..., 40
        got = ctx.records_summary(11, 10, offsets=b0)
    want = nb.get_summary(frec[10:] - b0[:, None])
    assert np.allclose(got, want, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("with_regressors", [False, True])
def test_concurrent_chains_are_bit_identical_to_sequential_ones(with_regressors):
    """nngp_chains_run[_regressors] (update_Gaussian.R:22-26: chains advance concurrently) -- three chains co-scheduled on one GPU,
    each on its own context / stream / host thread -- must return exactly what three nngp_chain_run calls return one after the
    other: every draw is keyed by (iter_start, chain_index), nothing by timing."""
    n, m, n_iter = 4000, 5, 12
    P = make_regression_problem(n, m, seed=61, n_extra_obs=100) if with_regressors else make_problem(n, m, seed=61, n_extra_obs=100)
    y = P["y"]
    var_y = float(np.var(y, ddof=1))
    p0 = [dict(shape=[np.log(0.08 + 0.02 * k)], beta_0=0.1 * k, log_scale=-0.1 * k, log_noise_variance=-0.5) for k in range(3)]
    rng = np.random.default_rng(3)
    fields = [P["field"] + 0.1 * rng.standard_normal(n) for _ in range(3)]
    betas = [0.1 * rng.standard_normal(P["X"].shape[1]) for _ in range(3)] if with_regressors else None

    def make():
        cs = []
        for k in range(3):
            c = nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"])
            if with_regressors:
                c.regressors_set(P["X"], y, xlocs=P["xlocs"], first_obs=P["first_obs"])
            else:
                c.obs_set(y)
            c.field_set(fields[k])
            cs.append(c)
        return cs

    seq, cs = [], make()
    try:
        for k, c in enumerate(cs):
            if with_regressors:
                seq.append(c.chain_run_regressors(p0[k], betas[k], P["solve_1XT1X"], P["chol_solve_1XT1X"], n_iter, var_y, thin=0.5,
                                                  n_chromatic=3, iter_start=0, chain_index=k + 1) + (c.field_get(),))
            else:
                seq.append(c.chain_run(p0[k], n_iter, var_y, thin=0.5, n_chromatic=3, iter_start=0, chain_index=k + 1) + (c.field_get(),))
    finally:
        for c in cs:
            c.close()
    cs = make()
    try:
        kw = dict(thin=0.5, n_chromatic=3, iter_start=0, chain_indices=[1, 2, 3])
        if with_regressors:
            con = nb.chains_run(cs, p0, n_iter, var_y, betas=betas, solve_1XT1X=P["solve_1XT1X"], chol_solve_1XT1X=P["chol_solve_1XT1X"], **kw)
        else:
            con = nb.chains_run(cs, p0, n_iter, var_y, **kw)
        for k in range(3):
            for a, b in zip(seq[k][1:-1], con[k][1:]):          # records, (beta records,) field records, accepts
                assert np.array_equal(a, b)
            assert np.array_equal(seq[k][-1], cs[k].field_get())
            for key in ("beta_0", "log_scale", "log_noise_variance", "logvar_sufficient", "logvar_ancillary"):
                assert seq[k][0][key] == con[k][0][key]
        # two chains on one context are refused
        with pytest.raises(nb.NNGPError):
            nb.chains_run([cs[0], cs[0]], p0[:2], 2, var_y)
    finally:
        for c in cs:
            c.close()
    if not with_regressors:   # max_concurrent = 1 (n_cores = 1) is the sequential schedule: the same records, from fresh contexts
        cs = make()
        try:
            one = nb.chains_run(cs, p0, n_iter, var_y, max_concurrent=1, **kw)
            for k in range(3):
                assert np.array_equal(one[k][1], con[k][1]) and np.array_equal(one[k][2], con[k][2])
        finally:
            for c in cs:
                c.close()


def test_sweep_loglik_host_equals_the_four_call_sequence():
    """nngp_sweep_loglik_host = nngp_field_set + nngp_gibbs_sweep + nngp_loglik + nngp_field_get in one call (one PCIe pass each way):
    the same field bit for bit and the same log-likelihood, with supplied normals and with Philox, from pageable and pinned buffers"""
    P = make_problem(20000, 10, seed=41)
    z = P["rng"].standard_normal(P["n"])
    b0, ls, lnv = 0.3, 0.1, -1.0
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        ctx.factor_build([1.0, 0.07, 0.0])
        ctx.factor_commit()
        ctx.obs_set(P["y"])
        ctx.field_set(P["field"])
        ctx.gibbs_sweep(b0, ls, lnv, n_sweeps=1, z=z)
        f_ref, ll_ref = ctx.field_get(), ctx.loglik(b0, ls)
        ctx.field_set(P["field"])
        ctx.gibbs_sweep(b0, ls, lnv, n_sweeps=2, seed=5)
        f_ref2, ll_ref2 = ctx.field_get(), ctx.loglik(b0, ls)
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        ctx.factor_build([1.0, 0.07, 0.0])
        ctx.factor_commit()
        ctx.obs_set(P["y"])
        f = P["field"].copy()
        ll = ctx.sweep_loglik_host(f, b0, ls, lnv, n_sweeps=1, z=z)
        assert np.array_equal(f, f_ref) and ll == ll_ref
        pinned = nb.PinnedArray(P["n"])
        pinned.array[:] = P["field"]
        ll2 = ctx.sweep_loglik_host(pinned.array, b0, ls, lnv, n_sweeps=2, seed=5)   # same per-context sweep counter as the reference run
        assert np.array_equal(pinned.array, f_ref2) and ll2 == ll_ref2
        pinned.free()
