"""Parity cases the round-1 review found missing: the GPU against the ORACLE at BASELINE's own sizes (config 3: n = 1M, m = 10;
config 4's shape: m = 20, Matern nu 0.75), the reference's default max-min ordering, and site columns longer than a tile
(e1 - e0 > 1024 entries) in the sweep, the transposition and the sharded ghost apply.  All through the C ABI."""
import numpy as np
import pytest

import nngp_b200 as nb
from oracle import oracle as O
from problems import make_problem, star_problem

pytestmark = pytest.mark.gpu
TOL = 1e-10


def rel_rows(a, b):
    return float(np.max(np.linalg.norm(a - b, axis=1) / np.linalg.norm(b, axis=1)))


def rel_vec(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def oracle_sweep(P, Lo, beta_0, ls, lnv, z, form):
    pd = O.precision_diag(Lo, P["NNarray"])
    rs = O.residuals_sum(P["locs_match"], P["n"], P["y"], np.full(P["n_obs"], beta_0))
    return O.chromatic_sweep(Lo, P["NNarray"], P["coloring"], pd, P["obs_per_loc"], rs, beta_0, ls, lnv, z, P["field"], form=form), pd


@pytest.mark.parametrize("n,m,covfun,cp,order", [
    (1_000_000, 10, "exponential_isotropic", [1.0, 0.05, 0.0], "random"),       # config 3
    (250_000, 20, "matern_isotropic", [1.0, 0.02, 0.75, 0.0], "random"),        # config 4's neighbour count / covariance
    (300_000, 10, "exponential_isotropic", [1.0, 0.05, 0.0], "maxmin"),         # the reference's default ordering at size
])
def test_gpu_equals_oracle_at_baseline_sizes(n, m, covfun, cp, order):
    """factor rows, precision_diag, log-lik, SpMV, triangular solve and one supplied-normal sweep, GPU vs oracle, full size"""
    locs = np.random.default_rng(1).random((n, 2))
    if order == "maxmin":
        locs = locs[nb.order_maxmin(locs) - 1]
    P = make_problem(n, m, seed=1, locs=locs)
    beta_0, ls, lnv = 0.3, 0.1, np.log(0.1)
    Lo = O.vecchia_Linv(cp, covfun, P["locs"], P["NNarray"])
    z = P["rng"].standard_normal(n)
    f_o, pd_o = oracle_sweep(P, Lo, beta_0, ls, lnv, z, "residual")
    # Factor rows: 1e-10 for the exponential family.  Matern, m = 20: the worst of the 250 000 rows sits at ~3e-10 -- 21 x 21 blocks
    # of a smoother kernel at range 0.02 have condition numbers ~1e4-1e5, which amplify the 1e-14-level differences between two
    # correct Bessel-K evaluations (the oracle's std::cyl_bessel_k vs the device's Temme series / per-build table); the bound for
    # that case is 2e-9 on the worst row and 1e-10 on the 99.9 % quantile of the rows.
    tol_rows = TOL if covfun.startswith("exponential") else 2e-9
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], covfun) as ctx:
        assert ctx.factor_build(cp) == 0
        Lg = ctx.factor_get()
        assert rel_rows(Lg, Lo) < tol_rows
        per_row = np.linalg.norm(Lg - Lo, axis=1) / np.linalg.norm(Lo, axis=1)
        assert np.quantile(per_row, 0.999) < TOL
        if covfun.startswith("matern"):        # the direct K_nu evaluation (no table) lands in the same place
            ctx.set_option("matern_table", 0)
            assert ctx.factor_build(cp) == 0
            assert rel_rows(ctx.factor_get(), Lo) < tol_rows
            ctx.set_option("matern_table", 1)
            assert ctx.factor_build(cp) == 0
        del Lg
        ctx.factor_commit()
        assert rel_vec(ctx.precision_diag(), pd_o) < tol_rows          # everything below inherits the factor rows' bound
        ctx.field_set(P["field"])
        ctx.obs_set(P["y"])
        ll_o = O.ll_compressed_sparse_chol(Lo, P["field"] - beta_0, P["NNarray"], ls)
        assert abs(ctx.loglik(beta_0, ls) - ll_o) < tol_rows * abs(ll_o)
        v = P["rng"].standard_normal(n)
        u_o = O.Linv_mult(Lo, v, P["NNarray"])
        assert rel_vec(ctx.spmv(v), u_o) < tol_rows
        assert rel_vec(ctx.sptrsv(u_o), v) < 1e-8                      # solve(L^-1, L^-1 v) = v; conditioning of a depth-~200 recursion
        ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=1, z=z)
        assert rel_vec(ctx.field_get(), f_o) < tol_rows
        mu = np.full(P["n_obs"], beta_0)
        assert abs(ctx.ssr() - O.ssr(P["locs_match"], P["y"], f_o, mu, beta_0)) < TOL * P["n_obs"]


@pytest.mark.parametrize("covfun,m,cp", [("exponential_isotropic", 10, [1.0, 0.07, 0.0]), ("exponential_isotropic", 5, [1.0, 0.05, 0.0]),
                                         ("matern_isotropic", 20, [1.0, 0.1, 0.6, 0.0]), ("exponential_isotropic", 7, [1.0, 0.1, 0.0])])
@pytest.mark.parametrize("layout", [nb.LAYOUT_COLOR, nb.LAYOUT_MORTON])
def test_parity_matrix_on_a_maxmin_ordering(covfun, m, cp, layout):
    """reordering = "maxmin" is the reference default (initialize.R:29): long-range early neighbours, long early columns, more
    colours.  Literal reference loop (one mat-vec per colour) as the sweep oracle."""
    n = 5000
    locs = np.random.default_rng(31).random((n, 2))
    locs = locs[nb.order_maxmin(locs) - 1]
    P = make_problem(n, m, seed=31, locs=locs, n_extra_obs=200)
    beta_0, ls, lnv = -0.2, 0.3, -0.9
    Lo = O.vecchia_Linv(cp, covfun, P["locs"], P["NNarray"])
    z = P["rng"].standard_normal(n)
    f_o, pd_o = oracle_sweep(P, Lo, beta_0, ls, lnv, z, "reference")
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], covfun, layout=layout) as ctx:
        assert ctx.factor_build(cp) == 0
        assert rel_rows(ctx.factor_get(), Lo) < TOL
        ctx.factor_commit()
        assert rel_vec(ctx.precision_diag(), pd_o) < TOL
        ctx.field_set(P["field"])
        ctx.obs_set(P["y"])
        ll_o = O.ll_compressed_sparse_chol(Lo, P["field"] - beta_0, P["NNarray"], ls)
        assert abs(ctx.loglik(beta_0, ls) - ll_o) < TOL * abs(ll_o)
        v = P["rng"].standard_normal(n)
        assert rel_vec(ctx.sptmv(v), O.sparse_chol_tmult(Lo, P["NNarray"], v)) < TOL
        assert rel_vec(ctx.sptrsv(v), O.sparse_chol_solve(Lo, P["NNarray"], v)) < 1e-9
        ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=1, z=z)
        assert rel_vec(ctx.field_get(), f_o) < TOL


@pytest.mark.parametrize("variant", [0, 2, 3])
def test_oversize_columns_in_sweep_and_transposition(variant):
    n, m, hubs = 6000, 5, 2
    P = star_problem(n, m, hubs, seed=41)
    cp = [1.0, 0.3, 0.0]
    beta_0, ls, lnv = 0.1, 0.2, -1.0
    Lo = O.vecchia_Linv(cp, "exponential_isotropic", P["locs"], P["NNarray"])
    z = P["rng"].standard_normal(2 * n)
    f = P["field"].copy()
    pd_o = O.precision_diag(Lo, P["NNarray"])
    rs = O.residuals_sum(P["locs_match"], n, P["y"], np.full(P["n_obs"], beta_0))
    for s in range(2):
        f = O.chromatic_sweep(Lo, P["NNarray"], P["coloring"], pd_o, P["obs_per_loc"], rs, beta_0, ls, lnv, z[s * n:(s + 1) * n], f, form="reference")
    for commit_variant in (0, 1):
        with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
            assert ctx.max_col > 1024                      # the hub columns do exceed a tile
            ctx.set_option("sweep_variant", variant)
            ctx.set_option("commit_variant", commit_variant)
            assert ctx.factor_build(cp) == 0
            ctx.factor_commit()
            assert rel_vec(ctx.precision_diag(), pd_o) < TOL
            ctx.field_set(P["field"])
            ctx.obs_set(P["y"])
            ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=2, z=z)
            assert rel_vec(ctx.field_get(), f) < TOL
            v = P["rng"].standard_normal(n)
            assert rel_vec(ctx.sptmv(v), O.sparse_chol_tmult(Lo, P["NNarray"], v)) < TOL


def test_oversize_columns_on_a_sharded_field():
    """hub sites are boundary sites of their owner and ghosts of every other rank: the oversize-tile push and the ghost apply of
    a long column, host-routed and with the fused peer-to-peer transport"""
    n, m, hubs = 6000, 5, 2
    P = star_problem(n, m, hubs, seed=43)
    cp = [1.0, 0.3, 0.0]
    beta_0, ls, lnv = 0.1, 0.2, -1.0
    z = P["rng"].standard_normal(2 * n)
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        ctx.factor_build(cp)
        ctx.factor_commit()
        ctx.field_set(P["field"])
        ctx.obs_set(P["y"])
        ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=2, z=z)
        f_ref = ctx.field_get()
    owner = nb.spatial_blocks(P["locs"], 3)
    for fused in (False, True):
        ctxs = []
        try:
            for r in range(3):
                plan = nb.shard_plan(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], owner, r, 3)
                c = nb.ShardedContext(plan, device=0, comm_id=None)
                c.factor_build(cp)
                c.factor_commit()
                c.field_set(P["field"][plan["local_sites"]])
                c.obs_set(P["y"][plan["obs_index"]])
                ctxs.append(c)
            if fused:
                nb.connect_local(ctxs)
                nb.group_sweep(ctxs, beta_0, ls, lnv, n_sweeps=2, z=z)
            else:
                for s in range(2):
                    nb.host_routed_sweep(ctxs, beta_0, ls, lnv, z=z[s * n:(s + 1) * n])
            f = np.full(n, np.nan)
            for c in ctxs:
                own = c.plan["owned"] == 1
                f[c.plan["local_sites"][own]] = c.field_get()[own]
            assert rel_vec(f, f_ref) < TOL
        finally:
            for c in ctxs:
                c.close()
