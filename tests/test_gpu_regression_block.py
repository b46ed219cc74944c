"""The regression block of nngp_chain_run_regressors (update_Gaussian.R:226-250) against the oracle chain on designs whose
products span several of op_atb's row chunks (kAtbRowsPerChunk = 4096 rows, nngp_b200.cu): the heavy-metals model of config 2,
and several chains advancing at once on one GPU, each with its own product buffers.  Both sides are driven by R's stream."""
import os

import numpy as np
import pytest

import nngp_b200 as nb
from oracle import oracle as O
from problems import assert_regression_chain_matches, make_regression_problem

pytestmark = pytest.mark.gpu

K = 4096   # kAtbRowsPerChunk


def chunks(rows):
    return -(-rows // K)


def test_config2_heavy_metals_regression_block_matches_oracle_chain():
    """config 2 as test_config2_heavy_metals_subset_runs_end_to_end builds it (real lon/lat data, exponential_sphere, m = 5,
    11 numeric + 3 factor location regressors, X$locs = 1..14), chain 1's initial state, 60 iterations so that the proposal
    variances adapt at iterations 25 and 50."""
    import pandas as pd
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "heavy_metals_subset.npz"), allow_pickle=False)
    df = pd.DataFrame(z["X_numeric"], columns=[str(s) for s in z["numeric_names"]])
    for k in ("minotype", "glwd31", "MAJOR1"):
        lv = z[f"levels_{k}"]
        df[k] = pd.Categorical(lv[z[f"factor_{k}"] - 1])
    lst = nb.mcmc_nngp_initialize(z["observed_locs"], z["observed_field"], X_locs=df, stationary_covfun="exponential_sphere", m=5, n_chains=3, seed=1)
    va, X, y = lst["vecchia_approx"], lst["X"], lst["observed_field"]
    assert X["locs"] == list(range(14))
    xlocs = np.array([c + 1 for c in X["locs"]], dtype=np.int32)
    assert chunks(va["n_obs"]) == 3 and chunks(va["n_locs"]) == 3 and X["X"].shape[1] + 1 > 8 * 16   # 3 x 3 chunks, 9 tiles
    st = lst["states"]["chain_1"]["params"]
    p0 = dict(shape=st["shape"], beta_0=st["beta_0"], log_scale=st["log_scale"], log_noise_variance=st["log_noise_variance"],
              logvar_sufficient=-2.0, logvar_ancillary=-2.0)
    n_iter, n_chromatic = 60, 5
    reg = dict(X=X["X"], xlocs=xlocs, first_obs=va["hctam_scol_1"], solve_1XT1X=X["solve_1XT1X"], chol_solve_1XT1X=X["chol_solve_1XT1X"],
               beta=st["beta"])
    ora = O.update_gaussian_chain(lst["locs"], va["NNarray"], va["coloring"], va["locs_match"], va["obs_per_loc"], y, "exponential_sphere",
                                  p0, st["field"], n_iter, 0.5, n_chromatic, 0, 1, 1, regressors=reg)
    var_y = float(np.var(y, ddof=1))
    with nb.NNGPContext(lst["locs"], va["NNarray"], va["coloring"], va["locs_match"], "exponential_sphere") as ctx:
        ctx.regressors_set(X["X"], y, xlocs=xlocs, first_obs=va["hctam_scol_1"])
        ctx.field_set(st["field"])
        dev = ctx.chain_run_regressors(p0, st["beta"], X["solve_1XT1X"], X["chol_solve_1XT1X"], n_iter, var_y, thin=0.5,
                                       n_chromatic=n_chromatic, iter_start=0, chain_index=1, rng_mode=nb.RNG_SUPPLIED)
        dev = dev + (ctx.field_get(), ctx.ssr())
    print(f"config 2: cond(solve_1XT1X) = {np.linalg.cond(X['solve_1XT1X']):.2e}")
    assert_regression_chain_matches(dev, ora, X["X"], y, va["locs_match"], "config 2")


def test_concurrent_chains_with_regressors_match_their_oracle_chains():
    """nngp_chains_run_regressors: three chains co-scheduled on one GPU (a context, stream and host thread each, every context with
    its own A^T B partial and output buffers) at 13 000 observations over 10 000 sites with 80 columns, each against the oracle
    chain with its own chain_index."""
    n, m, n_iter = 10000, 5, 50
    P = make_regression_problem(n, m, seed=29, n_extra_obs=3000, p_locs=20, p_obs=60)
    assert chunks(P["n_obs"]) == 4 and chunks(n) == 3
    y, var_y = P["y"], float(np.var(P["y"], ddof=1))
    p0 = [dict(shape=[np.log(0.08 + 0.02 * k)], beta_0=0.5 + 0.1 * k, log_scale=-0.2 - 0.1 * k, log_noise_variance=np.log(0.15),
               logvar_sufficient=-2.0, logvar_ancillary=-2.0) for k in range(3)]
    rng = np.random.default_rng(4)
    fields = [0.5 + P["w"] + 0.1 * rng.standard_normal(n) for _ in range(3)]
    betas = [0.1 * rng.standard_normal(P["X"].shape[1]) for _ in range(3)]
    cs = []
    try:
        for k in range(3):
            c = nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"])
            c.regressors_set(P["X"], y, xlocs=P["xlocs"], first_obs=P["first_obs"])
            c.field_set(fields[k])
            cs.append(c)
        con = nb.chains_run(cs, p0, n_iter, var_y, thin=0.5, n_chromatic=2, iter_start=0, chain_indices=[1, 2, 3], rng_mode=nb.RNG_SUPPLIED,
                            betas=betas, solve_1XT1X=P["solve_1XT1X"], chol_solve_1XT1X=P["chol_solve_1XT1X"])
        dev = [con[k] + (cs[k].field_get(), cs[k].ssr()) for k in range(3)]
    finally:
        for c in cs:
            c.close()
    for k in range(3):
        reg = dict(X=P["X"], xlocs=P["xlocs"], first_obs=P["first_obs"], solve_1XT1X=P["solve_1XT1X"],
                   chol_solve_1XT1X=P["chol_solve_1XT1X"], beta=betas[k])
        ora = O.update_gaussian_chain(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], P["obs_per_loc"], y, "exponential_isotropic",
                                      p0[k], fields[k], n_iter, 0.5, 2, 0, k + 1, 1, regressors=reg)
        assert_regression_chain_matches(dev[k], ora, P["X"], y, P["locs_match"], f"chain {k + 1}")
