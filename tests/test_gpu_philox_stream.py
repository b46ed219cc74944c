"""The on-device Philox stream, the sampler's default source of randomness, pinned to its reference (tests/philox_reference.py):
which normal each site receives in every sweep path, how the per-context sweep counter advances through every entry point that
sweeps, and whole Philox chains against the oracle chain run in Philox mode.  Every comparison prints its observed maximum
(pytest -rP shows them)."""
import itertools

import numpy as np
import pytest

import nngp_b200 as nb
from oracle import oracle as O
from philox_reference import chain_seed, philox_normals, sweep_normals
from problems import assert_regression_chain_matches, make_problem, make_regression_problem, star_problem

pytestmark = pytest.mark.gpu

TOL = 1e-10          # device against the oracle, as in test_gpu_parity.py
TOL_REPLAY = 1e-12   # a Philox call against a supplied-mode call handed the reference normals: same kernels, normals within ~1e-14
SEEDS = [0, 7, -3, 2 ** 32 + 5, 2 ** 45 + 17, chain_seed(4600, 2)]   # negative, past 32 bits, and a chain's key with bits in key1
B0, LS, LNV = 0.3, 0.2, -1.1
EPS = 2.0 ** -53
# |cospi(2 u2) - cos(2 pi u2)| <= 1.5e-15 (the rounding of 2 pi u2) times the radius sqrt(-2 log u1) <= sqrt(108 log 2) = 8.65, plus
# a few ulps of the radius for the device's and the reference's log and sqrt
GEN = 2e-15 * 8.65


def rel_vec(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def new_context(P, cp, covfun="exponential_isotropic", layout=nb.LAYOUT_MORTON):
    ctx = nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], covfun, layout=layout)
    assert ctx.factor_build(cp) == 0
    ctx.factor_commit()
    ctx.field_set(P["field"])
    ctx.obs_set(P["y"])
    return ctx


def oracle_sweeps(P, Lo, z, n_sweeps, form="reference"):
    """n_sweeps sweeps of update_Gaussian.R:257-275 from P's field with the normals z (hand-out order, sweep after sweep)"""
    n = P["n"]
    pd = O.precision_diag(Lo, P["NNarray"])
    rs = O.residuals_sum(P["locs_match"], n, P["y"], np.full(P["n_obs"], B0))
    f = P["field"].copy()
    for s in range(n_sweeps):
        f = O.chromatic_sweep(Lo, P["NNarray"], P["coloring"], pd, P["obs_per_loc"], rs, B0, LS, LNV, z[s * n:(s + 1) * n], f, form=form)
    return f


class ColourOne:
    """Reads the device's normals off colour 1.  A colour-1 site's conditional mean depends only on the starting field, so a Philox
    sweep and a supplied sweep with z = 0 from the same field differ there by z / sqrt(prec) alone:
        f_new = c0 - c1 a,  c0 = beta0 + (Qss w e_ls + e_ln resid) / prec + z / sqrt(prec),  c1 a = e_ls (L^T L w)_s / prec.
    Bound per site: the four roundings of c0 and f_new in each run, of quantities no larger than `scale` below, scaled back by
    sqrt(prec); the generators' difference (GEN); a few ulps of z for sqrt(1/prec) sqrt(prec) != 1."""

    def __init__(self, P, Lo, qss, f_zero):
        n, lm = P["n"], P["locs_match"] - 1
        self.c1 = P["coloring"] == 1
        e_ls, e_ln = np.exp(-LS), np.exp(-LNV)
        self.prec = e_ls * qss + e_ln * P["obs_per_loc"]
        w = P["field"] - B0
        LtLw = O.sparse_chol_tmult(Lo, P["NNarray"], O.Linv_mult(Lo, w, P["NNarray"]))
        resid = np.bincount(lm, weights=P["y"], minlength=n) - P["obs_per_loc"] * B0
        self.base = abs(B0) + (e_ls * (np.abs(LtLw) + qss * np.abs(w)) + e_ln * np.abs(resid)) / self.prec
        self.f_zero = f_zero

    def check(self, f_philox, seed, counter, label):
        c1, sp = self.c1, np.sqrt(self.prec[self.c1])
        got = (f_philox[c1] - self.f_zero[c1]) * sp
        want = philox_normals(seed, counter, c1.size)[c1]
        scale = self.base[c1] + np.maximum(np.abs(f_philox[c1]), np.abs(self.f_zero[c1])) + np.abs(want) / sp
        bound = 16 * EPS * scale * sp + GEN + 8 * EPS * np.abs(want)
        err = np.abs(got - want)
        print(f"{label} seed {seed} counter {counter}: {c1.sum()} colour-1 normals, max |dz| {err.max():.2e} "
              f"(bound here {bound.max():.2e}; worst err / bound {np.max(err / bound):.2f})")
        assert np.all(err <= bound), (label, seed, counter, float(err.max()), int(np.argmax(err / bound)))
        return float(err.max())


def colour_one_study(P, cp, seeds, counters, layout=nb.LAYOUT_MORTON, label=""):
    Lo = O.vecchia_Linv(cp, "exponential_isotropic", P["locs"], P["NNarray"])
    with new_context(P, cp, layout=layout) as cz:
        cz.gibbs_sweep(B0, LS, LNV, n_sweeps=1, z=np.zeros(P["n"]))
        reader = ColourOne(P, Lo, cz.precision_diag(), cz.field_get())
    worst = 0.0
    for seed in seeds:
        with new_context(P, cp, layout=layout) as ctx:          # a fresh context: the sweep counter starts at 0
            for k in counters:
                ctx.field_set(P["field"])
                ctx.gibbs_sweep(B0, LS, LNV, n_sweeps=1, seed=seed)
                worst = max(worst, reader.check(ctx.field_get(), seed, k, label))
    print(f"{label}: max |dz| over every seed and counter {worst:.2e} (suggested absolute bound 1e-13)")


@pytest.mark.parametrize("layout", [nb.LAYOUT_COLOR, nb.LAYOUT_MORTON])
def test_colour_one_reads_off_the_device_normals(layout):
    """the normal of every colour-1 site at counters 0, 1, 2 of a fresh context, for every seed, is the reference's"""
    P = make_problem(4000, 10, seed=51, n_extra_obs=400, drop_obs_frac=0.1)
    colour_one_study(P, [1.0, 0.08, 0.0], SEEDS, (0, 1, 2), layout=layout, label=f"layout {layout}")


def philox_against_supplied(P, cp, cases, n_sweeps, layout=nb.LAYOUT_MORTON, form="reference", label=""):
    """For each (sweep_variant, use_graph, seed): one Philox call of n_sweeps from P's field on one context, the same call in
    supplied mode with the reference normals in hand-out order on a second context (<= TOL_REPLAY), and the oracle's sweeps with
    those normals (<= TOL).  The Philox context's counter runs on from call to call."""
    Lo = O.vecchia_Linv(cp, "exponential_isotropic", P["locs"], P["NNarray"])
    worst = dict(replay=0.0, oracle=0.0)
    counter = 0
    with new_context(P, cp, layout=layout) as cph, new_context(P, cp, layout=layout) as csu:
        for variant, graph, seed in cases:
            for c in (cph, csu):
                c.set_option("sweep_variant", variant)
                c.set_option("use_graph", graph)
                c.field_set(P["field"])
            cph.gibbs_sweep(B0, LS, LNV, n_sweeps=n_sweeps, seed=seed)
            z = sweep_normals(seed, counter, n_sweeps, P["coloring"])
            counter += n_sweeps
            csu.gibbs_sweep(B0, LS, LNV, n_sweeps=n_sweeps, z=z)
            fp, fs = cph.field_get(), csu.field_get()
            fo = oracle_sweeps(P, Lo, z, n_sweeps, form=form)
            case = dict(label=label, variant=variant, use_graph=graph, seed=seed, counters=(counter - n_sweeps, counter - 1))
            gaps = dict(replay=rel_vec(fp, fs), oracle=rel_vec(fp, fo))
            for k in worst:
                worst[k] = max(worst[k], gaps[k])
            assert gaps["replay"] <= TOL_REPLAY, (case, gaps)
            assert gaps["oracle"] < TOL, (case, gaps)
    print(f"{label}: Philox vs supplied reference normals max rel {worst['replay']:.2e}, vs oracle {worst['oracle']:.2e}")


@pytest.mark.parametrize("layout", [nb.LAYOUT_COLOR, nb.LAYOUT_COLOR_MORTON, nb.LAYOUT_MORTON])
@pytest.mark.parametrize("m,d", [(5, 2), (10, 2), (31, 2), (12, 4)])
def test_philox_sweeps_draw_the_reference_normals_in_handout_order(m, d, layout):
    """three Philox sweeps in one call = the supplied-mode call handed the reference normals of counters k..k+2 colour by colour,
    for every sweep variant, with and without the captured graph, for every seed"""
    P = make_problem(3000, m, d=d, seed=61, n_extra_obs=200)
    cases = [(v, g, SEEDS[i % len(SEEDS)]) for i, (v, g) in enumerate(itertools.product(range(5), (1, 0)))]
    philox_against_supplied(P, [1.0, 0.08 if d == 2 else 0.3, 0.0], cases, 3, layout=layout, label=f"m={m} d={d} layout={layout}")


def test_philox_sweeps_through_oversize_column_tiles():
    """hub columns longer than a sweep tile (the whole-CTA path) draw the same normals"""
    P = star_problem(6000, 5, 2, seed=41)
    cases = [(v, 1, s) for v in (0, 2, 3) for s in (SEEDS[1], SEEDS[4])]
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        assert ctx.max_col > 1024
    philox_against_supplied(P, [1.0, 0.3, 0.0], cases, 3, label="star")


def test_sweep_counter_advances_in_every_entry_point_that_sweeps():
    """one context through gibbs_sweep (Philox and supplied), sweep_loglik_host, time_op's two sweeping ops and a final Philox
    sweep; every Philox step replayed in supplied mode on a second context with the normals of the counters it must have used.
    Then time_op_group over two contexts (repetitions + 1 sweeps each) and a Philox sweep on each."""
    P = make_problem(3000, 10, seed=71, n_extra_obs=200)
    cp, seed, n = [1.0, 0.08, 0.0], 2 ** 32 + 5, P["n"]
    worst = [0.0]

    def replay(rep, start, k, n_sweeps, s, got, what):
        rep.field_set(start)
        rep.gibbs_sweep(B0, LS, LNV, n_sweeps=n_sweeps, z=sweep_normals(s, k, n_sweeps, P["coloring"]))
        gap = rel_vec(got, rep.field_get())
        worst[0] = max(worst[0], gap)
        print(f"{what}: counters {k}..{k + n_sweeps - 1} under seed {s}: max rel {gap:.2e}")
        assert gap <= TOL_REPLAY, (what, k, gap)

    f0 = P["field"]
    with new_context(P, cp) as ctx, new_context(P, cp) as rep:
        ctx.gibbs_sweep(B0, LS, LNV, n_sweeps=3, seed=seed)                        # counters 0-2
        f1 = ctx.field_get()
        replay(rep, f0, 0, 3, seed, f1, "gibbs_sweep")
        z = P["rng"].standard_normal(2 * n)
        ctx.gibbs_sweep(B0, LS, LNV, n_sweeps=2, z=z)                              # supplied: 3-4
        rep.field_set(f1)
        rep.gibbs_sweep(B0, LS, LNV, n_sweeps=2, z=z)
        f2 = ctx.field_get()
        assert np.array_equal(f2, rep.field_get())
        fio = f2.copy()
        ctx.sweep_loglik_host(fio, B0, LS, LNV, n_sweeps=2, seed=seed)            # 5-6
        replay(rep, f2, 5, 2, seed, fio, "sweep_loglik_host")
        ctx.time_op("gibbs_sweep", reps=3)                                          # 7-9, time_op's own seed
        f3 = ctx.field_get()
        replay(rep, fio, 7, 3, 12345, f3, "time_op gibbs_sweep")
        ctx.time_op("sweep_loglik", reps=2)                                         # 10-11
        replay(rep, f3, 10, 2, 12345, ctx.field_get(), "time_op sweep_loglik")
        ctx.field_set(f0)
        ctx.gibbs_sweep(B0, LS, LNV, n_sweeps=1, seed=seed)                        # 12
        replay(rep, f0, 12, 1, seed, ctx.field_get(), "gibbs_sweep after time_op")
        with new_context(P, cp) as a, new_context(P, cp) as b:
            a.gibbs_sweep(B0, LS, LNV, n_sweeps=1, seed=seed)                      # a: 0
            b.gibbs_sweep(B0, LS, LNV, n_sweeps=2, seed=seed)                      # b: 0-1
            fa, fb = a.field_get(), b.field_get()
            nb.time_op_group([a, b], "gibbs_sweep", reps=3)                         # a: 1-4, b: 2-5
            replay(rep, fa, 1, 4, 12345, a.field_get(), "time_op_group, first context")
            replay(rep, fb, 2, 4, 12345, b.field_get(), "time_op_group, second context")
            for c, k in ((a, 5), (b, 6)):
                c.field_set(f0)
                c.gibbs_sweep(B0, LS, LNV, n_sweeps=1, seed=seed)
                replay(rep, f0, k, 1, seed, c.field_get(), f"gibbs_sweep after time_op_group (counter {k})")
    print(f"counter bookkeeping: max rel {worst[0]:.2e}")


def test_philox_stream_at_bench_size():
    """the benchmark's workload: n = 1M, m = 10, max-min ordering (the colours where the 6-CTA/SM build runs); colour 1 read off at
    counters 0 and 1, then two Philox sweeps against the reference normals and the oracle: sweep variant 0 (the default) with and
    without the captured graph, and variant 4 (the other one with the 6-CTA/SM build)"""
    n = 1_000_000
    locs = np.random.default_rng(1).random((n, 2))
    locs = locs[nb.order_maxmin(locs) - 1]
    P = make_problem(n, 10, seed=1, locs=locs)
    cp, seed = [1.0, 0.05, 0.0], chain_seed(4600, 2)
    colour_one_study(P, cp, [seed], (0, 1), label="n=1M")
    philox_against_supplied(P, cp, [(0, 1, seed), (0, 0, SEEDS[3]), (4, 1, SEEDS[2])], 2, form="residual", label="n=1M")


def assert_chain_matches(dev, ora, label):
    """same accept/reject sequence with at least one accept of each kind; records within 1e-8, field and field records within 1e-7,
    logvar_* within 1e-12"""
    pg, recg, frecg, accg, fg = dev
    po, fo, reco, freco, acco = ora
    gaps = dict(records=np.max(np.abs(recg - reco)), field=np.max(np.abs(fg - fo)), field_records=np.max(np.abs(frecg - freco)),
                logvar_ancillary=abs(pg["logvar_ancillary"] - po["logvar_ancillary"]),
                logvar_sufficient=abs(pg["logvar_sufficient"] - po["logvar_sufficient"]))
    print(f"{label}: accepts {int(accg[:, 0].sum())} ancillary, {int(accg[:, 1].sum())} sufficient of {accg.shape[0]}; "
          + ", ".join(f"{k} {v:.2e}" for k, v in gaps.items()))
    flips = np.argwhere(accg != acco)
    assert flips.size == 0, f"{label}: accept/reject differs at (iteration - 1, step) {flips[:5].tolist()}"
    assert np.all(accg.sum(axis=0) > 0), label
    assert gaps["records"] < 1e-8, (label, gaps)
    assert gaps["field"] < 1e-7 and gaps["field_records"] < 1e-7, (label, gaps)
    assert gaps["logvar_ancillary"] < 1e-12 and gaps["logvar_sufficient"] < 1e-12, (label, gaps)


# proposal variances small enough that both Metropolis steps accept several times in 50 iterations
LOGVAR = dict(logvar_ancillary=-6.0, logvar_sufficient=-4.0)


def chain_problem(covfun, n=1500, m=5, seed=41):
    P = make_problem(n, m, seed=seed)
    cp = [1.0, 0.1, 0.0] if covfun.startswith("exp") else [1.0, 0.1, 0.7, 0.0]
    w = O.sparse_chol_solve(O.vecchia_Linv(cp, covfun, P["locs"], P["NNarray"]), P["NNarray"], P["rng"].standard_normal(n))
    y = 1.0 + w + np.sqrt(0.1) * P["rng"].standard_normal(n)
    return P, w, y, np.arange(1, n + 1, dtype=np.int32)


@pytest.mark.parametrize("iter_start", [0, 4600])
@pytest.mark.parametrize("n_chromatic", [1, 3])
@pytest.mark.parametrize("covfun,shape", [("exponential_isotropic", [np.log(0.1)]), ("matern_isotropic", [np.log(0.1), 0.3])])
def test_philox_chain_run_matches_the_oracle_chain(covfun, shape, n_chromatic, iter_start):
    """nngp_chain_run in its default Philox mode against the oracle chain in Philox mode (key (iter_start << 20) ^ chain_index, R's
    stream for the scalars); then a second call on the same context with iter_start advanced, as mcmc_nngp_run's cycles do, against
    the oracle started at counter n_iter * n_chromatic"""
    n_iter = 50
    P, w, y, lm = chain_problem(covfun)
    p0 = dict(shape=shape, beta_0=0.9, log_scale=-0.2, log_noise_variance=np.log(0.2), **LOGVAR)
    var_y = np.var(y, ddof=1)
    ora = [O.update_gaussian_chain(P["locs"], P["NNarray"], P["coloring"], lm, np.ones(P["n"]), y, covfun, p0, 0.9 + w, n_iter, 0.5,
                                   n_chromatic, iter_start, 1, 0, rng="philox")]
    ora.append(O.update_gaussian_chain(P["locs"], P["NNarray"], P["coloring"], lm, np.ones(P["n"]), y, covfun, ora[0][0], ora[0][1],
                                       n_iter, 0.5, n_chromatic, iter_start + n_iter, 1, 0, rng="philox",
                                       sweep_counter=n_iter * n_chromatic))
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], lm, covfun) as ctx:
        ctx.field_set(0.9 + w)
        ctx.obs_set(y)
        p = p0
        for k in range(2):
            pg, recg, frecg, accg = ctx.chain_run(p, n_iter, var_y, thin=0.5, n_chromatic=n_chromatic, iter_start=iter_start + k * n_iter,
                                                  chain_index=1)
            assert_chain_matches((pg, recg, frecg, accg, ctx.field_get()), ora[k],
                                 f"{covfun} n_chromatic={n_chromatic} iter_start={iter_start + k * n_iter}")
            p = pg


@pytest.mark.parametrize("iter_start", [0, 4600])
def test_philox_chain_run_regressors_matches_the_oracle_chain(iter_start):
    """nngp_chain_run_regressors with location-level regressors (interweaving) in Philox mode against the oracle in Philox mode"""
    n, m, n_iter = 1500, 5, 50
    P = make_regression_problem(n, m, seed=23, n_extra_obs=300, p_locs=2, p_obs=1)
    p0 = dict(shape=[np.log(0.1)], beta_0=0.5, log_scale=-0.2, log_noise_variance=np.log(0.15), **LOGVAR)
    beta0 = 0.1 * np.ones(P["X"].shape[1])
    field0 = 0.5 + P["w"]
    reg = dict(X=P["X"], xlocs=P["xlocs"], first_obs=P["first_obs"], solve_1XT1X=P["solve_1XT1X"],
               chol_solve_1XT1X=P["chol_solve_1XT1X"], beta=beta0)
    ora = O.update_gaussian_chain(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], P["obs_per_loc"], P["y"],
                                  "exponential_isotropic", p0, field0, n_iter, 0.5, 2, iter_start, 3, 1, regressors=reg, rng="philox")
    var_y = float(np.var(P["y"], ddof=1))
    with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"]) as ctx:
        ctx.regressors_set(P["X"], P["y"], xlocs=P["xlocs"], first_obs=P["first_obs"])
        ctx.field_set(field0)
        dev = ctx.chain_run_regressors(p0, beta0, P["solve_1XT1X"], P["chol_solve_1XT1X"], n_iter, var_y, thin=0.5, n_chromatic=2,
                                       iter_start=iter_start, chain_index=3)
        dev = dev + (ctx.field_get(), ctx.ssr())
    assert_regression_chain_matches(dev, ora, P["X"], P["y"], P["locs_match"], f"regressors, Philox, iter_start={iter_start}")
    assert np.all(dev[4].sum(axis=0) > 0), "an accept of each kind"


def test_philox_chains_run_match_their_oracle_chains():
    """nngp_chains_run: three concurrent Philox chains, each keyed by its own chain_index, against three oracle chains"""
    n_iter, iter_start = 50, 10
    covfun = "exponential_isotropic"
    P, w, y, lm = chain_problem(covfun, seed=43)
    var_y = np.var(y, ddof=1)
    p0 = [dict(shape=[np.log(0.08 + 0.02 * k)], beta_0=0.9 + 0.1 * k, log_scale=-0.2 - 0.1 * k, log_noise_variance=np.log(0.2),
               **LOGVAR) for k in range(3)]
    rng = np.random.default_rng(5)
    fields = [0.9 + w + 0.1 * rng.standard_normal(P["n"]) for _ in range(3)]
    cs = []
    try:
        for k in range(3):
            c = nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], lm, covfun)
            c.field_set(fields[k])
            c.obs_set(y)
            cs.append(c)
        con = nb.chains_run(cs, p0, n_iter, var_y, thin=0.5, n_chromatic=2, iter_start=iter_start, chain_indices=[1, 2, 3])
        dev = [con[k] + (cs[k].field_get(),) for k in range(3)]
    finally:
        for c in cs:
            c.close()
    for k in range(3):
        ora = O.update_gaussian_chain(P["locs"], P["NNarray"], P["coloring"], lm, np.ones(P["n"]), y, covfun, p0[k], fields[k], n_iter,
                                      0.5, 2, iter_start, k + 1, 0, rng="philox")
        assert_chain_matches(dev[k], ora, f"chains_run chain {k + 1}")
