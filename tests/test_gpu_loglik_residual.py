"""The log-likelihood after a sweep is taken from the residual r = Linv (field - beta_0) the sweep keeps (loglik_from_residual = 1):
it must agree with the full pass (option 0) and the oracle however many sweeps r was patched over, it must never be used once
anything changed the field, the factor or beta_0 since the sweep, and slots or contexts it does not cover must get the full pass."""
import numpy as np
import pytest

import nngp_b200 as nb
from oracle import oracle as O
from problems import make_problem, make_regression_problem

pytestmark = pytest.mark.gpu

B0, LS, LNV = 0.3, 0.1, -1.0
EXP = ("exponential_isotropic", [1.0, 0.1, 0.0], [1.0, 0.07, 0.0])
MATERN = ("matern_isotropic", [1.0, 0.1, 0.75, 0.0], [1.0, 0.07, 0.75, 0.0])


def open_ctx(P, covfun, cp):
    ctx = nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], covfun)
    assert ctx.factor_build(cp) == 0
    ctx.factor_commit()
    ctx.field_set(P["field"])
    ctx.obs_set(P["y"])
    return ctx


def full_pass(ctx, beta_0, log_scale, slot=0):
    """the log-lik with the residual path switched off (switching clears the residual's validity, so switch back after)"""
    ctx.set_option("loglik_from_residual", 0)
    ll = ctx.loglik(beta_0, log_scale, slot)
    ctx.set_option("loglik_from_residual", 1)
    return ll


@pytest.mark.parametrize("covfun,cp", [EXP[:2], MATERN[:2]], ids=["exponential", "matern"])
def test_residual_loglik_agrees_with_full_pass_and_oracle(covfun, cp):
    worst = 0.0
    for d in (2, 3):
        for m in (5, 10, 20):
            P = make_problem(200_000, m, d=d, seed=100 + 10 * d + m)
            with open_ctx(P, covfun, cp) as ctx:
                Lg = ctx.factor_get()   # the factor's own accuracy is held to the oracle's by the parity tests
                ctx.gibbs_sweep(B0, LS, LNV, n_sweeps=1, seed=1)   # sets the parameters time_op's sweeps use
                for k in (1, 7, 2000):
                    ctx.time_op("gibbs_sweep", reps=k)              # one refresh of r, then k sweeps patching it
                    ll_r = ctx.loglik(B0, LS)
                    ll_f = full_pass(ctx, B0, LS)
                    ll_o = O.ll_compressed_sparse_chol(Lg, ctx.field_get() - B0, P["NNarray"], LS)
                    drift = abs(ll_r - ll_f) / abs(ll_f)
                    worst = max(worst, drift)
                    case = f"{covfun} d={d} m={m} after {k} sweeps"
                    assert drift < 1e-12, f"{case}: residual {ll_r!r} vs full pass {ll_f!r}"
                    assert abs(ll_r - ll_o) < 1e-10 * abs(ll_o), f"{case}: residual {ll_r!r} vs oracle {ll_o!r}"
    print(f"\n{covfun}: worst relative drift of the residual log-lik from the full pass: {worst:.3g}")


def test_state_changes_between_sweep_and_loglik_take_the_full_pass():
    """every entry point that changes the field, the current factor or beta_0 between the sweep and nngp_loglik (and the reads
    that are not known to leave r alone) must make the log-lik the full pass, bit for bit; where the call changes the state, the
    value must also differ from the stale residual's"""
    covfun, cp, cp2 = EXP
    P = make_problem(20_000, 10, seed=7)
    rng = np.random.default_rng(8)
    other = P["field"] + 0.5 * rng.standard_normal(P["n"])
    R = make_regression_problem(20_000, 10, seed=7, n_extra_obs=0, p_locs=1, p_obs=1)

    def init(ctx):
        ctx.field_set(P["field"])
        assert ctx.factor_build(cp) == 0
        ctx.factor_commit()

    def proposal_then(ctx, accept):
        assert ctx.factor_build(cp2, slot=1) == 0
        accept(ctx)

    def ancillary(ctx):
        assert ctx.factor_build(cp2, slot=1) == 0
        ctx.ancillary_propose(B0, 0.2, LNV)
        ctx.ancillary_accept()

    def chain(ctx):
        ctx.chain_run(dict(beta_0=B0, log_scale=LS, log_noise_variance=LNV, shape=np.log([0.1])), 3, var_y=10.0, n_chromatic=2,
                      keep_field=False)

    cases = {
        "field_set": (lambda ctx: ctx.field_set(other), True),
        "field_init": (lambda ctx: ctx.field_init(B0, LS, rng.standard_normal(P["n"])), True),
        "factor_build into the current slot": (lambda ctx: ctx.factor_build(cp2), True),
        "factor_commit of a proposal": (lambda ctx: proposal_then(ctx, lambda c: c.factor_commit(slot=1)), True),
        "factor_accept": (lambda ctx: proposal_then(ctx, lambda c: c.factor_accept()), True),
        "ancillary propose + accept": (ancillary, True),
        "beta0_moments": (lambda ctx: ctx.beta0_moments(LS), False),
        "chain_run": (chain, True),
        "regressors_set": (lambda ctx: ctx.regressors_set(R["X"], R["y"]), False),
    }
    with open_ctx(P, covfun, cp) as ctx:
        for name, (call, changes_state) in cases.items():
            init(ctx)
            ctx.gibbs_sweep(B0, LS, LNV, n_sweeps=3, seed=2)
            ll_stale = ctx.loglik(B0, LS)
            call(ctx)
            ll = ctx.loglik(B0, LS)
            assert ll == full_pass(ctx, B0, LS), name
            if changes_state:
                assert abs(ll - ll_stale) > 1e-6 * abs(ll_stale), f"{name}: the call did not change the log-lik (test is blind)"
        # a sweep at another beta_0, then the log-lik at the old one: r belongs to the new beta_0
        init(ctx)
        ctx.gibbs_sweep(B0 + 0.5, LS, LNV, n_sweeps=3, seed=2)
        ll = ctx.loglik(B0, LS)
        assert ll == full_pass(ctx, B0, LS)
        assert abs(ll - ctx.loglik(B0 + 0.5, LS)) > 1e-6 * abs(ll)


def test_proposal_slot_and_sharded_contexts_take_the_full_pass():
    covfun, cp, cp2 = EXP
    P = make_problem(30_000, 10, seed=9, n_extra_obs=300)
    with open_ctx(P, covfun, cp) as ctx:
        assert ctx.factor_build(cp2, slot=1) == 0
        ctx.gibbs_sweep(B0, LS, LNV, n_sweeps=3, seed=4)
        ll = ctx.loglik(B0, LS, 1)
        assert ll == full_pass(ctx, B0, LS, 1)
    owner = nb.spatial_blocks(P["locs"], 2)
    ctxs = []
    try:
        for r in range(2):
            plan = nb.shard_plan(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], owner, r, 2)
            c = nb.ShardedContext(plan, device=0, comm_id=None)
            c.factor_build(cp)
            c.factor_commit()
            c.field_set(P["field"][plan["local_sites"]])
            c.obs_set(P["y"][plan["obs_index"]])
            ctxs.append(c)
        for _ in range(2):
            nb.host_routed_sweep(ctxs, B0, LS, LNV, seed=4)
        for c in ctxs:
            ll = c.loglik(B0, LS)
            assert ll == full_pass(c, B0, LS)
    finally:
        for c in ctxs:
            c.close()


def test_residual_loglik_is_deterministic():
    covfun, cp, _ = EXP
    P = make_problem(50_000, 10, seed=11)
    runs = []
    for _ in range(2):
        with open_ctx(P, covfun, cp) as ctx:
            ctx.gibbs_sweep(B0, LS, LNV, n_sweeps=5, seed=6)
            lls = [ctx.loglik(B0, LS) for _ in range(3)]
            f = P["field"].copy()
            lls.append(ctx.sweep_loglik_host(f, B0, LS, LNV, n_sweeps=2, seed=7))
            runs.append((lls, f))
    (a, fa), (b, fb) = runs
    assert a[0] == a[1] == a[2] and a == b and np.array_equal(fa, fb)
