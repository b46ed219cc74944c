"""One step = the sweep's colours plus the log-likelihood from its residual, closed by loglik_residual_kernel: the log-determinant term
is kept per current factor and must follow every way a new factor becomes current; a step without sweeps must not move the Philox
counter; and the step must give the same field and log-lik bit for bit replayed from its graph, launched directly, with the closing
kernel as a programmatic dependent (sweep variants 0 and 4) or as a plain launch (2 and 3)."""
import numpy as np
import pytest

import nngp_b200 as nb
from oracle import oracle as O
from philox_reference import sweep_normals
from problems import make_problem

pytestmark = pytest.mark.gpu

B0, LS, LNV = 0.3, 0.1, -1.0
CP_A, CP_B = [1.0, 0.1, 0.0], [1.0, 0.07, 0.0]


def open_ctx(P, cp):
    ctx = nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"])
    assert ctx.factor_build(cp) == 0
    ctx.factor_commit()
    ctx.field_set(P["field"])
    ctx.obs_set(P["y"])
    return ctx


def full_pass(ctx, beta_0, log_scale):
    """the log-lik with the residual path switched off (switching clears the residual's validity, so switch back after)"""
    ctx.set_option("loglik_from_residual", 0)
    ll = ctx.loglik(beta_0, log_scale)
    ctx.set_option("loglik_from_residual", 1)
    return ll


def build_b_in_current_slot(ctx):
    assert ctx.factor_build(CP_B) == 0


def commit_b_from_proposal(ctx):
    assert ctx.factor_build(CP_B, slot=1) == 0
    ctx.factor_commit(slot=1)


def accept_b(ctx):
    assert ctx.factor_build(CP_B, slot=1) == 0
    ctx.factor_accept()


@pytest.mark.parametrize("make_b_current", [build_b_in_current_slot, commit_b_from_proposal, accept_b],
                         ids=["factor_build", "factor_commit_slot_1", "factor_accept"])
def test_log_determinant_follows_the_current_factor(make_b_current):
    """a step with factor A fills the kept log-determinant; once B is current the next step's log-lik must be B's, not A's"""
    P = make_problem(30_000, 10, seed=61)
    with open_ctx(P, CP_A) as ctx:
        f = P["field"].copy()
        ll_a = ctx.sweep_loglik_host(f, B0, LS, LNV, n_sweeps=2, seed=3)
        assert abs(ll_a - full_pass(ctx, B0, LS)) < 1e-12 * abs(ll_a)
        La = ctx.factor_get()
        make_b_current(ctx)
        ll_b = ctx.sweep_loglik_host(f, B0, LS, LNV, n_sweeps=2, seed=3)
        ll_b_full = full_pass(ctx, B0, LS)
        ll_a_same_field = O.ll_compressed_sparse_chol(La, f - B0, P["NNarray"], LS)
        print(f"\nstep log-lik with B {ll_b!r}, B's full pass {ll_b_full!r}, A's on the same field {ll_a_same_field!r}")
        assert abs(ll_b - ll_b_full) < 1e-12 * abs(ll_b_full)
        assert abs(ll_b - ll_a_same_field) > 1e-6 * abs(ll_b), "A and B give the same log-lik: the test is blind"
        # the log-lik taken on its own after a sweep reads the same kept term
        ctx.gibbs_sweep(B0, LS, LNV, n_sweeps=1, seed=4)
        assert abs(ctx.loglik(B0, LS) - full_pass(ctx, B0, LS)) < 1e-12 * abs(ll_b_full)


def test_step_without_sweeps_leaves_the_counter_alone():
    """sweep_loglik_host with n_sweeps = 0 takes the log-lik of the field it was given and advances no counter: the Philox sweep
    after it draws the normals of counter 1 (the one after the first sweep), replayed in supplied mode on a second context"""
    P = make_problem(4000, 10, seed=62)
    seed = 11
    with open_ctx(P, CP_A) as ctx, open_ctx(P, CP_A) as rep:
        ctx.gibbs_sweep(B0, LS, LNV, n_sweeps=1, seed=seed)                   # counter 0
        f = ctx.field_get()
        fio = f.copy()
        ll = ctx.sweep_loglik_host(fio, B0, LS, LNV, n_sweeps=0, seed=seed)   # no sweep
        assert np.array_equal(fio, f)
        assert abs(ll - full_pass(ctx, B0, LS)) < 1e-12 * abs(ll)
        ctx.field_set(f)
        ctx.gibbs_sweep(B0, LS, LNV, n_sweeps=1, seed=seed)                   # must be counter 1
        rep.field_set(f)
        rep.gibbs_sweep(B0, LS, LNV, n_sweeps=1, z=sweep_normals(seed, 1, 1, P["coloring"]))
        got, want = ctx.field_get(), rep.field_get()
        gap = float(np.max(np.abs(got - want)) / np.max(np.abs(want)))
        print(f"\nPhilox sweep after a step without sweeps vs counter 1 replayed: max rel {gap:.2e}")
        assert gap <= 1e-12


@pytest.mark.parametrize("variant", [0, 2, 3, 4])
def test_step_is_the_same_from_graph_and_direct_launches(variant):
    """time_op's step (its log-lik taken at beta_0 = 0, so the sweeps run at beta_0 = 0) and sweep_loglik_host's, graph on and off:
    the same field and log-lik bit for bit, and the same as a sweep followed by a separate log-lik call"""
    P = make_problem(30_000, 10, seed=63)
    res = {}
    for graph in (1, 0):
        with open_ctx(P, CP_A) as ctx:
            ctx.set_option("sweep_variant", variant)
            ctx.set_option("use_graph", graph)
            ctx.gibbs_sweep(0.0, LS, LNV, n_sweeps=1, seed=5)   # the sweep parameters time_op uses
            ctx.time_op("sweep_loglik", reps=3)
            f_t, ll_t = ctx.field_get(), ctx.loglik(0.0, LS)
            f = P["field"].copy()
            ll_h = ctx.sweep_loglik_host(f, 0.0, LS, LNV, n_sweeps=3, seed=6)
            ctx.field_set(P["field"])
            ctx.gibbs_sweep(0.0, LS, LNV, n_sweeps=3, seed=6)     # counters 7-9 here, 4-6 in the step above
            res[graph] = (f_t, ll_t, f, ll_h, ctx.loglik(0.0, LS))
    (f_t1, ll_t1, f1, ll_h1, ll_s1), (f_t0, ll_t0, f0, ll_h0, ll_s0) = res[1], res[0]
    assert np.array_equal(f_t1, f_t0) and ll_t1 == ll_t0
    assert np.array_equal(f1, f0) and ll_h1 == ll_h0
    assert ll_s1 == ll_s0
    # the step's own log-lik against the full pass of the field it returned
    with open_ctx(P, CP_A) as ctx:
        ctx.field_set(f1)
        assert abs(ll_h1 - ctx.loglik(0.0, LS)) < 1e-12 * abs(ll_h1)
