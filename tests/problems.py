"""Seeded synthetic NNGP problems shared by the parity tests, smoke() and bench.py."""
from __future__ import annotations

import json
import os
from decimal import Decimal, localcontext

import numpy as np

import nngp_b200 as nb


def make_problem(n, m, d=2, seed=0, n_extra_obs=0, drop_obs_frac=0.0, locs=None):
    """U(0,1)^d sites in the order generated (= reordering "random"), exact ordered NN, first-fit colouring, y = w + noise."""
    rng = np.random.default_rng(seed)
    if locs is None:
        locs = rng.random((n, d))
    nn = nb.find_ordered_nn(locs, m)
    coloring = nb.greedy_coloring(nn)
    sites = np.arange(1, n + 1, dtype=np.int32)
    if drop_obs_frac > 0:
        sites = sites[rng.random(n) >= drop_obs_frac]
    if n_extra_obs > 0:
        sites = np.concatenate([sites, rng.integers(1, n + 1, n_extra_obs).astype(np.int32)])
    locs_match = sites
    n_obs = locs_match.size
    obs_per_loc = np.bincount(locs_match - 1, minlength=n).astype(np.float64)
    y = rng.standard_normal(n_obs)
    field = 0.3 + rng.standard_normal(n)
    return dict(rng=rng, locs=locs, NNarray=nn, coloring=coloring, locs_match=locs_match, n_obs=n_obs,
                obs_per_loc=obs_per_loc, y=y, field=field, n=n, m=m, d=d)


def make_regression_problem(n, m, seed=0, n_extra_obs=0, p_locs=2, p_obs=1, range_=0.1, xlocs=None):
    """A Gaussian NNGP model WITH regressors as mcmc_nngp_initialize prepares it (initialize.R:116-137): X$X = centred
    cbind(X_locs[locs_match], X_obs) without intercept, X$locs = 1..p_locs, solve_1XT1X / chol_solve_1XT1X (upper factor),
    hctam_scol_1 = first observation of every site; y = beta_0 + X beta + w[locs_match] + noise with w drawn from the prior
    by the host utilities (no oracle, no GPU).
    xlocs (1-based, p_locs distinct columns of 1..p_locs + p_obs): X$locs in that order instead of the prefix; the l-th
    location-level column goes to column xlocs[l] of X$X and the observation-level columns fill the others in order."""
    P = make_problem(n, m, seed=seed, n_extra_obs=n_extra_obs)
    rng, lm = P["rng"], P["locs_match"] - 1
    n_obs = P["n_obs"]
    cols = []
    if p_locs:
        Xl = np.column_stack([P["locs"][:, 0]] + [rng.standard_normal(n) for _ in range(p_locs - 1)])
        cols.append(Xl[lm])
    if p_obs:
        cols.append(rng.standard_normal((n_obs, p_obs)))
    X = np.column_stack(cols)
    if xlocs is None:
        xlocs = np.arange(1, p_locs + 1)
    else:
        xlocs = np.asarray(xlocs)
        assert xlocs.size == p_locs and np.unique(xlocs).size == p_locs and xlocs.min() >= 1 and xlocs.max() <= X.shape[1]
        order = np.empty(X.shape[1], dtype=np.int64)
        order[xlocs - 1] = np.arange(p_locs)
        order[np.setdiff1d(np.arange(X.shape[1]), xlocs - 1)] = np.arange(p_locs, X.shape[1])
        X = X[:, order]
    X = X - X.mean(axis=0)                                                       # initialize.R:132
    one = np.column_stack([np.ones(n_obs), X])
    S = np.linalg.inv(one.T @ one)                                               # :135
    first = np.full(n, -1, dtype=np.int64)
    for o in range(n_obs - 1, -1, -1):
        first[lm[o]] = o
    beta_true = rng.standard_normal(X.shape[1])
    # a smooth field with roughly the right range (exact prior draws are not needed for these tests)
    w = np.sin(P["locs"][:, 0] / range_) * np.cos(P["locs"][:, 1] / range_) + 0.3 * rng.standard_normal(n)
    y = 0.7 + X @ beta_true + w[lm] + np.sqrt(0.1) * rng.standard_normal(n_obs)
    P.update(X=X, xlocs=xlocs.astype(np.int32), first_obs=(first + 1).astype(np.int32), solve_1XT1X=S,
             chol_solve_1XT1X=np.linalg.cholesky(S).T, beta_true=beta_true, y=y, w=w)
    return P


def assert_regression_chain_matches(dev, ora, X, y, locs_match, label, tol_rec=1e-8, tol_field=1e-7, tol_ssr=1e-7):
    """A device chain with regressors against the oracle chain driven by the same R stream.
    dev = (params, records, beta records, field records, accepts, final field, SSR of the context's y - X beta - field);
    ora = O.update_gaussian_chain(..., regressors=...) = (params, field, records, field records, accepts, beta records).
    Same accept/reject sequence with at least one accept (each accept rebuilds the interweaving matrices), records, beta records
    and the final beta within tol_rec, fields within tol_field, the SSR within tol_ssr relative.  Prints the largest
    differences (pytest -rP shows them)."""
    pg, recg, brecg, frecg, accg, fg, ssr_g = dev
    po, fo, reco, freco, acco, breco = ora
    lm = np.asarray(locs_match) - 1
    ssr_o = float(np.sum((y - X @ po["beta"] - fo[lm]) ** 2))
    gaps = dict(records=np.max(np.abs(recg - reco)), beta_records=np.max(np.abs(brecg - breco)),
                beta=np.max(np.abs(pg["beta"] - po["beta"])), field=np.max(np.abs(fg - fo)),
                field_records=np.max(np.abs(frecg - freco)), ssr_rel=abs(ssr_g - ssr_o) / ssr_o)
    print(f"{label}: accepts {int(accg.sum())} of {accg.size}; " + ", ".join(f"{k} {v:.2e}" for k, v in gaps.items()))
    flips = np.argwhere(accg != acco)
    assert flips.size == 0, f"{label}: accept/reject differs at (iteration - 1, step) {flips[:5].tolist()}"
    assert accg.sum() > 0, label
    for k in ("records", "beta_records", "beta"):
        assert gaps[k] < tol_rec, (label, k, gaps[k], tol_rec)
    for k in ("field", "field_records"):
        assert gaps[k] < tol_field, (label, k, gaps[k], tol_field)
    assert gaps["ssr_rel"] < tol_ssr, (label, gaps["ssr_rel"], tol_ssr)
    assert abs(pg["logvar_sufficient"] - po["logvar_sufficient"]) < 1e-12, label


# ---------------------------------------------------------------------------------------------------------------------------
# Kernel probes: a problem whose probe rows decouple into exact 2 x 2 blocks, so that the kernel value the factor build used for
# one distance can be read off a factor row.  Anchor A (site 1) sits at the origin; anchors 2..m sit 1e4 apart on the negative
# first axis, so that every kernel value between them, or between them and a probe, is exactly 0 in double; probe row i is the
# site (x_i, 0[, 0, 0]) and lists A in slot 1 and the far anchors in slots 2..m (a full row: the specialised kernels take it).
# With covparms (s2, 1, [nu,] tau) the block of a probe row is s2 [[1 + tau, rho], [rho, 1 + tau]] plus an identity-scaled
# diagonal part for the far anchors, hence
#     rho(x) = -Linv[i, 1] / Linv[i, 0] * (1 + tau),      Linv[i, 0]^-2 = s2 ((1 + tau) - rho^2 / (1 + tau)).
# ---------------------------------------------------------------------------------------------------------------------------
PROBE_REFERENCE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kernel_probe_reference.json")


def make_probe_problem(m, d, xs):
    """Probe rows m+1 .. m+len(xs) at (x, 0, ...); all-zero colouring (a context without sweeps), no observations."""
    xs = np.asarray(xs, dtype=np.float64)
    n = m + xs.size
    locs = np.zeros((n, d))
    locs[1:m, 0] = -1e4 * np.arange(1, m)
    locs[m:, 0] = xs
    nn = np.full((n, m + 1), nb.NA_INT, dtype=np.int32)
    nn[:, 0] = np.arange(1, n + 1)
    for k in range(1, m):                       # anchor rows: partial, every earlier anchor
        nn[k, 1:k + 1] = np.arange(1, k + 1)
    nn[m:, 1:] = np.arange(1, m + 1)
    return dict(locs=locs, NNarray=nn, coloring=np.zeros(n, dtype=np.int32), locs_match=np.zeros(0, dtype=np.int32), n=n, m=m, d=d)


def probe_covparms(nu, s2, tau):
    """isotropic covparms with range 1 (the scaled distance is x): exponential when nu is None"""
    return [s2, 1.0, tau] if nu is None else [s2, 1.0, nu, tau]


def load_probe_reference(path=PROBE_REFERENCE):
    """x (exact doubles) and, per family, the 50-digit rho split into a double and its remainder, and kappa = |x dlog(rho)/dx|"""
    with open(path) as f:
        ref = json.load(f)
    ref["x"] = np.array([float.fromhex(h) for h in ref["x"]])
    with localcontext() as ctx:
        ctx.prec = 80
        for fam in ref["families"]:
            hi = [float(r) for r in fam["rho"]]
            fam["rho_hi"] = np.array(hi)
            fam["rho_lo"] = np.array([float(Decimal(r) - Decimal(h)) for r, h in zip(fam["rho"], hi)])
            fam["kappa"] = np.array([float(k) for k in fam["kappa"]])
    return ref


# regimes of the device's Matern evaluation by the squared scaled distance s (kernels.cuh: MT_EMIN, MTS_E0, MT_ESCALED, MTS_E1,
# MT_EMAX); the specialised kernels read [2^-26, 2^6) from shared memory, the generic ones from the global table
PROBE_REGIMES = [(0.0, "s = 0"), (2.0 ** -1074, "exact K_nu, s < 2^-80"), (2.0 ** -80, "global table, [2^-80, 2^-26)"),
                 (2.0 ** -26, "smem table, [2^-26, 4)"), (4.0, "smem table e^x-scaled, [4, 2^6)"),
                 (2.0 ** 6, "global table e^x-scaled, [2^6, 2^20)"), (2.0 ** 20, "exact K_nu, s >= 2^20")]


def probe_regime(x):
    s = x * x
    return [name for lo, name in PROBE_REGIMES if s >= lo][-1]


def probe_errors(Linv, m, fam, s2, tau):
    """Per probe row: (relative error of rho, its bound, |conditional variance error|, its bound); NaN where not checked.
    rho >= 1e-280: relative to the 50-digit value, bound 1e-13 + kappa 2^-52 (kappa: the conditioning of rho in its argument, the
    rounding of s = x^2 and of sqrt(s) alone moves rho by kappa ulps).  Smaller rho: absolute 1e-280.  With tau = 0, probes where
    1 - rho^2 < 1e-10 are skipped (a singular block).  The conditional variance Linv[i, 0]^-2 is compared with
    s2 ((1 + tau) - rho_row^2 / (1 + tau)) for the rho read off the same row (checked above): this isolates the pivot arithmetic,
    whose bound is 8 ulps of s2 (1 + tau)."""
    L = Linv[m:]
    rho_hi, rho_lo, kappa = fam["rho_hi"], fam["rho_lo"], fam["kappa"]
    with np.errstate(invalid="ignore", divide="ignore"):      # tau = 0, x = 0: singular block (skipped below)
        got = -L[:, 1] / L[:, 0] * (1.0 + tau)
        var = 1.0 / L[:, 0] ** 2
    err = np.abs((got - rho_hi) - rho_lo)
    big = rho_hi >= 1e-280
    rel = np.where(big, err / np.where(big, rho_hi, 1.0), err)
    bound = np.where(big, 1e-13 + kappa * 2.0 ** -52, 1e-280)
    var_err = np.abs(var - s2 * ((1.0 + tau) - got ** 2 / (1.0 + tau)))
    var_bound = np.full(got.shape, 8 * np.spacing(s2 * (1.0 + tau)))
    if tau == 0.0:
        skip = 1.0 - rho_hi ** 2 < 1e-10
        rel[skip] = np.nan
        var_err[skip] = np.nan
    return rel, bound, var_err, var_bound


def probe_failures(Linv, m, ref, fam, s2, tau, label, worst=None, skip=None):
    """Messages for the probes over their bounds (regime, nu, x, the kernel instantiation); `worst` collects the largest relative
    error of rho per regime (Matern) or for the exponential family when given; probes where `skip` is true are not checked."""
    rel, bound, var_err, var_bound = probe_errors(Linv, m, fam, s2, tau)
    out = []
    for i, x in enumerate(ref["x"]):
        if skip is not None and skip[i]:
            continue
        reg = probe_regime(x)
        if worst is not None and np.isfinite(rel[i]) and fam["rho_hi"][i] >= 1e-280:
            key = reg if fam["nu"] is not None else "exponential"
            worst[key] = max(worst.get(key, 0.0), float(rel[i]))
        if not (rel[i] <= bound[i] or np.isnan(rel[i])) or not (var_err[i] <= var_bound[i] or np.isnan(var_err[i])):
            out.append(f"{label} {fam['covfun']} nu={fam['nu']!r} s2={s2} tau={tau} x={x!r} [{reg}]: rho rel err {rel[i]:.3g} "
                       f"(bound {bound[i]:.3g}), cond. variance err {var_err[i]:.3g} (bound {var_bound[i]:.3g})")
    return out
