#!/usr/bin/env python
"""bench.py -- headline benchmark of the NNGP hot path on B200 (contract: see the task statement / DESIGN.md section 6).

Metric (BASELINE.json): Gibbs sweeps/sec + Vecchia log-lik evals/sec at n = 1M, m = 10.  One STEP = one full chromatic
Gibbs sweep of the latent field (all colour classes, Philox normals) + one Vecchia log-likelihood evaluation.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N = 1: config 3 (synthetic U(0,1)^2 sites, n = 1 000 000, m = 10, exponential_isotropic, range 0.05, sigma^2 = 1, tau^2 = 0.1).
  `value` = steps/s, inputs resident in HBM, CUDA events on the library's stream; `e2e` = the same step through the C ABI with
  pinned HOST buffers (field in, field out, host field for the log-lik).
N > 1 (torchrun, one rank per GPU): ONE field of N x 1M sites sharded over the N GPUs by spatial blocks (SURVEY.md 8e, the
  north_star's multi-GPU split): boundary values pushed into the peers' ghost slots over NVLink from inside the sweep kernel,
  scalar all-reduce for the log-lik.  scaling = "weak" (1M sites per GPU); value = N x (steps/s of the whole field), i.e. steps/s
  counted in 1M-site blocks, so value_N / (N value_1) is the weak-scaling efficiency.  Extra keys: the same n = 1M field sharded
  over the N GPUs (strong scaling) and N independent replicas (one chain per GPU, no collective).
--mode sharded --sites 10000000 --nbrs 20 --covfun matern_isotropic : config 4.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

RANGE, SIGMA2, TAU2, NU = 0.05, 1.0, 0.1, 0.75


def algorithmic(n, m, d=2):
    """SURVEY.md 8(d): FP64 = 8 B, int32 = 4 B, each gathered operand counted once per use, no cache credit."""
    M = m + 1
    return {
        "gibbs_sweep": n * (M * 48 + 40),
        "loglik": n * M * 20,
        "factor_build": n * M * (4 + 8 * d + 8),
        "factor_build_flops": n * (M * (M + 1) / 2 * (3 * d + 35) + M ** 3 / 3 + M ** 2),
        "spmv": n * M * 20 + 8 * n,
    }


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def covparms(covfun, range_):
    return [1.0, range_, 0.0] if covfun.startswith("exponential") else [1.0, range_, NU, 0.0]


def stats(ms):
    ms = np.asarray(ms, dtype=np.float64)
    return {"median": float(np.median(ms)), "min": float(ms.min()), "mean": float(ms.mean()), "reps": int(ms.size)}


def git_sha():
    try:
        return subprocess.run(["git", "-C", ROOT, "rev-parse", "--short", "HEAD"], capture_output=True, text=True, timeout=5).stdout.strip() or None
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except Exception:
                continue
            for k, nm in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def pin_to_gpu_numa(local):
    """best effort: run this rank on the CPUs of the GPU's NUMA node, so that its pinned buffers and staging copies are local to
    the GPU's PCIe root (r01: 8 ranks all on NUMA 0 gave an 8-GPU e2e efficiency of 0.61)"""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=10).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/local_cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return spec
    except Exception:
        pass
    return None


def build_problem(n, m, seed, reordering="random"):
    """config 3 / 4 generator: U(0,1)^2 sites, ordering, exact ordered NN, first-fit colouring (host utilities of the library)"""
    import nngp_b200 as nb
    rng = np.random.default_rng(seed)
    locs = rng.random((n, 2))
    t = {}
    t0 = time.perf_counter()
    if reordering == "maxmin":
        locs = locs[nb.order_maxmin(locs) - 1]
    t["ordering_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    nn = nb.find_ordered_nn(locs, m)
    t["neighbours_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    coloring = nb.greedy_coloring(nn)
    t["colouring_s"] = time.perf_counter() - t0
    locs_match = np.arange(1, n + 1, dtype=np.int32)
    return rng, locs, nn, coloring, locs_match, t


DUMP_MAX_FIELD = 4_000_000   # float64 values (32 MB): a larger field is dumped as a fixed, seeded sample of this many sites


def dump_outputs(out_dir, field, loglik):
    """--dump-outputs: what the last timed step returns to a caller, the swept field and its Vecchia log-lik, as float64 .npy files,
    so that two builds run with the same arguments can be compared output for output"""
    os.makedirs(out_dir, exist_ok=True)
    if field.size > DUMP_MAX_FIELD:
        idx = np.sort(np.random.default_rng(0).choice(field.size, DUMP_MAX_FIELD, replace=False))
        np.save(os.path.join(out_dir, "field_sample.npy"), field[idx])
    else:
        np.save(os.path.join(out_dir, "field.npy"), field)
    np.save(os.path.join(out_dir, "loglik.npy"), np.array([loglik], dtype=np.float64))


# ---------------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle restatement of the reference's CPU path (R + GpGp + Matrix are not in this image)
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_chain_worker(args):
    n, m, seed, steps, warmup, form, reordering = args
    from oracle import oracle as O
    rng = np.random.default_rng(seed)
    locs = rng.random((n, 2))
    os.environ["NNGP_QUIET"] = "1"
    import nngp_b200 as nb   # host set-up utilities only (no CUDA call is made in this process)
    if reordering == "maxmin":
        locs = locs[nb.order_maxmin(locs) - 1]
    nn = nb.find_ordered_nn(locs, m)
    coloring = nb.greedy_coloring(nn)
    Linv = O.vecchia_Linv([1.0, RANGE, 0.0], "exponential_isotropic", locs, nn)
    pd = O.precision_diag(Linv, nn)
    w = O.sparse_chol_solve(Linv, nn, rng.standard_normal(n))
    y = w + np.sqrt(TAU2) * rng.standard_normal(n)
    lm = np.arange(1, n + 1, dtype=np.int32)
    rs = O.residuals_sum(lm, n, y, np.zeros(n))
    field = w.copy()
    times = []
    for s in range(warmup + steps):
        z = rng.standard_normal(n)
        t0 = time.perf_counter()
        field = O.chromatic_sweep(Linv, nn, coloring, pd, np.ones(n), rs, 0.0, np.log(SIGMA2), np.log(TAU2), z, field, form=form)
        ll = O.ll_compressed_sparse_chol(Linv, field, nn, np.log(SIGMA2))
        times.append(time.perf_counter() - t0)
    assert np.isfinite(ll)
    return times[warmup:]


def oracle_steps_per_sec(n, m, steps, warmup, procs, form="reference", reordering="maxmin"):
    import multiprocessing as mp
    args = [(n, m, 100 + k, steps, warmup, form, reordering) for k in range(procs)]
    if procs == 1:
        res = [_oracle_chain_worker(args[0])]
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            res = pool.map(_oracle_chain_worker, args)
    per_chain = [len(t) / sum(t) for t in res]
    return float(sum(per_chain)), float(np.mean([np.mean(t) for t in res]) * 1e3)


def workload_string(n, m, covfun, reordering, n_gpus):
    base = f"U(0,1)^2, n={n}, m={m}, {covfun} range {RANGE}" + (f" nu {NU}" if covfun.startswith("matern") else "") + f", sigma2 {SIGMA2}, tau2 {TAU2}, reordering={reordering}"
    if n_gpus == 1:
        return "config3: " + base
    return f"one field sharded over {n_gpus} GPUs by spatial blocks ({n // n_gpus} sites per GPU): " + base


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, a.ref_procs))
    # bounded sample: the reference-form sweep costs K full mat-vecs, ~1 s/step/chain at n = 1M.  The reference's only
    # parallelism is one chain per core (mclapply): `procs` independent chains of the 1M-site problem, aggregate steps/s.
    n = a.sites_per_gpu if a.ref_n is None else a.ref_n
    steps = max(1, min(a.steps, 3))
    warmup = min(a.warmup, 1)
    value, ms = oracle_steps_per_sec(n, a.m, steps, warmup, procs, reordering=a.reordering)
    scale = n / a.sites_per_gpu
    n_total = a.sites_per_gpu * a.gpus if a.n is None else a.n
    line = {
        "impl": "reference", "metric": "gibbs_sweep_plus_vecchia_loglik_per_sec", "value": value * scale, "unit": "steps/s (1M-site blocks)",
        "n_gpus": a.gpus, "steps": steps, "warmup": warmup, "ms_per_step": ms / scale, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_string(n_total, a.m, a.covfun, a.reordering, a.gpus),
                   "step": "1 chromatic Gibbs sweep (reference form: one sparse mat-vec per colour, update_Gaussian.R:257-275) + 1 Vecchia log-lik",
                   "reference_parallelism": f"{procs} independent chains of a {n}-site field, one per host core (mclapply, update_Gaussian.R:25); "
                                            "the reference has no way to split one field over cores"},
        "cpu_baseline": {"value": value * scale, "unit": "steps/s (1M-site blocks)", "cores": procs, "kind": "port",
                         "sample": f"oracle restatement (not R/GpGp): {procs} independent chains (one per core, as mclapply does), "
                                   f"n={n}, {steps} steps each" + ("" if scale == 1 else f", scaled by n/{a.sites_per_gpu}")},
        "e2e": {"value": value * scale, "unit": "steps/s (1M-site blocks)", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# our arm, one GPU
# ---------------------------------------------------------------------------------------------------------------------
def run_single(a):
    import torch
    import nngp_b200 as nb
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the NNGP hot path has no CPU fallback)")
    local = 0
    torch.cuda.set_device(local)
    n, m = (a.sites_per_gpu if a.n is None else a.n), a.m
    cp = covparms(a.covfun, RANGE)
    rng, locs, nn, coloring, locs_match, t_setup = build_problem(n, m, seed=1, reordering=a.reordering)
    t0 = time.perf_counter()
    ctx = nb.NNGPContext(locs, nn, coloring, locs_match, a.covfun, device=local)
    t_setup["ctx_create_s"] = time.perf_counter() - t0
    assert ctx.factor_build(cp) == 0
    ctx.factor_commit()
    ctx.field_init(0.0, np.log(SIGMA2), rng.standard_normal(n))          # w ~ NNGP prior by a triangular solve
    w = ctx.field_get()
    y = w + np.sqrt(TAU2) * rng.standard_normal(n)
    ctx.obs_set(y)
    beta_0, ls, lnv = 0.0, float(np.log(SIGMA2)), float(np.log(TAU2))
    ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=1, seed=0)                  # sets the sweep parameters used by time_op

    # ---- device-resident timing: W warm-up steps, then exactly K steps, CUDA events on the library's stream ----
    warm = max(a.warmup, 3)
    ctx.time_op("sweep_loglik", reps=warm)
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = nb.launch_count()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ms_steps, launches_per_step = ctx.time_op("sweep_loglik", reps=a.steps)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    launches = nb.launch_count() - launches0
    total_ms = float(ms_steps.sum())
    value = a.steps / (total_ms * 1e-3)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, ctx.field_get(), ctx.loglik(0.0, ls))   # nngp_time_op's step takes its log-lik at beta_0 = 0
    # component timings (same stream, same events; >= 50 repetitions, median and min -- SURVEY.md 8d)
    reps = max(50, min(a.steps, 200))
    comp = {}
    for key, op in (("sweep", "gibbs_sweep"), ("loglik", "loglik"), ("factor_build", "factor_build"), ("spmv_plus_sptrsv", "sptrsv"),
                    ("spmv", "spmv"), ("accept_transpose_precision_diag", "commit")):
        ctx.time_op(op, reps=3)
        comp[key] = stats(ctx.time_op(op, reps=reps)[0])
    clocks = sampler.stop()
    fp64_gflops = nb.fp64_peak(local)

    # ---- end to end through the C ABI with host buffers: field in -> sweep -> field out, host field -> log-lik ----
    def e2e_loop(field_h, steps):
        ll = 0.0
        for _ in range(steps):
            ctx.field_set(field_h)                            # H2D 8n bytes
            ctx.gibbs_sweep(beta_0, ls, lnv, 1, seed=0)
            ctx.field_get(out=field_h)                        # D2H 8n bytes
            ll = ctx.loglik_host(field_h, ls)                 # H2D 8n bytes, D2H 2 scalars
        return ll

    def e2e_loop_fused(field_h, steps):
        """the same step through ONE call: the field goes up, sweep + log-lik run on it, the new field comes down (the four-call
        sequence sends the field over PCIe a second time for nngp_loglik_host)"""
        ll = 0.0
        for _ in range(steps):
            ll = ctx.sweep_loglik_host(field_h, beta_0, ls, lnv, 1, seed=0)   # H2D 8n bytes, D2H 8n bytes + 2 scalars
        return ll

    def timed_e2e(field_h, steps, loop=None):
        loop = loop or e2e_loop
        loop(field_h, 3)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ll = loop(field_h, steps)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        assert np.isfinite(ll)
        return steps / dt

    # ---- the full reference iteration (2 factor rebuilds, ancillary solve, 10 sweeps, ...) behind one call; iter_start = 0 is the
    # adaptive phase in which proposals ARE accepted (the accept branch -- transposition + precision_diag, field copy -- is in) ----
    var_y = float(np.var(y, ddof=1))
    chain_params = {"shape": [np.log(RANGE)] + ([0.0] if a.covfun.startswith("matern") else []), "beta_0": 0.0, "log_scale": ls, "log_noise_variance": lnv}
    n_chain_it, n_adapt = (50, 700) if not a.no_chain else (2, 2)
    # the adaptive phase (update_Gaussian.R:153-157,209-213) shrinks the proposal variances until proposals are accepted: at n = 1M
    # the posterior of the covariance parameters is so narrow that this takes several hundred iterations from logvar = -2
    adapted, _, _, _ = ctx.chain_run(chain_params, n_adapt, var_y, thin=0.0, n_chromatic=10, iter_start=0, chain_index=1, keep_field=False)
    chain_params_t = dict(chain_params, **{k: adapted[k] for k in ("beta_0", "log_scale", "log_noise_variance", "logvar_sufficient", "logvar_ancillary")},
                          shape=list(adapted["shape"]))
    t0 = time.perf_counter()
    _, _, _, acc = ctx.chain_run(chain_params_t, n_chain_it, var_y, thin=0.0, n_chromatic=10, iter_start=n_adapt, chain_index=1, keep_field=False)
    chain_it_per_s = n_chain_it / (time.perf_counter() - t0)
    chain_accepts = [int(acc[:, 0].sum()), int(acc[:, 1].sum())]
    ctx.field_set(w)
    ctx.factor_build(cp)
    ctx.factor_commit()

    # ---- several chains per GPU (the reference's default is n_chains = 3, advanced concurrently): a sweep is a chain of
    # latency-bound colour stages, so co-scheduled chains fill each other's gaps ----
    multi = None
    if not a.no_multichain:
        others = []
        try:
            for k in range(2):
                c2 = nb.NNGPContext(locs, nn, coloring, locs_match, a.covfun, device=local)
                c2.factor_build(cp)
                c2.factor_commit()
                c2.field_set(w)
                c2.obs_set(y)
                c2.gibbs_sweep(beta_0, ls, lnv, 1, seed=k + 1)
                others.append(c2)
            r = 100
            one = nb.time_op_group([ctx], "gibbs_sweep", reps=r)
            two = nb.time_op_group([ctx, others[0]], "gibbs_sweep", reps=r)
            three = nb.time_op_group([ctx] + others, "gibbs_sweep", reps=r)
            three_step = nb.time_op_group([ctx] + others, "sweep_loglik", reps=r)
            t0 = time.perf_counter()
            res = nb.chains_run([ctx] + others, [chain_params] * 3, 20, var_y, thin=0.0, n_chromatic=10, iter_start=0,
                                chain_indices=[1, 2, 3], keep_field=False)
            chains3 = 3 * 20 / (time.perf_counter() - t0)
            multi = {"chains_per_gpu": 3, "sweeps_per_sec_1_chain": 1e3 * r / one, "sweeps_per_sec_2_chains": 2e3 * r / two,
                     "sweeps_per_sec_3_chains": 3e3 * r / three, "steps_per_sec_3_chains": 3e3 * r / three_step,
                     "chain_iterations_per_sec_3_chains": chains3,
                     "what": "aggregate over chains co-scheduled on ONE GPU (one context, stream and host thread per chain; nngp_time_op_group / nngp_chains_run)"}
            del res
        finally:
            for c2 in others:
                c2.close()
        ctx.field_set(w)
        ctx.factor_build(cp)
        ctx.factor_commit()

    # ---- mcmc_nngp_predict_field at n new sites (joint context over 2n sites; only the new rows are solved) ----
    pred_per_s = None
    if not a.no_predict:
        new_locs = np.random.default_rng(99).random((n, 2))
        joint = np.vstack([locs, new_locs])
        nn_j = nb.find_ordered_nn(joint, m)
        with nb.NNGPContext(joint, nn_j, np.zeros(2 * n, dtype=np.int32), np.zeros(0, dtype=np.int32), a.covfun, device=local) as pctx:
            pctx.factor_build(cp)
            zp = np.random.default_rng(5).standard_normal(n)
            pctx.predict_sample(n, w, beta_0, ls, zp)
            t0 = time.perf_counter()
            for _ in range(5):
                pctx.predict_sample(n, w, beta_0, ls, zp)
            pred_per_s = 5 / (time.perf_counter() - t0)

    e2e_steps = min(a.steps, 200)
    pinned = nb.PinnedArray(n)
    pinned.array[:] = ctx.field_get()
    e2e_four_calls = timed_e2e(pinned.array, e2e_steps)
    e2e_value = timed_e2e(pinned.array, e2e_steps, e2e_loop_fused)
    e2e_pageable = timed_e2e(ctx.field_get(), e2e_steps, e2e_loop_fused)
    pinned.free()

    # ---- the other ordering (the reference default is maxmin, initialize.R:29; "random" is its other option, :30) ----
    other = None
    if not a.no_other_ordering:
        oname = "random" if a.reordering == "maxmin" else "maxmin"
        rng2, locs2, nn2, col2, lm2, t2 = build_problem(n, m, seed=1, reordering=oname)
        with nb.NNGPContext(locs2, nn2, col2, lm2, a.covfun, device=local) as c2:
            c2.factor_build(cp)
            c2.factor_commit()
            c2.field_init(0.0, ls, rng2.standard_normal(n))
            w2 = c2.field_get()
            c2.obs_set(w2 + np.sqrt(TAU2) * rng2.standard_normal(n))
            c2.gibbs_sweep(beta_0, ls, lnv, 1, seed=0)
            c2.time_op("sweep_loglik", reps=3)
            o = {k: stats(c2.time_op(op, reps=reps)[0]) for k, op in (("sweep", "gibbs_sweep"), ("loglik", "loglik"), ("step", "sweep_loglik"),
                                                                       ("factor_build", "factor_build"), ("spmv_plus_sptrsv", "sptrsv"))}
            other = {"reordering": oname, "n_colors": c2.n_colors, "solve_levels": c2.n_levels, "longest_column": c2.max_col,
                     "steps_per_sec": 1e3 / o["step"]["median"], "ms": o, "setup": t2}

    peak, peak_src = measured_peaks()
    ab = algorithmic(n, m)
    traffic, traffic_meta = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and n == 1_000_000 and m == 10 and a.covfun == "exponential_isotropic":
        with open(tpath) as f:
            tj = json.load(f)
        traffic = tj["bytes"].get("gibbs_sweep_full")
        traffic_meta = {k: tj.get(k) for k in ("git_sha", "when", "how") if k in tj}
    sweep_ms = comp["sweep"]["median"]
    achieved = ab["gibbs_sweep"] / (sweep_ms * 1e-3) / 1e9
    fac_ms = comp["factor_build"]["median"]
    line = {
        "metric": "gibbs_sweep_plus_vecchia_loglik_per_sec", "value": value, "unit": "steps/s (1M-site blocks)", "n_gpus": 1, "steps": a.steps,
        "warmup": warm, "ms_per_step": total_ms / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_string(n, m, a.covfun, a.reordering, 1),
                   "step": "1 chromatic Gibbs sweep (all colours, Philox normals) + 1 Vecchia log-lik evaluation",
                   "parallelism": "single GPU",
                   "l2": "working set (factor + indices + transpose map, ~0.4 GB) exceeds the 126 MB L2; no explicit flush",
                   "n_colors": ctx.n_colors, "solve_levels": ctx.n_levels, "longest_column": ctx.max_col, "layout": ctx.layout, "setup": t_setup},
        "gibbs_sweeps_per_sec": 1e3 / sweep_ms, "loglik_evals_per_sec": 1e3 / comp["loglik"]["median"],
        "factor_builds_per_sec": 1e3 / fac_ms,
        "chain_iterations_per_sec": chain_it_per_s, "chain_accepts_ancillary_sufficient": chain_accepts,
        "chain_iteration": f"nngp_chain_run, {n_chain_it} iterations after {n_adapt} adaptive ones (proposal variances tuned, proposals are accepted: accept branch = transposition + precision_diag + field copy in the number): reference loop "
                           "update_Gaussian.R:101-314 (2 factor rebuilds, ancillary SpMV+SpTRSV, 2 log-liks, beta_0, 10 sweeps, noise steps), host wall clock",
        "multi_chain": multi,
        "predicted_field_samples_per_sec": pred_per_s,
        "predicted_field_sample": f"nngp_predict_sample through the C ABI with host buffers: one stored sample conditionally simulated at {n} new sites",
        "other_ordering": other,
        "ms": dict(comp, wall_timed_region=wall * 1e3),
        "roofline": {"bound": "hbm", "kernel": "gibbs_tile2_kernel (the K colour launches of one sweep, PDL-chained, replayed from one CUDA graph; 6 CTAs/SM build for colours that would not fit one wave at 5)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "frac_dram": (traffic / (sweep_ms * 1e-3) / 1e9 / peak) if traffic else None,
                     "traffic_source": "OFFLINE: profiles/traffic.json (ncu dram__bytes_read.sum + dram__bytes_write.sum summed over the colour launches of one warm sweep, "
                                       "--cache-control none); not measured in this run", "traffic_meta": traffic_meta,
                     "algorithmic_bytes_per_sweep": ab["gibbs_sweep"], "timing": "median of CUDA-event times, %d repetitions" % comp["sweep"]["reps"],
                     "loglik": {"achieved": ab["loglik"] / (comp["loglik"]["median"] * 1e-3) / 1e9, "frac": ab["loglik"] / (comp["loglik"]["median"] * 1e-3) / 1e9 / peak},
                     "factor_build": {"bound": "fp64", "flops_per_build": ab["factor_build_flops"], "achieved_gflops": ab["factor_build_flops"] / (fac_ms * 1e-3) / 1e9,
                                      "peak_gflops": fp64_gflops, "frac": ab["factor_build_flops"] / (fac_ms * 1e-3) / 1e9 / fp64_gflops if fp64_gflops else None,
                                      "peak_source": "nngp_fp64_peak: dependent-free DFMA chains on every SM, this run",
                                      "GBps": ab["factor_build"] / (fac_ms * 1e-3) / 1e9}},
        "e2e": {"value": e2e_value, "unit": "steps/s (1M-site blocks)", "h2d_bytes_per_step": 8 * n + 64, "d2h_bytes_per_step": 8 * n + 16,
                "what": "nngp_sweep_loglik_host: every step the field is uploaded from a pinned host buffer (nngp_host_alloc), swept once, its Vecchia "
                        "log-lik taken, and the new field + log-lik downloaded",
                "steps": e2e_steps, "pcie_GBps": e2e_value * (16 * n) / 1e9, "pageable_numpy_value": e2e_pageable,
                "four_calls_value": e2e_four_calls,
                "four_calls": "round-1 definition: nngp_field_set + nngp_gibbs_sweep + nngp_field_get + nngp_loglik_host (24 n bytes per step: the field "
                              "crosses PCIe a second time for the host-side log-lik call)"},
        "gpu_launches": int(launches), "launches_per_step": int(launches_per_step), "clocks": clocks, "git_sha": git_sha(),
    }
    if not a.no_cpu_baseline:
        v, ms = oracle_steps_per_sec(n, m, steps=2, warmup=0, procs=1, reordering=a.reordering)
        v2, ms2 = oracle_steps_per_sec(n, m, steps=2, warmup=0, procs=1, form="residual", reordering=a.reordering)
        line["cpu_baseline"] = {"value": v, "unit": "steps/s (1M-site blocks)", "cores": 1, "kind": "port",
                                "sample": f"oracle restatement (not R/GpGp), 1 thread, full n={n}: 2 steps of reference-form sweep (one mat-vec per colour) + log-lik",
                                "residual_form_value": v2,
                                "residual_form": "the same oracle with the O(n m) residual-maintained sweep the GPU kernel uses: separates the algorithmic gain from the hardware gain"}
    print(json.dumps(line), flush=True)
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# our arm, N GPUs: one field sharded by spatial blocks
# ---------------------------------------------------------------------------------------------------------------------
def shared_problem(dist, rank, n, m, seed, reordering, tag):
    """the (replicated) host-side structure is built once, by rank 0 with all host cores, and shared through /dev/shm"""
    shm = f"/dev/shm/nngp_bench_{os.environ.get('MASTER_PORT', '0')}_{tag}"
    t = None
    if rank == 0:
        import nngp_b200 as nb
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
        nb.set_host_threads(0)            # torchrun exports OMP_NUM_THREADS=1: rank 0 builds the shared structure with every core
        _, locs, nn, coloring, _, t = build_problem(n, m, seed=seed, reordering=reordering)
        np.save(shm + "_locs.npy", np.asfortranarray(locs))
        np.save(shm + "_nn.npy", np.asfortranarray(nn))
        np.save(shm + "_col.npy", coloring)
        del locs, nn, coloring
    dist.barrier()
    locs = np.load(shm + "_locs.npy", mmap_mode="r")
    nn = np.load(shm + "_nn.npy", mmap_mode="r")
    coloring = np.load(shm + "_col.npy", mmap_mode="r")
    dist.barrier()
    if rank == 0:
        for suffix in ("_locs.npy", "_nn.npy", "_col.npy"):
            os.remove(shm + suffix)        # the mappings stay valid
    return locs, nn, coloring, np.arange(1, n + 1, dtype=np.int32), t


def run_sharded(a):
    import torch
    import torch.distributed as dist
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if world < 2:
        raise SystemExit("--mode sharded needs torchrun with at least 2 ranks")
    numa = pin_to_gpu_numa(local)
    if rank == 0:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))                    # rank 0 builds the shared structure with every core
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)               # torchrun pins it to 1; the library is not loaded yet
    import nngp_b200 as nb
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n, m = (a.sites_per_gpu * world if a.n is None else a.n), a.m
    cp = covparms(a.covfun, RANGE)
    beta_0, ls, lnv = 0.0, float(np.log(SIGMA2)), float(np.log(TAU2))

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def make_field(n_, tag, transport):
        t0 = time.perf_counter()
        locs, nn, coloring, locs_match, t_host = shared_problem(dist, rank, n_, m, 1, a.reordering, tag)
        t1 = time.perf_counter()
        ctx, plan = nb.create_sharded_distributed(locs, nn, coloring, locs_match, a.covfun, local, dist, transport=transport)
        t2 = time.perf_counter()
        assert ctx.factor_build(cp) == 0
        ctx.factor_commit()
        w = np.random.default_rng(7).standard_normal(n_) * 0.5               # any field will do for throughput; same on all ranks
        y = w + np.sqrt(TAU2) * np.random.default_rng(8).standard_normal(n_)
        ctx.field_set(w[plan["local_sites"]])
        ctx.obs_set(y[plan["obs_index"]])
        ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=1, seed=1)
        return ctx, plan, {"host_structure_s": t1 - t0, "plan_and_ctx_s": t2 - t1, "host": t_host}, w[plan["local_sites"]]

    ctx, plan, t_setup, w_local = make_field(n, "weak", a.transport)
    warm = max(a.warmup, 3)
    ctx.time_op("sweep_loglik", reps=warm)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = nb.launch_count()
    barrier()
    ms_steps, launches_per_step = ctx.time_op("sweep_loglik", reps=a.steps)
    barrier()
    launches = nb.launch_count() - launches0
    reps = max(50, min(a.steps, 200))
    comp = {}
    for key, op in (("sweep", "gibbs_sweep"), ("loglik", "loglik"), ("factor_build", "factor_build")):
        ctx.time_op(op, reps=3)
        barrier()
        comp[key] = ctx.time_op(op, reps=reps)[0]
    # ---- a whole chain on the sharded field (reference loop update_Gaussian.R:101-314: 2 factor rebuilds, ancillary SpMV + sharded
    # triangular solve, 2 log-liks, beta_0, 10 sweeps, noise steps), every rank on its block, decisions on all-reduced scalars ----
    chain_it_per_s, solve_ms = None, None
    if a.transport == "p2p" and not a.no_chain:
        yv = np.random.default_rng(8).standard_normal(8)   # (var_y only has to be the same on every rank)
        var_y = float(1.0 + TAU2 + 0.0 * yv.sum())
        chain_params = {"shape": [np.log(RANGE)] + ([0.0] if a.covfun.startswith("matern") else []), "beta_0": 0.0, "log_scale": ls, "log_noise_variance": lnv}
        ctx.chain_run(chain_params, 2, var_y, thin=0.0, n_chromatic=10, iter_start=5000, chain_index=1, keep_field=False)
        n_it = 10
        barrier()
        t0 = time.perf_counter()
        ctx.chain_run(chain_params, n_it, var_y, thin=0.0, n_chromatic=10, iter_start=5000, chain_index=1, keep_field=False)
        barrier()
        chain_it_per_s = n_it / (time.perf_counter() - t0)
        ctx.field_set(w_local)
        assert ctx.factor_build(cp) == 0
        ctx.factor_commit()
        ctx.gibbs_sweep(beta_0, ls, lnv, n_sweeps=1, seed=1)
        ctx.time_op("sptrsv", reps=3)
        barrier()
        solve_ms = ctx.time_op("sptrsv", reps=20)[0]
    clocks = sampler.stop() if rank == 0 else None

    def maxred(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def sumred(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    total_ms, sweep_med, sweep_min, ll_med, ll_min, fac_med = maxred([float(ms_steps.sum()), float(np.median(comp["sweep"])), float(comp["sweep"].min()),
                                                                       float(np.median(comp["loglik"])), float(comp["loglik"].min()), float(np.median(comp["factor_build"]))])
    if solve_ms is not None:
        (solve_med,) = maxred([float(np.median(solve_ms))])
        (chain_it_per_s,) = [-v for v in maxred([-chain_it_per_s])]
    sp = np.asarray(plan["send_ptr"])
    pairs = int(((np.diff(sp).reshape(-1, world)) > 0).sum())
    halo_vals, n_ghost, n_local, pair_sum = sumred([float(sp[-1]), float(plan["n_ghost"]), float(plan["local_sites"].size), float(pairs)])

    # ---- end to end through the C ABI with pinned host buffers, every rank its block ----
    nl = plan["local_sites"].size
    pinned = nb.PinnedArray(nl)
    pinned.array[:] = w_local

    def e2e_loop(steps):
        ll = 0.0
        for _ in range(steps):
            ll = ctx.sweep_loglik_host(pinned.array, beta_0, ls, lnv, 1, seed=1)
        return ll

    e2e_steps = min(a.steps, 200)
    e2e_loop(3)
    barrier()
    t0 = time.perf_counter()
    ll = e2e_loop(e2e_steps)
    barrier()
    (e2e_dt,) = maxred([time.perf_counter() - t0])
    assert np.isfinite(ll)
    pinned.free()
    blocks = n / a.sites_per_gpu
    line = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        ab = algorithmic(n, m)
        achieved = ab["gibbs_sweep"] / (sweep_med * 1e-3) / 1e9
        steps_per_s = a.steps / (total_ms * 1e-3)
        line = {
            "metric": "gibbs_sweep_plus_vecchia_loglik_per_sec", "value": blocks * steps_per_s, "unit": "steps/s (1M-site blocks)", "n_gpus": world,
            "steps": a.steps, "warmup": warm, "ms_per_step": total_ms / a.steps, "higher_is_better": True, "scaling": "weak" if a.n is None else "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_string(n, m, a.covfun, a.reordering, world),
                       "step": "1 chromatic Gibbs sweep of the WHOLE field (boundary values pushed to the peers' ghost slots from inside the sweep kernel) + 1 Vecchia log-lik (scalar all-reduce)",
                       "value_definition": f"steps/s of the {n}-site field x {blocks:g} (1M-site blocks), so that value_N / (N value_1) is the weak-scaling efficiency",
                       "parallelism": f"field sharded over {world} GPUs by spatial blocks", "transport": a.transport, "n_colors": ctx.n_colors,
                       "halo_values_per_sweep": int(halo_vals), "halo_colour_peer_pairs": int(pair_sum), "ghost_sites_total": int(n_ghost),
                       "local_sites_total": int(n_local), "setup": t_setup, "numa_cpulist_rank0": numa,
                       "l2": "per-GPU working set (~0.4 GB per 1M sites) exceeds the 126 MB L2; no explicit flush"},
            "field_steps_per_sec": steps_per_s,
            "gibbs_sweeps_per_sec": 1e3 / sweep_med, "loglik_evals_per_sec": 1e3 / ll_med, "factor_builds_per_sec": 1e3 / fac_med,
            "ms": {"sweep": {"median": sweep_med, "min": sweep_min, "reps": reps}, "loglik": {"median": ll_med, "min": ll_min, "reps": reps},
                   "factor_build": {"median": fac_med, "reps": reps}},
            "chain_iterations_per_sec": chain_it_per_s,
            "chain_iteration": "nngp_chain_run on the sharded field: reference loop update_Gaussian.R:101-314 (2 factor rebuilds, ancillary SpMV + sharded triangular solve, 2 log-liks, beta_0, 10 sweeps, noise steps), every rank on its block, host wall clock",
            "spmv_plus_sptrsv_ms": solve_med if solve_ms is not None else None,
            "halo_us_per_colour_over_1gpu_block": None,
            "roofline": {"bound": "hbm", "kernel": "gibbs_tile2_kernel<SHARD> (whole-field sweep: K colour launches per rank, halo push / apply fused in; max over ranks)",
                         "achieved": achieved, "peak": peak * world, "unit": "GB/s", "frac": achieved / (peak * world), "traffic": None,
                         "peak_source": peak_src + f" x {world} GPUs", "algorithmic_bytes_per_sweep": ab["gibbs_sweep"],
                         "loglik": {"achieved": ab["loglik"] / (ll_med * 1e-3) / 1e9, "frac": ab["loglik"] / (ll_med * 1e-3) / 1e9 / (peak * world)}},
            "e2e": {"value": blocks * e2e_steps / e2e_dt, "unit": "steps/s (1M-site blocks)", "h2d_bytes_per_step": int(8 * n_local + 64 * world),
                    "d2h_bytes_per_step": int(8 * n_local + 16 * world), "steps": e2e_steps,
                    "what": "every rank: nngp_sweep_loglik_host on its block (owned + ghost sites): field up from a pinned host buffer, one sweep of the whole "
                            "field (halo exchange inside), all-reduced Vecchia log-lik, new field + log-lik down",
                    "pcie_GBps_per_rank": (16 * n_local / world) * e2e_steps / e2e_dt / 1e9},
            "gpu_launches": int(launches), "launches_per_step": int(launches_per_step), "clocks": clocks, "git_sha": git_sha(),
        }
    ctx.close()
    del ctx

    # ---- extras: the n = 1M field of the BASELINE metric split over the N GPUs (strong scaling), and N independent replicas ----
    if not a.no_extras and a.n is None:
        n1 = a.sites_per_gpu
        c1, p1, _, _ = make_field(n1, "strong", a.transport)
        c1.time_op("sweep_loglik", reps=warm)
        barrier()
        ms1, _ = c1.time_op("sweep_loglik", reps=min(a.steps, 300))
        barrier()
        sw1, _ = c1.time_op("gibbs_sweep", reps=50)
        (tot1, sw1m) = maxred([float(ms1.sum()), float(np.median(sw1))])
        c1.close()
        # replicas: every rank sweeps its own copy of the 1M-site field, no data-path collective
        locs, nn, coloring, locs_match, _ = shared_problem(dist, rank, n1, m, 1, a.reordering, "rep")
        with nb.NNGPContext(np.asarray(locs), np.asarray(nn), np.asarray(coloring), locs_match, a.covfun, device=local) as cr:
            cr.factor_build(cp)
            cr.factor_commit()
            wr = np.random.default_rng(7 + rank).standard_normal(n1) * 0.5
            cr.field_set(wr)
            cr.obs_set(wr + np.sqrt(TAU2) * np.random.default_rng(8).standard_normal(n1))
            cr.gibbs_sweep(beta_0, ls, lnv, 1, seed=rank)
            cr.time_op("sweep_loglik", reps=warm)
            barrier()
            msr, _ = cr.time_op("sweep_loglik", reps=min(a.steps, 300))
            barrier()
            (totr,) = maxred([float(msr.sum())])
        if rank == 0:
            line["strong_scaling_n1M"] = {"steps_per_sec": min(a.steps, 300) / (tot1 * 1e-3), "sweep_ms_median": sw1m,
                                          "what": f"the n = {n1} field of the BASELINE metric sharded over {world} GPUs (latency-bound: {ctx_colours(line)} dependent colour stages)"}
            line["replicas"] = {"steps_per_sec": world * min(a.steps, 300) / (totr * 1e-3),
                                "what": f"{world} independent chains of the n = {n1} field, one per GPU, no data-path collective (BASELINE config 5 / the reference's own parallelism)"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    dist.destroy_process_group()


def ctx_colours(line):
    return line["config"]["n_colors"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sites", "--n", dest="n", type=int, default=None, help="total sites (default: --sites-per-gpu x GPUs)")
    ap.add_argument("--sites-per-gpu", type=int, default=1_000_000)
    ap.add_argument("--nbrs", "--m", dest="m", type=int, default=10)
    ap.add_argument("--covfun", default="exponential_isotropic", choices=["exponential_isotropic", "matern_isotropic"])
    ap.add_argument("--reordering", default="maxmin", choices=["random", "maxmin"], help="maxmin = the reference default (initialize.R:29)")
    ap.add_argument("--ref-n", type=int, default=None, help="reference arm: run on a smaller n and scale (bounded sample)")
    ap.add_argument("--ref-procs", type=int, default=32, help="reference arm: at most this many independent chains (one per host core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-predict", action="store_true")
    ap.add_argument("--no-multichain", action="store_true")
    ap.add_argument("--no-other-ordering", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-chain", action="store_true")
    ap.add_argument("--mode", default="auto", choices=["auto", "single", "sharded"])
    ap.add_argument("--transport", default="p2p", choices=["p2p", "nccl"], help="sharded mode: halo transport")
    ap.add_argument("--range", dest="range_", type=float, default=None, help="covariance range (default 0.05; BASELINE config 4 is run with 0.02)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="single GPU: write the field and log-lik of the last timed step as DIR/field.npy (DIR/field_sample.npy, a seeded "
                         f"sample of {DUMP_MAX_FIELD} sites, above that size) and DIR/loglik.npy, float64")
    a = ap.parse_args()
    if a.range_ is not None:
        global RANGE
        RANGE = a.range_
    world = int(os.environ.get("WORLD_SIZE", "1"))
    sharded = a.mode == "sharded" or (a.mode == "auto" and world > 1)
    if a.dump_outputs and (a.impl == "reference" or sharded):
        ap.error("--dump-outputs is implemented for the single-GPU run of the library (--impl ours, one rank)")
    if a.impl == "reference":
        run_reference(a)
    elif sharded:
        run_sharded(a)
    else:
        run_single(a)


if __name__ == "__main__":
    main()
