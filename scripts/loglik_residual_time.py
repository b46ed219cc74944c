"""Times one step of bench.py's flagship workload (config 3: one sweep + one Vecchia log-lik, n = 1M, m = 10, exponential, max-min
order) with the log-lik taken from the sweep's residual (loglik_from_residual = 1) and with the full pass (0), alternating the two
in one process so that both see the same card, clocks and neighbours.  Development aid; not part of the bench contract.

    python scripts/loglik_residual_time.py [--rounds 5] [--reps 1000] [--n 1000000]
"""
import argparse
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import nngp_b200 as nb  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip() or "nvidia-smi gave no answer"
    except Exception as e:   # the numbers below still stand; say what is missing
        return f"nvidia-smi unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=1000)
    ap.add_argument("--n", type=int, default=1_000_000)
    a = ap.parse_args()
    if nb.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    print(f"card (name, power limit, max SM clock): {card()}", flush=True)
    rng, locs, nn, coloring, locs_match, _ = bench.build_problem(a.n, 10, seed=1, reordering="maxmin")
    ctx = nb.NNGPContext(locs, nn, coloring, locs_match, "exponential_isotropic")
    assert ctx.factor_build(bench.covparms("exponential_isotropic", bench.RANGE)) == 0
    ctx.factor_commit()
    ctx.field_init(0.0, np.log(bench.SIGMA2), rng.standard_normal(a.n))
    ctx.obs_set(ctx.field_get() + np.sqrt(bench.TAU2) * rng.standard_normal(a.n))
    ls = float(np.log(bench.SIGMA2))
    ctx.gibbs_sweep(0.0, ls, float(np.log(bench.TAU2)), n_sweeps=1, seed=0)   # the sweep parameters time_op uses, as in bench.py
    for opt in (0, 1):   # warm both paths
        ctx.set_option("loglik_from_residual", opt)
        ctx.time_op("sweep_loglik", reps=20)
    print(f"n={a.n}, m=10, maxmin order, {a.reps} steps per round (one sweep + one log-lik each), CUDA events per step", flush=True)
    per = {0: [], 1: []}
    for r in range(a.rounds):
        for opt in (0, 1):
            ctx.set_option("loglik_from_residual", opt)
            ms, launches = ctx.time_op("sweep_loglik", reps=a.reps)
            med, mn = float(np.median(ms)), float(ms.min())
            per[opt].append(med)
            print(f"round {r} option {opt} ({'residual' if opt else 'full pass'}): median {1e3 * med:.2f} us, min {1e3 * mn:.2f} us, "
                  f"{launches} launches/step, {1e3 / med:.0f} steps/s", flush=True)
    for opt in (0, 1):
        v = np.array(per[opt])
        print(f"option {opt}: median over rounds {1e3 * np.median(v):.2f} us/step, spread of round medians "
              f"{1e3 * (v.max() - v.min()):.2f} us ({100 * (v.max() - v.min()) / np.median(v):.2f} %)")
    gain = np.median(per[0]) / np.median(per[1]) - 1.0
    print(f"steps/s, residual over full pass: {100 * gain:+.1f} %")
    # the same state, both ways: after the last timed round (option 1) r is current
    ll_r = ctx.loglik(0.0, ls)
    ctx.set_option("loglik_from_residual", 0)
    ll_f = ctx.loglik(0.0, ls)
    print(f"log-lik after the last round: residual {ll_r!r}, full pass {ll_f!r}, relative difference {abs(ll_r - ll_f) / abs(ll_f):.3g}")
    ctx.close()


if __name__ == "__main__":
    main()
