"""Times the two halves of bench.py's flagship step (config 3: n = 1M, m = 10, exponential, max-min order): time_op's sweep alone and
its step (sweep + Vecchia log-lik), in rounds, CUDA events per repetition.  step - sweep is what the log-lik adds to a step.  --root
names the source tree whose library is loaded (default: this one), so that two builds can be run one after the other and compared.
Development aid; not part of the bench contract.

    python scripts/step_tail_time.py [--root DIR] [--rounds 5] [--reps 1000] [--n 1000000]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--reps", type=int, default=1000)
ap.add_argument("--n", type=int, default=1_000_000)
ap.add_argument("--label", default="")
a = ap.parse_args()
sys.path.insert(0, os.path.abspath(a.root))
import bench  # noqa: E402
import nngp_b200 as nb  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip() or "nvidia-smi gave no answer"
    except Exception as e:   # the numbers below still stand; say what is missing
        return f"nvidia-smi unavailable ({e})"


def main():
    if nb.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    print(f"{a.label} card (name, power limit, SM clock, max SM clock): {card()}", flush=True)
    rng, locs, nn, coloring, locs_match, _ = bench.build_problem(a.n, 10, seed=1, reordering="maxmin")
    ctx = nb.NNGPContext(locs, nn, coloring, locs_match, "exponential_isotropic")
    assert ctx.factor_build(bench.covparms("exponential_isotropic", bench.RANGE)) == 0
    ctx.factor_commit()
    ctx.field_init(0.0, np.log(bench.SIGMA2), rng.standard_normal(a.n))
    ctx.obs_set(ctx.field_get() + np.sqrt(bench.TAU2) * rng.standard_normal(a.n))
    ls = float(np.log(bench.SIGMA2))
    ctx.gibbs_sweep(0.0, ls, float(np.log(bench.TAU2)), n_sweeps=1, seed=0)   # the sweep parameters time_op uses, as in bench.py
    for op in ("gibbs_sweep", "sweep_loglik"):
        ctx.time_op(op, reps=50)
    rows = []
    for r in range(a.rounds):
        sw, _ = ctx.time_op("gibbs_sweep", reps=a.reps)
        st, launches = ctx.time_op("sweep_loglik", reps=a.reps)
        row = dict(round=r, sweep_us=1e3 * float(np.median(sw)), step_us=1e3 * float(np.median(st)), launches_per_step=launches)
        row["step_minus_sweep_us"] = row["step_us"] - row["sweep_us"]
        rows.append(row)
        print(f"{a.label} round {r}: sweep median {row['sweep_us']:.2f} us, step median {row['step_us']:.2f} us, "
              f"step - sweep {row['step_minus_sweep_us']:.2f} us, {launches} launches/step", flush=True)
    summary = {k: float(np.median([x[k] for x in rows])) for k in ("sweep_us", "step_us", "step_minus_sweep_us")}
    summary["step_spread_us"] = max(x["step_us"] for x in rows) - min(x["step_us"] for x in rows)
    summary["sweep_spread_us"] = max(x["sweep_us"] for x in rows) - min(x["sweep_us"] for x in rows)
    summary["loglik_after_last_round"] = ctx.loglik(0.0, ls)
    print(f"{a.label} summary {json.dumps(summary)}", flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
