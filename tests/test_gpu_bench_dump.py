"""bench.py --dump-outputs: the field and Vecchia log-lik of the last timed step, identical from run to run with the same arguments."""
import json

import numpy as np
import pytest

from test_bench_contract_cpu import run_bench

pytestmark = pytest.mark.gpu


def test_dump_outputs_writes_the_last_timed_step_and_repeats(tmp_path):
    import bench
    from oracle import oracle as O
    n, m = 20000, 10
    small = ("--n", str(n), "--steps", "7", "--warmup", "3", "--no-cpu-baseline", "--no-predict", "--no-multichain", "--no-other-ordering", "--no-chain")
    dumps = []
    for k in range(2):
        d = tmp_path / f"run{k}"
        r = run_bench(*small, "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 7
        assert sorted(p.name for p in d.iterdir()) == ["field.npy", "loglik.npy"]
        field, ll = np.load(d / "field.npy"), np.load(d / "loglik.npy")
        assert field.dtype == np.float64 and field.shape == (n,) and np.all(np.isfinite(field))
        assert ll.dtype == np.float64 and ll.shape == (1,)
        dumps.append((field, ll))
    np.testing.assert_allclose(dumps[1][0], dumps[0][0], rtol=1e-12, atol=0)
    np.testing.assert_allclose(dumps[1][1], dumps[0][1], rtol=1e-12, atol=0)
    # the log-lik written is the one of the field written (bench's problem: seed 1, maxmin order, sigma^2 = 1)
    _, locs, nn, _, _, _ = bench.build_problem(n, m, seed=1, reordering="maxmin")
    Linv = O.vecchia_Linv(bench.covparms("exponential_isotropic", bench.RANGE), "exponential_isotropic", locs, nn)
    ll_o = O.ll_compressed_sparse_chol(Linv, dumps[0][0], nn, np.log(bench.SIGMA2))
    assert abs(dumps[0][1][0] - ll_o) < 1e-10 * abs(ll_o)
