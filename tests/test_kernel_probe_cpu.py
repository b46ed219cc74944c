"""The kernel probe study on the CPU: the oracle's factor rows through the probe problems of tests/test_gpu_kernel_accuracy.py meet
the same bounds against the 50-digit reference, and that reference is what its generator writes."""
import os
import sys

import numpy as np
import pytest

from oracle import oracle as O
from problems import PROBE_REFERENCE, load_probe_reference, make_probe_problem, probe_covparms, probe_failures

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def libstdcxx_temme_cancels(nu, x):
    """std::cyl_bessel_k (the oracle's K_nu) forms Temme's coefficient (1/Gamma(1-mu) - 1/Gamma(1+mu)) / (2 mu), mu = nu - round(nu),
    as a difference for |mu| > eps: within 1e-9 of an integer order it loses ~log10(eps/|mu|) digits on the series side (x < 2),
    8e-7 relative at nu = 1 - 1e-9, x = 2 - ulp.  The device sums the Taylor series of 1/Gamma instead (device_math.cuh) and is
    held to the full bound there by tests/test_gpu_kernel_accuracy.py."""
    mu = abs(nu - round(nu)) if nu is not None else 1.0
    return (0.0 < mu < 1e-6) & (x > 0.0) & (x < 2.0)


@pytest.mark.parametrize("m", [1, 5, 20, 31])
def test_oracle_meets_the_probe_bounds(m):
    ref = load_probe_reference()
    P = make_probe_problem(m, 2, ref["x"])
    fails, worst = [], {}
    for fam in ref["families"]:
        skip = libstdcxx_temme_cancels(fam["nu"], ref["x"])
        for s2 in (1.0, 2.5):
            for tau in (0.0, 0.5):
                L = O.vecchia_Linv(probe_covparms(fam["nu"], s2, tau), fam["covfun"], P["locs"], P["NNarray"])
                if tau > 0:                                      # (tau = 0: the block of x = 0 is singular)
                    assert np.all(L[m:, 2:] == 0.0)              # the far anchors decouple exactly
                fails += probe_failures(L, m, ref, fam, s2, tau, f"oracle m={m}", worst, skip)
    print("worst relative error of rho per regime:", {k: f"{v:.2e}" for k, v in sorted(worst.items())})
    assert not fails, "\n".join(fails[:40])


def test_probe_reference_regenerates_bit_for_bit():
    pytest.importorskip("mpmath")
    sys.path.insert(0, GOLDEN)
    try:
        import make_kernel_probe_reference as G
    finally:
        sys.path.remove(GOLDEN)
    with open(PROBE_REFERENCE) as f:
        assert f.read() == G.dumps(G.reference())
