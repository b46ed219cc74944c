"""The device's covariance kernel values against 50-digit arithmetic, read off factor rows of probe problems (tests/problems.py:
make_probe_problem): every kernel instantiation of the factor build, the exponential family and GpGp's Matern over the smoothness
range (0, 1.5) the reference's transforms reach, at distances on and around every switch of the device's Matern evaluation (exact
K_nu, global table, shared-memory table, e^x-scaled octaves; Temme / continued fraction at x = 2), with and without a nugget, at unit
and non-unit variance (the table bakes the variance into its coefficients), with the table and with the direct K_nu."""
import numpy as np
import pytest

import nngp_b200 as nb
from problems import load_probe_reference, make_probe_problem, probe_covparms, probe_failures

pytestmark = pytest.mark.gpu


def factor_kernel(m, dt, factor_variant):
    """the instantiation launch_factor (csrc/nngp_b200.cu) selects"""
    M = m + 1
    if M in (6, 11) and dt in (2, 3):
        return f"reg<{M},{dt}>"
    if M == 21 and dt in (2, 3) and factor_variant == 1:
        return f"warp<21,{dt}>"
    if M == 21 and dt == 2:
        return "reg<21,2,MINB=1>"
    return f"generic<{8 if M <= 8 else 16 if M <= 16 else 24 if M <= 24 else 32}>"


@pytest.mark.parametrize("m,d", [(1, 2), (5, 2), (5, 3), (10, 2), (10, 3), (12, 2), (20, 2), (20, 3), (31, 2)])
def test_kernel_values_read_off_factor_rows(m, d):
    ref = load_probe_reference()
    P = make_probe_problem(m, d, ref["x"])
    fails, worst = [], {}
    for covfun in ("exponential_isotropic", "matern_isotropic"):
        fams = [f for f in ref["families"] if f["covfun"] == covfun]
        tables = (1, 0) if covfun.startswith("matern") else (1,)
        with nb.NNGPContext(P["locs"], P["NNarray"], P["coloring"], P["locs_match"], covfun) as ctx:
            for fv in ((0, 1) if m == 20 else (0,)):
                ctx.set_option("factor_variant", fv)
                for table in tables:
                    ctx.set_option("matern_table", table)
                    label = f"{factor_kernel(m, d, fv)} d={d} matern_table={table}"
                    for fam in fams:
                        for s2 in (1.0, 2.5):
                            for tau in (0.0, 0.5):
                                bad = ctx.factor_build(probe_covparms(fam["nu"], s2, tau))
                                L = ctx.factor_get()
                                if tau > 0:
                                    assert bad == 0, label
                                    assert np.all(L[m:, 2:] == 0.0), label      # the far anchors decouple exactly
                                fails += probe_failures(L, m, ref, fam, s2, tau, label, worst)
    print(f"\nm={m} d={d}: worst relative error of rho per regime:", {k: f"{v:.2e}" for k, v in sorted(worst.items())})
    assert not fails, f"{len(fails)} probes over their bounds:\n" + "\n".join(fails[:60])
