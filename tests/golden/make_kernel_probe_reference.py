"""Write tests/golden/kernel_probe_reference.json: the covariance kernels' correlation rho(x) at the probe distances, in 50-digit
arithmetic, for the kernel probe tests (tests/test_gpu_kernel_accuracy.py, tests/test_kernel_probe_cpu.py).

    python tests/golden/make_kernel_probe_reference.py

Needs mpmath.  The JSON it writes is committed, so the tests that read it do not; tests/test_kernel_probe_cpu.py regenerates it
and compares byte for byte when mpmath is importable.

Families: exponential, rho = exp(-x), and GpGp's Matern, rho = 2^(1-nu) / Gamma(nu) x^nu K_nu(x) (no sqrt(2 nu) factor), at smoothness
values that cross the device's switches: nl = (int)(nu + 1/2) of the upward recurrence (nu = 1/2, 3/2), mu = nu - nl = 0 (nu = 1/2,
1), and the ends of the range (0, 1.5) that the reference's transforms reach.  Distances (scaled, range 1): x = 0; the boundaries of
the device's evaluation regimes in s = x^2 -- 2^-80, 2^-26, 4 (also Temme / continued fraction at x = 2), 2^6, 2^20 -- with their
neighbouring doubles; and a seeded log-uniform handful inside every regime, 2^-50 .. 2000.  kappa = |x d log(rho) / dx| (exponential:
x; Matern: x K_{nu-1}(x) / K_nu(x)) is the conditioning of rho in its argument.
"""
import json
import math
import os
import random

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "kernel_probe_reference.json")
NUS = [0.05, 0.25, 0.4, 0.5 - 1e-12, 0.5, 0.5 + 1e-12, 0.75, 1 - 1e-9, 1.0, 1 + 1e-9, 1.1, 1.45, 1.499]
X_BOUNDARIES = [2.0 ** -40, 2.0 ** -13, 2.0, 8.0, 1024.0]        # s = 2^-80, 2^-26, 4, 2^6, 2^20
X_REGIMES = [2.0 ** -50, 2.0 ** -40, 2.0 ** -13, 2.0, 8.0, 1024.0, 2000.0]
PER_REGIME = 4
SEED = 20261020


def probe_distances():
    xs = [0.0]
    for b in X_BOUNDARIES:
        xs += [math.nextafter(b, 0.0), b, math.nextafter(b, math.inf)]
    rng = random.Random(SEED)                                      # Mersenne Twister: the same stream on every Python 3
    for lo, hi in zip(X_REGIMES[:-1], X_REGIMES[1:]):
        xs += sorted(math.exp(rng.uniform(math.log(lo), math.log(hi))) for _ in range(PER_REGIME))
    return xs


def reference():
    import mpmath as mp
    mp.mp.dps = 70
    xs = probe_distances()
    fams = []
    for nu in [None] + NUS:
        rho, kappa = [], []
        for x in xs:
            X = mp.mpf(x)
            if x == 0.0:
                r, k = mp.mpf(1), mp.mpf(0)
            elif nu is None:
                r, k = mp.exp(-X), X
            else:
                N = mp.mpf(nu)
                kn = mp.besselk(N, X)
                r = 2 ** (1 - N) / mp.gamma(N) * X ** N * kn
                k = X * mp.besselk(N - 1, X) / kn
            rho.append(mp.nstr(r, 50, min_fixed=1, max_fixed=0))
            kappa.append(mp.nstr(k, 6, min_fixed=1, max_fixed=0))
        fams.append({"covfun": "exponential_isotropic" if nu is None else "matern_isotropic", "nu": nu, "rho": rho, "kappa": kappa})
    return {"about": "rho(x) of the probe distances at 50 digits (mpmath); written by make_kernel_probe_reference.py",
            "x": [x.hex() for x in xs], "families": fams}


def dumps(ref):
    return json.dumps(ref, indent=1) + "\n"


def main():
    with open(OUT, "w") as f:
        f.write(dumps(reference()))
    print("wrote", OUT)


if __name__ == "__main__":
    main()
