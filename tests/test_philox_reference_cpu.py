"""The two transcriptions of the sampler's Philox normal stream the GPU tests compare the device with: tests/philox_reference.py
(vectorised numpy) and the oracle's plain C (oracle_philox_*), against Random123's known answers, against each other, and as a
source of standard normals."""
import numpy as np
import pytest
from scipy import stats

from oracle import oracle as O
from philox_reference import chain_seed, handout, normal_from_words, philox4x32_10, philox_key, philox_normals

# Random123 known-answer vectors for Philox4x32-10: (counter, key, output)
KAT = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
       ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
       ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]

# seeds as the ABI receives them: gibbs_sweep's seed (a negative one, >= 2^32, >= 2^45) and nngp_chain_run's, with iter_start >= 4096 so
# that its bits reach key1
SEEDS = [0, 1, 12345, -1, -7, 2 ** 32, 2 ** 32 + 3, 2 ** 45 + 11, chain_seed(0, 2), chain_seed(4096, 3), chain_seed(4600, 1)]
COUNTERS = [0, 1, 2, 12, 2 ** 31 - 1, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 5, 2 ** 40 + 3, 2 ** 64 - 1]


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_known_answers(ctr, key, want):
    got_np = [int(v) for v in philox4x32_10(*ctr, *key)]
    got_c = [int(v) for v in O.philox4x32_10(ctr, key)]
    assert got_np == list(want), [hex(v) for v in got_np]
    assert got_c == list(want), [hex(v) for v in got_c]


def test_keys_of_seeds():
    assert philox_key(0) == (0, 0x5EED5EED)
    assert philox_key(-1) == (0xFFFFFFFF, 0xFFFFFFFF ^ 0x5EED5EED)
    assert philox_key(2 ** 45 + 11) == (11, 2 ** 13 ^ 0x5EED5EED)
    assert chain_seed(4600, 1) == 4600 * 2 ** 20 + 1 and philox_key(chain_seed(4600, 1))[1] == 1 ^ 0x5EED5EED
    for s in SEEDS:
        assert O.philox_key(s) == philox_key(s), s


def test_numpy_and_c_generators_agree():
    """words bit for bit over a grid of sites, counters and keys; normals to 2e-15 max(1, |z|)"""
    sites = np.array([0, 1, 2, 3, 99, 2 ** 20 + 1, 2 ** 31, 2 ** 32 - 1], dtype=np.uint64)
    worst = 0.0
    for s in SEEDS:
        k0, k1 = philox_key(s)
        for k in COUNTERS:
            lo, hi = k & 0xFFFFFFFF, k >> 32
            words = np.stack(philox4x32_10(sites, lo, hi, 0x4E4E4750, k0, k1), axis=1)
            for i, g in enumerate(sites):
                assert np.array_equal(O.philox4x32_10((int(g), lo, hi, 0x4E4E4750), (k0, k1)), words[i]), (s, k, int(g))
            z = philox_normals(s, k, sites=sites)
            zc = np.array([O.philox_normal(int(g), k, s) for g in sites])
            worst = max(worst, float(np.max(np.abs(z - zc) / np.maximum(1.0, np.abs(z)))))
            coloring = np.ones(1000, dtype=np.int32)                    # one colour: hand-out order = site order
            z = philox_normals(s, k, 1000)
            zc = O.philox_handout(coloring, k, s)
            worst = max(worst, float(np.max(np.abs(z - zc) / np.maximum(1.0, np.abs(z)))))
    print(f"numpy vs C normals: max |dz| / max(1, |z|) = {worst:.2e}")
    assert worst <= 2e-15


def test_handout_order():
    """colour 1..K, ascending site index inside a colour, in numpy and in C"""
    rng = np.random.default_rng(3)
    coloring = rng.integers(1, 8, 5000).astype(np.int32)
    z = philox_normals(9, 4, 5000)
    h = handout(z, coloring)
    want = np.concatenate([z[coloring == c] for c in range(1, 8)])
    assert np.array_equal(h, want)
    assert np.max(np.abs(O.philox_handout(coloring, 4, 9) - h)) <= 2e-15 * max(1.0, np.max(np.abs(h)))


def test_stream_is_standard_normal():
    """4.2M normals over 65 536 sites x 64 counters (key bits past 32): moments within 5 standard errors, a KS test against Phi,
    lag-1 correlations along the site and the counter within 5 / sqrt(N)"""
    n_sites, n_ctr = 65536, 64
    Z = np.stack([philox_normals(chain_seed(4600, 1), k, n_sites) for k in range(1000, 1000 + n_ctr)])   # counter x site
    z = Z.ravel()
    N = z.size
    mean, var = z.mean(), z.var()
    c = z - mean
    skew = np.mean(c ** 3) / var ** 1.5
    kurt = np.mean(c ** 4) / var ** 2 - 3.0
    ks = stats.kstest(z, "norm")
    r_site = np.corrcoef(Z[:, :-1].ravel(), Z[:, 1:].ravel())[0, 1]
    r_ctr = np.corrcoef(Z[:-1].ravel(), Z[1:].ravel())[0, 1]
    print(f"N = {N}: mean {mean:.2e} var-1 {var - 1:.2e} skew {skew:.2e} excess kurtosis {kurt:.2e} KS p {ks.pvalue:.3f} "
          f"lag-1 site {r_site:.2e} counter {r_ctr:.2e}")
    assert abs(mean) < 5 / np.sqrt(N)
    assert abs(var - 1) < 5 * np.sqrt(2 / N)
    assert abs(skew) < 5 * np.sqrt(6 / N)
    assert abs(kurt) < 5 * np.sqrt(24 / N)
    assert ks.pvalue > 1e-3
    assert abs(r_site) < 5 / np.sqrt(N) and abs(r_ctr) < 5 / np.sqrt(N)


def test_extreme_words_give_finite_normals():
    """a = 0 gives the smallest u1 (2^-54, the largest radius, 8.62); a = 2^64 - 1 rounds u1 to 1 (radius 0)"""
    top = 0xFFFFFFFF
    for b in ((0, 0), (top, top), (0x80000000, 0), (0x40000000, 0)):       # u2 near 0, near 1, 1/2, 1/4
        z_small = normal_from_words(0, 0, *b)
        z_one = normal_from_words(top, top, *b)
        assert np.isfinite(z_small) and np.isfinite(z_one), b
        assert abs(z_small) <= np.sqrt(-2.0 * np.log(2.0 ** -54)) and z_one == 0.0, b
    assert abs(normal_from_words(0, 0, 0, 0) - np.sqrt(-2.0 * np.log(2.0 ** -54))) < 1e-14
