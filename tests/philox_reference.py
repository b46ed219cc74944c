"""Reference transcription of the sampler's on-device normal generator, in vectorised numpy (uint64 products, no loops over sites).

The contract it restates (device_math.cuh: philox4x32_10, philox_normal; nngp_b200.cu: set_sweep_params, nngp_chain_run):
  * the normal of reference site g (0-based, global on a sharded field) at sweep counter k under seed s is Philox4x32-10 with
    counter (g, k & 0xffffffff, k >> 32, 0x4e4e4750) and key (s & 0xffffffff, (s >> 32) ^ 0x5eed5eed), s = (uint64)(int64)seed;
  * a = (x << 32) | y, b = (z << 32) | w; u1 = ((a >> 11) + 0.5) 2^-53, u2 likewise from b; z = sqrt(-2 log u1) cos(2 pi u2)
    (the device takes cospi(2 u2); the two differ by the rounding of 2 pi u2, by less than 1.5e-15 sqrt(-2 log u1));
  * nngp_chain_run* key the sweeps with seed = (iter_start << 20) ^ chain_index;
  * supplied normals (and the oracle's rnorm) are handed out colour 1..K, ascending reference index inside a colour.
"""
from __future__ import annotations

import numpy as np

MASK32 = np.uint64(0xFFFFFFFF)
M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
COUNTER_TAG = 0x4E4E4750
KEY1_SALT = 0x5EED5EED


def philox4x32_10(x, y, z, w, k0, k1):
    """Philox4x32-10 (Salmon et al. 2011) on broadcastable arrays of 32-bit words; returns the four output words (uint64 arrays)"""
    x, y, z, w = np.broadcast_arrays(*(np.asarray(v, dtype=np.uint64) & MASK32 for v in (x, y, z, w)))
    k0, k1 = np.uint64(int(k0) & 0xFFFFFFFF), np.uint64(int(k1) & 0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = M0 * x, M1 * z                      # 32 x 32 -> 64 bits: exact in uint64
        x, y, z, w = (p1 >> np.uint64(32)) ^ y ^ k0, p1 & MASK32, (p0 >> np.uint64(32)) ^ w ^ k1, p0 & MASK32
        k0, k1 = (k0 + W0) & MASK32, (k1 + W1) & MASK32
    return x, y, z, w


def philox_key(seed):
    """(key0, key1) of a seed as set_sweep_params forms them: s = (uint64)(int64)seed"""
    s = int(seed) & 0xFFFFFFFFFFFFFFFF
    return s & 0xFFFFFFFF, (s >> 32) ^ KEY1_SALT


def normal_from_words(x, y, z, w):
    """Box-Muller on the two 53-bit uniforms the device forms from one Philox output block"""
    s32, s11 = np.uint64(32), np.uint64(11)
    a = (np.asarray(x, dtype=np.uint64) << s32) | np.asarray(y, dtype=np.uint64)
    b = (np.asarray(z, dtype=np.uint64) << s32) | np.asarray(w, dtype=np.uint64)
    u1 = ((a >> s11).astype(np.float64) + 0.5) * 2.0 ** -53
    u2 = ((b >> s11).astype(np.float64) + 0.5) * 2.0 ** -53
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


def philox_normals(seed, counter, n=None, sites=None):
    """normals of sites 0..n-1 (or of the given 0-based site ids) at sweep counter `counter` under `seed`"""
    g = np.arange(n, dtype=np.uint64) if sites is None else np.asarray(sites, dtype=np.uint64)
    k = int(counter) & 0xFFFFFFFFFFFFFFFF
    k0, k1 = philox_key(seed)
    return normal_from_words(*philox4x32_10(g, k & 0xFFFFFFFF, k >> 32, COUNTER_TAG, k0, k1))


def chain_seed(iter_start, chain_index):
    """the seed nngp_chain_run* key their sweeps with"""
    return ((int(iter_start) & 0xFFFFFFFF) << 20) ^ (int(chain_index) & 0xFFFFFFFF)


def handout(z_by_site, coloring):
    """normals indexed by site -> the order a supplied-mode sweep reads them: colour 1..K, ascending reference index inside a colour"""
    return np.asarray(z_by_site)[np.argsort(np.asarray(coloring), kind="stable")]


def sweep_normals(seed, counter, n_sweeps, coloring):
    """the z= argument that makes a supplied-mode call of n_sweeps sweeps draw what a Philox call starting at `counter` draws"""
    n = len(coloring)
    return np.concatenate([handout(philox_normals(seed, counter + s, n), coloring) for s in range(n_sweeps)])
