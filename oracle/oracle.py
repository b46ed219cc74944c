"""ctypes front-end of the CPU oracle (oracle/liboracle.so).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / ``--impl reference`` legs import this module.
The product package never does (tests/test_no_oracle_in_product.py enforces it).

All arrays follow R's conventions: column-major (Fortran order), float64, int32, 1-based indices, NA = INT_MIN.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

NA_INT = -2147483648
_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

COVFUN_IDS = {
    "exponential_isotropic": 0,
    "exponential_sphere": 1,
    "exponential_scaledim": 2,
    "exponential_spacetime": 3,
    "matern_isotropic": 4,
    "matern_sphere": 5,
    "matern_scaledim": 6,
    "matern_spacetime": 7,
}

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_lp = C.POINTER(C.c_int64)


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("nngp_oracle.c", "r_rng.c", "gpgp_order.c", "bessel_shim.cpp", "nngp_oracle.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["make", "-C", _HERE, "-s"], check=True)
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        _LIB.r_unif_rand.restype = C.c_double
        _LIB.r_norm_rand.restype = C.c_double
        _LIB.r_qnorm.restype = C.c_double
        _LIB.r_qnorm.argtypes = [C.c_double]
        _LIB.r_unif_index.restype = C.c_double
        _LIB.r_unif_index.argtypes = [C.c_double]
        _LIB.r_rbeta.restype = C.c_double
        _LIB.r_rbeta.argtypes = [C.c_double, C.c_double]
        _LIB.oracle_bessel_k.restype = C.c_double
        _LIB.oracle_bessel_k.argtypes = [C.c_double, C.c_double]
        _LIB.oracle_ll_compressed_sparse_chol.restype = C.c_double
        _LIB.oracle_obs_loglik.restype = C.c_double
        _LIB.oracle_ssr.restype = C.c_double
        _LIB.oracle_moral_graph.restype = C.c_int64
        _LIB.oracle_philox_normal.restype = C.c_double
        _LIB.oracle_philox_normal.argtypes = [C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32]
    return _LIB


def _f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64).ravel(order="F"))


def _i32(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.int32).ravel(order="F"))


def _d(a):
    return a.ctypes.data_as(_dp)


def _i(a):
    return a.ctypes.data_as(_ip)


# ---------------------------------------------------------------- R RNG
def set_seed(seed: int) -> None:
    lib().r_set_seed(C.c_uint32(seed & 0xFFFFFFFF))


def runif(n: int) -> np.ndarray:
    out = np.empty(n)
    lib().r_runif(C.c_int(n), _d(out))
    return out


def rnorm(n: int, mean: float = 0.0, sd: float = 1.0) -> np.ndarray:
    out = np.empty(n)
    lib().r_rnorm(C.c_int(n), C.c_double(mean), C.c_double(sd), _d(out))
    return out


def qnorm(p: float) -> float:
    return lib().r_qnorm(p)


def sample_perm(n: int) -> np.ndarray:
    out = np.empty(n, dtype=np.int32)
    lib().r_sample_perm(C.c_int(n), _i(out))
    return out


def sample_int(n: int, size: int) -> np.ndarray:
    """sample.int(n, size) without replacement (1-based)"""
    out = np.empty(size, dtype=np.int32)
    lib().r_sample_int(C.c_int(n), C.c_int(size), _i(out))
    return out


def rbeta(shape1: float, shape2: float) -> float:
    return lib().r_rbeta(float(shape1), float(shape2))


def bessel_k(nu: float, x: float) -> float:
    return lib().oracle_bessel_k(nu, x)


# ---------------------------------------------------------------- graph structure
def find_ordered_nn(locs: np.ndarray, m: int) -> np.ndarray:
    locs = np.asarray(locs, dtype=np.float64)
    n, d = locs.shape
    nn = np.empty(n * (m + 1), dtype=np.int32)
    lib().oracle_find_ordered_nn(_d(_f64(locs)), C.c_int(n), C.c_int(d), C.c_int(m), _i(nn))
    return nn.reshape((n, m + 1), order="F")


def order_maxmin_gpgp(locs: np.ndarray) -> np.ndarray:
    """GpGp::order_maxmin(locs) on R's stream (initialize.R:29): 1-based permutation; advances the stream by rnorm(n*d)
    and sample(n)"""
    locs = np.asarray(locs, dtype=np.float64)
    n, d = locs.shape
    out = np.empty(n, dtype=np.int32)
    lib().oracle_order_maxmin_gpgp(_d(_f64(locs)), C.c_int(n), C.c_int(d), _i(out))
    return out


def find_ordered_nn_gpgp(locs: np.ndarray, m: int) -> np.ndarray:
    """GpGp::find_ordered_nn(locs, m) on R's stream (initialize.R:93): the jitter consumes rnorm(n*d)"""
    locs = np.asarray(locs, dtype=np.float64)
    n, d = locs.shape
    nn = np.empty(n * (m + 1), dtype=np.int32)
    lib().oracle_find_ordered_nn_gpgp(_d(_f64(locs)), C.c_int(n), C.c_int(d), C.c_int(m), _i(nn))
    return nn.reshape((n, m + 1), order="F")


def moral_graph(NNarray: np.ndarray):
    n, M = NNarray.shape
    nn = _i32(NNarray)
    nnz = lib().oracle_moral_graph(_i(nn), C.c_int(n), C.c_int(M - 1), None, None)
    adj_p = np.empty(n + 1, dtype=np.int64)
    adj_i = np.empty(max(nnz, 1), dtype=np.int32)
    lib().oracle_moral_graph(_i(nn), C.c_int(n), C.c_int(M - 1), adj_p.ctypes.data_as(_lp), _i(adj_i))
    return adj_p, adj_i[:nnz]


def naive_greedy_coloring(adj_p: np.ndarray, adj_i: np.ndarray) -> np.ndarray:
    n = adj_p.shape[0] - 1
    cols = np.empty(n, dtype=np.int32)
    adj_p = np.ascontiguousarray(adj_p, dtype=np.int64)
    adj_i = np.ascontiguousarray(adj_i, dtype=np.int32)
    lib().oracle_naive_greedy_coloring(adj_p.ctypes.data_as(_lp), _i(adj_i), C.c_int(n), _i(cols))
    return cols


# ---------------------------------------------------------------- Vecchia factor and products
def vecchia_Linv(covparms, covfun_name: str, locs: np.ndarray, NNarray: np.ndarray, return_bad: bool = False):
    locs = np.asarray(locs, dtype=np.float64)
    n, d = locs.shape
    M = NNarray.shape[1]
    cp = _f64(covparms)
    out = np.empty(n * M)
    bad = lib().oracle_vecchia_linv(_d(cp), C.c_int(cp.size), C.c_int(COVFUN_IDS[covfun_name]), _d(_f64(locs)),
                                    C.c_int(n), C.c_int(d), _i(_i32(NNarray)), C.c_int(M - 1), _d(out))
    L = out.reshape((n, M), order="F")
    return (L, bad) if return_bad else L


def Linv_mult(Linv: np.ndarray, z: np.ndarray, NNarray: np.ndarray) -> np.ndarray:
    n, M = NNarray.shape
    out = np.empty(n)
    lib().oracle_linv_mult(_d(_f64(Linv)), _d(_f64(z)), _i(_i32(NNarray)), C.c_int(n), C.c_int(M - 1), _d(out))
    return out


def ll_compressed_sparse_chol(Linv, field, NNarray, log_scale: float) -> float:
    n, M = NNarray.shape
    return lib().oracle_ll_compressed_sparse_chol(_d(_f64(Linv)), _d(_f64(field)), _i(_i32(NNarray)), C.c_int(n),
                                                  C.c_int(M - 1), C.c_double(log_scale))


def precision_diag(Linv, NNarray) -> np.ndarray:
    n, M = NNarray.shape
    out = np.empty(n)
    lib().oracle_precision_diag(_d(_f64(Linv)), _i(_i32(NNarray)), C.c_int(n), C.c_int(M - 1), _d(out))
    return out


def sparse_chol_solve(Linv, NNarray, b) -> np.ndarray:
    n, M = NNarray.shape
    out = np.empty(n)
    lib().oracle_sparse_chol_solve(_d(_f64(Linv)), _i(_i32(NNarray)), C.c_int(n), C.c_int(M - 1), _d(_f64(b)), _d(out))
    return out


def sparse_chol_tmult(Linv, NNarray, u) -> np.ndarray:
    n, M = NNarray.shape
    out = np.empty(n)
    lib().oracle_sparse_chol_tmult(_d(_f64(Linv)), _i(_i32(NNarray)), C.c_int(n), C.c_int(M - 1), _d(_f64(u)), _d(out))
    return out


# ---------------------------------------------------------------- the product's Philox normals
def philox4x32_10(counter, key) -> np.ndarray:
    """Philox4x32-10 of four 32-bit counter words under two key words"""
    c = (C.c_uint32 * 4)(*[int(v) & 0xFFFFFFFF for v in counter])
    k = (C.c_uint32 * 2)(*[int(v) & 0xFFFFFFFF for v in key])
    out = (C.c_uint32 * 4)()
    lib().oracle_philox4x32_10(c, k, out)
    return np.array(out[:], dtype=np.uint64)


def philox_key(seed):
    """(key0, key1) of a seed: s = (uint64)(int64)seed"""
    k = (C.c_uint32 * 2)()
    lib().oracle_philox_key(C.c_int64(int(seed)), k)
    return k[0], k[1]


def philox_normal(site: int, counter: int, seed) -> float:
    k0, k1 = philox_key(seed)
    return lib().oracle_philox_normal(site, counter, k0, k1)


def philox_handout(coloring, counter: int, seed) -> np.ndarray:
    """the normals of one sweep at `counter` in hand-out order (colour 1..K, ascending site inside a colour)"""
    col = _i32(coloring)
    k0, k1 = philox_key(seed)
    out = np.empty(col.size)
    lib().oracle_philox_handout(_i(col), C.c_int(col.size), C.c_int(int(col.max())), C.c_uint64(counter), C.c_uint32(k0),
                                C.c_uint32(k1), _d(out))
    return out


# ---------------------------------------------------------------- sampler pieces
def chromatic_sweep(Linv, NNarray, coloring, precision_diag_, obs_per_loc, residuals_sum, beta_0, log_scale,
                    log_noise_variance, z, field, form: str = "reference") -> np.ndarray:
    n, M = NNarray.shape
    f = _f64(field).copy()
    coloring = _i32(coloring)
    fn = lib().oracle_chromatic_sweep_reference if form == "reference" else lib().oracle_chromatic_sweep_residual
    fn(_d(_f64(Linv)), _i(_i32(NNarray)), C.c_int(n), C.c_int(M - 1), _i(coloring), C.c_int(int(coloring.max())),
       _d(_f64(precision_diag_)), _d(_f64(obs_per_loc)), _d(_f64(residuals_sum)), C.c_double(beta_0),
       C.c_double(log_scale), C.c_double(log_noise_variance), _d(_f64(z)), _d(f))
    return f


def residuals_sum(locs_match, n, observed_field, mu) -> np.ndarray:
    lm = _i32(locs_match)
    out = np.empty(n)
    lib().oracle_residuals_sum(_i(lm), C.c_int(lm.size), C.c_int(n), _d(_f64(observed_field)), _d(_f64(mu)), _d(out))
    return out


def obs_loglik(locs_match, observed_field, field, mu, beta_0, log_noise_variance) -> float:
    lm = _i32(locs_match)
    return lib().oracle_obs_loglik(_i(lm), C.c_int(lm.size), _d(_f64(observed_field)), _d(_f64(field)), _d(_f64(mu)),
                                   C.c_double(beta_0), C.c_double(log_noise_variance))


def ssr(locs_match, observed_field, field, mu, beta_0) -> float:
    lm = _i32(locs_match)
    return lib().oracle_ssr(_i(lm), C.c_int(lm.size), _d(_f64(observed_field)), _d(_f64(field)), _d(_f64(mu)),
                            C.c_double(beta_0))


def beta0_moments(Linv, NNarray, field, log_scale):
    n, M = NNarray.shape
    mean = C.c_double()
    var = C.c_double()
    lib().oracle_beta0_moments(_d(_f64(Linv)), _i(_i32(NNarray)), C.c_int(n), C.c_int(M - 1), _d(_f64(field)),
                               C.c_double(log_scale), C.byref(mean), C.byref(var))
    return mean.value, var.value


def predict_field_sample(Linv_all, NN_all, n, field, beta_0, log_scale, z_pred) -> np.ndarray:
    nt, M = NN_all.shape
    n_pred = nt - n
    out = np.empty(n_pred)
    lib().oracle_predict_field_sample(_d(_f64(Linv_all)), _i(_i32(NN_all)), C.c_int(n), C.c_int(n_pred), C.c_int(M - 1),
                                      _d(_f64(field)), C.c_double(beta_0), C.c_double(log_scale), _d(_f64(z_pred)),
                                      _d(out))
    return out


class ChainParams(C.Structure):
    _fields_ = [("shape", C.c_double * 4), ("n_shape", C.c_int), ("beta_0", C.c_double), ("log_scale", C.c_double),
                ("log_noise_variance", C.c_double), ("logvar_sufficient", C.c_double), ("logvar_ancillary", C.c_double)]


class Regressors(C.Structure):
    _fields_ = [("p", C.c_int), ("X", C.POINTER(C.c_double)), ("n_xlocs", C.c_int), ("xlocs", C.POINTER(C.c_int)),
                ("first_obs", C.POINTER(C.c_int)), ("solve_1XT1X", C.POINTER(C.c_double)),
                ("chol_solve_1XT1X", C.POINTER(C.c_double)), ("beta", C.POINTER(C.c_double)),
                ("beta_records", C.POINTER(C.c_double))]


def update_gaussian_chain(locs, NNarray, coloring, locs_match, obs_per_loc, observed_field, covfun_name, params: dict,
                          field, n_iterations_update, field_thinning=1.0, n_chromatic=10, iter_start=0, chain_index=1,
                          sweep_form=0, regressors: dict | None = None, rng="R", sweep_counter=0):
    """One chain of mcmc_nngp_update_Gaussian. Returns (params, field, records, field_records, accept).
    regressors = dict(X, xlocs (1-based), first_obs (1-based), solve_1XT1X, chol_solve_1XT1X, beta): the model with
    regression coefficients (update_Gaussian.R:226-250); params then also carries "beta" and the tuple gets a sixth
    element, the beta records.
    rng = "R": every draw from R's stream, as the reference.  rng = "philox": the field normals as nngp_chain_run* draw them in
    NNGP_RNG_PHILOX mode -- Philox under seed (iter_start << 20) ^ chain_index, sweep j of the call at counter sweep_counter + j
    (the context's counter when the call starts), no rnorm for the field; the scalar draws stay on R's stream."""
    assert rng in ("R", "philox")
    locs = np.asarray(locs, dtype=np.float64)
    n, d = locs.shape
    M = NNarray.shape[1]
    p = ChainParams()
    shape = np.atleast_1d(np.asarray(params["shape"], dtype=np.float64))
    for k, v in enumerate(shape):
        p.shape[k] = v
    p.n_shape = shape.size
    p.beta_0 = params["beta_0"]
    p.log_scale = params["log_scale"]
    p.log_noise_variance = params["log_noise_variance"]
    p.logvar_sufficient = params.get("logvar_sufficient", -2.0)
    p.logvar_ancillary = params.get("logvar_ancillary", -2.0)
    f = _f64(field).copy()
    lm = _i32(locs_match)
    coloring = _i32(coloring)
    n_iter = int(n_iterations_update)
    rec = np.zeros(n_iter * (3 + shape.size))
    n_frec = int(round(n_iter * field_thinning))
    frec = np.zeros(max(n_frec, 1) * n)
    acc = np.zeros(2 * n_iter, dtype=np.int32)
    reg_ref, keep = None, []
    if regressors is not None:
        X = np.asfortranarray(regressors["X"], dtype=np.float64)
        P = X.shape[1]
        xl = _i32(np.atleast_1d(np.asarray(regressors.get("xlocs", []), dtype=np.int32)))
        fo = _i32(regressors["first_obs"]) if xl.size else np.zeros(1, dtype=np.int32)
        S = np.asfortranarray(regressors["solve_1XT1X"], dtype=np.float64)
        Ch = np.asfortranarray(regressors["chol_solve_1XT1X"], dtype=np.float64)
        beta = np.array(regressors["beta"], dtype=np.float64).ravel().copy()
        brec = np.zeros(max(n_iter * P, 1))
        assert X.shape[0] == lm.size and S.shape == (P + 1, P + 1) and Ch.shape == (P + 1, P + 1) and beta.size == P
        pd_ = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        r = Regressors(P, pd_(X), int(xl.size), xl.ctypes.data_as(C.POINTER(C.c_int)), fo.ctypes.data_as(C.POINTER(C.c_int)),
                       pd_(S), pd_(Ch), pd_(beta), pd_(brec))
        keep = [X, xl, fo, S, Ch, beta, brec]
        reg_ref = C.byref(r)
    fn = lib().oracle_update_gaussian_chain_rng
    fn.restype = C.c_int
    philox_seed = ((iter_start & 0xFFFFFFFF) << 20) ^ (chain_index & 0xFFFFFFFF)          # nngp_chain_run's key
    rc = fn(
        _d(_f64(locs)), C.c_int(n), C.c_int(d), _i(_i32(NNarray)), C.c_int(M - 1), _i(coloring),
        C.c_int(int(coloring.max())), _i(lm), C.c_int(lm.size), _d(_f64(obs_per_loc)), _d(_f64(observed_field)),
        C.c_int(COVFUN_IDS[covfun_name]), C.byref(p), _d(f), C.c_int(n_iter), C.c_double(field_thinning),
        C.c_int(n_chromatic), C.c_int(iter_start), C.c_int(chain_index), C.c_int(sweep_form), _d(rec), _d(frec), _i(acc),
        reg_ref, C.c_int(1 if rng == "philox" else 0), C.c_int64(philox_seed), C.c_uint64(sweep_counter))
    assert rc == 0
    out = dict(shape=np.array([p.shape[k] for k in range(shape.size)]), beta_0=p.beta_0, log_scale=p.log_scale,
               log_noise_variance=p.log_noise_variance, logvar_sufficient=p.logvar_sufficient,
               logvar_ancillary=p.logvar_ancillary)
    res = (out, f, rec.reshape((n_iter, 3 + shape.size), order="F"),
           frec[: n_frec * n].reshape((n_frec, n), order="F"), acc.reshape((n_iter, 2), order="F"))
    if regressors is not None:
        out["beta"] = keep[5]
        res = res + (keep[6][: n_iter * keep[5].size].reshape((n_iter, keep[5].size), order="F"),)
    return res
