"""NNGPContext: thin object wrapper over the context handle of the C ABI (one model graph + one chain state on one GPU)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L


class NNGPContext:
    """Device-resident Vecchia structure (vecchia_approx of the reference, Scripts/mcmc_nngp_initialize.R:80-110).

    All arrays use R's conventions: column-major, 1-based indices, NA = INT_MIN; `field` includes beta_0.
    """

    def __init__(self, locs, NNarray, coloring, locs_match, covfun_name="exponential_isotropic", device=0,
                 layout=L.LAYOUT_MORTON):
        locs = np.asarray(locs, dtype=np.float64)
        if locs.ndim == 1:
            locs = locs[:, None]
        NNarray = np.asarray(NNarray, dtype=np.int32)
        self.n, self.d = locs.shape
        self.m = NNarray.shape[1] - 1
        self.covfun_name = covfun_name
        lm = L.i32(locs_match)
        self.n_obs = lm.size
        self._id = None
        cid, st = C.c_int(-1), C.c_int(0)
        lib = L.load()
        lib.nngp_ctx_create(L.ci(self.n), L.ci(self.d), L.ci(self.m), L.dptr(L.f64(locs)), L.iptr(L.i32(NNarray)),
                            L.iptr(L.i32(coloring)), L.ci(self.n_obs), L.iptr(lm), L.ci(L.COVFUN_IDS[covfun_name]),
                            L.ci(device), L.ci(layout), C.byref(cid), C.byref(st))
        L.check(st)
        self._id = cid.value
        info = (C.c_int * 8)()
        lib.nngp_ctx_info(L.ci(self._id), info, C.byref(st))
        L.check(st)
        self.n_colors, self.n_levels, self.nnz, self.max_col = info[2], info[3], info[4], info[5]
        self.device, self.layout = info[6], info[7]

    # ---- lifecycle
    def close(self):
        if self._id is not None:
            st = C.c_int(0)
            L.load().nngp_ctx_destroy(L.ci(self._id), C.byref(st))
            self._id = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _call(self, name, *args):
        st = C.c_int(0)
        getattr(L.load(), name)(L.ci(self._id), *args, C.byref(st))
        L.check(st)

    OPTIONS = {"sweep_variant": 1, "solve_variant": 2, "use_graph": 3, "solve_ctas_per_sm": 4, "solve_sleep_ns": 5, "solve_level_copy": 6,
               "solve_window_ctas": 7, "commit_variant": 8, "matern_table": 9, "loglik_variant": 10, "shard_ghost_ctas": 11, "shard_ghost_first": 12, "factor_variant": 14,
               "loglik_from_residual": 15}

    def set_option(self, name: str, value: int):
        self._call("nngp_ctx_set_option", L.ci(self.OPTIONS[name]), L.ci(value))

    # ---- factor
    def factor_build(self, covparms, slot=L.SLOT_CURRENT) -> int:
        cp = L.f64(covparms)
        bad = C.c_int(0)
        self._call("nngp_factor_build", L.ci(slot), L.dptr(cp), L.ci(cp.size), C.byref(bad))
        return bad.value

    def factor_get(self, slot=L.SLOT_CURRENT) -> np.ndarray:
        out = np.empty(self.n * (self.m + 1))
        self._call("nngp_factor_get", L.ci(slot), L.dptr(out))
        return out.reshape((self.n, self.m + 1), order="F")

    def factor_accept(self):
        self._call("nngp_factor_accept")

    def factor_commit(self, slot=L.SLOT_CURRENT):
        self._call("nngp_factor_commit", L.ci(slot))

    def precision_diag(self) -> np.ndarray:
        out = np.empty(self.n)
        self._call("nngp_precision_diag", L.dptr(out))
        return out

    # ---- state
    def field_set(self, field):
        f = L.f64(field)
        assert f.size == self.n
        self._call("nngp_field_set", L.dptr(f))

    def field_get(self, out: np.ndarray | None = None) -> np.ndarray:
        """`out` may be a pinned buffer (L.PinnedArray(n).array): the download then lands in it without a staging copy"""
        if out is None:
            out = np.empty(self.n)
        assert out.dtype == np.float64 and out.size == self.n and out.flags.c_contiguous
        self._call("nngp_field_get", L.dptr(out))
        return out

    def obs_set(self, y_minus_xb):
        y = L.f64(y_minus_xb)
        assert y.size == self.n_obs
        self._call("nngp_obs_set", L.dptr(y))

    # ---- log-likelihood and products
    def loglik(self, beta_0, log_scale, slot=L.SLOT_CURRENT) -> float:
        out = C.c_double(0.0)
        self._call("nngp_loglik", L.ci(slot), L.cd(beta_0), L.cd(log_scale), C.byref(out))
        return out.value

    def loglik_host(self, z, log_scale, slot=L.SLOT_CURRENT) -> float:
        zz = L.f64(z)
        assert zz.size == self.n
        out = C.c_double(0.0)
        self._call("nngp_loglik_host", L.ci(slot), L.dptr(zz), L.cd(log_scale), C.byref(out))
        return out.value

    def _vec_op(self, name, v, slot):
        vv = L.f64(v)
        assert vv.size == self.n
        out = np.empty(self.n)
        self._call(name, L.ci(slot), L.dptr(vv), L.dptr(out))
        return out

    def spmv(self, v, slot=L.SLOT_CURRENT):
        return self._vec_op("nngp_spmv", v, slot)

    def sptmv(self, u, slot=L.SLOT_CURRENT):
        return self._vec_op("nngp_sptmv", u, slot)

    def sptrsv(self, b, slot=L.SLOT_CURRENT):
        return self._vec_op("nngp_sptrsv", b, slot)

    # ---- sampler steps
    def sweep_loglik_host(self, field_io: np.ndarray, beta_0, log_scale, log_noise_variance, n_sweeps=1, z=None, seed=0) -> float:
        """nngp_sweep_loglik_host: field_io (float64, C-contiguous, n values; may be pinned) is updated in place by n_sweeps sweeps;
        returns the Vecchia log-likelihood of the new field"""
        assert field_io.dtype == np.float64 and field_io.size == self.n and field_io.flags.c_contiguous
        ll = C.c_double(0.0)
        if z is None:
            self._call("nngp_sweep_loglik_host", L.ci(n_sweeps), L.cd(beta_0), L.cd(log_scale), L.cd(log_noise_variance), L.ci(L.RNG_PHILOX),
                       None, L.cd(seed), L.dptr(field_io), C.byref(ll))
        else:
            zz = L.f64(z)
            assert zz.size == getattr(self, "n_z", self.n) * n_sweeps
            self._call("nngp_sweep_loglik_host", L.ci(n_sweeps), L.cd(beta_0), L.cd(log_scale), L.cd(log_noise_variance), L.ci(L.RNG_SUPPLIED),
                       L.dptr(zz), L.cd(seed), L.dptr(field_io), C.byref(ll))
        return ll.value

    def gibbs_sweep(self, beta_0, log_scale, log_noise_variance, n_sweeps=1, z=None, seed=0):
        if z is None:
            self._call("nngp_gibbs_sweep", L.ci(n_sweeps), L.cd(beta_0), L.cd(log_scale), L.cd(log_noise_variance),
                       L.ci(L.RNG_PHILOX), None, L.cd(seed))
        else:
            zz = L.f64(z)
            assert zz.size == getattr(self, "n_z", self.n) * n_sweeps   # sharded contexts index the whole field's normals
            self._call("nngp_gibbs_sweep", L.ci(n_sweeps), L.cd(beta_0), L.cd(log_scale), L.cd(log_noise_variance),
                       L.ci(L.RNG_SUPPLIED), L.dptr(zz), L.cd(seed))

    def ancillary_propose(self, beta_0, delta_log_scale, log_noise_variance) -> float:
        out = C.c_double(0.0)
        self._call("nngp_ancillary_propose", L.cd(beta_0), L.cd(delta_log_scale), L.cd(log_noise_variance), C.byref(out))
        return out.value

    def ancillary_accept(self):
        self._call("nngp_ancillary_accept")

    def beta0_moments(self, log_scale):
        mean, var = C.c_double(0.0), C.c_double(0.0)
        self._call("nngp_beta0_moments", L.cd(log_scale), C.byref(mean), C.byref(var))
        return mean.value, var.value

    def ssr(self) -> float:
        out = C.c_double(0.0)
        self._call("nngp_ssr", C.byref(out))
        return out.value

    def field_init(self, beta_0, log_scale, z, slot=L.SLOT_CURRENT):
        zz = L.f64(z)
        assert zz.size == self.n
        self._call("nngp_field_init", L.ci(slot), L.cd(beta_0), L.cd(log_scale), L.dptr(zz))

    def chain_run(self, params: dict, n_iter, var_y, thin=1.0, n_chromatic=10, iter_start=0, chain_index=1,
                  rng_mode=L.RNG_PHILOX, keep_field=True):
        """nngp_chain_run: the whole reference loop (update_Gaussian.R:101-314, no regressors) behind the ABI."""
        shape = np.atleast_1d(np.asarray(params["shape"], dtype=np.float64))
        p = np.concatenate([[params["beta_0"], params["log_scale"], params["log_noise_variance"],
                             params.get("logvar_sufficient", -2.0), params.get("logvar_ancillary", -2.0)], shape])
        p = np.ascontiguousarray(p, dtype=np.float64)
        n_iter = int(n_iter)
        rec = np.zeros(n_iter * (3 + shape.size))
        n_frec = int(round(n_iter * thin))
        frec = np.zeros(max(n_frec, 1) * self.n) if keep_field else None
        acc = np.zeros(2 * n_iter, dtype=np.int32)
        self._call("nngp_chain_run", L.ci(shape.size), L.dptr(p), L.ci(n_iter), L.cd(thin), L.ci(n_chromatic),
                   L.ci(iter_start), L.ci(chain_index), L.ci(rng_mode), L.cd(var_y), L.dptr(rec),
                   L.dptr(frec) if keep_field else None, L.iptr(acc))
        out = dict(beta_0=p[0], log_scale=p[1], log_noise_variance=p[2], logvar_sufficient=p[3], logvar_ancillary=p[4],
                   shape=p[5:].copy())
        frec_m = frec[: n_frec * self.n].reshape((n_frec, self.n), order="F") if keep_field else None
        return out, rec.reshape((n_iter, 3 + shape.size), order="F"), frec_m, acc.reshape((n_iter, 2), order="F")

    def regressors_set(self, X, observed_field, xlocs=(), first_obs=None):
        """nngp_regressors_set: X$X (n_obs x p, centred, no intercept), observed_field, X$locs (1-based columns) and
        hctam_scol_1 stay resident on the device for chain_run_regressors."""
        Xf = np.asfortranarray(X, dtype=np.float64)
        y = L.f64(observed_field)
        xl = np.ascontiguousarray(xlocs, dtype=np.int32)
        fo = None if first_obs is None else np.ascontiguousarray(first_obs, dtype=np.int32)
        self._reg_p = Xf.shape[1]
        self._call("nngp_regressors_set", L.ci(Xf.shape[1]), Xf.ctypes.data_as(C.POINTER(C.c_double)), L.dptr(y), L.ci(xl.size),
                   L.iptr(xl) if xl.size else None, L.iptr(fo) if fo is not None else None)

    def chain_run_regressors(self, params: dict, beta, solve_1XT1X, chol_solve_1XT1X, n_iter, var_y, thin=1.0, n_chromatic=10,
                             iter_start=0, chain_index=1, rng_mode=L.RNG_PHILOX, keep_field=True):
        """nngp_chain_run_regressors: the reference loop with the regression updates (update_Gaussian.R:226-250) behind the ABI."""
        shape = np.atleast_1d(np.asarray(params["shape"], dtype=np.float64))
        p = np.concatenate([[params["beta_0"], params["log_scale"], params["log_noise_variance"],
                             params.get("logvar_sufficient", -2.0), params.get("logvar_ancillary", -2.0)], shape])
        p = np.ascontiguousarray(p, dtype=np.float64)
        b = np.array(beta, dtype=np.float64).ravel().copy()
        P1 = b.size + 1
        S = np.asfortranarray(solve_1XT1X, dtype=np.float64)
        Ch = np.asfortranarray(chol_solve_1XT1X, dtype=np.float64)
        assert S.shape == (P1, P1) and Ch.shape == (P1, P1) and b.size == getattr(self, "_reg_p", -1)
        n_iter = int(n_iter)
        rec = np.zeros(n_iter * (3 + shape.size))
        brec = np.zeros(max(n_iter * b.size, 1))
        n_frec = int(round(n_iter * thin))
        frec = np.zeros(max(n_frec, 1) * self.n) if keep_field else None
        acc = np.zeros(2 * n_iter, dtype=np.int32)
        self._call("nngp_chain_run_regressors", L.ci(shape.size), L.dptr(p), L.dptr(b), S.ctypes.data_as(C.POINTER(C.c_double)),
                   Ch.ctypes.data_as(C.POINTER(C.c_double)), L.ci(n_iter), L.cd(thin), L.ci(n_chromatic), L.ci(iter_start),
                   L.ci(chain_index), L.ci(rng_mode), L.cd(var_y), L.dptr(rec), L.dptr(brec),
                   L.dptr(frec) if keep_field else None, L.iptr(acc))
        out = dict(beta_0=p[0], log_scale=p[1], log_noise_variance=p[2], logvar_sufficient=p[3], logvar_ancillary=p[4],
                   shape=p[5:].copy(), beta=b)
        frec_m = frec[: n_frec * self.n].reshape((n_frec, self.n), order="F") if keep_field else None
        return (out, rec.reshape((n_iter, 3 + shape.size), order="F"), brec[: n_iter * b.size].reshape((n_iter, b.size), order="F"),
                frec_m, acc.reshape((n_iter, 2), order="F"))

    def records_summary(self, first_row: int, n_rows: int, offsets=None) -> np.ndarray:
        """get_summary (estimate.R:1-6) of the field samples kept on the device by the last chain_run; n x 5"""
        out = np.empty(self.n * 5)
        off = None if offsets is None else L.f64(offsets)
        self._call("nngp_records_summary", L.ci(first_row), L.ci(n_rows), None if off is None else L.dptr(off), L.dptr(out))
        return out.reshape((self.n, 5), order="F")

    def predict_sample(self, n_obs_sites, field, beta_0, log_scale, z_pred, slot=L.SLOT_CURRENT):
        f = L.f64(field)
        z = L.f64(z_pred)
        out = np.empty(self.n - n_obs_sites)
        self._call("nngp_predict_sample", L.ci(slot), L.ci(n_obs_sites), L.dptr(f), L.cd(beta_0), L.cd(log_scale),
                   L.dptr(z), L.dptr(out))
        return out

    # ---- measurement
    OPS = {"factor_build": 0, "loglik": 1, "gibbs_sweep": 2, "spmv": 3, "sptrsv": 4, "commit": 5, "sweep_loglik": 6}

    def time_op(self, op: str, reps=20, flush_l2=False):
        ms = np.zeros(reps)
        nl = C.c_int(0)
        self._call("nngp_time_op", L.ci(self.OPS[op]), L.ci(reps), L.ci(1 if flush_l2 else 0), L.dptr(ms), C.byref(nl))
        return ms, nl.value


def time_op_group(contexts, op: str, reps=20) -> float:
    """nngp_time_op_group: `reps` x op ("gibbs_sweep" or "sweep_loglik") enqueued on all contexts (one device) at once; ms until
    the last one finished"""
    ids = (C.c_int * len(contexts))(*[c._id for c in contexts])
    ms, st = C.c_double(0.0), C.c_int(0)
    L.load().nngp_time_op_group(ids, L.ci(len(contexts)), L.ci(NNGPContext.OPS[op]), L.ci(reps), C.byref(ms), C.byref(st))
    L.check(st)
    return ms.value


def fp64_peak(device=0) -> float:
    """measured FP64 FMA throughput of the device, GFLOP/s (nngp_fp64_peak)"""
    v, st = C.c_double(0.0), C.c_int(0)
    L.load().nngp_fp64_peak(L.ci(device), C.byref(v), C.byref(st))
    L.check(st)
    return v.value


def chains_run(contexts, params_list, n_iter, var_y, thin=1.0, n_chromatic=10, iter_start=0, chain_indices=None, rng_mode=L.RNG_PHILOX,
               keep_field=True, max_concurrent=None, betas=None, solve_1XT1X=None, chol_solve_1XT1X=None):
    """nngp_chains_run / nngp_chains_run_regressors: chain k on contexts[k], all advanced concurrently (the reference's mclapply
    over chains, update_Gaussian.R:22-26); max_concurrent = the reference's n_cores.  Returns one tuple per chain, laid out like
    NNGPContext.chain_run (or chain_run_regressors when betas is given)."""
    nc = len(contexts)
    assert nc >= 1 and len(params_list) == nc
    chain_indices = list(range(1, nc + 1)) if chain_indices is None else list(chain_indices)
    n = contexts[0].n
    assert all(c.n == n for c in contexts)
    shapes = [np.atleast_1d(np.asarray(p["shape"], dtype=np.float64)) for p in params_list]
    ns = shapes[0].size
    P = np.zeros((nc, 5 + ns))
    for k, p in enumerate(params_list):
        P[k] = np.concatenate([[p["beta_0"], p["log_scale"], p["log_noise_variance"], p.get("logvar_sufficient", -2.0),
                                p.get("logvar_ancillary", -2.0)], shapes[k]])
    n_iter = int(n_iter)
    n_frec = int(round(n_iter * thin))
    rec = np.zeros((nc, n_iter * (3 + ns)))
    frec = np.zeros((nc, max(n_frec, 1) * n)) if keep_field else None
    acc = np.zeros((nc, 2 * n_iter), dtype=np.int32)
    ids = (C.c_int * nc)(*[c._id for c in contexts])
    ci_arr = (C.c_int * nc)(*chain_indices)
    st = C.c_int(0)
    mc = nc if max_concurrent is None else max(1, int(max_concurrent))
    lib = L.load()
    if betas is None:
        lib.nngp_chains_run(L.ci(nc), ids, L.ci(ns), L.dptr(P), L.ci(n_iter), L.cd(thin), L.ci(n_chromatic), L.ci(iter_start), ci_arr,
                            L.ci(rng_mode), L.cd(var_y), L.ci(mc), L.dptr(rec), L.dptr(frec) if keep_field else None, L.iptr(acc), C.byref(st))
    else:
        B = np.ascontiguousarray(np.array(betas, dtype=np.float64).reshape(nc, -1))
        pb = B.shape[1]
        S = np.asfortranarray(solve_1XT1X, dtype=np.float64)
        Ch = np.asfortranarray(chol_solve_1XT1X, dtype=np.float64)
        assert S.shape == (pb + 1, pb + 1) and Ch.shape == (pb + 1, pb + 1)
        brec = np.zeros((nc, max(n_iter * pb, 1)))
        lib.nngp_chains_run_regressors(L.ci(nc), ids, L.ci(ns), L.dptr(P), L.dptr(B), S.ctypes.data_as(C.POINTER(C.c_double)),
                                       Ch.ctypes.data_as(C.POINTER(C.c_double)), L.ci(n_iter), L.cd(thin), L.ci(n_chromatic), L.ci(iter_start),
                                       ci_arr, L.ci(rng_mode), L.cd(var_y), L.ci(mc), L.dptr(rec), L.dptr(brec),
                                       L.dptr(frec) if keep_field else None, L.iptr(acc), C.byref(st))
    L.check(st)
    out = []
    for k in range(nc):
        po = dict(beta_0=P[k, 0], log_scale=P[k, 1], log_noise_variance=P[k, 2], logvar_sufficient=P[k, 3], logvar_ancillary=P[k, 4],
                  shape=P[k, 5:].copy())
        frec_m = frec[k, : n_frec * n].reshape((n_frec, n), order="F") if keep_field else None
        r = rec[k].reshape((n_iter, 3 + ns), order="F")
        a = acc[k].reshape((n_iter, 2), order="F")
        if betas is None:
            out.append((po, r, frec_m, a))
        else:
            po["beta"] = B[k].copy()
            out.append((po, r, brec[k, : n_iter * pb].reshape((n_iter, pb), order="F"), frec_m, a))
    return out


def find_ordered_nn(locs, m) -> np.ndarray:
    """GpGp::find_ordered_nn replacement (Scripts/mcmc_nngp_initialize.R:93): exact, ties by lower index."""
    locs = np.asarray(locs, dtype=np.float64)
    if locs.ndim == 1:
        locs = locs[:, None]
    n, d = locs.shape
    out = np.empty(n * (m + 1), dtype=np.int32)
    st = C.c_int(0)
    L.load().nngp_host_find_ordered_nn(L.dptr(L.f64(locs)), L.ci(n), L.ci(d), L.ci(m), L.iptr(out), C.byref(st))
    L.check(st)
    return out.reshape((n, m + 1), order="F")


def greedy_coloring(NNarray) -> np.ndarray:
    """moral graph + naive_greedy_coloring (initialize.R:103-110, Coloring.R:2-20) without the dense scratch."""
    NNarray = np.asarray(NNarray, dtype=np.int32)
    n, M = NNarray.shape
    out = np.empty(n, dtype=np.int32)
    K, st = C.c_int(0), C.c_int(0)
    L.load().nngp_host_greedy_coloring(L.iptr(L.i32(NNarray)), L.ci(n), L.ci(M - 1), L.iptr(out), C.byref(K), C.byref(st))
    L.check(st)
    return out


def order_maxmin(locs) -> np.ndarray:
    """exact max-min ordering, 1-based permutation (GpGp::order_maxmin is a randomised approximation of this)."""
    locs = np.asarray(locs, dtype=np.float64)
    if locs.ndim == 1:
        locs = locs[:, None]
    n, d = locs.shape
    out = np.empty(n, dtype=np.int32)
    st = C.c_int(0)
    L.load().nngp_host_order_maxmin(L.dptr(L.f64(locs)), L.ci(n), L.ci(d), L.iptr(out), C.byref(st))
    L.check(st)
    return out
