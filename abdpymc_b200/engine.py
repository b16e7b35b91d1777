"""``AbdEngine``: NumPy-facing wrapper over the C ABI of libabd_b200.so.

One engine = one cohort (or one shard of it) resident on one GPU.  Every method maps 1:1 to an
entry point of include/abd_b200.h; shapes follow the reference graph: ``i_raw`` is
(chains, gap, ind), ``waner`` (chains, ind), parameters (chains, 13 | 17).  A leading chain axis
may be omitted for a single chain.
"""

from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import AbdCohort, check

THETA13 = [
    "ab_n_perm", "ab_n_temp", "ab_n_rho", "ab_n_init", "ab_s_perm", "ab_s_rho", "ab_s_init",
    "it_n_b", "it_n_d", "it_n_sigma", "it_s_b", "it_s_d", "it_s_sigma",
]  # fmt: skip
#: PyMC value variables in declaration order (abd.py:424, 329-340, 367-388, 464-467)
Q17 = [
    "p_logodds__", "ab_n_perm_log__", "ab_n_temp_log__", "ab_n_rho_logodds__", "ab_n_init",
    "ab_s_perm_log__", "ab_s_rho_logodds__", "ab_s_p_waner_logodds__", "ab_s_tempinf_log__",
    "ab_s_tempvac_log__", "ab_s_init", "it_n_b", "it_n_d", "it_n_sigma_log__", "it_s_b", "it_s_d",
    "it_s_sigma_log__",
]  # fmt: skip
#: RV name and transform of each q17 slot
Q17_RV = [
    ("p", "logodds"), ("ab_n_perm", "log"), ("ab_n_temp", "log"), ("ab_n_rho", "logodds"),
    ("ab_n_init", None), ("ab_s_perm", "log"), ("ab_s_rho", "logodds"), ("ab_s_p_waner", "logodds"),
    ("ab_s_tempinf", "log"), ("ab_s_tempvac", "log"), ("ab_s_init", None), ("it_n_b", None),
    ("it_n_d", None), ("it_n_sigma", "log"), ("it_s_b", None), ("it_s_d", None), ("it_s_sigma", "log"),
]  # fmt: skip
Q_OF_THETA = [1, 2, 3, 4, 5, 6, 10, 11, 12, 13, 14, 15, 16]
Q_P, Q_PW = 0, 7


def backward(q17: np.ndarray) -> np.ndarray:
    """PyMC's default back-transforms (log -> exp, logodds -> sigmoid) applied slot-wise."""
    q17 = np.asarray(q17, dtype=np.float64)
    out = q17.copy()
    for k, (_, tr) in enumerate(Q17_RV):
        if tr == "log":
            out[..., k] = np.exp(q17[..., k])
        elif tr == "logodds":
            out[..., k] = 1.0 / (1.0 + np.exp(-q17[..., k]))
    return out


def forward(values: np.ndarray) -> np.ndarray:
    values = np.asarray(values, dtype=np.float64)
    out = values.copy()
    for k, (_, tr) in enumerate(Q17_RV):
        if tr == "log":
            out[..., k] = np.log(values[..., k])
        elif tr == "logodds":
            out[..., k] = np.log(values[..., k]) - np.log1p(-values[..., k])
    return out


def _ptr(a):
    """Address of a NumPy array for a void* argument (``.ctypes.data_as`` costs ~4 us per call)."""
    return None if a is None else a.ctypes.data


def _f64(a, shape):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a.reshape(shape)


class AbdEngine:
    def __init__(self, cohort, splits=None, ignore_pcrpos=False, device=0, totals=None, ind_offset=0):
        """``cohort``: abdpymc_b200.cohort.CohortArrays (or anything with the same attributes).
        ``splits``: None / () / (a,) / (a, b) as in abd.model (abd.py:396-410).
        ``totals``: (n_inds, n_rows_s, n_rows_n) of the WHOLE cohort when this engine holds one
        shard of the individuals; ``ind_offset``: global index of the shard's first individual."""
        self._lib = _lib.load()
        self._h = C.c_void_p()
        splits = tuple(splits or ())
        if any(not isinstance(s, (int, np.integer)) for s in splits):
            raise ValueError("splits must be ints")  # abd.py:621-622
        if len(splits) > 2:
            raise NotImplementedError("only implemented 1-3 time chunks (0-2 splits)")  # abd.py:882
        self.G, self.N = int(cohort.n_gaps), int(cohort.n_inds)
        self._out17 = {}
        self.splits = splits
        self.ignore_pcrpos = bool(ignore_pcrpos)
        self.device = device
        keep = []

        def arr(a, dt):
            a = np.ascontiguousarray(a, dtype=dt)
            keep.append(a)
            return a

        d = AbdCohort()
        d.n_gaps, d.n_inds, d.n_splits = self.G, self.N, len(splits)
        for k, s in enumerate(splits):
            d.splits[k] = int(s)
        vacs = arr(np.asarray(cohort.vacs).T != 0, np.uint8)  # (G, N), abd.py:413
        d.vacs = vacs.ctypes.data_as(_lib.c_uint8_p)
        if not ignore_pcrpos:  # abd.py:416-418
            pcr = arr(np.asarray(cohort.pcrpos).T != 0, np.uint8)
            d.pcrpos = pcr.ctypes.data_as(_lib.c_uint8_p)
        for a, name in ((1, "s"), (0, "n")):
            x, od, gap, ind = cohort.rows(a)
            setattr(d, f"n_rows_{name}", len(x))
            setattr(d, f"x_{name}", arr(x, np.float64).ctypes.data_as(_lib.c_double_p))
            setattr(d, f"od_{name}", arr(od, np.float64).ctypes.data_as(_lib.c_double_p))
            setattr(d, f"gap_{name}", arr(gap, np.int32).ctypes.data_as(_lib.c_int32_p))
            setattr(d, f"ind_{name}", arr(ind, np.int32).ctypes.data_as(_lib.c_int32_p))
        self.R_s, self.R_n = int(d.n_rows_s), int(d.n_rows_n)
        if totals is not None:
            d.total_inds, d.total_rows_s, d.total_rows_n = (int(v) for v in totals)
        d.ind_offset = int(ind_offset)
        check(self._lib.abd_create(C.byref(self._h), C.byref(d), int(device)))

    # ------------------------------------------------------------------------------ cache file
    def save_cache(self, path):
        """Write the preprocessed cohort (the device upload format) to ``path``; ``AbdEngine.from_cache`` reads it."""
        check(self._lib.abd_save_cache(self._h, str(path).encode()))

    @classmethod
    def from_cache(cls, path, device=0, splits=None, ignore_pcrpos=None):
        """An engine from a file written by ``save_cache``: no CSV parsing, no sorting -- read and upload.
        ``splits`` / ``ignore_pcrpos``, when given, must be what the cache was built with (ValueError otherwise)."""
        self = cls.__new__(cls)
        self._lib = _lib.load()
        self._h = C.c_void_p()
        check(self._lib.abd_create_from_cache(C.byref(self._h), str(path).encode(), int(device)))
        g, n, rs, rn = C.c_int32(), C.c_int32(), C.c_int64(), C.c_int64()
        check(self._lib.abd_sizes(self._h, C.byref(g), C.byref(n), C.byref(rs), C.byref(rn)))
        self.G, self.N, self.R_s, self.R_n = g.value, n.value, rs.value, rn.value
        ns, sp, hp = C.c_int32(), (C.c_int32 * 2)(), C.c_int32()
        check(self._lib.abd_cohort_info(self._h, C.byref(ns), sp, C.byref(hp)))
        self.splits = tuple(int(sp[k]) for k in range(ns.value))
        self.ignore_pcrpos = not hp.value
        self._out17, self.device = {}, device
        if splits is not None and tuple(splits or ()) != self.splits:
            self.close()
            raise ValueError(f"cache built with splits {self.splits}, asked for {tuple(splits or ())}")
        if ignore_pcrpos is not None and bool(ignore_pcrpos) != self.ignore_pcrpos:
            self.close()
            raise ValueError(f"cache built with ignore_pcrpos={self.ignore_pcrpos}")
        return self

    # ------------------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.abd_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ------------------------------------------------------------------------------ helpers
    def _state(self, C_, i_raw, waner):
        if i_raw is None and waner is None:
            return None, None
        if i_raw is None or waner is None:
            raise ValueError("pass both i_raw and waner, or neither (resident state)")
        return self._as_int8(i_raw, (C_, self.G, self.N)), self._as_int8(waner, (C_, self.N))

    @staticmethod
    def _as_int8(a, shape):
        """0/1 bytes for the C ABI.  One-byte inputs are passed through untouched (the kernels treat
        any non-zero byte as 1; a pinned buffer stays pinned); wider dtypes (PyMC holds the Bernoulli
        values as int64) are converted once."""
        a = np.asarray(a)
        if a.dtype.itemsize == 1 and a.flags.c_contiguous:
            return a.view(np.int8).reshape(shape)
        return np.ascontiguousarray(a != 0, dtype=np.int8).reshape(shape)

    @staticmethod
    def _chains(a, width):
        a = np.asarray(a, dtype=np.float64)
        if a.shape[-1] != width:
            raise ValueError(f"expected last dimension {width}, got {a.shape}")
        return 1 if a.ndim == 1 else int(a.shape[0]), a.ndim == 1

    def algorithmic_bytes_logp(self, n_chains):
        return int(self._lib.abd_algorithmic_bytes_logp(self._h, n_chains))

    def algorithmic_bytes_gibbs(self, n_chains):
        return int(self._lib.abd_algorithmic_bytes_gibbs(self._h, n_chains))

    @property
    def launch_count(self):
        return int(self._lib.abd_launch_count(self._h))

    def set_chain_offset(self, chain_offset):
        """Global index of this engine's first chain: keys the Philox streams of the Gibbs sweeps and of the HMC
        kernels, so that processes sharding the chains of one run (same seed) never share a stream."""
        check(self._lib.abd_set_chain_offset(self._h, int(chain_offset)))

    def state_touch(self):
        """Tell the library that the caller wrote into the resident int8 state (``state_dev`` pointers) itself."""
        check(self._lib.abd_state_touch(self._h))

    def set_tuning(self, rows_per_tile=0, chains_per_cta=0):
        check(self._lib.abd_set_tuning(self._h, int(rows_per_tile), int(chains_per_cta)))

    def last_plan(self) -> dict:
        """Grid plan of the most recent log-likelihood launch (tiles, chain groups, chains per CTA, shared memory,
        compact cell layout or not, resident CTAs per SM)."""
        out = np.zeros(6, dtype=np.int32)
        check(self._lib.abd_last_plan(self._h, _ptr(out)))
        keys = ("tiles", "chain_groups", "chains_per_cta", "smem_bytes", "compact_cells", "ctas_per_sm")
        return dict(zip(keys, (int(v) for v in out)))

    # ------------------------------------------------------------------------------ state
    def upload_state(self, i_raw, waner):
        i_raw = np.asarray(i_raw)
        C_ = 1 if i_raw.ndim == 2 else i_raw.shape[0]
        i8, w8 = self._state(C_, i_raw, waner)
        check(self._lib.abd_upload_state(self._h, C_, _ptr(i8), _ptr(w8)))
        return C_

    def download_state(self, n_chains):
        i8 = np.empty((n_chains, self.G, self.N), np.int8)
        w8 = np.empty((n_chains, self.N), np.int8)
        check(self._lib.abd_download_state(self._h, n_chains, _ptr(i8), _ptr(w8)))
        return i8, w8

    # ------------------------------------------------------------------------------ compute
    def loglik_grad(self, theta13, i_raw=None, waner=None):
        C_, single = self._chains(theta13, 13)
        th = _f64(theta13, (C_, 13))
        i8, w8 = self._state(C_, i_raw, waner)
        ll = np.empty(C_)
        g = np.empty((C_, 13))
        cnt = np.empty((C_, 2), np.int64)
        check(self._lib.abd_loglik_grad(self._h, C_, _ptr(th), _ptr(i8), _ptr(w8), _ptr(ll), _ptr(g), _ptr(cnt)))
        return (ll[0], g[0], cnt[0]) if single else (ll, g, cnt)

    def loglik_grad_resident(self, th_ptr, ll_ptr, g_ptr):
        """One chain, resident chain state, caller-owned buffers given as raw addresses (13 doubles in, 1 + 13 out):
        the per-leapfrog call of the PyTensor Op, without the argument handling of ``loglik_grad``."""
        rc = self._lib.abd_loglik_grad(self._h, 1, th_ptr, None, None, ll_ptr, g_ptr, None)
        if rc:
            check(rc)

    def logp_dlogp(self, q17, i_raw=None, waner=None):
        """Joint logp and gradient in PyMC's unconstrained space (what NUTS consumes).  The hot
        call of a host-driven sampler: output buffers and their addresses are cached per chain
        count, the results are returned as fresh copies."""
        C_, single = self._chains(q17, 17)
        q = _f64(q17, (C_, 17))
        i8, w8 = self._state(C_, i_raw, waner)
        buf = self._out17.get(C_)
        if buf is None:
            lp, g = np.empty(C_), np.empty((C_, 17))
            buf = self._out17[C_] = (lp, g, lp.ctypes.data, g.ctypes.data)
        lp, g, p_lp, p_g = buf
        rc = self._lib.abd_logp_dlogp(self._h, C_, q.ctypes.data, _ptr(i8), _ptr(w8), p_lp, p_g)
        if rc:
            check(rc)
        return (lp[0], g[0].copy()) if single else (lp.copy(), g.copy())

    def cond_logodds(self, theta13, p, p_w, i_raw=None, waner=None):
        C_, single = self._chains(theta13, 13)
        th = _f64(theta13, (C_, 13))
        pp, pw = _f64(p, (C_,)), _f64(p_w, (C_,))
        i8, w8 = self._state(C_, i_raw, waner)
        oi = np.empty((C_, self.G, self.N))
        ow = np.empty((C_, self.N))
        check(self._lib.abd_cond_logodds(self._h, C_, _ptr(th), _ptr(pp), _ptr(pw), _ptr(i8), _ptr(w8), _ptr(oi), _ptr(ow)))
        return (oi[0], ow[0]) if single else (oi, ow)

    def gibbs_sweep(self, theta13, p, p_w, i_raw=None, waner=None, seed=0, sweep=0,
                    mode=_lib.GIBBS_METROPOLIS, transit_p=0.8, download=True, inplace=False):
        """Returns (i_raw, waner, stats) -- updated copies (or (None, None, stats) when
        ``download=False``: the new state stays resident on the device).  ``inplace=True``: the
        int8 arrays passed in are updated in place in ONE call (abd_gibbs_sweep's in/out
        contract); with pinned arrays both directions then go over PCIe by SM copy kernels."""
        C_, single = self._chains(theta13, 13)
        th = _f64(theta13, (C_, 13))
        pp, pw = _f64(p, (C_,)), _f64(p_w, (C_,))
        i8, w8 = self._state(C_, i_raw, waner)
        st = np.zeros((C_, 2), np.int64)
        if inplace:
            if i8 is None or not (i8.flags.writeable and w8.flags.writeable and np.may_share_memory(i8, np.asarray(i_raw))):
                raise ValueError("inplace=True needs writable, contiguous one-byte i_raw / waner arrays")
            check(self._lib.abd_gibbs_sweep(self._h, C_, _ptr(th), _ptr(pp), _ptr(pw), _ptr(i8), _ptr(w8),
                                            int(seed), int(sweep), int(mode), float(transit_p), _ptr(st)))
            return i_raw, waner, (st[0] if single else st)
        if i8 is not None:
            check(self._lib.abd_upload_state(self._h, C_, _ptr(i8), _ptr(w8)))
        check(self._lib.abd_gibbs_sweep(self._h, C_, _ptr(th), _ptr(pp), _ptr(pw), None, None,
                                        int(seed), int(sweep), int(mode), float(transit_p), _ptr(st)))
        if not download:
            return None, None, (st[0] if single else st)
        i8, w8 = self.download_state(C_)
        return (i8[0], w8[0], st[0]) if single else (i8, w8, st)

    def deterministics(self, theta13, i_raw=None, waner=None):
        C_, single = self._chains(theta13, 13)
        th = _f64(theta13, (C_, 13))
        i8, w8 = self._state(C_, i_raw, waner)
        oi = np.empty((C_, self.G, self.N), np.int8)
        mn = np.empty((C_, self.G, self.N))
        ms = np.empty((C_, self.G, self.N))
        check(self._lib.abd_deterministics(self._h, C_, _ptr(th), _ptr(i8), _ptr(w8), _ptr(oi), _ptr(mn), _ptr(ms)))
        return (oi[0], mn[0], ms[0]) if single else (oi, mn, ms)

    def loglik_rows(self, theta13, i_raw=None, waner=None):
        """Pointwise log-likelihood of every OD row, (it_s_lik (C, R_s), it_n_lik (C, R_n)), rows in the cohort's order
        per antigen: the InferenceData's log_likelihood group (abd.py:459-469)."""
        C_, single = self._chains(theta13, 13)
        th = _f64(theta13, (C_, 13))
        i8, w8 = self._state(C_, i_raw, waner)
        ls, ln = np.empty((C_, self.R_s)), np.empty((C_, self.R_n))
        check(self._lib.abd_loglik_rows(self._h, C_, _ptr(th), _ptr(i8), _ptr(w8), _ptr(ls), _ptr(ln)))
        return (ls[0], ln[0]) if single else (ls, ln)

    # ------------------------------------------------------------------------------ device API
    # Arguments are raw device addresses (ints, e.g. torch.Tensor.data_ptr()) and a stream handle.
    def state_dev(self, n_chains):
        a, b = C.c_void_p(), C.c_void_p()
        check(self._lib.abd_state_dev(self._h, n_chains, C.byref(a), C.byref(b)))
        return a.value, b.value

    def sums_dev(self, C_, theta, theta_is_q17, i_raw, waner, sums, stream=0):
        check(self._lib.abd_sums_dev(self._h, C_, theta, int(theta_is_q17), i_raw, waner, sums, stream))

    def finalize_logp_dev(self, C_, q17, sums, out_logp, out_dlogp, stream=0):
        check(self._lib.abd_finalize_logp_dev(self._h, C_, q17, sums, out_logp, out_dlogp, stream))

    def finalize_loglik_dev(self, C_, theta13, sums, out_ll, out_grad, stream=0):
        check(self._lib.abd_finalize_loglik_dev(self._h, C_, theta13, sums, out_ll, out_grad, stream))

    def loglik_grad_dev(self, C_, theta13, i_raw, waner, out_ll, out_grad, stream=0):
        check(self._lib.abd_loglik_grad_dev(self._h, C_, theta13, i_raw, waner, out_ll, out_grad, stream))

    def logp_dlogp_dev(self, C_, q17, i_raw, waner, out_logp, out_dlogp, stream=0):
        check(self._lib.abd_logp_dlogp_dev(self._h, C_, q17, i_raw, waner, out_logp, out_dlogp, stream))

    def gibbs_sweep_dev(self, C_, theta, theta_is_q17, p, p_w, i_raw, waner, seed, sweep,
                        mode=_lib.GIBBS_METROPOLIS, transit_p=0.8, stats=None, stream=0):
        check(self._lib.abd_gibbs_sweep_dev(self._h, C_, theta, int(theta_is_q17), p, p_w, i_raw, waner,
                                            int(seed), int(sweep), int(mode), float(transit_p), stats, stream))

    def leapfrog_dev(self, C_, n_steps, q17, p17, grad17, logp, eps, inv_mass, i_raw, waner, stream=0):
        check(self._lib.abd_leapfrog_dev(self._h, C_, int(n_steps), q17, p17, grad17, logp, eps, inv_mass, i_raw, waner, stream))

    def leapfrog_status(self, C_):
        check(self._lib.abd_leapfrog_status(self._h, C_))

    def hmc_begin_dev(self, C_, q17, grad17, logp, linv_t, seed, it, qw, pw, gw, h0, stream=0):
        check(self._lib.abd_hmc_begin_dev(self._h, C_, q17, grad17, logp, linv_t, int(seed), int(it), qw, pw, gw, h0, stream))

    def hmc_end_dev(self, C_, q17, grad17, logp, qw, pw, gw, lpw, inv_mass, h0, seed, it, accept_out, da, eps, adapt,
                    target_accept, stream=0):
        check(self._lib.abd_hmc_end_dev(self._h, C_, q17, grad17, logp, qw, pw, gw, lpw, inv_mass, h0, int(seed), int(it),
                                        accept_out, da, eps, int(adapt), float(target_accept), stream))

    # the No-U-Turn tree on the device, see include/abd_b200.h
    def nuts_state_doubles(self, max_depth):
        return int(self._lib.abd_nuts_state_doubles(int(max_depth)))

    def nuts_begin_dev(self, C_, max_depth, q17, grad17, logp, linv_t, eps, seed, it, state, qw, pw, gw, eps_signed, any_active,
                       stream=0):
        check(self._lib.abd_nuts_begin_dev(self._h, C_, int(max_depth), q17, grad17, logp, linv_t, eps, int(seed), int(it), state,
                                           qw, pw, gw, eps_signed, any_active, stream))

    def nuts_leaf_dev(self, C_, max_depth, depth, leaf, qw, pw, gw, lpw, inv_mass, eps, seed, it, state, eps_signed, any_active,
                      stream=0):
        check(self._lib.abd_nuts_leaf_dev(self._h, C_, int(max_depth), int(depth), int(leaf), qw, pw, gw, lpw, inv_mass, eps,
                                          int(seed), int(it), state, eps_signed, any_active, stream))

    def nuts_extend_dev(self, C_, max_depth, depth, qw, pw, gw, lpw, inv_mass, eps, seed, it, state, eps_signed, any_active,
                        i_raw, waner, stream=0):
        check(self._lib.abd_nuts_extend_dev(self._h, C_, int(max_depth), int(depth), qw, pw, gw, lpw, inv_mass, eps, int(seed),
                                            int(it), state, eps_signed, any_active, i_raw, waner, stream))

    def nuts_end_dev(self, C_, max_depth, q17, grad17, logp, state, accept_out, depth_out, diverged_out, da, eps, adapt,
                     target_accept, stream=0):
        check(self._lib.abd_nuts_end_dev(self._h, C_, int(max_depth), q17, grad17, logp, state, accept_out, depth_out, diverged_out,
                                         da, eps, int(adapt), float(target_accept), stream))

    # peer exchange (fused all-reduce over NVLink), see include/abd_b200.h
    def xch_alloc(self, world, rank, max_chains) -> bytes:
        buf = C.create_string_buffer(64)
        check(self._lib.abd_xch_alloc(self._h, int(world), int(rank), int(max_chains), buf))
        return buf.raw

    def xch_connect(self, handles):
        blob = b"".join(handles)
        check(self._lib.abd_xch_connect(self._h, C.c_char_p(blob)))

    def logp_dlogp_sharded_dev(self, C_, q17, i_raw, waner, out_logp, out_dlogp, stream=0):
        check(self._lib.abd_logp_dlogp_sharded_dev(self._h, C_, q17, i_raw, waner, out_logp, out_dlogp, stream))

    def xch_status(self):
        check(self._lib.abd_xch_status(self._h))

    def leapfrog_sharded_dev(self, C_, q17, p17, grad17, logp, eps, inv_mass, i_raw, waner, stream=0):
        check(self._lib.abd_leapfrog_sharded_dev(self._h, C_, q17, p17, grad17, logp, eps, inv_mass, i_raw, waner, stream))

    def xch_stats(self, reset=False):
        """(ns waited for each peer [8], exchanges done): the fused all-reduce's cost apart from compute."""
        out = np.zeros(9, np.uint64)
        check(self._lib.abd_xch_stats(self._h, out.ctypes.data, int(reset)))
        return out[:8].copy(), int(out[8])

    def loglik_rows_dev(self, C_, theta13, i_raw, waner, out_s, out_n, stream=0):
        check(self._lib.abd_loglik_rows_dev(self._h, C_, theta13, i_raw, waner, out_s, out_n, stream))

    def deterministics_dev(self, C_, theta13, i_raw, waner, out_i, out_mu_n, out_mu_s, stream=0):
        check(self._lib.abd_deterministics_dev(self._h, C_, theta13, i_raw, waner, out_i, out_mu_n, out_mu_s, stream))

    def deterministics_accum_dev(self, C_, theta, theta_is_q17, i_raw, waner, sum_i, sum_mu_n, sum_mu_s, stream=0):
        """Adds the sum over chains of i, ab_n_mu, ab_s_mu (G, N) to the running totals (device pointers)."""
        check(self._lib.abd_deterministics_accum_dev(self._h, C_, theta, int(theta_is_q17), i_raw, waner, sum_i, sum_mu_n,
                                                     sum_mu_s, stream))

    def infection_probs_accum_dev(self, C_, q17, i_raw, waner, sum_i, sum_w, stream=0):
        """Adds, summed over the chains, the Rao-Blackwellised infection probabilities (G, N) to ``sum_i`` and the waner
        probabilities (N,) to ``sum_w`` (device pointers): the exact conditional probability of each constrained
        infection given the rest of the state, and of ab_s_waner = 1 given theta and i_raw."""
        check(self._lib.abd_infection_probs_accum_dev(self._h, C_, q17, i_raw, waner, sum_i, sum_w, stream))
