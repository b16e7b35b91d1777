"""Host-side mirror of the reference interface for the inference hot path (abdpymc/abd.py).

Same names, argument meaning and error behaviour as the reference for this path:

  ``model(data, splits=None, ignore_pcrpos=False)``   abd.py:396-442  -> pm.Model with the same RV
      names / dims (p, i_raw, ab_n_*, ab_s_*, it_*; Deterministics i, ab_n_mu, ab_s_mu with dims
      ("gap", "ind")), but the data likelihood is ONE opaque PyTensor Op backed by the CUDA
      library (``AbdLogLik``) wrapped in ``pm.Potential("loglik", ...)``.
  ``GpuBinaryGibbs``  the step method that replaces PyMC's BinaryGibbsMetropolis for ``i_raw`` and
      ``ab_s_waner`` (assigned implicitly by ``pm.sample`` at abd.py:922).
  ``main()``          ``abdpymc-infer`` with the reference's flags (abd.py:885-924).

PyMC / PyTensor / ArviZ are import-guarded: they are not installable in the offline build image,
so everything PyMC-facing here is written against the PyMC 5 API, executed against a protocol
stand-in in tests/test_gpu_pymc_glue.py (tests/fake_pymc.py) and against PyMC itself where it
exists (tests/test_pymc_parity.py, skipped otherwise).  Without PyMC, ``main()`` drives the
built-in sampler (abdpymc_b200.sampler) on the same model terms and writes the same variable
names to an .npz (or NetCDF when ArviZ is importable).  There is no CPU fallback for the
numerics: every path goes through libabd_b200.so.
"""

from __future__ import annotations

import argparse
import sys

import numpy as np

from .cohort import CohortArrays
from .engine import Q17, Q17_RV, Q_OF_THETA, Q_P, Q_PW, THETA13, AbdEngine, backward, forward

GAP_IND = "gap", "ind"  # abd.py:18

try:  # pragma: no cover - PyMC is absent from the build image
    import pymc as pm
    import pytensor.tensor as pt
    from pytensor.gradient import grad_undefined
    from pytensor.graph.basic import Apply
    from pytensor.graph.op import Op

    HAVE_PYMC = True
except ImportError:
    pm = pt = None
    Op = object
    HAVE_PYMC = False


def check_splits(splits, data=None):
    """abd.py:604-622, same messages."""
    if splits is not None:
        if any(split < 0 for split in splits):
            raise ValueError("split indexes must be positive")
        if sorted(splits) != list(splits):
            raise ValueError("splits must be in ascending order")
        if data is not None and splits and splits[-1] > data.n_gaps:
            raise ValueError(f"largest split must be less than n_gaps - 1, ({splits[-1]})")
        if len(splits) != len(set(splits)):
            raise ValueError("splits not unique")
        if any(not isinstance(split, (int, np.integer)) for split in splits):
            raise ValueError("splits must be ints")


def as_cohort(data) -> CohortArrays:
    """Accepts a CohortArrays or the reference's ``TiterData`` (abd.py:46-126: ``vacs``, ``pcrpos``
    (n_inds, n_gaps) and ``s.df`` / ``n.df`` with individual_i, elapsed_months, log_dilution, od)."""
    if isinstance(data, CohortArrays):
        return data
    rows = []
    for a, ag in ((0, data.n), (1, data.s)):
        df = ag.df
        rows.append((np.asarray(ag.idx_ind), np.asarray(ag.idx_gap), np.full(len(df), a),
                     df["log_dilution"].to_numpy(float), df["od"].to_numpy(float)))
    ind, gap, antigen, x, od = (np.concatenate(c) for c in zip(*rows))
    return CohortArrays(vacs=np.asarray(data.vacs), pcrpos=np.asarray(data.pcrpos), ind=ind, gap=gap, antigen=antigen,
                        x=x, od=od, t0=str(getattr(data, "t0", "2020-05")))


def make_engine(data, splits=None, ignore_pcrpos=False, device=0, **kw) -> AbdEngine:
    cohort = as_cohort(data)
    check_splits(splits, cohort)
    if splits is not None and len(splits) > 2:
        raise NotImplementedError("only implemented 1-3 time chunks (0-2 splits)")  # abd.py:881-882
    return AbdEngine(cohort, splits=splits, ignore_pcrpos=ignore_pcrpos, device=device, **kw)


# ------------------------------------------------------------------------------------------
# PyTensor Ops
# ------------------------------------------------------------------------------------------
class _Cache:
    """Shared by the Ops of one model and its ``GpuBinaryGibbs`` step.

    * Value and gradient come out of one kernel launch; NUTS asks for both at the same point.
    * The binaries (``i_raw`` 2.5 MB of int64 at 10k individuals, ``ab_s_waner``) only change once per
      Gibbs sweep, NUTS evaluates dozens of leapfrogs in between: they travel to the GPU only when they
      changed.  "Unchanged" is decided without touching their bytes on the hot path: PyTensor hands
      ``perform`` the SAME ndarray objects (the storage of the shared "extra values") until PyMC sets new
      ones, so object identity with the arrays seen last time is the test; when the objects are new
      (once per sweep) their contents are compared once with the host copy of what the sweep left on the
      device, and only a real difference (a new chain's initial point, a user evaluating some other
      point) costs an upload.  Inputs are assumed not to be mutated in place between calls (PyTensor /
      PyMC never do); ``strict=True`` compares contents on every call instead.
    """

    def __init__(self, engine, strict=False):
        self.engine, self.strict = engine, strict
        self.key, self.val = None, None
        self._seen = None   # (i_raw, waner) objects known to equal the resident state
        self._host = None   # one-byte copies of the resident state
        self._returned = None
        self.uploads = 0
        # buffers of the per-leapfrog call, allocated once
        self._th, self._ll, self._g = np.empty(13), np.empty(1), np.empty(13)
        self._ptrs = (self._th.ctypes.data, self._ll.ctypes.data, self._g.ctypes.data)

    def note_resident(self, i8, w8, as_returned=None):
        """The device state is now (i8, w8): called by the Gibbs step after a sweep.  ``as_returned``: the same state in
        the dtype handed back to PyMC (int64), so that the one comparison per step is between arrays of one dtype."""
        self._host, self._seen, self.key = (i8, w8), None, None
        self._returned = as_returned

    def binaries_resident(self, i_raw, waner) -> bool:
        if not self.strict and self._seen is not None and self._seen[0] is i_raw and self._seen[1] is waner:
            return True
        h = self._host
        r = self._returned
        if r is not None and r[0].dtype == getattr(i_raw, "dtype", None) and r[0].shape == np.shape(i_raw):
            h = r   # same dtype: a plain memory comparison
        if h is not None and h[0].shape == np.shape(i_raw) and np.array_equal(h[0], i_raw) and np.array_equal(h[1], waner):
            self._seen = (i_raw, waner)
            return True
        return False

    def ensure_resident(self, i_raw, waner):
        i_raw, waner = np.asarray(i_raw), np.asarray(waner)
        if self.binaries_resident(i_raw, waner):
            return
        i8 = np.ascontiguousarray(i_raw != 0, dtype=np.int8)
        w8 = np.ascontiguousarray(waner != 0, dtype=np.int8)
        self.engine.upload_state(i8, w8)
        self.uploads += 1
        self._host, self._seen, self.key = (i8, w8), (i_raw, waner), None

    def get(self, inputs):
        th = self._th
        th[:] = inputs[:13]
        self.ensure_resident(inputs[13], inputs[14])
        key = th.tobytes()
        if key != self.key:
            self.engine.loglik_grad_resident(*self._ptrs)   # chain state resident: 13 scalars in, 14 out
            self.key, self.val = key, (float(self._ll[0]), self._g.copy())
        return self.val


class AbdLogLik(Op):
    """loglik(theta13..., i_raw, ab_s_waner) -> scalar: the sum of the two observed Normal
    log-densities of abd.py:445-469 given the response model of abd.py:309-393."""

    __props__ = ()

    def __init__(self, engine, cache=None):
        self.engine = engine
        self.cache = cache or _Cache(engine)
        self.grad_op = None

    def make_node(self, *inputs):
        if len(inputs) != 15:
            raise ValueError("AbdLogLik takes the 13 likelihood scalars, i_raw and ab_s_waner")
        theta = [pt.as_tensor_variable(v).astype("float64") for v in inputs[:13]]
        binaries = [pt.as_tensor_variable(v) for v in inputs[13:]]
        return Apply(self, [*theta, *binaries], [pt.dscalar()])

    def perform(self, node, inputs, output_storage):
        output_storage[0][0] = np.asarray(self.cache.get(inputs)[0], dtype=np.float64)

    def grad(self, inputs, output_grads):
        if self.grad_op is None:
            self.grad_op = AbdLogLikGrad(self.engine, self.cache)
        (gz,) = output_grads
        parts = self.grad_op(*inputs)
        return [gz * g for g in parts] + [grad_undefined(self, 13, inputs[13]), grad_undefined(self, 14, inputs[14])]


class AbdLogLikGrad(Op):
    """d loglik / d theta13 (13 scalars), from the same launch as the value."""

    __props__ = ()

    def __init__(self, engine, cache):
        self.engine, self.cache = engine, cache

    def make_node(self, *inputs):
        inputs = [pt.as_tensor_variable(v) for v in inputs]
        return Apply(self, inputs, [pt.dscalar() for _ in range(13)])

    def perform(self, node, inputs, output_storage):
        g = self.cache.get(inputs)[1]
        for k in range(13):
            output_storage[k][0] = g[k:k + 1].reshape(())   # 0-d float64 views of the fresh copy


class AbdDeterministics(Op):
    """(i, ab_n_mu, ab_s_mu), each (gap, ind): abd.py:649 / 667, :341, :389-391."""

    __props__ = ()

    def __init__(self, engine, cache=None):
        self.engine, self.cache = engine, cache

    def make_node(self, *inputs):
        inputs = [pt.as_tensor_variable(v) for v in inputs]
        return Apply(self, inputs, [pt.bmatrix(), pt.dmatrix(), pt.dmatrix()])

    def perform(self, node, inputs, output_storage):
        th = np.array([float(v) for v in inputs[:13]], dtype=np.float64)
        if self.cache is not None:
            self.cache.ensure_resident(inputs[13], inputs[14])
            i, mn, ms = self.engine.deterministics(th)
        else:
            i, mn, ms = self.engine.deterministics(th, inputs[13], inputs[14])
        output_storage[0][0], output_storage[1][0], output_storage[2][0] = i, mn, ms


def model(data, splits=None, ignore_pcrpos=False, device=0):
    """Set up the antibody dynamics model (abd.py:396-442) with the GPU likelihood.

    Same RVs, priors and names as the reference; the only structural difference is that
    ``it_n_lik`` / ``it_s_lik`` (observed Normals) are replaced by ``pm.Potential("loglik")``.
    The engine is attached as ``model.abd_engine`` for ``GpuBinaryGibbs``."""
    if not HAVE_PYMC:
        raise ImportError("abdpymc_b200.abd.model needs PyMC; use abdpymc_b200.sampler without it")
    cohort = as_cohort(data)
    engine = make_engine(cohort, splits=splits, ignore_pcrpos=ignore_pcrpos, device=device)
    coords = dict(ind=np.arange(cohort.n_inds), gap=np.arange(cohort.n_gaps))  # abd.py:126
    with pm.Model(coords=coords) as m:
        p = pm.Beta("p", alpha=1, beta=cohort.n_gaps - 1)  # abd.py:424
        i_raw = pm.Bernoulli("i_raw", p, dims=GAP_IND)  # abd.py:427
        n_perm = pm.Gamma("ab_n_perm", mu=2.0, sigma=0.5)  # abd.py:329
        n_temp = pm.Gamma("ab_n_temp", mu=1.0, sigma=0.5)  # abd.py:333
        n_rho = pm.Beta("ab_n_rho", alpha=10.0, beta=1.0)  # abd.py:334
        n_init = pm.Normal("ab_n_init", -2, 1)  # abd.py:340
        s_perm = pm.Gamma("ab_s_perm", mu=2.0, sigma=0.5)  # abd.py:367
        s_rho = pm.Beta("ab_s_rho", alpha=10.0, beta=1.0)  # abd.py:371
        p_waner = pm.Beta("ab_s_p_waner", alpha=1.0, beta=1.0)  # abd.py:372
        waner = pm.Bernoulli("ab_s_waner", p=p_waner, dims="ind")  # abd.py:373
        pm.Gamma("ab_s_tempinf", mu=1.0, sigma=0.5)  # abd.py:377 -- prior only (abd.py:263-274 ignores temp)
        pm.Gamma("ab_s_tempvac", mu=1.0, sigma=0.5)  # abd.py:383
        s_init = pm.Normal("ab_s_init", -2, 1)  # abd.py:388
        n_b, n_d = pm.Normal("it_n_b", -1, 0.5), pm.Normal("it_n_d", 2, 0.5)  # abd.py:464-465
        n_sigma = pm.Exponential("it_n_sigma", 1)  # abd.py:467
        s_b, s_d = pm.Normal("it_s_b", -1, 0.5), pm.Normal("it_s_d", 2, 0.5)
        s_sigma = pm.Exponential("it_s_sigma", 1)
        theta = [n_perm, n_temp, n_rho, n_init, s_perm, s_rho, s_init, n_b, n_d, n_sigma, s_b, s_d, s_sigma]
        cache = _Cache(engine)
        pm.Potential("loglik", AbdLogLik(engine, cache)(*theta, i_raw, waner))
        i, mu_n, mu_s = AbdDeterministics(engine, cache)(*theta, i_raw, waner)
        pm.Deterministic("i", i, dims=GAP_IND)
        pm.Deterministic("ab_n_mu", mu_n, dims=GAP_IND)
        pm.Deterministic("ab_s_mu", mu_s, dims=GAP_IND)
    m.abd_engine, m.abd_cache = engine, cache
    return m


# ------------------------------------------------------------------------------------------
# PyMC step method
# ------------------------------------------------------------------------------------------
def point_to_q17(point) -> np.ndarray:
    """PyMC point dict (value-variable names, abd.py declaration order) -> q17."""
    return np.array([float(point[name]) for name in Q17], dtype=np.float64)


if HAVE_PYMC:  # pragma: no cover
    from pymc.step_methods.arraystep import BlockedStep
    from pymc.step_methods.compound import Competence

    class GpuBinaryGibbs(BlockedStep):
        """Drop-in for BinaryGibbsMetropolis over ``i_raw`` and ``ab_s_waner``:
        ``pm.sample(step=[GpuBinaryGibbs([m["i_raw"], m["ab_s_waner"]], model=m)])``.
        One ``step`` = one ``abd_gibbs_sweep`` (same per-bit transition kernel: flip proposed
        w.p. ``transit_p``, Metropolis accept; individuals updated in parallel, each in a
        uniformly random order)."""

        name = "gpu_binary_gibbs"
        stats_dtypes_shapes = {"p_jump": (float, []), "tune": (bool, [])}
        stats_dtypes = [{"p_jump": float, "tune": bool}]  # PyMC < 5.7 spelling

        def __new__(cls, vars=None, model=None, **kwargs):
            # BlockedStep.__new__ needs `vars`: fill in the model's two binary RVs when they are not given
            model = pm.modelcontext(model)
            if vars is None:
                vars = [model["i_raw"], model["ab_s_waner"]]
            return super().__new__(cls, vars=vars, model=model, **kwargs)

        def __init__(self, vars=None, model=None, transit_p=0.8, mode=0, seed=None, **kwargs):
            model = pm.modelcontext(model)
            vars = vars or [model["i_raw"], model["ab_s_waner"]]
            self.vars = [model.rvs_to_values.get(v, v) for v in vars]
            self.engine = model.abd_engine
            self.cache = getattr(model, "abd_cache", None)
            self.transit_p, self.mode = transit_p, mode
            self.seed = int(np.random.SeedSequence(seed).generate_state(1, dtype=np.uint64)[0])
            self.sweep, self.tune = 0, True
            self.model = model

        def step(self, point):
            q = point_to_q17(point)
            x = backward(q)
            if self.cache is not None:
                # the binaries NUTS has just been evaluating are already on the device: sweep them there,
                # and tell the Ops what the device holds afterwards (no upload on the next leapfrog)
                self.cache.ensure_resident(point["i_raw"], point["ab_s_waner"])
                i_raw, waner, st = self.engine.gibbs_sweep(x[Q_OF_THETA], x[Q_P], x[Q_PW], seed=self.seed, sweep=self.sweep,
                                                           mode=self.mode, transit_p=self.transit_p)
            else:
                i_raw, waner, st = self.engine.gibbs_sweep(x[Q_OF_THETA], x[Q_P], x[Q_PW], point["i_raw"],
                                                           point["ab_s_waner"], seed=self.seed, sweep=self.sweep,
                                                           mode=self.mode, transit_p=self.transit_p)
            self.sweep += 1
            new = dict(point)
            new["i_raw"] = i_raw.astype(np.asarray(point["i_raw"]).dtype)
            new["ab_s_waner"] = waner.astype(np.asarray(point["ab_s_waner"]).dtype)
            if self.cache is not None:
                self.cache.note_resident(i_raw, waner, (new["i_raw"], new["ab_s_waner"]))
            return new, [{"p_jump": float(st[1]) / max(float(st[0]), 1.0), "tune": self.tune}]

        def stop_tuning(self):
            self.tune = False

        @staticmethod
        def competence(var, has_grad):
            return Competence.COMPATIBLE if var.name in ("i_raw", "ab_s_waner") else Competence.INCOMPATIBLE


def pointwise_log_likelihood(engine, posterior, batch=64):
    """The InferenceData's ``log_likelihood`` group for the two observed nodes of the reference model
    (``it_s_lik`` / ``it_n_lik``, abd.py:459-469), which the GPU model replaces by one ``pm.Potential``:
    {"it_s_lik": (chain, draw, R_s), "it_n_lik": (chain, draw, R_n)} from posterior draws of the 13 likelihood
    scalars, ``i_raw`` (chain, draw, gap, ind) and ``ab_s_waner`` (chain, draw, ind) -- what ``az.loo`` / ``az.waic``
    read.  ``posterior``: mapping name -> array (an InferenceData's posterior group works)."""
    th = np.stack([np.asarray(posterior[n], dtype=np.float64) for n in THETA13], axis=-1)      # (chain, draw, 13)
    i_raw, w = np.asarray(posterior["i_raw"]), np.asarray(posterior["ab_s_waner"])
    n_c, n_d = th.shape[:2]
    flat_th = th.reshape(-1, 13)
    flat_i = i_raw.reshape((-1,) + i_raw.shape[2:])
    flat_w = w.reshape((-1,) + w.shape[2:])
    ls, ln = np.empty((n_c * n_d, engine.R_s)), np.empty((n_c * n_d, engine.R_n))
    for k in range(0, n_c * n_d, batch):
        a, b = engine.loglik_rows(flat_th[k:k + batch], flat_i[k:k + batch] != 0, flat_w[k:k + batch] != 0)
        ls[k:k + batch], ln[k:k + batch] = np.atleast_2d(a), np.atleast_2d(b)
    return {"it_s_lik": ls.reshape(n_c, n_d, -1), "it_n_lik": ln.reshape(n_c, n_d, -1)}


def infection_probabilities(engine, posterior, batch=64):
    """Rao-Blackwellised posterior infection and waner probabilities from posterior draws of the 17 scalars,
    ``i_raw`` (chain, draw, gap, ind) and ``ab_s_waner`` (chain, draw, ind): {"i_rb": (gap, ind), "ab_s_waner_rb": (ind,)},
    the average over the draws of the exact conditional probability of each constrained infection given the rest of the
    draw's state, and of ab_s_waner = 1 given the draw's scalars and i_raw.  They estimate the same quantities as the
    mean of the Deterministic ``i`` and of ``ab_s_waner`` over the draws, with smaller Monte-Carlo error.
    ``posterior``: mapping name -> array (an InferenceData's posterior group works)."""
    import torch

    x = np.stack([np.asarray(posterior[n], dtype=np.float64) for n, _ in Q17_RV], axis=-1)      # (chain, draw, 17)
    i_raw, w = np.asarray(posterior["i_raw"]), np.asarray(posterior["ab_s_waner"])
    q = forward(x.reshape(-1, 17))
    flat_i = i_raw.reshape((-1,) + i_raw.shape[2:])
    flat_w = w.reshape((-1,) + w.shape[2:])
    n = len(q)
    dev = torch.device("cuda", engine.device)
    sum_i = torch.zeros(engine.G, engine.N, dtype=torch.float64, device=dev)
    sum_w = torch.zeros(engine.N, dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    for k in range(0, n, batch):
        b = min(batch, n - k)
        qd = torch.from_numpy(np.ascontiguousarray(q[k:k + b])).to(dev)
        i8 = torch.from_numpy(np.ascontiguousarray(flat_i[k:k + b] != 0, dtype=np.int8)).to(dev)
        w8 = torch.from_numpy(np.ascontiguousarray(flat_w[k:k + b] != 0, dtype=np.int8)).to(dev)
        engine.infection_probs_accum_dev(b, qd.data_ptr(), i8.data_ptr(), w8.data_ptr(), sum_i.data_ptr(), sum_w.data_ptr(), st)
    torch.cuda.synchronize(dev)
    return {"i_rb": (sum_i / n).cpu().numpy(), "ab_s_waner_rb": (sum_w / n).cpu().numpy()}


# ------------------------------------------------------------------------------------------
# abdpymc-infer
# ------------------------------------------------------------------------------------------
def infer_builtin(cohort, splits, ignore_pcrpos, tune, draws, chains=4, device=0, seed=0, progress=None, gibbs_mode=0,
                  thinned=0, kernel="hmc", shard=None, rank=0, world=1, engine=None, rao_blackwell=False):
    """tune + draws iterations of the built-in HMC + GPU-Gibbs sampler.  Returns (result,
    {name: array (chain, draw, ...)}, last binary state) with the reference's posterior variable names.
    ``rao_blackwell``: ``result.means`` also holds the Rao-Blackwellised infection and waner probabilities
    ``i_rb`` (G, N) and ``ab_s_waner_rb`` (N,) (``SamplerConfig.rao_blackwell``).

    ``shard`` (one process per GPU, ``torch.distributed`` initialised, ``world`` ranks):
      "individuals": the cohort is split into contiguous blocks of individuals, one per rank; the 17 scalars
          are replicated and every evaluation all-reduces C x 16 sums inside the kernel (NVLink peer memory);
          every rank returns the same draws, Deterministic means / last state are gathered over the blocks;
      "chains": every rank holds the whole cohort and chains / world of the chains (no communication until the
          draws are gathered; RNG streams keyed by global chain)."""
    import torch

    from .sampler import AbdTarget, SamplerConfig, sample

    if engine is None:
        cohort = as_cohort(cohort)
        G, N = cohort.n_gaps, cohort.n_inds
    else:  # a ready engine (AbdEngine.from_cache): the cohort never exists on the host
        G, N = engine.G, engine.N
    rng = np.random.default_rng(seed)
    # PyMC-like initial point: prior means on the constrained scale, jittered in q space
    x0 = np.array([1.0 / G, 2, 1, 10 / 11, -2, 2, 10 / 11, 0.5, 1, 1, -2, -1, 2, 1, -1, 2, 1], dtype=np.float64)
    q0 = forward(x0)[None, :] + rng.uniform(-1, 1, size=(chains, 17))
    cfg = SamplerConfig(tune=tune, draws=draws, seed=seed, record_deterministics_every=1, thinned_deterministics=thinned,
                        kernel=kernel, rao_blackwell=rao_blackwell)
    if world > 1 and shard == "individuals":
        from .distributed import ShardedEngine, ShardedTarget

        check_splits(splits, cohort)
        sh = ShardedEngine(cohort, splits=splits, ignore_pcrpos=ignore_pcrpos, device_index=device, rank=rank, world=world,
                           fused=True, max_chains=chains)
        target = ShardedTarget(sh, chains, np.zeros((chains, G, N), np.int8), np.zeros((chains, N), np.int8), seed=seed,
                               gibbs_mode=gibbs_mode)
        cfg.thinned_deterministics = 0      # (G, N) draws of a sharded cohort are not gathered; the means are
        res = sample(target, torch.from_numpy(q0).to(target.device), cfg, progress=progress if rank == 0 else None)
        li, lw = target.state()
        post_last = dict(i_raw=target.gather_individuals(li), ab_s_waner=target.gather_individuals(lw))
        res.means = {k: target.gather_individuals(v) for k, v in res.means.items()}
        sh.close()
        return res, res.posterior(), post_last
    if engine is None:
        engine = make_engine(cohort, splits=splits, ignore_pcrpos=ignore_pcrpos, device=device)
    lo, hi = 0, chains
    if world > 1 and shard == "chains":
        from .cohort import shard_bounds

        lo, hi = shard_bounds(chains, rank, world)
        if hi <= lo:
            raise ValueError("fewer chains than GPUs")
        engine.set_chain_offset(lo)          # Philox streams keyed by GLOBAL chain: no two ranks share one
    c_loc = hi - lo
    target = AbdTarget(engine, c_loc, np.zeros((c_loc, G, N), np.int8), np.zeros((c_loc, N), np.int8), seed=seed,
                       gibbs_mode=gibbs_mode)
    res = sample(target, torch.from_numpy(q0[lo:hi]).to(target.device), cfg, progress=progress if rank == 0 else None)
    i_raw, waner = target.state()
    post_last = dict(i_raw=i_raw, ab_s_waner=waner)
    engine.close()
    if world > 1 and shard == "chains":
        import torch.distributed as dist

        parts = [None] * world
        dist.all_gather_object(parts, (res.q, res.logp, res.accept, res.step_size, res.means, res.thinned, post_last, c_loc))
        res.q, res.logp, res.accept = (np.concatenate([p[k] for p in parts], axis=0) for k in range(3))
        res.step_size = np.concatenate([p[3] for p in parts])
        tot = sum(p[7] for p in parts)
        res.means = {k: sum(p[4][k] * p[7] for p in parts) / tot for k in parts[0][4]}
        if res.thinned:
            res.thinned = {k: (v if k == "draw" else np.concatenate([p[5][k] for p in parts], axis=0)) for k, v in res.thinned.items()}
        post_last = {k: np.concatenate([p[6][k] for p in parts], axis=0) for k in post_last}
    return res, res.posterior(), post_last


def _write_builtin(args, data, res, post, last):
    out = args.netcdf or "abd_posterior.npz"
    if not out.endswith(".npz"):
        try:  # pragma: no cover - ArviZ is absent from the build image
            import arviz as az

            posterior = dict(post)
            dims, extra = {}, {}
            sample_stats = {"acceptance_rate": res.accept, "lp": res.logp, **res.stats}
            if res.thinned:  # the Deterministics only exist for the kept draws: thin everything alike
                keep = res.thinned["draw"]
                posterior = {k: v[:, keep] for k, v in posterior.items()}
                sample_stats = {k: v[:, keep] for k, v in sample_stats.items()}
                for name in ("i", "ab_n_mu", "ab_s_mu"):
                    posterior[name] = res.thinned[name]
                    dims[name] = list(GAP_IND)
                if "it_s_lik" in res.thinned:   # the reference's observed nodes (abd.py:459-469)
                    extra["log_likelihood"] = {k: res.thinned[k] for k in ("it_s_lik", "it_n_lik")}
                    if hasattr(data, "rows"):
                        extra["observed_data"] = {"it_s_lik": data.rows(1)[1], "it_n_lik": data.rows(0)[1]}
            idata = az.from_dict(posterior=posterior, sample_stats=sample_stats, dims=dims,
                                 coords={"gap": np.arange(data.n_gaps), "ind": np.arange(data.n_inds)}, **extra)
            if "i_rb" in res.means:   # no (chain, draw) axes: a Dataset, so that ArviZ does not prepend them
                import xarray as xr

                idata.add_groups(rao_blackwell=xr.Dataset(
                    {"i_rb": (GAP_IND, res.means["i_rb"]), "ab_s_waner_rb": ("ind", res.means["ab_s_waner_rb"])},
                    coords={"gap": np.arange(data.n_gaps), "ind": np.arange(data.n_inds)}))
            az.to_netcdf(idata, out)
            print(f"PyMC not installed: sampled with the built-in HMC+Gibbs driver in {res.wall_s:.1f} s; wrote {out}",
                  file=sys.stderr)
            return
        except ImportError:
            pass
    # no ArviZ: the same variables as a compressed .npz (posterior draws (chain, draw), sample_stats_* like the
    # InferenceData's sample_stats group, the Deterministics as posterior means + thinned draws, the last binary state)
    np.savez_compressed(out if out.endswith(".npz") else out + ".npz", **post, **{f"mean_{k}": v for k, v in res.means.items()},
                        **{f"last_{k}": v for k, v in last.items()}, step_size=res.step_size, wall_s=res.wall_s,
                        sample_stats_acceptance_rate=res.accept, sample_stats_lp=res.logp,
                        sample_stats_step_size=np.broadcast_to(res.step_size[:, None], res.accept.shape),
                        **{f"sample_stats_{k}": v for k, v in res.stats.items()},
                        **({"observed_data_it_s_lik": data.rows(1)[1], "observed_data_it_n_lik": data.rows(0)[1]}
                           if hasattr(data, "rows") else {}),
                        **{("thinned_draw" if k == "draw" else ("log_likelihood_" + k if k.endswith("_lik") else k)): v
                           for k, v in res.thinned.items()})
    print(f"PyMC not installed: sampled with the built-in HMC+Gibbs driver in {res.wall_s:.1f} s; wrote {out}", file=sys.stderr)


def _builtin_worker(rank, args, devices, port):
    """One process per GPU of --devices (spawned by main, or started by torchrun)."""
    import os

    world = len(devices)
    if world > 1:
        import torch
        import torch.distributed as dist

        os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1",
                          MASTER_PORT=str(port))
        torch.cuda.set_device(devices[rank])
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", devices[rank]))
    from pathlib import Path

    from .cohort import splits_from_t0

    splits = None
    if args.split_delta or args.split_omicron:
        t0 = (Path(args.ititers_data) / "t0.txt").read_text().strip()
        splits = splits_from_t0(t0, args.split_delta, args.split_omicron)
    # --cache: the preprocessed cohort as one binary file (no CSV parsing, no sorting); with the individuals
    # sharded every rank preprocesses its own block instead
    use_cache = bool(args.cache) and not (world > 1 and args.shard == "individuals")
    engine = None
    if use_cache and Path(args.cache).exists():
        engine = AbdEngine.from_cache(args.cache, device=devices[rank], splits=splits or (), ignore_pcrpos=args.ignore_pcrpos)
        data = type("Sizes", (), {"n_gaps": engine.G, "n_inds": engine.N})()
    else:
        data = CohortArrays.from_disk(args.ititers_data)
        if use_cache:
            engine = make_engine(data, splits=splits, ignore_pcrpos=args.ignore_pcrpos, device=devices[rank])
            if rank == 0:
                engine.save_cache(args.cache)
    res, post, last = infer_builtin(data, splits, args.ignore_pcrpos, args.tune, args.draws, chains=args.chains,
                                    device=devices[rank], progress=max(1, (args.tune + args.draws) // 10),
                                    gibbs_mode=args.gibbs_mode, thinned=args.thinned, kernel=args.kernel,
                                    shard=args.shard if world > 1 else None, rank=rank, world=world, engine=engine,
                                    rao_blackwell=args.rao_blackwell)
    if rank == 0:
        _write_builtin(args, data, res, post, last)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    return res


def main(argv=None):
    parser = argparse.ArgumentParser("abdpymc-infer")  # flags of abd.py:888-911
    parser.add_argument("--tune", help="Number of tuning steps.", type=int, required=True)
    parser.add_argument("--draws", help="Number of draws.", type=int, required=True)
    parser.add_argument("--cores", help="Number of cores", type=int)
    parser.add_argument("--ititers_data", help="Path to directory for generating TiterData object.", default="cohort_data")
    parser.add_argument("--split_delta", help="Split time chunk between delta and pre-delta", action="store_true")
    parser.add_argument("--split_omicron", help="Split time chunk between omicron and delta", action="store_true")
    parser.add_argument("--ignore_pcrpos", help="Ignore PCR+ data", action="store_true")
    parser.add_argument("--netcdf", help="Path of netCDF file to save.")
    parser.add_argument("--chains", type=int, default=4, help="(extension) chains batched on the GPU")
    parser.add_argument("--device", type=int, default=0, help="(extension) CUDA device")
    parser.add_argument("--devices", default=None,
                        help="(extension, PyMC-free driver) comma-separated CUDA devices of this node, one process each, e.g. "
                             "0,1,2,3,4,5,6,7; see --shard")
    parser.add_argument("--shard", default="individuals", choices=["individuals", "chains"],
                        help="(extension) with --devices: split the INDIVIDUALS over the GPUs (large cohorts; one fused "
                             "NVLink all-reduce of chains x 16 doubles per evaluation) or the CHAINS (no communication)")
    parser.add_argument("--cache", default=None,
                        help="(extension, PyMC-free driver) preprocessed-cohort file: read it if it exists (skips parsing "
                             "df.csv / vacs.txt / pcrpos.txt and the sorts of abd_create), otherwise build from "
                             "--ititers_data and write it")
    parser.add_argument("--thinned", type=int, default=250,
                        help="(extension, PyMC-free driver) evenly spaced draws of i / ab_n_mu / ab_s_mu kept per chain "
                             "(the downstream code uses <= 250: survival.py:109-114)")
    parser.add_argument("--kernel", default="hmc", choices=["hmc", "nuts"],
                        help="(extension, PyMC-free driver) transition for the 17 scalars: fused device-resident HMC "
                             "(default, fastest) or batched No-U-Turn trajectories")
    parser.add_argument("--gibbs_mode", type=int, default=0, choices=[0, 1, 2],
                        help="(extension) update rule of the indicator sweep: 0 BinaryGibbsMetropolis semantics, "
                             "1 single-site exact conditionals, 2 per-chunk block draw (include/abd_b200.h)")
    parser.add_argument("--rao_blackwell", action="store_true",
                        help="(extension, PyMC-free driver) also write the Rao-Blackwellised posterior infection and waner "
                             "probabilities (mean_i_rb (gap, ind), mean_ab_s_waner_rb (ind)): the same quantities as the "
                             "mean of i and of ab_s_waner, with smaller Monte-Carlo error")
    args = parser.parse_args(argv)
    if args.cores not in (None, 1):
        print(f"abdpymc-infer: --cores {args.cores} ignored -- the chains of a run are batched on the GPU(s) of this process "
              "(a CUDA context does not survive pm.sample's fork); use --chains / --devices", file=sys.stderr)

    if HAVE_PYMC:  # pragma: no cover
        import arviz as az

        data = CohortArrays.from_disk(args.ititers_data)
        splits = (None if (not args.split_delta) and (not args.split_omicron)
                  else data.calculate_splits(delta=args.split_delta, omicron=args.split_omicron))

        with model(data, splits=splits, ignore_pcrpos=args.ignore_pcrpos, device=args.device) as m:
            step = GpuBinaryGibbs([m["i_raw"], m["ab_s_waner"]], model=m, mode=args.gibbs_mode)
            # chains run in this process: CUDA contexts do not survive pm.sample's fork
            idata = pm.sample(tune=args.tune, draws=args.draws, cores=1, chains=args.chains, step=[step])
        az.to_netcdf(idata, args.netcdf)
        return idata

    devices = [int(d) for d in args.devices.split(",")] if args.devices else [args.device]
    if len(devices) == 1:
        return _builtin_worker(0, args, devices, 0)
    # several GPUs of this node: one process each (the CUDA context of this process is never created)
    import socket

    import torch.multiprocessing as mp

    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    mp.spawn(_builtin_worker, args=(args, devices, port), nprocs=len(devices), join=True)
    return None


if __name__ == "__main__":
    main()
