"""Built-in compound sampler: batched HMC over the 17 continuous value variables + the GPU
Gibbs sweep over the binary variables, for C chains in lockstep on one device.

The reference delegates sampling to PyMC (``pm.sample`` -> CompoundStep[NUTS,
BinaryGibbsMetropolis], abd.py:921-922).  PyMC is not installable offline, and even where it
is, a host round trip per leapfrog dominates once an evaluation costs microseconds (SURVEY.md
section 8f rank 1).  This driver keeps every chain's position, momentum, step size and mass
matrix in device tensors and calls the C ABI's device-pointer entry points directly; the model
terms it samples are exactly those of ``abd.model`` (same value variables, transforms, priors).

Kernel: Hamiltonian Monte Carlo with a dense mass matrix (the 17 scalars are strongly correlated,
e.g. ab_n_init against ab_n_perm), jittered trajectory length, step size by dual averaging
(Nesterov; Hoffman & Gelman 2014, the scheme PyMC's NUTS uses) and Stan-style windowed covariance
adaptation pooled over the chains of the batch.  It is *not* NUTS: trajectory length is fixed up to
jitter, which keeps all chains of a batch in lockstep (one kernel launch per leapfrog for all
chains).  ``SamplerConfig(kernel="nuts")`` runs batched No-U-Turn trees instead.  The binary block is
updated by ``abd_gibbs_sweep`` (Metropolised flips with BinaryGibbsMetropolis semantics by default).

``sample`` is one loop (warm-up windows, recording, result) over one of two transitions: ``_DeviceLoop``
for targets with the device-resident loop (``DeviceTarget``: ``AbdTarget``, ``distributed.ShardedTarget``),
``_HostLoop`` (torch ops) for any target with ``logp_dlogp``.  So the host logic is tested on CPU against
Gaussians with known moments (tests/test_host_logic.py).
"""

from __future__ import annotations

import time
from collections import deque
from dataclasses import dataclass, field
from functools import cached_property

import numpy as np
import torch

from .engine import Q17_RV, Q_OF_THETA, backward


class DeviceTarget:
    """A sampler target whose chain state (i_raw, waner) is resident on the GPU of ``engine``, for C chains: the
    device-resident transitions (abd_hmc_*_dev, abd_nuts_*_dev), the Gibbs sweep and the streaming Deterministic means.
    Subclasses add ``logp_dlogp_into`` and ``leapfrog_inplace``.  ``device_loop``: ``sample`` may run the loop that keeps
    every transition on the device."""

    device_loop = True
    dim = 17

    def __init__(self, engine, n_chains, device, seed, gibbs_mode, transit_p):
        self.engine, self.C, self.device = engine, n_chains, device
        self.seed, self.gibbs_mode, self.transit_p = seed, gibbs_mode, transit_p

    # the resident state's addresses are asked for on every use: the library reallocates the buffers when a
    # call with more chains than ever before arrives, and cached pointers would dangle silently
    @property
    def d_i(self):
        return self.engine.state_dev(self.C)[0]

    @property
    def d_w(self):
        return self.engine.state_dev(self.C)[1]

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def logp_dlogp(self, q):
        logp = torch.empty(self.C, dtype=torch.float64, device=self.device)
        grad = torch.empty(self.C, self.dim, dtype=torch.float64, device=self.device)
        self.logp_dlogp_into(q.contiguous(), logp, grad)
        return logp, grad

    def hmc_begin(self, q, grad, logp, linv_t, it, qw, pw, gw, h0):
        self.engine.hmc_begin_dev(self.C, q.data_ptr(), grad.data_ptr(), logp.data_ptr(), linv_t.data_ptr(), self.seed, it,
                                  qw.data_ptr(), pw.data_ptr(), gw.data_ptr(), h0.data_ptr(), self._stream())

    def hmc_end(self, q, grad, logp, qw, pw, gw, lpw, inv_mass, h0, it, acc, da, eps, adapt, target_accept):
        self.engine.hmc_end_dev(self.C, q.data_ptr(), grad.data_ptr(), logp.data_ptr(), qw.data_ptr(), pw.data_ptr(),
                                gw.data_ptr(), lpw.data_ptr(), inv_mass.data_ptr(), h0.data_ptr(), self.seed, it,
                                acc.data_ptr(), da.data_ptr(), eps.data_ptr(), adapt, target_accept, self._stream())

    def nuts_scratch(self, max_depth):
        f64 = dict(dtype=torch.float64, device=self.device)
        return (torch.zeros(self.C, self.engine.nuts_state_doubles(max_depth), **f64), torch.zeros(self.C, **f64),
                torch.zeros(max_depth + 1, dtype=torch.int32, device=self.device))

    def nuts_begin(self, D, q, grad, logp, linv_t, eps, it, state, qw, pw, gw, eps_signed, any_active):
        self.engine.nuts_begin_dev(self.C, D, q.data_ptr(), grad.data_ptr(), logp.data_ptr(), linv_t.data_ptr(), eps.data_ptr(),
                                   self.seed, it, state.data_ptr(), qw.data_ptr(), pw.data_ptr(), gw.data_ptr(),
                                   eps_signed.data_ptr(), any_active.data_ptr(), self._stream())

    def nuts_extend(self, D, j, qw, pw, gw, lpw, inv_mass, eps, it, state, eps_signed, any_active):
        """All 2^j leaves of one doubling (one leapfrog launch each, which also updates the trees) in one library call."""
        self.engine.nuts_extend_dev(self.C, D, j, qw.data_ptr(), pw.data_ptr(), gw.data_ptr(), lpw.data_ptr(), inv_mass.data_ptr(),
                                    eps.data_ptr(), self.seed, it, state.data_ptr(), eps_signed.data_ptr(), any_active.data_ptr(),
                                    self.d_i, self.d_w, self._stream())

    def nuts_end(self, D, q, grad, logp, state, acc, depth, div, da, eps, adapt, target_accept):
        self.engine.nuts_end_dev(self.C, D, q.data_ptr(), grad.data_ptr(), logp.data_ptr(), state.data_ptr(), acc.data_ptr(),
                                 depth.data_ptr(), div.data_ptr(), da.data_ptr(), eps.data_ptr(), adapt, target_accept,
                                 self._stream())

    def gibbs(self, q, sweep):
        """Sweep the binaries of every chain in place (on a sharded cohort: this rank's individuals, no collective --
        RNG streams are keyed by global individual)."""
        q = q.contiguous()
        self.engine.gibbs_sweep_dev(self.C, q.data_ptr(), 1, None, None, self.d_i, self.d_w, self.seed, sweep,
                                    mode=self.gibbs_mode, transit_p=self.transit_p, stream=self._stream())

    def accumulate_deterministics(self, q, sums):
        """Streaming posterior summaries: adds this state's i, ab_n_mu, ab_s_mu, summed over the chains,
        to ``sums`` (a dict of (G, N) float64 device tensors, created on first use) in ONE launch --
        no per-chain (C, G, N) arrays, no framework reductions."""
        G, N = self.engine.G, self.engine.N
        for name in ("i", "ab_n_mu", "ab_s_mu"):
            if name not in sums:
                sums[name] = torch.zeros(G, N, dtype=torch.float64, device=self.device)
        q = q.contiguous()
        self.engine.deterministics_accum_dev(self.C, q.data_ptr(), 1, self.d_i, self.d_w, sums["i"].data_ptr(),
                                             sums["ab_n_mu"].data_ptr(), sums["ab_s_mu"].data_ptr(), self._stream())

    def accumulate_infection_probs(self, q, sums):
        """Rao-Blackwellised posterior probabilities: adds this state's exact conditional infection probabilities
        ``sums["i_rb"]`` (G, N) and waner probabilities ``sums["ab_s_waner_rb"]`` (N,), summed over the chains, in one
        launch (float64 device tensors, created on first use).  Reads the state only; the chain is not touched."""
        G, N = self.engine.G, self.engine.N
        if "i_rb" not in sums:
            sums["i_rb"] = torch.zeros(G, N, dtype=torch.float64, device=self.device)
            sums["ab_s_waner_rb"] = torch.zeros(N, dtype=torch.float64, device=self.device)
        q = q.contiguous()
        self.engine.infection_probs_accum_dev(self.C, q.data_ptr(), self.d_i, self.d_w, sums["i_rb"].data_ptr(),
                                              sums["ab_s_waner_rb"].data_ptr(), self._stream())

    def state(self):
        """The binary state (i_raw (C, G, N), waner (C, N)); on a sharded cohort this rank's block of individuals."""
        torch.cuda.synchronize(self.device)
        return self.engine.download_state(self.C)

    def check_status(self):
        self.engine.leapfrog_status(self.C)


class AbdTarget(DeviceTarget):
    """The antibody-dynamics posterior on one GPU: joint logp + gradient over q17 for C chains
    with the chain state (i_raw, waner) resident on the device, and the Gibbs sweep over it."""

    def __init__(self, engine, n_chains, i_raw, waner, seed=0, gibbs_mode=0, transit_p=0.8):
        super().__init__(engine, n_chains, torch.device("cuda", engine.device), seed, gibbs_mode, transit_p)
        engine.upload_state(i_raw, waner)

    def logp_dlogp_into(self, q, logp, grad):
        self.engine.logp_dlogp_dev(self.C, q.data_ptr(), self.d_i, self.d_w, logp.data_ptr(), grad.data_ptr(), self._stream())

    def leapfrog_inplace(self, q, p, grad, logp, eps, inv_mass, n_steps):
        self.engine.leapfrog_dev(self.C, n_steps, q.data_ptr(), p.data_ptr(), grad.data_ptr(), logp.data_ptr(),
                                 eps.data_ptr(), inv_mass.data_ptr(), self.d_i, self.d_w, self._stream())

    @cached_property
    def _theta_of_q(self):   # per component of theta13: its back-transform (0 none, 1 exp, 2 sigmoid) and its column of q
        kinds = torch.tensor([{None: 0, "log": 1, "logodds": 2}[Q17_RV[j][1]] for j in Q_OF_THETA], device=self.device)
        return kinds, torch.tensor(Q_OF_THETA, device=self.device)

    def _theta13(self, q):
        kinds, idx = self._theta_of_q
        y = q.index_select(1, idx)
        return torch.where(kinds == 1, torch.exp(y), torch.where(kinds == 2, torch.sigmoid(y), y)).contiguous()

    def deterministics(self, q):
        """(i, ab_n_mu, ab_s_mu) of the current state, device tensors (C, G, N).  No host round
        trip: the back-transform of q runs on the device, the output buffers are reused."""
        G, N, C = self.engine.G, self.engine.N, self.C
        if not hasattr(self, "_det"):
            self._det = (torch.empty(C, G, N, dtype=torch.int8, device=self.device),
                         torch.empty(C, G, N, dtype=torch.float64, device=self.device),
                         torch.empty(C, G, N, dtype=torch.float64, device=self.device))
        oi, mn, ms = self._det
        th = self._theta13(q)
        self.engine.deterministics_dev(C, th.data_ptr(), self.d_i, self.d_w, oi.data_ptr(), mn.data_ptr(), ms.data_ptr(),
                                       self._stream())
        return oi, mn, ms

    def loglik_rows(self, q):
        """Pointwise log-likelihood of the current state: (it_s_lik (C, R_s), it_n_lik (C, R_n)) device tensors."""
        C, e = self.C, self.engine
        if not hasattr(self, "_llr"):
            self._llr = (torch.empty(C, e.R_s, dtype=torch.float64, device=self.device),
                         torch.empty(C, e.R_n, dtype=torch.float64, device=self.device))
        ls, ln = self._llr
        th = self._theta13(q)
        e.loglik_rows_dev(C, th.data_ptr(), self.d_i, self.d_w, ls.data_ptr(), ln.data_ptr(), self._stream())
        return ls, ln


@dataclass
class SamplerConfig:
    tune: int = 500
    draws: int = 500
    n_leapfrog: int = 5            # mean trajectory length in steps (tools/sampler_sweep.py: on the 10k cohort 4-5 steps
                                   # give 2-3 x the ESS/s of 12: the Gibbs <-> HMC alternation rate is what mixes)
    jitter: tuple = (0.6, 1.4)     # each trajectory: n_leapfrog x Uniform(jitter)
    target_accept: float = 0.8
    init_step: float = 0.05
    record_deterministics_every: int = 0   # 0 = never; k = accumulate means every k-th draw
    rao_blackwell: bool = False            # at the same draws, also average the exact conditional infection / waner
                                           # probabilities: means["i_rb"] (G, N), means["ab_s_waner_rb"] (N,)
    thinned_deterministics: int = 0        # keep this many evenly spaced draws of i / ab_n_mu / ab_s_mu per chain (the
                                           # consumers use <= 250: survival.py:109-114, timelines.py:289-301); 0 = none
    persistent_trajectories: bool = True   # run the whole transition on the device when the target can (``device_loop``);
                                           # False: torch ops driven from the host on any target
    single_step_launches: bool = True      # device HMC: one abd_leapfrog_dev launch per step rather than one persistent
                                           # launch per trajectory
    seed: int = 0
    kernel: str = "hmc"                    # "hmc": jittered fixed-length trajectories;
                                           # "nuts": batched multinomial No-U-Turn trajectories (what pm.sample runs for
                                           # the 17 scalars, abd.py:922), chains doubling in lockstep; tree bookkeeping on
                                           # the device when the target offers it (abd_nuts_*_dev), else torch ops
    max_treedepth: int = 8
    nuts_check_from_depth: int = 2         # device NUTS: depths below this are always built (no read-back of the "any chain
                                           # still doubling?" word before them: a read-back costs as much as two leaves)
    nuts_adaptive_checks: bool = True      # ... and so are the depths every tree of the last 32 iterations reached


@dataclass
class SamplerResult:
    q: np.ndarray                      # (chains, draws, dim) unconstrained draws
    logp: np.ndarray                   # (chains, draws)
    accept: np.ndarray                 # (chains, draws) acceptance probability of each HMC step
    step_size: np.ndarray              # (chains,)
    inv_mass: np.ndarray               # (dim, dim) adapted covariance (inverse mass matrix)
    wall_s: float
    n_grad_evals: int
    means: dict = field(default_factory=dict)   # posterior means of i, ab_n_mu, ab_s_mu (G, N); with rao_blackwell
                                                # also i_rb (G, N) and ab_s_waner_rb (N,)
    thinned: dict = field(default_factory=dict)  # i (int8), ab_n_mu, ab_s_mu (float32): (chains, kept draws, G, N); "draw" = their indexes
    stats: dict = field(default_factory=dict)   # NUTS: tree_depth, diverging (chains, draws); what PyMC puts in sample_stats
    wall_tune_s: float = 0.0           # the part of wall_s spent in the tuning iterations ...
    n_grad_evals_tune: int = 0         # ... and the gradient evaluations they took

    def posterior(self):
        """{RV name: (chains, draws)} on the constrained scale, named as abd.model names them."""
        x = backward(self.q)
        return {name: x[:, :, k] for k, (name, _) in enumerate(Q17_RV)} if x.shape[-1] == 17 else {}


class _DualAveraging:
    """Nesterov dual averaging of log step size, per chain (vectorised)."""

    def __init__(self, eps0, target, device, gamma=0.05, t0=10.0, kappa=0.75):
        self.mu = torch.log(10.0 * eps0)
        self.target, self.gamma, self.t0, self.kappa = target, gamma, t0, kappa
        self.h = torch.zeros_like(eps0)
        self.log_avg = torch.zeros_like(eps0)
        self.t = 0

    def update(self, accept):
        self.t += 1
        eta = 1.0 / (self.t + self.t0)
        self.h = (1 - eta) * self.h + eta * (self.target - accept)
        log_eps = self.mu - (self.t**0.5 / self.gamma) * self.h
        w = self.t ** (-self.kappa)
        self.log_avg = w * log_eps + (1 - w) * self.log_avg
        return torch.exp(log_eps)

    def final(self):
        return torch.exp(self.log_avg)


def _windows(tune):
    """Stan's warm-up schedule: fast initial buffer, doubling slow windows, fast final buffer.
    Returns the list of iteration indexes at which a slow window ends."""
    if tune < 150:
        return [int(tune * 0.5)] if tune >= 20 else []
    start, end, size, ends = 75, tune - 50, 25, []
    while start + size <= end:
        nxt = start + size
        if nxt + 2 * size > end:
            nxt = end
        ends.append(nxt)
        start, size = nxt, size * 2
    return ends


class _Thinned:
    """Evenly spaced draws of the three Deterministics, kept on the device until the end of the run
    (int8 i, float32 titers: 9 G N bytes per chain and kept draw)."""

    def __init__(self, target, cfg):
        n_keep = 0
        self.with_ll = hasattr(target, "loglik_rows")
        if cfg.thinned_deterministics and hasattr(target, "deterministics"):
            per_draw = 9 * target.C * target.engine.G * target.engine.N           # bytes per kept draw
            if self.with_ll:
                per_draw += 4 * target.C * (target.engine.R_s + target.engine.R_n)
            n_keep = int(min(cfg.thinned_deterministics, cfg.draws, max(1, (4 << 30) // per_draw)))  # at most 4 GiB
        self.keep = sorted(set(np.linspace(0, cfg.draws - 1, n_keep).round().astype(int).tolist())) if n_keep else []
        self.pos = {k: j for j, k in enumerate(self.keep)}
        if self.keep:
            G, N, C, dev = target.engine.G, target.engine.N, target.C, target.device
            self.i = torch.empty(len(self.keep), C, G, N, dtype=torch.int8, device=dev)
            self.mn = torch.empty(len(self.keep), C, G, N, dtype=torch.float32, device=dev)
            self.ms = torch.empty(len(self.keep), C, G, N, dtype=torch.float32, device=dev)
            if self.with_ll:   # the log_likelihood group of the kept draws (observed nodes it_s_lik / it_n_lik, abd.py:459-469)
                self.ls = torch.empty(len(self.keep), C, target.engine.R_s, dtype=torch.float32, device=dev)
                self.ln = torch.empty(len(self.keep), C, target.engine.R_n, dtype=torch.float32, device=dev)

    def record(self, target, k, q):
        j = self.pos.get(k)
        if j is not None:
            oi, mn, ms = target.deterministics(q)
            self.i[j].copy_(oi)
            self.mn[j].copy_(mn)
            self.ms[j].copy_(ms)
            if self.with_ll:
                ls, ln = target.loglik_rows(q)
                self.ls[j].copy_(ls)
                self.ln[j].copy_(ln)

    def result(self):
        if not self.keep:
            return {}
        out = {"draw": np.array(self.keep), "i": self.i.permute(1, 0, 2, 3).cpu().numpy(),
               "ab_n_mu": self.mn.permute(1, 0, 2, 3).cpu().numpy(), "ab_s_mu": self.ms.permute(1, 0, 2, 3).cpu().numpy()}
        if self.with_ll:
            out["it_s_lik"], out["it_n_lik"] = self.ls.permute(1, 0, 2).cpu().numpy(), self.ln.permute(1, 0, 2).cpu().numpy()
        return out


def _nuts_transition(target, q, logp, grad, eps, inv_mass, chol, gen, max_depth):
    """One No-U-Turn transition for a batch of chains (multinomial sampling inside sub-trees, biased
    progressive sampling between them, the generalised U-turn criterion on every balanced sub-tree:
    Betancourt 2017, as in Stan / PyMC).  The chains double in lockstep -- one batched logp + gradient
    evaluation per leaf serves them all -- and a chain that has terminated is masked.  Sub-tree U-turn
    checks use O(depth) momentum checkpoints per chain instead of recursion.
    Returns (q, logp, grad, mean acceptance statistic, tree depth, diverged, leaves evaluated)."""
    B, D = q.shape
    dev, f64 = q.device, torch.float64
    z = torch.randn(B, D, dtype=f64, device=dev, generator=gen)
    p0 = torch.linalg.solve_triangular(chol.T, z.T, upper=True).T          # p ~ N(0, M), M = Sigma^-1
    h0 = -logp + 0.5 * (z * z).sum(dim=1)
    e = eps[:, None]

    def turning(p_a, p_b, rho):  # either end of the span still moving against the span's momentum sum
        adj = rho - 0.5 * (p_a + p_b)
        return (((p_a @ inv_mass) * adj).sum(dim=1) <= 0) | (((p_b @ inv_mass) * adj).sum(dim=1) <= 0)

    q_l, p_l, g_l = q.clone(), p0.clone(), grad.clone()
    q_r, p_r, g_r = q.clone(), p0.clone(), grad.clone()
    q_prop, lp_prop, g_prop = q.clone(), logp.clone(), grad.clone()
    log_w = torch.zeros(B, dtype=f64, device=dev)          # log sum of exp(h0 - h) over the tree (start point: 0)
    rho = p0.clone()
    active = torch.ones(B, dtype=torch.bool, device=dev)
    depth = torch.zeros(B, dtype=torch.long, device=dev)
    diverged = torch.zeros(B, dtype=torch.bool, device=dev)
    sum_acc = torch.zeros(B, dtype=f64, device=dev)
    n_acc = torch.zeros(B, dtype=f64, device=dev)
    n_leaves = 0
    neg_inf = torch.full((B,), -float("inf"), dtype=f64, device=dev)
    for j in range(max_depth):
        if not bool(active.any()):
            break
        fwd = torch.rand(B, device=dev, generator=gen) < 0.5
        v = torch.where(fwd, 1.0, -1.0).to(f64)[:, None]
        fw = fwd[:, None]
        q_e, p_e, g_e = torch.where(fw, q_r, q_l), torch.where(fw, p_r, p_l), torch.where(fw, g_r, g_l)
        s_q, s_lp, s_g = q_e.clone(), lp_prop.clone(), g_e.clone()
        s_log_w, s_rho = neg_inf.clone(), torch.zeros(B, D, dtype=f64, device=dev)
        s_stop = ~active                                     # turned inside the sub-tree, diverged, or not running
        p_ck = torch.zeros(B, max(j, 1), D, dtype=f64, device=dev)
        rho_ck = torch.zeros(B, max(j, 1), D, dtype=f64, device=dev)
        for n in range(1 << j):
            run = ~s_stop
            if not bool(run.any()):
                break
            ph = p_e + 0.5 * v * e * g_e
            qn = q_e + v * e * (ph @ inv_mass)
            lpn, gn = target.logp_dlogp(qn)
            n_leaves += 1
            pn = ph + 0.5 * v * e * gn
            dh = h0 - (-lpn + 0.5 * ((pn @ inv_mass) * pn).sum(dim=1))
            dh = torch.where(torch.isfinite(dh), dh, neg_inf)
            div = run & (dh.abs() > 1000.0)          # PyMC's divergence threshold on the energy error
            ok = run & ~div
            r2 = run[:, None]
            q_e, p_e, g_e = torch.where(r2, qn, q_e), torch.where(r2, pn, p_e), torch.where(r2, gn, g_e)
            sum_acc = sum_acc + torch.where(run, torch.exp(torch.clamp(dh, max=0.0)), torch.zeros_like(dh))
            n_acc = n_acc + run.to(f64)
            new_w = torch.logaddexp(s_log_w, dh)
            take = ok & (torch.rand(B, dtype=f64, device=dev, generator=gen) < torch.exp(dh - new_w))
            t2 = take[:, None]
            s_q, s_lp, s_g = torch.where(t2, qn, s_q), torch.where(take, lpn, s_lp), torch.where(t2, gn, s_g)
            s_log_w = torch.where(ok, new_w, s_log_w)
            s_rho = s_rho + torch.where(ok[:, None], pn, torch.zeros_like(pn))
            diverged |= div
            s_stop = s_stop | div
            if j > 0:
                # checkpoints: leaf n closes the balanced sub-trees that start at the leaves whose
                # checkpoints sit at idx_min .. idx_max (n odd); an even leaf opens one at idx_max
                idx_max = bin(n >> 1).count("1")
                if n % 2 == 0:
                    p_ck[:, idx_max] = torch.where(ok[:, None], pn, p_ck[:, idx_max])
                    rho_ck[:, idx_max] = torch.where(ok[:, None], s_rho, rho_ck[:, idx_max])
                else:
                    trailing = (n ^ (n + 1)).bit_length() - 1          # number of trailing one bits of n
                    idx_min = idx_max - trailing + 1
                    for i in range(idx_max, idx_min - 1, -1):
                        span = s_rho - rho_ck[:, i] + p_ck[:, i]
                        s_stop = s_stop | (ok & turning(p_ck[:, i], pn, span))
        # merge the finished sub-tree (chains that neither turned inside it nor diverged)
        good = active & ~s_stop
        take = good & (torch.rand(B, dtype=f64, device=dev, generator=gen) < torch.exp(torch.clamp(s_log_w - log_w, max=0.0)))
        t2 = take[:, None]
        q_prop, lp_prop, g_prop = torch.where(t2, s_q, q_prop), torch.where(take, s_lp, lp_prop), torch.where(t2, s_g, g_prop)
        log_w = torch.where(good, torch.logaddexp(log_w, s_log_w), log_w)
        rho = rho + torch.where(good[:, None], s_rho, torch.zeros_like(s_rho))
        gr, gl = (good & fwd)[:, None], (good & ~fwd)[:, None]
        q_r, p_r, g_r = torch.where(gr, q_e, q_r), torch.where(gr, p_e, p_r), torch.where(gr, g_e, g_r)
        q_l, p_l, g_l = torch.where(gl, q_e, q_l), torch.where(gl, p_e, p_l), torch.where(gl, g_e, g_l)
        depth = depth + active.to(torch.long)
        active = good & ~turning(p_l, p_r, rho)
    return q_prop, lp_prop, g_prop, sum_acc / torch.clamp(n_acc, min=1.0), depth, diverged, n_leaves


class _HostLoop:
    """The transition as torch ops driven from the host, for any target with ``logp_dlogp(q) -> (logp, grad)``: momenta,
    trajectory jitter and accept decisions from one torch.Generator, step size by ``_DualAveraging``, the metric by
    torch.linalg."""

    def __init__(self, target, q0, cfg):
        dev, (C, D) = q0.device, q0.shape
        self.target, self.cfg, self.nuts = target, cfg, cfg.kernel == "nuts"
        self.gen = torch.Generator(device=dev)
        self.gen.manual_seed(cfg.seed)
        self.q = q0.clone().to(torch.float64)
        self.logp, self.grad = target.logp_dlogp(self.q)
        self.inv_mass = torch.eye(D, dtype=torch.float64, device=dev)   # Sigma = M^-1 (dense)
        self.chol = torch.eye(D, dtype=torch.float64, device=dev)       # Sigma = chol chol^T
        self.eps = torch.full((C,), cfg.init_step, dtype=torch.float64, device=dev)
        self.da = _DualAveraging(self.eps, cfg.target_accept, dev)

    def transition(self, it):
        """Moves q given the binaries; returns the number of gradient evaluations."""
        cfg, q, logp, grad, eps, inv_mass, gen = self.cfg, self.q, self.logp, self.grad, self.eps, self.inv_mass, self.gen
        if self.nuts:   # ---- NUTS over q given the binaries (abd.py:922 runs PyMC's) ----
            q, logp, grad, self.acc, self.depth, self.div, n_grad = _nuts_transition(self.target, q, logp, grad, eps, inv_mass,
                                                                                     self.chol, gen, cfg.max_treedepth)
        else:           # ---- HMC over q given the binaries ----
            C, D = q.shape
            # p ~ N(0, M) with M = Sigma^-1:  p = chol^-T z
            z = torch.randn(C, D, dtype=torch.float64, device=q.device, generator=gen)
            p = torch.linalg.solve_triangular(self.chol.T, z.T, upper=True).T
            h0 = -logp + 0.5 * (z * z).sum(dim=1)
            jitter = cfg.jitter[0] + (cfg.jitter[1] - cfg.jitter[0]) * torch.rand((), device=q.device, generator=gen).item()
            n_grad = L = max(1, int(round(cfg.n_leapfrog * jitter)))
            qn, pn, gn, lpn = q, p, grad, logp
            e = eps[:, None]
            for _ in range(L):
                pn = pn + 0.5 * e * gn
                qn = qn + e * (pn @ inv_mass)
                lpn, gn = self.target.logp_dlogp(qn)
                pn = pn + 0.5 * e * gn
            h1 = -lpn + 0.5 * ((pn @ inv_mass) * pn).sum(dim=1)
            dh = h0 - h1
            dh = torch.where(torch.isfinite(dh), dh, torch.full_like(dh, -float("inf")))
            self.acc = torch.exp(torch.clamp(dh, max=0.0))
            take = torch.rand(C, dtype=torch.float64, device=q.device, generator=gen) < self.acc
            q, grad, logp = torch.where(take[:, None], qn, q), torch.where(take[:, None], gn, grad), torch.where(take, lpn, logp)
        self.q, self.logp, self.grad = q, logp, grad
        if it < cfg.tune:
            self.eps = self.da.update(self.acc)
        return n_grad

    def refresh(self):
        self.logp, self.grad = self.target.logp_dlogp(self.q)

    def set_metric(self, x):
        n, D = x.shape
        cov = torch.cov(x.T)
        self.inv_mass = (n / (n + 5.0)) * cov + 1e-3 * (5.0 / (n + 5.0)) * torch.eye(D, dtype=cov.dtype, device=x.device)
        self.chol = torch.linalg.cholesky(self.inv_mass)  # Stan's shrinkage keeps it positive definite
        self.eps = self.da.final()  # restart step-size adaptation under the new metric
        self.da = _DualAveraging(self.eps, self.cfg.target_accept, x.device)

    def end_tuning(self):
        if self.da.t:
            self.eps = self.da.final()


class _DeviceLoop:
    """The transition on the device, no host synchronisation: abd_hmc_begin_dev, abd_leapfrog_dev (one launch per step, or
    one persistent launch per trajectory), abd_hmc_end_dev -- or abd_nuts_begin_dev, one abd_nuts_extend_dev per tree
    depth, abd_nuts_end_dev -- with the momenta, accept decisions and dual averaging in the kernels.  The host only picks
    the trajectory length and, at the end of a warm-up window, computes the metric."""

    def __init__(self, target, q0, cfg):
        dev, (C, D) = q0.device, q0.shape
        f64 = dict(dtype=torch.float64, device=dev)
        self.target, self.cfg, self.nuts = target, cfg, cfg.kernel == "nuts"
        self.rng = np.random.default_rng(cfg.seed)
        self.q = q0.clone().to(torch.float64).contiguous()
        self.logp, self.grad = torch.empty(C, **f64), torch.empty(C, D, **f64)
        target.logp_dlogp_into(self.q, self.logp, self.grad)
        self.inv_mass = torch.eye(D, **f64)
        self.linv_t = torch.eye(D, **f64)        # (chol^T)^-1 with inv_mass = chol chol^T
        self.eps = torch.full((C,), cfg.init_step, **f64)
        self.da = torch.zeros(C, 4, **f64)       # mu, hbar, log_avg, t
        self.da[:, 0] = torch.log(10.0 * self.eps)
        self.qw, self.pw, self.gw = torch.empty(C, D, **f64), torch.empty(C, D, **f64), torch.empty(C, D, **f64)
        self.lpw, self.h0, self.acc = torch.empty(C, **f64), torch.empty(C, **f64), torch.empty(C, **f64)
        if self.nuts:
            self.TD = int(min(max(cfg.max_treedepth, 1), 10))   # maximum tree depth
            self.tree, self.eps_signed, self.any_active = target.nuts_scratch(self.TD)
            self.depth, self.div = torch.zeros(C, **f64), torch.zeros(C, **f64)
            self.recent_depths = deque(maxlen=32)

    def transition(self, it):
        """Moves q given the binaries; returns the number of gradient evaluations."""
        tgt, cfg, adapt = self.target, self.cfg, it < self.cfg.tune
        q, grad, logp, eps, qw, pw, gw, lpw = self.q, self.grad, self.logp, self.eps, self.qw, self.pw, self.gw, self.lpw
        if not self.nuts:
            L = max(1, int(round(cfg.n_leapfrog * (cfg.jitter[0] + (cfg.jitter[1] - cfg.jitter[0]) * self.rng.random()))))
            tgt.hmc_begin(q, grad, logp, self.linv_t, it, qw, pw, gw, self.h0)
            if cfg.single_step_launches:   # L overlapped launches: 14.7 us per step (one persistent launch: 16.8)
                for _ in range(L):
                    tgt.leapfrog_inplace(qw, pw, gw, lpw, eps, self.inv_mass, 1)
            else:
                tgt.leapfrog_inplace(qw, pw, gw, lpw, eps, self.inv_mass, L)
            tgt.hmc_end(q, grad, logp, qw, pw, gw, lpw, self.inv_mass, self.h0, it, self.acc, self.da, eps, adapt,
                        cfg.target_accept)
            return L
        # the chains double in lockstep: depth j adds 2^j leaves (one leapfrog launch each, which also updates the trees);
        # one word is read back per depth: does any chain still want to double?
        TD, tree, eps_signed, any_active = self.TD, self.tree, self.eps_signed, self.any_active
        tgt.nuts_begin(TD, q, grad, logp, self.linv_t, eps, it, tree, qw, pw, gw, eps_signed, any_active)
        # Depths below `check_from` are built without asking (a read-back costs as much as two leaves): the shallowest
        # tree of the last 32 iterations, never below cfg.nuts_check_from_depth.  Building a depth no chain wanted
        # changes nothing (its leaves are masked on the device), it only costs their launches.
        recent = self.recent_depths
        check_from = max(cfg.nuts_check_from_depth, min(recent)) if cfg.nuts_adaptive_checks and recent \
            else cfg.nuts_check_from_depth
        flags, n_grad = None, 0
        for j in range(TD):
            tgt.nuts_extend(TD, j, qw, pw, gw, lpw, self.inv_mass, eps, it, tree, eps_signed, any_active)
            n_grad += 1 << j
            if j + 1 < TD and j + 1 >= check_from:
                flags = any_active.tolist()       # [k]: did any chain want depth k?  (one read-back, all depths)
                if flags[j + 1] == 0:
                    break
        # lockstep depth of this tree: the first depth nobody wanted
        recent.append(TD if flags is None else next((k for k in range(1, TD + 1) if flags[k] == 0), TD))
        tgt.nuts_end(TD, q, grad, logp, tree, self.acc, self.depth, self.div, self.da, eps, adapt, cfg.target_accept)
        return n_grad

    def refresh(self):
        self.target.logp_dlogp_into(self.q, self.logp, self.grad)

    def set_metric(self, x):
        # 17 x 17 linear algebra on the host (a handful of times per run; the first cuSOLVER
        # call alone would cost more than all of them)
        x = x.cpu().numpy()
        n, D = x.shape
        cov = np.cov(x.T)
        im = (n / (n + 5.0)) * cov + 1e-3 * (5.0 / (n + 5.0)) * np.eye(D)  # Stan's shrinkage keeps it positive definite
        chol = np.linalg.cholesky(im)
        dev = self.q.device
        self.inv_mass = torch.from_numpy(np.ascontiguousarray(im)).to(dev)
        self.linv_t = torch.from_numpy(np.ascontiguousarray(np.linalg.inv(chol.T))).to(dev)
        # restart step-size adaptation under the new metric from the averaged step
        self.eps = torch.exp(self.da[:, 2]).contiguous()
        self.da.zero_()
        self.da[:, 0] = torch.log(10.0 * self.eps)

    def end_tuning(self):
        self.eps = torch.where(self.da[:, 3] > 0, torch.exp(self.da[:, 2]), self.eps).contiguous()


def sample(target, q0, cfg: SamplerConfig = SamplerConfig(), progress=None) -> SamplerResult:
    """Run tune + draws iterations of [HMC or NUTS on q | binaries] then [Gibbs on binaries | q].  The transitions run on
    the device when the target has the device-resident loop (``device_loop``) and ``cfg.persistent_trajectories`` is set,
    otherwise as torch ops driven from the host."""
    if cfg.kernel not in ("hmc", "nuts"):
        raise ValueError(f"unknown kernel {cfg.kernel!r}: 'hmc' or 'nuts'")
    on_device = cfg.persistent_trajectories and getattr(target, "device_loop", False)
    run = (_DeviceLoop if on_device else _HostLoop)(target, q0, cfg)
    dev = q0.device
    C, D = q0.shape
    f64 = dict(dtype=torch.float64, device=dev)

    def sync():
        if dev.type == "cuda":
            torch.cuda.synchronize(dev)

    ends = _windows(cfg.tune)
    win_start = 75 if cfg.tune >= 150 else 0
    win_draws = []
    total = cfg.tune + cfg.draws
    out_q = torch.empty(cfg.draws, C, D, **f64)
    out_lp, out_acc = torch.empty(cfg.draws, C, **f64), torch.empty(cfg.draws, C, **f64)
    out_depth, out_div = torch.zeros(cfg.draws, C, **f64), torch.zeros(cfg.draws, C, **f64)   # NUTS tree statistics
    means, n_means, n_grad = {}, 0, 0
    thin = _Thinned(target, cfg)
    has_gibbs = hasattr(target, "gibbs")
    t0 = time.perf_counter()
    wall_tune, n_grad_tune = 0.0, 0
    for it in range(total):
        n_grad += run.transition(it)
        if has_gibbs:   # Gibbs over the binaries given q, then logp / grad at the new state
            target.gibbs(run.q, it)
            run.refresh()
            n_grad += 1
        if it < cfg.tune:
            if ends and win_start <= it:
                win_draws.append(run.q.clone())
            if ends and it + 1 == ends[0]:
                run.set_metric(torch.stack(win_draws).reshape(-1, D))
                win_draws, win_start = [], ends.pop(0)
            if it + 1 == cfg.tune:
                run.end_tuning()
                sync()     # once per run: the draws are timed on their own as well
                wall_tune, n_grad_tune = time.perf_counter() - t0, n_grad
        else:
            k = it - cfg.tune
            out_q[k].copy_(run.q)
            out_lp[k].copy_(run.logp)
            out_acc[k].copy_(run.acc)
            if run.nuts:
                out_depth[k].copy_(run.depth)
                out_div[k].copy_(run.div)
            thin.record(target, k, run.q)
            every = cfg.record_deterministics_every
            if every and k % every == 0 and hasattr(target, "accumulate_deterministics"):
                target.accumulate_deterministics(run.q, means)   # sums over chains; divided once at the end
                if cfg.rao_blackwell:
                    target.accumulate_infection_probs(run.q, means)
                n_means += C
        if progress and (it + 1) % progress == 0:
            print(f"  iter {it + 1}/{total}  step {run.eps.mean().item():.4f}  accept {run.acc.mean().item():.2f}", flush=True)
    sync()
    if on_device:
        target.check_status()
    wall = time.perf_counter() - t0
    stats = {"tree_depth": out_depth.T.cpu().numpy().astype(np.int64), "diverging": out_div.T.cpu().numpy() != 0} if run.nuts else {}
    return SamplerResult(
        q=out_q.permute(1, 0, 2).cpu().numpy(), logp=out_lp.T.cpu().numpy(), accept=out_acc.T.cpu().numpy(),
        step_size=run.eps.cpu().numpy(), inv_mass=run.inv_mass.cpu().numpy(), wall_s=wall, n_grad_evals=n_grad,
        means={k: (v / n_means).cpu().numpy() for k, v in means.items()}, thinned=thin.result(), stats=stats,
        wall_tune_s=wall_tune, n_grad_evals_tune=n_grad_tune,
    )
