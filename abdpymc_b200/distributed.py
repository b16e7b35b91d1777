"""Multi-GPU sharding of the hot path: one process per GPU, ``torch.distributed`` for plumbing.

Two axes shard naturally (SURVEY.md section 8e):

* **individuals** -- given the 17 scalars every likelihood term, Bernoulli term and Gibbs update
  of individual n depends only on column n (abd.py:343, 393 gather per (gap, ind); the
  constraints abd.py:560-862 are column-wise).  Rank r holds a contiguous block of individuals
  (``CohortArrays.shard``) and the matching slice of every chain's ``i_raw`` / ``waner``.  One
  evaluation = local raw sums (``abd_sums_dev``) -> ONE all-reduce of C x 16 doubles ->
  ``abd_finalize_logp_dev`` on every rank.  The Gibbs sweep needs no collective at all.
* **chains** -- fully independent: replicate the cohort, give each rank its own chains, no
  collective on the data path.

The reference has no distributed code of any kind (pm.sample(cores=K) forks independent chain
processes, abd.py:922); this module is the B200-native counterpart of that chain-level process
parallelism plus the individual sharding large cohorts need.
"""

from __future__ import annotations

import os

import numpy as np
import torch
import torch.distributed as dist

from .cohort import CohortArrays, shard_bounds
from .engine import AbdEngine
from .sampler import DeviceTarget

N_SUMS = 16


def dist_env():
    """(rank, world, local_rank) from the torchrun environment (1 process = 1 GPU)."""
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def init_process_group(backend=None, device=None):
    """Initialise torch.distributed from the torchrun environment; no-op for a single process.
    NCCL when a CUDA device is given, gloo otherwise (CPU tests)."""
    rank, world, _ = dist_env()
    if world == 1 or dist.is_initialized():
        return dist if world > 1 else None
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29577")
    backend = backend or ("nccl" if device is not None else "gloo")
    kw = {"device_id": device} if (device is not None and backend == "nccl") else {}
    dist.init_process_group(backend, rank=rank, world_size=world, **kw)
    return dist


def chain_slice(n_chains: int, rank: int, world: int) -> slice:
    """Chains owned by ``rank`` when chains are sharded (contiguous, sizes differ by <= 1)."""
    lo, hi = shard_bounds(n_chains, rank, world)
    return slice(lo, hi)


def cohort_totals(cohort: CohortArrays) -> tuple:
    """(n_inds, n_rows_s, n_rows_n) of the whole cohort: what every shard's engine must be told
    so that the finaliser uses global Bernoulli / likelihood constants."""
    return cohort.n_inds, int((cohort.antigen == 1).sum()), int((cohort.antigen == 0).sum())


def shard_cohort(cohort: CohortArrays, rank: int, world: int):
    """(shard, totals, ind_offset, slice of individuals) for individual sharding."""
    lo, hi = shard_bounds(cohort.n_inds, rank, world)
    return cohort.shard(rank, world), cohort_totals(cohort), lo, slice(lo, hi)


def allreduce_sums(sums, group=None):
    """Sum the per-shard raw sums (C x 16 doubles, every entry additive over individuals) over
    all ranks, in place.  ``sums``: torch tensor on the device the process group runs on."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    return sums


class ShardedEngine:
    """Individual-sharded evaluation of the joint logp + gradient on this rank's GPU.

    Every rank builds the engine of its shard with the global totals; ``logp_dlogp`` runs
    sums -> all-reduce -> finalise and leaves identical (logp, dlogp) tensors on every rank.
    """

    def __init__(self, cohort: CohortArrays, splits=None, ignore_pcrpos=False, device_index=0, rank=None, world=None,
                 group=None, fused=False, max_chains=64):
        """``fused=True``: the all-reduce is done INSIDE the logp kernel over NVLink peer memory
        (``abd_logp_dlogp_sharded_dev``: every rank's finishing CTA stores its sums into all peers'
        exchange buffers and waits for theirs) -- one launch per evaluation, no NCCL call.  Needs
        an initialised process group once, to exchange the CUDA IPC handles."""
        env_rank, env_world, _ = dist_env()
        self.rank = env_rank if rank is None else rank
        self.world = env_world if world is None else world
        self.group = group
        shard, totals, offset, self.ind_slice = shard_cohort(cohort, self.rank, self.world)
        self.device = torch.device("cuda", device_index)
        self.engine = AbdEngine(shard, splits=splits, ignore_pcrpos=ignore_pcrpos, device=device_index, totals=totals,
                                ind_offset=offset)
        self.G, self.N_local, self.N_total = self.engine.G, self.engine.N, cohort.n_inds
        self._bufs = {}
        self.fused = bool(fused) and self.world > 1
        if self.fused:
            mine = self.engine.xch_alloc(self.world, self.rank, max_chains)
            handles = [None] * self.world
            dist.all_gather_object(handles, mine, group=group)
            self.engine.xch_connect(handles)
            dist.barrier(group=group)  # every rank has mapped every buffer before the first launch

    def _buffers(self, C):
        if C not in self._bufs:
            self._bufs[C] = (
                torch.zeros(C, N_SUMS, dtype=torch.float64, device=self.device),
                torch.zeros(C, dtype=torch.float64, device=self.device),
                torch.zeros(C, 17, dtype=torch.float64, device=self.device),
            )
        return self._bufs[C]

    def upload_state(self, i_raw, waner):
        """``i_raw`` (C, G, N_total), ``waner`` (C, N_total): keeps this rank's individuals."""
        i_raw, waner = np.asarray(i_raw), np.asarray(waner)
        return self.engine.upload_state(np.ascontiguousarray(i_raw[..., self.ind_slice]),
                                        np.ascontiguousarray(waner[..., self.ind_slice]))

    def logp_dlogp(self, q17, n_chains=None, out=None, outg=None):
        """``q17``: torch (C, 17) float64 tensor on this rank's device (identical on all ranks).
        Uses the resident chain state.  Returns (logp (C,), dlogp (C, 17)) device tensors (``out`` /
        ``outg`` when given, otherwise buffers reused by the next call)."""
        C = q17.shape[0] if n_chains is None else n_chains
        sums, out_, outg_ = self._buffers(C)
        out = out_ if out is None else out
        outg = outg_ if outg is None else outg
        st = torch.cuda.current_stream(self.device).cuda_stream
        d_i, d_w = self.engine.state_dev(C)
        if self.fused:
            self.engine.logp_dlogp_sharded_dev(C, q17.data_ptr(), d_i, d_w, out.data_ptr(), outg.data_ptr(), st)
            return out, outg
        self.engine.sums_dev(C, q17.data_ptr(), 1, d_i, d_w, sums.data_ptr(), st)
        allreduce_sums(sums, self.group)
        self.engine.finalize_logp_dev(C, q17.data_ptr(), sums.data_ptr(), out.data_ptr(), outg.data_ptr(), st)
        return out, outg

    def exchange_wait_us(self, reset=True):
        """Mean time (us) the finishing CTA of an evaluation spent waiting for its slowest peer's contribution
        -- launch skew between the ranks plus NVLink latency -- since the last reset (fused engines only)."""
        ns, n = self.engine.xch_stats(reset=reset)
        return float(ns.max()) / max(n, 1) / 1e3

    def close(self):
        self.engine.close()


class ShardedTarget(DeviceTarget):
    """The posterior of an INDIVIDUAL-SHARDED cohort as a sampler target (same interface as
    ``sampler.AbdTarget``): every rank holds a contiguous block of individuals and the matching slice of
    every chain's binary state; the 17 scalars, their momenta, step sizes and the metric are replicated.

    * logp + gradient / leapfrog steps: local sums, all-reduce of C x 16 doubles fused into the launch
      over NVLink peer memory (``fused=True``) -- every rank obtains bitwise identical results, so the
      replicated HMC state never diverges; or ``abd_sums_dev`` -> NCCL / gloo all-reduce ->
      ``abd_finalize_logp_dev`` (``fused=False``; the sampler then runs its host-driven loop).
    * momentum refresh / accept (``abd_hmc_begin_dev`` / ``abd_hmc_end_dev``): Philox streams keyed by
      (seed; iteration, chain) -- the same seed on every rank gives the same momenta and decisions.
    * Gibbs sweep: local, no communication (individuals are conditionally independent given the
      scalars; streams keyed by GLOBAL individual, so the draws do not depend on the sharding).
    What abd.py:922 runs as NUTS + BinaryGibbsMetropolis on one CPU core per chain.  Its draws of the (G, N)
    Deterministics are not gathered over the ranks, so it has no ``deterministics`` / ``loglik_rows``."""

    def __init__(self, sharded: ShardedEngine, n_chains, i_raw, waner, seed=0, gibbs_mode=0, transit_p=0.8):
        super().__init__(sharded.engine, n_chains, sharded.device, seed, gibbs_mode, transit_p)
        self.sh, self.device_loop = sharded, sharded.fused
        sharded.upload_state(i_raw, waner)          # (C, G, N_total) / (C, N_total): this rank keeps its block

    def logp_dlogp_into(self, q, logp, grad):
        self.sh.logp_dlogp(q, self.C, out=logp, outg=grad)

    def leapfrog_inplace(self, q, p, grad, logp, eps, inv_mass, n_steps):
        """One launch per step, the exchange fused into it (fused engines only)."""
        for _ in range(n_steps):
            self.engine.leapfrog_sharded_dev(self.C, q.data_ptr(), p.data_ptr(), grad.data_ptr(), logp.data_ptr(), eps.data_ptr(),
                                             inv_mass.data_ptr(), self.d_i, self.d_w, self._stream())

    def check_status(self):
        super().check_status()
        if self.sh.fused:
            self.engine.xch_status()

    def gather_individuals(self, local, axis=-1):
        """Concatenate per-rank blocks of individuals (NumPy arrays) along ``axis`` on every rank."""
        parts = [None] * self.sh.world
        dist.all_gather_object(parts, np.ascontiguousarray(local), group=self.sh.group)
        return np.concatenate(parts, axis=axis)
