#!/usr/bin/env python3
"""The compound sampler (HMC + Gibbs) on an INDIVIDUAL-SHARDED cohort over >= 2 GPUs of one node
(distributed.ShardedTarget), against the same sampler on the unsharded cohort on one GPU.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29595 tools/sharded_sampler_check.py [n_inds] [n_chains] [tune] [draws]

Checks (exit code non-zero on failure, one JSON line on rank 0):
  * every rank ends with bitwise identical draws of the 17 scalars (replicated HMC state never diverges);
  * the fused path (all-reduce inside the kernel) and the NCCL path (host-driven loop) agree with the
    unsharded run: identical Gibbs / accept decisions, scalars equal to rounding, over the first iterations
    (tiles are summed in another order, so the runs may part after many iterations -- both remain valid chains);
  * the binary state gathered from the shards equals the unsharded state after those iterations.
"""
import json
import os
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from abdpymc_b200.cohort import synthetic_cohort  # noqa: E402
from abdpymc_b200.distributed import ShardedEngine, ShardedTarget  # noqa: E402
from abdpymc_b200.engine import AbdEngine, forward  # noqa: E402
from abdpymc_b200.sampler import AbdTarget, SamplerConfig, sample  # noqa: E402

n_inds = int(sys.argv[1]) if len(sys.argv) > 1 else 3000
C = int(sys.argv[2]) if len(sys.argv) > 2 else 2
tune = int(sys.argv[3]) if len(sys.argv) > 3 else 30
draws = int(sys.argv[4]) if len(sys.argv) > 4 else 30
SPLITS = (14, 20)
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)

co = synthetic_cohort(n_inds)
G, N = co.n_gaps, co.n_inds
x0 = np.array([1.0 / G, 2, 1, 10 / 11, -2, 2, 10 / 11, 0.5, 1, 1, -2, -1, 2, 1, -1, 2, 1], dtype=np.float64)
q0 = forward(x0)[None, :] + np.random.default_rng(3).uniform(-0.5, 0.5, size=(C, 17))
i0, w0 = np.zeros((C, G, N), np.int8), np.zeros((C, N), np.int8)
cfg = SamplerConfig(tune=tune, draws=draws, seed=5, record_deterministics_every=1)
# a short run from a small fixed step for the step-by-step comparison with the unsharded sampler (rounding
# differences of the tile sums grow along a long adapted run; both remain valid chains)
cfg_short = SamplerConfig(tune=3, draws=8, seed=5, init_step=0.002, record_deterministics_every=1)
cfg_nuts = SamplerConfig(tune=2, draws=6, seed=5, init_step=0.002, kernel="nuts", max_treedepth=4)
ok, info = True, {}

runs = {}
for name, fused in (("fused", True), ("nccl", False)):
    se = ShardedEngine(co, splits=SPLITS, device_index=local, rank=rank, world=world, fused=fused, max_chains=C)
    tgt = ShardedTarget(se, C, i0, w0, seed=11)
    short = sample(tgt, torch.from_numpy(q0).to(dev), cfg_short)
    li, lw = tgt.state()
    state = (tgt.gather_individuals(li), tgt.gather_individuals(lw))
    means = {k: tgt.gather_individuals(v) for k, v in short.means.items()}
    res = sample(tgt, torch.from_numpy(q0).to(dev), cfg)
    nuts = sample(tgt, torch.from_numpy(q0).to(dev), cfg_nuts) if fused else None   # device No-U-Turn tree on the sharded cohort
    runs[name] = (res, state, means, short, nuts)
    # every rank holds the same draws
    t = torch.from_numpy(np.ascontiguousarray(res.q)).to(dev)
    parts = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(parts, t)
    same = all(torch.equal(parts[0], u) for u in parts)
    ok &= same
    info[f"{name}_identical_on_all_ranks"] = same
    info[f"{name}_iterations_per_s"] = (tune + draws) / res.wall_s
    info[f"{name}_mean_accept"] = float(res.accept.mean())
    if fused:
        info["fused_exchange_wait_us"] = se.exchange_wait_us()
    se.close()

if rank == 0:
    with AbdEngine(co, splits=SPLITS, device=local) as eng:
        tgt = AbdTarget(eng, C, i0, w0, seed=11)
        ref = sample(tgt, torch.from_numpy(q0).to(dev), cfg_short)
        ri, rw = tgt.state()
        sample(tgt, torch.from_numpy(q0).to(dev), cfg)             # bring the binary state to where the sharded run was
        ref_nuts = sample(tgt, torch.from_numpy(q0).to(dev), cfg_nuts)
    # the fused sharded run against the fused unsharded run: the same algorithm step for step
    res, state, means, short, nuts = runs["fused"]
    err = float(np.max(np.abs(short.q - ref.q) / np.maximum(1.0, np.abs(ref.q))))
    info["fused_vs_unsharded_rel_err_short_run"] = err
    ok &= err < 1e-8
    # (the long adapted runs in between may have parted by rounding: compare the NUTS runs only loosely unless they did not)
    info["nuts_tree_depth_sharded"], info["nuts_tree_depth_unsharded"] = float(nuts.stats["tree_depth"].mean()), float(ref_nuts.stats["tree_depth"].mean())
    ok &= bool(np.isfinite(nuts.q).all()) and abs(info["nuts_tree_depth_sharded"] - info["nuts_tree_depth_unsharded"]) < 1.5
    info["fused_state_bits_differing"] = int((state[0] != ri).sum() + (state[1] != rw).sum())
    ok &= info["fused_state_bits_differing"] == 0
    for k in ("i", "ab_n_mu", "ab_s_mu"):
        ok &= bool(np.allclose(means[k], ref.means[k], rtol=1e-9, atol=1e-9))
    # the long adapted runs (fused: device-resident loop; NCCL: host-driven loop with another RNG for the momenta)
    # are only compared loosely: both must have moved to the same region
    res_n = runs["nccl"][0]
    info["nccl_logp_mean"], info["fused_logp_mean"] = float(res_n.logp[:, -10:].mean()), float(res.logp[:, -10:].mean())
    ok &= bool(np.isfinite(res.q).all() and np.isfinite(res_n.q).all())
    info["logp_start"] = float(min(res.logp[:, 0].min(), res_n.logp[:, 0].min()))
    ok &= info["nccl_logp_mean"] > info["logp_start"] and info["fused_logp_mean"] > info["logp_start"]  # both climbing
    ok &= info["fused_mean_accept"] > 0.3 and info["nccl_mean_accept"] > 0.3

flag = torch.tensor([1.0 if ok else 0.0], device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0:
    print(json.dumps({"ok": bool(flag.item()), "world": world, "n_inds": n_inds, "chains": C, "tune": tune, "draws": draws, **info}))
dist.destroy_process_group()
sys.exit(0 if flag.item() else 1)
