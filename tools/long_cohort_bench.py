#!/usr/bin/env python3
"""What the 128-bit gap-mask layout (cohorts of 64..127 gaps) costs on the GPU.

The bench cohort (10 000 individuals, G = 31) and two longer versions of it: every individual's schedule (OD rows,
vaccinations, PCR+ months) repeated at +31 and +62 months (G = 62 and 93), OD values simulated again.  Per cohort,
in one process, with CUDA events:
  k_sums       us per fused logp + gradient launch on the resident state, 4 and 128 chains
  k_gibbs      us per Gibbs sweep (Metropolis, 4 chains)
  sampler      device HMC + Gibbs iterations / s (4 chains)
  per row / per cell   k_sums time at 4 chains over OD rows and over (individual, gap) cells
The G = 62 cohort runs on its own 64-bit layout and with ABD_B200_MASK_BITS=128 (same cohort, wider masks).

    python tools/long_cohort_bench.py [--iters 200] [--out DIR]

Prints one JSON line (device name and power limit included).  Every timed window re-reads its inputs from the
previous launch's L2: the cohort arrays (tens of MB) fit the 126 MB L2, so the numbers are L2-resident.
"""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from abdpymc_b200.cohort import CohortArrays, simulate, synthetic_cohort  # noqa: E402

SPLITS = (14, 20)


def repeated(co: CohortArrays, times: int) -> CohortArrays:
    """The cohort followed `times` times as long: each individual's schedule repeated every G months."""
    G = co.n_gaps
    rows = [(co.ind, co.gap + k * G, co.antigen, co.x) for k in range(times)]
    longer = CohortArrays(vacs=np.tile(co.vacs, times), pcrpos=np.tile(co.pcrpos, times),
                          ind=np.concatenate([r[0] for r in rows]), gap=np.concatenate([r[1] for r in rows]),
                          antigen=np.concatenate([r[2] for r in rows]), x=np.concatenate([r[3] for r in rows]),
                          od=np.zeros(len(co.ind) * times), t0=co.t0)
    return simulate(longer, lam0=0.04, seed=42)


def device_info():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        smi = "unknown"
    return {"device": name, "power_limit_and_max_sm_clock": smi}


def time_us(fn, iters):
    import torch

    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / iters


def measure(co, label, iters):
    import torch

    from abdpymc_b200.engine import AbdEngine, backward, forward
    from abdpymc_b200.sampler import AbdTarget, SamplerConfig, sample
    from oracle import abd_oracle as ora

    G, N = co.n_gaps, co.n_inds
    rng = np.random.default_rng(7)
    out = {"label": label, "G": G, "N": N, "rows": int(co.n_rows),
           "cells": int(len(np.unique(co.ind.astype(np.int64) * 256 + co.gap + 128 * co.antigen)))}
    dev = torch.device("cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    with AbdEngine(co, splits=SPLITS) as eng:
        for C in (4, 128):
            q = np.stack([ora.forward(ora.sample_prior(rng, G)) for _ in range(C)])
            eng.upload_state((rng.random((C, G, N)) < 0.04).astype(np.int8), (rng.random((C, N)) < 0.5).astype(np.int8))
            di, dw = eng.state_dev(C)
            tq = torch.from_numpy(q).to(dev)
            lp = torch.empty(C, dtype=torch.float64, device=dev)
            g = torch.empty(C, 17, dtype=torch.float64, device=dev)
            out[f"k_sums_us_c{C}"] = time_us(lambda: eng.logp_dlogp_dev(C, tq.data_ptr(), di, dw, lp.data_ptr(), g.data_ptr(), st),
                                             iters)
            out[f"plan_c{C}"] = eng.last_plan()
            if C == 4:
                sweep = [0]

                def gibbs():
                    eng.gibbs_sweep_dev(C, tq.data_ptr(), 1, None, None, di, dw, 11, sweep[0], 0, 0.8, None, st)
                    sweep[0] += 1

                out["k_gibbs_us_per_sweep_c4"] = time_us(gibbs, max(iters // 4, 20))
        out["us_per_row_c4"] = out["k_sums_us_c4"] / out["rows"]
        out["us_per_cell_c4"] = out["k_sums_us_c4"] / out["cells"]
        C = 4
        tgt = AbdTarget(eng, C, (rng.random((C, G, N)) < 0.04).astype(np.int8), (rng.random((C, N)) < 0.5).astype(np.int8),
                        seed=3)
        x0 = np.array([1.0 / G, 2, 1, 10 / 11, -2, 2, 10 / 11, 0.5, 1, 1, -2, -1, 2, 1, -1, 2, 1], dtype=np.float64)
        q0 = torch.from_numpy(forward(x0)[None, :].repeat(C, 0)).to(dev)
        sample(tgt, q0, SamplerConfig(tune=20, draws=20, seed=1))  # warm-up (plans, tilings, modules)
        torch.cuda.synchronize()
        n_it = 300
        t = time.perf_counter()
        res = sample(tgt, q0, SamplerConfig(tune=n_it // 2, draws=n_it - n_it // 2, seed=2))
        torch.cuda.synchronize()
        out["sampler_iters_per_s_c4"] = n_it / (time.perf_counter() - t)
        assert np.isfinite(backward(res.q)).all()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--n_inds", type=int, default=10_000)
    ap.add_argument("--out", default=None, help="directory for the JSON result")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("long_cohort_bench.py measures the GPU: no CUDA device")
    from abdpymc_b200 import build

    build.build()
    base = synthetic_cohort(args.n_inds)
    res = {"info": device_info(), "inputs": "L2-resident (cohort arrays < 126 MB, re-read every launch)", "runs": []}
    for times in (1, 2, 3):
        co = base if times == 1 else repeated(base, times)
        res["runs"].append(measure(co, f"G{co.n_gaps}", args.iters))
        if times == 2:
            os.environ["ABD_B200_MASK_BITS"] = "128"
            try:
                res["runs"].append(measure(co, f"G{co.n_gaps}_mask128", args.iters))
            finally:
                del os.environ["ABD_B200_MASK_BITS"]
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).mkdir(parents=True, exist_ok=True)
        (Path(args.out) / "long_cohort_bench.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
