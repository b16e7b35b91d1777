#!/usr/bin/env python3
"""What the Rao-Blackwellised infection / waner probabilities (abd_infection_probs_accum_dev, k_infprob_accum) cost on
the GPU and what they buy.  In one process, with CUDA events, on the bench cohort (10 000 individuals, G = 31, splits
(14, 20)) and its 3x longer version (G = 93: the last chunk is [20, 93), 73 options):
  k_infprob     us per accumulation: 10k x 4 and 10k x 128 chains, G = 93 x 4, 10k x 4 without splits
  k_gibbs_blk   us per blocked Gibbs sweep at 10k x 4 (the kernel evaluates about as many likelihoods)
  sampler       device HMC + Gibbs iterations / s at 10k x 4, means recorded every draw, without and with
                rao_blackwell, alternated
  se_ratio      median over (gap, individual) with posterior probability in [0.01, 0.99] of the Monte-Carlo
                standard error across 32 chains of the Rao-Blackwellised mean over that of the mean of the draws of i
                (and the same for ab_s_waner), from one 32-chain run of the sampler on the 1 000-individual cohort

    python tools/infection_probs_bench.py [--iters 200] [--out DIR]

Prints one JSON line (device name and power limit included).  The cohort arrays fit the 126 MB L2, so the kernel
times are L2-resident.
"""
import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from long_cohort_bench import device_info, repeated, time_us  # noqa: E402

from abdpymc_b200.cohort import synthetic_cohort  # noqa: E402

SPLITS = (14, 20)


def kernel_times(eng, rng, chain_counts, iters, with_blk=False):
    import torch

    from oracle import abd_oracle as ora

    G, N = eng.G, eng.N
    dev = torch.device("cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    out = {}
    for C in chain_counts:
        q = torch.from_numpy(np.stack([ora.forward(ora.sample_prior(rng, G)) for _ in range(C)])).to(dev)
        eng.upload_state((rng.random((C, G, N)) < 0.04).astype(np.int8), (rng.random((C, N)) < 0.5).astype(np.int8))
        di, dw = eng.state_dev(C)
        si = torch.zeros(G, N, dtype=torch.float64, device=dev)
        sw = torch.zeros(N, dtype=torch.float64, device=dev)
        out[f"k_infprob_us_c{C}"] = time_us(
            lambda: eng.infection_probs_accum_dev(C, q.data_ptr(), di, dw, si.data_ptr(), sw.data_ptr(), st), iters)
        if with_blk and C == 4:
            sweep = [0]

            def blk():
                eng.gibbs_sweep_dev(C, q.data_ptr(), 1, None, None, di, dw, 11, sweep[0], 2, 0.8, None, st)
                sweep[0] += 1

            out["k_gibbs_blk_us_per_sweep_c4"] = time_us(blk, iters)
    return out


def sampler_rates(co, reps=3, n_it=400):
    import torch

    from abdpymc_b200.engine import AbdEngine, forward
    from abdpymc_b200.sampler import AbdTarget, SamplerConfig, sample

    G, N, C = co.n_gaps, co.n_inds, 4
    rng = np.random.default_rng(3)
    x0 = np.array([1.0 / G, 2, 1, 10 / 11, -2, 2, 10 / 11, 0.5, 1, 1, -2, -1, 2, 1, -1, 2, 1], dtype=np.float64)
    q0 = torch.from_numpy(forward(x0)[None, :].repeat(C, 0)).to("cuda:0")
    rates = {False: [], True: []}
    with AbdEngine(co, splits=SPLITS) as eng:
        tgt = AbdTarget(eng, C, (rng.random((C, G, N)) < 0.04).astype(np.int8), (rng.random((C, N)) < 0.5).astype(np.int8),
                        seed=3)
        for rb in (False, True):   # warm-up (plans, tilings, modules)
            sample(tgt, q0, SamplerConfig(tune=20, draws=20, seed=1, record_deterministics_every=1, rao_blackwell=rb))
        for _ in range(reps):
            for rb in (False, True):
                torch.cuda.synchronize()
                t = time.perf_counter()
                sample(tgt, q0, SamplerConfig(tune=n_it // 2, draws=n_it - n_it // 2, seed=2, record_deterministics_every=1,
                                              rao_blackwell=rb))
                torch.cuda.synchronize()
                rates[rb].append(n_it / (time.perf_counter() - t))
    return {"sampler_iters_per_s_c4": rates[False], "sampler_iters_per_s_c4_rao_blackwell": rates[True]}


def se_ratio(n_inds=1000, C=32, tune=500, draws=2000):
    """Per-chain means of i / ab_s_waner and of their Rao-Blackwellised versions, through per-chain launches."""
    import torch

    from abdpymc_b200.engine import AbdEngine, forward
    from abdpymc_b200.sampler import AbdTarget, SamplerConfig, sample

    co = synthetic_cohort(n_inds)
    G, N = co.n_gaps, co.n_inds
    dev = torch.device("cuda:0")
    f64 = dict(dtype=torch.float64, device=dev)

    class PerChain(AbdTarget):
        def accumulate_deterministics(self, q, sums):
            if "i" not in sums:
                sums.update(i=torch.zeros(C, G, N, **f64), w=torch.zeros(C, N, **f64), i_rb=torch.zeros(C, G, N, **f64),
                            w_rb=torch.zeros(C, N, **f64))
            q = q.contiguous()
            e, st, di, dw = self.engine, self._stream(), self.d_i, self.d_w
            for c in range(C):
                qc = q.data_ptr() + 8 * 17 * c
                e.deterministics_accum_dev(1, qc, 1, di + c * G * N, dw + c * N, sums["i"][c].data_ptr(), None, None, st)
                e.infection_probs_accum_dev(1, qc, di + c * G * N, dw + c * N, sums["i_rb"][c].data_ptr(),
                                            sums["w_rb"][c].data_ptr(), st)
            torch.cuda.synchronize(dev)
            sums["w"] += torch.from_numpy(self.engine.download_state(C)[1]).to(dev, torch.float64)

    rng = np.random.default_rng(1)
    x0 = np.array([1.0 / G, 2, 1, 10 / 11, -2, 2, 10 / 11, 0.5, 1, 1, -2, -1, 2, 1, -1, 2, 1], dtype=np.float64)
    q0 = torch.from_numpy(forward(x0)[None, :] + rng.uniform(-1, 1, size=(C, 17))).to(dev)
    with AbdEngine(co, splits=SPLITS) as eng:
        tgt = PerChain(eng, C, np.zeros((C, G, N), np.int8), np.zeros((C, N), np.int8), seed=5)
        res = sample(tgt, q0, SamplerConfig(tune=tune, draws=draws, seed=5, record_deterministics_every=1))
    m = res.means   # already divided by C x draws: per-chain means are C times these
    out = {}
    for plain, rb in (("i", "i_rb"), ("w", "w_rb")):
        a, b = m[plain] * C, m[rb] * C
        p = a.mean(axis=0)
        sel = (p >= 0.01) & (p <= 0.99)
        sa, sb = a.std(axis=0, ddof=1)[sel], b.std(axis=0, ddof=1)[sel]
        keep = sa > 0
        out[f"se_ratio_{plain}"] = float(np.median(sb[keep] / sa[keep]))
        out[f"n_elements_{plain}"] = int(keep.sum())
    out.update(se_ratio_setup=f"{n_inds} individuals, splits {SPLITS}, {C} chains, tune {tune}, draws {draws}")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", default=None, help="directory for the JSON result")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("infection_probs_bench.py measures the GPU: no CUDA device")
    from abdpymc_b200 import build
    from abdpymc_b200.engine import AbdEngine

    build.build()
    rng = np.random.default_rng(7)
    base = synthetic_cohort(10_000)
    res = {"info": device_info(), "inputs": "L2-resident (cohort arrays < 126 MB, re-read every launch)"}
    with AbdEngine(base, splits=SPLITS) as eng:
        res["G31_splits"] = kernel_times(eng, rng, (4, 128), args.iters, with_blk=True)
    with AbdEngine(base, splits=()) as eng:
        res["G31_no_splits"] = kernel_times(eng, rng, (4,), args.iters)
    with AbdEngine(repeated(base, 3), splits=SPLITS) as eng:
        res["G93_splits"] = kernel_times(eng, rng, (4,), max(args.iters // 4, 20))
    res["sampler_10k"] = sampler_rates(base)
    res["se_ratio"] = se_ratio()
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).mkdir(parents=True, exist_ok=True)
        (Path(args.out) / "infection_probs_bench.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
