#!/usr/bin/env python3
"""Benchmark of the abdpymc inference hot path on B200 (see DESIGN.md, "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): the simulated
10 000-individual cohort of SURVEY.md section 8d (bootstrap of the bundled 1520-individual
schedule, forward-simulated with the reference's default dynamics), 31 monthly gaps, splits
(14, 20), 4 chains per GPU.  With N > 1 GPUs every rank holds the whole cohort and its own 4
chains (chain sharding: no data-path collective, weak scaling).

One STEP = EVALS_PER_STEP (256) consecutive batched logp+grad evaluations of all 4 chains --
a block of NUTS leapfrogs -- replayed as one CUDA graph.  Consecutive evaluations rotate over
independent replicas of the cohort + chain state whose total footprint exceeds twice the L2
(126 MB), so every evaluation streams its inputs from HBM ("inputs larger than L2").
`value` = chain evaluations per second (C * 256 * K / device time, max over ranks, CUDA events).
`e2e` = the same metric through the host-pointer C-ABI call abd_logp_dlogp(q17, i_raw, waner)
with pinned HOST buffers: every call copies all three inputs to the device and the results back.
The `gibbs` object reports abd_gibbs_sweep the same way (its own timed regions).
--dump-outputs DIR writes what the last timed step returned to its caller, DIR/logp.npy (C,) and
DIR/dlogp.npy (C, 17), float64, all ranks' chains: the inputs are seeded, so two builds can be
compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
# the benchmark leaves the tree as it found it (which may be read-only): no __pycache__ directories
sys.dont_write_bytecode = True

N_INDS = 10_000
N_CHAINS = 4
SPLITS = (14, 20)
EVALS_PER_STEP = 256
# what the benchmark cohort was simulated with (cohort.SimParams; simulation.py defaults).  The S
# response of the model has no temp factor (abd.py:263-274), so ab_s_temp* have no counterpart.
SIM_TRUTH = {"ab_n_perm": 2.0, "ab_n_temp": 1.5, "ab_n_rho": 0.95, "ab_n_init": -2.0, "ab_s_perm": 2.0, "ab_s_rho": 0.95,
             "ab_s_init": -2.0, "it_n_b": -2.2, "it_n_d": 1.6, "it_n_sigma": 0.1, "it_s_b": -2.2, "it_s_d": 1.6,
             "it_s_sigma": 0.1}
L2_BYTES = 126e6
METRIC = "logp+grad evals/s (10k individuals, joint logp + 17-dim gradient, per chain)"


# ------------------------------------------------------------------------------------------
def workload(n_inds=N_INDS, n_chains=N_CHAINS, seed=0, chain_offset=0):
    from abdpymc_b200.cohort import synthetic_cohort
    from abdpymc_b200.engine import forward

    co = synthetic_cohort(n_inds)
    rng = np.random.default_rng(1000 + seed + chain_offset)

    def gam(mu, sd, size):
        return rng.gamma(mu * mu / sd**2, sd**2 / mu, size)

    C = n_chains
    vals = np.stack([
        np.clip(rng.beta(1, co.n_gaps - 1, C), 1e-4, 1 - 1e-4), gam(2, .5, C), gam(1, .5, C), rng.beta(10, 1, C),
        rng.normal(-2, 1, C), gam(2, .5, C), rng.beta(10, 1, C), np.clip(rng.beta(1, 1, C), 1e-4, 1 - 1e-4),
        gam(1, .5, C), gam(1, .5, C), rng.normal(-2, 1, C), rng.normal(-1, .5, C), rng.normal(2, .5, C),
        rng.exponential(1, C) + 0.05, rng.normal(-1, .5, C), rng.normal(2, .5, C), rng.exponential(1, C) + 0.05,
    ], axis=1)  # fmt: skip
    q = forward(vals)
    i_raw = (rng.random((C, co.n_gaps, co.n_inds)) < 0.04).astype(np.int8)
    w = (rng.random((C, co.n_inds)) < 0.5).astype(np.int8)
    return co, q, vals, i_raw, w


def workload_name(co, n_chains=N_CHAINS):
    """config.workload: one string for both arms (the driver compares them)."""
    return (f"simulated {co.n_inds}-individual cohort (G={co.n_gaps}, {co.n_rows} OD rows), {n_chains} chains per GPU, "
            f"splits {list(SPLITS)}")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


ISSUE_PEAK_GINST = 148 * 4 * 1.965   # warp instructions / ns: 148 SMs x 4 schedulers x 1 per clock at clocks.max.sm


def ncu_issue(kernel, t_launch_s):
    """The second roof: instruction issue.  Warp instructions per launch from the committed ncu capture
    (smsp__inst_executed.sum, static) / this run's launch duration, against 148 SMs x 4 schedulers x 1.965 GHz."""
    p = ROOT / "profiles" / "ncu_traffic.json"
    try:
        n = float(json.loads(p.read_text())[kernel]["warp_inst"])
    except Exception:
        return None
    ach = n / t_launch_s / 1e9
    return {"warp_inst_per_launch": n, "achieved_ginst_per_s": ach, "peak_ginst_per_s": ISSUE_PEAK_GINST,
            "frac": ach / ISSUE_PEAK_GINST, "source": "static: smsp__inst_executed.sum of the committed ncu capture (profiles/ncu_traffic.json)"}


TRAFFIC_SOURCE = ("static: dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture "
                  "of this kernel on this workload (profiles/ncu_traffic.json, profiles/README.md); not re-measured in this run")


def ncu_traffic(kernel):
    p = ROOT / "profiles" / "ncu_traffic.json"
    if p.exists():
        try:
            d = json.loads(p.read_text()).get(kernel)
            return None if d is None else int(d["dram_bytes_read"]) + int(d["dram_bytes_write"])
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------------
# CPU baseline: the oracle's restatement of the reference's dense (G,G,N) formulation
# ------------------------------------------------------------------------------------------
_CPU = {}


def _cpu_init(n_sub, dense):
    from oracle import abd_oracle as ora

    os.environ["OMP_NUM_THREADS"] = "1"
    co, q, vals, i_raw, w = workload()
    sub = co.take(np.arange(n_sub))
    _CPU.update(o=ora.Oracle(sub, splits=SPLITS, dense=dense), q=q, i_raw=i_raw[:, :, :n_sub], w=w[:, :n_sub])


def _cpu_eval(k):
    c = k % N_CHAINS
    t = time.perf_counter()
    _CPU["o"].logp_dlogp(_CPU["q"][c], _CPU["i_raw"][c], _CPU["w"][c])
    return time.perf_counter() - t


def _cpu_eval_value(k):
    """Value only (no gradient): what one BinaryGibbsMetropolis proposal costs the reference."""
    c = k % N_CHAINS
    t = time.perf_counter()
    _CPU["o"].logp(_CPU["q"][c], _CPU["i_raw"][c], _CPU["w"][c])
    return time.perf_counter() - t


def cpu_throughput(n_sub, dense, cores, steps, warmup, fn=None):
    """steps x (one logp+grad evaluation on n_sub individuals on each of `cores` processes).
    Returns (chain-evals/s extrapolated linearly to N_INDS individuals, seconds per step)."""
    import multiprocessing as mp

    fn = fn or _cpu_eval
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_cpu_init, initargs=(n_sub, dense)) as pool:
        for _ in range(warmup):
            pool.map(fn, range(cores), chunksize=1)
        t0 = time.perf_counter()
        for _ in range(steps):
            pool.map(fn, range(cores), chunksize=1)
        dt = time.perf_counter() - t0
    evals = steps * cores * (n_sub / N_INDS)
    return evals / dt, dt / steps


def cpu_c_port(seconds=3.0):
    """The compiled CPU port (oracle/abd_oracle_c.c: plain C, OpenMP over individuals and OD rows, recurrence
    form) on all host threads, whole 10k cohort: joint logp + gradient evaluations per second.  Never fatal."""
    try:
        from oracle import c_oracle

        co, q, _, i_raw, w = workload()
        threads = min(os.cpu_count() or 1, 64)
        o = c_oracle.COracle(co, splits=SPLITS, threads=threads)
        for c in range(N_CHAINS):
            o.logp_dlogp(q[c], i_raw[c], w[c])
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds or n < 8:
            o.logp_dlogp(q[n % N_CHAINS], i_raw[n % N_CHAINS], w[n % N_CHAINS])
            n += 1
        dt = time.perf_counter() - t0
        return {"value": n / dt, "unit": "evals/s", "threads": threads, "kind": "port",
                "sample": f"{n} joint logp+grad evaluations of the whole {co.n_inds}-individual cohort in {dt:.1f} s, one process, "
                          f"{threads} OpenMP threads",
                "what": "oracle/abd_oracle_c.c: the O(G N) recurrence form in plain C (gcc -O2 -fopenmp), checked against the "
                        "reference-generated goldens; the algorithmically fair compiled CPU implementation of this path"}
    except Exception as exc:  # a missing compiler on some box must not cost the bench line
        return {"unavailable": f"{type(exc).__name__}: {exc}"[:200]}


def cpu_c_gibbs(seconds=3.0):
    """One Gibbs sweep of one chain over the whole 10k cohort by the compiled CPU port (abd_c_gibbs_sweep: the
    sweep exactly as the CUDA kernel schedules it -- same Philox streams, same decisions --, OpenMP over
    individuals, the flipped bit's individual re-evaluated per proposal), all host threads.  Never fatal."""
    try:
        from oracle import c_oracle

        co, _, vals, i_raw, w = workload()
        th = vals[:, [1, 2, 3, 4, 5, 6, 10, 11, 12, 13, 14, 15, 16]]
        threads = min(os.cpu_count() or 1, 64)
        o = c_oracle.COracle(co, splits=SPLITS, threads=threads)
        o.gibbs_sweep(th[0], vals[0, 0], vals[0, 7], i_raw[0], w[0], 1, 0, 0)
        n, t0, props = 0, time.perf_counter(), 0
        while time.perf_counter() - t0 < seconds or n < 2:
            c = n % N_CHAINS
            props += o.gibbs_sweep(th[c], vals[c, 0], vals[c, 7], i_raw[c], w[c], 1, n, c)[2][0]
            n += 1
        dt = time.perf_counter() - t0
        return {"value": n / dt, "unit": "sweeps/s", "threads": threads, "kind": "port", "proposals_per_sweep": props / n,
                "sample": f"{n} sweeps of one chain over all {co.n_inds} individuals in {dt:.1f} s, one process, {threads} OpenMP threads",
                "what": "oracle/abd_oracle_c.c abd_c_gibbs_sweep: the kernel's sweep restated in plain C (bit-identical decisions to "
                        "the NumPy restatement the GPU sweep is tested against); measured, not extrapolated"}
    except Exception as exc:
        return {"unavailable": f"{type(exc).__name__}: {exc}"[:200]}


def cpu_baseline():
    """The bounded CPU sample reported next to the GPU number (rank 0, N = 1 only).  Runs
    before CUDA is initialised in this process (the pool forks)."""
    cores = min(os.cpu_count() or 1, 64)
    n_sub, steps = 5000, 20
    v_dense, _ = cpu_throughput(n_sub, True, cores, steps, 1)
    v_scan, _ = cpu_throughput(N_INDS, False, cores, steps, 1)
    # Gibbs on the CPU: the reference's BinaryGibbsMetropolis evaluates the WHOLE model's logp (value
    # only) once per proposed flip, 0.8 (G N + N) proposals per sweep and chain (SURVEY 3.3); one
    # sweep at 10k individuals takes hours, so it is extrapolated from timed value-only evaluations
    v_val, _ = cpu_throughput(n_sub, True, cores, 8, 1, fn=_cpu_eval_value)
    co = workload()[0]
    proposals = 0.8 * (co.n_gaps * co.n_inds + co.n_inds)
    c_port = cpu_c_port()  # (after the pools above: its OpenMP threads must not exist when they fork)
    c_gibbs = cpu_c_gibbs()
    return {"value": v_dense, "unit": "evals/s", "cores": cores, "kind": "port",
            "gibbs": {"value": v_val / proposals, "unit": "sweeps/s", "logp_value_evals_per_s": v_val,
                      "proposals_per_sweep": proposals, "c_port": c_gibbs,
                      "sample": f"extrapolated: {cores} processes x 8 value-only dense-formulation logp evaluations on the "
                                f"first {n_sub} individuals (scaled to {N_INDS}), one evaluation per proposed flip, "
                                f"0.8 (G N + N) proposals per sweep (BinaryGibbsMetropolis, transit_p = 0.8)"},
            "sample": (f"{steps} steps x {cores} processes x 1 dense-formulation logp+grad evaluation on the first {n_sub} of "
                       f"{N_INDS} individuals, scaled by {n_sub}/{N_INDS}; PyMC is not installable offline, so this is "
                       "the NumPy restatement of the reference graph (oracle/abd_oracle.py)"),
            "recurrence_port_evals_per_s": v_scan,
            "c_port": c_port}


def run_reference(args):
    """--impl reference: the reference's own CPU formulation (restated: PyMC is not installable
    offline), all host cores, same metric / config; rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cores = min(os.cpu_count() or 1, 64)
    steps, warmup = max(args.steps, 1), max(args.warmup, 0)
    # one dense evaluation costs ~65 us per individual per core: bound the whole run to ~100 s
    budget_s = 100.0
    n_sub = int(min(N_INDS, max(250, budget_s / ((steps + warmup) * 65e-6 * 1.5))))
    value, s_per_step = cpu_throughput(n_sub, True, cores, steps, warmup)
    sample = (f"each step = 1 logp+grad evaluation of the dense (G,G,N) formulation on the first {n_sub} of the "
              f"{N_INDS} individuals on each of {cores} processes; throughput scaled by {n_sub}/{N_INDS} (cost is linear in N)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": s_per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(workload()[0]),
                   "reference": "NumPy restatement of abd.py's dense formulation (oracle/abd_oracle.py); PyMC unavailable offline"},
        "cpu_baseline": {"value": value, "unit": "evals/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        # beside the reference's own (dense) formulation: the compiled O(G N) port of the same path on the same cores
        "fair_port": cpu_c_port(),
    }
    emit(line)


# ------------------------------------------------------------------------------------------
def _timed_us(fn, n, dist, dev, warm=5):
    """Average device time (us) of n calls of fn on the current stream, max over ranks."""
    import torch

    for _ in range(warm):
        fn()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) / n * 1e3


def bench_create(co, device):
    """SURVEY 8f-4: how a large cohort reaches the GPU.  Seconds for (a) the reference's route, text files ->
    arrays (pd.read_csv of df.csv, np.loadtxt of vacs.txt / pcrpos.txt: TiterData.from_disk, abd.py:171-202),
    (b) abd_create from in-memory arrays (sorts, CSR / cell tables, packing, upload), (c) abd_create_from_cache
    from the binary cache file abd_save_cache wrote (read + upload)."""
    import tempfile

    from abdpymc_b200.cohort import CohortArrays
    from abdpymc_b200.engine import AbdEngine

    res = {"n_inds": co.n_inds, "n_rows": co.n_rows}
    with tempfile.TemporaryDirectory() as td:
        t = time.perf_counter()
        co.to_disk(Path(td) / "cohort_data")
        res["write_text_files_s"] = time.perf_counter() - t
        t = time.perf_counter()
        back = CohortArrays.from_disk(Path(td) / "cohort_data")
        res["parse_text_files_s"] = time.perf_counter() - t
        assert back.n_rows == co.n_rows
        t = time.perf_counter()
        eng = AbdEngine(co, splits=SPLITS, device=device)
        res["abd_create_s"] = time.perf_counter() - t
        cache = Path(td) / "cohort.abdcache"
        t = time.perf_counter()
        eng.save_cache(cache)
        res["abd_save_cache_s"] = time.perf_counter() - t
        res["cache_file_mb"] = cache.stat().st_size / 1e6
        eng.close()
        t = time.perf_counter()
        eng = AbdEngine.from_cache(cache, device=device, splits=SPLITS)
        res["abd_create_from_cache_s"] = time.perf_counter() - t
        eng.close()
    res["speedup_cache_vs_text_route"] = (res["parse_text_files_s"] + res["abd_create_s"]) / res["abd_create_from_cache_s"]
    return res


def bench_sharded(dist, rank, world, local, dev, K, n_big=100_000, chain_counts=(4, 32), block=32):
    """BASELINE configs[3].  One evaluation = joint logp + gradient of all C chains on the 100k cohort.
    `one_gpu`: the whole cohort on rank 0's GPU (the baseline the speed-ups are quoted against; the other
    ranks idle).  With world > 1: individuals split into `world` contiguous blocks, the C x 16 sums exchanged
    per evaluation by NCCL (three launches + a collective, host-driven) or inside the kernel over NVLink peer
    memory (one launch; host-driven, and as a CUDA graph of `block` evaluations, which removes the launch skew
    between the ranks' host threads).  Everything here re-evaluates ONE cohort back to back (L2-resident on
    every side, the access pattern of consecutive leapfrogs)."""
    import torch

    from abdpymc_b200.cohort import synthetic_cohort
    from abdpymc_b200.distributed import ShardedEngine
    from abdpymc_b200.engine import AbdEngine

    big = synthetic_cohort(n_big)
    out = {"workload": f"simulated {n_big}-individual cohort (G={big.n_gaps}, {big.n_rows} OD rows) sharded by individual over "
                       f"{world} GPU(s), splits {list(SPLITS)}", "unit": "us per evaluation of all C chains", "by_chains": {}}
    side = torch.cuda.Stream(device=dev)
    n_rep = max(3, min(20, K))
    if rank == 0:
        out["create"] = bench_create(big, local)
    for Csh in chain_counts:
        rngb = np.random.default_rng(77)
        ib = (rngb.random((Csh, big.n_gaps, big.n_inds)) < 0.04).astype(np.int8)
        wb = (rngb.random((Csh, big.n_inds)) < 0.5).astype(np.int8)
        tqs = torch.from_numpy(workload(n_inds=1000, n_chains=Csh, chain_offset=0)[1]).to(dev)  # identical q on every rank
        res = {}
        # -- baseline: the whole cohort on one GPU (rank 0), a graph of `block` evaluations
        t1 = torch.zeros(1, dtype=torch.float64, device=dev)
        lp1 = torch.zeros(Csh, dtype=torch.float64, device=dev)
        if rank == 0:
            with AbdEngine(big, splits=SPLITS, device=local) as e1g:
                e1g.upload_state(ib, wb)
                di, dw = e1g.state_dev(Csh)
                o1 = torch.zeros(Csh, dtype=torch.float64, device=dev)
                o2 = torch.zeros(Csh, 17, dtype=torch.float64, device=dev)
                with torch.cuda.stream(side):
                    e1g.logp_dlogp_dev(Csh, tqs.data_ptr(), di, dw, o1.data_ptr(), o2.data_ptr(), side.cuda_stream)
                side.synchronize()
                g1 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g1, stream=side):
                    for _ in range(block):
                        e1g.logp_dlogp_dev(Csh, tqs.data_ptr(), di, dw, o1.data_ptr(), o2.data_ptr(), side.cuda_stream)
                t1[0] = _timed_us(g1.replay, n_rep, None, dev, warm=2) / block
                lp1.copy_(o1)
                plan1 = e1g.last_plan()
                del g1
        if dist:
            dist.broadcast(t1, 0)
            dist.broadcast(lp1, 0)
        us1 = float(t1.item())
        res["one_gpu"] = {"us_per_eval": us1, "evals_per_s": Csh / us1 * 1e6}
        if rank == 0:
            res["one_gpu"]["plan"] = plan1
        if dist:
            se = ShardedEngine(big, splits=SPLITS, device_index=local, rank=rank, world=world)
            se.upload_state(ib, wb)
            us_nccl = _timed_us(lambda: se.logp_dlogp(tqs), max(50, 10 * n_rep), dist, dev, warm=10)
            lp_n = se.logp_dlogp(tqs)[0].clone()
            se.close()
            sf = ShardedEngine(big, splits=SPLITS, device_index=local, rank=rank, world=world, fused=True, max_chains=Csh)
            sf.upload_state(ib, wb)
            us_fused = _timed_us(lambda: sf.logp_dlogp(tqs), max(50, 10 * n_rep), dist, dev, warm=10)
            lp_f = sf.logp_dlogp(tqs)[0].clone()
            sf.exchange_wait_us(reset=True)
            with torch.cuda.stream(side):
                sf.logp_dlogp(tqs)
            side.synchronize()
            dist.barrier()
            gf = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gf, stream=side):
                for _ in range(block):
                    sf.logp_dlogp(tqs)
            sf.exchange_wait_us(reset=True)
            us_graph = _timed_us(gf.replay, n_rep, dist, dev, warm=2) / block
            wait_us = sf.exchange_wait_us(reset=True)
            tw = torch.tensor([wait_us], dtype=torch.float64, device=dev)
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
            sf.engine.xch_status()
            plan_f = sf.engine.last_plan()
            del gf
            sf.close()
            rel = float(((lp_f - lp1).abs() / lp1.abs()).max())
            res["nccl"] = {"us_per_eval": us_nccl, "speedup_vs_1gpu": us1 / us_nccl,
                           "collective": f"torch.distributed all_reduce(SUM) of {Csh} x 16 float64 per evaluation (NCCL), host-driven"}
            res["fused_peer_allreduce"] = {
                "us_per_eval": us_fused, "speedup_vs_1gpu": us1 / us_fused, "host_driven": True,
                "bitwise_equal_to_nccl_path": bool(torch.equal(lp_f, lp_n)), "rel_err_vs_one_gpu": rel}
            res["fused_peer_allreduce_graph"] = {
                "us_per_eval": us_graph, "speedup_vs_1gpu": us1 / us_graph, "evals_per_s": Csh / us_graph * 1e6,
                "exchange_wait_us_per_eval_max_over_ranks": float(tw.item()), "plan_rank0": plan_f,
                "note": f"CUDA graph of {block} evaluations per rank; exchange_wait = mean time the finishing CTA spent waiting "
                        "for its slowest peer's sums (launch skew + NVLink latency), measured in the kernel with %globaltimer"}
        out["by_chains"][str(Csh)] = res
    # ---- the compound sampler (device HMC + Gibbs) on the same cohort, 4 chains: one GPU holds the whole cohort
    #      (world == 1), or the individuals are sharded with the all-reduce inside every leapfrog launch ----
    from abdpymc_b200.engine import forward
    from abdpymc_b200.sampler import AbdTarget, SamplerConfig, sample

    Cs, G, N = 4, big.n_gaps, big.n_inds
    x0 = np.array([1.0 / G, 2, 1, 10 / 11, -2, 2, 10 / 11, 0.5, 1, 1, -2, -1, 2, 1, -1, 2, 1], dtype=np.float64)
    q0 = forward(x0)[None, :] + np.random.default_rng(9).uniform(-0.5, 0.5, size=(Cs, 17))
    cfg = SamplerConfig(tune=150, draws=150, seed=3)
    zi, zw = np.zeros((Cs, G, N), np.int8), np.zeros((Cs, N), np.int8)
    if dist:
        from abdpymc_b200.distributed import ShardedTarget

        sh = ShardedEngine(big, splits=SPLITS, device_index=local, rank=rank, world=world, fused=True, max_chains=Cs)
        tgt = ShardedTarget(sh, Cs, zi, zw, seed=5)
        dist.barrier()
        r = sample(tgt, torch.from_numpy(q0).to(dev), cfg)
        tw = torch.tensor([r.wall_s], dtype=torch.float64, device=dev)
        dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        wall = float(tw.item())
        sh.close()
    else:
        with AbdEngine(big, splits=SPLITS, device=local) as e1g:
            r = sample(AbdTarget(e1g, Cs, zi, zw, seed=5), torch.from_numpy(q0).to(dev), cfg)
        wall = r.wall_s
    out["sampler"] = {"chains": Cs, "iterations_per_s": (cfg.tune + cfg.draws) / wall, "mean_accept": float(r.accept.mean()),
                      "what": f"device HMC + Gibbs, {cfg.tune} + {cfg.draws} iterations from the all-zero indicator state (burn-in "
                              "regime: many accepted flips), " + ("individuals sharded, fused NVLink all-reduce in every leapfrog "
                              "launch, Gibbs sweeps local" if dist else "whole cohort on one GPU")}
    return out


def bench_ess(eng, co, C, dev, rank, world, dist, tune_n, draws_n, cpu):
    """A bounded run of the built-in sampler with C chains per GPU; every rank samples its own chains (chain
    sharding: no collective; Philox streams keyed by global chain), diagnostics over all world x C chains."""
    import torch

    G, N = co.n_gaps, co.n_inds
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    from abdpymc_b200 import diagnostics as dg
    from abdpymc_b200.sampler import AbdTarget, SamplerConfig, sample

    from abdpymc_b200.engine import forward

    # every rank samples its own C chains (chain sharding: no collective), seeds differ by rank
    eng.set_chain_offset(rank * C)
    tgt = AbdTarget(eng, C, np.zeros((C, G, N), np.int8), np.zeros((C, N), np.int8), seed=1)
    cfg = SamplerConfig(tune=tune_n, draws=draws_n, seed=1 + rank)
    # PyMC-like initial point: prior means on the constrained scale, jittered in q space (abd.infer_builtin)
    x0 = np.array([1.0 / G, 2, 1, 10 / 11, -2, 2, 10 / 11, 0.5, 1, 1, -2, -1, 2, 1, -1, 2, 1], dtype=np.float64)
    q0 = forward(x0)[None, :] + np.random.default_rng(1 + rank).uniform(-1, 1, size=(C, 17))
    barrier()
    res = sample(tgt, torch.from_numpy(q0).to(dev), cfg)
    draws_q, wall = res.q, res.wall_s
    if dist:  # gather every rank's draws on all ranks: diagnostics over world x C chains, slowest rank's wall time
        tdraw = torch.from_numpy(np.ascontiguousarray(res.q)).to(dev)
        parts = [torch.empty_like(tdraw) for _ in range(world)]
        dist.all_gather(parts, tdraw)
        draws_q = torch.cat(parts, dim=0).cpu().numpy()
        tw = torch.tensor([res.wall_s], dtype=torch.float64, device=dev)
        dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        wall = float(tw.item())
    from abdpymc_b200.engine import Q17_RV, backward as _bw

    xq = _bw(draws_q)
    summ = dg.summary({name: xq[:, :, k] for k, (name, _) in enumerate(Q17_RV)})
    res.wall_s = wall
    vals_ess = sorted(v["ess_bulk"] for v in summ.values())
    # R-hat gate: an ESS/s is only quoted for quantities whose chains agree (rank-normalised split R-hat <= 1.05);
    # if any of the 17 scalars fails it the run as a whole is reported as not converged and min ESS/s is null
    RHAT_MAX = 1.05
    bad = sorted(name for name, v in summ.items() if not (v["rhat"] <= RHAT_MAX))
    ok_ess = sorted(v["ess_bulk"] for v in summ.values() if v["rhat"] <= RHAT_MAX)
    converged = not bad
    # Gibbs sweeps on the chains' states at the end of the run (the stationary regime: few accepted flips)
    tq_end = torch.from_numpy(res.q[:, -1, :].copy()).to(dev)
    torch.cuda.synchronize()
    e0.record()
    for k in range(50):
        tgt.gibbs(tq_end, 10_000 + k)
    e1.record()
    torch.cuda.synchronize()
    # wall time of the whole run (tune + draws) is charged to the draws kept
    ess = {"sampler": f"built-in batched HMC (dense metric) + GPU Metropolised-Gibbs sweep, device-resident transitions, "
                      f"{world * C} chains x ({tune_n} tune + {draws_n} draws)" + (f" on {world} GPUs" if world > 1 else ""),
           "chains": world * C, "wall_s": res.wall_s, "iterations_per_s": (tune_n + draws_n) / res.wall_s,
           "converged": converged, "rhat_gate": RHAT_MAX, "not_converged": bad,
           "min_bulk_ess_per_s": (vals_ess[0] / res.wall_s) if converged else None,
           "median_bulk_ess_per_s": (vals_ess[len(vals_ess) // 2] / res.wall_s) if converged else None,
           "min_bulk_ess_per_s_over_converged_quantities": (ok_ess[0] / res.wall_s) if ok_ess else None,
           "n_converged_quantities": len(ok_ess),
           "max_rhat": max(v["rhat"] for v in summ.values()), "grad_evals": res.n_grad_evals,
           "gibbs_sweeps_per_s_stationary": world * C * 50 / (e0.elapsed_time(e1) / 1e3),
           "posterior": {name: {"mean": float(np.mean(xq[:, :, k])), "sd": float(np.std(xq[:, :, k])),
                                "ess_bulk": float(summ[name]["ess_bulk"]), "rhat": float(summ[name]["rhat"]),
                                "simulated_with": SIM_TRUTH.get(name)}
                         for k, (name, _) in enumerate(Q17_RV)},
           "note": "PyMC is not installable offline, so there is no measured PyMC-CPU ESS/s beside it (cpu_extrapolation "
                   "scales this run's ESS per iteration by the CPU cost of one iteration); the slowest-mixing "
                   "parameters are those coupled to the latent infection indicators (data-augmentation Gibbs); "
                   "quantities that fail the R-hat gate get no ESS/s"}
    if cpu and cpu.get("gibbs"):
        # one iteration of the reference's compound step = one NUTS draw (>= the 5 leapfrogs used here) + one
        # BinaryGibbsMetropolis sweep; its chains run one per core.  Same ESS per iteration assumed.
        t_iter = 1.0 / (cpu["gibbs"]["value"] / cpu["cores"]) + cfg.n_leapfrog / (cpu["value"] / cpu["cores"])
        ess_per_iter = (vals_ess[0] if converged else (ok_ess[0] if ok_ess else float("nan"))) / (tune_n + draws_n)
        ess["cpu_extrapolation"] = {
            "seconds_per_iteration_per_chain": t_iter, "min_bulk_ess_per_s": ess_per_iter / t_iter,
            "how": f"this run's min bulk ESS per iteration ({world * C} chains) / CPU seconds per iteration of one chain on "
                   f"one core (1 Gibbs sweep + {cfg.n_leapfrog} logp+grad evaluations of the restated reference, "
                   "cpu_baseline), chains in parallel on separate cores"}

    return ess


def dump_outputs(directory, last_step, dist, rank, world):
    """logp.npy / dlogp.npy of the last timed step, every rank's chains in rank order (written by rank 0)."""
    import torch

    arrays = {}
    for name, t in zip(("logp", "dlogp"), last_step):
        if dist:
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            t = torch.cat(parts)
        arrays[name] = t.cpu().numpy()
    if rank == 0:
        d = Path(directory)
        d.mkdir(parents=True, exist_ok=True)
        for name, a in arrays.items():
            np.save(d / f"{name}.npy", a.astype(np.float64))


# ------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch

    from abdpymc_b200 import build
    from abdpymc_b200.engine import AbdEngine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    C, K, W = N_CHAINS, args.steps, max(args.warmup, 3)
    cpu = cpu_baseline() if (world == 1 and not args.no_cpu_baseline and not args.profile) else None
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        build.build()
    if dist:
        dist.barrier()

    co, q, vals, i_raw, w = workload(chain_offset=rank * N_CHAINS)
    G, N = co.n_gaps, co.n_inds
    th13 = vals[:, [1, 2, 3, 4, 5, 6, 10, 11, 12, 13, 14, 15, 16]].copy()
    p, pw = vals[:, 0].copy(), vals[:, 7].copy()

    eng0 = AbdEngine(co, splits=SPLITS, device=local)
    a_logp = eng0.algorithmic_bytes_logp(C)
    a_gibbs = eng0.algorithmic_bytes_gibbs(C)
    n_rep = int(np.ceil(2 * L2_BYTES / a_logp)) + 1
    engines = [eng0] + [AbdEngine(co, splits=SPLITS, device=local) for _ in range(n_rep - 1)]
    states = []
    for e in engines:
        e.upload_state(i_raw, w)
        states.append(e.state_dev(C))

    tq = torch.from_numpy(q).to(dev)
    if args.profile:
        tth = torch.from_numpy(th13).to(dev)
        tp, tpw = torch.from_numpy(p).to(dev), torch.from_numpy(pw).to(dev)
        o1 = torch.zeros(C, dtype=torch.float64, device=dev)
        o2 = torch.zeros(C, 17, dtype=torch.float64, device=dev)
        for k in range(max(K, 1) * 8):
            j = k % n_rep
            engines[j].logp_dlogp_dev(C, tq.data_ptr(), states[j][0], states[j][1], o1.data_ptr(), o2.data_ptr(), 0)
        for k in range(max(K, 1)):
            j = k % n_rep
            engines[j].gibbs_sweep_dev(C, tth.data_ptr(), 0, tp.data_ptr(), tpw.data_ptr(), states[j][0], states[j][1], 1, k)
        for k in range(max(K, 1)):  # the per-chunk block draw (k_gibbs_blk)
            j = k % n_rep
            engines[j].gibbs_sweep_dev(C, tth.data_ptr(), 0, tp.data_ptr(), tpw.data_ptr(), states[j][0], states[j][1], 1,
                                       100 + k, mode=2)
        # the throughput regime: 128 chains per launch (BASELINE configs[4], one GPU's share)
        CB = 128
        _, qb, _, ib, wb = workload(n_chains=CB)
        eng_b = AbdEngine(co, splits=SPLITS, device=local)
        eng_b.upload_state(ib, wb)
        sb = eng_b.state_dev(CB)
        tqb = torch.from_numpy(qb).to(dev)
        ob1 = torch.zeros(CB, dtype=torch.float64, device=dev)
        ob2 = torch.zeros(CB, 17, dtype=torch.float64, device=dev)
        for k in range(max(K, 1)):
            eng_b.logp_dlogp_dev(CB, tqb.data_ptr(), sb[0], sb[1], ob1.data_ptr(), ob2.data_ptr(), 0)
        torch.cuda.synchronize()
        print("profile run done:", o1.cpu().numpy())
        return
    out = torch.zeros(C, dtype=torch.float64, device=dev)
    outg = torch.zeros(C, 17, dtype=torch.float64, device=dev)
    side = torch.cuda.Stream(device=dev)

    def enqueue_block(stream_handle, start=0):
        for k in range(EVALS_PER_STEP):
            j = (start + k) % n_rep
            engines[j].logp_dlogp_dev(C, tq.data_ptr(), states[j][0], states[j][1], out.data_ptr(), outg.data_ptr(),
                                      stream_handle)

    # warm every replica outside capture (first call allocates scratch), then capture one step
    with torch.cuda.stream(side):
        enqueue_block(side.cuda_stream)
    side.synchronize()
    check_lp = out.cpu().numpy().copy()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        enqueue_block(side.cuda_stream)

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    launches0 = sum(e.launch_count for e in engines)
    for _ in range(W):
        graph.replay()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        e0.record()
        for _ in range(K):
            graph.replay()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        last_step = (out.clone(), outg.clone())
        # keep the sampler alive long enough for at least a few samples under load
        t_end = time.time() + max(0.0, 0.6 - ms / 1e3)
        while time.time() < t_end:
            graph.replay()
        torch.cuda.synchronize()
    clocks = clk.summary()
    assert np.array_equal(out.cpu().numpy(), check_lp), "graph replay changed the result"
    if dist:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_step, dist, rank, world)
    n_launch = K * EVALS_PER_STEP
    value = world * C * n_launch / (ms / 1e3)
    t_kernel = ms / 1e3 / n_launch

    # ---- L2-resident variant (what consecutive NUTS leapfrogs on ONE cohort see) ----
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2, stream=side):
        for _ in range(EVALS_PER_STEP):
            eng0.logp_dlogp_dev(C, tq.data_ptr(), states[0][0], states[0][1], out.data_ptr(), outg.data_ptr(), side.cuda_stream)
    for _ in range(W):
        g2.replay()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(K):
        g2.replay()
    e1.record()
    torch.cuda.synchronize()
    ms_l2 = e0.elapsed_time(e1)

    # ---- the same block issued over S streams (independent evaluation requests: what S PyMC worker
    #      processes -- pm.sample(cores=S), one chain group each -- present to one GPU).  A single
    #      stream leaves the SMs idle while a launch's last CTA finalises and the next one starts;
    #      independent streams fill those gaps.  HBM-cold replicas as in the headline region. ----
    concurrent = {}
    for S in (2, 4):
        if n_rep < 2 * S:
            continue
        streams = [torch.cuda.Stream(device=dev) for _ in range(S - 1)]
        outs = [(torch.zeros_like(out), torch.zeros_like(outg)) for _ in range(S)]
        gS = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gS, stream=side):
            fork = torch.cuda.Event()
            fork.record(side)
            for st in streams:
                st.wait_event(fork)
            m = n_rep - n_rep % S  # engine j always runs on stream j % S: its scratch is never shared by two streams
            for k in range(EVALS_PER_STEP):
                j, sidx = k % m, k % S
                stream = side if sidx == 0 else streams[sidx - 1]
                o, og = outs[sidx]
                engines[j].logp_dlogp_dev(C, tq.data_ptr(), states[j][0], states[j][1], o.data_ptr(), og.data_ptr(),
                                          stream.cuda_stream)
            for st in streams:
                join = torch.cuda.Event()
                join.record(st)
                side.wait_event(join)
        for _ in range(W):
            gS.replay()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(K):
            gS.replay()
        e1.record()
        torch.cuda.synchronize()
        ms_S = e0.elapsed_time(e1)
        if dist:
            t = torch.tensor([ms_S], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_S = float(t.item())
        assert all(np.array_equal(o.cpu().numpy(), check_lp) for o, _ in outs), "concurrent streams changed the result"
        concurrent[f"{S}_streams"] = {"value": world * C * n_launch / (ms_S / 1e3), "unit": "evals/s",
                                      "avg_us_per_launch": ms_S / n_launch * 1e3,
                                      "hbm_frac": a_logp / (ms_S / 1e3 / n_launch) / 1e9 / measured_peak_gbs()[0]}
        del gS
    concurrent["note"] = ("the headline block issued round-robin over S streams inside one CUDA graph (independent evaluation "
                          "requests, e.g. S PyMC worker processes sharing the GPU); `value` stays the single-stream number")

    # ---- inside one persistent trajectory launch (abd_leapfrog_dev): L dependent leapfrog steps, each
    #      one full logp+grad evaluation at a new position; no launch / re-staging between them ----
    traj = None
    try:
        L = 64
        tq2, tp2, tg2 = tq.clone(), torch.zeros_like(tq), outg.clone()
        teps = torch.full((C,), 1e-4, dtype=torch.float64, device=dev)
        tmass = torch.eye(17, dtype=torch.float64, device=dev)
        with torch.cuda.stream(side):
            for _ in range(W):
                eng0.leapfrog_dev(C, L, tq2.data_ptr(), tp2.data_ptr(), tg2.data_ptr(), out.data_ptr(), teps.data_ptr(),
                                  tmass.data_ptr(), states[0][0], states[0][1], side.cuda_stream)
            e0.record()
            for _ in range(K):
                eng0.leapfrog_dev(C, L, tq2.data_ptr(), tp2.data_ptr(), tg2.data_ptr(), out.data_ptr(), teps.data_ptr(),
                                  tmass.data_ptr(), states[0][0], states[0][1], side.cuda_stream)
            e1.record()
        side.synchronize()
        eng0.leapfrog_status(C)
        ms_traj = e0.elapsed_time(e1)
        traj = {"value": world * C * L * K / (ms_traj / 1e3), "unit": "evals/s", "us_per_step": ms_traj / (K * L) * 1e3,
                "note": f"abd_leapfrog_dev: {L} dependent leapfrog steps per persistent launch, binary state staged once"}
    except Exception as ex:  # the grid does not fit at once on this device
        traj = {"unavailable": str(ex)[:200]}

    # ---- BASELINE configs[4], one GPU's share: 128 chains batched in one launch (throughput regime) ----
    CB = 128
    cob, qb, _, ib, wb = workload(n_chains=CB, chain_offset=rank * CB)
    eng_b = AbdEngine(co, splits=SPLITS, device=local)
    eng_b.upload_state(ib, wb)
    sb = eng_b.state_dev(CB)
    tqb = torch.from_numpy(qb).to(dev)
    outb = torch.zeros(CB, dtype=torch.float64, device=dev)
    outgb = torch.zeros(CB, 17, dtype=torch.float64, device=dev)
    with torch.cuda.stream(side):
        for _ in range(W):
            eng_b.logp_dlogp_dev(CB, tqb.data_ptr(), sb[0], sb[1], outb.data_ptr(), outgb.data_ptr(), side.cuda_stream)
    n_b = max(8, min(64, K))
    reps_b = []
    for _ in range(3):  # median of three repeats (a single block of ~40 launches is at the mercy of one hiccup)
        with torch.cuda.stream(side):
            e0.record()
            for _ in range(n_b):
                eng_b.logp_dlogp_dev(CB, tqb.data_ptr(), sb[0], sb[1], outb.data_ptr(), outgb.data_ptr(), side.cuda_stream)
            e1.record()
        side.synchronize()
        reps_b.append(e0.elapsed_time(e1))
    ms_b = sorted(reps_b)[1]
    a_b = eng_b.algorithmic_bytes_logp(CB)
    batched = {"chains": CB, "value": world * CB * n_b / (ms_b / 1e3), "unit": "evals/s", "avg_launch_us": ms_b / n_b * 1e3,
               "issue": ncu_issue("k_sums_128", ms_b / n_b / 1e3),
               "algorithmic_bytes_packed_state": int(CB * (8 * N + 216) + 2 * G * N + 20 * co.n_rows + 8 * (N + 1)),
               "algorithmic_bytes_per_launch": a_b, "hbm_frac": a_b / (ms_b / n_b / 1e3) / 1e9 / measured_peak_gbs()[0],
               "note": "one launch evaluates 128 chains; algorithmic_bytes_per_launch is SURVEY 8d's formula (int8 boundary "
                       "state, 40 MB); the kernel reads the packed resident copy instead (8 bytes per individual and chain)"}
    eng_b.close()
    del tqb, outb, outgb

    # ---- Deterministics (i, ab_n_mu, ab_s_mu of every (gap, individual): what a recorded draw costs):
    #      k_determ is the write-bound kernel of the path, 17 G N bytes out + G N + N bytes in per chain ----
    determ = {}
    for CD in (C, 128):
        cod, _, vd, idd, wdd = workload(n_chains=CD, chain_offset=rank * CD)
        eng_d = AbdEngine(co, splits=SPLITS, device=local)
        eng_d.upload_state(idd, wdd)
        sd = eng_d.state_dev(CD)
        thd = torch.from_numpy(vd[:, [1, 2, 3, 4, 5, 6, 10, 11, 12, 13, 14, 15, 16]].copy()).to(dev)
        oi = torch.empty(CD, G, N, dtype=torch.int8, device=dev)
        omn = torch.empty(CD, G, N, dtype=torch.float64, device=dev)
        oms = torch.empty(CD, G, N, dtype=torch.float64, device=dev)
        with torch.cuda.stream(side):
            for _ in range(W):
                eng_d.deterministics_dev(CD, thd.data_ptr(), sd[0], sd[1], oi.data_ptr(), omn.data_ptr(), oms.data_ptr(),
                                         side.cuda_stream)
            e0.record()
            n_d = 20
            for _ in range(n_d):
                eng_d.deterministics_dev(CD, thd.data_ptr(), sd[0], sd[1], oi.data_ptr(), omn.data_ptr(), oms.data_ptr(),
                                         side.cuda_stream)
            e1.record()
        side.synchronize()
        t_d = e0.elapsed_time(e1) / n_d / 1e3
        a_d = CD * (18 * G * N + N)
        determ[f"{CD}_chains"] = {"avg_launch_us": t_d * 1e6, "algorithmic_bytes_per_launch": a_d, "achieved_gbs": a_d / t_d / 1e9,
                                  "hbm_frac": a_d / t_d / 1e9 / measured_peak_gbs()[0],
                                  "outputs_larger_than_l2": bool(CD * 17 * G * N > L2_BYTES)}
        eng_d.close()
        del oi, omn, oms
    determ["note"] = ("abd_deterministics_dev (k_determ), the bandwidth-bound kernel of the path: one thread per (individual, chain) "
                      "runs the recurrence and writes int8 i and f64 ab_n_mu / ab_s_mu coalesced over individuals")

    # ---- e2e: host-pointer C-ABI call, pinned host buffers, all inputs copied every call ----
    hq = torch.from_numpy(q).pin_memory()
    hi = torch.from_numpy(i_raw).pin_memory()
    hw = torch.from_numpy(w).pin_memory()
    n_e2e = max(50, min(2000, K * 8))
    for k in range(W * 4):
        engines[k % n_rep].logp_dlogp(hq.numpy(), hi.numpy(), hw.numpy())
    barrier()
    t0 = time.perf_counter()
    for k in range(n_e2e):
        lp, gr = engines[k % n_rep].logp_dlogp(hq.numpy(), hi.numpy(), hw.numpy())
    dt_e2e = time.perf_counter() - t0
    t0 = time.perf_counter()
    for k in range(n_e2e):
        lp2, gr2 = engines[k % n_rep].logp_dlogp(hq.numpy())  # chain state already resident
    dt_res = time.perf_counter() - t0
    if dist:
        t = torch.tensor([dt_e2e, dt_res], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt_e2e, dt_res = (float(v) for v in t.tolist())
    assert np.array_equal(lp, check_lp) and np.array_equal(lp2, check_lp)

    # ---- Gibbs sweeps ----
    tth = torch.from_numpy(th13).to(dev)
    tp, tpw = torch.from_numpy(p).to(dev), torch.from_numpy(pw).to(dev)
    n_sw = max(10, min(200, K))
    for k in range(3):
        engines[k % n_rep].gibbs_sweep_dev(C, tth.data_ptr(), 0, tp.data_ptr(), tpw.data_ptr(), states[k % n_rep][0],
                                           states[k % n_rep][1], 1, k, stream=side.cuda_stream)
    barrier()
    with torch.cuda.stream(side):
        e0.record()
        for k in range(n_sw):
            j = k % n_rep
            engines[j].gibbs_sweep_dev(C, tth.data_ptr(), 0, tp.data_ptr(), tpw.data_ptr(), states[j][0], states[j][1],
                                       1, 3 + k, stream=side.cuda_stream)
        e1.record()
    barrier()
    ms_gibbs = e0.elapsed_time(e1)
    # the other two update rules on the same states (ABD_GIBBS_HEATBATH, ABD_GIBBS_BLOCKED)
    ms_modes = {}
    for mode_name, mode_id in (("heatbath", 1), ("blocked", 2)):
        with torch.cuda.stream(side):
            engines[0].gibbs_sweep_dev(C, tth.data_ptr(), 0, tp.data_ptr(), tpw.data_ptr(), states[0][0], states[0][1], 1, 0,
                                       mode=mode_id, stream=side.cuda_stream)
            e0.record()
            for k in range(n_sw):
                j = k % n_rep
                engines[j].gibbs_sweep_dev(C, tth.data_ptr(), 0, tp.data_ptr(), tpw.data_ptr(), states[j][0], states[j][1],
                                           1, 500 + k, mode=mode_id, stream=side.cuda_stream)
            e1.record()
        barrier()
        ms_modes[mode_name] = e0.elapsed_time(e1)
        if dist:
            t = torch.tensor([ms_modes[mode_name]], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_modes[mode_name] = float(t.item())
    for e in engines:
        e.upload_state(i_raw, w)
    n_sw_e2e = max(5, min(50, K))
    t0 = time.perf_counter()
    for k in range(n_sw_e2e):
        engines[k % n_rep].gibbs_sweep(th13, p, pw, hi.numpy(), hw.numpy(), seed=1, sweep=k, inplace=True)
    dt_gibbs_e2e = time.perf_counter() - t0
    if dist:
        t = torch.tensor([ms_gibbs, dt_gibbs_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_gibbs, dt_gibbs_e2e = (float(v) for v in t.tolist())
    launches = sum(e.launch_count for e in engines) - launches0
    for e in engines[1:]:
        e.close()

    # ---- the PyMC-facing path (Op.perform / step protocol) driven through the protocol stand-in (tests/fake_pymc.py;
    #      PyMC is not installable offline): host cost per NUTS leapfrog and per Gibbs step at 10k individuals ----
    op_path = None
    try:
        sys.path.insert(0, str(ROOT / "tests"))
        import fake_pymc

        fabd = fake_pymc.load_abd_with_fake_pymc()
        from abdpymc_b200.engine import Q17 as _Q17, THETA13 as _TH13

        m = fabd.model(co, splits=SPLITS, device=local)
        node = m["loglik"].owner
        val_op, grad_op = node.op, fabd.AbdLogLikGrad(m.abd_engine, m.abd_cache)
        i64, w64 = i_raw[0].astype(np.int64), w[0].astype(np.int64)     # PyMC holds Bernoulli values as int64
        st_val, st_grad = [[None]], [[None] for _ in range(13)]

        def leapfrog_eval(theta13):
            inputs = [np.float64(v) for v in theta13] + [i64, w64]
            val_op.perform(node, inputs, st_val)
            grad_op.perform(None, inputs, st_grad)

        n_op = max(200, min(2000, K * 20))
        for k in range(20):
            leapfrog_eval(th13[0] * (1 + 1e-6 * k))
        t0 = time.perf_counter()
        for k in range(n_op):
            leapfrog_eval(th13[0] * (1 + 1e-6 * (k + 20)))
        dt_op = time.perf_counter() - t0
        step = fabd.GpuBinaryGibbs(model=m, seed=3)
        point = {**{name: np.float64(q[0][k]) for k, name in enumerate(_Q17)}, "i_raw": i64, "ab_s_waner": w64}
        point, _ = step.step(point)
        n_st = max(5, min(30, K))
        t0 = time.perf_counter()
        for _ in range(n_st):
            point, _ = step.step(point)
        dt_step = time.perf_counter() - t0
        op_path = {"us_per_leapfrog": dt_op / n_op * 1e6, "us_per_gibbs_step": dt_step / n_st * 1e6, "chains": 1,
                   "uploads_of_the_binaries": int(m.abd_cache.uploads),
                   "what": "AbdLogLik.perform + AbdLogLikGrad.perform at a new parameter point with unchanged binaries (one kernel "
                           "launch, 13 scalars in / 14 out; i_raw stays on the GPU between Gibbs steps), and "
                           "GpuBinaryGibbs.step (sweep on the resident state + download of the new int8 state + int64 conversion for "
                           "PyMC's point); driven through tests/fake_pymc.py, the stand-in for the PyMC 5 protocol"}
        m.abd_engine.close()
    except Exception as ex:  # never let the optional leg take the headline down
        op_path = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}

    # ---- individual sharding (BASELINE configs[3]): the 100k-individual cohort on ONE GPU (baseline, rank 0)
    #      and split over the ranks, C = 4 and C = 32 chains; NCCL all-reduce against the all-reduce fused into
    #      the kernel over NVLink peer memory, host-driven and as a CUDA graph ----
    sharded = None
    if not args.no_sharded:
        sharded = bench_sharded(dist, rank, world, local, dev, K)

    # ---- ESS/s of the built-in HMC + GPU-Gibbs sampler on the same cohort (bounded runs): the headline's 4 chains,
    #      and 128 chains per GPU (BASELINE configs[4]: 1024 chains over 8 GPUs, chain-parallel ESS/s) ----
    ess = ess128 = nuts = None
    if not args.no_ess:
        ess = bench_ess(eng0, co, C, dev, rank, world, dist, args.ess_tune, args.ess_draws, cpu)
        eng128 = AbdEngine(co, splits=SPLITS, device=local)
        ess128 = bench_ess(eng128, co, 128, dev, rank, world, dist, args.ess128_tune, args.ess128_draws, None)
        eng128.close()
        # what pm.sample runs for the 17 scalars is NUTS (abd.py:922): the device-resident No-U-Turn tree + the same sweep
        from abdpymc_b200.engine import forward as _fw
        from abdpymc_b200.sampler import AbdTarget as _T, SamplerConfig as _SC, sample as _sample

        x0 = np.array([1.0 / G, 2, 1, 10 / 11, -2, 2, 10 / 11, 0.5, 1, 1, -2, -1, 2, 1, -1, 2, 1], dtype=np.float64)
        q0n = _fw(x0)[None, :] + np.random.default_rng(11 + rank).uniform(-1, 1, size=(C, 17))
        eng0.set_chain_offset(rank * C)
        rn = _sample(_T(eng0, C, np.zeros((C, G, N), np.int8), np.zeros((C, N), np.int8), seed=2), torch.from_numpy(q0n).to(dev),
                     _SC(tune=600, draws=400, seed=2 + rank, kernel="nuts"))
        nuts = {"iterations_per_s": 1000 / rn.wall_s, "chains": C, "mean_tree_depth": float(rn.stats["tree_depth"].mean()),
                "mean_leapfrogs_per_iteration": rn.n_grad_evals / 1000 - 1, "diverging_fraction": float(rn.stats["diverging"].mean()),
                "mean_accept": float(rn.accept.mean()),
                # the 400 draws on their own (adapted step size and metric; the trees of early tuning are several times deeper)
                "draws_per_s_after_tuning": 400 / (rn.wall_s - rn.wall_tune_s),
                "mean_leapfrogs_per_draw": (rn.n_grad_evals - rn.n_grad_evals_tune) / 400 - 1,
                "what": "device No-U-Turn tree (abd_nuts_extend_dev: ONE launch per leaf for all chains -- the leapfrog step, and its "
                        "finishing warp folds the new state into the chain's tree --, one read-back per tree depth, none for the depths every recent tree reached) + Gibbs "
                        "sweep; 600 tune (deep trees early on) + 400 draws, rate over all 1000 iterations"}

    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak_gbs()
    ach = a_logp / t_kernel / 1e9
    flops = C * (60.0 * co.n_rows + 12.0 * G * N)
    t_sweep = ms_gibbs / 1e3 / n_sw
    ach_g = a_gibbs / t_sweep / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {
            "workload": workload_name(co, C),
            "step": f"{EVALS_PER_STEP} consecutive batched logp+grad evaluations (one CUDA graph replay)",
            "l2": f"inputs larger than L2: evaluations rotate over {n_rep} cohort+state replicas ({n_rep * a_logp / 1e6:.0f} MB > 2 x 126 MB L2)",
            "parallelism": "chains sharded across GPUs, cohort replicated, no collective" if world > 1 else "1 GPU",
        },
        "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                     "traffic": ncu_traffic("k_sums"), "traffic_source": TRAFFIC_SOURCE, "kernel": "k_sums",
                     "algorithmic_bytes_per_launch": a_logp,
                     "avg_launch_us": t_kernel * 1e6, "peak_source": peak_src,
                     "issue": ncu_issue("k_sums", t_kernel),
                     # the second, honest bound (SURVEY 8d): fp64 work, 60 R + 12 G N flop-equivalents per chain evaluation
                     "fp64": {"flops_per_launch": flops, "achieved_tflops": flops / t_kernel / 1e12,
                              "nominal_peak_tflops": 37.0, "frac_of_nominal": flops / t_kernel / 1e12 / 37.0,
                              "note": "the kernel is bound by fp64 issue / latency, not by HBM: ~1.4 algorithmic bytes "
                                      "per OD row against ~60 fp64-heavy instructions (DESIGN.md section 4)"}},
        "cpu_baseline": cpu,
        "e2e": {"value": world * C * n_e2e / dt_e2e, "unit": "evals/s",
                "h2d_bytes_per_step": int(C * (17 * 8 + G * N + N)), "d2h_bytes_per_step": int(C * 18 * 8),
                "call": "abd_logp_dlogp(q17, i_raw, waner) with pinned host buffers, one call per step (the library pulls pinned "
                        "chain state with an SM copy kernel over PCIe instead of the copy engine; q17 / results by cudaMemcpyAsync)"},
        "e2e_resident_state": {"value": world * C * n_e2e / dt_res, "unit": "evals/s",
                               "h2d_bytes_per_step": int(C * 17 * 8), "d2h_bytes_per_step": int(C * 18 * 8),
                               "call": "abd_logp_dlogp(q17, NULL, NULL): chain state left on the device by the Gibbs sweep"},
        "l2_resident": {"value": world * C * n_launch / (ms_l2 / 1e3), "unit": "evals/s",
                        "avg_launch_us": ms_l2 / n_launch * 1e3,
                        "note": "same cohort re-evaluated back to back (the access pattern of consecutive NUTS leapfrogs)"},
        "concurrent_streams": concurrent,
        "persistent_trajectory": traj,
        "batched_128_chains": batched,
        "deterministics": determ,
        "gibbs": {"metric": "Gibbs sweeps/s (all G*N+N binary variables of one chain)", "value": world * C * n_sw / (ms_gibbs / 1e3),
                  "unit": "sweeps/s", "avg_launch_us": t_sweep * 1e6,
                  "regime": "states drawn at random (4 % infections, 50 % waners): the burn-in regime, many accepted flips",
                  "other_update_rules": {name: {"value": world * C * n_sw / (v / 1e3), "unit": "sweeps/s"} for name, v in ms_modes.items()},
                  "roofline": {"bound": "hbm", "achieved": ach_g, "peak": peak, "unit": "GB/s", "frac": ach_g / peak,
                               "traffic": ncu_traffic("k_gibbs"), "traffic_source": TRAFFIC_SOURCE, "kernel": "k_gibbs",
                               "algorithmic_bytes_per_launch": a_gibbs, "issue": ncu_issue("k_gibbs", t_sweep),
                               "fp64": {"flops_per_launch": C * N * G * (4.0 * G + 60.0 * co.n_rows / N),
                                        "achieved_tflops": C * N * G * (4.0 * G + 60.0 * co.n_rows / N) / t_sweep / 1e12,
                                        "nominal_peak_tflops": 37.0,
                                        "note": "SURVEY 8d: N G (4 G + 60 R / N) fp64 flop-equivalents per chain sweep; the sweep is "
                                                "bound by instruction issue (sequential per-individual decisions), not HBM"}},
                  "e2e": {"value": world * C * n_sw_e2e / dt_gibbs_e2e, "unit": "sweeps/s",
                          "h2d_bytes_per_step": int(C * (G * N + N + 15 * 8)), "d2h_bytes_per_step": int(C * (G * N + N + 16))}},
        "pymc_op_path": op_path, "sharded_100k": sharded, "ess": ess, "ess_128_chains": ess128, "nuts": nuts,
        "gpu_launches": int(n_launch), "gpu_launches_host_api": int(launches), "clocks": clocks,
    }
    emit(line)
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ess", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the 100k-individual (individual-sharded) leg")
    ap.add_argument("--ess-tune", type=int, default=2000)
    ap.add_argument("--ess-draws", type=int, default=6000)
    ap.add_argument("--ess128-tune", type=int, default=2000)
    ap.add_argument("--ess128-draws", type=int, default=2000)
    ap.add_argument("--profile", action="store_true",
                    help="short run for ncu: a few un-captured logp+grad launches and Gibbs sweeps, no JSON line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's logp and gradient of every chain as DIR/logp.npy, DIR/dlogp.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.profile):
        ap.error("--dump-outputs needs the timed CUDA path (not --impl reference or --profile)")
    # Exactly ONE line goes to stdout (rank 0's JSON): libraries that chat on stdout (NCCL prints its
    # version there) are sent to stderr for the whole run.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


_REAL_STDOUT = None


def emit(line: dict) -> None:
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


if __name__ == "__main__":
    main()
