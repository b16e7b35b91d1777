#!/usr/bin/env python3
"""Developer tool (run on the GPU box): build variants of libabd_b200.so with extra nvcc flags and time the
three hot launches with each: logp+grad at 4 chains (same cohort re-evaluated back to back, CUDA graph),
logp+grad at 128 chains, one Gibbs sweep of 4 chains -- 10k-individual benchmark cohort.

    python tools/variants.py base= minb4="-DABD_SUMS_MINB=4" ...
    python tools/variants.py --probe            (internal: measure the library named by ABD_B200_LIB)
"""
import json
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def probe():
    import numpy as np
    import torch

    import bench
    from abdpymc_b200.engine import AbdEngine

    dev = torch.device("cuda:0")
    out = {}
    side = torch.cuda.Stream()

    def graph_time(fn, n_inner, reps):
        with torch.cuda.stream(side):
            fn(side.cuda_stream)
        side.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for _ in range(n_inner):
                fn(side.cuda_stream)
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        best = 1e30
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                g.replay()
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / (reps * n_inner) * 1e3)
        return best

    for C, n_inner, reps in ((4, 128, 10), (128, 4, 5)):
        co, q, vals, i_raw, w = bench.workload(n_chains=C)
        eng = AbdEngine(co, splits=bench.SPLITS)
        eng.upload_state(i_raw, w)
        di, dw = eng.state_dev(C)
        tq = torch.from_numpy(q).to(dev)
        o1 = torch.zeros(C, dtype=torch.float64, device=dev)
        o2 = torch.zeros(C, 17, dtype=torch.float64, device=dev)
        out[f"logp_us_C{C}"] = graph_time(lambda st: eng.logp_dlogp_dev(C, tq.data_ptr(), di, dw, o1.data_ptr(), o2.data_ptr(), st),
                                          n_inner, reps)
        torch.cuda.synchronize()
        out[f"logp_sum_C{C}"] = float(o1.sum().item())
        if C == 4:
            th = torch.from_numpy(vals[:, [1, 2, 3, 4, 5, 6, 10, 11, 12, 13, 14, 15, 16]].copy()).to(dev)
            tp, tpw = torch.from_numpy(vals[:, 0].copy()).to(dev), torch.from_numpy(vals[:, 7].copy()).to(dev)
            for mode, name in ((0, "gibbs_us_C4"), (2, "gibbs_blk_us_C4")):
                eng.upload_state(i_raw, w)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                with torch.cuda.stream(side):
                    for k in range(3):
                        eng.gibbs_sweep_dev(C, th.data_ptr(), 0, tp.data_ptr(), tpw.data_ptr(), di, dw, 1, k, mode=mode,
                                            stream=side.cuda_stream)
                    side.synchronize()
                    eng.upload_state(i_raw, w)
                    e0.record()
                    for k in range(20):
                        eng.gibbs_sweep_dev(C, th.data_ptr(), 0, tp.data_ptr(), tpw.data_ptr(), di, dw, 1, 3 + k, mode=mode,
                                            stream=side.cuda_stream)
                    e1.record()
                side.synchronize()
                out[name] = e0.elapsed_time(e1) / 20 * 1e3
                # the same sweep once the states have settled under these parameters (few accepted flips: what a sampler sees)
                with torch.cuda.stream(side):
                    for k in range(60):
                        eng.gibbs_sweep_dev(C, th.data_ptr(), 0, tp.data_ptr(), tpw.data_ptr(), di, dw, 1, 23 + k, mode=mode,
                                            stream=side.cuda_stream)
                    e0.record()
                    for k in range(20):
                        eng.gibbs_sweep_dev(C, th.data_ptr(), 0, tp.data_ptr(), tpw.data_ptr(), di, dw, 1, 83 + k, mode=mode,
                                            stream=side.cuda_stream)
                    e1.record()
                side.synchronize()
                out[name.replace("_us_", "_settled_us_")] = e0.elapsed_time(e1) / 20 * 1e3
                si, sw = eng.download_state(C)
                out[name.replace("_us_", "_state_")] = int(si.sum()) * 1000003 + int(sw.sum())
        eng.close()
    print("PROBE " + json.dumps(out))


def main():
    if "--probe" in sys.argv:
        return probe()
    variants = [a.split("=", 1) for a in sys.argv[1:]]
    outdir = ROOT / "build" / "variants"
    outdir.mkdir(parents=True, exist_ok=True)

    def build(nv):
        name, flags = nv
        so = outdir / f"libabd_{name}.so"
        cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", *flags.split(),
               "-Xcompiler", "-fPIC", "-shared", "-o", str(so), str(ROOT / "abdpymc_b200/csrc/abd_b200.cu")]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return name, so, r.returncode, r.stderr[-500:]

    with ThreadPoolExecutor(8) as ex:
        built = list(ex.map(build, variants))
    rows = []
    for name, so, rc, err in built:
        if rc:
            print(f"{name}: build failed: {err}")
            continue
        env = dict(os.environ, ABD_B200_LIB=str(so))
        r = subprocess.run([sys.executable, __file__, "--probe"], capture_output=True, text=True, env=env)
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("PROBE ")]
        if not line:
            print(f"{name}: probe failed: {r.stderr[-800:]}")
            continue
        d = json.loads(line[0][6:])
        rows.append((name, d))
        print(f"{name:>16}: " + "  ".join(f"{k}={v:.2f}" if isinstance(v, float) and "us" in k else f"{k}={v}" for k, v in d.items()),
              flush=True)
    (outdir / "results.json").write_text(json.dumps(rows, indent=1))


if __name__ == "__main__":
    main()
