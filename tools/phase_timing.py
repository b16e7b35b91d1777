#!/usr/bin/env python3
"""Developer tool: per-phase timeline of k_sums (needs the -DABD_PHASE_TIMING debug build)."""
import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
dbg = ROOT / "build" / "libabd_b200_dbg.so"
dbg.parent.mkdir(exist_ok=True)
import os
subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-DABD_PHASE_TIMING", *os.environ.get("ABD_EXTRA_FLAGS", "").split(), "-Xcompiler", "-fPIC",
                "-shared", "-o", str(dbg), str(ROOT / "abdpymc_b200/csrc/abd_b200.cu")], check=True)
from abdpymc_b200 import _lib  # noqa: E402

_lib.LIB_PATH = dbg
import bench  # noqa: E402
from abdpymc_b200.engine import AbdEngine  # noqa: E402

C_ = int(sys.argv[1]) if len(sys.argv) > 1 else 4
co, q, vals, i_raw, w = bench.workload(n_chains=C_)
eng = AbdEngine(co, splits=bench.SPLITS)
if len(sys.argv) > 2:
    eng.set_tuning(int(sys.argv[2]), 0)
eng.upload_state(i_raw, w)
di, dw = eng.state_dev(C_)
dev = torch.device("cuda:0")
tq = torch.from_numpy(q).to(dev)
out = torch.zeros(C_, dtype=torch.float64, device=dev)
outg = torch.zeros(C_, 17, dtype=torch.float64, device=dev)
lib = _lib.load()
L = int(sys.argv[3]) if len(sys.argv) > 3 else 0
if L:
    a = np.random.default_rng(0).normal(size=(17, 17))
    tm = torch.from_numpy(1e-6 * (a @ a.T / 17 + np.eye(17))).to(dev)
    te = torch.full((C_,), 1e-3, dtype=torch.float64, device=dev)
    eng.logp_dlogp_dev(C_, tq.data_ptr(), di, dw, out.data_ptr(), outg.data_ptr(), 0)
    torch.cuda.synchronize()
for rep in range(4):
    torch.cuda.synchronize()
    if L:
        qq, pp, gg = tq.clone(), torch.zeros_like(tq), outg.clone()
        eng.leapfrog_dev(C_, L, qq.data_ptr(), pp.data_ptr(), gg.data_ptr(), out.data_ptr(), te.data_ptr(), tm.data_ptr(), di, dw, 0)
    else:
        eng.logp_dlogp_dev(C_, tq.data_ptr(), di, dw, out.data_ptr(), outg.data_ptr(), 0)
    torch.cuda.synchronize()
n = 4096
buf = np.zeros((n, 16), np.uint64)
lib.abd_debug_phase_times.argtypes = [C.c_void_p, C.c_int]
lib.abd_debug_phase_times(buf.ctypes.data_as(C.c_void_p), n)
buf = buf[buf[:, 0] > 0].astype(np.int64)
t0 = buf[:, 0].min()
rel = (buf[:, :9] - t0) / 1e3
names = ["start", "staged+tab", "phase0 done", "tma arrived", "cells done", "rows done", "partial written", "ticket", "end"]
print(f"{len(buf)} CTAs (all chains); times in us relative to the first CTA start")
for k, nm in enumerate(names):
    col = rel[:, k]
    print(f"  {nm:16s} min {col.min():7.2f}  median {np.median(col):7.2f}  max {col.max():7.2f}")
per = len(buf) // C_
for c in range(C_):
    blk = rel[c * per:(c + 1) * per]
    print(f"  chain {c}: start median {np.median(blk[:, 0]):.2f}  phase0 done {np.median(blk[:, 2]):.2f}  rows done {np.median(blk[:, 5]):.2f}  end max {blk[:, 8].max():.2f}")
last = buf[buf[:, 11] > buf[:, 0]]
if len(last):
    r = (last[0, [7, 9, 10, 11, 8]] - t0) / 1e3
    print(f"  last CTA: ticket {r[0]:.2f}  partials read {r[1]:.2f}  totals {r[2]:.2f}  finalised {r[3]:.2f}  end {r[4]:.2f}")
for k, nm in ((12, "columns+constrain"), (13, "pow table (warp 4)"), (14, "params (warp 6)"), (15, "dilution table (warp 7)")):
    col = (buf[:, k] - buf[:, 1]) / 1e3
    print(f"  phase 0 detail, after the dependency wait: {nm:24s} median {np.median(col):6.2f}  max {col.max():6.2f}")
print("  durations (median): " + ", ".join(f"{names[k + 1]} {np.median(rel[:, k + 1] - rel[:, k]):.2f}" for k in range(8)))
