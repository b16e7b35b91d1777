#!/usr/bin/env python3
"""Developer tool: kernel spans (first CTA start .. last CTA end) and the gaps between consecutive
k_sums launches inside a CUDA graph (needs the -DABD_PHASE_TIMING debug build)."""
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
dbg = ROOT / "build" / "libabd_b200_dbg.so"
dbg.parent.mkdir(exist_ok=True)
subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-DABD_PHASE_TIMING", "-Xcompiler", "-fPIC",
                "-shared", "-o", str(dbg), str(ROOT / "abdpymc_b200/csrc/abd_b200.cu")], check=True)
os.environ["ABD_B200_LIB"] = str(dbg)
from abdpymc_b200 import _lib  # noqa: E402

_lib.LIB_PATH = dbg
import bench  # noqa: E402
from abdpymc_b200.engine import AbdEngine  # noqa: E402

C_ = int(sys.argv[1]) if len(sys.argv) > 1 else 4
co, q, vals, i_raw, w = bench.workload(n_chains=C_)
eng = AbdEngine(co, splits=bench.SPLITS)
eng.upload_state(i_raw, w)
di, dw = eng.state_dev(C_)
dev = torch.device("cuda:0")
tq = torch.from_numpy(q).to(dev)
out = torch.zeros(C_, dtype=torch.float64, device=dev)
outg = torch.zeros(C_, 17, dtype=torch.float64, device=dev)
lib = _lib.load()
lib.abd_debug_spans.argtypes = [C.c_void_p, C.c_int]
side = torch.cuda.Stream()
with torch.cuda.stream(side):
    eng.logp_dlogp_dev(C_, tq.data_ptr(), di, dw, out.data_ptr(), outg.data_ptr(), side.cuda_stream)
side.synchronize()
g = torch.cuda.CUDAGraph()
n = 32
with torch.cuda.graph(g, stream=side):
    for _ in range(n):
        eng.logp_dlogp_dev(C_, tq.data_ptr(), di, dw, out.data_ptr(), outg.data_ptr(), side.cuda_stream)
for _ in range(3):
    g.replay()
torch.cuda.synchronize()
lib.abd_debug_spans(None, 1)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
g.replay()
e1.record()
torch.cuda.synchronize()
buf = np.zeros((256, 2), np.uint64)
lib.abd_debug_spans(buf.ctypes.data_as(C.c_void_p), 0)
s = buf[:n].astype(np.int64)
span = (s[:, 1] - s[:, 0]) / 1e3
gap = (s[1:, 0] - s[:-1, 1]) / 1e3
print(f"C={C_}: graph of {n} launches {e0.elapsed_time(e1) * 1e3 / n:.2f} us/launch; "
      f"kernel span median {np.median(span):.2f} (min {span.min():.2f}, max {span.max():.2f}); gap start-after-end median {np.median(gap):.2f} "
      f"(min {gap.min():.2f}, max {gap.max():.2f})")
