"""Grid family (csrc/grid_sweep.cu) at a chosen shape: emRR sweeps on synthetic genotypes, ms per sweep-kernel launch from the library's CUDA events
(bwgr_profile; EmStepper keeps everything resident).  usage: python tools/grid_probe.py n p [EM model] [nsweeps]"""
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bwgr_b200 as bw  # noqa: E402

n, p = int(sys.argv[1]), int(sys.argv[2])
model = sys.argv[3] if len(sys.argv) > 3 else "emRR"
ns = int(sys.argv[4]) if len(sys.argv) > 4 else 5
gen = torch.Generator(device="cuda").manual_seed(1)
X = torch.randint(0, 3, (p, n), generator=gen, device="cuda", dtype=torch.int8)
y = np.random.default_rng(3).normal(size=n)
torch.cuda.synchronize()
for path in ((bw.PATH_GRID,) if os.environ.get("GRID_ONLY") else (bw.PATH_GRID, bw.PATH_AUTO)):
    try:
        with bw.Genotypes(device=0, path=path) as g:
            g.load(X)
            st = bw.EmStepper(model, y, g)
            st.sweeps(2)
            g.profile(True)
            st.sweeps(ns)
            pr = g.profile_read()
            g.profile(False)
            st.end()
            print("path %d: %s n=%d p=%d: sweep kernel %.3f ms per launch (%d launches), epilogue %.3f ms" % (
                path, model, n, p, pr["sweep"]["ms"] / max(1, pr["sweep"]["launches"]), pr["sweep"]["launches"],
                pr["epilogue"]["ms"] / max(1, pr["epilogue"]["launches"])), flush=True)
    except bw.BwgrError as e:
        print("path %d: %s" % (path, e))
