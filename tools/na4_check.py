"""Blocked family beyond three 128-row atoms per worker (n = 52k-70k, NA = 4): parity against the oracle."""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "tests"))
import bwgr_b200 as bw, oracle as O
from conftest import synth
for n in (52000, 60000, 70000):
    X, y = synth(n, 700, seed=2)
    ref = O.em("emRR", y, X.astype(np.float32), it=4)
    try:
        with bw.Genotypes(X, path=2) as g:
            out = bw.emRR(y, g, it=4)
        print(n, "err", np.abs(out["b"] - ref["b"]).max() / np.abs(ref["b"]).max(), out["h2"], ref["h2"], flush=True)
    except Exception as e:
        print(n, "FAILED", str(e)[:100], flush=True)
