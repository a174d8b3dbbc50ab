"""Batched Gibbs systems and one-pass fitted values against their one-system-at-a-time counterparts, on one GPU, in one call.

  python tools/gibbs_batch_bench.py [--n 10000] [--p 50000] [--traits 20] [--folds 5] [--it 3] [--old-lib PATH] [--out FILE]

1. BayesB on `traits` x `folds` row-masked systems (BASELINE config 4's shape: 20 traits x 5 CV folds at 10k x 50k): one
   bwgr_gibbs_fit_sys call against the same systems fitted one after another by single-system calls on the same store.  Both run `it`
   sweeps (burn-in 1) instead of the reference's 1,500; the per-sweep time is scaled linearly to 1,500 sweeps, and the output says so.
2. Fitted values mu + X b of k = 1, 20, 100 systems: one bwgr_fitted_sys call against k calls of bwgr_fitted of the library at
   --old-lib (a build of the commit before bwgr_fitted_sys, whose bwgr_fitted is the one-system GEMV), run in a subprocess; hat is
   compared bit for bit.

Times are host clocks around calls that end in a stream synchronise (median of --reps after a warm-up).  The genotypes (n p bytes)
are larger than the 126 MB L2, so every pass reads them from HBM.  The card's name and power limit are printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    """name, power limit, max SM clock of GPU 0 (read-only query)."""
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    except OSError as ex:
        return "unknown (%s)" % ex
    return q.stdout.strip() if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def data(n, p, k, seed=4):
    rng = np.random.default_rng(seed)
    f = rng.uniform(0.05, 0.5, size=p).astype(np.float32)
    X = np.empty((n, p), dtype=np.int8, order="F")
    for j0 in range(0, p, 4096):  # column blocks: the float draws of the whole matrix would not fit a small host
        j1 = min(p, j0 + 4096)
        X[:, j0:j1] = (rng.random((n, j1 - j0), dtype=np.float32) < f[j0:j1]) + (rng.random((n, j1 - j0), dtype=np.float32) < f[j0:j1])
    Y = np.asfortranarray(rng.normal(size=(n, k)))
    return X, Y, rng


def timed(fn, reps):
    fn()  # warm-up: module load, buffers of this shape
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), r


def effects(p, k):
    """b (p x k) and mu (k) of the fitted-values timing, float32 values, the same in both arms."""
    rng = np.random.default_rng(99)
    return rng.normal(size=(p, k)).astype(np.float32).astype(np.float64), rng.normal(size=k).astype(np.float32).astype(np.float64)


def old_gemv(args):
    """Subprocess arm: k calls of bwgr_fitted of the library at --old-lib, through its C ABI alone (that build has none of the new
    entry points the Python binding declares); writes {k: seconds} and the hat of the largest k."""
    import ctypes as C
    lib = C.CDLL(args.old_lib)
    lib.bwgr_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.bwgr_destroy.argtypes = [C.c_void_p]
    lib.bwgr_geno_load_i8.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int]
    lib.bwgr_fitted.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
    X, _, _ = data(args.n, args.p, 1)
    B, mu = effects(args.p, max(args.ks))
    B = np.ascontiguousarray(B.T)  # one contiguous b per call
    h = C.c_void_p()
    assert lib.bwgr_create(0, C.byref(h)) == 0
    assert lib.bwgr_geno_load_i8(h, X.ctypes.data_as(C.c_void_p), args.n, args.p, args.n, 0) == 0
    hat = np.empty((max(args.ks), args.n))

    def run(k):
        for t in range(k):
            assert lib.bwgr_fitted(h, B[t].ctypes.data_as(C.c_void_p), float(mu[t]), hat[t].ctypes.data_as(C.c_void_p)) == 0
        return hat[:k].T.copy()

    res = {}
    for k in args.ks:
        res[str(k)], out = timed(lambda: run(k), args.reps)
    lib.bwgr_destroy(h)
    np.save(args.old_arm, out)
    with open(args.old_arm + ".json", "w") as fh:
        json.dump(res, fh)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10000)
    ap.add_argument("--p", type=int, default=50000)
    ap.add_argument("--traits", type=int, default=20)
    ap.add_argument("--folds", type=int, default=5)
    ap.add_argument("--it", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ks", type=int, nargs="+", default=[1, 20, 100])
    ap.add_argument("--old-lib", default=None, help="libbwgr_b200.so of the parent commit (one-system GEMV); omit to skip that arm")
    ap.add_argument("--old-arm", default=None, help=argparse.SUPPRESS)  # internal: run the old-GEMV arm, write here
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.old_arm:
        return old_gemv(args)
    import tempfile

    import bwgr_b200 as bw
    lines = {"card": card(), "shape": "n %d x p %d, int8 store" % (args.n, args.p)}
    k = args.traits * args.folds
    X, Y0, rng = data(args.n, args.p, args.traits)
    # trait t of fold f: column f * traits + t; fold f holds out a fifth of the rows (a random partition)
    Y = np.asfortranarray(np.tile(Y0, (1, args.folds)))
    fold = rng.permutation(args.n) % args.folds
    M = np.asfortranarray(np.repeat(np.stack([fold != f for f in range(args.folds)], axis=1), args.traits, axis=1))
    with bw.Genotypes(X) as g:
        kw = dict(it=args.it, bi=1, seed=11)
        t0 = time.perf_counter()
        batched = bw.gibbs_fit("BayesB", Y, g, row_mask=M, **kw)
        tb = time.perf_counter() - t0
        t0 = time.perf_counter()
        seq = [bw.gibbs_fit("BayesB", Y[:, s], g, row_mask=M[:, s:s + 1], chain0=s, **kw) for s in range(k)]
        ts = time.perf_counter() - t0
        same = all(np.array_equal(batched["b"][:, s], r["b"]) for s, r in enumerate(seq))
        lines["gibbs"] = {
            "what": "BayesB, %d traits x %d masked folds = %d systems; %d sweeps each, scaled linearly to 1500 sweeps" % (args.traits, args.folds, k, args.it),
            "batched_one_call_s": tb, "sequential_%d_calls_s" % k: ts,
            "batched_s_per_1500_sweeps": tb / args.it * 1500, "sequential_s_per_1500_sweeps": ts / args.it * 1500,
            "speedup": ts / tb, "posterior_means_bit_identical": bool(same)}
        # fitted values
        B, mu = effects(args.p, max(args.ks))
        fv = {}
        hat_new = None
        for kk in args.ks:
            sec, hat_new = timed(lambda: g.fitted(B[:, :kk], mu[:kk]), args.reps)
            fv[str(kk)] = {"one_pass_ms": sec * 1e3}
    if args.old_lib:
        with tempfile.TemporaryDirectory() as td:
            arm = os.path.join(td, "old")
            cmd = [sys.executable, os.path.abspath(__file__), "--old-arm", arm, "--old-lib", os.path.abspath(args.old_lib), "--n", str(args.n), "--p", str(args.p), "--reps", str(args.reps),
                   "--ks"] + [str(v) for v in args.ks]
            subprocess.run(cmd, check=True)
            old = json.load(open(arm + ".json"))
            hat_old = np.load(arm + ".npy")
        for kk in args.ks:
            fv[str(kk)]["per_system_gemv_ms"] = old[str(kk)] * 1e3
            fv[str(kk)]["speedup"] = old[str(kk)] / (fv[str(kk)]["one_pass_ms"] * 1e-3)
        fv["hat_bit_identical_to_parent_k%d" % max(args.ks)] = bool(np.array_equal(hat_old, hat_new))
    lines["fitted_values"] = fv
    txt = json.dumps(lines, indent=1)
    print(txt)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
