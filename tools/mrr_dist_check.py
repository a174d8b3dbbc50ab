#!/usr/bin/env python
"""Row-sharded MRR3 / MRR3F over the ranks of one node against the single-GPU fit of the same data (run under torchrun).

  torchrun --nproc-per-node N tools/mrr_dist_check.py
      parity checks; rank 0 prints MRR DIST CHECK OK / FAILED (exit status 0 / 1)
  torchrun --nproc-per-node N tools/mrr_dist_check.py --time n p k [--sweeps S] [--general]
      ms per MRR3 iteration at n x p with k traits, rows split evenly over the ranks; one JSON line on rank 0.  With one process the
      store is not sharded; --general forces the general path (BWGR_MRR=general, one process only).  The genotypes are made on the
      GPU in eight seeded row chunks, so every world size fits the same data.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import bwgr_b200 as bw  # noqa: E402

UNSUPPORTED = -5
KEYS = ("b", "h2", "GC", "vb", "ve", "mu", "MSx")


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def same_on_all_ranks(x):
    """True on every rank iff x is bit-identical to rank 0's x (broadcast and compare)."""
    t = torch.tensor(np.ascontiguousarray(x), device="cuda")
    t0 = t.clone()
    dist.broadcast(t0, src=0)
    flag = torch.tensor([0 if bool((t == t0).all().item()) else 1], device="cuda")
    dist.all_reduce(flag)
    return flag.item() == 0


def mrr_traits(X, k, seed):
    """k correlated traits with 5 % of the markers causal (the shape mrr(Y, gen) is used on)."""
    rng = np.random.default_rng(seed)
    p = X.shape[1]
    Lc = np.linalg.cholesky(0.5 * np.ones((k, k)) + 0.5 * np.eye(k))
    B = (rng.normal(size=(p, k)) @ Lc.T) * (rng.random((p, 1)) < 0.05)
    G = X.astype(np.float64) @ B
    return np.asfortranarray(G / G.std(0) + rng.normal(size=G.shape))


def check(rank, world, local):
    import oracle as O
    from conftest import synth
    ok = True

    def report(name, good, text):
        """good: rank 0's verdict (text is rank 0's); every rank records it"""
        nonlocal ok
        flag = torch.tensor([0 if good else 1], device="cuda")
        dist.broadcast(flag, src=0)
        ok = ok and flag.item() == 0
        if rank == 0:
            print("%-38s %s  %s" % (name, "ok  " if flag.item() == 0 else "FAIL", text), flush=True)

    n, p = 4096, 1500
    X, y = synth(n, p, seed=5)
    rows = np.array_split(np.arange(n), world)[rank]
    g = bw.Genotypes(device=local, path=bw.PATH_BLOCKED).enable_row_sharding()
    g.load(np.ascontiguousarray(X[rows]))
    g1 = bw.Genotypes(X, device=local, path=bw.PATH_BLOCKED) if rank == 0 else None

    def against_one_gpu(name, fit, Y, kw, store, store1, Xo=None, oracle_tol=None):
        """the sharded fit against the one-GPU fit of the same global data (1e-5 relative, the same Its) and, optionally, the oracle"""
        out = fit(np.ascontiguousarray(Y[rows]), store, **kw)
        same = same_on_all_ranks(out["b"])
        good, text = same, "b identical on every rank: %s" % same
        if rank == 0:
            ref = fit(Y, store1, **kw)
            errs = {key: rel(out[key], ref[key]) for key in KEYS}
            errs["hat"] = rel(out["hat"], ref["hat"][rows])
            worst = max(errs, key=errs.get)
            good = good and errs[worst] <= 1e-5 and out["Its"] == ref["Its"]
            text = "vs 1 GPU: max rel %.1e (%s), Its %d/%d; %s" % (errs[worst], worst, out["Its"], ref["Its"], text)
            if oracle_tol is not None:
                o = O.mrr3(Y, Xo.astype(np.float64), f32_variant=fit is bw.MRR3F, **kw)
                eo = max(rel(out["b"], o["b"]), rel(out["hat"], o["hat"][rows]), rel(out["h2"], o["h2"]))
                good = good and eo <= oracle_tol
                text += "; vs oracle %.1e" % eo
        report(name, good, text)
        return out

    # 1. k = 4 after 1, 3 and 12 sweeps; 2. k = 20 (config 3's trait count)
    Y4 = mrr_traits(X, 4, 11)
    for its in (1, 3, 12):
        against_one_gpu("MRR3 k=4 maxit=%d" % its, bw.MRR3, Y4, dict(maxit=its), g, g1, X, oracle_tol=2e-4)
    against_one_gpu("MRR3 k=20 maxit=3", bw.MRR3, mrr_traits(X, 20, 12), dict(maxit=3), g, g1)
    # 3. to convergence at the default tol: the same Its on every rank and on one GPU
    out = against_one_gpu("MRR3 k=4 to convergence", bw.MRR3, Y4, {}, g, g1)
    its = same_on_all_ranks(np.array([out["Its"]]))
    report("Its equal on every rank", its, "Its %d" % out["Its"])
    # 4. options that change the host's variance block, the mean, or the system
    for name, kw in (("updateMu", dict(updateMu=True)), ("HCS", dict(HCS=True)), ("OneVarB", dict(OneVarB=True))):
        against_one_gpu("MRR3 %s maxit=4" % name, bw.MRR3, Y4, dict(kw, maxit=4), g, g1)
    against_one_gpu("MRR3F maxit=4", bw.MRR3F, Y4, dict(maxit=4), g, g1)

    # 5. CNT(gen) through the centred loader; rank 0 holds none of the rows with the smallest code of column j
    j = int(np.argmin((X == X.min(axis=0)).sum(axis=0)))
    order = np.argsort(X[:, j] == X[:, j].min(), kind="stable")
    Xo, Yo = X[order], Y4[order]
    Xc = O.cnt(Xo.astype(np.float64)).astype(np.float64)
    gc = bw.Genotypes(device=local, path=bw.PATH_BLOCKED).enable_row_sharding()
    gc.load(np.ascontiguousarray(Xc[rows]), centred_ok=True)
    codes = np.array_equal(gc.unpack(), Xo[rows] - Xo.min(axis=0))
    lacking = int((Xo[np.array_split(np.arange(n), world)[0]].min(axis=0) > Xo.min(axis=0)).sum())
    report("centred loader: common constants", same_on_all_ranks(np.array([int(codes)])) and codes,
           "rank 0 lacks the smallest code of %d columns" % lacking)
    gc1 = bw.Genotypes(Xc, device=local, path=bw.PATH_BLOCKED, centred_ok=True) if rank == 0 else None
    against_one_gpu("mrr(Y, CNT(gen)) maxit=6", bw.MRR3, Yo, dict(maxit=6), gc, gc1)
    gc.close()
    if gc1 is not None:
        gc1.close()

    # 6. several systems through the sharded sweep: emRR on 4 traits (separates sweep-kernel faults from the MRR3 host driver)
    out = bw.em_fit("emRR", Y4[rows], g, it=10)
    good = same_on_all_ranks(out["b"])
    text = ""
    if rank == 0:
        ref = bw.em_fit("emRR", Y4, g1, it=10)
        e = max(rel(out["b"], ref["b"]), rel(out["hat"], ref["hat"][rows]))
        good, text = good and e <= 1e-4, "vs 1 GPU: max rel %.1e" % e
    report("emRR nsys=4", good, text)

    # 8. refusals taken together (the subprocess timeout of the test is the guard against a hang), then the same handles fit again
    Yn = Y4.copy()
    if rank == 1:
        Yn[rows[0], 0] = np.nan
    for name, Yr, kw in (("NaN in Y on rank 1 only", Yn, {}), ("InnerGS", Y4, dict(InnerGS=True))):
        try:
            bw.MRR3(np.ascontiguousarray(Yr[rows]), g, maxit=3, **kw)
            code, msg = 0, ""
        except bw.BwgrError as err:
            code, msg = err.code, str(err)
        flag = torch.tensor([0 if code == UNSUPPORTED and "row-sharded" in msg else 1], device="cuda")
        dist.all_reduce(flag)
        report("refused on every rank: " + name, flag.item() == 0, msg[:100])
    out = bw.em_fit("emRR", y[rows], g, it=10)
    good = same_on_all_ranks(out["b"])
    text = ""
    if rank == 0:
        ref = bw.em_fit("emRR", y, g1, it=10)
        e = max(rel(out["b"], ref["b"]), rel(out["hat"], ref["hat"][rows]))
        good, text = good and e <= 1e-4, "vs 1 GPU: max rel %.1e" % e
    report("emRR after the refusals", good, text)
    g.close()
    if g1 is not None:
        g1.close()
    return ok


def make_rows(n, p, k, chunks, device):
    """Row chunks `chunks` of the eight seeded chunks of an n x p genotype matrix (codes 0..2, column-major as a (p, rows) int8
    tensor) and of its k traits (rows x k, host)."""
    f = torch.tensor(np.random.default_rng(7).uniform(0.05, 0.5, size=p), dtype=torch.float32, device=device)[:, None]
    beta = torch.tensor(np.random.default_rng(8).normal(size=(p, k)) * (np.random.default_rng(9).random((p, 1)) < 0.01),
                        dtype=torch.float32, device=device)
    scale = 1.0 / np.sqrt(max(1.0, float((beta[:, 0] != 0).sum().item())) * 0.4)
    nc = n // 8
    xs, ys = [], []
    for c in chunks:
        gen = torch.Generator(device=device).manual_seed(1000 + c)
        Xc = ((torch.rand((p, nc), generator=gen, device=device) < f).to(torch.int8)
              + (torch.rand((p, nc), generator=gen, device=device) < f).to(torch.int8))
        G = Xc.t().float() @ beta
        ys.append((G * scale + torch.randn((nc, k), generator=gen, device=device)).double().cpu().numpy())
        xs.append(Xc)
    X = torch.cat(xs, dim=1).contiguous() if len(xs) > 1 else xs[0]
    return X, np.asfortranarray(np.concatenate(ys, axis=0))


def timing(rank, world, local, n, p, k, sweeps, general):
    assert n % 8 == 0 and 8 % world == 0, "n must split into 8 chunks and world must divide 8"
    if general:
        assert world == 1, "--general times the one-GPU general path"
        os.environ["BWGR_MRR"] = "general"
    per = 8 // world
    X, Y = make_rows(n, p, k, range(rank * per, (rank + 1) * per), torch.device("cuda", local))
    g = bw.Genotypes(device=local, path=bw.PATH_BLOCKED if world > 1 else bw.PATH_AUTO)
    if world > 1:
        g.enable_row_sharding()
    g.load(X)
    del X
    torch.cuda.empty_cache()

    def run(maxit):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        out = bw.MRR3(Y, g, maxit=maxit, tol=1e-30)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return time.perf_counter() - t0, out["Its"]

    line = {"tool": "mrr_dist_check", "n": n, "p": p, "k": k, "gpus": world, "rows_per_gpu": n // world,
            "path": "general" if general else "fast"}
    try:
        run(1)  # warm-up: module loads, workspace
        t1, i1 = run(1)
        t2, i2 = run(1 + sweeps)
        line.update(sweeps_timed=i2 - i1, ms_per_iteration=round(1e3 * (t2 - t1) / (i2 - i1), 3), fit_s_at_1_sweep=round(t1, 3))
    except bw.BwgrError as err:  # a shape no path takes is a result too
        line["error"] = str(err)
    g.close()
    if rank == 0:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                           capture_output=True, text=True)
        line["gpu"] = q.stdout.strip()
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--time", nargs=3, type=int, metavar=("N", "P", "K"))
    ap.add_argument("--sweeps", type=int, default=10)
    ap.add_argument("--general", action="store_true")
    a = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if a.time:
        timing(rank, world, local, *a.time, a.sweeps, a.general)
        ok = True
    else:
        assert world > 1, "the parity checks need two or more processes"
        ok = check(rank, world, local)
    if world > 1:
        flag = torch.tensor([0 if ok else 1], device="cuda")
        dist.all_reduce(flag)
        ok = flag.item() == 0
        dist.destroy_process_group()
    if rank == 0 and not a.time:
        print("MRR DIST CHECK", "OK" if ok else "FAILED", flush=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
