"""Multi-GPU sharding of INDEPENDENT fits (folds x traits x chains x seeds; SURVEY 8e, BASELINE config 4).

One process per GPU (torchrun / torch.distributed).  Systems are partitioned over ranks, every rank keeps the packed
genotypes (they are shared by all fits) and runs its share through the ordinary single-GPU entry points; there is NO
data-path collective -- only the host-side gather of the small result vectors at the end, which is what the reference's
caller does with `lapply` results (R/cv.R:80).  The single large fit (config 5) shards rows instead and needs a per-block
exchange inside the sweep kernel; see DESIGN.md section 6.  A row-sharded store (Genotypes.enable_row_sharding) takes the EM
and Gibbs fits and MRR3 / MRR3F (bw.MRR3(Y[rows], g)) on their fast path.
"""
import numpy as np


def partition(nsys, world):
    """Balanced contiguous split of nsys systems over `world` ranks: [(start, stop)] * world (empty ranges allowed)."""
    base, rem = divmod(int(nsys), int(world))
    out, s = [], 0
    for r in range(world):
        e = s + base + (1 if r < rem else 0)
        out.append((s, e))
        s = e
    return out


def _merge(parts, axis_keys):
    """Concatenate per-rank result dicts along the system axis (last axis of arrays, stacked scalars)."""
    parts = [p for p in parts if p is not None]
    out = {}
    for key in parts[0]:
        vals = [np.atleast_1d(np.asarray(p[key])) for p in parts]
        out[key] = np.concatenate(vals, axis=-1)
    return out


def fit_sharded(fit_fn, Y, row_mask=None, group=None, offset_kw=None, **kw):
    """Run `fit_fn(Y_cols, row_mask=mask_cols, **kw)` (e.g. functools.partial(bw.em_fit, "emBC", gen=store)) on this
    rank's share of the columns of Y (n x nsys) and gather every rank's result dict on all ranks.  Works on any
    torch.distributed backend (nccl on the GPU box, gloo in the CPU tests); without an initialised process group it
    degenerates to one rank.  offset_kw: name of a keyword that receives the index of the rank's first column, e.g. "chain0"
    with bw.gibbs_fit (one chain per column), so that the sharded systems draw the streams of the one-GPU fit."""
    import torch.distributed as dist
    Y = np.asarray(Y)
    nsys = Y.shape[1]
    if dist.is_available() and dist.is_initialized():
        rank, world = dist.get_rank(group), dist.get_world_size(group)
    else:
        rank, world = 0, 1
    s, e = partition(nsys, world)[rank]
    mine = None
    if e > s:
        m = None if row_mask is None else np.asarray(row_mask)[:, s:e]
        fkw = dict(kw) if offset_kw is None else dict(kw, **{offset_kw: s})
        res = fit_fn(Y[:, s:e], row_mask=m, **fkw) if row_mask is not None else fit_fn(Y[:, s:e], **fkw)
        mine = {k: np.asarray(v) for k, v in res.items()}
    if world == 1:
        return _merge([mine], None)
    gathered = [None] * world
    dist.all_gather_object(gathered, mine, group=group)  # host gather of O((n + p) * nsys) results, not on the data path
    return _merge(gathered, None)


def cv_tasks(nfolds, ntraits, world):
    """emCV-style work list (R/cv.R:13-22): one fit per (fold, trait), fold-major, split contiguously over the ranks so
    that a rank touches as few folds as possible (one row-subset genotype store per fold it works on).
    Returns, per rank, a list of (fold, [traits])."""
    tasks = [(f, t) for f in range(nfolds) for t in range(ntraits)]
    out = []
    for s, e in partition(len(tasks), world):
        groups = {}
        for f, t in tasks[s:e]:
            groups.setdefault(f, []).append(t)
        out.append(sorted(groups.items()))
    return out


def fit_cv_sharded(fit_fn, load_fn, Y, held_out, group=None, **kw):
    """k-fold x trait batch of fits sharded over the ranks, each fold fitted on its own ROW-SUBSET store -- literally what the
    reference's emCV does with gen[-w,] -- so that the fits of a fold run on the blocked whole-GPU kernel family (no row masks).

    load_fn(keep_rows) -> Genotypes store of the rows kept by a fold; fit_fn(Ycols, store, **kw) -> result dict (system axis
    last); Y: n x ntraits; held_out: list of row-index arrays, one per fold.  Every rank gets the dict of all (fold, trait)
    results, keys as fit_fn returns them, system axis ordered fold-major.  No data-path collective (host gather only)."""
    import torch.distributed as dist
    Y = np.asarray(Y)
    n, ntraits = Y.shape
    if dist.is_available() and dist.is_initialized():
        rank, world = dist.get_rank(group), dist.get_world_size(group)
    else:
        rank, world = 0, 1
    mine = []
    for f, traits in cv_tasks(len(held_out), ntraits, world)[rank]:
        keep = np.setdiff1d(np.arange(n), np.asarray(held_out[f]))
        store = load_fn(keep)
        try:
            res = fit_fn(Y[np.ix_(keep, traits)], store, **kw)
        finally:
            store.close()
        res = {k: np.asarray(v) for k, v in res.items() if np.asarray(v).ndim == 0 or np.asarray(v).shape[-1] == len(traits)
               and k != "hat"}
        mine.append(((f, traits), res))
    gathered = [mine]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, mine, group=group)
    parts = [res for per_rank in gathered for _, res in per_rank]
    return _merge(parts, None)
