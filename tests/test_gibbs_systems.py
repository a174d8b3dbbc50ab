"""Several traits / CV folds of a Gibbs sampler in one call (bwgr_gibbs_fit_sys), and the fitted values of k systems in one pass over
the genotype store (bwgr_fitted_sys).

System s = t * nchains + c of a fit fits column t of Y and draws from Philox chain chain0 + s.  The draws are addressed by (sweep,
marker, chain), not by row, so a row-masked system is the sampler on the rows its mask keeps under the same chain index: each
system is checked against the oracle's replay of that physical subset (O.gibbs(..., draws="philox", chain=chain0 + s)) with the bar
and the no-near-tie conditions of test_gibbs_replay.py.  The seeds below pass those conditions for every system of their case
(test_replay_seeds_have_no_near_ties checks that on the CPU)."""
import ctypes as C
import os
import re
from unittest import mock

import numpy as np
import pytest

import oracle as O
from conftest import ROOT, synth
from test_gibbs_replay import _close, _gibbs_keys, _margins_ok

IT, BI = 10, 4
CHAIN0 = 5
NCOL, NCHAIN = 3, 2
# per model: seed of the masked replay case (3 columns x 2 chains) and of the unmasked several-trait case
MASKED_SEEDS = {"BayesRR": 1, "BayesA": 1, "BayesB": 2, "BayesC": 1, "BayesL": 1, "BayesCpi": 1, "BayesDpi": 9}
TRAIT_SEEDS = {"BayesRR": 2, "BayesA": 2, "BayesB": 8, "BayesC": 2, "BayesL": 2, "BayesCpi": 2, "BayesDpi": 6}


def _columns(tpod, masked):
    """Three phenotype columns on tpod's genotypes (tpod's y plus noise) and, for the masked case, three row masks keeping ~80 %."""
    y, gen = tpod
    rng = np.random.default_rng(77)
    n = y.size
    Y = np.asfortranarray(np.stack([y] + [y + 0.5 * rng.normal(size=n) for _ in range(NCOL - 1)], axis=1))
    M = np.asfortranarray(rng.random((n, NCOL)) < 0.8) if masked else None
    return Y, M, gen


def _replays(model, Y, M, X, seed, nchain, chain0):
    """(r32, r64) of every system: column t on the rows of its mask under chain chain0 + t * nchain + c."""
    out = []
    for t in range(Y.shape[1]):
        rows = np.ones(Y.shape[0], dtype=bool) if M is None else M[:, t]
        for c in range(nchain):
            kw = dict(it=IT, bi=BI, seed=seed, draws="philox", chain=chain0 + t * nchain + c)
            out.append((O.gibbs(model, Y[rows, t], X[rows], **kw), O.gibbs(model, Y[rows, t], X[rows], use_double=True, **kw)))
    return out


def _system(out, s):
    return {k: (v[:, s] if np.ndim(v) == 2 else v[s]) for k, v in out.items() if k != "PVAL" and np.ndim(v) >= 1}


# ---- CPU ----------------------------------------------------------------------------------------------------------------------

def test_entry_points_declared_and_exported():
    """bwgr_gibbs_fit_sys and bwgr_fitted_sys are declared in the header, listed by the binding and exported by the library."""
    from bwgr_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        from bwgr_b200 import build
        build.build()
    hdr = open(os.path.join(ROOT, "include", "bwgr_b200.h")).read()
    declared = set(re.findall(r"BWGR_API [\w\s\*]*?\b(bwgr_\w+)\(", hdr))
    cdll = _lib.load()
    for name in ("bwgr_gibbs_fit_sys", "bwgr_fitted_sys"):
        assert name in declared and name in _lib.SYMBOLS
        assert getattr(cdll, name) is not None
    # the ctypes mirror of bwgr_gibbs_sys_params has the header's fields in the header's order
    body = hdr.partition("} bwgr_gibbs_sys_params;")[0].rpartition("typedef struct {")[2]
    fields = re.findall(r"\b(\w+);", re.sub(r"/\*.*?\*/", "", body, flags=re.S))
    assert fields == [f for f, _ in _lib.GibbsSysParams._fields_]


def test_fit_sharded_offset_kw():
    """fit_sharded(offset_kw=...) hands every rank the index of its first column under that keyword; without it nothing is added."""
    from bwgr_b200 import dist as D
    import torch.distributed as tdist
    Y = np.zeros((4, 6))
    seen = []

    def fit(Yc, **kw):
        seen.append(kw)
        return {"b": np.zeros((2, Yc.shape[1]))}

    D.fit_sharded(fit, Y)
    D.fit_sharded(fit, Y, offset_kw="chain0")
    assert seen == [{}, {"chain0": 0}]
    seen.clear()
    with mock.patch.object(tdist, "is_available", return_value=True), mock.patch.object(tdist, "is_initialized", return_value=True), \
            mock.patch.object(tdist, "get_rank", return_value=1), mock.patch.object(tdist, "get_world_size", return_value=2), \
            mock.patch.object(tdist, "all_gather_object", side_effect=lambda out, obj, group=None: out.__setitem__(slice(None), [obj, obj])):
        res = D.fit_sharded(fit, Y, offset_kw="chain0")
    assert seen == [{"chain0": 3}] and res["b"].shape == (2, 6)


def test_replay_seeds_have_no_near_ties(tpod):
    """Every system of the GPU replay cases below is free of near-ties at its seed (the oracle alone decides this)."""
    X = tpod[1].astype(np.float64)
    for masked, seeds in ((True, MASKED_SEEDS), (False, TRAIT_SEEDS)):
        Y, M, _ = _columns(tpod, masked)
        for model, seed in seeds.items():
            for s, (r32, r64) in enumerate(_replays(model, Y, M, X, seed, NCHAIN, CHAIN0)):
                _margins_ok(r32, r64, "%s masked=%s system %d" % (model, masked, s))


# ---- GPU ----------------------------------------------------------------------------------------------------------------------

STORES = [(1, "int8"), (1, "2bit"), (3, "int8")]


@pytest.mark.gpu
@pytest.mark.parametrize("path,store", STORES, ids=["small_n-int8", "small_n-2bit", "grid-int8"])
@pytest.mark.parametrize("model", list(O.GIBBS_MODELS))
def test_masked_systems_replay(tpod, model, path, store):
    """3 masked columns x 2 chains, chain0 = 5, on the small-n and grid families: system s replays O.gibbs on the rows of its mask
    under chain 5 + s; hat of every row (the held-out ones included) is mu + X b of that system."""
    bw = pytest.importorskip("bwgr_b200")
    Y, M, gen = _columns(tpod, True)
    X = gen.astype(np.float64)
    seed = MASKED_SEEDS[model]
    storage = bw.STORE_2BIT if store == "2bit" else bw.STORE_I8
    with bw.Genotypes(gen, storage=storage, path=path) as g:
        out = bw.gibbs_fit(model, Y, g, it=IT, bi=BI, seed=seed, nchains=NCHAIN, row_mask=M, chain0=CHAIN0)
    assert out["b"].shape == (X.shape[1], NCOL * NCHAIN) and out["hat"].shape == (X.shape[0], NCOL * NCHAIN)
    keys = [k for k in _gibbs_keys(model) if k != "hat"]
    for s, (r32, r64) in enumerate(_replays(model, Y, M, X, seed, NCHAIN, CHAIN0)):
        case = "masked %s path %d %s system %d" % (model, path, store, s)
        _margins_ok(r32, r64, case)
        one = _system(out, s)
        _close(one, r32, r64, keys, case, exact=("d",))
        ref = one["mu"] + X @ one["b"]
        held = ~M[:, s // NCHAIN]
        assert held.any()
        np.testing.assert_allclose(one["hat"][held], ref[held], rtol=0, atol=1e-5 * np.abs(ref).max())
        np.testing.assert_allclose(one["hat"], ref, rtol=0, atol=1e-5 * np.abs(ref).max())


@pytest.mark.gpu
@pytest.mark.parametrize("model", list(O.GIBBS_MODELS))
def test_several_traits_blocked_replay(tpod, model):
    """3 unmasked columns x 2 chains on the blocked family: every system replays as its own chain (chain0 = 5)."""
    bw = pytest.importorskip("bwgr_b200")
    Y, _, gen = _columns(tpod, False)
    X = gen.astype(np.float64)
    seed = TRAIT_SEEDS[model]
    with bw.Genotypes(gen, path=2) as g:
        out = bw.gibbs_fit(model, Y, g, it=IT, bi=BI, seed=seed, nchains=NCHAIN, chain0=CHAIN0)
    for s, (r32, r64) in enumerate(_replays(model, Y, None, X, seed, NCHAIN, CHAIN0)):
        case = "traits %s blocked system %d" % (model, s)
        _margins_ok(r32, r64, case)
        _close(_system(out, s), r32, r64, _gibbs_keys(model), case, exact=("d",))


def _old_entry(bw, g, model, y, nchains, seed):
    """bwgr_gibbs_fit called directly (the single-trait entry point)."""
    from bwgr_b200 import _lib
    nc, n, p = nchains, g.n, g.p
    bufs = {k: np.zeros(shape, order="F") for k, shape in
            (("mu", (nc,)), ("b", (p, nc)), ("d", (p, nc)), ("hat", (n, nc)), ("vb", (p, nc)), ("scal", (bw.api.NSCAL, nc)))}
    par = _lib.GibbsParams(bw.api._GIBBS[model], nc, IT, BI, 0.95, 5.0, 0.5, seed)
    ptr = {k: v.ctypes.data_as(C.c_void_p) for k, v in bufs.items()}
    out = _lib.GibbsOut(ptr["mu"], ptr["b"], ptr["d"], ptr["hat"], ptr["vb"], ptr["scal"])
    y = np.ascontiguousarray(y, dtype=np.float64)
    _lib.check(g.lib.bwgr_gibbs_fit(g.h, C.byref(par), y.ctypes.data_as(C.c_void_p), C.byref(out)))
    return bufs


@pytest.mark.gpu
@pytest.mark.parametrize("nchains", [1, 3])
@pytest.mark.parametrize("path", [1, 2, 3])
def test_one_column_equals_single_trait_entry(tpod, path, nchains):
    """bwgr_gibbs_fit_sys with nsys = 1, no mask, chain0 = 0 gives bwgr_gibbs_fit's outputs bit for bit."""
    bw = pytest.importorskip("bwgr_b200")
    y, gen = tpod
    for model in ("BayesB", "BayesCpi"):
        with bw.Genotypes(gen, path=path) as g:
            ref = _old_entry(bw, g, model, y, nchains, 21)
            out = bw.gibbs_fit(model, y[:, None], g, it=IT, bi=BI, seed=21, nchains=nchains)
        want = {"mu": ref["mu"], "b": ref["b"], "hat": ref["hat"], "d": ref["d"], "ve": ref["scal"][1], "h2": ref["scal"][2],
                "vb": ref["vb"] if model == "BayesB" else ref["scal"][0], "pi": ref["scal"][4]}
        for key, v in out.items():
            if key in want:
                assert np.array_equal(np.asarray(v), want[key]), (model, key)


@pytest.mark.gpu
def test_column_shard_draws_the_streams_of_the_whole_fit(tpod):
    """Columns 3..5 of a 6-column masked fit, fitted alone with chain0 = 3 * nchains, are bit-identical to those columns of the whole
    fit (small-n family: one CTA per system, nothing shared between systems)."""
    bw = pytest.importorskip("bwgr_b200")
    y, gen = tpod
    rng = np.random.default_rng(5)
    n = y.size
    Y = np.asfortranarray(np.stack([y + 0.3 * rng.normal(size=n) for _ in range(6)], axis=1))
    M = np.asfortranarray(rng.random((n, 6)) < 0.75)
    nc = 2
    with bw.Genotypes(gen, path=1) as g:
        whole = bw.gibbs_fit("BayesB", Y, g, it=IT, bi=BI, seed=9, nchains=nc, row_mask=M)
        part = bw.gibbs_fit("BayesB", Y[:, 3:], g, it=IT, bi=BI, seed=9, nchains=nc, row_mask=M[:, 3:], chain0=3 * nc)
    for key, v in part.items():
        assert np.array_equal(np.asarray(v), np.asarray(whole[key])[..., 3 * nc:]), key


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1037, 10000])
@pytest.mark.parametrize("store", ["int8", "2bit", "float32"])
def test_fitted_values_of_k_systems(n, store):
    """One pass over the store for k systems gives every column bit-identical to the fitted values of that column alone."""
    bw = pytest.importorskip("bwgr_b200")
    p = 700
    gen, _ = synth(n, p, seed=n)
    rng = np.random.default_rng(3)
    if store == "float32":
        G = (gen - gen.mean(0)).astype(np.float32).astype(np.float64)
        kw = dict(storage=bw.STORE_F32)
    else:
        G = gen
        kw = dict(storage=bw.STORE_2BIT if store == "2bit" else bw.STORE_I8)
    with bw.Genotypes(G, **kw) as g:
        assert g.info()["storage"] == kw["storage"]
        for k in (1, 3, 37, 100):
            B = rng.normal(size=(p, k)).astype(np.float32).astype(np.float64)
            B[rng.random((p, k)) < 0.2] = 0.0  # exact zeros: the single-system pass skips them, the k-system pass does not
            mu = rng.normal(size=k).astype(np.float32).astype(np.float64)
            hat = g.fitted(B, mu)
            assert hat.shape == (n, k)
            for t in range(k):
                one = g.fitted(B[:, t], mu[t])
                assert np.array_equal(hat[:, t], one), (store, n, k, t)
            ref = mu + G.astype(np.float64) @ B
            np.testing.assert_allclose(hat, ref, rtol=0, atol=1e-5 * np.abs(ref).max())


@pytest.mark.gpu
def test_errors_leave_the_handle_usable(tpod):
    """nsys < 1, NaN in Y, a mask column keeping one row -> BWGR_ERR_ARG; more than 32 masked systems whose residual does not fit one
    SM -> BWGR_ERR_UNSUPPORTED.  After each, a valid fit on the same handle succeeds."""
    bw = pytest.importorskip("bwgr_b200")
    from bwgr_b200 import _lib
    y, gen = tpod
    n = y.size
    Y = np.stack([y, y], axis=1)

    def valid(g, yy):
        out = bw.gibbs_fit("BayesB", yy, g, it=3, bi=1, seed=2)
        assert np.isfinite(out["b"]).all()

    with bw.Genotypes(gen) as g:
        # nsys = 0 through the C entry directly (the Python mirror derives nsys from Y)
        par = _lib.GibbsSysParams(_lib.GibbsParams(2, 1, 3, 1, 0.95, 5.0, 0.5, 2), 0, None, 0)
        out = _lib.GibbsOut(*([None] * 6))
        assert g.lib.bwgr_gibbs_fit_sys(g.h, C.byref(par), Y.ctypes.data_as(C.c_void_p), C.byref(out)) == -1
        valid(g, y)
        bad = Y.copy()
        bad[7, 1] = np.nan
        with pytest.raises(bw.BwgrError) as ei:
            bw.gibbs_fit("BayesB", bad, g, it=3, bi=1)
        assert ei.value.code == -1
        valid(g, Y)
        M = np.ones((n, 2), dtype=bool)
        M[1:, 1] = False
        with pytest.raises(bw.BwgrError) as ei:
            bw.gibbs_fit("BayesB", Y, g, it=3, bi=1, row_mask=M)
        assert ei.value.code == -1
        valid(g, Y)
    # 33 masked systems at n = 40,000: the small-n family cannot hold the residual, the grid family takes at most 32 systems
    big_n, k = 40000, 33
    rng = np.random.default_rng(1)
    G = rng.integers(0, 3, size=(big_n, 8)).astype(np.int8)
    Yb = rng.normal(size=(big_n, k))
    Mb = rng.random((big_n, k)) < 0.8
    with bw.Genotypes(G) as g:
        with pytest.raises(bw.BwgrError) as ei:
            bw.gibbs_fit("BayesB", Yb, g, it=3, bi=1, row_mask=Mb)
        assert ei.value.code == -5
        out = bw.gibbs_fit("BayesB", Yb[:, :32], g, it=3, bi=1, row_mask=Mb[:, :32])
        assert np.isfinite(out["b"]).all()
