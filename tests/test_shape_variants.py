"""The sweep-kernel variants that only larger shapes select, against the oracle.

Every sweep kernel picks a variant from the shape at launch time: the small-n family how many 16-row chunks a thread holds and how
deep its cp.async ring is, the general MRR3 path how many residual rows a thread keeps in registers (NJ, or 0 for a slab in shared
memory), the blocked family how many 128-row atoms a worker has, its topology (clustered or flat) and how many systems share a
solve warp.  Each case below first shows that its shape reaches the variant it is meant to test, on the device it runs on:
  - blocked family: from the sweep's trace header {CTAs, blocks, 32, look-ahead D} (BWGR_TRACE);
  - small-n family and general MRR3 path (no trace): from the selection arithmetic of the launch code, restated below with the
    device's SM count and opt-in shared memory.  n is chosen from those two numbers, so each case lands in its bucket; a bucket
    that cannot be reached fails the case.
n is ragged everywhere (51 rows short of a multiple of 128, so the last CTA or thread holds a partial slab), and so is p.

The bars are the suite's: _close_em (1e-4, widened by the float oracle's distance to its float64 recipe), the Philox replay's _close,
and 1e-6 for the float64 state of the general MRR3 path (2e-4 for the rotated float32 path).  The replay seeds were chosen on the
oracle alone at the shapes a B200 (148 SMs, 227 KB of opt-in shared memory) selects; test_replay_seeds_have_no_near_ties checks them
there on the CPU, and every GPU case checks its own margins again on the device it runs on."""
import functools

import numpy as np
import pytest

import oracle as O
from conftest import synth
from test_gibbs_replay import _close, _gibbs_keys, _kmup_state, _margins_ok
from test_gibbs_systems import BI, IT, _replays, _system
from test_gpu_parity import RTOL, _close_em, _close_mrr

B200 = (148, 232448)  # SMs, opt-in shared memory per block (bytes): the geometry the replay seeds were chosen at
P = 333               # markers of the univariate cases: 3 blocks of 128, the last one ragged
P_MRR = 237           # markers of the MRR3 cases
CHAIN0 = 5


def _ld(n):
    return -(-n // 128) * 128


def _pick(target_ld, pred, what):
    """The ragged n = ld - 51 nearest to target_ld (ld a multiple of 128) that satisfies pred(n); a bucket no n reaches fails."""
    for ld in sorted(range(128, 2 * target_ld + 128, 128), key=lambda v: abs(v - target_ld)):
        if pred(ld - 51):
            return ld - 51
    raise AssertionError("no row count reaches " + what)


def _geometry():
    import torch
    pr = torch.cuda.get_device_properties(0)
    return pr.multi_processor_count, pr.shared_memory_per_block_optin


# ---- small-n family (csrc/small_n.cu) -------------------------------------------------------------------------------------------

def _small_n_plan(n, optin, two_bit=False, masked=False, gibbs=False, weighted=False):
    """(fits, ring, T, chunks): small_n_fits, launch_small_model and small_n_smem restated.  A thread owns 16-row chunks of the
    residual; T = clamp(ceil(chunks / 32) * 32, 32, 1024) threads, so n > 16 T rows gives a thread several chunks (the
    single == false path).  The ring is the deepest of 8, 4, 2 whose shared memory fits; the family takes the store if ring 2 fits at
    T = 1024 with the Gibbs draw buffer."""
    ld = _ld(n)
    chunks = ld // 16
    T = min(1024, max(32, -(-chunks // 32) * 32))
    col = ld // 4 if two_bit else ld

    def smem(ring, T, gibbs):
        return (4 * ld + ring * col + (ld if masked else 0) + 64 * 4 + (2 * T * 16 if gibbs else 0) + 2 * T * 4 + 16 +
                (4 * ld + 16 if weighted else 0))

    ring = next((r for r in (8, 4, 2) if smem(r, T, gibbs) <= optin), None)
    return smem(2, 1024, True) <= optin, ring, T, chunks


def _small_n_n(geo, target, ring, **kw):
    """n near `target` rows where the small-n family takes the store and launches ring `ring` with several chunks per thread."""
    def ok(n):
        fits, r, T, chunks = _small_n_plan(n, geo[1], **kw)
        return fits and r == ring and chunks > T
    return _pick(_ld(target), ok, "small-n ring %d with several chunks per thread (%s)" % (ring, kw))


def _assert_small_n(n, geo, ring, case, **kw):
    fits, r, T, chunks = _small_n_plan(n, geo[1], **kw)
    print("VARIANT %-36s n %6d  small-n ring %s, %d threads, %d chunks (%d..%d per thread)" % (case, n, r, T, chunks, chunks // T, -(-chunks // T)))
    assert fits and r == ring and chunks > T, (case, n, fits, r, T, chunks)


# ---- general MRR3 path (csrc/mrr_gen.cu) ----------------------------------------------------------------------------------------

def _mrr_gen_plan(n, sms):
    """(NJ, rows_per_cta, CTAs): grid_geometry (fit.cu) and launch_mrr_gen_sweep restated.  rows_per_cta = max(64, ceil(ld / SMs)
    rounded up to 16); a thread keeps ceil(rows_per_cta / 32) rows per trait in registers, the kernel instance with NJ = 2, 4, 8, 12 or
    16 such rows, or NJ = 0 (slab in shared memory) above 512 rows per CTA."""
    ld = _ld(n)
    rp = max(64, -(-(-(-ld // sms)) // 16) * 16)
    nj = -(-rp // 32)
    return next((v for v in (2, 4, 8, 12, 16) if nj <= v), 0), rp, -(-ld // rp)


# rows per CTA of each NJ case: the top of its bucket, so that every register slot j < NJ holds rows (above 512 for NJ = 0)
MRR_RP = {2: 64, 4: 128, 8: 256, 12: 384, 16: 512, 0: 560}
# traits of each NJ case: together they put a trait in every slot q of warp w's traits w + 8 q
MRR_K = {2: 32, 4: 9, 8: 9, 12: 20, 16: 5, 0: 17}


def _mrr_n(geo, nj):
    rp = MRR_RP[nj]
    return _pick(rp * geo[0], lambda n: _mrr_gen_plan(n, geo[0])[:2] == (nj, rp), "MRR3 general NJ = %d at %d rows per CTA" % (nj, rp))


# ---- blocked family (csrc/sweep_pipe.cu): the plan from the trace header ---------------------------------------------------------

def _clusters(sms):
    return min(18, max(2, (sms - 36) // 8))  # plan_pipe's first choice (fit.cu): leave 36 SMs to the next sweep's Gram band


def _n_clustered(geo, rows):
    """n whose first-choice clustered plan gives each of the 7 x clusters workers `rows` rows."""
    return (7 * _clusters(geo[0]) * rows) // 128 * 128 - 51


def _n_flat(geo, rows):
    """n whose flat plan (one solver CTA + SMs - 1 workers) gives each worker `rows` rows."""
    return ((geo[0] - 1) * rows) // 128 * 128 - 51


def _traced(monkeypatch, tmp_path, fit):
    """Run fit() with BWGR_TRACE set: (its result, the trace header or None if no blocked sweep ran)."""
    trace = tmp_path / "trace.bin"
    if trace.exists():
        trace.unlink()
    monkeypatch.setenv("BWGR_TRACE", str(trace))
    try:
        out = fit()
    finally:
        monkeypatch.delenv("BWGR_TRACE")
    if not trace.exists():
        return out, None
    hdr = np.fromfile(trace, dtype=np.int64, count=4)
    trace.unlink()
    return out, hdr


def _assert_plan(hdr, n, p, topology, atoms, case, lookahead=None):
    """Topology, rows per worker and row atoms of the blocked sweep from its header {CTAs, blocks, 32, D}.  Clustered: 8 CTAs per
    cluster, 7 of them workers; flat: W workers + 1 solver CTA, and W = ceil(ld / R).  R = ceil(ceil(ld / W) / 16) * 16 with
    ld = ceil(n / 128) * 128, atoms = ceil(R / 128)."""
    assert hdr is not None, (case, "no blocked sweep ran")
    ctas = int(hdr[0])
    assert hdr[1] == -(-p // 128) and hdr[2] == 32, (case, hdr)
    ld = _ld(n)
    Rf = -(-(-(-ld // (ctas - 1))) // 16) * 16
    is_flat = -(-ld // Rf) == ctas - 1  # the header is the flat plan's W + 1 CTAs
    W = 7 * ctas // 8 if topology == "clustered" else ctas - 1
    R = -(-(-(-ld // W)) // 16) * 16
    print("VARIANT %-36s n %6d  blocked %s, %d CTAs, %d workers x %d rows, %d atoms, look-ahead %d" % (case, n, topology, ctas, W, R, -(-R // 128), hdr[3]))
    if topology == "clustered":
        assert ctas % 8 == 0 and not is_flat, (case, "not clustered", hdr)
    else:
        assert is_flat, (case, "not the flat plan", hdr)
    assert R <= 512 and -(-R // 128) == atoms, (case, R, atoms)
    if lookahead is not None:
        assert hdr[3] == lookahead, (case, hdr)


# ---- data and oracle fits ------------------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def _data(n, p, k=1, seed=20261021):
    X, Y = synth(n, p, k=k, seed=seed)
    return X, np.asfortranarray(Y.reshape(n, -1))


@functools.lru_cache(maxsize=None)
def _xf(n, p, k=1):
    return _data(n, p, k)[0].astype(np.float32)


@functools.lru_cache(maxsize=None)
def _em_ref(model, n, p, k, t, it):
    """(float oracle, float64 oracle) of column t."""
    X, Y = _data(n, p, k)
    Xf = _xf(n, p, k)
    return O.em(model, Y[:, t], Xf, it=it), O.em(model, Y[:, t], Xf, it=it, use_double=True)


def _close_em_cols(out, model, n, p, k, cols, it, case):
    for t in cols:
        ref, ref64 = _em_ref(model, n, p, k, t, it)
        o = {key: (v[..., t] if np.ndim(v) else v) for key, v in out.items()}
        try:
            _close_em(o, ref, model, ref64)
        except AssertionError as e:
            raise AssertionError((case, model, "system", t, str(e)))


def _gibbs_case(bw, model, g, Y, seed, nchain=1, chain0=0, M=None):
    return bw.gibbs_fit(model, Y, g, it=IT, bi=BI, seed=seed, nchains=nchain, row_mask=M, chain0=chain0)


def _check_replays(out, reps, model, case, M=None, X=None, nchain=1):
    keys = [k for k in _gibbs_keys(model) if M is None or k != "hat"]
    for s, (r32, r64) in enumerate(reps):
        c = "%s %s system %d" % (case, model, s)
        _margins_ok(r32, r64, c)
        one = _system(out, s)
        _close(one, r32, r64, keys, c, exact=("d",))
        if M is not None:  # fitted values of every row, the held-out ones included
            ref = one["mu"] + X @ one["b"]
            np.testing.assert_allclose(one["hat"], ref, rtol=0, atol=1e-5 * np.abs(ref).max())


def _masks(n, k, seed=3):
    fold = np.random.default_rng(seed).integers(0, 3, size=n)
    return np.asfortranarray(np.stack([fold != t for t in range(k)], axis=1))


# Replay cases: (name, model) -> seed.  Every system of every case is free of near-ties at its seed at the B200's shapes.
SEEDS = {
    ("clustered3", "BayesA"): 1, ("clustered3", "BayesB"): 3, ("clustered3", "BayesC"): 1, ("clustered3", "BayesL"): 1,
    ("clustered3", "BayesDpi"): 1,
    ("flat4", "BayesB"): 3,
    ("traits2", "BayesA"): 8, ("traits2", "BayesB"): 8,
    ("ring2", "BayesA"): 1, ("ring2", "BayesB"): 1,
    ("masked", "BayesB"): 2, ("masked", "BayesCpi"): 2,
    ("2bit", "BayesC"): 3,
}
KMUP2_SEED = 1


def _replay_shape(name, geo):
    """(n, columns, chains, masked) of a replay case."""
    return {"clustered3": (_n_clustered(geo, 320), 1, 1, False),
            "flat4": (_n_flat(geo, 416), 1, 1, False),
            "traits2": (_n_clustered(geo, 320), 3, 2, False),  # 6 systems: flat, 2 atoms
            "ring2": (_small_n_n(geo, 30000, 2, gibbs=True), 1, 1, False),
            "masked": (_small_n_n(geo, 24000, 4, masked=True), 3, 1, True),
            "2bit": (_small_n_n(geo, 40000, 2, two_bit=True, gibbs=True), 1, 1, False)}[name]


def _replay(name, model, geo):
    """Data of a replay case and the oracle's (float, float64) replays of its systems."""
    n, k, nchain, masked = _replay_shape(name, geo)
    X, Y = _data(n, P, 3)
    Y = Y[:, :k]
    M = _masks(n, k) if masked else None
    chain0 = 0 if (k, nchain) == (1, 1) else CHAIN0
    return n, X, Y, M, nchain, chain0, _replays(model, Y, M, X.astype(np.float64), SEEDS[name, model], nchain, chain0)


def _kmup2_case(geo):
    """KMUP2 on rows drawn with replacement on the small-n family: n, the genotypes, the sweep's inputs and its (float, float64)
    replays.  With the row mask, the multiplicities and the draw buffer in shared memory, ring 2 fits only up to ld = 17,280 on a
    B200, so n settles near 17,000 rather than 20,000 (still several chunks per thread)."""
    n = _small_n_n(geo, 20000, 2, masked=True, gibbs=True, weighted=True)
    X, Y = _data(n, P, 3)
    Xd = X.astype(np.float64)
    y = Y[:, 0]
    rng = np.random.default_rng(8)
    use = np.sort(rng.integers(0, n, int(0.8 * n))).astype(np.float64)
    b0, d0, e, L = _kmup_state(y, P)
    xx = (Xd ** 2).sum(0)
    args = (use, b0, d0, xx, e, L, 0.5 * float(np.var(y)), 0.4)
    kw = dict(seed=KMUP2_SEED, draws="philox")
    return n, X, args, (O.kmup2(Xd, *args, **kw), O.kmup2(Xd, *args, use_double=True, **kw))


# ---- CPU --------------------------------------------------------------------------------------------------------------------------

def test_replay_seeds_have_no_near_ties():
    """Every system of every replay case below, at the shapes a B200 selects, is free of near-ties at its seed."""
    for name, model in SEEDS:
        for s, (r32, r64) in enumerate(_replay(name, model, B200)[-1]):
            _margins_ok(r32, r64, "%s %s system %d" % (name, model, s))
    _, _, _, (r32, r64) = _kmup2_case(B200)
    _margins_ok(r32, r64, "kmup2 repeated rows")


def test_selection_arithmetic_reaches_every_bucket_on_a_b200():
    """The row counts the cases choose on a B200 land where the issue's table says they do."""
    sms, optin = B200
    assert _small_n_plan(_small_n_n(B200, 17000, 8), optin)[1:] == (8, 1024, 1064)
    assert [_mrr_gen_plan(_mrr_n(B200, nj), sms)[0] for nj in MRR_RP] == list(MRR_RP)
    assert not _small_n_plan(_replay_shape("2bit", B200)[0], optin)[0]  # the int8 store does not fit the small-n family there


# ---- GPU: small-n family ----------------------------------------------------------------------------------------------------------

def _bw():
    return pytest.importorskip("bwgr_b200")


@pytest.mark.gpu
def test_small_n_several_chunks_per_thread_em():
    """int8 store, unmasked, ~17,000 rows: 1,024 threads, some with 2 chunks, ring 8; p > 2,048 so that the marker order in shared
    memory is refilled.  emRR, emBB, emBC, emBL and lasso after 8 sweeps."""
    bw = _bw()
    geo = _geometry()
    n, p = _small_n_n(geo, 17000, 8), 2111
    _assert_small_n(n, geo, 8, "em int8 unmasked")
    X, Y = _data(n, p)
    with bw.Genotypes(X, path=bw.PATH_SMALL_N) as g:
        for model in ("emRR", "emBB", "emBC", "emBL", "lasso"):
            out = bw.em_fit(model, Y[:, 0], g, it=8)
            ref, ref64 = _em_ref(model, n, p, 1, 0, 8)
            _close_em(out, ref, model, ref64)


@pytest.mark.gpu
def test_small_n_masked_folds_em():
    """Three row-masked systems (CV folds) at ~24,000 rows: several chunks per thread, ring 4; emBC against per-subset oracle fits."""
    bw = _bw()
    geo = _geometry()
    n = _small_n_n(geo, 24000, 4, masked=True)
    _assert_small_n(n, geo, 4, "emBC masked", masked=True)
    X, Y = _data(n, P, 3)
    M = _masks(n, 3)
    with bw.Genotypes(X, path=bw.PATH_SMALL_N) as g:
        out = bw.em_fit("emBC", Y, g, it=8, row_mask=M)
    for t in range(3):
        keep = M[:, t]
        Xk = X[keep].astype(np.float32)
        ref = O.em("emBC", Y[keep, t], Xk, it=8)
        ref64 = O.em("emBC", Y[keep, t], Xk, it=8, use_double=True)
        nb = np.abs(ref["b"] - ref64["b"]).max()
        assert np.abs(out["b"][:, t] - ref["b"]).max() <= RTOL * np.abs(ref["b"]).max() + nb, t
        assert abs(out["h2"][t] - ref["h2"]) <= RTOL + abs(ref["h2"] - ref64["h2"]), t
        assert abs(out["Ve"][t] - ref["Ve"]) <= RTOL * abs(ref["Ve"]) + abs(ref["Ve"] - ref64["Ve"]), t


@pytest.mark.gpu
@pytest.mark.parametrize("name,model,kw", [("masked", "BayesB", dict(masked=True)), ("masked", "BayesCpi", dict(masked=True)),
                                           ("ring2", "BayesA", {}), ("ring2", "BayesB", {}),
                                           ("2bit", "BayesC", dict(two_bit=True))])
def test_small_n_gibbs_replay(name, model, kw):
    """Gibbs samplers on the small-n family with several chunks per thread: three masked systems through bwgr_gibbs_fit_sys (each
    replayed on its rows under chain 5 + s), unmasked chains at ~30,000 rows, and the 2-bit store at ~40,000 rows (beyond the int8
    store); all at ring 2."""
    bw = _bw()
    geo = _geometry()
    n, X, Y, M, nchain, chain0, reps = _replay(name, model, geo)
    _assert_small_n(n, geo, 2, "%s %s" % (name, model), gibbs=True, **kw)
    storage = bw.STORE_2BIT if name == "2bit" else bw.STORE_I8
    with bw.Genotypes(X, storage=storage, path=bw.PATH_SMALL_N) as g:
        out = _gibbs_case(bw, model, g, Y, SEEDS[name, model], nchain, chain0, M)
    _check_replays(out, reps, model, "small-n " + name, M, X.astype(np.float64))


@pytest.mark.gpu
def test_small_n_2bit_store_beyond_int8():
    """~40,000 rows: the int8 store does not fit the small-n family, the 2-bit store does (2-3 chunks per thread, 4-byte cp.async
    columns, ring 4 for EM): emRR against the oracle."""
    bw = _bw()
    geo = _geometry()
    n = _replay_shape("2bit", geo)[0]
    assert not _small_n_plan(n, geo[1])[0]
    _assert_small_n(n, geo, 4, "emRR 2-bit", two_bit=True)
    X, Y = _data(n, P, 3)
    with bw.Genotypes(X, path=bw.PATH_SMALL_N) as g:
        with pytest.raises(bw.BwgrError) as ei:
            bw.emRR(Y[:, 0], g, it=2)
        assert ei.value.code == -5
    with bw.Genotypes(X, storage=bw.STORE_2BIT, path=bw.PATH_SMALL_N) as g:
        out = bw.em_fit("emRR", Y[:, 0], g, it=8)
    ref, ref64 = _em_ref("emRR", n, P, 3, 0, 8)
    _close_em(out, ref, "emRR", ref64)


@pytest.mark.gpu
def test_small_n_2bit_equals_int8_with_several_chunks():
    """~20,000 rows, which both stores take with several chunks per thread (ring 4 on int8, ring 8 on 2-bit): the same arithmetic
    gives the same bits."""
    bw = _bw()
    geo = _geometry()
    n = _small_n_n(geo, 20000, 4)
    _assert_small_n(n, geo, 4, "int8 ~20k")
    _assert_small_n(n, geo, 8, "2-bit ~20k", two_bit=True)
    X, Y = _data(n, P, 3)
    for model in ("emRR", "emBC"):
        with bw.Genotypes(X, storage=bw.STORE_I8, path=bw.PATH_SMALL_N) as g:
            a = bw.em_fit(model, Y[:, 0], g, it=6)
        with bw.Genotypes(X, storage=bw.STORE_2BIT, path=bw.PATH_SMALL_N) as g:
            b = bw.em_fit(model, Y[:, 0], g, it=6)
        assert np.array_equal(a["b"], b["b"]) and np.array_equal(a["hat"], b["hat"]), model


@pytest.mark.gpu
def test_small_n_kmup2_repeated_rows():
    """KMUP2 on rows drawn with replacement (row multiplicities in the dot products) with several chunks per thread: the Philox replay."""
    bw = _bw()
    geo = _geometry()
    n, X, args, (r32, r64) = _kmup2_case(geo)
    _assert_small_n(n, geo, 2, "kmup2 repeated rows", masked=True, gibbs=True, weighted=True)
    use = args[0]
    assert np.unique(use).size < use.size
    _margins_ok(r32, r64, "kmup2 repeated rows")
    with bw.Genotypes(X, path=bw.PATH_SMALL_N) as g:
        out = bw.KMUP2(g, *args, seed=KMUP2_SEED)
    assert np.array_equal(out["d"], r64["d"])
    _close(out, r32, r64, ("b", "e"), "kmup2 repeated rows")


# ---- GPU: general MRR3 path -------------------------------------------------------------------------------------------------------

def _mrr_Y(X, k, missing, seed=8):
    rng = np.random.default_rng(seed)
    p = X.shape[1]
    Lc = np.linalg.cholesky(0.5 * np.ones((k, k)) + 0.5 * np.eye(k))
    B = (rng.normal(size=(p, k)) @ Lc.T) * (rng.random((p, 1)) < 0.05)
    G = X.astype(np.float64) @ B
    Y = G / G.std(0) + rng.normal(size=G.shape)
    if missing:
        Y[rng.random(Y.shape) < missing] = np.nan
    return np.asfortranarray(Y)


def _mrr_fit(monkeypatch, tmp_path, g, Y, **kw):
    """bw.MRR3 with the trace on: (result, trace header or None)."""
    return _traced(monkeypatch, tmp_path, lambda: _bw().MRR3(Y, g, **kw))


@pytest.mark.gpu
@pytest.mark.parametrize("nj", list(MRR_RP))
def test_mrr3_general_every_nj(monkeypatch, tmp_path, nj):
    """The general MRR3 path with 25 % of Y missing at the row count of each register variant NJ (and NJ = 0, the slab in shared
    memory), the traits spread over every slot of warp w's traits w + 8 q: 1 and 3 sweeps against the oracle at 1e-6."""
    bw = _bw()
    geo = _geometry()
    n, k = _mrr_n(geo, nj), MRR_K[nj]
    got, rp, grid = _mrr_gen_plan(n, geo[0])
    print("VARIANT %-36s n %6d  MRR3 general NJ %d, %d rows per CTA, %d CTAs, k %d" % ("mrr3 NJ %d" % nj, n, got, rp, grid, k))
    assert got == nj and grid <= geo[0]
    X, _ = _data(n, P_MRR)
    Y = _mrr_Y(X, k, 0.25)
    Xd = X.astype(np.float64)
    with bw.Genotypes(X) as g:
        for its in (1, 3):
            ref = O.mrr3(Y, Xd, maxit=its)
            out, hdr = _mrr_fit(monkeypatch, tmp_path, g, Y, maxit=its)
            assert hdr is None  # no blocked sweep: the general path ran
            assert out["Its"] == ref["Its"] == its
            _close_mrr(out, ref, 1e-6)
            np.testing.assert_allclose(out["cnvB"], ref["cnvB"], atol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("nj", [8, 0])
def test_mrr3_general_innergs(monkeypatch, tmp_path, nj):
    """InnerGS (two k x k matrices per marker in the ring) at a register variant and at NJ = 0, complete Y: 3 sweeps against the
    oracle at the suite's InnerGS bar."""
    bw = _bw()
    geo = _geometry()
    n, k = _mrr_n(geo, nj), MRR_K[nj]
    assert _mrr_gen_plan(n, geo[0])[0] == nj
    X, _ = _data(n, P_MRR)
    Y = _mrr_Y(X, k, 0.0)
    with bw.Genotypes(X) as g:
        out, hdr = _mrr_fit(monkeypatch, tmp_path, g, Y, maxit=3, InnerGS=True)
    assert hdr is None
    _close_mrr(out, O.mrr3(Y, X.astype(np.float64), maxit=3, InnerGS=True), 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 16])
def test_mrr3_rotated_one_and_sixteen_traits(monkeypatch, tmp_path, k):
    """The rotated fast path (k systems on the blocked family, flat, 1 atom) at k = 1 and k = 16 (two systems per solve warp), complete
    Y, 1 and 3 sweeps at the fast path's 2e-4.  (At k = 32 the blocked plan does not fit shared memory at any row count, and MRR3
    runs on the general path: test_mrr3_thirty_two_traits_blocked_refuses.)"""
    bw = _bw()
    n = 3000 - 51
    X, _ = _data(n, P_MRR)
    Y = _mrr_Y(X, k, 0.0)
    with bw.Genotypes(X) as g:
        for its in (1, 3):
            out, hdr = _mrr_fit(monkeypatch, tmp_path, g, Y, maxit=its)
            _assert_plan(hdr, n, P_MRR, "flat", 1, "mrr3 rotated k %d" % k)
            _close_mrr(out, O.mrr3(Y, X.astype(np.float64), maxit=its), 2e-4)


@pytest.mark.gpu
def test_mrr3_thirty_two_traits_blocked_refuses(monkeypatch, tmp_path):
    """k = 32, complete Y, at a row count where the blocked plan needs 4 atoms: (4 + 1) x 128 TMEM columns > 512, so bwgr_mrr3_fit
    falls back to the general path (NJ = 16 there), which matches the oracle at its float64 bar."""
    bw = _bw()
    geo = _geometry()
    n, k = _n_flat(geo, 416), 32
    nj, rp, _ = _mrr_gen_plan(n, geo[0])
    print("VARIANT %-36s n %6d  MRR3 general NJ %d, %d rows per CTA" % ("mrr3 k 32 blocked refuses", n, nj, rp))
    assert nj == 16
    X, _ = _data(n, P_MRR)
    Y = _mrr_Y(X, k, 0.0)
    with bw.Genotypes(X) as g:
        out, hdr = _mrr_fit(monkeypatch, tmp_path, g, Y, maxit=2)
    assert hdr is None
    _close_mrr(out, O.mrr3(Y, X.astype(np.float64), maxit=2), 1e-6)


# ---- GPU: blocked family ----------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("model", list(O.EM_MODELS))
def test_blocked_three_atoms_em(monkeypatch, tmp_path, model):
    """One system, clustered, 3 row atoms per worker (~31,000 rows): the ten EM solvers after 6 sweeps."""
    bw = _bw()
    geo = _geometry()
    n = _n_clustered(geo, 320)
    X, Y = _data(n, P, 3)
    with bw.Genotypes(X, path=bw.PATH_BLOCKED) as g:
        out, hdr = _traced(monkeypatch, tmp_path, lambda: bw.em_fit(model, Y[:, 0], g, it=6))
    _assert_plan(hdr, n, P, "clustered", 3, "em 3 atoms " + model)
    ref, ref64 = _em_ref(model, n, P, 3, 0, 6)
    _close_em(out, ref, model, ref64)


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["BayesA", "BayesB", "BayesC", "BayesL", "BayesDpi"])
def test_blocked_three_atoms_gibbs_replay(monkeypatch, tmp_path, model):
    """One chain, clustered, 3 row atoms: BayesA (linear chain), BayesB, BayesC, BayesL and BayesDpi against the Philox replay."""
    bw = _bw()
    geo = _geometry()
    n, X, Y, M, nchain, chain0, reps = _replay("clustered3", model, geo)
    with bw.Genotypes(X, path=bw.PATH_BLOCKED) as g:
        out, hdr = _traced(monkeypatch, tmp_path, lambda: _gibbs_case(bw, model, g, Y, SEEDS["clustered3", model]))
    _assert_plan(hdr, n, P, "clustered", 3, "gibbs 3 atoms " + model)
    _check_replays(out, reps, model, "blocked 3 atoms")


@pytest.mark.gpu
def test_blocked_flat_topology_one_gpu(monkeypatch, tmp_path):
    """~61,000 rows on one GPU: beyond the clustered plan, the flat one (one solver CTA, SMs - 1 workers, 4 atoms, look-ahead 1):
    emRR, emBC and a BayesB replay."""
    bw = _bw()
    geo = _geometry()
    n, X, Y, M, nchain, chain0, reps = _replay("flat4", "BayesB", geo)
    with bw.Genotypes(X, path=bw.PATH_BLOCKED) as g:
        for model in ("emRR", "emBC"):
            out, hdr = _traced(monkeypatch, tmp_path, lambda: bw.em_fit(model, Y[:, 0], g, it=6))
            _assert_plan(hdr, n, P, "flat", 4, "flat " + model, lookahead=1)
            ref, ref64 = _em_ref(model, n, P, 3, 0, 6)
            _close_em(out, ref, model, ref64)
        out, hdr = _traced(monkeypatch, tmp_path, lambda: _gibbs_case(bw, "BayesB", g, Y, SEEDS["flat4", "BayesB"]))
    _assert_plan(hdr, n, P, "flat", 4, "flat BayesB", lookahead=1)
    _check_replays(out, reps, "BayesB", "blocked flat")


SYS_MODELS = ("emRR", "emBB", "emBC", "emEN", "lasso")


@pytest.mark.gpu
@pytest.mark.parametrize("ns", [8, 9, 16])
def test_blocked_systems_per_solve_warp(monkeypatch, tmp_path, ns):
    """ns systems on the blocked family at ~3,000 rows (flat, 1 atom): with ns > 8 a solve warp runs several systems (32 systems do
    not fit the blocked plan: their solver CTA needs 278,816 bytes of shared memory at the smallest ring, against the 224,256 the
    plan allows on a B200; they run on the small-n and grid families).  emRR (in-warp
    substitution) and the scalar chains emBB, emBC, emEN, lasso: every column against its own oracle fit."""
    bw = _bw()
    n = 3000 - 51
    X, Y = _data(n, P, 32)
    with bw.Genotypes(X, path=bw.PATH_BLOCKED) as g:
        for model in SYS_MODELS:
            out, hdr = _traced(monkeypatch, tmp_path, lambda: bw.em_fit(model, Y[:, :ns], g, it=6))
            _assert_plan(hdr, n, P, "flat", 1, "%d systems %s" % (ns, model))
            _close_em_cols(out, model, n, P, 32, range(ns), 6, "%d systems" % ns)


# (case, systems, models, topology, atoms, n from the geometry)
MULTI = {
    "9 systems flat 3 atoms": (9, ("emRR", "emBC"), "flat", 3, lambda geo: _n_flat(geo, 288)),
    "2 systems linear flat 3 atoms": (2, ("emRR",), "flat", 3, lambda geo: _n_flat(geo, 288)),
    "2 systems chain clustered 3 atoms": (2, ("emBC",), "clustered", 3, lambda geo: _n_clustered(geo, 320)),
    "4 systems 3 atoms": (4, ("emRR", "emBC"), "flat", 3, lambda geo: _n_flat(geo, 288)),
    "4 systems 4 atoms": (4, ("emRR", "emBC"), "flat", 4, lambda geo: _n_flat(geo, 416)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(MULTI))
def test_blocked_systems_at_several_atoms(monkeypatch, tmp_path, case):
    """Several systems with 3 or 4 row atoms: 9 systems (flat); 2 systems, which go flat for a linear rule (the 32 x 32-inverse
    solve) and clustered for a chain; 4 systems at 3 and 4 atoms, flat.  Every column against its own oracle fit.
    4 systems never take the clustered topology: its solver CTA would need 242,976 bytes of shared memory (sring 3, the partial
    inboxes of 7 workers), more than the 223,232 the plan allows on a B200 (opt-in less 9 KB of static shared memory)."""
    bw = _bw()
    ns, models, topology, atoms, nf = MULTI[case]
    n = nf(_geometry())
    X, Y = _data(n, P, 9)
    with bw.Genotypes(X, path=bw.PATH_BLOCKED) as g:
        for model in models:
            out, hdr = _traced(monkeypatch, tmp_path, lambda: bw.em_fit(model, Y[:, :ns], g, it=6))
            _assert_plan(hdr, n, P, topology, atoms, "%s %s" % (case, model))
            _close_em_cols(out, model, n, P, 9, range(ns), 6, case)


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["BayesA", "BayesB"])
def test_blocked_gibbs_traits_two_atoms(monkeypatch, tmp_path, model):
    """3 columns x 2 chains through bwgr_gibbs_fit_sys at ~31,000 rows (6 systems: flat, 2 atoms): every system replays as chain 5 + s."""
    bw = _bw()
    geo = _geometry()
    n, X, Y, M, nchain, chain0, reps = _replay("traits2", model, geo)
    with bw.Genotypes(X, path=bw.PATH_BLOCKED) as g:
        out, hdr = _traced(monkeypatch, tmp_path, lambda: _gibbs_case(bw, model, g, Y, SEEDS["traits2", model], nchain, chain0))
    _assert_plan(hdr, n, P, "flat", 2, "gibbs traits " + model)
    _check_replays(out, reps, model, "blocked traits")

