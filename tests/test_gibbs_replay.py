"""The stochastic solvers draw for draw: every device draw is counter-addressed Philox4x32-10, so the oracle can consume the same
draws (O.gibbs / O.kmup / O.kmup2 / O.wgr with draws="philox") and each chain becomes a deterministic function of its seed.

The reference of every GPU case is the float64 replay on the same float draws.  The bar is RTOL relative to the output's scale,
widened by the float replay's own distance to the float64 one (as _close_em of test_gpu_parity.py does for the EM solvers).

A replay makes accept / reject decisions (spike-slab and Kuo-Mallick inclusion tests, Marsaglia-Tsang acceptances).  A decision the
device and the replay could take differently on float rounding alone would make the comparison meaningless, so every case asserts
at its fixed seed that no decision was near a tie:
  - inclusion tests: min |u - q| > MARGIN_Q = 1e-5.  The float replay evaluates ||e1||^2 - ||e2||^2 as the reference does, as the
    difference of two O(n) float sums; its q strays from the float64 one by up to 1e-6 on tpod and 6e-4 at 10,000 rows (so that
    distance cannot serve as the threshold there).  The device forms the difference in closed form,
    b1 (2 x'e + xx (2 b0 - b1)), whose float error moves q by orders of magnitude less than 1e-5 at these sizes; d must
    then agree exactly, which the comparisons assert;
  - Marsaglia-Tsang: min |log u - (0.5 x^2 + d - d v + d log v)| / (1 + d) > MT_MARGIN = 2e-6, about ten times the float rounding
    (a few ulp of terms of size d) by which the device's and the host's evaluations of that test can differ.
A seed that failed these would be refused, not retried; the seeds below pass them.

The statistical tests of test_gpu_parity.py stay: they are the only link to the reference's own RNG semantics."""
import numpy as np
import pytest

import oracle as O
from conftest import synth

RTOL = 1e-4
MARGIN_Q = 1e-5
MT_MARGIN = 2e-6
SEED_HI = (1 << 33) + 12345  # above 2^32: the high key word (seed_hi) takes part


# ---- numpy restatement of the generator and of the counters of each draw site -------------------------------------------------

def _philox(c0, c1, c2, c3, seed):
    """Philox4x32-10 over arrays of counters, key = (seed & 0xFFFFFFFF, seed >> 32)."""
    M0, M1, W0, W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), 0x9E3779B9, 0xBB67AE85
    c = [np.asarray(v, dtype=np.uint64) & np.uint64(0xFFFFFFFF) for v in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    m32 = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & m32, (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1), p0 & m32]
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    return c


def _u01(x):
    return ((x >> np.uint64(8)) + np.uint64(1)).astype(np.float32) * np.float32(1.0 / 16777216.0)


def _normals(c):
    # log in float64 rounded to float32: the correctly rounded logf (numpy's own float32 log may differ by an ulp)
    r = np.sqrt(np.float32(-2.0) * np.log(_u01(c[0]).astype(np.float64)).astype(np.float32))
    t = np.pi * (np.float32(2.0) * _u01(c[1])).astype(np.float64)
    return r * np.cos(t).astype(np.float32), r * np.sin(t).astype(np.float32)


def _marker_draws(markers, sweep, chain, seed):
    c = _philox(markers, sweep, chain, 0, seed)
    z1, z2 = _normals(c)
    return z1, z2, _u01(c[2])


def test_philox_known_answers():
    """The oracle's Philox4x32-10 gives the known answers tests/kat_philox.cu checks for the device's."""
    import ctypes as C
    lib = O.lib()
    cases = [((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
             ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), "408f276d 41c83b0e a20bc7c6 6d5451fd"),
             ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), "d16cfe09 94fdcceb 5001e420 24126ea1")]
    for ctr, key, want in cases:
        c = (C.c_uint32 * 4)(*ctr)
        out = (C.c_uint32 * 4)()
        lib.orc_philox4x32_10(c, C.c_uint32(key[0]), C.c_uint32(key[1]), out)
        assert " ".join("%08x" % v for v in out) == want
        assert " ".join("%08x" % int(v) for v in _philox(*ctr, key[0] | (key[1] << 32))) == want


def test_replay_draw_sites_land_on_their_counters():
    """A short replay takes each draw from the counter the device uses: marker draws (marker, sweep, chain, 0) and wgr's intercept
    (0xFFFFFFFE, sweep, 0, 0), checked against numpy recomputations of those counters."""
    import ctypes as C
    lib = O.lib()
    # marker draws as the source hands them out
    for marker, sweep, chain in ((0, 0, 0), (7, 3, 2), (123456, 77, 1)):
        out = np.zeros(4, dtype=np.float32)
        lib.orc_marker_draws(C.c_uint32(marker), C.c_uint32(sweep), C.c_uint32(chain), C.c_float(0.0), C.c_uint64(SEED_HI),
                             out.ctypes.data_as(C.POINTER(C.c_float)))
        z1, z2, u = _marker_draws(marker, sweep, chain, SEED_HI)
        np.testing.assert_array_equal(out[:3], np.array([z1, z2, u], dtype=np.float32))
    # KMUP on disjoint unit columns with e = 0, b = 0: b_j = sd z1_j (pi = 0); d_j = [u_j < q_j] and excluded b_j = sd z2_j (pi > 0)
    p = 64
    X = np.eye(p)
    L, Ve = 3.0, 2.0
    sd = np.sqrt(Ve / (1.0 + L))
    z1, z2, u = _marker_draws(np.arange(p), 0, 0, SEED_HI)
    r = O.kmup(X, np.zeros(p), np.ones(p), np.ones(p), np.zeros(p), np.full(p, L), Ve, 0.0, seed=SEED_HI, draws="philox", use_double=True)
    np.testing.assert_allclose(r["b"], sd * z1.astype(np.float64), rtol=1e-15)
    r = O.kmup(X, np.zeros(p), np.ones(p), np.ones(p), np.zeros(p), np.full(p, L), Ve, 0.5, seed=SEED_HI, draws="philox", use_double=True)
    assert np.array_equal(r["u"], u.astype(np.float64))
    np.testing.assert_array_equal(r["d"], (u < r["q"]).astype(np.float64))
    np.testing.assert_allclose(r["b"], np.where(r["d"] == 1, sd * z1.astype(np.float64), sd * z2.astype(np.float64)), rtol=1e-15)
    assert 0 < r["d"].sum() < p
    # wgr's intercept draw: with pi = 0 and BRR, mu after one iteration = mean(y) + mean(e) + (Ve / n) z, z from (0xFFFFFFFE, 0, 0, 0)
    n, p = 50, 4
    rng = np.random.default_rng(1)
    X = rng.normal(size=(n, p))
    y = rng.normal(size=n)
    w = O.wgr(y, X, it=1, bi=1, th=1, seed=SEED_HI, draws="philox", use_double=True)
    w2 = O.wgr(y, X, it=1, bi=1, th=1, seed=SEED_HI, draws="philox", use_double=True)
    assert w["mu"] == w2["mu"] and np.array_equal(w["b"], w2["b"])  # deterministic in the seed
    zm, _ = _normals(_philox(0xFFFFFFFE, 0, 0, 0, SEED_HI))
    e = y - y.mean() - X @ w["b"]
    assert abs(w["mu"] - (y.mean() + e.mean() + w["Ve"] / n * float(zm))) <= 1e-5 * max(1.0, abs(w["mu"]))


def test_default_draws_unchanged_by_the_draw_sites():
    """draws="mt" (the default) is the reference's stream: the same seed gives the same chain, another seed another one, and the
    Philox replay is a different chain (the two sources are not mixed up)."""
    rng = np.random.default_rng(4)
    X = rng.integers(0, 3, size=(60, 20)).astype(np.float64)
    y = X @ rng.normal(size=20) * 0.1 + rng.normal(size=60)
    a = O.gibbs("BayesB", y, X, it=20, bi=5, seed=3)
    b = O.gibbs("BayesB", y, X, it=20, bi=5, seed=3)
    c = O.gibbs("BayesB", y, X, it=20, bi=5, seed=3, draws="philox")
    assert np.array_equal(a["b"], b["b"]) and "q" not in a
    assert not np.array_equal(a["b"], c["b"])


# ---- GPU ----------------------------------------------------------------------------------------------------------------------

def _margins_ok(r32, r64, case):
    """The no-near-tie conditions of the module docstring, at the case's fixed seed."""
    if r64["q"].size:
        assert r32["q"].size == r64["q"].size, case
        print("REPLAY %-40s min |u - q| = %.2e, max |q_float - q_float64| = %.2e" % (case, r64["margin"], np.abs(r32["q"] - r64["q"]).max()))
        assert r64["margin"] > MARGIN_Q, (case, "inclusion test near a tie", r64["margin"])
    assert r64["mt_margin"] > MT_MARGIN, (case, "Marsaglia-Tsang test near a tie", r64["mt_margin"])


def _close(out, r32, r64, keys, case, exact=()):
    """|device - float64 replay| <= RTOL * scale + |float replay - float64 replay|, key by key; keys in `exact` must agree to 1e-6
    (the inclusion indicators and their posterior means)."""
    for key in keys:
        a, ref, f = (np.asarray(v[key], dtype=np.float64) for v in (out, r64, r32))
        diff = float(np.abs(a - ref).max())
        if key in exact:
            bar = 1e-6
        else:
            bar = RTOL * max(float(np.abs(ref).max()), 1e-3 if ref.ndim == 0 else 0.0) + float(np.abs(f - ref).max())
        print("REPLAY %-40s %-4s max|dev - replay| = %.3e  bar %.3e" % (case, key, diff, bar))
        assert diff <= bar, (case, key, diff, bar)


def _gibbs_keys(model):
    keys = ["b", "vb", "mu", "ve", "h2", "hat"]
    if model in ("BayesB", "BayesC", "BayesCpi", "BayesDpi"):
        keys.append("d")
    if model in ("BayesCpi", "BayesDpi"):
        keys.append("pi")
    return keys


@pytest.fixture(scope="module")
def ragged():
    X, y = synth(1000, 333, seed=20261020)
    return y, X


GIBBS_SEEDS = {"tpod": 11, "ragged": 5}


@pytest.mark.gpu
@pytest.mark.parametrize("data", ["tpod", "ragged"])
@pytest.mark.parametrize("path", [1, 2, 3])
@pytest.mark.parametrize("model", list(O.GIBBS_MODELS))
def test_gibbs_replay(tpod, ragged, model, path, data):
    """The seven Gibbs samplers on the small-n (1), blocked (2) and grid (3) families against the replay: 10 sweeps, burn-in 4."""
    bw = pytest.importorskip("bwgr_b200")
    y, gen = tpod if data == "tpod" else ragged
    X = gen.astype(np.float64)
    seed = GIBBS_SEEDS[data]
    kw = dict(it=10, bi=4, seed=seed, draws="philox")
    r32, r64 = O.gibbs(model, y, X, **kw), O.gibbs(model, y, X, use_double=True, **kw)
    case = "gibbs %s %s path %d" % (model, data, path)
    _margins_ok(r32, r64, case)
    with bw.Genotypes(gen, path=path) as g:
        out = bw.gibbs_fit(model, y, g, it=10, bi=4, seed=seed)
    _close(out, r32, r64, _gibbs_keys(model), case, exact=("d",))


@pytest.mark.gpu
@pytest.mark.parametrize("path", [1, 2])
@pytest.mark.parametrize("model", list(O.GIBBS_MODELS))
def test_gibbs_replay_three_chains(tpod, model, path):
    """nchains = 3: chain c of the device replays with chain index c."""
    bw = pytest.importorskip("bwgr_b200")
    y, gen = tpod
    X = gen.astype(np.float64)
    with bw.Genotypes(gen, path=path) as g:
        out = bw.gibbs_fit(model, y, g, it=10, bi=4, seed=32, nchains=3)
    for c in range(3):
        kw = dict(it=10, bi=4, seed=32, draws="philox", chain=c)
        r32, r64 = O.gibbs(model, y, X, **kw), O.gibbs(model, y, X, use_double=True, **kw)
        case = "gibbs %s tpod path %d chain %d" % (model, path, c)
        _margins_ok(r32, r64, case)
        one = {k: (v[:, c] if np.ndim(v) == 2 else v[c]) for k, v in out.items() if k != "PVAL" and np.ndim(v) >= 1}
        _close(one, r32, r64, _gibbs_keys(model), case, exact=("d",))


@pytest.mark.gpu
def test_bayesb_blocked_many_workers_share_rows():
    """BayesB at 10,000 x 1,000 on the blocked family, where many workers share each block of rows: 4 sweeps."""
    bw = pytest.importorskip("bwgr_b200")
    gen, y = synth(10000, 1000, seed=7)
    X = gen.astype(np.float64)
    kw = dict(it=4, bi=1, seed=4, draws="philox")
    r32, r64 = O.gibbs("BayesB", y, X, **kw), O.gibbs("BayesB", y, X, use_double=True, **kw)
    _margins_ok(r32, r64, "gibbs BayesB 10000x1000")
    with bw.Genotypes(gen, path=2) as g:
        out = bw.gibbs_fit("BayesB", y, g, it=4, bi=1, seed=4)
    _close(out, r32, r64, _gibbs_keys("BayesB"), "gibbs BayesB 10000x1000 path 2", exact=("d",))


def _kmup_state(y, p, seed=0):
    rng = np.random.default_rng(seed)
    return rng.normal(size=p) * 0.01, np.ones(p), y - y.mean(), np.full(p, 37.0)


@pytest.mark.gpu
def test_kmup_draw_probe():
    """Disjoint unit columns (n = p, xx = 1), e = 0, b = 0: KMUP's effects are sd z1_j (pi = 0); at pi = 0.999 every marker is
    excluded and takes sd z2_j; at pi = 0.5 both branches occur and d_j = [u_j < q_j].  This isolates the generator from the
    chains: the device's effects agree with the numpy recomputation of the draws to a few ulp."""
    bw = pytest.importorskip("bwgr_b200")
    p = 256
    X = np.eye(p, dtype=np.int8)
    L, Ve = np.full(p, 3.0), 2.0
    sd = np.sqrt(Ve / 4.0)
    z1, z2, u = (v.astype(np.float64) for v in _marker_draws(np.arange(p), 0, 0, SEED_HI))
    for pi in (0.0, 0.5, 0.999):
        kw = dict(seed=SEED_HI, draws="philox")
        r32 = O.kmup(X, np.zeros(p), np.ones(p), np.ones(p), np.zeros(p), L, Ve, pi, **kw)
        r64 = O.kmup(X, np.zeros(p), np.ones(p), np.ones(p), np.zeros(p), L, Ve, pi, use_double=True, **kw)
        _margins_ok(r32, r64, "probe pi %g" % pi)
        out = bw.KMUP(X, np.zeros(p), np.ones(p), np.ones(p), np.zeros(p), L, Ve, pi, seed=SEED_HI)
        d = np.ones(p) if pi == 0 else (u < r64["q"]).astype(np.float64)
        want = np.where(d == 1, sd * z1, sd * z2)
        ulp = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)
        print("REPLAY probe pi %g: max |dev - draws| / ulp = %.1f" % (pi, float((np.abs(out["b"] - want) / ulp).max())))
        assert np.array_equal(out["d"], d), pi
        assert np.all(np.abs(out["b"] - want) <= 8 * ulp), pi
        if pi == 0.5:
            assert 0 < out["d"].sum() < p
        if pi == 0.999:
            assert out["d"].sum() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("store", ["int8", "2bit", "grid", "float32"])
def test_kmup_replay(tpod, store):
    """One KMUP sweep with pi > 0 on each store: d exactly, b and e to the bar."""
    bw = pytest.importorskip("bwgr_b200")
    y, gen = tpod
    X = gen.astype(np.float64)
    if store == "float32":
        X = (X - X.mean(0)).astype(np.float32).astype(np.float64)
    p = X.shape[1]
    b0, d0, e, L = _kmup_state(y, p)
    xx = (X ** 2).sum(0)
    Ve = 0.5 * float(np.var(y))
    kw = dict(seed=31, draws="philox")
    r32 = O.kmup(X, b0, d0, xx, e, L, Ve, 0.5, **kw)
    r64 = O.kmup(X, b0, d0, xx, e, L, Ve, 0.5, use_double=True, **kw)
    _margins_ok(r32, r64, "kmup " + store)
    sk = {"int8": dict(), "2bit": dict(storage=bw.STORE_2BIT), "grid": dict(path=3), "float32": dict(storage=bw.STORE_F32)}[store]
    with bw.Genotypes(X if store == "float32" else gen, **sk) as g:
        out = bw.KMUP(g, b0, d0, xx, e, L, Ve, 0.5, seed=31)
    assert np.array_equal(out["d"], r64["d"])
    _close(out, r32, r64, ("b", "e"), "kmup " + store)


@pytest.mark.gpu
@pytest.mark.parametrize("repeats", [False, True])
def test_kmup2_replay(tpod, repeats):
    """One KMUP2 sweep over a row subset, and over a Use with repeated rows."""
    bw = pytest.importorskip("bwgr_b200")
    y, gen = tpod
    X = gen.astype(np.float64)
    n, p = X.shape
    rng = np.random.default_rng(8)
    use = np.sort(rng.integers(0, n, 150) if repeats else rng.choice(n, 120, replace=False)).astype(np.float64)
    assert (len(np.unique(use)) < use.size) == repeats
    b0, d0, e, L = _kmup_state(y, p)
    xx = (X ** 2).sum(0)
    Ve = 0.5 * float(np.var(y))
    kw = dict(seed=41, draws="philox")
    r32 = O.kmup2(X, use, b0, d0, xx, e, L, Ve, 0.4, **kw)
    r64 = O.kmup2(X, use, b0, d0, xx, e, L, Ve, 0.4, use_double=True, **kw)
    _margins_ok(r32, r64, "kmup2 repeats=%s" % repeats)
    out = bw.KMUP2(gen, use, b0, d0, xx, e, L, Ve, 0.4, seed=41)
    assert np.array_equal(out["d"], r64["d"])
    _close(out, r32, r64, ("b", "e"), "kmup2 repeats=%s" % repeats)


WGR_MODES = {"BRR": dict(), "BayesA": dict(iv=True), "BayesB": dict(iv=True, pi=0.9), "BayesC": dict(pi=0.9), "de": dict(de=True)}


@pytest.mark.gpu
@pytest.mark.parametrize("bag,rp", [(1.0, False), (0.5, False), (0.5, True), (0.45, False)])
@pytest.mark.parametrize("mode", list(WGR_MODES))
def test_wgr_replay(tpod, mode, bag, rp):
    """wgr native (bag = 1) and bagged (bag < 1, rows without / with replacement; 0.45 leaves n * bag fractional): 8 iterations,
    burn-in 2, th = 2."""
    bw = pytest.importorskip("bwgr_b200")
    y, gen = tpod
    X = gen.astype(np.float64)
    kw = dict(it=8, bi=2, th=2, bag=bag, rp=rp, seed=19, **WGR_MODES[mode])
    r32 = O.wgr(y, X, draws="philox", **kw)
    r64 = O.wgr(y, X, draws="philox", use_double=True, **kw)
    case = "wgr %s bag %g rp %s" % (mode, bag, rp)
    _margins_ok(r32, r64, case)
    with bw.Genotypes(gen) as g:
        out = bw.wgr(y, g, **kw)
    keys = ["b", "mu", "Ve", "hat", "Vb"] + (["d"] if WGR_MODES[mode].get("pi", 0) > 0 else [])
    _close(out, r32, r64, keys, case, exact=("d",))
