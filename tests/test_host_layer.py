"""One genotype store serves fits of every kernel family and state shape back to back.

Each fit builds its own state and hands it back when it ends, so nothing a fit leaves on the handle (per-marker variances, block
inverses, Gibbs posterior sums, a row mask, grid accumulators, the wgr driver's state, MRR3's centred columns) may change the next
one: every fit below must give the same bits as the same fit on a new store of the same genotypes."""
import numpy as np
import pytest

from conftest import synth

N, P = 3000, 2000


def _fits(bw):
    """(name, fit(g), path the store is tuned to) in the order they run on the shared store."""
    X, y = synth(N, P, seed=11)
    mask = np.random.default_rng(5).random(N) < 0.8
    Y4 = np.asfortranarray(np.stack([y + 0.3 * np.random.default_rng(t).normal(size=N) for t in range(4)], axis=1))
    return X, [
        ("emBA", lambda g: bw.emBA(y, g, it=8), bw.PATH_AUTO),                                    # per-marker variances, blocked
        ("emRR", lambda g: bw.emRR(y, g, it=8), bw.PATH_AUTO),                                    # block inverses
        ("BayesB", lambda g: bw.BayesB(y, g, it=12, bi=4, seed=3), bw.PATH_AUTO),                 # posterior sums, natural order
        ("emBC masked", lambda g: bw.emBC(y, g, it=8, row_mask=mask), bw.PATH_AUTO),              # small-n family, row mask
        ("emRR grid", lambda g: bw.emRR(y, g, it=8), bw.PATH_GRID),                               # grid family
        ("wgr", lambda g: bw.wgr(y, g, it=12, bi=4, seed=3), bw.PATH_AUTO),                       # wgr driver state
        ("MRR3", lambda g: bw.MRR3(Y4, g, maxit=4), bw.PATH_AUTO),                                # xx_over, sx_dev, cshift
        ("emRR again", lambda g: bw.emRR(y, g, it=8), bw.PATH_AUTO),
    ]


def _same(name, a, b):
    assert a.keys() == b.keys(), name
    for key in a:
        assert np.array_equal(np.asarray(a[key]), np.asarray(b[key]), equal_nan=True), (name, key)


@pytest.mark.gpu
def test_fits_on_one_store_match_fresh_stores():
    bw = pytest.importorskip("bwgr_b200")
    X, fits = _fits(bw)
    with bw.Genotypes(X) as shared:
        for name, fit, path in fits:
            shared.set_tuning(path=path)
            got = fit(shared)
            with bw.Genotypes(X, path=path) as fresh:
                want = fit(fresh)
            _same(name, got, want)
