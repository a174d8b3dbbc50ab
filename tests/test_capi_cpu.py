"""CPU-side checks of the boundary: the shared object loads, exports every symbol include/bwgr_b200.h
declares, and fails loudly (no CPU fallback) when there is no device."""
import os
import re

import pytest

from conftest import ROOT


def _lib():
    from bwgr_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        from bwgr_b200 import build
        build.build()
    return _lib


def test_header_symbols_exported():
    L = _lib()
    hdr = open(os.path.join(ROOT, "include", "bwgr_b200.h")).read()
    declared = sorted(set(re.findall(r"BWGR_API [\w\s\*]*?\b(bwgr_\w+)\(", hdr)))
    assert declared == sorted(L.SYMBOLS)
    cdll = L.load()
    for s in declared:
        assert getattr(cdll, s) is not None
    assert cdll.bwgr_version() >= 100


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import bwgr_b200 as bw
    with pytest.raises(bw.BwgrError) as ei:
        bw.Genotypes()
    assert ei.value.code == -2 and "no CPU path" in str(ei.value)


def test_product_does_not_touch_oracle():
    """The oracle is test infrastructure: nothing under bwgr_b200/ or include/ may reference it."""
    for base in ("bwgr_b200", "include"):
        for dp, _, fs in os.walk(os.path.join(ROOT, base)):
            for f in fs:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                    txt = open(os.path.join(dp, f), errors="ignore").read()
                    assert "oracle" not in txt.lower(), os.path.join(dp, f)


def test_cv_host_logic():
    """emCV / mcmcCV host side (R/cv.R): hold-out sets and the predictive-ability summary, no device involved."""
    import numpy as np
    from bwgr_b200 import api
    hs = api._cv_holdouts(196, k=5, n=3, llo=None, seed=7)
    assert len(hs) == 3 and all(len(w) == 39 and len(set(w.tolist())) == 39 and w.max() < 196 for w in hs)  # round(N/k) rows each
    assert [w.tolist() for w in hs] == [w.tolist() for w in api._cv_holdouts(196, 5, 3, None, 7)]            # seed-reproducible
    lev = np.array(list("aabbbcc"))
    assert [w.tolist() for w in api._cv_holdouts(7, 5, 5, lev, 1)] == [[0, 1], [2, 3, 4], [5, 6]]             # leave-level-out
    assert [w.tolist() for w in api._cv_holdouts(5, 5, 5, np.array(list("zzaaz")), 1)] == [[0, 1, 4], [2, 3]]  # levels in order of appearance
    rng = np.random.default_rng(0)
    obs = rng.normal(size=50)
    M = np.stack([obs + rng.normal(size=50) * s for s in (2.0, 0.1, 0.7)] + [obs], axis=1)
    pooled = api._cv_summary([M[:25], M[25:]], ["m1", "m2", "m3"], avg=True)
    assert list(pooled) == ["m2", "m3", "m1"]                                                                  # sorted, best first
    assert pooled["m2"] == round(float(np.corrcoef(M[:, 1], obs)[0, 1]), 4)
    per = api._cv_summary([M[:25], M[25:]], ["m1", "m2", "m3"], avg=False)
    assert list(per) == ["CV_1", "CV_2"] and per["CV_2"]["m3"] == round(float(np.corrcoef(M[25:, 2], obs[25:])[0, 1]), 4)


@pytest.mark.parametrize("level", [0, 1, 2, -1])
def test_float64_loader_narrowing_paths(level):
    """The loader of R's double matrix (store.cu load_f64_common -> csrc/host_narrow.cpp): every code path (plain, AVX2, AVX-512)
    narrows exact integer codes bit for bit and flags anything else -- fractions, NaN, infinities, out-of-range codes -- wherever in
    the column it sits (vector body or scalar tail)."""
    import ctypes as C

    import numpy as np
    cdll = _lib().load()
    rng = np.random.default_rng(level + 5)

    def run(col, use_shift=0, shift=0.0, lo=-128, hi=127):
        col = np.ascontiguousarray(col, dtype=np.float64)
        out = np.full(col.size, 77, dtype=np.int8)
        mn = C.c_double()
        rc = cdll.bwgr_debug_narrow(col.ctypes.data, col.size, out.ctypes.data, use_shift, float(shift), lo, hi, level, C.byref(mn))
        return rc, out, mn.value

    if run(np.zeros(4))[0] == -1:
        pytest.skip("this CPU lacks the instruction set of level %d" % level)
    for n in (1, 3, 15, 16, 17, 31, 64, 1000, 1003):
        col = rng.integers(-128, 128, size=n).astype(np.float64)
        rc, out, mn = run(col)
        assert rc == 0 and np.array_equal(out, col.astype(np.int8)) and mn == col.min()
        codes = rng.integers(0, 3, size=n)
        rc, out, _ = run(codes, lo=0, hi=2)
        assert rc == 0 and np.array_equal(out, codes.astype(np.int8))
        # centred column: codes + a constant, float32-resolution noise allowed
        shift = -0.73125
        rc, out, _ = run(codes + shift + rng.uniform(-5e-5, 5e-5, size=n), use_shift=1, shift=shift, lo=0, hi=2)
        assert rc == 0 and np.array_equal(out, codes.astype(np.int8))
        for bad in (0.5, np.nan, np.inf, -np.inf, 128.0, -129.0, 3e9, 1e300, 1.0000001):
            for pos in {0, n // 2, n - 1}:
                c2 = col.copy()
                c2[pos] = bad
                assert run(c2)[0] == 1, (n, bad, pos)
                if bad != 1.0000001:
                    c3 = codes.astype(np.float64) + shift
                    c3[pos] = bad
                    assert run(c3, use_shift=1, shift=shift, lo=0, hi=2)[0] == 1, (n, bad, pos, "shifted")
        c2 = codes.astype(np.float64)
        c2[n // 2] = 3.0
        assert run(c2, lo=0, hi=2)[0] == 1
