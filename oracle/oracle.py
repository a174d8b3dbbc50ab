"""ctypes front end of the CPU oracle (oracle/bwgr_oracle.hpp).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's CPU legs.
The product package bwgr_b200 never imports this module.  Function names and returned keys
mirror the reference's R-facing lists (Rcpp20260726ai.cpp:348-353 etc.).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBS = {}

EM_MODELS = {"emRR": 0, "emBA": 1, "emBB": 2, "emBC": 3, "emBL": 4, "emEN": 5, "emDE": 6, "emML": 7, "emBCpi": 8, "lasso": 9}
GIBBS_MODELS = {"BayesRR": 0, "BayesA": 1, "BayesB": 2, "BayesC": 3, "BayesL": 4, "BayesCpi": 5, "BayesDpi": 6}

MRR3_DEFAULTS = dict(
    maxit=500, tol=10e-9, cores=1, TH=False, NLfactor=0.0, InnerGS=False, NoInv=False, HCS=False, XFA=False,
    ACS=False, NumXFA=3, R2=0.5, gc0=0.5, df0=1.0, updateMu=False, weight_prior_h2=0.01, weight_prior_gc=0.01,
    PenCor=0.0, MinCor=1.0, uncorH2below=0.0, roundGCupFrom=1.0, roundGCupTo=1.0, roundGCdownFrom=1.0,
    roundGCdownTo=0.0, bucketGCfrom=1.0, bucketGCto=1.0, DeflateMax=0.9, DeflateBy=0.0, OneVarB=False, OneVarE=False)


def build(native=False):
    target = "native" if native else "all"
    subprocess.check_call(["make", "-s", "-C", _HERE, target])
    return os.path.join(_HERE, "build", "liboracle_native.so" if native else "liboracle.so")


def lib(native=False):
    key = bool(native)
    if key not in _LIBS:
        path = os.path.join(_HERE, "build", "liboracle_native.so" if native else "liboracle.so")
        src_m = max(os.path.getmtime(os.path.join(_HERE, f)) for f in ("bwgr_oracle.hpp", "oracle_capi.cpp"))
        if native or not os.path.exists(path) or os.path.getmtime(path) < src_m:
            path = build(native)
        _LIBS[key] = C.CDLL(path)
    return _LIBS[key]


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def _f32(a):
    return np.asfortranarray(np.asarray(a, dtype=np.float32))


def perm(p, n_iter):
    out = np.empty((n_iter, p), dtype=np.int32)
    lib().orc_perm(C.c_int(p), C.c_int(n_iter), _p(out, C.c_int32))
    return out


def em(model, y, gen, df=10.0, R2=0.5, Pi=0.75, alpha=0.02, it=-1, use_double=False, native=False):
    y = _f32(y)
    X = _f32(gen)
    n, p = X.shape
    mu = C.c_double()
    its = C.c_int()
    b, d, vbv = (np.zeros(p) for _ in range(3))
    hat = np.zeros(n)
    scal = np.zeros(6)
    rc = lib(native).orc_em(C.c_int(EM_MODELS[model]), C.c_int(int(use_double)), _p(y, C.c_float), _p(X, C.c_float),
                            C.c_int(n), C.c_int(p), C.c_float(df), C.c_float(R2), C.c_float(Pi), C.c_float(alpha),
                            C.c_int(it), C.byref(mu), _p(b, C.c_double), _p(d, C.c_double), _p(hat, C.c_double),
                            _p(vbv, C.c_double), _p(scal, C.c_double), C.byref(its))
    assert rc == 0
    Va, Ve, h2, Vg, pi_out, lmb_out = scal
    out = {"mu": mu.value, "b": b, "hat": hat, "its": its.value}
    if model == "emRR":
        out.update(Va=Va, Ve=Ve, h2=h2)
    elif model == "emBA":
        out.update(Vb=vbv, Ve=Ve, h2=h2)
    elif model == "emBB":
        out.update(d=d, Vb=vbv, Ve=Ve, h2=h2)
    elif model == "emBC":
        out.update(d=d, Vg=Vg, Va=Va, Ve=Ve, h2=h2)
    elif model == "emBL":
        out.update(h2=h2)
    elif model == "emEN":
        out.update(Va=Va, Ve=Ve, h2=h2)
    elif model == "emDE":
        out.update(Vb=vbv, Ve=Ve, h2=h2)
    elif model == "emML":
        out.update(h2=h2, Vb=Vg, Va=Va, Ve=Ve)
    elif model == "emBCpi":
        out.update(d=d, pi=pi_out, Vg=Vg, Va=Va, Ve=Ve, h2=h2)
    elif model == "lasso":
        out.update(h2=h2, Lmb=lmb_out)
    return out


def emML_weighted(y, gen, D, it=-1, use_double=False):
    """emML(y, gen, D) with marker weights (Rcpp20260726ai.cpp:463-521, P_WEIGHTS)."""
    y = _f32(y)
    X = _f32(gen)
    n, p = X.shape
    D = np.ascontiguousarray(D, dtype=np.float64)
    mu = C.c_double()
    its = C.c_int()
    b = np.zeros(p)
    hat = np.zeros(n)
    scal = np.zeros(6)
    lib().orc_emml_weighted(C.c_int(int(use_double)), _p(y, C.c_float), _p(X, C.c_float), C.c_int(n), C.c_int(p), _p(D, C.c_double), C.c_int(it),
                            C.byref(mu), _p(b, C.c_double), _p(hat, C.c_double), _p(scal, C.c_double), C.byref(its))
    return {"mu": mu.value, "b": b, "hat": hat, "h2": scal[2], "Vb": scal[3], "Va": scal[0], "Ve": scal[1], "its": its.value}


class _Margins:
    """Decision record of a replay on the device's Philox draws (see orc::PhiloxDraws)."""

    def __init__(self, cap):
        self.q, self.u = np.zeros(cap), np.zeros(cap)
        self.nq, self.mt = C.c_int(), np.zeros(1)
        self.args = (_p(self.q, C.c_double), _p(self.u, C.c_double), C.c_int(cap), C.byref(self.nq), _p(self.mt, C.c_double))

    def add_to(self, out):
        k = self.nq.value
        assert k <= self.q.size
        # q / u: the inclusion probability and the uniform of every accept / reject decision, in the order they were made;
        # margin: the smallest |u - q|; mt_margin: the smallest normalised Marsaglia-Tsang acceptance margin
        out.update(q=self.q[:k].copy(), u=self.u[:k].copy(), margin=float(np.abs(self.u[:k] - self.q[:k]).min()) if k else np.inf,
                   mt_margin=float(self.mt[0]))
        return out


def gibbs(model, y, X, it=1500, bi=500, pi=0.95, df=5.0, R2=0.5, seed=1, draws="mt", chain=0, use_double=False):
    """draws = "mt": the reference's draw order on one std::mt19937_64 stream; "philox": the device's counter-addressed draws of chain
    `chain`, with the decision record of _Margins.  use_double (philox only): the same recipe in float64 on the same float draws."""
    y = _f32(y)
    X = _f32(X)
    n, p = X.shape
    mu = C.c_double()
    b, d, vbv = (np.zeros(p) for _ in range(3))
    hat = np.zeros(n)
    scal = np.zeros(5)
    if draws == "philox":
        m = _Margins(int(it) * p)
        rc = lib().orc_gibbs_philox(C.c_int(GIBBS_MODELS[model]), C.c_int(int(use_double)), C.c_int(chain), _p(y, C.c_float), _p(X, C.c_float),
                                    C.c_int(n), C.c_int(p), C.c_float(it), C.c_float(bi), C.c_float(pi), C.c_float(df), C.c_float(R2),
                                    C.c_uint64(seed), C.byref(mu), _p(b, C.c_double), _p(d, C.c_double), _p(hat, C.c_double),
                                    _p(vbv, C.c_double), _p(scal, C.c_double), *m.args)
    else:
        assert draws == "mt" and chain == 0 and not use_double
        m = None
        rc = lib().orc_gibbs(C.c_int(GIBBS_MODELS[model]), _p(y, C.c_float), _p(X, C.c_float), C.c_int(n), C.c_int(p),
                             C.c_float(it), C.c_float(bi), C.c_float(pi), C.c_float(df), C.c_float(R2),
                             C.c_uint64(seed), C.byref(mu), _p(b, C.c_double), _p(d, C.c_double), _p(hat, C.c_double),
                             _p(vbv, C.c_double), _p(scal, C.c_double))
    assert rc == 0
    vb, ve, h2, MSx, pi_out = scal
    out = {"mu": mu.value, "b": b, "hat": hat, "ve": ve, "h2": h2, "MSx": MSx}
    if m is not None:
        m.add_to(out)
    out["vb"] = vbv if model in ("BayesA", "BayesB", "BayesL", "BayesDpi") else vb
    if model in ("BayesB", "BayesC", "BayesCpi", "BayesDpi"):
        out["d"] = d
    if model in ("BayesCpi", "BayesDpi"):  # these two return pi and PVAL instead of MSx (:914-919, :982-987)
        del out["MSx"]
        out["pi"] = pi_out
        with np.errstate(divide="ignore"):
            out["PVAL"] = -np.log(1.0 - d)
    return out


def _kmup_philox(X, use, b, d, xx, e, L, Ve, pi, seed, use_double):
    """One KMUP (use None) or KMUP2 sweep on the device's Philox draws, in the ratio form the device evaluates."""
    X = _f32(X)
    n, p = X.shape
    b, d, xx, e, L = (np.array(v, dtype=np.float64).ravel() for v in (b, d, xx, e, L))
    if use is not None:
        use = np.array(use, dtype=np.float32).ravel()
    e_out = np.zeros(n if use is None else use.size)
    m = _Margins(p)
    rc = lib().orc_kmup_philox(C.c_int(int(use_double)), _p(X, C.c_float), C.c_int(n), C.c_int(p), None if use is None else _p(use, C.c_float),
                               C.c_int(0 if use is None else use.size), _p(b, C.c_double), _p(d, C.c_double), _p(xx, C.c_double),
                               _p(e, C.c_double), _p(e_out, C.c_double), _p(L, C.c_double), C.c_double(Ve), C.c_double(pi),
                               C.c_uint64(seed), *m.args)
    assert rc == 0
    return m.add_to({"b": b, "d": d, "e": e_out})


def kmup(X, b, d, xx, e, L, Ve, pi, seed=1, ratio_form=False, draws="mt", use_double=False):
    """draws = "philox": the device's draws of a standalone sweep (sweep 0, chain 0), ratio form, use_double as for gibbs()."""
    if draws == "philox":
        return _kmup_philox(X, None, b, d, xx, e, L, Ve, pi, seed, use_double)
    assert draws == "mt" and not use_double
    X = _f32(X)
    n, p = X.shape
    b, d, xx, e, L = (np.array(v, dtype=np.float32) for v in (b, d, xx, e, L))
    lib().orc_kmup(_p(X, C.c_float), C.c_int(n), C.c_int(p), _p(b, C.c_float), _p(d, C.c_float), _p(xx, C.c_float),
                   _p(e, C.c_float), _p(L, C.c_float), C.c_float(Ve), C.c_float(pi), C.c_uint64(seed),
                   C.c_int(int(ratio_form)))
    return {"b": b, "d": d, "e": e}


def kmup2(X, use, b, d, xx, E, L, Ve, pi, seed=1, ratio_form=False, draws="mt", use_double=False):
    """draws = "philox": as kmup()."""
    if draws == "philox":
        return _kmup_philox(X, use, b, d, xx, E, L, Ve, pi, seed, use_double)
    assert draws == "mt" and not use_double
    X = _f32(X)
    n, p = X.shape
    use = np.array(use, dtype=np.float32)
    b, d, xx, E, L = (np.array(v, dtype=np.float32) for v in (b, d, xx, E, L))
    e_out = np.zeros(use.size, dtype=np.float32)
    lib().orc_kmup2(_p(X, C.c_float), C.c_int(n), C.c_int(p), _p(use, C.c_float), C.c_int(use.size), _p(b, C.c_float), _p(d, C.c_float),
                    _p(xx, C.c_float), _p(E, C.c_float), _p(e_out, C.c_float), _p(L, C.c_float), C.c_float(Ve), C.c_float(pi),
                    C.c_uint64(seed), C.c_int(int(ratio_form)))
    return {"b": b, "d": d, "e": e_out}


def gs(which, y, e, gen, b, Lmb, xx, cxx, maxit=50):
    """GSRR / GSFLM (Rcpp20260726ai.cpp:1564-1628)."""
    X = _f32(gen)
    n, p = X.shape
    y, e, b, Lmb, xx = (np.array(v, dtype=np.float32) for v in (y, e, b, Lmb, xx))
    vb = np.zeros(p, dtype=np.float32)
    scal = np.zeros(4)
    lib().orc_gs(C.c_int(0 if which == "GSRR" else 1), _p(y, C.c_float), _p(e, C.c_float), _p(X, C.c_float), C.c_int(n), C.c_int(p),
                 _p(b, C.c_float), _p(Lmb, C.c_float), _p(xx, C.c_float), C.c_float(cxx), C.c_int(maxit), _p(vb, C.c_float), _p(scal, C.c_double))
    return {"mu": scal[0], "b": b, "h2": scal[1], "e": e, "Lmb": Lmb, "vb": vb, "its": int(scal[3])}


def cnt(X):
    X = np.array(_f32(X), order="F")
    lib().orc_cnt_imp(C.c_int(0), _p(X, C.c_float), C.c_int(X.shape[0]), C.c_int(X.shape[1]))
    return X


def imp(X):
    X = np.array(_f32(X), order="F")
    lib().orc_cnt_imp(C.c_int(1), _p(X, C.c_float), C.c_int(X.shape[0]), C.c_int(X.shape[1]))
    return X


def eigk_rank(values, VarK=0.95):
    """pk of R/wgr.R:25: which.max((cumsum(V) / length(V)) > VarK) (1 if the condition never holds)."""
    V = np.asarray(values, dtype=np.float64)
    return int(np.argmax(np.cumsum(V) / V.size > VarK)) + 1


def wgr(y, X, it=1500, bi=500, th=1, iv=False, de=False, pi=0.0, df=5.0, R2=0.5, seed=1, ratio_form=False, bag=1.0, eigK=None, VarK=0.95, rp=False,
        draws="mt", use_double=False):
    """draws = "philox": the device's draws (native or bagged; not eigK), KMUP sweeps in the ratio form; use_double: the KMUP sweeps
    in float64 on the same float draws."""
    y = np.ascontiguousarray(y, dtype=np.float64)
    X = np.asfortranarray(X, dtype=np.float64)
    n, p = X.shape
    b, d, Vb = (np.zeros(p) for _ in range(3))
    hat = np.zeros(n)
    scal = np.zeros(4)
    if draws == "philox":
        assert eigK is None
        m = _Margins(int(it) * p)
        rc = lib().orc_wgr_philox(C.c_int(int(use_double)), _p(y, C.c_double), _p(X, C.c_double), C.c_int(n), C.c_int(p), C.c_int(it), C.c_int(bi),
                                  C.c_int(th), C.c_double(bag), C.c_int(int(rp)), C.c_int(int(iv)), C.c_int(int(de)), C.c_double(pi),
                                  C.c_double(df), C.c_double(R2), C.c_uint64(seed), _p(b, C.c_double), _p(d, C.c_double), _p(Vb, C.c_double),
                                  _p(hat, C.c_double), _p(scal, C.c_double), *m.args)
        assert rc == 0
        mu, Ve, Va, cxx = scal
        return m.add_to({"mu": mu, "b": b, "Vb": Vb if (iv or de) else Va, "d": d, "Ve": Ve, "hat": hat, "cxx": cxx})
    assert draws == "mt" and not use_double
    if eigK is not None:  # R/wgr.R:23-33 (bag == 1)
        assert bag == 1.0
        pk = eigk_rank(eigK["values"], VarK)
        U = np.asfortranarray(np.asarray(eigK["vectors"], dtype=np.float64)[:, :pk])
        V = np.ascontiguousarray(np.asarray(eigK["values"], dtype=np.float64)[:pk])
        u = np.zeros(n)
        scal = np.zeros(5)
        lib().orc_wgr_eigk(_p(y, C.c_double), _p(X, C.c_double), C.c_int(n), C.c_int(p), _p(U, C.c_double), _p(V, C.c_double), C.c_int(pk),
                           C.c_int(it), C.c_int(bi), C.c_int(th), C.c_int(int(iv)), C.c_int(int(de)), C.c_double(pi), C.c_double(df),
                           C.c_double(R2), C.c_uint64(seed), C.c_int(int(ratio_form)), _p(b, C.c_double), _p(d, C.c_double),
                           _p(Vb, C.c_double), _p(hat, C.c_double), _p(u, C.c_double), _p(scal, C.c_double))
        mu, Ve, Va, cxx, Vk = scal
        return {"mu": mu, "b": b, "Vb": Vb if (iv or de) else Va, "d": d, "Ve": Ve, "hat": hat, "u": u, "Vk": Vk, "cxx": cxx}
    if bag != 1.0 and rp:  # R/wgr.R:68, rows drawn with replacement
        lib().orc_wgr_bag_rp(_p(y, C.c_double), _p(X, C.c_double), C.c_int(n), C.c_int(p), C.c_int(it), C.c_int(bi), C.c_int(th),
                             C.c_double(bag), C.c_int(1), C.c_int(int(iv)), C.c_int(int(de)), C.c_double(pi), C.c_double(df), C.c_double(R2),
                             C.c_uint64(seed), C.c_int(int(ratio_form)), _p(b, C.c_double), _p(d, C.c_double), _p(Vb, C.c_double),
                             _p(hat, C.c_double), _p(scal, C.c_double))
        mu, Ve, Va, cxx = scal
        return {"mu": mu, "b": b, "Vb": Vb if (iv or de) else Va, "d": d, "Ve": Ve, "hat": hat, "cxx": cxx}
    if bag != 1.0:
        lib().orc_wgr_bag(_p(y, C.c_double), _p(X, C.c_double), C.c_int(n), C.c_int(p), C.c_int(it), C.c_int(bi), C.c_int(th),
                          C.c_double(bag), C.c_int(int(iv)), C.c_int(int(de)), C.c_double(pi), C.c_double(df), C.c_double(R2),
                          C.c_uint64(seed), C.c_int(int(ratio_form)), _p(b, C.c_double), _p(d, C.c_double), _p(Vb, C.c_double),
                          _p(hat, C.c_double), _p(scal, C.c_double))
        mu, Ve, Va, cxx = scal
        return {"mu": mu, "b": b, "Vb": Vb if (iv or de) else Va, "d": d, "Ve": Ve, "hat": hat, "cxx": cxx}
    lib().orc_wgr(_p(y, C.c_double), _p(X, C.c_double), C.c_int(n), C.c_int(p), C.c_int(it), C.c_int(bi), C.c_int(th),
                  C.c_int(int(iv)), C.c_int(int(de)), C.c_double(pi), C.c_double(df), C.c_double(R2), C.c_uint64(seed),
                  C.c_int(int(ratio_form)), _p(b, C.c_double), _p(d, C.c_double), _p(Vb, C.c_double),
                  _p(hat, C.c_double), _p(scal, C.c_double))
    mu, Ve, Va, cxx = scal
    return {"mu": mu, "b": b, "Vb": Vb if (iv or de) else Va, "d": d, "Ve": Ve, "hat": hat, "cxx": cxx}


def mrr3(Y, X, f32_variant=False, **kw):
    par = dict(MRR3_DEFAULTS)
    for key, v in kw.items():
        if key == "NonLinearFactor":
            key = "NLfactor"
        if key not in par:
            raise TypeError("unknown MRR3 argument %r" % key)
        par[key] = v
    Y = np.asfortranarray(Y, dtype=np.float64)
    X = np.asfortranarray(X, dtype=np.float64)
    n, k = Y.shape
    p = X.shape[1]
    pv = np.array([float(par[name]) for name in MRR3_DEFAULTS], dtype=np.float64)
    maxit = int(par["maxit"])
    mu, h2, ve, MSx = (np.zeros(k) for _ in range(4))
    b = np.zeros((p, k), order="F")
    W = np.zeros((p, k), order="F")
    hat = np.zeros((n, k), order="F")
    GC = np.zeros((k, k), order="F")
    vb = np.zeros((k, k), order="F")
    cnv = np.zeros(3 * maxit)
    its = C.c_int()
    lib().orc_mrr3(C.c_int(int(f32_variant)), _p(Y, C.c_double), _p(X, C.c_double), C.c_int(n), C.c_int(k), C.c_int(p),
                   _p(pv, C.c_double), _p(mu, C.c_double), _p(b, C.c_double), _p(hat, C.c_double), _p(h2, C.c_double),
                   _p(GC, C.c_double), _p(vb, C.c_double), _p(ve, C.c_double), _p(MSx, C.c_double), _p(cnv, C.c_double),
                   _p(W, C.c_double), C.byref(its))
    q = its.value
    return {"mu": mu, "b": b, "hat": hat, "h2": h2, "GC": GC, "vb": vb, "ve": ve, "MSx": MSx, "cnvB": cnv[:q],
            "cnvH2": cnv[maxit:maxit + q], "cnvV": cnv[2 * maxit:2 * maxit + q], "b_Weights": W, "Its": q}

TWO_DESIGN = {"BayesA2": 0, "BayesB2": 1, "BayesRR2": 2, "emML2": 3}


def two_design(model, y, X1, X2, it=1500, bi=500, pi=0.95, df=5.0, R2=0.5, seed=1, D1=None, D2=None):
    """BayesA2 / BayesB2 / BayesRR2 / emML2 (Rcpp20260726ai.cpp:990-1305): y = mu + X1 b1 + X2 b2 + e.  Keys as the reference's lists."""
    y = _f32(y)
    X1, X2 = _f32(X1), _f32(X2)
    n, p1 = X1.shape
    p2 = X2.shape[1]
    b1, d1, vb1 = (np.zeros(p1) for _ in range(3))
    b2, d2, vb2 = (np.zeros(p2) for _ in range(3))
    hat, u1, u2 = (np.zeros(n) for _ in range(3))
    scal = np.zeros(8)
    D1 = None if D1 is None else np.ascontiguousarray(D1, dtype=np.float64)
    D2 = None if D2 is None else np.ascontiguousarray(D2, dtype=np.float64)
    rc = lib().orc_two_design(C.c_int(TWO_DESIGN[model]), _p(y, C.c_float), _p(X1, C.c_float), _p(X2, C.c_float), C.c_int(n), C.c_int(p1),
                  C.c_int(p2), C.c_float(it), C.c_float(bi), C.c_float(pi), C.c_float(df), C.c_float(R2), C.c_uint64(seed),
                  _p(D1, C.c_double) if D1 is not None else None, _p(D2, C.c_double) if D2 is not None else None,
                  _p(b1, C.c_double), _p(b2, C.c_double), _p(d1, C.c_double), _p(d2, C.c_double), _p(vb1, C.c_double),
                  _p(vb2, C.c_double), _p(hat, C.c_double), _p(u1, C.c_double), _p(u2, C.c_double), _p(scal, C.c_double))
    assert rc == 0
    mu, ve, h2, s1, s2, MSx1, MSx2, its = scal
    if model == "emML2":
        return {"mu": mu, "b1": b1, "b2": b2, "Vb1": s1, "Vb2": s2, "Ve": ve, "u1": u1, "u2": u2, "MSx1": MSx1, "MSx2": MSx2, "h2": h2,
                "hat": hat}
    out = {"hat": hat, "mu": mu, "b1": b1, "b2": b2, "vb1": s1 if model == "BayesRR2" else vb1, "vb2": s2 if model == "BayesRR2" else vb2,
           "ve": ve, "h2": h2}
    if model == "BayesB2":
        out["d1"], out["d2"] = d1, d2
    return out
