"""Host-side mirror of the reference's R-facing functions for the marker-effect update loop.

Same names, argument names/defaults and returned list keys as the reference's exports
(R/RcppExports.R:12-65, :180; R/wgr.R:2-8), implemented over the C ABI of include/bwgr_b200.h.
`gen` / `X` may be a numpy matrix (float or int8, n x p) or an already loaded `Genotypes` store,
which removes the per-call n x p conversion the reference pays (src/RcppExports.cpp:115-116).
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import EmOut, EmParams, GibbsOut, GibbsParams, GibbsSysParams, check

STORE_I8, STORE_2BIT, STORE_F32 = 0, 1, 2
PATH_AUTO, PATH_SMALL_N, PATH_BLOCKED, PATH_GRID = 0, 1, 2, 3
_EM = {"emRR": 0, "emBA": 1, "emBB": 2, "emBC": 3, "emBL": 4, "emEN": 5, "emDE": 6, "emML": 7, "emBCpi": 8, "lasso": 9}
_GIBBS = {"BayesRR": 0, "BayesA": 1, "BayesB": 2, "BayesC": 3, "BayesL": 4, "BayesCpi": 5, "BayesDpi": 6}
NSCAL = 6  # BWGR_NSCAL of include/bwgr_b200.h


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _need(cond, what):
    """The C ABI takes plain pointers and reads g.n / g.p elements from them: a short vector must be an error here, not a
    host out-of-bounds read there (BWGR_ERR_ARG, like the C side's own argument checks)."""
    if not cond:
        raise _lib.BwgrError(-1, what)


class Genotypes:
    """Genotype matrix resident in HBM (int8 column-major or 2-bit packed) behind one bwgr_handle."""

    def __init__(self, X=None, storage=STORE_I8, device=0, path=PATH_AUTO, grid=0, centred_ok=False):
        self.lib = _lib.load()
        h = C.c_void_p()
        check(self.lib.bwgr_create(device, C.byref(h)))
        self.h = h
        self.n = self.p = 0
        check(self.lib.bwgr_set_tuning(self.h, -1, path, grid))
        if X is not None:
            self.load(X, storage, centred_ok=centred_ok)

    def load(self, X, storage=STORE_I8, centred_ok=False):
        if hasattr(X, "data_ptr"):  # torch tensor
            import torch
            assert X.dtype == torch.int8 and X.dim() == 2
            # torch is row-major: a (p, n) contiguous tensor is the column-major n x p matrix
            p, n = X.shape
            assert X.is_contiguous()
            fn = self.lib.bwgr_geno_load_i8_device if X.is_cuda else self.lib.bwgr_geno_load_i8
            if X.is_cuda:  # the handle copies on its own non-blocking stream: the kernels that produced X must have finished
                torch.cuda.current_stream(X.device).synchronize()
            check(fn(self.h, C.c_void_p(X.data_ptr()), n, p, n, storage))
        else:
            X = np.asarray(X)
            n, p = X.shape
            if X.dtype == np.int8:
                Xf = np.asfortranarray(X)
                check(self.lib.bwgr_geno_load_i8(self.h, _ptr(Xf), n, p, n, storage))
            else:
                Xf = np.asfortranarray(X, dtype=np.float64)
                fn = self.lib.bwgr_geno_load_f64_centred if centred_ok else self.lib.bwgr_geno_load_f64
                try:
                    check(fn(self.h, _ptr(Xf), n, p, n, storage))
                except _lib.BwgrError as err:
                    # real-valued genotypes (NA cells imputed with column means, R/wgr.R:13-19; IMP() / CNT() output): the float32
                    # store, the type the reference itself computes in -- served by the grid family
                    if err.code != -1 or storage != STORE_I8 or "non-integer" not in str(err):
                        raise
                    check(self.lib.bwgr_geno_load_f64(self.h, _ptr(Xf), n, p, n, STORE_F32))
        self.n, self.p = int(n), int(p)
        return self

    def load_bed(self, prefix, storage=STORE_I8, missing=-1):
        """PLINK binary fileset `prefix`.bed / .bim / .fam -> store (additive count of allele A1).  missing: see bwgr_geno_load_bed.
        Returns the number of missing calls met."""
        def lines(path):
            with open(path, "rb") as f:
                return sum(1 for _ in f)
        n, p = lines(prefix + ".fam"), lines(prefix + ".bim")
        nm = C.c_int64()
        check(self.lib.bwgr_geno_load_bed(self.h, (prefix + ".bed").encode(), n, p, storage, int(missing), C.byref(nm)))
        self.n, self.p = int(n), int(p)
        return int(nm.value)

    def enable_row_sharding(self, group=None):
        """One large fit sharded by rows over the ranks of a torch.distributed group (one process per GPU of a node):
        call before load(); every rank then loads ITS rows and passes ITS rows of y to the usual fit functions.
        The host framework only carries 128 + 64 bytes per rank here (NCCL id, IPC handle of the exchange ring)."""
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        uid = np.zeros(128, dtype=np.uint8)
        if rank == 0:
            check(self.lib.bwgr_dist_unique_id(_ptr(uid)))
        box = [uid.tobytes()]
        dist.broadcast_object_list(box, src=0, group=group)
        uid = np.frombuffer(box[0], dtype=np.uint8).copy()
        ipc = np.zeros(64, dtype=np.uint8)
        check(self.lib.bwgr_dist_init(self.h, rank, world, _ptr(uid), _ptr(ipc)))
        allh = [None] * world
        dist.all_gather_object(allh, ipc.tobytes(), group=group)
        blob = np.frombuffer(b"".join(allh), dtype=np.uint8).copy()
        check(self.lib.bwgr_dist_connect(self.h, _ptr(blob)))
        self.rank, self.world = rank, world
        return self

    def set_tuning(self, block=-1, path=-1, grid=-1):
        check(self.lib.bwgr_set_tuning(self.h, block, path, grid))

    def set_stream(self, stream_ptr):
        check(self.lib.bwgr_set_stream(self.h, C.c_void_p(stream_ptr)))

    def info(self):
        n, p, ldb, tot = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
        st = C.c_int()
        check(self.lib.bwgr_geno_info(self.h, C.byref(n), C.byref(p), C.byref(ldb), C.byref(st), C.byref(tot)))
        return {"n": n.value, "p": p.value, "ld_bytes": ldb.value, "storage": st.value, "total_bytes": tot.value}

    def unpack(self):
        out = np.empty((self.n, self.p), dtype=np.int8, order="F")
        check(self.lib.bwgr_geno_unpack_i8(self.h, _ptr(out)))
        return out

    def raw(self):
        out = np.empty(self.info()["total_bytes"], dtype=np.uint8)
        check(self.lib.bwgr_geno_raw(self.h, _ptr(out)))
        return out

    def stats(self):
        xx, sx = np.empty(self.p), np.empty(self.p)
        check(self.lib.bwgr_geno_stats(self.h, _ptr(xx), _ptr(sx)))
        return xx, sx

    def fitted(self, b, mu=0.0):
        """mu + X b on the store: b is p (bwgr_fitted) or p x k with mu a scalar or k values (bwgr_fitted_sys: k systems, one pass
        over the store, hat n x k)."""
        b = np.asarray(b, dtype=np.float64)
        if b.ndim == 1:
            b = np.ascontiguousarray(b)
            _need(b.size == self.p, "b must have p = %d values" % self.p)
            hat = np.empty(self.n)
            check(self.lib.bwgr_fitted(self.h, _ptr(b), float(mu), _ptr(hat)))
            return hat
        _need(b.ndim == 2 and b.shape[0] == self.p and b.shape[1] >= 1, "b must be p x k with p = %d" % self.p)
        B = np.asfortranarray(b)
        k = B.shape[1]
        m = np.ascontiguousarray(np.broadcast_to(np.asarray(mu, dtype=np.float64), (k,)))
        hat = np.empty((self.n, k), order="F")
        check(self.lib.bwgr_fitted_sys(self.h, k, _ptr(B), _ptr(m), _ptr(hat)))
        return hat

    def gram_blocks(self, perm, block=128):
        perm = np.ascontiguousarray(perm, dtype=np.int32)
        nb = (self.p + block - 1) // block
        out = np.empty((nb, block, block), dtype=np.int32)
        check(self.lib.bwgr_debug_gram(self.h, _ptr(perm), block, _ptr(out)))
        return out

    def gram_band(self, perm):
        """The Gram band the pipelined sweep consumes ([nblocks][128][256] floats) from the same dispatch as a fit; returns (band, kind)
        with kind 4 = FP4 path, 8 = E4M3 / int8 path."""
        perm = np.ascontiguousarray(perm, dtype=np.int32)
        nb = (self.p + 127) // 128
        out = np.empty((nb, 128, 256), dtype=np.float32)
        kind = C.c_int()
        check(self.lib.bwgr_debug_gram_band(self.h, _ptr(perm), _ptr(out), C.byref(kind)))
        return out, kind.value

    def profile(self, enable=True):
        check(self.lib.bwgr_profile(self.h, int(enable)))

    def profile_read(self):
        ms = np.zeros(4)
        cnt = np.zeros(4, dtype=np.int64)
        check(self.lib.bwgr_profile_read(self.h, _ptr(ms), _ptr(cnt)))
        return {k: {"ms": float(ms[i]), "launches": int(cnt[i])} for i, k in enumerate(("gram", "sweep", "epilogue", "block_inverse"))}

    def launch_count(self):
        return int(self.lib.bwgr_launch_count(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.lib.bwgr_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def trim():
    """Return the device / pinned blocks kept from closed stores and fits to the driver (bwgr_trim)."""
    _lib.load().bwgr_trim()


def _store(gen, **kw):
    if isinstance(gen, Genotypes):
        if gen.p == 0:  # same status and text as the C ABI gives for a call before bwgr_geno_load_*
            raise _lib.BwgrError(-3, "no genotypes loaded")
        return gen, False
    return Genotypes(gen, **kw), True


class _EmBuffers:
    def __init__(self, n, p, nsys):
        self.mu = np.zeros(nsys)
        self.b = np.zeros((p, nsys), order="F")
        self.d = np.zeros((p, nsys), order="F")
        self.hat = np.zeros((n, nsys), order="F")
        self.vb = np.zeros((p, nsys), order="F")
        self.scal = np.zeros((NSCAL, nsys), order="F")
        self.its = np.zeros(nsys, dtype=np.int32)
        self.c = EmOut(_ptr(self.mu), _ptr(self.b), _ptr(self.d), _ptr(self.hat), _ptr(self.vb), _ptr(self.scal),
                       _ptr(self.its))

    def result(self, model, squeeze):
        def v(a):
            return a[:, 0].copy() if squeeze else a

        def s(a):
            return float(a[0]) if squeeze else a.copy()

        Va, Ve, h2, Vg, pi_out, lmb_out = (self.scal[i] for i in range(NSCAL))
        out = {"mu": s(self.mu), "b": v(self.b), "hat": v(self.hat)}
        if model == "emRR":
            out.update(Va=s(Va), Ve=s(Ve), h2=s(h2))
        elif model == "emBA":
            out.update(Vb=v(self.vb), Ve=s(Ve), h2=s(h2))
        elif model == "emBB":
            out.update(d=v(self.d), Vb=v(self.vb), Ve=s(Ve), h2=s(h2))
        elif model == "emBC":
            out.update(d=v(self.d), Vg=s(Vg), Va=s(Va), Ve=s(Ve), h2=s(h2))
        elif model == "emBL":
            out.update(h2=s(h2))
        elif model == "emEN":
            out.update(Va=s(Va), Ve=s(Ve), h2=s(h2))
        elif model == "emDE":  # Rcpp20260726ai.cpp:300-305
            out.update(Vb=v(self.vb), Ve=s(Ve), h2=s(h2))
        elif model == "emML":  # :513-519
            out.update(h2=s(h2), Vb=s(Vg), Va=s(Va), Ve=s(Ve))
        elif model == "emBCpi":  # :1541-1545
            out.update(d=v(self.d), pi=s(pi_out), Vg=s(Vg), Va=s(Va), Ve=s(Ve), h2=s(h2))
        elif model == "lasso":  # :1495-1497
            out.update(h2=s(h2), Lmb=s(lmb_out))
        out["its"] = int(self.its[0]) if squeeze else self.its.copy()
        return out


def _em_params(model, y, nsys, it, df, R2, Pi, alpha, row_mask, n, weights=None):
    mask = None
    if row_mask is not None:
        mask = np.asfortranarray(np.asarray(row_mask).reshape(n, nsys, order="F") != 0, dtype=np.uint8)
    par = EmParams(_EM[model], nsys, it, df, R2, Pi, alpha, _ptr(mask), _ptr(weights))
    return par, (mask, weights)


def em_fit(model, y, gen, df=10.0, R2=0.5, Pi=0.75, alpha=0.02, it=-1, row_mask=None, weights=None, **store_kw):
    """Generic entry: y is n (one fit) or n x k (k independent fits sharing gen)."""
    g, own = _store(gen, **store_kw)
    try:
        y = np.asarray(y, dtype=np.float64)
        squeeze = y.ndim == 1
        Y = np.asfortranarray(y.reshape(g.n, -1, order="F"))
        nsys = Y.shape[1]
        if weights is not None:
            weights = np.ascontiguousarray(weights, dtype=np.float64)
            _need(weights.size == g.p, "marker weights must have p = %d values" % g.p)
        par, mask = _em_params(model, Y, nsys, it, df, R2, Pi, alpha, row_mask, g.n, weights)
        buf = _EmBuffers(g.n, g.p, nsys)
        check(g.lib.bwgr_em_fit(g.h, C.byref(par), _ptr(Y), C.byref(buf.c)))
        del mask
        return buf.result(model, squeeze)
    finally:
        if own:
            g.close()


class EmStepper:
    """begin / sweeps / end split of one EM fit, for timing sweeps with everything resident."""

    def __init__(self, model, y, gen, df=10.0, R2=0.5, Pi=0.75, alpha=0.02):
        self.g = gen
        self.model = model
        y = np.asarray(y, dtype=np.float64)
        self.squeeze = y.ndim == 1
        self.Y = np.asfortranarray(y.reshape(gen.n, -1, order="F"))
        self.par, self._mask = _em_params(model, self.Y, self.Y.shape[1], -1, df, R2, Pi, alpha, None, gen.n)
        check(gen.lib.bwgr_em_begin(gen.h, C.byref(self.par), _ptr(self.Y)))

    def sweeps(self, k=1):
        check(self.g.lib.bwgr_em_sweeps(self.g.h, k))

    def end(self):
        buf = _EmBuffers(self.g.n, self.g.p, self.Y.shape[1])
        check(self.g.lib.bwgr_em_end(self.g.h, C.byref(buf.c)))
        return buf.result(self.model, self.squeeze)


def emRR(y, gen, df=10, R2=0.5, **kw):
    return em_fit("emRR", y, gen, df=df, R2=R2, **kw)


def emBA(y, gen, df=10, R2=0.5, **kw):
    return em_fit("emBA", y, gen, df=df, R2=R2, **kw)


def emBB(y, gen, df=10, R2=0.5, Pi=0.75, **kw):
    return em_fit("emBB", y, gen, df=df, R2=R2, Pi=Pi, **kw)


def emBC(y, gen, df=10, R2=0.5, Pi=0.75, **kw):
    return em_fit("emBC", y, gen, df=df, R2=R2, Pi=Pi, **kw)


def emBL(y, gen, R2=0.5, alpha=0.02, **kw):
    return em_fit("emBL", y, gen, R2=R2, alpha=alpha, **kw)


def emEN(y, gen, R2=0.5, alpha=0.02, **kw):
    return em_fit("emEN", y, gen, R2=R2, alpha=alpha, **kw)


def emDE(y, gen, R2=0.5, **kw):
    return em_fit("emDE", y, gen, R2=R2, **kw)


def emML(y, gen, D=None, **kw):
    """emML(y, gen, D = NULL) (Rcpp20260726ai.cpp:463-521); D = optional marker weights: the penalty of marker j is Lmb / D[j] (:495)."""
    return em_fit("emML", y, gen, weights=D, **kw)


def emBCpi(y, gen, df=10, R2=0.5, Pi=0.75, **kw):
    return em_fit("emBCpi", y, gen, df=df, R2=R2, Pi=Pi, **kw)


def lasso(y, gen, **kw):
    return em_fit("lasso", y, gen, **kw)


def gibbs_fit(model, y, X, it=1500, bi=500, pi=0.95, df=5.0, R2=0.5, seed=1, nchains=1, row_mask=None, chain0=0, **store_kw):
    """Generic entry of the seven samplers.  y is n (one trait) or n x k (k traits / CV folds sharing X, one call); row_mask (n x k, like
    em_fit's) fits column t on the rows it keeps.  Column t runs `nchains` chains: system s = t * nchains + c draws from Philox chain
    chain0 + s.  A 1-D y without a mask returns what the single-trait call returns (a trailing chain axis when nchains > 1); an n x k y
    returns arrays with a trailing system axis of k * nchains, and hat covers every row, the ones a mask leaves out included."""
    g, own = _store(X, **store_kw)
    try:
        y = np.asarray(y, dtype=np.float64)
        _need(y.ndim in (1, 2) and y.shape[0] == g.n and y.size % g.n == 0, "y has %d rows, the genotype store %d" % (y.shape[0], g.n))
        Y = np.asfortranarray(y.reshape(g.n, -1, order="F"))
        k = Y.shape[1]
        nc = max(1, int(nchains))
        ns = k * nc
        mask = None
        if row_mask is not None:
            mask = np.asfortranarray(np.asarray(row_mask).reshape(g.n, k, order="F") != 0, dtype=np.uint8)
        mu = np.zeros(ns)
        b = np.zeros((g.p, ns), order="F")
        d = np.zeros((g.p, ns), order="F")
        hat = np.zeros((g.n, ns), order="F")
        vb = np.zeros((g.p, ns), order="F")
        scal = np.zeros((NSCAL, ns), order="F")
        par = GibbsSysParams(GibbsParams(_GIBBS[model], nc, int(it), int(bi), pi, df, R2, seed), k, _ptr(mask), int(chain0))
        out = GibbsOut(_ptr(mu), _ptr(b), _ptr(d), _ptr(hat), _ptr(vb), _ptr(scal))
        check(g.lib.bwgr_gibbs_fit_sys(g.h, C.byref(par), _ptr(Y), C.byref(out)))
        sq = ns == 1 and y.ndim == 1

        def v(a):
            return a[:, 0].copy() if sq else a

        res = {"mu": float(mu[0]) if sq else mu, "b": v(b), "hat": v(hat),
               "ve": float(scal[1, 0]) if sq else scal[1].copy(), "h2": float(scal[2, 0]) if sq else scal[2].copy(),
               "MSx": float(scal[3, 0]) if sq else scal[3].copy()}
        if model in ("BayesA", "BayesB", "BayesL", "BayesDpi"):
            res["vb"] = v(vb)
        else:
            res["vb"] = float(scal[0, 0]) if sq else scal[0].copy()
        if model in ("BayesB", "BayesC", "BayesCpi", "BayesDpi"):
            res["d"] = v(d)
        if model in ("BayesCpi", "BayesDpi"):  # these two return pi and PVAL = -log(1 - D) in place of MSx (:914-919, :982-987)
            del res["MSx"]
            res["pi"] = float(scal[4, 0]) if sq else scal[4].copy()
            with np.errstate(divide="ignore"):
                res["PVAL"] = -np.log(1.0 - res["d"])
        return res
    finally:
        if own:
            g.close()


def BayesRR(y, X, it=1500, bi=500, df=5, R2=0.5, **kw):
    return gibbs_fit("BayesRR", y, X, it=it, bi=bi, df=df, R2=R2, **kw)


def BayesA(y, X, it=1500, bi=500, df=5, R2=0.5, **kw):
    return gibbs_fit("BayesA", y, X, it=it, bi=bi, df=df, R2=R2, **kw)


def BayesB(y, X, it=1500, bi=500, pi=0.95, df=5, R2=0.5, **kw):
    return gibbs_fit("BayesB", y, X, it=it, bi=bi, pi=pi, df=df, R2=R2, **kw)


def BayesC(y, X, it=1500, bi=500, pi=0.95, df=5, R2=0.5, **kw):
    return gibbs_fit("BayesC", y, X, it=it, bi=bi, pi=pi, df=df, R2=R2, **kw)


def BayesL(y, X, it=1500, bi=500, df=5, R2=0.5, **kw):
    return gibbs_fit("BayesL", y, X, it=it, bi=bi, df=df, R2=R2, **kw)


def BayesCpi(y, X, it=1500, bi=500, df=5, R2=0.5, **kw):
    return gibbs_fit("BayesCpi", y, X, it=it, bi=bi, df=df, R2=R2, **kw)


def BayesDpi(y, X, it=1500, bi=500, df=5, R2=0.5, **kw):
    return gibbs_fit("BayesDpi", y, X, it=it, bi=bi, df=df, R2=R2, **kw)


def KMUP(X, b, d, xx, e, L, Ve, pi, seed=1, **store_kw):
    """One Kuo-Mallick sweep, drop-in for KMUP(X,b,d,xx,e,L,Ve,pi) (Rcpp20260726ai.cpp:12-38): returns (b, d, e)
    like the reference's list.  X: matrix or Genotypes store."""
    g, own = _store(X, **store_kw)
    try:
        b, d, xx, e, L = (np.array(v, dtype=np.float64) for v in (b, d, xx, e, L))
        _need(b.size == g.p and d.size == g.p and xx.size == g.p and L.size == g.p, "KMUP: b, d, xx, L must have p = %d values" % g.p)
        _need(e.size == g.n, "KMUP: e must have n = %d values" % g.n)
        check(g.lib.bwgr_kmup_sweep(g.h, _ptr(b), _ptr(d), _ptr(xx), _ptr(e), _ptr(L), float(Ve), float(pi), int(seed)))
        return {"b": b, "d": d, "e": e}
    finally:
        if own:
            g.close()


def KMUP2(X, Use, b, d, xx, E, L, Ve, pi, seed=1, **store_kw):
    """The bagged Kuo-Mallick sweep, drop-in for KMUP2(X,Use,b,d,xx,E,L,Ve,pi) (Rcpp20260726ai.cpp:41-77): Use = 0-based rows; a row
    named more than once (sampling with replacement) counts once per occurrence in the dot products, as in the reference's H / e0.
    Returns (b, d, e) with e the residuals of the rows in use in the order of Use, like the reference's list."""
    g, own = _store(X, **store_kw)
    try:
        Use = np.array(Use, dtype=np.float64).ravel()
        b, d, xx, E, L = (np.array(v, dtype=np.float64) for v in (b, d, xx, E, L))
        _need(b.size == g.p and d.size == g.p and xx.size == g.p and L.size == g.p, "KMUP2: b, d, xx, L must have p = %d values" % g.p)
        _need(E.size == g.n, "KMUP2: E must have n = %d values" % g.n)
        _need(Use.size >= 2, "KMUP2: Use must name at least 2 rows")
        e = np.zeros(Use.size)
        check(g.lib.bwgr_kmup2_sweep(g.h, _ptr(Use), int(Use.size), _ptr(b), _ptr(d), _ptr(xx), _ptr(E), _ptr(e), _ptr(L), float(Ve),
                                     float(pi), int(seed)))
        return {"b": b, "d": d, "e": e}
    finally:
        if own:
            g.close()


def _gs(which, y, e, gen, b, Lmb, xx, cxx, maxit, **store_kw):
    g, own = _store(gen, **store_kw)
    try:
        y, e, b, Lmb, xx = (np.array(v, dtype=np.float64) for v in (y, e, b, Lmb, xx))
        _need(y.size == g.n and e.size == g.n, "GSRR / GSFLM: y and e must have n = %d values" % g.n)
        _need(b.size == g.p and Lmb.size == g.p and xx.size == g.p, "GSRR / GSFLM: b, Lmb, xx must have p = %d values" % g.p)
        vb = np.zeros(g.p)
        scal = np.zeros(4)
        check(g.lib.bwgr_gs_fit(g.h, which, _ptr(y), _ptr(e), _ptr(b), _ptr(Lmb), _ptr(xx), float(cxx), int(maxit), _ptr(vb), _ptr(scal)))
        return {"mu": float(scal[0]), "b": b, "h2": float(scal[1]), "e": e, "Lmb": Lmb, "vb": vb, "its": int(scal[3])}
    finally:
        if own:
            g.close()


def GSRR(y, e, gen, b, Lmb, xx, cxx, maxit=50, **kw):
    """GSRR(y, e, gen, b, Lmb, xx, cxx, maxit = 50) (Rcpp20260726ai.cpp:1597-1628): same arguments, same list (mu, b, h2, e, Lmb, vb)."""
    return _gs(0, y, e, gen, b, Lmb, xx, cxx, maxit, **kw)


def GSFLM(y, e, gen, b, Lmb, xx, cxx, maxit=50, **kw):
    """GSFLM(y, e, gen, b, Lmb, xx, cxx, maxit = 50) (Rcpp20260726ai.cpp:1564-1594)."""
    return _gs(1, y, e, gen, b, Lmb, xx, cxx, maxit, **kw)


def wgr(y, X, it=1500, bi=500, th=1, bag=1, rp=False, iv=False, de=False, pi=0, df=5, R2=0.5, eigK=None, VarK=0.95,
        verb=False, seed=1, **store_kw):
    """wgr() of R/wgr.R:2-8 with the MCMC loop native (one C call instead of `it` KMUP round trips).
    Model map (man/wgr.Rd:185): BRR pi=0,iv=F; BayesA iv=T; BayesB pi>0,iv=T; BayesC pi>0,iv=F; BayesL de=T."""
    # R/wgr.R:11-19, :35-40: missing genotypes take their column mean (the float32 store serves real-valued genotypes); individuals
    # without a phenotype leave the fit and keep their fitted value
    gen0 = None
    if not isinstance(X, Genotypes) and not hasattr(X, "data_ptr"):
        X = np.asarray(X)
        if X.dtype.kind == "f" and np.isnan(X).any():
            X = np.array(X, dtype=np.float64)
            cm = np.nan_to_num(np.nanmean(X, axis=0), nan=0.0)  # x[is.nan(x)] = 0: an all-missing column
            X[np.isnan(X)] = np.broadcast_to(cm, X.shape)[np.isnan(X)]
        y = np.asarray(y, dtype=np.float64)
        if np.isnan(y).any():
            gen0, keep = X, ~np.isnan(y)
            X, y = X[keep], y[keep]
            if eigK is not None:
                eigK = {"values": eigK["values"], "vectors": np.asarray(eigK["vectors"])[keep], "vectors0": np.asarray(eigK["vectors"])}
    if eigK is not None:
        out = _wgr_eigk(y, X, eigK, VarK, it, bi, th, bag, iv, de, pi, df, R2, seed, store_kw)
    else:
        out = _wgr_native(y, X, it, bi, th, bag, rp, iv, de, pi, df, R2, seed, store_kw)
    if gen0 is not None:  # :143-150: HAT = B0 + gen0 %*% B (+ U0 %*% H)
        out["hat"] = out["mu"] + np.asarray(gen0, dtype=np.float64) @ out["b"]
        if eigK is not None:
            out["hat"] = out["hat"] + out["u"]
    return out


def _wgr_eigk(y, X, eigK, VarK, it, bi, th, bag, iv, de, pi, df, R2, seed, store_kw):
    """wgr with the polygenic term (R/wgr.R:23-33, :74-84, :116-119, :124, :145-150): the reference's own R loop, one Kuo-Mallick sweep
    over the leading eigenvectors of the kernel (real-valued: the float32 store) and one over the markers per iteration, both on the
    device through the KMUP entry point; the variance draws of the driver on the host, like R's.  bag must be 1: with bag != 1 the
    reference hands KMUP2's residual of the rows in use back to KMUP2 as the full residual (:81-87) and reads out of bounds."""
    if bag != 1:
        raise _lib.BwgrError(-5, "wgr: eigK with bag != 1 reads out of bounds in the reference (R/wgr.R:81-87); not reproduced")
    if de:
        iv = True
    V = np.asarray(eigK["values"], dtype=np.float64)
    vec = np.asarray(eigK["vectors"], dtype=np.float64)
    pk = int(np.argmax(np.cumsum(V) / V.size > VarK)) + 1  # which.max(cumsum(V) / length(V) > VarK)
    U = np.asfortranarray(vec[:, :pk])
    U0 = np.asarray(eigK.get("vectors0", vec), dtype=np.float64)[:, :pk]
    V = V[:pk]
    y = np.ascontiguousarray(y, dtype=np.float64)
    g, own = _store(X, **store_kw)
    gu = Genotypes(device=store_kw.get("device", 0))
    try:
        _need(y.size == g.n and U.shape[0] == g.n, "y has %d values, eigK$vectors %d rows, the genotype store %d rows" % (y.size, U.shape[0], g.n))
        check(gu.lib.bwgr_geno_load_f64(gu.h, _ptr(U), g.n, pk, g.n, STORE_F32))
        gu.n, gu.p = g.n, pk
        n, p = g.n, g.p
        rng = np.random.default_rng(seed)
        xxi, sxi = g.stats()
        xx = np.asarray(xxi, dtype=np.float64)
        MSx = float(((xx - np.asarray(sxi, dtype=np.float64) ** 2 / n) / (n - 1)).sum())  # sum(apply(X, 2, var))
        post = set(range(bi, it + 1, th))  # seq(bi, it, th)
        mc = len(post)
        b, d, h = np.zeros(p), np.ones(p), np.zeros(pk)
        mu = float(y.mean())
        e = y - mu
        Va, Ve = MSx, 1.0
        Vb = np.full(p, Va)
        Vk = np.ones(pk)
        L = Vb / Ve  # sic (:55)
        vy = float(y.var(ddof=1))
        Sb, Se, Sk = R2 * df * vy / MSx, (1 - R2) * df * vy, R2 * vy * (df + 2)
        xxK = np.full(pk, float(bag))
        B0 = VA = VE = VP = 0.0
        VB, D, B, H = np.zeros(p), np.zeros(p), np.zeros(p), np.zeros(pk)
        Vp = 0.0
        for i in range(1, it + 1):
            s = int(rng.integers(1, 2 ** 62))
            up = KMUP(gu, h, np.zeros(pk), xxK, e, Ve / (V * Vk), Ve, 0, seed=s)
            h, e = up["b"], up["e"]
            up = KMUP(g, b, d, xx, e, L, Ve, pi, seed=s + 1)
            if pi > 0:
                d = up["d"]
            b, e = up["b"], up["e"]
            if iv:
                Vb = np.sqrt(b * b * Ve / MSx) if de else (Sb + b * b) / rng.chisquare(df + 1, size=p)
            else:
                Va = float((b @ b + Sb) / rng.chisquare(df + p))
                Vb = np.full(p, Va)
            Vp = float(((h * h / V).sum() + Sk) / rng.chisquare(df + pk))
            Vk = np.full(pk, Vp)
            Ve = float((e @ e + Se) / rng.chisquare(n * bag + df))
            L = Ve / Vb
            e = y - g.fitted(b, mu) - U @ h  # :124 (e = y - mu - X b - U h)
            mu0 = rng.normal(e.mean(), Ve / n)  # sic: the sd argument is Ve / n (:125)
            mu += mu0
            e = e - mu0
            if i in post:
                B0 += mu; B += b; D += d; VE += Ve; H += h; VP += Vp
                if iv:
                    VB += Vb
                else:
                    VA += Va
        B0 /= mc; D /= mc; B = B / mc / D.mean(); VE /= mc; H /= mc; VP /= mc
        poly = U0 @ H
        hat = g.fitted(B, B0) + U @ H  # B0 + gen0 %*% B + U0 %*% H on the rows of the fit
        return {"mu": B0, "b": B, "Vb": VB / mc if iv else VA / mc, "d": D, "Ve": VE, "hat": hat, "u": poly, "Vk": VP, "cxx": float(xx.mean() * bag)}
    finally:
        gu.close()
        if own:
            g.close()


def _wgr_native(y, X, it, bi, th, bag, rp, iv, de, pi, df, R2, seed, store_kw):
    g, own = _store(X, **store_kw)
    try:
        y = np.ascontiguousarray(y, dtype=np.float64)
        _need(y.size == g.n, "y has %d values, the genotype store %d rows" % (y.size, g.n))
        b, d, Vb = (np.zeros(g.p) for _ in range(3))
        hat = np.zeros(g.n)
        scal = np.zeros(4)
        if bag != 1:  # R/wgr.R:21, :68, :87: a fresh row sample per iteration, swept by KMUP2
            check(g.lib.bwgr_wgr_fit_bag(g.h, _ptr(y), int(it), int(bi), int(th), float(bag), int(bool(rp)), int(bool(iv)), int(bool(de)),
                                         float(pi), float(df), float(R2), int(seed), _ptr(b), _ptr(d), _ptr(Vb), _ptr(hat), _ptr(scal)))
        else:
            check(g.lib.bwgr_wgr_fit(g.h, _ptr(y), int(it), int(bi), int(th), int(bool(iv)), int(bool(de)), float(pi), float(df),
                                     float(R2), int(seed), _ptr(b), _ptr(d), _ptr(Vb), _ptr(hat), _ptr(scal)))
        return {"mu": float(scal[0]), "b": b, "Vb": Vb if (iv or de) else float(scal[2]), "d": d, "Ve": float(scal[1]),
                "hat": hat, "cxx": float(scal[3])}
    finally:
        if own:
            g.close()


class _TwoDesigns:
    """The two marker matrices of a two-design solver as two stores, and the reference's set-up of both (xx, MSx = sum of column variances)."""

    def __init__(self, y, X1, X2, store_kw):
        self.y = np.ascontiguousarray(y, dtype=np.float64)
        self.g, self.own = [], []
        try:
            for X in (X1, X2):
                g, own = _store(X, **store_kw)
                self.g.append(g); self.own.append(own)
            _need(self.g[0].n == self.g[1].n == self.y.size, "y, X1 and X2 must have the same number of rows")
            self.n, self.p = self.g[0].n, [self.g[0].p, self.g[1].p]
            self.xx, self.MSx = [], []
            for g in self.g:
                xx, sx = (np.asarray(v, dtype=np.float64) for v in g.stats())
                self.xx.append(xx)
                self.MSx.append(float(((xx - sx * sx / self.n) / (self.n - 1)).sum()))
        except Exception:
            self.close()
            raise

    def sweep(self, q, b, d, e, L, Ve, pi, seed):
        """One Kuo-Mallick sweep over design q on the device (natural marker order, shared residual)."""
        return KMUP(self.g[q], b, d, self.xx[q], e, L, Ve, pi, seed=seed)

    def close(self):
        for g, own in zip(self.g, self.own):
            if own:
                g.close()


def emML2(y, X1, X2, D1=None, D2=None, **store_kw):
    """emML2(y, X1, X2, D1 = NULL, D2 = NULL) (Rcpp20260726ai.cpp:1221-1305): y = mu + X1 b1 + X2 b2 + e, ridge sweeps over both designs
    with one residual (the device's Kuo-Mallick sweep in its deterministic limit Ve -> 0, pi = 0: b1 = (x'e + xx b0) / (xx + Lmb)),
    variance components from u'cY / n with u1 = X1 b1, u2 = X2 b2 formed on the device every sweep; same list."""
    T = _TwoDesigns(y, X1, X2, store_kw)
    try:
        n, y = T.n, T.y
        Dw = [None if D is None else np.asarray(D, dtype=np.float64) for D in (D1, D2)]
        for q in range(2):
            _need(Dw[q] is None or Dw[q].size == T.p[q], "emML2: D%d must have one weight per marker" % (q + 1))
        b = [np.zeros(T.p[0]), np.zeros(T.p[1])]
        u = [np.zeros(n), np.zeros(n)]
        Lmb = list(T.MSx)
        vb = [0.0, 0.0]
        mu = float(np.float32(y.mean()))
        e = y - mu
        ve = 0.0
        for numit in range(350):
            bc = [b[0].copy(), b[1].copy()]
            for q in range(2):
                L = np.full(T.p[q], Lmb[q]) if Dw[q] is None else Lmb[q] / Dw[q]
                up = T.sweep(q, b[q], np.ones(T.p[q]), e, L, 1e-30, 0.0, 1)
                b[q], e = up["b"], up["e"]
            for q in range(2):  # :1275-1276 (formed afresh like the reference: the variance components feed back on them)
                u[q] = T.g[q].fitted(b[q])
            eM = e.mean()
            mu += eM
            e = e - eM
            cY = u[0] + u[1] + e
            ve = float(e @ cY / n)
            for q in range(2):
                vb[q] = float(u[q] @ cY / n) / T.MSx[q]
                Lmb[q] = ve / vb[q]
            if np.abs(bc[0] - b[0]).sum() + np.abs(bc[1] - b[1]).sum() < 10e-8:
                break
        return {"mu": mu, "b1": b[0], "b2": b[1], "Vb1": vb[0], "Vb2": vb[1], "Ve": ve, "u1": u[0], "u2": u[1], "MSx1": T.MSx[0],
                "MSx2": T.MSx[1], "h2": 1 - ve / float(y.var(ddof=1)), "hat": mu + u[0] + u[1], "its": numit + 1}
    finally:
        T.close()


def _gibbs2(model, y, X1, X2, it, bi, pi, df, R2, seed, store_kw):
    """BayesA2 :990-1069, BayesB2 :1072-1154, BayesRR2 :1157-1218: per iteration one Kuo-Mallick sweep per design on the device (BayesB2's
    marker step IS KMUP's, :1106-1118; the others are its pi = 0 case), the variance draws on the host.  A marker's variance draw depends
    on its own effect only and is not read again before the sweep ends, so drawing all of them after the sweep is the same sampler."""
    T = _TwoDesigns(y, X1, X2, store_kw)
    try:
        n, y, P = T.n, T.y, T.p
        it, bi = int(it), int(bi)
        rng = np.random.default_rng(seed)
        vy = float(y.var(ddof=1))
        Sb = [R2 * df * vy / T.MSx[q] for q in range(2)]
        Se = (1 - R2) * df * vy
        mu, ve = float(y.mean()), vy
        e = y - mu
        b = [np.zeros(P[q]) for q in range(2)]
        d = [np.zeros(P[q]) for q in range(2)]
        vb = [np.full(P[q], Sb[q]) for q in range(2)]
        vbs = [0.0, 0.0]
        L = [np.full(P[q], T.MSx[q]) if model == "BayesRR2" else ve / vb[q] for q in range(2)]
        MU = VE = 0.0
        B = [np.zeros(P[q]) for q in range(2)]
        D = [np.zeros(P[q]) for q in range(2)]
        VB = [np.zeros(P[q]) for q in range(2)]
        VBs = [0.0, 0.0]
        for i in range(it):
            for q in range(2):
                up = T.sweep(q, b[q], d[q], e, L[q], ve, pi if model == "BayesB2" else 0.0, int(rng.integers(1, 2 ** 62)))
                b[q], e = up["b"], up["e"]
                if model == "BayesB2":
                    d[q] = up["d"]
                if model != "BayesRR2":
                    vb[q] = (Sb[q] + b[q] * b[q]) / rng.chisquare(df + 1, size=P[q])
            eM = rng.normal(e.mean(), np.sqrt(ve / n))
            mu += eM
            e = e - eM
            ve = float((e @ e + Se) / rng.chisquare(n + df))
            for q in range(2):
                if model == "BayesRR2":
                    vbs[q] = float((Sb[q] + b[q] @ b[q]) / rng.chisquare(df + P[q]))
                    L[q] = np.full(P[q], ve / vbs[q])
                else:
                    L[q] = ve / vb[q]
            if i > bi:  # sic: it - bi - 1 draws are summed and divided by it - bi (:1062-1065)
                MU += mu; VE += ve
                for q in range(2):
                    B[q] += b[q]; D[q] += d[q]; VB[q] += vb[q]; VBs[q] += vbs[q]
        mc = float(it - bi)
        MU /= mc; VE /= mc
        B = [v / mc for v in B]; D = [v / mc for v in D]; VB = [v / mc for v in VB]; VBs = [v / mc for v in VBs]
        vg = VBs[0] * T.MSx[0] + VBs[1] * T.MSx[1] if model == "BayesRR2" else float(VB[0].sum() + VB[1].sum())
        hat = T.g[0].fitted(B[0], MU) + T.g[1].fitted(B[1])  # fit = X1 B1 + X2 B2 + MU (:1063-1064)
        out = {"hat": hat, "mu": MU, "b1": B[0], "b2": B[1], "vb1": VBs[0] if model == "BayesRR2" else VB[0],
               "vb2": VBs[1] if model == "BayesRR2" else VB[1], "ve": VE, "h2": vg / (vg + VE)}
        if model == "BayesB2":
            out["d1"], out["d2"] = D[0], D[1]
        return out
    finally:
        T.close()


def BayesA2(y, X1, X2, it=1500, bi=500, df=5, R2=0.5, seed=1, **kw):
    """BayesA2(y, X1, X2, it = 1500, bi = 500, df = 5, R2 = 0.5) (Rcpp20260726ai.cpp:990-1069)."""
    return _gibbs2("BayesA2", y, X1, X2, it, bi, 0.0, df, R2, seed, kw)


def BayesB2(y, X1, X2, it=1500, bi=500, pi=0.95, df=5, R2=0.5, seed=1, **kw):
    """BayesB2(y, X1, X2, it = 1500, bi = 500, pi = 0.95, df = 5, R2 = 0.5) (Rcpp20260726ai.cpp:1072-1154)."""
    return _gibbs2("BayesB2", y, X1, X2, it, bi, pi, df, R2, seed, kw)


def BayesRR2(y, X1, X2, it=1500, bi=500, df=5, R2=0.5, seed=1, **kw):
    """BayesRR2(y, X1, X2, it = 1500, bi = 500, df = 5, R2 = 0.5) (Rcpp20260726ai.cpp:1157-1218)."""
    return _gibbs2("BayesRR2", y, X1, X2, it, bi, 0.0, df, R2, seed, kw)


_MRR3_DEFAULTS = dict(
    maxit=500, tol=10e-9, cores=1, TH=False, NLfactor=0.0, InnerGS=False, NoInv=False, HCS=False, XFA=False,
    ACS=False, NumXFA=3, R2=0.5, gc0=0.5, df0=1.0, updateMu=False, weight_prior_h2=0.01, weight_prior_gc=0.01,
    PenCor=0.0, MinCor=1.0, uncorH2below=0.0, roundGCupFrom=1.0, roundGCupTo=1.0, roundGCdownFrom=1.0,
    roundGCdownTo=0.0, bucketGCfrom=1.0, bucketGCto=1.0, DeflateMax=0.9, DeflateBy=0.0, OneVarB=False, OneVarE=False)


def MRR3(Y, X, f32_variant=False, verbose=False, **kw):
    """MRR3(Y, X, ...) of R/RcppExports.R:180 (same argument names and defaults, same returned list).
    The marker loop runs as k rotated ridge systems in the blocked sweep kernel (csrc/mrr.cu).
    X may be a row-sharded store (Genotypes.enable_row_sharding): every rank passes its rows of Y and gets the common
    b / mu / h2 / GC / vb / ve / MSx / Its and hat for its rows.  Only the fast path runs sharded (complete Y, no InnerGS, TH,
    NLfactor or MRR3F NoInv); otherwise every rank raises BwgrError(BWGR_ERR_UNSUPPORTED)."""
    par = dict(_MRR3_DEFAULTS)
    for key, v in kw.items():
        if key not in par:
            raise TypeError("unknown MRR3 argument %r" % key)
        par[key] = v
    g, own = _store(X, centred_ok=True)  # MRR3 centres every column itself (:378-379): X and CNT(X) are the same model
    try:
        Y = np.asfortranarray(Y, dtype=np.float64)
        _need(Y.ndim == 2 and Y.shape[0] == g.n, "Y must be n x k with n = %d rows" % g.n)
        n, k = Y.shape
        p = g.p
        pv = np.array([float(par[name]) for name in _MRR3_DEFAULTS], dtype=np.float64)
        maxit = int(par["maxit"])
        mu, h2, ve, MSx = (np.zeros(k) for _ in range(4))
        b = np.zeros((p, k), order="F")
        W = np.zeros((p, k), order="F")
        hat = np.zeros((n, k), order="F")
        GC = np.zeros((k, k), order="F")
        vb = np.zeros((k, k), order="F")
        cnv = np.zeros(3 * maxit)
        its = C.c_int()
        check(g.lib.bwgr_mrr3_fit(g.h, int(bool(f32_variant)), _ptr(Y), k, _ptr(pv), _ptr(mu), _ptr(b), _ptr(hat), _ptr(h2),
                                  _ptr(GC), _ptr(vb), _ptr(ve), _ptr(MSx), _ptr(cnv), _ptr(W), C.byref(its)))
        q = its.value
        return {"mu": mu, "b": b, "hat": hat, "h2": h2, "GC": GC, "vb": vb, "ve": ve, "MSx": MSx, "cnvB": cnv[:q],
                "cnvH2": cnv[maxit:maxit + q], "cnvV": cnv[2 * maxit:2 * maxit + q], "b_Weights": W, "Its": q}
    finally:
        if own:
            g.close()


def MRR3F(Y, X, **kw):
    return MRR3(Y, X, f32_variant=True, **kw)


def mrr(Y, X, **kw):  # R/mix.R:1271
    return MRR3(Y, X, **kw)


def mrr_float(Y, X, **kw):  # R/mix.R:1273
    return MRR3F(Y, X, **kw)


# ---- cross-validation drivers (R/cv.R:2-216): the batched callers of the marker-effect loop --------------------------------
EMCV_MODELS = ("emRR", "emEN", "emBL", "emDE", "emBA", "emBB", "emBC", "emML", "emBCpi", "lasso")  # R/cv.R:24-26
MCMCCV_MODELS = ("BayesA", "BayesB", "BayesC", "BayesL", "BayesCpi", "BayesDpi", "BayesRR")          # R/cv.R:132-133


def _cv_holdouts(n_rows, k, n, llo, seed):
    """The held-out row sets: `n` random draws of round(N/k) rows (R/cv.R:6-10 -- random hold-outs, not a partition; the
    draws come from numpy, not from R's sample()), or one set per level of `llo` (leave-level-out, R/cv.R:45-48)."""
    if llo is not None:
        llo = np.asarray(llo)
        lev, first = np.unique(llo, return_index=True)
        return [np.flatnonzero(llo == v) for v in lev[np.argsort(first)]]  # unique(as.character(llo)): order of first appearance
    rng = np.random.default_rng(seed)
    nk = int(round(n_rows / k))
    return [np.sort(rng.choice(n_rows, nk, replace=False)) for _ in range(n)]


def _cv_summary(gebv, models, avg):
    """sCV of R/cv.R:86-101: predictive ability = correlation of each model's column with OBSERVATION, over the pooled
    hold-outs (avg, sorted decreasing) or per hold-out; rounded to four digits like the reference."""
    def pa(M):  # cor(..., use = 'p') of R/cv.R:88 / :97: pairwise-complete rows for every (model, OBSERVATION) pair
        obs = M[:, -1]
        out = np.full(M.shape[1] - 1, np.nan)
        with np.errstate(invalid="ignore", divide="ignore"):
            for j in range(M.shape[1] - 1):
                ok = np.isfinite(M[:, j]) & np.isfinite(obs)
                if ok.sum() > 1:
                    out[j] = np.corrcoef(M[ok, j], obs[ok])[0, 1]
        return out
    if avg:
        c = pa(np.concatenate(gebv, axis=0))
        order = np.argsort(-c, kind="stable")
        return {models[i]: round(float(c[i]), 4) for i in order}
    return {"CV_%d" % (i + 1): {m: round(float(v), 4) for m, v in zip(models, pa(M))} for i, M in enumerate(gebv)}


def _cv_world(group):
    """(rank, world) of the torch.distributed group the hold-outs are dealt over; (0, 1) without an initialised process group."""
    try:
        import torch.distributed as dist
    except ImportError:
        return 0, 1, None
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group), dist
    return 0, 1, None


def _cv_run(models, fit_one, y, gen, holdouts, tbv, avg, ReturnGebv, group=None, store=None):
    """The hold-outs are independent fits (SURVEY 8e, "independent folds": no communication): under torch.distributed rank r
    takes hold-outs r, r + world, ... on its own GPU (LOCAL_RANK) and the per-hold-out results are gathered on the host, so
    every rank returns the full summary.  `store(X_keep, device)` builds the per-hold-out genotype store (tests inject a stub)."""
    import os
    y = np.asarray(y, dtype=np.float64)
    X = np.asarray(gen)
    obs = y if tbv is None else np.asarray(tbv, dtype=np.float64)
    rank, world, dist = _cv_world(group)
    device = int(os.environ.get("LOCAL_RANK", rank)) if world > 1 else 0
    if store is None:
        def store(Xk, dev):
            return Genotypes(np.asfortranarray(Xk), device=dev)
    mine = []
    for idx in range(rank, len(holdouts), world):
        w = holdouts[idx]
        keep = np.setdiff1d(np.arange(X.shape[0]), w)
        with store(X[keep], device) as g:  # gen[-w, ] packed ONCE per hold-out, shared by every model of the panel
            B = np.stack([fit_one(m, y[keep], g)["b"] for m in models], axis=1)
        M = np.concatenate([X[w].astype(np.float64) @ B, obs[w][:, None]], axis=1)  # gen[w, ] %*% b | OBSERVATION
        mine.append((idx, M, B))
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, mine, group=group)
        mine = sorted((item for per_rank in gathered for item in per_rank), key=lambda item: item[0])
    gebv = [M for _, M, _ in mine]
    B0 = [B for _, _, B in mine]
    cv = _cv_summary(gebv, list(models), avg)
    if not ReturnGebv:
        return cv
    beta = np.mean(B0, axis=0)  # R/cv.R:102-106
    return {"cv": cv, "hat": X.astype(np.float64) @ beta + np.nanmean(y), "beta": beta}


def emCV(y, gen, k=5, n=5, Pi=0.75, alpha=0.02, df=10, R2=0.5, avg=True, llo=None, tbv=None, ReturnGebv=False, seed=1,
         group=None):
    """emCV of R/cv.R:2-108: ten EM solvers per hold-out, predictive correlation of gen[w, ] b with the held-out
    observations.  Per fold the training rows are packed once into one device store and all ten fits run on it."""
    def fit_one(m, yk, g):
        kw = {"emRR": dict(R2=R2, df=df), "emEN": dict(alpha=alpha, R2=R2), "emBL": dict(alpha=alpha, R2=R2), "emDE": dict(R2=R2),
              "emBA": dict(R2=R2, df=df), "emBB": dict(Pi=Pi, R2=R2, df=df), "emBC": dict(Pi=Pi, R2=R2, df=df), "emML": {},
              "emBCpi": {}, "lasso": {}}[m]  # R/cv.R:13-22 (emML, emBCpi and lasso run on their defaults)
        return em_fit(m, yk, g, **kw)
    return _cv_run(EMCV_MODELS, fit_one, y, gen, _cv_holdouts(np.asarray(gen).shape[0], k, n, llo, seed), tbv, avg, ReturnGebv,
                   group=group)


def mcmcCV(y, gen, k=5, n=5, it=1500, bi=500, pi=0.95, df=5, R2=0.5, avg=True, llo=None, tbv=None, ReturnGebv=False, seed=1,
           group=None):
    """mcmcCV of R/cv.R:110-216: the seven Gibbs samplers per hold-out.  Deliberate deviation: every column is labelled with the
    model that produced it; the reference fits BayesRR, BayesCpi, BayesDpi as f5..f7 (cv.R:128-130) but names those columns BayesCpi,
    BayesDpi, BayesRR (:132-133), i.e. its last three labels are rotated."""
    def fit_one(m, yk, g):
        kw = dict(R2=R2, df=df, it=it, bi=bi, seed=seed)
        if m in ("BayesB", "BayesC"):
            kw["pi"] = pi
        return gibbs_fit(m, yk, g, **kw)
    return _cv_run(MCMCCV_MODELS, fit_one, y, gen, _cv_holdouts(np.asarray(gen).shape[0], k, n, llo, seed), tbv, avg, ReturnGebv,
                   group=group)
