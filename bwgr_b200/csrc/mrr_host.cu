// mrr_host.cu -- MRR3 / MRR3F (bwgr_mrr3_fit): the k x k linear algebra and variance block on the host, the rotated fast path on
// the fit engine's pipelined sweep (mrr.cu), and the general path (mrr_gen.cu).
#include "host.h"

using namespace bwgr;
using namespace bwgr::host;

namespace {
// ---- small dense symmetric helpers for the k x k part of MRR3 (column-major, double) ----------------------------------
using Mat = std::vector<double>;
// cyclic Jacobi: A = V diag(w) V', eigenvalues ascending (what Eigen's SelfAdjointEigenSolver returns, :639)
void sym_eig(const Mat& Ain, int k, std::vector<double>& w, Mat& V) {
  Mat A(Ain);
  V.assign((size_t)k * k, 0.0);
  for (int i = 0; i < k; i++) V[i + (size_t)i * k] = 1.0;
  for (int sweep = 0; sweep < 64; sweep++) {
    double off = 0;
    for (int i = 0; i < k; i++) for (int j = 0; j < i; j++) off += A[i + (size_t)j * k] * A[i + (size_t)j * k];
    if (off < 1e-300) break;
    for (int pI = 0; pI < k - 1; pI++)
      for (int q = pI + 1; q < k; q++) {
        const double apq = A[pI + (size_t)q * k];
        if (std::fabs(apq) < 1e-300) continue;
        const double theta = (A[q + (size_t)q * k] - A[pI + (size_t)pI * k]) / (2.0 * apq);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), sn = t * c;
        for (int r = 0; r < k; r++) {
          const double arp = A[r + (size_t)pI * k], arq = A[r + (size_t)q * k];
          A[r + (size_t)pI * k] = c * arp - sn * arq; A[r + (size_t)q * k] = sn * arp + c * arq;
        }
        for (int r = 0; r < k; r++) {
          const double apr = A[pI + (size_t)r * k], aqr = A[q + (size_t)r * k];
          A[pI + (size_t)r * k] = c * apr - sn * aqr; A[q + (size_t)r * k] = sn * apr + c * aqr;
        }
        for (int r = 0; r < k; r++) {
          const double vrp = V[r + (size_t)pI * k], vrq = V[r + (size_t)q * k];
          V[r + (size_t)pI * k] = c * vrp - sn * vrq; V[r + (size_t)q * k] = sn * vrp + c * vrq;
        }
      }
  }
  std::vector<int> idx(k);
  for (int i = 0; i < k; i++) idx[i] = i;
  std::sort(idx.begin(), idx.end(), [&](int a, int b) { return A[a + (size_t)a * k] < A[b + (size_t)b * k]; });
  w.resize(k);
  Mat Vs((size_t)k * k);
  for (int c = 0; c < k; c++) { w[c] = A[idx[c] + (size_t)idx[c] * k]; for (int r = 0; r < k; r++) Vs[r + (size_t)c * k] = V[r + (size_t)idx[c] * k]; }
  V.swap(Vs);
}
bool chol_ok(const Mat& Ain, int k) {  // LLT success test (:603-607)
  Mat A(Ain);
  for (int j = 0; j < k; j++) {
    double d = A[j + (size_t)j * k];
    for (int c = 0; c < j; c++) d -= A[j + (size_t)c * k] * A[j + (size_t)c * k];
    if (!(d > 0)) return false;
    d = std::sqrt(d);
    A[j + (size_t)j * k] = d;
    for (int i = j + 1; i < k; i++) {
      double v = A[i + (size_t)j * k];
      for (int c = 0; c < j; c++) v -= A[i + (size_t)c * k] * A[j + (size_t)c * k];
      A[i + (size_t)j * k] = v / d;
    }
  }
  return true;
}
void sym_pinv(const Mat& A, int k, Mat& out) {  // completeOrthogonalDecomposition().pseudoInverse() of a symmetric matrix (:648)
  std::vector<double> w; Mat V;
  sym_eig(A, k, w, V);
  double wmax = 0;
  for (double v : w) wmax = std::max(wmax, std::fabs(v));
  const double tol = wmax * k * 2.220446049250313e-16;
  out.assign((size_t)k * k, 0.0);
  for (int c = 0; c < k; c++) {
    if (std::fabs(w[c]) <= tol) continue;
    const double iw = 1.0 / w[c];
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) out[i + (size_t)j * k] += iw * V[i + (size_t)c * k] * V[j + (size_t)c * k];
  }
}

// MRR3's argument list after (Y, X), in the order of R/RcppExports.R:180
struct MrrFlags {
  int maxit; double tol; bool TH; double NLfactor; bool InnerGS, NoInv, HCS, XFA, ACS; int NumXFA; double R2, gc0, df0; bool updateMu;
  double wph2, wpgc, PenCor, MinCor, uncorH2below, rUpFrom, rUpTo, rDownFrom, rDownTo, bkFrom, bkTo, DeflateMax, DeflateBy;
  bool OneVarB, OneVarE;
  explicit MrrFlags(const double* par) {
    int q = 0;
    maxit = (int)par[q++]; tol = par[q++]; q++; TH = par[q++] != 0; NLfactor = par[q++];
    InnerGS = par[q++] != 0; NoInv = par[q++] != 0; HCS = par[q++] != 0; XFA = par[q++] != 0; ACS = par[q++] != 0;
    NumXFA = (int)par[q++]; R2 = par[q++]; gc0 = par[q++]; df0 = par[q++]; updateMu = par[q++] != 0;
    wph2 = par[q++]; wpgc = par[q++]; PenCor = par[q++]; MinCor = par[q++]; uncorH2below = par[q++];
    rUpFrom = par[q++]; rUpTo = par[q++]; rDownFrom = par[q++]; rDownTo = par[q++]; bkFrom = par[q++]; bkTo = par[q++];
    DeflateMax = par[q++]; DeflateBy = par[q++]; OneVarB = par[q++] != 0; OneVarE = par[q++] != 0;
  }
};
// The state of MRR3's outer loop that survives from sweep to sweep, the same on the rotated fast path and the general path.
struct MrrVar {
  Mat vb, iG, GC, Sb;
  std::vector<double> vbInit;
  double Deflate = 1, inflate = 0;
  std::vector<double> mu, vy, MSx, nn;  // per trait: mean and variance of y, sum of the marker variances, observations (the path's)
  std::vector<double> ve, iVe, veInit, h2, Se, iNp;
  std::vector<double> cnvB, cnvH2, cnvV;  // convergence records (:662-666)
  int numit = 0;
};
// Output arrays of bwgr_mrr3_fit (any may be null)
struct MrrOut {
  double *mu, *b, *hat, *h2, *GC, *vb, *ve, *MSx, *cnv, *W;
  int* its;
};

// Starting values (:394-432) from V.vy, V.MSx and V.nn.
void mrr_start(const MrrFlags& F, int k, MrrVar& V) {
  auto M = [k](int r, int c) { return (size_t)r + (size_t)c * k; };
  Mat& vb = V.vb;
  vb.assign((size_t)k * k, 0.0); V.iG.assign((size_t)k * k, 0.0); V.GC.assign((size_t)k * k, 0.0);
  for (auto* v : {&V.vbInit, &V.ve, &V.iVe, &V.veInit, &V.h2, &V.Se, &V.iNp}) v->resize(k);
  for (int t = 0; t < k; t++) {
    V.ve[t] = V.vy[t] * (1 - F.R2); V.iVe[t] = 1.0 / V.ve[t]; V.veInit[t] = V.ve[t];
    V.vbInit[t] = V.vy[t] * F.R2 / V.MSx[t]; vb[M(t, t)] = V.vbInit[t]; V.iG[M(t, t)] = 1.0 / V.vbInit[t]; V.h2[t] = 1 - V.ve[t] / V.vy[t];
    V.Se[t] = V.ve[t] * F.df0; V.iNp[t] = 1.0 / (V.nn[t] + F.df0 - 1.0);
  }
  for (int i = 0; i < k; i++) for (int j = 0; j < i; j++) { const double v = F.gc0 * std::sqrt(vb[M(i, i)] * vb[M(j, j)]); vb[M(i, j)] = v; vb[M(j, i)] = v; }
  V.Sb = vb;
  for (auto& v : V.Sb) v *= F.df0;
}

// Residual variances of one sweep (:536-543) from e'y of trait t at ey[t * stride].
void mrr_residual_var(const MrrFlags& F, int k, const double* ey, int stride, MrrVar& V) {
  for (int t = 0; t < k; t++) { V.ve[t] = (ey[(size_t)t * stride] + V.Se[t]) * V.iNp[t]; V.h2[t] = 1 - V.ve[t] / V.vy[t]; }
  if (F.wph2 > 0) for (int t = 0; t < k; t++) V.ve[t] = V.ve[t] * (1 - F.wph2) + F.wph2 * V.veInit[t];
  if (F.OneVarE) { double m = 0; for (int t = 0; t < k; t++) m += V.ve[t]; m /= k; for (int t = 0; t < k; t++) V.ve[t] = m; }
  for (int t = 0; t < k; t++) V.iVe[t] = 1.0 / V.ve[t];
}

// Convergence records of one sweep (:662-666) from |beta0 - b|^2 of every trait; vb0 and h20 are vb and h2 before the sweep.
// False: the outer loop ends here.
bool mrr_record(const MrrFlags& F, int k, const double* db, const Mat& vb0, const std::vector<double>& h20, MrrVar& V) {
  double mx = -1e300;
  for (int t = 0; t < k; t++) mx = std::max(mx, db[t]);
  const double cnv = std::log10(mx);
  V.cnvB.push_back(cnv);
  if (cnv != cnv) return false;  // :663
  { double sH = 0; for (int t = 0; t < k; t++) sH += (h20[t] - V.h2[t]) * (h20[t] - V.h2[t]); V.cnvH2.push_back(std::log10(sH)); }
  { double sV = 0; for (size_t i = 0; i < V.vb.size(); i++) sV += (vb0[i] - V.vb[i]) * (vb0[i] - V.vb[i]); V.cnvV.push_back(std::log10(sV)); }
  ++V.numit;
  return !(cnv < std::log10(F.tol));
}

// The outputs (:676-700) both paths share; b, hat and W are the path's own.
void mrr_copy_out(const MrrFlags& F, int k, const MrrVar& V, const MrrOut& o) {
  for (int t = 0; t < k; t++) {
    if (o.mu) o.mu[t] = V.mu[t];
    if (o.h2) o.h2[t] = V.h2[t];
    if (o.ve) o.ve[t] = V.ve[t];
    if (o.MSx) o.MSx[t] = V.MSx[t];
  }
  if (o.GC) for (int i = 0; i < k * k; i++) o.GC[i] = V.GC[i];
  if (o.vb) for (int i = 0; i < k * k; i++) o.vb[i] = V.vb[i];
  if (o.cnv)
    for (int i = 0; i < V.numit; i++) { o.cnv[i] = V.cnvB[i]; o.cnv[F.maxit + i] = V.cnvH2[i]; o.cnv[2 * F.maxit + i] = V.cnvV[i]; }
  if (o.its) *o.its = V.numit;
}
// Genetic (co)variances of one sweep (:559-648): TildeHat and the traces Tr (TrXSX, or TrDinvXSX under TH) in, vb / GC / iG out.
// Shared by the rotated fast path and the general path; double, on the host (k <= 32).
void mrr_varcomp(const MrrFlags& F, int k, const Mat& TildeHat, const std::vector<double>& Tr, const std::vector<double>& h2, MrrVar& V) {
  auto M = [k](int r, int c) { return (size_t)r + (size_t)c * k; };
  Mat &vb = V.vb, &iG = V.iG, &GC = V.GC, A;
  const Mat& Sb = V.Sb;
  const std::vector<double>& vbInit = V.vbInit;
  double &Deflate = V.Deflate, &inflate = V.inflate;
  const double df0 = F.df0, wph2 = F.wph2, wpgc = F.wpgc, gc0 = F.gc0, PenCor = F.PenCor, MinCor = F.MinCor, uncorH2below = F.uncorH2below;
  const double rUpFrom = F.rUpFrom, rUpTo = F.rUpTo, rDownFrom = F.rDownFrom, rDownTo = F.rDownTo, bkFrom = F.bkFrom, bkTo = F.bkTo;
  const double DeflateMax = F.DeflateMax, DeflateBy = F.DeflateBy, bucketMean = 0.5 * (F.bkFrom + F.bkTo);
  const bool ACS = F.ACS, HCS = F.HCS, XFA = F.XFA, OneVarB = F.OneVarB;
  const int NumXFA = F.NumXFA;
  const bool rebuild = !F.NoInv || F.TH;  // :628, :647: with NoInv (and no TH) the correlations are not bent and iG keeps its start value
  for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) {
    if (i == j) vb[M(i, i)] = (TildeHat[M(i, i)] + Sb[M(i, i)]) / (Tr[i] + df0);
    else vb[M(i, j)] = (TildeHat[M(i, j)] + TildeHat[M(j, i)] + Sb[M(i, j)]) / (Tr[i] + Tr[j] + df0);
  }
  if (wph2 > 0) for (int i = 0; i < k; i++) vb[M(i, i)] = vb[M(i, i)] * (1 - wph2) + wph2 * vbInit[i];
  if (wpgc > 0) {
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++)
      GC[M(i, j)] = (i != j) ? (1.0 - wpgc) * vb[M(i, j)] / std::sqrt(vb[M(i, i)] * vb[M(j, j)]) + gc0 * wpgc : 1.0;
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) if (i != j) vb[M(i, j)] = GC[M(i, j)] * std::sqrt(vb[M(i, i)] * vb[M(j, j)]);
  } else {
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) GC[M(i, j)] = vb[M(i, j)] / std::sqrt(vb[M(i, i)] * vb[M(j, j)]);
  }
  auto top_factors = [&](double add, double scale) {  // :593-600, :612-617
    std::vector<double> ew; Mat ev;
    sym_eig(GC, k, ew, ev);
    Mat UDU((size_t)k * k, 0.0);
    for (int fI = 0; fI < NumXFA && fI < k; fI++) {
      const int c = k - fI - 1;
      for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) UDU[M(i, j)] += ew[c] * ev[M(i, c)] * ev[M(j, c)];
    }
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) GC[M(i, j)] = (UDU[M(i, j)] + add) * scale;
    for (int i = 0; i < k; i++) GC[M(i, i)] = 1;
  };
  if (ACS) {
    double gs = 0;
    for (double v : GC) gs += v;
    gs = (gs - k) / ((k * (k - 1))) / 2.0;
    top_factors(gs, 0.5);
  } else if (HCS) {
    double gs = 0;
    for (int i = 0; i < k; i++) for (int j = 0; j < i; j++) gs += GC[M(i, j)];
    gs = gs / ((k * (k - 1)) / 2);
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) GC[M(i, j)] = (i != j) ? gs : 1.0;
  } else if (XFA) {
    top_factors(0.0, 1.0);
  }
  for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) if (i != j) {  // :619-626
    double& g = GC[M(i, j)];
    if (MinCor < 1 && g < MinCor) g = 0;
    if (PenCor > 0) g = std::tanh(PenCor * std::fabs(g)) * g;
    if (rDownFrom < 1 && g < rDownFrom) g = rDownTo;
    if (rUpFrom < 1 && g > rUpFrom) g = rUpTo;
    if (bkFrom < 1 && g > bkFrom && g < bkTo) g = bucketMean;
    if (uncorH2below > 0 && (h2[i] < uncorH2below || h2[j] < uncorH2below)) g = 0;
  }
  if (rebuild) {  // bending (:629-644)
    A = GC;
    if (DeflateBy > 0) {
      for (auto& v : A) v *= Deflate;
      for (int i = 0; i < k; i++) A[M(i, i)] = 1;
      if (!chol_ok(A, k) && Deflate > DeflateMax) {
        Deflate -= DeflateBy;
        A = GC;
        for (auto& v : A) v *= Deflate;
        for (int i = 0; i < k; i++) A[M(i, i)] = 1;
      }
    }
    std::vector<double> ew; Mat ev;
    sym_eig(A, k, ew, ev);
    if (ew[0] < 0) {
      inflate = std::fabs(ew[0] * 1.1);
      for (int i = 0; i < k; i++) A[M(i, i)] += inflate;
      for (auto& v : A) v /= (1.0 + inflate);
      GC = A;
    }
  }
  if (OneVarB) {
    double tmp = 0;
    for (int i = 0; i < k; i++) tmp += TildeHat[M(i, i)];
    tmp /= k;
    for (size_t i = 0; i < vb.size(); i++) vb[i] = GC[i] * tmp;
  } else {
    const Mat dv(vb);
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) vb[M(i, j)] = GC[M(i, j)] * std::sqrt(dv[M(i, i)] * dv[M(j, j)]);
  }
  if (rebuild) sym_pinv(vb, k, iG);
}

// MRR3 / MRR3F on the general device path (mrr_gen.cu): per-trait observation masks, InnerGS, NLfactor, TH, MRR3F's NoInv system.
// Host side = the reference's set-up (:359-432) and the k x k variance block; everything O(n), O(p) or O(n p) is a kernel.
int mrr3_general(bwgr_handle* h, int f32_variant, const double* Y, int k, const MrrFlags& F, const MrrOut& out) {
  if (h->storage != BWGR_STORE_I8 || !h->x8) return fail(BWGR_ERR_UNSUPPORTED, "MRR3 (general path) reads the int8 store");
  if (h->world > 1) return fail(BWGR_ERR_UNSUPPORTED, "MRR3 does not run on a row-sharded store");
  const int64_t n = h->n, p = h->p, ld = h->ld;
  const int maxit = F.maxit, kk = k * k;
  const bool innergs = F.InnerGS, noinv_system = f32_variant && F.NoInv, NonLinear = F.NLfactor != 0;
  const int nmat = innergs ? 2 : 1;
  auto M = [k](int r, int c) { return (size_t)r + (size_t)c * k; };
  CU(cudaSetDevice(h->device));
  // ---- incidence, counts, centred phenotypes (:359-376)
  MrrVar V;
  std::vector<double> &nn = V.nn, &mu = V.mu, &vy = V.vy, &MSx = V.MSx;
  nn.resize(k); mu.resize(k); vy.resize(k); MSx.assign(k, 0.0);
  std::vector<uint32_t> zb((size_t)ld, 0u);
  std::vector<double> ysum(k), yh((size_t)k * ld, 0.0);
  for (int t = 0; t < k; t++) {
    double sum = 0; int64_t cnt = 0;
    for (int64_t i = 0; i < n; i++) { const double v = Y[(size_t)t * n + i]; if (v == v) { zb[i] |= 1u << t; sum += v; cnt++; } }
    if (cnt < 2) return fail(BWGR_ERR_ARG, "MRR3: trait %d has fewer than two observations", t + 1);
    nn[t] = (double)cnt; mu[t] = sum / (double)cnt;
    double s1 = 0, s2 = 0;
    for (int64_t i = 0; i < n; i++) {
      const double v = Y[(size_t)t * n + i];
      if (v == v) { const double c = v - mu[t]; yh[(size_t)t * ld + i] = c; s1 += c; s2 += c * c; }
    }
    ysum[t] = s1; vy[t] = s2 / (nn[t] - 1.0);
    if (!(vy[t] > 0)) return fail(BWGR_ERR_ARG, "MRR3: trait %d has no variance", t + 1);
  }
  // ---- launch geometry: one CTA per row slab, all co-resident
  int rp = 0, grid = 0;
  grid_geometry(h, &rp, &grid);
  const size_t smem = mrr_gen_smem(k, rp, innergs);
  if (smem > h->smem_optin || grid > h->num_sms)
    return fail(BWGR_ERR_UNSUPPORTED, "MRR3 (general path): %lld rows x %d traits do not fit the shared memory of %d SMs", (long long)n, k, h->num_sms);
  DevBuf<uint32_t> zbits; DevBuf<double> yd, ed, bd, bold, fixd, meand, tilded, sold, Wd, xsxd, dinvd, small;
  DevBuf<unsigned long long> accd; DevBuf<int> permd;
  const size_t nsmall = (size_t)2 * kk + 11 * 32;  // iG | vb | iVe | se | ey | cnv | trd | par(2 x 32) | shift | see | scale(2 x 32)
  if (zbits.alloc(ld) != cudaSuccess || yd.alloc((size_t)k * ld) != cudaSuccess || ed.alloc((size_t)k * ld) != cudaSuccess ||
      bd.alloc((size_t)p * k) != cudaSuccess || bold.alloc((size_t)p * k) != cudaSuccess || fixd.alloc((size_t)p * 2 * k) != cudaSuccess ||
      meand.alloc(p) != cudaSuccess || tilded.alloc((size_t)p * k) != cudaSuccess || sold.alloc((size_t)p * nmat * kk) != cudaSuccess ||
      (NonLinear && Wd.alloc((size_t)p * k) != cudaSuccess) || (F.TH && (xsxd.alloc((size_t)p * k) != cudaSuccess || dinvd.alloc((size_t)p * k) != cudaSuccess)) ||
      small.alloc(nsmall + kk) != cudaSuccess || accd.alloc((size_t)p * 32 * kGridCopies) != cudaSuccess || grid > 255 ||
      permd.alloc(p + 32) != cudaSuccess)
    return fail(BWGR_ERR_CUDA, "cudaMalloc(MRR3 general workspace) failed");
  double *d_iG = small.p, *d_vb = small.p + kk, *d_iVe = d_vb + kk, *d_se = d_iVe + 32, *d_ey = d_se + 32, *d_cnv = d_ey + 32,
         *d_trd = d_cnv + 32, *d_par = d_trd + 32, *d_shift = d_par + 64, *d_see = d_shift + 32, *d_scale = d_see + 32, *d_th = small.p + nsmall;
  cudaStream_t st = h->stream;
  CU(cudaMemcpyAsync(zbits.p, zb.data(), sizeof(uint32_t) * ld, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(yd.p, yh.data(), sizeof(double) * k * ld, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(ed.p, yd.p, sizeof(double) * k * ld, cudaMemcpyDeviceToDevice, st));  // e = y (:435)
  CU(cudaMemsetAsync(bd.p, 0, sizeof(double) * p * k, st));
  // ---- masked column statistics (:381-392) and tilde = X_c'y (:420) from one pass over the store
  std::vector<double> sxz((size_t)p * k), sxxz((size_t)p * k), tilde((size_t)p * k), fixed((size_t)p * 2 * k), meanv(p), xsx;
  {
    DevBuf<double> a1, a2;
    if (a1.alloc((size_t)p * k) != cudaSuccess || a2.alloc((size_t)p * k) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    launch_mrr_gen_colstats(h->view(), zbits.p, yd.p, k, a1.p, a2.p, tilded.p, st);
    h->launches++;
    CU(cudaMemcpyAsync(sxz.data(), a1.p, sizeof(double) * p * k, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(sxxz.data(), a2.p, sizeof(double) * p * k, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(tilde.data(), tilded.p, sizeof(double) * p * k, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  std::vector<double> TrXSX(k), see(k);
  for (int t = 0; t < k; t++) see[t] = vy[t] * (nn[t] - 1.0);  // e = y at the start
  if (F.TH) xsx.resize((size_t)p * k);
  for (int64_t j = 0; j < p; j++) {
    const double m = h->h_sx[j] / (double)n;  // X.colwise().mean() over all n0 rows (:378)
    meanv[j] = m;
    for (int t = 0; t < k; t++) {
      const size_t q = (size_t)j * k + t;
      const double XX = sxxz[q] - 2.0 * m * sxz[q] + m * m * nn[t];  // sum_i (x - m)^2 z_it
      const double sc = sxz[q] - m * nn[t];                           // sum_i (x - m) z_it
      const double qq = sc / nn[t], v = XX / nn[t] - qq * qq;         // XSX (:386-388)
      fixed[(size_t)j * 2 * k + t] = XX; fixed[(size_t)j * 2 * k + k + t] = sc;
      MSx[t] += v;
      if (F.TH) xsx[q] = v * nn[t];                                   // :423
      tilde[q] -= m * ysum[t];
    }
  }
  for (int t = 0; t < k; t++) {
    if (!(MSx[t] > 0)) return fail(BWGR_ERR_ARG, "genotypes have no variance");
    TrXSX[t] = nn[t] * MSx[t];
  }
  CU(cudaMemcpyAsync(fixd.p, fixed.data(), sizeof(double) * p * 2 * k, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(meand.p, meanv.data(), sizeof(double) * p, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(tilded.p, tilde.data(), sizeof(double) * p * k, cudaMemcpyHostToDevice, st));
  if (F.TH) CU(cudaMemcpyAsync(xsxd.p, xsx.data(), sizeof(double) * p * k, cudaMemcpyHostToDevice, st));
  mrr_start(F, k, V);
  Mat TildeHat((size_t)kk);
  std::vector<int> order(p), irgs(32);
  for (int64_t j = 0; j < p; j++) order[j] = (int)j;
  for (int j = 0; j < 32; j++) irgs[j] = j;
  std::vector<double> W, bh, hsmall(32 * 4 + kk), trd(k);
  if (NonLinear) { W.assign((size_t)p * k, 1.0); CU(cudaMemcpyAsync(Wd.p, W.data(), sizeof(double) * p * k, cudaMemcpyHostToDevice, st)); }
  int rc = 0;
  MrrGenArgs a;
  a.g = h->view(); a.k = k; a.rows_per_cta = rp; a.innergs = innergs ? 1 : 0; a.perm = permd.p; a.irgs = permd.p + p; a.zbits = zbits.p;
  a.e = ed.p; a.b = bd.p; a.fixed = fixd.p; a.mean = meand.p; a.sol = sold.p; a.se0 = d_se; a.acc = accd.p; a.scale = d_scale; a.err = h->err.p;
  while (V.numit < maxit) {
    const Mat vb0(V.vb); const std::vector<double> h20(V.h2);
    const int numit = V.numit;
    CU(cudaMemcpyAsync(bold.p, bd.p, sizeof(double) * p * k, cudaMemcpyDeviceToDevice, st));  // beta0 (:475)
    std::shuffle(order.begin(), order.end(), std::mt19937(numit));                           // :483-484, cumulative
    std::shuffle(irgs.begin(), irgs.begin() + k, std::mt19937(numit));
    CU(cudaMemcpyAsync(permd.p, order.data(), sizeof(int) * p, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(permd.p + p, irgs.data(), sizeof(int) * 32, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_iG, V.iG.data(), sizeof(double) * kk, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_vb, V.vb.data(), sizeof(double) * kk, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_iVe, V.iVe.data(), sizeof(double) * k, cudaMemcpyHostToDevice, st));
    // MRR3 applies the marker weights in the solve (:504); MRR3F never does (its weights are an output only)
    launch_mrr_gen_systems((int)p, k, fixd.p, (NonLinear && !f32_variant) ? Wd.p : nullptr, d_iG, d_vb, d_iVe, noinv_system ? 1 : 0,
                           innergs ? 1 : 0, sold.p, st);
    launch_mrr_gen_colred(ed.p, nullptr, ld, (int)n, k, d_se, st);
    {  // fixed-point scale of the grid sums of this sweep: |x'e_t| <= sqrt(max_j x_j'x_j) |e_t| (Cauchy-Schwarz, also for the sum of
       // the per-CTA magnitudes); 16 x headroom for the growth of |e_t| inside a sweep, 2^52 of range
      std::vector<double> scl(64, 0.0);
      for (int t = 0; t < k; t++) {
        int ex = 0;
        std::frexp(16.0 * std::sqrt(h->xx_max * see[t]) + 1e-300, &ex);
        scl[t] = std::ldexp(1.0, 52 - ex); scl[32 + t] = std::ldexp(1.0, ex - 52);
      }
      CU(cudaMemcpyAsync(d_scale, scl.data(), sizeof(double) * 64, cudaMemcpyHostToDevice, st));
      CU(cudaMemsetAsync(accd.p, 0, sizeof(unsigned long long) * p * 32 * kGridCopies, st));
      const cudaError_t le = launch_mrr_gen_sweep(a, grid, st);
      if (le != cudaSuccess) return fail(BWGR_ERR_CUDA, "MRR3 general sweep launch failed: %s", cudaGetErrorString(le));
    }
    launch_mrr_gen_colred(ed.p, yd.p, ld, (int)n, k, d_ey, st);  // e.y (:536)
    launch_mrr_gen_colred(ed.p, ed.p, ld, (int)n, k, d_see, st);  // |e_t|^2: the next sweep's fixed-point range
    h->launches += 5;
    CU(cudaMemcpyAsync(hsmall.data(), d_ey, sizeof(double) * k, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(see.data(), d_see, sizeof(double) * k, cudaMemcpyDeviceToHost, st));
    if (NonLinear) { bh.resize((size_t)p * k); CU(cudaMemcpyAsync(bh.data(), bd.p, sizeof(double) * p * k, cudaMemcpyDeviceToHost, st)); }
    CU(cudaStreamSynchronize(st));
    rc = check_err_flag(h, "MRR3 general sweep");
    if (rc) return rc;
    if (NonLinear) {  // :524-533
      std::vector<double> tmpW(p);
      for (int t = 0; t < k; t++) {
        double maxW = -INFINITY, minW = INFINITY;
        for (int64_t j = 0; j < p; j++) { const double v = std::fabs(bh[(size_t)j * k + t]); maxW = std::max(maxW, v); minW = std::min(minW, v); }
        double sw = 0;
        for (int64_t j = 0; j < p; j++) { tmpW[j] = F.NLfactor * (std::fabs(bh[(size_t)j * k + t]) - minW) / (maxW - minW) + (1.0 - F.NLfactor); sw += tmpW[j]; }
        const double mw = sw / (double)p;
        for (int64_t j = 0; j < p; j++) W[(size_t)j * k + t] = tmpW[j] + (1.0 - mw);
      }
      CU(cudaMemcpyAsync(Wd.p, W.data(), sizeof(double) * p * k, cudaMemcpyHostToDevice, st));
    }
    mrr_residual_var(F, k, hsmall.data(), 1, V);
    // ---- tilde-hat (:546-556) and the convergence sums (:662)
    if (F.TH) {
      std::vector<double> par(64, 0.0);
      for (int t = 0; t < k; t++) { par[t] = V.ve[t]; par[k + t] = V.iG[M(t, t)]; }
      CU(cudaMemcpyAsync(d_par, par.data(), sizeof(double) * 2 * k, cudaMemcpyHostToDevice, st));
      launch_mrr_gen_pk(2, xsxd.p, nullptr, dinvd.p, d_par, (int)p, k, d_trd, st);
      launch_mrr_gen_pk(0, bd.p, tilded.p, dinvd.p, nullptr, (int)p, k, d_th, st);
      h->launches++;
    } else {
      launch_mrr_gen_pk(0, bd.p, tilded.p, nullptr, nullptr, (int)p, k, d_th, st);
    }
    launch_mrr_gen_pk(1, bold.p, bd.p, nullptr, nullptr, (int)p, k, d_cnv, st);
    h->launches += 2;
    CU(cudaMemcpyAsync(hsmall.data(), d_cnv, sizeof(double) * 64, cudaMemcpyDeviceToHost, st));  // cnv | trd
    CU(cudaMemcpyAsync(hsmall.data() + 128, d_th, sizeof(double) * kk, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) TildeHat[M(i, j)] = hsmall[128 + (size_t)i * k + j];
    for (int t = 0; t < k; t++) trd[t] = hsmall[32 + t];
    mrr_varcomp(F, k, TildeHat, F.TH ? trd : TrXSX, V.h2, V);
    if (F.updateMu) {  // :651-655; iN is 1 / (n_t - 1) by now (:395)
      launch_mrr_gen_colred(ed.p, nullptr, ld, (int)n, k, d_se, st);
      std::vector<double> sh(k);
      CU(cudaMemcpyAsync(sh.data(), d_se, sizeof(double) * k, cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      for (int t = 0; t < k; t++) { sh[t] /= (nn[t] - 1.0); mu[t] += sh[t]; }
      CU(cudaMemcpyAsync(d_shift, sh.data(), sizeof(double) * k, cudaMemcpyHostToDevice, st));
      launch_mrr_gen_shift(ed.p, zbits.p, ld, (int)n, k, d_shift, st);
      CU(cudaStreamSynchronize(st));
      h->launches += 2;
    }
    if (!mrr_record(F, k, hsmall.data(), vb0, h20, V)) break;
  }
  // ---- outputs (:676-700): hat = X_c b + mu = X b + (mu - sum_j mean_j b_j)
  bh.resize((size_t)p * k);
  CU(cudaMemcpyAsync(bh.data(), bd.p, sizeof(double) * p * k, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (out.hat) {
    std::vector<float> bt((size_t)k * p), m0(k), hh;
    for (int t = 0; t < k; t++) {
      double shift = 0;
      for (int64_t j = 0; j < p; j++) { const double v = bh[(size_t)j * k + t]; shift += meanv[j] * v; bt[(size_t)t * p + j] = (float)v; }
      m0[t] = (float)(mu[t] - shift);
    }
    if ((rc = fitted_values(h, k, bt.data(), true, m0.data(), hh))) return rc;
    for (size_t i = 0; i < hh.size(); i++) out.hat[i] = hh[i];
  }
  if (out.b) for (int t = 0; t < k; t++) for (int64_t j = 0; j < p; j++) out.b[(size_t)t * p + j] = bh[(size_t)j * k + t];
  if (out.W) for (int t = 0; t < k; t++) for (int64_t j = 0; j < p; j++) out.W[(size_t)t * p + j] = NonLinear ? W[(size_t)j * k + t] : 1.0;
  mrr_copy_out(F, k, V, out);
  return 0;
}
}  // namespace

extern "C" {

// MRR3 / MRR3F with the marker loop on the device (see mrr.cu).  Fast path = complete Y and the direct k x k solve:
// NaN in Y, InnerGS, NLfactor != 0, TH, and MRR3F's NoInv system return BWGR_ERR_UNSUPPORTED (never a CPU fallback).
int bwgr_mrr3_fit(bwgr_handle* h, int f32_variant, const double* Y, int k, const double* par, double* mu_out, double* b_out,
                  double* hat_out, double* h2_out, double* GC_out, double* vb_out, double* ve_out, double* MSx_out, double* cnv_out,
                  double* W_out, int* its_out) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!Y || !par) return fail(BWGR_ERR_ARG, "null argument");
  if (k < 1 || k > 32) return fail(BWGR_ERR_UNSUPPORTED, "MRR3 on the B200 path takes 1..32 traits (k=%d)", k);
  const MrrFlags F(par);
  const MrrOut out{mu_out, b_out, hat_out, h2_out, GC_out, vb_out, ve_out, MSx_out, cnv_out, W_out, its_out};
  const int maxit = F.maxit;
  if (maxit < 1) return fail(BWGR_ERR_ARG, "maxit < 1");
  // n: this rank's rows (all of them on one GPU); ng: the individuals every sum over individuals runs over
  const int64_t n = h->n, p = h->p, ld = h->ld, ng = h->n_global;
  const bool dist = h->world > 1;
  bool missing = false;
  for (int64_t i = 0; i < n * k && !missing; i++) missing = !(Y[i] == Y[i]);
  // Everything the rotation cannot express -- missing phenotypes (per-trait XX), the inner Gauss-Seidel solve, marker weights,
  // MRR3F's NoInv system, the tilde-hat estimator -- runs on the general device path (mrr_gen.cu); BWGR_MRR=general forces it.
  const char* force = getenv("BWGR_MRR");
  const bool options = F.TH || F.NLfactor != 0 || F.InnerGS || (f32_variant && F.NoInv);
  const bool forced = force && !strcmp(force, "general");
  if (dist) {
    // A row-sharded store has the fast path only, and every rank must take the same road: the reasons any rank has to refuse are
    // all-reduced before any other collective, and then every rank refuses or none does.
    PipePlan pl;
    const bool no_fit = !h->hx_connected || h->storage != BWGR_STORE_I8 || !(h->xx_max < 16777216.0) || !plan_pipe(h, M_MRR, k, &pl);
    double why[4] = {missing ? 1.0 : 0.0, options ? 1.0 : 0.0, forced ? 1.0 : 0.0, no_fit ? 1.0 : 0.0};
    int rc = dist_allreduce_host(h, why, 4, true);
    if (rc) return rc;
    if (why[0] || why[1] || why[2] || why[3])
      return fail(BWGR_ERR_UNSUPPORTED, "the general MRR3 path does not run on a row-sharded store (%s)",
                  why[0] ? "missing phenotypes on some rank" : why[1] ? "TH, NLfactor, InnerGS or MRR3F's NoInv" :
                  why[2] ? "BWGR_MRR=general on some rank" : "the shard does not fit the pipelined blocked sweep on some rank");
  } else if (missing || options || forced) {
    return mrr3_general(h, f32_variant, Y, k, F, out);
  }
  auto M = [k](int r, int c) { return (size_t)r + (size_t)c * k; };
  // ---- setup (:359-432), double on the host
  MrrVar V;
  V.mu.assign(k, 0.0); V.vy.assign(k, 0.0); V.nn.assign(k, (double)ng);
  for (int t = 0; t < k; t++)
    for (int64_t i = 0; i < n; i++) V.mu[t] += Y[(size_t)t * n + i];
  int rc = dist_allreduce_host(h, V.mu.data(), k, false);
  if (rc) return rc;
  for (int t = 0; t < k; t++) {
    V.mu[t] /= (double)ng;
    for (int64_t i = 0; i < n; i++) { const double v = Y[(size_t)t * n + i] - V.mu[t]; V.vy[t] += v * v; }
  }
  if ((rc = dist_allreduce_host(h, V.vy.data(), k, false))) return rc;
  for (int t = 0; t < k; t++) V.vy[t] /= ((double)ng - 1.0);
  std::vector<float> xxc(p), sxf(p);
  double msx = 0;
  for (int64_t j = 0; j < p; j++) {
    const double c = h->h_xx[j] - h->h_sx[j] * h->h_sx[j] / (double)ng;  // XX(J,t) = sum (x - mean)^2, same for every trait (:382-385)
    xxc[j] = (float)c; sxf[j] = (float)h->h_sx[j];
    msx += c / (double)ng;                                              // XSX (:386-388): the centred column sums to zero
  }
  if (!(msx > 0)) return fail(BWGR_ERR_ARG, "genotypes have no variance");
  const double TrXSX = (double)ng * msx;
  V.MSx.assign(k, msx);
  mrr_start(F, k, V);
  // ---- device state through the common fit machinery: k systems of the rotated ridge rule
  FitSpec s;
  s.model = M_MRR; s.nsys = k; s.shuffled = true; s.row_mask = nullptr;
  s.df = 0; s.R2 = (float)F.R2; s.Pi = 0; s.alpha = 0; s.pi = 0; s.it = maxit; s.bi = 0; s.seed = 0;
  FitGuard guard{h};
  rc = fit_begin(h, s, Y);
  if (rc == BWGR_ERR_UNSUPPORTED && !dist)  // the shape does not fit the pipelined blocked sweep (row slabs above 512 rows): general path
    return mrr3_general(h, f32_variant, Y, k, F, out);
  if (rc) return rc;
  Fit& f = *h->fit;
  f.skip_epilogue = true;
  DevBuf<float> tilde, e_alt, b_alt, b_old, Tdev, amax;
  DevBuf<double> red, red2;
  if (f.xx_over.alloc(p) != cudaSuccess || f.sx_dev.alloc(p) != cudaSuccess || f.cshift.alloc(32) != cudaSuccess ||
      tilde.alloc((size_t)k * p) != cudaSuccess || e_alt.alloc((size_t)k * ld) != cudaSuccess || b_alt.alloc((size_t)k * p) != cudaSuccess ||
      b_old.alloc((size_t)k * p) != cudaSuccess || Tdev.alloc(2 * 32 * 32) != cudaSuccess || amax.alloc(32) != cudaSuccess ||
      red.alloc((size_t)k * k + 3 * k) != cudaSuccess || red2.alloc((size_t)k * k) != cudaSuccess)
    return fail(BWGR_ERR_CUDA, "cudaMalloc(MRR3 workspace) failed");
  CU(cudaMemcpyAsync(f.xx_over.p, xxc.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.sx_dev.p, sxf.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemsetAsync(e_alt.p, 0, sizeof(float) * k * ld, h->stream));
  // f.y holds the raw Y, f.e = Y - mu (fit_begin): centre y in place for the e.y reductions (:536)
  CU(cudaMemcpyAsync(f.y.p, f.e.p, sizeof(float) * k * ld, cudaMemcpyDeviceToDevice, h->stream));
  launch_xty(h->view(), f.y.p, k, tilde.p, h->stream);  // tilde = X'y (:420)
  h->launches++;
  if (dist) NC(nccl().AllReduce(tilde.p, tilde.p, (size_t)k * p, ncclFloat, ncclSum, h->comm, h->stream));
  std::vector<double> hred((size_t)k * k + 3 * k);
  std::vector<float> Tf(32 * 32), Tif(32 * 32), hmax(32);
  std::vector<SysScalars> sc(f.sc0);
  Mat TildeHat((size_t)k * k);
  while (V.numit < maxit) {
    const Mat vb0(V.vb); const std::vector<double> h20(V.h2);
    const std::vector<double>& iVe = V.iVe;
    // ---- rotation of this sweep: S^-1 iG S^-1 = U Lambda U', T = S U, T^-1 = U' S^-1
    Mat Ms((size_t)k * k), U; std::vector<double> lam;
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) Ms[M(i, j)] = V.iG[M(i, j)] / std::sqrt(iVe[i] * iVe[j]);
    sym_eig(Ms, k, lam, U);
    for (int sI = 0; sI < k; sI++) for (int t = 0; t < k; t++) {
      Tf[sI * k + t] = (float)(std::sqrt(iVe[sI]) * U[M(sI, t)]);       // T[s][t]
      Tif[sI * k + t] = (float)(U[M(t, sI)] / std::sqrt(iVe[t]));        // Tinv[s][t] = U[t][s] / S_t
    }
    CU(cudaMemcpyAsync(Tdev.p, Tf.data(), sizeof(float) * k * k, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(Tdev.p + 1024, Tif.data(), sizeof(float) * k * k, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(b_old.p, f.b.p, sizeof(float) * k * p, cudaMemcpyDeviceToDevice, h->stream));  // beta0 (:475)
    CU(cudaMemsetAsync(amax.p, 0, sizeof(float) * 32, h->stream));
    launch_rotate(f.e.p, e_alt.p, ld, (int)n, k, Tdev.p, nullptr, amax.p, h->num_sms, h->stream);
    launch_rotate(f.b.p, b_alt.p, p, (int)p, k, Tdev.p, nullptr, nullptr, h->num_sms, h->stream);
    h->launches += 2;
    f.e.swap(e_alt); f.b.swap(b_alt);
    // the fixed-point words of X_B'E the ranks exchange are summable only at one scale: max|e| over all individuals
    if (dist) NC(nccl().AllReduce(amax.p, amax.p, 32, ncclFloat, ncclMax, h->comm, h->stream));
    CU(cudaMemcpyAsync(hmax.data(), amax.p, sizeof(float) * 32, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int t = 0; t < k; t++) {
      SysScalars& c = sc[t];
      c.lmb = (float)std::max(lam[t], 0.0);
      set_e_scale(c, hmax[t]);
      c.done = 0; c.sweep = V.numit;
    }
    CU(cudaMemcpyAsync(f.sc.p, sc.data(), sizeof(SysScalars) * k, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemsetAsync(f.cshift.p, 0, sizeof(float) * 32, h->stream));
    rc = fit_sweeps(h, 1);  // marker order shuffle(mt19937(numit)) (:483), centred Gram band, k-system sweep
    if (rc) return rc;
    // ---- back to trait space: E = (E~ + c) T^-1, b = b~ T^-1
    launch_rotate(f.e.p, e_alt.p, ld, (int)n, k, Tdev.p + 1024, f.cshift.p, nullptr, h->num_sms, h->stream);
    launch_rotate(f.b.p, b_alt.p, p, (int)p, k, Tdev.p + 1024, nullptr, nullptr, h->num_sms, h->stream);
    f.e.swap(e_alt); f.b.swap(b_alt);
    // ---- reductions of the sweep epilogue: b'tilde (:549), e.y (:536), |beta0 - b|^2 (:662), column sums of e (:652)
    launch_pair_reduce(f.b.p, tilde.p, p, p, (int)p, k, 0, red.p, h->stream);
    launch_pair_reduce(f.e.p, f.y.p, ld, ld, (int)n, k, 0, red2.p, h->stream);
    launch_pair_reduce(b_old.p, f.b.p, p, p, (int)p, k, 1, red.p + (size_t)k * k, h->stream);
    launch_pair_reduce(f.e.p, nullptr, ld, ld, (int)n, k, 2, red.p + (size_t)k * k + k, h->stream);
    h->launches += 6;
    if (dist) {  // e.y and the column sums of e run over individuals; b'tilde and |beta0 - b|^2 are the same on every rank
      NC(nccl().AllReduce(red2.p, red2.p, (size_t)k * k, ncclDouble, ncclSum, h->comm, h->stream));
      NC(nccl().AllReduce(red.p + (size_t)k * k + k, red.p + (size_t)k * k + k, (size_t)k, ncclDouble, ncclSum, h->comm, h->stream));
    }
    std::vector<double> ey((size_t)k * k), small(2 * k);
    CU(cudaMemcpyAsync(hred.data(), red.p, sizeof(double) * ((size_t)k * k + 2 * k), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(ey.data(), red2.p, sizeof(double) * k * k, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) TildeHat[M(i, j)] = hred[(size_t)i * k + j];
    for (int t = 0; t < 2 * k; t++) small[t] = hred[(size_t)k * k + t];
    rc = check_err_flag(h, "MRR3 sweep");
    if (rc) return rc;
    // ---- variance components (:536-648), double
    mrr_residual_var(F, k, ey.data(), k + 1, V);  // e.y of trait t: the diagonal of the k x k products
    { const std::vector<double> Tr((size_t)k, TrXSX); mrr_varcomp(F, k, TildeHat, Tr, V.h2, V); }
    if (F.updateMu) {  // :651-655 (complete Y: Z = 1)
      std::vector<float> sh(k);
      for (int t = 0; t < k; t++) { const double m = small[k + t] / ((double)ng - 1.0); V.mu[t] += m; sh[t] = (float)(-m); }
      // e -= m: a rotation by the identity with a shift
      std::vector<float> I((size_t)k * k, 0.0f);
      for (int t = 0; t < k; t++) I[(size_t)t * k + t] = 1.0f;
      CU(cudaMemcpyAsync(Tdev.p, I.data(), sizeof(float) * k * k, cudaMemcpyHostToDevice, h->stream));
      CU(cudaMemcpyAsync(f.cshift.p, sh.data(), sizeof(float) * k, cudaMemcpyHostToDevice, h->stream));
      launch_rotate(f.e.p, e_alt.p, ld, (int)n, k, Tdev.p, f.cshift.p, nullptr, h->num_sms, h->stream);
      f.e.swap(e_alt);
      CU(cudaStreamSynchronize(h->stream));
    }
    if (!mrr_record(F, k, small.data(), vb0, h20, V)) break;
  }
  // ---- outputs (:676-700): hat = X_c b + mu = X b + (mu - sum_j mean_j b_j)
  std::vector<float> hb((size_t)k * p), m0(k), hh;
  CU(cudaMemcpyAsync(hb.data(), f.b.p, sizeof(float) * k * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  for (int t = 0; t < k; t++) {
    double shift = 0;
    for (int64_t j = 0; j < p; j++) shift += (h->h_sx[j] / (double)ng) * (double)hb[(size_t)t * p + j];
    m0[t] = (float)(V.mu[t] - shift);
  }
  rc = fitted_values(h, k, f.b.p, false, m0.data(), hh);
  if (rc) return rc;
  if (hat_out) for (size_t i = 0; i < hh.size(); i++) hat_out[i] = hh[i];
  if (b_out) for (size_t i = 0; i < hb.size(); i++) b_out[i] = hb[i];
  if (W_out) for (size_t i = 0; i < (size_t)k * p; i++) W_out[i] = 1.0;
  mrr_copy_out(F, k, V, out);
  dump_trace(h);
  return 0;
}

}  // extern "C"
