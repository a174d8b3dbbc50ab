// oracle_capi.cpp -- C entry points over bwgr_oracle.hpp for ctypes (tests, smoke, bench CPU arm).
// TEST INFRASTRUCTURE ONLY: see the header of bwgr_oracle.hpp.  All matrices are column-major.
#include "bwgr_oracle.hpp"

#include <cstdio>

namespace {
template <class R>
void em_run(int model, const float* y, const float* X, int n, int p, float df, float R2, float Pi, float alpha, int it,
            double* mu, double* b, double* d, double* hat, double* vbv, double* scal, int* its, const double* D = nullptr) {
  std::vector<R> yy(y, y + n);
  std::vector<R> XX;
  const R* Xp;
  if constexpr (sizeof(R) == sizeof(float)) {
    Xp = reinterpret_cast<const R*>(X);
  } else {
    XX.assign(X, X + (size_t)n * p);
    Xp = XX.data();
  }
  orc::EmPar<R> P;
  P.df = df; P.R2 = R2; P.Pi = Pi; P.alpha = alpha; P.it = it; P.D = D;
  orc::EmOut<R> o;
  orc::em_fit<R>(model, yy.data(), Xp, n, p, P, o);
  *mu = o.mu;
  for (int j = 0; j < p; j++) b[j] = o.b[j];
  for (int j = 0; j < p; j++) d[j] = o.d.empty() ? 0.0 : (double)o.d[j];
  for (int j = 0; j < p; j++) vbv[j] = o.vbv.empty() ? 0.0 : (double)o.vbv[j];
  for (int i = 0; i < n; i++) hat[i] = o.hat[i];
  scal[0] = o.Va; scal[1] = o.Ve; scal[2] = o.h2; scal[3] = o.Vg; scal[4] = o.pi; scal[5] = o.Lmb;
  *its = o.its;
}
}  // namespace

extern "C" {

// Cumulative marker orders of sweeps 0..n_iter-1: out[i*p + jj] (Rcpp20260726ai.cpp:329-331).
int orc_perm(int p, int n_iter, int32_t* out) {
  orc::Shuffler sh(p);
  for (int i = 0; i < n_iter; i++) {
    sh.next(i);
    std::memcpy(out + (size_t)i * p, sh.order.data(), sizeof(int) * p);
  }
  return 0;
}

// Univariate EM fit. use_double=0: float32 like the reference; 1: same recipe in float64 (to bound
// float noise).  it<0: the reference's hard-coded sweep count.  scal = {Va, Ve, h2, Vg, pi, Lmb}.
int orc_em(int model, int use_double, const float* y, const float* X, int n, int p, float df, float R2, float Pi,
           float alpha, int it, double* mu, double* b, double* d, double* hat, double* vbv, double* scal, int* its) {
  if (model < 0 || model > 9) return -1;
  if (use_double) em_run<double>(model, y, X, n, p, df, R2, Pi, alpha, it, mu, b, d, hat, vbv, scal, its);
  else em_run<float>(model, y, X, n, p, df, R2, Pi, alpha, it, mu, b, d, hat, vbv, scal, its);
  return 0;
}

// emML with marker weights D (Rcpp20260726ai.cpp:463-521, P_WEIGHTS branch)
int orc_emml_weighted(int use_double, const float* y, const float* X, int n, int p, const double* D, int it, double* mu, double* b,
                      double* hat, double* scal, int* its) {
  std::vector<double> d(p), vbv(p);
  if (use_double) em_run<double>(7, y, X, n, p, 10, 0.5f, 0.75f, 0.02f, it, mu, b, d.data(), hat, vbv.data(), scal, its, D);
  else em_run<float>(7, y, X, n, p, 10, 0.5f, 0.75f, 0.02f, it, mu, b, d.data(), hat, vbv.data(), scal, its, D);
  return 0;
}

// Univariate Gibbs fit (float32 state). scal = {vb, ve, h2, MSx, pi}.
int orc_gibbs(int model, const float* y, const float* X, int n, int p, float it, float bi, float pi, float df, float R2,
              uint64_t seed, double* mu, double* b, double* d, double* hat, double* vbv, double* scal) {
  if (model < 0 || model > 6) return -1;
  orc::GibbsOut<float> o;
  orc::Rng rng(seed);
  orc::gibbs_fit<float>(model, y, X, n, p, it, bi, pi, df, R2, rng, o);
  *mu = o.mu;
  for (int j = 0; j < p; j++) { b[j] = o.b[j]; d[j] = o.d[j]; vbv[j] = o.vbv[j]; }
  for (int i = 0; i < n; i++) hat[i] = o.hat[i];
  scal[0] = o.vb; scal[1] = o.ve; scal[2] = o.h2; scal[3] = o.MSx; scal[4] = o.pi;
  return 0;
}

int orc_kmup(const float* X, int n, int p, float* b, float* d, const float* xx, float* e, const float* L, float Ve,
             float pi, uint64_t seed, int ratio_form) {
  orc::Rng rng(seed);
  orc::kmup(X, n, p, b, d, xx, e, L, Ve, pi, rng, ratio_form != 0);
  return 0;
}

int orc_kmup2(const float* X, int n, int p, const float* use, int nuse, float* b, float* d, const float* xx, const float* E, float* e_out,
              const float* L, float Ve, float pi, uint64_t seed, int ratio_form) {
  orc::Rng rng(seed);
  orc::kmup2(X, n, p, use, nuse, b, d, xx, E, e_out, L, Ve, pi, rng, ratio_form != 0);
  return 0;
}

// which = 0 GSRR, 1 GSFLM; scal = {mu, h2, vna, its}
int orc_gs(int which, const float* y, float* e, const float* X, int n, int p, float* b, float* Lmb, const float* xx, float cxx, int maxit,
           float* vb, double* scal) {
  const orc::GsOut o = orc::gs_solver(which != 0, y, e, X, n, p, b, Lmb, xx, cxx, maxit, vb);
  scal[0] = o.mu; scal[1] = o.h2; scal[2] = o.vna; scal[3] = o.its;
  return 0;
}

int orc_cnt_imp(int which, float* X, int n, int p) {
  if (which == 0) orc::cnt_columns(X, n, p); else orc::imp_columns(X, n, p);
  return 0;
}

// two-design solvers.  model: 0 BayesA2, 1 BayesB2, 2 BayesRR2, 3 emML2.  scal = {mu, ve, h2, vb1 (scalar), vb2 (scalar), MSx1, MSx2, its}
int orc_two_design(int model, const float* y, const float* X1, const float* X2, int n, int p1, int p2, float it, float bi, float pi, float df,
                   float R2, uint64_t seed, const double* D1, const double* D2, double* b1, double* b2, double* d1, double* d2, double* vb1,
                   double* vb2, double* hat, double* u1, double* u2, double* scal) {
  orc::TwoDesignOut o;
  if (model == 3) orc::emml2_fit(y, X1, X2, n, p1, p2, D1, D2, o);
  else orc::gibbs2_fit(model, y, X1, X2, n, p1, p2, it, bi, pi, df, R2, seed, o);
  auto cp = [](const std::vector<float>& v, double* out) { if (out) for (size_t i = 0; i < v.size(); i++) out[i] = v[i]; };
  cp(o.b1, b1); cp(o.b2, b2); cp(o.d1, d1); cp(o.d2, d2); cp(o.vb1, vb1); cp(o.vb2, vb2); cp(o.hat, hat); cp(o.u1, u1); cp(o.u2, u2);
  scal[0] = o.mu; scal[1] = o.ve; scal[2] = o.h2; scal[3] = o.vb1s; scal[4] = o.vb2s; scal[5] = o.MSx1; scal[6] = o.MSx2; scal[7] = o.its;
  return 0;
}

// scal = {mu, Ve, Va, cxx}
int orc_wgr(const double* y, const double* X, int n, int p, int it, int bi, int th, int iv, int de, double pi, double df,
            double R2, uint64_t seed, int ratio_form, double* b, double* d, double* Vb, double* hat, double* scal) {
  orc::WgrOut o;
  orc::Rng rng(seed);
  orc::wgr<float>(y, X, n, p, it, bi, th, iv != 0, de != 0, pi, df, R2, rng, ratio_form != 0, o);
  for (int j = 0; j < p; j++) { b[j] = o.b[j]; d[j] = o.d[j]; Vb[j] = o.Vb[j]; }
  for (int i = 0; i < n; i++) hat[i] = o.hat[i];
  scal[0] = o.mu; scal[1] = o.Ve; scal[2] = o.Va; scal[3] = o.cxx;
  return 0;
}

// wgr with the polygenic term (eigK): U n x pk, V pk; scal = {mu, Ve, Va, cxx, Vk}; u = U0 %*% H
int orc_wgr_eigk(const double* y, const double* X, int n, int p, const double* U, const double* V, int pk, int it, int bi, int th, int iv,
                 int de, double pi, double df, double R2, uint64_t seed, int ratio_form, double* b, double* d, double* Vb, double* hat,
                 double* u, double* scal) {
  orc::WgrOut o;
  orc::Rng rng(seed);
  orc::wgr<float>(y, X, n, p, it, bi, th, iv != 0, de != 0, pi, df, R2, rng, ratio_form != 0, o, 1.0, U, V, pk);
  for (int j = 0; j < p; j++) { b[j] = o.b[j]; d[j] = o.d[j]; Vb[j] = o.Vb[j]; }
  for (int i = 0; i < n; i++) { hat[i] = o.hat[i]; u[i] = o.u[i]; }
  scal[0] = o.mu; scal[1] = o.Ve; scal[2] = o.Va; scal[3] = o.cxx; scal[4] = o.Vk;
  return 0;
}

int orc_wgr_bag(const double* y, const double* X, int n, int p, int it, int bi, int th, double bag, int iv, int de, double pi, double df,
                double R2, uint64_t seed, int ratio_form, double* b, double* d, double* Vb, double* hat, double* scal) {
  orc::WgrOut o;
  orc::Rng rng(seed);
  orc::wgr<float>(y, X, n, p, it, bi, th, iv != 0, de != 0, pi, df, R2, rng, ratio_form != 0, o, bag);
  for (int j = 0; j < p; j++) { b[j] = o.b[j]; d[j] = o.d[j]; Vb[j] = o.Vb[j]; }
  for (int i = 0; i < n; i++) hat[i] = o.hat[i];
  scal[0] = o.mu; scal[1] = o.Ve; scal[2] = o.Va; scal[3] = o.cxx;
  return 0;
}

// wgr(bag, rp): rp != 0 draws the rows of every iteration with replacement (R/wgr.R:68)
int orc_wgr_bag_rp(const double* y, const double* X, int n, int p, int it, int bi, int th, double bag, int rp, int iv, int de, double pi,
                   double df, double R2, uint64_t seed, int ratio_form, double* b, double* d, double* Vb, double* hat, double* scal) {
  orc::WgrOut o;
  orc::Rng rng(seed);
  orc::wgr<float>(y, X, n, p, it, bi, th, iv != 0, de != 0, pi, df, R2, rng, ratio_form != 0, o, bag, nullptr, nullptr, 0, rp != 0);
  for (int j = 0; j < p; j++) { b[j] = o.b[j]; d[j] = o.d[j]; Vb[j] = o.Vb[j]; }
  for (int i = 0; i < n; i++) hat[i] = o.hat[i];
  scal[0] = o.mu; scal[1] = o.Ve; scal[2] = o.Va; scal[3] = o.cxx;
  return 0;
}

// MRR3 (f32_variant=0, float64) / MRR3F (f32_variant=1, float32).  par[] in the order of the R
// signature after (Y,X): maxit,tol,cores,TH,NLfactor,InnerGS,NoInv,HCS,XFA,ACS,NumXFA,R2,gc0,df0,
// updateMu,weight_prior_h2,weight_prior_gc,PenCor,MinCor,uncorH2below,roundGCupFrom,roundGCupTo,
// roundGCdownFrom,roundGCdownTo,bucketGCfrom,bucketGCto,DeflateMax,DeflateBy,OneVarB,OneVarE  (30 values).
// cnv: 3*maxit doubles (cnvB | cnvH2 | cnvV, each maxit long, first *its valid).
int orc_mrr3(int f32_variant, const double* Y, const double* X, int n, int k, int p, const double* par, double* mu,
             double* b, double* hat, double* h2, double* GC, double* vb, double* ve, double* MSx, double* cnv,
             double* W, int* its) {
  auto run = [&](auto tag) {
    using R = decltype(tag);
    orc::MrrPar<R> P;
    int q = 0;
    P.maxit = (int)par[q++]; P.tol = (R)par[q++]; q++; P.TH = par[q++] != 0; P.NLfactor = (R)par[q++];
    P.InnerGS = par[q++] != 0; P.NoInv = par[q++] != 0; P.HCS = par[q++] != 0; P.XFA = par[q++] != 0; P.ACS = par[q++] != 0;
    P.NumXFA = (int)par[q++]; P.R2 = (R)par[q++]; P.gc0 = (R)par[q++]; P.df0 = (R)par[q++]; P.updateMu = par[q++] != 0;
    P.weight_prior_h2 = (R)par[q++]; P.weight_prior_gc = (R)par[q++]; P.PenCor = (R)par[q++]; P.MinCor = (R)par[q++];
    P.uncorH2below = (R)par[q++]; P.roundGCupFrom = (R)par[q++]; P.roundGCupTo = (R)par[q++];
    P.roundGCdownFrom = (R)par[q++]; P.roundGCdownTo = (R)par[q++]; P.bucketGCfrom = (R)par[q++];
    P.bucketGCto = (R)par[q++]; P.DeflateMax = (R)par[q++]; P.DeflateBy = (R)par[q++]; P.OneVarB = par[q++] != 0;
    P.OneVarE = par[q++] != 0;
    std::vector<R> Yr(Y, Y + (size_t)n * k), Xr(X, X + (size_t)n * p);
    orc::MrrOut<R> o;
    orc::mrr3<R>(Yr.data(), Xr.data(), n, k, p, P, f32_variant != 0, o);
    for (int t = 0; t < k; t++) { mu[t] = o.mu[t]; h2[t] = o.h2[t]; ve[t] = o.ve[t]; MSx[t] = o.MSx[t]; }
    for (size_t i = 0; i < (size_t)p * k; i++) { b[i] = o.b[i]; W[i] = o.W[i]; }
    for (size_t i = 0; i < (size_t)n * k; i++) hat[i] = o.hat[i];
    for (int i = 0; i < k * k; i++) { GC[i] = o.GC[i]; vb[i] = o.vb[i]; }
    for (int i = 0; i < o.its; i++) { cnv[i] = o.cnvB[i]; cnv[P.maxit + i] = o.cnvH2[i]; cnv[2 * P.maxit + i] = o.cnvV[i]; }
    *its = o.its;
  };
  if (f32_variant) run(float{}); else run(double{});
  return 0;
}

}  // extern "C"

// ---- replays on the device's Philox draws (orc::PhiloxDraws) --------------------------------------------------------------------
// use_double = 1 runs the same recipe in float64 on the same float draws.  Every replay reports how close its accept / reject
// decisions came to the other outcome: q / u (the inclusion probability and the uniform of each decision, at most qcap of them,
// *nq = how many there were) and mt[0] = the smallest normalised Marsaglia-Tsang acceptance margin.
namespace {
void margins_out(const orc::PhiloxDraws& rng, double* q, double* u, int qcap, int* nq, double* mt) {
  *nq = (int)rng.q.size();
  for (int i = 0; i < *nq && i < qcap; i++) { q[i] = rng.q[i]; u[i] = rng.uq[i]; }
  mt[0] = rng.mt_margin;
}
template <class R>
void gibbs_philox_run(int model, const float* y, const float* X, int n, int p, float it, float bi, float pi, float df, float R2,
                      orc::PhiloxDraws& rng, double* mu, double* b, double* d, double* hat, double* vbv, double* scal) {
  std::vector<R> yy(y, y + n), XX(X, X + (size_t)n * p);
  orc::GibbsOut<R> o;
  orc::gibbs_fit<R>(model, yy.data(), XX.data(), n, p, it, bi, pi, df, R2, rng, o);
  *mu = o.mu;
  for (int j = 0; j < p; j++) { b[j] = o.b[j]; d[j] = o.d[j]; vbv[j] = o.vbv[j]; }
  for (int i = 0; i < n; i++) hat[i] = o.hat[i];
  scal[0] = o.vb; scal[1] = o.ve; scal[2] = o.h2; scal[3] = o.MSx; scal[4] = o.pi;
}
template <class R>
void kmup_philox_run(const float* X, int n, int p, const float* use, int nuse, double* b, double* d, const double* xx, const double* e,
                     double* e_out, const double* L, double Ve, double pi, orc::PhiloxDraws& rng) {
  std::vector<R> XX(X, X + (size_t)n * p), bb(b, b + p), dd(d, d + p), x2(xx, xx + p), LL(L, L + p), ee(e, e + n), eo(use ? nuse : n);
  for (int j = 0; j < p; j++) { bb[j] = (R)(float)b[j]; dd[j] = (R)(float)d[j]; x2[j] = (R)(float)xx[j]; LL[j] = (R)(float)L[j]; }
  for (int i = 0; i < n; i++) ee[i] = (R)(float)e[i];
  if (use) orc::kmup2<R>(XX.data(), n, p, use, nuse, bb.data(), dd.data(), x2.data(), ee.data(), eo.data(), LL.data(), (R)(float)Ve,
                         (R)(float)pi, rng, true);
  else { orc::kmup<R>(XX.data(), n, p, bb.data(), dd.data(), x2.data(), ee.data(), LL.data(), (R)(float)Ve, (R)(float)pi, rng, true); eo = ee; }
  for (int j = 0; j < p; j++) { b[j] = bb[j]; d[j] = dd[j]; }
  for (size_t i = 0; i < eo.size(); i++) e_out[i] = eo[i];
}
}  // namespace

extern "C" {

// Gibbs fit of chain `chain`; scal as orc_gibbs.
int orc_gibbs_philox(int model, int use_double, int chain, const float* y, const float* X, int n, int p, float it, float bi, float pi,
                     float df, float R2, uint64_t seed, double* mu, double* b, double* d, double* hat, double* vbv, double* scal, double* q,
                     double* u, int qcap, int* nq, double* mt) {
  if (model < 0 || model > 6) return -1;
  orc::PhiloxDraws rng(seed);
  rng.set_chain(chain);
  if (use_double) gibbs_philox_run<double>(model, y, X, n, p, it, bi, pi, df, R2, rng, mu, b, d, hat, vbv, scal);
  else gibbs_philox_run<float>(model, y, X, n, p, it, bi, pi, df, R2, rng, mu, b, d, hat, vbv, scal);
  margins_out(rng, q, u, qcap, nq, mt);
  return 0;
}

// One KMUP sweep (use = NULL; e_out has n values) or KMUP2 sweep over the rows `use` (e_out has nuse values), at sweep 0, chain 0,
// in the ratio form the device evaluates.  b and d are updated in place.
int orc_kmup_philox(int use_double, const float* X, int n, int p, const float* use, int nuse, double* b, double* d, const double* xx,
                    const double* e, double* e_out, const double* L, double Ve, double pi, uint64_t seed, double* q, double* u, int qcap,
                    int* nq, double* mt) {
  orc::PhiloxDraws rng(seed);
  if (use_double) kmup_philox_run<double>(X, n, p, use, nuse, b, d, xx, e, e_out, L, Ve, pi, rng);
  else kmup_philox_run<float>(X, n, p, use, nuse, b, d, xx, e, e_out, L, Ve, pi, rng);
  margins_out(rng, q, u, qcap, nq, mt);
  return 0;
}

// wgr (bag = 1: native; bag != 1: bagged, rp as orc_wgr_bag_rp), KMUP sweeps in the ratio form; scal as orc_wgr.
int orc_wgr_philox(int use_double, const double* y, const double* X, int n, int p, int it, int bi, int th, double bag, int rp, int iv, int de,
                   double pi, double df, double R2, uint64_t seed, double* b, double* d, double* Vb, double* hat, double* scal, double* q,
                   double* u, int qcap, int* nq, double* mt) {
  orc::WgrOut o;
  orc::PhiloxDraws rng(seed);
  if (use_double) orc::wgr<double>(y, X, n, p, it, bi, th, iv != 0, de != 0, pi, df, R2, rng, true, o, bag, nullptr, nullptr, 0, rp != 0);
  else orc::wgr<float>(y, X, n, p, it, bi, th, iv != 0, de != 0, pi, df, R2, rng, true, o, bag, nullptr, nullptr, 0, rp != 0);
  for (int j = 0; j < p; j++) { b[j] = o.b[j]; d[j] = o.d[j]; Vb[j] = o.Vb[j]; }
  for (int i = 0; i < n; i++) hat[i] = o.hat[i];
  scal[0] = o.mu; scal[1] = o.Ve; scal[2] = o.Va; scal[3] = o.cxx;
  margins_out(rng, q, u, qcap, nq, mt);
  return 0;
}

// Known-answer check of the restated generator: out[4] = Philox4x32-10(counter, key)
int orc_philox4x32_10(const uint32_t* counter, uint32_t k0, uint32_t k1, uint32_t* out) {
  uint32_t c[4] = {counter[0], counter[1], counter[2], counter[3]};
  orc::philox::philox4x32_10(c, k0, k1);
  for (int i = 0; i < 4; i++) out[i] = c[i];
  return 0;
}

// The draws of one marker update at (marker, sweep, chain): {z1, z2, u, chi(nu)} (chi with nu <= 0: not drawn, 1)
int orc_marker_draws(uint32_t marker, uint32_t sweep, uint32_t chain, float nu, uint64_t seed, float* out) {
  orc::PhiloxDraws rng(seed);
  rng.set_chain((int)chain);
  rng.set_sweep((int)sweep);
  rng.set_marker((int)marker);
  out[0] = rng.z1; out[1] = rng.z2; out[2] = rng.u;
  out[3] = nu > 0 ? (float)rng.chi_marker(nu) : 1.0f;
  return 0;
}

}  // extern "C"
