// bwgr_oracle.hpp -- CPU restatement of bWGR's marker-effect update loop.
//
// *** TEST INFRASTRUCTURE ONLY. ***  Nothing under bwgr_b200/ (the product) may
// include, link or call this file.  Only tests/, __graft_entry__.smoke() and the
// cpu_baseline / --impl reference legs of bench.py use it, and only as the checker /
// the CPU arm, never as the thing shipped.
//
// Provenance: dependency-free C++17 restatement (plain loops, no Eigen/Rcpp/Rmath) of
//   /root/reference/src/Rcpp20260726ai.cpp      (univariate EM + Gibbs + KMUP, float32)
//   /root/reference/src/RcppEigen20230423.cpp   (MRR3 float64 :318-701, MRR3F float32 :704-1079)
//   /root/reference/R/wgr.R                     (wgr MCMC driver :2-169)
// The reference ships no tests or golden vectors for this path, and R / Rcpp / RcppEigen are absent from this image.
//   PARITY PINNED (round 2) -- the reference's own sources are compiled UNMODIFIED against stand-in RcppEigen / Rcpp headers
//   (oracle/shim/RcppEigen.h) into oracle/_ref/libbwgr_ref.so (oracle/Makefile, target `ref`: Rcpp20260726ai.cpp whole,
//   RcppEigen20230423.cpp:317-1079 = MRR3 + MRR3F).  tests/test_ref_pin.py runs both on the same inputs: the ten EM solvers,
//   the seven Gibbs samplers (same std::mt19937_64 stream, draw for draw), KMUP, and MRR3 / MRR3F under every flag incl.
//   missing phenotypes agree to float reassociation (1e-15 for the float64 MRR3); tests/golden/tpod_em.npz (<model>_ref__*) and
//   tpod_mrr3.npz are REFERENCE-EXECUTED outputs of that library (oracle/make_golden.py).  What the stand-in headers cannot
//   pin is Eigen's own packet order of float reductions and R's RNG stream (Gibbs parity vs R stays statistical).
// Also pinned: the libstdc++ std::shuffle/std::mt19937 marker order (known answers in SURVEY.md section 8a) and tpod.
//
// Third-party arithmetic restated here (absent from /root/reference):
//   Eigen (via CRAN RcppEigen, version unpinned by DESCRIPTION:15): dot / squaredNorm / sum are
//     restated with Eigen's linear-vectorised redux order for 16-byte packets (two packet
//     accumulators, then horizontal add), LLT, self-adjoint EVD (Jacobi here) and the
//     pseudo-inverse (EVD based here; vb is symmetric).
//   Rmath (R >= 4.0): rnorm / rchisq / rbinom -> std::mt19937_64 + <random> distributions.
//     R's RNG stream is irreproducible outside R; Gibbs parity with it is statistical (posterior means).  PhiloxDraws replays the
//     device's own draws instead, which makes each chain a deterministic function of the seed.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <random>
#include <vector>

namespace orc {

// ------------------------------------------------------------------------------------------------
// Eigen-style reductions (redux_impl<..., LinearVectorizedTraversal, NoUnrolling>), packet = 16 B.
// ------------------------------------------------------------------------------------------------
template <class R, class F>
static inline R reduce_sum(int n, F f) {
  constexpr int W = 16 / (int)sizeof(R);
  if (n <= 0) return R(0);
  const int a2 = (n / (2 * W)) * (2 * W), a1 = (n / W) * W;
  R res;
  if (a1) {
    R p0[W], p1[W];
    for (int l = 0; l < W; l++) p0[l] = f(l);
    if (a1 > W) {
      for (int l = 0; l < W; l++) p1[l] = f(W + l);
      for (int i = 2 * W; i < a2; i += 2 * W)
        for (int l = 0; l < W; l++) {
          p0[l] += f(i + l);
          p1[l] += f(i + W + l);
        }
      for (int l = 0; l < W; l++) p0[l] += p1[l];
      if (a1 > a2)
        for (int l = 0; l < W; l++) p0[l] += f(a2 + l);
    }
    if (W == 4) res = (p0[0] + p0[2 % W]) + (p0[1 % W] + p0[3 % W]);
    else res = p0[0] + p0[1 % W];
    for (int i = a1; i < n; i++) res += f(i);
  } else {
    res = f(0);
    for (int i = 1; i < n; i++) res += f(i);
  }
  return res;
}
template <class R> static inline R vsum(const R* x, int n) { return reduce_sum<R>(n, [&](int i) { return x[i]; }); }
template <class R> static inline R vdot(const R* x, const R* y, int n) { return reduce_sum<R>(n, [&](int i) { return x[i] * y[i]; }); }
template <class R> static inline R vsq(const R* x, int n) { return reduce_sum<R>(n, [&](int i) { return x[i] * x[i]; }); }
template <class R> static inline R vmean(const R* x, int n) { return vsum(x, n) / (R)n; }
// fvar: Rcpp20260726ai.cpp:7-9
template <class R> static inline R fvar(const R* x, int n) {
  const R m = vmean(x, n);
  return reduce_sum<R>(n, [&](int i) { R t = x[i] - m; return t * t; }) / (R)(n - 1);
}
template <class R> static inline void axpy_sub(R* e, const R* x, R s, int n) {  // e -= x*s
  for (int i = 0; i < n; i++) e[i] -= x[i] * s;
}
// ||e - x*s||^2 as Eigen evaluates (e1 = e - x*s; e1.squaredNorm()): temp then norm.
template <class R> static inline R sq_after(const R* e, const R* x, R s, R* tmp, int n) {
  for (int i = 0; i < n; i++) tmp[i] = e[i] - x[i] * s;
  return vsq(tmp, n);
}

// The marker order of every shuffled solver: std::shuffle(order, std::mt19937(iter)), cumulative.
// Rcpp20260726ai.cpp:329-331 (and :101-103, :155-158, :214-217, :372-374, :424-427).
struct Shuffler {
  std::vector<int> order;
  explicit Shuffler(int p) : order(p) { for (int j = 0; j < p; j++) order[j] = j; }
  void next(int iter) { std::shuffle(order.begin(), order.end(), std::mt19937(iter)); }
};

// ------------------------------------------------------------------------------------------------
// Univariate EM solvers.  X: n x p column-major, same element type as the arithmetic (the
// reference casts R doubles to Eigen::MatrixXf, RcppExports.cpp:115).
// ------------------------------------------------------------------------------------------------
enum EmModel { EM_RR = 0, EM_BA = 1, EM_BB = 2, EM_BC = 3, EM_BL = 4, EM_EN = 5, EM_DE = 6, EM_ML = 7, EM_BCPI = 8, EM_LASSO = 9 };

template <class R>
struct EmOut {
  R mu = 0;
  std::vector<R> b, d, hat, vbv;  // vbv: per-marker Vb (emBA/emBB)
  R Va = 0, Ve = 0, h2 = 0, Vg = 0;
  R pi = 0, Lmb = 0;  // emBCpi's updated Pi; lasso's final penalty
  int its = 0;
};

template <class R>
struct EmPar {
  R df = 10, R2 = 0.5, Pi = 0.75, alpha = 0.02;
  int it = -1;  // <0: the reference's hard-coded count (200; emEN maxit 300)
  const double* D = nullptr;  // emML: optional marker weights (:471-475), p values, cast to float like the reference does
};

template <class R>
static void xx_vx(const R* X, int n, int p, std::vector<R>& xx, std::vector<R>* vx) {
  xx.resize(p);
  if (vx) vx->resize(p);
  for (int j = 0; j < p; j++) {
    const R* x = X + (size_t)j * n;
    xx[j] = vsq(x, n);
    if (vx) (*vx)[j] = fvar(x, n);
  }
}
template <class R>
static void fitted(const R* X, int n, int p, const std::vector<R>& b, R mu, std::vector<R>& hat) {
  hat.assign(n, R(0));  // fit = gen*b (column-oriented gemv), then + mu
  for (int j = 0; j < p; j++) {
    const R bj = b[j];
    const R* x = X + (size_t)j * n;
    for (int i = 0; i < n; i++) hat[i] += x[i] * bj;
  }
  for (int i = 0; i < n; i++) hat[i] += mu;
}

// emRR: Rcpp20260726ai.cpp:308-354
template <class R>
static void emRR(const R* y, const R* X, int n, int p, const EmPar<R>& P, EmOut<R>& o) {
  const int it = P.it < 0 ? 200 : P.it;
  const R df = P.df, R2 = P.R2;
  std::vector<R> xx, vx;
  xx_vx(X, n, p, xx, &vx);
  R MSx = vsum(vx.data(), p);
  R Lmb = MSx;
  R Rho = MSx * (1 - R2) / R2;
  R vy = fvar(y, n);
  R ve = R(0.5) * vy;
  R vb = ve / MSx;
  R Se = (1 - R2) * (df + 2) * vy;
  R Sb = R2 * (df + 2) * vy / MSx;
  R mu = vmean(y, n);
  std::vector<R> b(p, R(0)), e(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  Shuffler sh(p);
  for (int i = 0; i < it; i++) {
    sh.next(i);
    for (int jj = 0; jj < p; jj++) {
      const int j = sh.order[jj];
      const R* x = X + (size_t)j * n;
      const R b0 = b[j];
      b[j] = (vdot(x, e.data(), n) + xx[j] * b0) / (xx[j] + Lmb);
      axpy_sub(e.data(), x, b[j] - b0, n);
    }
    vb = (vsq(b.data(), p) + Sb) / (p + df);
    ve = (vsq(e.data(), n) + Se) / (n + df);
    Lmb = std::sqrt(Rho * ve / vb);
    const R eM = vmean(e.data(), n);
    mu += eM;
    for (int r = 0; r < n; r++) e[r] -= eM;
  }
  o.its = it; o.mu = mu; o.b = b; o.Va = vb; o.Ve = ve; o.h2 = 1 - ve / vy;
  fitted(X, n, p, b, mu, o.hat);
}

// emBA: Rcpp20260726ai.cpp:80-128 (note: e is updated twice per marker, :108 and :111)
template <class R>
static void emBA(const R* y, const R* X, int n, int p, const EmPar<R>& P, EmOut<R>& o) {
  const int it = P.it < 0 ? 200 : P.it;
  const R df = P.df, R2 = P.R2;
  R ve = 1;
  std::vector<R> b(p, R(0)), vb(p, R(1)), Lmb(p);
  for (int j = 0; j < p; j++) Lmb[j] = ve * (R(1) / vb[j]);
  R vy = fvar(y, n);
  std::vector<R> xx, vx;
  xx_vx(X, n, p, xx, &vx);
  R MSx = vsum(vx.data(), p);
  R Sb = R2 * (df + 2) * vy / MSx;
  R Se = (1 - R2) * (df + 2) * vy;
  R mu = vmean(y, n);
  std::vector<R> e(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  Shuffler sh(p);
  for (int i = 0; i < it; i++) {
    sh.next(i);
    for (int jj = 0; jj < p; jj++) {
      const int j = sh.order[jj];
      const R* x = X + (size_t)j * n;
      const R b0 = b[j];
      const R b1 = (vdot(x, e.data(), n) + xx[j] * b0) / (xx[j] + Lmb[j]);
      axpy_sub(e.data(), x, b1 - b0, n);
      b[j] = b1;
      vb[j] = (Sb + b[j] * b[j]) / (df + 1);
      axpy_sub(e.data(), x, b1 - b0, n);
    }
    ve = (vsq(e.data(), n) + Se) / (n + df);
    for (int j = 0; j < p; j++) Lmb[j] = ve * (R(1) / vb[j]);
    const R eM = vmean(e.data(), n);
    mu += eM;
    for (int r = 0; r < n; r++) e[r] -= eM;
  }
  o.its = it; o.mu = mu; o.b = b; o.vbv = vb; o.Ve = ve; o.h2 = 1 - ve / vy;
  fitted(X, n, p, b, mu, o.hat);
}

// emBB: Rcpp20260726ai.cpp:131-187
template <class R>
static void emBB(const R* y, const R* X, int n, int p, const EmPar<R>& P, EmOut<R>& o) {
  const int it = P.it < 0 ? 200 : P.it;
  const R df = P.df, R2 = P.R2;
  R Pi = P.Pi;
  R ve = 1;
  std::vector<R> d(p, R(0)), b(p, R(0)), vb(p, R(1)), Lmb(p);
  for (int j = 0; j < p; j++) Lmb[j] = ve * (R(1) / vb[j]);
  R vy = fvar(y, n);
  if (Pi > R(0.5)) Pi = 1 - Pi;
  std::vector<R> xx, vx;
  xx_vx(X, n, p, xx, &vx);
  R MSx = vsum(vx.data(), p) * Pi;
  R Sb = R2 * (df + 2) * vy / MSx;
  R Se = (1 - R2) * (df + 2) * vy;
  R mu = vmean(y, n);
  std::vector<R> e(n), t1(n), t2(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  const R Pi0 = (1 - Pi) / Pi;
  Shuffler sh(p);
  for (int i = 0; i < it; i++) {
    const R C = R(-0.5) / std::sqrt(ve);
    sh.next(i);
    for (int jj = 0; jj < p; jj++) {
      const int j = sh.order[jj];
      const R* x = X + (size_t)j * n;
      const R b0 = b[j];
      const R b1 = (vdot(x, e.data(), n) + xx[j] * b0) / (xx[j] + Lmb[j]);
      const R n1 = sq_after(e.data(), x, b1 - b0, t1.data(), n);
      const R n2 = sq_after(e.data(), x, R(0) - b0, t2.data(), n);
      const R LR = Pi0 * std::exp(C * (n2 - n1));
      d[j] = (1 / (1 + LR));
      b[j] = b1 * d[j];
      vb[j] = (Sb + b[j] * b[j]) / (df + 1);
      axpy_sub(e.data(), x, b[j] - b0, n);
    }
    ve = (vsq(e.data(), n) + Se) / (n + df);
    for (int j = 0; j < p; j++) Lmb[j] = ve * (R(1) / vb[j]);
    const R eM = vmean(e.data(), n);
    mu += eM;
    for (int r = 0; r < n; r++) e[r] -= eM;
  }
  o.its = it; o.mu = mu; o.b = b; o.d = d; o.vbv = vb; o.Ve = ve; o.h2 = 1 - ve / vy;
  fitted(X, n, p, b, mu, o.hat);
}

// emBC: Rcpp20260726ai.cpp:190-247 (note ve=Sa, va=Se initialisation, :209-210)
template <class R>
static void emBC(const R* y, const R* X, int n, int p, const EmPar<R>& P, EmOut<R>& o) {
  const int it = P.it < 0 ? 200 : P.it;
  const R df = P.df, R2 = P.R2;
  R Pi = P.Pi;
  std::vector<R> d(p, R(0)), b(p, R(0));
  R vy = fvar(y, n);
  if (Pi > R(0.5)) Pi = 1 - Pi;
  std::vector<R> xx, vx;
  xx_vx(X, n, p, xx, &vx);
  R MSx = vsum(vx.data(), p) * Pi * (1 - Pi);
  R Sa = R2 * (df + 2) * vy / MSx;
  R Se = (1 - R2) * (df + 2) * vy;
  R mu = vmean(y, n);
  std::vector<R> e(n), t1(n), t2(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  R ve = Sa;
  R va = Se;
  R Lmb = ve / va;
  const R Pi0 = (1 - Pi) / Pi;
  Shuffler sh(p);
  for (int i = 0; i < it; i++) {
    const R C = R(-0.5) / std::sqrt(ve);
    sh.next(i);
    for (int jj = 0; jj < p; jj++) {
      const int j = sh.order[jj];
      const R* x = X + (size_t)j * n;
      const R b0 = b[j];
      const R b1 = (vdot(x, e.data(), n) + xx[j] * b0) / (xx[j] + Lmb);
      const R n1 = sq_after(e.data(), x, b1 - b0, t1.data(), n);
      const R n2 = sq_after(e.data(), x, R(0) - b0, t2.data(), n);
      const R LR = Pi0 * std::exp(C * (n2 - n1));
      d[j] = (1 / (1 + LR));
      b[j] = b1 * d[j];
      axpy_sub(e.data(), x, b[j] - b0, n);
    }
    ve = (vsq(e.data(), n) + Se) / (n + df);
    va = (vsq(b.data(), p) + Sa) / (p + df) / (vmean(d.data(), p) - Pi);
    Lmb = ve / va;
    const R eM = vmean(e.data(), n);
    mu += eM;
    for (int r = 0; r < n; r++) e[r] -= eM;
  }
  o.its = it; o.mu = mu; o.b = b; o.d = d; o.Vg = va * MSx; o.Va = va; o.Ve = ve; o.h2 = 1 - ve / vy;
  fitted(X, n, p, b, mu, o.hat);
}

// emBL: Rcpp20260726ai.cpp:357-397
template <class R>
static void emBL(const R* y, const R* X, int n, int p, const EmPar<R>& P, EmOut<R>& o) {
  const int it = P.it < 0 ? 200 : P.it;
  R h2 = P.R2;
  const R alpha = P.alpha;
  std::vector<R> b(p, R(0));
  R mu = vmean(y, n);
  std::vector<R> e(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  std::vector<R> xx;
  xx_vx<R>(X, n, p, xx, nullptr);
  const R cxx = vmean(xx.data(), p);
  const R Lmb1 = cxx * ((1 - h2) / h2) * alpha * R(0.5);
  const R Lmb2 = cxx * ((1 - h2) / h2) * (1 - alpha);
  Shuffler sh(p);
  for (int i = 0; i < it; i++) {
    sh.next(i);
    for (int jj = 0; jj < p; jj++) {
      const int j = sh.order[jj];
      const R* x = X + (size_t)j * n;
      const R b0 = b[j];
      const R OLS = (vdot(x, e.data(), n) + xx[j] * b0);
      const R Half_L2 = R(0.5) * OLS / (xx[j] + cxx);
      R G;
      if (OLS > 0) {
        G = R(0.5) * (OLS - Lmb1) / (Lmb2 + xx[j]);
        b[j] = (G > 0) ? G + Half_L2 : Half_L2;
      } else {
        G = R(0.5) * (OLS + Lmb1) / (Lmb2 + xx[j]);
        b[j] = (G < 0) ? G + Half_L2 : Half_L2;
      }
      axpy_sub(e.data(), x, b[j] - b0, n);
    }
    const R eM = vmean(e.data(), n);
    mu += eM;
    for (int r = 0; r < n; r++) e[r] -= eM;
  }
  o.its = it; o.mu = mu; o.b = b;
  fitted(X, n, p, b, mu, o.hat);
  o.h2 = 1 - fvar(e.data(), n) / fvar(y, n);
}

// emEN: Rcpp20260726ai.cpp:400-460
template <class R>
static void emEN(const R* y, const R* X, int n, int p, const EmPar<R>& P, EmOut<R>& o) {
  const int maxit = P.it < 0 ? 300 : P.it;
  const R tol = R(10e-11f);
  const R R2 = P.R2, alpha = P.alpha;
  std::vector<R> b(p, R(0)), bc(p);
  R mu = vmean(y, n);
  std::vector<R> e(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  std::vector<R> xx, vx;
  xx_vx(X, n, p, xx, &vx);
  const R cxx = vsum(vx.data(), p) * (1 - R2) / R2;
  R Ve = 0, Va = 0;
  const R Sy = std::sqrt(fvar(y, n));
  R Lmb = cxx;
  R Lmb1 = R(0.5) * Lmb * alpha * Sy;
  R Lmb2 = Lmb * (1 - alpha);
  R trAC22 = 0;
  for (int k = 0; k < p; k++) trAC22 += R(1.0) / (xx[k] + Lmb);
  int numit = 0;
  Shuffler sh(p);
  while (numit < maxit) {
    bc = b;
    sh.next(numit);
    for (int jj = 0; jj < p; jj++) {
      const int j = sh.order[jj];
      const R* x = X + (size_t)j * n;
      const R b0 = b[j];
      const R OLS = (vdot(x, e.data(), n) + xx[j] * b0);
      R b1;
      if (OLS > 0) { b1 = (OLS - Lmb1) / (Lmb2 + xx[j]); if (b1 < 0) b1 = 0; }
      else         { b1 = (OLS + Lmb1) / (Lmb2 + xx[j]); if (b1 > 0) b1 = 0; }
      b[j] = b1;
      axpy_sub(e.data(), x, b1 - b0, n);
    }
    const R eM = vmean(e.data(), n);
    mu += eM;
    for (int r = 0; r < n; r++) e[r] -= eM;
    Ve = vdot(e.data(), y, n) / (n - 1);
    Va = (vsq(b.data(), p) + trAC22 * Ve) / p;
    Lmb = Ve / Va;
    Lmb1 = R(0.5) * Lmb * alpha * Sy;
    Lmb2 = Lmb * (1 - alpha);
    ++numit;
    const R cnv = reduce_sum<R>(p, [&](int j) { return std::fabs(bc[j] - b[j]); });
    if (cnv < tol) break;
  }
  o.its = numit; o.mu = mu; o.b = b; o.Va = Va * cxx; o.Ve = Ve; o.h2 = Va * cxx / (Va * cxx + Ve);
  fitted(X, n, p, b, mu, o.hat);
}

// emDE: Rcpp20260726ai.cpp:250-306.  Ridge step with a per-marker penalty that the sweep epilogue re-estimates
// (double-exponential flavour); stops on sum |b_old - b_new| < 1e-5 or after 300 sweeps.
template <class R>
static void emDE(const R* y, const R* X, int n, int p, const EmPar<R>& P, EmOut<R>& o) {
  const int maxit = P.it < 0 ? 300 : P.it;
  const R tol = R(10e-6f), R2 = P.R2;
  R mu = vmean(y, n);
  std::vector<R> e(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  std::vector<R> xx, vx;
  xx_vx(X, n, p, xx, &vx);
  for (int k = 0; k < p; k++) if (xx[k] == 0) xx[k] = R(0.1f);  // :261
  const R cxx = vsum(vx.data(), p) * (1 - R2) / R2;
  R Ve = 0;
  std::vector<R> Vb(p, R(0)), b(p, R(0)), Lmb(p, (R)p + cxx), bc(p);
  int numit = 0;
  Shuffler sh(p);
  while (numit < maxit) {
    bc = b;
    sh.next(numit);
    for (int jj = 0; jj < p; jj++) {
      const int j = sh.order[jj];
      const R* x = X + (size_t)j * n;
      const R b0 = b[j];
      const R b1 = (vdot(x, e.data(), n) + xx[j] * b0) / (Lmb[j] + xx[j]);
      b[j] = b1;
      axpy_sub(e.data(), x, b1 - b0, n);
    }
    const R eM = vmean(e.data(), n);
    mu += eM;
    for (int r = 0; r < n; r++) e[r] -= eM;
    Ve = vdot(e.data(), y, n) / (n - 1);
    for (int j = 0; j < p; j++) Vb[j] = b[j] * b[j] + Ve / (xx[j] + Lmb[j] + R(0.0001f));
    for (int j = 0; j < p; j++) Lmb[j] = std::sqrt(cxx * Ve / Vb[j]);
    ++numit;
    const R cnv = reduce_sum<R>(p, [&](int j) { return std::fabs(bc[j] - b[j]); });
    if (cnv < tol) break;
  }
  const R sVb = vsum(Vb.data(), p);
  o.its = numit; o.mu = mu; o.b = b; o.vbv = Vb; o.Ve = Ve; o.h2 = sVb / (sVb + Ve);
  fitted(X, n, p, b, mu, o.hat);
}

// emML: Rcpp20260726ai.cpp:463-520 with D = NULL (no marker weights).  Ridge step; the variance components come from
// the moment identities ve = (y-mu)'e/n, vb = (y-mu)'(y-mu-e)/(n MSx); hat is y - e.
template <class R>
static void emML(const R* y, const R* X, int n, int p, const EmPar<R>& P, EmOut<R>& o) {
  const int maxit = P.it < 0 ? 300 : P.it;
  const R tol = R(10e-8f);
  R mu = vmean(y, n), ve = 0, vb = 0;
  std::vector<R> b(p, R(0)), bc(p), e(n), yc(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  std::vector<R> xx, vx;
  xx_vx(X, n, p, xx, &vx);
  const R MSx = vsum(vx.data(), p);
  R Lmb = MSx;
  int numit = 0;
  Shuffler sh(p);
  while (numit < maxit) {
    bc = b;
    sh.next(numit);
    for (int jj = 0; jj < p; jj++) {
      const int j = sh.order[jj];
      const R* x = X + (size_t)j * n;
      const R b0 = b[j];
      if (P.D) b[j] = (vdot(x, e.data(), n) + xx[j] * b0) / (xx[j] + Lmb / (R)(float)P.D[j]);  // :495-496
      else b[j] = (vdot(x, e.data(), n) + xx[j] * b0) / (xx[j] + Lmb);
      axpy_sub(e.data(), x, b[j] - b0, n);
    }
    const R eM = vmean(e.data(), n);
    mu += eM;
    for (int r = 0; r < n; r++) e[r] -= eM;
    for (int r = 0; r < n; r++) yc[r] = y[r] - mu;
    ve = vdot(yc.data(), e.data(), n) / (R)n;
    vb = reduce_sum<R>(n, [&](int r) { return yc[r] * (yc[r] - e[r]); }) / (R)(n * MSx);
    Lmb = ve / vb;
    ++numit;
    const R cnv = reduce_sum<R>(p, [&](int j) { return std::fabs(bc[j] - b[j]); });
    if (cnv < tol) break;
  }
  o.its = numit; o.mu = mu; o.b = b; o.Vg = vb; o.Va = vb * MSx; o.Ve = ve; o.h2 = vb * MSx / (vb * MSx + ve);
  o.hat.resize(n);
  for (int r = 0; r < n; r++) o.hat[r] = y[r] - e[r];
}

// emBCpi: Rcpp20260726ai.cpp:1502-1546.  emBC's step in the natural marker order, with the mixture proportion
// re-estimated after every sweep from the mean inclusion (and MSx, Sa with it).
template <class R>
static void emBCpi(const R* y, const R* X, int n, int p, const EmPar<R>& P, EmOut<R>& o) {
  const int it = P.it < 0 ? 200 : P.it;
  const R df = P.df, R2 = P.R2;
  R Pi = P.Pi;
  std::vector<R> d(p, R(0)), b(p, R(0));
  const R vy = fvar(y, n);
  if (Pi > R(0.5)) Pi = 1 - Pi;
  std::vector<R> xx, vx;
  xx_vx(X, n, p, xx, &vx);
  const R PriorPi = Pi, svx = vsum(vx.data(), p);
  R MSx = svx * Pi * (1 - Pi);
  R Sa = R2 * (df + 2) * vy / MSx;
  const R Se = (1 - R2) * (df + 2) * vy;
  R mu = vmean(y, n);
  std::vector<R> e(n), t1(n), t2(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  R ve = Sa, va = Se, Lmb = ve / va, Pi0 = (1 - Pi) / Pi;
  for (int i = 0; i < it; i++) {
    const R C = R(-0.5) / std::sqrt(ve);
    for (int j = 0; j < p; j++) {
      const R* x = X + (size_t)j * n;
      const R b0 = b[j];
      const R b1 = (vdot(x, e.data(), n) + xx[j] * b0) / (xx[j] + Lmb);
      const R n1 = sq_after(e.data(), x, b1 - b0, t1.data(), n);
      const R n2 = sq_after(e.data(), x, R(0) - b0, t2.data(), n);
      const R LR = Pi0 * std::exp(C * (n2 - n1));
      d[j] = 1 / (1 + LR);
      b[j] = b1 * d[j];
      axpy_sub(e.data(), x, b[j] - b0, n);
    }
    const R dm = vmean(d.data(), p);
    Pi = ((1 - dm) * p + PriorPi * df) / (p + df);
    Pi0 = (1 - Pi) / Pi;
    MSx = svx * Pi * (1 - Pi);
    Sa = R2 * (df + 2) * vy / MSx;
    ve = (vsq(e.data(), n) + Se) / (n + df);
    va = (vsq(b.data(), p) + Sa) / (p + df) / (dm - Pi);
    Lmb = ve / va;
    const R eM = vmean(e.data(), n);
    mu += eM;
    for (int r = 0; r < n; r++) e[r] -= eM;
  }
  o.its = it; o.mu = mu; o.b = b; o.d = d; o.pi = Pi; o.Vg = va * MSx; o.Va = va; o.Ve = ve; o.h2 = 1 - ve / vy;
  fitted(X, n, p, b, mu, o.hat);
}

// lasso: Rcpp20260726ai.cpp:1463-1500.  Soft-threshold coordinate descent in the natural order; the penalty is
// re-estimated after every sweep from how much of each marker's x'e the threshold removed.
template <class R>
static void lasso(const R* y, const R* X, int n, int p, const EmPar<R>& P, EmOut<R>& o) {
  const int maxit = P.it < 0 ? 300 : P.it;
  const R tol = R(10e-8f);
  R mu = vmean(y, n);
  std::vector<R> b(p, R(0)), bc(p), yx(p, R(0)), e(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  std::vector<R> xx;
  xx_vx<R>(X, n, p, xx, nullptr);
  R Lmb = vmean(xx.data(), p) / p;
  int numit = 0;
  while (numit < maxit) {
    bc = b;
    for (int j = 0; j < p; j++) {
      const R* x = X + (size_t)j * n;
      axpy_sub(e.data(), x, -b[j], n);  // e += x b_j
      yx[j] = vdot(e.data(), x, n);
      if (yx[j] > 0) { b[j] = (yx[j] - Lmb) / xx[j]; if (b[j] < 0) b[j] = 0; }
      else           { b[j] = (yx[j] + Lmb) / xx[j]; if (b[j] > 0) b[j] = 0; }
      axpy_sub(e.data(), x, b[j], n);
    }
    R tmp = 0;
    for (int j = 0; j < p; j++) tmp += std::fabs(yx[j]) - std::fabs(b[j] * xx[j]);
    Lmb = R(2) * tmp / p;
    Lmb = R(2) * std::sqrt(std::fabs(Lmb));
    const R eM = vmean(e.data(), n);
    mu += eM;
    for (int r = 0; r < n; r++) e[r] -= eM;
    ++numit;
    const R cnv = reduce_sum<R>(p, [&](int j) { return std::fabs(bc[j] - b[j]); });
    if (cnv < tol) break;
  }
  o.its = numit; o.mu = mu; o.b = b; o.Lmb = Lmb; o.h2 = 1 - (vdot(e.data(), y, n) / (n - 1)) / fvar(y, n);
  o.hat.resize(n);
  for (int r = 0; r < n; r++) o.hat[r] = y[r] - e[r];
}

template <class R>
static void em_fit(int model, const R* y, const R* X, int n, int p, const EmPar<R>& P, EmOut<R>& o) {
  switch (model) {
    case EM_RR: emRR(y, X, n, p, P, o); break;
    case EM_BA: emBA(y, X, n, p, P, o); break;
    case EM_BB: emBB(y, X, n, p, P, o); break;
    case EM_BC: emBC(y, X, n, p, P, o); break;
    case EM_BL: emBL(y, X, n, p, P, o); break;
    case EM_EN: emEN(y, X, n, p, P, o); break;
    case EM_DE: emDE(y, X, n, p, P, o); break;
    case EM_ML: emML(y, X, n, p, P, o); break;
    case EM_BCPI: emBCpi(y, X, n, p, P, o); break;
    case EM_LASSO: lasso(y, X, n, p, P, o); break;
  }
}

// ------------------------------------------------------------------------------------------------
// Draw sources.  The samplers below ask for every random number at a named site:
//   effect(m, s)    marker effect  ~ N(m, s)          excluded(s)    excluded effect ~ N(0, s)
//   include(q)      inclusion test, true with prob. q  chi_marker(nu) per-marker chi-square
//   intercept(m, s) intercept of a Gibbs sweep         chi_e(nu), chi_b(nu)  residual / marker variance of a Gibbs sweep
//   wgr_Ve, wgr_Va, wgr_mu0, wgr_Vb(j, .), wgr_Vp  the draws of wgr's driver      rows(...)  wgr's row sample of one iteration
// and tell the source where they are (set_sweep, set_marker, set_chain).
// ------------------------------------------------------------------------------------------------
// Rng: the stand-in for Rmath (R::rnorm / R::rchisq / R::rbinom), one std::mt19937_64 stream consumed in the reference's order.
struct Rng {
  std::mt19937_64 g;
  explicit Rng(uint64_t seed) : g(seed) {}
  double rnorm(double m, double s) { std::normal_distribution<double> d(0.0, 1.0); return m + s * d(g); }
  double rchisq(double df) { std::chi_squared_distribution<double> d(df); return d(g); }
  // R::rbinom(1, p): NaN in -> NaN out (so "== 1" is false)
  double rbinom1(double p) {
    if (!(p == p)) return std::numeric_limits<double>::quiet_NaN();
    std::uniform_real_distribution<double> u(0.0, 1.0);
    return u(g) < p ? 1.0 : 0.0;
  }
  void set_sweep(int) {}
  void set_marker(int) {}
  double effect(double m, double s) { return rnorm(m, s); }
  double excluded(double s) { return rnorm(0, s); }
  bool include(double q) { return rbinom1(q) == 1; }
  double chi_marker(double nu) { return rchisq(nu); }
  double intercept(double m, double s) { return rnorm(m, s); }
  double chi_e(double nu) { return rchisq(nu); }
  double chi_b(double nu) { return rchisq(nu); }
  double wgr_Ve(double nu) { return rchisq(nu); }
  double wgr_Va(double nu) { return rchisq(nu); }
  double wgr_mu0(double m, double s) { return rnorm(m, s); }
  double wgr_Vb(int, double nu) { return rchisq(nu); }
  double wgr_Vp(double nu) { return rchisq(nu); }
  // sample(n, nuse, rp) of R/wgr.R:68, unsorted, in rows[0, nuse)
  void rows(int n, int nuse, bool rp, std::vector<int>& rows) {
    if (rp) {
      rows.resize(std::max(n, nuse));
      std::uniform_int_distribution<int> pick(0, n - 1);
      for (int r = 0; r < nuse; r++) rows[r] = pick(g);
    } else {
      for (int r = 0; r < n; r++) rows[r] = r;
      for (int r = 0; r < nuse; r++) { std::uniform_int_distribution<int> pick(r, n - 1); std::swap(rows[r], rows[pick(g)]); }
    }
  }
};

// PhiloxDraws: the device's counter-addressed draws (Philox4x32-10, key = the seed), restated on the host so that a chain is a
// deterministic function of the seed and can be compared with the device draw for draw.  Counters:
//   marker draws z1, z2, u    (marker, sweep, chain, 0)        per-marker chi-square   (marker, sweep, chain, 1 + (attempt << 8))
//   Gibbs sweep epilogue      (0xFFFFFFFF, sweep, chain, p): intercept p = 0, chi_e p = 1, chi_b p = 2
//   wgr driver                (0xFFFFFFFE, sweep, 0, p): mu0 p = 0, Ve p = 1, Va p = 2       wgr per-marker Vb  (marker, sweep, 0, 3)
// Every draw is made in float, as on the device; the sampler may then run in float or double on the same draws.  wgr's row samples
// come from std::mt19937_64(seed ^ 0x9E3779B97F4A7C15) with int64 uniform_int_distribution, as in the C ABI's bagged driver.
// The source records how close every accept / reject decision came to the other outcome: q[] (the inclusion probability of each
// include() call) and u[] (the uniform it was tested with), and mt_margin, the smallest |log u - (0.5 x^2 + d - d v + d log v)| / (1 + d)
// of every Marsaglia-Tsang acceptance test.
namespace philox {
inline void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
  for (int r = 0; r < 10; r++) {
    const uint64_t p0 = (uint64_t)M0 * c[0], p1 = (uint64_t)M1 * c[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1, n3 = (uint32_t)p0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += W0; k1 += W1;
  }
}
inline float u01(uint32_t x) { return (float)((x >> 8) + 1) * (1.0f / 16777216.0f); }  // (0, 1], 24 bits
// sincospi(t) as sin / cos of pi t in double, rounded to float
inline void box_muller(uint32_t a, uint32_t b, float& z0, float& z1) {
  const float r = std::sqrt(-2.0f * std::log(u01(a)));
  const double t = 3.14159265358979323846 * (double)(2.0f * u01(b));
  z0 = r * (float)std::cos(t);
  z1 = r * (float)std::sin(t);
}
// chi-square(nu) = 2 Gamma(nu / 2) by Marsaglia-Tsang, each attempt its own counter; a < 1 is boosted by u^(1/a)
inline float rchisq(float nu, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t purpose, uint32_t k0, uint32_t k1, double& margin) {
  float a = 0.5f * nu;
  const bool boost = a < 1.0f;
  if (boost) a += 1.0f;
  const float d = a - (1.0f / 3.0f), cc = 1.0f / std::sqrt(9.0f * d);
  float out = d, ub = 1.0f;
  for (uint32_t att = 0; att < 64; att++) {
    uint32_t c[4] = {c0, c1, c2, purpose + (att << 8)};
    philox4x32_10(c, k0, k1);
    float x, unused;
    box_muller(c[0], c[1], x, unused);
    const float u = u01(c[2]);
    ub = u01(c[3]);
    float v = 1.0f + cc * x;
    if (v <= 0.0f) continue;
    v = v * v * v;
    const float lhs = std::log(u), rhs = 0.5f * x * x + d - d * v + d * std::log(v);
    margin = std::min(margin, (double)std::fabs(lhs - rhs) / (1.0 + d));
    if (lhs < rhs) { out = d * v; break; }
  }
  if (boost) out *= std::pow(ub, 1.0f / (0.5f * nu));
  return 2.0f * out;
}
}  // namespace philox

struct PhiloxDraws {
  uint32_t k0, k1, chain = 0, sweep = 0, marker = 0;
  float z1 = 0, z2 = 0, u = 0;
  std::vector<float> q, uq;
  double mt_margin = std::numeric_limits<double>::infinity();
  uint64_t seed;
  std::mt19937_64 row_gen;
  explicit PhiloxDraws(uint64_t s) : k0((uint32_t)s), k1((uint32_t)(s >> 32)), seed(s), row_gen(s ^ 0x9E3779B97F4A7C15ull) {}
  void set_chain(int c) { chain = (uint32_t)c; }
  void set_sweep(int i) { sweep = (uint32_t)i; }
  void set_marker(int j) {
    marker = (uint32_t)j;
    uint32_t c[4] = {marker, sweep, chain, 0u};
    philox::philox4x32_10(c, k0, k1);
    philox::box_muller(c[0], c[1], z1, z2);
    u = philox::u01(c[2]);
  }
  double effect(double m, double s) { return m + s * (double)z1; }
  double excluded(double s) { return s * (double)z2; }
  bool include(double qj) { q.push_back((float)qj); uq.push_back(u); return (double)u < qj; }
  double chi_marker(double nu) { return philox::rchisq((float)nu, marker, sweep, chain, 1u, k0, k1, mt_margin); }
  double scalar_normal(uint32_t c0, uint32_t ch) {
    uint32_t c[4] = {c0, sweep, ch, 0u};
    philox::philox4x32_10(c, k0, k1);
    float z, unused;
    philox::box_muller(c[0], c[1], z, unused);
    return z;
  }
  double intercept(double m, double s) { return m + s * scalar_normal(0xFFFFFFFFu, chain); }
  double chi_e(double nu) { return philox::rchisq((float)nu, 0xFFFFFFFFu, sweep, chain, 1u, k0, k1, mt_margin); }
  double chi_b(double nu) { return philox::rchisq((float)nu, 0xFFFFFFFFu, sweep, chain, 2u, k0, k1, mt_margin); }
  double wgr_mu0(double m, double s) { return m + s * scalar_normal(0xFFFFFFFEu, 0u); }
  double wgr_Ve(double nu) { return philox::rchisq((float)nu, 0xFFFFFFFEu, sweep, 0u, 1u, k0, k1, mt_margin); }
  double wgr_Va(double nu) { return philox::rchisq((float)nu, 0xFFFFFFFEu, sweep, 0u, 2u, k0, k1, mt_margin); }
  double wgr_Vb(int j, double nu) { return philox::rchisq((float)nu, (uint32_t)j, sweep, 0u, 3u, k0, k1, mt_margin); }
  // wgr with eigK has no device counters (its driver draws with numpy): a replay of it is not defined
  double wgr_Vp(double) { return std::numeric_limits<double>::quiet_NaN(); }
  void rows(int n, int nuse, bool rp, std::vector<int>& rows) {
    if (rp) {
      rows.resize(std::max(n, nuse));
      std::uniform_int_distribution<int64_t> pick(0, n - 1);
      for (int r = 0; r < nuse; r++) rows[r] = (int)pick(row_gen);
    } else {
      for (int r = 0; r < n; r++) rows[r] = r;
      for (int r = 0; r < nuse; r++) { std::uniform_int_distribution<int64_t> pick(r, n - 1); std::swap(rows[r], rows[pick(row_gen)]); }
    }
  }
};

// ------------------------------------------------------------------------------------------------
// Univariate Gibbs samplers (float32 state; natural marker order).
// ------------------------------------------------------------------------------------------------
enum GibbsModel { GB_RR = 0, GB_A = 1, GB_B = 2, GB_C = 3, GB_L = 4, GB_CPI = 5, GB_DPI = 6 };

template <class R>
struct GibbsOut {
  R mu = 0, vb = 0, ve = 0, h2 = 0, MSx = 0, pi = 0;  // pi: BayesCpi / BayesDpi (1 - mean inclusion)
  std::vector<R> b, d, hat, vbv;
};

// BayesRR :812-855, BayesA :589-635, BayesB :638-699, BayesC :702-759, BayesL :762-809, BayesCpi :858-919,
// BayesDpi :922-987 of Rcpp20260726ai.cpp.  BayesL = BayesA with Lmb_j = sqrt(Phi ve / vb_j) after the first sweep;
// BayesCpi = BayesC started at pi = 0.5 whose prior scale Sb follows the mean inclusion (the mixing odds Pi0 stay fixed);
// BayesDpi = per-marker variances with the Kuo-Mallick style acceptance min(1, (1 - pi) exp(C(|e1|^2 - |e2|^2))), pi = mean(d).
template <class R, class Draws>
static void gibbs_fit(int model, const R* y, const R* X, int n, int p, R it_f, R bi_f, R pi, R df, R R2,
                      Draws& rng, GibbsOut<R>& o) {
  const int iit = (int)it_f, ibi = (int)bi_f;
  const R MCMC = it_f - bi_f;
  std::vector<R> xx, vx;
  xx_vx(X, n, p, xx, &vx);
  const R MSx = vsum(vx.data(), p);
  const R vy = fvar(y, n);
  if (model == GB_CPI || model == GB_DPI) pi = R(0.5f);  // :870, :934 (not an argument of these two)
  const bool c_like = (model == GB_C || model == GB_CPI);
  R Sb = c_like ? df * R2 * vy / MSx / (1 - pi) : R2 * df * vy / MSx;
  const R Se = c_like ? df * (1 - R2) * vy : (1 - R2) * df * vy;
  const R Phi = MSx * (1 - R2) / R2;  // BayesL :773
  const bool per_marker = (model == GB_A || model == GB_B || model == GB_L || model == GB_DPI);
  const bool spike = (model == GB_B || model == GB_C || model == GB_CPI || model == GB_DPI);
  R PiSum = 0;
  std::vector<R> d(p, R(0)), b(p, R(0)), D(p, R(0)), B(p, R(0)), VBv(p, R(0));
  std::vector<R> vbv(p, Sb), Lmbv(p);
  R ve = vy, vb = Sb, VB = 0, MU = 0, VE = 0;
  for (int j = 0; j < p; j++) Lmbv[j] = ve * (R(1) / vbv[j]);
  R Lmb = ve / vb;
  R mu = vmean(y, n);
  std::vector<R> e(n), t1(n), t2(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  const R Pi0 = pi / (R(1.0) - pi);
  for (int i = 0; i < iit; i++) {
    const R C = R(-0.5) / std::sqrt(ve);
    rng.set_sweep(i);
    for (int j = 0; j < p; j++) {
      rng.set_marker(j);
      const R* x = X + (size_t)j * n;
      const R L = per_marker ? Lmbv[j] : Lmb;
      const R b0 = b[j];
      const R sd = std::sqrt(ve / (xx[j] + L));
      const R b1 = (R)rng.effect((vdot(x, e.data(), n) + xx[j] * b0) / (xx[j] + L), sd);
      if (model == GB_CPI || model == GB_DPI) {  // both draw b2 before the test (:886, :951)
        const R b2 = (R)rng.excluded(sd);
        const R n1 = sq_after(e.data(), x, b1 - b0, t1.data(), n);
        const R n2 = sq_after(e.data(), x, (model == GB_DPI ? b2 : R(0)) - b0, t2.data(), n);
        R pj;
        if (model == GB_CPI) pj = R(1.0) / (R(1.0) + Pi0 * std::exp(C * (n2 - n1)));
        else { pj = (1 - pi) * std::exp(C * (n1 - n2)); if (pj > 1) pj = 1; }
        if (rng.include(pj)) { b[j] = b1; d[j] = 1; }
        else { b[j] = b2; d[j] = 0; }
      } else if (spike) {
        const R n1 = sq_after(e.data(), x, b1 - b0, t1.data(), n);
        const R n2 = sq_after(e.data(), x, R(0) - b0, t2.data(), n);
        const R LR = Pi0 * std::exp(C * (n2 - n1));
        const R pj = R(1.0) / (R(1.0) + LR);
        if (rng.include(pj)) { b[j] = b1; d[j] = 1; }
        else { b[j] = (R)rng.excluded(sd); d[j] = 0; }
      } else {
        b[j] = b1;
      }
      if (per_marker) vbv[j] = (Sb + b[j] * b[j]) / (R)rng.chi_marker(df + 1);
      axpy_sub(e.data(), x, b[j] - b0, n);
    }
    const R eM = (R)rng.intercept(vmean(e.data(), n), std::sqrt(ve / n));
    mu += eM;
    for (int r = 0; r < n; r++) e[r] -= eM;
    if (model == GB_RR) {  // :841-843 (ve first, then vb)
      ve = (vsq(e.data(), n) + Se) / (R)rng.chi_e(n + df);
      vb = (vsq(b.data(), p) + Sb) / (R)rng.chi_b(p + df);
      Lmb = ve / vb;
    } else if (c_like) {  // :745-747, :903-907 (vb first, then ve)
      vb = (vsq(b.data(), p) + Sb) / (R)rng.chi_b(df + p);
      ve = (vsq(e.data(), n) + Se) / (R)rng.chi_e(n + df);
      Lmb = ve / vb;
      if (model == GB_CPI) { pi = vmean(d.data(), p); Sb = df * R2 * vy / MSx / (1 - pi); }  // Pi0 is NOT refreshed (:906-907)
    } else {
      ve = (vsq(e.data(), n) + Se) / (R)rng.chi_e(n + df);
      if (model == GB_L) for (int j = 0; j < p; j++) Lmbv[j] = std::sqrt(Phi * ve / vbv[j]);  // :799
      else for (int j = 0; j < p; j++) Lmbv[j] = ve * (R(1) / vbv[j]);
      if (model == GB_DPI) pi = vmean(d.data(), p);  // :969
    }
    if (i > ibi) {  // sic: i>ibi yet divided by it-bi (:624-627)
      MU += mu; VE += ve;
      for (int j = 0; j < p; j++) B[j] += b[j];
      if (spike) for (int j = 0; j < p; j++) D[j] += d[j];
      if (per_marker) for (int j = 0; j < p; j++) VBv[j] += vbv[j];
      else VB += vb;
      PiSum += pi;
    }
  }
  MU /= MCMC; VE /= MCMC;
  for (int j = 0; j < p; j++) { B[j] /= MCMC; D[j] /= MCMC; VBv[j] /= MCMC; }
  VB /= MCMC;
  R vg = per_marker ? vsum(VBv.data(), p) : VB * MSx;
  if (model == GB_CPI || model == GB_DPI) o.pi = 1 - PiSum / MCMC;  // :911, :975
  if (model == GB_CPI) vg = VB * MSx / o.pi;                         // :913
  o.mu = MU; o.b = B; o.d = D; o.vbv = VBv; o.vb = VB; o.ve = VE; o.h2 = vg / (vg + VE); o.MSx = MSx;
  fitted(X, n, p, B, MU, o.hat);
}

// KMUP: Rcpp20260726ai.cpp:12-38.  One Kuo-Mallick sweep, state updated in place.
// ratio_form=false restates the reference literally (exp(C*||e1||^2) etc., which underflows to
// NaN -> "else" branch for large n*Ve); ratio_form=true is the algebraically identical
// 1/(1+pi/(1-pi)*exp(C*(||e2||^2-||e1||^2))) that the CUDA path implements.
template <class R, class Draws>
static void kmup(const R* X, int n, int p, R* b, R* d, const R* xx, R* e, const R* L, R Ve, R pi, Draws& rng, bool ratio_form) {
  std::vector<R> e1(n), e2(n);
  const R C = R(-0.5f) / std::sqrt(Ve);
  for (int j = 0; j < p; j++) {
    rng.set_marker(j);
    const R* x = X + (size_t)j * n;
    const R b0 = b[j];
    const R sd = std::sqrt(Ve / (xx[j] + L[j]));
    const R b1 = (R)rng.effect((vdot(x, e, n) + xx[j] * b0) / (xx[j] + L[j]), sd);
    const R b2 = (R)rng.excluded(sd);
    for (int i = 0; i < n; i++) e1[i] = e[i] - x[i] * (b1 - b0);
    if (pi > 0) {
      for (int i = 0; i < n; i++) e2[i] = e[i] - x[i] * (b2 - b0);
      R pj;
      if (ratio_form) {
        pj = R(1.0f) / (R(1.0f) + (pi / (1 - pi)) * std::exp(C * (vsq(e2.data(), n) - vsq(e1.data(), n))));
      } else {
        const R cj = (1 - pi) * std::exp(C * vsq(e1.data(), n));
        const R dj = (pi)*std::exp(C * vsq(e2.data(), n));
        pj = cj / (cj + dj);
      }
      if (rng.include(pj)) { b[j] = b1; d[j] = 1; std::memcpy(e, e1.data(), sizeof(R) * n); }
      else { b[j] = b2; d[j] = 0; std::memcpy(e, e2.data(), sizeof(R) * n); }
    } else {
      d[j] = 1; b[j] = b1; std::memcpy(e, e1.data(), sizeof(R) * n);
    }
  }
}


// ------------------------------------------------------------------------------------------------
// Two-design solvers (SURVEY 8f rank 3): y = mu + X1 b1 + X2 b2 + e, the per-marker step of the univariate solvers looped over two
// marker matrices with one shared residual.  BayesA2 :990-1069, BayesB2 :1072-1154, BayesRR2 :1157-1218, emML2 :1221-1305 of
// Rcpp20260726ai.cpp.  Draws are made in the reference's order (the marker's variance right after its effect).
// ------------------------------------------------------------------------------------------------
enum TwoDesignModel { TD_A2 = 0, TD_B2 = 1, TD_RR2 = 2 };
struct TwoDesignOut {
  float mu = 0, ve = 0, h2 = 0, vb1s = 0, vb2s = 0, MSx1 = 0, MSx2 = 0;
  int its = 0;
  std::vector<float> b1, b2, d1, d2, vb1, vb2, hat, u1, u2;
};
static inline void gibbs2_fit(int model, const float* y, const float* X1, const float* X2, int n, int p1, int p2, float it_f, float bi_f,
                              float pi, float df, float R2, uint64_t seed, TwoDesignOut& o) {
  Rng rng(seed);
  const int iit = (int)it_f, ibi = (int)bi_f;
  const int P[2] = {p1, p2};
  const float* X[2] = {X1, X2};
  std::vector<float> xx[2], vx[2], b[2], d[2], vbv[2], Lv[2], B[2], D[2], VBv[2];
  float MSx[2], Sb[2], Lmb[2], vbs[2] = {0, 0}, VBs[2] = {0, 0};
  const float vy = fvar(y, n);
  for (int q = 0; q < 2; q++) {
    xx_vx(X[q], n, P[q], xx[q], &vx[q]);
    MSx[q] = vsum(vx[q].data(), P[q]);
    Sb[q] = R2 * df * vy / MSx[q];
    Lmb[q] = MSx[q];  // BayesRR2 :1181
    b[q].assign(P[q], 0.0f); d[q].assign(P[q], 0.0f); B[q].assign(P[q], 0.0f); D[q].assign(P[q], 0.0f); VBv[q].assign(P[q], 0.0f);
    vbv[q].assign(P[q], Sb[q]);
  }
  const float Se = (1 - R2) * df * vy;
  float mu = vmean(y, n), ve = vy, MU = 0, VE = 0;
  for (int q = 0; q < 2; q++) { Lv[q].resize(P[q]); for (int j = 0; j < P[q]; j++) Lv[q][j] = ve * (1.0f / vbv[q][j]); }
  std::vector<float> e(n), e1(n), e2(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  for (int i = 0; i < iit; i++) {
    const float C = -0.5f / std::sqrt(ve);
    for (int q = 0; q < 2; q++) {
      for (int j = 0; j < P[q]; j++) {
        const float* x = X[q] + (size_t)j * n;
        const float b0 = b[q][j];
        const float L = model == TD_RR2 ? Lmb[q] : Lv[q][j];
        const float sd = std::sqrt(ve / (xx[q][j] + L));
        const float bt1 = (float)rng.rnorm((vdot(x, e.data(), n) + xx[q][j] * b0) / (xx[q][j] + L), sd);
        float bn = bt1;
        if (model == TD_B2) {  // :1106-1118
          const float bt2 = (float)rng.rnorm(0, sd);
          for (int r = 0; r < n; r++) { e1[r] = e[r] - x[r] * (bt1 - b0); e2[r] = e[r] - x[r] * (bt2 - b0); }
          const float cj = (1 - pi) * std::exp(C * vsq(e1.data(), n));
          const float dj = (pi)*std::exp(C * vsq(e2.data(), n));
          const float pj = cj / (cj + dj);
          if (rng.rbinom1(pj) == 1) { bn = bt1; d[q][j] = 1; } else { bn = bt2; d[q][j] = 0; }
        }
        b[q][j] = bn;
        if (model != TD_RR2) vbv[q][j] = (Sb[q] + bn * bn) / (float)rng.rchisq(df + 1);
        for (int r = 0; r < n; r++) e[r] -= x[r] * (bn - b0);
      }
    }
    const float eM = (float)rng.rnorm(vmean(e.data(), n), std::sqrt(ve / n));
    mu += eM;
    for (int r = 0; r < n; r++) e[r] -= eM;
    ve = (vsq(e.data(), n) + Se) / (float)rng.rchisq(n + df);
    for (int q = 0; q < 2; q++) {
      if (model == TD_RR2) { vbs[q] = (Sb[q] + vsq(b[q].data(), P[q])) / (float)rng.rchisq(df + P[q]); Lmb[q] = ve / vbs[q]; }
      else for (int j = 0; j < P[q]; j++) Lv[q][j] = ve * (1.0f / vbv[q][j]);
    }
    if (i > ibi) {
      MU += mu; VE += ve;
      for (int q = 0; q < 2; q++) {
        for (int j = 0; j < P[q]; j++) { B[q][j] += b[q][j]; D[q][j] += d[q][j]; VBv[q][j] += vbv[q][j]; }
        VBs[q] += vbs[q];
      }
    }
  }
  const float MCMC = it_f - bi_f;
  MU /= MCMC; VE /= MCMC;
  for (int q = 0; q < 2; q++) {
    for (int j = 0; j < P[q]; j++) { B[q][j] /= MCMC; D[q][j] /= MCMC; VBv[q][j] /= MCMC; }
    VBs[q] /= MCMC;
  }
  const float vg = model == TD_RR2 ? VBs[0] * MSx[0] + VBs[1] * MSx[1] : vsum(VBv[0].data(), p1) + vsum(VBv[1].data(), p2);
  o.h2 = vg / (vg + VE);
  o.mu = MU; o.ve = VE; o.vb1s = VBs[0]; o.vb2s = VBs[1]; o.MSx1 = MSx[0]; o.MSx2 = MSx[1];
  o.b1 = B[0]; o.b2 = B[1]; o.d1 = D[0]; o.d2 = D[1]; o.vb1 = VBv[0]; o.vb2 = VBv[1];
  o.hat.assign(n, 0.0f);
  for (int q = 0; q < 2; q++)
    for (int j = 0; j < P[q]; j++) {
      const float* x = X[q] + (size_t)j * n;
      for (int r = 0; r < n; r++) o.hat[r] += x[r] * B[q][j];
    }
  for (int r = 0; r < n; r++) o.hat[r] += MU;
}

// emML2 :1221-1305: natural marker order, at most 350 sweeps, stop when sum |db| < 1e-7; D1 / D2 = optional marker weights
// (penalty Lmb / D[j]).
static inline void emml2_fit(const float* y, const float* X1, const float* X2, int n, int p1, int p2, const double* D1, const double* D2,
                             TwoDesignOut& o) {
  const int maxit = 350;
  const float tol = 10e-8f;
  const int P[2] = {p1, p2};
  const float* X[2] = {X1, X2};
  const double* Dw[2] = {D1, D2};
  std::vector<float> xx[2], vx[2], b[2], bc[2], dw[2], u[2];
  float MSx[2], Lmb[2], vb[2] = {0, 0};
  for (int q = 0; q < 2; q++) {
    xx_vx(X[q], n, P[q], xx[q], &vx[q]);
    MSx[q] = vsum(vx[q].data(), P[q]);
    Lmb[q] = MSx[q];
    b[q].assign(P[q], 0.0f);
    dw[q].assign(P[q], 1.0f);
    if (Dw[q]) for (int j = 0; j < P[q]; j++) dw[q][j] = (float)Dw[q][j];
    u[q].assign(n, 0.0f);
  }
  float mu = vmean(y, n), ve = 0;
  std::vector<float> e(n), cY(n);
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  int numit = 0;
  while (numit < maxit) {
    float cnv = 0;
    for (int q = 0; q < 2; q++) {
      bc[q] = b[q];
      for (int j = 0; j < P[q]; j++) {
        const float* x = X[q] + (size_t)j * n;
        const float b0 = b[q][j];
        const float bn = Dw[q] ? (vdot(x, e.data(), n) + xx[q][j] * b0) / (xx[q][j] + Lmb[q] / dw[q][j])
                               : (vdot(x, e.data(), n) + xx[q][j] * b0) / (xx[q][j] + Lmb[q]);
        b[q][j] = bn;
        for (int r = 0; r < n; r++) e[r] -= x[r] * (bn - b0);
      }
    }
    for (int q = 0; q < 2; q++) {  // u = X b, column by column like Eigen's gemv
      std::fill(u[q].begin(), u[q].end(), 0.0f);
      for (int j = 0; j < P[q]; j++) {
        const float* x = X[q] + (size_t)j * n;
        const float bj = b[q][j];
        for (int r = 0; r < n; r++) u[q][r] += x[r] * bj;
      }
    }
    const float eM = vmean(e.data(), n);
    mu += eM;
    for (int r = 0; r < n; r++) { e[r] -= eM; cY[r] = u[0][r] + u[1][r] + e[r]; }
    ve = vdot(e.data(), cY.data(), n) / (float)n;
    for (int q = 0; q < 2; q++) { vb[q] = (vdot(u[q].data(), cY.data(), n) / (float)n) / MSx[q]; Lmb[q] = ve / vb[q]; }
    ++numit;
    for (int q = 0; q < 2; q++) cnv += reduce_sum<float>(P[q], [&](int j) { return std::fabs(bc[q][j] - b[q][j]); });
    if (cnv < tol) break;
  }
  o.its = numit; o.mu = mu; o.ve = ve; o.vb1s = vb[0]; o.vb2s = vb[1]; o.MSx1 = MSx[0]; o.MSx2 = MSx[1];
  o.h2 = 1 - ve / fvar(y, n);
  o.b1 = b[0]; o.b2 = b[1]; o.u1 = u[0]; o.u2 = u[1];
  o.hat.resize(n);
  for (int r = 0; r < n; r++) o.hat[r] = mu + u[0][r] + u[1][r];
}

// KMUP2: Rcpp20260726ai.cpp:41-77.  The bagged sweep of wgr(bag != 1): only the rows `use` enter; note (H.e0 + b0) without the xx
// factor (:59, sic) and xx scaled by bg = n0 / n.  e_out has length nuse.
template <class R, class Draws>
static void kmup2(const R* X, int n0, int p, const float* use, int nuse, R* b, R* d, const R* xx, const R* E, R* e_out, const R* L, R Ve,
                  R pi, Draws& rng, bool ratio_form) {
  const int n = nuse;
  const R C = R(-0.5f) / std::sqrt(Ve);
  const R bg = (R)((float)n0 / (float)n);
  std::vector<R> e0(n), H(n), e1(n), e2(n);
  for (int k = 0; k < n; k++) e0[k] = E[(int)use[k]];
  for (int j = 0; j < p; j++) {
    rng.set_marker(j);
    for (int x = 0; x < n; x++) H[x] = X[(size_t)j * n0 + (int)use[x]];
    const R b0 = b[j];
    const R sd = std::sqrt(Ve / (xx[j] * bg + L[j]));
    const R b1 = (R)rng.effect((vdot(H.data(), e0.data(), n) + b0) / (xx[j] * bg + L[j]), sd);
    const R b2 = (R)rng.excluded(sd);
    for (int i = 0; i < n; i++) e1[i] = e0[i] - H[i] * (b1 - b0);
    if (pi > 0) {
      for (int i = 0; i < n; i++) e2[i] = e0[i] - H[i] * (b2 - b0);
      R pj;
      if (ratio_form) pj = R(1.0f) / (R(1.0f) + (pi / (1 - pi)) * std::exp(C * (vsq(e2.data(), n) - vsq(e1.data(), n))));
      else {
        const R cj = (1 - pi) * std::exp(C * vsq(e1.data(), n));
        const R dj = (pi)*std::exp(C * vsq(e2.data(), n));
        pj = cj / (cj + dj);
      }
      if (rng.include(pj)) { b[j] = b1; d[j] = 1; e0 = e1; }
      else { b[j] = b2; d[j] = 0; e0 = e2; }
    } else {
      d[j] = 1; b[j] = b1; e0 = e1;
    }
  }
  std::memcpy(e_out, e0.data(), sizeof(R) * n);
}

// GSRR :1597-1628 / GSFLM :1564-1594: the warm-start Gauss-Seidel solvers of mm() (R/mix.R:890-892); natural marker order, the
// state (b, e, Lmb) is the caller's.  flm = false: GSRR (one variance), true: GSFLM (per-marker variances).  Returns sweeps done.
struct GsOut { float mu = 0, h2 = 0, vna = 0; int its = 0; };
static inline GsOut gs_solver(bool flm, const float* y, float* e, const float* X, int n, int p, float* b, float* Lmb, const float* xx,
                              float cxx, int maxit, float* Vb) {
  const float tol = 10e-8f, phi = cxx;
  std::vector<float> e0(e, e + n), bc(p);
  const float vy = fvar(y, n);
  float vna = vdot(y, e, n) / (n - 1);
  float mu = vmean(e, n);
  for (int i = 0; i < n; i++) e[i] -= mu;
  int numit = 0;
  while (numit < maxit) {
    std::copy(b, b + p, bc.begin());
    for (int j = 0; j < p; j++) {
      const float* x = X + (size_t)j * n;
      const float b0 = b[j];
      const float b1 = (vdot(x, e, n) + xx[j] * b0) / (Lmb[j] + xx[j] + 0.01f);
      b[j] = b1;
      axpy_sub(e, x, b1 - b0, n);
    }
    const float eM = vmean(e, n);
    mu += eM;
    for (int i = 0; i < n; i++) e[i] -= eM;
    vna = vdot(e, e0.data(), n) / n;
    if (flm) {
      for (int j = 0; j < p; j++) Vb[j] = b[j] * b[j] + vna / (xx[j] + Lmb[j]);
      for (int j = 0; j < p; j++) Lmb[j] = std::sqrt(phi * vna / Vb[j]);
    } else {
      const float vg = (vy - vna) / phi, LmbTmp = vna / vg;
      for (int j = 0; j < p; j++) { Vb[j] = vg; Lmb[j] = LmbTmp; }
    }
    ++numit;
    float cnv = 0;
    for (int j = 0; j < p; j++) cnv += std::fabs(bc[j] - b[j]);
    if (cnv < tol) break;
  }
  GsOut o;
  o.mu = mu; o.h2 = 1.0f - vna / vy; o.vna = vna; o.its = numit;
  return o;
}

// CNT :1308-1313 (column centring) and IMP :1316-1335 (NaN -> column mean of the observed values), in place
static inline void cnt_columns(float* X, int n, int p) {
  for (int j = 0; j < p; j++) { float* x = X + (size_t)j * n; const float m = vmean(x, n); for (int i = 0; i < n; i++) x[i] -= m; }
}
static inline void imp_columns(float* X, int n, int p) {
  for (int j = 0; j < p; j++) {
    float* x = X + (size_t)j * n;
    bool hasna = false;
    for (int i = 0; i < n; i++) if (std::isnan(x[i])) { hasna = true; break; }
    if (!hasna) continue;
    float sum = 0; int cnt = 0;
    for (int i = 0; i < n; i++) if (!std::isnan(x[i])) { sum += x[i]; cnt++; }
    const float EXP = sum / cnt;
    for (int i = 0; i < n; i++) if (std::isnan(x[i])) x[i] = EXP;
  }
}

// wgr(): R/wgr.R:2-169 with eigK=NULL, no NA; bag != 1 resamples the rows of every iteration (:68: Use = sort(sample(n, n*bag, rp)) - 1,
// without replacement unless rp) and sweeps them with KMUP2.  The driver arithmetic is R's (double);
// every KMUP call crosses the Rcpp boundary, i.e. casts X,b,d,xx,e,L to float and back
// (RcppExports.cpp:16-31).
// eigK (bag == 1 only: with bag != 1 the reference hands KMUP2's nuse-long residual back to KMUP2 as E, :81-87, and reads out of
// bounds): Ud = the first pk eigenvectors (n x pk, column-major), Vd their eigenvalues; pk is chosen by the caller (:25).
struct WgrOut {
  double mu = 0, Ve = 0, Va = 0, cxx = 0, Vk = 0;
  std::vector<double> b, d, Vb, hat, u;
};
// K: the arithmetic of the KMUP sweeps (float, as across the Rcpp boundary; double for a float64 replay of the same draws).
template <class K, class Draws>
static void wgr(const double* y, const double* Xd, int n, int p, int it, int bi, int th, bool iv, bool de,
                double pi, double df, double R2, Draws& rng, bool ratio_form, WgrOut& o, double bag = 1.0,
                const double* Ud = nullptr, const double* Vd = nullptr, int pk = 0, bool rp = false) {
  if (de) iv = true;
  const bool bagged = bag != 1.0;
  if (bagged) df = df / (bag * bag);  // :21
  const int nuse = bagged ? (int)(n * bag) : n;
  std::vector<int> rows(n);
  std::vector<float> usef(nuse);
  std::vector<K> esub(nuse);
  std::vector<K> Xf((size_t)n * p);
  for (size_t i = 0; i < Xf.size(); i++) Xf[i] = (K)(float)Xd[i];
  std::vector<int> post;
  for (int v = bi; v <= it; v += th) post.push_back(v);  // seq(bi,it,th)
  const int mc = (int)post.size();
  std::vector<double> xx(p), b(p, 0.0), d(p, 1.0), e(n), Vb(p), L(p);
  double MSx = 0;
  for (int j = 0; j < p; j++) {
    const double* x = Xd + (size_t)j * n;
    double s = 0, ss = 0;
    for (int i = 0; i < n; i++) { s += x[i]; ss += x[i] * x[i]; }
    xx[j] = ss * bag;  // :49
    const double m = s / n;
    double v = 0;
    for (int i = 0; i < n; i++) v += (x[i] - m) * (x[i] - m);
    MSx += v / (n - 1);
  }
  double mu = 0;
  for (int i = 0; i < n; i++) mu += y[i];
  mu /= n;
  for (int i = 0; i < n; i++) e[i] = y[i] - mu;
  double Va = MSx, Ve = 1;
  for (int j = 0; j < p; j++) { Vb[j] = Va; L[j] = Vb[j] / Ve; }  // sic L=Vb/Ve at start (wgr.R:55)
  double vy = 0;
  { double m = 0; for (int i = 0; i < n; i++) m += y[i]; m /= n; for (int i = 0; i < n; i++) vy += (y[i] - m) * (y[i] - m); vy /= (n - 1); }
  const double Sb = R2 * df * vy / MSx, Se = (1 - R2) * df * vy;
  double B0 = 0, VA = 0, VE = 0;
  std::vector<double> VB(p, 0.0), D(p, 0.0), B(p, 0.0);
  std::vector<K> bf(p), dfl(p), xxf(p), ef(n), Lf(p);
  // polygenic term (:23-33, :60): h = effects of the eigenvectors, xxK = bag, Vk = 1, Sk = R2 var(y) (df + 2)
  const bool poly = Ud != nullptr && pk > 0;
  std::vector<double> h(pk, 0.0), H(pk, 0.0), Vk(pk, 1.0);
  std::vector<K> Uf((size_t)n * pk), hf(pk), dhf(pk), xxKf(pk, (K)(float)bag), Lkf(pk);
  for (size_t i = 0; i < Uf.size(); i++) Uf[i] = (K)(float)Ud[i];
  const double Sk = R2 * vy * (df + 2);
  double Vp = 0, VP = 0;
  size_t next_post = 0;
  for (int i = 1; i <= it; i++) {
    rng.set_sweep(i - 1);
    for (int j = 0; j < p; j++) { bf[j] = (K)(float)b[j]; dfl[j] = (K)(float)d[j]; xxf[j] = (K)(float)xx[j]; Lf[j] = (K)(float)L[j]; }
    for (int r = 0; r < n; r++) ef[r] = (K)(float)e[r];
    if (poly) {  // :77-84: Lk = Ve / (V Vk); KMUP(U, h, dh, xxK, e, Lk, Ve, 0)
      for (int q = 0; q < pk; q++) { Lkf[q] = (K)(float)(Ve / (Vd[q] * Vk[q])); hf[q] = (K)(float)h[q]; dhf[q] = 0; }
      kmup(Uf.data(), n, pk, hf.data(), dhf.data(), xxKf.data(), ef.data(), Lkf.data(), (K)(float)Ve, K(0), rng, ratio_form);
      for (int q = 0; q < pk; q++) h[q] = hf[q];
    }
    if (bagged) {  // :68, :87: a fresh sorted row sample, swept by KMUP2; e becomes the residual of the rows in use
      // sample(n, n*bag, rp): with rp = TRUE rows may repeat; KMUP2 then counts a repeated row once per draw (:51-60)
      rng.rows(n, nuse, rp, rows);
      std::sort(rows.begin(), rows.begin() + nuse);
      for (int r = 0; r < nuse; r++) usef[r] = (float)rows[r];
      kmup2(Xf.data(), n, p, usef.data(), nuse, bf.data(), dfl.data(), xxf.data(), ef.data(), esub.data(), Lf.data(), (K)(float)Ve,
            (K)(float)pi, rng, ratio_form);
    } else {
      kmup(Xf.data(), n, p, bf.data(), dfl.data(), xxf.data(), ef.data(), Lf.data(), (K)(float)Ve, (K)(float)pi, rng, ratio_form);
    }
    if (pi > 0) for (int j = 0; j < p; j++) d[j] = dfl[j];
    for (int j = 0; j < p; j++) b[j] = bf[j];
    for (int r = 0; r < n; r++) e[r] = ef[r];
    if (iv) {
      if (de) for (int j = 0; j < p; j++) Vb[j] = std::sqrt(b[j] * b[j] * Ve / MSx);
      else for (int j = 0; j < p; j++) Vb[j] = (Sb + b[j] * b[j]) / rng.wgr_Vb(j, df + 1);
    } else {
      double bb = 0;
      for (int j = 0; j < p; j++) bb += b[j] * b[j];
      Va = (bb + Sb) / rng.wgr_Va(df + p);
      for (int j = 0; j < p; j++) Vb[j] = Va;
    }
    if (poly) {  // :116-119
      double hh = 0;
      for (int q = 0; q < pk; q++) hh += h[q] * h[q] / Vd[q];
      Vp = (hh + Sk) / rng.wgr_Vp(df + pk);
      for (int q = 0; q < pk; q++) Vk[q] = Vp;
    }
    double ee = 0;
    if (bagged) for (int r = 0; r < nuse; r++) ee += (double)esub[r] * (double)esub[r];
    else for (int r = 0; r < n; r++) ee += e[r] * e[r];
    Ve = (ee + Se) / rng.wgr_Ve(n * bag + df);  // :121
    for (int j = 0; j < p; j++) L[j] = Ve / Vb[j];
    for (int r = 0; r < n; r++) e[r] = y[r] - mu;  // e = y-mu-X%*%b
    for (int j = 0; j < p; j++) {
      const double bj = b[j];
      if (bj == 0.0) continue;
      const double* x = Xd + (size_t)j * n;
      for (int r = 0; r < n; r++) e[r] -= x[r] * bj;
    }
    if (poly)  // :124: ... - U %*% h
      for (int q = 0; q < pk; q++) {
        const double* u = Ud + (size_t)q * n;
        for (int r = 0; r < n; r++) e[r] -= u[r] * h[q];
      }
    double em = 0;
    for (int r = 0; r < n; r++) em += e[r];
    em /= n;
    const double mu0 = rng.wgr_mu0(em, Ve / n);  // sic: sd argument is Ve/n (wgr.R:125)
    mu += mu0;
    for (int r = 0; r < n; r++) e[r] -= mu0;
    if (next_post < post.size() && post[next_post] == i) {
      next_post++;
      B0 += mu; VE += Ve;
      for (int j = 0; j < p; j++) { B[j] += b[j]; D[j] += d[j]; }
      if (iv) for (int j = 0; j < p; j++) VB[j] += Vb[j];
      else VA += Va;
      if (poly) { for (int q = 0; q < pk; q++) H[q] += h[q]; VP += Vp; }
    }
  }
  B0 /= mc;
  double mD = 0;
  for (int j = 0; j < p; j++) { D[j] /= mc; mD += D[j]; }
  mD /= p;
  for (int j = 0; j < p; j++) B[j] = B[j] / mc / mD;
  VE /= mc;
  if (iv) for (int j = 0; j < p; j++) VB[j] /= mc;
  else VA /= mc;
  o.mu = B0; o.b = B; o.d = D; o.Ve = VE; o.Va = VA; o.Vb = VB;
  double cxx = 0;
  for (int j = 0; j < p; j++) cxx += xx[j];
  o.cxx = cxx / p;
  o.hat.assign(n, B0);
  for (int j = 0; j < p; j++) {
    const double* x = Xd + (size_t)j * n;
    for (int r = 0; r < n; r++) o.hat[r] += x[r] * B[j];
  }
  if (poly) {  // :145-150: poly = U0 %*% (H / mc); HAT += poly
    o.Vk = VP / mc;
    o.u.assign(n, 0.0);
    for (int q = 0; q < pk; q++) {
      const double* u = Ud + (size_t)q * n;
      for (int r = 0; r < n; r++) o.u[r] += u[r] * (H[q] / mc);
    }
    for (int r = 0; r < n; r++) o.hat[r] += o.u[r];
  }
}

// ------------------------------------------------------------------------------------------------
// Small dense k x k helpers for MRR3 (column-major, leading dimension k).
// ------------------------------------------------------------------------------------------------
template <class R>
static bool llt_factor(std::vector<R>& A, int k) {  // lower Cholesky in place; false if not PD
  bool ok = true;
  for (int j = 0; j < k; j++) {
    R s = A[j + (size_t)j * k];
    for (int t = 0; t < j; t++) s -= A[j + (size_t)t * k] * A[j + (size_t)t * k];
    if (!(s > 0)) ok = false;
    const R l = std::sqrt(s);
    A[j + (size_t)j * k] = l;
    for (int i = j + 1; i < k; i++) {
      R v = A[i + (size_t)j * k];
      for (int t = 0; t < j; t++) v -= A[i + (size_t)t * k] * A[j + (size_t)t * k];
      A[i + (size_t)j * k] = v / l;
    }
  }
  return ok;
}
template <class R>
static void llt_solve(const std::vector<R>& Lm, int k, std::vector<R>& x) {  // x := (L L')^{-1} x
  for (int i = 0; i < k; i++) {
    R s = x[i];
    for (int t = 0; t < i; t++) s -= Lm[i + (size_t)t * k] * x[t];
    x[i] = s / Lm[i + (size_t)i * k];
  }
  for (int i = k - 1; i >= 0; i--) {
    R s = x[i];
    for (int t = i + 1; t < k; t++) s -= Lm[t + (size_t)i * k] * x[t];
    x[i] = s / Lm[i + (size_t)i * k];
  }
}
// Symmetric eigen-decomposition (cyclic Jacobi), eigenvalues ascending like SelfAdjointEigenSolver.
template <class R>
static void sym_evd(const std::vector<R>& Ain, int k, std::vector<R>& w, std::vector<R>& V) {
  std::vector<double> A(Ain.begin(), Ain.end()), Q((size_t)k * k, 0.0);
  for (int i = 0; i < k; i++) Q[i + (size_t)i * k] = 1.0;
  for (int sweep = 0; sweep < 100; sweep++) {
    double off = 0;
    for (int i = 0; i < k; i++) for (int j = 0; j < i; j++) off += A[i + (size_t)j * k] * A[i + (size_t)j * k];
    if (off < 1e-300) break;
    for (int pI = 0; pI < k - 1; pI++)
      for (int q = pI + 1; q < k; q++) {
        const double apq = A[pI + (size_t)q * k];
        if (std::fabs(apq) < 1e-300) continue;
        const double app = A[pI + (size_t)pI * k], aqq = A[q + (size_t)q * k];
        const double tau = (aqq - app) / (2 * apq);
        const double t = (tau >= 0 ? 1.0 : -1.0) / (std::fabs(tau) + std::sqrt(1 + tau * tau));
        const double c = 1 / std::sqrt(1 + t * t), s = t * c;
        for (int r = 0; r < k; r++) {
          const double arp = A[r + (size_t)pI * k], arq = A[r + (size_t)q * k];
          A[r + (size_t)pI * k] = c * arp - s * arq;
          A[r + (size_t)q * k] = s * arp + c * arq;
        }
        for (int r = 0; r < k; r++) {
          const double apr = A[pI + (size_t)r * k], aqr = A[q + (size_t)r * k];
          A[pI + (size_t)r * k] = c * apr - s * aqr;
          A[q + (size_t)r * k] = s * apr + c * aqr;
        }
        for (int r = 0; r < k; r++) {
          const double qrp = Q[r + (size_t)pI * k], qrq = Q[r + (size_t)q * k];
          Q[r + (size_t)pI * k] = c * qrp - s * qrq;
          Q[r + (size_t)q * k] = s * qrp + c * qrq;
        }
      }
  }
  std::vector<int> idx(k);
  for (int i = 0; i < k; i++) idx[i] = i;
  std::sort(idx.begin(), idx.end(), [&](int a, int b2) { return A[a + (size_t)a * k] < A[b2 + (size_t)b2 * k]; });
  w.resize(k); V.resize((size_t)k * k);
  for (int c = 0; c < k; c++) {
    w[c] = (R)A[idx[c] + (size_t)idx[c] * k];
    for (int r = 0; r < k; r++) V[r + (size_t)c * k] = (R)Q[r + (size_t)idx[c] * k];
  }
}
// Pseudo-inverse of a symmetric matrix (stands in for completeOrthogonalDecomposition().pseudoInverse()).
template <class R>
static void sym_pinv(const std::vector<R>& A, int k, std::vector<R>& out) {
  std::vector<R> w, V;
  sym_evd(A, k, w, V);
  R mx = 0;
  for (int i = 0; i < k; i++) mx = std::max(mx, (R)std::fabs(w[i]));
  const R thr = mx * (R)k * std::numeric_limits<R>::epsilon();
  out.assign((size_t)k * k, R(0));
  for (int c = 0; c < k; c++) {
    if (std::fabs(w[c]) <= thr) continue;
    const R iw = R(1) / w[c];
    for (int j = 0; j < k; j++) {
      const R vj = V[j + (size_t)c * k] * iw;
      for (int i = 0; i < k; i++) out[i + (size_t)j * k] += V[i + (size_t)c * k] * vj;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// MRR3 (R=double, f32_variant=false; RcppEigen20230423.cpp:318-701) and
// MRR3F (R=float,  f32_variant=true;  :704-1079).  Differences (SURVEY 7.3): MRR3 recomputes the
// system with marker weights and so ignores NoInv in the solve (:503-507); MRR3F honours NoInv but
// never applies W in the solve.
// ------------------------------------------------------------------------------------------------
template <class R>
struct MrrPar {
  int maxit = 500; R tol = R(10e-9); bool TH = false; R NLfactor = 0; bool InnerGS = false, NoInv = false,
      HCS = false, XFA = false, ACS = false; int NumXFA = 3; R R2 = R(0.5), gc0 = R(0.5), df0 = R(1.0);
  bool updateMu = false; R weight_prior_h2 = R(0.01), weight_prior_gc = R(0.01), PenCor = 0, MinCor = 1,
      uncorH2below = 0, roundGCupFrom = 1, roundGCupTo = 1, roundGCdownFrom = 1, roundGCdownTo = 0,
      bucketGCfrom = 1, bucketGCto = 1, DeflateMax = R(0.9), DeflateBy = 0; bool OneVarB = false, OneVarE = false;
};
template <class R>
struct MrrOut {
  int k = 0, its = 0;
  std::vector<R> mu, b, hat, h2, GC, vb, ve, MSx, cnvB, cnvH2, cnvV, W;
};

template <class R>
static void mrr3(const R* Yin, const R* Xin, int n0, int k, int p, const MrrPar<R>& P, bool f32_variant, MrrOut<R>& o) {
  auto M = [](int r, int c, int ld) { return (size_t)r + (size_t)c * ld; };
  std::vector<R> Y(Yin, Yin + (size_t)n0 * k), X(Xin, Xin + (size_t)n0 * p), Z((size_t)n0 * k);
  for (int i = 0; i < n0; i++) for (int j = 0; j < k; j++) {
    if (std::isnan(Y[M(i, j, n0)])) { Z[M(i, j, n0)] = 0; Y[M(i, j, n0)] = 0; } else Z[M(i, j, n0)] = 1;
  }
  std::vector<R> n(k), iN(k), mu(k), y((size_t)n0 * k);
  for (int t = 0; t < k; t++) { n[t] = vsum(&Z[M(0, t, n0)], n0); iN[t] = R(1) / n[t]; }
  for (int t = 0; t < k; t++) mu[t] = vsum(&Y[M(0, t, n0)], n0) * iN[t];
  for (int t = 0; t < k; t++) for (int i = 0; i < n0; i++) y[M(i, t, n0)] = (Y[M(i, t, n0)] - mu[t]) * Z[M(i, t, n0)];
  for (int j = 0; j < p; j++) {  // centre X (:378-379)
    const R m = vmean(&X[M(0, j, n0)], n0);
    for (int i = 0; i < n0; i++) X[M(i, j, n0)] -= m;
  }
  std::vector<R> XX((size_t)p * k), XSX((size_t)p * k), MSx(k), TrXSX(k);
  for (int j = 0; j < p; j++) for (int t = 0; t < k; t++) {
    const R* x = &X[M(0, j, n0)]; const R* z = &Z[M(0, t, n0)];
    XX[M(j, t, p)] = reduce_sum<R>(n0, [&](int i) { return x[i] * x[i] * z[i]; });
    const R sx = reduce_sum<R>(n0, [&](int i) { return x[i] * z[i]; });
    const R q = sx * iN[t];
    XSX[M(j, t, p)] = XX[M(j, t, p)] * iN[t] - q * q;
  }
  for (int t = 0; t < k; t++) { MSx[t] = vsum(&XSX[M(0, t, p)], p); TrXSX[t] = n[t] * MSx[t]; }
  for (int t = 0; t < k; t++) iN[t] = R(1) / (n[t] - 1);
  std::vector<R> vy(k), ve(k), iVe(k), vbInit(k), veInit(k), h2(k);
  for (int t = 0; t < k; t++) { vy[t] = vsq(&y[M(0, t, n0)], n0) * iN[t]; ve[t] = vy[t] * (1 - P.R2); iVe[t] = R(1) / ve[t]; }
  std::vector<R> vb((size_t)k * k, R(0)), TildeHat((size_t)k * k), iG((size_t)k * k, R(0));
  for (int t = 0; t < k; t++) { vbInit[t] = (vy[t] * P.R2) / MSx[t]; veInit[t] = ve[t]; vb[M(t, t, k)] = vbInit[t];
    iG[M(t, t, k)] = R(1) / vbInit[t]; h2[t] = 1 - ve[t] / vy[t]; }
  for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) if (i > j) {
    const R tmp = P.gc0 * std::sqrt(vb[M(i, i, k)] * vb[M(j, j, k)]);
    vb[M(i, j, k)] = tmp; vb[M(j, i, k)] = tmp;
  }
  std::vector<R> tilde((size_t)p * k);  // X' y
  for (int j = 0; j < p; j++) for (int t = 0; t < k; t++) tilde[M(j, t, p)] = vdot(&X[M(0, j, n0)], &y[M(0, t, n0)], n0);
  std::vector<R> TrDinvXSX(k), Dinv((size_t)p * k);
  if (P.TH) for (int t = 0; t < k; t++) for (int j = 0; j < p; j++) XSX[M(j, t, p)] *= n[t];
  std::vector<R> Sb(vb), Se(ve), iNp(k);
  for (auto& v : Sb) v *= P.df0;
  for (int t = 0; t < k; t++) { Se[t] = ve[t] * P.df0; iNp[t] = R(1) / (n[t] + P.df0 - 1); }
  std::vector<R> LHS((size_t)k * k), RHS(k), b((size_t)p * k, R(0)), b0(k), b1(k), e(y);
  std::vector<R> A(vb), GC((size_t)k * k, R(0)), beta0, vb0, ve0, h20, CNV1, CNV2, CNV3;
  const R bucketMean = R(0.5) * (P.bucketGCfrom + P.bucketGCto);
  R inflate = 0, Deflate = 1, cnv = 10, gs, tmp;
  int numit = 0;
  const R logtol = std::log10(P.tol);
  std::vector<int> RGS(p), IRGS(k);
  for (int j = 0; j < p; j++) RGS[j] = j;
  for (int j = 0; j < k; j++) IRGS[j] = j;
  const bool NonLinear = P.NLfactor != 0;
  std::vector<R> W((size_t)p * k, R(1)), iVeWj(iVe), tmpW(p), ew, ev, UDU((size_t)k * k), xe(k);
  (void)cnv;
  while (numit < P.maxit) {
    beta0 = b; vb0 = vb; ve0 = ve; h20 = h2;
    std::shuffle(RGS.begin(), RGS.end(), std::mt19937(numit));
    std::shuffle(IRGS.begin(), IRGS.end(), std::mt19937(numit));
    for (int j = 0; j < p; j++) {
      const int J = RGS[j];
      const R* x = &X[M(0, J, n0)];
      for (int t = 0; t < k; t++) b0[t] = b[M(J, t, p)];
      for (int t = 0; t < k; t++) xe[t] = vdot(x, &e[M(0, t, n0)], n0);  // X.col(J)' * e
      const bool noinv_system = f32_variant && P.NoInv;
      if (!f32_variant) for (int t = 0; t < k; t++) iVeWj[t] = iVe[t] * W[M(J, t, p)];  // :504
      if (noinv_system) {  // :878-882 (MRR3F only; MRR3 overwrites it, :503-507)
        for (int c = 0; c < k; c++) for (int r = 0; r < k; r++)
          LHS[M(r, c, k)] = vb[M(r, c, k)] * (XX[M(J, c, p)] * iVeWj[c]);
        for (int t = 0; t < k; t++) LHS[M(t, t, k)] += 1;
        std::vector<R> r0(k);
        for (int t = 0; t < k; t++) r0[t] = (xe[t] + XX[M(J, t, p)] * b0[t]) * iVeWj[t];
        for (int r = 0; r < k; r++) { R s = 0; for (int c = 0; c < k; c++) s += vb[M(r, c, k)] * r0[c]; RHS[r] = s; }
      } else {
        LHS = iG;
        for (int t = 0; t < k; t++) LHS[M(t, t, k)] += XX[M(J, t, p)] * iVeWj[t];
        for (int t = 0; t < k; t++) RHS[t] = (xe[t] + XX[M(J, t, p)] * b0[t]) * iVeWj[t];
      }
      if (P.InnerGS) {
        for (int t = 0; t < k; t++) b1[t] = b[M(J, t, p)];
        for (int i = 0; i < k; i++) {
          const int ri = IRGS[i];
          R s = 0;
          for (int t = 0; t < k; t++) s += LHS[M(t, ri, k)] * b1[t];
          b1[ri] = (RHS[ri] - s + LHS[M(ri, ri, k)] * b1[ri]) / LHS[M(ri, ri, k)];
        }
      } else {
        std::vector<R> Lc(LHS);
        llt_factor(Lc, k);
        b1 = RHS;
        llt_solve(Lc, k, b1);
      }
      for (int t = 0; t < k; t++) {
        b[M(J, t, p)] = b1[t];
        const R dlt = b1[t] - b0[t];
        R* et = &e[M(0, t, n0)]; const R* zt = &Z[M(0, t, n0)];
        for (int i = 0; i < n0; i++) et[i] = et[i] - (x[i] * dlt) * zt[i];
      }
    }
    if (NonLinear) {
      for (int t = 0; t < k; t++) {
        R maxW = -std::numeric_limits<R>::infinity(), minW = std::numeric_limits<R>::infinity();
        for (int j = 0; j < p; j++) { const R a = std::fabs(b[M(j, t, p)]); maxW = std::max(maxW, a); minW = std::min(minW, a); }
        for (int j = 0; j < p; j++) tmpW[j] = P.NLfactor * (std::fabs(b[M(j, t, p)]) - minW) / (maxW - minW) + (R(1.0) - P.NLfactor);
        const R m = vmean(tmpW.data(), p);
        for (int j = 0; j < p; j++) W[M(j, t, p)] = tmpW[j] + (R(1.0) - m);
      }
    }
    for (int t = 0; t < k; t++) {
      ve[t] = vdot(&e[M(0, t, n0)], &y[M(0, t, n0)], n0);
      ve[t] = (ve[t] + Se[t]) * iNp[t];
      h2[t] = 1 - ve[t] / vy[t];
    }
    if (P.weight_prior_h2 > 0) for (int t = 0; t < k; t++) ve[t] = ve[t] * (1 - P.weight_prior_h2) + P.weight_prior_h2 * veInit[t];
    if (P.OneVarE) { tmp = vmean(ve.data(), k); for (int t = 0; t < k; t++) ve[t] = tmp; }
    for (int t = 0; t < k; t++) { iVe[t] = R(1) / ve[t]; iVeWj[t] = iVe[t]; }
    if (P.TH) {
      for (int t = 0; t < k; t++) {
        R s = 0;
        for (int j = 0; j < p; j++) { Dinv[M(j, t, p)] = R(1) / (XSX[M(j, t, p)] / ve[t] + iG[M(t, t, k)]); s += XSX[M(j, t, p)] * Dinv[M(j, t, p)]; }
        TrDinvXSX[t] = s;
      }
      for (int i = 0; i < k; i++) for (int j = 0; j < k; j++)
        TildeHat[M(i, j, k)] = reduce_sum<R>(p, [&](int m) { return b[M(m, i, p)] * (Dinv[M(m, j, p)] * tilde[M(m, j, p)]); });
    } else {
      for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) TildeHat[M(i, j, k)] = vdot(&b[M(0, i, p)], &tilde[M(0, j, p)], p);
    }
    const std::vector<R>& Tr = P.TH ? TrDinvXSX : TrXSX;
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) {
      if (i == j) vb[M(i, i, k)] = (TildeHat[M(i, i, k)] + Sb[M(i, i, k)]) / (Tr[i] + P.df0);
      else vb[M(i, j, k)] = (TildeHat[M(i, j, k)] + TildeHat[M(j, i, k)] + Sb[M(i, j, k)]) / (Tr[i] + Tr[j] + P.df0);
    }
    if (P.weight_prior_h2 > 0) for (int i = 0; i < k; i++) vb[M(i, i, k)] = vb[M(i, i, k)] * (1 - P.weight_prior_h2) + P.weight_prior_h2 * vbInit[i];
    if (P.weight_prior_gc > 0) {
      for (int i = 0; i < k; i++) for (int j = 0; j < k; j++)
        GC[M(i, j, k)] = (i != j) ? (R(1.0) - P.weight_prior_gc) * vb[M(i, j, k)] / std::sqrt(vb[M(i, i, k)] * vb[M(j, j, k)]) + P.gc0 * P.weight_prior_gc : R(1);
      for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) if (i != j) vb[M(i, j, k)] = GC[M(i, j, k)] * std::sqrt(vb[M(i, i, k)] * vb[M(j, j, k)]);
    } else {
      for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) GC[M(i, j, k)] = vb[M(i, j, k)] / std::sqrt(vb[M(i, i, k)] * vb[M(j, j, k)]);
    }
    auto top_factors = [&](R add, R scale) {
      sym_evd(GC, k, ew, ev);
      std::fill(UDU.begin(), UDU.end(), R(0));
      for (int f = 0; f < P.NumXFA; f++) {
        const int c = k - f - 1;
        for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) UDU[M(i, j, k)] += ew[c] * ev[M(i, c, k)] * ev[M(j, c, k)];
      }
      for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) GC[M(i, j, k)] = (UDU[M(i, j, k)] + add) * scale;
      for (int i = 0; i < k; i++) GC[M(i, i, k)] = 1;
    };
    if (P.ACS) {
      gs = (vsum(GC.data(), k * k) - k) / ((k * (k - 1))) / R(2.0);
      top_factors(gs, R(0.5));
    } else if (P.HCS) {
      gs = 0;
      for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) if (i > j) gs += GC[M(i, j, k)];
      gs = gs / ((k * (k - 1)) / 2);
      for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) GC[M(i, j, k)] = (i != j) ? gs : R(1);
    } else if (P.XFA) {
      top_factors(R(0), R(1));
    }
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) if (i != j) {
      R& g = GC[M(i, j, k)];
      if (P.MinCor < 1 && g < P.MinCor) g = 0;
      if (P.PenCor > 0) g = std::tanh(P.PenCor * std::fabs(g)) * g;
      if (P.roundGCdownFrom < 1 && g < P.roundGCdownFrom) g = P.roundGCdownTo;
      if (P.roundGCupFrom < 1 && g > P.roundGCupFrom) g = P.roundGCupTo;
      if (P.bucketGCfrom < 1 && g > P.bucketGCfrom && g < P.bucketGCto) g = bucketMean;
      if (P.uncorH2below > 0 && (h2[i] < P.uncorH2below || h2[j] < P.uncorH2below)) g = 0;
    }
    if (!P.NoInv || P.TH) {
      A = GC;
      if (P.DeflateBy > 0) {
        for (auto& v : A) v *= Deflate;
        for (int i = 0; i < k; i++) A[M(i, i, k)] = 1;
        std::vector<R> Lc(A);
        if (!llt_factor(Lc, k) && Deflate > P.DeflateMax) {
          Deflate -= P.DeflateBy;
          A = GC;
          for (auto& v : A) v *= Deflate;
          for (int i = 0; i < k; i++) A[M(i, i, k)] = 1;
        }
      }
      sym_evd(A, k, ew, ev);
      const R MinDVb = ew[0];
      if (MinDVb < 0) {
        inflate = std::fabs(MinDVb * R(1.1));
        for (int i = 0; i < k; i++) A[M(i, i, k)] += inflate;
        for (auto& v : A) v /= (R(1.0) + inflate);
        GC = A;
      }
    }
    if (P.OneVarB) {
      tmp = 0;
      for (int i = 0; i < k; i++) tmp += TildeHat[M(i, i, k)];
      tmp /= k;
      for (size_t i = 0; i < vb.size(); i++) vb[i] = GC[i] * tmp;
    } else {
      for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) vb[M(i, j, k)] = GC[M(i, j, k)] * std::sqrt(vb[M(i, i, k)] * vb[M(j, j, k)]);
    }
    if (!P.NoInv || P.TH) sym_pinv(vb, k, iG);
    if (P.updateMu) {
      for (int t = 0; t < k; t++) {
        const R m = vsum(&e[M(0, t, n0)], n0) * iN[t];
        mu[t] += m;
        for (int i = 0; i < n0; i++) e[M(i, t, n0)] = (e[M(i, t, n0)] - m) * Z[M(i, t, n0)];
      }
    }
    R mx = -std::numeric_limits<R>::infinity();
    for (int t = 0; t < k; t++) {
      const R s = reduce_sum<R>(p, [&](int j) { const R dd = beta0[M(j, t, p)] - b[M(j, t, p)]; return dd * dd; });
      mx = std::max(mx, s);
    }
    cnv = std::log10(mx);
    CNV1.push_back(cnv);
    if (std::isnan(cnv)) break;
    CNV2.push_back(std::log10(reduce_sum<R>(k, [&](int t) { const R dd = h20[t] - h2[t]; return dd * dd; })));
    CNV3.push_back(std::log10(reduce_sum<R>(k * k, [&](int t) { const R dd = vb0[t] - vb[t]; return dd * dd; })));
    ++numit;
    if (cnv < logtol) break;
  }
  o.k = k; o.its = numit; o.mu = mu; o.b = b; o.h2 = h2; o.GC = GC; o.vb = vb; o.ve = ve; o.MSx = MSx; o.W = W;
  CNV1.resize(numit); CNV2.resize(numit); CNV3.resize(numit);
  o.cnvB = CNV1; o.cnvH2 = CNV2; o.cnvV = CNV3;
  o.hat.assign((size_t)n0 * k, R(0));
  for (int t = 0; t < k; t++) {
    R* h = &o.hat[M(0, t, n0)];
    for (int j = 0; j < p; j++) { const R bj = b[M(j, t, p)]; const R* x = &X[M(0, j, n0)]; for (int i = 0; i < n0; i++) h[i] += x[i] * bj; }
    for (int i = 0; i < n0; i++) h[i] += mu[t];
  }
}

}  // namespace orc
