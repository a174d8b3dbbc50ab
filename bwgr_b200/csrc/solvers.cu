// solvers.cu -- the solver entry points of the C ABI on top of the fit engine (fit.cu): the EM solvers, GSRR / GSFLM, the Gibbs
// samplers, KMUP / KMUP2, wgr, and the fitted values of the store.
#include "host.h"

using namespace bwgr;
using namespace bwgr::host;

extern "C" {

static int em_spec(const bwgr_em_params* par, FitSpec* s) {
  if (!par) return fail(BWGR_ERR_ARG, "params NULL");
  if (par->model < 0 || par->model > BWGR_EM_LASSO) return fail(BWGR_ERR_ARG, "bad EM model %d", par->model);
  s->model = par->model; s->nsys = par->nsys; s->row_mask = par->row_mask;
  s->shuffled = !(par->model == BWGR_EM_BCPI || par->model == BWGR_EM_LASSO);  // these two walk the markers in order (:1523, :1477)
  s->df = (float)par->df; s->R2 = (float)par->R2; s->Pi = (float)par->Pi; s->alpha = (float)par->alpha; s->pi = 0;
  s->it = par->it < 0 ? (model_has_cnv(par->model) ? 300 : 200) : par->it;  // maxit of the solvers with a stopping rule, else 200 sweeps
  s->bi = 0; s->seed = 0;
  return 0;
}

int bwgr_em_begin(bwgr_handle* h, const bwgr_em_params* par, const double* y) {
  FitSpec s;
  int rc = em_spec(par, &s);
  if (rc) return rc;
  if (par->weights) {  // emML(y, gen, D): the weighted penalty Lmb / d_j (:495-496) travels in the per-marker slot
    if (par->model != BWGR_EM_ML) return fail(BWGR_ERR_ARG, "marker weights belong to emML");
    if (par->nsys != 1 || par->row_mask) return fail(BWGR_ERR_UNSUPPORTED, "emML with marker weights: one unmasked system");
    s.model = M_EMMLD;
  }
  rc = fit_begin(h, s, y);
  if (rc || !par->weights) return rc;
  Fit& f = *h->fit;
  const int64_t p = h->p;
  std::vector<float> w(p), l0(p);
  for (int64_t j = 0; j < p; j++) {
    w[j] = (float)par->weights[j];
    if (!(w[j] > 0.0f)) { h->fit.reset(); return fail(BWGR_ERR_ARG, "marker weights must be positive"); }
    l0[j] = f.sc0[0].lmb / w[j];
  }
  if (f.wts.alloc(p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  CU(cudaMemcpyAsync(f.wts.p, w.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.vbv.p, l0.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int bwgr_em_sweeps(bwgr_handle* h, int nsweeps) {
  if (!h) return fail(BWGR_ERR_ARG, "null handle");
  return fit_sweeps(h, nsweeps);
}

int bwgr_em_end(bwgr_handle* h, bwgr_em_out* out) {
  if (!h || !h->fit) return fail(BWGR_ERR_STATE, "no fit in progress");
  if (!out) return fail(BWGR_ERR_ARG, "out NULL");
  FitGuard guard{h};
  Fit& f = *h->fit;
  const int64_t n = h->n, p = h->p, ld = h->ld;
  const int ns = f.nsys;
  int rc = check_err_flag(h, "sweep");
  if (rc) return rc;
  dump_trace(h);
  std::vector<SysScalars> sc(ns);
  CU(cudaMemcpyAsync(sc.data(), f.sc.p, sizeof(SysScalars) * ns, cudaMemcpyDeviceToHost, h->stream));
  std::vector<float> hb((size_t)ns * p), hd, hv, hh, he;
  std::vector<uint8_t> hmask;  // row masks of masked systems (emBL's var(e))
  CU(cudaMemcpyAsync(hb.data(), f.b.p, sizeof(float) * hb.size(), cudaMemcpyDeviceToHost, h->stream));
  if (f.d.p && out->d) { hd.resize((size_t)ns * p); CU(cudaMemcpyAsync(hd.data(), f.d.p, sizeof(float) * hd.size(), cudaMemcpyDeviceToHost, h->stream)); }
  if (f.vbv.p && (out->vb || f.model == M_EMDE)) { hv.resize((size_t)ns * p); CU(cudaMemcpyAsync(hv.data(), f.vbv.p, sizeof(float) * hv.size(), cudaMemcpyDeviceToHost, h->stream)); }
  if (f.model == M_EMBL) { he.resize((size_t)ns * ld); CU(cudaMemcpyAsync(he.data(), f.e.p, sizeof(float) * he.size(), cudaMemcpyDeviceToHost, h->stream)); }
  CU(cudaStreamSynchronize(h->stream));
  std::vector<float> mu(ns);
  for (int t = 0; t < ns; t++) mu[t] = sc[t].mu;
  if ((rc = fitted_values(h, ns, f.b.p, false, mu.data(), hh))) return rc;
  for (int t = 0; t < ns; t++) {
    const SysScalars& c = sc[t];
    if (out->mu) out->mu[t] = c.mu;
    if (out->its) out->its[t] = c.its;
    double Va = 0, Ve = c.ve, h2 = 0, Vg = 0, pi_out = 0, lmb_out = 0;
    switch (f.model) {
      case M_EMRR: Va = c.vb; h2 = 1.0f - c.ve / f.vy[t]; break;
      case M_EMBA: case M_EMBB: h2 = 1.0f - c.ve / f.vy[t]; break;
      case M_EMBC: Va = c.vb; Vg = c.vb * f.MSx[t]; h2 = 1.0f - c.ve / f.vy[t]; break;
      case M_EMBL: {
        // var(e) over the rows the system uses (:391): a masked system's held-out rows never enter e (they stay 0)
        std::vector<float> ev;
        if (f.masked && hmask.empty()) {
          hmask.resize((size_t)ns * ld);
          CU(cudaMemcpy(hmask.data(), f.mask.p, hmask.size(), cudaMemcpyDeviceToHost));
        }
        for (int64_t i = 0; i < n; i++)
          if (!f.masked || hmask[(size_t)t * ld + i]) ev.push_back(he[(size_t)t * ld + i]);
        if (h->world > 1) {  // var(e) over all individuals (:391)
          double sums[2] = {0, 0};
          for (float v : ev) sums[0] += v;
          rc = dist_allreduce_host(h, sums, 1, false);
          if (rc) return rc;
          const float me = (float)(sums[0] / (double)h->n_global);
          for (float v : ev) { const float tt = v - me; sums[1] += (double)tt * tt; }
          rc = dist_allreduce_host(h, sums + 1, 1, false);
          if (rc) return rc;
          h2 = 1.0f - ((float)sums[1] / (float)(h->n_global - 1)) / f.vy[t];
        } else {
          h2 = 1.0f - fvar_f(ev) / f.vy[t];
        }
        Ve = 0; break;
      }
      case M_EMEN: { const float va = c.vb * f.cxx[t]; Va = va; h2 = va / (va + c.ve); break; }
      case M_EMDE: {  // Vb_j of the last sweep from the penalty it produced: Lmb_j = sqrt(cxx Ve / Vb_j) (:293-296, :305)
        float sv = 0;
        if (!hv.empty() || out->vb) {
          for (int64_t j = 0; j < p; j++) {
            const float L = hv.empty() ? 0.0f : hv[(size_t)t * p + j];
            const float vbj = (c.its > 0 && L > 0) ? c.cxx * c.ve / (L * L) : 0.0f;
            if (!hv.empty()) hv[(size_t)t * p + j] = vbj;
            sv += vbj;
          }
        }
        h2 = sv / (sv + c.ve);
        break;
      }
      case M_EMMLD:
      case M_EMML: Vg = c.vb; Va = c.vb * c.MSx; h2 = Va / (Va + c.ve); break;                  // :508-515 (Vg slot = Vb)
      case M_EMBCPI: Va = c.vb; Vg = c.vb * c.MSx; h2 = 1.0f - c.ve / f.vy[t]; pi_out = c.Pi; break;  // :1539-1545
      case M_LASSO: h2 = 1.0f - c.ve / f.vy[t]; Ve = 0; lmb_out = c.lmb; break;                       // :1494-1497
      default: break;
    }
    if (out->scal) {
      double* sc_out = out->scal + (size_t)BWGR_NSCAL * t;
      sc_out[0] = Va; sc_out[1] = Ve; sc_out[2] = h2; sc_out[3] = Vg; sc_out[4] = pi_out; sc_out[5] = lmb_out;
    }
  }
  if (out->b) for (size_t i = 0; i < hb.size(); i++) out->b[i] = hb[i];
  if (out->d && !hd.empty()) for (size_t i = 0; i < hd.size(); i++) out->d[i] = hd[i];
  if (out->vb && !hv.empty()) for (size_t i = 0; i < hv.size(); i++) out->vb[i] = hv[i];
  if (out->hat) for (size_t i = 0; i < hh.size(); i++) out->hat[i] = hh[i];
  return 0;
}

int bwgr_em_fit(bwgr_handle* h, const bwgr_em_params* par, const double* y, bwgr_em_out* out) {
  FitGuard guard{h};
  int rc = bwgr_em_begin(h, par, y);
  if (rc) return rc;
  Fit& f = *h->fit;
  std::vector<SysScalars> sc;
  rc = model_has_cnv(f.model) ? fit_sweeps_until_done(h, sc) : fit_sweeps(h, f.it_target);
  if (rc) return rc;
  return bwgr_em_end(h, out);
}

// ---- GSRR / GSFLM: warm-start Gauss-Seidel (Rcpp20260726ai.cpp:1564-1628) ---------------------------------------------
int bwgr_gs_fit(bwgr_handle* h, int which, const double* y, double* e, double* b, double* Lmb, const double* xx, double cxx, int maxit,
                double* vb, double* scal) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!y || !e || !b || !Lmb || !xx) return fail(BWGR_ERR_ARG, "null argument");
  if (which < 0 || which > 1 || maxit < 1) return fail(BWGR_ERR_ARG, "bad which / maxit");
  const int64_t n = h->n, p = h->p, ld = h->ld;
  FitSpec s;
  s.model = which == 0 ? M_GSRR : M_GSFLM; s.nsys = 1; s.shuffled = false; s.row_mask = nullptr;  // natural marker order (:1581)
  s.df = 10; s.R2 = 0.5f; s.Pi = 0; s.alpha = 0; s.pi = 0; s.it = maxit; s.bi = 0; s.seed = 0;
  // fit_begin on the residual as passed in: mu = mean(e), e <- e - mu (:1574), and the y slot keeps e0 for vna = e.e0/n (:1587)
  FitGuard guard{h};
  int rc = fit_begin(h, s, e);
  if (rc) return rc;
  Fit& f = *h->fit;
  std::vector<float> yv(n), hb(p), hl(p), hx(p);
  for (int64_t i = 0; i < n; i++) { if (!(y[i] == y[i])) return fail(BWGR_ERR_ARG, "y contains NaN"); yv[i] = (float)y[i]; }
  for (int64_t j = 0; j < p; j++) { hb[j] = (float)b[j]; hl[j] = (float)Lmb[j] + 0.01f; hx[j] = (float)xx[j]; }
  SysScalars c = f.sc0[0];
  c.vy = fvar_f(yv);      // float vy = fvar(y) (:1571)
  c.cxx = (float)cxx;     // phi
  f.sc0[0] = c; f.vy[0] = c.vy;
  if (f.xx_over.alloc(p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  CU(cudaMemcpyAsync(f.b.p, hb.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.vbv.p, hl.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.xx_over.p, hx.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.sc.p, &c, sizeof(SysScalars), cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  std::vector<SysScalars> scv;
  if ((rc = fit_sweeps_until_done(h, scv))) return rc;
  const SysScalars& sc = scv[0];
  rc = check_err_flag(h, "sweep");
  if (rc) return rc;
  std::vector<float> he(ld);
  CU(cudaMemcpyAsync(he.data(), f.e.p, sizeof(float) * ld, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(hb.data(), f.b.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(hl.data(), f.vbv.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  for (int64_t i = 0; i < n; i++) e[i] = he[i];
  for (int64_t j = 0; j < p; j++) {
    b[j] = hb[j];
    const float L = hl[j] - 0.01f;
    Lmb[j] = L;
    if (vb) vb[j] = which == 0 ? sc.vb : sc.cxx * sc.ve / (L * L);  // GSFLM: Lmb_j = sqrt(phi vna / Vb_j) (:1589)
  }
  if (scal) { scal[0] = sc.mu; scal[1] = 1.0f - sc.ve / c.vy; scal[2] = sc.ve; scal[3] = sc.its; }
  return 0;
}

// ---- Gibbs -------------------------------------------------------------------------------------------
// nsys phenotype columns x nchains chains = S systems; system s = t * nchains + c fits column t (on the rows of its mask) and draws
// from Philox chain chain0 + s.  bwgr_gibbs_fit is the case nsys = 1, no mask, chain0 = 0.
int bwgr_gibbs_fit_sys(bwgr_handle* h, const bwgr_gibbs_sys_params* sp, const double* Y, bwgr_gibbs_out* out) {
  if (!h || !sp || !out || !Y) return fail(BWGR_ERR_ARG, "null argument");
  if (!h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  const bwgr_gibbs_params* par = &sp->base;
  if (par->model < 0 || par->model > BWGR_GIBBS_DPI) return fail(BWGR_ERR_ARG, "bad Gibbs model %d", par->model);
  static const int kGibbsModel[] = {M_BRR, M_BA, M_BB, M_BC, M_BL, M_BCPI, M_BDPI};
  const bool has_pi = par->model == BWGR_GIBBS_CPI || par->model == BWGR_GIBBS_DPI;  // these two start at pi = 0.5 (:870, :934), not an argument
  if (par->it < 1 || par->bi < 0 || par->bi >= par->it) return fail(BWGR_ERR_ARG, "need 0 <= bi < it");
  if (sp->nsys < 1) return fail(BWGR_ERR_ARG, "bad nsys %d", sp->nsys);
  if (sp->chain0 < 0) return fail(BWGR_ERR_ARG, "bad chain0 %d", sp->chain0);
  const int nc = par->nchains < 1 ? 1 : par->nchains;
  if ((int64_t)sp->nsys * nc > 4096) return fail(BWGR_ERR_ARG, "nsys x nchains = %lld systems (at most 4096)", (long long)sp->nsys * nc);
  const int ns = sp->nsys * nc;
  const int64_t n = h->n, p = h->p;
  std::vector<double> yy((size_t)ns * n);
  std::vector<uint8_t> mm(sp->row_mask ? (size_t)ns * n : 0);
  for (int s = 0; s < ns; s++) {
    const size_t t = (size_t)(s / nc);
    memcpy(yy.data() + (size_t)s * n, Y + t * n, sizeof(double) * n);
    if (sp->row_mask) memcpy(mm.data() + (size_t)s * n, sp->row_mask + t * n, (size_t)n);
  }
  FitSpec s;
  s.model = kGibbsModel[par->model]; s.nsys = ns; s.shuffled = false; s.row_mask = sp->row_mask ? mm.data() : nullptr;
  s.df = (float)par->df; s.R2 = (float)par->R2; s.Pi = 0; s.alpha = 0; s.pi = has_pi ? 0.5f : (float)par->pi;
  s.it = par->it; s.bi = par->bi; s.seed = par->seed; s.chain0 = sp->chain0;
  FitGuard guard{h};
  int rc = fit_begin(h, s, yy.data());
  if (rc) return rc;
  Fit& f = *h->fit;
  rc = fit_sweeps(h, par->it);
  if (rc) return rc;
  rc = check_err_flag(h, "gibbs sweep");
  if (rc) return rc;
  dump_trace(h);
  std::vector<SysScalars> sc(ns);
  CU(cudaMemcpyAsync(sc.data(), f.sc.p, sizeof(SysScalars) * ns, cudaMemcpyDeviceToHost, h->stream));
  std::vector<float> B((size_t)ns * p), D, V;
  CU(cudaMemcpyAsync(B.data(), f.B.p, sizeof(float) * B.size(), cudaMemcpyDeviceToHost, h->stream));
  if (f.D.p) { D.resize((size_t)ns * p); CU(cudaMemcpyAsync(D.data(), f.D.p, sizeof(float) * D.size(), cudaMemcpyDeviceToHost, h->stream)); }
  if (f.VBv.p) { V.resize((size_t)ns * p); CU(cudaMemcpyAsync(V.data(), f.VBv.p, sizeof(float) * V.size(), cudaMemcpyDeviceToHost, h->stream)); }
  CU(cudaStreamSynchronize(h->stream));
  const float MCMC = (float)par->it - (float)par->bi;  // sic (:626): divisor it-bi although i>bi keeps it-bi-1 draws
  std::vector<float> Bm(B.size()), MU(ns), hh;
  for (size_t i = 0; i < B.size(); i++) Bm[i] = B[i] / MCMC;
  for (int c = 0; c < ns; c++) MU[c] = (float)(sc[c].MU / MCMC);
  if ((rc = fitted_values(h, ns, Bm.data(), true, MU.data(), hh))) return rc;  // every row, the ones a mask leaves out included
  for (int c = 0; c < ns; c++) {
    const float VE = (float)(sc[c].VE / MCMC), VBs = (float)(sc[c].VB / MCMC);
    float vg;
    if (f.VBv.p) { double sv = 0; for (int64_t j = 0; j < p; j++) sv += V[(size_t)c * p + j] / MCMC; vg = (float)sv; }
    else vg = VBs * f.MSx[c];
    const float pi_out = has_pi ? 1.0f - (float)(sc[c].PI / MCMC) : 0.0f;  // :911, :975
    if (f.model == M_BCPI) vg = VBs * f.MSx[c] / pi_out;                   // :913
    if (out->mu) out->mu[c] = MU[c];
    if (out->scal) {
      double* sc_out = out->scal + (size_t)BWGR_NSCAL * c;
      sc_out[0] = VBs; sc_out[1] = VE; sc_out[2] = vg / (vg + VE); sc_out[3] = f.MSx[c]; sc_out[4] = pi_out; sc_out[5] = 0;
    }
    if (out->vb) {
      if (f.VBv.p) for (int64_t j = 0; j < p; j++) out->vb[(size_t)c * p + j] = V[(size_t)c * p + j] / MCMC;
      else out->vb[c] = VBs;
    }
  }
  if (out->b) for (size_t i = 0; i < Bm.size(); i++) out->b[i] = Bm[i];
  if (out->d && !D.empty()) for (size_t i = 0; i < D.size(); i++) out->d[i] = D[i] / MCMC;
  if (out->hat) for (size_t i = 0; i < hh.size(); i++) out->hat[i] = hh[i];
  return 0;
}

int bwgr_gibbs_fit(bwgr_handle* h, const bwgr_gibbs_params* par, const double* y, bwgr_gibbs_out* out) {
  if (!par) return fail(BWGR_ERR_ARG, "null argument");
  bwgr_gibbs_sys_params sp;
  sp.base = *par; sp.nsys = 1; sp.row_mask = nullptr; sp.chain0 = 0;
  return bwgr_gibbs_fit_sys(h, &sp, y, out);
}

// Common start of KMUP / wgr: a one-system M_KMUP fit whose state (b, d, e, per-marker L, Ve, pi) is set by the caller.
// Row multiplicities of a sweep over rows drawn with replacement (Use with repeats, :41-77): cnt [n] on the host -> the uint8 and
// float copies on the device, and xx_sys = H'H over the rows in use with their multiplicities (the scale of the rule's
// likelihood ratio).  The 0/1 mask (cnt != 0) is the caller's.
static int set_row_multiplicities(bwgr_handle* h, const uint8_t* cnt) {
  Fit& f = *h->fit;
  const int64_t n = h->n, ld = h->ld;
  std::vector<uint8_t> c8((size_t)ld, 0);
  std::vector<float> cf((size_t)ld, 0.0f);
  for (int64_t i = 0; i < n; i++) { c8[i] = cnt[i]; cf[i] = (float)cnt[i]; }
  if (f.cnt.alloc(ld) != cudaSuccess || f.row_w.alloc(ld) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  CU(cudaMemcpyAsync(f.cnt.p, c8.data(), (size_t)ld, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.row_w.p, cf.data(), sizeof(float) * ld, cudaMemcpyHostToDevice, h->stream));
  ColStatBufs cs;
  const int rc = rows_col_stats(h, cs, f.cnt.p, true, f.xx_sys.p, nullptr, nullptr);
  if (rc) return rc;
  CU(cudaStreamSynchronize(h->stream));  // c8 / cf / the scratch go out of scope
  f.weighted = true;
  return 0;
}

static int kmup_begin(bwgr_handle* h, const double* b, const double* d, const double* xx, const double* e, const double* L,
                      double Ve, double pi, uint64_t seed, const uint8_t* row_mask = nullptr, double xx_scale = 1.0,
                      const uint8_t* row_cnt = nullptr) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!b || !e || !L) return fail(BWGR_ERR_ARG, "null argument");
  if (!(Ve > 0)) return fail(BWGR_ERR_ARG, "Ve must be positive");
  const int64_t n = h->n, p = h->p, ld = h->ld;
  FitSpec s;
  // row_mask = the bagged sweep KMUP2 (:41-77): the rows in use as a mask on the small-n family, xx_scale = bg = n0 / n (:47)
  s.model = row_mask ? M_KMUP2 : M_KMUP; s.nsys = 1; s.shuffled = false; s.row_mask = row_mask; s.row_cnt = row_mask ? row_cnt : nullptr;
  s.df = 5; s.R2 = 0.5f; s.Pi = 0; s.alpha = 0; s.pi = (float)pi; s.it = 1; s.bi = 0; s.seed = seed;
  if (row_mask && !xx) return fail(BWGR_ERR_ARG, "KMUP2 needs xx");
  int rc = fit_begin(h, s, e);  // y := e (only its mean/variance feed unused defaults)
  if (rc) return rc;
  Fit& f = *h->fit;
  std::vector<float> he(ld, 0.0f), hb(p), hd(p, 1.0f), hl(p);
  float emax = 0;
  for (int64_t i = 0; i < n; i++) { he[i] = (float)e[i]; emax = std::max(emax, std::fabs(he[i])); }
  for (int64_t j = 0; j < p; j++) { hb[j] = (float)b[j]; hl[j] = (float)L[j]; if (d) hd[j] = (float)d[j]; }
  SysScalars c = f.sc0[0];
  c.mu = 0; c.ve = (float)Ve; c.pi_mix = (float)pi; c.C = -0.5f / std::sqrt((float)Ve);  // C = -0.5/sqrt(Ve) (:17, sic)
  c.sweep = 0; c.burn = 0;
  set_e_scale(c, emax);
  f.sc0[0] = c;
  f.skip_epilogue = true;  // the state is advanced by the caller's sweeps alone (KMUP) or by the wgr driver's steps
  CU(cudaMemcpyAsync(f.e.p, he.data(), sizeof(float) * ld, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.b.p, hb.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.d.p, hd.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.vbv.p, hl.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.sc.p, &c, sizeof(SysScalars), cudaMemcpyHostToDevice, h->stream));
  if (xx) {
    std::vector<float> hx(p);
    for (int64_t j = 0; j < p; j++) hx[j] = (float)xx[j] * (float)xx_scale;
    if (f.xx_over.alloc(p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    CU(cudaMemcpyAsync(f.xx_over.p, hx.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  }
  if (s.row_cnt) {  // repeated rows: multiplicities for the dot products, and H'H with a row counted as often as it was drawn
    rc = set_row_multiplicities(h, s.row_cnt);
    if (rc) return rc;
  }
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

// One sweep of the KMUP / KMUP2 fit kmup_begin set up, and its read-out: b, d and the residuals, e_out[q] = e[rows[q]] (KMUP2: the
// rows of Use, in that order) or, with rows null, all n rows.
static int kmup_sweep_out(bwgr_handle* h, const char* where, double* b, double* d, double* e_out, const double* rows, int64_t nrows) {
  Fit& f = *h->fit;
  int rc = fit_sweeps(h, 1);
  if (rc) return rc;
  rc = check_err_flag(h, where);
  if (rc) return rc;
  const int64_t n = h->n, p = h->p;
  std::vector<float> he(n), hb(p), hd(p);
  CU(cudaMemcpyAsync(he.data(), f.e.p, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(hb.data(), f.b.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(hd.data(), f.d.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (rows) for (int64_t q = 0; q < nrows; q++) e_out[q] = he[(int64_t)rows[q]];
  else for (int64_t i = 0; i < n; i++) e_out[i] = he[i];
  for (int64_t j = 0; j < p; j++) { b[j] = hb[j]; if (d) d[j] = hd[j]; }
  return 0;
}

// KMUP(X,b,d,xx,e,L,Ve,pi) (:12-38): one sweep, state updated in place.  X = the handle's store.
int bwgr_kmup_sweep(bwgr_handle* h, double* b, double* d, const double* xx, double* e, const double* L, double Ve, double pi,
                    uint64_t seed) {
  FitGuard guard{h};
  const int rc = kmup_begin(h, b, d, xx, e, L, Ve, pi, seed);
  if (rc) return rc;
  return kmup_sweep_out(h, "kmup sweep", b, d, e, nullptr, 0);
}

// Fitted values of the handle's store: hat = mu + X b.  What the reference's drivers form as X * b (emML2's u1 = X1 * b1,
// Rcpp20260726ai.cpp:1275-1276; the fit of the two-design samplers :1063, :1151, :1212; wgr's gen0 %*% B, R/wgr.R:147).
int bwgr_fitted_sys(bwgr_handle* h, int k, const double* B, const double* mu, double* hat) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!B || !mu || !hat) return fail(BWGR_ERR_ARG, "null argument");
  if (k < 1) return fail(BWGR_ERR_ARG, "bad k %d", k);
  if (h->world > 1) return fail(BWGR_ERR_UNSUPPORTED, "bwgr_fitted on a row-sharded store");
  if (h->col_offset.size()) return fail(BWGR_ERR_UNSUPPORTED, "this store holds integer codes + a constant per column: use the solvers that centre the columns themselves");
  CU(cudaSetDevice(h->device));
  const int64_t n = h->n, p = h->p;
  std::vector<float> bf((size_t)k * p), m0(k), hh;
  for (size_t j = 0; j < bf.size(); j++) bf[j] = (float)B[j];
  for (int t = 0; t < k; t++) m0[t] = (float)mu[t];
  const int rc = fitted_values(h, k, bf.data(), true, m0.data(), hh);
  if (rc) return rc;
  for (size_t i = 0; i < (size_t)k * n; i++) hat[i] = hh[i];
  return 0;
}

int bwgr_fitted(bwgr_handle* h, const double* b, double mu, double* hat) { return bwgr_fitted_sys(h, 1, b, &mu, hat); }

// wgr(y, X, it, bi, th, bag, rp, iv, de, pi, df, R2, eigK = NULL) (R/wgr.R:2-169) with the MCMC loop on the device.
// bag = 1: `it` KMUP sweeps, each followed by the driver's step on the device (wgr_mode).
// bag != 1 (:21, :49, :68, :87, :121): every iteration sweeps a fresh sorted sample of floor(n * bag) rows with KMUP2, estimates Ve
// from their residuals, and rebuilds e = y - mu - X b over all rows.  The row samples come from std::mt19937_64(seed), not from R's
// sample().
static int wgr_fit(bwgr_handle* h, const double* y, int it, int bi, int th, double bag, int rp, int iv, int de, double pi, double df,
                   double R2, uint64_t seed, double* b, double* d, double* Vb, double* hat, double* scal) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!y) return fail(BWGR_ERR_ARG, "y is NULL");
  if (it < 1 || bi < 1 || bi > it || th < 1) return fail(BWGR_ERR_ARG, "need 1 <= bi <= it and th >= 1");
  const bool bagged = bag != 1.0;
  const int64_t n = h->n, p = h->p, ld = h->ld;
  const int64_t nuse = (int64_t)((double)n * bag);
  if (bagged && (!(bag > 0) || nuse < 2 || (!rp && nuse > n))) return fail(BWGR_ERR_ARG, "bag must give 2 <= n * bag (<= n rows without replacement)");
  if (de) iv = 1;  // R/wgr.R:10
  if (bagged) df = df / (bag * bag);  // :21
  // initial state (R/wgr.R:46-59): b = 0, d = 1, mu = mean(y), e = y - mu, Va = MSx, Vb = Va, Ve = 1, L = Vb/Ve (sic)
  double mu = 0;
  for (int64_t i = 0; i < n; i++) { if (!(y[i] == y[i])) return fail(BWGR_ERR_ARG, "y contains NaN"); mu += y[i]; }
  mu /= (double)n;
  double vy = 0;
  for (int64_t i = 0; i < n; i++) vy += (y[i] - mu) * (y[i] - mu);
  vy /= (double)(n - 1);
  double MSx = 0, sxx = 0;
  for (int64_t j = 0; j < p; j++) { MSx += (h->h_xx[j] - h->h_sx[j] * h->h_sx[j] / (double)n) / ((double)n - 1.0); sxx += h->h_xx[j] * bag; }
  if (!(MSx > 0)) return fail(BWGR_ERR_ARG, "genotypes have no variance");
  std::vector<double> e0(n), b0(p, 0.0), d0(p, 1.0), L0(p, MSx), xxb(p);
  for (int64_t i = 0; i < n; i++) e0[i] = y[i] - mu;
  for (int64_t j = 0; j < p; j++) xxb[j] = h->h_xx[j] * bag;  // xx = crossprod * bag (:49)
  std::mt19937_64 gen(seed ^ 0x9E3779B97F4A7C15ull);
  std::vector<int64_t> rows(n);
  std::vector<uint8_t> mask((size_t)ld, 0), cnt((size_t)ld, 0);
  std::vector<float> cntf((size_t)ld, 0.0f);
  bool overflow = false;
  auto draw = [&]() {  // Use = sort(sample(n, n * bag, rp)) (:68) as a mask (+ the multiplicity of every row when rp = TRUE)
    std::fill(mask.begin(), mask.end(), 0);
    if (rp) {
      std::fill(cnt.begin(), cnt.end(), 0);
      std::uniform_int_distribution<int64_t> pick(0, n - 1);
      for (int64_t r = 0; r < nuse; r++) { const int64_t q = pick(gen); mask[q] = 1; if (cnt[q] == 255) overflow = true; else cnt[q]++; }
      for (int64_t r = 0; r < n; r++) cntf[r] = (float)cnt[r];
      return;
    }
    for (int64_t r = 0; r < n; r++) rows[r] = r;
    for (int64_t r = 0; r < nuse; r++) { std::uniform_int_distribution<int64_t> pick(r, n - 1); std::swap(rows[r], rows[pick(gen)]); mask[rows[r]] = 1; }
  };
  FitGuard guard{h};
  int rc;
  if (bagged) {
    draw();
    rc = kmup_begin(h, b0.data(), d0.data(), xxb.data(), e0.data(), L0.data(), 1.0, pi, seed, mask.data(), (double)((float)n / (float)nuse),
                    rp ? cnt.data() : nullptr);
  } else {
    rc = kmup_begin(h, b0.data(), d0.data(), nullptr, e0.data(), L0.data(), 1.0, pi, seed);
  }
  if (rc) return rc;
  Fit& f = *h->fit;
  {
    SysScalars c = f.sc0[0];
    c.mu = (float)mu;
    CU(cudaMemcpyAsync(f.sc.p, &c, sizeof(SysScalars), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  if (f.wst.alloc(1) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  CU(cudaMemsetAsync(f.wst.p, 0, sizeof(WgrState), h->stream));
  WgrArgs& w = f.wgr_args;
  memset(&w, 0, sizeof w);
  w.n = (int)n; w.p = (int)p; w.ld = ld; w.e = f.e.p; w.b = f.b.p; w.d = f.d.p; w.L = f.vbv.p;
  w.B = f.B.p; w.D = f.D.p; w.VB = f.VBv.p; w.sc = f.sc.p; w.st = f.wst.p; w.iv = iv; w.de = de;
  w.Sb = (float)(R2 * df * vy / MSx); w.Se = (float)((1 - R2) * df * vy); w.df = (float)df; w.MSx = (float)MSx;  // :58-59
  w.it = it; w.bi = bi; w.th = th; w.seed_lo = (uint32_t)seed; w.seed_hi = (uint32_t)(seed >> 32);
  if (!bagged) {
    f.wgr_mode = true;
    if ((rc = fit_sweeps(h, it))) return rc;
  } else {
    DevBuf<float> yd, hatd;
    if (yd.alloc(ld) != cudaSuccess || hatd.alloc(ld) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    std::vector<float> yf(ld, 0.0f);
    for (int64_t i = 0; i < n; i++) yf[i] = (float)y[i];
    CU(cudaMemcpyAsync(yd.p, yf.data(), sizeof(float) * ld, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    // phase 1 weighs e^2 by the byte (0/1 or the multiplicity); Ve's chi-square has n * bag + df degrees of freedom (:121), n * bag
    // unrounded although the sample holds floor(n * bag) rows
    w.mask = rp ? f.cnt.p : f.mask.p; w.nsub = (float)((double)n * bag); w.y = yd.p; w.hat = hatd.p;
    ColStatBufs cs;
    for (int i = 0; i < it; i++) {
      if (i > 0) {  // this iteration's rows: mask, and H'H of every marker over them (the rule's likelihood-ratio scale)
        draw();
        CU(cudaMemcpyAsync(f.mask.p, mask.data(), (size_t)ld, cudaMemcpyHostToDevice, h->stream));
        if (rp) {
          if (overflow) return fail(BWGR_ERR_UNSUPPORTED, "wgr(rp = TRUE): a row was drawn more than 255 times in one iteration");
          CU(cudaMemcpyAsync(f.cnt.p, cnt.data(), (size_t)ld, cudaMemcpyHostToDevice, h->stream));
          CU(cudaMemcpyAsync(f.row_w.p, cntf.data(), sizeof(float) * ld, cudaMemcpyHostToDevice, h->stream));
        }
        if ((rc = rows_col_stats(h, cs, rp ? f.cnt.p : f.mask.p, rp, f.xx_sys.p, nullptr, nullptr))) return rc;
      }
      if ((rc = fit_sweeps(h, 1))) return rc;                                    // KMUP2 over the rows in use
      launch_wgr_bag_phase(w, 1, h->num_sms, h->stream);                          // Vb (with the old Ve), Va, Ve from the rows in use
      if ((rc = fit_hat(h, 1, f.b.p, reinterpret_cast<const float*>(f.sc.p), hatd.p))) return rc;  // mu + X b  (SysScalars starts with mu)
      launch_wgr_bag_phase(w, 2, h->num_sms, h->stream);                          // e = y - hat, intercept draw, L, posterior sums
      h->launches += 3;
    }
  }
  rc = check_err_flag(h, bagged ? "wgr (bagged) sweep" : "wgr sweep");
  if (rc) return rc;
  if (!bagged) dump_trace(h);
  WgrState st;
  CU(cudaMemcpyAsync(&st, f.wst.p, sizeof st, cudaMemcpyDeviceToHost, h->stream));
  std::vector<float> B(p), D(p), V(p);
  CU(cudaMemcpyAsync(B.data(), f.B.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(D.data(), f.D.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(V.data(), f.VBv.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  const double mc = (double)((it - bi) / th + 1);  // length(seq(bi, it, th)) (:41-42)
  double mD = 0;
  for (int64_t j = 0; j < p; j++) mD += D[j] / mc;
  mD /= (double)p;
  std::vector<float> Bm(p), hh;
  for (int64_t j = 0; j < p; j++) Bm[j] = (float)(B[j] / mc / mD);  // B = B/mc/mean(D) (:143)
  const float B0 = (float)(st.B0 / mc);
  rc = fitted_values(h, 1, Bm.data(), true, &B0, hh);  // HAT = B0 + gen0 %*% B (:152)
  if (rc) return rc;
  if (b) for (int64_t j = 0; j < p; j++) b[j] = Bm[j];
  if (d) for (int64_t j = 0; j < p; j++) d[j] = D[j] / mc;
  if (Vb && iv) for (int64_t j = 0; j < p; j++) Vb[j] = V[j] / mc;
  if (hat) for (int64_t i = 0; i < n; i++) hat[i] = hh[i];
  if (scal) { scal[0] = B0; scal[1] = st.VE / mc; scal[2] = iv ? 0.0 : st.VA / mc; scal[3] = sxx / (double)p; }
  return 0;
}

int bwgr_wgr_fit(bwgr_handle* h, const double* y, int it, int bi, int th, int iv, int de, double pi, double df, double R2,
                 uint64_t seed, double* b, double* d, double* Vb, double* hat, double* scal) {
  return wgr_fit(h, y, it, bi, th, 1.0, 0, iv, de, pi, df, R2, seed, b, d, Vb, hat, scal);
}

// Rows of one bagged iteration as a 0/1 mask plus the multiplicity of every row.  use: 0-based row indices as R passes them
// (doubles).  *repeats = some row occurs more than once (sampling with replacement, rp = TRUE).
static int use_to_mask(const double* use, int64_t nuse, int64_t n, std::vector<uint8_t>& mask, std::vector<uint8_t>& cnt, bool* repeats) {
  mask.assign((size_t)n, 0);
  cnt.assign((size_t)n, 0);
  *repeats = false;
  for (int64_t q = 0; q < nuse; q++) {
    const int64_t r = (int64_t)use[q];
    if (r < 0 || r >= n) return fail(BWGR_ERR_ARG, "Use[%lld] = %lld is not a row of X", (long long)q, (long long)r);
    if (cnt[r] == 255) return fail(BWGR_ERR_UNSUPPORTED, "KMUP2: row %lld occurs more than 255 times in Use", (long long)r);
    if (mask[r]) *repeats = true;
    mask[r] = 1;
    cnt[r]++;
  }
  return 0;
}

// KMUP2(X,Use,b,d,xx,E,L,Ve,pi) (:41-77): one Kuo-Mallick sweep over the rows Use.  b, d updated in place; e_out [nuse] = the
// residuals of the rows in use, in the order of Use (the reference's third list element).  Runs on the small-n family (row mask).
int bwgr_kmup2_sweep(bwgr_handle* h, const double* use, int64_t nuse, double* b, double* d, const double* xx, const double* E,
                     double* e_out, const double* L, double Ve, double pi, uint64_t seed) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!use || !E || !e_out || nuse < 2) return fail(BWGR_ERR_ARG, "KMUP2: bad Use / E / e_out");
  const int64_t n = h->n;
  std::vector<uint8_t> mask, cnt;
  bool repeats = false;
  int rc = use_to_mask(use, nuse, n, mask, cnt, &repeats);
  if (rc) return rc;
  FitGuard guard{h};
  rc = kmup_begin(h, b, d, xx, E, L, Ve, pi, seed, mask.data(), (double)((float)n / (float)nuse), repeats ? cnt.data() : nullptr);
  if (rc) return rc;
  return kmup_sweep_out(h, "kmup2 sweep", b, d, e_out, use, nuse);
}

// wgr(y,X,it,bi,th,bag,rp,iv,de,pi,df,R2): bwgr_wgr_fit with row bagging (see wgr_fit); bag = 1 is bwgr_wgr_fit.  Same outputs.
int bwgr_wgr_fit_bag(bwgr_handle* h, const double* y, int it, int bi, int th, double bag, int rp, int iv, int de, double pi, double df,
                     double R2, uint64_t seed, double* b, double* d, double* Vb, double* hat, double* scal) {
  return wgr_fit(h, y, it, bi, th, bag, rp, iv, de, pi, df, R2, seed, b, d, Vb, hat, scal);
}

}  // extern "C"
