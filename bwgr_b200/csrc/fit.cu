// fit.cu -- the fit engine every solver shares: the kernel family and geometry of a fit, its initial state (SURVEY A.1), the marker
// orders (libstdc++'s std::shuffle, cumulative, Rcpp20260726ai.cpp:329-331), the sweeps with their Gram bands and epilogues, and the
// fitted values.  All host work is O(p) or O(n) per sweep and overlapped with the GPU; every sweep runs in a CUDA kernel.
#include "host.h"

namespace bwgr::host {

float fvar_f(const std::vector<float>& x) {  // fvar, Rcpp20260726ai.cpp:7-9 (sums in double, rounded once)
  double m = 0;
  for (float v : x) m += v;
  const float mean = (float)(m / (double)x.size());
  double s = 0;
  for (float v : x) { const float t = v - mean; s += (double)t * t; }
  return (float)s / (float)(x.size() - 1);
}

bool plan_pipe(const bwgr_handle* h, int model, int ns, PipePlan* pl) {
  if (h->storage != BWGR_STORE_I8 || ns > 32) return false;
  int sms = h->grid > 1 ? std::min(h->grid, h->num_sms) : h->num_sms;  // CTAs of the flat topology
  if (h->world > 1 && h->grid <= 1 && h->x2f.p && h->comm_side && h->num_sms > 64) {
    // row-sharded fit, flat topology: the per-block chain is latency-bound, so ~104 CTAs sweep as fast as 148 and the SMs left idle
    // compute the next sweep's Gram band meanwhile (measured at 50k x 50k: 104 CTAs 1.54 ms per sweep, 120: 1.68, 148: 1.84)
    const int want = h->num_sms - 44;
    if ((h->ld + want - 2) / (want - 1) <= 496) sms = want;
  }
  if (sms < 2) return false;
  const int W0 = sms - 1;
  const int R = (int)(((h->ld + W0 - 1) / W0 + 15) / 16 * 16);
  if (R > 512) return false;
  const int W = (int)((h->ld + R - 1) / R);
  const int NA = (R + 127) / 128, N = ((4 * ns + 15) / 16) * 16;
  if ((NA + 1) * N > 512) return false;
  int D = 1;
  // one linear system on uncentred columns: the in-block solve applies the precomputed block inverse (block_inv.cu).
  // (MRR3's centred systems keep the stepwise solve.)
  const int full_inv = model_is_linear(model) && ns == 1 && model != M_MRR;
  pl->cl = 0; pl->nclusters = 0;
  // Clustered topology (sweep_pipe.cu): thread-block clusters of one solver + seven workers; steps travel through distributed shared
  // memory, and every worker adds its partial sums to L2 grid-sum words: one L2 hop per block.
  // Single GPU at the default grid, at most three systems; otherwise the flat topology (one solver CTA, two-hop L2 tree).  Row-sharded
  // fits use the flat one: a clustered variant with a third (NVLink) hop after the cluster exchange measured 1.79 ms against 1.43 ms per sweep.
  if (h->world <= 1 && h->grid <= 1 && sweep_pipe_cluster_ok(model, ns, full_inv)) {
    {
      // The sweep is latency-bound: 14 clusters sweep as fast as 15 (measured 1.226 against 1.235 ms at 50k x 50k), and every SM left
      // idle works on the next sweep's Gram band meanwhile (fit_sweeps).  First choice: leave at least 36 SMs; if the rows per
      // worker then exceed the tile (512), take every cluster that fits.
      const int cap_side = std::max(2, (h->num_sms - 36) / 8);
      for (int nbuf = D + 2; nbuf >= D + 1; nbuf--)
      for (int pass = 0; pass < 2; pass++) {
        // rows per worker depend on the number of co-resident clusters, which depends on the shared memory per CTA: iterate
        int C = pass == 0 ? std::min(18, cap_side) : 18;
        for (int iter = 0; iter < 4 && C >= 2; iter++) {
          const int Wc = 7 * C;
          const int Rc = (int)(((h->ld + Wc - 1) / Wc + 15) / 16 * 16);
          if (Rc > 512) { C = 0; break; }
          const size_t smem = sweep_pipe_smem(Rc, ns, model, nbuf, 3, full_inv, 1);
          if (smem > h->smem_optin - 9216) { C = 0; break; }  // the kernel's static shared memory (barriers, system scalars) is ~9 KB
          const int Cmax = std::min(18, sweep_pipe_max_clusters(model, smem));
          if (Cmax >= C) break;
          C = Cmax;
        }
        if (C >= 2) {
          const int Wc = 7 * C;
          const int Rc = (int)(((h->ld + Wc - 1) / Wc + 15) / 16 * 16);
          const int NAc = (Rc + 127) / 128;
          if ((NAc + 1) * N <= 512 && sweep_pipe_smem(Rc, ns, model, nbuf, 3, full_inv, 1) <= h->smem_optin - 9216) {
            pl->R = Rc; pl->W = Wc; pl->nbuf = nbuf; pl->D = D; pl->sring = 3; pl->full_inv = full_inv; pl->cl = 1; pl->nclusters = C;
            return true;
          }
        }
      }
    }
  }
  for (; D >= 0; D--) {
    for (int sring = 3; sring >= 2; sring--)
      for (int nbuf = std::min(8, D + 3); nbuf >= D + 1; nbuf--)
        if (sweep_pipe_smem(R, ns, model, nbuf, sring, full_inv, 0) <= h->smem_optin - 8192) {
          pl->R = R; pl->W = W; pl->nbuf = nbuf; pl->D = D; pl->sring = sring; pl->full_inv = full_inv;
          return true;
        }
  }
  return false;
}

void grid_geometry(bwgr_handle* h, int* rp, int* grid) {
  int r = (int)((h->ld + h->num_sms - 1) / h->num_sms);
  r = std::max(64, (r + 15) / 16 * 16);
  *rp = r;
  *grid = (int)((h->ld + r - 1) / r);
}

// path: the BWGR_PATH_* to honour
static int choose_path(bwgr_handle* h, const FitSpec& s, int path, Family* family) {
  const GenoView g = h->view();
  const bool small_ok = h->storage != BWGR_STORE_F32 && small_n_fits(g, s.row_mask != nullptr, h->smem_optin, s.row_cnt != nullptr);
  PipePlan pl;
  const bool blocked_ok = !s.row_mask && plan_pipe(h, s.model, s.nsys, &pl);
  int grp = 0, ggrid = 0;
  grid_geometry(h, &grp, &ggrid);
  const bool grid_ok = (h->storage == BWGR_STORE_I8 || h->storage == BWGR_STORE_F32) && h->world <= 1 && s.nsys <= 32 && s.model != M_MRR &&
                       ggrid <= 255 && grid_sweep_smem(s.nsys, grp, s.row_mask != nullptr, h->storage == BWGR_STORE_F32) <= h->smem_optin;
  if (path == BWGR_PATH_SMALL_N) {
    if (!small_ok) return fail(BWGR_ERR_UNSUPPORTED, "small-n path: residual of n=%lld does not fit one SM", (long long)h->n);
    *family = Family::SmallN;
  } else if (path == BWGR_PATH_BLOCKED) {
    if (!blocked_ok) return fail(BWGR_ERR_UNSUPPORTED, "blocked path needs the int8 store, no row mask, nsys<=32 and n <= 512 rows x grid");
    *family = Family::Blocked;
  } else if (path == BWGR_PATH_GRID) {
    if (!grid_ok) return fail(BWGR_ERR_UNSUPPORTED, "grid path needs the int8 or float32 store, one GPU, nsys<=32 and the row slabs of all systems in shared memory");
    *family = Family::Grid;
  } else {
    const bool prefer_small = small_ok && (s.row_mask || s.nsys >= 8 || h->n <= 1024);
    if (prefer_small) *family = Family::SmallN;
    else if (blocked_ok) *family = Family::Blocked;
    else if (small_ok) *family = Family::SmallN;
    else if (grid_ok) *family = Family::Grid;
    else return fail(BWGR_ERR_UNSUPPORTED, "no kernel family fits n=%lld nsys=%d storage=%d", (long long)h->n, s.nsys, h->storage);
  }
  return 0;
}

// Column statistics over the rows a system uses -- a 0/1 row mask, or (cnt) the multiplicity of every row -- with
// xx_j = sum_i w_i x_ij^2 as floats into xx_sys [p].  With xx / sx, both sums also come back as host doubles, and the float
// conversion runs on the host.
int rows_col_stats(bwgr_handle* h, ColStatBufs& s, const uint8_t* rows, bool cnt, float* xx_sys, std::vector<double>* xx, std::vector<double>* sx) {
  const int64_t p = h->p;
  const bool exact = !cnt && h->storage != BWGR_STORE_F32;
  if (exact) {
    if (s.xx_i.n < (size_t)p && (s.xx_i.alloc(p) != cudaSuccess || s.sx_i.alloc(p) != cudaSuccess)) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    launch_col_stats_masked(h->view(), rows, s.xx_i.p, s.sx_i.p, h->stream);
  } else {
    if (s.xx_d.n < (size_t)p && (s.xx_d.alloc(p) != cudaSuccess || s.sx_d.alloc(p) != cudaSuccess)) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    if (cnt) launch_col_stats_cnt(h->view(), rows, s.xx_d.p, s.sx_d.p, h->stream);
    else launch_col_stats_f32(h->view(), rows, s.xx_d.p, s.sx_d.p, h->stream);
  }
  h->launches++;
  if (!xx) {
    if (exact) launch_ll_to_float(s.xx_i.p, xx_sys, (int)p, h->stream);
    else launch_d_to_float(s.xx_d.p, xx_sys, (int)p, h->stream);
    h->launches++;
    return 0;
  }
  xx->resize(p); sx->resize(p);
  if (exact) {
    std::vector<long long> hx(p), hs(p);
    CU(cudaMemcpyAsync(hx.data(), s.xx_i.p, sizeof(long long) * p, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(hs.data(), s.sx_i.p, sizeof(long long) * p, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    xx->assign(hx.begin(), hx.end()); sx->assign(hs.begin(), hs.end());  // exact: |sums| < 2^45
  } else {
    CU(cudaMemcpyAsync(xx->data(), s.xx_d.p, sizeof(double) * p, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(sx->data(), s.sx_d.p, sizeof(double) * p, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  std::vector<float> xf(p);
  for (int64_t j = 0; j < p; j++) xf[j] = (float)(*xx)[j];
  CU(cudaMemcpyAsync(xx_sys, xf.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int fit_begin(bwgr_handle* h, const FitSpec& s, const double* y) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!y) return fail(BWGR_ERR_ARG, "y is NULL");
  if (s.nsys < 1 || s.nsys > 4096) return fail(BWGR_ERR_ARG, "bad nsys %d", s.nsys);
  if (h->has_offset && s.model != M_MRR)
    return fail(BWGR_ERR_UNSUPPORTED, "this store holds integer codes + a constant per column (bwgr_geno_load_f64_centred): only the solvers that "
                                      "centre the columns themselves (MRR3 / MRR3F) can use it");
  CU(cudaSetDevice(h->device));
  h->fit.reset();
  std::unique_ptr<Fit> fit(new Fit(h));
  Fit& f = *fit;
  const bool dist = h->world > 1;
  if (dist) {
    if (!h->hx_connected) return fail(BWGR_ERR_STATE, "row-sharded handle: call bwgr_dist_connect before fitting");
    if (s.row_mask) return fail(BWGR_ERR_UNSUPPORTED, "row-sharded fits take unmasked systems");
    if (s.model == M_KMUP || s.model == M_KMUP2) return fail(BWGR_ERR_UNSUPPORTED, "row sharding covers the EM and Gibbs solvers and MRR3's fast path");
  }
  // row-sharded fits and MRR3's rotated systems run on the pipelined blocked sweep only
  int rc = choose_path(h, s, dist || s.model == M_MRR ? BWGR_PATH_BLOCKED : h->path, &f.family);
  if (rc) return rc;
  const int64_t n = h->n, p = h->p, ld = h->ld;
  const int ns = s.nsys;
  f.model = s.model; f.nsys = ns; f.shuffled = s.shuffled; f.masked = s.row_mask != nullptr;
  f.seed = s.seed; f.chain0 = s.chain0; f.it_target = s.it;

  // ---- per-system row masks and column statistics
  std::vector<float> n_eff(ns, (float)(dist ? h->n_global : n));
  std::vector<std::vector<double>> xx_s, sx_s;  // masked systems only
  if (f.masked) {
    std::vector<uint8_t> m((size_t)ns * ld, 0);
    for (int t = 0; t < ns; t++) {
      int cnt = 0;
      for (int64_t i = 0; i < n; i++) { const uint8_t v = s.row_mask[(size_t)t * n + i] ? 1 : 0; m[(size_t)t * ld + i] = v; cnt += v; }
      if (cnt < 2) return fail(BWGR_ERR_ARG, "row_mask of system %d keeps %d rows", t, cnt);
      n_eff[t] = (float)cnt;
    }
    if (f.mask.alloc(m.size()) != cudaSuccess || f.xx_sys.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    CU(cudaMemcpyAsync(f.mask.p, m.data(), m.size(), cudaMemcpyHostToDevice, h->stream));
    xx_s.resize(ns); sx_s.resize(ns);
    ColStatBufs cs;
    for (int t = 0; t < ns; t++)
      if ((rc = rows_col_stats(h, cs, f.mask.p + (size_t)t * ld, false, f.xx_sys.p + (size_t)t * p, &xx_s[t], &sx_s[t]))) return rc;
  }

  // ---- initial state per system (SURVEY A.1), float arithmetic
  f.sc0.assign(ns, SysScalars());
  f.vy.assign(ns, 0); f.MSx.assign(ns, 0); f.cxx.assign(ns, 0);
  std::vector<float> hy((size_t)ns * ld, 0.0f), he((size_t)ns * ld, 0.0f);
  std::vector<float> hvb;  // initial per-marker variance
  float vbv_init = 1.0f;
  for (int t = 0; t < ns; t++) {
    std::vector<float> yt;
    yt.reserve(n);
    for (int64_t i = 0; i < n; i++) {
      const double v = y[(size_t)t * n + i];
      if (!(v == v)) return fail(BWGR_ERR_ARG, "y contains NaN (man/em.Rd:38 forbids NA in y)");
      hy[(size_t)t * ld + i] = (float)v;
      if (!f.masked || s.row_mask[(size_t)t * n + i]) yt.push_back((float)v);
    }
    const float nn = n_eff[t];
    const std::vector<double>& xx = f.masked ? xx_s[t] : h->h_xx;
    const std::vector<double>& sx = f.masked ? sx_s[t] : h->h_sx;
    double svx = 0, sxx = 0, tr = 0;
    for (int64_t j = 0; j < p; j++) {
      const double v = (xx[j] - sx[j] * sx[j] / (double)nn) / ((double)nn - 1.0);
      svx += (double)(float)v;
      sxx += xx[j];
    }
    const float sum_vx = (float)svx;
    float vy, mu;
    if (!dist) {
      vy = fvar_f(yt);
      double sm = 0;
      for (float v : yt) sm += v;
      mu = (float)(sm / (double)yt.size());
    } else {  // mean and variance of y over ALL individuals (two small all-reduces)
      double sm = 0;
      for (float v : yt) sm += v;
      rc = dist_allreduce_host(h, &sm, 1, false);
      if (rc) return rc;
      mu = (float)(sm / (double)h->n_global);
      double ss = 0;
      for (float v : yt) { const float tt = v - mu; ss += (double)tt * tt; }
      rc = dist_allreduce_host(h, &ss, 1, false);
      if (rc) return rc;
      vy = (float)ss / (float)(h->n_global - 1);
    }
    SysScalars c;
    memset(&c, 0, sizeof c);
    c.mu = mu; c.df = s.df; c.R2 = s.R2; c.alpha = s.alpha; c.vy = vy; c.n_eff = nn; c.pi_mix = s.pi;
    c.burn = s.bi; c.sweep = 0;
    const float df = s.df, R2 = s.R2;
    float Pi = s.Pi;
    switch (s.model) {
      case M_EMRR: {  // Rcpp20260726ai.cpp:317-324
        const float MSx = sum_vx;
        c.MSx = MSx; c.lmb = MSx; c.Rho = MSx * (1 - R2) / R2; c.ve = 0.5f * vy; c.vb = c.ve / MSx;
        c.Se = (1 - R2) * (df + 2) * vy; c.Sb = R2 * (df + 2) * vy / MSx;
        break;
      }
      case M_EMBA: {  // :84-97
        const float MSx = sum_vx;
        c.MSx = MSx; c.ve = 1; c.Sb = R2 * (df + 2) * vy / MSx; c.Se = (1 - R2) * (df + 2) * vy;
        vbv_init = 1.0f;
        break;
      }
      case M_EMBB: {  // :135-154
        if (Pi > 0.5f) Pi = 1 - Pi;
        const float MSx = sum_vx * Pi;
        c.MSx = MSx; c.ve = 1; c.Sb = R2 * (df + 2) * vy / MSx; c.Se = (1 - R2) * (df + 2) * vy;
        c.Pi = Pi; c.Pi0 = (1 - Pi) / Pi;
        vbv_init = 1.0f;
        break;
      }
      case M_EMBC: {  // :196-213 (ve = Sa, va = Se: sic)
        if (Pi > 0.5f) Pi = 1 - Pi;
        const float MSx = sum_vx * Pi * (1 - Pi);
        c.MSx = MSx; c.Sa = R2 * (df + 2) * vy / MSx; c.Se = (1 - R2) * (df + 2) * vy;
        c.ve = c.Sa; c.vb = c.Se; c.lmb = c.ve / c.vb; c.Pi = Pi; c.Pi0 = (1 - Pi) / Pi;
        break;
      }
      case M_EMBL: {  // :359-370
        const float h2 = R2;
        const float cxx = (float)(sxx / (double)p);
        c.cxx = cxx;
        c.lmb1 = cxx * ((1 - h2) / h2) * s.alpha * 0.5f;
        c.lmb2 = cxx * ((1 - h2) / h2) * (1 - s.alpha);
        break;
      }
      case M_EMEN: {  // :412-419
        const float cxx = sum_vx * (1 - R2) / R2;
        c.cxx = cxx; c.Sy = std::sqrt(vy); c.lmb = cxx;
        c.lmb1 = 0.5f * cxx * s.alpha * c.Sy; c.lmb2 = cxx * (1 - s.alpha);
        for (int64_t j = 0; j < p; j++) tr += 1.0 / ((double)(float)xx[j] + (double)cxx);
        c.trAC22 = (float)tr;
        break;
      }
      case M_EMDE: {  // :262-270 ; the per-marker slot carries Lmb_j
        const float cxx = sum_vx * (1 - R2) / R2;
        c.cxx = cxx;
        vbv_init = (float)p + cxx;
        break;
      }
      case M_EMMLD:
      case M_EMML: {  // :480-486
        c.MSx = sum_vx; c.lmb = sum_vx;
        break;
      }
      case M_GSRR: case M_GSFLM: break;  // warm start: the caller's state is uploaded by bwgr_gs_fit
      case M_EMBCPI: {  // :1508-1520 (emBC's start; the prior Pi is kept for the per-sweep update of Pi)
        if (Pi > 0.5f) Pi = 1 - Pi;
        const float MSx = sum_vx * Pi * (1 - Pi);
        c.MSx = MSx; c.Sa = R2 * (df + 2) * vy / MSx; c.Se = (1 - R2) * (df + 2) * vy;
        c.ve = c.Sa; c.vb = c.Se; c.lmb = c.ve / c.vb; c.Pi = Pi; c.Pi0 = (1 - Pi) / Pi;
        c.cxx = sum_vx; c.pi_mix = Pi;
        break;
      }
      case M_LASSO: {  // :1470-1472
        c.lmb = (float)(sxx / (double)p) / (float)p;
        break;
      }
      case M_BRR: case M_BA: case M_BB: case M_BL: case M_BDPI: {  // :822-827, :598-609, :649-665, :771-783, :931-944
        const float MSx = sum_vx;
        c.MSx = MSx; c.Sb = R2 * df * vy / MSx; c.Se = (1 - R2) * df * vy; c.ve = vy; c.vb = c.Sb; c.lmb = c.ve / c.vb;
        c.Pi0 = s.pi / (1.0f - s.pi);
        c.Rho = MSx * (1 - R2) / R2;  // BayesL's Phi (:773)
        c.Pi = s.pi;                  // BayesDpi: pi = 0.5 at the start (:934), then the mean inclusion
        vbv_init = c.Sb;
        break;
      }
      case M_BCPI:  // :866-880 = BayesC started at pi = 0.5
      case M_BC: {  // :712-726
        const float MSx = sum_vx;
        c.MSx = MSx; c.Sb = df * R2 * vy / MSx / (1 - s.pi); c.Se = df * (1 - R2) * vy; c.ve = vy; c.vb = c.Sb;
        c.lmb = c.ve / c.vb; c.Pi0 = s.pi / (1.0f - s.pi); c.Pi = s.pi;
        break;
      }
      case M_MRR: {  // rotated MRR3 systems: lambda and scales are set per sweep by the driver
        c.MSx = sum_vx; c.ve = 1; c.vb = 1; c.lmb = 1;
        break;
      }
      case M_KMUP2:
      case M_KMUP: {  // state comes from the caller (KMUP :12-38) or from the wgr driver (R/wgr.R:46-59)
        c.MSx = sum_vx; c.ve = 1; c.vb = 1; c.lmb = 1;
        break;
      }
      default: return fail(BWGR_ERR_ARG, "bad model %d", s.model);
    }
    c.C = -0.5f / std::sqrt(c.ve);
    {  // fixed-point scale of the residuals, from max|y - mu|
      float emax = 0;
      for (float v : yt) emax = std::max(emax, std::fabs(v - mu));
      if (dist) {  // the fixed-point scale must be the same on every rank
        double em = emax;
        rc = dist_allreduce_host(h, &em, 1, true);
        if (rc) return rc;
        emax = (float)em;
      }
      set_e_scale(c, emax);
    }
    f.sc0[t] = c;
    f.vy[t] = vy; f.MSx[t] = c.MSx; f.cxx[t] = c.cxx;
    for (int64_t i = 0; i < n; i++)
      if (!f.masked || s.row_mask[(size_t)t * n + i]) he[(size_t)t * ld + i] = hy[(size_t)t * ld + i] - mu;
    if (model_has_vbj(s.model)) hvb.resize((size_t)ns * p), std::fill(hvb.begin() + (size_t)t * p, hvb.begin() + (size_t)(t + 1) * p, vbv_init);
  }

  // ---- device state
  const bool gibbs = model_is_gibbs(s.model);
  if (f.y.alloc((size_t)ns * ld) != cudaSuccess || f.e.alloc((size_t)ns * ld) != cudaSuccess ||
      f.b.alloc((size_t)ns * p) != cudaSuccess || f.sc.alloc(ns) != cudaSuccess || f.perm.alloc((size_t)kPermRing * p) != cudaSuccess)
    return fail(BWGR_ERR_CUDA, "cudaMalloc(fit state) failed");
  if (model_has_d(s.model) && f.d.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  if (model_has_vbj(s.model) && f.vbv.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  if (model_has_cnv(s.model) && f.b_prev.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  if (gibbs) {
    if (f.B.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    CU(cudaMemsetAsync(f.B.p, 0, sizeof(float) * ns * p, h->stream));
    if (f.d.p) { if (f.D.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed"); CU(cudaMemsetAsync(f.D.p, 0, sizeof(float) * ns * p, h->stream)); }
    if (f.vbv.p) { if (f.VBv.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed"); CU(cudaMemsetAsync(f.VBv.p, 0, sizeof(float) * ns * p, h->stream)); }
  }
  CU(cudaMemcpyAsync(f.y.p, hy.data(), sizeof(float) * hy.size(), cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.e.p, he.data(), sizeof(float) * he.size(), cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemsetAsync(f.b.p, 0, sizeof(float) * ns * p, h->stream));
  if (f.d.p) CU(cudaMemsetAsync(f.d.p, 0, sizeof(float) * ns * p, h->stream));
  if (f.vbv.p) CU(cudaMemcpyAsync(f.vbv.p, hvb.data(), sizeof(float) * hvb.size(), cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.sc.p, f.sc0.data(), sizeof(SysScalars) * ns, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));

  f.h_perm_bytes = sizeof(int) * kPermRing * p;
  CU(pinned_alloc(reinterpret_cast<void**>(&f.h_perm), f.h_perm_bytes));
  for (int i = 0; i < kPermRing; i++) CU(cudaEventCreateWithFlags(&f.perm_free[i], cudaEventDisableTiming));
  f.order.resize(p);
  for (int64_t j = 0; j < p; j++) f.order[j] = (int)j;

  if (f.family == Family::Blocked) {
    f.nblocks = (int)((p + kBlk - 1) / kBlk);
    PipePlan pl;
    if (!plan_pipe(h, s.model, ns, &pl)) return fail(BWGR_ERR_UNSUPPORTED, "the shape does not fit the pipelined blocked sweep");
    if (dist) {
      // the per-rank Gram bands are summed in float by ncclAllReduce: exact (= independent of the sharding) only below 2^24.
      // |G_jk| <= max_j xx_j (Cauchy-Schwarz) over ALL individuals; h_xx holds the all-reduced column statistics.
      if (!(h->xx_max < 16777216.0))
        return fail(BWGR_ERR_UNSUPPORTED, "row-sharded fit: max_j sum_i x_ij^2 = %.0f >= 2^24, the float sum of the per-GPU Gram bands would depend on the sharding", h->xx_max);
      // stale words of a previous fit (another nsys = another ring layout) must not be mistaken for this fit's: zero my ring,
      // then a collective as the barrier that no peer writes into it before it is clean
      CU(cudaMemsetAsync(h->hx_own.p, 0, sizeof(unsigned long long) * h->hx_own.n, h->stream));
      double one = 1;
      rc = dist_allreduce_host(h, &one, 1, false);
      if (rc) return rc;
    }
    f.rows_per_cta = pl.R; f.nworkers = pl.W; f.grid = pl.cl ? pl.nclusters * 8 : pl.W + 1; f.nbuf = pl.nbuf; f.sring = pl.sring; f.lookahead = pl.D; f.full_inv = pl.full_inv; f.nband = pl.D + 1;
    f.cl = pl.cl; f.nclusters = pl.nclusters;
    const size_t gram_n = (size_t)f.nblocks * kBlk * kBlk * f.nband;
    if (!s.shuffled) {  // natural order: one Gram band per genotype store, kept on the handle
      if (h->gram_nat_band != f.nband || h->gram_nat.n != gram_n) {
        h->gram_nat_band = 0;
        if (h->gram_nat.alloc(gram_n) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(Gram band) failed");
      } else {
        f.gram_cached = true;
      }
      f.gram_p = h->gram_nat.p;
    } else {
      if (f.gram.alloc(gram_n) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(Gram band) failed");
      f.gram_p = f.gram.p;
      // the clustered sweep occupies 8 x nclusters of the SMs: the next sweep's Gram band (a function of the marker order only)
      // is computed on the others meanwhile
      f.overlap = (h->world <= 1 || h->comm_side) && h->wait32 && h->x2f.p && f.nband == 2 &&
                  f.grid + 8 <= h->num_sms;  // at least a few SMs are left idle by the sweep
      if (f.overlap && f.gram2.alloc(gram_n) != cudaSuccess) { cudaGetLastError(); f.overlap = false; }
    }
    if (f.full_inv && f.tinv.alloc((size_t)f.nblocks * kBlk * kBlk) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(block inverses) failed");
    if (f.part.alloc((size_t)8 * ns * 128 * 161) != cudaSuccess || f.dew.alloc((size_t)f.nblocks * ns * 136) != cudaSuccess)
      return fail(BWGR_ERR_CUDA, "cudaMalloc(blocked workspace) failed");
    // clustered topology: two sets of the grid-sum words of h, used by alternate sweeps; each sweep zeroes the other set
    if (f.cl) {
      if (f.hsum.alloc((size_t)2 * f.nblocks * ns * 128 * kGridCopies) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(grid sums of h) failed");
      CU(cudaMemsetAsync(f.hsum.p, 0, sizeof(unsigned long long) * f.hsum.n, h->stream));
    }
    CU(cudaMemsetAsync(f.dew.p, 0, sizeof(unsigned long long) * f.dew.n, h->stream));
  }
  if (f.family == Family::Grid) {
    grid_geometry(h, &f.rows_per_cta, &f.grid);
    // unmasked systems: blocks of markers per grid sum, if the block ring fits next to the residual slabs (else one marker per sum)
    f.grid_blocked = !f.masked && s.model != M_KMUP2 &&
                     grid_block_smem(ns, f.rows_per_cta, h->storage == BWGR_STORE_F32, model_is_gibbs(s.model)) <= h->smem_optin;
    const size_t words = f.grid_blocked ? grid_block_acc_words(ns, (int)p) : (size_t)p * kGridCopies * 32;
    if (f.gridacc.alloc(words) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(grid accumulators) failed");
  }
  h->fit = std::move(fit);
  return 0;
}

// Fixed-point quantum of g = x'e: a power of two such that 64 x the Cauchy-Schwarz bound stays below 2^50.
static void g_fixed_point(bwgr_handle* h, const Fit& f, float* quantum, float* limit) {
  const double xxmax = std::max(1.0, h->xx_max);
  double yy = 0;
  for (size_t t = 0; t < f.vy.size(); t++) yy = std::max(yy, (double)f.vy[t] * (double)(h->n - 1));
  const double bound = 64.0 * (f.weighted ? 256.0 : 1.0) * std::sqrt(xxmax * std::max(yy, 1e-30));  // row multiplicities <= 255
  int ex;
  std::frexp(bound, &ex);
  *quantum = (float)std::ldexp(1.0, ex - 50);
  *limit = (float)std::ldexp(1.0, ex);
}

// The fit's state as the sweep kernels and the epilogue take it.  The rule divides by the per-system xx of masked systems, else by
// the caller's (KMUP) or the centred (MRR3) xx when the fit has one, else by the store's; the blocked family never has masked
// systems.  Only the KMUP2 rule reads xx2.
static SweepState sweep_state(const bwgr_handle* h) {
  const Fit& f = *h->fit;
  SweepState s;
  s.g = h->view(); s.nsys = f.nsys;
  s.e = f.e.p; s.b = f.b.p; s.d = f.d.p; s.vbv = f.vbv.p;
  s.xx = f.masked ? f.xx_sys.p : (f.xx_over.p ? f.xx_over.p : h->xx_f.p); s.xx_per_sys = f.masked ? 1 : 0;
  s.xx2 = f.model == M_KMUP2 ? f.xx_over.p : nullptr;
  s.mask = f.mask.p; s.sc = f.sc.p;
  s.seed_lo = (uint32_t)f.seed; s.seed_hi = (uint32_t)(f.seed >> 32); s.chain0 = f.chain0;
  s.err = h->err.p;
  return s;
}

// Row-sharded fit: the uncentred Gram band of this rank's rows -> the band over all individuals (exact: integers below 2^24 in
// fp32), centred afterwards when the fit's columns are (MRR3), with the same arithmetic as one GPU's Gram kernel.
static int sum_gram_band(bwgr_handle* h, float* gram, const int* perm, ncclComm_t comm, cudaStream_t st) {
  const Fit& f = *h->fit;
  NC(nccl().AllReduce(gram, gram, (size_t)f.nblocks * kBlk * kBlk * f.nband, ncclFloat, ncclSum, comm, st));
  if (f.sx_dev.p) {
    launch_gram_centre(gram, perm, (int)h->p, f.nblocks, f.nband, f.sx_dev.p, 1.0f / (float)h->n_global, st);
    h->launches++;
  }
  return 0;
}

int fit_sweeps(bwgr_handle* h, int nsweeps) {
  if (!h || !h->fit) return fail(BWGR_ERR_STATE, "no fit in progress");
  Fit& f = *h->fit;
  CU(cudaSetDevice(h->device));
  const int64_t p = h->p;
  const SweepState state = sweep_state(h);
  float quantum = 1, limit = 1;
  if (f.family == Family::Grid) g_fixed_point(h, f, &quantum, &limit);
  for (int k = 0; k < nsweeps; k++) {
    const int sweep = f.sweeps_issued;
    const int slot = sweep % kPermRing;
    const int* d_perm = nullptr;
    // the marker order of sweep `sw` (cumulative shuffles, Rcpp20260726ai.cpp:329-331) goes up on stream `st`
    auto upload_order = [&](int sw, cudaStream_t st) -> cudaError_t {
      const int sl = sw % kPermRing;
      if (cudaError_t e = cudaEventSynchronize(f.perm_free[sl])) return e;  // returns at once before the slot's first use
      int* hp = f.h_perm + (size_t)sl * p;
      if (f.shuffled) std::shuffle(f.order.begin(), f.order.end(), std::mt19937(sw));
      memcpy(hp, f.order.data(), sizeof(int) * p);
      return cudaMemcpyAsync(f.perm.p + (size_t)sl * p, hp, sizeof(int) * p, cudaMemcpyHostToDevice, st);
    };
    const bool ahead = f.overlap && f.gram_ahead == sweep;  // order and Gram band of this sweep were issued on the side stream
    if (f.overlap) f.gram_p = (sweep & 1) ? f.gram2.p : f.gram.p;
    if (!ahead && (f.shuffled || (f.family == Family::Blocked && f.sweeps_issued == 0)))  // natural order: the identity is uploaded once (slot 0)
      CU(upload_order(sweep, h->stream));
    if (f.shuffled) d_perm = f.perm.p + (size_t)slot * p;
    else if (f.family == Family::Blocked) d_perm = f.perm.p;  // identity order, uploaded once (slot 0)
    if (model_has_cnv(f.model)) CU(cudaMemcpyAsync(f.b_prev.p, f.b.p, sizeof(float) * f.nsys * p, cudaMemcpyDeviceToDevice, h->stream));
    if (f.family == Family::Blocked) {
      if (ahead) {
        CU(cudaStreamWaitEvent(h->stream, h->side_done[sweep & 1], 0));
      } else if (f.shuffled || !f.gram_cached) {
        cudaEvent_t pe = h->prof_begin(0);
        // row shards: each rank's band is uncentred (integers below 2^24 in fp32, so the float all-reduce is exact) and is
        // centred once the sum is complete
        const float* sx_in_kernel = h->world > 1 ? nullptr : f.sx_dev.p;
        if (h->x2f.p && f.nband == 2) {
          const cudaError_t ge = launch_gram_fp4(h->x2f.p, h->ld, (int)h->p, (int)h->n_global, d_perm, f.nblocks, f.gram_p, h->err.p, h->num_sms, sx_in_kernel, h->stream);
          if (ge != cudaSuccess) return fail(BWGR_ERR_CUDA, "FP4 Gram launch failed: %s", cudaGetErrorString(ge));
        } else launch_gram_tc(h->gram_view(), d_perm, f.nblocks, f.gram_p, 1, f.nband, h->fp8_codes, h->err.p, h->num_sms, sx_in_kernel, h->stream);
        h->prof_end(pe);
        h->launches++;
        f.gram_cached = true;
        if (!f.shuffled && f.gram_p == h->gram_nat.p) h->gram_nat_band = f.nband;
        if (h->world > 1) {
          int rc = sum_gram_band(h, f.gram_p, d_perm, h->comm, h->stream);
          if (rc) return rc;
        }
      }
      if (f.full_inv) {  // the step coefficients change every sweep (lambda), the inverses with them
        cudaEvent_t pi = h->prof_begin(3);
        launch_block_inverse(f.model, d_perm, (int)p, f.nblocks, f.gram_p, f.nband, state.xx, state.vbv, state.sc, f.tinv.p, h->stream);
        h->prof_end(pi);
        h->launches++;
      }
      if (!f.cl) CU(cudaMemsetAsync(f.part.p, 0, sizeof(unsigned long long) * f.part.n, h->stream));
      PipeArgs a;
      memset(&a, 0, sizeof a);
      a.s = state; a.model = rule_model(f.model); a.perm = d_perm; a.nblocks = f.nblocks; a.gram = f.gram_p; a.nband = f.nband; a.tinv = f.full_inv ? f.tinv.p : nullptr;
      a.sx = f.sx_dev.p; a.cshift = f.cshift.p; a.n_total = (int)h->n_global;
      a.part = f.part.p; a.hred = f.part.p + (size_t)8 * f.nsys * 128 * 160; a.dew = f.dew.p; a.tag = ++f.tag;
      a.rows_per_cta = f.rows_per_cta; a.nworkers = f.nworkers; a.D = f.lookahead; a.nbuf = f.nbuf; a.sring = f.sring;
      a.world = h->world; a.rank = h->rank; a.gen0 = h->dist_gen;
      a.cl = f.cl; a.nclusters = f.nclusters;
      if (f.cl) {
        const size_t set = f.hsum.n / 2;
        a.hsum = f.hsum.p + (sweep & 1) * set; a.hsum_next = f.hsum.p + ((sweep + 1) & 1) * set;
      }
      for (int r = 0; r < 8; r++) a.hx[r] = h->hx[r];
      if (h->world > 1) h->dist_gen += (unsigned long long)f.nblocks;
      if (getenv("BWGR_TRACE")) {
        const size_t tn = (size_t)f.grid * f.nblocks * 32;
        if (f.trace.n != tn) { f.trace.alloc(tn); cudaMemsetAsync(f.trace.p, 0, sizeof(long long) * f.trace.n, h->stream); }
        a.trace = f.trace.p;
      }
      if (f.overlap) { a.started = h->started.p; a.started_val = ++h->started_seq; }
      cudaEvent_t pe = h->prof_begin(1);
      const cudaError_t le = launch_sweep_pipe(a, h->stream);
      h->prof_end(pe);
      if (le != cudaSuccess) return fail(BWGR_ERR_CUDA, "pipelined sweep launch failed: %s", cudaGetErrorString(le));
      h->launches++;
      if (f.overlap) {
        // the flag is also set when the sweep has drained, whatever happened inside it: the side stream never waits forever
        const CUdeviceptr flag = reinterpret_cast<CUdeviceptr>(h->started.p);
        if (h->write32(h->stream, flag, a.started_val, 0) != CUDA_SUCCESS) return fail(BWGR_ERR_CUDA, "cuStreamWriteValue32 failed");
        const bool more = k + 1 < nsweeps || sweep + 1 < f.it_target;
        if (more && !h->profiling) {  // sweep + 1: order + Gram band on the SMs this sweep leaves idle, as soon as it is resident
          if (h->wait32(h->side, flag, a.started_val, CU_STREAM_WAIT_VALUE_GEQ) != CUDA_SUCCESS) return fail(BWGR_ERR_CUDA, "cuStreamWaitValue32 failed");
          CU(upload_order(sweep + 1, h->side));
          const int* np_ = f.perm.p + (size_t)((sweep + 1) % kPermRing) * p;
          float* gn = ((sweep + 1) & 1) ? f.gram2.p : f.gram.p;
          const cudaError_t ge = launch_gram_fp4(h->x2f.p, h->ld, (int)h->p, (int)h->n_global, np_, f.nblocks, gn, h->err.p, h->num_sms,
                                                 h->world > 1 ? nullptr : f.sx_dev.p, h->side, true);
          if (ge != cudaSuccess) return fail(BWGR_ERR_CUDA, "FP4 Gram launch failed: %s", cudaGetErrorString(ge));
          if (h->world > 1) {  // row shards: its own communicator, so it never queues behind (or ahead of) the main stream's
            int rc = sum_gram_band(h, gn, np_, h->comm_side, h->side);
            if (rc) return rc;
          }
          CU(cudaEventRecord(h->side_done[(sweep + 1) & 1], h->side));
          f.gram_ahead = sweep + 1;
          h->launches++;
        }
      }
    } else if (f.family == Family::Grid) {
      GridArgs a;
      memset(&a, 0, sizeof a);
      a.s = state; a.model = f.model; a.perm = d_perm;
      a.s.mask = f.weighted ? f.cnt.p : f.mask.p;  // row multiplicities ride in the mask bytes (they weigh the dot products only)
      a.blocked = f.grid_blocked ? 1 : 0;
      {  // cross products are bounded by max_j x_j'x_j (Cauchy-Schwarz): one unit = 1 (exact integers) unless that exceeds 2^50
        int ex = 0;
        std::frexp(std::max(1.0, h->xx_max), &ex);
        a.gram_quantum = h->storage == BWGR_STORE_F32 ? (float)std::ldexp(1.0, ex - 50) : (float)std::ldexp(1.0, std::max(0, ex - 50));
      }
      a.acc = f.gridacc.p; a.g_quantum = quantum; a.rows_per_cta = f.rows_per_cta;
      CU(cudaMemsetAsync(f.gridacc.p, 0, sizeof(unsigned long long) * f.gridacc.n, h->stream));
      cudaEvent_t pe = h->prof_begin(1);
      const cudaError_t le = launch_grid_sweep(a, f.grid, h->stream);
      h->prof_end(pe);
      if (le != cudaSuccess) return fail(BWGR_ERR_CUDA, "grid sweep launch failed: %s", cudaGetErrorString(le));
      h->launches++;
    } else {
      SmallNArgs a;
      memset(&a, 0, sizeof a);
      a.s = state; a.model = rule_model(f.model); a.perms = d_perm; a.row_w = f.weighted ? f.row_w.p : nullptr;
      cudaEvent_t pe = h->prof_begin(1);
      const cudaError_t le = launch_small_n(a, h->smem_optin, h->stream);
      h->prof_end(pe);
      if (le != cudaSuccess) return fail(BWGR_ERR_CUDA, "small-n sweep launch failed: %s", cudaGetErrorString(le));
      h->launches++;
    }
    if (f.shuffled) CU(cudaEventRecord(f.perm_free[slot], h->stream));
    if (f.wgr_mode) {
      cudaEvent_t pe2 = h->prof_begin(2);
      launch_wgr_step(f.wgr_args, h->num_sms, h->stream);
      h->prof_end(pe2);
      h->launches += 2;
    } else if (!f.skip_epilogue) {
      EpilogueArgs ea;
      memset(&ea, 0, sizeof ea);
      if (h->world > 1) {
        if (f.esum.n < (size_t)4 * f.nsys && (f.esum.alloc((size_t)4 * f.nsys) != cudaSuccess || f.emaxv.alloc(f.nsys) != cudaSuccess))
          return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
      }
      ea.s = state; ea.model = f.model; ea.y = f.y.p; ea.b_prev = f.b_prev.p; ea.wts = f.wts.p;
      ea.B = f.B.p; ea.D = f.D.p; ea.VBv = f.VBv.p;
      cudaEvent_t pe2 = h->prof_begin(2);
      if (h->world > 1) {  // sums over individuals: per rank, then all-reduced; everything else is replicated
        launch_epilogue_partial(ea, f.esum.p, f.emaxv.p, h->stream);
        NC(nccl().AllReduce(f.esum.p, f.esum.p, (size_t)4 * f.nsys, ncclDouble, ncclSum, h->comm, h->stream));
        NC(nccl().AllReduce(f.emaxv.p, f.emaxv.p, (size_t)f.nsys, ncclFloat, ncclMax, h->comm, h->stream));
        ea.esum = f.esum.p; ea.emaxv = f.emaxv.p;
        h->launches++;
      }
      launch_epilogue(ea, h->stream);
      h->prof_end(pe2);
      h->launches++;
    }
    f.sweeps_issued++;
    cudaError_t le = cudaGetLastError();
    if (le != cudaSuccess) return fail(BWGR_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(le));
  }
  return 0;
}

// fit_sweeps until every system has met its stopping rule (checked on the device each sweep) or it_target sweeps are issued, polling
// in batches to keep the host off the path.  sc: the systems' scalars as last read.
int fit_sweeps_until_done(bwgr_handle* h, std::vector<SysScalars>& sc) {
  Fit& f = *h->fit;
  sc.resize(f.nsys);
  for (int done_all = 0; f.sweeps_issued < f.it_target && !done_all;) {
    if (int rc = fit_sweeps(h, std::min(4, f.it_target - f.sweeps_issued))) return rc;
    CU(cudaMemcpyAsync(sc.data(), f.sc.p, sizeof(SysScalars) * f.nsys, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    done_all = 1;
    for (auto& c : sc) done_all &= c.done;
  }
  return 0;
}

constexpr int kHatSplits = 64;           // column splits of the fitted values (they fix each row's summation order)
constexpr size_t kHatWorkBytes = 512u << 20;  // bound of the partial sums [k][splits][ld] of one launch of the fitted values

// hat[t] = mu[t] + X b_t for the k systems of b [k][p] into hat [k][ld] (device buffers): one launch per group of systems whose partial
// sums fit kHatWorkBytes (all k at once up to n ~ 10^5 for k = 16)
int fit_hat(bwgr_handle* h, int k, const float* b_dev, const float* mu_dev, float* hat_dev) {
  const size_t per_sys = (size_t)kHatSplits * h->ld;
  int per = (int)std::max<size_t>(1, std::min<size_t>((size_t)k, kHatWorkBytes / (per_sys * sizeof(float))));
  if (per < k && per >= kHatChunk) per -= per % kHatChunk;
  if (h->hat_work.n < (size_t)per * per_sys && h->hat_work.alloc((size_t)per * per_sys) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  for (int t0 = 0; t0 < k; t0 += per) {
    const int kc = std::min(per, k - t0);
    launch_gemv_hat(h->view(), b_dev + (size_t)t0 * h->p, kc, mu_dev + t0, hat_dev + (size_t)t0 * h->ld, h->hat_work.p, kHatSplits, h->stream);
    h->launches += 2;
  }
  return 0;
}

// Fitted values of nsys systems read back to the host: hat[t * n + i] = mu[t] + x_i'b_t.  b: nsys x p floats, on the device or, with
// b_on_host, on the host.
int fitted_values(bwgr_handle* h, int nsys, const float* b, bool b_on_host, const float* mu, std::vector<float>& hat) {
  const int64_t n = h->n, p = h->p, ld = h->ld;
  DevBuf<float> bdev, mudev, hatd;
  if ((b_on_host && bdev.alloc((size_t)nsys * p) != cudaSuccess) || mudev.alloc(nsys) != cudaSuccess || hatd.alloc((size_t)nsys * ld) != cudaSuccess)
    return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  if (b_on_host) CU(cudaMemcpyAsync(bdev.p, b, sizeof(float) * nsys * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(mudev.p, mu, sizeof(float) * nsys, cudaMemcpyHostToDevice, h->stream));
  const int rc = fit_hat(h, nsys, b_on_host ? bdev.p : b, mudev.p, hatd.p);
  if (rc) return rc;
  hat.resize((size_t)nsys * n);
  CU(cudaMemcpy2DAsync(hat.data(), sizeof(float) * n, hatd.p, sizeof(float) * ld, sizeof(float) * n, nsys, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

// debug (BWGR_TRACE=file): header {CTAs, blocks, 32, look-ahead D}, then the raw int64 stamps of the last sweep, [cta][block][32]
void dump_trace(bwgr_handle* h) {
  const Fit& f = *h->fit;
  if (!f.trace.p || !getenv("BWGR_TRACE")) return;
  cudaStreamSynchronize(h->stream);
  std::vector<long long> tr(f.trace.n);
  cudaMemcpy(tr.data(), f.trace.p, tr.size() * sizeof(long long), cudaMemcpyDeviceToHost);
  if (FILE* fp = fopen(getenv("BWGR_TRACE"), "wb")) {
    const long long hdr[4] = {f.grid, f.nblocks, 32, f.lookahead};
    fwrite(hdr, sizeof(long long), 4, fp);
    fwrite(tr.data(), sizeof(long long), tr.size(), fp);
    fclose(fp);
  }
}

Fit::~Fit() {
  // an order upload for a sweep that never ran (an EM fit stopped early) may still be reading h_perm on the side stream
  cudaStreamSynchronize(h->stream);
  if (h->side) cudaStreamSynchronize(h->side);
  pinned_free(h_perm, h_perm_bytes);
  for (cudaEvent_t ev : perm_free) if (ev) cudaEventDestroy(ev);
}

}  // namespace bwgr::host
