// epilogue.cu -- per-sweep reductions and hyper-parameter updates (K9 of SURVEY 2c), one CTA per system.
//
// Restates, in the reference's float arithmetic, the block that follows the marker loop in every solver:
//   emRR  Rcpp20260726ai.cpp:338-343   emBA :113-117   emBB :171-175   emBC :229-234
//   emBL  :389-391                     emEN :440-450
//   emDE  :288-298   emML :498-506   emBCpi :1529-1538   lasso :1487-1492
//   BayesRR :839-844   BayesA :620-624   BayesB :683-687   BayesC :743-748
//   BayesL :795-800   BayesCpi :900-908   BayesDpi :966-970
// Sums over rows / markers are accumulated in double and rounded once (the reference sums in float
// packets; both are within float reassociation noise of each other).
#include <cooperative_groups.h>

#include "kernels.h"

namespace bwgr {

namespace {

__device__ double block_sum(double v, double* sh) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : 0.0;
  if (threadIdx.x < 32) r = warp_sum(r);
  __syncthreads();
  if (threadIdx.x == 0) sh[0] = r;
  __syncthreads();
  return sh[0];
}

// A cluster of kEpiCl CTAs per system: one CTA alone spends ~100 k cycles on the double-precision sums over n rows and p markers
// (ncu: a single SM busy for 52 us at 50k x 50k); the partial sums meet in CTA 0 through distributed shared memory, in rank order.
constexpr int kEpiCl = 8;

__global__ void __cluster_dims__(kEpiCl, 1, 1) __launch_bounds__(1024) epilogue_kernel(EpilogueArgs a) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  __shared__ double sh[32];
  __shared__ double part[kEpiCl][8];
  __shared__ float s_eM, s_ve, s_cxx, s_lmb;
  __shared__ int s_acc;
  const int cr = (int)cluster.block_rank();
  const int sys = blockIdx.x / kEpiCl, tid = threadIdx.x, T = blockDim.x * kEpiCl, gt = cr * (int)blockDim.x + tid;
  SysScalars* scp = a.s.sc + sys;
  if (scp->done) return;
  float* e = a.s.e + (size_t)sys * a.s.g.ld;
  const float* y = a.y + (size_t)sys * a.s.g.ld;
  float* b = a.s.b + (size_t)sys * a.s.g.p;
  const float* d = a.s.d ? a.s.d + (size_t)sys * a.s.g.p : nullptr;
  float* vbv = a.s.vbv ? a.s.vbv + (size_t)sys * a.s.g.p : nullptr;
  const uint8_t* mask = a.s.mask ? a.s.mask + (size_t)sys * a.s.g.ld : nullptr;
  const int model = a.model;

  double se = 0, see = 0, sey = 0, sy = 0;
  float emax = 0.0f;
  if (!a.esum)  // row-sharded fit: the sums over individuals were taken per rank and all-reduced (a.esum)
    for (int i0 = gt; i0 < a.s.g.n; i0 += 8 * T) {  // one CTA walks the vector: eight loads in flight per thread, or latency is all there is
      float ev[8], yv[8];
#pragma unroll
      for (int u = 0; u < 8; u++) {
        const int i = i0 + u * T;
        const bool ok = i < a.s.g.n && (!mask || mask[i]);
        ev[u] = ok ? e[i] : 0.0f;
        yv[u] = ok ? y[i] : 0.0f;
      }
#pragma unroll
      for (int u = 0; u < 8; u++) {
        const double ed = ev[u], yd = yv[u];
        se += ed; see += ed * ed; sey += ed * yd; sy += yd;
        emax = fmaxf(emax, fabsf(ev[u]));
      }
    }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) emax = fmaxf(emax, __shfl_xor_sync(0xffffffffu, emax, o));
  __shared__ float sh_max[32];
  if ((tid & 31) == 0) sh_max[tid >> 5] = emax;
  __syncthreads();
  emax = 0.0f;
  for (int w = 0; w < (int)(blockDim.x >> 5); w++) emax = fmaxf(emax, sh_max[w]);
  double sbb = 0, sd = 0, scnv = 0;
  for (int j0 = gt; j0 < a.s.g.p; j0 += 8 * T) {
    float bv[8], dv[8], pv[8];
#pragma unroll
    for (int u = 0; u < 8; u++) {
      const int j = j0 + u * T;
      const bool ok = j < a.s.g.p;
      bv[u] = ok ? b[j] : 0.0f;
      dv[u] = (ok && d) ? d[j] : 0.0f;
      pv[u] = (ok && a.b_prev) ? a.b_prev[(size_t)sys * a.s.g.p + j] : bv[u];
    }
#pragma unroll
    for (int u = 0; u < 8; u++) {
      const double bj = bv[u];
      sbb += bj * bj;
      sd += (double)dv[u];
      scnv += fabs((double)pv[u] - bj);
    }
  }
  se = block_sum(se, sh); see = block_sum(see, sh); sey = block_sum(sey, sh); sy = block_sum(sy, sh);
  sbb = block_sum(sbb, sh); sd = block_sum(sd, sh); scnv = block_sum(scnv, sh);
  if (tid == 0) {  // this CTA's sums into CTA 0's table
    double* dst = cluster.map_shared_rank(&part[0][0], 0) + cr * 8;
    dst[0] = se; dst[1] = see; dst[2] = sey; dst[3] = sy; dst[4] = sbb; dst[5] = sd; dst[6] = scnv; dst[7] = (double)emax;
  }
  cluster.sync();
  if (cr == 0 && tid == 0) {
    se = see = sey = sy = sbb = sd = scnv = 0.0; emax = 0.0f;
    for (int c = 0; c < kEpiCl; c++) {
      se += part[c][0]; see += part[c][1]; sey += part[c][2]; sy += part[c][3]; sbb += part[c][4]; sd += part[c][5]; scnv += part[c][6];
      emax = fmaxf(emax, (float)part[c][7]);
    }
  }
  if (a.esum) {
    se = a.esum[4 * sys + 0]; see = a.esum[4 * sys + 1]; sey = a.esum[4 * sys + 2]; sy = a.esum[4 * sys + 3];
    emax = a.emaxv[sys];
  }

  if (cr == 0 && tid == 0) {
    SysScalars s = *scp;
    const float n = s.n_eff, p = (float)a.s.g.p;
    const float ee = (float)see, bb = (float)sbb;
    float eM = (float)(se / (double)n);
    int accumulate = 0;
    if (!model_is_gibbs(model)) {
      switch (model) {
        case M_EMRR:
          s.vb = (bb + s.Sb) / (p + s.df);
          s.ve = (ee + s.Se) / (n + s.df);
          s.lmb = sqrtf(s.Rho * s.ve / s.vb);
          break;
        case M_EMBA:
        case M_EMBB:
          s.ve = (ee + s.Se) / (n + s.df);
          break;
        case M_EMBC:
          s.ve = (ee + s.Se) / (n + s.df);
          s.vb = (bb + s.Sa) / (p + s.df) / ((float)(sd / (double)a.s.g.p) - s.Pi);
          s.lmb = s.ve / s.vb;
          break;
        case M_EMEN: {
          const float ey = (float)(sey - (double)eM * sy);  // e (after mean removal) . y
          s.ve = ey / (n - 1.0f);
          s.vb = (bb + s.trAC22 * s.ve) / p;
          const float L = s.ve / s.vb;
          s.lmb = L;
          s.lmb1 = 0.5f * L * s.alpha * s.Sy;
          s.lmb2 = L * (1.0f - s.alpha);
          s.cnv = (float)scnv;
          if (s.cnv < 10e-11f) s.done = 1;
          break;
        }
        case M_EMDE: {  // :288-298 ; the per-marker penalties follow below, once Ve is known to every thread
          const float ey = (float)(sey - (double)eM * sy);
          s.ve = ey / (n - 1.0f);
          s.cnv = (float)scnv;
          if (s.cnv < 10e-6f) s.done = 1;
          break;
        }
        case M_EMMLD:
        case M_EMML: {  // :498-506 ; (y-mu)'e and (y-mu)'(y-mu) with the updated mu and the centred e, from the running sums
          const double mu1 = (double)s.mu + (double)eM;
          const double yce = sey - (double)eM * sy;
          const double syy = ((double)n - 1.0) * (double)s.vy + sy * sy / (double)n;
          const double ycyc = syy - 2.0 * mu1 * sy + (double)n * mu1 * mu1;
          s.ve = (float)(yce / (double)n);
          s.vb = (float)((ycyc - yce) / ((double)n * (double)s.MSx));
          s.lmb = s.ve / s.vb;
          s.cnv = (float)scnv;
          if (s.cnv < 10e-8f) s.done = 1;
          break;
        }
        case M_EMBCPI: {  // :1529-1536 ; pi_mix = the prior Pi, cxx = sum of the marker variances
          const float dm = (float)(sd / (double)a.s.g.p);
          s.Pi = ((1.0f - dm) * p + s.pi_mix * s.df) / (p + s.df);
          s.Pi0 = (1.0f - s.Pi) / s.Pi;
          s.MSx = s.cxx * s.Pi * (1.0f - s.Pi);
          s.Sa = s.R2 * (s.df + 2.0f) * s.vy / s.MSx;
          s.ve = (ee + s.Se) / (n + s.df);
          s.vb = (bb + s.Sa) / (p + s.df) / (dm - s.Pi);
          s.lmb = s.ve / s.vb;
          break;
        }
        case M_LASSO: {  // :1487-1492 ; d_j = |x_j'e~| - |b_j xx_j| was left by the rule
          const float tmp = 2.0f * (float)sd / p;
          s.lmb = 2.0f * sqrtf(fabsf(tmp));
          s.ve = (float)(sey - (double)eM * sy) / (n - 1.0f);  // for h2 = 1 - (e'y/(n-1))/var(y) (:1494)
          s.cnv = (float)scnv;
          if (s.cnv < 10e-8f) s.done = 1;
          break;
        }
        case M_GSRR:
        case M_GSFLM: {  // :1586-1590, :1618-1624 ; the y slot holds e0 (the residual as passed in); cxx = phi
          s.ve = (float)(sey - (double)eM * sy) / n;  // vna = e . e0 / n, e after the mean removal
          if (model == M_GSRR) { s.vb = (s.vy - s.ve) / s.cxx; s.lmb = s.ve / s.vb; }
          s.cnv = (float)scnv;
          if (s.cnv < 10e-8f) s.done = 1;
          break;
        }
        default: break;  // emBL, M_MRR: mean removal only (M_MRR: none, see below)
      }
      s.C = -0.5f / sqrtf(s.ve);
      if (model == M_MRR) eM = 0.0f;
      s.its += 1;
    } else {
      // Gibbs: intercept draw, then variances (counter = (0xFFFFFFFF, sweep, chain, purpose))
      const uint32_t chain = (uint32_t)(a.s.chain0 + sys), sw = (uint32_t)s.sweep;
      uint32_t c[4] = {0xFFFFFFFFu, sw, chain, 0u};
      philox4x32_10(c, a.s.seed_lo, a.s.seed_hi);
      float z, z2;
      box_muller(c[0], c[1], z, z2);
      eM = eM + sqrtf(s.ve / n) * z;
      const float ee2 = (float)(see - 2.0 * (double)eM * se + (double)n * (double)eM * (double)eM);
      const float chi_e = rchisq_philox(n + s.df, 0xFFFFFFFFu, sw, chain, 1u, a.s.seed_lo, a.s.seed_hi);
      if (model == M_BRR || model == M_BC || model == M_BCPI) {
        const float chi_b = rchisq_philox(p + s.df, 0xFFFFFFFFu, sw, chain, 2u, a.s.seed_lo, a.s.seed_hi);
        s.ve = (ee2 + s.Se) / chi_e;
        s.vb = (bb + s.Sb) / chi_b;
        s.lmb = s.ve / s.vb;
        if (model == M_BCPI) {  // :906-907 ; the mixing odds Pi0 stay as they were
          s.Pi = (float)(sd / (double)a.s.g.p);
          s.Sb = s.df * s.R2 * s.vy / s.MSx / (1.0f - s.Pi);
        }
      } else {
        s.ve = (ee2 + s.Se) / chi_e;
        if (model == M_BDPI) s.Pi = (float)(sd / (double)a.s.g.p);  // :969
      }
      s.C = -0.5f / sqrtf(s.ve);
      if (s.sweep > s.burn) {  // sic: i > bi, divided later by it-bi (:624-627)
        accumulate = 1;
        s.MU += (double)(s.mu + eM); s.VE += (double)s.ve; s.VB += (double)s.vb; s.PI += (double)s.Pi;
        s.post_count += 1;
      }
    }
    s.mu += eM;
    s.sweep += 1;
    set_e_scale(s, emax + fabsf(eM));
    *scp = s;
    s_eM = eM;
    s_acc = accumulate;
    s_ve = s.ve; s_cxx = s.cxx; s_lmb = s.lmb;
  }
  cluster.sync();
  if (cr != 0 && tid == 0) {  // the scalars every CTA needs for its share of the element-wise passes
    s_eM = *cluster.map_shared_rank(&s_eM, 0); s_acc = *cluster.map_shared_rank(&s_acc, 0);
    s_ve = *cluster.map_shared_rank(&s_ve, 0); s_cxx = *cluster.map_shared_rank(&s_cxx, 0); s_lmb = *cluster.map_shared_rank(&s_lmb, 0);
  }
  cluster.sync();  // CTA 0 stays until its shared memory has been read
  const float eM = s_eM;
  if (model == M_EMDE && vbv) {  // :293-296 ; Vb_j = b_j^2 + Ve/(xx_j + Lmb_j + 1e-4), Lmb_j = sqrt(cxx Ve / Vb_j)
    const float* xx = a.s.xx + (a.s.xx_per_sys ? (size_t)sys * a.s.g.p : 0);
    const float Ve = s_ve, cxx = s_cxx;
    for (int j = gt; j < a.s.g.p; j += T) {
      float xxj = xx[j];
      if (xxj == 0.0f) xxj = 0.1f;  // :261
      const float Vb = b[j] * b[j] + Ve / (xxj + vbv[j] + 0.0001f);
      vbv[j] = sqrtf(cxx * Ve / Vb);
    }
  }
  if (model == M_EMMLD && vbv && a.wts) {  // :495 ; the penalty of marker j is Lmb / d_j
    for (int j = gt; j < a.s.g.p; j += T) vbv[j] = s_lmb / a.wts[j];
  }
  if ((model == M_GSRR || model == M_GSFLM) && vbv) {  // the per-marker slot carries Lmb_j + 0.01 (the rule's denominator)
    const float* xx = a.s.xx + (a.s.xx_per_sys ? (size_t)sys * a.s.g.p : 0);
    const float vna = s_ve, phi = s_cxx;
    for (int j = gt; j < a.s.g.p; j += T) {
      if (model == M_GSRR) vbv[j] = s_lmb + 0.01f;  // :1621-1623
      else {                                        // :1588-1589 ; Vb_j = b_j^2 + vna/(xx_j + Lmb_j), Lmb_j = sqrt(phi vna / Vb_j)
        const float Vb = b[j] * b[j] + vna / (xx[j] + (vbv[j] - 0.01f));
        vbv[j] = sqrtf(phi * vna / Vb) + 0.01f;
      }
    }
  }
  if (eM != 0.0f)
    for (int i0 = gt; i0 < a.s.g.n; i0 += 8 * T) {
      float ev[8];
#pragma unroll
      for (int u = 0; u < 8; u++) { const int i = i0 + u * T; ev[u] = i < a.s.g.n ? e[i] : 0.0f; }
#pragma unroll
      for (int u = 0; u < 8; u++) { const int i = i0 + u * T; if (i < a.s.g.n && (!mask || mask[i])) e[i] = ev[u] - eM; }
    }
  if (s_acc && a.B) {
    float* B = a.B + (size_t)sys * a.s.g.p;
    for (int j = gt; j < a.s.g.p; j += T) B[j] += b[j];
    if (a.D && d) { float* D = a.D + (size_t)sys * a.s.g.p; for (int j = gt; j < a.s.g.p; j += T) D[j] += d[j]; }
    if (a.VBv && vbv) { float* V = a.VBv + (size_t)sys * a.s.g.p; for (int j = gt; j < a.s.g.p; j += T) V[j] += vbv[j]; }
  }
}

// ---- wgr(): the R-level MCMC step restated on the device (R/wgr.R:91-136, eigK = NULL, bag = 1) ----------------
// Kernel A (one CTA): e'e, b'b, mean(e) -> Va (pi/iv dependent), Ve, intercept draw; kernel B (grid): per-marker Vb, L = Ve/Vb,
// posterior sums, e -= mu0.  The residual the reference rebuilds each iteration (e = y - mu - X b, :124) is the one the sweep
// maintains, so it is not recomputed.
__global__ void __launch_bounds__(1024) wgr_scalars_kernel(WgrArgs a) {
  __shared__ double sh[32];
  __shared__ float sh_max[32];
  const int tid = threadIdx.x, T = blockDim.x;
  const int phase = a.phase;
  double se = 0, see = 0, sbb = 0;
  float emax = 0.0f;
  if (phase == 2) {  // bagged wgr: the residual is rebuilt from the fitted values every iteration (e = y - mu - X b, :124)
    for (int i = tid; i < a.n; i += T) { const float ef = a.y[i] - a.hat[i]; a.e[i] = ef; se += (double)ef; emax = fmaxf(emax, fabsf(ef)); }
  } else {
    for (int i = tid; i < a.n; i += T) {
      // KMUP2 returns the residuals of the rows in use only (:76): crossprod(e) is theirs, a row drawn c times (rp = TRUE) enters c
      // times (the mask byte is 0/1, or the multiplicity)
      const double wv = phase == 1 ? (double)a.mask[i] : 1.0;
      if (wv == 0.0) continue;
      const double ev = a.e[i];
      se += wv * ev; see += wv * ev * ev; emax = fmaxf(emax, fabsf(a.e[i]));
    }
    for (int j = tid; j < a.p; j += T) { const double bj = a.b[j]; sbb += bj * bj; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) emax = fmaxf(emax, __shfl_xor_sync(0xffffffffu, emax, o));
  if ((tid & 31) == 0) sh_max[tid >> 5] = emax;
  se = block_sum(se, sh); see = block_sum(see, sh); sbb = block_sum(sbb, sh);
  if (tid == 0) {
    emax = 0.0f;
    for (int w = 0; w < (T >> 5); w++) emax = fmaxf(emax, sh_max[w]);
    SysScalars s = *a.sc;
    WgrState w = *a.st;
    const uint32_t sw = (uint32_t)s.sweep;
    const int i = s.sweep + 1;  // R's 1-based iteration
    const float n = (float)a.n, p = (float)a.p;
    if (phase != 2) {
      w.Ve_old = s.ve;
      if (!a.iv) w.Va = ((float)sbb + a.Sb) / rchisq_philox(a.df + p, 0xFFFFFFFEu, sw, 0u, 2u, a.seed_lo, a.seed_hi);  // :113
      const float nres = phase == 1 ? a.nsub : n;                                                                       // n * bag (:121)
      w.Ve = ((float)see + a.Se) / rchisq_philox(nres + a.df, 0xFFFFFFFEu, sw, 0u, 1u, a.seed_lo, a.seed_hi);            // :121
    }
    if (phase != 1) {
      uint32_t c[4] = {0xFFFFFFFEu, sw, 0u, 0u};
      philox4x32_10(c, a.seed_lo, a.seed_hi);
      float z, z2;
      box_muller(c[0], c[1], z, z2);
      w.mu0 = (float)(se / (double)n) + (w.Ve / n) * z;  // sic: rnorm(1, mean(e), Ve/n), the sd argument is Ve/n (:125)
      s.mu += w.mu0;
      w.post = (i >= a.bi && i <= a.it && ((i - a.bi) % a.th) == 0) ? 1 : 0;
      if (w.post) { w.B0 += (double)s.mu; w.VE += (double)w.Ve; if (!a.iv) w.VA += (double)w.Va; w.post_count += 1; }
      s.ve = w.Ve;
      s.C = -0.5f / sqrtf(s.ve);
      s.sweep += 1;
      s.its += 1;
      set_e_scale(s, emax + fabsf(w.mu0));
      *a.sc = s;
    }
    *a.st = w;
  }
}

__global__ void __launch_bounds__(256) ll_to_float_kernel(const long long* __restrict__ src, float* __restrict__ dst, int n) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < n) dst[i] = (float)src[i];
}

__global__ void __launch_bounds__(256) wgr_markers_kernel(WgrArgs a) {
  const WgrState w = *a.st;
  const uint32_t sw = (uint32_t)(a.sc->sweep - 1);  // the sweep the scalar kernel just closed
  const int stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  for (int j = t0; j < a.p; j += stride) {
    const float bj = a.b[j];
    float Vb;
    if (a.iv) {
      if (a.de) Vb = sqrtf(bj * bj * w.Ve_old / a.MSx);                                                         // :97, :106
      else Vb = (a.Sb + bj * bj) / rchisq_philox(a.df + 1.0f, (uint32_t)j, sw, 0u, 3u, a.seed_lo, a.seed_hi);      // :100, :109
    } else {
      Vb = w.Va;
    }
    a.L[j] = w.Ve / Vb;                                                                                          // :122
    if (w.post) {
      a.B[j] += bj;
      a.D[j] += a.d[j];
      if (a.iv) a.VB[j] += Vb;
    }
  }
  if (w.mu0 != 0.0f)
    for (int i = t0; i < a.n; i += stride) a.e[i] -= w.mu0;
}

// Row-sharded fit: this rank's part of the sums over individuals, [nsys][4] doubles {sum e, sum e^2, sum e y, sum y} and
// max|e| per system; ncclAllReduce (sum / max) runs between this kernel and epilogue_kernel.
__global__ void __launch_bounds__(1024) epilogue_partial_kernel(EpilogueArgs a, double* out, float* emax_out) {
  __shared__ double sh[32];
  __shared__ float sh_max[32];
  const int sys = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
  const float* e = a.s.e + (size_t)sys * a.s.g.ld;
  const float* y = a.y + (size_t)sys * a.s.g.ld;
  double se = 0, see = 0, sey = 0, sy = 0;
  float emax = 0.0f;
  for (int i = tid; i < a.s.g.n; i += T) {
    const double ev = e[i], yv = y[i];
    se += ev; see += ev * ev; sey += ev * yv; sy += yv;
    emax = fmaxf(emax, fabsf(e[i]));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) emax = fmaxf(emax, __shfl_xor_sync(0xffffffffu, emax, o));
  if ((tid & 31) == 0) sh_max[tid >> 5] = emax;
  se = block_sum(se, sh); see = block_sum(see, sh); sey = block_sum(sey, sh); sy = block_sum(sy, sh);
  if (tid == 0) {
    emax = 0.0f;
    for (int w = 0; w < (T >> 5); w++) emax = fmaxf(emax, sh_max[w]);
    out[4 * sys + 0] = se; out[4 * sys + 1] = see; out[4 * sys + 2] = sey; out[4 * sys + 3] = sy;
    emax_out[sys] = emax;
  }
}

}  // namespace

void launch_epilogue_partial(const EpilogueArgs& a, double* out, float* emax_out, cudaStream_t st) {
  epilogue_partial_kernel<<<a.s.nsys, 1024, 0, st>>>(a, out, emax_out);
}

// bagged wgr: phase 1 (variances) before the fitted values are rebuilt, phase 2 (intercept, posterior sums, per-marker part) after
void launch_wgr_bag_phase(const WgrArgs& a, int phase, int num_sms, cudaStream_t st) {
  WgrArgs b = a;
  b.phase = phase;
  wgr_scalars_kernel<<<1, 1024, 0, st>>>(b);
  if (phase == 2) wgr_markers_kernel<<<num_sms, 256, 0, st>>>(b);
}

void launch_ll_to_float(const long long* src, float* dst, int n, cudaStream_t st) {
  ll_to_float_kernel<<<(n + 255) / 256, 256, 0, st>>>(src, dst, n);
}

void launch_wgr_step(const WgrArgs& a, int num_sms, cudaStream_t st) {
  wgr_scalars_kernel<<<1, 1024, 0, st>>>(a);
  wgr_markers_kernel<<<num_sms, 256, 0, st>>>(a);
}

void launch_epilogue(const EpilogueArgs& a, cudaStream_t st) { epilogue_kernel<<<a.s.nsys * kEpiCl, 1024, 0, st>>>(a); }

}  // namespace bwgr
