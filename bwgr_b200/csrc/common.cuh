// common.cuh -- shared device/host definitions of the B200 marker-effect update loop.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

namespace bwgr {

// Unified model ids used on the device (EM = bwgr_em_model, Gibbs = 10 + bwgr_gibbs_model).
enum Model : int {
  M_EMRR = 0, M_EMBA = 1, M_EMBB = 2, M_EMBC = 3, M_EMBL = 4, M_EMEN = 5,
  M_EMDE = 6, M_EMML = 7, M_EMBCPI = 8, M_LASSO = 9,  // the rest of emCV's panel (R/cv.R:13-22)
  M_BRR = 10, M_BA = 11, M_BB = 12, M_BC = 13, M_KMUP = 14, M_MRR = 15 /* rotated MRR3 trait: ridge, per-system lambda */,
  M_BL = 16, M_BCPI = 17, M_BDPI = 18,                 // the rest of mcmcCV's panel (R/cv.R:124-130)
  M_GSRR = 19, M_GSFLM = 20,                           // warm-start Gauss-Seidel solvers of mm() (Rcpp20260726ai.cpp:1564-1628)
  M_EMMLD = 21,                                        // emML with marker weights D: penalty Lmb / d_j (:495-496)
  M_KMUP2 = 22                                         // the bagged Kuo-Mallick sweep of wgr(bag != 1) (:41-77): row subset, (H'e0 + b0) numerator
};
// Several solvers share one per-marker rule and differ only in the sweep epilogue: the sweep kernels are instantiated per
// RULE, the epilogue and the host recipes see the full model.  emML :463 steps like emRR, emBCpi :1502 like emBC,
// BayesCpi :858 like BayesC (its mixing odds Pi0 are never refreshed, only the prior scale Sb follows the inclusion rate).
// GSRR / GSFLM :1583, :1615 step like emDE with the per-marker slot carrying Lmb_j + 0.01 (their denominator is Lmb_j + xx_j + 0.01).
__host__ __device__ constexpr int rule_model(int m) {
  // emML with weights steps like emDE too: the per-marker slot carries Lmb / d_j, refreshed by the epilogue after every sweep
  return m == M_EMML ? M_EMRR : m == M_EMBCPI ? M_EMBC : m == M_BCPI ? M_BC : (m == M_GSRR || m == M_GSFLM || m == M_EMMLD) ? M_EMDE : m;
}
// The one list of rules the sweep kernels are instantiated for: calls f(std::integral_constant<int, rule_model(m)>()), or nothing
// when m is not a model id.  A kernel family leaves out, with if constexpr on the constant, the rules it is never launched with.
template <class F>
void with_rule(int m, F&& f) {
  switch (rule_model(m)) {
    case M_EMRR: f(std::integral_constant<int, M_EMRR>()); break;
    case M_EMBA: f(std::integral_constant<int, M_EMBA>()); break;
    case M_EMBB: f(std::integral_constant<int, M_EMBB>()); break;
    case M_EMBC: f(std::integral_constant<int, M_EMBC>()); break;
    case M_EMBL: f(std::integral_constant<int, M_EMBL>()); break;
    case M_EMEN: f(std::integral_constant<int, M_EMEN>()); break;
    case M_EMDE: f(std::integral_constant<int, M_EMDE>()); break;
    case M_LASSO: f(std::integral_constant<int, M_LASSO>()); break;
    case M_BRR: f(std::integral_constant<int, M_BRR>()); break;
    case M_BA: f(std::integral_constant<int, M_BA>()); break;
    case M_BB: f(std::integral_constant<int, M_BB>()); break;
    case M_BC: f(std::integral_constant<int, M_BC>()); break;
    case M_KMUP: f(std::integral_constant<int, M_KMUP>()); break;
    case M_MRR: f(std::integral_constant<int, M_MRR>()); break;
    case M_BL: f(std::integral_constant<int, M_BL>()); break;
    case M_BDPI: f(std::integral_constant<int, M_BDPI>()); break;
    case M_KMUP2: f(std::integral_constant<int, M_KMUP2>()); break;
    default: break;
  }
}

// Per-system scalar state, device resident, updated by the sweep epilogue.
struct SysScalars {
  // hyper-parameters read by the marker rule
  float mu, ve, vb, lmb, lmb1, lmb2, C, Pi, Pi0, Sb, Se, Sa, df, cxx;
  // constants of the fit
  float R2, alpha, vy, MSx, Rho, trAC22, Sy, pi_mix;
  float n_eff;  // rows used by this system (row masks)
  // fixed-point scale of the residuals for the tensor-core passes: e = q * e_q, |q| <= 2^30 (power of two)
  float e_q, e_qinv;
  float cnv;    // emEN: sum |b_old - b_new| of the last sweep
  int its;      // sweeps done
  int done;     // emEN convergence reached
  int sweep;    // absolute sweep index (Gibbs: RNG counter)
  int burn, post_count;
  // posterior accumulators (Gibbs)
  double MU, VE, VB, PI;
};

// Fixed-point scale of the residuals for the next sweep, from bound >= max|e|: |e| may grow 8x before it saturates 2^30.
__host__ __device__ inline void set_e_scale(SysScalars& s, float bound) {
  int ex = 0;
  if (bound > 0.0f && bound < 3.0e38f) frexpf(bound, &ex);
  if (ex < -60) ex = -60;
  s.e_q = ldexpf(1.0f, ex + 3 - 30);
  s.e_qinv = ldexpf(1.0f, 30 - 3 - ex);
}

struct MarkerDraws {  // pre-generated per marker per sweep (Gibbs only)
  float z1, z2, u, chi;
};

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 counter-based RNG (Salmon et al. 2011). key = seed, counter = (marker, sweep,
// chain, purpose) so every draw is addressable and independent of the launch geometry.
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint64_t p0 = (uint64_t)M0 * c[0], p1 = (uint64_t)M1 * c[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1, n3 = (uint32_t)p0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += W0; k1 += W1;
  }
}
__host__ __device__ inline float u01(uint32_t x) {  // (0,1], 24 bits
  return ((x >> 8) + 1) * (1.0f / 16777216.0f);
}
__device__ inline void box_muller(uint32_t a, uint32_t b, float& z0, float& z1) {
  const float r = sqrtf(-2.0f * logf(u01(a)));
  float s, c;
  sincospif(2.0f * u01(b), &s, &c);
  z0 = r * c; z1 = r * s;
}
// chi-square(nu) = 2*Gamma(nu/2) by Marsaglia-Tsang (2000); attempts are separate Philox counters.
__device__ inline float rchisq_philox(float nu, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t purpose, uint32_t k0,
                                      uint32_t k1) {
  float a = 0.5f * nu;
  const bool boost = a < 1.0f;
  if (boost) a += 1.0f;
  const float d = a - (1.0f / 3.0f), cc = rsqrtf(9.0f * d);
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
    if (logf(u) < 0.5f * x * x + d - d * v + d * logf(v)) { out = d * v; break; }
  }
  if (boost) out *= powf(ub, 1.0f / (0.5f * nu));
  return 2.0f * out;
}
// Draws of one marker update: z1 (effect), z2 (excluded effect), u (inclusion), chi (df+1).
__device__ inline MarkerDraws marker_draws(int model, uint32_t marker, uint32_t sweep, uint32_t chain, float df,
                                           uint32_t k0, uint32_t k1) {
  MarkerDraws m;
  uint32_t c[4] = {marker, sweep, chain, 0u};
  philox4x32_10(c, k0, k1);
  box_muller(c[0], c[1], m.z1, m.z2);
  m.u = u01(c[2]);
  m.chi = 1.0f;
  if (model == M_BA || model == M_BB || model == M_BL || model == M_BDPI) m.chi = rchisq_philox(df + 1.0f, marker, sweep, chain, 1u, k0, k1);
  return m;
}

// ---------------------------------------------------------------------------------------------
// The per-marker update rule (SURVEY 8a). In: g = x_j'e, xx = ||x_j||^2, b0, per-marker variance
// vbj (BA/BB families) or per-marker lambda (KMUP). Out: new effect, residual step de
// (e -= x_j*de), inclusion d, new per-marker variance.
// The spike-slab likelihood ratio uses ||e2||^2-||e1||^2 = b1*(2g + xx*(2*b0-b1)) in closed form.
// ---------------------------------------------------------------------------------------------
struct RuleOut { float b, de, d, vbj; };

// The ridge penalty of marker j as the rule sees it.  vbj is the per-marker slot: a variance (emBA/emBB/BayesA/B/L/Dpi),
// or the penalty itself (KMUP's L[j], emDE's Lmb[j] :281).  BayesL :790-799: ve/vb_j in the first sweep, sqrt(Phi ve/vb_j) after.
template <int MODEL>
__device__ __forceinline__ float marker_lambda(float vbj, const SysScalars& s) {
  if constexpr (MODEL == M_EMBA || MODEL == M_EMBB || MODEL == M_BA || MODEL == M_BB || MODEL == M_BDPI) return s.ve * (1.0f / vbj);
  else if constexpr (MODEL == M_BL) return s.sweep == 0 ? s.ve * (1.0f / vbj) : sqrtf(s.Rho * s.ve / vbj);
  else if constexpr (MODEL == M_EMDE || MODEL == M_KMUP || MODEL == M_KMUP2) return vbj;
  else return s.lmb;
}

template <int MODEL>
__device__ __forceinline__ RuleOut marker_rule(float g, float xx, float b0, float vbj, const SysScalars& s,
                                               const MarkerDraws& dr, float xx2 = 0.0f) {
  RuleOut o;
  o.d = 1.0f; o.vbj = vbj;
  if constexpr (MODEL == M_EMRR || MODEL == M_MRR) {  // Rcpp20260726ai.cpp:335 ; MRR3 rotated system
    o.b = (g + xx * b0) / (xx + s.lmb);
    o.de = o.b - b0;
  } else if constexpr (MODEL == M_EMDE) {  // :281-283 (vbj carries Lmb[j]; the epilogue re-estimates it)
    o.b = (g + xx * b0) / (vbj + xx);
    o.de = o.b - b0;
  } else if constexpr (MODEL == M_LASSO) {  // :1478-1486 ; d carries |x'e~| - |b xx|, which the epilogue sums into the next penalty (:1487-1489)
    const float yx = g + xx * b0;
    float b1;
    if (yx > 0.0f) { b1 = (yx - s.lmb) / xx; if (b1 < 0.0f) b1 = 0.0f; }
    else           { b1 = (yx + s.lmb) / xx; if (b1 > 0.0f) b1 = 0.0f; }
    o.b = b1;
    o.d = fabsf(yx) - fabsf(b1 * xx);
    o.de = b1 - b0;
  } else if constexpr (MODEL == M_EMBA) {  // :107-111 (e updated twice)
    const float lmb = s.ve * (1.0f / vbj);
    const float b1 = (g + xx * b0) / (xx + lmb);
    o.b = b1;
    o.vbj = (s.Sb + b1 * b1) / (s.df + 1.0f);
    o.de = 2.0f * (b1 - b0);
  } else if constexpr (MODEL == M_EMBB || MODEL == M_EMBC) {  // :162-169, :221-227
    const float lmb = (MODEL == M_EMBB) ? s.ve * (1.0f / vbj) : s.lmb;
    const float b1 = (g + xx * b0) / (xx + lmb);
    const float LR = s.Pi0 * expf(s.C * (b1 * (2.0f * g + xx * (2.0f * b0 - b1))));
    o.d = 1.0f / (1.0f + LR);
    o.b = b1 * o.d;
    if (MODEL == M_EMBB) o.vbj = (s.Sb + o.b * o.b) / (s.df + 1.0f);
    o.de = o.b - b0;
  } else if constexpr (MODEL == M_EMBL) {  // :378-386
    const float OLS = g + xx * b0;
    const float Half = 0.5f * OLS / (xx + s.cxx);
    if (OLS > 0.0f) {
      const float G = 0.5f * (OLS - s.lmb1) / (s.lmb2 + xx);
      o.b = (G > 0.0f) ? G + Half : Half;
    } else {
      const float G = 0.5f * (OLS + s.lmb1) / (s.lmb2 + xx);
      o.b = (G < 0.0f) ? G + Half : Half;
    }
    o.de = o.b - b0;
  } else if constexpr (MODEL == M_EMEN) {  // :431-438
    const float OLS = g + xx * b0;
    float b1;
    if (OLS > 0.0f) { b1 = (OLS - s.lmb1) / (s.lmb2 + xx); if (b1 < 0.0f) b1 = 0.0f; }
    else            { b1 = (OLS + s.lmb1) / (s.lmb2 + xx); if (b1 > 0.0f) b1 = 0.0f; }
    o.b = b1;
    o.de = b1 - b0;
  } else if constexpr (MODEL == M_BRR || MODEL == M_BA || MODEL == M_BL) {  // :835, :615-618, :790-793
    const float lmb = marker_lambda<MODEL>(vbj, s);
    const float sd = sqrtf(s.ve / (xx + lmb));
    o.b = (g + xx * b0) / (xx + lmb) + sd * dr.z1;
    if (MODEL == M_BA || MODEL == M_BL) o.vbj = (s.Sb + o.b * o.b) / dr.chi;
    o.de = o.b - b0;
  } else if constexpr (MODEL == M_BDPI) {  // :949-964 ; accept b1 with probability min(1, (1-pi) exp(C(|e1|^2 - |e2|^2))), s.Pi = pi
    const float lmb = s.ve * (1.0f / vbj);
    const float sd = sqrtf(s.ve / (xx + lmb));
    const float b1 = (g + xx * b0) / (xx + lmb) + sd * dr.z1, b2 = sd * dr.z2;
    const float diff = (b2 - b1) * (-2.0f * g + xx * (b1 + b2 - 2.0f * b0));  // ||e2||^2-||e1||^2, e2 = e - x(b2-b0)
    float pj = (1.0f - s.Pi) * expf(-s.C * diff);
    if (pj > 1.0f) pj = 1.0f;
    if (dr.u < pj) { o.b = b1; o.d = 1.0f; } else { o.b = b2; o.d = 0.0f; }
    o.vbj = (s.Sb + o.b * o.b) / dr.chi;
    o.de = o.b - b0;
  } else if constexpr (MODEL == M_BB || MODEL == M_BC) {  // :670-681, :731-741
    const float lmb = (MODEL == M_BB) ? s.ve * (1.0f / vbj) : s.lmb;
    const float sd = sqrtf(s.ve / (xx + lmb));
    const float b1 = (g + xx * b0) / (xx + lmb) + sd * dr.z1;
    const float LR = s.Pi0 * expf(s.C * (b1 * (2.0f * g + xx * (2.0f * b0 - b1))));
    const float pj = 1.0f / (1.0f + LR);
    if (dr.u < pj) { o.b = b1; o.d = 1.0f; } else { o.b = sd * dr.z2; o.d = 0.0f; }
    if (MODEL == M_BB) o.vbj = (s.Sb + o.b * o.b) / dr.chi;
    o.de = o.b - b0;
  } else if constexpr (MODEL == M_KMUP) {  // :19-35 ; vbj carries L[j]
    const float sd = sqrtf(s.ve / (xx + vbj));
    const float b1 = (g + xx * b0) / (xx + vbj) + sd * dr.z1;
    if (s.pi_mix > 0.0f) {
      const float b2 = sd * dr.z2;
      const float diff = (b2 - b1) * (-2.0f * g + xx * (b1 + b2 - 2.0f * b0));  // ||e2||^2-||e1||^2
      const float pj = 1.0f / (1.0f + (s.pi_mix / (1.0f - s.pi_mix)) * expf(s.C * diff));
      if (dr.u < pj) { o.b = b1; o.d = 1.0f; } else { o.b = b2; o.d = 0.0f; }
    } else {
      o.b = b1; o.d = 1.0f;
    }
    o.de = o.b - b0;
  } else if constexpr (MODEL == M_KMUP2) {  // :60-74 ; g = H'e0 and xx = H'H over the rows in use, xx2 = the caller's xx(j) * bg, vbj = L[j]
    const float den = xx2 + vbj, sd = sqrtf(s.ve / den);
    const float b1 = (g + b0) / den + sd * dr.z1;  // sic: b0 enters without its xx (:60)
    if (s.pi_mix > 0.0f) {
      const float b2 = sd * dr.z2;
      const float diff = (b2 - b1) * (-2.0f * g + xx * (b1 + b2 - 2.0f * b0));  // ||e2||^2-||e1||^2 of the rows in use
      const float pj = 1.0f / (1.0f + (s.pi_mix / (1.0f - s.pi_mix)) * expf(s.C * diff));
      if (dr.u < pj) { o.b = b1; o.d = 1.0f; } else { o.b = b2; o.d = 0.0f; }
    } else {
      o.b = b1; o.d = 1.0f;
    }
    o.de = o.b - b0;
  }
  return o;
}

// Linear rules: the residual step of marker i is  de_i = a_i * g_i + c_i  with a_i, c_i independent of g
// (g_i = current x_i'e).  emRR :335, emBA :107-111 (de = 2*(b1-b0)), BayesRR :835, BayesA :615, rotated MRR3, emDE :281,
// emML :492, BayesL :790.
__host__ __device__ constexpr bool model_is_linear(int m) {
  return m == M_EMRR || m == M_EMBA || m == M_MRR || m == M_BRR || m == M_BA || m == M_EMDE || m == M_EMML || m == M_BL || m == M_GSRR ||
         m == M_GSFLM || m == M_EMMLD;
}
struct LinCoef { float a, c, kappa; };
template <int MODEL>
__device__ __forceinline__ LinCoef lin_coef(float xx, float b0, float vbj, const SysScalars& s, const MarkerDraws& dr) {
  const float lmb = marker_lambda<MODEL>(vbj, s);
  const float alpha = 1.0f / (xx + lmb);
  LinCoef o;
  o.kappa = (MODEL == M_EMBA) ? 2.0f : 1.0f;
  float c = -lmb * b0 * alpha;                       // (g + xx*b0)*alpha - b0 = g*alpha - lmb*b0*alpha
  if (MODEL == M_BRR || MODEL == M_BA || MODEL == M_BL) c += sqrtf(s.ve * alpha) * dr.z1;
  o.a = o.kappa * alpha;
  o.c = o.kappa * c;
  return o;
}

__host__ __device__ constexpr bool model_is_gibbs(int m) { return (m >= M_BRR && m <= M_KMUP) || (m >= M_BL && m <= M_BDPI) || m == M_KMUP2; }
__host__ __device__ constexpr bool model_has_vbj(int m) {
  return m == M_EMBA || m == M_EMBB || m == M_BA || m == M_BB || m == M_KMUP || m == M_EMDE || m == M_BL || m == M_BDPI || m == M_GSRR ||
         m == M_GSFLM || m == M_EMMLD || m == M_KMUP2;
}
// the rule itself rewrites the per-marker slot (KMUP's L and emDE's Lmb are inputs of the sweep: caller / epilogue own them)
__host__ __device__ constexpr bool model_rule_writes_vbj(int m) { return model_has_vbj(m) && m != M_KMUP && m != M_KMUP2 && m != M_EMDE && m != M_GSRR && m != M_GSFLM && m != M_EMMLD; }
__host__ __device__ constexpr bool model_has_d(int m) {
  return m == M_EMBB || m == M_EMBC || m == M_BB || m == M_BC || m == M_KMUP || m == M_EMBCPI || m == M_LASSO || m == M_BCPI || m == M_BDPI || m == M_KMUP2;
}
// solvers that stop on sum |b_old - b_new| < tol (emEN :449, emDE :297, emML :505, lasso :1492)
__host__ __device__ constexpr bool model_has_cnv(int m) { return m == M_EMEN || m == M_EMDE || m == M_EMML || m == M_LASSO || m == M_GSRR || m == M_GSFLM || m == M_EMMLD; }

// int8 genotype byte (two's complement) -> float, on the FMA/ALU pipes (no I2F):
// place u = (byte ^ 0x80) = x + 128 in the mantissa of 2^23 and subtract 2^23 + 128 (exact).
__device__ __forceinline__ float byte_to_float(uint32_t word_xored, int byte_idx) {
  uint32_t r;
  const uint32_t sel = 0x7440u | (uint32_t)byte_idx;  // result bytes {u_i, 0x00, 0x00, 0x4B} from (word, 0x4B000000)
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(word_xored), "r"(0x4B000000u), "r"(sel));
  return __uint_as_float(r) - 8388736.0f;
}

// 2-bit store: expand 4 packed bytes (16 rows, row r in bits 2*(r%4) of byte r/4) into 16 int8 bytes.
__device__ __forceinline__ uint4 expand_2bit(uint32_t pk) {
  uint32_t w[4];
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const uint32_t byte = (pk >> (8 * q)) & 0xFFu;
    w[q] = (byte & 3u) | (((byte >> 2) & 3u) << 8) | (((byte >> 4) & 3u) << 16) | (((byte >> 6) & 3u) << 24);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace bwgr
