// grid_sweep.cu -- the third kernel family ("grid"): the reference's per-marker step (dot -> rule -> residual update), literally, with the
// individuals spread over the whole GPU.  It takes what the other two families cannot: any n on one GPU (the small-n family needs the
// residual of a system in ONE SM's shared memory, the blocked family at most 512 rows per worker, i.e. n <= ~75k), row-masked systems
// (CV folds) at any n, every rule of common.cuh.  Up to 32 systems share one pass over the genotypes.
//
// One persistent cooperative grid; CTA c keeps its row slab of the residuals (and masks) of all systems in shared memory for the whole
// sweep and streams its slab of the genotype columns in marker order through a cp.async ring.  Per marker: slab dot products -> ONE
// grid-wide sum through L2 (the accumulator word of device.cuh, one atomic per system and CTA) -> the rule, evaluated by every CTA
// alike -> rank-one update of the slab.  The integer sums are order-free: every CTA reads bit-identical totals, takes bit-identical
// decisions, and a fit is bit-reproducible.  The per-marker chain is latency-bound (~2-3 us per marker): this family is the fallback,
// not the fast path.
// HBM traffic per sweep: n p bytes.
#include "device.cuh"

namespace bwgr {

namespace {

constexpr int kT = 256;  // threads per CTA
constexpr int kD = 4;    // markers in flight

struct GridSmem {
  float* E;          // [ns][rp]
  uint8_t* M;        // [ns][rp] (masked fits): 0/1, or the multiplicity of a row drawn with replacement (KMUP2, rp = TRUE)
  unsigned char* xs[kD];  // [rp] int8 or [rp] float
  float* vin[kD];    // b0[32] | vbj[32] | xx[32] | xx2
  SysScalars* sc;    // [ns]
  MarkerDraws* dr;   // [2][32]
  int* Js;           // [kD]
};

__host__ __device__ inline size_t grid_carve(unsigned char* base, int ns, int rp, bool masked, int xbytes, GridSmem* s) {
  size_t o = 0;
  auto take = [&](size_t bytes) { unsigned char* q = base ? base + o : nullptr; o = (o + bytes + 15) & ~(size_t)15; return q; };
  float* E = reinterpret_cast<float*>(take(sizeof(float) * (size_t)ns * rp));
  unsigned char* xs[kD];
  for (int d = 0; d < kD; d++) xs[d] = take((size_t)rp * xbytes);
  uint8_t* M = reinterpret_cast<uint8_t*>(take(masked ? (size_t)ns * rp : 0));
  float* vin[kD];
  for (int d = 0; d < kD; d++) vin[d] = reinterpret_cast<float*>(take(sizeof(float) * 100));
  SysScalars* sc = reinterpret_cast<SysScalars*>(take(sizeof(SysScalars) * (size_t)ns));
  MarkerDraws* dr = reinterpret_cast<MarkerDraws*>(take(sizeof(MarkerDraws) * 64));
  int* Js = reinterpret_cast<int*>(take(sizeof(int) * kD));
  if (s) {
    s->E = E; s->M = M; s->sc = sc; s->dr = dr; s->Js = Js;
    for (int d = 0; d < kD; d++) { s->xs[d] = xs[d]; s->vin[d] = vin[d]; }
  }
  return o;
}

// XT = int8_t (integer store) or float (real-valued store: NA-imputed / centred genotypes, what the reference holds as MatrixXf)
template <int MODEL, class XT>
__global__ void __launch_bounds__(kT, 1) grid_sweep_kernel(GridArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_abort;
  __shared__ float s_de[32];
  __shared__ float s_wred[8][33];
  GridSmem s;
  const int ns = a.s.nsys, rp = a.rows_per_cta, p = a.s.g.p;
  const bool masked = a.s.mask != nullptr;
  grid_carve(smem_raw, ns, rp, masked, (int)sizeof(XT), &s);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, G = (int)gridDim.x, cta = blockIdx.x;
  const int64_t ld = a.s.g.ld, r0 = (int64_t)cta * rp;
  for (int q = tid; q < ns * rp; q += kT) {
    const int t = q / rp, i = q - t * rp;
    const bool in = r0 + i < ld;
    s.E[q] = in ? a.s.e[(size_t)t * ld + r0 + i] : 0.0f;
    if (masked) s.M[q] = in ? a.s.mask[(size_t)t * ld + r0 + i] : (uint8_t)0;
  }
  for (int q = tid; q < kD * rp * (int)sizeof(XT); q += kT) s.xs[0][q] = 0;  // the ring slots are contiguous (rp is a multiple of 16)
  if (tid < ns) s.sc[tid] = a.s.sc[tid];
  if (tid == 0) s_abort = 0;
  const int nch = rp * (int)sizeof(XT) / 16;  // 16-byte chunks of a slab
  constexpr int kRowsPerChunk = 16 / (int)sizeof(XT);
  const float* xxbase = a.s.xx;
  int Jnext = a.perm ? a.perm[0] : 0;
  auto prefetch = [&](int m) {
    if (m < p) {
      const int J = Jnext, slot = m % kD;
      if (m + 1 < p) Jnext = a.perm ? a.perm[m + 1] : m + 1;
      const unsigned char* col = sizeof(XT) == 1 ? reinterpret_cast<const unsigned char*>(a.s.g.x8 + (int64_t)J * ld + r0)
                                                 : reinterpret_cast<const unsigned char*>(a.s.g.xf + (int64_t)J * ld + r0);
      for (int c = tid; c < nch; c += kT)
        if (r0 + (int64_t)kRowsPerChunk * c < ld) cp_async16(s.xs[slot] + 16 * c, col + 16 * c);
      float* v = s.vin[slot];
      if (tid < 32) { if (tid < ns) cp_async4(v + tid, a.s.b + (size_t)tid * p + J); }
      else if (tid < 64) { const int t = tid - 32; if (t < ns && a.s.vbv) cp_async4(v + 32 + t, a.s.vbv + (size_t)t * p + J); }
      else if (tid < 96) { const int t = tid - 64; if (t < ns) cp_async4(v + 64 + t, xxbase + (a.s.xx_per_sys ? (size_t)t * p : 0) + J); }
      else if (tid == 96 && a.s.xx2) cp_async4(v + 96, a.s.xx2 + J);
      if (tid == 0) s.Js[slot] = J;
    }
    cp_async_commit();
  };
  __syncthreads();  // the zeroed ring slots are in place before any cp.async lands in them
  for (int m = 0; m < kD - 1; m++) prefetch(m);
  __syncthreads();
  if (model_is_gibbs(MODEL) && warp == 1 && lane < ns)  // draws of marker 0
    s.dr[lane] = marker_draws(MODEL, (uint32_t)s.Js[0], (uint32_t)s.sc[lane].sweep, (uint32_t)(a.s.chain0 + lane), s.sc[lane].df, a.s.seed_lo, a.s.seed_hi);
  const unsigned long long t_start = globaltimer_ns();
  const double inv_q = (double)a.g_quantum;  // value of one fixed-point unit
  const double qinv = 1.0 / (double)a.g_quantum;
  for (int m = 0; m < p; m++) {
    cp_async_wait<kD - 2>();
    __syncthreads();  // marker m's slot has landed; step m - 1 is finished by every thread
    prefetch(m + kD - 1);
    const int slot = m % kD;
    const XT* xs = reinterpret_cast<const XT*>(s.xs[slot]);
    const float* vin = s.vin[slot];
    // ---- slab dot products g_s = x'e_s
    if (ns == 1) {
      float acc = 0.0f;
      if (masked) for (int i = tid; i < rp; i += kT) acc = fmaf((float)xs[i] * (float)s.M[i], s.E[i], acc);
      else for (int i = tid; i < rp; i += kT) acc = fmaf((float)xs[i], s.E[i], acc);
      acc = warp_sum(acc);
      if (lane == 0) s_wred[warp][0] = acc;
    } else {
      for (int t0 = 0; t0 < ns; t0 += 8) {
        float acc[8];
#pragma unroll
        for (int q = 0; q < 8; q++) acc[q] = 0.0f;
        for (int i = tid; i < rp; i += kT) {
          const float x = (float)xs[i];
#pragma unroll
          for (int q = 0; q < 8; q++)
            if (t0 + q < ns) acc[q] = fmaf(masked ? x * (float)s.M[(t0 + q) * rp + i] : x, s.E[(t0 + q) * rp + i], acc[q]);
        }
#pragma unroll
        for (int q = 0; q < 8; q++) {
          if (t0 + q < ns) {
            const float v = warp_sum(acc[q]);
            if (lane == 0) s_wred[warp][t0 + q] = v;
          }
        }
      }
    }
    __syncthreads();
    if (warp == 0) {
      const bool on = lane < ns;
      if (on) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < 8; w++) v += (double)s_wred[w][lane];
        grid_add(a.acc + ((size_t)m * kGridCopies + (cta & (kGridCopies - 1))) * 32 + lane, v * qinv, a.s.err);
      }
      const long long tot = grid_wait_total(a.acc + (size_t)m * kGridCopies * 32 + (on ? lane : 0), on, G, a.s.err, t_start, &s_abort);
      if (on) {
        const float g = (float)((double)tot * inv_q);
        const SysScalars& sc = s.sc[lane];
        float de = 0.0f;
        if (!sc.done) {
          MarkerDraws dr;
          if (model_is_gibbs(MODEL)) dr = s.dr[(m & 1) * 32 + lane];
          else { dr.z1 = dr.z2 = dr.u = 0.0f; dr.chi = 1.0f; }
          const float vbj = a.s.vbv ? vin[32 + lane] : 0.0f;
          const RuleOut r = marker_rule<MODEL>(g, vin[64 + lane], vin[lane], vbj, sc, dr, a.s.xx2 ? vin[96] : 0.0f);
          de = r.de;
          if (cta == 0) {
            const size_t q = (size_t)lane * p + s.Js[slot];
            a.s.b[q] = r.b;
            if (model_has_d(MODEL) && a.s.d) a.s.d[q] = r.d;
            if (model_rule_writes_vbj(MODEL) && a.s.vbv) a.s.vbv[q] = r.vbj;
          }
        }
        s_de[lane] = de;
      }
    } else if (model_is_gibbs(MODEL) && warp == 1 && lane < ns && m + 1 < p) {  // the next marker's draws, off the chain
      s.dr[((m + 1) & 1) * 32 + lane] = marker_draws(MODEL, (uint32_t)s.Js[(m + 1) % kD], (uint32_t)s.sc[lane].sweep, (uint32_t)(a.s.chain0 + lane),
                                                     s.sc[lane].df, a.s.seed_lo, a.s.seed_hi);
    }
    __syncthreads();
    if (s_abort) return;  // the host reports the error flag; the residuals of this launch are not written back
    // ---- e_s -= x de_s (on the rows the system uses)
    for (int t = 0; t < ns; t++) {
      const float de = s_de[t];
      if (de == 0.0f) continue;
      float* Et = s.E + (size_t)t * rp;
      if (masked) {
        const uint8_t* Mt = s.M + (size_t)t * rp;
        for (int i = tid; i < rp; i += kT) Et[i] = fmaf(Mt[i] ? -(float)xs[i] : 0.0f, de, Et[i]);  // the byte may be a row multiplicity: it weighs the dot products only
      } else {
        for (int i = tid; i < rp; i += kT) Et[i] = fmaf(-(float)xs[i], de, Et[i]);
      }
    }
  }
  cp_async_wait<0>();
  __syncthreads();
  for (int q = tid; q < ns * rp; q += kT) {
    const int t = q / rp, i = q - t * rp;
    if (r0 + i < ld) a.s.e[(size_t)t * ld + r0 + i] = s.E[q];
  }
}

// ---- blocks of kGB markers per grid sum (unmasked systems) -----------------------------------------------------------------------
// One L2 round trip per BLOCK instead of per marker: the round carries the dot products of the block's markers with the residuals as
// they stand at the start of the block, and the cross products x_j'x_i of the block (integers for the int8 store: exact).  Every CTA
// then walks the block alike: the dot of marker j is corrected by the steps already taken in the block,
// g_j = g_j(stale) - sum_{i<j} (x_j'x_i) de_i -- the same algebra as the blocked family, on CUDA cores -- and the residual slab gets the
// block's update at once.  The cross products do not depend on the residuals: they are summed one block AHEAD, by the warps that do
// not poll, while the polling warps (one thread per word) wait for the current block's totals; before the wait a CTA only has its 16
// dot products to add.  Measured at n = 100,000 (profiles/r2_grid_block_probe.txt): 0.51 us per marker (1.88 one marker per sum).
constexpr int kGB = 16;                       // markers per block (measured: 32 is 10 % slower per marker, the chain and the payload grow)
constexpr int kGP = kGB * (kGB - 1) / 2;      // cross products per block
constexpr int kGR = 3;                        // blocks in flight
constexpr int kJR = kGR + 1;                  // marker indices are staged one block further ahead
constexpr int kTB = 1024;                     // threads per CTA of the blocked variant: its phases are short dependent chains, 32 warps hide them
static_assert(kGB <= 32 && kGB * 32 + kGP <= kTB, "one dot warp per marker, one polling thread per word");

struct GridBlockSmem {
  float* E;                 // [ns][rp]
  unsigned char* xs[kGR];   // [kGB][rp] int8 / float
  float* vin[kGR];          // [kGB][100]
  int* Js[kJR];             // [kGB]
  float* tot;               // [kGB * ns + kGP] the block's totals: dots (marker-major, stale) | cross products j (j - 1) / 2 + i
  float* de;                // [kGB][32]
  SysScalars* sc;           // [ns]
  MarkerDraws* dr;          // [2][kGB][32]
  unsigned char* pj;        // [kGP] pair index pr = j (j - 1) / 2 + i (i < j) -> j
};

__host__ __device__ inline size_t grid_block_carve(unsigned char* base, int ns, int rp, int xbytes, bool gibbs, GridBlockSmem* s) {
  size_t o = 0;
  auto take = [&](size_t bytes) { unsigned char* q = base ? base + o : nullptr; o = (o + bytes + 15) & ~(size_t)15; return q; };
  float* E = reinterpret_cast<float*>(take(sizeof(float) * (size_t)ns * rp));
  unsigned char* xs[kGR];
  for (int d = 0; d < kGR; d++) xs[d] = take((size_t)kGB * rp * xbytes);
  float* vin[kGR];
  for (int d = 0; d < kGR; d++) vin[d] = reinterpret_cast<float*>(take(sizeof(float) * kGB * 100));
  int* Js[kJR];
  for (int d = 0; d < kJR; d++) Js[d] = reinterpret_cast<int*>(take(sizeof(int) * kGB));
  float* tot = reinterpret_cast<float*>(take(sizeof(float) * (kGB * 32 + kGP)));
  float* de = reinterpret_cast<float*>(take(sizeof(float) * kGB * 32));
  SysScalars* sc = reinterpret_cast<SysScalars*>(take(sizeof(SysScalars) * (size_t)ns));
  MarkerDraws* dr = reinterpret_cast<MarkerDraws*>(take(gibbs ? sizeof(MarkerDraws) * 2 * kGB * 32 : 0));
  unsigned char* pj = take(kGP);
  if (s) {
    s->E = E; s->tot = tot; s->de = de; s->sc = sc; s->dr = dr; s->pj = pj;
    for (int d = 0; d < kGR; d++) { s->xs[d] = xs[d]; s->vin[d] = vin[d]; }
    for (int d = 0; d < kJR; d++) s->Js[d] = Js[d];
  }
  return o;
}

__host__ __device__ inline int grid_block_words(int ns) { return (kGB * ns + kGP + 31) / 32 * 32; }

template <int MODEL, class XT>
__global__ void __launch_bounds__(kTB, 1) grid_block_kernel(GridArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_abort;
  GridBlockSmem s;
  const int ns = a.s.nsys, rp = a.rows_per_cta, p = a.s.g.p;
  grid_block_carve(smem_raw, ns, rp, (int)sizeof(XT), model_is_gibbs(MODEL), &s);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, G = (int)gridDim.x, cta = blockIdx.x;
  const int64_t ld = a.s.g.ld, r0 = (int64_t)cta * rp;
  const int nblk = (p + kGB - 1) / kGB, W = grid_block_words(ns), ndot = kGB * ns;
  for (int q = tid; q < ns * rp; q += kTB) {
    const int t = q / rp, i = q - t * rp;
    s.E[q] = (r0 + i < ld) ? a.s.e[(size_t)t * ld + r0 + i] : 0.0f;
  }
  for (int q = tid; q < kGR * kGB * rp * (int)sizeof(XT); q += kTB) s.xs[0][q] = 0;  // slots are contiguous
  for (int q = tid; q < kGR * kGB * 100; q += kTB) s.vin[0][q] = 0.0f;
  if (tid < ns) s.sc[tid] = a.s.sc[tid];
  if (tid == 0) s_abort = 0;
  for (int j = 1 + warp; j < kGB; j += kTB / 32)
    for (int i = lane; i < j; i += 32) s.pj[j * (j - 1) / 2 + i] = (unsigned char)j;
  __syncthreads();  // the zeroed ring slots are in place before any cp.async lands in them
  const int nch = rp * (int)sizeof(XT) / 16;
  constexpr int kRowsPerChunk = 16 / (int)sizeof(XT);
  // marker indices of block blk -> shared memory, by sixteen threads of the last warp (their L2 round trip stays off everybody's path:
  // the indices are used one step later)
  auto load_js = [&](int blk) {
    const int j = tid - (kTB - 32);
    if (j >= 0 && j < kGB && blk < nblk) {
      const int m = blk * kGB + j;
      s.Js[blk % kJR][j] = m < p ? (a.perm ? a.perm[m] : m) : 0;
    }
  };
  auto prefetch = [&](int blk) {
    if (blk < nblk) {
      const int slot = blk % kGR, nb = min(kGB, p - blk * kGB);
      const int* Jv = s.Js[blk % kJR];
      // the block's column slabs as (marker, 16-byte chunk) pairs dealt over the CTA: one pass, no per-marker loop on every thread
      for (int q = tid; q < nb * nch; q += kTB) {
        const int j = q / nch, c = q - j * nch;
        if (r0 + (int64_t)kRowsPerChunk * c < ld) {
          const int64_t off = (int64_t)Jv[j] * ld + r0;
          const unsigned char* col = sizeof(XT) == 1 ? reinterpret_cast<const unsigned char*>(a.s.g.x8 + off) : reinterpret_cast<const unsigned char*>(a.s.g.xf + off);
          cp_async16(s.xs[slot] + (size_t)j * rp * sizeof(XT) + 16 * c, col + 16 * c);
        }
      }
      // the markers' inputs (b0 | vb_j | xx per system), dealt from the other end of the CTA
      for (int q = kTB - 1 - tid; q < nb * 96; q += kTB) {
        const int j = q / 96, w = (q - j * 96) >> 5, t = q & 31;
        if (t < ns) {
          const int J = Jv[j];
          float* v = s.vin[slot] + j * 100 + 32 * w + t;
          if (w == 0) cp_async4(v, a.s.b + (size_t)t * p + J);
          else if (w == 1) { if (a.s.vbv) cp_async4(v, a.s.vbv + (size_t)t * p + J); }
          else cp_async4(v, a.s.xx + (a.s.xx_per_sys ? (size_t)t * p : 0) + J);
        }
      }
    }
    cp_async_commit();
  };
  auto draws_for = [&](int blk) {  // Gibbs draws of a block's markers, one (marker, system) per thread of warps 1..7
    if (!model_is_gibbs(MODEL) || blk >= nblk) return;
    const int nb = min(kGB, p - blk * kGB);
    for (int q = tid - 32; q < nb * ns; q += kTB - 32) {
      if (q < 0) break;
      const int j = q / ns, t = q - j * ns;
      s.dr[((blk & 1) * kGB + j) * 32 + t] = marker_draws(MODEL, (uint32_t)s.Js[blk % kJR][j], (uint32_t)s.sc[t].sweep, (uint32_t)(a.s.chain0 + t),
                                                          s.sc[t].df, a.s.seed_lo, a.s.seed_hi);
    }
  };
  const unsigned long long t_start = globaltimer_ns();
  const double inv_q = (double)a.g_quantum, qinv = 1.0 / (double)a.g_quantum;
  const double inv_qG = (double)a.gram_quantum, qinvG = 1.0 / (double)a.gram_quantum;
  // cross products x_j'x_i (i < j) of a block: E-independent, so they are summed over the grid one block AHEAD of their use -- while the
  // polling warps wait for the current block's totals -- by the warps w0, w0 + 1, ... of the CTA
  auto cross_tasks = [&](int blk, int w0) {
    if (blk >= nblk) return;
    const XT* xs = reinterpret_cast<const XT*>(s.xs[blk % kGR]);
    unsigned long long* accw = a.acc + ((size_t)blk * kGridCopies + (cta & (kGridCopies - 1))) * W + ndot;
    for (int pr = warp - w0; pr < kGP; pr += kTB / 32 - w0) {
      const int j = s.pj[pr], i2 = pr - j * (j - 1) / 2;
      double v;
      if constexpr (sizeof(XT) == 1) {
        const int* wj = reinterpret_cast<const int*>(xs + (size_t)j * rp);
        const int* wi = reinterpret_cast<const int*>(xs + (size_t)i2 * rp);
        int acc = 0;
        for (int q = lane; q < rp / 4; q += 32) acc = __dp4a(wj[q], wi[q], acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        v = (double)acc * qinvG;
      } else {
        const float* fj = reinterpret_cast<const float*>(xs + (size_t)j * rp);
        const float* fi = reinterpret_cast<const float*>(xs + (size_t)i2 * rp);
        float acc = 0.0f;
        for (int q = lane; q < rp; q += 32) acc = fmaf(fj[q], fi[q], acc);
        v = (double)warp_sum(acc) * qinvG;
      }
      if (lane == 0) atomicAdd(accw + pr, grid_word(v));
    }
  };
  const int nw = ndot + kGP;            // words of a block: one polling thread each (nw <= 16 * 32 + 120 < kTB)
  const int npollw = (nw + 31) / 32;    // the polling warps; the others work ahead while these wait
  for (int b = 0; b < kGR; b++) load_js(b);
  __syncthreads();
  for (int b = 0; b < kGR - 1; b++) prefetch(b);
  draws_for(0);
  cp_async_wait<0>();
  __syncthreads();
  cross_tasks(0, 0);
  for (int blk = 0; blk < nblk; blk++) {
    cp_async_wait<0>();    // block blk + 1's slab (issued one whole block ago) has landed, block blk's long since
    __syncthreads();  // ... for every thread; block blk - 1 is finished by every thread
    prefetch(blk + kGR - 1);
    const int slot = blk % kGR, nb = min(kGB, p - blk * kGB);
    const int* Jcur = s.Js[blk % kJR];
    const XT* xs = reinterpret_cast<const XT*>(s.xs[slot]);
    unsigned long long* accw = a.acc + ((size_t)blk * kGridCopies + (cta & (kGridCopies - 1))) * W;
    // ---- the block's dot tasks (marker j with the residuals as they stand), one warp each
    if (warp < nb) {
      const int j = warp;
      const XT* xj = xs + (size_t)j * rp;
      if (ns == 1) {
        float acc = 0.0f;
        for (int i = lane; i < rp; i += 32) acc = fmaf((float)xj[i], s.E[i], acc);
        const double v = (double)warp_sum(acc) * qinv;
        if (lane == 0) grid_add(accw + j, v, a.s.err);
      } else {
        for (int t0 = 0; t0 < ns; t0 += 4) {
          const int nt = min(4, ns - t0);
          float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
          for (int i = lane; i < rp; i += 32) {
            const float x = (float)xj[i];
#pragma unroll
            for (int q = 0; q < 4; q++)
              if (q < nt) acc[q] = fmaf(x, s.E[(t0 + q) * rp + i], acc[q]);
          }
#pragma unroll
          for (int q = 0; q < 4; q++) {
            if (q < nt) {
              const double v = (double)warp_sum(acc[q]) * qinv;
              if (lane == 0) grid_add(accw + j * ns + t0 + q, v, a.s.err);
            }
          }
        }
      }
    }
    load_js(blk + kGR);
    if (warp >= npollw) {
      cross_tasks(blk + 1, npollw);  // next block's cross products, under this block's wait
    } else if (tid < nw && !(tid < ndot && tid / ns >= nb)) {  // markers past the end of the last block are never added
      // ---- the block's totals, one word per polling thread: a word is complete when its low byte counts all the CTAs of its copy
      const unsigned long long* src = a.acc + (size_t)blk * kGridCopies * W + tid;
      unsigned int spins = 0;
      for (;;) {
        long long tot = 0;
        bool done = true;
#pragma unroll
        for (int c = 0; c < kGridCopies; c++) {
          const unsigned long long w = ld_relaxed_u64(src + (size_t)c * W);
          done &= grid_word_count(w) == grid_copy_count(G, c);
          tot += grid_word_value(w);
        }
        if (done) { s.tot[tid] = (float)((double)tot * (tid < ndot ? inv_q : inv_qG)); break; }
        if ((++spins & 0x3ffu) == 0) {
          if (*reinterpret_cast<volatile int*>(a.s.err) != 0) { s_abort = 1; break; }
          if (globaltimer_ns() - t_start > kGridTimeoutNs) { atomicExch(a.s.err, 3); s_abort = 1; break; }
        }
      }
    }
    __syncthreads();
    if (s_abort) return;
    // ---- the block's chain, by every CTA alike: lane t of warp 0 walks system t; the other warps draw for the next block
    if (warp == 0) {
      if (lane < ns) {
        const SysScalars& sc = s.sc[lane];
        const float* vin = s.vin[slot];
        float de[kGB];
#pragma unroll
        for (int j = 0; j < kGB; j++) {
          de[j] = 0.0f;
          if (j < nb && !sc.done) {
            float g = s.tot[j * ns + lane];
#pragma unroll
            for (int i = 0; i < j; i++) g = fmaf(-s.tot[ndot + j * (j - 1) / 2 + i], de[i], g);
            MarkerDraws dr;
            if (model_is_gibbs(MODEL)) dr = s.dr[((blk & 1) * kGB + j) * 32 + lane];
            else { dr.z1 = dr.z2 = dr.u = 0.0f; dr.chi = 1.0f; }
            const float* v = vin + j * 100;
            const RuleOut r = marker_rule<MODEL>(g, v[64 + lane], v[lane], a.s.vbv ? v[32 + lane] : 0.0f, sc, dr, 0.0f);
            de[j] = r.de;
            if (cta == 0) {
              const size_t q = (size_t)lane * p + Jcur[j];
              a.s.b[q] = r.b;
              if (model_has_d(MODEL) && a.s.d) a.s.d[q] = r.d;
              if (model_rule_writes_vbj(MODEL) && a.s.vbv) a.s.vbv[q] = r.vbj;
            }
          }
          s.de[j * 32 + lane] = de[j];
        }
      }
    } else {
      draws_for(blk + 1);
    }
    __syncthreads();
    // ---- e_t -= sum_j x_j de_jt
    for (int i = tid; i < rp; i += kTB) {
      float x[kGB];
#pragma unroll
      for (int j = 0; j < kGB; j++) x[j] = (float)xs[(size_t)j * rp + i];
      for (int t = 0; t < ns; t++) {
        float acc = 0.0f;
#pragma unroll
        for (int j = 0; j < kGB; j++) acc = fmaf(x[j], s.de[j * 32 + t], acc);
        s.E[t * rp + i] -= acc;
      }
    }
  }
  cp_async_wait<0>();
  __syncthreads();
  for (int q = tid; q < ns * rp; q += kTB) {
    const int t = q / rp, i = q - t * rp;
    if (r0 + i < ld) a.s.e[(size_t)t * ld + r0 + i] = s.E[q];
  }
}

template <int MODEL>
cudaError_t launch_grid_model(const GridArgs& a, int grid, cudaStream_t st) {
  const bool real = a.s.g.storage == 2;
  size_t smem = grid_sweep_smem(a.s.nsys, a.rows_per_cta, a.s.mask != nullptr, real);
  int threads = kT;
  const void* fn = real ? reinterpret_cast<const void*>(grid_sweep_kernel<MODEL, float>) : reinterpret_cast<const void*>(grid_sweep_kernel<MODEL, int8_t>);
  if (a.blocked) {
    if constexpr (MODEL != M_KMUP2) {
      smem = grid_block_smem(a.s.nsys, a.rows_per_cta, real, model_is_gibbs(MODEL));
      fn = real ? reinterpret_cast<const void*>(grid_block_kernel<MODEL, float>) : reinterpret_cast<const void*>(grid_block_kernel<MODEL, int8_t>);
      threads = kTB;
    }
  }
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  GridArgs args = a;
  void* params[] = {&args};
  return cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(threads), params, smem, st);
}

}  // namespace

size_t grid_block_smem(int nsys, int rows_per_cta, bool real_store, bool gibbs) {
  return grid_block_carve(nullptr, nsys, rows_per_cta, real_store ? 4 : 1, gibbs, nullptr) + 16;
}
size_t grid_block_acc_words(int nsys, int p) { return (size_t)((p + kGB - 1) / kGB) * kGridCopies * grid_block_words(nsys); }

size_t grid_sweep_smem(int nsys, int rows_per_cta, bool masked, bool real_store) {
  return grid_carve(nullptr, nsys, rows_per_cta, masked, real_store ? 4 : 1, nullptr) + 16;
}

// Every rule but MRR3's rotated systems, which run on the pipelined blocked sweep only.
cudaError_t launch_grid_sweep(const GridArgs& a, int grid, cudaStream_t st) {
  cudaError_t e = cudaErrorInvalidValue;
  with_rule(a.model, [&](auto rule) {
    constexpr int M = decltype(rule)::value;
    if constexpr (M != M_MRR) e = launch_grid_model<M>(a, grid, st);
  });
  return e;
}

}  // namespace bwgr
