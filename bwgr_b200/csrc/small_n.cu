// small_n.cu -- "small-n batching" path: one persistent CTA per system (trait / fold / chain).
//
// The residual vector of a system lives in this SM's shared memory for the whole sweep, so the CTA
// runs the reference's per-marker step literally (Rcpp20260726ai.cpp:332-337 and siblings):
//   g = x_j'e  ->  scalar rule  ->  e -= x_j * de
// Each thread owns fixed 16-row chunks of e (no cross-thread hazard on e), genotype columns are
// streamed from HBM/L2 through a cp.async ring in marker order (the order is known up front), and
// the only block-wide synchronisation per marker is the one barrier of the dot-product reduction.
// Independent systems = independent CTAs: no communication (SURVEY 8e, "replicas").
#include "device.cuh"

namespace bwgr {

namespace {

// kRing = genotype columns in flight per CTA (8, 4 or 2 depending on how much shared memory e leaves).
template <int MODEL, int kRing>
__global__ void __launch_bounds__(1024, 1) small_n_sweep_kernel(SmallNArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int sys = blockIdx.x;
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = T >> 5;
  const int ld = (int)a.s.g.ld, p = a.s.g.p;
  const int nchunks = ld >> 4;
  const bool two_bit = a.s.g.storage != 0;
  const int col_bytes = two_bit ? (ld >> 2) : ld;  // bytes of one column slot in the ring

  // e in shared memory, quarter-chunk major: rows 16c + 4q .. 16c + 4q + 3 of chunk c sit at float4 index q * nchunks + c, so that the
  // threads of a warp (consecutive chunks) read consecutive 16-byte words.  (Row-major, thread c's four float4 are 64 bytes apart from
  // thread c + 1's: a 4-way bank conflict on every one of the twelve accesses per marker -- ncu: 1.8e9 conflict cycles, short-scoreboard
  // stall 7.5 per issue at the config-4 shape.)
  float* e_s = reinterpret_cast<float*>(smem_raw);                          // [ld]
  auto e_idx = [&](int i) { return ((((i >> 2) & 3) * nchunks + (i >> 4)) << 2) + (i & 3); };
  unsigned char* ring = smem_raw + (size_t)ld * 4;                          // [kRing][col_bytes]
  unsigned char* mask_s = ring + (size_t)kRing * col_bytes;                 // [ld] (only if mask)
  float* red = reinterpret_cast<float*>(mask_s + (a.s.mask ? ld : 0));        // [2][32]
  MarkerDraws* draws = reinterpret_cast<MarkerDraws*>(red + 64);            // [2][T] (Gibbs)
  int* ord_s = reinterpret_cast<int*>(draws + (model_is_gibbs(MODEL) ? 2 * T : 0));  // [2][T]: the marker order, two chunks of T positions
  // KMUP2 on rows drawn with replacement (R/wgr.R:68, rp = TRUE): H'e0 counts a row as often as it was drawn (:57-60), the residual
  // of a repeated row is one value.  Multiplicities as floats in e's layout, multiplied into the dot product only.
  const float* w_s = nullptr;
  if constexpr (MODEL == M_KMUP2)
    if (a.row_w) w_s = reinterpret_cast<const float*>((reinterpret_cast<uintptr_t>(ord_s + 2 * T) + 15) & ~(uintptr_t)15);
  __shared__ SysScalars sc;

  if (tid == 0) sc = a.s.sc[sys];
  __syncthreads();
  if (sc.done) return;

  float* e_g = a.s.e + (size_t)sys * ld;
  for (int i = tid; i < ld; i += T) e_s[e_idx(i)] = e_g[i];
  if (a.s.mask)
    for (int i = tid; i < ld; i += T) mask_s[i] = a.s.mask[(size_t)sys * ld + i];
  if (w_s)
    for (int i = tid; i < ld; i += T) const_cast<float*>(w_s)[e_idx(i)] = a.row_w[i];

  float* b = a.s.b + (size_t)sys * p;
  float* dvec = a.s.d ? a.s.d + (size_t)sys * p : nullptr;
  float* vbv = a.s.vbv ? a.s.vbv + (size_t)sys * p : nullptr;
  const float* xx = a.s.xx + (a.s.xx_per_sys ? (size_t)sys * p : 0);
  const int* order = a.perms;  // nullptr = natural order
  const int sweep = sc.sweep;
  const uint32_t chain = (uint32_t)(a.s.chain0 + sys);

  // the order is read through shared memory: straight from global memory the index load sat in front of every column address and
  // every per-marker input (a dependent L2 round trip per marker in every thread)
  // (pm, pb) = (pos % T, (pos / T) & 1), kept incrementally: T is a run-time value and an integer division costs ~20 instructions,
  // three of them per marker were a third of the instruction stream of a kernel that is issue-bound
  int pm = 0, pb = 0;
  const bool single = nchunks <= T;
  auto marker_ahead = [&](int pos, int d) {  // marker at position pos + d, 0 <= d < T
    int m = pm + d, bsel = pb;
    if (m >= T) { m -= T; bsel ^= 1; }
    return order ? ord_s[bsel * T + m] : pos + d;
  };
  if (order)
    for (int k = 0; k < 2; k++) { const int q = k * T + tid; if (q < p) ord_s[k * T + tid] = order[q]; }
  __syncthreads();
  auto issue_col = [&](int pos, int j) {
    if (pos < p) {
      unsigned char* slot = ring + (size_t)(pos % kRing) * col_bytes;
      if (!two_bit) {
        const int8_t* src = a.s.g.x8 + (int64_t)j * a.s.g.ld;
        for (int c = tid; c < nchunks; c += T) cp_async16(slot + 16 * c, src + 16 * c);
      } else {
        const uint8_t* src = a.s.g.x2 + (int64_t)j * a.s.g.ldb;
        for (int c = tid; c < nchunks; c += T) cp_async4(slot + 4 * c, src + 4 * c);
      }
    }
    cp_async_commit();
  };

#pragma unroll 1
  for (int q = 0; q < kRing - 1; q++) issue_col(q, marker_ahead(0, q));
  __syncthreads();  // e_s, mask_s visible

  // per-marker inputs, prefetched two markers ahead (a permutation visits a marker once per sweep: nothing read early is stale)
  int jA = marker_ahead(0, 0), jB = p > 1 ? marker_ahead(0, 1) : 0;
  float bA = b[jA], xA = xx[jA], vA = vbv ? vbv[jA] : 0.0f;
  float bB = b[jB], xB = xx[jB], vB = vbv ? vbv[jB] : 0.0f;
  float hA = 0.0f, hB = 0.0f;  // KMUP2: the second per-marker scale
  if constexpr (MODEL == M_KMUP2) { hA = a.s.xx2[jA]; hB = a.s.xx2[jB]; }

#pragma unroll 1
  for (int pos = 0; pos < p; pos++) {
    const int j = jA;
    const float b0 = bA, xxj = xA, vbj = vA, xx2j = hA;
    jA = jB; bA = bB; xA = xB; vA = vB; hA = hB;
    if (order && pos > 0 && pm == 0) {  // chunk pos / T + 1 of the order replaces chunk pos / T - 1 (nobody reads that any more)
      const int q = pos + T + tid;
      if (q < p) ord_s[(pb ^ 1) * T + tid] = order[q];
    }
    if (pos + 2 < p) {
      jB = marker_ahead(pos, 2);
      bB = b[jB]; xB = xx[jB]; vB = vbv ? vbv[jB] : 0.0f;
      if constexpr (MODEL == M_KMUP2) hB = a.s.xx2[jB];
    }
    if (model_is_gibbs(MODEL) && pm == 0) {  // draws of the next T markers, one per thread
      const int q = pos + tid;
      if (q < p)
        draws[pb * T + tid] = marker_draws(MODEL, (uint32_t)marker_ahead(pos, tid), (uint32_t)sweep, chain, sc.df, a.s.seed_lo, a.s.seed_hi);
    }
    issue_col(pos + kRing - 1, pos + kRing - 1 < p ? marker_ahead(pos, kRing - 1) : 0);
    cp_async_wait<kRing - 1>();

    // ---- g = x_j' e over this thread's chunks
    const unsigned char* slot = ring + (size_t)(pos % kRing) * col_bytes;
    float acc = 0.0f;
    // one chunk per thread (n <= 16 T rows, the usual case): the sixteen genotypes of the thread are converted once and stay in
    // registers for the residual update
    float xf[16];
    if (single) {
      if (tid < nchunks) {
        const int c = tid;
        uint4 w = two_bit ? expand_2bit(*reinterpret_cast<const uint32_t*>(slot + 4 * c))
                          : *reinterpret_cast<const uint4*>(slot + 16 * c);
        if (a.s.mask) {
          const uint4 m = *reinterpret_cast<const uint4*>(mask_s + 16 * c);
          w.x &= m.x * 0xFFu; w.y &= m.y * 0xFFu; w.z &= m.z * 0xFFu; w.w &= m.w * 0xFFu;
        }
        const uint32_t ww[4] = {w.x ^ 0x80808080u, w.y ^ 0x80808080u, w.z ^ 0x80808080u, w.w ^ 0x80808080u};
        const float4* ev = reinterpret_cast<const float4*>(e_s) + c;
        float a4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int q = 0; q < 4; q++) {
          float4 e4 = ev[(size_t)q * nchunks];
          if (w_s) { const float4 w4 = reinterpret_cast<const float4*>(w_s)[(size_t)q * nchunks + c]; e4.x *= w4.x; e4.y *= w4.y; e4.z *= w4.z; e4.w *= w4.w; }
#pragma unroll
          for (int k = 0; k < 4; k++) xf[4 * q + k] = byte_to_float(ww[q], k);
          a4[q] = fmaf(xf[4 * q + 0], e4.x, a4[q]); a4[q] = fmaf(xf[4 * q + 1], e4.y, a4[q]);
          a4[q] = fmaf(xf[4 * q + 2], e4.z, a4[q]); a4[q] = fmaf(xf[4 * q + 3], e4.w, a4[q]);
        }
        acc = (a4[0] + a4[1]) + (a4[2] + a4[3]);
      }
    } else
    for (int c = tid; c < nchunks; c += T) {
      uint4 w = two_bit ? expand_2bit(*reinterpret_cast<const uint32_t*>(slot + 4 * c))
                        : *reinterpret_cast<const uint4*>(slot + 16 * c);
      if (a.s.mask) {
        const uint4 m = *reinterpret_cast<const uint4*>(mask_s + 16 * c);
        w.x &= m.x * 0xFFu; w.y &= m.y * 0xFFu; w.z &= m.z * 0xFFu; w.w &= m.w * 0xFFu;
      }
      const uint32_t ww[4] = {w.x ^ 0x80808080u, w.y ^ 0x80808080u, w.z ^ 0x80808080u, w.w ^ 0x80808080u};
      const float4* ev = reinterpret_cast<const float4*>(e_s) + c;
#pragma unroll
      for (int q = 0; q < 4; q++) {
        float4 e4 = ev[(size_t)q * nchunks];
        if (w_s) { const float4 w4 = reinterpret_cast<const float4*>(w_s)[(size_t)q * nchunks + c]; e4.x *= w4.x; e4.y *= w4.y; e4.z *= w4.z; e4.w *= w4.w; }
        acc = fmaf(byte_to_float(ww[q], 0), e4.x, acc);
        acc = fmaf(byte_to_float(ww[q], 1), e4.y, acc);
        acc = fmaf(byte_to_float(ww[q], 2), e4.z, acc);
        acc = fmaf(byte_to_float(ww[q], 3), e4.w, acc);
      }
    }
    acc = warp_sum(acc);
    float* rbuf = red + (pos & 1) * 32;
    if (lane == 0) rbuf[warp] = acc;
    __syncthreads();
    float g = (lane < nwarps) ? rbuf[lane] : 0.0f;
    g = warp_sum(g);

    // ---- rule (every thread, identical inputs -> identical result)
    MarkerDraws dr;
    if (model_is_gibbs(MODEL)) dr = draws[pb * T + pm];
    else { dr.z1 = dr.z2 = dr.u = 0.0f; dr.chi = 1.0f; }
    const RuleOut r = marker_rule<MODEL>(g, xxj, b0, vbj, sc, dr, xx2j);
    if (tid == 0) {
      b[j] = r.b;
      if (model_has_d(MODEL) && dvec) dvec[j] = r.d;
      if (model_rule_writes_vbj(MODEL) && vbv) vbv[j] = r.vbj;
    }

    // ---- e -= x_j * de on this thread's chunks
    if (r.de != 0.0f && single) {
      if (tid < nchunks) {
        float4* ev = reinterpret_cast<float4*>(e_s) + tid;
#pragma unroll
        for (int q = 0; q < 4; q++) {
          float4 e4 = ev[(size_t)q * nchunks];
          e4.x = fmaf(-xf[4 * q + 0], r.de, e4.x); e4.y = fmaf(-xf[4 * q + 1], r.de, e4.y);
          e4.z = fmaf(-xf[4 * q + 2], r.de, e4.z); e4.w = fmaf(-xf[4 * q + 3], r.de, e4.w);
          ev[(size_t)q * nchunks] = e4;
        }
      }
    } else if (r.de != 0.0f) {
      for (int c = tid; c < nchunks; c += T) {
        uint4 w = two_bit ? expand_2bit(*reinterpret_cast<const uint32_t*>(slot + 4 * c))
                          : *reinterpret_cast<const uint4*>(slot + 16 * c);
        if (a.s.mask) {
          const uint4 m = *reinterpret_cast<const uint4*>(mask_s + 16 * c);
          w.x &= m.x * 0xFFu; w.y &= m.y * 0xFFu; w.z &= m.z * 0xFFu; w.w &= m.w * 0xFFu;
        }
        const uint32_t ww[4] = {w.x ^ 0x80808080u, w.y ^ 0x80808080u, w.z ^ 0x80808080u, w.w ^ 0x80808080u};
        float4* ev = reinterpret_cast<float4*>(e_s) + c;
#pragma unroll
        for (int q = 0; q < 4; q++) {
          float4 e4 = ev[(size_t)q * nchunks];
          e4.x = fmaf(-byte_to_float(ww[q], 0), r.de, e4.x);
          e4.y = fmaf(-byte_to_float(ww[q], 1), r.de, e4.y);
          e4.z = fmaf(-byte_to_float(ww[q], 2), r.de, e4.z);
          e4.w = fmaf(-byte_to_float(ww[q], 3), r.de, e4.w);
          ev[(size_t)q * nchunks] = e4;
        }
      }
    }
    if (++pm == T) { pm = 0; pb ^= 1; }
  }
  cp_async_wait<0>();
  __syncthreads();
  for (int i = tid; i < ld; i += T) e_g[i] = e_s[e_idx(i)];
}

}  // namespace

static size_t small_n_smem(const SmallNArgs& a, int ring, int T) {
  const size_t ld = (size_t)a.s.g.ld;
  const size_t col_bytes = a.s.g.storage ? (ld >> 2) : ld;
  return ld * 4 + (size_t)ring * col_bytes + (a.s.mask ? ld : 0) + 64 * 4 +
         (model_is_gibbs(a.model) ? 2 * (size_t)T * sizeof(MarkerDraws) : 0) + 2 * (size_t)T * sizeof(int) + 16 + (a.row_w ? ld * 4 + 16 : 0);
}

// Largest n this path takes: e (4 B/row) + two ring slots must fit the 227 KB of one SM.
bool small_n_fits(const GenoView& g, bool masked, size_t smem_limit, bool weighted) {
  SmallNArgs a;
  a.s.g = g; a.s.mask = masked ? reinterpret_cast<const uint8_t*>(1) : nullptr; a.model = M_BB;
  a.row_w = weighted ? reinterpret_cast<const float*>(1) : nullptr;
  return small_n_smem(a, 2, 1024) <= smem_limit;
}

template <int MODEL>
static cudaError_t launch_small_model(const SmallNArgs& a, size_t smem_limit, cudaStream_t st) {
  const int nchunks = (int)(a.s.g.ld >> 4);
  int T = ((nchunks + 31) / 32) * 32;
  if (T > 1024) T = 1024;
  if (T < 32) T = 32;
#define BWGR_TRY_RING(RING)                                                                                       \
  {                                                                                                               \
    const size_t smem = small_n_smem(a, RING, T);                                                                 \
    if (smem <= smem_limit) {                                                                                     \
      const cudaError_t e =                                                                                       \
          cudaFuncSetAttribute(small_n_sweep_kernel<MODEL, RING>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
      if (e != cudaSuccess) return e;                                                                             \
      small_n_sweep_kernel<MODEL, RING><<<a.s.nsys, T, smem, st>>>(a);                                            \
      return cudaSuccess;                                                                                         \
    }                                                                                                             \
  }
  BWGR_TRY_RING(8)
  BWGR_TRY_RING(4)
  BWGR_TRY_RING(2)
#undef BWGR_TRY_RING
  return cudaErrorInvalidValue;
}

// Every rule but MRR3's rotated systems, which run on the pipelined blocked sweep only.
cudaError_t launch_small_n(const SmallNArgs& a, size_t smem_limit, cudaStream_t st) {
  cudaError_t e = cudaErrorInvalidValue;
  with_rule(a.model, [&](auto rule) {
    constexpr int M = decltype(rule)::value;
    if constexpr (M != M_MRR) e = launch_small_model<M>(a, smem_limit, st);
  });
  return e;
}

}  // namespace bwgr
