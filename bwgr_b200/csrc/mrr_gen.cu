// mrr_gen.cu -- the GENERAL multivariate ridge sweep (MRR3 / MRR3F, RcppEigen20230423.cpp:318-701, :704-1079): per-trait
// observation masks (missing phenotypes, :359-365), the inner Gauss-Seidel solve (:510-514), marker weights (NLfactor, :504,
// :524-533), MRR3F's NoInv system (:878-882) and the tilde-hat variance estimator (TH, :423, :549-571).
//
// With missing phenotypes XX(J,t) differs per trait, so the k x k system of a marker no longer diagonalises once per sweep
// (the rotation of mrr.cu) and the marker walk is a strict chain of p dependent k x k solves.  What the chain does NOT depend
// on is factored out of it:
//   * mrr_gen_systems_kernel: the system matrix of EVERY marker of the sweep, inverted up front (one warp per marker,
//     Gauss-Jordan in shared memory, float64), so a chain step is one k x k mat-vec;
//   * mrr_gen_sweep_kernel: one persistent cooperative grid; CTA c keeps its row slab of the k residual columns and of the
//     observation mask in shared memory for the whole sweep (float64: this path is the reference's MRR3 arithmetic), streams
//     its slab of the genotype columns in marker order through a cp.async ring together with the marker's matrix and
//     vectors, and per marker: slab dot products -> one grid-wide sum through L2 (the accumulator words of device.cuh: each warp
//     adds its fixed-point partials with one atomic each; integer sums are order-free, so all CTAs read bit-identical totals and no
//     broadcast is needed) -> mat-vec (or the inner Gauss-Seidel walk) -> masked rank-one update of the slab.  Column centring (:378-379) is analytic: x_c'e = x'e - mean_J * sum(e), with the
//     running column sums of e carried in registers.
// HBM traffic per sweep: n p bytes of genotypes + 8 k^2 p bytes of matrices; the bound is the grid sum's latency per marker.
#include "device.cuh"

namespace bwgr {

namespace {

constexpr int kGT = 256;  // threads of a sweep CTA
constexpr int kGD = 4;    // ring depth (markers in flight)

// 8 B, through L1
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

// Per marker, one pass over the column: masked integer sums sxz[j][t] = sum_i x z_t, sxxz[j][t] = sum_i x^2 z_t (exact), and
// xty[j][t] = sum_i x y_t (float64).  One warp per marker, eight markers per CTA: the eight warps walk the rows together, so the
// k phenotype columns and the mask words they all read come from L1 (one CTA per marker re-read them from L2 for every marker:
// 8 k n bytes each, 400 GB at 50k x 50k x 20).
__global__ void __launch_bounds__(256) mrr_gen_colstats_kernel(GenoView g, const uint32_t* __restrict__ zbits,
                                                               const double* __restrict__ y, int k, double* __restrict__ sxz,
                                                               double* __restrict__ sxxz, double* __restrict__ xty) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = blockIdx.x * 8 + warp;
  if (j >= g.p) return;
  const int8_t* col = g.x8 + (int64_t)j * g.ld;
  int s1[32], s2[32];
  double s3[32];
#pragma unroll
  for (int t = 0; t < 32; t++) { s1[t] = 0; s2[t] = 0; s3[t] = 0.0; }
  for (int i = lane; i < g.n; i += 32) {
    const int x = col[i];
    const uint32_t zb = zbits[i];
    const double xd = (double)x;
#pragma unroll
    for (int t = 0; t < 32; t++) {
      if (t < k) {
        const int m = -(int)((zb >> t) & 1u);
        s1[t] += m & x;
        s2[t] += m & (x * x);
        s3[t] = fma(xd, y[(size_t)t * g.ld + i], s3[t]);  // y is zero where unobserved
      }
    }
  }
#pragma unroll
  for (int t = 0; t < 32; t++) {
    if (t < k) {
      long long a = s1[t], c = s2[t];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); c += __shfl_xor_sync(0xffffffffu, c, o); }
      const double d = warp_sum(s3[t]);
      if (lane == 0) {
        sxz[(size_t)j * k + t] = (double)a;
        sxxz[(size_t)j * k + t] = (double)c;
        xty[(size_t)j * k + t] = d;
      }
    }
  }
}

// The k x k system of every marker of the sweep (one warp per marker).  fixed[j] = {XX(j,0..k) | ...}; W = marker weights
// [p][k] or nullptr; iG / vb column-major k x k; wv_t = iVe_t * W(j,t); d_t = XX(j,t) * wv_t.
//   direct solve, traditional system (:505-507):  sol_j = (iG + diag(d))^-1 diag(wv)               b1 = sol_j * r
//   direct solve, NoInv system of MRR3F (:878-882): LHS = vb diag(d) + I, of which LLT reads the lower triangle;
//                                                  sol_j = sym(LHS)^-1 vb diag(wv)
//   inner Gauss-Seidel (:510-514): sol_j = [LHS | PRE] with RHS = PRE * r
// where r_t = x_c'e_t + XX(j,t) b0_t is what the chain supplies.
__global__ void __launch_bounds__(32) mrr_gen_systems_kernel(int p, int k, int fstride, const double* __restrict__ fixed,
                                                             const double* __restrict__ W, const double* __restrict__ iG,
                                                             const double* __restrict__ vb, const double* __restrict__ iVe,
                                                             int noinv_system, int innergs, double* __restrict__ sol) {
  __shared__ double aug[32 * 65];
  __shared__ double dv[32], wv[32];
  const int J = blockIdx.x, lane = threadIdx.x, kk = k * k, st = 2 * k + 1;
  if (lane < k) {
    const double w = iVe[lane] * (W ? W[(size_t)J * k + lane] : 1.0);
    wv[lane] = w;
    dv[lane] = fixed[(size_t)J * fstride + lane] * w;
  }
  __syncwarp();
  if (innergs) {
    double* lhs = sol + (size_t)J * 2 * kk;
    double* pre = lhs + kk;
    if (lane < k)
      for (int c = 0; c < k; c++) {
        const double id = lane == c ? 1.0 : 0.0;
        lhs[lane * k + c] = noinv_system ? vb[lane + (size_t)c * k] * dv[c] + id : iG[lane + (size_t)c * k] + id * dv[c];
        pre[lane * k + c] = noinv_system ? vb[lane + (size_t)c * k] * wv[c] : id * wv[c];
      }
    return;
  }
  if (lane < k)
    for (int c = 0; c < k; c++) {
      const int rr = lane > c ? lane : c, cc = lane > c ? c : lane;  // the triangle LLT reads
      const double id = rr == cc ? 1.0 : 0.0;
      aug[lane * st + c] = noinv_system ? vb[rr + (size_t)cc * k] * dv[cc] + id : iG[rr + (size_t)cc * k] + id * dv[cc];
      aug[lane * st + k + c] = lane == c ? 1.0 : 0.0;
    }
  __syncwarp();
  for (int piv = 0; piv < k; piv++) {  // Gauss-Jordan without pivoting (symmetric positive definite systems)
    const double ip = 1.0 / aug[piv * st + piv];
    __syncwarp();
    if (lane == piv)
      for (int c = 0; c < 2 * k; c++) aug[piv * st + c] *= ip;
    __syncwarp();
    if (lane < k && lane != piv) {
      const double f = aug[lane * st + piv];
      for (int c = 0; c < 2 * k; c++) aug[lane * st + c] = fma(-f, aug[piv * st + c], aug[lane * st + c]);
    }
    __syncwarp();
  }
  if (lane < k) {
    double* out = sol + (size_t)J * kk + (size_t)lane * k;
    for (int c = 0; c < k; c++) {
      double v;
      if (noinv_system) {
        v = 0.0;
        for (int m = 0; m < k; m++) v = fma(aug[lane * st + k + m], vb[m + (size_t)c * k], v);
      } else {
        v = aug[lane * st + k + c];
      }
      out[c] = v * wv[c];
    }
  }
}

struct GenSmem {
  double* E;        // [k][rp]
  uint32_t* zb;     // [rp]
  double* dl;       // [32]
  int* Js;          // [kGD]
  int* irgs;        // [32]
  double* mats[kGD];
  double* vec[kGD];
  int8_t* xs[kGD];
};

__device__ __forceinline__ GenSmem carve(unsigned char* base, int ke, int rp, int nmat, int k) {
  GenSmem s;
  size_t o = 0;
  s.E = reinterpret_cast<double*>(base + o); o += sizeof(double) * (size_t)ke * rp;
  s.dl = reinterpret_cast<double*>(base + o); o += sizeof(double) * 32;
  for (int d = 0; d < kGD; d++) { s.mats[d] = reinterpret_cast<double*>(base + o); o += sizeof(double) * (size_t)nmat * k * k; }
  for (int d = 0; d < kGD; d++) { s.vec[d] = reinterpret_cast<double*>(base + o); o += sizeof(double) * (3 * k + 1); }
  o = (o + 15) & ~(size_t)15;
  for (int d = 0; d < kGD; d++) { s.xs[d] = reinterpret_cast<int8_t*>(base + o); o += (size_t)rp; }
  s.zb = reinterpret_cast<uint32_t*>(base + o); o += sizeof(uint32_t) * (size_t)rp;
  s.Js = reinterpret_cast<int*>(base + o); o += sizeof(int) * kGD;
  s.irgs = reinterpret_cast<int*>(base + o);
  return s;
}

// int8 genotype byte -> double on the integer and FP64 pipes (no I2F): u = x + 128 in the low mantissa bits of 2^52, minus 2^52 + 128
__device__ __forceinline__ double byte_to_double(int8_t x) {
  return __hiloint2double(0x43300000, (int)((uint32_t)(uint8_t)x ^ 0x80u)) - 4503599627370624.0;
}

// NJ > 0: a thread keeps its share of the residual slab in registers for the whole sweep -- the traits of its warp (w, w + 8, w + 16,
// w + 24) x the rows lane + 32 j, j < NJ (rows_per_cta <= 32 NJ) -- together with the observation bits of those rows: the dot products
// and the rank-one update of a marker touch no memory but the marker's genotype bytes.  NJ = 0: the slab lives in shared memory
// (row slabs above 512 rows).
template <int NJ>
__global__ void __launch_bounds__(kGT, 1) mrr_gen_sweep_kernel(MrrGenArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_abort;
  constexpr int NJR = NJ > 0 ? NJ : 1;
  const int k = a.k, rp = a.rows_per_cta, nmat = a.innergs ? 2 : 1, kk = k * k;
  const GenSmem s = carve(smem_raw, NJ > 0 ? 0 : k, rp, nmat, k);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, G = (int)gridDim.x, cta = blockIdx.x;
  const int64_t r0 = (int64_t)cta * rp;
  const int p = a.g.p;
  // slab of the residuals and of the observation mask
  double er[4][NJR];
  uint32_t zr[NJR];
  if constexpr (NJ > 0) {
#pragma unroll
    for (int j = 0; j < NJ; j++) {
      const int i = lane + 32 * j;
      const bool in = i < rp && r0 + i < a.g.ld;
      zr[j] = in ? a.zbits[r0 + i] : 0u;
#pragma unroll
      for (int q = 0; q < 4; q++) er[q][j] = (in && warp + 8 * q < k) ? a.e[(size_t)(warp + 8 * q) * a.g.ld + r0 + i] : 0.0;
    }
  } else {
    for (int q = tid; q < k * rp; q += kGT) {
      const int t = q / rp, i = q - t * rp;
      s.E[q] = (r0 + i < a.g.ld) ? a.e[(size_t)t * a.g.ld + r0 + i] : 0.0;
    }
    for (int i = tid; i < rp; i += kGT) s.zb[i] = (r0 + i < a.g.ld) ? a.zbits[r0 + i] : 0u;
  }
  if (tid < 32) s.irgs[tid] = (a.irgs && tid < k) ? a.irgs[tid] : tid;
  if (tid == 0) s_abort = 0;
  for (int q = tid; q < kGD * rp; q += kGT) s.xs[0][q] = 0;  // the four slots are contiguous
  double se = (warp == 0 && lane < k) ? a.se0[lane] : 0.0;  // running column sum of e_t over ALL rows (identical in every CTA)
  double sc4[4];  // fixed-point scale of this warp's traits; inverse scale of lane t's trait
#pragma unroll
  for (int q = 0; q < 4; q++) sc4[q] = (warp + 8 * q < k) ? a.scale[warp + 8 * q] : 0.0;
  const double inv_scale = lane < k ? a.scale[32 + lane] : 0.0;
  const int nch = rp / 16;
  int Jnext = 0;  // marker of the NEXT prefetch, read one step early so that its L2 round trip is not in front of the address arithmetic
  auto prefetch = [&](int m) {
    if (m < p) {
      const int J = Jnext, slot = m % kGD;
      if (m + 1 < p) Jnext = a.perm[m + 1];
      const int8_t* col = a.g.x8 + (int64_t)J * a.g.ld + r0;
      for (int c = tid; c < nch; c += kGT)
        if (r0 + 16 * c < a.g.ld) cp_async16(s.xs[slot] + 16 * c, col + 16 * c);  // rows past the padded column stay as they are: e = z = 0 there
      const double* src = a.sol + (size_t)J * nmat * kk;
      for (int c = tid; c < nmat * kk; c += kGT) cp_async8(s.mats[slot] + c, src + c);
      if (tid < 2 * k) cp_async8(s.vec[slot] + tid, a.fixed + (size_t)J * 2 * k + tid);
      else if (tid < 3 * k) cp_async8(s.vec[slot] + tid, a.b + (size_t)J * k + (tid - 2 * k));
      else if (tid == 3 * k) cp_async8(s.vec[slot] + 3 * k, a.mean + J);
      if (tid == 0) s.Js[slot] = J;
    }
    cp_async_commit();
  };
  Jnext = a.perm[0];
  __syncthreads();  // the zeroed ring slots are in place before any cp.async lands in them
  for (int m = 0; m < kGD - 1; m++) prefetch(m);
  const unsigned long long t_start = globaltimer_ns();
  for (int m = 0; m < p; m++) {
    cp_async_wait<kGD - 2>();
    __syncthreads();  // marker m's slot has landed for every thread; step m - 1 is finished by every thread
    prefetch(m + kGD - 1);
    const int slot = m % kGD;
    const int8_t* xs = s.xs[slot];
    const double* vec = s.vec[slot];
    const double* mats = s.mats[slot];
    // ---- slab dot products x'e_t: warp w takes traits w, w + 8, w + 16, w + 24
    double xr[NJR];
    {
      double acc[4] = {0.0, 0.0, 0.0, 0.0};
      if constexpr (NJ > 0) {
#pragma unroll
        for (int j = 0; j < NJ; j++) {
          const int i = lane + 32 * j;
          xr[j] = i < rp ? byte_to_double(xs[i]) : 0.0;
#pragma unroll
          for (int q = 0; q < 4; q++) acc[q] = fma(xr[j], er[q][j], acc[q]);
        }
      } else {
        for (int i = lane; i < rp; i += 32) {
          const double x = byte_to_double(xs[i]);
#pragma unroll
          for (int q = 0; q < 4; q++) {
            const int t = warp + 8 * q;
            if (t < k) acc[q] = fma(x, s.E[t * rp + i], acc[q]);
          }
        }
      }
      unsigned long long* accw = a.acc + ((size_t)m * kGridCopies + (cta & (kGridCopies - 1))) * 32;
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const int t = warp + 8 * q;
        if (t < k) {
          const double v = warp_sum(acc[q]) * sc4[q];
          if (lane == 0) grid_add(accw + t, v, a.err);
        }
      }
    }
    if (warp == 0) {
      const bool on = lane < k;
      const long long tot = grid_wait_total(a.acc + (size_t)m * kGridCopies * 32 + (on ? lane : 0), on, G, a.err, t_start, &s_abort);
      const double dot = (double)tot * inv_scale;
      const double XXt = on ? vec[lane] : 0.0, sxzc = on ? vec[k + lane] : 0.0, b0 = on ? vec[2 * k + lane] : 0.0;
      const double mean = vec[3 * k];
      const double r = on ? dot - mean * se + XXt * b0 : 0.0;  // x_c'e_t + XX(J,t) b0_t  (:506)
      double b1 = 0.0;
      if (!a.innergs) {
        for (int c = 0; c < k; c++) {
          const double rc = shfl_d(r, c);
          if (on) b1 = fma(mats[lane * k + c], rc, b1);
        }
      } else {
        double RHS = 0.0;
        for (int c = 0; c < k; c++) {
          const double rc = shfl_d(r, c);
          if (on) RHS = fma(mats[kk + lane * k + c], rc, RHS);
        }
        b1 = b0;
        for (int i = 0; i < k; i++) {  // :511-514, in the sweep's inner order
          const int ri = s.irgs[i];
          const double sdot = warp_sum(on ? mats[lane * k + ri] * b1 : 0.0);  // LHS.col(ri) . b1
          const double bri = shfl_d(b1, ri), Rri = shfl_d(RHS, ri), dg = mats[ri * k + ri];
          const double nb = (Rri - sdot + dg * bri) / dg;
          if (lane == ri) b1 = nb;
        }
      }
      if (on) {
        const double dlt = b1 - b0;
        s.dl[lane] = dlt;
        se -= dlt * sxzc;  // sum_i (x_iJ - mean_J) z_it
        if (cta == 0) a.b[(size_t)s.Js[slot] * k + lane] = b1;
      }
    }
    __syncthreads();
    if (s_abort) return;  // the host reports the error flag; the residuals of this launch are not written back
    // ---- e_t -= (x - mean) (b1_t - b0_t) on the observed rows (:518)
    {
      const double mean = vec[3 * k];
      double dl[4];
#pragma unroll
      for (int q = 0; q < 4; q++) dl[q] = (warp + 8 * q < k) ? s.dl[warp + 8 * q] : 0.0;
      if constexpr (NJ > 0) {
#pragma unroll
        for (int j = 0; j < NJ; j++) {
          const double x = xr[j] - mean;
#pragma unroll
          for (int q = 0; q < 4; q++) er[q][j] = fma(-x, ((zr[j] >> (warp + 8 * q)) & 1u) ? dl[q] : 0.0, er[q][j]);
        }
      } else {
        for (int i = lane; i < rp; i += 32) {
          const double x = byte_to_double(xs[i]) - mean;
          const uint32_t zb = s.zb[i];
          double ev[4];
#pragma unroll
          for (int q = 0; q < 4; q++) ev[q] = (warp + 8 * q < k) ? s.E[(warp + 8 * q) * rp + i] : 0.0;
#pragma unroll
          for (int q = 0; q < 4; q++) ev[q] = fma(-x, ((zb >> (warp + 8 * q)) & 1u) ? dl[q] : 0.0, ev[q]);
#pragma unroll
          for (int q = 0; q < 4; q++)
            if (warp + 8 * q < k) s.E[(warp + 8 * q) * rp + i] = ev[q];
        }
      }
    }
  }
  cp_async_wait<0>();
  __syncthreads();
  if constexpr (NJ > 0) {
#pragma unroll
    for (int j = 0; j < NJ; j++) {
      const int i = lane + 32 * j;
      if (i < rp && r0 + i < a.g.ld) {
#pragma unroll
        for (int q = 0; q < 4; q++)
          if (warp + 8 * q < k) a.e[(size_t)(warp + 8 * q) * a.g.ld + r0 + i] = er[q][j];
      }
    }
  } else {
    for (int q = tid; q < k * rp; q += kGT) {
      const int t = q / rp, i = q - t * rp;
      if (r0 + i < a.g.ld) a.e[(size_t)t * a.g.ld + r0 + i] = s.E[q];
    }
  }
}

// out[t] = sum_i A[t][i] * (B ? B[t][i] : 1)   (matrices [k][ld], float64; one CTA per trait, fixed order)
__global__ void __launch_bounds__(256) mrr_gen_colred_kernel(const double* __restrict__ A, const double* __restrict__ B, int64_t ld,
                                                             int n, double* __restrict__ out) {
  __shared__ double sh[8];
  const int t = blockIdx.x, tid = threadIdx.x;
  const double* a = A + (size_t)t * ld;
  const double* b = B ? B + (size_t)t * ld : nullptr;
  double s = 0.0;
  for (int i = tid; i < n; i += 256) s += b ? a[i] * b[i] : a[i];
  s = warp_sum(s);
  if ((tid & 31) == 0) sh[tid >> 5] = s;
  __syncthreads();
  if (tid == 0) {
    double r = 0.0;
    for (int w = 0; w < 8; w++) r += sh[w];
    out[t] = r;
  }
}

// [p][k] reductions of the sweep epilogue.  mode 0: out[i*k + j] = sum_m A[m][i] * B[m][j] * (C ? C[m][j] : 1)  (b' tilde, :549, or
// b' (Dinv o tilde), :547);  mode 1: out[i] = sum_m (A[m][i] - B[m][i])^2 (:662);  mode 2 (TH, :543-545): C[m][i] =
// 1 / (A[m][i] / par[i] + par[k + i]) written, out[i] = sum_m A[m][i] * C[m][i]
__global__ void __launch_bounds__(256) mrr_gen_pk_kernel(int mode, const double* __restrict__ A, const double* __restrict__ B,
                                                         double* __restrict__ Cm, const double* __restrict__ par, int p, int k,
                                                         double* __restrict__ out) {
  __shared__ double sh[8];
  const int i = blockIdx.x, j = blockIdx.y, tid = threadIdx.x;
  double s = 0.0;
  for (int m = tid; m < p; m += 256) {
    if (mode == 0) {
      const double w = B[(size_t)m * k + j] * (Cm ? Cm[(size_t)m * k + j] : 1.0);
      s = fma(A[(size_t)m * k + i], w, s);
    } else if (mode == 1) {
      const double d = A[(size_t)m * k + i] - B[(size_t)m * k + i];
      s = fma(d, d, s);
    } else {
      const double x = A[(size_t)m * k + i];
      const double dv = 1.0 / (x / par[i] + par[k + i]);
      Cm[(size_t)m * k + i] = dv;
      s = fma(x, dv, s);
    }
  }
  s = warp_sum(s);
  if ((tid & 31) == 0) sh[tid >> 5] = s;
  __syncthreads();
  if (tid == 0) {
    double r = 0.0;
    for (int w = 0; w < 8; w++) r += sh[w];
    out[mode == 0 ? i * k + j : i] = r;
  }
}

// e_t = (e_t - shift_t) on the observed rows (updateMu, :651-655)
__global__ void __launch_bounds__(256) mrr_gen_shift_kernel(double* __restrict__ e, const uint32_t* __restrict__ zbits, int64_t ld,
                                                            int n, int k, const double* __restrict__ shift) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const uint32_t zb = zbits[i];
  for (int t = 0; t < k; t++)
    if ((zb >> t) & 1u) e[(size_t)t * ld + i] -= shift[t];
}

}  // namespace

size_t mrr_gen_smem(int k, int rows_per_cta, int innergs) {
  const int nmat = innergs ? 2 : 1;
  size_t o = (rows_per_cta <= 512 ? 0 : sizeof(double) * (size_t)k * rows_per_cta) + sizeof(double) * 32;
  o += (size_t)kGD * sizeof(double) * ((size_t)nmat * k * k + 3 * k + 1);
  o = (o + 15) & ~(size_t)15;
  o += (size_t)kGD * rows_per_cta + sizeof(uint32_t) * (size_t)rows_per_cta + sizeof(int) * (kGD + 32);
  return o + 16;
}

void launch_mrr_gen_colstats(const GenoView& g, const uint32_t* zbits, const double* y, int k, double* sxz, double* sxxz,
                             double* xty, cudaStream_t st) {
  mrr_gen_colstats_kernel<<<(g.p + 7) / 8, 256, 0, st>>>(g, zbits, y, k, sxz, sxxz, xty);
}

void launch_mrr_gen_systems(int p, int k, const double* fixed, const double* W, const double* iG, const double* vb,
                            const double* iVe, int noinv_system, int innergs, double* sol, cudaStream_t st) {
  mrr_gen_systems_kernel<<<p, 32, 0, st>>>(p, k, 2 * k, fixed, W, iG, vb, iVe, noinv_system, innergs, sol);
}

cudaError_t launch_mrr_gen_sweep(const MrrGenArgs& a, int grid, cudaStream_t st) {
  const size_t smem = mrr_gen_smem(a.k, a.rows_per_cta, a.innergs);
  const int nj = (a.rows_per_cta + 31) / 32;
  const void* fn = nj <= 2    ? reinterpret_cast<const void*>(mrr_gen_sweep_kernel<2>)
                   : nj <= 4  ? reinterpret_cast<const void*>(mrr_gen_sweep_kernel<4>)
                   : nj <= 8  ? reinterpret_cast<const void*>(mrr_gen_sweep_kernel<8>)
                   : nj <= 12 ? reinterpret_cast<const void*>(mrr_gen_sweep_kernel<12>)
                   : nj <= 16 ? reinterpret_cast<const void*>(mrr_gen_sweep_kernel<16>)
                              : reinterpret_cast<const void*>(mrr_gen_sweep_kernel<0>);
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  MrrGenArgs args = a;
  void* params[] = {&args};
  return cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kGT), params, smem, st);
}

void launch_mrr_gen_colred(const double* A, const double* B, int64_t ld, int n, int k, double* out, cudaStream_t st) {
  mrr_gen_colred_kernel<<<k, 256, 0, st>>>(A, B, ld, n, out);
}

void launch_mrr_gen_pk(int mode, const double* A, const double* B, double* C, const double* par, int p, int k, double* out,
                       cudaStream_t st) {
  mrr_gen_pk_kernel<<<dim3(k, mode == 0 ? k : 1), 256, 0, st>>>(mode, A, B, C, par, p, k, out);
}

void launch_mrr_gen_shift(double* e, const uint32_t* zbits, int64_t ld, int n, int k, const double* shift, cudaStream_t st) {
  mrr_gen_shift_kernel<<<(n + 255) / 256, 256, 0, st>>>(e, zbits, ld, n, k, shift);
}

}  // namespace bwgr
