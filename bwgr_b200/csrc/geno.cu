// geno.cu -- genotype store kernels: packing (f64 -> int8 -> 2-bit), unpack, integer-exact column
// statistics (K4 of SURVEY 2c; replaces xx[j]=squaredNorm / fvar at Rcpp20260726ai.cpp:312-316) and
// the final GEBV pass hat = mu + X b (K10; :346).  All HBM-bound streaming kernels: 16-byte
// vector loads, one column per CTA (stats) or a row tile x column split per CTA (gemv).
#include "kernels.h"

namespace bwgr {

__global__ void pack_f64_kernel(const double* __restrict__ src, int64_t ld_src, int n, int pc, int8_t* __restrict__ dst,
                                int64_t ld, int lo, int hi, int* bad) {
  const int j = blockIdx.x;
  const double* s = src + (int64_t)j * ld_src;
  int8_t* d = dst + (int64_t)j * ld;
  for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < ld; i += gridDim.y * blockDim.x) {
    int8_t v = 0;
    if (i < n) {
      const double x = s[i];
      const double r = rint(x);
      if (!(x == r) || r < (double)lo || r > (double)hi) atomicExch(bad, 1);
      else v = (int8_t)(int)r;
    }
    d[i] = v;
  }
}
void launch_pack_f64(const double* src, int64_t ld_src, int n, int pc, int8_t* dst, int64_t ld, int lo, int hi, int* bad,
                     cudaStream_t st) {
  dim3 grid((unsigned)pc, (unsigned)((ld + 1023) / 1024 > 64 ? 64 : (ld + 1023) / 1024));  // columns on x (p can exceed the 65,535 limit of y)
  pack_f64_kernel<<<grid, 256, 0, st>>>(src, ld_src, n, pc, dst, ld, lo, hi, bad);
}

// PLINK .bed (variant-major): column j = ceil(n/4) bytes, sample i in bits 2*(i%4) of byte i/4: 00 = two copies of allele A1, 10 = one,
// 11 = none, 01 = missing.  Decoded to the additive count of A1 (what `plink --recode A` writes).  missing: 0..2 = that code,
// -2 = the rounded mean of the column's observed codes (integer stand-in for IMP, Rcpp20260726ai.cpp:1316-1335), -1 = an error (*bad).
// nmiss += the number of missing calls.
__global__ void __launch_bounds__(256) decode_bed_kernel(const uint8_t* __restrict__ bed, int64_t bpc, int n, int8_t* __restrict__ dst, int64_t ld,
                                                         int missing, int* bad, unsigned long long* nmiss) {
  __shared__ int s_sum, s_cnt, s_fill;
  const uint8_t* col = bed + (int64_t)blockIdx.x * bpc;
  int8_t* d = dst + (int64_t)blockIdx.x * ld;
  if (threadIdx.x == 0) { s_sum = 0; s_cnt = 0; s_fill = missing >= 0 ? missing : 0; }
  __syncthreads();
  int sum = 0, cnt = 0, miss = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int c = (col[i >> 2] >> (2 * (i & 3))) & 3;
    if (c == 1) miss++;
    else { sum += c == 0 ? 2 : c == 2 ? 1 : 0; cnt++; }
  }
  if (miss) {
    atomicAdd(nmiss, (unsigned long long)miss);
    if (missing == -1) atomicExch(bad, 1);
  }
  if (missing == -2) {
    atomicAdd(&s_sum, sum); atomicAdd(&s_cnt, cnt);
    __syncthreads();
    if (threadIdx.x == 0) s_fill = s_cnt > 0 ? (int)rintf((float)s_sum / (float)s_cnt) : 0;
    __syncthreads();
  }
  const int fill = s_fill;
  for (int i = threadIdx.x; i < ld; i += blockDim.x) {
    int v = 0;
    if (i < n) {
      const int c = (col[i >> 2] >> (2 * (i & 3))) & 3;
      v = c == 0 ? 2 : c == 2 ? 1 : c == 3 ? 0 : fill;
    }
    d[i] = (int8_t)v;
  }
}
void launch_decode_bed(const uint8_t* bed, int64_t bytes_per_col, int n, int p, int8_t* dst, int64_t ld, int missing, int* bad,
                       unsigned long long* nmiss, cudaStream_t st) {
  decode_bed_kernel<<<(unsigned)p, 256, 0, st>>>(bed, bytes_per_col, n, dst, ld, missing, bad, nmiss);
}

__global__ void check_range_kernel(const int8_t* __restrict__ src, int64_t ld, int n, int lo, int hi, int* bad) {
  const int8_t* s = src + (int64_t)blockIdx.x * ld;
  for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < n; i += gridDim.y * blockDim.x) {
    const int v = s[i];
    if (v < lo || v > hi) atomicExch(bad, 1);
  }
}
void launch_check_range_i8(const int8_t* src, int64_t ld, int n, int p, int lo, int hi, int* bad, cudaStream_t st) {
  dim3 grid((unsigned)p, (unsigned)((n + 1023) / 1024 > 64 ? 64 : (n + 1023) / 1024));  // columns on x (p can exceed the 65,535 limit of y)
  check_range_kernel<<<grid, 256, 0, st>>>(src, ld, n, lo, hi, bad);
}

__global__ void zero_pad_kernel(int8_t* x, int64_t ld, int n) {
  int8_t* c = x + (int64_t)blockIdx.x * ld;
  for (int i = n + threadIdx.x; i < ld; i += blockDim.x) c[i] = 0;
}
void launch_zero_pad(int8_t* x, int64_t ld, int n, int p, cudaStream_t st) {
  if (ld > n) zero_pad_kernel<<<p, 128, 0, st>>>(x, ld, n);
}

// 2-bit packing: byte k of a column holds rows 4k..4k+3, row r in bits 2*(r%4).
__global__ void pack_2bit_kernel(const int8_t* __restrict__ src, int64_t ld, int n, uint8_t* __restrict__ dst,
                                 int64_t ldb, int* bad) {
  const int8_t* s = src + (int64_t)blockIdx.x * ld;
  uint8_t* d = dst + (int64_t)blockIdx.x * ldb;
  for (int k = blockIdx.y * blockDim.x + threadIdx.x; k < ldb; k += gridDim.y * blockDim.x) {
    uint32_t byte = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const int r = 4 * k + q;
      int v = 0;
      if (r < n) {
        v = s[r];
        if (v < 0 || v > 2) { atomicExch(bad, 1); v = 0; }
      }
      byte |= (uint32_t)v << (2 * q);
    }
    d[k] = (uint8_t)byte;
  }
}
void launch_pack_2bit(const int8_t* src, int64_t ld, int n, int p, uint8_t* dst, int64_t ldb, int* bad, cudaStream_t st) {
  dim3 grid((unsigned)p, (unsigned)((ldb + 255) / 256 > 64 ? 64 : (ldb + 255) / 256));  // columns on x (p can exceed the 65,535 limit of y)
  pack_2bit_kernel<<<grid, 256, 0, st>>>(src, ld, n, dst, ldb, bad);
}
// Gram shadow copy: 16 rows per 32-bit word, interleaved so that the kernel expands it with one shift and one mask per
// output word: the code of row 16g + 4q + k sits at bits [8k + 2q, 8k + 2q + 1], i.e. (w >> 2q) & 0x03030303 is the four
// bytes of rows 4q .. 4q+3.  Codes must be 0..3 (else *bad).
__global__ void pack_2bit_gram_kernel(const int8_t* __restrict__ src, int64_t ld, uint32_t* __restrict__ dst, int64_t ldw,
                                      int* bad) {
  const uint4* s = reinterpret_cast<const uint4*>(src + (int64_t)blockIdx.x * ld);
  uint32_t* d = dst + (int64_t)blockIdx.x * ldw;
  for (int64_t g = blockIdx.y * blockDim.x + threadIdx.x; g < ldw; g += (int64_t)gridDim.y * blockDim.x) {
    const uint4 v = s[g];  // rows 16g .. 16g+15 (pad rows are zero)
    const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
    uint32_t out = 0, any = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      any |= w4[q] & 0xFCFCFCFCu;
      out |= (w4[q] & 0x03030303u) << (2 * q);
    }
    if (any) atomicExch(bad, 1);
    d[g] = out;
  }
}
void launch_pack_2bit_gram(const int8_t* src, int64_t ld, int p, uint8_t* dst, int* bad, cudaStream_t st) {
  const int64_t ldw = ld / 16;
  dim3 grid((unsigned)p, (unsigned)((ldw + 255) / 256 > 64 ? 64 : (ldw + 255) / 256));  // columns on x (p can exceed the 65,535 limit of y)
  pack_2bit_gram_kernel<<<grid, 256, 0, st>>>(src, ld, reinterpret_cast<uint32_t*>(dst), ldw, bad);
}
__global__ void unpack_2bit_kernel(const uint8_t* __restrict__ src, int64_t ldb, int n, int8_t* __restrict__ dst,
                                   int64_t ld) {
  const uint8_t* s = src + (int64_t)blockIdx.x * ldb;
  int8_t* d = dst + (int64_t)blockIdx.x * ld;
  for (int r = blockIdx.y * blockDim.x + threadIdx.x; r < ld; r += gridDim.y * blockDim.x)
    d[r] = (r < n) ? (int8_t)((s[r >> 2] >> (2 * (r & 3))) & 3) : (int8_t)0;
}
void launch_unpack_2bit(const uint8_t* src, int64_t ldb, int n, int p, int8_t* dst, int64_t ld, cudaStream_t st) {
  dim3 grid((unsigned)p, (unsigned)((ld + 1023) / 1024 > 64 ? 64 : (ld + 1023) / 1024));  // columns on x (p can exceed the 65,535 limit of y)
  unpack_2bit_kernel<<<grid, 256, 0, st>>>(src, ldb, n, dst, ld);
}

// Column statistics, one CTA per column, dp4a for sum and sum of squares (int32 partials are safe:
// 127^2 * 16 rows per lane-iteration, promoted to int64 before the block reduction).
template <bool MASKED>
__global__ void __launch_bounds__(256) col_stats_kernel(GenoView g, const uint8_t* __restrict__ mask, long long* xx,
                                                        long long* sx) {
  const int j = blockIdx.x;
  long long s1 = 0, s2 = 0;
  if (g.storage == 0) {
    const uint4* col = reinterpret_cast<const uint4*>(g.x8 + (int64_t)j * g.ld);
    const int nv = (int)(g.ld >> 4);
    for (int v = threadIdx.x; v < nv; v += blockDim.x) {
      uint4 w = __ldg(col + v);
      if (MASKED) {  // mask bytes are 0/1; 0x01*0xFF = 0xFF selects the genotype byte
        const uint4 m = __ldg(reinterpret_cast<const uint4*>(mask) + v);
        w.x &= m.x * 0xFFu; w.y &= m.y * 0xFFu; w.z &= m.z * 0xFFu; w.w &= m.w * 0xFFu;
      }
      int a = 0, q = 0;
      a = __dp4a((int)w.x, 0x01010101, a); a = __dp4a((int)w.y, 0x01010101, a);
      a = __dp4a((int)w.z, 0x01010101, a); a = __dp4a((int)w.w, 0x01010101, a);
      q = __dp4a((int)w.x, (int)w.x, q); q = __dp4a((int)w.y, (int)w.y, q);
      q = __dp4a((int)w.z, (int)w.z, q); q = __dp4a((int)w.w, (int)w.w, q);
      s1 += a; s2 += q;
    }
  } else {
    const uint8_t* col = g.x2 + (int64_t)j * g.ldb;
    for (int k = threadIdx.x; k < g.ldb; k += blockDim.x) {
      const uint32_t byte = col[k];
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const int r = 4 * k + q;
        int v = (byte >> (2 * q)) & 3;
        if (MASKED && r < g.n && !mask[r]) v = 0;
        s1 += v; s2 += v * v;
      }
    }
  }
  __shared__ long long r1[8], r2[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if ((threadIdx.x & 31) == 0) { r1[threadIdx.x >> 5] = s1; r2[threadIdx.x >> 5] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    long long a = 0, q = 0;
    for (int w = 0; w < 8; w++) { a += r1[w]; q += r2[w]; }
    sx[j] = a; xx[j] = q;
  }
}
void launch_col_stats(const GenoView& g, long long* xx, long long* sx, cudaStream_t st) {
  col_stats_kernel<false><<<g.p, 256, 0, st>>>(g, nullptr, xx, sx);
}
void launch_col_stats_masked(const GenoView& g, const uint8_t* mask, long long* xx, long long* sx, cudaStream_t st) {
  col_stats_kernel<true><<<g.p, 256, 0, st>>>(g, mask, xx, sx);
}

// float32 store: xx_j = sum x^2, sx_j = sum x in double, fixed order (one CTA per marker)
__global__ void __launch_bounds__(256) col_stats_f32_kernel(GenoView g, const uint8_t* __restrict__ mask, double* __restrict__ xx,
                                                            double* __restrict__ sx) {
  __shared__ double sh1[8], sh2[8];
  const int j = blockIdx.x, tid = threadIdx.x;
  const float* col = g.xf + (int64_t)j * g.ld;
  double s1 = 0, s2 = 0;
  for (int i = tid; i < g.n; i += 256) {
    if (mask && !mask[i]) continue;
    const double v = (double)col[i];
    s1 += v; s2 += v * v;
  }
  s1 = warp_sum(s1); s2 = warp_sum(s2);
  if ((tid & 31) == 0) { sh1[tid >> 5] = s1; sh2[tid >> 5] = s2; }
  __syncthreads();
  if (tid == 0) {
    double a = 0, c = 0;
    for (int w = 0; w < 8; w++) { a += sh1[w]; c += sh2[w]; }
    sx[j] = a; xx[j] = c;
  }
}
void launch_col_stats_f32(const GenoView& g, const uint8_t* mask, double* xx, double* sx, cudaStream_t st) {
  col_stats_f32_kernel<<<g.p, 256, 0, st>>>(g, mask, xx, sx);
}
// Row multiplicities (KMUP2 on rows sampled with replacement, R/wgr.R:68 with rp = TRUE): xx_j = sum_i c_i x_ij^2, sx_j = sum_i c_i x_ij
// for any store, in double (exact for the integer stores: every partial sum is an integer below 2^53).  One CTA per marker.
__global__ void __launch_bounds__(256) col_stats_cnt_kernel(GenoView g, const uint8_t* __restrict__ cnt, double* __restrict__ xx,
                                                            double* __restrict__ sx) {
  __shared__ double sh1[8], sh2[8];
  const int j = blockIdx.x, tid = threadIdx.x;
  double s1 = 0, s2 = 0;
  for (int i = tid; i < g.n; i += 256) {
    const double c = (double)cnt[i];
    if (c == 0.0) continue;
    double v;
    if (g.storage == 0) v = (double)g.x8[(int64_t)j * g.ld + i];
    else if (g.storage == 1) v = (double)((g.x2[(int64_t)j * g.ldb + (i >> 2)] >> (2 * (i & 3))) & 3);
    else v = (double)g.xf[(int64_t)j * g.ld + i];
    s1 += c * v; s2 += c * v * v;
  }
  s1 = warp_sum(s1); s2 = warp_sum(s2);
  if ((tid & 31) == 0) { sh1[tid >> 5] = s1; sh2[tid >> 5] = s2; }
  __syncthreads();
  if (tid == 0) {
    double a = 0, c = 0;
    for (int w = 0; w < 8; w++) { a += sh1[w]; c += sh2[w]; }
    sx[j] = a; xx[j] = c;
  }
}
void launch_col_stats_cnt(const GenoView& g, const uint8_t* cnt, double* xx, double* sx, cudaStream_t st) {
  col_stats_cnt_kernel<<<g.p, 256, 0, st>>>(g, cnt, xx, sx);
}
__global__ void __launch_bounds__(256) d_to_float_kernel(const double* __restrict__ src, float* __restrict__ dst, int n) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < n) dst[i] = (float)src[i];
}
void launch_d_to_float(const double* src, float* dst, int n, cudaStream_t st) { d_to_float_kernel<<<(n + 255) / 256, 256, 0, st>>>(src, dst, n); }

// hat[t] = mu[t] + X b_t for k systems with one stream of X.
// Split `y` of a column split takes the columns j = y, y + splits, ...; every row's partial sum of a system runs over them in increasing j
// as one FMA chain, and a second kernel adds the splits in a fixed order (deterministic; k = 1 is the single-system fitted values).
// A row's chain does not depend on which thread holds the row or on the other systems, so a thread takes R rows x KC systems:
// each genotype is converted once and used KC times, each b_tj (staged in shared memory, kHatCols columns of the split at a time) R times.
// CTAs of the same (row tile, split) and consecutive system chunks are adjacent in launch order (blockIdx.x = chunk): they read the
// same X tile at about the same time, so HBM serves it once and L2 the rest.
// A zero b_tj is not skipped: acc starts at +0 and an FMA never turns it into -0, so fmaf(x, 0, acc) == acc for every finite x.
constexpr int kHatCols = 128;
constexpr int kHatThreads = 256;

template <int R>
__device__ __forceinline__ void hat_rows(const GenoView& g, int64_t j, int64_t row0, float (&x)[R]) {
  static_assert(R == 4 || R == 16, "rows per thread");
  if (g.storage == 2) {  // float32 store
    const float4* v = reinterpret_cast<const float4*>(g.xf + j * g.ld + row0);
#pragma unroll
    for (int q = 0; q < R / 4; q++) {
      const float4 f = __ldg(v + q);
      x[4 * q + 0] = f.x; x[4 * q + 1] = f.y; x[4 * q + 2] = f.z; x[4 * q + 3] = f.w;
    }
    return;
  }
  uint32_t w[R / 4];
  if (g.storage == 0) {
    if constexpr (R == 16) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(g.x8 + j * g.ld + row0));
      w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    } else {
      w[0] = __ldg(reinterpret_cast<const uint32_t*>(g.x8 + j * g.ld + row0));
    }
  } else {  // 2-bit store: R / 4 packed bytes
    uint32_t pk;
    if constexpr (R == 16) pk = __ldg(reinterpret_cast<const uint32_t*>(g.x2 + j * g.ldb + (row0 >> 2)));
    else pk = __ldg(g.x2 + j * g.ldb + (row0 >> 2));
    const uint4 v = expand_2bit(pk);
    w[0] = v.x;
    if constexpr (R == 16) { w[1] = v.y; w[2] = v.z; w[3] = v.w; }
  }
#pragma unroll
  for (int q = 0; q < R / 4; q++) {
    const uint32_t xw = w[q] ^ 0x80808080u;
#pragma unroll
    for (int t = 0; t < 4; t++) x[4 * q + t] = byte_to_float(xw, t);
  }
}

// work[t][y][row] = sum over the columns of split y of x_row,j b_tj, for the KC systems of chunk blockIdx.x
template <int R, int KC>
__global__ void __launch_bounds__(kHatThreads) gemv_hat_partial_kernel(GenoView g, const float* __restrict__ b, int k,
                                                                      float* __restrict__ work, int splits) {
  static_assert(KC == 1 || KC % 4 == 0, "systems per thread");
  __shared__ __align__(16) float bs[KC == 1 ? 1 : kHatCols][KC];
  const int t0 = blockIdx.x * KC, split = blockIdx.z;
  const int64_t row0 = ((int64_t)blockIdx.y * kHatThreads + threadIdx.x) * R;
  const bool live = row0 < g.ld;  // KC > 1: no early return, the thread takes part in staging b
  float acc[R][KC];
#pragma unroll
  for (int r = 0; r < R; r++)
#pragma unroll
    for (int t = 0; t < KC; t++) acc[r][t] = 0.0f;
  if constexpr (KC == 1) {  // one system: b_j read in place, zero effects cost no load
    if (!live) return;
    for (int64_t j = split; j < g.p; j += splits) {
      const float bj = __ldg(b + j);
      if (bj == 0.0f) continue;
      float x[R];
      hat_rows<R>(g, j, row0, x);
#pragma unroll
      for (int r = 0; r < R; r++) acc[r][0] = fmaf(x[r], bj, acc[r][0]);
    }
    float* out = work + (int64_t)split * g.ld + row0;
#pragma unroll
    for (int q = 0; q < R; q += 4) *reinterpret_cast<float4*>(out + q) = make_float4(acc[q][0], acc[q + 1][0], acc[q + 2][0], acc[q + 3][0]);
  } else {
    const int ncol = (g.p - split + splits - 1) / splits;
    for (int m0 = 0; m0 < ncol; m0 += kHatCols) {
      const int mc = min(kHatCols, ncol - m0);
      __syncthreads();  // the previous columns' b are consumed
      for (int q = threadIdx.x; q < kHatCols * KC; q += kHatThreads) {
        const int t = q / kHatCols, m = q - t * kHatCols;
        bs[m][t] = (m < mc && t0 + t < k) ? __ldg(b + (int64_t)(t0 + t) * g.p + split + (int64_t)splits * (m0 + m)) : 0.0f;
      }
      __syncthreads();
      if (!live) continue;
#pragma unroll 2
      for (int m = 0; m < mc; m++) {
        float x[R];
        hat_rows<R>(g, split + (int64_t)splits * (m0 + m), row0, x);
#pragma unroll
        for (int t4 = 0; t4 < KC; t4 += 4) {
          const float4 bt = *reinterpret_cast<const float4*>(&bs[m][t4]);
#pragma unroll
          for (int r = 0; r < R; r++) {
            acc[r][t4 + 0] = fmaf(x[r], bt.x, acc[r][t4 + 0]); acc[r][t4 + 1] = fmaf(x[r], bt.y, acc[r][t4 + 1]);
            acc[r][t4 + 2] = fmaf(x[r], bt.z, acc[r][t4 + 2]); acc[r][t4 + 3] = fmaf(x[r], bt.w, acc[r][t4 + 3]);
          }
        }
      }
    }
    if (!live) return;
#pragma unroll
    for (int t = 0; t < KC; t++) {
      if (t0 + t >= k) break;
      float* out = work + ((int64_t)(t0 + t) * splits + split) * g.ld + row0;
#pragma unroll
      for (int q = 0; q < R; q += 4) *reinterpret_cast<float4*>(out + q) = make_float4(acc[q][t], acc[q + 1][t], acc[q + 2][t], acc[q + 3][t]);
    }
  }
}


__global__ void __launch_bounds__(256) gemv_hat_reduce_kernel(const float* __restrict__ work, int64_t ld, int n, int splits,
                                                              const float* __restrict__ mu, float* __restrict__ hat) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, t = blockIdx.y;
  if (i >= n) return;
  const float* w = work + (int64_t)t * splits * ld + i;
  float s = 0.0f;
  for (int y = 0; y < splits; y++) s += w[(int64_t)y * ld];
  hat[(int64_t)t * ld + i] = s + mu[t];
}

template <int R, int KC>
static void launch_hat_partial(const GenoView& g, const float* b, int k, float* work, int splits, cudaStream_t st) {
  const int rows = kHatThreads * R;
  dim3 grid((unsigned)((k + KC - 1) / KC), (unsigned)((g.ld + rows - 1) / rows), (unsigned)splits);
  gemv_hat_partial_kernel<R, KC><<<grid, kHatThreads, 0, st>>>(g, b, k, work, splits);
}

void launch_gemv_hat(const GenoView& g, const float* b, int k, const float* mu, float* hat, float* work, int splits, cudaStream_t st) {
  if (k == 1) launch_hat_partial<16, 1>(g, b, k, work, splits, st);
  else if (k <= 4) launch_hat_partial<16, 4>(g, b, k, work, splits, st);
  else launch_hat_partial<4, kHatChunk>(g, b, k, work, splits, st);
  gemv_hat_reduce_kernel<<<dim3((unsigned)((g.n + 255) / 256), (unsigned)k), 256, 0, st>>>(work, g.ld, g.n, splits, mu, hat);
}

}  // namespace bwgr
