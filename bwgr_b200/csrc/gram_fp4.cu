// gram_fp4.cu -- the Gram band [X_b'X_b | X_{b-1}'X_b] of a sweep on the block-scaled FP4 tensor-core path.
//
// When every genotype is a code 0, 1 or 2 (SimZ / tpod / any biallelic SNP matrix) the codes are exact in E2M1 (0 -> 0x0,
// 1 -> 0x2, 2 -> 0x4), products are 0, 1, 2 or 4 and the fp32 sums stay below 2^24 (checked at load time: max_j xx_j < 2^24),
// so tcgen05.mma kind::mxf4 with every block scale = 2^0 gives the EXACT integer Gram at twice the E4M3 rate and half the
// shared-memory bytes per row (gram_tc.cu is bound by the shared-memory pipe, not by the tensor pipe).
//
// Per block b of 128 markers ONE instruction shape: M = 128 (markers of block b), N = 256 (markers of block b | block b + 1),
// K = 64 genotype rows:  D = X_b' [X_b | X_{b+1}]  -> columns 0..127 are the diagonal block of b, columns 128..255 are row-for-row
// the cross block the sweep's look-ahead needs for block b + 1 (row r = marker r of block b, column c = marker c of block b + 1),
// written into block b + 1's band -- the same [p/128][128][256] float layout gram_tc.cu produces.
//
// Source: a packed 2-bit shadow copy (`launch_pack_2bit_fp4`): word k of a column holds rows 16k .. 16k+15, nibble i = rows
// 16k + i (low two bits) and 16k + 8 + i (high two bits), so the E2M1 nibbles of rows 16k..16k+7 are (w & 0x33333333) << 1 and
// those of rows 16k+8..16k+15 are (w >> 1) & 0x66666666: two ALU operations per eight rows, 0.25 bytes per genotype from HBM.
//
// Warp roles (672 threads): warps 0-3 and 9-20 (512 producers) expand packed chunks into the K-major SWIZZLE_128B tiles (a 128-byte
// tile row = 256 genotype rows of one marker), six stages of loads in flight per thread (the gather is DRAM-latency-bound: with 256
// producers and four stages the kernel took 0.41 ms and, next to the sweep on the side stream, finished 92 us late every sweep; with
// 512 and six it takes 0.39 ms and is never waited for); warp 4 issues the MMAs and owns TMEM (256 accumulator columns + a region of
// scale bytes 0x7F = 2^0), warps 5-8 drain the accumulator.  One CTA per SM; persistent over blocks, or one CTA per block when the
// launch shares the GPU with the sweep.
#include <stdint.h>
#include <string.h>

#include "device.cuh"

namespace bwgr {

namespace {

constexpr int kStages = 6;
constexpr int kProducers = 512;             // warps 0-3 and 9-20: one packed 16-byte chunk of one marker of each tile per thread and stage
constexpr int kThreads = kProducers + 160;  // + MMA warp (4) + four epilogue warps (5-8)
constexpr int kStageBytes = 2 * 128 * 128;  // two tiles (block b, block b + 1) x 128 markers x 128 bytes (256 rows as FP4)
constexpr uint32_t kAccCols = 256, kSfCol = 256, kSfCols = 64, kTmemCols = 512;

// block-scaled instruction descriptor (cute/arch/mma_sm100_desc.hpp, InstrDescriptorBlockScaled): A, B = E2M1 (kind::mxf4 format 1),
// both K-major, N = 256, scale format UE8M0, M = 128, K = 64, scale-factor ids 0
constexpr uint32_t kIdescMxf4 = (1u << 7) | (1u << 10) | ((256u >> 3) << 17) | (1u << 23) | ((128u >> 4) << 24);
__device__ __forceinline__ void umma_mxf4(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t sfa, uint32_t sfb, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::mxf4.block_scale.scale_vec::2X [%0], %1, %2, %3, [%4], [%5], p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(kIdescMxf4), "r"(sfa), "r"(sfb), "r"(accumulate) : "memory");
}

struct Fp4Smem {
  uint64_t full[kStages], empty[kStages], tmem_full, tmem_empty;
  uint32_t tmem_base;
  float sxc[256];  // column sums of the markers of block b | block b + 1 (centred Gram)
};

__global__ void __launch_bounds__(kThreads, 1) gram_fp4_kernel(const uint8_t* __restrict__ x2f, int64_t ldb, int64_t ld, int p, int n,
                                                          const int* __restrict__ perm, int nblocks, float* __restrict__ gram,
                                                          int* err, const float* __restrict__ sx, float inv_n) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* tiles = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  Fp4Smem* S = reinterpret_cast<Fp4Smem*>(tiles + kStages * kStageBytes);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkg = (int)((ld + 255) >> 8);  // stages of 256 genotype rows per block

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; s++) { mbar_init(&S->full[s], kProducers); mbar_init(&S->empty[s], 1); }
    mbar_init(&S->tmem_full, 1); mbar_init(&S->tmem_empty, 4);
    fence_mbar_init();
  }
  if (warp == 4) tmem_alloc(&S->tmem_base, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = S->tmem_base;
  if (warp >= 5 && warp <= 8) {
    // every block scale = 0x7F (UE8M0 2^0): the whole scale region is filled with that byte, so whichever rows / columns / byte
    // lanes of it the scale_vec::2X layout addresses read 1.0
    const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + kSfCol;
    const uint32_t one = 0x7F7F7F7Fu;
#pragma unroll
    for (int c = 0; c < (int)kSfCols; c += 4)
      asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %1, %1, %1};" ::"r"(taddr + (uint32_t)c), "r"(one) : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp < 4 || warp >= 9) {
    // ===================== producer: packed 2-bit chunks -> E2M1 nibbles, SWIZZLE_128B K-major tiles =====================
    // thread t: packed chunk c = t & 3 (64 rows = 32 bytes of FP4 = one K step of one marker) of marker m0 of both tiles; four
    // consecutive threads read 64 contiguous bytes of one packed column
    const int t = warp < 4 ? threadIdx.x : threadIdx.x - 160;  // 0..511
    const int c = t & 3, m0 = t >> 2;
    uint32_t it = 0;
    bool ok = true;
    for (int blk = blockIdx.x; blk < nblocks && ok; blk += gridDim.x) {
      const uint8_t* colp[2];
      bool val[2];
#pragma unroll
      for (int i = 0; i < 2; i++) {  // i = tile
        const int pos = (blk + i) * 128 + m0;
        val[i] = pos < p;
        colp[i] = x2f + (int64_t)(val[i] ? perm[pos] : 0) * ldb;
      }
      // kPf stages of packed chunks in flight per thread (16 bytes x 2 markers each): the gather is latency-bound (DRAM latency under
      // load is about two stage times), L2 serves the second reader of every tile (block b's tile 1 is block b + 1's tile 0, fetched
      // by a neighbouring CTA at about the same time)
      constexpr int kPf = 6;
      uint4 q[kPf][2];
      auto load_stage = [&](int kg, uint4 (&dst)[2]) {
        const int64_t off = (int64_t)kg * 64 + c * 16;  // byte offset inside the packed column
#pragma unroll
        for (int i = 0; i < 2; i++) dst[i] = (val[i] && kg < nkg && off < ldb) ? __ldg(reinterpret_cast<const uint4*>(colp[i] + off)) : make_uint4(0, 0, 0, 0);
      };
      // loads go out two stages at a time: the four threads of a marker then ask for one whole 128-byte line of its packed column
      // (two 64-byte visits to the same DRAM page at different times cost two activations)
#pragma unroll
      for (int s0 = 0; s0 < kPf - 2; s0++) load_stage(s0, q[s0]);
      for (int kg0 = 0; kg0 < nkg && ok; kg0 += kPf) {
#pragma unroll
        for (int u = 0; u < kPf; u++) {
          const int kg = kg0 + u;
          if (kg >= nkg || !ok) break;
          if ((u & 1) == 0) { load_stage(kg + kPf - 2, q[(u + kPf - 2) % kPf]); load_stage(kg + kPf - 1, q[(u + kPf - 1) % kPf]); }
          const uint32_t stage = it % kStages, phase = (it / kStages) & 1u;
          ok = mbar_wait(&S->empty[stage], phase ^ 1u, err);
          const uint32_t tbase = smem_u32(tiles + stage * kStageBytes);
#pragma unroll
          for (int i = 0; i < 2; i++) {
            const int m = m0;
            const uint32_t rowb = tbase + (uint32_t)(i * 16384 + (m >> 3) * 1024 + (m & 7) * 128);
            const uint4 pk = q[u][i];
            const uint32_t sw = (uint32_t)m & 7u;
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rowb + ((((uint32_t)(2 * c)) ^ sw) << 4)),
                         "r"((pk.x & 0x33333333u) << 1), "r"((pk.x >> 1) & 0x66666666u), "r"((pk.y & 0x33333333u) << 1), "r"((pk.y >> 1) & 0x66666666u) : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rowb + ((((uint32_t)(2 * c + 1)) ^ sw) << 4)),
                         "r"((pk.z & 0x33333333u) << 1), "r"((pk.z >> 1) & 0x66666666u), "r"((pk.w & 0x33333333u) << 1), "r"((pk.w >> 1) & 0x66666666u) : "memory");
          }
          fence_proxy_async();
          mbar_arrive(&S->full[stage]);
          it++;
        }
      }
    }
  } else if (warp == 4) {
    // ===================== MMA issuer =====================
    uint32_t it = 0, bi = 0;
    bool ok = true;
    const uint32_t sfa = tmem_base + kSfCol, sfb = tmem_base + kSfCol + 16;
    for (int blk = blockIdx.x; blk < nblocks && ok; blk += gridDim.x, bi++) {
      ok = mbar_wait(&S->tmem_empty, (bi & 1u) ^ 1u, err);
      tc_fence_after();
      for (int kg = 0; kg < nkg && ok; kg++, it++) {
        const uint32_t stage = it % kStages, phase = (it / kStages) & 1u;
        ok = mbar_wait(&S->full[stage], phase, err);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t desc = desc_k_sw128(smem_u32(tiles + stage * kStageBytes));  // A = tile of block b; B = both tiles (256 rows)
#pragma unroll
          for (int k4 = 0; k4 < 4; k4++)
            umma_mxf4(tmem_base, desc + (uint64_t)(k4 * 2), desc + (uint64_t)(k4 * 2), sfa, sfb, (kg | k4) != 0 ? 1u : 0u);
          umma_commit(&S->empty[stage]);
        }
        __syncwarp();
      }
      if (elect_one()) umma_commit(&S->tmem_full);
      __syncwarp();
    }
  } else if (warp <= 8) {
    // ===================== epilogue: TMEM -> registers -> HBM =====================
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    uint32_t bi = 0;
    bool ok = true;
    for (int blk = blockIdx.x; blk < nblocks && ok; blk += gridDim.x, bi++) {
      ok = mbar_wait(&S->tmem_full, bi & 1u, err);
      tc_fence_after();
      float* out_d = gram + ((size_t)blk * 128 + row) * 256;              // diagonal block of b
      float* out_c = gram + ((size_t)(blk + 1) * 128 + row) * 256 + 128;  // cross block of b + 1 (its row r = marker r of block b)
      float sxr = 0.0f;
      if (sx) {  // centred Gram (gram_centre)
        const int pos = blk * 128 + row;
        sxr = pos < p ? sx[perm[pos]] : 0.0f;
        named_bar(1, 128);
        for (int q = row; q < 256; q += 128) { const int pq = blk * 128 + q; S->sxc[q] = pq < p ? sx[perm[pq]] : 0.0f; }
        named_bar(1, 128);
      }
#pragma unroll
      for (int c = 0; c < 8; c++) {
        uint32_t v[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)c * 32u;
        tmem_ld_x32(taddr, v);
        tmem_ld_wait();
        if (sx) {
#pragma unroll
          for (int q = 0; q < 32; q++) v[q] = __float_as_uint(gram_centre(__uint_as_float(v[q]), sxr, S->sxc[c * 32 + q], inv_n));
        }
        if (c < 4) {
#pragma unroll
          for (int q = 0; q < 32; q += 4) *reinterpret_cast<uint4*>(out_d + c * 32 + q) = make_uint4(v[q], v[q + 1], v[q + 2], v[q + 3]);
        } else if (blk + 1 < nblocks) {
#pragma unroll
          for (int q = 0; q < 32; q += 4) *reinterpret_cast<uint4*>(out_c + (c - 4) * 32 + q) = make_uint4(v[q], v[q + 1], v[q + 2], v[q + 3]);
        }
      }
      if (blk == 0) {  // block 0 has no predecessor: its cross half is never read by the sweep, but keep it defined
#pragma unroll
        for (int q = 0; q < 128; q += 4) *reinterpret_cast<uint4*>(gram + (size_t)row * 256 + 128 + q) = make_uint4(0, 0, 0, 0);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&S->tmem_empty);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, kTmemCols);
}

// int8 store -> the packed shadow this kernel reads: word k of a column = rows 16k .. 16k+15, nibble i = {row 16k+i, row 16k+8+i}
__global__ void pack_2bit_fp4_kernel(const int8_t* __restrict__ src, int64_t ld, uint32_t* __restrict__ dst, int64_t ldw, int* bad) {
  const uint4* s = reinterpret_cast<const uint4*>(src + (int64_t)blockIdx.x * ld);
  uint32_t* d = dst + (int64_t)blockIdx.x * ldw;
  for (int64_t g = blockIdx.y * blockDim.x + threadIdx.x; g < ldw; g += (int64_t)gridDim.y * blockDim.x) {
    const uint4 v = s[g];  // rows 16g .. 16g+15 as bytes (pad rows are zero)
    const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
    uint32_t out = 0, any = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      any |= w4[q] & 0xFCFCFCFCu;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const int r = 4 * q + k;  // row inside the word
        const uint32_t code = (w4[q] >> (8 * k)) & 3u;
        out |= code << (4 * (r & 7) + 2 * (r >> 3));
      }
    }
    // a code 3 has both bits of its field set (E2M1 could hold 3, but not as code << 1)
    if (any || (out & (out >> 1) & 0x55555555u)) atomicExch(bad, 1);
    d[g] = out;
  }
}

}  // namespace

void launch_pack_2bit_fp4(const int8_t* src, int64_t ld, int p, uint8_t* dst, int* bad, cudaStream_t st) {
  const int64_t ldw = ld / 16;
  dim3 grid((unsigned)p, (unsigned)((ldw + 255) / 256 > 64 ? 64 : (ldw + 255) / 256));
  pack_2bit_fp4_kernel<<<grid, 256, 0, st>>>(src, ld, reinterpret_cast<uint32_t*>(dst), ldw, bad);
}

// gram: [nblocks][128][256] floats (band 2).  x2f: the packed shadow, ld / 4 bytes per column.
cudaError_t launch_gram_fp4(const uint8_t* x2f, int64_t ld, int p, int n, const int* perm, int nblocks, float* gram, int* err,
                            int num_sms, const float* sx, cudaStream_t st, bool block_per_cta) {
  const size_t smem = (size_t)kStages * kStageBytes + sizeof(Fp4Smem) + 1024;
  cudaError_t e = cudaFuncSetAttribute(gram_fp4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  // block_per_cta: one short CTA per marker block instead of a persistent grid -- the hardware hands blocks to whichever SMs are
  // free, which is what a launch that shares the GPU with the clustered sweep needs
  const int grid = block_per_cta || nblocks < num_sms ? nblocks : num_sms;
  gram_fp4_kernel<<<grid, kThreads, smem, st>>>(x2f, ld / 4, ld, p, n, perm, nblocks, gram, err, sx, 1.0f / (float)n);
  return cudaGetLastError();
}

}  // namespace bwgr
