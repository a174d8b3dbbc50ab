// gram_tc.cu -- Gram blocks X_B' X_B on the 5th-gen tensor cores (K6 of SURVEY 2c; not in the reference,
// required by the blocked exact Gauss-Seidel reformulation).
//
// For every block of 128 markers (in this sweep's order) G = X_B' X_B is a 128 x 128 x n int8 GEMM with
// exact int32 accumulation: tcgen05.mma kind::i8, M = N = 128, K = 32 per instruction, accumulator in
// TMEM.  A and B are the SAME shared-memory tile (marker-major, K = rows contiguous), staged as the
// canonical K-major SWIZZLE_128B layout: row m of the tile holds 128 consecutive genotype rows of marker m,
// 16-byte chunk c stored at chunk (c ^ (m & 7)); 8-row groups are 1024 B apart (SBO = 1024).
// Columns of a block are scattered in HBM when the order is shuffled (emRR & co, Rcpp20260726ai.cpp:331),
// so the tile is gathered with 16-byte cp.async (8 consecutive lanes = one 128-byte line of one column).
//
// Warp roles (416 threads): warps 0-3 gather (cp.async producer; with the packed source warps 9-12 join them), warp 4
// issues the MMAs (one elected lane) and owns the TMEM allocation, warps 5-8 drain the accumulator (tcgen05.ld -> st.global).
// Two accumulator stages (2 x 128 TMEM columns) overlap the drain of block i with the MMAs of block i+1.
// One CTA per SM, persistent over blocks.  HBM traffic: every genotype byte is read exactly once.
#include "device.cuh"

namespace bwgr {

namespace {

constexpr int kTileBytes = 128 * 128;
// NBAND = 1: diagonal blocks X_b'X_b only.  NBAND = 2: [X_b'X_b | X_{b-1}'X_b] (one-block look-ahead of the
// pipelined sweep, sweep_pipe.cu): row r of block b holds NBAND*128 entries, x_{b,r}'X_b then x_{b-1,r}'X_b.
// The gather is latency-bound: keep (almost) the whole 227 KB of shared memory in flight.
// A stage holds kSub consecutive 128-row atoms of every column of the band, so one visit to a column reads kSub*128
// contiguous bytes (DRAM pages are reused instead of re-opened per 128 B).
template <int NBAND> struct GramCfg {
  static constexpr int kSub = NBAND == 1 ? 4 : 2;
  static constexpr int kStages = 3;
  static constexpr int kLag = 2;
};
// kind::f8f6f4 with both operands E4M3 and an F32 accumulator.  Genotype codes 0..7 stored as int8 are, read as E4M3,
// the subnormals code * 2^-9: the SAME bytes feed this (4x faster) instruction, every product code_i*code_j*2^-18 is
// exact, and so is the fp32 sum while max_j xx_j < 2^24 -- the epilogue rescales by 2^18 and lands on the exact integer.
constexpr uint32_t kIdescF8 = (1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
__device__ __forceinline__ void umma_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

template <int NBAND>
struct GramSmem {
  uint64_t full[GramCfg<NBAND>::kStages], empty[GramCfg<NBAND>::kStages], tmem_full[2], tmem_empty[2];
  uint32_t tmem_base;
  float sxc[128];  // column sums of this block's markers (centred Gram)
};

// PACKED: the tiles are expanded from the 2-bit shadow copy g.x2 (codes 0..3) instead of gathered from the int8 store
template <int NBAND, bool FP8, bool PACKED>
__global__ void __launch_bounds__(416, 1) gram_tc_kernel(GenoView g, const int* __restrict__ perm, int nblocks,
                                                         int32_t* __restrict__ gram, int out_f32, int* err,
                                                         const float* __restrict__ sx, float inv_n) {
  constexpr int kStages = GramCfg<NBAND>::kStages;
  constexpr int kLag = GramCfg<NBAND>::kLag;  // cp.async groups kept in flight per producer thread
  constexpr int kSub = GramCfg<NBAND>::kSub;
  constexpr int kStageBytes = NBAND * kSub * kTileBytes;
  constexpr uint32_t kAccCols = NBAND * 128;  // TMEM columns of one accumulator stage
  using Sm = GramSmem<NBAND>;
  extern __shared__ unsigned char smem_raw[];
  // tiles first (1024 B aligned for SWIZZLE_128B), bookkeeping after them
  unsigned char* tiles = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  Sm* S = reinterpret_cast<Sm*>(tiles + kStages * kStageBytes);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkt = (int)(g.ld >> 7);  // K tiles of 128 rows (ld is a multiple of 128)
  const int nkg = (nkt + GramCfg<NBAND>::kSub - 1) / GramCfg<NBAND>::kSub;  // stages per block

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; s++) { mbar_init(&S->full[s], PACKED ? 256 : 128); mbar_init(&S->empty[s], 1); }
    for (int s = 0; s < 2; s++) { mbar_init(&S->tmem_full[s], 1); mbar_init(&S->tmem_empty[s], 4); }
    fence_mbar_init();
  }
  if (warp == 4) tmem_alloc(&S->tmem_base, 2u * kAccCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = S->tmem_base;

  if (PACKED && (warp < 4 || warp >= 9)) {
    // ===================== producer: 2-bit packed source (codes 0..3), expanded to bytes in flight =====================
    // The gather is what bounds this kernel (~4.3 TB/s of cp.async at 50k x 50k whatever the MMA kind); reading the packed
    // shadow copy moves 4x fewer bytes.  A 16-byte packed chunk = 64 rows of one marker = half a 128-row atom: it is
    // loaded into registers one stage ahead, expanded with two shift/mask steps per word and stored as four swizzled
    // 16-byte chunks.  Stage = kSub atoms, i.e. CPC = 2*kSub packed chunks per marker.
    // Eight producer warps (0-3 and 9-12): the expansion, not the gather, is what this producer costs.
    constexpr int CPC = 2 * kSub;          // packed 16-byte chunks per marker per stage
    constexpr int NIT = CPC / 2;           // chunks per thread per band per stage (128 markers * CPC chunks / 256 threads)
    constexpr int NLD = NIT * NBAND;
    constexpr int MSTEP = 256 / CPC;       // marker stride between a thread's chunks
    const int t = warp < 4 ? threadIdx.x : threadIdx.x - 160;  // 0..255
    const int c = t % CPC, m0 = t / CPC;   // this thread's chunk within the stage and its first marker; markers m0 + MSTEP*i
    uint32_t it = 0;
    bool ok = true;
    uint4 cur[NLD], nxt[NLD];
    auto load_stage = [&](const uint8_t* const (&colp)[NBAND][NIT], const bool (&val)[NBAND][NIT], int kg, uint4 (&dst)[NLD]) {
#pragma unroll
      for (int d = 0; d < NBAND; d++)
#pragma unroll
        for (int i = 0; i < NIT; i++) {
          const int64_t off = ((int64_t)kg * CPC + c) * 16;  // byte offset inside the packed column
          dst[d * NIT + i] = (val[d][i] && off < g.ldb) ? __ldg(reinterpret_cast<const uint4*>(colp[d][i] + off)) : make_uint4(0, 0, 0, 0);
        }
    };
    for (int blk = blockIdx.x; blk < nblocks && ok; blk += gridDim.x) {
      const uint8_t* colp[NBAND][NIT];
      bool val[NBAND][NIT];
#pragma unroll
      for (int d = 0; d < NBAND; d++)
#pragma unroll
        for (int i = 0; i < NIT; i++) {
          const int m = m0 + MSTEP * i;
          const int pos = (blk - d) * 128 + m;
          val[d][i] = pos >= 0 && pos < g.p;
          colp[d][i] = g.x2 + (int64_t)(val[d][i] ? perm[pos] : 0) * g.ldb;
        }
      load_stage(colp, val, 0, cur);
      for (int kg = 0; kg < nkg && ok; kg++, it++) {
        if (kg + 1 < nkg) load_stage(colp, val, kg + 1, nxt);
        const uint32_t stage = it % kStages, phase = (it / kStages) & 1u;
        ok = mbar_wait(&S->empty[stage], phase ^ 1u, err);
        const uint32_t tbase = smem_u32(tiles + stage * kStageBytes);
        const int sub = c >> 1;  // atom of this chunk; rows 64*(c&1) .. +63 inside it -> output chunks 4*(c&1) .. +3
#pragma unroll
        for (int d = 0; d < NBAND; d++)
#pragma unroll
          for (int i = 0; i < NIT; i++) {
            const int m = m0 + MSTEP * i;
            const uint4 pk = cur[d * NIT + i];
            const uint32_t w4[4] = {pk.x, pk.y, pk.z, pk.w};
            const uint32_t rowb = tbase + (sub * NBAND + d) * kTileBytes + m * 128;
#pragma unroll
            for (int q = 0; q < 4; q++) {  // packed word q = rows 16q .. 16q+15 of the half atom = one 16-byte output chunk
              // interleaved shadow layout (geno.cu): bytes of rows 4r .. 4r+3 = (w >> 2r) & 0x03030303
              const uint32_t oc = (uint32_t)(4 * (c & 1) + q);
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rowb + ((oc ^ ((uint32_t)m & 7u)) << 4)),
                           "r"(w4[q] & 0x03030303u), "r"((w4[q] >> 2) & 0x03030303u), "r"((w4[q] >> 4) & 0x03030303u),
                           "r"((w4[q] >> 6) & 0x03030303u) : "memory");
            }
          }
        fence_proxy_async();
        mbar_arrive(&S->full[stage]);
        if (kg + 1 < nkg) {
#pragma unroll
          for (int q = 0; q < NLD; q++) cur[q] = nxt[q];
        }
      }
    }
  } else if (warp < 4) {
    // ===================== producer: gather tiles from the int8 store with cp.async =====================
    const int t = threadIdx.x;  // 0..127
    uint32_t it = 0;            // tile counter (runs over blocks and K tiles)
    bool ok = true;
    for (int blk = blockIdx.x; blk < nblocks && ok; blk += gridDim.x) {
      const int8_t* colp[NBAND][8];
      uint32_t nbytes[NBAND][8];
#pragma unroll
      for (int d = 0; d < NBAND; d++)
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const int m = i * 16 + (t >> 3);
          const int pos = (blk - d) * 128 + m;
          const bool valid = pos >= 0 && pos < g.p;
          const int j = valid ? perm[pos] : 0;
          colp[d][i] = g.x8 + (int64_t)j * g.ld + ((t & 7) << 4);
          nbytes[d][i] = valid ? 16u : 0u;
        }
      for (int kg = 0; kg < nkg && ok; kg++, it++) {
        const uint32_t stage = it % kStages, phase = (it / kStages) & 1u;
        ok = mbar_wait(&S->empty[stage], phase ^ 1u, err);
        const uint32_t tbase = smem_u32(tiles + stage * kStageBytes);
#pragma unroll
        for (int sub = 0; sub < kSub; sub++) {
          const int kt = kg * kSub + sub;
          if (kt < nkt) {
#pragma unroll
            for (int d = 0; d < NBAND; d++)
#pragma unroll
              for (int i = 0; i < 8; i++) {
                const int m = i * 16 + (t >> 3);
                const uint32_t dst = tbase + (sub * NBAND + d) * kTileBytes + m * 128 + ((((uint32_t)t & 7u) ^ ((uint32_t)m & 7u)) << 4);
                cp_async16_zfill(dst, colp[d][i] + (int64_t)kt * 128, nbytes[d][i]);
              }
          }
        }
        cp_async_commit();
        if (it >= kLag) {
          cp_async_wait<kLag>();
          fence_proxy_async();
          mbar_arrive(&S->full[(it - kLag) % kStages]);
        }
      }
    }
    // drain: signal the last (up to kLag) tiles
    cp_async_wait<0>();
    fence_proxy_async();
    for (uint32_t q = (it > kLag ? it - kLag : 0); q < it; q++) mbar_arrive(&S->full[q % kStages]);
  } else if (warp == 4) {
    // ===================== MMA issuer =====================
    uint32_t it = 0, bi = 0;
    bool ok = true;
    for (int blk = blockIdx.x; blk < nblocks && ok; blk += gridDim.x, bi++) {
      const uint32_t as = bi & 1u, aphase = (bi >> 1) & 1u;
      ok = mbar_wait(&S->tmem_empty[as], aphase ^ 1u, err);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + as * kAccCols;
      for (int kg = 0; kg < nkg && ok; kg++, it++) {
        const uint32_t stage = it % kStages, phase = (it / kStages) & 1u;
        ok = mbar_wait(&S->full[stage], phase, err);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int sub = 0; sub < kSub; sub++) {
            const int kt = kg * kSub + sub;
            if (kt < nkt) {
              const uint64_t desc = desc_k_sw128(smem_u32(tiles + stage * kStageBytes + sub * NBAND * kTileBytes));
#pragma unroll
              for (int d = 0; d < NBAND; d++) {
                const uint64_t bdesc = desc_k_sw128(smem_u32(tiles + stage * kStageBytes + (sub * NBAND + d) * kTileBytes));
#pragma unroll
                for (int k4 = 0; k4 < 4; k4++) {
                  // band d >= 1 is stored transposed: row r = marker r of block b-d, columns = markers of block b, so that
                  // the sweep's correction threads (one per marker of block b) read it coalesced
                  const uint32_t acc = (kt | k4) != 0 ? 1u : 0u;
                  if (FP8) {
                    if (d == 0) umma_f8(tmem_d, desc + (uint64_t)(k4 * 2), desc + (uint64_t)(k4 * 2), kIdescF8, acc);
                    else umma_f8(tmem_d + (uint32_t)d * 128u, bdesc + (uint64_t)(k4 * 2), desc + (uint64_t)(k4 * 2), kIdescF8, acc);
                  } else {
                    if (d == 0) umma_i8(tmem_d, desc + (uint64_t)(k4 * 2), desc + (uint64_t)(k4 * 2), idesc_i8(128, 0), acc);
                    else umma_i8(tmem_d + (uint32_t)d * 128u, bdesc + (uint64_t)(k4 * 2), desc + (uint64_t)(k4 * 2), idesc_i8(128, 0), acc);
                  }
                }
              }
            }
          }
          umma_commit(&S->empty[stage]);  // frees the stage when these MMAs have read it
        }
        __syncwarp();
      }
      if (elect_one()) umma_commit(&S->tmem_full[as]);
      __syncwarp();
    }
  } else if (warp <= 8) {
    // ===================== epilogue: TMEM -> registers -> HBM =====================
    const int quarter = warp & 3;  // TMEM lanes this warp may touch
    const int row = quarter * 32 + lane;
    uint32_t bi = 0;
    bool ok = true;
    for (int blk = blockIdx.x; blk < nblocks && ok; blk += gridDim.x, bi++) {
      const uint32_t as = bi & 1u, aphase = (bi >> 1) & 1u;
      ok = mbar_wait(&S->tmem_full[as], aphase, err);
      tc_fence_after();
      int32_t* out = gram + ((size_t)blk * 128 + row) * (NBAND * 128);
      // centred Gram (gram_centre)
      float sxr0 = 0.0f, sxr1 = 0.0f;
      if (sx) {
        const int pos0 = blk * 128 + row, pos1 = (blk - 1) * 128 + row;
        sxr0 = pos0 < g.p ? sx[perm[pos0]] : 0.0f;
        sxr1 = (pos1 >= 0 && pos1 < g.p) ? sx[perm[pos1]] : 0.0f;
        named_bar(1, 128);  // previous block's reads of sxc are done
        S->sxc[row] = sxr0;
        named_bar(1, 128);
      }
#pragma unroll
      for (int c = 0; c < 4 * NBAND; c++) {
        uint32_t v[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + as * kAccCols + (uint32_t)c * 32u;
        tmem_ld_x32(taddr, v);
        tmem_ld_wait();
        if (FP8) {  // accumulator = exact integer * 2^-18 in fp32
#pragma unroll
          for (int q = 0; q < 32; q++) {
            const float f = __uint_as_float(v[q]) * 262144.0f;
            v[q] = out_f32 ? __float_as_uint(f) : (uint32_t)__float2int_rn(f);
          }
        } else if (out_f32) {
#pragma unroll
          for (int q = 0; q < 32; q++) v[q] = __float_as_uint(__int2float_rn((int)v[q]));
        }
        if (sx && out_f32) {
          const float sr = c < 4 ? sxr0 : sxr1;
#pragma unroll
          for (int q = 0; q < 32; q++) v[q] = __float_as_uint(gram_centre(__uint_as_float(v[q]), sr, S->sxc[(c & 3) * 32 + q], inv_n));
        }
        if (ok) {
#pragma unroll
          for (int q = 0; q < 32; q += 4)
            *reinterpret_cast<uint4*>(out + c * 32 + q) = make_uint4(v[q], v[q + 1], v[q + 2], v[q + 3]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&S->tmem_empty[as]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, 2u * kAccCols);
}

// Centres a band the kernel above (or gram_fp4.cu) wrote uncentred: row r of block b, column c of band d is x_{b-d,r}'x_{b,c}.
// One CTA per band row; block 0's cross half (no predecessor) is left as it is, as the Gram kernels leave it.
__global__ void __launch_bounds__(128) gram_centre_kernel(float* __restrict__ gram, const int* __restrict__ perm, int p, int nband,
                                                          const float* __restrict__ sx, float inv_n) {
  const int blk = blockIdx.x >> 7, r = blockIdx.x & 127, c = threadIdx.x;
  const int pc = blk * 128 + c;
  const float sxc = pc < p ? sx[perm[pc]] : 0.0f;
  float* row = gram + (size_t)blockIdx.x * nband * 128;
  for (int d = 0; d < nband && d <= blk; d++) {
    const int pr = (blk - d) * 128 + r;
    const float sxr = pr < p ? sx[perm[pr]] : 0.0f;
    row[d * 128 + c] = gram_centre(row[d * 128 + c], sxr, sxc, inv_n);
  }
}

}  // namespace

void launch_gram_centre(float* gram, const int* perm, int p, int nblocks, int nband, const float* sx, float inv_n, cudaStream_t st) {
  gram_centre_kernel<<<nblocks * 128, 128, 0, st>>>(gram, perm, p, nband, sx, inv_n);
}

template <int NBAND, bool FP8>
static void launch_gram_band(const GenoView& g, const int* perm, int nblocks, void* gram, int out_f32, int* err, int num_sms,
                             const float* sx, cudaStream_t st) {
  const size_t smem = (size_t)GramCfg<NBAND>::kStages * GramCfg<NBAND>::kSub * NBAND * kTileBytes + sizeof(GramSmem<NBAND>) + 1024;
  const int grid = nblocks < num_sms ? nblocks : num_sms;
  const float inv_n = 1.0f / (float)g.n;
  int32_t* out = static_cast<int32_t*>(gram);
#define BWGR_GRAM_LAUNCH(PACKED)                                                                                            \
  do {                                                                                                                      \
    cudaFuncSetAttribute(gram_tc_kernel<NBAND, FP8, PACKED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);       \
    gram_tc_kernel<NBAND, FP8, PACKED><<<grid, 416, smem, st>>>(g, perm, nblocks, out, out_f32, err, sx, inv_n);            \
  } while (0)
  if (FP8 && g.x2) BWGR_GRAM_LAUNCH(true);   // packed 2-bit shadow copy: codes 0..3, exact E4M3 products
  else BWGR_GRAM_LAUNCH(false);
#undef BWGR_GRAM_LAUNCH
}
void launch_gram_tc(const GenoView& g, const int* perm, int nblocks, void* gram, int out_f32, int nband, int fp8_codes,
                    int* err, int num_sms, const float* sx, cudaStream_t st) {
  if (fp8_codes) {
    if (nband == 2) launch_gram_band<2, true>(g, perm, nblocks, gram, out_f32, err, num_sms, sx, st);
    else launch_gram_band<1, true>(g, perm, nblocks, gram, out_f32, err, num_sms, sx, st);
  } else {
    if (nband == 2) launch_gram_band<2, false>(g, perm, nblocks, gram, out_f32, err, num_sms, sx, st);
    else launch_gram_band<1, false>(g, perm, nblocks, gram, out_f32, err, num_sms, sx, st);
  }
}

}  // namespace bwgr
