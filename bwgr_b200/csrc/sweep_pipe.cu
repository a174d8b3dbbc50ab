// sweep_pipe.cu -- the blocked exact Gauss-Seidel / Gibbs sweep, v5: streaming CTAs + one solver CTA,
// pipelined with a one-block look-ahead (K1 + K5 + K2 of SURVEY 2c).
//
// One persistent cooperative kernel per sweep, grid = W workers + 1 solver.
//
//   worker w (one per SM) owns the row slab [w*R, (w+1)*R) of every genotype column and the matching slab
//   of the residuals E (float master copy + four signed int8 limbs of its 31-bit fixed-point image, both in
//   shared memory).  Warp roles: 0 = tcgen05 issuer, 1-4 = TMEM epilogue, 5-8 = cp.async gather of the
//   X tiles (SWIZZLE_128B layout, ring of nbuf tiles, each genotype byte read from HBM once per sweep).
//   Per block b of 128 markers in this sweep's order (Rcpp20260726ai.cpp:331):
//     U(b):  E_slab -= X_b dE_b        tcgen05.mma kind::i8, A = tile (MN-major), B = int8 limbs of dE_b
//     G(c):  h_c partial = X_c' E      c = b+1+D; A = tile (K-major), B = limbs of E; exact int32 in TMEM
//   The integer partial of h_c goes to an L2 accumulator with one 64-bit red per marker: (value << 8) + 1,
//   so every word carries its own arrival count and nobody needs a fence or a grid barrier.
//
//   solver (the last CTA) polls h_b, forms the up-to-date  g_b = h_b - (X_b'X_{b-1}) dE_{b-1}  (D = 1:
//   h_b was taken before block b-1 was applied -- this is what takes the worker pipeline and the two L2
//   round trips off the critical path; the cross Gram block comes from gram_tc.cu, band 2), runs the
//   in-block sequential solve on the Gram block X_b'X_b and publishes dE_b as 64-bit self-validating words
//   (int32 fixed-point step | launch tag).  Linear rules (emRR, emBA, BayesRR, BayesA, rotated MRR3) are a
//   unit-lower-triangular system: one system applies the block inverse precomputed by block_inv.cu as a single
//   lower-triangular mat-vec on four warps; two systems step through 32-marker blocks with 32x32 inverses computed
//   one block ahead; more systems use an in-warp substitution.  The other rules walk the scalar chain.
//   Row-sharded fits (several GPUs): the reduced partial of a rank is stored into every peer's exchange ring (NVLink).
//   Either way the result is the reference's Gauss-Seidel order up to float reassociation.
//
// Critical path per block with D = 1: cross-Gram correction + in-block solve.  Everything else (gather,
// both tensor-core passes, quantisation, L2 round trips) runs beside it.
#include <string.h>

#include "device.cuh"

namespace bwgr {

namespace {

constexpr int kT = 512;
constexpr int kAtomBytes = 128 * 128;  // one 128-row atom of an X tile: 128 markers x 128 B
constexpr uint32_t kSpin = 1u << 21;
constexpr int kTS = 36;                // row stride (floats) of a 32x32 Gram tile in shared memory
constexpr int kTileF = 32 * kTS;       // floats per Gram tile
constexpr int kMS = 132;               // k/4 stride of a 32x32 inverse
constexpr int kSolveWarps = 8, kInvWarp0 = 4, kCorrWarp0 = 8, kPreWarp0 = 12;
constexpr int kDewStride = 136;        // 64-bit words per (block, system) of the published step
constexpr int kRing = 8;               // blocks of partial / reduced h kept in flight (ring in L2)
constexpr int kWPad = 160;             // worker slots per (block, system, marker) row of the partials
constexpr int kRedWarp = 9;            // worker warp that reduces its share of the partials

// genotype bytes are streamed once per sweep: L2 evict-first keeps the small hot arrays (Gram band, b, xx, order) resident
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void cp_async16_stream(uint32_t dst, const void* src, uint32_t nbytes, uint64_t pol) {
  asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2, %3;" ::"r"(dst), "l"(src), "r"(nbytes), "l"(pol) : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// Bounded wait.  A protocol bug or a dead peer must not hang the GPU: on time-out (or when another CTA
// already raised the error flag) the thread turns `dead` and every later wait returns at once.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, bool& dead, int* err) {
  if (dead) return;
  for (uint32_t spin = 0; spin < kSpin; spin++) {
    if (mbar_try(bar, parity)) return;
    if ((spin & 1023u) == 1023u && *reinterpret_cast<volatile int*>(err) != 0) break;
  }
  dead = true;
  atomicCAS(err, 0, 2);
}
__device__ __forceinline__ uint64_t desc_mn_sw128(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(kAtomBytes >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, int& v0, int& v1, int& v2, int& v3) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v0), "=r"(v1), "=r"(v2), "=r"(v3) : "r"(taddr) : "memory");
}
__device__ __forceinline__ long long combine_limbs(int s0, int s1, int s2, int s3) {
  return (long long)s0 + ((long long)s1 << 8) + ((long long)s2 << 16) + ((long long)s3 << 24);
}
// q (|q| <= 2^30) -> four balanced signed int8 limbs, q = l0 + 2^8 l1 + 2^16 l2 + 2^24 l3
__device__ __forceinline__ void split_limbs(int q, int& l0, int& l1, int& l2, int& l3) {
  l0 = (int)(signed char)(q & 0xFF); q = (q - l0) >> 8;
  l1 = (int)(signed char)(q & 0xFF); q = (q - l1) >> 8;
  l2 = (int)(signed char)(q & 0xFF); q = (q - l2) >> 8;
  l3 = q;
}
// byte offset of element (row n, K byte kb) inside one K-major SWIZZLE_128B atom stack
__device__ __forceinline__ uint32_t sw128_off(int n, int kb) {
  return (uint32_t)((n >> 3) * 1024 + (n & 7) * 128 + ((((kb >> 4) ^ (n & 7)) & 7) << 4) + (kb & 15));
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// system scope: the exchange ring of a row-sharded fit is written by peer GPUs over NVLink
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// ---- thread-block clusters (clustered topology: rank 0 of every cluster of 8 is a solver, ranks 1..7 are its workers) ----
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_idx() { uint32_t r; asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// remote shared-memory store that counts its bytes on the destination CTA's mbarrier (no flag, no polling)
__device__ __forceinline__ void st_async_u32(uint32_t raddr, uint32_t v, uint32_t rbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(raddr), "r"(v), "r"(rbar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
constexpr int kClSize = 8;             // CTAs per cluster: one solver + seven workers
constexpr int kClWorkers = kClSize - 1;
constexpr int kDeStride = 132;         // 32-bit words per (parity, system) of a worker's step inbox: 128 steps + the scale (+ pad)
constexpr int kAtomsPerGroup = 2;      // row atoms whose U epilogue / G issue are handled together (see the worker)
constexpr int kCommWarp0 = 4;          // clustered solver: warps 4-7 wait for the grid sums of h (they are idle whenever CL is eligible)
constexpr unsigned int kPollBackoffNs = 128;  // their sleep between polls (they share the SM with the solve chain)
// word of (block b, system s, marker m) among the grid-sum words of h (PipeArgs::hsum); copy c at + 32 c
__host__ __device__ inline size_t hsum_word(int b, int ns, int s, int m) { return (((size_t)b * ns + s) * 4 + (m >> 5)) * kGridCopies * 32 + (m & 31); }

// Self-validating 64-bit words of the grid reduction: (signed value << 12) | tag, tag = 1 + (use index of the ring slot) mod 4095
// (never 0 = freshly zeroed memory; consecutive uses of a slot always differ).  |value| < 2^51: a rank's sum of 143 worker
// partials of 2^30 * 2 * 512 rows is < 2^48.
constexpr int kTagBits = 12;
__device__ __forceinline__ unsigned long long tag_of(unsigned long long use) { return use % 4095ull + 1ull; }
__device__ __forceinline__ unsigned long long pack_word(long long v, unsigned long long tag) { return ((unsigned long long)v << kTagBits) | tag; }
__device__ __forceinline__ bool word_ok(unsigned long long w, unsigned long long tag) { return (w & ((1ull << kTagBits) - 1ull)) == tag; }
__device__ __forceinline__ long long word_val(unsigned long long w) { return (long long)w >> kTagBits; }

// per (system, marker) inputs of the solve; per marker: xx and the marker id
struct MarkerSys { float b0, vbj, a, c; };
struct MarkerCol { float xx, sx; int j, pad; };

// index of the 32x32 tile (hi, lo), lo <= hi, in the packed triangle
__device__ __forceinline__ int tri(int hi, int lo) { return hi * (hi + 1) / 2 + lo; }

struct Sync {
  // worker
  uint64_t tile_full[8], tile_empty[8], dl_full[2], u_done, el_full, g_done, g_empty;
  // solver
  uint64_t raw_ready[3], in_ready[3], solve_done[3], corr_ready[32], de_ready[32][4];
  // clustered topology: step inbox of a worker, grid sums of h ready for the solve warps
  uint64_t de_in[2], h_ready[2];
  // per 128-row atom: U accumulator complete (tcgen05.commit) / new residual limbs of the atom written (128 epilogue threads)
  uint64_t u_done_at[4], el_full_at[4];
  uint32_t tmem_base;
};

struct WLayout { int NA, N, nbuf; size_t xs, el, dl, es, dq, di, total; };
__host__ __device__ inline WLayout worker_layout(int R, int ns, int nbuf, bool cl = false) {
  WLayout L;
  L.NA = (R + 127) / 128; L.N = ((4 * ns + 15) / 16) * 16; L.nbuf = nbuf;
  size_t o = 0;
  L.xs = o; o += (size_t)nbuf * L.NA * kAtomBytes;
  L.el = o; o += (size_t)L.NA * (L.N / 8) * 1024;
  L.dl = o; o += (size_t)2 * (L.N / 8) * 1024;
  L.es = o; o += (size_t)ns * L.NA * 128 * 4;
  L.dq = o; o += (size_t)2 * 32 * 4;
  L.di = o; o += cl ? (size_t)2 * ns * kDeStride * 4 : 0;  // step inbox, written by the cluster's solver (st.async)
  L.total = o;
  return L;
}
struct SLayout { size_t gs, mt, ms, mc, drw, tc, dh, rb, cs, hs, total; };
// sring = blocks of solve inputs in flight in the solver CTA (2 or 3)
__host__ __device__ inline SLayout solver_layout(int ns, bool gibbs, bool use_inv, int sring, bool cl = false) {
  SLayout L;
  size_t o = 0;
  L.gs = o; o += (size_t)sring * 10 * kTileF * 4;                        // Gram triangle
  L.mt = o; o += use_inv ? (size_t)sring * ns * 4 * 8 * kMS * 4 : 0;       // 32x32 inverses
  L.ms = o; o += (size_t)sring * ns * 128 * sizeof(MarkerSys);
  L.mc = o; o += (size_t)sring * 128 * sizeof(MarkerCol);
  L.drw = o; o += gibbs ? (size_t)sring * ns * 128 * sizeof(MarkerDraws) : 0;
  L.tc = o; o += (size_t)2 * ns * 128 * 4;                               // cross-Gram correction, double buffered by block parity
  L.dh = o; o += (size_t)ns * 128 * 4;                                   // dE of the block being solved
  L.rb = o; o += (size_t)kSolveWarps * 32 * 4;
  L.cs = o; o += (size_t)32 * 2 * 4 + 2 * 4 * 4;  // running mean shift per system (centred columns): {current, before the last block}
  o = (o + 15) & ~(size_t)15;
  L.hs = o; o += cl ? (size_t)2 * ns * 128 * 8 : 0;  // h summed over the whole grid [parity][system][marker]
  L.total = o;
  return L;
}
__host__ __device__ inline bool pipe_use_inv(int model, int ns) { return model_is_linear(model) && ns <= 2; }

template <int MODEL, bool CL>
__global__ void __launch_bounds__(kT, 1) sweep_pipe_kernel(PipeArgs a) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ Sync S;
  __shared__ SysScalars sc[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ns = a.s.nsys, p = a.s.g.p, W = a.nworkers, D = a.D, nblocks = a.nblocks;
  unsigned char* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  // clustered topology (CL): rank 0 of every cluster is a solver (all solvers run the identical solve on the identical integer
  // sums, like the ranks of a row-sharded fit), ranks 1..7 are its workers; worker index = cluster * 7 + rank - 1
  const int crank = CL ? (int)cluster_ctarank() : 0, cluster = CL ? (int)cluster_idx() : 0;
  const bool is_solver = CL ? crank == 0 : (int)blockIdx.x == W;
  const int widx = CL ? cluster * kClWorkers + crank - 1 : (int)blockIdx.x;
  const bool writer = !CL || cluster == 0;  // the solver that writes b / d / vb back to HBM
  bool dead = false;

  if (tid < ns) sc[tid] = a.s.sc[tid];
  if (tid == 0) {
    for (int i = 0; i < 8; i++) { mbar_init(&S.tile_full[i], 128); mbar_init(&S.tile_empty[i], 1); }
    for (int i = 0; i < 4; i++) { mbar_init(&S.u_done_at[i], 1); mbar_init(&S.el_full_at[i], 128); }
    mbar_init(&S.dl_full[0], 128); mbar_init(&S.dl_full[1], 128);
    mbar_init(&S.u_done, 1); mbar_init(&S.el_full, 128); mbar_init(&S.g_done, 1); mbar_init(&S.g_empty, 128);
    const int nsw = ns < kSolveWarps ? ns : kSolveWarps;
    for (int i = 0; i < 3; i++) { mbar_init(&S.raw_ready[i], 128); mbar_init(&S.in_ready[i], 128); mbar_init(&S.solve_done[i], a.tinv ? 4 : nsw); }
    for (int s = 0; s < 32; s++) {
      mbar_init(&S.corr_ready[s], 128);
      for (int d = 0; d < 4; d++) mbar_init(&S.de_ready[s][d], 1);
    }
    for (int i = 0; i < 2; i++) { mbar_init(&S.de_in[i], 1); mbar_init(&S.h_ready[i], 128); }
    fence_mbar_init();
    if (CL && !is_solver)  // expected bytes of the first two steps (every later phase is armed by the consumer of the phase before)
      for (int i = 0; i < 2 && i < nblocks; i++) mbar_expect_tx(&S.de_in[i], (uint32_t)(ns * 129 * 4));
  }
  if (CL) cluster_sync_all();  // every CTA's barriers exist before the first remote store

  if (!is_solver) {
    // =====================================================================================================
    // worker
    // =====================================================================================================
    const WLayout L = worker_layout(a.rows_per_cta, ns, a.nbuf, CL);
    const int R = a.rows_per_cta, NA = L.NA, N = L.N, RS = NA * 128, nbuf = L.nbuf;
    const int row0 = widx * R;
    const uint32_t* dein = reinterpret_cast<const uint32_t*>(base + L.di);
    unsigned char* Xs = base + L.xs;
    unsigned char* EL = base + L.el;
    unsigned char* DL = base + L.dl;
    float* Es = reinterpret_cast<float*>(base + L.es);
    float* dqs = reinterpret_cast<float*>(base + L.dq);
    {  // zero tiles and operand regions once: pad rows / chunks / limb columns stay zero for the whole kernel
      uint4* z = reinterpret_cast<uint4*>(base);
      const int nz = (int)(L.es >> 4);
      for (int i = tid; i < nz; i += kT) z[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    bool bad = false;
    for (int s = 0; s < ns; s++)
      for (int i = tid; i < RS; i += kT) {
        const int r = row0 + i;
        const float e = (i < R && r < a.s.g.ld) ? a.s.e[(size_t)s * a.s.g.ld + r] : 0.0f;
        Es[s * RS + i] = e;
        if (i < R) {
          const float sv = e * sc[s].e_qinv;
          if (!(fabsf(sv) <= 1073741824.0f)) bad = true;
          int l0, l1, l2, l3;
          split_limbs(__float2int_rn(sv), l0, l1, l2, l3);
          unsigned char* atom = EL + (size_t)(i >> 7) * (N / 8) * 1024;
          const int kb = i & 127;
          atom[sw128_off(4 * s + 0, kb)] = (unsigned char)l0; atom[sw128_off(4 * s + 1, kb)] = (unsigned char)l1;
          atom[sw128_off(4 * s + 2, kb)] = (unsigned char)l2; atom[sw128_off(4 * s + 3, kb)] = (unsigned char)l3;
        }
      }
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < (NA + 1) * N) tmem_cols <<= 1;
    if (warp == 0) tmem_alloc(&S.tmem_base, tmem_cols);
    fence_proxy_async();  // initial limbs (generic stores) -> tensor core
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = S.tmem_base;
    const uint32_t tmem_g = tmem_base + (uint32_t)(NA * N);
    const bool tracing = a.trace != nullptr;
#define WSTAMP(blk, k) do { if (tracing) { long long* tp_ = a.trace + ((size_t)blockIdx.x * nblocks + (blk)) * 32 + (k); tp_[0] = (long long)globaltimer_ns(); tp_[16] = clock64(); } } while (0)

    if (warp == 0) {
      // ------------------------------------------------------------------ tcgen05 issuer
      const uint32_t idesc_g = idesc_i8(N, 0), idesc_u = idesc_i8(N, 1);
      // The row atoms of the slab are handled in groups of two (kAtomsPerGroup): the U pass commits group by group, the epilogue
      // updates E and writes the new limbs group by group (both atoms of a group in flight at once: the epilogue is latency-bound),
      // and the MMAs of G(c) over a group are issued as soon as that group's limbs are in shared memory (el_full_at[g]; `use` = use
      // number of those barriers, < 0 = the limbs written at start-up).  The two tensor-core passes and the epilogue overlap by halves.
      auto issue_g = [&](int c, int use) {
        const unsigned char* Xt = Xs + (size_t)(c % nbuf) * NA * kAtomBytes;
        mbar_wait(&S.tile_full[c % nbuf], (uint32_t)(c / nbuf) & 1u, dead, a.s.err);
        if (c > 0) mbar_wait(&S.g_empty, (uint32_t)(c - 1) & 1u, dead, a.s.err);
        for (int g = 0; g * kAtomsPerGroup < NA; g++) {
          if (use >= 0) mbar_wait(&S.el_full_at[g], (uint32_t)use & 1u, dead, a.s.err);
          tc_fence_after();
          if (elect_one()) {
            for (int at = g * kAtomsPerGroup; at < NA && at < (g + 1) * kAtomsPerGroup; at++) {
              const uint64_t ad = desc_k_sw128(smem_u32(Xt + (size_t)at * kAtomBytes));
              const uint64_t bd = desc_k_sw128(smem_u32(EL + (size_t)at * (N / 8) * 1024));
#pragma unroll
              for (int k4 = 0; k4 < 4; k4++) umma_i8(tmem_g, ad + (uint64_t)(2 * k4), bd + (uint64_t)(2 * k4), idesc_g, (at | k4) != 0);
            }
            if ((g + 1) * kAtomsPerGroup >= NA) umma_commit(&S.g_done);
          }
          __syncwarp();
        }
      };
      const int npro = (D < nblocks - 1 ? D : nblocks - 1);
      for (int c = 0; c <= npro; c++) issue_g(c, -1);
      for (int b = 0; b < nblocks; b++) {
        const unsigned char* Xt = Xs + (size_t)(b % nbuf) * NA * kAtomBytes;
        mbar_wait(&S.dl_full[b & 1], (uint32_t)(b >> 1) & 1u, dead, a.s.err);
        tc_fence_after();
        if (tracing && lane == 0) WSTAMP(b, 8);
        if (elect_one()) {
          const uint64_t bd = desc_k_sw128(smem_u32(DL + (size_t)(b & 1) * (N / 8) * 1024));
          for (int at = 0; at < NA; at++) {
            const uint64_t ad = desc_mn_sw128(smem_u32(Xt + (size_t)at * kAtomBytes));
#pragma unroll
            for (int k4 = 0; k4 < 4; k4++)
              umma_i8(tmem_base + (uint32_t)(at * N), ad + (uint64_t)(k4 * (4096 >> 4)), bd + (uint64_t)(2 * k4), idesc_u, k4 != 0);
            if ((at % kAtomsPerGroup) == kAtomsPerGroup - 1 || at == NA - 1) umma_commit(&S.u_done_at[at / kAtomsPerGroup]);  // the epilogue starts on this group while the next one is multiplied
          }
          umma_commit(&S.tile_empty[b % nbuf]);
          if (tracing) WSTAMP(b, 2);
        }
        __syncwarp();
        const int c = b + 1 + D;
        if (c < nblocks) {
          issue_g(c, b);
          if (tracing && lane == 0) WSTAMP(b, 5);
        }
      }
    } else if (warp <= 4) {
      // ------------------------------------------------------------------ TMEM epilogue (thread = TMEM lane)
      const int quarter = warp & 3;
      const int q = quarter * 32 + lane;
      const uint32_t tlane = (uint32_t)(quarter * 32) << 16;
      const bool t0 = tracing && q == 0;
      auto g_epilogue = [&](int c) {
        mbar_wait(&S.g_done, (uint32_t)c & 1u, dead, a.s.err);
        if (t0) WSTAMP(c, 6);
        tc_fence_after();
        // partial of marker q, system s -> part[c % ring][s][this worker][q] (full 32-byte sectors): (value << 12) | block tag
        unsigned long long* hb = a.part + (((size_t)(c % kRing) * ns) * kWPad + (CL ? 0 : blockIdx.x)) * 128 + q;
        const unsigned long long tagc = tag_of((unsigned long long)(c / kRing));
        for (int s = 0; s < ns; s++) {
          int s0, s1, s2, s3;
          tmem_ld4(tmem_g + tlane + (uint32_t)(4 * s), s0, s1, s2, s3);
          tmem_ld_wait();
          const long long gq = combine_limbs(s0, s1, s2, s3);
          // CL: straight into copy (worker % kGridCopies) of the grid-sum word of (block c, system s, marker q)
          if (CL) grid_add(a.hsum + hsum_word(c, ns, s, q) + (widx % kGridCopies) * 32, gq, a.s.err);
          else st_relaxed_u64(hb + (size_t)s * kWPad * 128, pack_word(gq, tagc));
        }
        tc_fence_before();
        mbar_arrive(&S.g_empty);
        if (t0) WSTAMP(c, 7);
      };
      const int npro = (D < nblocks - 1 ? D : nblocks - 1);
      for (int c = 0; c <= npro; c++) g_epilogue(c);
      for (int b = 0; b < nblocks; b++) {
        // ---- the step of block b, published by the solver: (int32 q << 32) | tag per marker, then the scale
        {
          const unsigned long long* wv = a.dew + (size_t)b * ns * kDewStride;
          unsigned char* dl = DL + (size_t)(b & 1) * (N / 8) * 1024;
          // epilogue warp e receives the systems s = e, e+4, ...: lane l polls step words l, l+32, l+64, l+96 and lane 0 the
          // scale word as well (one L2 round trip when the step is already there), then writes the limbs of those markers
          if (CL) mbar_wait(&S.de_in[b & 1], (uint32_t)(b >> 1) & 1u, dead, a.s.err);
          for (int s = quarter; s < ns; s += 4) {
            const unsigned long long* ws = wv + (size_t)s * kDewStride;
            unsigned long long v[4] = {0, 0, 0, 0}, vq = 0;
            uint32_t spin = 0;
            if (CL) {  // the step arrived in this CTA's inbox (st.async from the cluster's solver)
              const uint32_t* di = dein + (size_t)((b & 1) * ns + s) * kDeStride;
#pragma unroll
              for (int t = 0; t < 4; t++) v[t] = (unsigned long long)di[32 * t + lane] << 32;
              vq = (unsigned long long)di[128] << 32;
            }
            while (!CL && !dead) {
              bool ok = true;
#pragma unroll
              for (int t = 0; t < 4; t++) { v[t] = ld_relaxed_u64(ws + 32 * t + lane); ok = ok && ((uint32_t)v[t] == a.tag); }
              if (lane == 0) { vq = ld_relaxed_u64(ws + 128); ok = ok && ((uint32_t)vq == a.tag); }
              if (__all_sync(0xffffffffu, ok)) break;
              if (++spin > kSpin || ((spin & 255u) == 255u && *reinterpret_cast<volatile int*>(a.s.err) != 0)) { dead = true; atomicCAS(a.s.err, 0, 3); }
            }
            if (lane == 0) dqs[(b & 1) * 32 + s] = __uint_as_float((uint32_t)(vq >> 32));
#pragma unroll
            for (int t = 0; t < 4; t++) {
              const int m = 32 * t + lane;
              int l0, l1, l2, l3;
              split_limbs(dead ? 0 : (int)(uint32_t)(v[t] >> 32), l0, l1, l2, l3);
              dl[sw128_off(4 * s + 0, m)] = (unsigned char)l0; dl[sw128_off(4 * s + 1, m)] = (unsigned char)l1;
              dl[sw128_off(4 * s + 2, m)] = (unsigned char)l2; dl[sw128_off(4 * s + 3, m)] = (unsigned char)l3;
            }
          }
          if (t0) WSTAMP(b, 0);
          // this inbox slot is next used by block b + 2, whose step cannot be sent before this worker's partial of b + 2
          if (CL && q == 0 && b + 2 < nblocks) mbar_expect_tx(&S.de_in[b & 1], (uint32_t)(ns * 129 * 4));
          fence_proxy_async();
          mbar_arrive(&S.dl_full[b & 1]);
          named_bar(1, 128);  // the scales (dqs) of all systems visible to the four epilogue warps
          if (t0) WSTAMP(b, 1);
        }
        // ---- E_slab -= X_b dE_b, then the limbs of the new residual (B operand of the next G pass)
        // group by group (two row atoms each), as the issuer commits them
        for (int g = 0; g * kAtomsPerGroup < NA; g++) {
          mbar_wait(&S.u_done_at[g], (uint32_t)b & 1u, dead, a.s.err);
          if (t0 && g == 0) WSTAMP(b, 3);
          tc_fence_after();
          const int at0 = g * kAtomsPerGroup;
          for (int s = 0; s < ns; s++) {
            int acc[kAtomsPerGroup][4];
#pragma unroll
            for (int u = 0; u < kAtomsPerGroup; u++)
              if (at0 + u < NA) tmem_ld4(tmem_base + tlane + (uint32_t)((at0 + u) * N + 4 * s), acc[u][0], acc[u][1], acc[u][2], acc[u][3]);
            tmem_ld_wait();
            const float dqv = dqs[(b & 1) * 32 + s], eqi = sc[s].e_qinv;
#pragma unroll
            for (int u = 0; u < kAtomsPerGroup; u++) {
              const int at = at0 + u, i = at * 128 + q;
              if (at < NA && i < R) {
                // uq * dq in two exact float pieces (uq = 2^24 hi + lo, |hi| < 2^22, 0 <= lo < 2^24; dq is a power of two)
                const long long uq = combine_limbs(acc[u][0], acc[u][1], acc[u][2], acc[u][3]);
                const float hi = (float)(int)(uq >> 24) * 16777216.0f, lo = (float)(int)(uq & 0xFFFFFF);
                const float e = fmaf(-lo, dqv, fmaf(-hi, dqv, Es[s * RS + i]));
                Es[s * RS + i] = e;
                const float sv = e * eqi;
                if (!(fabsf(sv) <= 1073741824.0f)) bad = true;
                int l0, l1, l2, l3;
                split_limbs(__float2int_rn(sv), l0, l1, l2, l3);
                unsigned char* atom = EL + (size_t)at * (N / 8) * 1024;
                atom[sw128_off(4 * s + 0, q)] = (unsigned char)l0; atom[sw128_off(4 * s + 1, q)] = (unsigned char)l1;
                atom[sw128_off(4 * s + 2, q)] = (unsigned char)l2; atom[sw128_off(4 * s + 3, q)] = (unsigned char)l3;
              }
            }
          }
          tc_fence_before();
          fence_proxy_async();
          mbar_arrive(&S.el_full_at[g]);
        }
        if (t0) WSTAMP(b, 4);
        const int c = b + 1 + D;
        if (c < nblocks) g_epilogue(c);
      }
      // residuals back to HBM
      named_bar(1, 128);
      for (int s = 0; s < ns; s++)
        for (int i = q; i < R; i += 128) {
          const int r = row0 + i;
          if (r < a.s.g.ld) a.s.e[(size_t)s * a.s.g.ld + r] = Es[s * RS + i];
        }
    } else if ((warp >= 5 && warp <= 8) || (warp >= 10 && warp <= 13)) {
      // ------------------------------------------------------------------ X tile gather
      // two groups of four warps take alternate tiles; a group waits for its own tile to land before it signals it,
      // so a tile is announced the moment it is complete and the other group's tile stays in flight meanwhile.
      // A ring of one tile (the plans without look-ahead) has one group: with two, the group of tile t + 2 could wait on the
      // parity of a tile_empty phase two uses ahead, which reads as complete, and overwrite the tile still in use.
      const int grp = warp >= 10 ? 1 : 0, ngrp = nbuf >= 2 ? 2 : 1;
      const int lw = warp - (grp ? 10 : 5);
      const int nchunk = R >> 4;
      const bool act = lane < nchunk && row0 + 16 * lane < a.s.g.ld;
      const uint32_t choff = (uint32_t)((lane >> 3) * kAtomBytes + ((lane & 7) << 4));
      const int8_t* xrow = a.s.g.x8 + row0 + 16 * lane;
      const uint64_t pol = policy_evict_first();
      for (int t = grp; t < nblocks && grp < ngrp; t += ngrp) {
        const int buf = t % nbuf;
        const int pos = t * 128 + lw + 4 * lane;
        const int myid = pos < p ? a.perm[pos] : -1;
        if (t >= nbuf) mbar_wait(&S.tile_empty[buf], (uint32_t)(t / nbuf - 1) & 1u, dead, a.s.err);
        const uint32_t dst = smem_u32(Xs + (size_t)buf * NA * kAtomBytes);
#pragma unroll 8
        for (int i = 0; i < 32; i++) {
          const int m = lw + 4 * i;
          const int j = __shfl_sync(0xffffffffu, myid, i);
          if (lane < nchunk) {
            const uint32_t dm = dst + (uint32_t)(m * 128) + (choff ^ (uint32_t)((m & 7) << 4));
            const bool ok = act && j >= 0;
            cp_async16_stream(dm, ok ? xrow + (int64_t)j * a.s.g.ld : a.s.g.x8, ok ? 16u : 0u, pol);
          }
        }
        cp_async_commit();
        if (tracing && lw == 0 && lane == 0) WSTAMP(t, 12);
        cp_async_wait<0>();
        fence_proxy_async();
        mbar_arrive(&S.tile_full[buf]);
        if (tracing && lw == 0 && lane == 0) WSTAMP(t, 13);
      }
    } else if (warp == kRedWarp && CL) {
      // ------------------------------------------------------------------ zero the grid-sum words of the next launch
      // (this warp is idle in the clustered topology; the words are in use again only after this launch has ended)
      const size_t n16 = (size_t)nblocks * ns * 128 * kGridCopies / 2;
      uint4* z = reinterpret_cast<uint4*>(a.hsum_next);
      for (size_t i = (size_t)widx * 32 + lane; i < n16; i += (size_t)W * 32) z[i] = make_uint4(0, 0, 0, 0);
    } else if (warp == kRedWarp) {
      // ------------------------------------------------------------------ second hop of the grid reduction
      // row (block c, system s, marker m) of the partials is summed by worker (s*128 + m) % W; plain loads and one store,
      // no atomics (143 x 128 L2 atomics per block cost ~7 us; this tree costs two L2 round trips)
      for (int c = 0; c < nblocks; c++) {
        const unsigned long long tagc = tag_of((unsigned long long)(c / kRing));
        // row-sharded fit: the slot / tag of the exchange ring follow the global block sequence number (never re-zeroed)
        const unsigned long long gen = a.gen0 + (unsigned long long)c;
        const unsigned long long tagx = tag_of(gen / kRing);
        const size_t xslot = (size_t)(gen % kRing);
        for (int task = blockIdx.x; task < ns * 128; task += W) {
          const unsigned long long* row = a.part + ((size_t)(c % kRing) * ns + (task >> 7)) * kWPad * 128 + (task & 127);  // stride 128 words per worker
          long long sum = 0;
          uint32_t spin = 0;
          while (!dead) {  // all W <= 160 words of the row in flight at once; re-read the whole row until every tag matches
            bool ok = true;
            sum = 0;
#pragma unroll
            for (int k = 0; k < 5; k++) {
              const int w = 32 * k + lane;
              if (w < W) {
                const unsigned long long v = ld_relaxed_u64(row + (size_t)w * 128);
                ok = ok && word_ok(v, tagc);
                sum += word_val(v);
              }
            }
            if (__all_sync(0xffffffffu, ok)) break;
            if (++spin > kSpin || ((spin & 255u) == 255u && *reinterpret_cast<volatile int*>(a.s.err) != 0)) { dead = true; atomicCAS(a.s.err, 0, 3); sum = 0; }
          }
          if (tracing && lane == 0 && task == (int)blockIdx.x) WSTAMP(c, 14);
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
          if (a.world > 1) {
            // third hop over NVLink: this rank's reduced word goes straight into every rank's exchange ring (peer stores);
            // each solver then sums the `world` words of a marker in rank order -- identical integers on every GPU
            if (lane < a.world) st_relaxed_sys_u64(a.hx[lane] + ((xslot * a.world + a.rank) * ns) * 128 + task, pack_word(sum, tagx));
          } else if (lane == 0) {
            st_relaxed_u64(a.hred + (size_t)(c % kRing) * ns * 128 + task, pack_word(sum, tagc));
          }
          if (tracing && lane == 0 && task == (int)blockIdx.x) WSTAMP(c, 15);
        }
      }
    }
    if (bad) atomicExch(a.s.err, 4);
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, tmem_cols);
#undef WSTAMP
    if (CL) cluster_sync_all();  // nobody leaves while a peer may still store into its shared memory
    return;
  }

  // =======================================================================================================
  // solver
  // =======================================================================================================
  constexpr bool kLinear = model_is_linear(MODEL);
  constexpr bool kGibbs = model_is_gibbs(MODEL);
  // Gibbs spike-slab rules (BayesB :670-681, BayesC :731-741, KMUP :19-32, BayesDpi :949-964): everything that does not depend on g is folded
  // into four per-marker numbers one block ahead, and the Bernoulli(pj) draw u < 1/(1 + R exp(x)) is taken as
  // x < log((1/u - 1)/R): the dependent chain per marker is one shuffle, five FMAs and a compare (no exp, no division).
  constexpr bool kSlabDraw = MODEL == M_BB || MODEL == M_BC || MODEL == M_KMUP || MODEL == M_BDPI;
  // EM spike-slab rules (emBB :162-169, emBC :221-227): the reciprocal 1/(xx + lambda) and xx b0/(xx + lambda) are folded one
  // block ahead as well; the chain keeps one exp and one reciprocal (the inclusion weight d = 1/(1 + LR) is a value here).
  constexpr bool kSlabEM = MODEL == M_EMBB || MODEL == M_EMBC;
  // Thresholding rules (emEN :431-436, lasso :1478-1486, emBL :378-386): the reciprocals of their denominators are folded one
  // block ahead, the chain keeps an FMA, a compare / clip and a multiply (no division).
  constexpr bool kFoldEM = MODEL == M_EMEN || MODEL == M_LASSO || MODEL == M_EMBL;
  // T = (I + A L)^-1 of every block precomputed (block_inv.cu): one system, linear rule, uncentred columns.  The in-block solve
  // is then one lower-triangular mat-vec, spread over four warps
  const bool full_inv = a.tinv != nullptr;
  const bool use_inv = !full_inv && pipe_use_inv(MODEL, ns);
  const int sring = a.sring;
  const SLayout L = solver_layout(ns, kGibbs, use_inv, sring, CL);
  float* Gs = reinterpret_cast<float*>(base + L.gs);
  float* Mt = reinterpret_cast<float*>(base + L.mt);
  MarkerSys* msys = reinterpret_cast<MarkerSys*>(base + L.ms);
  MarkerCol* mcol = reinterpret_cast<MarkerCol*>(base + L.mc);
  MarkerDraws* drw = reinterpret_cast<MarkerDraws*>(base + L.drw);
  float* tcor = reinterpret_cast<float*>(base + L.tc);
  float* dehist = reinterpret_cast<float*>(base + L.dh);
  float* rb = reinterpret_cast<float*>(base + L.rb);
  float* cs = reinterpret_cast<float*>(base + L.cs);
  long long* hsum = reinterpret_cast<long long*>(base + L.hs);
  // a worker's step inbox sits at the same shared-window offset in every CTA of this launch
  const uint32_t dein_u32 = smem_u32(base) + (uint32_t)worker_layout(a.rows_per_cta, ns, a.nbuf, CL).di;
  const bool centred = a.sx != nullptr;
  const float inv_n = 1.0f / (float)a.n_total;
  if (tid < 64) cs[tid] = 0.0f;
  const int gstride = a.nband * 128;  // floats per Gram row in HBM
  const int nsw = ns < kSolveWarps ? ns : kSolveWarps;
  __syncthreads();
  const bool tracing = a.trace != nullptr;
#define SSTAMPW(blk, k) do { if (tracing && lane == 0) { long long* tp_ = a.trace + ((size_t)blockIdx.x * nblocks + (blk)) * 32 + (k); tp_[0] = (long long)globaltimer_ns(); tp_[16] = clock64(); } } while (0)
#define SSTAMP(blk, k) do { if (tracing && warp == 0 && lane == 0) { long long* tp_ = a.trace + ((size_t)blockIdx.x * nblocks + (blk)) * 32 + (k); tp_[0] = (long long)globaltimer_ns(); tp_[16] = clock64(); } } while (0)

  if (warp < kSolveWarps) {
    if (use_inv && warp >= kInvWarp0) {
      // ------------------------------------------------------------------ inverses of the diagonal blocks (ns <= 2: solve warps 4-7 are free)
      // invert the four 32x32 diagonal blocks of I + A L (E-independent), one block of markers ahead of the solve
      for (int nb = 0; nb < nblocks; nb++) {
        const int slot = nb % sring;
        mbar_wait(&S.raw_ready[slot], (uint32_t)(nb / sring) & 1u, dead, a.s.err);
        const float* Gb = Gs + (size_t)slot * 10 * kTileF;
        for (int task = warp - kInvWarp0; task < ns * 4; task += 4) {
          const int s = task >> 2, d = task & 3;
          const MarkerSys* mk = msys + ((size_t)slot * ns + s) * 128 + 32 * d;
          const float* gt = Gb + (size_t)tri(d, d) * kTileF;
          // column `lane` of M = (I + A L)^-1 by right-looking substitution: once x_k is final, every later partial sum
          // takes its term at once (31-k independent FMAs), so the dependent chain is two FMAs per step
          float x[32], sacc[32];
#pragma unroll
          for (int i = 0; i < 32; i++) sacc[i] = 0.0f;
#pragma unroll
          for (int k = 0; k < 32; k++) {
            x[k] = fmaf(-mk[k].a, sacc[k], (k == lane) ? 1.0f : 0.0f);
            const float4* grow = reinterpret_cast<const float4*>(gt + k * kTS);  // row k = column k (symmetric tile)
#pragma unroll
            for (int i4 = (k + 1) / 4; i4 < 8; i4++) {
              const float4 gv = grow[i4];
              if (4 * i4 + 0 > k) sacc[4 * i4 + 0] = fmaf(gv.x, x[k], sacc[4 * i4 + 0]);
              if (4 * i4 + 1 > k) sacc[4 * i4 + 1] = fmaf(gv.y, x[k], sacc[4 * i4 + 1]);
              if (4 * i4 + 2 > k) sacc[4 * i4 + 2] = fmaf(gv.z, x[k], sacc[4 * i4 + 2]);
              if (4 * i4 + 3 > k) sacc[4 * i4 + 3] = fmaf(gv.w, x[k], sacc[4 * i4 + 3]);
            }
          }
          // M[i][c] (c = lane) stored as Mt4[c/4][i][c%4] with a padded c/4 stride: conflict-free both ways
          float* mt = Mt + ((size_t)(slot * ns + s) * 4 + d) * 8 * kMS + (lane >> 2) * kMS + (lane & 3);
#pragma unroll
          for (int i = 0; i < 32; i++) mt[4 * i] = x[i];
        }
        mbar_arrive(&S.in_ready[slot]);
        if (tracing && warp == kInvWarp0 && lane == 0) { long long* tp_ = a.trace + ((size_t)blockIdx.x * nblocks + nb) * 32 + 3; tp_[0] = (long long)globaltimer_ns(); tp_[16] = clock64(); }
      }
    }
    if (CL && warp >= kCommWarp0) {
      // ------------------------------------------------------------------ clustered topology: gather h_b
      // every worker has added its partial to the grid-sum words of h_b (one atomic per (system, marker): the only L2 hop of a
      // block); these warps wait for the words, all copies of a word in flight at once, and hand the total (an integer: the same
      // on every solver) to the solve warps through shared memory -- the solve warps never wait on L2 themselves.
      const int ct = tid - kCommWarp0 * 32;  // 0..127
      const unsigned long long t_start = globaltimer_ns();
      for (int b = 0; b < nblocks; b++) {
        const int slot = b & 1;
        // h_b cannot be complete before the step of block b - 2 is published (the workers' G(b) follows U(b - 2)): sleep on that
        // barrier, not on the words, so that a long solve chain is not slowed by these warps' polls.  The hsum slot is next used by
        // block b + 2 for the same reason.
        if (b >= 2) mbar_wait(&S.solve_done[(b - 2) % sring], (uint32_t)((b - 2) / sring) & 1u, dead, a.s.err);
        for (int pair = ct; pair < ns * 128; pair += 128) {
          long long tot = 0;
          if (!dead) {
            int ab = 0;
            tot = grid_wait_total(a.hsum + hsum_word(b, ns, pair >> 7, pair & 127), true, W, a.s.err, t_start, &ab, kPollBackoffNs);
            if (__shfl_sync(0xffffffffu, ab, 0)) { dead = true; tot = 0; }
          }
          hsum[(size_t)slot * ns * 128 + pair] = tot;
        }
        mbar_arrive(&S.h_ready[slot]);
        if (b == 0 && ct == 0 && cluster == 0 && a.started) {  // every worker has added its partial: the whole grid is resident
          *reinterpret_cast<volatile unsigned int*>(a.started) = a.started_val;
          __threadfence_system();
        }
        if (tracing && ct == 0) { long long* tp_ = a.trace + ((size_t)blockIdx.x * nblocks + b) * 32 + 4; tp_[0] = (long long)globaltimer_ns(); tp_[16] = clock64(); }
        // until the partials of the next block arrive these warps are idle: three of them take one tile each of the lower-
        // triangular product dE = T r of the block they just delivered ((2,2), (3,2), (3,3)); the solve warps add the tile sums in
        // the same order as when they compute all tiles themselves, so the result is bit-identical to the flat topology
        if (full_inv && !sc[0].done) {
          named_bar(4, 256);  // r of all 128 markers is in shared memory
          const int hw = warp - kCommWarp0;  // 0: tile (2,2); 1: (3,2); 2: (3,3)
          if (hw < 3) {
            const int tw = hw == 0 ? 2 : 3, tt = hw == 1 ? 2 : hw == 0 ? 2 : 3;
            const float* Gb = Gs + (size_t)(b % sring) * 10 * kTileF;
            const float* trow = Gb + (size_t)tri(tw, tt) * kTileF + lane * kTS;
            const float* rv4 = rb + 32 * tt;
            float fa[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int k4 = 0; k4 < 8; k4++) {
              const float4 tv = *reinterpret_cast<const float4*>(trow + 4 * k4);
              const float4 rv = *reinterpret_cast<const float4*>(rv4 + 4 * k4);
              fa[0] = fmaf(tv.x, rv.x, fa[0]); fa[1] = fmaf(tv.y, rv.y, fa[1]);
              fa[2] = fmaf(tv.z, rv.z, fa[2]); fa[3] = fmaf(tv.w, rv.w, fa[3]);
            }
            rb[128 + hw * 32 + lane] = (fa[0] + fa[1]) + (fa[2] + fa[3]);
          }
          named_bar(5, 256);
        }
      }
    }
    if (full_inv && warp < 4) {
      // ------------------------------------------------------------------ one system on four solve warps
      // warp w owns markers 32w .. 32w+31 of the block (lane = marker)
      const int w = warp;
      float* mxs = cs + 64;  // [2][4] block maxima of |dE| per warp, double buffered by block parity
      for (int b = 0; b < nblocks; b++) {
        const int nvalid = min(128, p - b * 128);
        const int slot = b % sring;
        const float* Gb = Gs + (size_t)slot * 10 * kTileF;
        const MarkerCol* mc = mcol + slot * 128;
        mbar_wait(&S.in_ready[slot], (uint32_t)(b / sring) & 1u, dead, a.s.err);
        const SysScalars Sy = sc[0];
        const MarkerSys* mk = msys + (size_t)slot * 128;
        const MarkerDraws* drb = drw + (size_t)slot * 128;
        const int jj = 32 * w + lane;
        float g;
        {
          long long qq = 0;
          uint32_t spins = 0;
          if (CL) {
            mbar_wait(&S.h_ready[b & 1], (uint32_t)(b >> 1) & 1u, dead, a.s.err);
            qq = dead ? 0 : hsum[(size_t)(b & 1) * 128 + jj];
          } else if (a.world > 1) {
            const unsigned long long gen = a.gen0 + (unsigned long long)b;
            const unsigned long long tagx = tag_of(gen / kRing);
            const unsigned long long* gx = a.hx[a.rank] + ((size_t)(gen % kRing) * a.world) * 128 + jj;
            // the words of all ranks in flight at once (one NVLink-written L2 round trip, not `world` of them)
            unsigned long long wv[8];
            while (!dead) {
              bool ok = true;
#pragma unroll
              for (int src = 0; src < 8; src++) {
                wv[src] = src < a.world ? ld_relaxed_sys_u64(gx + (size_t)src * 128) : tagx;
                ok = ok && word_ok(wv[src], tagx);
              }
              if (__all_sync(0xffffffffu, ok)) break;
              if (++spins > kSpin || ((spins & 255u) == 255u && *reinterpret_cast<volatile int*>(a.s.err) != 0)) { dead = true; atomicCAS(a.s.err, 0, 3); }
            }
#pragma unroll
            for (int src = 0; src < 8; src++) qq += dead ? 0 : word_val(wv[src]);  // tag-only filler words carry value 0
          } else {
            const unsigned long long* gq = a.hred + (size_t)(b % kRing) * 128 + jj;
            const unsigned long long tagb = tag_of((unsigned long long)(b / kRing));
            unsigned long long wv = 0;
            while (!dead) {
              wv = ld_relaxed_u64(gq);
              if (__all_sync(0xffffffffu, word_ok(wv, tagb))) break;
              if (++spins > kSpin || ((spins & 255u) == 255u && *reinterpret_cast<volatile int*>(a.s.err) != 0)) { dead = true; atomicCAS(a.s.err, 0, 3); }
            }
            qq = dead ? 0 : word_val(wv);
          }
          if (w == 0) SSTAMPW(b, 8);
          if (!CL && b == 0 && w == 0 && lane == 0 && a.started) {  // flat topology: the first reduced h means every worker is resident
            *reinterpret_cast<volatile unsigned int*>(a.started) = a.started_val;
            __threadfence_system();
          }
          g = (float)((double)qq * (double)Sy.e_q);
        }
        if (D > 0 && b > 0) {
          mbar_wait(&S.corr_ready[0], (uint32_t)(b - 1) & 1u, dead, a.s.err);
          g -= tcor[(b & 1) * ns * 128 + jj];
        }
        if (w == 0) SSTAMPW(b, 9);
        const float av = mk[jj].a;
        const float r = fmaf(av, g, mk[jj].c);
        float de = 0.0f;
        if (Sy.done) {
          dehist[jj] = 0.0f;
          __syncwarp();
          if (lane == 0) mbar_arrive(&S.de_ready[0][w]);
        } else {
          // dE = T r: all right-hand sides through shared memory, then every warp takes its 32 rows of the lower-triangular
          // product at once -- no dependent 32-marker steps left in the chain
          rb[jj] = r;
          named_bar(4, CL ? 256 : 128);
#pragma unroll
          for (int t = 0; t < 4; t++) {
            if (CL && t >= 2) {  // tiles (2,2), (3,2), (3,3) come from the comm warps: same tile sums, added in the same order
              if (t == 2) named_bar(5, 256);
              if (t <= w) de += rb[128 + (w == 2 ? 0 : t - 1) * 32 + lane];
              continue;
            }
            if (t <= w) {
              const float* trow = Gb + (size_t)tri(w, t) * kTileF + lane * kTS;
              const float* rv4 = rb + 32 * t;
              float fa[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
              for (int k4 = 0; k4 < 8; k4++) {
                const float4 tv = *reinterpret_cast<const float4*>(trow + 4 * k4);
                const float4 rv = *reinterpret_cast<const float4*>(rv4 + 4 * k4);
                fa[0] = fmaf(tv.x, rv.x, fa[0]); fa[1] = fmaf(tv.y, rv.y, fa[1]);
                fa[2] = fmaf(tv.z, rv.z, fa[2]); fa[3] = fmaf(tv.w, rv.w, fa[3]);
              }
              de += (fa[0] + fa[1]) + (fa[2] + fa[3]);
            }
          }
          dehist[jj] = de;
          __syncwarp();
          if (lane == 0) mbar_arrive(&S.de_ready[0][w]);
        }
        if (w == 3) SSTAMPW(b, 10);
        // block maximum of |dE| over the four warps -> the fixed-point scale of the published step
        float mx = fabsf(de);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if (lane == 0) mxs[(b & 1) * 4 + w] = mx;
        named_bar(3, 128);
        mx = fmaxf(fmaxf(mxs[(b & 1) * 4 + 0], mxs[(b & 1) * 4 + 1]), fmaxf(mxs[(b & 1) * 4 + 2], mxs[(b & 1) * 4 + 3]));
        // frexp exponent of the block maximum by exponent-field arithmetic (mx = m 2^ex, 0.5 <= m < 1; subnormals clamp below anyway)
        int ex = 0;
        if (mx > 0.0f && mx < 3.0e38f) ex = (int)((__float_as_uint(mx) >> 23) & 0xFFu) - 126;
        if (ex < -90) ex = -90;
        const float dq = __uint_as_float((uint32_t)(ex - 30 + 127) << 23), dqinv = __uint_as_float((uint32_t)(30 - ex + 127) << 23);
        if (!(mx < 3.0e38f)) atomicExch(a.s.err, 4);
        unsigned long long* wv = a.dew + (size_t)b * kDewStride;
        const bool valid = jj < nvalid && !Sy.done;
        const int qv = valid ? __float2int_rn(de * dqinv) : 0;
        if (CL) {  // the step goes straight into the inbox of each of this cluster's workers
          const uint32_t off = dein_u32 + (uint32_t)((b & 1) * kDeStride + jj) * 4u, boff = smem_u32(&S.de_in[b & 1]);
#pragma unroll
          for (int wr = 1; wr <= kClWorkers; wr++) st_async_u32(mapa_u32(off, (uint32_t)wr), (uint32_t)qv, mapa_u32(boff, (uint32_t)wr));
          if (w == 3 && lane == 0) {
            const uint32_t soff = dein_u32 + (uint32_t)((b & 1) * kDeStride + 128) * 4u;
#pragma unroll
            for (int wr = 1; wr <= kClWorkers; wr++) st_async_u32(mapa_u32(soff, (uint32_t)wr), __float_as_uint(dq), mapa_u32(boff, (uint32_t)wr));
          }
        } else {
          st_relaxed_u64(wv + jj, ((unsigned long long)(uint32_t)qv << 32) | a.tag);
          if (w == 3 && lane == 0) st_relaxed_u64(wv + 128, ((unsigned long long)__float_as_uint(dq) << 32) | a.tag);
        }
        if (w == 3) SSTAMPW(b, 11);
        if (valid && writer) {
          const float deq = (float)qv * dq;  // the step actually applied to E (a 31-bit integer times a power of two, rounded once)
          const MarkerSys in = mk[jj];
          const float bnew = fmaf(deq, (MODEL == M_EMBA) ? 0.5f : 1.0f, in.b0);
          float vnew = in.vbj;
          if (MODEL == M_EMBA) vnew = (Sy.Sb + bnew * bnew) / (Sy.df + 1.0f);
          if (MODEL == M_BA || MODEL == M_BL) vnew = (Sy.Sb + bnew * bnew) / drb[jj].chi;
          const int j = mc[jj].j;
          a.s.b[j] = bnew;
          if (model_rule_writes_vbj(MODEL) && a.s.vbv) a.s.vbv[j] = vnew;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.solve_done[slot]);
      }
    }
    // -------------------------------------------------------------------- solve warps (one system at a time)
    if (!full_inv && warp < nsw) {
      for (int b = 0; b < nblocks; b++) {
        const int nvalid = min(128, p - b * 128);
        const int slot = b % sring;
        const float* Gb = Gs + (size_t)slot * 10 * kTileF;
        const MarkerCol* mc = mcol + slot * 128;
        mbar_wait(&S.in_ready[slot], (uint32_t)(b / sring) & 1u, dead, a.s.err);
        for (int s = warp; s < ns; s += kSolveWarps) {
          const SysScalars Sy = sc[s];
          const MarkerSys* mk = msys + ((size_t)slot * ns + s) * 128;
          const MarkerDraws* drb = drw + ((size_t)slot * ns + s) * 128;
          float g[4], de[4];
          {
            long long qq[4] = {0, 0, 0, 0};
            uint32_t spins = 0;
            if (CL) {
              mbar_wait(&S.h_ready[b & 1], (uint32_t)(b >> 1) & 1u, dead, a.s.err);
#pragma unroll
              for (int t = 0; t < 4; t++) qq[t] = dead ? 0 : hsum[(size_t)((b & 1) * ns + s) * 128 + 32 * t + lane];
            } else if (a.world > 1) {
              const unsigned long long gen = a.gen0 + (unsigned long long)b;
              const unsigned long long tagx = tag_of(gen / kRing);
              const unsigned long long* gx = a.hx[a.rank] + ((size_t)(gen % kRing) * a.world * ns + s) * 128;
              for (int src = 0; src < a.world; src++) {
                const unsigned long long* gq = gx + (size_t)src * ns * 128;
                long long w4[4] = {0, 0, 0, 0};
                while (!dead) {
                  bool ok = true;
#pragma unroll
                  for (int t = 0; t < 4; t++) {
                    const unsigned long long w = ld_relaxed_sys_u64(gq + 32 * t + lane);
                    ok = ok && word_ok(w, tagx);
                    w4[t] = word_val(w);
                  }
                  if (__all_sync(0xffffffffu, ok)) break;
                  if (++spins > kSpin || ((spins & 255u) == 255u && *reinterpret_cast<volatile int*>(a.s.err) != 0)) { dead = true; atomicCAS(a.s.err, 0, 3); }
                }
#pragma unroll
                for (int t = 0; t < 4; t++) qq[t] += w4[t];
              }
            } else {
              const unsigned long long* gq = a.hred + ((size_t)(b % kRing) * ns + s) * 128;
              const unsigned long long tagb = tag_of((unsigned long long)(b / kRing));
              while (!dead) {
                bool ok = true;
#pragma unroll
                for (int t = 0; t < 4; t++) {
                  const unsigned long long w = ld_relaxed_u64(gq + 32 * t + lane);
                  ok = ok && word_ok(w, tagb);
                  qq[t] = word_val(w);
                }
                if (__all_sync(0xffffffffu, ok)) break;
                if (++spins > kSpin || ((spins & 255u) == 255u && *reinterpret_cast<volatile int*>(a.s.err) != 0)) { dead = true; atomicCAS(a.s.err, 0, 3); }
              }
            }
            if (s == 0) SSTAMP(b, 8);
            if (!CL && b == 0 && s == 0 && lane == 0 && a.started) {
              *reinterpret_cast<volatile unsigned int*>(a.started) = a.started_val;
              __threadfence_system();
            }
#pragma unroll
            for (int t = 0; t < 4; t++) {
              g[t] = (float)((double)qq[t] * (double)Sy.e_q);
              de[t] = 0.0f;
            }
          }
          if (D > 0 && b > 0) {
            mbar_wait(&S.corr_ready[s], (uint32_t)(b - 1) & 1u, dead, a.s.err);
#pragma unroll
            for (int t = 0; t < 4; t++) g[t] -= tcor[((b & 1) * ns + s) * 128 + 32 * t + lane];
          }
          if (centred) {  // x_c'e_true = x'e_stored + c * sx with c as of the residual h_b was taken from
            const float cuse = cs[2 * s + ((D > 0 && b > 0) ? 1 : 0)];
#pragma unroll
            for (int t = 0; t < 4; t++) g[t] = fmaf(cuse, mc[32 * t + lane].sx, g[t]);
          }
          if (s == 0) SSTAMP(b, 9);
          float nb[4] = {0.f, 0.f, 0.f, 0.f}, nd[4] = {1.f, 1.f, 1.f, 1.f}, nv[4] = {1.f, 1.f, 1.f, 1.f};
          float* dh = dehist + s * 128;
          if (Sy.done) {
            // converged system (emEN): no update
            if (D > 0) {
#pragma unroll
              for (int d = 0; d < 4; d++) dh[32 * d + lane] = 0.0f;
              __syncwarp();
              if (lane == 0) for (int d = 0; d < 4; d++) mbar_arrive(&S.de_ready[s][d]);
            }
          } else if (kLinear) {
            float r[4], av[4];
#pragma unroll
            for (int t = 0; t < 4; t++) { av[t] = mk[32 * t + lane].a; r[t] = fmaf(av[t], g[t], mk[32 * t + lane].c); }
            float* rbs = rb + warp * 32;
#pragma unroll
            for (int d = 0; d < 4; d++) {
              float acc;
              if (use_inv) {
                // de_d = M_d r_d : broadcast r_d through shared memory, 128-bit loads down the k axis
                __syncwarp();
                rbs[lane] = r[d];
                __syncwarp();
                const float* mt = Mt + ((size_t)(slot * ns + s) * 4 + d) * 8 * kMS + 4 * lane;
                float ac[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int k4 = 0; k4 < 8; k4++) {
                  const float4 mv = *reinterpret_cast<const float4*>(mt + k4 * kMS);
                  const float4 rv = *reinterpret_cast<const float4*>(rbs + 4 * k4);
                  ac[0] = fmaf(mv.x, rv.x, ac[0]); ac[1] = fmaf(mv.y, rv.y, ac[1]);
                  ac[2] = fmaf(mv.z, rv.z, ac[2]); ac[3] = fmaf(mv.w, rv.w, ac[3]);
                }
                acc = (ac[0] + ac[1]) + (ac[2] + ac[3]);
              } else {
                // in-warp forward substitution of the 32x32 unit-lower-triangular diagonal block
                const float* grow = Gb + (size_t)tri(d, d) * kTileF + lane * kTS;
                float ag[32];
#pragma unroll
                for (int k4 = 0; k4 < 8; k4++) {
                  const float4 gv = *reinterpret_cast<const float4*>(grow + 4 * k4);
                  ag[4 * k4 + 0] = -av[d] * gv.x; ag[4 * k4 + 1] = -av[d] * gv.y;
                  ag[4 * k4 + 2] = -av[d] * gv.z; ag[4 * k4 + 3] = -av[d] * gv.w;
                }
                // x_k (final) -> x_{k+1} is the chain.  The broadcast of lane k+1 is taken off it: its value BEFORE step k is shuffled
                // out ahead, and every lane applies step k to it with the owner's own coefficient and FMA (same bits).
                float x = r[d];
                float xk = __shfl_sync(0xffffffffu, x, 0);
                const float* gcol = Gb + (size_t)tri(d, d) * kTileF;
#pragma unroll
                for (int k = 0; k < 31; k++) {
                  const float pre = __shfl_sync(0xffffffffu, x, k + 1);
                  const float cn = -mk[32 * d + k + 1].a * gcol[(k + 1) * kTS + k];
                  if (lane > k) x = fmaf(ag[k], xk, x);
                  xk = fmaf(cn, xk, pre);
                }
                acc = x;
              }
              de[d] = acc;
              __syncwarp();
              rbs[lane] = acc;
              if (D > 0) dh[32 * d + lane] = acc;
              __syncwarp();
              if (D > 0 && lane == 0) mbar_arrive(&S.de_ready[s][d]);
              if (d < 3) {
#pragma unroll
                for (int d2 = 0; d2 < 4; d2++) {
                  if (d2 > d) {
                    // r_d2 -= a * sum_k G[32 d2 + lane][32 d + k] * de_d[k]
                    const float* grow = Gb + (size_t)tri(d2, d) * kTileF + lane * kTS;
                    float fa[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                    for (int k4 = 0; k4 < 8; k4++) {
                      const float4 gv = *reinterpret_cast<const float4*>(grow + 4 * k4);
                      const float4 dv = *reinterpret_cast<const float4*>(rbs + 4 * k4);
                      fa[0] = fmaf(gv.x, dv.x, fa[0]); fa[1] = fmaf(gv.y, dv.y, fa[1]);
                      fa[2] = fmaf(gv.z, dv.z, fa[2]); fa[3] = fmaf(gv.w, dv.w, fa[3]);
                    }
                    r[d2] = fmaf(-av[d2], (fa[0] + fa[1]) + (fa[2] + fa[3]), r[d2]);
                  }
                }
              }
            }
          } else {
            // The chain: g of marker jj -> rule -> step -> g of marker jj + 1.  Lane jj + 1 owns that g, but its broadcast does not
            // have to sit on the chain: its value BEFORE step jj is shuffled out while the rule of jj is evaluated, and every lane
            // applies step jj to it with the same fused multiply-add the owner uses (same bits).  Chain per marker = rule + one FMA.
            // The marker's own inputs (coefficients, draws, xx) are read one marker ahead: their shared-memory latency would otherwise
            // open every link of the chain (the loop has no early exit for the same reason: markers past the end of the last block
            // are walked with a zero step).
            float gc = __shfl_sync(0xffffffffu, g[0], 0);
            MarkerSys in_n = mk[0];
            MarkerDraws dr_n;
            if (kGibbs) dr_n = drb[0];
            else { dr_n.z1 = dr_n.z2 = dr_n.u = 0.0f; dr_n.chi = 1.0f; }
            float xx_n = mc[0].xx;
#pragma unroll
            for (int t = 0; t < 4; t++) {
              // unroll measured on wgr BayesB at 10k x 50k (profiles/r2_wgr_bayesb_fold_variants.txt): 4 -> 2.93, 8 -> 2.54, 16 -> 2.47, 32 -> 3.8 ms
#pragma unroll (MODEL == M_KMUP ? 16 : 8)
              for (int i = 0; i < 32; i++) {
                const int jj = 32 * t + i;
                const bool valid = jj < nvalid;
                const MarkerSys in = in_n;
                const MarkerDraws dr = dr_n;
                const float xxj_ = xx_n;
                {
                  const int jn = jj < 127 ? jj + 1 : 127;
                  in_n = mk[jn];
                  if (kGibbs) dr_n = drb[jn];
                  xx_n = mc[jn].xx;
                }
                // marker jj + 1 as its owner has it now (steps 0 .. jj-1 applied), and the Gram element that couples it to marker jj
                const float gnext = i < 31 ? __shfl_sync(0xffffffffu, g[t], i + 1) : __shfl_sync(0xffffffffu, g[t < 3 ? t + 1 : 3], 0);
                const float Gnext = i < 31 ? Gb[(size_t)tri(t, t) * kTileF + i * kTS + i + 1] : Gb[(size_t)tri(t < 3 ? t + 1 : 3, t) * kTileF + i * kTS];
                RuleOut ro;
                if (kSlabDraw) {
                  // ||e2||^2 - ||e1||^2 in closed form: KMUP and BayesDpi (:953-955) compare the two draws, BayesB/C the draw against
                  // b = 0 (:673):   q = (b2 - b1) (xx (b1 + b2 - 2 b0) - 2 g)   resp.   q = b1 (xx (2 b0 - b1) + 2 g),   b1 = a g + c.
                  // Both factors are affine in g.  C times the second one's coefficients were formed with the marker's other inputs one
                  // block ahead (P in dr.z1; Q in dr.chi, or in in.vbj for the rules that draw a chi-square and recompute vbj), so the
                  // chain per marker is g -> two FMAs side by side -> multiply -> compare -> select the step -> FMA into the next g.
                  // (Forming P and Q inside this loop instead was measured slower: the chain's warp is issue-bound too.)
                  constexpr bool kTwoDraws = MODEL == M_KMUP || MODEL == M_BDPI, kChi = MODEL == M_BB || MODEL == M_BDPI;
                  const float b2 = dr.z2, b1 = fmaf(gc, in.a, in.c);
                  const float f1 = kTwoDraws ? fmaf(gc, -in.a, b2 - in.c) : b1;
                  const bool take = f1 * fmaf(gc, dr.z1, kChi ? in.vbj : dr.chi) < dr.u;  // C q < threshold
                  ro.de = take ? fmaf(gc, in.a, in.c - in.b0) : b2 - in.b0;
                  ro.b = take ? b1 : b2; ro.d = take ? 1.0f : 0.0f;
                  ro.vbj = kChi ? (Sy.Sb + ro.b * ro.b) / dr.chi : in.vbj;
                } else if (kSlabEM) {
                  const float xxj = xxj_, b1 = fmaf(gc, in.a, in.c);
                  const float LR = Sy.Pi0 * expf(Sy.C * (b1 * fmaf(xxj, 2.0f * in.b0 - b1, 2.0f * gc)));
                  ro.d = __frcp_rn(1.0f + LR);
                  ro.b = b1 * ro.d;
                  ro.de = ro.b - in.b0;
                  ro.vbj = MODEL == M_EMBB ? (Sy.Sb + ro.b * ro.b) / (Sy.df + 1.0f) : in.vbj;
                } else if (kFoldEM) {
                  const float OLS = fmaf(xxj_, in.b0, gc);
                  if (MODEL == M_EMBL) {  // in.a = 0.5/(Lmb2 + xx), in.c = 0.5/(xx + cxx)
                    const float Half = OLS * in.c;
                    const float G = (OLS > 0.0f ? OLS - Sy.lmb1 : OLS + Sy.lmb1) * in.a;
                    const bool keep = OLS > 0.0f ? G > 0.0f : G < 0.0f;
                    ro.b = keep ? G + Half : Half;
                    ro.d = 1.0f;
                  } else {                // in.a = 1/(Lmb2 + xx) (emEN) or 1/xx (lasso)
                    const float l1 = MODEL == M_LASSO ? Sy.lmb : Sy.lmb1;
                    const float t = OLS > 0.0f ? fmaxf(OLS - l1, 0.0f) : fminf(OLS + l1, 0.0f);
                    ro.b = t * in.a;
                    ro.d = MODEL == M_LASSO ? fabsf(OLS) - fabsf(t) : 1.0f;  // lasso: |x'e~| - |b xx| for the next penalty
                  }
                  ro.de = ro.b - in.b0;
                  ro.vbj = in.vbj;
                } else {
                  ro = marker_rule<MODEL>(gc, xxj_, in.b0, in.vbj, Sy, dr);
                }
                if (!valid) ro.de = 0.0f;
                if (lane == i && valid) { nb[t] = ro.b; nd[t] = ro.d; nv[t] = ro.vbj; de[t] = ro.de; }
                // row jj of the Gram block to the right of (and inside) its diagonal tile: stored as tile (tt, t)
#pragma unroll
                for (int tt = 0; tt < 4; tt++)
                  if (tt >= t) g[tt] = fmaf(-Gb[(size_t)tri(tt, t) * kTileF + i * kTS + lane], ro.de, g[tt]);
                gc = fmaf(-Gnext, ro.de, gnext);
              }
              if (D > 0) {
                dh[32 * t + lane] = de[t];
                __syncwarp();
                if (lane == 0) mbar_arrive(&S.de_ready[s][t]);
              }
            }
          }
          if (centred) {  // c += sum_k mean_k dE_k (this block's contribution to the mean of the fitted values)
            float sm = 0.0f;
#pragma unroll
            for (int t = 0; t < 4; t++) sm = fmaf(mc[32 * t + lane].sx, de[t], sm);
            sm = warp_sum(sm) * inv_n;
            __syncwarp();
            if (lane == 0) { const float cc = cs[2 * s]; cs[2 * s + 1] = cc; cs[2 * s] = cc + sm; }
            __syncwarp();
          }
          if (s == 0) SSTAMP(b, 10);
          // quantise dE to 31-bit fixed point relative to the block maximum and publish it
          float mx = fmaxf(fmaxf(fabsf(de[0]), fabsf(de[1])), fmaxf(fabsf(de[2]), fabsf(de[3])));
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
          int ex = 0;
          if (mx > 0.0f && mx < 3.0e38f) frexpf(mx, &ex);
          if (ex < -90) ex = -90;
          const float dq = ldexpf(1.0f, ex - 30), dqinv = ldexpf(1.0f, 30 - ex);
          if (!(mx < 3.0e38f)) atomicExch(a.s.err, 4);
          unsigned long long* wv = a.dew + ((size_t)b * ns + s) * kDewStride;
          int qv[4];
#pragma unroll
          for (int t = 0; t < 4; t++) {
            const int jj = 32 * t + lane;
            const bool valid = jj < nvalid && !Sy.done;
            qv[t] = valid ? __float2int_rn(de[t] * dqinv) : 0;
            if (CL) {
              const uint32_t off = dein_u32 + (uint32_t)(((b & 1) * ns + s) * kDeStride + jj) * 4u, boff = smem_u32(&S.de_in[b & 1]);
#pragma unroll
              for (int wr = 1; wr <= kClWorkers; wr++) st_async_u32(mapa_u32(off, (uint32_t)wr), (uint32_t)qv[t], mapa_u32(boff, (uint32_t)wr));
            } else {
              st_relaxed_u64(wv + jj, ((unsigned long long)(uint32_t)qv[t] << 32) | a.tag);
            }
          }
          if (CL) {
            if (lane == 0) {
              const uint32_t soff = dein_u32 + (uint32_t)(((b & 1) * ns + s) * kDeStride + 128) * 4u, boff = smem_u32(&S.de_in[b & 1]);
#pragma unroll
              for (int wr = 1; wr <= kClWorkers; wr++) st_async_u32(mapa_u32(soff, (uint32_t)wr), __float_as_uint(dq), mapa_u32(boff, (uint32_t)wr));
            }
          } else if (lane == 0) st_relaxed_u64(wv + 128, ((unsigned long long)__float_as_uint(dq) << 32) | a.tag);
          if (s == 0) SSTAMP(b, 11);
#pragma unroll
          for (int t = 0; t < 4; t++) {
            const int jj = 32 * t + lane;
            if (jj < nvalid && !Sy.done && writer) {
              const float deq = (float)qv[t] * dq;  // the step actually applied to E (a 31-bit integer times a power of two, rounded once)
              const MarkerSys in = mk[jj];
              float bnew, dnew = nd[t], vnew = nv[t];
              if (kLinear) {
                bnew = fmaf(deq, (MODEL == M_EMBA) ? 0.5f : 1.0f, in.b0);
                if (MODEL == M_EMBA) vnew = (Sy.Sb + bnew * bnew) / (Sy.df + 1.0f);
                if (MODEL == M_BA || MODEL == M_BL) vnew = (Sy.Sb + bnew * bnew) / drb[jj].chi;
              } else {
                bnew = nb[t];
              }
              const int j = mc[jj].j;
              a.s.b[(size_t)s * p + j] = bnew;
              if (model_has_d(MODEL) && a.s.d) a.s.d[(size_t)s * p + j] = dnew;
              if (model_rule_writes_vbj(MODEL) && a.s.vbv) a.s.vbv[(size_t)s * p + j] = vnew;
            }
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.solve_done[slot]);
      }
      if (centred && a.cshift && lane == 0 && writer)
        for (int s = warp; s < ns; s += kSolveWarps) a.cshift[s] = cs[2 * s];
    }
  } else if (warp < kPreWarp0) {
    // -------------------------------------------------------------------- cross-Gram correction (D = 1)
    // thread = row i of block b+1:  t[s][i] = sum_k (x_{b+1,i}' x_{b,k}) dE_b[s][k], consumed 32 markers at a time
    if (D > 0) {
      constexpr int kCS = 256;  // floats per Gram row when the band is 2 (the only band with D = 1): immediate offsets
      const int i = (warp - kCorrWarp0) * 32 + lane;
      for (int b = 0; b + 1 < nblocks; b++) {
        // cross block of block b+1, stored transposed: ct[k * gstride] = x_{b,k}' x_{b+1,i}  (a warp reads 128 B per k)
        const float* ct = a.gram + (size_t)(b + 1) * 128 * kCS + 128 + i;
        // two 32-marker chunks of the row in flight at any time (64 registers): chunk d+2 is fetched into the set that
        // chunk d just released, two solve steps (~1000 cycles) before it is needed -- an L2 hit thanks to the prefetch
        float c0[32], c1[32];
#pragma unroll
        for (int k = 0; k < 32; k++) c0[k] = __ldg(ct + k * kCS);
#pragma unroll
        for (int k = 0; k < 32; k++) c1[k] = __ldg(ct + (32 + k) * kCS);
        if (b + 2 < nblocks) {  // pull the cross block of block b+2 into L2 now: row i of it, 4 lines of 128 B
          const float* nxt = a.gram + ((size_t)(b + 2) * 128 + i) * kCS + 128;
#pragma unroll
          for (int q4 = 0; q4 < 4; q4++) prefetch_l2(nxt + 32 * q4);
        }
        auto chunk = [&](const float (&cv)[32], int d) {
          for (int s = 0; s < ns; s++) {
            mbar_wait(&S.de_ready[s][d], (uint32_t)b & 1u, dead, a.s.err);
            const float4* dv = reinterpret_cast<const float4*>(dehist + s * 128 + 32 * d);
            float fa[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int k4 = 0; k4 < 8; k4++) {
              const float4 v = dv[k4];
              fa[0] = fmaf(cv[4 * k4 + 0], v.x, fa[0]); fa[1] = fmaf(cv[4 * k4 + 1], v.y, fa[1]);
              fa[2] = fmaf(cv[4 * k4 + 2], v.z, fa[2]); fa[3] = fmaf(cv[4 * k4 + 3], v.w, fa[3]);
            }
            const float part = (fa[0] + fa[1]) + (fa[2] + fa[3]);
            float* tc = tcor + (((b + 1) & 1) * ns + s) * 128 + i;  // buffer of block b+1 (a late solve warp may still read block b's)
            if (d == 0) *tc = part; else *tc += part;
            if (d == 3) mbar_arrive(&S.corr_ready[s]);
          }
        };
        chunk(c0, 0);
#pragma unroll
        for (int k = 0; k < 32; k++) c0[k] = __ldg(ct + (64 + k) * kCS);
        chunk(c1, 1);
#pragma unroll
        for (int k = 0; k < 32; k++) c1[k] = __ldg(ct + (96 + k) * kCS);
        chunk(c0, 2);
        chunk(c1, 3);
      }
    }
  } else {
    // -------------------------------------------------------------------- prefetch of the solve inputs (ring of sring blocks)
    // thread ht = marker ht of the block.  Marker ids are fetched two blocks ahead and the per-marker scalars one block
    // ahead into registers, so the HBM round trips of these tiny gathers never sit on the per-block path.
    const int ht = (warp - kPreWarp0) * 32 + lane;  // 0..127
#define PSTAMP(k) do { if (tracing && ht == 0) { long long* tp_ = a.trace + ((size_t)blockIdx.x * nblocks + nb) * 32 + (k); tp_[0] = (long long)globaltimer_ns(); tp_[16] = clock64(); } } while (0)
    constexpr int kPipeSys = 2;  // systems whose scalars are register-pipelined (more systems: loaded in place)
    auto perm_at = [&](int blk) { const int pos = blk * 128 + ht; return (blk < nblocks && pos < p) ? a.perm[pos] : -1; };
    int j_cur = perm_at(0), j_nxt = perm_at(1);
    float xx_cur = j_cur >= 0 ? a.s.xx[j_cur] : 1.0f, sx_cur = (j_cur >= 0 && a.sx) ? a.sx[j_cur] : 0.0f, b_cur[kPipeSys], v_cur[kPipeSys];
#pragma unroll
    for (int s = 0; s < kPipeSys; s++) {
      b_cur[s] = (s < ns && j_cur >= 0) ? a.s.b[(size_t)s * p + j_cur] : 0.0f;
      v_cur[s] = (s < ns && j_cur >= 0 && model_has_vbj(MODEL) && a.s.vbv) ? a.s.vbv[(size_t)s * p + j_cur] : 1.0f;
    }
    const int rr0 = ht >> 3, c4 = ht & 7;
    for (int nb = 0; nb < nblocks; nb++) {
      const int slot = nb % sring;
      if (nb >= sring) mbar_wait(&S.solve_done[slot], (uint32_t)(nb / sring - 1) & 1u, dead, a.s.err);
      PSTAMP(0);
      // Gram triangle of block nb: linear rules read tile (hi, lo) = G[32 hi + r][32 lo + c];
      // the scalar chain reads the transposed triangle, stored in the same slots
      {
        float* Gb = Gs + (size_t)slot * 10 * kTileF;
        // with the precomputed block inverse the solver needs T_b (lower triangle), not the Gram block itself
        const int tstride = full_inv ? 128 : gstride;
        const float* src = full_inv ? a.tinv + (size_t)nb * 128 * 128 : a.gram + (size_t)nb * 128 * gstride;
#pragma unroll
        for (int it = 0; it < 20; it++) {
          constexpr int kHi[10] = {0, 1, 1, 2, 2, 2, 3, 3, 3, 3}, kLo[10] = {0, 0, 1, 0, 1, 2, 0, 1, 2, 3};
          const int tile = it >> 1, rr = rr0 + 16 * (it & 1);
          const int hi = kHi[tile], lo = kLo[tile];
          const int grow_ = kLinear ? 32 * hi + rr : 32 * lo + rr, gcol = kLinear ? 32 * lo + 4 * c4 : 32 * hi + 4 * c4;
          cp_async16_zfill(smem_u32(Gb + (size_t)tile * kTileF + rr * kTS + 4 * c4), src + (size_t)grow_ * tstride + gcol, 16u);
        }
        cp_async_commit();
      }
      PSTAMP(1);
      // issue the gathers of the following blocks now; they are consumed in the next iteration
      const int j_nn = perm_at(nb + 2);
      float xx_nxt = 1.0f, sx_nxt = 0.0f, b_nxt[kPipeSys], v_nxt[kPipeSys];
      if (j_nxt >= 0) { xx_nxt = a.s.xx[j_nxt]; if (a.sx) sx_nxt = a.sx[j_nxt]; }
#pragma unroll
      for (int s = 0; s < kPipeSys; s++) {
        b_nxt[s] = (s < ns && j_nxt >= 0) ? a.s.b[(size_t)s * p + j_nxt] : 0.0f;
        v_nxt[s] = (s < ns && j_nxt >= 0 && model_has_vbj(MODEL) && a.s.vbv) ? a.s.vbv[(size_t)s * p + j_nxt] : 1.0f;
      }
      {
        const int j = j_cur;
        MarkerCol mcv;
        mcv.xx = xx_cur; mcv.sx = sx_cur; mcv.j = j; mcv.pad = 0;
        mcol[slot * 128 + ht] = mcv;
        for (int s = 0; s < ns; s++) {
          MarkerSys in = {0.0f, 1.0f, 0.0f, 0.0f};
          if (j >= 0 && !sc[s].done) {
            if (s < kPipeSys) { in.b0 = b_cur[s < kPipeSys ? s : 0]; in.vbj = v_cur[s < kPipeSys ? s : 0]; }
            else {
              in.b0 = a.s.b[(size_t)s * p + j];
              in.vbj = (model_has_vbj(MODEL) && a.s.vbv) ? a.s.vbv[(size_t)s * p + j] : 1.0f;
            }
            MarkerDraws dr;
            dr.z1 = dr.z2 = dr.u = 0.0f; dr.chi = 1.0f;
            if (kGibbs) {
              dr = marker_draws(MODEL, (uint32_t)j, (uint32_t)sc[s].sweep, (uint32_t)(a.s.chain0 + s), sc[s].df, a.s.seed_lo, a.s.seed_hi);
              drw[((size_t)slot * ns + s) * 128 + ht] = dr;
            }
            if (kLinear) {
              const LinCoef lc = lin_coef<MODEL>(mcv.xx, in.b0, in.vbj, sc[s], dr);
              in.a = lc.a; in.c = lc.c;
            }
            if (kFoldEM) {
              if (MODEL == M_EMBL) { in.a = 0.5f / (sc[s].lmb2 + mcv.xx); in.c = 0.5f / (mcv.xx + sc[s].cxx); }
              else in.a = 1.0f / (MODEL == M_LASSO ? mcv.xx : sc[s].lmb2 + mcv.xx);
            }
            if (kSlabEM) {
              const float lmb = MODEL == M_EMBB ? sc[s].ve * (1.0f / in.vbj) : sc[s].lmb;
              const float ia = 1.0f / (mcv.xx + lmb);
              in.a = ia;                          // b1 = g * ia + c
              in.c = mcv.xx * in.b0 * ia;
            }
            if (kSlabDraw) {
              const float lmb = (MODEL == M_BB || MODEL == M_BDPI) ? sc[s].ve * (1.0f / in.vbj) : MODEL == M_BC ? sc[s].lmb : in.vbj;  // KMUP: vbj carries L[j]
              const float ia = 1.0f / (mcv.xx + lmb), sd = sqrtf(sc[s].ve * ia);
              const float ratio = MODEL == M_KMUP ? sc[s].pi_mix / (1.0f - sc[s].pi_mix) : sc[s].Pi0;
              in.a = ia;                                   // b1 = g * ia + c
              in.c = fmaf(mcv.xx * in.b0, ia, sd * dr.z1);
              dr.z2 = sd * dr.z2;                          // the excluded draw b2
              // accept b1 iff C*q < this.  BayesDpi: u < min(1, (1-pi) exp(-C q))  <=>  C q < log((1-pi)/u)
              if (MODEL == M_BDPI) dr.u = logf((1.0f - sc[s].Pi) / dr.u);
              else dr.u = (MODEL == M_KMUP && !(sc[s].pi_mix > 0.0f)) ? 3.0e38f : logf((1.0f / dr.u - 1.0f) / ratio);
              {  // the chain's second factor times C as P g + Q (see the chain): C (xx (b1 + b2 - 2 b0) - 2 g) resp. C (xx (2 b0 - b1) + 2 g)
                const bool two = MODEL == M_KMUP || MODEL == M_BDPI;
                const float P = sc[s].C * (two ? fmaf(mcv.xx, ia, -2.0f) : fmaf(-mcv.xx, ia, 2.0f));
                const float Q = sc[s].C * (mcv.xx * (two ? (in.c + dr.z2) - 2.0f * in.b0 : 2.0f * in.b0 - in.c));
                dr.z1 = P;
                if (MODEL == M_BB || MODEL == M_BDPI) in.vbj = Q;  // these rules recompute vbj from their chi-square draw
                else dr.chi = Q;                                   // KMUP, BayesC: no chi-square draw per marker
              }
              drw[((size_t)slot * ns + s) * 128 + ht] = dr;
            }
          }
          msys[((size_t)slot * ns + s) * 128 + ht] = in;
        }
      }
      PSTAMP(2);
      cp_async_wait<0>();
      if (use_inv) mbar_arrive(&S.raw_ready[slot]);
      else mbar_arrive(&S.in_ready[slot]);
      PSTAMP(7);
      j_cur = j_nxt; j_nxt = j_nn; xx_cur = xx_nxt; sx_cur = sx_nxt;
#pragma unroll
      for (int s = 0; s < kPipeSys; s++) { b_cur[s] = b_nxt[s]; v_cur[s] = v_nxt[s]; }
    }
#undef PSTAMP
  }
#undef SSTAMP
#undef SSTAMPW
  if (CL) {
    __syncthreads();
    cluster_sync_all();  // nobody leaves while a peer may still store into its shared memory
  }
}

template <int MODEL>
cudaError_t launch_model(const PipeArgs& a, size_t smem, cudaStream_t st) {
  PipeArgs args = a;
  if (a.cl) {
    cudaError_t e = cudaFuncSetAttribute(sweep_pipe_kernel<MODEL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(a.nclusters * kClSize); cfg.blockDim = dim3(kT); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = kClSize; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, sweep_pipe_kernel<MODEL, true>, args);
  }
  cudaError_t e = cudaFuncSetAttribute(sweep_pipe_kernel<MODEL, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  void* params[] = {&args};
  return cudaLaunchCooperativeKernel((void*)sweep_pipe_kernel<MODEL, false>, dim3(a.nworkers + 1), dim3(kT), params, smem, st);
}

// co-resident clusters of kClSize CTAs with `smem` bytes of dynamic shared memory each (0 on error)
template <int MODEL>
int max_clusters_model(size_t smem) {
  if (cudaFuncSetAttribute(sweep_pipe_kernel<MODEL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { cudaGetLastError(); return 0; }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = dim3(kClSize * 32); cfg.blockDim = dim3(kT); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = kClSize; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, sweep_pipe_kernel<MODEL, true>, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

}  // namespace

// Shared memory of one CTA (both roles use the same launch) and the largest tile ring that fits.
size_t sweep_pipe_smem(int rows_per_cta, int nsys, int model, int nbuf, int sring, int full_inv, int cl) {
  const size_t w = worker_layout(rows_per_cta, nsys, nbuf, cl != 0).total;
  const size_t s = solver_layout(nsys, model_is_gibbs(model), !full_inv && pipe_use_inv(model, nsys), sring, cl != 0).total;
  return (w > s ? w : s) + 1024;
}

// The clustered topology needs the solver's warps 4-7 free (comm warps) and no in-kernel 32 x 32 inverses.  At most three systems:
// four never fitted next to the partial inboxes the solver once had, and without them are not measured (the comm warps would
// wait for four words per thread one after the other).
bool sweep_pipe_cluster_ok(int model, int nsys, int full_inv) {
  return nsys <= 3 && !(!full_inv && pipe_use_inv(model, nsys));
}
// Every rule but KMUP2's, which always comes with a row mask (the pipelined sweep takes unmasked systems only).
int sweep_pipe_max_clusters(int model, size_t smem) {
  int n = 0;
  with_rule(model, [&](auto rule) {
    constexpr int M = decltype(rule)::value;
    if constexpr (M != M_KMUP2) n = max_clusters_model<M>(smem);
  });
  return n;
}

cudaError_t launch_sweep_pipe(const PipeArgs& a, cudaStream_t st) {
  const size_t smem = sweep_pipe_smem(a.rows_per_cta, a.s.nsys, a.model, a.nbuf, a.sring, a.tinv != nullptr, a.cl);
  cudaError_t e = cudaErrorInvalidValue;
  with_rule(a.model, [&](auto rule) {
    constexpr int M = decltype(rule)::value;
    if constexpr (M != M_KMUP2) e = launch_model<M>(a, smem, st);
  });
  return e;
}

}  // namespace bwgr
