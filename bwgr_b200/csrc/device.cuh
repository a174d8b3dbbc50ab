// device.cuh -- the inline-PTX wrappers that more than one kernel file uses, and the L2 grid-sum word.  Device code only: the
// kernel .cu files include it, the host layer (host.h, kernels.h) does not.
#pragma once
#include "kernels.h"

namespace bwgr {

// ---- shared memory, mbarriers ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// one elected lane of a converged warp: the form ptxas turns into back-to-back UTC*MMA issue (a plain `lane == 0` branch makes it
// wrap every tcgen05.mma in a per-lane loop, ~250 cycles per instruction)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return done != 0;
}
// Bounded wait of the Gram kernels: a protocol bug must not hang the GPU (it sets *err = 2 and lets the kernel drain).
constexpr uint32_t kMbarSpinLimit = 1u << 22;
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, int* err) {
  for (uint32_t spin = 0; spin < kMbarSpinLimit; spin++)
    if (mbar_try(bar, parity)) return true;
  atomicExch(err, 2);
  return false;
}
__device__ __forceinline__ void named_bar(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
// generic-proxy stores to shared memory -> visible to the tensor core (async proxy)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- cp.async ---------------------------------------------------------------------------------------------------------------
// 16 B, L2 only; src_bytes < 16 zero-fills the rest (0 = a zero chunk, nothing is read)
__device__ __forceinline__ void cp_async16_zfill(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
// 16 B, L2 only
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
// 4 B, through L1
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- global memory, timer ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ---- tcgen05: tensor memory and the int8 MMA ---------------------------------------------------------------------------------
// K-major operand, SWIZZLE_128B: 128-byte rows, 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t desc_k_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);  // start address, 16 B units
  d |= (uint64_t)1 << 16;                    // leading byte offset (unused for swizzled K-major) = 16 B
  d |= (uint64_t)(1024 >> 4) << 32;          // stride byte offset: 8 rows x 128 B
  d |= (uint64_t)1 << 46;                    // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                    // SWIZZLE_128B
  return d;
}
// kind::i8 instruction descriptor: D = S32, A = B = signed int8, B K-major, A K-major (a_mn = 0) or MN-major (1), M = 128, N
__host__ __device__ constexpr uint32_t idesc_i8(int N, int a_mn) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)(N >> 3) << 17) | ((128u >> 4) << 24);
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on `bar` when the MMAs issued so far have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// one warp: ncols TMEM columns, base address written to *dst (shared memory); the permit is given up at once
__device__ __forceinline__ void tmem_alloc(uint32_t* dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
// called by the allocating warp after a block-wide barrier that follows every thread's last TMEM access
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t ncols) {
  tc_fence_after();
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols) : "memory");
}
// 32 consecutive columns of this warp's 32 TMEM lanes (lane = row); complete after tmem_ld_wait()
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- the L2 grid sum (grid family, general MRR3, clustered sweep) ------------------------------------------------------------
// A sum over the CTAs of a grid lives in 64-bit words of global memory, zeroed before the launch: (fixed-point sum << 8) + arrivals.
// Every CTA adds its fixed-point partial, plus one, with a single atomic, so the low byte counts the CTAs that have added and the
// data is its own flag (one L2 hop, no fence, no barrier).  Integer sums are order-free: every CTA reads bit-identical totals.
// Same-address atomics serialise in L2, so each sum has kGridCopies copies (kernels.h) and CTA c adds to copy c % kGridCopies.
constexpr unsigned long long kGridTimeoutNs = 120000000000ull;  // two minutes without the grid: err = 3

__device__ __forceinline__ unsigned long long grid_word(double v) { return ((unsigned long long)__double2ll_rn(v) << 8) + 1ull; }
__device__ __forceinline__ int grid_word_count(unsigned long long w) { return (int)(w & 0xffull); }
__device__ __forceinline__ long long grid_word_value(unsigned long long w) { return (long long)w >> 8; }
// arrivals that complete copy c of a word in a grid of G CTAs (the CTAs with cta % kGridCopies == c)
__device__ __forceinline__ int grid_copy_count(int G, int c) { return (G + kGridCopies - 1 - c) / kGridCopies; }
// adds the partial v (fixed-point units) to a word; |v| >= 2^52 leaves the fixed-point range of the sum: err = 4
__device__ __forceinline__ void grid_add(unsigned long long* w, double v, int* err) {
  if (!(fabs(v) < 4503599627370496.0)) atomicExch(err, 4);
  atomicAdd(w, grid_word(v));
}
// the same with an integer partial (the sweep's exact fixed-point sums)
__device__ __forceinline__ void grid_add(unsigned long long* w, long long v, int* err) {
  if (!(v < 4503599627370496ll && v > -4503599627370496ll)) atomicExch(err, 4);
  atomicAdd(w, ((unsigned long long)v << 8) + 1ull);
}
// Warp-collective wait for the words of one marker, copy c at w + 32 c: returns the lane's total once the words of every lane with
// `on` set are complete.  Every 4096 spins lane 0 looks at the error flag and, two minutes after t_start, raises err = 3; either ends
// the wait for the whole warp with *abort = 1 (the total is then meaningless).  backoff_ns > 0: the warp sleeps that long between
// polls (it issues nothing meanwhile: a poller that shares its SM with a latency-bound chain leaves the chain the issue slots).
__device__ __forceinline__ long long grid_wait_total(const unsigned long long* w, bool on, int G, int* err, unsigned long long t_start,
                                                     int* abort, unsigned int backoff_ns = 0) {
  unsigned long long v[kGridCopies];
  unsigned int spins = 0;
  for (;;) {
    bool pending = false;
#pragma unroll
    for (int c = 0; c < kGridCopies; c++) v[c] = ld_relaxed_u64(w + c * 32);
#pragma unroll
    for (int c = 0; c < kGridCopies; c++) pending |= grid_word_count(v[c]) != grid_copy_count(G, c);
    if (!__any_sync(0xffffffffu, on && pending)) break;
    if (backoff_ns) __nanosleep(backoff_ns);
    if ((++spins & 0xfffu) == 0) {
      int ab = 0;
      if ((threadIdx.x & 31) == 0) {
        if (*reinterpret_cast<volatile int*>(err) != 0) ab = 1;
        else if (globaltimer_ns() - t_start > kGridTimeoutNs) { atomicExch(err, 3); ab = 1; }
        if (ab) *abort = 1;
      }
      if (__shfl_sync(0xffffffffu, ab, 0)) break;
    }
  }
  long long tot = 0;
#pragma unroll
  for (int c = 0; c < kGridCopies; c++) tot += grid_word_value(v[c]);
  return tot;
}

// ---- centred Gram band (MRR3 centres every column, RcppEigen20230423.cpp:378-379) ----------------------------------------------
// x_ci'x_ck = x_i'x_k - sx_i sx_k / n, rounded as one FMA on the exact integer entry g.  The Gram kernels apply it in their epilogue
// and gram_centre_kernel to a band that was summed over the ranks of a row-sharded fit: the same operands, so the same bits.
__device__ __forceinline__ float gram_centre(float g, float sx_i, float sx_k, float inv_n) { return fmaf(-(sx_i * inv_n), sx_k, g); }

}  // namespace bwgr
