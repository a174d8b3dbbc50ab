// kernels.h -- internal launch interface between the C-ABI host layer (host.h and its .cu files) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace bwgr {

// ---- genotype store -----------------------------------------------------------------------------
struct GenoView {
  const int8_t* x8 = nullptr;   // int8 store: column j at x8 + j*ld
  const uint8_t* x2 = nullptr;  // 2-bit store: column j at x2 + j*ldb, row r in byte r/4, bits 2*(r%4)
  const float* xf = nullptr;    // float32 store (storage 2, real-valued genotypes): column j at xf + j*ld; grid family only
  int64_t ld = 0, ldb = 0;
  int n = 0, p = 0;
  int storage = 0;
};

// f64 (device staging chunk, column-major ld_src) -> int8 store columns [j0, j0+pc); *bad != 0 if a value
// is not an integer in range.
void launch_pack_f64(const double* src, int64_t ld_src, int n, int pc, int8_t* dst, int64_t ld, int lo, int hi,
                     int* bad, cudaStream_t st);
// int8 store -> 2-bit store (values must be in {0,1,2}; else *bad)
void launch_pack_2bit(const int8_t* src, int64_t ld, int n, int p, uint8_t* dst, int64_t ldb, int* bad, cudaStream_t st);
// packed shadow copy for the Gram kernel (interleaved 2-bit layout, see geno.cu); dst: ld/4 bytes per column
void launch_pack_2bit_gram(const int8_t* src, int64_t ld, int p, uint8_t* dst, int* bad, cudaStream_t st);
void launch_unpack_2bit(const uint8_t* src, int64_t ldb, int n, int p, int8_t* dst, int64_t ld, cudaStream_t st);
void launch_check_range_i8(const int8_t* src, int64_t ld, int n, int p, int lo, int hi, int* bad, cudaStream_t st);
// PLINK .bed payload (variant-major, after the 3 magic bytes) -> int8 store, additive count of allele A1; see geno.cu
void launch_decode_bed(const uint8_t* bed, int64_t bytes_per_col, int n, int p, int8_t* dst, int64_t ld, int missing, int* bad,
                       unsigned long long* nmiss, cudaStream_t st);
// zero rows [n, ld) of every column
void launch_zero_pad(int8_t* x, int64_t ld, int n, int p, cudaStream_t st);
// integer-exact column statistics: xx_j = sum x^2, sx_j = sum x (as int64)
void launch_col_stats(const GenoView& g, long long* xx, long long* sx, cudaStream_t st);
// masked variant for a system with a row mask (uint8 n): xx, sx over used rows
void launch_col_stats_masked(const GenoView& g, const uint8_t* mask, long long* xx, long long* sx, cudaStream_t st);
// float32 store: column statistics in double (mask: optional uint8 [n], rows used)
void launch_col_stats_f32(const GenoView& g, const uint8_t* mask, double* xx, double* sx, cudaStream_t st);
// row multiplicities cnt[i] (uint8) instead of a 0/1 mask; any store
void launch_col_stats_cnt(const GenoView& g, const uint8_t* cnt, double* xx, double* sx, cudaStream_t st);
void launch_d_to_float(const double* src, float* dst, int n, cudaStream_t st);
// hat[t] = mu[t] + X b_t for k systems, one stream of X (deterministic two-stage reduction; each system's sum does not depend on k).
// b: [k][p], mu: [k], hat: [k][ld], work: [k][splits][ld] floats (all device).
constexpr int kHatChunk = 16;  // systems per thread when k > 4
void launch_gemv_hat(const GenoView& g, const float* b, int k, const float* mu, float* hat, float* work, int splits, cudaStream_t st);

// ---- the state of a fit's systems, as every sweep kernel and the epilogue read it ----------------
// The order puts fields that are read together (b and d, vbv and xx, the seed words and chain0) in one 16-byte word of the
// parameter bank, where one instruction loads them; the sweep kernels keep the registers they had with their own copies.
struct SweepState {
  GenoView g;
  int nsys;
  const uint8_t* mask;     // [nsys][ld] or nullptr
  float* e;                // [nsys][ld]  residuals (state, persists across launches)
  float* b;                // [nsys][p]
  float* d;                // [nsys][p] or nullptr
  float* vbv;              // [nsys][p] per-marker variance (or KMUP lambda) or nullptr
  const float* xx;         // [nxx][p]  (nxx = 1 shared or nsys when masked)
  const float* xx2;        // KMUP2: the caller's xx(j) * bg [p] (the rule's denominator; xx carries H'H of the rows in use), else nullptr
  SysScalars* sc;          // [nsys]
  int xx_per_sys;
  uint32_t seed_lo, seed_hi;
  int chain0;              // chain id offset for the RNG counter
  int* err;                // device error flag
};

// ---- small-n path: one persistent CTA per system -------------------------------------------------
struct SmallNArgs {
  SweepState s;
  int model;               // the rule (rule_model)
  const int* perms;        // [p] marker order of this sweep, or nullptr for natural order
  const float* row_w;      // KMUP2 on rows sampled with replacement: [ld] row multiplicities as floats (nsys = 1), or nullptr
};
cudaError_t launch_small_n(const SmallNArgs& a, size_t smem_limit, cudaStream_t st);
bool small_n_fits(const GenoView& g, bool masked, size_t smem_limit, bool weighted = false);

// ---- blocked path ---------------------------------------------------------------------------------
constexpr int kBlk = 128;  // markers per block

// Gram blocks G[blk][i][j] = x_{perm[blk*128+i]}' x_{perm[blk*128+j]} (int32), tcgen05 kind::i8.
// out_f32: write the (exact) int32 accumulators converted to float, the form the sweep consumes.
// nband = 2: row r of block b holds [x_{b,r}'X_b | x_{b-1,r}'X_b] (256 entries): the cross block (stored transposed) feeds
// the one-block look-ahead of the pipelined sweep.
// fp8_codes != 0: all genotypes are codes 0..7 and n*49 < 2^24 -> kind::f8f6f4 on the same bytes (exact, see gram_tc.cu);
// with g.x2 set as well (the packed shadow of a store whose codes are 0..3) the tiles are expanded from the 2-bit copy.
// sx != nullptr (float output): the Gram of the CENTRED columns, x_i'x_k - sx_i sx_k / n (MRR3).
void launch_gram_tc(const GenoView& g, const int* perm, int nblocks, void* gram, int out_f32, int nband, int fp8_codes,
                    int* err, int num_sms, const float* sx, cudaStream_t st);
// FP4 path (gram_fp4.cu): band-2 Gram of a store whose codes are all 0..2, from the packed shadow of launch_pack_2bit_fp4
// (ld / 4 bytes per column); exact, twice the E4M3 rate.  gram: [nblocks][128][256] floats.
void launch_pack_2bit_fp4(const int8_t* src, int64_t ld, int p, uint8_t* dst, int* bad, cudaStream_t st);
cudaError_t launch_gram_fp4(const uint8_t* x2f, int64_t ld, int p, int n, const int* perm, int nblocks, float* gram, int* err,
                            int num_sms, const float* sx, cudaStream_t st, bool block_per_cta = false);
// Centres an uncentred float band in place (gram_tc.cu): what sx != nullptr does inside the Gram kernels, bit for bit, for a band
// summed over the ranks of a row-sharded fit first (sx = column sums and inv_n = 1 / n over all individuals).
void launch_gram_centre(float* gram, const int* perm, int p, int nblocks, int nband, const float* sx, float inv_n, cudaStream_t st);
// host_narrow.cpp: one column of R's double matrix -> int8 codes, exactly (nonzero = not an integer code in [lo, hi])
int narrow_column(const double* src, int64_t n, int8_t* out, int lo, int hi);
int narrow_column_shifted(const double* src, int64_t n, int8_t* out, double shift, int lo, int hi);
double column_min(const double* src, int64_t n);

// Pipelined blocked sweep (sweep_pipe.cu): nworkers streaming CTAs + one solver CTA, look-ahead D (0 or 1).
struct PipeArgs {
  SweepState s;          // unmasked systems: xx is one [p] for all
  int model;             // the rule (rule_model)
  const int* perm;       // this sweep's marker order [p] (device)
  int nblocks;
  const float* gram;     // [nblocks][128][nband*128] Gram band as float (exact below 2^24)
  int nband;
  const float* tinv;     // [nblocks][128][128] (I + A L)^-1 of every block (block_inv.cu), given exactly when the sweep
                         // has one linear system on uncentred columns; else nullptr
  const float* sx;       // [p] column sums, or nullptr.  Non-null = the columns are centred (MRR3): the Gram band is the
                         // centred one and g gets the running mean-shift term c * sx_j (the workers stay uncentred)
  float* cshift;         // [nsys] out: the mean shift c accumulated over the sweep (e_true = e_stored + c)
  int n_total;           // individuals over all ranks: the mean shift is sum_j sx_j dE_j / n_total
  unsigned long long* part;  // [8][nsys][128][160] per-worker integer partials of h: (value << 12) | block tag; zeroed before launch
  unsigned long long* hred;  // [8][nsys][128] reduced h, same word format; zeroed before launch
  // row-sharded fit over `world` GPUs of a node: hx[r] = rank r's exchange ring [8][world][nsys][128] mapped into this
  // process (peer memory over NVLink); gen0 = global sequence number of this launch's block 0 (slot / tag of the ring)
  int world, rank;
  unsigned long long* hx[8];
  unsigned long long gen0;
  unsigned long long* dew;  // [nblocks][nsys][136] published steps: (int32 q << 32) | tag, word 128 = (float scale << 32) | tag
  int rows_per_cta;      // multiple of 16, <= 512
  int nworkers;
  int D;                 // look-ahead depth
  int nbuf;              // X tiles in the ring of a worker (>= D + 1)
  int sring;             // blocks of solve inputs in flight in the solver CTA (2 or 3)
  uint32_t tag;          // unique per launch, never 0
  // clustered topology: nclusters thread-block clusters of 8 CTAs = one solver + seven workers each (nworkers = 7 * nclusters);
  // hsum = [nblocks][nsys][4][kGridCopies][32] L2 grid-sum words of h (device.cuh), word (block, system, marker m) at
  // [block][system][m / 32][copy][m % 32]; zero at launch.  hsum_next = the set of the next launch: this launch zeroes it
  unsigned long long* hsum;
  unsigned long long* hsum_next;
  long long* trace;      // optional [nblocks][16] clock64 stamps (BWGR_TRACE), else nullptr
  int cl, nclusters;
  // optional: cluster 0 stores started_val here once the first grid sum is complete, i.e. when every CTA of the launch is
  // resident -- a side stream waits on it (cuStreamWaitValue32) before it fills the SMs this launch leaves idle
  unsigned int* started;
  unsigned int started_val;
};
cudaError_t launch_sweep_pipe(const PipeArgs& a, cudaStream_t st);
size_t sweep_pipe_smem(int rows_per_cta, int nsys, int model, int nbuf, int sring, int full_inv, int cl);
bool sweep_pipe_cluster_ok(int model, int nsys, int full_inv);
int sweep_pipe_max_clusters(int model, size_t smem);
// T_b = (I + A_b L_b)^-1 for every 128-marker block of the sweep (linear rules, one system): [nblocks][128][128] float
void launch_block_inverse(int model, const int* perm, int p, int nblocks, const float* gram, int nband, const float* xx,
                          const float* vbv, const SysScalars* sc, float* tinv, cudaStream_t st);

// Sweep epilogue (both paths use the same arithmetic): reductions + hyper-parameter update +
// e -= mean(e). One CTA per system.
struct EpilogueArgs {
  SweepState s;                     // xx: emDE's per-marker penalty update needs xx_j
  int model;                        // the full model
  const float* y; const float* b_prev;  // b_prev: convergence (model_has_cnv)
  const float* wts;                 // emML with marker weights: d_j (one system)
  float* B; float* D; float* VBv;
  // row-sharded fit: all-reduced sums over individuals [nsys][4] {sum e, sum e^2, sum e.y, sum y} and max|e| [nsys]; else nullptr
  const double* esum; const float* emaxv;
};
void launch_epilogue(const EpilogueArgs& a, cudaStream_t st);
void launch_epilogue_partial(const EpilogueArgs& a, double* out, float* emax_out, cudaStream_t st);

// wgr() driver step (R/wgr.R:91-136), after each Kuo-Mallick sweep: variance draws, intercept, posterior sums.
struct WgrState {      // device resident, one per fit
  float Ve_old, Ve, Va, mu0;
  int post;            // this iteration is saved (i %in% seq(bi, it, th))
  int post_count;
  double B0, VE, VA;   // posterior sums
};
struct WgrArgs {
  int n, p; int64_t ld;
  float* e; const float* b; const float* d; float* L;   // L = vbv of the sweep (per-marker lambda)
  float* B; float* D; float* VB;                        // posterior sums [p]
  SysScalars* sc; WgrState* st;
  int iv, de; float Sb, Se, df, MSx; int it, bi, th;
  uint32_t seed_lo, seed_hi;
  // wgr(bag != 1): phase 1 = variances from the rows in use (mask, nsub); phase 2 = e := y - hat (hat = mu + X b), intercept draw,
  // posterior sums.  phase 0 = the unbagged step.
  int phase; const uint8_t* mask; float nsub; const float* y; const float* hat;
};
void launch_wgr_step(const WgrArgs& a, int num_sms, cudaStream_t st);
void launch_wgr_bag_phase(const WgrArgs& a, int phase, int num_sms, cudaStream_t st);
void launch_ll_to_float(const long long* src, float* dst, int n, cudaStream_t st);

// ---- multivariate ridge helpers (mrr.cu) ---------------------------------------------------------------------------
// tilde[t][j] = x_j' Y[t]   (Y: [k][ld] float, out: [k][p])
void launch_xty(const GenoView& g, const float* Y, int k, float* out, cudaStream_t st);
// out[t][i] = sum_s (in[s][i] + shift[s]) * T[s*k + t], matrices [k][ld]; amax[t] (zeroed by the caller) = max_i |out[t][i]|
void launch_rotate(const float* in, float* out, int64_t ld, int len, int k, const float* T, const float* shift, float* amax,
                   int num_sms, cudaStream_t st);
// mode 0: out[t1*k+t2] = A[t1].B[t2]; mode 1: out[t] = |A[t]-B[t]|^2; mode 2: out[t] = sum A[t]   (double)
void launch_pair_reduce(const float* A, const float* B, int64_t lda, int64_t ldb, int len, int k, int mode, double* out,
                        cudaStream_t st);

// ---- grid family (grid_sweep.cu): the per-marker step with the individuals spread over the whole GPU; any n, row masks, every rule ----
// copies of each L2 grid-sum word of the grid family and the general MRR3 sweep (the word format is in device.cuh); a power of two
// (4, 8 and 16 measured alike with grid_block_kernel)
constexpr int kGridCopies = 8;
struct GridArgs {
  SweepState s;           // nsys <= 32; a mask byte may be a row multiplicity (KMUP2 on rows drawn with replacement)
  int model;              // the full model
  unsigned long long* acc;  // [p][kGridCopies][32]: (fixed-point sum << 8) + arrivals; zeroed before launch
  float g_quantum;        // value of one fixed-point unit of g
  float gram_quantum;     // blocked variant: value of one fixed-point unit of a cross product x_j'x_i (<= 1 for the int8 store: exact)
  const int* perm;        // marker order of this sweep [p], or nullptr = natural order
  int blocked;            // blocked variant (unmasked systems): acc is [nblocks][kGridCopies][grid_block_words(nsys)]
  int rows_per_cta;       // multiple of 16; grid * rows_per_cta >= ld
};
size_t grid_block_smem(int nsys, int rows_per_cta, bool real_store, bool gibbs);
size_t grid_block_acc_words(int nsys, int p);
size_t grid_sweep_smem(int nsys, int rows_per_cta, bool masked, bool real_store);
cudaError_t launch_grid_sweep(const GridArgs& a, int grid, cudaStream_t st);

// ---- general multivariate ridge sweep (mrr_gen.cu): missing phenotypes, InnerGS, marker weights, NoInv, TH --------------
struct MrrGenArgs {
  GenoView g;
  int k;
  int rows_per_cta;       // multiple of 16; grid * rows_per_cta >= ld
  int innergs;            // sol holds [LHS | PRE] per marker and the chain walks the inner Gauss-Seidel order
  const int* perm;        // marker order of this sweep [p]
  const int* irgs;        // inner order [k] (InnerGS) or nullptr
  const uint32_t* zbits;  // [ld] bit t = trait t observed in row i
  double* e;              // [k][ld] residuals (zero where unobserved)
  double* b;              // [p][k] effects, marker-major
  const double* fixed;    // [p][2k]: XX(j, 0..k) | sum_i (x_ij - mean_j) z_it
  const double* mean;     // [p] column means
  const double* sol;      // [p][nmat * k * k] from launch_mrr_gen_systems
  const double* se0;      // [k] column sums of e at launch
  unsigned long long* acc;  // [p][kGridCopies][32] the grid sums of marker position m: (fixed-point sum << 8) + arrivals; zeroed before launch
  const double* scale;    // [64]: fixed-point scale of trait t (a power of two) | its inverse
  int* err;
};
size_t mrr_gen_smem(int k, int rows_per_cta, int innergs);
// masked integer column sums and X'y in one pass: sxz, sxxz, xty are [p][k] (y: [k][ld] float64, zero where unobserved)
void launch_mrr_gen_colstats(const GenoView& g, const uint32_t* zbits, const double* y, int k, double* sxz, double* sxxz,
                             double* xty, cudaStream_t st);
void launch_mrr_gen_systems(int p, int k, const double* fixed, const double* W, const double* iG, const double* vb,
                            const double* iVe, int noinv_system, int innergs, double* sol, cudaStream_t st);
cudaError_t launch_mrr_gen_sweep(const MrrGenArgs& a, int grid, cudaStream_t st);
void launch_mrr_gen_colred(const double* A, const double* B, int64_t ld, int n, int k, double* out, cudaStream_t st);
void launch_mrr_gen_pk(int mode, const double* A, const double* B, double* C, const double* par, int p, int k, double* out,
                       cudaStream_t st);
void launch_mrr_gen_shift(double* e, const uint32_t* zbits, int64_t ld, int n, int k, const double* shift, cudaStream_t st);

}  // namespace bwgr
