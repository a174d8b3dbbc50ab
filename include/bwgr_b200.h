/* bwgr_b200.h -- C ABI of the B200-native marker-effect update loop (drop-in for bWGR's hot path).
 *
 * Every entry point takes plain pointers and sizes (R's own memory: double, column-major) and
 * writes into caller-allocated outputs, so the Rcpp shim that replaces the reference's generated
 * glue (src/RcppExports.cpp:14-1233) is a one-to-one forwarding stub (see INTEGRATION.md).
 * All functions return 0 on success or a negative bwgr_status; bwgr_last_error() gives the text.
 * There is no CPU fallback: without a CUDA device (or with the CUDA library missing) every
 * compute call fails with BWGR_ERR_CUDA.
 *
 * Citations are file:line under the reference tree (alenxav/bWGR).
 */
#ifndef BWGR_B200_H
#define BWGR_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define BWGR_API __attribute__((visibility("default")))
#else
#define BWGR_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bwgr_handle bwgr_handle; /* one per GPU (= per rank); owns the genotype store */

enum bwgr_status {
  BWGR_OK = 0,
  BWGR_ERR_ARG = -1,     /* bad argument (shape, NULL, non-integer genotype ...) */
  BWGR_ERR_CUDA = -2,    /* CUDA runtime / launch failure, or no device */
  BWGR_ERR_STATE = -3,   /* call order (no genotypes loaded, no fit in progress ...) */
  BWGR_ERR_NUMERIC = -4, /* fixed-point range exceeded / kernel watchdog */
  BWGR_ERR_UNSUPPORTED = -5
};

/* Genotype storage in HBM: column-major, one marker per column. */
enum bwgr_storage {
  BWGR_STORE_I8 = 0,  /* int8, leading dimension padded to 128 rows */
  BWGR_STORE_2BIT = 1, /* codes {0,1,2} packed 4 per byte (little end first), unpacked on the fly */
  BWGR_STORE_F32 = 2   /* float32, the type the reference computes in (Eigen::MatrixXf): ANY real-valued genotypes -- NA cells imputed
                          with column means (R/wgr.R:13-19), IMP() / CNT() output.  Served by the grid family only (bwgr_geno_load_f64). */
};

/* Univariate EM solvers of src/Rcpp20260726ai.cpp. */
enum bwgr_em_model {
  BWGR_EM_RR = 0, /* emRR :308-354 */
  BWGR_EM_BA = 1, /* emBA :80-128  */
  BWGR_EM_BB = 2, /* emBB :131-187 */
  BWGR_EM_BC = 3, /* emBC :190-247 */
  BWGR_EM_BL = 4, /* emBL :357-397 */
  BWGR_EM_EN = 5, /* emEN :400-460 */
  /* the rest of emCV's ten-model panel (R/cv.R:13-22) */
  BWGR_EM_DE = 6,   /* emDE   :250-306   */
  BWGR_EM_ML = 7,   /* emML   :463-520 (D = NULL) */
  BWGR_EM_BCPI = 8, /* emBCpi :1502-1546 */
  BWGR_EM_LASSO = 9 /* lasso  :1463-1500 */
};

/* Univariate Gibbs samplers of src/Rcpp20260726ai.cpp. */
enum bwgr_gibbs_model {
  BWGR_GIBBS_RR = 0, /* BayesRR :812-855 */
  BWGR_GIBBS_A = 1,  /* BayesA  :589-635 */
  BWGR_GIBBS_B = 2,  /* BayesB  :638-699 */
  BWGR_GIBBS_C = 3,  /* BayesC  :702-759 */
  /* the rest of mcmcCV's seven-model panel (R/cv.R:124-130) */
  BWGR_GIBBS_L = 4,   /* BayesL   :762-809 */
  BWGR_GIBBS_CPI = 5, /* BayesCpi :858-919 (pi starts at 0.5; params.pi is ignored) */
  BWGR_GIBBS_DPI = 6  /* BayesDpi :922-987 (same) */
};

#define BWGR_NSCAL 6 /* scalars per system in bwgr_em_out.scal / bwgr_gibbs_out.scal */

/* Which kernel family runs the sweep. AUTO picks SMALL_N when several systems share X and the
 * residual of one system fits one SM's shared memory, BLOCKED otherwise, and GRID (the per-marker step with the individuals spread
 * over the whole GPU: any n, row masks, every rule, <= 32 systems; latency-bound) when neither takes the shape -- n above ~75k on one
 * GPU, or row-masked systems whose residual does not fit one SM. */
enum bwgr_path { BWGR_PATH_AUTO = 0, BWGR_PATH_SMALL_N = 1, BWGR_PATH_BLOCKED = 2, BWGR_PATH_GRID = 3 };

/* ---- lifetime ---------------------------------------------------------------------------- */
BWGR_API int bwgr_create(int device, bwgr_handle** out);
BWGR_API void bwgr_destroy(bwgr_handle* h);
BWGR_API const char* bwgr_last_error(void);
BWGR_API int bwgr_version(void);
/* Device and pinned-host blocks released by destroyed handles are kept for reuse by the next handle of the process (an R session
 * calls emRR(y, gen) repeatedly on the same shapes; cudaFree of gigabyte blocks is slow and erratic).  Bound: BWGR_CACHE_GB
 * (default 24, 0 = keep nothing).  bwgr_trim() returns everything held to the driver. */
BWGR_API void bwgr_trim(void);
/* Use the caller's CUDA stream (cudaStream_t as void*) for all work of this handle; NULL = the
 * handle's own stream. Lets a host framework time the library with its own events. */
BWGR_API int bwgr_set_stream(bwgr_handle* h, void* cuda_stream);
/* Tuning knobs: block = markers per block of the blocked sweep (128); path = bwgr_path;
 * grid = persistent CTAs (0 = one per SM; grid > 1 runs the blocked sweep in its flat topology on that many CTAs).
 * Negative values leave a knob unchanged. A shape the blocked sweep cannot take on `grid` CTAs (more than 512 rows per CTA, or
 * a solver that does not fit one SM) returns BWGR_ERR_UNSUPPORTED under path = BLOCKED; under AUTO another family takes it. */
BWGR_API int bwgr_set_tuning(bwgr_handle* h, int block, int path, int grid);

/* ---- genotype store (replaces the per-call double->float copy of RcppExports.cpp:115-116) -- */
/* X: host, column-major, n x p, leading dimension ld (>= n). Values must be integers in
 * [-128,127] (I8) or {0,1,2} (2BIT); anything else -> BWGR_ERR_ARG (no silent rounding). */
BWGR_API int bwgr_geno_load_f64(bwgr_handle* h, const double* X, int64_t n, int64_t p, int64_t ld, int storage);
/* The same for a caller whose solver centres the columns itself (MRR3 / MRR3F, RcppEigen20230423.cpp:378-379): a column may be
 * "integer codes + one constant", e.g. CNT(gen) (Rcpp20260726ai.cpp:1308; the reference's own example mrr(Y, CNT(gen)), man/mvr.Rd:144-153).
 * The codes are stored, the constants dropped; the other solvers refuse such a store (BWGR_ERR_UNSUPPORTED). */
BWGR_API int bwgr_geno_load_f64_centred(bwgr_handle* h, const double* X, int64_t n, int64_t p, int64_t ld, int storage);
/* On-disk ingestion: a PLINK .bed file (variant-major; n = lines of the .fam file, p = lines of the .bim file) decoded on the device
 * to the additive count of allele A1 (0/1/2, like `plink --recode A`).  missing: 0..2 = code given to missing calls, -2 = the rounded
 * mean of the marker's observed codes (an integer stand-in for IMP, Rcpp20260726ai.cpp:1316-1335), -1 = missing calls are an error.
 * *nmissing_out (optional) = the number of missing calls met. */
BWGR_API int bwgr_geno_load_bed(bwgr_handle* h, const char* path, int64_t n, int64_t p, int storage, int missing, int64_t* nmissing_out);
BWGR_API int bwgr_geno_load_i8(bwgr_handle* h, const int8_t* X, int64_t n, int64_t p, int64_t ld, int storage);
/* Same, X already resident in device memory (int8, column-major). */
BWGR_API int bwgr_geno_load_i8_device(bwgr_handle* h, const int8_t* dX, int64_t n, int64_t p, int64_t ld, int storage);
/* Round trip for the bit-exactness tests: unpack the store to host int8 (n x p, ld = n). */
BWGR_API int bwgr_geno_unpack_i8(bwgr_handle* h, int8_t* X_out);
/* Raw bytes of the store as laid out in HBM (size from bwgr_geno_info). */
BWGR_API int bwgr_geno_raw(bwgr_handle* h, uint8_t* bytes_out);
BWGR_API int bwgr_geno_info(bwgr_handle* h, int64_t* n, int64_t* p, int64_t* ld_bytes, int* storage, int64_t* total_bytes);
/* Integer-exact column statistics (reference: xx[j]=squaredNorm, :312-316): xx_j = sum x^2, sx_j = sum x. */
BWGR_API int bwgr_geno_stats(bwgr_handle* h, double* xx, double* sx);

/* ---- univariate EM family ----------------------------------------------------------------- */
typedef struct {
  int model;     /* bwgr_em_model */
  int nsys;      /* systems (traits / folds) sharing the genotypes; y is n x nsys */
  int it;        /* sweeps; <0 = the reference's hard-coded 200 (emEN, emDE, emML, lasso: maxit 300 with their tol) */
  double df, R2, Pi, alpha; /* reference defaults: 10, 0.5, 0.75, 0.02 */
  const uint8_t* row_mask;  /* optional n x nsys, 1 = row used by the system (CV folds); NULL = all */
  const double* weights;    /* emML only: optional marker weights D [p] (Rcpp20260726ai.cpp:471-475; one system, no row mask); NULL = none */
} bwgr_em_params;

typedef struct {
  double* mu;   /* [nsys] */
  double* b;    /* [p x nsys] */
  double* d;    /* [p x nsys] inclusion (emBB, emBC, emBCpi) or NULL */
  double* hat;  /* [n x nsys] */
  double* vb;   /* [p x nsys] per-marker Vb (emBA, emBB, emDE) or NULL */
  double* scal; /* [BWGR_NSCAL x nsys]: Va, Ve, h2, Vg (as each model defines them; emML: Vg slot = Vb), pi (emBCpi), Lmb (lasso) */
  int* its;     /* [nsys] sweeps done */
} bwgr_em_out;

/* Whole fit, the call the Rcpp shim makes for emRR/emBA/emBB/emBC/emBL/emEN/emDE/emML/emBCpi/lasso. */
BWGR_API int bwgr_em_fit(bwgr_handle* h, const bwgr_em_params* par, const double* y, bwgr_em_out* out);
/* Same fit split in three so that a harness can time sweeps with everything resident in HBM. */
BWGR_API int bwgr_em_begin(bwgr_handle* h, const bwgr_em_params* par, const double* y);
BWGR_API int bwgr_em_sweeps(bwgr_handle* h, int nsweeps); /* asynchronous on the handle's stream */
BWGR_API int bwgr_em_end(bwgr_handle* h, bwgr_em_out* out);

/* ---- univariate Gibbs family --------------------------------------------------------------- */
typedef struct {
  int model;    /* bwgr_gibbs_model */
  int nchains;  /* independent chains of the same model on the same y (one seed; the chain index enters the Philox counter, so the chains draw from disjoint streams) */
  int it, bi;   /* reference defaults 1500, 500 */
  double pi, df, R2; /* 0.95, 5, 0.5 */
  uint64_t seed;
} bwgr_gibbs_params;

typedef struct {
  double* mu;   /* [nchains] (bwgr_gibbs_fit_sys: [S] here and below) */
  double* b;    /* [p x nchains] posterior means */
  double* d;    /* [p x nchains] (BayesB/C/Cpi/Dpi; the reference's PVAL is -log(1 - d)) or NULL */
  double* hat;  /* [n x nchains] */
  double* vb;   /* [p x nchains] (BayesA/B/L/Dpi) or [nchains] (BayesRR/C/Cpi) */
  double* scal; /* [BWGR_NSCAL x nchains]: vb (scalar models), ve, h2, MSx, pi (BayesCpi/Dpi), reserved */
} bwgr_gibbs_out;

BWGR_API int bwgr_gibbs_fit(bwgr_handle* h, const bwgr_gibbs_params* par, const double* y, bwgr_gibbs_out* out);

/* Several traits / CV folds in one call (not in the reference: its samplers take one y).  Column t of Y runs base.nchains chains, so
 * there are S = nsys * nchains systems; system s = t * nchains + c draws from Philox chain index chain0 + s (disjoint streams; a caller
 * that splits the columns over GPUs passes its first system as chain0 and gets the draws of the one-GPU fit).  A masked system fits
 * its column on the rows its mask keeps: the draws are addressed by (sweep, marker, chain), so it is the fit of those rows alone under
 * the same chain index, with MSx and the variance draws from those rows.  Every output of bwgr_gibbs_out has S columns; hat covers
 * all n rows, the held-out ones included (their prediction).  bwgr_gibbs_fit = nsys 1, no mask, chain0 0.
 * BWGR_ERR_ARG: nsys < 1, NaN in Y, a mask column that keeps fewer than 2 rows.  BWGR_ERR_UNSUPPORTED: a mask on a row-sharded
 * store, or a shape no kernel family takes (more than 32 masked systems whose residual does not fit one SM). */
typedef struct {
  bwgr_gibbs_params base;   /* model, nchains, it, bi, pi, df, R2, seed: as for bwgr_gibbs_fit */
  int nsys;                 /* phenotype columns of Y (traits / folds) */
  const uint8_t* row_mask;  /* optional n x nsys, 1 = row used by that column's systems; NULL = all */
  int chain0;               /* Philox chain index of the first system */
} bwgr_gibbs_sys_params;
BWGR_API int bwgr_gibbs_fit_sys(bwgr_handle* h, const bwgr_gibbs_sys_params* par, const double* Y /* n x nsys */,
                                bwgr_gibbs_out* out);

/* One Kuo-Mallick sweep, drop-in for KMUP(X,b,d,xx,e,L,Ve,pi) (:12-38); b,d,e updated in place.
 * The inclusion probability uses BayesB's ratio form (:673-674), algebraically identical to
 * :25-27 but free of the exp underflow (SURVEY appendix). */
BWGR_API int bwgr_kmup_sweep(bwgr_handle* h, double* b, double* d, const double* xx, double* e, const double* L, double Ve,
                    double pi, uint64_t seed);

/* hat[n] = mu + X b on the handle's store: the X * b the reference's drivers form around the marker loop (emML2's u1 = X1 * b1,
 * Rcpp20260726ai.cpp:1275-1276; the fitted values of the two-design samplers :1063, :1151, :1212; wgr's gen0 %*% B, R/wgr.R:147). */
BWGR_API int bwgr_fitted(bwgr_handle* h, const double* b, double mu, double* hat);
/* The same for k systems with one pass over the store: hat[:, t] = mu[t] + X B[:, t].  B: p x k, mu: [k], hat: n x k (column-major).
 * Every column is bit-identical to bwgr_fitted of that column alone (the summation order of a row does not depend on k). */
BWGR_API int bwgr_fitted_sys(bwgr_handle* h, int k, const double* B, const double* mu, double* hat);

/* KMUP2(X,Use,b,d,xx,E,L,Ve,pi) (:41-77), the bagged sweep of wgr(bag != 1): only the rows Use (0-based, as R passes them) enter.
 * b, d updated in place; e_out [nuse] = the residuals of the rows in use, in the order of Use (the reference's third list element).
 * A row named more than once (sampling with replacement, rp = TRUE) counts once per occurrence in H'e0, H'H and ||e||^2, as in the
 * reference's H / e0 (:51-60): row multiplicities (<= 255) in the dot products, on the small-n family when the residual and the
 * multiplicities of n rows fit one SM's shared memory, else on the grid family (any n, int8 or float32 store). */
BWGR_API int bwgr_kmup2_sweep(bwgr_handle* h, const double* use, int64_t nuse, double* b, double* d, const double* xx, const double* E,
                     double* e_out, const double* L, double Ve, double pi, uint64_t seed);

/* GSRR / GSFLM(y, e, gen, b, Lmb, xx, cxx, maxit = 50) (:1564-1628): the warm-start Gauss-Seidel solvers mm() calls inside its
 * back-fitting loop (R/mix.R:890-892).  which = 0 GSRR, 1 GSFLM.  In / out: e [n], b [p], Lmb [p] (the state the caller carries from
 * one outer iteration to the next); out: vb [p]; scal = {mu, h2, vna (the residual variance e.e0/n), sweeps done}. */
BWGR_API int bwgr_gs_fit(bwgr_handle* h, int which, const double* y, double* e, double* b, double* Lmb, const double* xx, double cxx,
                int maxit, double* vb, double* scal);

/* wgr(y,X,it,bi,th,bag=1,rp,iv,de,pi,df,R2) with the MCMC loop native (R/wgr.R:2-169; eigK=NULL).
 * scal = {mu, Ve, Va, cxx}; Vb is [p] when iv/de, else scal[2]. */
BWGR_API int bwgr_wgr_fit(bwgr_handle* h, const double* y, int it, int bi, int th, int iv, int de, double pi, double df,
                 double R2, uint64_t seed, double* b, double* d, double* Vb, double* hat, double* scal);

/* wgr(..., bag, rp) for bag != 1 (R/wgr.R:21, :49, :68, :87, :121): a fresh sorted sample of floor(n * bag) rows per iteration (drawn
 * with std::mt19937_64(seed), not R's sample()), swept by KMUP2; rp = TRUE draws them with replacement (bag > 1 allowed) and sweeps with row multiplicities (see
 * bwgr_kmup2_sweep).  bag = 1 forwards to bwgr_wgr_fit. */
BWGR_API int bwgr_wgr_fit_bag(bwgr_handle* h, const double* y, int it, int bi, int th, double bag, int rp, int iv, int de, double pi,
                     double df, double R2, uint64_t seed, double* b, double* d, double* Vb, double* hat, double* scal);

/* ---- multivariate ridge -------------------------------------------------------------------- */
/* MRR3 / MRR3F (src/RcppEigen20230423.cpp:318-701, :704-1079). par[30] = the arguments after
 * (Y,X) in the order of R/RcppExports.R:180. Y: n x k column-major.
 * cnv: 3*maxit doubles (cnvB | cnvH2 | cnvV).
 * Two device paths, chosen by the arguments (never a CPU fallback):
 *  - complete Y, direct k x k solve (the default flags, HCS / XFA / ACS / updateMu / OneVarB / OneVarE / NoInv for MRR3 and all the GC
 *    and h2 shaping arguments): k rotated ridge systems on the pipelined blocked sweep, float32 device state (csrc/mrr.cu);
 *  - everything else -- NaN in Y (missing phenotypes, :359-365), InnerGS = TRUE (:510-514), TH = TRUE (:423, :549-571), NLfactor != 0
 *    (:524-533), MRR3F with NoInv = TRUE (:878-882): one k x k system per marker with per-trait observation masks, float64 device
 *    state (csrc/mrr_gen.cu); needs the int8 store.
 * On a row-sharded store (bwgr_dist_*) only the first path runs: each rank passes its rows of Y and gets the common b, mu, h2, GC,
 * vb, ve, MSx, cnv and Its, and hat for its rows.  Whether the fit can run is decided by all ranks together: if any rank meets
 * something only the general path handles (NaN in its rows of Y, InnerGS, TH, NLfactor, MRR3F's NoInv, BWGR_MRR=general) or a
 * shard the pipelined sweep cannot take, every rank returns BWGR_ERR_UNSUPPORTED.
 * BWGR_ERR_UNSUPPORTED: k > 32; a trait with fewer than two observations is BWGR_ERR_ARG. */
BWGR_API int bwgr_mrr3_fit(bwgr_handle* h, int f32_variant, const double* Y, int k, const double* par, double* mu, double* b,
                  double* hat, double* h2, double* GC, double* vb, double* ve, double* MSx, double* cnv, double* W,
                  int* its);

/* ---- one large fit sharded by rows over the GPUs of a node (SURVEY 8e, BASELINE config 5) ---------------------
 * Not in the reference (single process, single thread).  One process per GPU; every rank loads ITS rows of X and passes
 * ITS rows of y.  b / variance components come back identical on every rank, hat holds the rank's rows.
 * Per 128-marker block the reduced partial X_B'E of a rank is stored straight into every peer's exchange ring inside the
 * sweep kernel (peer memory over NVLink, no host involvement); NCCL all-reduces the per-sweep Gram band and scalars.
 * Call order on every rank: bwgr_create -> bwgr_dist_init -> (exchange the 64-byte handles) -> bwgr_dist_connect ->
 * bwgr_geno_load_* -> fits.  Supports the blocked family (unmasked systems, int8 store): the EM and Gibbs solvers and MRR3 /
 * MRR3F's rotated fast path (bwgr_mrr3_fit; a refusal there is taken by all ranks together, so no rank waits in a collective the
 * others never reach).  bwgr_geno_load_f64_centred agrees each column's constant over the ranks. */
BWGR_API int bwgr_dist_unique_id(void* id128);  /* rank 0 creates it, the host framework broadcasts the 128 bytes */
BWGR_API int bwgr_dist_init(bwgr_handle* h, int rank, int world, const void* id128, void* ipc_handle_out64);
BWGR_API int bwgr_dist_connect(bwgr_handle* h, const void* ipc_handles_all /* world x 64 bytes, rank order */);

/* ---- introspection for tests and the bench -------------------------------------------------- */
/* Kernels launched by this handle since creation (the bench's gpu_launches claim). */
BWGR_API int64_t bwgr_launch_count(bwgr_handle* h);
/* Per-kernel device timing for the roofline report: when enabled, CUDA events bracket every kernel
 * of the sweep loop on the handle's stream. read: ms[4] / counts[4] = {gram, sweep, epilogue, block inverses} summed
 * since enable (synchronises the stream). */
BWGR_API int bwgr_profile(bwgr_handle* h, int enable);
BWGR_API int bwgr_profile_read(bwgr_handle* h, double* ms, int64_t* counts);
/* Gram blocks X_B' X_B of one sweep order (perm[p], block markers each), int32, [nblocks][block][block];
 * the tcgen05 kernel's output, exposed so tests can check it bit-exactly. */
/* Host-side test hook of the float64 loader's narrowing paths (csrc/host_narrow.cpp); needs no GPU.  level: -1 = the path the
 * loader uses on this CPU, 0 plain, 1 AVX2, 2 AVX-512 (-1 returned if the CPU lacks it).  Returns 1 if any value is not an
 * integer code in [lo, hi] (to 1e-4 after subtracting `shift` when use_shift), else 0. */
BWGR_API int bwgr_debug_narrow(const double* src, int64_t n, int8_t* out, int use_shift, double shift, int lo, int hi, int level,
                               double* min_out);
BWGR_API int bwgr_debug_gram_band(bwgr_handle* h, const int32_t* perm, float* gram_out /* [nblocks][128][256] */, int* kind_out);
BWGR_API int bwgr_debug_gram(bwgr_handle* h, const int32_t* perm, int block, int32_t* gram_out);

#ifdef __cplusplus
}
#endif
#endif /* BWGR_B200_H */
