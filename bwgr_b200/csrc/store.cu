// store.cu -- the genotype store: its loaders (R's double matrix narrowed by a pool of host threads, int8 from host or device,
// PLINK .bed), the column statistics and Gram shadow copies every load finishes with, and the store accessors.
#include <sched.h>
#include <atomic>
#include <thread>

#include "host.h"

using namespace bwgr;
using namespace bwgr::host;

static int finish_store(bwgr_handle* h, int storage) {
  // column statistics from the int8 copy, then optional 2-bit packing
  GenoView g8 = h->view();
  g8.storage = 0;
  if (h->xx_i.alloc(h->p) != cudaSuccess || h->sx_i.alloc(h->p) != cudaSuccess || h->xx_f.alloc(h->p) != cudaSuccess)
    return fail(BWGR_ERR_CUDA, "cudaMalloc(stats) failed");
  launch_col_stats(g8, h->xx_i.p, h->sx_i.p, h->stream);
  h->launches++;
  h->n_global = h->n;
  if (h->world > 1) {  // row shards: the column statistics are sums over all individuals
    if (storage != BWGR_STORE_I8) return fail(BWGR_ERR_UNSUPPORTED, "row-sharded fits take the int8 store");
    NC(nccl().AllReduce(h->xx_i.p, h->xx_i.p, (size_t)h->p, ncclInt64, ncclSum, h->comm, h->stream));
    NC(nccl().AllReduce(h->sx_i.p, h->sx_i.p, (size_t)h->p, ncclInt64, ncclSum, h->comm, h->stream));
    double ng = (double)h->n;
    int rcn = dist_allreduce_host(h, &ng, 1, false);
    if (rcn) return rcn;
    h->n_global = (int64_t)ng;
  }
  std::vector<long long> xx(h->p), sx(h->p);
  CU(cudaMemcpyAsync(xx.data(), h->xx_i.p, sizeof(long long) * h->p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(sx.data(), h->sx_i.p, sizeof(long long) * h->p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->h_xx.assign(xx.begin(), xx.end());
  h->h_sx.assign(sx.begin(), sx.end());
  h->xx_max = 0;
  for (double v : h->h_xx) h->xx_max = std::max(h->xx_max, v);
  std::vector<float> xf(h->p);
  for (int64_t j = 0; j < h->p; j++) xf[j] = (float)xx[j];
  CU(cudaMemcpyAsync(h->xx_f.p, xf.data(), sizeof(float) * h->p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  int flag = 0, rc = 0;
  // row shards: which Gram kernel runs, and so the band's layout, the sweep's geometry and the collectives of a fit, must be the
  // same on every rank -- a code any rank holds counts for all
  auto agree = [h](int* f) -> int {
    double v = *f;
    const int r = dist_allreduce_host(h, &v, 1, true);
    *f = v != 0.0 ? 1 : 0;
    return r;
  };
  {  // codes 0..7 everywhere?  (one more streaming pass at load time)
    h->fp8_codes = 0;
    if (h->xx_max < 16777216.0) {  // every Gram entry and every partial sum of non-negative codes is bounded by max_j xx_j
      launch_check_range_i8(h->x8, h->ld, (int)h->n, (int)h->p, 0, 7, h->err.p, h->stream);
      h->launches++;
      if ((rc = take_err_flag(h, &flag)) || (rc = agree(&flag))) return rc;
      h->fp8_codes = flag ? 0 : 1;
    }
  }
  h->x2f.release();
  if (h->fp8_codes && storage == BWGR_STORE_I8) {  // FP4 Gram shadow copy (gram_fp4.cu): only when every code is 0, 1 or 2
    flag = 1;
    if (h->x2f.alloc((size_t)(h->ld / 4) * h->p) == cudaSuccess) {
      launch_pack_2bit_fp4(h->x8, h->ld, (int)h->p, h->x2f.p, h->err.p, h->stream);
      h->launches++;
      if ((rc = take_err_flag(h, &flag))) return rc;
    }
    if ((rc = agree(&flag))) return rc;
    if (flag) h->x2f.release();  // a code 3..7 (or no room for the copy): the E4M3 path
  }
  h->x2g.release();
  if (h->fp8_codes && storage == BWGR_STORE_I8 && !h->x2f.p) {  // E4M3 Gram shadow copy (codes 0..3)
    flag = 1;
    if (h->x2g.alloc((size_t)(h->ld / 4) * h->p) == cudaSuccess) {
      launch_pack_2bit_gram(h->x8, h->ld, (int)h->p, h->x2g.p, h->err.p, h->stream);
      h->launches++;
      if ((rc = take_err_flag(h, &flag))) return rc;
    }
    if ((rc = agree(&flag))) return rc;
    if (flag) h->x2g.release();  // a code 3..7 (or no room for the copy): keep the int8 gather
  }
  CU(cudaGetLastError());  // a store kernel that failed to launch must not go unnoticed
  h->storage = BWGR_STORE_I8;
  if (storage == BWGR_STORE_2BIT) {
    h->ldb = h->ld / 4;
    if (h->x2.alloc((size_t)h->ldb * h->p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(2-bit store) failed");
    launch_pack_2bit(h->x8, h->ld, (int)h->n, (int)h->p, h->x2.p, h->ldb, h->err.p, h->stream);
    h->launches++;
    rc = check_err_flag(h, "bwgr_geno_load (2-bit needs codes {0,1,2})");
    if (rc) { h->x2.release(); return rc; }
    h->storage = BWGR_STORE_2BIT;
    h->x8_own.release();  // the 2-bit store is the only copy kept in HBM
    h->x8 = nullptr;
  }
  return 0;
}

static int prepare_store(bwgr_handle* h, int64_t n, int64_t p, int storage) {
  if (!h) return fail(BWGR_ERR_ARG, "null handle");
  if (n < 2 || p < 1 || n > (int64_t)1 << 30 || p > (int64_t)1 << 30) return fail(BWGR_ERR_ARG, "bad shape n=%lld p=%lld", (long long)n, (long long)p);
  if (storage != BWGR_STORE_I8 && storage != BWGR_STORE_2BIT && storage != BWGR_STORE_F32) return fail(BWGR_ERR_ARG, "bad storage %d", storage);
  CU(cudaSetDevice(h->device));
  h->fit.reset();
  h->x2.release();
  h->gram_nat.release(); h->gram_nat_band = 0;
  h->x2g.release(); h->x2f.release();
  h->n = n; h->p = p;
  h->ld = (n + 127) / 128 * 128;
  h->ldb = 0;
  h->xf_own.release();
  if (storage == BWGR_STORE_F32) {
    if (h->world > 1) return fail(BWGR_ERR_UNSUPPORTED, "row-sharded fits take the int8 store");
    h->x8_own.release(); h->x8 = nullptr;
    if (h->xf_own.alloc((size_t)h->ld * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(%lld bytes) for genotypes failed", (long long)(h->ld * p * 4));
    return 0;
  }
  if (h->x8_own.alloc((size_t)h->ld * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(%lld bytes) for genotypes failed", (long long)(h->ld * p));
  h->x8 = h->x8_own.p;
  return 0;
}

extern "C" {

// Host side of emRR(y, gen) on R's double matrix: exact narrowing to int8 codes (host_narrow.cpp) by a pool of host threads into
// pinned staging buffers, each chunk of columns copied to the device while the next ones are narrowed.
// offsets != nullptr (the centred loader): a column may be "integer codes + one constant" (CNT(gen), or any integer-valued
// column): the constant -- the fractional part of the first value plus the column minimum, so that the stored codes start at 0 --
// goes to offsets[j]; the codes must still be integers to 1e-4, the resolution of a float32 column mean.  mins (row-sharded store):
// the column minima over all ranks, so that every rank shifts a column by the same integer.
static int narrow_columns(const double* X, int64_t ld_src, int64_t n, int64_t ld_dst, int64_t j0, int64_t j1, int8_t* dst, int lo, int hi, double* offsets,
                          const double* mins) {
  int flag = 0;
  for (int64_t j = j0; j < j1; j++) {
    const double* src = X + j * ld_src;
    int8_t* out = dst + (j - j0) * ld_dst;
    if (offsets) {
      const double v0 = src[0];
      double frac = v0 - std::floor(v0);
      if (!(frac == frac) || frac < 1e-4 || frac > 1.0 - 1e-4) frac = 0.0;
      // also for an integer-valued column: the solver centres anyway, and codes starting at 0 keep the store on the FP4 / E4M3 Gram paths
      const double base = std::nearbyint((mins ? mins[j] : bwgr::column_min(src, n)) - frac);
      flag |= bwgr::narrow_column_shifted(src, n, out, frac + base, lo, hi);
      offsets[j] = frac + base;
    } else {
      flag |= bwgr::narrow_column(src, n, out, lo, hi);
    }
    for (int64_t i = n; i < ld_dst; i++) out[i] = 0;
  }
  return flag;
}

// host threads the loader may keep busy: the cores this process may run on, capped by the cgroup CPU quota (a container that
// over-subscribes its quota is throttled for the rest of every scheduling period -- stalls of tens of milliseconds)
static int loader_threads() {
  if (const char* e = getenv("BWGR_LOAD_THREADS")) { const int v = atoi(e); if (v > 0) return std::min(v, 256); }
  int nt = (int)std::thread::hardware_concurrency();
  cpu_set_t cs;
  if (sched_getaffinity(0, sizeof cs, &cs) == 0) nt = std::min(nt > 0 ? nt : 1 << 20, CPU_COUNT(&cs));
  if (FILE* f = fopen("/sys/fs/cgroup/cpu.max", "r")) {
    long long quota = 0, period = 0;
    if (fscanf(f, "%lld %lld", &quota, &period) == 2 && quota > 0 && period > 0) nt = std::min<long long>(nt, std::max<long long>(1, quota / period));
    fclose(f);
  }
  return std::max(1, std::min(nt, 64));
}

// BWGR_STORE_F32: R's double matrix narrowed to float32, the type the reference itself computes in (Eigen::MatrixXf arguments,
// RcppExports.cpp:115-116) -- any real-valued genotypes: NA cells imputed with column means (R/wgr.R:13-19), IMP() / CNT() output.
static int load_f64_real(bwgr_handle* h, const double* X, int64_t n, int64_t p, int64_t ld) {
  int rc = prepare_store(h, n, p, BWGR_STORE_F32);
  if (rc) return rc;
  h->col_offset.clear(); h->has_offset = false;
  const int64_t ldd = h->ld;
  const int64_t chunk_cols = std::max<int64_t>(1, std::min<int64_t>(p, ((int64_t)64 << 20) / (ldd * 4)));
  float* stage[2] = {nullptr, nullptr};
  const size_t bytes = (size_t)chunk_cols * ldd * sizeof(float);
  if (pinned_alloc(reinterpret_cast<void**>(&stage[0]), bytes) != cudaSuccess || pinned_alloc(reinterpret_cast<void**>(&stage[1]), bytes) != cudaSuccess) {
    pinned_free(stage[0], bytes); pinned_free(stage[1], bytes);
    return fail(BWGR_ERR_CUDA, "staging allocation failed");
  }
  cudaEvent_t done[2];
  cudaEventCreateWithFlags(&done[0], cudaEventDisableTiming); cudaEventCreateWithFlags(&done[1], cudaEventDisableTiming);
  bool used[2] = {false, false}, bad = false;
  cudaError_t ce = cudaSuccess;
  for (int64_t j0 = 0, c = 0; j0 < p && ce == cudaSuccess; j0 += chunk_cols, c++) {
    const int sl = (int)(c & 1);
    const int64_t pc = std::min(chunk_cols, p - j0);
    if (used[sl]) ce = cudaEventSynchronize(done[sl]);
    float* dst = stage[sl];
    for (int64_t j = 0; j < pc; j++) {
      const double* src = X + (size_t)(j0 + j) * ld;
      float* col = dst + (size_t)j * ldd;
      for (int64_t i = 0; i < n; i++) { const double v = src[i]; if (!(v - v == 0.0)) bad = true; col[i] = (float)v; }
      for (int64_t i = n; i < ldd; i++) col[i] = 0.0f;
    }
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(h->xf_own.p + j0 * ldd, dst, (size_t)pc * ldd * sizeof(float), cudaMemcpyHostToDevice, h->stream);
    if (ce == cudaSuccess) ce = cudaEventRecord(done[sl], h->stream);
    used[sl] = true;
  }
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(h->stream);
  cudaEventDestroy(done[0]); cudaEventDestroy(done[1]);
  pinned_free(stage[0], bytes); pinned_free(stage[1], bytes);
  if (ce != cudaSuccess) return fail(BWGR_ERR_CUDA, "bwgr_geno_load_f64: %s", cudaGetErrorString(ce));
  if (bad) return fail(BWGR_ERR_ARG, "bwgr_geno_load_f64: NaN or infinite genotype (impute first: R/wgr.R:13-19)");
  // column statistics in double
  DevBuf<double> dxx, dsx;
  if (dxx.alloc(p) != cudaSuccess || dsx.alloc(p) != cudaSuccess || h->xx_f.alloc(p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(stats) failed");
  launch_col_stats_f32(h->view(), nullptr, dxx.p, dsx.p, h->stream);
  launch_d_to_float(dxx.p, h->xx_f.p, (int)p, h->stream);
  h->launches += 2;
  h->h_xx.resize(p); h->h_sx.resize(p);
  CU(cudaMemcpyAsync(h->h_xx.data(), dxx.p, sizeof(double) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(h->h_sx.data(), dsx.p, sizeof(double) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->xx_max = 0;
  for (double v : h->h_xx) h->xx_max = std::max(h->xx_max, v);
  h->n_global = h->n;
  h->storage = BWGR_STORE_F32;
  h->fp8_codes = 0;
  h->x2f.release(); h->x2g.release();
  return 0;
}

static int load_f64_common(bwgr_handle* h, const double* X, int64_t n, int64_t p, int64_t ld, int storage, bool allow_offset) {
  if (!X || ld < n) return fail(BWGR_ERR_ARG, "bad X / ld");
  if (storage == BWGR_STORE_F32) return load_f64_real(h, X, n, p, ld);
  int rc = prepare_store(h, n, p, storage);
  if (rc) return rc;
  h->col_offset.clear(); h->has_offset = false;
  if (allow_offset) h->col_offset.assign((size_t)p, 0.0);
  double* offs = allow_offset ? h->col_offset.data() : nullptr;
  const int lo = storage == BWGR_STORE_2BIT ? 0 : -128, hi = storage == BWGR_STORE_2BIT ? 2 : 127;
  std::vector<double> mins;  // row-sharded centred store: column minima over all ranks (min = -max of the negated values)
  if (allow_offset && h->world > 1) {
    mins.resize((size_t)p);
    std::vector<std::thread> pool;
    const int nthr = (int)std::min<int64_t>(loader_threads(), p);
    for (int t = 0; t < nthr; t++)
      pool.emplace_back([&, t]() { for (int64_t j = t; j < p; j += nthr) mins[(size_t)j] = -bwgr::column_min(X + j * ld, n); });
    for (auto& th : pool) th.join();
    rc = dist_allreduce_host(h, mins.data(), (int)p, true);
    if (rc) return rc;
    for (double& v : mins) v = -v;
  }
  const double* gmins = mins.empty() ? nullptr : mins.data();
  const int64_t ldd = h->ld;
  constexpr int kStage = 4;
  const int64_t chunk_cols = std::max<int64_t>(1, std::min<int64_t>(p, ((int64_t)32 << 20) / ldd));
  const size_t chunk_bytes = (size_t)chunk_cols * ldd;
  int8_t* stage[kStage] = {};
  cudaEvent_t done[kStage] = {};
  auto release_staging = [&]() { for (int i = 0; i < kStage; i++) { pinned_free(stage[i], chunk_bytes); if (done[i]) cudaEventDestroy(done[i]); } };
  for (int i = 0; i < kStage; i++) {
    if (pinned_alloc(reinterpret_cast<void**>(&stage[i]), chunk_bytes) != cudaSuccess) { release_staging(); return fail(BWGR_ERR_CUDA, "staging allocation failed"); }
    if (cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming) != cudaSuccess) { release_staging(); return fail(BWGR_ERR_CUDA, "cudaEventCreate failed"); }
  }
  const int64_t nchunk = (p + chunk_cols - 1) / chunk_cols;
  const int nthr = (int)std::min<int64_t>(loader_threads(), p);
  const int nslice = (int)std::min<int64_t>(chunk_cols, 2 * nthr);  // tasks per chunk
  // task t = (chunk t / nslice, slice t % nslice), handed out in order; a chunk may be written once the copy that last read its
  // staging buffer has finished (`released`, advanced by this thread), and is copied once all its slices are in (`left`)
  std::atomic<int64_t> next_task(0), released(kStage);
  std::vector<std::atomic<int>> left((size_t)nchunk);
  for (auto& l : left) l.store(nslice);
  std::atomic<int> bad(0), stop(0);
  auto worker = [&]() {
    for (;;) {
      const int64_t t = next_task.fetch_add(1);
      const int64_t c = t / nslice;
      if (c >= nchunk) return;
      while (c >= released.load(std::memory_order_acquire)) { if (stop.load()) return; std::this_thread::yield(); }
      const int sl = (int)(t % nslice);
      const int64_t j0 = c * chunk_cols, pc = std::min(chunk_cols, p - j0);
      const int64_t a = pc * sl / nslice, b = pc * (sl + 1) / nslice;
      if (b > a && narrow_columns(X, ld, n, ldd, j0 + a, j0 + b, stage[c % kStage] + a * ldd, lo, hi, offs, gmins)) bad.store(1);
      left[(size_t)c].fetch_sub(1, std::memory_order_release);
    }
  };
  std::vector<std::thread> pool;
  for (int t = 0; t < nthr; t++) pool.emplace_back(worker);
  cudaError_t ce = cudaSuccess;
  int64_t synced = 0;  // copies known to have finished
  for (int64_t c = 0; c < nchunk && ce == cudaSuccess; c++) {
    while (left[(size_t)c].load(std::memory_order_acquire) > 0) {
      if (synced < c && cudaEventQuery(done[synced % kStage]) == cudaSuccess) released.store(++synced + kStage, std::memory_order_release);
      else std::this_thread::yield();
    }
    const int64_t j0 = c * chunk_cols, pc = std::min(chunk_cols, p - j0);
    ce = cudaMemcpyAsync(h->x8_own.p + j0 * ldd, stage[c % kStage], (size_t)pc * ldd, cudaMemcpyHostToDevice, h->stream);
    if (ce == cudaSuccess) ce = cudaEventRecord(done[c % kStage], h->stream);
    while (ce == cudaSuccess && synced <= c && c + 1 < nchunk && c + 1 >= synced + kStage) {  // the next chunk cannot start before an older copy ends
      ce = cudaEventSynchronize(done[synced % kStage]);
      released.store(++synced + kStage, std::memory_order_release);
    }
  }
  stop.store(1);
  for (auto& th : pool) th.join();
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(h->stream);
  release_staging();
  cudaGetLastError();
  if (ce != cudaSuccess) return fail(BWGR_ERR_CUDA, "bwgr_geno_load_f64: %s", cudaGetErrorString(ce));
  if (bad.load()) return fail(BWGR_ERR_ARG, "bwgr_geno_load_f64: non-integer or out-of-range genotype");
  if (allow_offset) for (double v : h->col_offset) if (v != 0.0) { h->has_offset = true; break; }
  return finish_store(h, storage);
}
int bwgr_geno_load_f64(bwgr_handle* h, const double* X, int64_t n, int64_t p, int64_t ld, int storage) {
  return load_f64_common(h, X, n, p, ld, storage, false);
}
int bwgr_geno_load_f64_centred(bwgr_handle* h, const double* X, int64_t n, int64_t p, int64_t ld, int storage) {
  return load_f64_common(h, X, n, p, ld, storage, true);
}

// On-disk ingestion (SURVEY 8f rank 4): a PLINK .bed file is already 2 bits per genotype; it is read in chunks of columns, uploaded as
// is (n/4 bytes per marker instead of R's 8n) and decoded on the device.  n, p = the line counts of the .fam / .bim files.
int bwgr_geno_load_bed(bwgr_handle* h, const char* path, int64_t n, int64_t p, int storage, int missing, int64_t* nmissing_out) {
  if (!path) return fail(BWGR_ERR_ARG, "path is NULL");
  if (missing < -2 || missing > 2) return fail(BWGR_ERR_ARG, "missing must be -2 (rounded column mean), -1 (reject) or a code 0..2");
  int rc = prepare_store(h, n, p, storage);
  if (rc) return rc;
  h->col_offset.clear(); h->has_offset = false;
  FILE* fp = fopen(path, "rb");
  if (!fp) return fail(BWGR_ERR_ARG, "cannot open %s", path);
  unsigned char magic[3] = {0, 0, 0};
  if (fread(magic, 1, 3, fp) != 3 || magic[0] != 0x6C || magic[1] != 0x1B) { fclose(fp); return fail(BWGR_ERR_ARG, "%s is not a PLINK .bed file", path); }
  if (magic[2] != 0x01) { fclose(fp); return fail(BWGR_ERR_UNSUPPORTED, "%s is sample-major; only the variant-major .bed layout is read", path); }
  const int64_t bpc = (n + 3) / 4;
  const int64_t chunk_cols = std::max<int64_t>(1, std::min<int64_t>(p, ((int64_t)64 << 20) / bpc));
  uint8_t* stage = nullptr;
  DevBuf<uint8_t> dbed;
  DevBuf<unsigned long long> dmiss;
  const size_t stage_bytes = (size_t)chunk_cols * bpc;
  if (pinned_alloc(reinterpret_cast<void**>(&stage), stage_bytes) != cudaSuccess || dbed.alloc(stage_bytes) != cudaSuccess || dmiss.alloc(1) != cudaSuccess) {
    pinned_free(stage, stage_bytes);
    fclose(fp);
    return fail(BWGR_ERR_CUDA, "staging allocation failed");
  }
  cudaMemsetAsync(dmiss.p, 0, sizeof(unsigned long long), h->stream);
  cudaError_t ce = cudaSuccess;
  bool short_read = false;
  for (int64_t j0 = 0; j0 < p && ce == cudaSuccess; j0 += chunk_cols) {
    const int64_t pc = std::min(chunk_cols, p - j0);
    if (fread(stage, 1, (size_t)pc * bpc, fp) != (size_t)pc * bpc) { short_read = true; break; }
    ce = cudaMemcpyAsync(dbed.p, stage, (size_t)pc * bpc, cudaMemcpyHostToDevice, h->stream);
    if (ce != cudaSuccess) break;
    launch_decode_bed(dbed.p, bpc, (int)n, (int)pc, h->x8_own.p + j0 * h->ld, h->ld, missing, h->err.p, dmiss.p, h->stream);
    h->launches++;
    ce = cudaStreamSynchronize(h->stream);  // the staging buffer is reused by the next fread
  }
  fclose(fp);
  unsigned long long nm = 0;
  if (ce == cudaSuccess) ce = cudaMemcpy(&nm, dmiss.p, sizeof nm, cudaMemcpyDeviceToHost);
  pinned_free(stage, stage_bytes);
  if (short_read) return fail(BWGR_ERR_ARG, "%s is shorter than 3 + p * ceil(n/4) bytes (n=%lld, p=%lld)", path, (long long)n, (long long)p);
  if (ce != cudaSuccess) return fail(BWGR_ERR_CUDA, "bwgr_geno_load_bed: %s", cudaGetErrorString(ce));
  if (nmissing_out) *nmissing_out = (int64_t)nm;
  rc = check_err_flag(h, "bwgr_geno_load_bed (missing genotype calls and missing = -1)");
  if (rc) return rc;
  return finish_store(h, storage);
}

static int load_i8_common(bwgr_handle* h, const int8_t* X, int64_t n, int64_t p, int64_t ld, int storage, cudaMemcpyKind kind) {
  if (!X || ld < n) return fail(BWGR_ERR_ARG, "bad X / ld");
  int rc = prepare_store(h, n, p, storage);
  if (rc) return rc;
  CU(cudaMemcpy2DAsync(h->x8_own.p, h->ld, X, ld, n, p, kind, h->stream));
  launch_zero_pad(h->x8_own.p, h->ld, (int)n, (int)p, h->stream);
  h->launches++;
  return finish_store(h, storage);
}
int bwgr_geno_load_i8(bwgr_handle* h, const int8_t* X, int64_t n, int64_t p, int64_t ld, int storage) {
  return load_i8_common(h, X, n, p, ld, storage, cudaMemcpyHostToDevice);
}
int bwgr_geno_load_i8_device(bwgr_handle* h, const int8_t* dX, int64_t n, int64_t p, int64_t ld, int storage) {
  return load_i8_common(h, dX, n, p, ld, storage, cudaMemcpyDeviceToDevice);
}

int bwgr_geno_info(bwgr_handle* h, int64_t* n, int64_t* p, int64_t* ld_bytes, int* storage, int64_t* total_bytes) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  const int64_t ldb = h->storage == BWGR_STORE_2BIT ? h->ldb : h->storage == BWGR_STORE_F32 ? h->ld * 4 : h->ld;
  if (n) *n = h->n;
  if (p) *p = h->p;
  if (ld_bytes) *ld_bytes = ldb;
  if (storage) *storage = h->storage;
  if (total_bytes) *total_bytes = ldb * h->p;
  return 0;
}

int bwgr_geno_raw(bwgr_handle* h, uint8_t* out) {
  if (!h || !h->p || !out) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  const void* src = h->storage == BWGR_STORE_2BIT ? (const void*)h->x2.p : h->storage == BWGR_STORE_F32 ? (const void*)h->xf_own.p : (const void*)h->x8;
  const int64_t ldb = h->storage == BWGR_STORE_2BIT ? h->ldb : h->storage == BWGR_STORE_F32 ? h->ld * 4 : h->ld;
  CU(cudaMemcpyAsync(out, src, (size_t)ldb * h->p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int bwgr_geno_unpack_i8(bwgr_handle* h, int8_t* out) {
  if (!h || !h->p || !out) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (h->storage == BWGR_STORE_F32) return fail(BWGR_ERR_UNSUPPORTED, "the float32 store holds real-valued genotypes: read it with bwgr_geno_raw");
  if (h->storage == BWGR_STORE_I8) {
    CU(cudaMemcpy2DAsync(out, h->n, h->x8, h->ld, h->n, h->p, cudaMemcpyDeviceToHost, h->stream));
  } else {
    DevBuf<int8_t> tmp;
    if (tmp.alloc((size_t)h->ld * h->p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    launch_unpack_2bit(h->x2.p, h->ldb, (int)h->n, (int)h->p, tmp.p, h->ld, h->stream);
    h->launches++;
    CU(cudaMemcpy2DAsync(out, h->n, tmp.p, h->ld, h->n, h->p, cudaMemcpyDeviceToHost, h->stream));
  }
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int bwgr_geno_stats(bwgr_handle* h, double* xx, double* sx) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (xx) std::copy(h->h_xx.begin(), h->h_xx.end(), xx);
  if (sx) std::copy(h->h_sx.begin(), h->h_sx.end(), sx);
  return 0;
}

}  // extern "C"
