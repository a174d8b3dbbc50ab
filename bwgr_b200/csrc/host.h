// host.h -- the types and helpers the host translation units of the C ABI (include/bwgr_b200.h) share: handle.cu, store.cu,
// fit.cu, solvers.cu and mrr_host.cu.
#pragma once
#include <cuda.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <random>
#include <string>
#include <utility>
#include <vector>

#include "../../include/bwgr_b200.h"
#include "kernels.h"

namespace bwgr::host {

int fail(int code, const char* fmt, ...);

#define CU(call)                                                                                      \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess) return fail(BWGR_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

// Device and pinned-host blocks released by a handle are kept for the next one: the drop-in creates and destroys a store and a
// fit per emRR(y, gen) call, and cudaFree / cudaFreeHost of gigabyte blocks cost anything from 3 to 200 ms each on a busy
// driver (measured: tools/load_probe.py).  Exact-size reuse, bounded (BWGR_CACHE_GB, default 24; 0 = off), emptied by bwgr_trim().
struct BlockCache {
  struct Blk { void* p; size_t bytes; int dev; bool host; };
  std::mutex mu;
  std::vector<Blk> blocks;
  size_t held = 0;
  static size_t limit() {
    static const size_t lim = [] { const char* e = getenv("BWGR_CACHE_GB"); return (size_t)((e ? atof(e) : 24.0) * 1073741824.0); }();
    return lim;
  }
  void* take(size_t bytes, int dev, bool host) {
    std::lock_guard<std::mutex> l(mu);
    for (size_t i = 0; i < blocks.size(); i++)
      if (blocks[i].bytes == bytes && blocks[i].dev == dev && blocks[i].host == host) {
        void* p = blocks[i].p;
        held -= bytes;
        blocks.erase(blocks.begin() + (long)i);
        return p;
      }
    return nullptr;
  }
  static void drop(const Blk& b) { if (b.host) cudaFreeHost(b.p); else { int cur = 0; cudaGetDevice(&cur); cudaSetDevice(b.dev); cudaFree(b.p); cudaSetDevice(cur); } }
  void give(void* p, size_t bytes, int dev, bool host) {
    if (bytes > limit() || bytes < 4096) { drop({p, bytes, dev, host}); return; }
    std::lock_guard<std::mutex> l(mu);
    blocks.push_back({p, bytes, dev, host});
    held += bytes;
    while (held > limit() && !blocks.empty()) { held -= blocks.front().bytes; drop(blocks.front()); blocks.erase(blocks.begin()); }
  }
  void trim() {
    std::lock_guard<std::mutex> l(mu);
    for (auto& b : blocks) drop(b);
    blocks.clear(); held = 0;
  }
};
BlockCache& block_cache();

template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  int dev = 0;
  bool cacheable = true;  // false: memory other processes have mapped (cudaIpc)
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;  // a copy would hand the same block back to the cache twice
  DevBuf& operator=(const DevBuf&) = delete;
  void swap(DevBuf& o) { std::swap(p, o.p); std::swap(n, o.n); std::swap(dev, o.dev); std::swap(cacheable, o.cacheable); }
  cudaError_t alloc(size_t count) {
    release();
    n = count;
    if (!count) return cudaSuccess;
    const size_t bytes = count * sizeof(T);
    cudaGetDevice(&dev);
    if (cacheable) {
      if (void* q = block_cache().take(bytes, dev, false)) {
        p = static_cast<T*>(q);
        // a fresh cudaMalloc block usually reads as zeros; keep that for the small state buffers (the big ones are stores and
        // bands their producers overwrite in full)
        if (bytes <= ((size_t)256 << 20)) { cudaError_t e = cudaMemset(p, 0, bytes); if (e != cudaSuccess) return e; return cudaDeviceSynchronize(); }
        return cudaSuccess;
      }
    }
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&p), bytes);
    if (e != cudaSuccess && cacheable) {  // the cache may be what fills the device
      cudaGetLastError();
      block_cache().trim();
      e = cudaMalloc(reinterpret_cast<void**>(&p), bytes);
    }
    if (e != cudaSuccess) { p = nullptr; n = 0; }
    return e;
  }
  void release() {
    if (p) {
      if (cacheable) {
        int cur = 0;
        cudaGetDevice(&cur);
        if (cur != dev) cudaSetDevice(dev);
        cudaDeviceSynchronize();  // what cudaFree would have implied: nothing in flight still uses the block
        if (cur != dev) cudaSetDevice(cur);
        block_cache().give(p, n * sizeof(T), dev, false);
      } else {
        cudaFree(p);
      }
    }
    p = nullptr; n = 0;
  }
  ~DevBuf() { release(); }
};

inline cudaError_t pinned_alloc(void** p, size_t bytes) {
  if ((*p = block_cache().take(bytes, -1, true))) return cudaSuccess;
  return cudaMallocHost(p, bytes);
}
inline void pinned_free(void* p, size_t bytes) { if (p) block_cache().give(p, bytes, -1, true); }

// NCCL is resolved at run time (dlopen): a single-GPU user of the library never needs it.
struct NcclApi {
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*CommSplit)(ncclComm_t, int, int, ncclComm_t*, void*) = nullptr;  // optional (NCCL >= 2.18)
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
};
NcclApi& nccl();
#define NC(call)                                                                                                     \
  do {                                                                                                               \
    ncclResult_t r_ = (call);                                                                                        \
    if (r_ != ncclSuccess) return fail(BWGR_ERR_CUDA, "%s failed: %s", #call, nccl().GetErrorString ? nccl().GetErrorString(r_) : "?"); \
  } while (0)

constexpr int kPermRing = 8;

// Kernel family of a fit: small_n.cu (one CTA per system), sweep_pipe.cu (pipelined blocked sweep) or grid_sweep.cu
enum class Family { SmallN, Blocked, Grid };

// The state of one fit, from fit_begin to the end of the fit (the handle's `fit` is null between fits).
struct Fit {
  explicit Fit(const bwgr_handle* h) : h(h) {}
  ~Fit();
  const bwgr_handle* h;
  int model = 0;        // device Model id
  int nsys = 0;
  int it_target = 0;    // sweeps requested by the reference recipe
  int sweeps_issued = 0;
  bool shuffled = true; // EM: shuffled order; Gibbs: natural
  Family family = Family::SmallN;
  bool grid_blocked = false;            // grid family: its blocked variant (unmasked systems)
  DevBuf<unsigned long long> gridacc;   // its per-marker accumulator words
  bool masked = false;
  int rows_per_cta = 0, grid = 0, nblocks = 0;
  bool gram_cached = false;
  uint64_t seed = 0;
  int chain0 = 0;                       // Philox chain index of system 0
  std::vector<SysScalars> sc0;
  std::vector<float> vy, MSx, cxx;      // per system constants needed for outputs
  std::vector<int> order;               // host marker order (cumulative shuffles)
  DevBuf<float> y, e, b, d, vbv, b_prev, B, D, VBv, xx_sys, gram;
  DevBuf<uint8_t> mask, cnt;            // cnt / row_w: row multiplicities of a bagged sweep with replacement (uint8 and float)
  DevBuf<float> row_w;
  bool weighted = false;
  DevBuf<SysScalars> sc;
  DevBuf<int> perm;                     // [kPermRing][p]
  DevBuf<long long> trace;
  // pipelined sweep (sweep_pipe.cu)
  int lookahead = 0, nbuf = 0, sring = 2, nworkers = 0, nband = 1, full_inv = 0, cl = 0, nclusters = 0;
  DevBuf<float> tinv;                   // (I + A L)^-1 of every block of the current sweep (block_inv.cu)
  uint32_t tag = 0;
  DevBuf<unsigned long long> dew, part, hsum;
  DevBuf<float> wts;  // emML: marker weights d_j
  float* gram_p = nullptr;              // Gram band in use: f.gram (per fit) or the handle's natural-order cache
  // Gram band of sweep s + 1 computed on the handle's side stream while sweep s runs (the clustered sweep leaves SMs idle)
  bool overlap = false;
  DevBuf<float> gram2;                  // band buffer of the odd sweeps (f.gram: even sweeps)
  int gram_ahead = -1;                  // sweep whose band has been issued on the side stream (-1: none)
  // single Kuo-Mallick sweep / wgr driver
  DevBuf<float> xx_over;                // caller's xx (KMUP takes it as an argument, :12) / centred xx (MRR3)
  DevBuf<double> esum; DevBuf<float> emaxv;  // row-sharded fit: all-reduced epilogue sums
  DevBuf<float> sx_dev, cshift;         // MRR3: column sums (centred columns) and the per-system mean shift of a sweep
  bool skip_epilogue = false;
  bool wgr_mode = false;
  DevBuf<WgrState> wst;
  WgrArgs wgr_args;
  int* h_perm = nullptr;                // pinned [kPermRing][p]
  size_t h_perm_bytes = 0;
  cudaEvent_t perm_free[kPermRing] = {};
};

struct FitSpec {
  int model;      // device Model
  int nsys;
  bool shuffled;
  const uint8_t* row_mask;  // host, n x nsys or null
  const uint8_t* row_cnt = nullptr;  // KMUP2 on rows drawn with replacement: multiplicity of every row (host, n; nsys = 1), row_mask = cnt != 0
  float df, R2, Pi, alpha, pi;
  int it, bi;
  uint64_t seed;
  int chain0 = 0;  // Philox chain index of system 0 (Gibbs): system t draws from chain chain0 + t
};

// Held by a one-shot entry point from the start of its fit to its return: the fit is released whatever the exit, so a failed call
// leaves no fit that bwgr_em_sweeps / bwgr_em_end could continue.
struct FitGuard {
  bwgr_handle* h;
  ~FitGuard();
};

// Geometry of the pipelined sweep: W streaming CTAs (row slabs of R rows, R <= 512) + one solver CTA, look-ahead D,
// nbuf X tiles per worker.  False if the shape does not fit one SM's shared memory / TMEM.
struct PipePlan { int R, W, nbuf, D, sring, full_inv, cl, nclusters; };
bool plan_pipe(const bwgr_handle* h, int model, int ns, PipePlan* pl);
// rows per CTA and CTAs of the grid family for this store
void grid_geometry(bwgr_handle* h, int* rp, int* grid);

// Device scratch of rows_col_stats: exact int64 sums (int8 store, 0/1 mask) or double sums, allocated on first use
struct ColStatBufs {
  DevBuf<long long> xx_i, sx_i;
  DevBuf<double> xx_d, sx_d;
};
int rows_col_stats(bwgr_handle* h, ColStatBufs& s, const uint8_t* rows, bool cnt, float* xx_sys, std::vector<double>* xx, std::vector<double>* sx);
int take_err_flag(bwgr_handle* h, int* flag);
int check_err_flag(bwgr_handle* h, const char* where);
int dist_allreduce_host(bwgr_handle* h, double* v, int cnt, bool is_max);
float fvar_f(const std::vector<float>& x);
int fit_begin(bwgr_handle* h, const FitSpec& s, const double* y);
int fit_sweeps(bwgr_handle* h, int nsweeps);
int fit_sweeps_until_done(bwgr_handle* h, std::vector<SysScalars>& sc);
int fit_hat(bwgr_handle* h, int k, const float* b_dev, const float* mu_dev, float* hat_dev);
int fitted_values(bwgr_handle* h, int nsys, const float* b, bool b_on_host, const float* mu, std::vector<float>& hat);
void dump_trace(bwgr_handle* h);

}  // namespace bwgr::host

struct bwgr_handle {
  template <class T> using DevBuf = bwgr::host::DevBuf<T>;
  int device = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  int num_sms = 0;
  size_t smem_optin = 0;
  // genotype store
  DevBuf<int8_t> x8_own;
  const int8_t* x8 = nullptr;
  DevBuf<float> xf_own;  // float32 store (BWGR_STORE_F32): real-valued genotypes, grid family only
  DevBuf<uint8_t> x2;
  DevBuf<uint8_t> x2f;  // packed 2-bit shadow in the layout gram_fp4.cu expands to E2M1 nibbles (codes 0..2 only)
  DevBuf<uint8_t> x2g;  // packed 2-bit shadow of an int8 store with codes 0..2: what the Gram kernel gathers (4x fewer bytes)
  int64_t n = 0, p = 0, ld = 0, ldb = 0;
  int storage = BWGR_STORE_I8;
  DevBuf<long long> xx_i, sx_i;
  DevBuf<float> xx_f;
  std::vector<double> h_xx, h_sx;
  double xx_max = 0;  // max_j h_xx[j]: bounds every Gram entry and every |x_j'x_k| (Cauchy-Schwarz)
  std::vector<double> col_offset;  // bwgr_geno_load_f64_centred: x = code + col_offset[j]
  bool has_offset = false;
  DevBuf<int> err;
  // tuning
  int path = BWGR_PATH_AUTO, grid = 0;
  DevBuf<float> gram_nat;  // Gram band of the natural marker order (Gibbs / KMUP / wgr): depends on the store only
  int gram_nat_band = 0;
  DevBuf<float> hat_work;  // partial sums of the fitted values (fit_hat), also used with no fit in progress (bwgr_fitted_sys)
  // row-sharded fit over the GPUs of a node (bwgr_dist_*)
  int world = 1, rank = 0;
  int64_t n_global = 0;
  ncclComm_t comm = nullptr;
  ncclComm_t comm_side = nullptr;  // second communicator over the same ranks: collectives of the side stream (Gram band computed ahead)
  DevBuf<unsigned long long> hx_own;        // this rank's exchange ring [8][world][32][128]
  unsigned long long* hx[8] = {};           // every rank's ring as seen from this process (peer memory)
  bool hx_connected = false;
  unsigned long long dist_gen = 0;          // global block sequence number (same on every rank)
  DevBuf<double> dscratch;                  // small all-reduce scratch
  // side stream for work that overlaps the clustered sweep, gated by a flag word the sweep kernel stores (stream memory operations)
  cudaStream_t side = nullptr;
  cudaEvent_t side_done[2] = {nullptr, nullptr};
  DevBuf<unsigned int> started;
  unsigned int started_seq = 0;
  CUresult (*wait32)(CUstream, CUdeviceptr, cuuint32_t, unsigned int) = nullptr;
  CUresult (*write32)(CUstream, CUdeviceptr, cuuint32_t, unsigned int) = nullptr;
  int fp8_codes = 0;  // all genotypes are codes 0..7 (and n small enough): the Gram kernel may use the exact E4M3 path
  int64_t launches = 0;
  std::unique_ptr<bwgr::host::Fit> fit;  // the fit in progress, if any
  // optional per-kernel timing (bwgr_profile)
  bool profiling = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_ev[4];  // gram, sweep, epilogue, block inverses
  double prof_ms[4] = {0, 0, 0, 0};
  int64_t prof_n[4] = {0, 0, 0, 0};
  cudaEvent_t prof_begin(int cls) {
    if (!profiling) return nullptr;
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    prof_ev[cls].push_back({a, b});
    cudaEventRecord(a, stream);
    return b;
  }
  void prof_end(cudaEvent_t b) { if (b) cudaEventRecord(b, stream); }
  void prof_collect() {
    for (int c = 0; c < 4; c++) {
      for (auto& pr : prof_ev[c]) {
        float ms = 0;
        cudaEventSynchronize(pr.second);
        cudaEventElapsedTime(&ms, pr.first, pr.second);
        prof_ms[c] += ms; prof_n[c]++;
        cudaEventDestroy(pr.first); cudaEventDestroy(pr.second);
      }
      prof_ev[c].clear();
    }
  }

  bwgr::GenoView view() const {
    bwgr::GenoView g;
    g.x8 = x8; g.x2 = x2.p; g.xf = xf_own.p; g.ld = ld; g.ldb = ldb; g.n = (int)n; g.p = (int)p;
    g.storage = storage;
    return g;
  }
  // view handed to the Gram kernel: the int8 store plus, when it exists, the packed shadow copy
  bwgr::GenoView gram_view() const {
    bwgr::GenoView g = view();
    if (x2g.p) { g.x2 = x2g.p; g.ldb = ld / 4; }
    return g;
  }
};

inline bwgr::host::FitGuard::~FitGuard() { if (h) h->fit.reset(); }
