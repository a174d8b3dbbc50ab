// capi.cu -- the thin extern "C" layer of include/bwgr_b200.h: handle, genotype store, and the host
// orchestration of a fit (what stays C++ behind Rcpp in the drop-in; SURVEY 8b).
//
// Host responsibilities, all O(p) or O(n) per sweep and overlapped with the GPU through the stream:
//   * the marker order of every shuffled solver -- std::shuffle(order, std::mt19937(sweep)), cumulative
//     (Rcpp20260726ai.cpp:329-331) -- produced with libstdc++ itself and uploaded ahead of use;
//   * initial hyper-parameters per solver (SURVEY A.1), in float like the reference;
//   * choosing the kernel family (small-n CTA-per-system vs blocked whole-GPU sweep).
// There is deliberately no CPU compute path: every sweep runs in the CUDA kernels of this directory.
#include <cuda.h>
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <atomic>
#include <mutex>
#include <sched.h>
#include <thread>
#include <vector>

#include "../../include/bwgr_b200.h"
#include "kernels.h"

using namespace bwgr;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

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
BlockCache& block_cache() { static BlockCache* c = new BlockCache; return *c; }  // never destroyed: no CUDA calls at process exit

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

constexpr int kPermRing = 8;

struct Fit {
  bool active = false;
  int model = 0;        // device Model id
  int nsys = 0;
  int it_target = 0;    // sweeps requested by the reference recipe
  int sweeps_issued = 0;
  bool shuffled = true; // EM: shuffled order; Gibbs: natural
  bool blocked = false;
  bool gridfam = false;                 // grid family (grid_sweep.cu)
  bool grid_blocked = false;            // ... its blocked variant (unmasked systems)
  DevBuf<unsigned long long> gridacc;   // its per-marker accumulator words
  bool masked = false;
  int rows_per_cta = 0, grid = 0, nblocks = 0;
  bool gram_cached = false;
  uint64_t seed = 0;
  int chain0 = 0;                       // Philox chain index of system 0
  std::vector<SysScalars> sc0;
  std::vector<float> vy, MSx, cxx;      // per system constants needed for outputs
  std::vector<int> order;               // host marker order (cumulative shuffles)
  DevBuf<float> y, e, b, d, vbv, b_prev, B, D, VBv, xx_sys, gram, work;
  DevBuf<uint8_t> mask, cnt;            // cnt / row_w: row multiplicities of a bagged sweep with replacement (uint8 and float)
  DevBuf<float> row_w;
  bool weighted = false;
  DevBuf<SysScalars> sc;
  DevBuf<int> perm;                     // [kPermRing][p]
  DevBuf<long long> trace;
  // pipelined sweep (sweep_pipe.cu)
  int lookahead = 0, nbuf = 0, sring = 2, nworkers = 0, nc = 1, nband = 1, full_inv = 0, cl = 0, nclusters = 0;
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
  bool perm_ev_valid[kPermRing] = {};
  void reset() {
    active = false;
    if (h_perm) { pinned_free(h_perm, h_perm_bytes); h_perm = nullptr; }
    for (int i = 0; i < kPermRing; i++)
      if (perm_free[i]) { cudaEventDestroy(perm_free[i]); perm_free[i] = nullptr; perm_ev_valid[i] = false; }
  }
};

}  // namespace

namespace {
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
NcclApi& nccl() {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (lib) {
      api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(lib, "ncclGetUniqueId"));
      api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(lib, "ncclCommInitRank"));
      api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(dlsym(lib, "ncclAllReduce"));
      api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(lib, "ncclCommDestroy"));
      api.CommSplit = reinterpret_cast<decltype(api.CommSplit)>(dlsym(lib, "ncclCommSplit"));
      api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(lib, "ncclGetErrorString"));
      api.ok = api.GetUniqueId && api.CommInitRank && api.AllReduce && api.CommDestroy;
    }
  }
  return api;
}
#define NC(call)                                                                                                     \
  do {                                                                                                               \
    ncclResult_t r_ = (call);                                                                                        \
    if (r_ != ncclSuccess) return fail(BWGR_ERR_CUDA, "%s failed: %s", #call, nccl().GetErrorString ? nccl().GetErrorString(r_) : "?"); \
  } while (0)
}  // namespace

struct bwgr_handle {
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
  Fit fit;
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

  GenoView view() const {
    GenoView g;
    g.x8 = x8; g.x2 = x2.p; g.xf = xf_own.p; g.ld = ld; g.ldb = ldb; g.n = (int)n; g.p = (int)p;
    g.storage = storage;
    return g;
  }
};

namespace {

// view handed to the Gram kernel: the int8 store plus, when it exists, the packed shadow copy
GenoView gram_view(const bwgr_handle* h) {
  GenoView g = h->view();
  if (h->x2g.p) { g.x2 = h->x2g.p; g.ldb = h->ld / 4; }
  return g;
}

// Reads the device error word into *flag (0: no kernel raised one) and clears it.
int take_err_flag(bwgr_handle* h, int* flag) {
  *flag = 0;
  CU(cudaMemcpyAsync(flag, h->err.p, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (*flag) CU(cudaMemsetAsync(h->err.p, 0, sizeof(int), h->stream));
  return 0;
}

int check_err_flag(bwgr_handle* h, const char* where) {
  int flag = 0;
  const int rc = take_err_flag(h, &flag);
  if (rc || !flag) return rc;
  const char* what = flag == 1 ? "non-integer or out-of-range genotype" : flag == 2 ? "tensor-core pipeline watchdog"
                     : flag == 3 ? "grid barrier watchdog" : flag == 4 ? "fixed-point range of g exceeded" : "device error";
  return fail(flag == 1 ? BWGR_ERR_ARG : BWGR_ERR_NUMERIC, "%s: %s", where, what);
}

// Row-sharded fit: all-reduce `cnt` host doubles over the ranks (sum or max) through a device scratch buffer.
int dist_allreduce_host(bwgr_handle* h, double* v, int cnt, bool is_max) {
  if (h->world <= 1) return 0;
  if (h->dscratch.n < (size_t)cnt && h->dscratch.alloc(std::max(cnt, 256)) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  CU(cudaMemcpyAsync(h->dscratch.p, v, sizeof(double) * cnt, cudaMemcpyHostToDevice, h->stream));
  NC(nccl().AllReduce(h->dscratch.p, h->dscratch.p, (size_t)cnt, ncclDouble, is_max ? ncclMax : ncclSum, h->comm, h->stream));
  CU(cudaMemcpyAsync(v, h->dscratch.p, sizeof(double) * cnt, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int finish_store(bwgr_handle* h, int storage) {
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

int prepare_store(bwgr_handle* h, int64_t n, int64_t p, int storage) {
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

// ---- host-side helpers that mirror the reference's float arithmetic -------------------------------
float fvar_f(const std::vector<float>& x) {  // fvar, Rcpp20260726ai.cpp:7-9 (sums in double, rounded once)
  double m = 0;
  for (float v : x) m += v;
  const float mean = (float)(m / (double)x.size());
  double s = 0;
  for (float v : x) { const float t = v - mean; s += (double)t * t; }
  return (float)s / (float)(x.size() - 1);
}

// Held by a one-shot entry point from the start of its fit to its return: the fit is released whatever the exit, so a failed call
// leaves no fit that bwgr_em_sweeps / bwgr_em_end could continue.
struct FitGuard {
  bwgr_handle* h;
  ~FitGuard() { if (h) h->fit.reset(); }
};

}  // namespace

extern "C" {

const char* bwgr_last_error(void) { return g_err.c_str(); }
int bwgr_version(void) { return 100; }
void bwgr_trim(void) { block_cache().trim(); }

int bwgr_create(int device, bwgr_handle** out) {
  if (!out) return fail(BWGR_ERR_ARG, "out is NULL");
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return fail(BWGR_ERR_CUDA, "no CUDA device: this library has no CPU path");
  if (device < 0 || device >= count) return fail(BWGR_ERR_ARG, "device %d out of range (%d devices)", device, count);
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(BWGR_ERR_UNSUPPORTED, "device %d is sm_%d%d; this build targets sm_100a (B200) only", device, prop.major, prop.minor);
  bwgr_handle* h = new bwgr_handle();
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  h->smem_optin = prop.sharedMemPerBlockOptin;
  if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return fail(BWGR_ERR_CUDA, "cudaStreamCreate failed"); }
  h->stream = h->own_stream;
  {  // side stream + stream memory operations (driver entry points through the runtime: no link against libcuda)
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    void *fw = nullptr, *fs = nullptr;
    cudaDriverEntryPointQueryResult q1, q2;
    if (cudaStreamCreateWithPriority(&h->side, cudaStreamNonBlocking, lo) == cudaSuccess &&
        cudaEventCreateWithFlags(&h->side_done[0], cudaEventDisableTiming) == cudaSuccess &&
        cudaEventCreateWithFlags(&h->side_done[1], cudaEventDisableTiming) == cudaSuccess && h->started.alloc(1) == cudaSuccess &&
        cudaGetDriverEntryPoint("cuStreamWaitValue32", &fw, cudaEnableDefault, &q1) == cudaSuccess && q1 == cudaDriverEntryPointSuccess &&
        cudaGetDriverEntryPoint("cuStreamWriteValue32", &fs, cudaEnableDefault, &q2) == cudaSuccess && q2 == cudaDriverEntryPointSuccess) {
      h->wait32 = reinterpret_cast<decltype(h->wait32)>(fw);
      h->write32 = reinterpret_cast<decltype(h->write32)>(fs);
      cudaMemset(h->started.p, 0, sizeof(unsigned int));
    }
    cudaGetLastError();
  }
  if (h->err.alloc(1) != cudaSuccess) { delete h; return fail(BWGR_ERR_CUDA, "cudaMalloc failed"); }
  cudaMemset(h->err.p, 0, sizeof(int));
  *out = h;
  return 0;
}

void bwgr_destroy(bwgr_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  h->fit.reset();
  for (int r = 0; r < h->world; r++)
    if (r != h->rank && h->hx[r]) cudaIpcCloseMemHandle(h->hx[r]);
  if (h->comm_side && nccl().ok) nccl().CommDestroy(h->comm_side);
  if (h->comm && nccl().ok) nccl().CommDestroy(h->comm);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  if (h->side) cudaStreamDestroy(h->side);
  for (int i = 0; i < 2; i++) if (h->side_done[i]) cudaEventDestroy(h->side_done[i]);
  delete h;
}

int bwgr_set_stream(bwgr_handle* h, void* s) {
  if (!h) return fail(BWGR_ERR_ARG, "null handle");
  CU(cudaStreamSynchronize(h->stream));
  h->stream = s ? reinterpret_cast<cudaStream_t>(s) : h->own_stream;
  return 0;
}

int bwgr_set_tuning(bwgr_handle* h, int block, int path, int grid) {
  if (!h) return fail(BWGR_ERR_ARG, "null handle");
  if (block >= 0 && block != kBlk) return fail(BWGR_ERR_UNSUPPORTED, "only block=%d is built", kBlk);
  if (path >= 0) {
    if (path > BWGR_PATH_GRID) return fail(BWGR_ERR_ARG, "bad path %d", path);
    h->path = path;
  }
  if (grid >= 0) h->grid = grid;
  return 0;
}

int64_t bwgr_launch_count(bwgr_handle* h) { return h ? h->launches : 0; }

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
    return fail(BWGR_ERR_CUDA, "cudaMallocHost(staging) failed");
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
  // the pinned staging buffers are kept for the life of the process (cudaMallocHost / cudaFreeHost cost tens of milliseconds
  // each and would otherwise be paid by every emRR(y, gen) call of the drop-in, which creates and destroys its store)
  static int8_t* s_stage[kStage] = {};
  static size_t s_stage_bytes = 0;
  static std::mutex s_mu;
  std::lock_guard<std::mutex> lock(s_mu);
  if (s_stage_bytes < chunk_bytes) {
    bool ok = true;
    for (int i = 0; i < kStage; i++) { if (s_stage[i]) cudaFreeHost(s_stage[i]); s_stage[i] = nullptr; }
    s_stage_bytes = 0;
    for (int i = 0; i < kStage && ok; i++) ok = cudaMallocHost(reinterpret_cast<void**>(&s_stage[i]), chunk_bytes) == cudaSuccess;
    if (!ok) {
      for (int i = 0; i < kStage; i++) { if (s_stage[i]) cudaFreeHost(s_stage[i]); s_stage[i] = nullptr; }
      return fail(BWGR_ERR_CUDA, "cudaMallocHost(staging) failed");
    }
    s_stage_bytes = chunk_bytes;
  }
  cudaEvent_t done[kStage] = {};
  for (int i = 0; i < kStage; i++)
    if (cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaEventCreate failed");
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
      if (b > a && narrow_columns(X, ld, n, ldd, j0 + a, j0 + b, s_stage[c % kStage] + a * ldd, lo, hi, offs, gmins)) bad.store(1);
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
    ce = cudaMemcpyAsync(h->x8_own.p + j0 * ldd, s_stage[c % kStage], (size_t)pc * ldd, cudaMemcpyHostToDevice, h->stream);
    if (ce == cudaSuccess) ce = cudaEventRecord(done[c % kStage], h->stream);
    while (ce == cudaSuccess && synced <= c && c + 1 < nchunk && c + 1 >= synced + kStage) {  // the next chunk cannot start before an older copy ends
      ce = cudaEventSynchronize(done[synced % kStage]);
      released.store(++synced + kStage, std::memory_order_release);
    }
  }
  stop.store(1);
  for (auto& th : pool) th.join();
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(h->stream);
  for (int i = 0; i < kStage; i++) cudaEventDestroy(done[i]);
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
  if (cudaMallocHost(reinterpret_cast<void**>(&stage), (size_t)chunk_cols * bpc) != cudaSuccess || dbed.alloc((size_t)chunk_cols * bpc) != cudaSuccess ||
      dmiss.alloc(1) != cudaSuccess) {
    if (stage) cudaFreeHost(stage);
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
  cudaFreeHost(stage);
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
    CU(cudaStreamSynchronize(h->stream));
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

// =====================================================================================================
// Fit orchestration shared by the EM and Gibbs families
// =====================================================================================================
namespace {

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

// Geometry of the pipelined sweep: W streaming CTAs (row slabs of R rows, R <= 512) + one solver CTA, look-ahead D,
// nbuf X tiles per worker.  False if the shape does not fit one SM's shared memory / TMEM.
struct PipePlan { int R, W, nbuf, D, sring, full_inv, cl, nclusters; };
bool plan_pipe(const bwgr_handle* h, int model, int ns, PipePlan* pl) {
  if (h->storage != BWGR_STORE_I8 || ns > 32) return false;
  int sms = h->grid > 1 ? std::min(h->grid, h->num_sms) : h->num_sms;  // CTAs of the flat topology
  if (h->world > 1 && h->grid <= 1 && h->x2f.p && h->comm_side && h->num_sms > 64) {
    // row-sharded fit, flat topology: the per-block chain is latency-bound, so ~104 CTAs sweep as fast as 148 and the SMs left idle
    // compute the next sweep's Gram band meanwhile (measured at 50k x 50k: 104 CTAs 1.54 ms per sweep, 120: 1.68, 148: 1.84)
    const int want = h->num_sms - 44;
    if ((h->ld + want - 2) / (want - 1) <= 496) sms = want;
  }
  if (sms < 2) return false;
  const int W0 = sms - 1;
  const int R = (int)(((h->ld + W0 - 1) / W0 + 15) / 16 * 16);
  if (R > 512) return false;
  const int W = (int)((h->ld + R - 1) / R);
  const int NA = (R + 127) / 128, N = ((4 * ns + 15) / 16) * 16;
  if ((NA + 1) * N > 512) return false;
  int D = 1;
  // one linear system on uncentred columns: the in-block solve applies the precomputed block inverse (block_inv.cu).
  // (MRR3's centred systems keep the stepwise solve.)
  const int full_inv = model_is_linear(model) && ns == 1 && model != M_MRR;
  pl->cl = 0; pl->nclusters = 0;
  // Clustered topology (sweep_pipe.cu): thread-block clusters of one solver + seven workers; steps travel through distributed shared
  // memory, and every worker adds its partial sums to L2 grid-sum words: one L2 hop per block.
  // Single GPU at the default grid, at most three systems; otherwise the flat topology (one solver CTA, two-hop L2 tree).  Row-sharded
  // fits use the flat one: a clustered variant with a third (NVLink) hop after the cluster exchange measured 1.79 ms against 1.43 ms per sweep.
  if (h->world <= 1 && h->grid <= 1 && sweep_pipe_cluster_ok(model, ns, full_inv)) {
    {
      // The sweep is latency-bound: 14 clusters sweep as fast as 15 (measured 1.226 against 1.235 ms at 50k x 50k), and every SM left
      // idle works on the next sweep's Gram band meanwhile (capi.cu fit_sweeps).  First choice: leave at least 36 SMs; if the rows per
      // worker then exceed the tile (512), take every cluster that fits.
      const int cap_side = std::max(2, (h->num_sms - 36) / 8);
      for (int nbuf = D + 2; nbuf >= D + 1; nbuf--)
      for (int pass = 0; pass < 2; pass++) {
        // rows per worker depend on the number of co-resident clusters, which depends on the shared memory per CTA: iterate
        int C = pass == 0 ? std::min(18, cap_side) : 18;
        for (int iter = 0; iter < 4 && C >= 2; iter++) {
          const int Wc = 7 * C;
          const int Rc = (int)(((h->ld + Wc - 1) / Wc + 15) / 16 * 16);
          if (Rc > 512) { C = 0; break; }
          const size_t smem = sweep_pipe_smem(Rc, ns, model, nbuf, 3, full_inv, 1);
          if (smem > h->smem_optin - 9216) { C = 0; break; }  // the kernel's static shared memory (barriers, system scalars) is ~9 KB
          const int Cmax = std::min(18, sweep_pipe_max_clusters(model, smem));
          if (Cmax >= C) break;
          C = Cmax;
        }
        if (C >= 2) {
          const int Wc = 7 * C;
          const int Rc = (int)(((h->ld + Wc - 1) / Wc + 15) / 16 * 16);
          const int NAc = (Rc + 127) / 128;
          if ((NAc + 1) * N <= 512 && sweep_pipe_smem(Rc, ns, model, nbuf, 3, full_inv, 1) <= h->smem_optin - 9216) {
            pl->R = Rc; pl->W = Wc; pl->nbuf = nbuf; pl->D = D; pl->sring = 3; pl->full_inv = full_inv; pl->cl = 1; pl->nclusters = C;
            return true;
          }
        }
      }
    }
  }
  for (; D >= 0; D--) {
    for (int sring = 3; sring >= 2; sring--)
      for (int nbuf = std::min(8, D + 3); nbuf >= D + 1; nbuf--)
        if (sweep_pipe_smem(R, ns, model, nbuf, sring, full_inv, 0) <= h->smem_optin - 8192) {
          pl->R = R; pl->W = W; pl->nbuf = nbuf; pl->D = D; pl->sring = sring; pl->full_inv = full_inv;
          return true;
        }
  }
  return false;
}

// rows per CTA and CTAs of the grid family for this store
void grid_geometry(bwgr_handle* h, int* rp, int* grid) {
  int r = (int)((h->ld + h->num_sms - 1) / h->num_sms);
  r = std::max(64, (r + 15) / 16 * 16);
  *rp = r;
  *grid = (int)((h->ld + r - 1) / r);
}

// family: 0 = small-n, 1 = blocked, 2 = grid; path: the BWGR_PATH_* to honour
int choose_path(bwgr_handle* h, const FitSpec& s, int path, int* family) {
  const GenoView g = h->view();
  const bool small_ok = h->storage != BWGR_STORE_F32 && small_n_fits(g, s.row_mask != nullptr, h->smem_optin, s.row_cnt != nullptr);
  PipePlan pl;
  const bool blocked_ok = !s.row_mask && plan_pipe(h, s.model, s.nsys, &pl);
  int grp = 0, ggrid = 0;
  grid_geometry(h, &grp, &ggrid);
  const bool grid_ok = (h->storage == BWGR_STORE_I8 || h->storage == BWGR_STORE_F32) && h->world <= 1 && s.nsys <= 32 && s.model != M_MRR &&
                       ggrid <= 255 && grid_sweep_smem(s.nsys, grp, s.row_mask != nullptr, h->storage == BWGR_STORE_F32) <= h->smem_optin;
  if (path == BWGR_PATH_SMALL_N) {
    if (!small_ok) return fail(BWGR_ERR_UNSUPPORTED, "small-n path: residual of n=%lld does not fit one SM", (long long)h->n);
    *family = 0;
  } else if (path == BWGR_PATH_BLOCKED) {
    if (!blocked_ok) return fail(BWGR_ERR_UNSUPPORTED, "blocked path needs the int8 store, no row mask, nsys<=32 and n <= 512 rows x grid");
    *family = 1;
  } else if (path == BWGR_PATH_GRID) {
    if (!grid_ok) return fail(BWGR_ERR_UNSUPPORTED, "grid path needs the int8 or float32 store, one GPU, nsys<=32 and the row slabs of all systems in shared memory");
    *family = 2;
  } else {
    const bool prefer_small = small_ok && (s.row_mask || s.nsys >= 8 || h->n <= 1024);
    if (prefer_small) *family = 0;
    else if (blocked_ok) *family = 1;
    else if (small_ok) *family = 0;
    else if (grid_ok) *family = 2;
    else return fail(BWGR_ERR_UNSUPPORTED, "no kernel family fits n=%lld nsys=%d storage=%d", (long long)h->n, s.nsys, h->storage);
  }
  return 0;
}

// Device scratch of rows_col_stats: exact int64 sums (int8 store, 0/1 mask) or double sums, allocated on first use
struct ColStatBufs {
  DevBuf<long long> xx_i, sx_i;
  DevBuf<double> xx_d, sx_d;
};

// Column statistics over the rows a system uses -- a 0/1 row mask, or (cnt) the multiplicity of every row -- with
// xx_j = sum_i w_i x_ij^2 as floats into slot t of f.xx_sys.  With xx / sx, both sums also come back as host doubles, and the float
// conversion runs on the host.
int rows_col_stats(bwgr_handle* h, ColStatBufs& s, const uint8_t* rows, bool cnt, int t, std::vector<double>* xx, std::vector<double>* sx) {
  const int64_t p = h->p;
  float* xx_sys = h->fit.xx_sys.p + (size_t)t * p;
  const bool exact = !cnt && h->storage != BWGR_STORE_F32;
  if (exact) {
    if (s.xx_i.n < (size_t)p && (s.xx_i.alloc(p) != cudaSuccess || s.sx_i.alloc(p) != cudaSuccess)) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    launch_col_stats_masked(h->view(), rows, s.xx_i.p, s.sx_i.p, h->stream);
  } else {
    if (s.xx_d.n < (size_t)p && (s.xx_d.alloc(p) != cudaSuccess || s.sx_d.alloc(p) != cudaSuccess)) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    if (cnt) launch_col_stats_cnt(h->view(), rows, s.xx_d.p, s.sx_d.p, h->stream);
    else launch_col_stats_f32(h->view(), rows, s.xx_d.p, s.sx_d.p, h->stream);
  }
  h->launches++;
  if (!xx) {
    if (exact) launch_ll_to_float(s.xx_i.p, xx_sys, (int)p, h->stream);
    else launch_d_to_float(s.xx_d.p, xx_sys, (int)p, h->stream);
    h->launches++;
    return 0;
  }
  xx->resize(p); sx->resize(p);
  if (exact) {
    std::vector<long long> hx(p), hs(p);
    CU(cudaMemcpyAsync(hx.data(), s.xx_i.p, sizeof(long long) * p, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(hs.data(), s.sx_i.p, sizeof(long long) * p, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    xx->assign(hx.begin(), hx.end()); sx->assign(hs.begin(), hs.end());  // exact: |sums| < 2^45
  } else {
    CU(cudaMemcpyAsync(xx->data(), s.xx_d.p, sizeof(double) * p, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(sx->data(), s.sx_d.p, sizeof(double) * p, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  std::vector<float> xf(p);
  for (int64_t j = 0; j < p; j++) xf[j] = (float)(*xx)[j];
  CU(cudaMemcpyAsync(xx_sys, xf.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int fit_begin(bwgr_handle* h, const FitSpec& s, const double* y) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!y) return fail(BWGR_ERR_ARG, "y is NULL");
  if (s.nsys < 1 || s.nsys > 4096) return fail(BWGR_ERR_ARG, "bad nsys %d", s.nsys);
  if (h->has_offset && s.model != M_MRR)
    return fail(BWGR_ERR_UNSUPPORTED, "this store holds integer codes + a constant per column (bwgr_geno_load_f64_centred): only the solvers that "
                                      "centre the columns themselves (MRR3 / MRR3F) can use it");
  CU(cudaSetDevice(h->device));
  Fit& f = h->fit;
  f.reset();
  int family = 0;
  const bool dist = h->world > 1;
  if (dist) {
    if (!h->hx_connected) return fail(BWGR_ERR_STATE, "row-sharded handle: call bwgr_dist_connect before fitting");
    if (s.row_mask) return fail(BWGR_ERR_UNSUPPORTED, "row-sharded fits take unmasked systems");
    if (s.model == M_KMUP || s.model == M_KMUP2) return fail(BWGR_ERR_UNSUPPORTED, "row sharding covers the EM and Gibbs solvers and MRR3's fast path");
  }
  // row-sharded fits and MRR3's rotated systems run on the pipelined blocked sweep only
  int rc = choose_path(h, s, dist || s.model == M_MRR ? BWGR_PATH_BLOCKED : h->path, &family);
  if (rc) return rc;
  const bool blocked = family == 1;
  const int64_t n = h->n, p = h->p, ld = h->ld;
  const int ns = s.nsys;
  f.model = s.model; f.nsys = ns; f.shuffled = s.shuffled; f.blocked = blocked; f.gridfam = family == 2; f.masked = s.row_mask != nullptr; f.weighted = false;
  f.sweeps_issued = 0; f.seed = s.seed; f.chain0 = s.chain0; f.gram_cached = false; f.skip_epilogue = false; f.wgr_mode = false; f.gram_p = nullptr;
  f.overlap = false; f.gram_ahead = -1;
  if (h->side) CU(cudaStreamSynchronize(h->side));  // a band computed ahead for a sweep the previous fit never ran
  f.xx_over.release(); f.wst.release(); f.sx_dev.release(); f.cshift.release(); f.wts.release();
  f.it_target = s.it;

  // ---- per-system row masks and column statistics
  std::vector<float> n_eff(ns, (float)(dist ? h->n_global : n));
  std::vector<std::vector<double>> xx_s, sx_s;  // masked systems only
  if (f.masked) {
    std::vector<uint8_t> m((size_t)ns * ld, 0);
    for (int t = 0; t < ns; t++) {
      int cnt = 0;
      for (int64_t i = 0; i < n; i++) { const uint8_t v = s.row_mask[(size_t)t * n + i] ? 1 : 0; m[(size_t)t * ld + i] = v; cnt += v; }
      if (cnt < 2) return fail(BWGR_ERR_ARG, "row_mask of system %d keeps %d rows", t, cnt);
      n_eff[t] = (float)cnt;
    }
    if (f.mask.alloc(m.size()) != cudaSuccess || f.xx_sys.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    CU(cudaMemcpyAsync(f.mask.p, m.data(), m.size(), cudaMemcpyHostToDevice, h->stream));
    xx_s.resize(ns); sx_s.resize(ns);
    ColStatBufs cs;
    for (int t = 0; t < ns; t++)
      if ((rc = rows_col_stats(h, cs, f.mask.p + (size_t)t * ld, false, t, &xx_s[t], &sx_s[t]))) return rc;
  }

  // ---- initial state per system (SURVEY A.1), float arithmetic
  f.sc0.assign(ns, SysScalars());
  f.vy.assign(ns, 0); f.MSx.assign(ns, 0); f.cxx.assign(ns, 0);
  std::vector<float> hy((size_t)ns * ld, 0.0f), he((size_t)ns * ld, 0.0f);
  std::vector<float> hvb;  // initial per-marker variance
  float vbv_init = 1.0f;
  for (int t = 0; t < ns; t++) {
    std::vector<float> yt;
    yt.reserve(n);
    for (int64_t i = 0; i < n; i++) {
      const double v = y[(size_t)t * n + i];
      if (!(v == v)) return fail(BWGR_ERR_ARG, "y contains NaN (man/em.Rd:38 forbids NA in y)");
      hy[(size_t)t * ld + i] = (float)v;
      if (!f.masked || s.row_mask[(size_t)t * n + i]) yt.push_back((float)v);
    }
    const float nn = n_eff[t];
    const std::vector<double>& xx = f.masked ? xx_s[t] : h->h_xx;
    const std::vector<double>& sx = f.masked ? sx_s[t] : h->h_sx;
    double svx = 0, sxx = 0, tr = 0;
    for (int64_t j = 0; j < p; j++) {
      const double v = (xx[j] - sx[j] * sx[j] / (double)nn) / ((double)nn - 1.0);
      svx += (double)(float)v;
      sxx += xx[j];
    }
    const float sum_vx = (float)svx;
    float vy, mu;
    if (!dist) {
      vy = fvar_f(yt);
      double sm = 0;
      for (float v : yt) sm += v;
      mu = (float)(sm / (double)yt.size());
    } else {  // mean and variance of y over ALL individuals (two small all-reduces)
      double sm = 0;
      for (float v : yt) sm += v;
      rc = dist_allreduce_host(h, &sm, 1, false);
      if (rc) return rc;
      mu = (float)(sm / (double)h->n_global);
      double ss = 0;
      for (float v : yt) { const float tt = v - mu; ss += (double)tt * tt; }
      rc = dist_allreduce_host(h, &ss, 1, false);
      if (rc) return rc;
      vy = (float)ss / (float)(h->n_global - 1);
    }
    SysScalars c;
    memset(&c, 0, sizeof c);
    c.mu = mu; c.df = s.df; c.R2 = s.R2; c.alpha = s.alpha; c.vy = vy; c.n_eff = nn; c.pi_mix = s.pi;
    c.burn = s.bi; c.sweep = 0;
    const float df = s.df, R2 = s.R2;
    float Pi = s.Pi;
    switch (s.model) {
      case M_EMRR: {  // Rcpp20260726ai.cpp:317-324
        const float MSx = sum_vx;
        c.MSx = MSx; c.lmb = MSx; c.Rho = MSx * (1 - R2) / R2; c.ve = 0.5f * vy; c.vb = c.ve / MSx;
        c.Se = (1 - R2) * (df + 2) * vy; c.Sb = R2 * (df + 2) * vy / MSx;
        break;
      }
      case M_EMBA: {  // :84-97
        const float MSx = sum_vx;
        c.MSx = MSx; c.ve = 1; c.Sb = R2 * (df + 2) * vy / MSx; c.Se = (1 - R2) * (df + 2) * vy;
        vbv_init = 1.0f;
        break;
      }
      case M_EMBB: {  // :135-154
        if (Pi > 0.5f) Pi = 1 - Pi;
        const float MSx = sum_vx * Pi;
        c.MSx = MSx; c.ve = 1; c.Sb = R2 * (df + 2) * vy / MSx; c.Se = (1 - R2) * (df + 2) * vy;
        c.Pi = Pi; c.Pi0 = (1 - Pi) / Pi;
        vbv_init = 1.0f;
        break;
      }
      case M_EMBC: {  // :196-213 (ve = Sa, va = Se: sic)
        if (Pi > 0.5f) Pi = 1 - Pi;
        const float MSx = sum_vx * Pi * (1 - Pi);
        c.MSx = MSx; c.Sa = R2 * (df + 2) * vy / MSx; c.Se = (1 - R2) * (df + 2) * vy;
        c.ve = c.Sa; c.vb = c.Se; c.lmb = c.ve / c.vb; c.Pi = Pi; c.Pi0 = (1 - Pi) / Pi;
        break;
      }
      case M_EMBL: {  // :359-370
        const float h2 = R2;
        const float cxx = (float)(sxx / (double)p);
        c.cxx = cxx;
        c.lmb1 = cxx * ((1 - h2) / h2) * s.alpha * 0.5f;
        c.lmb2 = cxx * ((1 - h2) / h2) * (1 - s.alpha);
        break;
      }
      case M_EMEN: {  // :412-419
        const float cxx = sum_vx * (1 - R2) / R2;
        c.cxx = cxx; c.Sy = std::sqrt(vy); c.lmb = cxx;
        c.lmb1 = 0.5f * cxx * s.alpha * c.Sy; c.lmb2 = cxx * (1 - s.alpha);
        for (int64_t j = 0; j < p; j++) tr += 1.0 / ((double)(float)xx[j] + (double)cxx);
        c.trAC22 = (float)tr;
        break;
      }
      case M_EMDE: {  // :262-270 ; the per-marker slot carries Lmb_j
        const float cxx = sum_vx * (1 - R2) / R2;
        c.cxx = cxx;
        vbv_init = (float)p + cxx;
        break;
      }
      case M_EMMLD:
      case M_EMML: {  // :480-486
        c.MSx = sum_vx; c.lmb = sum_vx;
        break;
      }
      case M_GSRR: case M_GSFLM: break;  // warm start: the caller's state is uploaded by bwgr_gs_fit
      case M_EMBCPI: {  // :1508-1520 (emBC's start; the prior Pi is kept for the per-sweep update of Pi)
        if (Pi > 0.5f) Pi = 1 - Pi;
        const float MSx = sum_vx * Pi * (1 - Pi);
        c.MSx = MSx; c.Sa = R2 * (df + 2) * vy / MSx; c.Se = (1 - R2) * (df + 2) * vy;
        c.ve = c.Sa; c.vb = c.Se; c.lmb = c.ve / c.vb; c.Pi = Pi; c.Pi0 = (1 - Pi) / Pi;
        c.cxx = sum_vx; c.pi_mix = Pi;
        break;
      }
      case M_LASSO: {  // :1470-1472
        c.lmb = (float)(sxx / (double)p) / (float)p;
        break;
      }
      case M_BRR: case M_BA: case M_BB: case M_BL: case M_BDPI: {  // :822-827, :598-609, :649-665, :771-783, :931-944
        const float MSx = sum_vx;
        c.MSx = MSx; c.Sb = R2 * df * vy / MSx; c.Se = (1 - R2) * df * vy; c.ve = vy; c.vb = c.Sb; c.lmb = c.ve / c.vb;
        c.Pi0 = s.pi / (1.0f - s.pi);
        c.Rho = MSx * (1 - R2) / R2;  // BayesL's Phi (:773)
        c.Pi = s.pi;                  // BayesDpi: pi = 0.5 at the start (:934), then the mean inclusion
        vbv_init = c.Sb;
        break;
      }
      case M_BCPI:  // :866-880 = BayesC started at pi = 0.5
      case M_BC: {  // :712-726
        const float MSx = sum_vx;
        c.MSx = MSx; c.Sb = df * R2 * vy / MSx / (1 - s.pi); c.Se = df * (1 - R2) * vy; c.ve = vy; c.vb = c.Sb;
        c.lmb = c.ve / c.vb; c.Pi0 = s.pi / (1.0f - s.pi); c.Pi = s.pi;
        break;
      }
      case M_MRR: {  // rotated MRR3 systems: lambda and scales are set per sweep by the driver
        c.MSx = sum_vx; c.ve = 1; c.vb = 1; c.lmb = 1;
        break;
      }
      case M_KMUP2:
      case M_KMUP: {  // state comes from the caller (KMUP :12-38) or from the wgr driver (R/wgr.R:46-59)
        c.MSx = sum_vx; c.ve = 1; c.vb = 1; c.lmb = 1;
        break;
      }
      default: return fail(BWGR_ERR_ARG, "bad model %d", s.model);
    }
    c.C = -0.5f / std::sqrt(c.ve);
    {  // fixed-point scale of the residuals, from max|y - mu|
      float emax = 0;
      for (float v : yt) emax = std::max(emax, std::fabs(v - mu));
      if (dist) {  // the fixed-point scale must be the same on every rank
        double em = emax;
        rc = dist_allreduce_host(h, &em, 1, true);
        if (rc) return rc;
        emax = (float)em;
      }
      set_e_scale(c, emax);
    }
    f.sc0[t] = c;
    f.vy[t] = vy; f.MSx[t] = c.MSx; f.cxx[t] = c.cxx;
    for (int64_t i = 0; i < n; i++)
      if (!f.masked || s.row_mask[(size_t)t * n + i]) he[(size_t)t * ld + i] = hy[(size_t)t * ld + i] - mu;
    if (model_has_vbj(s.model)) hvb.resize((size_t)ns * p), std::fill(hvb.begin() + (size_t)t * p, hvb.begin() + (size_t)(t + 1) * p, vbv_init);
  }

  // ---- device state (buffers a previous fit on this handle left behind must not leak into this one)
  const bool gibbs = model_is_gibbs(s.model);
  if (!model_has_d(s.model)) f.d.release();
  if (!model_has_vbj(s.model)) f.vbv.release();
  if (!model_has_cnv(s.model)) f.b_prev.release();
  if (!gibbs) { f.B.release(); f.D.release(); f.VBv.release(); }
  if (!f.masked) { f.mask.release(); f.xx_sys.release(); }
  if (f.y.alloc((size_t)ns * ld) != cudaSuccess || f.e.alloc((size_t)ns * ld) != cudaSuccess ||
      f.b.alloc((size_t)ns * p) != cudaSuccess || f.sc.alloc(ns) != cudaSuccess || f.perm.alloc((size_t)kPermRing * p) != cudaSuccess)
    return fail(BWGR_ERR_CUDA, "cudaMalloc(fit state) failed");
  if (model_has_d(s.model) && f.d.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  if (model_has_vbj(s.model) && f.vbv.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  if (model_has_cnv(s.model) && f.b_prev.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  if (gibbs) {
    if (f.B.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    CU(cudaMemsetAsync(f.B.p, 0, sizeof(float) * ns * p, h->stream));
    if (f.d.p) { if (f.D.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed"); CU(cudaMemsetAsync(f.D.p, 0, sizeof(float) * ns * p, h->stream)); }
    if (f.vbv.p) { if (f.VBv.alloc((size_t)ns * p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed"); CU(cudaMemsetAsync(f.VBv.p, 0, sizeof(float) * ns * p, h->stream)); }
  }
  CU(cudaMemcpyAsync(f.y.p, hy.data(), sizeof(float) * hy.size(), cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.e.p, he.data(), sizeof(float) * he.size(), cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemsetAsync(f.b.p, 0, sizeof(float) * ns * p, h->stream));
  if (f.d.p) CU(cudaMemsetAsync(f.d.p, 0, sizeof(float) * ns * p, h->stream));
  if (f.vbv.p) CU(cudaMemcpyAsync(f.vbv.p, hvb.data(), sizeof(float) * hvb.size(), cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.sc.p, f.sc0.data(), sizeof(SysScalars) * ns, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));

  f.h_perm_bytes = sizeof(int) * kPermRing * p;
  CU(pinned_alloc(reinterpret_cast<void**>(&f.h_perm), f.h_perm_bytes));
  for (int i = 0; i < kPermRing; i++) CU(cudaEventCreateWithFlags(&f.perm_free[i], cudaEventDisableTiming));
  f.order.resize(p);
  for (int64_t j = 0; j < p; j++) f.order[j] = (int)j;

  if (blocked) {
    f.nblocks = (int)((p + kBlk - 1) / kBlk);
    PipePlan pl;
    if (!plan_pipe(h, s.model, ns, &pl)) return fail(BWGR_ERR_UNSUPPORTED, "the shape does not fit the pipelined blocked sweep");
    if (dist) {
      // the per-rank Gram bands are summed in float by ncclAllReduce: exact (= independent of the sharding) only below 2^24.
      // |G_jk| <= max_j xx_j (Cauchy-Schwarz) over ALL individuals; h_xx holds the all-reduced column statistics.
      if (!(h->xx_max < 16777216.0))
        return fail(BWGR_ERR_UNSUPPORTED, "row-sharded fit: max_j sum_i x_ij^2 = %.0f >= 2^24, the float sum of the per-GPU Gram bands would depend on the sharding", h->xx_max);
      // stale words of a previous fit (another nsys = another ring layout) must not be mistaken for this fit's: zero my ring,
      // then a collective as the barrier that no peer writes into it before it is clean
      CU(cudaMemsetAsync(h->hx_own.p, 0, sizeof(unsigned long long) * h->hx_own.n, h->stream));
      double one = 1;
      rc = dist_allreduce_host(h, &one, 1, false);
      if (rc) return rc;
    }
    f.rows_per_cta = pl.R; f.nworkers = pl.W; f.grid = pl.cl ? pl.nclusters * 8 : pl.W + 1; f.nbuf = pl.nbuf; f.sring = pl.sring; f.lookahead = pl.D; f.full_inv = pl.full_inv; f.nband = pl.D + 1;
    f.cl = pl.cl; f.nclusters = pl.nclusters;
    f.nc = std::max(1, 16 / ns);
    f.tag = 0;
    const size_t gram_n = (size_t)f.nblocks * kBlk * kBlk * f.nband;
    if (!s.shuffled) {  // natural order: one Gram band per genotype store, kept on the handle
      if (h->gram_nat_band != f.nband || h->gram_nat.n != gram_n) {
        h->gram_nat_band = 0;
        if (h->gram_nat.alloc(gram_n) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(Gram band) failed");
      } else {
        f.gram_cached = true;
      }
      f.gram_p = h->gram_nat.p;
    } else {
      if (f.gram.alloc(gram_n) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(Gram band) failed");
      f.gram_p = f.gram.p;
      // the clustered sweep occupies 8 x nclusters of the SMs: the next sweep's Gram band (a function of the marker order only)
      // is computed on the others meanwhile
      f.overlap = (h->world <= 1 || h->comm_side) && h->wait32 && h->x2f.p && f.nband == 2 &&
                  f.grid + 8 <= h->num_sms;  // at least a few SMs are left idle by the sweep
      if (f.overlap && f.gram2.alloc(gram_n) != cudaSuccess) { cudaGetLastError(); f.overlap = false; }
    }
    if (!f.overlap) f.gram2.release();
    f.gram_ahead = -1;
    if (f.full_inv && f.tinv.alloc((size_t)f.nblocks * kBlk * kBlk) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(block inverses) failed");
    if (!f.full_inv) f.tinv.release();
    if (f.part.alloc((size_t)8 * ns * 128 * 161) != cudaSuccess || f.dew.alloc((size_t)f.nblocks * ns * 136) != cudaSuccess)
      return fail(BWGR_ERR_CUDA, "cudaMalloc(blocked workspace) failed");
    // clustered topology: two sets of the grid-sum words of h, used by alternate sweeps; each sweep zeroes the other set
    if (f.cl) {
      if (f.hsum.alloc((size_t)2 * f.nblocks * ns * 128 * kGridCopies) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(grid sums of h) failed");
      CU(cudaMemsetAsync(f.hsum.p, 0, sizeof(unsigned long long) * f.hsum.n, h->stream));
    } else {
      f.hsum.release();
    }
    CU(cudaMemsetAsync(f.dew.p, 0, sizeof(unsigned long long) * f.dew.n, h->stream));
  }
  if (f.gridfam) {
    grid_geometry(h, &f.rows_per_cta, &f.grid);
    // unmasked systems: blocks of markers per grid sum, if the block ring fits next to the residual slabs (else one marker per sum)
    f.grid_blocked = !f.masked && s.model != M_KMUP2 &&
                     grid_block_smem(ns, f.rows_per_cta, h->storage == BWGR_STORE_F32, model_is_gibbs(s.model)) <= h->smem_optin;
    const size_t words = f.grid_blocked ? grid_block_acc_words(ns, (int)p) : (size_t)p * kGridCopies * 32;
    if (f.gridacc.alloc(words) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(grid accumulators) failed");
  }
  f.active = true;
  return 0;
}

// Fixed-point quantum of g = x'e: a power of two such that 64 x the Cauchy-Schwarz bound stays below 2^50.
void g_fixed_point(bwgr_handle* h, const Fit& f, float* quantum, float* limit) {
  const double xxmax = std::max(1.0, h->xx_max);
  double yy = 0;
  for (size_t t = 0; t < f.vy.size(); t++) yy = std::max(yy, (double)f.vy[t] * (double)(h->n - 1));
  const double bound = 64.0 * (f.weighted ? 256.0 : 1.0) * std::sqrt(xxmax * std::max(yy, 1e-30));  // row multiplicities <= 255
  int ex;
  std::frexp(bound, &ex);
  *quantum = (float)std::ldexp(1.0, ex - 50);
  *limit = (float)std::ldexp(1.0, ex);
}

// The fit's state as the sweep kernels and the epilogue take it.  The rule divides by the per-system xx of masked systems, else by
// the caller's (KMUP) or the centred (MRR3) xx when the fit has one, else by the store's; the blocked family never has masked
// systems.  Only the KMUP2 rule reads xx2.
SweepState sweep_state(const bwgr_handle* h) {
  const Fit& f = h->fit;
  SweepState s;
  s.g = h->view(); s.nsys = f.nsys;
  s.e = f.e.p; s.b = f.b.p; s.d = f.d.p; s.vbv = f.vbv.p;
  s.xx = f.masked ? f.xx_sys.p : (f.xx_over.p ? f.xx_over.p : h->xx_f.p); s.xx_per_sys = f.masked ? 1 : 0;
  s.xx2 = f.model == M_KMUP2 ? f.xx_over.p : nullptr;
  s.mask = f.mask.p; s.sc = f.sc.p;
  s.seed_lo = (uint32_t)f.seed; s.seed_hi = (uint32_t)(f.seed >> 32); s.chain0 = f.chain0;
  s.err = h->err.p;
  return s;
}

// Row-sharded fit: the uncentred Gram band of this rank's rows -> the band over all individuals (exact: integers below 2^24 in
// fp32), centred afterwards when the fit's columns are (MRR3), with the same arithmetic as one GPU's Gram kernel.
int sum_gram_band(bwgr_handle* h, float* gram, const int* perm, ncclComm_t comm, cudaStream_t st) {
  const Fit& f = h->fit;
  NC(nccl().AllReduce(gram, gram, (size_t)f.nblocks * kBlk * kBlk * f.nband, ncclFloat, ncclSum, comm, st));
  if (f.sx_dev.p) {
    launch_gram_centre(gram, perm, (int)h->p, f.nblocks, f.nband, f.sx_dev.p, 1.0f / (float)h->n_global, st);
    h->launches++;
  }
  return 0;
}

int fit_sweeps(bwgr_handle* h, int nsweeps) {
  Fit& f = h->fit;
  if (!h || !f.active) return fail(BWGR_ERR_STATE, "no fit in progress");
  CU(cudaSetDevice(h->device));
  const int64_t p = h->p;
  const SweepState state = sweep_state(h);
  float quantum = 1, limit = 1;
  if (f.gridfam) g_fixed_point(h, f, &quantum, &limit);
  for (int k = 0; k < nsweeps; k++) {
    const int sweep = f.sweeps_issued;
    const int slot = sweep % kPermRing;
    const int* d_perm = nullptr;
    // the marker order of sweep `sw` (cumulative shuffles, Rcpp20260726ai.cpp:329-331) goes up on stream `st`
    auto upload_order = [&](int sw, cudaStream_t st) -> cudaError_t {
      const int sl = sw % kPermRing;
      if (f.perm_ev_valid[sl]) { cudaError_t e = cudaEventSynchronize(f.perm_free[sl]); if (e != cudaSuccess) return e; }
      int* hp = f.h_perm + (size_t)sl * p;
      if (f.shuffled) std::shuffle(f.order.begin(), f.order.end(), std::mt19937(sw));
      memcpy(hp, f.order.data(), sizeof(int) * p);
      return cudaMemcpyAsync(f.perm.p + (size_t)sl * p, hp, sizeof(int) * p, cudaMemcpyHostToDevice, st);
    };
    const bool ahead = f.overlap && f.gram_ahead == sweep;  // order and Gram band of this sweep were issued on the side stream
    if (f.overlap) f.gram_p = (sweep & 1) ? f.gram2.p : f.gram.p;
    if (!ahead && (f.shuffled || (f.blocked && f.sweeps_issued == 0)))  // natural order: the identity is uploaded once (slot 0)
      CU(upload_order(sweep, h->stream));
    if (f.shuffled) d_perm = f.perm.p + (size_t)slot * p;
    else if (f.blocked) d_perm = f.perm.p;  // identity order, uploaded once (slot 0)
    if (model_has_cnv(f.model)) CU(cudaMemcpyAsync(f.b_prev.p, f.b.p, sizeof(float) * f.nsys * p, cudaMemcpyDeviceToDevice, h->stream));
    if (f.blocked) {
      if (ahead) {
        CU(cudaStreamWaitEvent(h->stream, h->side_done[sweep & 1], 0));
      } else if (f.shuffled || !f.gram_cached) {
        cudaEvent_t pe = h->prof_begin(0);
        // row shards: each rank's band is uncentred (integers below 2^24 in fp32, so the float all-reduce is exact) and is
        // centred once the sum is complete
        const float* sx_in_kernel = h->world > 1 ? nullptr : f.sx_dev.p;
        if (h->x2f.p && f.nband == 2) {
          const cudaError_t ge = launch_gram_fp4(h->x2f.p, h->ld, (int)h->p, (int)h->n_global, d_perm, f.nblocks, f.gram_p, h->err.p, h->num_sms, sx_in_kernel, h->stream);
          if (ge != cudaSuccess) return fail(BWGR_ERR_CUDA, "FP4 Gram launch failed: %s", cudaGetErrorString(ge));
        } else launch_gram_tc(gram_view(h), d_perm, f.nblocks, f.gram_p, 1, f.nband, h->fp8_codes, h->err.p, h->num_sms, sx_in_kernel, h->stream);
        h->prof_end(pe);
        h->launches++;
        f.gram_cached = true;
        if (!f.shuffled && f.gram_p == h->gram_nat.p) h->gram_nat_band = f.nband;
        if (h->world > 1) {
          int rc = sum_gram_band(h, f.gram_p, d_perm, h->comm, h->stream);
          if (rc) return rc;
        }
      }
      if (f.full_inv) {  // the step coefficients change every sweep (lambda), the inverses with them
        cudaEvent_t pi = h->prof_begin(3);
        launch_block_inverse(f.model, d_perm, (int)p, f.nblocks, f.gram_p, f.nband, state.xx, state.vbv, state.sc, f.tinv.p, h->stream);
        h->prof_end(pi);
        h->launches++;
      }
      if (!f.cl) CU(cudaMemsetAsync(f.part.p, 0, sizeof(unsigned long long) * f.part.n, h->stream));
      PipeArgs a;
      memset(&a, 0, sizeof a);
      a.s = state; a.model = rule_model(f.model); a.perm = d_perm; a.nblocks = f.nblocks; a.gram = f.gram_p; a.nband = f.nband; a.tinv = f.full_inv ? f.tinv.p : nullptr;
      a.sx = f.sx_dev.p; a.cshift = f.cshift.p; a.n_total = (int)h->n_global;
      a.part = f.part.p; a.hred = f.part.p + (size_t)8 * f.nsys * 128 * 160; a.dew = f.dew.p; a.tag = ++f.tag;
      a.rows_per_cta = f.rows_per_cta; a.nworkers = f.nworkers; a.D = f.lookahead; a.nbuf = f.nbuf; a.sring = f.sring;
      a.world = h->world; a.rank = h->rank; a.gen0 = h->dist_gen;
      a.cl = f.cl; a.nclusters = f.nclusters;
      if (f.cl) {
        const size_t set = f.hsum.n / 2;
        a.hsum = f.hsum.p + (sweep & 1) * set; a.hsum_next = f.hsum.p + ((sweep + 1) & 1) * set;
      }
      for (int r = 0; r < 8; r++) a.hx[r] = h->hx[r];
      if (h->world > 1) h->dist_gen += (unsigned long long)f.nblocks;
      if (getenv("BWGR_TRACE")) {
        const size_t tn = (size_t)f.grid * f.nblocks * 32;  // a previous fit on this handle may have had another geometry
        if (f.trace.n != tn) { f.trace.alloc(tn); cudaMemsetAsync(f.trace.p, 0, sizeof(long long) * f.trace.n, h->stream); }
        a.trace = f.trace.p;
      }
      if (f.overlap) { a.started = h->started.p; a.started_val = ++h->started_seq; }
      cudaEvent_t pe = h->prof_begin(1);
      const cudaError_t le = launch_sweep_pipe(a, h->stream);
      h->prof_end(pe);
      if (le != cudaSuccess) return fail(BWGR_ERR_CUDA, "pipelined sweep launch failed: %s", cudaGetErrorString(le));
      h->launches++;
      if (f.overlap) {
        // the flag is also set when the sweep has drained, whatever happened inside it: the side stream never waits forever
        const CUdeviceptr flag = reinterpret_cast<CUdeviceptr>(h->started.p);
        if (h->write32(h->stream, flag, a.started_val, 0) != CUDA_SUCCESS) return fail(BWGR_ERR_CUDA, "cuStreamWriteValue32 failed");
        const bool more = k + 1 < nsweeps || sweep + 1 < f.it_target;
        if (more && !h->profiling) {  // sweep + 1: order + Gram band on the SMs this sweep leaves idle, as soon as it is resident
          if (h->wait32(h->side, flag, a.started_val, CU_STREAM_WAIT_VALUE_GEQ) != CUDA_SUCCESS) return fail(BWGR_ERR_CUDA, "cuStreamWaitValue32 failed");
          CU(upload_order(sweep + 1, h->side));
          const int* np_ = f.perm.p + (size_t)((sweep + 1) % kPermRing) * p;
          float* gn = ((sweep + 1) & 1) ? f.gram2.p : f.gram.p;
          const cudaError_t ge = launch_gram_fp4(h->x2f.p, h->ld, (int)h->p, (int)h->n_global, np_, f.nblocks, gn, h->err.p, h->num_sms,
                                                 h->world > 1 ? nullptr : f.sx_dev.p, h->side, true);
          if (ge != cudaSuccess) return fail(BWGR_ERR_CUDA, "FP4 Gram launch failed: %s", cudaGetErrorString(ge));
          if (h->world > 1) {  // row shards: its own communicator, so it never queues behind (or ahead of) the main stream's
            int rc = sum_gram_band(h, gn, np_, h->comm_side, h->side);
            if (rc) return rc;
          }
          CU(cudaEventRecord(h->side_done[(sweep + 1) & 1], h->side));
          f.gram_ahead = sweep + 1;
          h->launches++;
        }
      }
    } else if (f.gridfam) {
      GridArgs a;
      memset(&a, 0, sizeof a);
      a.s = state; a.model = f.model; a.perm = d_perm;
      a.s.mask = f.weighted ? f.cnt.p : f.mask.p;  // row multiplicities ride in the mask bytes (they weigh the dot products only)
      a.blocked = f.grid_blocked ? 1 : 0;
      {  // cross products are bounded by max_j x_j'x_j (Cauchy-Schwarz): one unit = 1 (exact integers) unless that exceeds 2^50
        int ex = 0;
        std::frexp(std::max(1.0, h->xx_max), &ex);
        a.gram_quantum = h->storage == BWGR_STORE_F32 ? (float)std::ldexp(1.0, ex - 50) : (float)std::ldexp(1.0, std::max(0, ex - 50));
      }
      a.acc = f.gridacc.p; a.g_quantum = quantum; a.rows_per_cta = f.rows_per_cta;
      CU(cudaMemsetAsync(f.gridacc.p, 0, sizeof(unsigned long long) * f.gridacc.n, h->stream));
      cudaEvent_t pe = h->prof_begin(1);
      const cudaError_t le = launch_grid_sweep(a, f.grid, h->stream);
      h->prof_end(pe);
      if (le != cudaSuccess) return fail(BWGR_ERR_CUDA, "grid sweep launch failed: %s", cudaGetErrorString(le));
      h->launches++;
    } else {
      SmallNArgs a;
      memset(&a, 0, sizeof a);
      a.s = state; a.model = rule_model(f.model); a.perms = d_perm; a.row_w = f.weighted ? f.row_w.p : nullptr;
      cudaEvent_t pe = h->prof_begin(1);
      const cudaError_t le = launch_small_n(a, h->smem_optin, h->stream);
      h->prof_end(pe);
      if (le != cudaSuccess) return fail(BWGR_ERR_CUDA, "small-n sweep launch failed: %s", cudaGetErrorString(le));
      h->launches++;
    }
    if (f.shuffled) { CU(cudaEventRecord(f.perm_free[slot], h->stream)); f.perm_ev_valid[slot] = true; }
    if (f.wgr_mode) {
      cudaEvent_t pe2 = h->prof_begin(2);
      launch_wgr_step(f.wgr_args, h->num_sms, h->stream);
      h->prof_end(pe2);
      h->launches += 2;
    } else if (!f.skip_epilogue) {
      EpilogueArgs ea;
      memset(&ea, 0, sizeof ea);
      if (h->world > 1) {
        if (f.esum.n < (size_t)4 * f.nsys && (f.esum.alloc((size_t)4 * f.nsys) != cudaSuccess || f.emaxv.alloc(f.nsys) != cudaSuccess))
          return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
      }
      ea.s = state; ea.model = f.model; ea.y = f.y.p; ea.b_prev = f.b_prev.p; ea.wts = f.wts.p;
      ea.B = f.B.p; ea.D = f.D.p; ea.VBv = f.VBv.p;
      cudaEvent_t pe2 = h->prof_begin(2);
      if (h->world > 1) {  // sums over individuals: per rank, then all-reduced; everything else is replicated
        launch_epilogue_partial(ea, f.esum.p, f.emaxv.p, h->stream);
        NC(nccl().AllReduce(f.esum.p, f.esum.p, (size_t)4 * f.nsys, ncclDouble, ncclSum, h->comm, h->stream));
        NC(nccl().AllReduce(f.emaxv.p, f.emaxv.p, (size_t)f.nsys, ncclFloat, ncclMax, h->comm, h->stream));
        ea.esum = f.esum.p; ea.emaxv = f.emaxv.p;
        h->launches++;
      }
      launch_epilogue(ea, h->stream);
      h->prof_end(pe2);
      h->launches++;
    }
    f.sweeps_issued++;
    cudaError_t le = cudaGetLastError();
    if (le != cudaSuccess) return fail(BWGR_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(le));
  }
  return 0;
}

constexpr int kHatSplits = 64;           // column splits of the fitted values (they fix each row's summation order)
constexpr size_t kHatWorkBytes = 512u << 20;  // bound of the partial sums [k][splits][ld] of one launch of the fitted values

// hat[t] = mu[t] + X b_t for the k systems of b [k][p] into hat [k][ld] (device buffers): one launch per group of systems whose partial
// sums fit kHatWorkBytes (all k at once up to n ~ 10^5 for k = 16)
int fit_hat(bwgr_handle* h, int k, const float* b_dev, const float* mu_dev, float* hat_dev) {
  Fit& f = h->fit;
  const size_t per_sys = (size_t)kHatSplits * h->ld;
  int per = (int)std::max<size_t>(1, std::min<size_t>((size_t)k, kHatWorkBytes / (per_sys * sizeof(float))));
  if (per < k && per >= kHatChunk) per -= per % kHatChunk;
  if (f.work.n < (size_t)per * per_sys && f.work.alloc((size_t)per * per_sys) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  for (int t0 = 0; t0 < k; t0 += per) {
    const int kc = std::min(per, k - t0);
    launch_gemv_hat(h->view(), b_dev + (size_t)t0 * h->p, kc, mu_dev + t0, hat_dev + (size_t)t0 * h->ld, f.work.p, kHatSplits, h->stream);
    h->launches += 2;
  }
  return 0;
}

// Fitted values of nsys systems read back to the host: hat[t * n + i] = mu[t] + x_i'b_t.  b: nsys x p floats, on the device or, with
// b_on_host, on the host.
int fitted_values(bwgr_handle* h, int nsys, const float* b, bool b_on_host, const float* mu, std::vector<float>& hat) {
  const int64_t n = h->n, p = h->p, ld = h->ld;
  DevBuf<float> bdev, mudev, hatd;
  if ((b_on_host && bdev.alloc((size_t)nsys * p) != cudaSuccess) || mudev.alloc(nsys) != cudaSuccess || hatd.alloc((size_t)nsys * ld) != cudaSuccess)
    return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  if (b_on_host) CU(cudaMemcpyAsync(bdev.p, b, sizeof(float) * nsys * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(mudev.p, mu, sizeof(float) * nsys, cudaMemcpyHostToDevice, h->stream));
  const int rc = fit_hat(h, nsys, b_on_host ? bdev.p : b, mudev.p, hatd.p);
  if (rc) return rc;
  hat.resize((size_t)nsys * n);
  CU(cudaMemcpy2DAsync(hat.data(), sizeof(float) * n, hatd.p, sizeof(float) * ld, sizeof(float) * n, nsys, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

}  // namespace

extern "C" {

static int em_spec(const bwgr_em_params* par, FitSpec* s) {
  if (!par) return fail(BWGR_ERR_ARG, "params NULL");
  if (par->model < 0 || par->model > BWGR_EM_LASSO) return fail(BWGR_ERR_ARG, "bad EM model %d", par->model);
  s->model = par->model; s->nsys = par->nsys; s->row_mask = par->row_mask;
  s->shuffled = !(par->model == BWGR_EM_BCPI || par->model == BWGR_EM_LASSO);  // these two walk the markers in order (:1523, :1477)
  s->df = (float)par->df; s->R2 = (float)par->R2; s->Pi = (float)par->Pi; s->alpha = (float)par->alpha; s->pi = 0;
  s->it = par->it < 0 ? (model_has_cnv(par->model) ? 300 : 200) : par->it;  // maxit of the solvers with a stopping rule, else 200 sweeps
  s->bi = 0; s->seed = 0;
  return 0;
}

int bwgr_em_begin(bwgr_handle* h, const bwgr_em_params* par, const double* y) {
  FitSpec s;
  int rc = em_spec(par, &s);
  if (rc) return rc;
  if (par->weights) {  // emML(y, gen, D): the weighted penalty Lmb / d_j (:495-496) travels in the per-marker slot
    if (par->model != BWGR_EM_ML) return fail(BWGR_ERR_ARG, "marker weights belong to emML");
    if (par->nsys != 1 || par->row_mask) return fail(BWGR_ERR_UNSUPPORTED, "emML with marker weights: one unmasked system");
    s.model = M_EMMLD;
  }
  rc = fit_begin(h, s, y);
  if (rc || !par->weights) return rc;
  Fit& f = h->fit;
  const int64_t p = h->p;
  std::vector<float> w(p), l0(p);
  for (int64_t j = 0; j < p; j++) {
    w[j] = (float)par->weights[j];
    if (!(w[j] > 0.0f)) { f.reset(); return fail(BWGR_ERR_ARG, "marker weights must be positive"); }
    l0[j] = f.sc0[0].lmb / w[j];
  }
  if (f.wts.alloc(p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  CU(cudaMemcpyAsync(f.wts.p, w.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.vbv.p, l0.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int bwgr_em_sweeps(bwgr_handle* h, int nsweeps) {
  if (!h) return fail(BWGR_ERR_ARG, "null handle");
  return fit_sweeps(h, nsweeps);
}

// debug (BWGR_TRACE=file): header {CTAs, blocks, 32, look-ahead D}, then the raw int64 stamps of the last sweep, [cta][block][32]
static void dump_trace(bwgr_handle* h) {
  Fit& f = h->fit;
  if (!f.trace.p || !getenv("BWGR_TRACE")) return;
  cudaStreamSynchronize(h->stream);
  std::vector<long long> tr(f.trace.n);
  cudaMemcpy(tr.data(), f.trace.p, tr.size() * sizeof(long long), cudaMemcpyDeviceToHost);
  if (FILE* fp = fopen(getenv("BWGR_TRACE"), "wb")) {
    const long long hdr[4] = {f.grid, f.nblocks, 32, f.lookahead};
    fwrite(hdr, sizeof(long long), 4, fp);
    fwrite(tr.data(), sizeof(long long), tr.size(), fp);
    fclose(fp);
  }
}

int bwgr_em_end(bwgr_handle* h, bwgr_em_out* out) {
  if (!h || !h->fit.active) return fail(BWGR_ERR_STATE, "no fit in progress");
  if (!out) return fail(BWGR_ERR_ARG, "out NULL");
  FitGuard guard{h};
  Fit& f = h->fit;
  const int64_t n = h->n, p = h->p, ld = h->ld;
  const int ns = f.nsys;
  int rc = check_err_flag(h, "sweep");
  if (rc) return rc;
  dump_trace(h);
  std::vector<SysScalars> sc(ns);
  CU(cudaMemcpyAsync(sc.data(), f.sc.p, sizeof(SysScalars) * ns, cudaMemcpyDeviceToHost, h->stream));
  std::vector<float> hb((size_t)ns * p), hd, hv, hh, he;
  std::vector<uint8_t> hmask;  // row masks of masked systems (emBL's var(e))
  CU(cudaMemcpyAsync(hb.data(), f.b.p, sizeof(float) * hb.size(), cudaMemcpyDeviceToHost, h->stream));
  if (f.d.p && out->d) { hd.resize((size_t)ns * p); CU(cudaMemcpyAsync(hd.data(), f.d.p, sizeof(float) * hd.size(), cudaMemcpyDeviceToHost, h->stream)); }
  if (f.vbv.p && (out->vb || f.model == M_EMDE)) { hv.resize((size_t)ns * p); CU(cudaMemcpyAsync(hv.data(), f.vbv.p, sizeof(float) * hv.size(), cudaMemcpyDeviceToHost, h->stream)); }
  if (f.model == M_EMBL) { he.resize((size_t)ns * ld); CU(cudaMemcpyAsync(he.data(), f.e.p, sizeof(float) * he.size(), cudaMemcpyDeviceToHost, h->stream)); }
  CU(cudaStreamSynchronize(h->stream));
  std::vector<float> mu(ns);
  for (int t = 0; t < ns; t++) mu[t] = sc[t].mu;
  if ((rc = fitted_values(h, ns, f.b.p, false, mu.data(), hh))) return rc;
  for (int t = 0; t < ns; t++) {
    const SysScalars& c = sc[t];
    if (out->mu) out->mu[t] = c.mu;
    if (out->its) out->its[t] = c.its;
    double Va = 0, Ve = c.ve, h2 = 0, Vg = 0, pi_out = 0, lmb_out = 0;
    switch (f.model) {
      case M_EMRR: Va = c.vb; h2 = 1.0f - c.ve / f.vy[t]; break;
      case M_EMBA: case M_EMBB: h2 = 1.0f - c.ve / f.vy[t]; break;
      case M_EMBC: Va = c.vb; Vg = c.vb * f.MSx[t]; h2 = 1.0f - c.ve / f.vy[t]; break;
      case M_EMBL: {
        // var(e) over the rows the system uses (:391): a masked system's held-out rows never enter e (they stay 0)
        std::vector<float> ev;
        if (f.masked && hmask.empty()) {
          hmask.resize((size_t)ns * ld);
          CU(cudaMemcpy(hmask.data(), f.mask.p, hmask.size(), cudaMemcpyDeviceToHost));
        }
        for (int64_t i = 0; i < n; i++)
          if (!f.masked || hmask[(size_t)t * ld + i]) ev.push_back(he[(size_t)t * ld + i]);
        if (h->world > 1) {  // var(e) over all individuals (:391)
          double sums[2] = {0, 0};
          for (float v : ev) sums[0] += v;
          rc = dist_allreduce_host(h, sums, 1, false);
          if (rc) return rc;
          const float me = (float)(sums[0] / (double)h->n_global);
          for (float v : ev) { const float tt = v - me; sums[1] += (double)tt * tt; }
          rc = dist_allreduce_host(h, sums + 1, 1, false);
          if (rc) return rc;
          h2 = 1.0f - ((float)sums[1] / (float)(h->n_global - 1)) / f.vy[t];
        } else {
          h2 = 1.0f - fvar_f(ev) / f.vy[t];
        }
        Ve = 0; break;
      }
      case M_EMEN: { const float va = c.vb * f.cxx[t]; Va = va; h2 = va / (va + c.ve); break; }
      case M_EMDE: {  // Vb_j of the last sweep from the penalty it produced: Lmb_j = sqrt(cxx Ve / Vb_j) (:293-296, :305)
        float sv = 0;
        if (!hv.empty() || out->vb) {
          for (int64_t j = 0; j < p; j++) {
            const float L = hv.empty() ? 0.0f : hv[(size_t)t * p + j];
            const float vbj = (c.its > 0 && L > 0) ? c.cxx * c.ve / (L * L) : 0.0f;
            if (!hv.empty()) hv[(size_t)t * p + j] = vbj;
            sv += vbj;
          }
        }
        h2 = sv / (sv + c.ve);
        break;
      }
      case M_EMMLD:
      case M_EMML: Vg = c.vb; Va = c.vb * c.MSx; h2 = Va / (Va + c.ve); break;                  // :508-515 (Vg slot = Vb)
      case M_EMBCPI: Va = c.vb; Vg = c.vb * c.MSx; h2 = 1.0f - c.ve / f.vy[t]; pi_out = c.Pi; break;  // :1539-1545
      case M_LASSO: h2 = 1.0f - c.ve / f.vy[t]; Ve = 0; lmb_out = c.lmb; break;                       // :1494-1497
      default: break;
    }
    if (out->scal) {
      double* sc_out = out->scal + (size_t)BWGR_NSCAL * t;
      sc_out[0] = Va; sc_out[1] = Ve; sc_out[2] = h2; sc_out[3] = Vg; sc_out[4] = pi_out; sc_out[5] = lmb_out;
    }
  }
  if (out->b) for (size_t i = 0; i < hb.size(); i++) out->b[i] = hb[i];
  if (out->d && !hd.empty()) for (size_t i = 0; i < hd.size(); i++) out->d[i] = hd[i];
  if (out->vb && !hv.empty()) for (size_t i = 0; i < hv.size(); i++) out->vb[i] = hv[i];
  if (out->hat) for (size_t i = 0; i < hh.size(); i++) out->hat[i] = hh[i];
  return 0;
}

int bwgr_em_fit(bwgr_handle* h, const bwgr_em_params* par, const double* y, bwgr_em_out* out) {
  FitGuard guard{h};
  int rc = bwgr_em_begin(h, par, y);
  if (rc) return rc;
  Fit& f = h->fit;
  if (model_has_cnv(f.model)) {
    // convergence is checked on the device each sweep; poll in batches to keep the host off the path
    int done_all = 0;
    std::vector<SysScalars> sc(f.nsys);
    while (f.sweeps_issued < f.it_target && !done_all) {
      rc = fit_sweeps(h, std::min(4, f.it_target - f.sweeps_issued));
      if (rc) return rc;
      CU(cudaMemcpyAsync(sc.data(), f.sc.p, sizeof(SysScalars) * f.nsys, cudaMemcpyDeviceToHost, h->stream));
      CU(cudaStreamSynchronize(h->stream));
      done_all = 1;
      for (auto& c : sc) done_all &= c.done;
    }
  } else {
    rc = fit_sweeps(h, f.it_target);
    if (rc) return rc;
  }
  return bwgr_em_end(h, out);
}


// ---- GSRR / GSFLM: warm-start Gauss-Seidel (Rcpp20260726ai.cpp:1564-1628) ---------------------------------------------
int bwgr_gs_fit(bwgr_handle* h, int which, const double* y, double* e, double* b, double* Lmb, const double* xx, double cxx, int maxit,
                double* vb, double* scal) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!y || !e || !b || !Lmb || !xx) return fail(BWGR_ERR_ARG, "null argument");
  if (which < 0 || which > 1 || maxit < 1) return fail(BWGR_ERR_ARG, "bad which / maxit");
  const int64_t n = h->n, p = h->p, ld = h->ld;
  FitSpec s;
  s.model = which == 0 ? M_GSRR : M_GSFLM; s.nsys = 1; s.shuffled = false; s.row_mask = nullptr;  // natural marker order (:1581)
  s.df = 10; s.R2 = 0.5f; s.Pi = 0; s.alpha = 0; s.pi = 0; s.it = maxit; s.bi = 0; s.seed = 0;
  // fit_begin on the residual as passed in: mu = mean(e), e <- e - mu (:1574), and the y slot keeps e0 for vna = e.e0/n (:1587)
  FitGuard guard{h};
  int rc = fit_begin(h, s, e);
  if (rc) return rc;
  Fit& f = h->fit;
  std::vector<float> yv(n), hb(p), hl(p), hx(p);
  for (int64_t i = 0; i < n; i++) { if (!(y[i] == y[i])) return fail(BWGR_ERR_ARG, "y contains NaN"); yv[i] = (float)y[i]; }
  for (int64_t j = 0; j < p; j++) { hb[j] = (float)b[j]; hl[j] = (float)Lmb[j] + 0.01f; hx[j] = (float)xx[j]; }
  SysScalars c = f.sc0[0];
  c.vy = fvar_f(yv);      // float vy = fvar(y) (:1571)
  c.cxx = (float)cxx;     // phi
  f.sc0[0] = c; f.vy[0] = c.vy;
  if (f.xx_over.alloc(p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  CU(cudaMemcpyAsync(f.b.p, hb.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.vbv.p, hl.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.xx_over.p, hx.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.sc.p, &c, sizeof(SysScalars), cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  SysScalars sc;
  int done = 0;
  while (f.sweeps_issued < maxit && !done) {
    rc = fit_sweeps(h, std::min(4, maxit - f.sweeps_issued));
    if (rc) return rc;
    CU(cudaMemcpyAsync(&sc, f.sc.p, sizeof(SysScalars), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    done = sc.done;
  }
  rc = check_err_flag(h, "sweep");
  if (rc) return rc;
  std::vector<float> he(ld);
  CU(cudaMemcpyAsync(he.data(), f.e.p, sizeof(float) * ld, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(hb.data(), f.b.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(hl.data(), f.vbv.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  for (int64_t i = 0; i < n; i++) e[i] = he[i];
  for (int64_t j = 0; j < p; j++) {
    b[j] = hb[j];
    const float L = hl[j] - 0.01f;
    Lmb[j] = L;
    if (vb) vb[j] = which == 0 ? sc.vb : sc.cxx * sc.ve / (L * L);  // GSFLM: Lmb_j = sqrt(phi vna / Vb_j) (:1589)
  }
  if (scal) { scal[0] = sc.mu; scal[1] = 1.0f - sc.ve / c.vy; scal[2] = sc.ve; scal[3] = sc.its; }
  return 0;
}

// ---- Gibbs -------------------------------------------------------------------------------------------
// nsys phenotype columns x nchains chains = S systems; system s = t * nchains + c fits column t (on the rows of its mask) and draws
// from Philox chain chain0 + s.  bwgr_gibbs_fit is the case nsys = 1, no mask, chain0 = 0.
int bwgr_gibbs_fit_sys(bwgr_handle* h, const bwgr_gibbs_sys_params* sp, const double* Y, bwgr_gibbs_out* out) {
  if (!h || !sp || !out || !Y) return fail(BWGR_ERR_ARG, "null argument");
  if (!h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  const bwgr_gibbs_params* par = &sp->base;
  if (par->model < 0 || par->model > BWGR_GIBBS_DPI) return fail(BWGR_ERR_ARG, "bad Gibbs model %d", par->model);
  static const int kGibbsModel[] = {M_BRR, M_BA, M_BB, M_BC, M_BL, M_BCPI, M_BDPI};
  const bool has_pi = par->model == BWGR_GIBBS_CPI || par->model == BWGR_GIBBS_DPI;  // these two start at pi = 0.5 (:870, :934), not an argument
  if (par->it < 1 || par->bi < 0 || par->bi >= par->it) return fail(BWGR_ERR_ARG, "need 0 <= bi < it");
  if (sp->nsys < 1) return fail(BWGR_ERR_ARG, "bad nsys %d", sp->nsys);
  if (sp->chain0 < 0) return fail(BWGR_ERR_ARG, "bad chain0 %d", sp->chain0);
  const int nc = par->nchains < 1 ? 1 : par->nchains;
  if ((int64_t)sp->nsys * nc > 4096) return fail(BWGR_ERR_ARG, "nsys x nchains = %lld systems (at most 4096)", (long long)sp->nsys * nc);
  const int ns = sp->nsys * nc;
  const int64_t n = h->n, p = h->p;
  std::vector<double> yy((size_t)ns * n);
  std::vector<uint8_t> mm(sp->row_mask ? (size_t)ns * n : 0);
  for (int s = 0; s < ns; s++) {
    const size_t t = (size_t)(s / nc);
    memcpy(yy.data() + (size_t)s * n, Y + t * n, sizeof(double) * n);
    if (sp->row_mask) memcpy(mm.data() + (size_t)s * n, sp->row_mask + t * n, (size_t)n);
  }
  FitSpec s;
  s.model = kGibbsModel[par->model]; s.nsys = ns; s.shuffled = false; s.row_mask = sp->row_mask ? mm.data() : nullptr;
  s.df = (float)par->df; s.R2 = (float)par->R2; s.Pi = 0; s.alpha = 0; s.pi = has_pi ? 0.5f : (float)par->pi;
  s.it = par->it; s.bi = par->bi; s.seed = par->seed; s.chain0 = sp->chain0;
  FitGuard guard{h};
  int rc = fit_begin(h, s, yy.data());
  if (rc) return rc;
  Fit& f = h->fit;
  rc = fit_sweeps(h, par->it);
  if (rc) return rc;
  rc = check_err_flag(h, "gibbs sweep");
  if (rc) return rc;
  dump_trace(h);
  std::vector<SysScalars> sc(ns);
  CU(cudaMemcpyAsync(sc.data(), f.sc.p, sizeof(SysScalars) * ns, cudaMemcpyDeviceToHost, h->stream));
  std::vector<float> B((size_t)ns * p), D, V;
  CU(cudaMemcpyAsync(B.data(), f.B.p, sizeof(float) * B.size(), cudaMemcpyDeviceToHost, h->stream));
  if (f.D.p) { D.resize((size_t)ns * p); CU(cudaMemcpyAsync(D.data(), f.D.p, sizeof(float) * D.size(), cudaMemcpyDeviceToHost, h->stream)); }
  if (f.VBv.p) { V.resize((size_t)ns * p); CU(cudaMemcpyAsync(V.data(), f.VBv.p, sizeof(float) * V.size(), cudaMemcpyDeviceToHost, h->stream)); }
  CU(cudaStreamSynchronize(h->stream));
  const float MCMC = (float)par->it - (float)par->bi;  // sic (:626): divisor it-bi although i>bi keeps it-bi-1 draws
  std::vector<float> Bm(B.size()), MU(ns), hh;
  for (size_t i = 0; i < B.size(); i++) Bm[i] = B[i] / MCMC;
  for (int c = 0; c < ns; c++) MU[c] = (float)(sc[c].MU / MCMC);
  if ((rc = fitted_values(h, ns, Bm.data(), true, MU.data(), hh))) return rc;  // every row, the ones a mask leaves out included
  for (int c = 0; c < ns; c++) {
    const float VE = (float)(sc[c].VE / MCMC), VBs = (float)(sc[c].VB / MCMC);
    float vg;
    if (f.VBv.p) { double sv = 0; for (int64_t j = 0; j < p; j++) sv += V[(size_t)c * p + j] / MCMC; vg = (float)sv; }
    else vg = VBs * f.MSx[c];
    const float pi_out = has_pi ? 1.0f - (float)(sc[c].PI / MCMC) : 0.0f;  // :911, :975
    if (f.model == M_BCPI) vg = VBs * f.MSx[c] / pi_out;                   // :913
    if (out->mu) out->mu[c] = MU[c];
    if (out->scal) {
      double* sc_out = out->scal + (size_t)BWGR_NSCAL * c;
      sc_out[0] = VBs; sc_out[1] = VE; sc_out[2] = vg / (vg + VE); sc_out[3] = f.MSx[c]; sc_out[4] = pi_out; sc_out[5] = 0;
    }
    if (out->vb) {
      if (f.VBv.p) for (int64_t j = 0; j < p; j++) out->vb[(size_t)c * p + j] = V[(size_t)c * p + j] / MCMC;
      else out->vb[c] = VBs;
    }
  }
  if (out->b) for (size_t i = 0; i < Bm.size(); i++) out->b[i] = Bm[i];
  if (out->d && !D.empty()) for (size_t i = 0; i < D.size(); i++) out->d[i] = D[i] / MCMC;
  if (out->hat) for (size_t i = 0; i < hh.size(); i++) out->hat[i] = hh[i];
  return 0;
}

int bwgr_gibbs_fit(bwgr_handle* h, const bwgr_gibbs_params* par, const double* y, bwgr_gibbs_out* out) {
  if (!par) return fail(BWGR_ERR_ARG, "null argument");
  bwgr_gibbs_sys_params sp;
  sp.base = *par; sp.nsys = 1; sp.row_mask = nullptr; sp.chain0 = 0;
  return bwgr_gibbs_fit_sys(h, &sp, y, out);
}

// Common start of KMUP / wgr: a one-system M_KMUP fit whose state (b, d, e, per-marker L, Ve, pi) is set by the caller.
// Row multiplicities of a sweep over rows drawn with replacement (Use with repeats, :41-77): cnt [n] on the host -> the uint8 and
// float copies on the device, and xx_sys = H'H over the rows in use with their multiplicities (the scale of the rule's
// likelihood ratio).  The 0/1 mask (cnt != 0) is the caller's.
static int set_row_multiplicities(bwgr_handle* h, const uint8_t* cnt) {
  Fit& f = h->fit;
  const int64_t n = h->n, ld = h->ld;
  std::vector<uint8_t> c8((size_t)ld, 0);
  std::vector<float> cf((size_t)ld, 0.0f);
  for (int64_t i = 0; i < n; i++) { c8[i] = cnt[i]; cf[i] = (float)cnt[i]; }
  if (f.cnt.alloc(ld) != cudaSuccess || f.row_w.alloc(ld) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  CU(cudaMemcpyAsync(f.cnt.p, c8.data(), (size_t)ld, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.row_w.p, cf.data(), sizeof(float) * ld, cudaMemcpyHostToDevice, h->stream));
  ColStatBufs cs;
  const int rc = rows_col_stats(h, cs, f.cnt.p, true, 0, nullptr, nullptr);
  if (rc) return rc;
  CU(cudaStreamSynchronize(h->stream));  // c8 / cf / the scratch go out of scope
  f.weighted = true;
  return 0;
}

static int kmup_begin(bwgr_handle* h, const double* b, const double* d, const double* xx, const double* e, const double* L,
                      double Ve, double pi, uint64_t seed, const uint8_t* row_mask = nullptr, double xx_scale = 1.0,
                      const uint8_t* row_cnt = nullptr) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!b || !e || !L) return fail(BWGR_ERR_ARG, "null argument");
  if (!(Ve > 0)) return fail(BWGR_ERR_ARG, "Ve must be positive");
  const int64_t n = h->n, p = h->p, ld = h->ld;
  FitSpec s;
  // row_mask = the bagged sweep KMUP2 (:41-77): the rows in use as a mask on the small-n family, xx_scale = bg = n0 / n (:47)
  s.model = row_mask ? M_KMUP2 : M_KMUP; s.nsys = 1; s.shuffled = false; s.row_mask = row_mask; s.row_cnt = row_mask ? row_cnt : nullptr;
  s.df = 5; s.R2 = 0.5f; s.Pi = 0; s.alpha = 0; s.pi = (float)pi; s.it = 1; s.bi = 0; s.seed = seed;
  if (row_mask && !xx) return fail(BWGR_ERR_ARG, "KMUP2 needs xx");
  int rc = fit_begin(h, s, e);  // y := e (only its mean/variance feed unused defaults)
  if (rc) return rc;
  Fit& f = h->fit;
  std::vector<float> he(ld, 0.0f), hb(p), hd(p, 1.0f), hl(p);
  float emax = 0;
  for (int64_t i = 0; i < n; i++) { he[i] = (float)e[i]; emax = std::max(emax, std::fabs(he[i])); }
  for (int64_t j = 0; j < p; j++) { hb[j] = (float)b[j]; hl[j] = (float)L[j]; if (d) hd[j] = (float)d[j]; }
  SysScalars c = f.sc0[0];
  c.mu = 0; c.ve = (float)Ve; c.pi_mix = (float)pi; c.C = -0.5f / std::sqrt((float)Ve);  // C = -0.5/sqrt(Ve) (:17, sic)
  c.sweep = 0; c.burn = 0;
  set_e_scale(c, emax);
  f.sc0[0] = c;
  f.skip_epilogue = true;  // the state is advanced by the caller's sweeps alone (KMUP) or by the wgr driver's steps
  CU(cudaMemcpyAsync(f.e.p, he.data(), sizeof(float) * ld, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.b.p, hb.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.d.p, hd.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.vbv.p, hl.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.sc.p, &c, sizeof(SysScalars), cudaMemcpyHostToDevice, h->stream));
  if (xx) {
    std::vector<float> hx(p);
    for (int64_t j = 0; j < p; j++) hx[j] = (float)xx[j] * (float)xx_scale;
    if (f.xx_over.alloc(p) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    CU(cudaMemcpyAsync(f.xx_over.p, hx.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  }
  if (s.row_cnt) {  // repeated rows: multiplicities for the dot products, and H'H with a row counted as often as it was drawn
    rc = set_row_multiplicities(h, s.row_cnt);
    if (rc) return rc;
  }
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

// One sweep of the KMUP / KMUP2 fit kmup_begin set up, and its read-out: b, d and the residuals, e_out[q] = e[rows[q]] (KMUP2: the
// rows of Use, in that order) or, with rows null, all n rows.
static int kmup_sweep_out(bwgr_handle* h, const char* where, double* b, double* d, double* e_out, const double* rows, int64_t nrows) {
  Fit& f = h->fit;
  int rc = fit_sweeps(h, 1);
  if (rc) return rc;
  rc = check_err_flag(h, where);
  if (rc) return rc;
  const int64_t n = h->n, p = h->p;
  std::vector<float> he(n), hb(p), hd(p);
  CU(cudaMemcpyAsync(he.data(), f.e.p, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(hb.data(), f.b.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(hd.data(), f.d.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (rows) for (int64_t q = 0; q < nrows; q++) e_out[q] = he[(int64_t)rows[q]];
  else for (int64_t i = 0; i < n; i++) e_out[i] = he[i];
  for (int64_t j = 0; j < p; j++) { b[j] = hb[j]; if (d) d[j] = hd[j]; }
  return 0;
}

// KMUP(X,b,d,xx,e,L,Ve,pi) (:12-38): one sweep, state updated in place.  X = the handle's store.
int bwgr_kmup_sweep(bwgr_handle* h, double* b, double* d, const double* xx, double* e, const double* L, double Ve, double pi,
                    uint64_t seed) {
  FitGuard guard{h};
  const int rc = kmup_begin(h, b, d, xx, e, L, Ve, pi, seed);
  if (rc) return rc;
  return kmup_sweep_out(h, "kmup sweep", b, d, e, nullptr, 0);
}

// Fitted values of the handle's store: hat = mu + X b.  What the reference's drivers form as X * b (emML2's u1 = X1 * b1,
// Rcpp20260726ai.cpp:1275-1276; the fit of the two-design samplers :1063, :1151, :1212; wgr's gen0 %*% B, R/wgr.R:147).
int bwgr_fitted_sys(bwgr_handle* h, int k, const double* B, const double* mu, double* hat) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!B || !mu || !hat) return fail(BWGR_ERR_ARG, "null argument");
  if (k < 1) return fail(BWGR_ERR_ARG, "bad k %d", k);
  if (h->world > 1) return fail(BWGR_ERR_UNSUPPORTED, "bwgr_fitted on a row-sharded store");
  if (h->col_offset.size()) return fail(BWGR_ERR_UNSUPPORTED, "this store holds integer codes + a constant per column: use the solvers that centre the columns themselves");
  CU(cudaSetDevice(h->device));
  const int64_t n = h->n, p = h->p;
  std::vector<float> bf((size_t)k * p), m0(k), hh;
  for (size_t j = 0; j < bf.size(); j++) bf[j] = (float)B[j];
  for (int t = 0; t < k; t++) m0[t] = (float)mu[t];
  const int rc = fitted_values(h, k, bf.data(), true, m0.data(), hh);
  if (rc) return rc;
  for (size_t i = 0; i < (size_t)k * n; i++) hat[i] = hh[i];
  return 0;
}

int bwgr_fitted(bwgr_handle* h, const double* b, double mu, double* hat) { return bwgr_fitted_sys(h, 1, b, &mu, hat); }

// wgr(y, X, it, bi, th, bag, rp, iv, de, pi, df, R2, eigK = NULL) (R/wgr.R:2-169) with the MCMC loop on the device.
// bag = 1: `it` KMUP sweeps, each followed by the driver's step on the device (wgr_mode).
// bag != 1 (:21, :49, :68, :87, :121): every iteration sweeps a fresh sorted sample of floor(n * bag) rows with KMUP2, estimates Ve
// from their residuals, and rebuilds e = y - mu - X b over all rows.  The row samples come from std::mt19937_64(seed), not from R's
// sample().
static int wgr_fit(bwgr_handle* h, const double* y, int it, int bi, int th, double bag, int rp, int iv, int de, double pi, double df,
                   double R2, uint64_t seed, double* b, double* d, double* Vb, double* hat, double* scal) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!y) return fail(BWGR_ERR_ARG, "y is NULL");
  if (it < 1 || bi < 1 || bi > it || th < 1) return fail(BWGR_ERR_ARG, "need 1 <= bi <= it and th >= 1");
  const bool bagged = bag != 1.0;
  const int64_t n = h->n, p = h->p, ld = h->ld;
  const int64_t nuse = (int64_t)((double)n * bag);
  if (bagged && (!(bag > 0) || nuse < 2 || (!rp && nuse > n))) return fail(BWGR_ERR_ARG, "bag must give 2 <= n * bag (<= n rows without replacement)");
  if (de) iv = 1;  // R/wgr.R:10
  if (bagged) df = df / (bag * bag);  // :21
  // initial state (R/wgr.R:46-59): b = 0, d = 1, mu = mean(y), e = y - mu, Va = MSx, Vb = Va, Ve = 1, L = Vb/Ve (sic)
  double mu = 0;
  for (int64_t i = 0; i < n; i++) { if (!(y[i] == y[i])) return fail(BWGR_ERR_ARG, "y contains NaN"); mu += y[i]; }
  mu /= (double)n;
  double vy = 0;
  for (int64_t i = 0; i < n; i++) vy += (y[i] - mu) * (y[i] - mu);
  vy /= (double)(n - 1);
  double MSx = 0, sxx = 0;
  for (int64_t j = 0; j < p; j++) { MSx += (h->h_xx[j] - h->h_sx[j] * h->h_sx[j] / (double)n) / ((double)n - 1.0); sxx += h->h_xx[j] * bag; }
  if (!(MSx > 0)) return fail(BWGR_ERR_ARG, "genotypes have no variance");
  std::vector<double> e0(n), b0(p, 0.0), d0(p, 1.0), L0(p, MSx), xxb(p);
  for (int64_t i = 0; i < n; i++) e0[i] = y[i] - mu;
  for (int64_t j = 0; j < p; j++) xxb[j] = h->h_xx[j] * bag;  // xx = crossprod * bag (:49)
  std::mt19937_64 gen(seed ^ 0x9E3779B97F4A7C15ull);
  std::vector<int64_t> rows(n);
  std::vector<uint8_t> mask((size_t)ld, 0), cnt((size_t)ld, 0);
  std::vector<float> cntf((size_t)ld, 0.0f);
  bool overflow = false;
  auto draw = [&]() {  // Use = sort(sample(n, n * bag, rp)) (:68) as a mask (+ the multiplicity of every row when rp = TRUE)
    std::fill(mask.begin(), mask.end(), 0);
    if (rp) {
      std::fill(cnt.begin(), cnt.end(), 0);
      std::uniform_int_distribution<int64_t> pick(0, n - 1);
      for (int64_t r = 0; r < nuse; r++) { const int64_t q = pick(gen); mask[q] = 1; if (cnt[q] == 255) overflow = true; else cnt[q]++; }
      for (int64_t r = 0; r < n; r++) cntf[r] = (float)cnt[r];
      return;
    }
    for (int64_t r = 0; r < n; r++) rows[r] = r;
    for (int64_t r = 0; r < nuse; r++) { std::uniform_int_distribution<int64_t> pick(r, n - 1); std::swap(rows[r], rows[pick(gen)]); mask[rows[r]] = 1; }
  };
  FitGuard guard{h};
  int rc;
  if (bagged) {
    draw();
    rc = kmup_begin(h, b0.data(), d0.data(), xxb.data(), e0.data(), L0.data(), 1.0, pi, seed, mask.data(), (double)((float)n / (float)nuse),
                    rp ? cnt.data() : nullptr);
  } else {
    rc = kmup_begin(h, b0.data(), d0.data(), nullptr, e0.data(), L0.data(), 1.0, pi, seed);
  }
  if (rc) return rc;
  Fit& f = h->fit;
  {
    SysScalars c = f.sc0[0];
    c.mu = (float)mu;
    CU(cudaMemcpyAsync(f.sc.p, &c, sizeof(SysScalars), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  if (f.wst.alloc(1) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  CU(cudaMemsetAsync(f.wst.p, 0, sizeof(WgrState), h->stream));
  WgrArgs& w = f.wgr_args;
  memset(&w, 0, sizeof w);
  w.n = (int)n; w.p = (int)p; w.ld = ld; w.e = f.e.p; w.b = f.b.p; w.d = f.d.p; w.L = f.vbv.p;
  w.B = f.B.p; w.D = f.D.p; w.VB = f.VBv.p; w.sc = f.sc.p; w.st = f.wst.p; w.iv = iv; w.de = de;
  w.Sb = (float)(R2 * df * vy / MSx); w.Se = (float)((1 - R2) * df * vy); w.df = (float)df; w.MSx = (float)MSx;  // :58-59
  w.it = it; w.bi = bi; w.th = th; w.seed_lo = (uint32_t)seed; w.seed_hi = (uint32_t)(seed >> 32);
  if (!bagged) {
    f.wgr_mode = true;
    if ((rc = fit_sweeps(h, it))) return rc;
  } else {
    DevBuf<float> yd, hatd;
    if (yd.alloc(ld) != cudaSuccess || hatd.alloc(ld) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    std::vector<float> yf(ld, 0.0f);
    for (int64_t i = 0; i < n; i++) yf[i] = (float)y[i];
    CU(cudaMemcpyAsync(yd.p, yf.data(), sizeof(float) * ld, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    // phase 1 weighs e^2 by the byte (0/1 or the multiplicity); Ve's chi-square has n * bag + df degrees of freedom (:121), n * bag
    // unrounded although the sample holds floor(n * bag) rows
    w.mask = rp ? f.cnt.p : f.mask.p; w.nsub = (float)((double)n * bag); w.y = yd.p; w.hat = hatd.p;
    ColStatBufs cs;
    for (int i = 0; i < it; i++) {
      if (i > 0) {  // this iteration's rows: mask, and H'H of every marker over them (the rule's likelihood-ratio scale)
        draw();
        CU(cudaMemcpyAsync(f.mask.p, mask.data(), (size_t)ld, cudaMemcpyHostToDevice, h->stream));
        if (rp) {
          if (overflow) return fail(BWGR_ERR_UNSUPPORTED, "wgr(rp = TRUE): a row was drawn more than 255 times in one iteration");
          CU(cudaMemcpyAsync(f.cnt.p, cnt.data(), (size_t)ld, cudaMemcpyHostToDevice, h->stream));
          CU(cudaMemcpyAsync(f.row_w.p, cntf.data(), sizeof(float) * ld, cudaMemcpyHostToDevice, h->stream));
        }
        if ((rc = rows_col_stats(h, cs, rp ? f.cnt.p : f.mask.p, rp, 0, nullptr, nullptr))) return rc;
      }
      if ((rc = fit_sweeps(h, 1))) return rc;                                    // KMUP2 over the rows in use
      launch_wgr_bag_phase(w, 1, h->num_sms, h->stream);                          // Vb (with the old Ve), Va, Ve from the rows in use
      if ((rc = fit_hat(h, 1, f.b.p, reinterpret_cast<const float*>(f.sc.p), hatd.p))) return rc;  // mu + X b  (SysScalars starts with mu)
      launch_wgr_bag_phase(w, 2, h->num_sms, h->stream);                          // e = y - hat, intercept draw, L, posterior sums
      h->launches += 3;
    }
  }
  rc = check_err_flag(h, bagged ? "wgr (bagged) sweep" : "wgr sweep");
  if (rc) return rc;
  if (!bagged) dump_trace(h);
  WgrState st;
  CU(cudaMemcpyAsync(&st, f.wst.p, sizeof st, cudaMemcpyDeviceToHost, h->stream));
  std::vector<float> B(p), D(p), V(p);
  CU(cudaMemcpyAsync(B.data(), f.B.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(D.data(), f.D.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(V.data(), f.VBv.p, sizeof(float) * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  const double mc = (double)((it - bi) / th + 1);  // length(seq(bi, it, th)) (:41-42)
  double mD = 0;
  for (int64_t j = 0; j < p; j++) mD += D[j] / mc;
  mD /= (double)p;
  std::vector<float> Bm(p), hh;
  for (int64_t j = 0; j < p; j++) Bm[j] = (float)(B[j] / mc / mD);  // B = B/mc/mean(D) (:143)
  const float B0 = (float)(st.B0 / mc);
  rc = fitted_values(h, 1, Bm.data(), true, &B0, hh);  // HAT = B0 + gen0 %*% B (:152)
  if (rc) return rc;
  if (b) for (int64_t j = 0; j < p; j++) b[j] = Bm[j];
  if (d) for (int64_t j = 0; j < p; j++) d[j] = D[j] / mc;
  if (Vb && iv) for (int64_t j = 0; j < p; j++) Vb[j] = V[j] / mc;
  if (hat) for (int64_t i = 0; i < n; i++) hat[i] = hh[i];
  if (scal) { scal[0] = B0; scal[1] = st.VE / mc; scal[2] = iv ? 0.0 : st.VA / mc; scal[3] = sxx / (double)p; }
  return 0;
}

int bwgr_wgr_fit(bwgr_handle* h, const double* y, int it, int bi, int th, int iv, int de, double pi, double df, double R2,
                 uint64_t seed, double* b, double* d, double* Vb, double* hat, double* scal) {
  return wgr_fit(h, y, it, bi, th, 1.0, 0, iv, de, pi, df, R2, seed, b, d, Vb, hat, scal);
}

// Rows of one bagged iteration as a 0/1 mask plus the multiplicity of every row.  use: 0-based row indices as R passes them
// (doubles).  *repeats = some row occurs more than once (sampling with replacement, rp = TRUE).
static int use_to_mask(const double* use, int64_t nuse, int64_t n, std::vector<uint8_t>& mask, std::vector<uint8_t>& cnt, bool* repeats) {
  mask.assign((size_t)n, 0);
  cnt.assign((size_t)n, 0);
  *repeats = false;
  for (int64_t q = 0; q < nuse; q++) {
    const int64_t r = (int64_t)use[q];
    if (r < 0 || r >= n) return fail(BWGR_ERR_ARG, "Use[%lld] = %lld is not a row of X", (long long)q, (long long)r);
    if (cnt[r] == 255) return fail(BWGR_ERR_UNSUPPORTED, "KMUP2: row %lld occurs more than 255 times in Use", (long long)r);
    if (mask[r]) *repeats = true;
    mask[r] = 1;
    cnt[r]++;
  }
  return 0;
}

// KMUP2(X,Use,b,d,xx,E,L,Ve,pi) (:41-77): one Kuo-Mallick sweep over the rows Use.  b, d updated in place; e_out [nuse] = the
// residuals of the rows in use, in the order of Use (the reference's third list element).  Runs on the small-n family (row mask).
int bwgr_kmup2_sweep(bwgr_handle* h, const double* use, int64_t nuse, double* b, double* d, const double* xx, const double* E,
                     double* e_out, const double* L, double Ve, double pi, uint64_t seed) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!use || !E || !e_out || nuse < 2) return fail(BWGR_ERR_ARG, "KMUP2: bad Use / E / e_out");
  const int64_t n = h->n;
  std::vector<uint8_t> mask, cnt;
  bool repeats = false;
  int rc = use_to_mask(use, nuse, n, mask, cnt, &repeats);
  if (rc) return rc;
  FitGuard guard{h};
  rc = kmup_begin(h, b, d, xx, E, L, Ve, pi, seed, mask.data(), (double)((float)n / (float)nuse), repeats ? cnt.data() : nullptr);
  if (rc) return rc;
  return kmup_sweep_out(h, "kmup2 sweep", b, d, e_out, use, nuse);
}

// wgr(y,X,it,bi,th,bag,rp,iv,de,pi,df,R2): bwgr_wgr_fit with row bagging (see wgr_fit); bag = 1 is bwgr_wgr_fit.  Same outputs.
int bwgr_wgr_fit_bag(bwgr_handle* h, const double* y, int it, int bi, int th, double bag, int rp, int iv, int de, double pi, double df,
                     double R2, uint64_t seed, double* b, double* d, double* Vb, double* hat, double* scal) {
  return wgr_fit(h, y, it, bi, th, bag, rp, iv, de, pi, df, R2, seed, b, d, Vb, hat, scal);
}

}  // extern "C"

namespace {
// ---- small dense symmetric helpers for the k x k part of MRR3 (column-major, double) ----------------------------------
using Mat = std::vector<double>;
// cyclic Jacobi: A = V diag(w) V', eigenvalues ascending (what Eigen's SelfAdjointEigenSolver returns, :639)
void sym_eig(const Mat& Ain, int k, std::vector<double>& w, Mat& V) {
  Mat A(Ain);
  V.assign((size_t)k * k, 0.0);
  for (int i = 0; i < k; i++) V[i + (size_t)i * k] = 1.0;
  for (int sweep = 0; sweep < 64; sweep++) {
    double off = 0;
    for (int i = 0; i < k; i++) for (int j = 0; j < i; j++) off += A[i + (size_t)j * k] * A[i + (size_t)j * k];
    if (off < 1e-300) break;
    for (int pI = 0; pI < k - 1; pI++)
      for (int q = pI + 1; q < k; q++) {
        const double apq = A[pI + (size_t)q * k];
        if (std::fabs(apq) < 1e-300) continue;
        const double theta = (A[q + (size_t)q * k] - A[pI + (size_t)pI * k]) / (2.0 * apq);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), sn = t * c;
        for (int r = 0; r < k; r++) {
          const double arp = A[r + (size_t)pI * k], arq = A[r + (size_t)q * k];
          A[r + (size_t)pI * k] = c * arp - sn * arq; A[r + (size_t)q * k] = sn * arp + c * arq;
        }
        for (int r = 0; r < k; r++) {
          const double apr = A[pI + (size_t)r * k], aqr = A[q + (size_t)r * k];
          A[pI + (size_t)r * k] = c * apr - sn * aqr; A[q + (size_t)r * k] = sn * apr + c * aqr;
        }
        for (int r = 0; r < k; r++) {
          const double vrp = V[r + (size_t)pI * k], vrq = V[r + (size_t)q * k];
          V[r + (size_t)pI * k] = c * vrp - sn * vrq; V[r + (size_t)q * k] = sn * vrp + c * vrq;
        }
      }
  }
  std::vector<int> idx(k);
  for (int i = 0; i < k; i++) idx[i] = i;
  std::sort(idx.begin(), idx.end(), [&](int a, int b) { return A[a + (size_t)a * k] < A[b + (size_t)b * k]; });
  w.resize(k);
  Mat Vs((size_t)k * k);
  for (int c = 0; c < k; c++) { w[c] = A[idx[c] + (size_t)idx[c] * k]; for (int r = 0; r < k; r++) Vs[r + (size_t)c * k] = V[r + (size_t)idx[c] * k]; }
  V.swap(Vs);
}
bool chol_ok(const Mat& Ain, int k) {  // LLT success test (:603-607)
  Mat A(Ain);
  for (int j = 0; j < k; j++) {
    double d = A[j + (size_t)j * k];
    for (int c = 0; c < j; c++) d -= A[j + (size_t)c * k] * A[j + (size_t)c * k];
    if (!(d > 0)) return false;
    d = std::sqrt(d);
    A[j + (size_t)j * k] = d;
    for (int i = j + 1; i < k; i++) {
      double v = A[i + (size_t)j * k];
      for (int c = 0; c < j; c++) v -= A[i + (size_t)c * k] * A[j + (size_t)c * k];
      A[i + (size_t)j * k] = v / d;
    }
  }
  return true;
}
void sym_pinv(const Mat& A, int k, Mat& out) {  // completeOrthogonalDecomposition().pseudoInverse() of a symmetric matrix (:648)
  std::vector<double> w; Mat V;
  sym_eig(A, k, w, V);
  double wmax = 0;
  for (double v : w) wmax = std::max(wmax, std::fabs(v));
  const double tol = wmax * k * 2.220446049250313e-16;
  out.assign((size_t)k * k, 0.0);
  for (int c = 0; c < k; c++) {
    if (std::fabs(w[c]) <= tol) continue;
    const double iw = 1.0 / w[c];
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) out[i + (size_t)j * k] += iw * V[i + (size_t)c * k] * V[j + (size_t)c * k];
  }
}

// MRR3's argument list after (Y, X), in the order of R/RcppExports.R:180
struct MrrFlags {
  int maxit; double tol; bool TH; double NLfactor; bool InnerGS, NoInv, HCS, XFA, ACS; int NumXFA; double R2, gc0, df0; bool updateMu;
  double wph2, wpgc, PenCor, MinCor, uncorH2below, rUpFrom, rUpTo, rDownFrom, rDownTo, bkFrom, bkTo, DeflateMax, DeflateBy;
  bool OneVarB, OneVarE;
  explicit MrrFlags(const double* par) {
    int q = 0;
    maxit = (int)par[q++]; tol = par[q++]; q++; TH = par[q++] != 0; NLfactor = par[q++];
    InnerGS = par[q++] != 0; NoInv = par[q++] != 0; HCS = par[q++] != 0; XFA = par[q++] != 0; ACS = par[q++] != 0;
    NumXFA = (int)par[q++]; R2 = par[q++]; gc0 = par[q++]; df0 = par[q++]; updateMu = par[q++] != 0;
    wph2 = par[q++]; wpgc = par[q++]; PenCor = par[q++]; MinCor = par[q++]; uncorH2below = par[q++];
    rUpFrom = par[q++]; rUpTo = par[q++]; rDownFrom = par[q++]; rDownTo = par[q++]; bkFrom = par[q++]; bkTo = par[q++];
    DeflateMax = par[q++]; DeflateBy = par[q++]; OneVarB = par[q++] != 0; OneVarE = par[q++] != 0;
  }
};
// The state of MRR3's outer loop that survives from sweep to sweep, the same on the rotated fast path and the general path.
struct MrrVar {
  Mat vb, iG, GC, Sb;
  std::vector<double> vbInit;
  double Deflate = 1, inflate = 0;
  std::vector<double> mu, vy, MSx, nn;  // per trait: mean and variance of y, sum of the marker variances, observations (the path's)
  std::vector<double> ve, iVe, veInit, h2, Se, iNp;
  std::vector<double> cnvB, cnvH2, cnvV;  // convergence records (:662-666)
  int numit = 0;
};
// Output arrays of bwgr_mrr3_fit (any may be null)
struct MrrOut {
  double *mu, *b, *hat, *h2, *GC, *vb, *ve, *MSx, *cnv, *W;
  int* its;
};

// Starting values (:394-432) from V.vy, V.MSx and V.nn.
void mrr_start(const MrrFlags& F, int k, MrrVar& V) {
  auto M = [k](int r, int c) { return (size_t)r + (size_t)c * k; };
  Mat& vb = V.vb;
  vb.assign((size_t)k * k, 0.0); V.iG.assign((size_t)k * k, 0.0); V.GC.assign((size_t)k * k, 0.0);
  for (auto* v : {&V.vbInit, &V.ve, &V.iVe, &V.veInit, &V.h2, &V.Se, &V.iNp}) v->resize(k);
  for (int t = 0; t < k; t++) {
    V.ve[t] = V.vy[t] * (1 - F.R2); V.iVe[t] = 1.0 / V.ve[t]; V.veInit[t] = V.ve[t];
    V.vbInit[t] = V.vy[t] * F.R2 / V.MSx[t]; vb[M(t, t)] = V.vbInit[t]; V.iG[M(t, t)] = 1.0 / V.vbInit[t]; V.h2[t] = 1 - V.ve[t] / V.vy[t];
    V.Se[t] = V.ve[t] * F.df0; V.iNp[t] = 1.0 / (V.nn[t] + F.df0 - 1.0);
  }
  for (int i = 0; i < k; i++) for (int j = 0; j < i; j++) { const double v = F.gc0 * std::sqrt(vb[M(i, i)] * vb[M(j, j)]); vb[M(i, j)] = v; vb[M(j, i)] = v; }
  V.Sb = vb;
  for (auto& v : V.Sb) v *= F.df0;
}

// Residual variances of one sweep (:536-543) from e'y of trait t at ey[t * stride].
void mrr_residual_var(const MrrFlags& F, int k, const double* ey, int stride, MrrVar& V) {
  for (int t = 0; t < k; t++) { V.ve[t] = (ey[(size_t)t * stride] + V.Se[t]) * V.iNp[t]; V.h2[t] = 1 - V.ve[t] / V.vy[t]; }
  if (F.wph2 > 0) for (int t = 0; t < k; t++) V.ve[t] = V.ve[t] * (1 - F.wph2) + F.wph2 * V.veInit[t];
  if (F.OneVarE) { double m = 0; for (int t = 0; t < k; t++) m += V.ve[t]; m /= k; for (int t = 0; t < k; t++) V.ve[t] = m; }
  for (int t = 0; t < k; t++) V.iVe[t] = 1.0 / V.ve[t];
}

// Convergence records of one sweep (:662-666) from |beta0 - b|^2 of every trait; vb0 and h20 are vb and h2 before the sweep.
// False: the outer loop ends here.
bool mrr_record(const MrrFlags& F, int k, const double* db, const Mat& vb0, const std::vector<double>& h20, MrrVar& V) {
  double mx = -1e300;
  for (int t = 0; t < k; t++) mx = std::max(mx, db[t]);
  const double cnv = std::log10(mx);
  V.cnvB.push_back(cnv);
  if (cnv != cnv) return false;  // :663
  { double sH = 0; for (int t = 0; t < k; t++) sH += (h20[t] - V.h2[t]) * (h20[t] - V.h2[t]); V.cnvH2.push_back(std::log10(sH)); }
  { double sV = 0; for (size_t i = 0; i < V.vb.size(); i++) sV += (vb0[i] - V.vb[i]) * (vb0[i] - V.vb[i]); V.cnvV.push_back(std::log10(sV)); }
  ++V.numit;
  return !(cnv < std::log10(F.tol));
}

// The outputs (:676-700) both paths share; b, hat and W are the path's own.
void mrr_copy_out(const MrrFlags& F, int k, const MrrVar& V, const MrrOut& o) {
  for (int t = 0; t < k; t++) {
    if (o.mu) o.mu[t] = V.mu[t];
    if (o.h2) o.h2[t] = V.h2[t];
    if (o.ve) o.ve[t] = V.ve[t];
    if (o.MSx) o.MSx[t] = V.MSx[t];
  }
  if (o.GC) for (int i = 0; i < k * k; i++) o.GC[i] = V.GC[i];
  if (o.vb) for (int i = 0; i < k * k; i++) o.vb[i] = V.vb[i];
  if (o.cnv)
    for (int i = 0; i < V.numit; i++) { o.cnv[i] = V.cnvB[i]; o.cnv[F.maxit + i] = V.cnvH2[i]; o.cnv[2 * F.maxit + i] = V.cnvV[i]; }
  if (o.its) *o.its = V.numit;
}
// Genetic (co)variances of one sweep (:559-648): TildeHat and the traces Tr (TrXSX, or TrDinvXSX under TH) in, vb / GC / iG out.
// Shared by the rotated fast path and the general path; double, on the host (k <= 32).
void mrr_varcomp(const MrrFlags& F, int k, const Mat& TildeHat, const std::vector<double>& Tr, const std::vector<double>& h2, MrrVar& V) {
  auto M = [k](int r, int c) { return (size_t)r + (size_t)c * k; };
  Mat &vb = V.vb, &iG = V.iG, &GC = V.GC, A;
  const Mat& Sb = V.Sb;
  const std::vector<double>& vbInit = V.vbInit;
  double &Deflate = V.Deflate, &inflate = V.inflate;
  const double df0 = F.df0, wph2 = F.wph2, wpgc = F.wpgc, gc0 = F.gc0, PenCor = F.PenCor, MinCor = F.MinCor, uncorH2below = F.uncorH2below;
  const double rUpFrom = F.rUpFrom, rUpTo = F.rUpTo, rDownFrom = F.rDownFrom, rDownTo = F.rDownTo, bkFrom = F.bkFrom, bkTo = F.bkTo;
  const double DeflateMax = F.DeflateMax, DeflateBy = F.DeflateBy, bucketMean = 0.5 * (F.bkFrom + F.bkTo);
  const bool ACS = F.ACS, HCS = F.HCS, XFA = F.XFA, OneVarB = F.OneVarB;
  const int NumXFA = F.NumXFA;
  const bool rebuild = !F.NoInv || F.TH;  // :628, :647: with NoInv (and no TH) the correlations are not bent and iG keeps its start value
  for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) {
    if (i == j) vb[M(i, i)] = (TildeHat[M(i, i)] + Sb[M(i, i)]) / (Tr[i] + df0);
    else vb[M(i, j)] = (TildeHat[M(i, j)] + TildeHat[M(j, i)] + Sb[M(i, j)]) / (Tr[i] + Tr[j] + df0);
  }
  if (wph2 > 0) for (int i = 0; i < k; i++) vb[M(i, i)] = vb[M(i, i)] * (1 - wph2) + wph2 * vbInit[i];
  if (wpgc > 0) {
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++)
      GC[M(i, j)] = (i != j) ? (1.0 - wpgc) * vb[M(i, j)] / std::sqrt(vb[M(i, i)] * vb[M(j, j)]) + gc0 * wpgc : 1.0;
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) if (i != j) vb[M(i, j)] = GC[M(i, j)] * std::sqrt(vb[M(i, i)] * vb[M(j, j)]);
  } else {
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) GC[M(i, j)] = vb[M(i, j)] / std::sqrt(vb[M(i, i)] * vb[M(j, j)]);
  }
  auto top_factors = [&](double add, double scale) {  // :593-600, :612-617
    std::vector<double> ew; Mat ev;
    sym_eig(GC, k, ew, ev);
    Mat UDU((size_t)k * k, 0.0);
    for (int fI = 0; fI < NumXFA && fI < k; fI++) {
      const int c = k - fI - 1;
      for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) UDU[M(i, j)] += ew[c] * ev[M(i, c)] * ev[M(j, c)];
    }
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) GC[M(i, j)] = (UDU[M(i, j)] + add) * scale;
    for (int i = 0; i < k; i++) GC[M(i, i)] = 1;
  };
  if (ACS) {
    double gs = 0;
    for (double v : GC) gs += v;
    gs = (gs - k) / ((k * (k - 1))) / 2.0;
    top_factors(gs, 0.5);
  } else if (HCS) {
    double gs = 0;
    for (int i = 0; i < k; i++) for (int j = 0; j < i; j++) gs += GC[M(i, j)];
    gs = gs / ((k * (k - 1)) / 2);
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) GC[M(i, j)] = (i != j) ? gs : 1.0;
  } else if (XFA) {
    top_factors(0.0, 1.0);
  }
  for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) if (i != j) {  // :619-626
    double& g = GC[M(i, j)];
    if (MinCor < 1 && g < MinCor) g = 0;
    if (PenCor > 0) g = std::tanh(PenCor * std::fabs(g)) * g;
    if (rDownFrom < 1 && g < rDownFrom) g = rDownTo;
    if (rUpFrom < 1 && g > rUpFrom) g = rUpTo;
    if (bkFrom < 1 && g > bkFrom && g < bkTo) g = bucketMean;
    if (uncorH2below > 0 && (h2[i] < uncorH2below || h2[j] < uncorH2below)) g = 0;
  }
  if (rebuild) {  // bending (:629-644)
    A = GC;
    if (DeflateBy > 0) {
      for (auto& v : A) v *= Deflate;
      for (int i = 0; i < k; i++) A[M(i, i)] = 1;
      if (!chol_ok(A, k) && Deflate > DeflateMax) {
        Deflate -= DeflateBy;
        A = GC;
        for (auto& v : A) v *= Deflate;
        for (int i = 0; i < k; i++) A[M(i, i)] = 1;
      }
    }
    std::vector<double> ew; Mat ev;
    sym_eig(A, k, ew, ev);
    if (ew[0] < 0) {
      inflate = std::fabs(ew[0] * 1.1);
      for (int i = 0; i < k; i++) A[M(i, i)] += inflate;
      for (auto& v : A) v /= (1.0 + inflate);
      GC = A;
    }
  }
  if (OneVarB) {
    double tmp = 0;
    for (int i = 0; i < k; i++) tmp += TildeHat[M(i, i)];
    tmp /= k;
    for (size_t i = 0; i < vb.size(); i++) vb[i] = GC[i] * tmp;
  } else {
    const Mat dv(vb);
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) vb[M(i, j)] = GC[M(i, j)] * std::sqrt(dv[M(i, i)] * dv[M(j, j)]);
  }
  if (rebuild) sym_pinv(vb, k, iG);
}

// MRR3 / MRR3F on the general device path (mrr_gen.cu): per-trait observation masks, InnerGS, NLfactor, TH, MRR3F's NoInv system.
// Host side = the reference's set-up (:359-432) and the k x k variance block; everything O(n), O(p) or O(n p) is a kernel.
int mrr3_general(bwgr_handle* h, int f32_variant, const double* Y, int k, const MrrFlags& F, const MrrOut& out) {
  if (h->storage != BWGR_STORE_I8 || !h->x8) return fail(BWGR_ERR_UNSUPPORTED, "MRR3 (general path) reads the int8 store");
  if (h->world > 1) return fail(BWGR_ERR_UNSUPPORTED, "MRR3 does not run on a row-sharded store");
  const int64_t n = h->n, p = h->p, ld = h->ld;
  const int maxit = F.maxit, kk = k * k;
  const bool innergs = F.InnerGS, noinv_system = f32_variant && F.NoInv, NonLinear = F.NLfactor != 0;
  const int nmat = innergs ? 2 : 1;
  auto M = [k](int r, int c) { return (size_t)r + (size_t)c * k; };
  CU(cudaSetDevice(h->device));
  // ---- incidence, counts, centred phenotypes (:359-376)
  MrrVar V;
  std::vector<double> &nn = V.nn, &mu = V.mu, &vy = V.vy, &MSx = V.MSx;
  nn.resize(k); mu.resize(k); vy.resize(k); MSx.assign(k, 0.0);
  std::vector<uint32_t> zb((size_t)ld, 0u);
  std::vector<double> ysum(k), yh((size_t)k * ld, 0.0);
  for (int t = 0; t < k; t++) {
    double sum = 0; int64_t cnt = 0;
    for (int64_t i = 0; i < n; i++) { const double v = Y[(size_t)t * n + i]; if (v == v) { zb[i] |= 1u << t; sum += v; cnt++; } }
    if (cnt < 2) return fail(BWGR_ERR_ARG, "MRR3: trait %d has fewer than two observations", t + 1);
    nn[t] = (double)cnt; mu[t] = sum / (double)cnt;
    double s1 = 0, s2 = 0;
    for (int64_t i = 0; i < n; i++) {
      const double v = Y[(size_t)t * n + i];
      if (v == v) { const double c = v - mu[t]; yh[(size_t)t * ld + i] = c; s1 += c; s2 += c * c; }
    }
    ysum[t] = s1; vy[t] = s2 / (nn[t] - 1.0);
    if (!(vy[t] > 0)) return fail(BWGR_ERR_ARG, "MRR3: trait %d has no variance", t + 1);
  }
  // ---- launch geometry: one CTA per row slab, all co-resident
  int rp = 0, grid = 0;
  grid_geometry(h, &rp, &grid);
  const size_t smem = mrr_gen_smem(k, rp, innergs);
  if (smem > h->smem_optin || grid > h->num_sms)
    return fail(BWGR_ERR_UNSUPPORTED, "MRR3 (general path): %lld rows x %d traits do not fit the shared memory of %d SMs", (long long)n, k, h->num_sms);
  DevBuf<uint32_t> zbits; DevBuf<double> yd, ed, bd, bold, fixd, meand, tilded, sold, Wd, xsxd, dinvd, small;
  DevBuf<unsigned long long> accd; DevBuf<int> permd;
  const size_t nsmall = (size_t)2 * kk + 11 * 32;  // iG | vb | iVe | se | ey | cnv | trd | par(2 x 32) | shift | see | scale(2 x 32)
  if (zbits.alloc(ld) != cudaSuccess || yd.alloc((size_t)k * ld) != cudaSuccess || ed.alloc((size_t)k * ld) != cudaSuccess ||
      bd.alloc((size_t)p * k) != cudaSuccess || bold.alloc((size_t)p * k) != cudaSuccess || fixd.alloc((size_t)p * 2 * k) != cudaSuccess ||
      meand.alloc(p) != cudaSuccess || tilded.alloc((size_t)p * k) != cudaSuccess || sold.alloc((size_t)p * nmat * kk) != cudaSuccess ||
      (NonLinear && Wd.alloc((size_t)p * k) != cudaSuccess) || (F.TH && (xsxd.alloc((size_t)p * k) != cudaSuccess || dinvd.alloc((size_t)p * k) != cudaSuccess)) ||
      small.alloc(nsmall + kk) != cudaSuccess || accd.alloc((size_t)p * 32 * kGridCopies) != cudaSuccess || grid > 255 ||
      permd.alloc(p + 32) != cudaSuccess)
    return fail(BWGR_ERR_CUDA, "cudaMalloc(MRR3 general workspace) failed");
  double *d_iG = small.p, *d_vb = small.p + kk, *d_iVe = d_vb + kk, *d_se = d_iVe + 32, *d_ey = d_se + 32, *d_cnv = d_ey + 32,
         *d_trd = d_cnv + 32, *d_par = d_trd + 32, *d_shift = d_par + 64, *d_see = d_shift + 32, *d_scale = d_see + 32, *d_th = small.p + nsmall;
  cudaStream_t st = h->stream;
  CU(cudaMemcpyAsync(zbits.p, zb.data(), sizeof(uint32_t) * ld, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(yd.p, yh.data(), sizeof(double) * k * ld, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(ed.p, yd.p, sizeof(double) * k * ld, cudaMemcpyDeviceToDevice, st));  // e = y (:435)
  CU(cudaMemsetAsync(bd.p, 0, sizeof(double) * p * k, st));
  // ---- masked column statistics (:381-392) and tilde = X_c'y (:420) from one pass over the store
  std::vector<double> sxz((size_t)p * k), sxxz((size_t)p * k), tilde((size_t)p * k), fixed((size_t)p * 2 * k), meanv(p), xsx;
  {
    DevBuf<double> a1, a2;
    if (a1.alloc((size_t)p * k) != cudaSuccess || a2.alloc((size_t)p * k) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
    launch_mrr_gen_colstats(h->view(), zbits.p, yd.p, k, a1.p, a2.p, tilded.p, st);
    h->launches++;
    CU(cudaMemcpyAsync(sxz.data(), a1.p, sizeof(double) * p * k, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(sxxz.data(), a2.p, sizeof(double) * p * k, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(tilde.data(), tilded.p, sizeof(double) * p * k, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  std::vector<double> TrXSX(k), see(k);
  for (int t = 0; t < k; t++) see[t] = vy[t] * (nn[t] - 1.0);  // e = y at the start
  if (F.TH) xsx.resize((size_t)p * k);
  for (int64_t j = 0; j < p; j++) {
    const double m = h->h_sx[j] / (double)n;  // X.colwise().mean() over all n0 rows (:378)
    meanv[j] = m;
    for (int t = 0; t < k; t++) {
      const size_t q = (size_t)j * k + t;
      const double XX = sxxz[q] - 2.0 * m * sxz[q] + m * m * nn[t];  // sum_i (x - m)^2 z_it
      const double sc = sxz[q] - m * nn[t];                           // sum_i (x - m) z_it
      const double qq = sc / nn[t], v = XX / nn[t] - qq * qq;         // XSX (:386-388)
      fixed[(size_t)j * 2 * k + t] = XX; fixed[(size_t)j * 2 * k + k + t] = sc;
      MSx[t] += v;
      if (F.TH) xsx[q] = v * nn[t];                                   // :423
      tilde[q] -= m * ysum[t];
    }
  }
  for (int t = 0; t < k; t++) {
    if (!(MSx[t] > 0)) return fail(BWGR_ERR_ARG, "genotypes have no variance");
    TrXSX[t] = nn[t] * MSx[t];
  }
  CU(cudaMemcpyAsync(fixd.p, fixed.data(), sizeof(double) * p * 2 * k, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(meand.p, meanv.data(), sizeof(double) * p, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(tilded.p, tilde.data(), sizeof(double) * p * k, cudaMemcpyHostToDevice, st));
  if (F.TH) CU(cudaMemcpyAsync(xsxd.p, xsx.data(), sizeof(double) * p * k, cudaMemcpyHostToDevice, st));
  mrr_start(F, k, V);
  Mat TildeHat((size_t)kk);
  std::vector<int> order(p), irgs(32);
  for (int64_t j = 0; j < p; j++) order[j] = (int)j;
  for (int j = 0; j < 32; j++) irgs[j] = j;
  std::vector<double> W, bh, hsmall(32 * 4 + kk), trd(k);
  if (NonLinear) { W.assign((size_t)p * k, 1.0); CU(cudaMemcpyAsync(Wd.p, W.data(), sizeof(double) * p * k, cudaMemcpyHostToDevice, st)); }
  int rc = 0;
  MrrGenArgs a;
  a.g = h->view(); a.k = k; a.rows_per_cta = rp; a.innergs = innergs ? 1 : 0; a.perm = permd.p; a.irgs = permd.p + p; a.zbits = zbits.p;
  a.e = ed.p; a.b = bd.p; a.fixed = fixd.p; a.mean = meand.p; a.sol = sold.p; a.se0 = d_se; a.acc = accd.p; a.scale = d_scale; a.err = h->err.p;
  while (V.numit < maxit) {
    const Mat vb0(V.vb); const std::vector<double> h20(V.h2);
    const int numit = V.numit;
    CU(cudaMemcpyAsync(bold.p, bd.p, sizeof(double) * p * k, cudaMemcpyDeviceToDevice, st));  // beta0 (:475)
    std::shuffle(order.begin(), order.end(), std::mt19937(numit));                           // :483-484, cumulative
    std::shuffle(irgs.begin(), irgs.begin() + k, std::mt19937(numit));
    CU(cudaMemcpyAsync(permd.p, order.data(), sizeof(int) * p, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(permd.p + p, irgs.data(), sizeof(int) * 32, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_iG, V.iG.data(), sizeof(double) * kk, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_vb, V.vb.data(), sizeof(double) * kk, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_iVe, V.iVe.data(), sizeof(double) * k, cudaMemcpyHostToDevice, st));
    // MRR3 applies the marker weights in the solve (:504); MRR3F never does (its weights are an output only)
    launch_mrr_gen_systems((int)p, k, fixd.p, (NonLinear && !f32_variant) ? Wd.p : nullptr, d_iG, d_vb, d_iVe, noinv_system ? 1 : 0,
                           innergs ? 1 : 0, sold.p, st);
    launch_mrr_gen_colred(ed.p, nullptr, ld, (int)n, k, d_se, st);
    {  // fixed-point scale of the grid sums of this sweep: |x'e_t| <= sqrt(max_j x_j'x_j) |e_t| (Cauchy-Schwarz, also for the sum of
       // the per-CTA magnitudes); 16 x headroom for the growth of |e_t| inside a sweep, 2^52 of range
      std::vector<double> scl(64, 0.0);
      for (int t = 0; t < k; t++) {
        int ex = 0;
        std::frexp(16.0 * std::sqrt(h->xx_max * see[t]) + 1e-300, &ex);
        scl[t] = std::ldexp(1.0, 52 - ex); scl[32 + t] = std::ldexp(1.0, ex - 52);
      }
      CU(cudaMemcpyAsync(d_scale, scl.data(), sizeof(double) * 64, cudaMemcpyHostToDevice, st));
      CU(cudaMemsetAsync(accd.p, 0, sizeof(unsigned long long) * p * 32 * kGridCopies, st));
      const cudaError_t le = launch_mrr_gen_sweep(a, grid, st);
      if (le != cudaSuccess) return fail(BWGR_ERR_CUDA, "MRR3 general sweep launch failed: %s", cudaGetErrorString(le));
    }
    launch_mrr_gen_colred(ed.p, yd.p, ld, (int)n, k, d_ey, st);  // e.y (:536)
    launch_mrr_gen_colred(ed.p, ed.p, ld, (int)n, k, d_see, st);  // |e_t|^2: the next sweep's fixed-point range
    h->launches += 5;
    CU(cudaMemcpyAsync(hsmall.data(), d_ey, sizeof(double) * k, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(see.data(), d_see, sizeof(double) * k, cudaMemcpyDeviceToHost, st));
    if (NonLinear) { bh.resize((size_t)p * k); CU(cudaMemcpyAsync(bh.data(), bd.p, sizeof(double) * p * k, cudaMemcpyDeviceToHost, st)); }
    CU(cudaStreamSynchronize(st));
    rc = check_err_flag(h, "MRR3 general sweep");
    if (rc) return rc;
    if (NonLinear) {  // :524-533
      std::vector<double> tmpW(p);
      for (int t = 0; t < k; t++) {
        double maxW = -INFINITY, minW = INFINITY;
        for (int64_t j = 0; j < p; j++) { const double v = std::fabs(bh[(size_t)j * k + t]); maxW = std::max(maxW, v); minW = std::min(minW, v); }
        double sw = 0;
        for (int64_t j = 0; j < p; j++) { tmpW[j] = F.NLfactor * (std::fabs(bh[(size_t)j * k + t]) - minW) / (maxW - minW) + (1.0 - F.NLfactor); sw += tmpW[j]; }
        const double mw = sw / (double)p;
        for (int64_t j = 0; j < p; j++) W[(size_t)j * k + t] = tmpW[j] + (1.0 - mw);
      }
      CU(cudaMemcpyAsync(Wd.p, W.data(), sizeof(double) * p * k, cudaMemcpyHostToDevice, st));
    }
    mrr_residual_var(F, k, hsmall.data(), 1, V);
    // ---- tilde-hat (:546-556) and the convergence sums (:662)
    if (F.TH) {
      std::vector<double> par(64, 0.0);
      for (int t = 0; t < k; t++) { par[t] = V.ve[t]; par[k + t] = V.iG[M(t, t)]; }
      CU(cudaMemcpyAsync(d_par, par.data(), sizeof(double) * 2 * k, cudaMemcpyHostToDevice, st));
      launch_mrr_gen_pk(2, xsxd.p, nullptr, dinvd.p, d_par, (int)p, k, d_trd, st);
      launch_mrr_gen_pk(0, bd.p, tilded.p, dinvd.p, nullptr, (int)p, k, d_th, st);
      h->launches++;
    } else {
      launch_mrr_gen_pk(0, bd.p, tilded.p, nullptr, nullptr, (int)p, k, d_th, st);
    }
    launch_mrr_gen_pk(1, bold.p, bd.p, nullptr, nullptr, (int)p, k, d_cnv, st);
    h->launches += 2;
    CU(cudaMemcpyAsync(hsmall.data(), d_cnv, sizeof(double) * 64, cudaMemcpyDeviceToHost, st));  // cnv | trd
    CU(cudaMemcpyAsync(hsmall.data() + 128, d_th, sizeof(double) * kk, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) TildeHat[M(i, j)] = hsmall[128 + (size_t)i * k + j];
    for (int t = 0; t < k; t++) trd[t] = hsmall[32 + t];
    mrr_varcomp(F, k, TildeHat, F.TH ? trd : TrXSX, V.h2, V);
    if (F.updateMu) {  // :651-655; iN is 1 / (n_t - 1) by now (:395)
      launch_mrr_gen_colred(ed.p, nullptr, ld, (int)n, k, d_se, st);
      std::vector<double> sh(k);
      CU(cudaMemcpyAsync(sh.data(), d_se, sizeof(double) * k, cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      for (int t = 0; t < k; t++) { sh[t] /= (nn[t] - 1.0); mu[t] += sh[t]; }
      CU(cudaMemcpyAsync(d_shift, sh.data(), sizeof(double) * k, cudaMemcpyHostToDevice, st));
      launch_mrr_gen_shift(ed.p, zbits.p, ld, (int)n, k, d_shift, st);
      CU(cudaStreamSynchronize(st));
      h->launches += 2;
    }
    if (!mrr_record(F, k, hsmall.data(), vb0, h20, V)) break;
  }
  // ---- outputs (:676-700): hat = X_c b + mu = X b + (mu - sum_j mean_j b_j)
  bh.resize((size_t)p * k);
  CU(cudaMemcpyAsync(bh.data(), bd.p, sizeof(double) * p * k, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (out.hat) {
    std::vector<float> bt((size_t)k * p), m0(k), hh;
    for (int t = 0; t < k; t++) {
      double shift = 0;
      for (int64_t j = 0; j < p; j++) { const double v = bh[(size_t)j * k + t]; shift += meanv[j] * v; bt[(size_t)t * p + j] = (float)v; }
      m0[t] = (float)(mu[t] - shift);
    }
    if ((rc = fitted_values(h, k, bt.data(), true, m0.data(), hh))) return rc;
    for (size_t i = 0; i < hh.size(); i++) out.hat[i] = hh[i];
  }
  if (out.b) for (int t = 0; t < k; t++) for (int64_t j = 0; j < p; j++) out.b[(size_t)t * p + j] = bh[(size_t)j * k + t];
  if (out.W) for (int t = 0; t < k; t++) for (int64_t j = 0; j < p; j++) out.W[(size_t)t * p + j] = NonLinear ? W[(size_t)j * k + t] : 1.0;
  mrr_copy_out(F, k, V, out);
  return 0;
}
}  // namespace

extern "C" {

// MRR3 / MRR3F with the marker loop on the device (see mrr.cu).  Fast path = complete Y and the direct k x k solve:
// NaN in Y, InnerGS, NLfactor != 0, TH, and MRR3F's NoInv system return BWGR_ERR_UNSUPPORTED (never a CPU fallback).
int bwgr_mrr3_fit(bwgr_handle* h, int f32_variant, const double* Y, int k, const double* par, double* mu_out, double* b_out,
                  double* hat_out, double* h2_out, double* GC_out, double* vb_out, double* ve_out, double* MSx_out, double* cnv_out,
                  double* W_out, int* its_out) {
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (!Y || !par) return fail(BWGR_ERR_ARG, "null argument");
  if (k < 1 || k > 32) return fail(BWGR_ERR_UNSUPPORTED, "MRR3 on the B200 path takes 1..32 traits (k=%d)", k);
  const MrrFlags F(par);
  const MrrOut out{mu_out, b_out, hat_out, h2_out, GC_out, vb_out, ve_out, MSx_out, cnv_out, W_out, its_out};
  const int maxit = F.maxit;
  if (maxit < 1) return fail(BWGR_ERR_ARG, "maxit < 1");
  // n: this rank's rows (all of them on one GPU); ng: the individuals every sum over individuals runs over
  const int64_t n = h->n, p = h->p, ld = h->ld, ng = h->n_global;
  const bool dist = h->world > 1;
  bool missing = false;
  for (int64_t i = 0; i < n * k && !missing; i++) missing = !(Y[i] == Y[i]);
  // Everything the rotation cannot express -- missing phenotypes (per-trait XX), the inner Gauss-Seidel solve, marker weights,
  // MRR3F's NoInv system, the tilde-hat estimator -- runs on the general device path (mrr_gen.cu); BWGR_MRR=general forces it.
  const char* force = getenv("BWGR_MRR");
  const bool options = F.TH || F.NLfactor != 0 || F.InnerGS || (f32_variant && F.NoInv);
  const bool forced = force && !strcmp(force, "general");
  if (dist) {
    // A row-sharded store has the fast path only, and every rank must take the same road: the reasons any rank has to refuse are
    // all-reduced before any other collective, and then every rank refuses or none does.
    PipePlan pl;
    const bool no_fit = !h->hx_connected || h->storage != BWGR_STORE_I8 || !(h->xx_max < 16777216.0) || !plan_pipe(h, M_MRR, k, &pl);
    double why[4] = {missing ? 1.0 : 0.0, options ? 1.0 : 0.0, forced ? 1.0 : 0.0, no_fit ? 1.0 : 0.0};
    int rc = dist_allreduce_host(h, why, 4, true);
    if (rc) return rc;
    if (why[0] || why[1] || why[2] || why[3])
      return fail(BWGR_ERR_UNSUPPORTED, "the general MRR3 path does not run on a row-sharded store (%s)",
                  why[0] ? "missing phenotypes on some rank" : why[1] ? "TH, NLfactor, InnerGS or MRR3F's NoInv" :
                  why[2] ? "BWGR_MRR=general on some rank" : "the shard does not fit the pipelined blocked sweep on some rank");
  } else if (missing || options || forced) {
    return mrr3_general(h, f32_variant, Y, k, F, out);
  }
  auto M = [k](int r, int c) { return (size_t)r + (size_t)c * k; };
  // ---- setup (:359-432), double on the host
  MrrVar V;
  V.mu.assign(k, 0.0); V.vy.assign(k, 0.0); V.nn.assign(k, (double)ng);
  for (int t = 0; t < k; t++)
    for (int64_t i = 0; i < n; i++) V.mu[t] += Y[(size_t)t * n + i];
  int rc = dist_allreduce_host(h, V.mu.data(), k, false);
  if (rc) return rc;
  for (int t = 0; t < k; t++) {
    V.mu[t] /= (double)ng;
    for (int64_t i = 0; i < n; i++) { const double v = Y[(size_t)t * n + i] - V.mu[t]; V.vy[t] += v * v; }
  }
  if ((rc = dist_allreduce_host(h, V.vy.data(), k, false))) return rc;
  for (int t = 0; t < k; t++) V.vy[t] /= ((double)ng - 1.0);
  std::vector<float> xxc(p), sxf(p);
  double msx = 0;
  for (int64_t j = 0; j < p; j++) {
    const double c = h->h_xx[j] - h->h_sx[j] * h->h_sx[j] / (double)ng;  // XX(J,t) = sum (x - mean)^2, same for every trait (:382-385)
    xxc[j] = (float)c; sxf[j] = (float)h->h_sx[j];
    msx += c / (double)ng;                                              // XSX (:386-388): the centred column sums to zero
  }
  if (!(msx > 0)) return fail(BWGR_ERR_ARG, "genotypes have no variance");
  const double TrXSX = (double)ng * msx;
  V.MSx.assign(k, msx);
  mrr_start(F, k, V);
  // ---- device state through the common fit machinery: k systems of the rotated ridge rule
  FitSpec s;
  s.model = M_MRR; s.nsys = k; s.shuffled = true; s.row_mask = nullptr;
  s.df = 0; s.R2 = (float)F.R2; s.Pi = 0; s.alpha = 0; s.pi = 0; s.it = maxit; s.bi = 0; s.seed = 0;
  FitGuard guard{h};
  rc = fit_begin(h, s, Y);
  if (rc == BWGR_ERR_UNSUPPORTED && !dist)  // the shape does not fit the pipelined blocked sweep (row slabs above 512 rows): general path
    return mrr3_general(h, f32_variant, Y, k, F, out);
  if (rc) return rc;
  Fit& f = h->fit;
  f.skip_epilogue = true;
  DevBuf<float> tilde, e_alt, b_alt, b_old, Tdev, amax;
  DevBuf<double> red, red2;
  if (f.xx_over.alloc(p) != cudaSuccess || f.sx_dev.alloc(p) != cudaSuccess || f.cshift.alloc(32) != cudaSuccess ||
      tilde.alloc((size_t)k * p) != cudaSuccess || e_alt.alloc((size_t)k * ld) != cudaSuccess || b_alt.alloc((size_t)k * p) != cudaSuccess ||
      b_old.alloc((size_t)k * p) != cudaSuccess || Tdev.alloc(2 * 32 * 32) != cudaSuccess || amax.alloc(32) != cudaSuccess ||
      red.alloc((size_t)k * k + 3 * k) != cudaSuccess || red2.alloc((size_t)k * k) != cudaSuccess)
    return fail(BWGR_ERR_CUDA, "cudaMalloc(MRR3 workspace) failed");
  CU(cudaMemcpyAsync(f.xx_over.p, xxc.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(f.sx_dev.p, sxf.data(), sizeof(float) * p, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemsetAsync(e_alt.p, 0, sizeof(float) * k * ld, h->stream));
  // f.y holds the raw Y, f.e = Y - mu (fit_begin): centre y in place for the e.y reductions (:536)
  CU(cudaMemcpyAsync(f.y.p, f.e.p, sizeof(float) * k * ld, cudaMemcpyDeviceToDevice, h->stream));
  launch_xty(h->view(), f.y.p, k, tilde.p, h->stream);  // tilde = X'y (:420)
  h->launches++;
  if (dist) NC(nccl().AllReduce(tilde.p, tilde.p, (size_t)k * p, ncclFloat, ncclSum, h->comm, h->stream));
  std::vector<double> hred((size_t)k * k + 3 * k);
  std::vector<float> Tf(32 * 32), Tif(32 * 32), hmax(32);
  std::vector<SysScalars> sc(f.sc0);
  Mat TildeHat((size_t)k * k);
  while (V.numit < maxit) {
    const Mat vb0(V.vb); const std::vector<double> h20(V.h2);
    const std::vector<double>& iVe = V.iVe;
    // ---- rotation of this sweep: S^-1 iG S^-1 = U Lambda U', T = S U, T^-1 = U' S^-1
    Mat Ms((size_t)k * k), U; std::vector<double> lam;
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) Ms[M(i, j)] = V.iG[M(i, j)] / std::sqrt(iVe[i] * iVe[j]);
    sym_eig(Ms, k, lam, U);
    for (int sI = 0; sI < k; sI++) for (int t = 0; t < k; t++) {
      Tf[sI * k + t] = (float)(std::sqrt(iVe[sI]) * U[M(sI, t)]);       // T[s][t]
      Tif[sI * k + t] = (float)(U[M(t, sI)] / std::sqrt(iVe[t]));        // Tinv[s][t] = U[t][s] / S_t
    }
    CU(cudaMemcpyAsync(Tdev.p, Tf.data(), sizeof(float) * k * k, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(Tdev.p + 1024, Tif.data(), sizeof(float) * k * k, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(b_old.p, f.b.p, sizeof(float) * k * p, cudaMemcpyDeviceToDevice, h->stream));  // beta0 (:475)
    CU(cudaMemsetAsync(amax.p, 0, sizeof(float) * 32, h->stream));
    launch_rotate(f.e.p, e_alt.p, ld, (int)n, k, Tdev.p, nullptr, amax.p, h->num_sms, h->stream);
    launch_rotate(f.b.p, b_alt.p, p, (int)p, k, Tdev.p, nullptr, nullptr, h->num_sms, h->stream);
    h->launches += 2;
    f.e.swap(e_alt); f.b.swap(b_alt);
    // the fixed-point words of X_B'E the ranks exchange are summable only at one scale: max|e| over all individuals
    if (dist) NC(nccl().AllReduce(amax.p, amax.p, 32, ncclFloat, ncclMax, h->comm, h->stream));
    CU(cudaMemcpyAsync(hmax.data(), amax.p, sizeof(float) * 32, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int t = 0; t < k; t++) {
      SysScalars& c = sc[t];
      c.lmb = (float)std::max(lam[t], 0.0);
      set_e_scale(c, hmax[t]);
      c.done = 0; c.sweep = V.numit;
    }
    CU(cudaMemcpyAsync(f.sc.p, sc.data(), sizeof(SysScalars) * k, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemsetAsync(f.cshift.p, 0, sizeof(float) * 32, h->stream));
    rc = fit_sweeps(h, 1);  // marker order shuffle(mt19937(numit)) (:483), centred Gram band, k-system sweep
    if (rc) return rc;
    // ---- back to trait space: E = (E~ + c) T^-1, b = b~ T^-1
    launch_rotate(f.e.p, e_alt.p, ld, (int)n, k, Tdev.p + 1024, f.cshift.p, nullptr, h->num_sms, h->stream);
    launch_rotate(f.b.p, b_alt.p, p, (int)p, k, Tdev.p + 1024, nullptr, nullptr, h->num_sms, h->stream);
    f.e.swap(e_alt); f.b.swap(b_alt);
    // ---- reductions of the sweep epilogue: b'tilde (:549), e.y (:536), |beta0 - b|^2 (:662), column sums of e (:652)
    launch_pair_reduce(f.b.p, tilde.p, p, p, (int)p, k, 0, red.p, h->stream);
    launch_pair_reduce(f.e.p, f.y.p, ld, ld, (int)n, k, 0, red2.p, h->stream);
    launch_pair_reduce(b_old.p, f.b.p, p, p, (int)p, k, 1, red.p + (size_t)k * k, h->stream);
    launch_pair_reduce(f.e.p, nullptr, ld, ld, (int)n, k, 2, red.p + (size_t)k * k + k, h->stream);
    h->launches += 6;
    if (dist) {  // e.y and the column sums of e run over individuals; b'tilde and |beta0 - b|^2 are the same on every rank
      NC(nccl().AllReduce(red2.p, red2.p, (size_t)k * k, ncclDouble, ncclSum, h->comm, h->stream));
      NC(nccl().AllReduce(red.p + (size_t)k * k + k, red.p + (size_t)k * k + k, (size_t)k, ncclDouble, ncclSum, h->comm, h->stream));
    }
    std::vector<double> ey((size_t)k * k), small(2 * k);
    CU(cudaMemcpyAsync(hred.data(), red.p, sizeof(double) * ((size_t)k * k + 2 * k), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(ey.data(), red2.p, sizeof(double) * k * k, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) TildeHat[M(i, j)] = hred[(size_t)i * k + j];
    for (int t = 0; t < 2 * k; t++) small[t] = hred[(size_t)k * k + t];
    rc = check_err_flag(h, "MRR3 sweep");
    if (rc) return rc;
    // ---- variance components (:536-648), double
    mrr_residual_var(F, k, ey.data(), k + 1, V);  // e.y of trait t: the diagonal of the k x k products
    { const std::vector<double> Tr((size_t)k, TrXSX); mrr_varcomp(F, k, TildeHat, Tr, V.h2, V); }
    if (F.updateMu) {  // :651-655 (complete Y: Z = 1)
      std::vector<float> sh(k);
      for (int t = 0; t < k; t++) { const double m = small[k + t] / ((double)ng - 1.0); V.mu[t] += m; sh[t] = (float)(-m); }
      // e -= m: a rotation by the identity with a shift
      std::vector<float> I((size_t)k * k, 0.0f);
      for (int t = 0; t < k; t++) I[(size_t)t * k + t] = 1.0f;
      CU(cudaMemcpyAsync(Tdev.p, I.data(), sizeof(float) * k * k, cudaMemcpyHostToDevice, h->stream));
      CU(cudaMemcpyAsync(f.cshift.p, sh.data(), sizeof(float) * k, cudaMemcpyHostToDevice, h->stream));
      launch_rotate(f.e.p, e_alt.p, ld, (int)n, k, Tdev.p, f.cshift.p, nullptr, h->num_sms, h->stream);
      f.e.swap(e_alt);
      CU(cudaStreamSynchronize(h->stream));
    }
    if (!mrr_record(F, k, small.data(), vb0, h20, V)) break;
  }
  // ---- outputs (:676-700): hat = X_c b + mu = X b + (mu - sum_j mean_j b_j)
  std::vector<float> hb((size_t)k * p), m0(k), hh;
  CU(cudaMemcpyAsync(hb.data(), f.b.p, sizeof(float) * k * p, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  for (int t = 0; t < k; t++) {
    double shift = 0;
    for (int64_t j = 0; j < p; j++) shift += (h->h_sx[j] / (double)ng) * (double)hb[(size_t)t * p + j];
    m0[t] = (float)(V.mu[t] - shift);
  }
  rc = fitted_values(h, k, f.b.p, false, m0.data(), hh);
  if (rc) return rc;
  if (hat_out) for (size_t i = 0; i < hh.size(); i++) hat_out[i] = hh[i];
  if (b_out) for (size_t i = 0; i < hb.size(); i++) b_out[i] = hb[i];
  if (W_out) for (size_t i = 0; i < (size_t)k * p; i++) W_out[i] = 1.0;
  mrr_copy_out(F, k, V, out);
  dump_trace(h);
  return 0;
}

// ---- row sharding over the GPUs of a node ------------------------------------------------------------------------------
int bwgr_dist_unique_id(void* id128) {
  if (!id128) return fail(BWGR_ERR_ARG, "null argument");
  if (!nccl().ok) return fail(BWGR_ERR_UNSUPPORTED, "libnccl.so.2 not found");
  ncclUniqueId id;
  NC(nccl().GetUniqueId(&id));
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  memcpy(id128, &id, 128);
  return 0;
}

int bwgr_dist_init(bwgr_handle* h, int rank, int world, const void* id128, void* ipc_out) {
  if (!h || !id128 || !ipc_out) return fail(BWGR_ERR_ARG, "null argument");
  if (world < 2 || world > 8 || rank < 0 || rank >= world) return fail(BWGR_ERR_ARG, "need 2 <= world <= 8 and 0 <= rank < world");
  if (!nccl().ok) return fail(BWGR_ERR_UNSUPPORTED, "libnccl.so.2 not found");
  if (h->p) return fail(BWGR_ERR_STATE, "bwgr_dist_init must precede bwgr_geno_load_*");
  CU(cudaSetDevice(h->device));
  ncclUniqueId id;
  memcpy(&id, id128, 128);
  NC(nccl().CommInitRank(&h->comm, world, id, rank));
  if (nccl().CommSplit && nccl().CommSplit(h->comm, 0, rank, &h->comm_side, nullptr) != ncclSuccess) h->comm_side = nullptr;
  h->hx_own.cacheable = false;  // peers map it (cudaIpc): never handed to another owner
  if (h->hx_own.alloc((size_t)8 * world * 32 * 128) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc(exchange ring) failed");
  CU(cudaMemset(h->hx_own.p, 0, sizeof(unsigned long long) * h->hx_own.n));
  cudaIpcMemHandle_t mh;
  CU(cudaIpcGetMemHandle(&mh, h->hx_own.p));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(ipc_out, &mh, 64);
  h->world = world; h->rank = rank; h->dist_gen = 0; h->hx_connected = false;
  return 0;
}

int bwgr_dist_connect(bwgr_handle* h, const void* ipc_all) {
  if (!h || !ipc_all) return fail(BWGR_ERR_ARG, "null argument");
  if (h->world < 2) return fail(BWGR_ERR_STATE, "bwgr_dist_init first");
  CU(cudaSetDevice(h->device));
  for (int r = 0; r < h->world; r++) {
    if (r == h->rank) { h->hx[r] = h->hx_own.p; continue; }
    cudaIpcMemHandle_t mh;
    memcpy(&mh, static_cast<const unsigned char*>(ipc_all) + 64 * r, 64);
    void* ptr = nullptr;
    CU(cudaIpcOpenMemHandle(&ptr, mh, cudaIpcMemLazyEnablePeerAccess));
    h->hx[r] = static_cast<unsigned long long*>(ptr);
  }
  h->hx_connected = true;
  return 0;
}

int bwgr_profile(bwgr_handle* h, int enable) {
  if (!h) return fail(BWGR_ERR_ARG, "null handle");
  h->prof_collect();
  if (enable) { for (int c = 0; c < 4; c++) { h->prof_ms[c] = 0; h->prof_n[c] = 0; } }
  h->profiling = enable != 0;
  return 0;
}
int bwgr_profile_read(bwgr_handle* h, double* ms, int64_t* counts) {
  if (!h) return fail(BWGR_ERR_ARG, "null handle");
  CU(cudaStreamSynchronize(h->stream));
  h->prof_collect();
  for (int c = 0; c < 4; c++) { if (ms) ms[c] = h->prof_ms[c]; if (counts) counts[c] = h->prof_n[c]; }
  return 0;
}

// The band the pipelined sweep consumes, produced by the SAME dispatch as in a fit (FP4 shadow when the store has one):
// out [nblocks][128][256] floats, row r of block b = [x_{b,r}'X_b | x_{b-1,r}'X_b].  *kind_out: 4 = FP4 path, 8 = E4M3 / int8 path.
int bwgr_debug_gram_band(bwgr_handle* h, const int32_t* perm, float* gram_out, int* kind_out) {
  if (h && h->storage == BWGR_STORE_F32) return fail(BWGR_ERR_UNSUPPORTED, "the Gram kernels read the integer stores");
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (h->storage != BWGR_STORE_I8) return fail(BWGR_ERR_UNSUPPORTED, "Gram kernel needs the int8 store");
  CU(cudaSetDevice(h->device));
  const int64_t p = h->p;
  const int nblocks = (int)((p + kBlk - 1) / kBlk);
  DevBuf<int> dperm;
  DevBuf<float> dg;
  if (dperm.alloc(p) != cudaSuccess || dg.alloc((size_t)nblocks * kBlk * kBlk * 2) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  CU(cudaMemcpyAsync(dperm.p, perm, sizeof(int) * p, cudaMemcpyHostToDevice, h->stream));
  if (h->x2f.p) {
    const cudaError_t ge = launch_gram_fp4(h->x2f.p, h->ld, (int)p, (int)h->n, dperm.p, nblocks, dg.p, h->err.p, h->num_sms, nullptr, h->stream);
    if (ge != cudaSuccess) return fail(BWGR_ERR_CUDA, "FP4 Gram launch failed: %s", cudaGetErrorString(ge));
  } else {
    launch_gram_tc(gram_view(h), dperm.p, nblocks, dg.p, 1, 2, h->fp8_codes, h->err.p, h->num_sms, nullptr, h->stream);
  }
  if (kind_out) *kind_out = h->x2f.p ? 4 : 8;
  h->launches++;
  CU(cudaMemcpyAsync(gram_out, dg.p, sizeof(float) * dg.n, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return check_err_flag(h, "gram band");
}

int bwgr_debug_gram(bwgr_handle* h, const int32_t* perm, int block, int32_t* gram_out) {
  if (h && h->storage == BWGR_STORE_F32) return fail(BWGR_ERR_UNSUPPORTED, "the Gram kernels read the integer stores");
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (block != kBlk) return fail(BWGR_ERR_UNSUPPORTED, "only block=%d is built", kBlk);
  if (h->storage != BWGR_STORE_I8) return fail(BWGR_ERR_UNSUPPORTED, "Gram kernel needs the int8 store");
  CU(cudaSetDevice(h->device));
  const int64_t p = h->p;
  const int nblocks = (int)((p + kBlk - 1) / kBlk);
  DevBuf<int> dperm;
  DevBuf<int32_t> dg;
  if (dperm.alloc(p) != cudaSuccess || dg.alloc((size_t)nblocks * kBlk * kBlk) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  CU(cudaMemcpyAsync(dperm.p, perm, sizeof(int) * p, cudaMemcpyHostToDevice, h->stream));
  launch_gram_tc(gram_view(h), dperm.p, nblocks, dg.p, 0, 1, h->fp8_codes, h->err.p, h->num_sms, nullptr, h->stream);
  h->launches++;
  CU(cudaMemcpyAsync(gram_out, dg.p, sizeof(int32_t) * dg.n, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return check_err_flag(h, "gram");
}

}  // extern "C"
