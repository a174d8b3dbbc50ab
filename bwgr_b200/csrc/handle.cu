// handle.cu -- the handle's life cycle and tuning, the device error flag, the all-reduce of host values, row sharding over the GPUs
// of a node, per-kernel profiling and the Gram debug entry points.
#include <dlfcn.h>
#include <cstdarg>

#include "host.h"

using namespace bwgr;
using namespace bwgr::host;

static thread_local std::string g_err;

namespace bwgr::host {

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

BlockCache& block_cache() { static BlockCache* c = new BlockCache; return *c; }  // never destroyed: no CUDA calls at process exit

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

}  // namespace bwgr::host

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

// The Gram debug entry points: the store checks, the permutation upload, the launch -- band: the float band the pipelined sweep
// consumes, by the same dispatch as in a fit; else the int32 diagonal blocks -- the read-back and the device error flag.
static int debug_gram(bwgr_handle* h, const int32_t* perm, int block, bool band, void* out, int* kind_out) {
  if (h && h->storage == BWGR_STORE_F32) return fail(BWGR_ERR_UNSUPPORTED, "the Gram kernels read the integer stores");
  if (!h || !h->p) return fail(BWGR_ERR_STATE, "no genotypes loaded");
  if (block != kBlk) return fail(BWGR_ERR_UNSUPPORTED, "only block=%d is built", kBlk);
  if (h->storage != BWGR_STORE_I8) return fail(BWGR_ERR_UNSUPPORTED, "Gram kernel needs the int8 store");
  CU(cudaSetDevice(h->device));
  const int64_t p = h->p;
  const int nblocks = (int)((p + kBlk - 1) / kBlk);
  DevBuf<int> dperm;
  DevBuf<float> dg;  // float (band) or int32 words
  if (dperm.alloc(p) != cudaSuccess || dg.alloc((size_t)nblocks * kBlk * kBlk * (band ? 2 : 1)) != cudaSuccess) return fail(BWGR_ERR_CUDA, "cudaMalloc failed");
  CU(cudaMemcpyAsync(dperm.p, perm, sizeof(int) * p, cudaMemcpyHostToDevice, h->stream));
  if (band && h->x2f.p) {
    const cudaError_t ge = launch_gram_fp4(h->x2f.p, h->ld, (int)p, (int)h->n, dperm.p, nblocks, dg.p, h->err.p, h->num_sms, nullptr, h->stream);
    if (ge != cudaSuccess) return fail(BWGR_ERR_CUDA, "FP4 Gram launch failed: %s", cudaGetErrorString(ge));
  } else {
    launch_gram_tc(h->gram_view(), dperm.p, nblocks, dg.p, band ? 1 : 0, band ? 2 : 1, h->fp8_codes, h->err.p, h->num_sms, nullptr, h->stream);
  }
  if (kind_out) *kind_out = h->x2f.p ? 4 : 8;
  h->launches++;
  CU(cudaMemcpyAsync(out, dg.p, sizeof(float) * dg.n, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return check_err_flag(h, band ? "gram band" : "gram");
}

// out [nblocks][128][256] floats, row r of block b = [x_{b,r}'X_b | x_{b-1,r}'X_b].  *kind_out: 4 = FP4 path, 8 = E4M3 / int8 path.
int bwgr_debug_gram_band(bwgr_handle* h, const int32_t* perm, float* gram_out, int* kind_out) { return debug_gram(h, perm, kBlk, true, gram_out, kind_out); }
int bwgr_debug_gram(bwgr_handle* h, const int32_t* perm, int block, int32_t* gram_out) { return debug_gram(h, perm, block, false, gram_out, nullptr); }

}  // extern "C"
