// Error plumbing, tensor-map encoding and device checks for libisx.
#include <stdarg.h>

#include "../../include/isx.h"
#include "isx_common.cuh"
#include "isx_internal.h"

static thread_local char g_err[1024] = "";

void isx_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* isx_last_error(void) { return g_err; }
extern "C" int isx_version(void) { return ISX_VERSION; }

extern "C" int isx_device_check(int device) {
  int count = 0;
  ISX_CHECK_CUDA(cudaGetDeviceCount(&count));
  ISX_REQUIRE(device >= 0 && device < count, "isx_device_check: device %d not present (%d visible)", device, count);
  cudaDeviceProp prop;
  ISX_CHECK_CUDA(cudaGetDeviceProperties(&prop, device));
  ISX_REQUIRE(prop.major == 10, "isx: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
              prop.major, prop.minor);
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Peer memory (BASELINE config 3: the feature rows of every rank land in every rank's matrix).  A rank exports the
// cudaMalloc allocation behind its row matrix as a 64-byte IPC handle, the other ranks of the box map it into their own
// address space (peer access over NVLink / NVSwitch enabled lazily by the driver) and PUSH their rows into it with plain
// device-to-device copies -- copy engines, no SM, no collective kernel competing with the persistent conv CTAs.
// ---------------------------------------------------------------------------------------------
extern "C" int isx_ipc_export(const void* ptr, void* handle64, int64_t* offset) {
  ISX_REQUIRE(ptr && handle64 && offset, "isx_ipc_export: null pointer");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  // the handle names the whole allocation: report where `ptr` lies inside it
  typedef CUresult (*RangeFn)(CUdeviceptr*, size_t*, CUdeviceptr);
  static RangeFn range = nullptr;
  if (!range) {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuMemGetAddressRange", &f, cudaEnableDefault, &qres);
    ISX_REQUIRE(e == cudaSuccess && qres == cudaDriverEntryPointSuccess && f, "isx_ipc_export: cuMemGetAddressRange unavailable");
    range = reinterpret_cast<RangeFn>(f);
  }
  CUdeviceptr base = 0;
  size_t size = 0;
  ISX_REQUIRE(range(&base, &size, reinterpret_cast<CUdeviceptr>(ptr)) == CUDA_SUCCESS, "isx_ipc_export: %p is not a device allocation", ptr);
  cudaIpcMemHandle_t h;
  ISX_CHECK_CUDA(cudaIpcGetMemHandle(&h, reinterpret_cast<void*>(base)));
  memcpy(handle64, &h, 64);
  *offset = static_cast<int64_t>(reinterpret_cast<CUdeviceptr>(ptr) - base);
  return 0;
}

extern "C" int isx_ipc_open(const void* handle64, void** base_out) {
  ISX_REQUIRE(handle64 && base_out, "isx_ipc_open: null pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  ISX_CHECK_CUDA(cudaIpcOpenMemHandle(base_out, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}

extern "C" int isx_copy_d2d_async(void* dst, const void* src, int64_t bytes, isx_stream stream) {
  ISX_REQUIRE(dst && src && bytes >= 0, "isx_copy_d2d_async: bad arguments");
  ISX_CHECK_CUDA(cudaMemcpyAsync(dst, src, static_cast<size_t>(bytes), cudaMemcpyDeviceToDevice, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

extern "C" int isx_ipc_close(void* base) {
  ISX_REQUIRE(base, "isx_ipc_close: null pointer");
  ISX_CHECK_CUDA(cudaIpcCloseMemHandle(base));
  return 0;
}

// cuTensorMapEncodeTiled is fetched through the runtime so that libisx.so does not link libcuda
// (the library must load -- symbols only -- on a box without a driver for the CPU test tier).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || p == nullptr) {
    isx_set_error("cuTensorMapEncodeTiled not available from the driver (%s)", cudaGetErrorString(e));
    return nullptr;
  }
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

int isx_make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                       const uint64_t* strides_bytes, const uint32_t* box, bool swizzle128, const uint32_t* elem_strides) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return 3;
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bx[5];
  cuuint32_t es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = elem_strides ? elem_strides[i] : 1;
  }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) {
    isx_set_error("tensor map base %p is not 16-byte aligned", base);
    return 3;
  }
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    isx_set_error("cuTensorMapEncodeTiled failed (CUresult %d) rank=%d dims=[%llu,%llu,%llu,%llu] box=[%u,%u,%u,%u]",
                  (int)r, rank, (unsigned long long)dims[0], rank > 1 ? (unsigned long long)dims[1] : 0ull,
                  rank > 2 ? (unsigned long long)dims[2] : 0ull, rank > 3 ? (unsigned long long)dims[3] : 0ull, box[0],
                  rank > 1 ? box[1] : 0u, rank > 2 ? box[2] : 0u, rank > 3 ? box[3] : 0u);
    return 3;
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------
// contexts (handles): options, launch counter, per-family CUDA-event timing, SM count
// ---------------------------------------------------------------------------------------------
#include <vector>

struct IsxProfRec { cudaEvent_t e0, e1; int family; double work; };
struct IsxProfiler {
  bool on = false;
  std::vector<IsxProfRec> recs;
  std::vector<cudaEvent_t> pool;
  size_t pool_next = 0;
  cudaEvent_t open[ISX_PROF_FAMILIES];
  double open_work[ISX_PROF_FAMILIES];
  bool is_open[ISX_PROF_FAMILIES] = {};
  cudaEvent_t event() {
    if (pool_next == pool.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      pool.push_back(e);
    }
    return pool[pool_next++];
  }
};
static const size_t kMaxRecs = 32768;

static thread_local IsxContext* t_current = nullptr;   // bound with isx_make_current
static thread_local IsxContext* t_default = nullptr;   // this thread's private default context

static void query_device(IsxContext* c, int device) {
  c->device = device;
  int sms = 0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) c->num_sms = sms;
  cudaGetLastError();  // a thread without a usable device keeps the B200 default; the first launch reports the real error
}

IsxContext* isx_ctx() {
  if (t_current) return t_current;
  if (!t_default) {
    t_default = new IsxContext();
    t_default->prof = new IsxProfiler();
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) query_device(t_default, dev);
    cudaGetLastError();
  }
  return t_default;
}

extern "C" int isx_create(int device, isx_handle* out) {
  ISX_REQUIRE(out != nullptr, "isx_create: null handle pointer");
  if (int rc = isx_device_check(device)) return rc;
  IsxContext* c = new IsxContext();
  c->prof = new IsxProfiler();
  query_device(c, device);
  *out = c;
  return 0;
}

extern "C" int isx_destroy(isx_handle h) {
  IsxContext* c = static_cast<IsxContext*>(h);
  if (!c) return 0;
  if (t_current == c) t_current = nullptr;
  for (cudaEvent_t e : c->prof->pool) cudaEventDestroy(e);
  delete c->prof;
  delete c;
  return 0;
}

extern "C" int isx_make_current(isx_handle h) {
  t_current = static_cast<IsxContext*>(h);   // NULL: back to the thread's default context
  return 0;
}

extern "C" int isx_sm_count(void) { return isx_ctx()->num_sms; }

void isx_prof_begin(int family, double work, cudaStream_t s) {
  IsxProfiler& P = *isx_ctx()->prof;
  if (!P.on || P.recs.size() >= kMaxRecs) return;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(s, &cs);
  if (cs != cudaStreamCaptureStatusNone) return;
  P.open[family] = P.event();
  P.open_work[family] = work;
  P.is_open[family] = true;
  cudaEventRecord(P.open[family], s);
}
void isx_prof_end(int family, cudaStream_t s) {
  IsxProfiler& P = *isx_ctx()->prof;
  if (!P.on || !P.is_open[family]) return;
  IsxProfRec r;
  r.e0 = P.open[family];
  r.e1 = P.event();
  r.family = family;
  r.work = P.open_work[family];
  cudaEventRecord(r.e1, s);
  P.recs.push_back(r);
  P.is_open[family] = false;
}

extern "C" unsigned long long isx_launch_count(void) { return isx_ctx()->launches; }
extern "C" int isx_prof_enable(int on) {
  IsxProfiler& P = *isx_ctx()->prof;
  P.on = on != 0;
  P.recs.clear();
  P.pool_next = 0;
  for (int f = 0; f < ISX_PROF_FAMILIES; ++f) P.is_open[f] = false;
  return 0;
}
// After a device synchronisation: per family {launches, total ms, total work (FLOPs or bytes)}; out[3*family + k].
extern "C" int isx_prof_collect(double* out, int n_out) {
  ISX_REQUIRE(out && n_out >= 3 * ISX_PROF_FAMILIES, "isx_prof_collect: need %d doubles", 3 * ISX_PROF_FAMILIES);
  IsxProfiler& P = *isx_ctx()->prof;
  for (int i = 0; i < 3 * ISX_PROF_FAMILIES; ++i) out[i] = 0.0;
  for (const IsxProfRec& r : P.recs) {
    float ms = 0.f;
    ISX_CHECK_CUDA(cudaEventElapsedTime(&ms, r.e0, r.e1));
    out[3 * r.family + 0] += 1.0;
    out[3 * r.family + 1] += ms;
    out[3 * r.family + 2] += r.work;
  }
  P.recs.clear();
  P.pool_next = 0;
  return 0;
}
