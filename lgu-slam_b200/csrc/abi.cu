// abi.cu -- library identification + error plumbing of the C ABI (include/lgu_corr.h).
#include <array>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <unordered_map>
#include <vector>
#define LGU_STR2(x) #x
#define LGU_STR(x) LGU_STR2(x)
#include "common.cuh"

namespace lgu {
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return LGU_ERR_LAUNCH;
  }
  return LGU_OK;
}

// ---- one-time launch plumbing ------------------------------------------------------------------------------------
static std::mutex g_plumb_mutex;

int optin_smem(const void* kernel, int bytes, const char* who) {
  struct Done { int dev; const void* kernel; int bytes; };
  static std::vector<Done> done;                                // a few dozen (device, kernel) pairs at most
  int dev = 0;
  cudaGetDevice(&dev);
  {
    std::lock_guard<std::mutex> lk(g_plumb_mutex);
    for (const auto& d : done)
      if (d.dev == dev && d.kernel == kernel && d.bytes >= bytes) return LGU_OK;
  }
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) {
    set_error("%s: cannot opt in to %d B of shared memory: %s", who, bytes, cudaGetErrorString(e));
    return LGU_ERR_LAUNCH;
  }
  std::lock_guard<std::mutex> lk(g_plumb_mutex);
  for (auto& d : done)
    if (d.dev == dev && d.kernel == kernel) { d.bytes = bytes; return LGU_OK; }
  done.push_back({dev, kernel, bytes});
  return LGU_OK;
}

namespace {
// The device, then every argument that reaches the encoder: rank-dependent entries past `rank` stay zero.
constexpr int kMaxRank = 5;
typedef std::array<uint64_t, 6 + 3 * kMaxRank> MapKey;
struct KeyHash {
  size_t operator()(const MapKey& k) const {
    uint64_t h = 1469598103934665603ull;
    for (uint64_t x : k) h = (h ^ x) * 1099511628211ull;
    return (size_t)h;
  }
};
constexpr size_t kMapCacheMax = 512;
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
}  // namespace

int encode_tensor_map(CUtensorMap* map, CUtensorMapDataType dt, int rank, const void* base, const uint64_t* dims,
                      const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle swz, CUtensorMapL2promotion l2) {
  static std::unordered_map<MapKey, CUtensorMap, KeyHash> cache;
  static const EncodeTiledFn encode = [] {                       // resolved once; static initialisation is thread-safe
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
                    q == cudaDriverEntryPointSuccess;
    return ok ? reinterpret_cast<EncodeTiledFn>(p) : nullptr;
  }();
  if (rank < 1 || rank > kMaxRank) {
    set_error("encode_tensor_map: rank %d is outside 1..%d", rank, kMaxRank);
    return LGU_ERR_LAUNCH;
  }
  int dev = 0;
  cudaGetDevice(&dev);
  MapKey key{(uint64_t)dev, (uint64_t)reinterpret_cast<uintptr_t>(base), (uint64_t)dt, (uint64_t)rank, (uint64_t)swz,
             (uint64_t)l2};
  for (int i = 0; i < rank; ++i) {
    key[6 + i] = dims[i];
    key[6 + kMaxRank + i] = box[i];
  }
  for (int i = 0; i + 1 < rank; ++i) key[6 + 2 * kMaxRank + i] = strides_bytes[i];
  {
    std::lock_guard<std::mutex> lk(g_plumb_mutex);
    auto it = cache.find(key);
    if (it != cache.end()) {
      *map = it->second;
      return LGU_OK;
    }
  }
  if (encode == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return LGU_ERR_LAUNCH;
  }
  const cuuint32_t elem_strides[kMaxRank] = {1, 1, 1, 1, 1};
  const CUresult r = encode(map, dt, (cuuint32_t)rank, const_cast<void*>(base), dims, strides_bytes, box, elem_strides,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, swz, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char d[128];
    int n = 0;
    for (int i = 0; i < rank; ++i) n += snprintf(d + n, sizeof(d) - n, i ? " x %llu" : "%llu", (unsigned long long)dims[i]);
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d, dims %s)", (int)r, rank, d);
    return LGU_ERR_LAUNCH;
  }
  std::lock_guard<std::mutex> lk(g_plumb_mutex);
  if (cache.size() >= kMapCacheMax) cache.clear();               // geometry churn: start over (maps are cheap to redo)
  cache[key] = *map;
  return LGU_OK;
}

int num_sms() {
  struct Known { int dev, sms; };
  static std::vector<Known> known;
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  {
    std::lock_guard<std::mutex> lk(g_plumb_mutex);
    for (const auto& k : known)
      if (k.dev == dev) return k.sms;
  }
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return kNumSMs;
  std::lock_guard<std::mutex> lk(g_plumb_mutex);
  known.push_back({dev, sms});
  return sms;
}
}  // namespace lgu

extern "C" {
// ---- peer-visible device memory (the gathered output buffer of the sharded backend, lgu-slam_b200/sharded.py) ---------
int lgu_peer_alloc(long long bytes, void** ptr, void* handle64) {
  LGU_REQUIRE(bytes > 0 && ptr != nullptr && handle64 != nullptr, "lgu_peer_alloc: bad arguments");
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, (size_t)bytes);                 // a plain cudaMalloc allocation: exportable by CUDA IPC
  if (e != cudaSuccess) {
    lgu::set_error("lgu_peer_alloc: cudaMalloc(%lld) failed: %s", bytes, cudaGetErrorString(e));
    return LGU_ERR_LAUNCH;
  }
  cudaIpcMemHandle_t h;
  e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    lgu::set_error("lgu_peer_alloc: cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    return LGU_ERR_LAUNCH;
  }
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(handle64, &h, 64);
  *ptr = p;
  return LGU_OK;
}
int lgu_peer_open(const void* handle64, void** ptr) {
  LGU_REQUIRE(handle64 != nullptr && ptr != nullptr, "lgu_peer_open: bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  // opened with the CALLER's device current: the mapping (and peer access to the owning GPU) belongs to the device whose
  // kernels will store through it
  cudaError_t e = cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) {
    lgu::set_error("lgu_peer_open: cudaIpcOpenMemHandle failed: %s", cudaGetErrorString(e));
    return LGU_ERR_LAUNCH;
  }
  return LGU_OK;
}
int lgu_peer_close(void* ptr) {
  cudaError_t e = cudaIpcCloseMemHandle(ptr);
  if (e != cudaSuccess) {
    lgu::set_error("lgu_peer_close: %s", cudaGetErrorString(e));
    return LGU_ERR_LAUNCH;
  }
  return LGU_OK;
}
int lgu_peer_free(void* ptr) {
  cudaError_t e = cudaFree(ptr);
  if (e != cudaSuccess) {
    lgu::set_error("lgu_peer_free: %s", cudaGetErrorString(e));
    return LGU_ERR_LAUNCH;
  }
  return LGU_OK;
}

int lgu_abi_version(void) { return 1; }
const char* lgu_build_info(void) {
  return "lgu_corr sm_100a, nvcc " LGU_STR(__CUDACC_VER_MAJOR__) "." LGU_STR(__CUDACC_VER_MINOR__) ", built " __DATE__;
}
const char* lgu_last_error_string(void) { return lgu::g_err; }
}
