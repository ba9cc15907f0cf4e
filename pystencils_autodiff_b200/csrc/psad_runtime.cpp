// psad_runtime.cpp — host runtime behind include/psad.h.
//
// Replaces, for the torch_native path of the reference, the generated C++ wrapper + pybind11 module + nvcc JIT
// (/root/reference/src/pystencils_autodiff/backends/astnodes.py:95-186, framework_integration/printer.py:88-145):
// specialised CUDA source -> NVRTC -> sm_100a cubin (content-addressed on-disk cache, like the reference's md5
// keyed object cache, backends/astnodes.py:157-166) -> cuModuleLoadData -> cuLaunchKernel on the caller's stream
// with tensor maps encoded per launch.  libcuda / libnvrtc / libnccl are dlopen'ed lazily so that the library
// loads (and compiles cubins) on a machine without a GPU.
#include "../../include/psad.h"

#include <dlfcn.h>
#include <sys/stat.h>
#include <unistd.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "kernels/psad_args.h"

// NVTX ranges around compile / launch / halo exchange (header-only NVTX 3: the calls are a null-pointer test until a
// profiler injects itself, so they stay in the launch path unconditionally).  Without the CUDA headers they vanish.
#if defined(__has_include)
#if __has_include(<nvtx3/nvToolsExt.h>)
#include <nvtx3/nvToolsExt.h>
#define PSAD_HAVE_NVTX 1
#endif
#endif
struct NvtxRange {
#ifdef PSAD_HAVE_NVTX
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
#else
  explicit NvtxRange(const char*) {}
#endif
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};

// ---------------------------------------------------------------------------------------------------------------
// error handling
static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...) {
  char buf[4096];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

extern "C" const char* psad_last_error(void) { return g_err.c_str(); }
extern "C" int psad_abi_version(void) { return PSAD_ABI_VERSION; }
extern "C" void psad_free(void* p) { free(p); }

// ---------------------------------------------------------------------------------------------------------------
// minimal driver-API / NVRTC / NCCL declarations (resolved with dlsym; no CUDA headers needed to build)
typedef int CUresult;
typedef int CUdevice;
typedef struct CUctx_st* CUcontext;
typedef struct CUmod_st* CUmodule;
typedef struct CUfunc_st* CUfunction;
typedef struct CUstream_st* CUstream;
typedef unsigned long long CUdeviceptr;
struct alignas(64) CUtensorMap { unsigned long long opaque[16]; };
struct CUipcMemHandle { char reserved[64]; };
enum { CU_IPC_MEM_LAZY_ENABLE_PEER_ACCESS = 1 };

enum { CU_DEVICE_ATTRIBUTE_MULTIPROCESSOR_COUNT = 16, CU_DEVICE_ATTRIBUTE_COMPUTE_CAPABILITY_MAJOR = 75,
       CU_DEVICE_ATTRIBUTE_COMPUTE_CAPABILITY_MINOR = 76, CU_DEVICE_ATTRIBUTE_MAX_SHARED_MEMORY_PER_BLOCK_OPTIN = 97 };
enum { CU_FUNC_ATTRIBUTE_SHARED_SIZE_BYTES = 1, CU_FUNC_ATTRIBUTE_LOCAL_SIZE_BYTES = 3, CU_FUNC_ATTRIBUTE_NUM_REGS = 4,
       CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES = 8 };
enum { CU_TENSOR_MAP_DATA_TYPE_FLOAT16 = 6, CU_TENSOR_MAP_DATA_TYPE_FLOAT32 = 7, CU_TENSOR_MAP_DATA_TYPE_FLOAT64 = 8 };

struct Driver {
  void* lib = nullptr;
  CUresult (*cuInit)(unsigned);
  CUresult (*cuDeviceGet)(CUdevice*, int);
  CUresult (*cuDeviceGetAttribute)(int*, int, CUdevice);
  CUresult (*cuCtxGetCurrent)(CUcontext*);
  CUresult (*cuCtxSetCurrent)(CUcontext);
  CUresult (*cuCtxGetDevice)(CUdevice*);
  CUresult (*cuCtxPushCurrent)(CUcontext);
  CUresult (*cuCtxPopCurrent)(CUcontext*);
  CUresult (*cuDevicePrimaryCtxRetain)(CUcontext*, CUdevice);
  CUresult (*cuModuleLoadData)(CUmodule*, const void*);
  CUresult (*cuModuleUnload)(CUmodule);
  CUresult (*cuModuleGetFunction)(CUfunction*, CUmodule, const char*);
  CUresult (*cuFuncSetAttribute)(CUfunction, int, int);
  CUresult (*cuFuncGetAttribute)(int*, int, CUfunction);
  CUresult (*cuOccupancyMaxActiveBlocksPerMultiprocessor)(int*, CUfunction, int, size_t);
  CUresult (*cuLaunchKernel)(CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned,
                             CUstream, void**, void**);
  CUresult (*cuGetErrorString)(CUresult, const char**);
  CUresult (*cuTensorMapEncodeTiled)(CUtensorMap*, int, unsigned, void*, const unsigned long long*,
                                     const unsigned long long*, const unsigned*, const unsigned*, int, int, int, int);
  // optional (peer halos): resolved separately so that an old driver still loads the library
  CUresult (*cuIpcGetMemHandle)(CUipcMemHandle*, CUdeviceptr) = nullptr;
  CUresult (*cuIpcOpenMemHandle)(CUdeviceptr*, CUipcMemHandle, unsigned) = nullptr;     // the handle travels by value
  CUresult (*cuIpcCloseMemHandle)(CUdeviceptr) = nullptr;
  CUresult (*cuMemGetAddressRange)(CUdeviceptr*, size_t*, CUdeviceptr) = nullptr;
  CUresult (*cuMemsetD32Async)(CUdeviceptr, unsigned, size_t, CUstream) = nullptr;
};
static Driver g_drv;
static std::once_flag g_drv_once;
static std::string g_drv_err;

template <typename T> static bool sym(void* lib, const char* name, T& fn, std::string& err) {
  fn = reinterpret_cast<T>(dlsym(lib, name));
  if (!fn) { err = std::string("missing symbol ") + name; return false; }
  return true;
}

static void load_driver() {
  void* lib = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) { g_drv_err = std::string("cannot load libcuda.so.1 (no NVIDIA driver on this machine): ") + dlerror(); return; }
  Driver d; d.lib = lib; std::string e;
  bool ok = sym(lib, "cuInit", d.cuInit, e) && sym(lib, "cuDeviceGet", d.cuDeviceGet, e) &&
            sym(lib, "cuDeviceGetAttribute", d.cuDeviceGetAttribute, e) && sym(lib, "cuCtxGetCurrent", d.cuCtxGetCurrent, e) &&
            sym(lib, "cuCtxSetCurrent", d.cuCtxSetCurrent, e) && sym(lib, "cuCtxGetDevice", d.cuCtxGetDevice, e) &&
            sym(lib, "cuCtxPushCurrent_v2", d.cuCtxPushCurrent, e) && sym(lib, "cuCtxPopCurrent_v2", d.cuCtxPopCurrent, e) &&
            sym(lib, "cuDevicePrimaryCtxRetain", d.cuDevicePrimaryCtxRetain, e) &&
            sym(lib, "cuModuleLoadData", d.cuModuleLoadData, e) && sym(lib, "cuModuleUnload", d.cuModuleUnload, e) &&
            sym(lib, "cuModuleGetFunction", d.cuModuleGetFunction, e) && sym(lib, "cuFuncSetAttribute", d.cuFuncSetAttribute, e) &&
            sym(lib, "cuFuncGetAttribute", d.cuFuncGetAttribute, e) &&
            sym(lib, "cuOccupancyMaxActiveBlocksPerMultiprocessor", d.cuOccupancyMaxActiveBlocksPerMultiprocessor, e) &&
            sym(lib, "cuLaunchKernel", d.cuLaunchKernel, e) && sym(lib, "cuGetErrorString", d.cuGetErrorString, e) &&
            sym(lib, "cuTensorMapEncodeTiled", d.cuTensorMapEncodeTiled, e);
  if (!ok) { g_drv_err = e; return; }
  {
    std::string ignore;   // optional: peer halos
    sym(lib, "cuIpcGetMemHandle", d.cuIpcGetMemHandle, ignore);
    sym(lib, "cuIpcOpenMemHandle_v2", d.cuIpcOpenMemHandle, ignore);
    sym(lib, "cuIpcCloseMemHandle", d.cuIpcCloseMemHandle, ignore);
    sym(lib, "cuMemGetAddressRange_v2", d.cuMemGetAddressRange, ignore);
    sym(lib, "cuMemsetD32Async", d.cuMemsetD32Async, ignore);
  }
  CUresult r = d.cuInit(0);
  if (r != 0) { g_drv_err = "cuInit failed with code " + std::to_string(r); return; }
  g_drv = d;
}

static int need_driver() {
  std::call_once(g_drv_once, load_driver);
  if (!g_drv.lib) return fail(PSAD_ERR_NO_DRIVER, "%s", g_drv_err.c_str());
  return 0;
}

static int cu_fail(CUresult r, const char* what) {
  const char* s = nullptr;
  if (g_drv.cuGetErrorString) g_drv.cuGetErrorString(r, &s);
  return fail(PSAD_ERR_CUDA, "%s failed: %s (CUresult %d)", what, s ? s : "?", r);
}
#define CU_CHECK(call) do { CUresult _r = (call); if (_r != 0) return cu_fail(_r, #call); } while (0)

// make sure the calling thread has a current context (torch's primary context when called from PyTorch).  A thread
// without one (an autograd worker that has not touched the runtime API yet) gets `preferred` — the context a kernel
// was loaded in — or, with no preference, the primary context of device 0.
static int ensure_context(CUcontext preferred = nullptr) {
  CUcontext ctx = nullptr;
  CU_CHECK(g_drv.cuCtxGetCurrent(&ctx));
  if (ctx) return 0;
  if (preferred) {
    CU_CHECK(g_drv.cuCtxSetCurrent(preferred));
    return 0;
  }
  CUdevice dev;
  CU_CHECK(g_drv.cuDeviceGet(&dev, 0));
  CU_CHECK(g_drv.cuDevicePrimaryCtxRetain(&ctx, dev));
  CU_CHECK(g_drv.cuCtxSetCurrent(ctx));
  return 0;
}

// NVRTC
typedef struct _nvrtcProgram* nvrtcProgram;
struct Nvrtc {
  void* lib = nullptr;
  int (*nvrtcCreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*);
  int (*nvrtcDestroyProgram)(nvrtcProgram*);
  int (*nvrtcCompileProgram)(nvrtcProgram, int, const char* const*);
  int (*nvrtcGetProgramLogSize)(nvrtcProgram, size_t*);
  int (*nvrtcGetProgramLog)(nvrtcProgram, char*);
  int (*nvrtcGetCUBINSize)(nvrtcProgram, size_t*);
  int (*nvrtcGetCUBIN)(nvrtcProgram, char*);
  const char* (*nvrtcGetErrorString)(int);
  int (*nvrtcVersion)(int*, int*);
};
static Nvrtc g_rtc;
static std::once_flag g_rtc_once;
static std::string g_rtc_err;

static void load_nvrtc() {
  const char* names[] = {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so"};
  void* lib = nullptr;
  for (const char* n : names) { lib = dlopen(n, RTLD_NOW | RTLD_LOCAL); if (lib) break; }
  if (!lib) { g_rtc_err = std::string("cannot load libnvrtc: ") + dlerror(); return; }
  Nvrtc n; n.lib = lib; std::string e;
  bool ok = sym(lib, "nvrtcCreateProgram", n.nvrtcCreateProgram, e) && sym(lib, "nvrtcDestroyProgram", n.nvrtcDestroyProgram, e) &&
            sym(lib, "nvrtcCompileProgram", n.nvrtcCompileProgram, e) && sym(lib, "nvrtcGetProgramLogSize", n.nvrtcGetProgramLogSize, e) &&
            sym(lib, "nvrtcGetProgramLog", n.nvrtcGetProgramLog, e) && sym(lib, "nvrtcGetCUBINSize", n.nvrtcGetCUBINSize, e) &&
            sym(lib, "nvrtcGetCUBIN", n.nvrtcGetCUBIN, e) && sym(lib, "nvrtcGetErrorString", n.nvrtcGetErrorString, e) &&
            sym(lib, "nvrtcVersion", n.nvrtcVersion, e);
  if (!ok) { g_rtc_err = e; return; }
  g_rtc = n;
}

static int need_nvrtc() {
  std::call_once(g_rtc_once, load_nvrtc);
  if (!g_rtc.lib) return fail(PSAD_ERR_NO_DRIVER, "%s", g_rtc_err.c_str());
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// configuration
static std::mutex g_cfg_mutex;
static std::string g_include_dir, g_cache_dir;
static std::atomic<uint64_t> g_launches{0};

static void mkdir_p(const std::string& path) {
  std::string cur;
  for (size_t i = 0; i < path.size(); ++i) {
    cur += path[i];
    if (path[i] == '/' || i + 1 == path.size()) mkdir(cur.c_str(), 0755);
  }
}

extern "C" int psad_init(const char* kernel_include_dir, const char* cache_dir) {
  if (!kernel_include_dir || !cache_dir) return fail(PSAD_ERR_INVALID, "psad_init: null argument");
  std::lock_guard<std::mutex> lock(g_cfg_mutex);
  g_include_dir = kernel_include_dir;
  g_cache_dir = cache_dir;
  mkdir_p(g_cache_dir);
  struct stat st;
  if (stat((g_include_dir + "/psad_common.cuh").c_str(), &st) != 0)
    return fail(PSAD_ERR_IO, "psad_init: %s/psad_common.cuh not found", kernel_include_dir);
  return 0;
}

extern "C" uint64_t psad_launch_count(void) { return g_launches.load(); }

extern "C" int psad_device_info(int* device, int* sm_count, int* cc_major, int* cc_minor, size_t* smem_optin) {
  if (int rc = need_driver()) return rc;
  if (int rc = ensure_context()) return rc;
  CUdevice dev;
  CU_CHECK(g_drv.cuCtxGetDevice(&dev));
  int v;
  if (device) *device = dev;
  if (sm_count) { CU_CHECK(g_drv.cuDeviceGetAttribute(&v, CU_DEVICE_ATTRIBUTE_MULTIPROCESSOR_COUNT, dev)); *sm_count = v; }
  if (cc_major) { CU_CHECK(g_drv.cuDeviceGetAttribute(&v, CU_DEVICE_ATTRIBUTE_COMPUTE_CAPABILITY_MAJOR, dev)); *cc_major = v; }
  if (cc_minor) { CU_CHECK(g_drv.cuDeviceGetAttribute(&v, CU_DEVICE_ATTRIBUTE_COMPUTE_CAPABILITY_MINOR, dev)); *cc_minor = v; }
  if (smem_optin) { CU_CHECK(g_drv.cuDeviceGetAttribute(&v, CU_DEVICE_ATTRIBUTE_MAX_SHARED_MEMORY_PER_BLOCK_OPTIN, dev)); *smem_optin = (size_t)v; }
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// compilation + cubin cache
static bool read_file(const std::string& path, std::vector<char>& out) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) return false;
  fseek(f, 0, SEEK_END);
  long n = ftell(f);
  if (n < 0) { fclose(f); return false; }
  fseek(f, 0, SEEK_SET);
  out.resize((size_t)n);
  size_t got = n ? fread(out.data(), 1, (size_t)n, f) : 0;
  fclose(f);
  return got == (size_t)n;
}

static int compile_to_cache(const char* source, const char* cache_key, const char* const* options, int n_options,
                            int* cache_hit, char** log_out, std::string* cubin_path_out) {
  if (!source || !cache_key) return fail(PSAD_ERR_INVALID, "psad_compile: null argument");
  std::string inc, cache;
  {
    std::lock_guard<std::mutex> lock(g_cfg_mutex);
    inc = g_include_dir;
    cache = g_cache_dir;
  }
  if (inc.empty()) return fail(PSAD_ERR_INVALID, "psad_init() has not been called");
  const std::string path = cache + "/" + cache_key + ".cubin";
  if (cubin_path_out) *cubin_path_out = path;
  if (log_out) *log_out = nullptr;
  struct stat st;
  if (stat(path.c_str(), &st) == 0 && st.st_size > 0) {
    if (cache_hit) *cache_hit = 1;
    return 0;
  }
  if (cache_hit) *cache_hit = 0;
  if (int rc = need_nvrtc()) return rc;

  nvrtcProgram prog;
  std::string name = std::string(cache_key) + ".cu";
  int r = g_rtc.nvrtcCreateProgram(&prog, source, name.c_str(), 0, nullptr, nullptr);
  if (r != 0) return fail(PSAD_ERR_NVRTC, "nvrtcCreateProgram: %s", g_rtc.nvrtcGetErrorString(r));
  std::vector<std::string> opts = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo", "-I" + inc};
  for (int i = 0; i < n_options; ++i) opts.push_back(options[i]);
  std::vector<const char*> copts;
  for (auto& o : opts) copts.push_back(o.c_str());
  r = g_rtc.nvrtcCompileProgram(prog, (int)copts.size(), copts.data());
  size_t log_size = 0;
  g_rtc.nvrtcGetProgramLogSize(prog, &log_size);
  std::string log(log_size, '\0');
  if (log_size > 1) g_rtc.nvrtcGetProgramLog(prog, &log[0]);
  if (log_out && log_size > 1) *log_out = strdup(log.c_str());
  if (r != 0) {
    g_rtc.nvrtcDestroyProgram(&prog);
    return fail(PSAD_ERR_NVRTC, "NVRTC compilation of %s failed: %s\n%s", name.c_str(), g_rtc.nvrtcGetErrorString(r), log.c_str());
  }
  size_t n = 0;
  r = g_rtc.nvrtcGetCUBINSize(prog, &n);
  if (r != 0 || n == 0) { g_rtc.nvrtcDestroyProgram(&prog); return fail(PSAD_ERR_NVRTC, "nvrtcGetCUBINSize failed"); }
  std::vector<char> cubin(n);
  r = g_rtc.nvrtcGetCUBIN(prog, cubin.data());
  g_rtc.nvrtcDestroyProgram(&prog);
  if (r != 0) return fail(PSAD_ERR_NVRTC, "nvrtcGetCUBIN failed");

  mkdir_p(cache);
  const std::string tmp = path + ".tmp" + std::to_string((long)getpid());
  FILE* f = fopen(tmp.c_str(), "wb");
  if (!f) return fail(PSAD_ERR_IO, "cannot write %s", tmp.c_str());
  const size_t written = fwrite(cubin.data(), 1, n, f);
  if (fclose(f) != 0 || written != n) {
    unlink(tmp.c_str());
    return fail(PSAD_ERR_IO, "short write to %s (disk full?)", tmp.c_str());
  }
  if (rename(tmp.c_str(), path.c_str()) != 0) {
    unlink(tmp.c_str());
    return fail(PSAD_ERR_IO, "cannot rename %s", tmp.c_str());
  }
  // keep the specialised source beside the cubin (the reference keeps its generated .cu too)
  FILE* s = fopen((cache + "/" + cache_key + ".cu").c_str(), "w");
  if (s) { fputs(source, s); fclose(s); }
  return 0;
}

extern "C" int psad_compile(const char* source, const char* cache_key, const char* const* options, int n_options,
                            int* cache_hit, char** log) {
  NvtxRange nvtx("psad_compile");
  return compile_to_cache(source, cache_key, options, n_options, cache_hit, log, nullptr);
}

// ---------------------------------------------------------------------------------------------------------------
// kernel objects
// One remembered launch: what was passed (the key) and everything derived from it that does not depend on the scalars —
// the parameter block, the grid and the encoded tensor maps.  A time loop or an autograd Function launches the same
// kernel on the same few buffers over and over; re-validating the arguments and re-encoding every tensor map
// (cuTensorMapEncodeTiled) on each launch was most of the host cost of a launch.
struct LaunchKey {
  int n_fields;
  int has_range;
  int has_peer;
  psad_field_arg_t fields[PSAD_MAX_FIELDS];
  psad_range_t range;
  psad_peer_t peer;      // with expect zeroed: like the scalars it changes from launch to launch
};
struct alignas(64) TensorMaps { CUtensorMap m[3 * PSAD_MAX_FIELDS]; };   // peer kernels: [local | lower | upper neighbour]
struct LaunchEntry {
  LaunchKey key;
  PsadArgs args;
  unsigned grid[3];
  int empty;
  TensorMaps tm;
  unsigned long long stamp;
};
static const int PSAD_LAUNCH_CACHE = 16;

struct psad_kernel {
  psad_plan_t plan;
  CUmodule module = nullptr;
  CUfunction fn = nullptr;
  CUcontext ctx = nullptr;  // the context the module was loaded in
  int sm_count = 0;
  int occupancy = 1;  // resident CTAs per SM for this kernel (march: persistent grid = sm_count * occupancy)
  std::string name;
  std::mutex cache_mutex;                 // launches of one kernel may come from several threads (autograd workers)
  std::vector<LaunchEntry*> cache;        // most recently used launches, at most PSAD_LAUNCH_CACHE
  unsigned long long cache_clock = 0;
  ~psad_kernel() { for (LaunchEntry* e : cache) delete e; }
};
static std::atomic<unsigned long long> g_cache_hits{0}, g_cache_misses{0};

extern "C" int psad_kernel_create(const char* source, const char* kernel_name, const char* cache_key,
                                  const char* const* options, int n_options, const psad_plan_t* plan,
                                  psad_kernel_t* out) {
  if (!kernel_name || !plan || !out) return fail(PSAD_ERR_INVALID, "psad_kernel_create: null argument");
  if (plan->abi_version != PSAD_ABI_VERSION) return fail(PSAD_ERR_INVALID, "plan ABI version %d != %d", plan->abi_version, PSAD_ABI_VERSION);
  if (plan->n_fields < 1 || plan->n_fields > PSAD_MAX_FIELDS || plan->n_scalars < 0 || plan->n_scalars > PSAD_MAX_SCALARS ||
      plan->ndim < 1 || plan->ndim > 3 || plan->threads < 32 || plan->threads > 1024)
    return fail(PSAD_ERR_INVALID, "psad_kernel_create: plan out of range");
  std::string path;
  if (int rc = compile_to_cache(source, cache_key, options, n_options, nullptr, nullptr, &path)) return rc;
  if (int rc = need_driver()) return rc;
  if (int rc = ensure_context()) return rc;
  std::vector<char> cubin;
  if (!read_file(path, cubin)) return fail(PSAD_ERR_IO, "cannot read %s", path.c_str());
  psad_kernel* k = new psad_kernel();
  k->plan = *plan;
  k->name = kernel_name;
  g_drv.cuCtxGetCurrent(&k->ctx);
  CUresult r = g_drv.cuModuleLoadData(&k->module, cubin.data());
  if (r != 0) { delete k; return cu_fail(r, "cuModuleLoadData"); }
  r = g_drv.cuModuleGetFunction(&k->fn, k->module, kernel_name);
  if (r != 0) { g_drv.cuModuleUnload(k->module); delete k; return cu_fail(r, "cuModuleGetFunction"); }
  if (plan->smem_bytes > 48 * 1024) {
    r = g_drv.cuFuncSetAttribute(k->fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, plan->smem_bytes);
    if (r != 0) { g_drv.cuModuleUnload(k->module); delete k; return cu_fail(r, "cuFuncSetAttribute(max dynamic smem)"); }
  }
  CUdevice dev;
  g_drv.cuCtxGetDevice(&dev);
  g_drv.cuDeviceGetAttribute(&k->sm_count, CU_DEVICE_ATTRIBUTE_MULTIPROCESSOR_COUNT, dev);
  int occ = 0;
  if (g_drv.cuOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k->fn, plan->threads, (size_t)plan->smem_bytes) == 0 && occ > 0)
    k->occupancy = occ;
  if (plan->ctas_per_sm > 0 && plan->ctas_per_sm < k->occupancy) k->occupancy = plan->ctas_per_sm;
  *out = k;
  return 0;
}

extern "C" int psad_kernel_destroy(psad_kernel_t k) {
  if (!k) return 0;
  if (k->module && g_drv.lib) g_drv.cuModuleUnload(k->module);
  delete k;
  return 0;
}

extern "C" int psad_kernel_attributes(psad_kernel_t k, int* num_regs, int* static_smem, int* local_bytes,
                                      int* max_ctas_per_sm) {
  if (!k) return fail(PSAD_ERR_INVALID, "null kernel");
  if (num_regs) CU_CHECK(g_drv.cuFuncGetAttribute(num_regs, CU_FUNC_ATTRIBUTE_NUM_REGS, k->fn));
  if (static_smem) CU_CHECK(g_drv.cuFuncGetAttribute(static_smem, CU_FUNC_ATTRIBUTE_SHARED_SIZE_BYTES, k->fn));
  if (local_bytes) CU_CHECK(g_drv.cuFuncGetAttribute(local_bytes, CU_FUNC_ATTRIBUTE_LOCAL_SIZE_BYTES, k->fn));
  if (max_ctas_per_sm)
    CU_CHECK(g_drv.cuOccupancyMaxActiveBlocksPerMultiprocessor(max_ctas_per_sm, k->fn, k->plan.threads, (size_t)k->plan.smem_bytes));
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// launch
static inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }

// Everything a launch needs that does not touch the device: the parameter block (shapes, strides, iteration / write
// ranges), the work decomposition of march kernels and the grid.  *empty = 1 when there is nothing to write.
static int build_args(const psad_plan_t& P, const char* kname, int sm_count, int occupancy, const psad_field_arg_t* fields,
                      int n_fields, const double* scalars, int n_scalars, const psad_range_t* range, PsadArgs& A,
                      unsigned grid[3], int* empty) {
  if (n_fields != P.n_fields) return fail(PSAD_ERR_INVALID, "%s: expected %d fields, got %d", kname, P.n_fields, n_fields);
  if (n_scalars != P.n_scalars) return fail(PSAD_ERR_INVALID, "%s: expected %d scalars, got %d", kname, P.n_scalars, n_scalars);
  if (n_scalars > 0 && !scalars) return fail(PSAD_ERR_INVALID, "null scalars");
  const int nd = P.ndim;
  *empty = 0;
  grid[0] = grid[1] = grid[2] = 1;
  memset(&A, 0, sizeof(A));
  // normalise to (z, y, x): leading dims of extent 1
  for (int d = 0; d < 3; ++d) A.shape[d] = 1;
  for (int d = 0; d < nd; ++d) A.shape[3 - nd + d] = fields[0].shape[d];
  for (int f = 0; f < n_fields; ++f) {
    if (!fields[f].ptr) return fail(PSAD_ERR_INVALID, "%s: field %d has a null pointer", kname, f);
    for (int d = 0; d < nd; ++d) {
      if (fields[f].shape[d] != fields[0].shape[d])
        return fail(PSAD_ERR_INVALID, "%s: all fields of a kernel must share one spatial shape (field %d, dim %d: %lld vs %lld)",
                    kname, f, d, (long long)fields[f].shape[d], (long long)fields[0].shape[d]);
      A.stride[f][3 - nd + d] = fields[f].stride[d];
    }
    A.stride[f][3] = fields[f].stride[3];
    A.ptr[f] = fields[f].ptr;
  }
  for (int i = 0; i < n_scalars; ++i) A.scalar[i] = scalars[i];
  for (int d = 0; d < 3; ++d) { A.it_lo[d] = 0; A.it_hi[d] = A.shape[d]; A.wr_lo[d] = 0; A.wr_hi[d] = A.shape[d]; }
  if (range) {
    for (int d = 0; d < nd; ++d) {
      const int e = 3 - nd + d;
      A.it_lo[e] = range->iter_lo[d]; A.it_hi[e] = range->iter_hi[d];
      A.wr_lo[e] = range->write_lo[d]; A.wr_hi[e] = range->write_hi[d];
      if (A.wr_lo[e] < 0 || A.wr_hi[e] > A.shape[e])
        return fail(PSAD_ERR_INVALID, "%s: write range [%lld, %lld) outside the array extent %lld in dim %d", kname,
                    A.wr_lo[e], A.wr_hi[e], A.shape[e], d);
      // Evaluated cells read c + offset.  The generic kernel with interior iteration (boundary 0) reads unguarded, so
      // every evaluated cell must keep `ghost_layers` cells to each array edge; everywhere else out-of-array reads are
      // zero-filled (TMA boxes of the march kernels) or index-guarded ('zeros'), but the evaluated cell must exist.
      const long long margin = (P.boundary == 0 && P.kind == PSAD_KIND_GENERIC) ? P.ghost_layers : 0;
      if (A.it_hi[e] > A.it_lo[e] && (A.it_lo[e] < margin || A.it_hi[e] > A.shape[e] - margin))
        return fail(PSAD_ERR_INVALID, "%s: iteration range [%lld, %lld) in dim %d must lie inside [%lld, %lld) of the array "
                    "(extent %lld, %d ghost layers, boundary %s)", kname, A.it_lo[e], A.it_hi[e], d, margin,
                    A.shape[e] - margin, A.shape[e], P.ghost_layers, P.boundary == 0 ? "none" : "zeros");
    }
  } else if (P.boundary == 0 && P.ghost_layers > 0) {
    for (int d = 0; d < nd; ++d) {
      const int e = 3 - nd + d;
      A.it_lo[e] = P.ghost_layers;
      A.it_hi[e] = A.shape[e] - P.ghost_layers;
    }
  }
  for (int d = 0; d < 3; ++d) {
    if (A.it_hi[d] < A.it_lo[d]) A.it_hi[d] = A.it_lo[d];
    if (A.wr_hi[d] <= A.wr_lo[d]) { *empty = 1; return 0; }  // nothing to write
  }

  if (P.kind == PSAD_KIND_GENERIC) {
    // x over threads (coalesced), y / z over blockIdx.y / blockIdx.z with grid-stride loops in the kernel
    const long long nx = A.wr_hi[2] - A.wr_lo[2], ny = A.wr_hi[1] - A.wr_lo[1], nz = A.wr_hi[0] - A.wr_lo[0];
    long long gx = cdiv(nx, P.threads);
    if (gx > 65535) gx = 65535;
    grid[0] = (unsigned)gx;
    // enough blocks to fill the machine a few times over, few enough that every block walks many rows
    const long long want = (long long)sm_count * 32;
    long long gy = ny < 65535 ? ny : 65535, gz = nz < 65535 ? nz : 65535;
    if (gx * gy * gz > want) {
      gz = want / (gx * gy);
      if (gz < 1) { gz = 1; gy = want / gx; if (gy < 1) gy = 1; }
    }
    grid[1] = (unsigned)gy;
    grid[2] = (unsigned)gz;
  } else if (P.kind == PSAD_KIND_MARCH) {
    if (nd < 2) return fail(PSAD_ERR_INVALID, "march kernels need 2 or 3 spatial dims");
    if (A.wr_lo[2] != 0 || A.wr_hi[2] != A.shape[2] || A.wr_lo[1] < 0)
      return fail(PSAD_ERR_INVALID, "march kernels write full rows: the x range must be the whole axis");
    // Kernels fusing several steps take launch ranges too: the iteration range bounds every intermediate field (0
    // outside it, what the next single-step launch would have read there), the write range the stored planes.  A
    // slab needs s * g valid ghost planes around the written planes for s fused steps (datahandling.slab_ranges).
    A.tiles_x = (int)cdiv(A.shape[2], P.tile_x);
    A.tiles_y = (int)cdiv(A.shape[1], P.tile_y);
    long long span = (nd == 3) ? (A.wr_hi[0] - A.wr_lo[0]) : A.tiles_y;
    const long long tiles = (long long)A.tiles_x * (nd == 3 ? A.tiles_y : 1);
    const long long cap = (long long)sm_count * occupancy;
    long long n_chunks;
    if (P.chunk > 0) {
      n_chunks = cdiv(span, P.chunk);
    } else {
      // Static round-robin over a persistent grid: pick the chunk count that minimises the steps of the busiest
      // CTA, ceil(items / grid) * (chunk + warm-up planes).  Long chunks amortise the HZL+HZH warm-up planes,
      // many chunks even out the tail.
      const long long warm = (nd == 3) ? P.reserved[0] : 0;
      long long best = -1, best_nc = 1;
      const long long max_nc = span < 512 ? span : 512;
      for (long long nc = 1; nc <= max_nc; ++nc) {
        const long long ch = cdiv(span, nc);
        if (cdiv(span, ch) != nc) continue;
        if (nd == 3 && ch < 8 && nc > 1) break;
        const long long cost = cdiv(tiles * nc, cap) * (ch + warm);
        if (best < 0 || cost < best) { best = cost; best_nc = nc; }
      }
      n_chunks = best_nc;
    }
    long long chunk = cdiv(span, n_chunks);
    n_chunks = cdiv(span, chunk);
    A.chunk = (int)chunk;
    A.n_chunks = (int)n_chunks;
    A.n_items = tiles * n_chunks;
    grid[0] = (unsigned)(A.n_items < cap ? A.n_items : cap);
    for (int f = 0; f < n_fields; ++f) {
      const psad_field_plan_t& fp = P.field[f];
      if (A.stride[f][2] != 1) return fail(PSAD_ERR_INVALID, "%s: field %d is not contiguous along x", kname, f);
      if (((uintptr_t)A.ptr[f]) % 16 != 0) return fail(PSAD_ERR_INVALID, "%s: field %d pointer is not 16-byte aligned", kname, f);
      if ((A.stride[f][1] * fp.elem_size) % 16 != 0 || (nd == 3 && (A.stride[f][0] * fp.elem_size) % 16 != 0))
        return fail(PSAD_ERR_INVALID, "%s: field %d row/plane pitch is not a multiple of 16 bytes", kname, f);
      if (fp.tma && fp.elem_size != 2 && fp.elem_size != 4 && fp.elem_size != 8)
        return fail(PSAD_ERR_INVALID, "TMA fields must be float16/float32/float64");
    }
  } else {
    return fail(PSAD_ERR_INVALID, "unknown kernel kind %d", P.kind);
  }
  return 0;
}

// Peer halos: what psad_kernel_launch_peer checks and derives without touching a device.
static int check_peer(const psad_plan_t& P, const char* kname, int n_fields, const psad_peer_t* peer) {
  const bool peer_kernel = P.reserved[2] == 1;
  if (peer_kernel != (peer != nullptr))
    return fail(PSAD_ERR_INVALID, "%s: %s", kname, peer_kernel ? "a peer-halo kernel needs psad_kernel_launch_peer"
                                                               : "not a peer-halo kernel (plan.reserved[2] != 1)");
  if (!peer) return 0;
  if (P.kind != PSAD_KIND_MARCH || P.ndim != 3) return fail(PSAD_ERR_INVALID, "%s: peer halos need a 3-D march kernel", kname);
  if (peer->ghost_planes < 1) return fail(PSAD_ERR_INVALID, "%s: peer halos need at least one ghost plane", kname);
  for (int s = 0; s < 2; ++s) {
    const void* flag = s ? peer->flag_hi : peer->flag_lo;
    if (!flag) continue;
    if ((s ? peer->hi_planes : peer->lo_planes) < 2 * peer->ghost_planes + 1)
      return fail(PSAD_ERR_INVALID, "%s: the %s neighbour's array has too few planes", kname, s ? "upper" : "lower");
    for (int f = 0; f < n_fields; ++f)
      if (P.field[f].tma && !(s ? peer->hi_ptr[f] : peer->lo_ptr[f]))
        return fail(PSAD_ERR_INVALID, "%s: field %d has no %s-neighbour array", kname, f, s ? "upper" : "lower");
  }
  return 0;
}

static int fill_peer_args(const char* kname, const psad_peer_t* peer, PsadArgs& A) {
  const int g = peer->ghost_planes;
  if (A.shape[0] < 2 * g + 1) return fail(PSAD_ERR_INVALID, "%s: the array has too few planes for %d ghost planes", kname, g);
  A.peer_flag_lo = static_cast<const unsigned*>(peer->flag_lo);
  A.peer_flag_hi = static_cast<const unsigned*>(peer->flag_hi);
  A.peer_error = static_cast<unsigned*>(peer->error_flag);
  A.peer_expect = peer->expect;
  static const bool no_rot = getenv("PSAD_PEER_NO_ROTATION") != nullptr;
  A.chunk_rot = no_rot ? 0 : A.n_chunks / 2;
  A.peer_lo_end = g;
  A.peer_hi_begin = (int)A.shape[0] - g;
  A.peer_lo_shift = (int)peer->lo_planes - 2 * g;     // ghost plane p of the lower block = the neighbour's plane p + n_lo
  A.peer_hi_shift = (int)A.shape[0] - 2 * g;          // ghost plane p of the upper block = the neighbour's plane p - n
  return 0;
}

extern "C" int psad_plan_launch(const psad_plan_t* plan, int sm_count, int ctas_per_sm, const psad_field_arg_t* fields,
                                int n_fields, const double* scalars, int n_scalars, const psad_range_t* range,
                                void* args_out, size_t args_bytes, unsigned grid_out[3]) {
  if (!plan || !fields || !args_out || !grid_out) return fail(PSAD_ERR_INVALID, "psad_plan_launch: null argument");
  if (args_bytes != sizeof(PsadArgs)) return fail(PSAD_ERR_INVALID, "psad_plan_launch: parameter block is %zu bytes", sizeof(PsadArgs));
  int empty = 0;
  PsadArgs A;
  if (int rc = build_args(*plan, "plan", sm_count, ctas_per_sm, fields, n_fields, scalars, n_scalars, range, A, grid_out, &empty)) return rc;
  if (empty) grid_out[0] = 0;
  memcpy(args_out, &A, sizeof(A));
  return 0;
}

extern "C" size_t psad_args_size(void) { return sizeof(PsadArgs); }

extern "C" int psad_plan_launch_peer(const psad_plan_t* plan, int sm_count, int ctas_per_sm, const psad_field_arg_t* fields,
                                     int n_fields, const double* scalars, int n_scalars, const psad_range_t* range,
                                     const psad_peer_t* peer, void* args_out, size_t args_bytes, unsigned grid_out[3]) {
  if (!plan || !fields || !args_out || !grid_out || !peer) return fail(PSAD_ERR_INVALID, "psad_plan_launch_peer: null argument");
  if (args_bytes != sizeof(PsadArgs)) return fail(PSAD_ERR_INVALID, "psad_plan_launch_peer: parameter block is %zu bytes", sizeof(PsadArgs));
  if (int rc = check_peer(*plan, "plan", n_fields, peer)) return rc;
  int empty = 0;
  PsadArgs A;
  if (int rc = build_args(*plan, "plan", sm_count, ctas_per_sm, fields, n_fields, scalars, n_scalars, range, A, grid_out, &empty)) return rc;
  if (int rc = fill_peer_args("plan", peer, A)) return rc;
  if (empty) grid_out[0] = 0;
  memcpy(args_out, &A, sizeof(A));
  return 0;
}

static int encode_one_map(const psad_plan_t& P, const psad_field_plan_t& fp, void* base, const unsigned long long gdim[3],
                          const unsigned long long gstr[2], CUtensorMap* out) {
  const int nd = P.ndim;
  // L2 promotion of TMA requests: 0 none, 1 64B, 2 128B, 3 256B (PSAD_L2PROMO overrides for experiments)
  static const int l2promo = getenv("PSAD_L2PROMO") ? atoi(getenv("PSAD_L2PROMO")) : 3;
  unsigned box[3] = {(unsigned)fp.box[0], (unsigned)fp.box[1], (unsigned)(nd == 3 ? fp.box[2] : 1)};
  unsigned estr[3] = {1, 1, 1};
  for (int d = 0; d < nd; ++d)
    if (box[d] < 1 || box[d] > 256) return fail(PSAD_ERR_INVALID, "TMA box dim %d = %u out of range", d, box[d]);
  const int dtype = fp.elem_size == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                    : fp.elem_size == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64;
  CUresult r = g_drv.cuTensorMapEncodeTiled(out, dtype,
                                            (unsigned)nd, base, gdim, gstr, box, estr,
                                            /*interleave none*/ 0, /*swizzle none*/ 0, /*L2 promotion*/ l2promo, /*oob fill: zeros*/ 0);
  if (r != 0) return cu_fail(r, "cuTensorMapEncodeTiled");
  return 0;
}

static int encode_tensor_maps(const psad_plan_t& P, const PsadArgs& A, int n_fields, const psad_peer_t* peer, TensorMaps& TM) {
  int n_tma_total = 0;
  for (int f = 0; f < n_fields; ++f) n_tma_total += P.field[f].tma ? 1 : 0;
  int n_tma = 0;
  for (int f = 0; f < n_fields; ++f) {
    const psad_field_plan_t& fp = P.field[f];
    if (!fp.tma) continue;
    unsigned long long gdim[3] = {(unsigned long long)A.shape[2], (unsigned long long)A.shape[1], (unsigned long long)A.shape[0]};
    unsigned long long gstr[2] = {(unsigned long long)A.stride[f][1] * fp.elem_size, (unsigned long long)A.stride[f][0] * fp.elem_size};
    if (int rc = encode_one_map(P, fp, A.ptr[f], gdim, gstr, &TM.m[n_tma])) return rc;
    if (peer) {
      // the neighbours' arrays have this array's row / plane pitch and their own number of planes; a missing neighbour
      // gets a copy of the local map (never used: the kernel takes that branch only with a non-null flag)
      const void* nb[2] = {peer->flag_lo ? peer->lo_ptr[f] : nullptr, peer->flag_hi ? peer->hi_ptr[f] : nullptr};
      const long long planes[2] = {peer->lo_planes, peer->hi_planes};
      for (int s = 0; s < 2; ++s) {
        CUtensorMap* dst = &TM.m[(s + 1) * n_tma_total + n_tma];
        if (!nb[s]) { *dst = TM.m[n_tma]; continue; }
        if (((uintptr_t)nb[s]) % 16 != 0) return fail(PSAD_ERR_INVALID, "peer array of field %d is not 16-byte aligned", f);
        unsigned long long pdim[3] = {gdim[0], gdim[1], (unsigned long long)planes[s]};
        if (int rc = encode_one_map(P, fp, const_cast<void*>(nb[s]), pdim, gstr, dst)) return rc;
      }
    }
    ++n_tma;
  }
  return 0;
}

static int launch_impl(psad_kernel_t k, const psad_field_arg_t* fields, int n_fields, const double* scalars, int n_scalars,
                       const psad_range_t* range, const psad_peer_t* peer, void* stream) {
  if (!k || !fields) return fail(PSAD_ERR_INVALID, "psad_kernel_launch: null argument");
  NvtxRange nvtx(k->name.c_str());
  const psad_plan_t& P = k->plan;
  if (n_fields != P.n_fields) return fail(PSAD_ERR_INVALID, "%s: expected %d fields, got %d", k->name.c_str(), P.n_fields, n_fields);
  if (n_scalars != P.n_scalars) return fail(PSAD_ERR_INVALID, "%s: expected %d scalars, got %d", k->name.c_str(), P.n_scalars, n_scalars);
  if (n_scalars > 0 && !scalars) return fail(PSAD_ERR_INVALID, "null scalars");
  if (int rc = check_peer(P, k->name.c_str(), n_fields, peer)) return rc;
  static const bool debug = getenv("PSAD_DEBUG") != nullptr;
  static const bool no_cache = getenv("PSAD_NO_LAUNCH_CACHE") != nullptr;

  // the calling thread needs the kernel's context: none current (an autograd worker) -> make it current; another device's
  // context current -> push ours for the duration of the launch
  CUcontext cur = nullptr;
  CU_CHECK(g_drv.cuCtxGetCurrent(&cur));
  bool pushed = false;
  if (cur == nullptr) {
    CU_CHECK(g_drv.cuCtxSetCurrent(k->ctx));
  } else if (cur != k->ctx) {
    CU_CHECK(g_drv.cuCtxPushCurrent(k->ctx));
    pushed = true;
  }
  struct PopGuard { bool on; ~PopGuard() { if (on) { CUcontext c; g_drv.cuCtxPopCurrent(&c); } } } guard{pushed};

  // parameter block + tensor maps: from the launch cache when this (buffers, shapes, strides, range, peers) was seen before
  LaunchKey key;
  memset(&key, 0, sizeof(key));
  key.n_fields = n_fields;
  memcpy(key.fields, fields, sizeof(psad_field_arg_t) * (size_t)n_fields);
  if (range) { key.has_range = 1; key.range = *range; }
  if (peer) { key.has_peer = 1; key.peer = *peer; key.peer.expect = 0; }
  PsadArgs A;
  TensorMaps TM;
  unsigned grid[3];
  int empty = 0;
  bool hit = false;
  if (!no_cache) {
    std::lock_guard<std::mutex> lock(k->cache_mutex);
    for (LaunchEntry* e : k->cache) {
      if (memcmp(&e->key, &key, sizeof(key)) == 0) {
        A = e->args; TM = e->tm; empty = e->empty;
        grid[0] = e->grid[0]; grid[1] = e->grid[1]; grid[2] = e->grid[2];
        e->stamp = ++k->cache_clock;
        hit = true;
        break;
      }
    }
  }
  if (hit) {
    g_cache_hits.fetch_add(1, std::memory_order_relaxed);
  } else {
    g_cache_misses.fetch_add(1, std::memory_order_relaxed);
    if (int rc = build_args(P, k->name.c_str(), k->sm_count, k->occupancy, fields, n_fields, scalars, n_scalars, range, A, grid, &empty)) return rc;
    if (peer)
      if (int rc = fill_peer_args(k->name.c_str(), peer, A)) return rc;
    if (!empty && P.kind == PSAD_KIND_MARCH)
      if (int rc = encode_tensor_maps(P, A, n_fields, peer, TM)) return rc;
    if (!no_cache) {
      LaunchEntry* e = new LaunchEntry();
      e->key = key; e->args = A; e->tm = TM; e->empty = empty;
      e->grid[0] = grid[0]; e->grid[1] = grid[1]; e->grid[2] = grid[2];
      std::lock_guard<std::mutex> lock(k->cache_mutex);
      e->stamp = ++k->cache_clock;
      if ((int)k->cache.size() >= PSAD_LAUNCH_CACHE) {          // evict the least recently used launch
        size_t victim = 0;
        for (size_t i = 1; i < k->cache.size(); ++i) if (k->cache[i]->stamp < k->cache[victim]->stamp) victim = i;
        delete k->cache[victim];
        k->cache[victim] = e;
      } else {
        k->cache.push_back(e);
      }
    }
  }
  if (empty || grid[0] == 0) return 0;
  for (int i = 0; i < n_scalars; ++i) A.scalar[i] = scalars[i];      // scalars are not part of the key
  if (peer) A.peer_expect = peer->expect;                           // nor is the launch counter
  void* params[2] = {&A, &TM};   // both are copied by cuLaunchKernel (the kernel declares as many maps as it uses)
  if (debug)
    fprintf(stderr, "[psad] %s grid=%u threads=%d smem=%d items=%lld tiles=%dx%d chunks=%d chunk=%d occ=%d cache=%s%s\n", k->name.c_str(), grid[0],
            P.threads, P.smem_bytes, A.n_items, A.tiles_x, A.tiles_y, A.n_chunks, A.chunk, k->occupancy, hit ? "hit" : "miss",
            peer ? " peer" : "");
  CUresult r = g_drv.cuLaunchKernel(k->fn, grid[0], grid[1], grid[2], (unsigned)P.threads, 1, 1, (unsigned)P.smem_bytes, (CUstream)stream, params, nullptr);
  if (r != 0) return cu_fail(r, "cuLaunchKernel");
  g_launches.fetch_add(1);
  return 0;
}

extern "C" int psad_kernel_launch(psad_kernel_t k, const psad_field_arg_t* fields, int n_fields,
                                  const double* scalars, int n_scalars, const psad_range_t* range, void* stream) {
  return launch_impl(k, fields, n_fields, scalars, n_scalars, range, nullptr, stream);
}

extern "C" int psad_kernel_launch_peer(psad_kernel_t k, const psad_field_arg_t* fields, int n_fields, const double* scalars,
                                       int n_scalars, const psad_range_t* range, const psad_peer_t* peer, void* stream) {
  if (!peer) return fail(PSAD_ERR_INVALID, "psad_kernel_launch_peer: null peer description");
  return launch_impl(k, fields, n_fields, scalars, n_scalars, range, peer, stream);
}

// ---- CUDA IPC plumbing for peer halos ---------------------------------------------------------------------------
struct IpcMapping { CUipcMemHandle handle; CUdeviceptr base; int refs; };
static std::mutex g_ipc_mutex;
static std::vector<IpcMapping> g_ipc;

static int need_ipc() {
  if (int rc = need_driver()) return rc;
  if (!g_drv.cuIpcGetMemHandle || !g_drv.cuIpcOpenMemHandle || !g_drv.cuIpcCloseMemHandle || !g_drv.cuMemGetAddressRange)
    return fail(PSAD_ERR_NO_DRIVER, "this driver lacks the CUDA IPC entry points needed for peer halos");
  return ensure_context();
}

extern "C" int psad_ipc_export(const void* ptr, void* handle_64, uint64_t* offset) {
  if (!ptr || !handle_64 || !offset) return fail(PSAD_ERR_INVALID, "psad_ipc_export: null argument");
  if (int rc = need_ipc()) return rc;
  CUdeviceptr base = 0;
  size_t size = 0;
  CU_CHECK(g_drv.cuMemGetAddressRange(&base, &size, (CUdeviceptr)(uintptr_t)ptr));
  CUipcMemHandle h;
  CUresult r = g_drv.cuIpcGetMemHandle(&h, base);
  if (r != 0) return cu_fail(r, "cuIpcGetMemHandle (allocations of an expandable-segments / VMM allocator cannot be exported)");
  memcpy(handle_64, &h, sizeof(h));
  *offset = (uint64_t)((CUdeviceptr)(uintptr_t)ptr - base);
  return 0;
}

extern "C" int psad_ipc_open(const void* handle_64, uint64_t offset, void** ptr_out) {
  if (!handle_64 || !ptr_out) return fail(PSAD_ERR_INVALID, "psad_ipc_open: null argument");
  if (int rc = need_ipc()) return rc;
  CUipcMemHandle h;
  memcpy(&h, handle_64, sizeof(h));
  std::lock_guard<std::mutex> lock(g_ipc_mutex);
  for (IpcMapping& m : g_ipc) {
    if (memcmp(&m.handle, &h, sizeof(h)) == 0) {           // an allocation can be opened only once per process
      ++m.refs;
      *ptr_out = (void*)(uintptr_t)(m.base + offset);
      return 0;
    }
  }
  CUdeviceptr base = 0;
  CUresult r = g_drv.cuIpcOpenMemHandle(&base, h, CU_IPC_MEM_LAZY_ENABLE_PEER_ACCESS);
  if (r != 0) return cu_fail(r, "cuIpcOpenMemHandle");
  g_ipc.push_back(IpcMapping{h, base, 1});
  *ptr_out = (void*)(uintptr_t)(base + offset);
  return 0;
}

extern "C" int psad_ipc_close(void* ptr) {
  if (!ptr) return 0;
  if (int rc = need_ipc()) return rc;
  std::lock_guard<std::mutex> lock(g_ipc_mutex);
  // the mapping with the largest base not above ptr
  int best = -1;
  for (size_t i = 0; i < g_ipc.size(); ++i)
    if (g_ipc[i].base <= (CUdeviceptr)(uintptr_t)ptr && (best < 0 || g_ipc[i].base > g_ipc[best].base)) best = (int)i;
  if (best < 0) return fail(PSAD_ERR_INVALID, "psad_ipc_close: not a pointer returned by psad_ipc_open");
  if (--g_ipc[best].refs == 0) {
    CUresult r = g_drv.cuIpcCloseMemHandle(g_ipc[best].base);
    g_ipc.erase(g_ipc.begin() + best);
    if (r != 0) return cu_fail(r, "cuIpcCloseMemHandle");
  }
  return 0;
}

extern "C" int psad_stream_write_u32(void* dst, uint32_t value, void* stream) {
  if (!dst) return fail(PSAD_ERR_INVALID, "psad_stream_write_u32: null pointer");
  if (int rc = need_driver()) return rc;
  if (!g_drv.cuMemsetD32Async) return fail(PSAD_ERR_NO_DRIVER, "cuMemsetD32Async is not available");
  CU_CHECK(g_drv.cuMemsetD32Async((CUdeviceptr)(uintptr_t)dst, value, 1, (CUstream)stream));
  return 0;
}

// A stream-ordered wait on the neighbours' launch counters for launches that do not wait themselves (kernels outside the
// peer protocol, or with a shorter reach than the launch before them): one thread of a built-in kernel spins until both
// counters have reached `expect` (psad_wait_peer, bounded), everything behind it on the stream starts after that.
static const char* k_peer_wait_source =
    "#include \"psad_args.h\"\n#include \"psad_common.cuh\"\n"
    "extern \"C\" __global__ void psad_peer_wait_kernel(const unsigned* lo, const unsigned* hi, unsigned expect, unsigned* error) {\n"
    "  if (lo) psad_wait_peer(lo, expect, error);\n"
    "  if (hi) psad_wait_peer(hi, expect, error);\n"
    "}\n";
struct WaitKernel { CUcontext ctx; CUmodule module; CUfunction fn; };
static std::mutex g_wait_mutex;
static std::vector<WaitKernel> g_wait_kernels;   // one per context (one per GPU a process drives)

extern "C" int psad_peer_wait(const void* flag_lo, const void* flag_hi, uint32_t expect, void* error_flag, void* stream) {
  if (!flag_lo && !flag_hi) return 0;
  if (int rc = need_driver()) return rc;
  if (int rc = ensure_context()) return rc;
  CUcontext ctx = nullptr;
  CU_CHECK(g_drv.cuCtxGetCurrent(&ctx));
  CUfunction fn = nullptr;
  {
    std::lock_guard<std::mutex> lock(g_wait_mutex);
    for (const WaitKernel& w : g_wait_kernels)
      if (w.ctx == ctx) fn = w.fn;
    if (!fn) {
      std::string path;
      if (int rc = compile_to_cache(k_peer_wait_source, "psad_peer_wait_v1", nullptr, 0, nullptr, nullptr, &path)) return rc;
      std::vector<char> cubin;
      if (!read_file(path, cubin)) return fail(PSAD_ERR_IO, "cannot read %s", path.c_str());
      WaitKernel w{ctx, nullptr, nullptr};
      CUresult r = g_drv.cuModuleLoadData(&w.module, cubin.data());
      if (r != 0) return cu_fail(r, "cuModuleLoadData(psad_peer_wait)");
      r = g_drv.cuModuleGetFunction(&w.fn, w.module, "psad_peer_wait_kernel");
      if (r != 0) { g_drv.cuModuleUnload(w.module); return cu_fail(r, "cuModuleGetFunction(psad_peer_wait_kernel)"); }
      g_wait_kernels.push_back(w);
      fn = w.fn;
    }
  }
  unsigned e = expect;
  void* params[4] = {&flag_lo, &flag_hi, &e, &error_flag};
  CUresult r = g_drv.cuLaunchKernel(fn, 1, 1, 1, 1, 1, 1, 0, (CUstream)stream, params, nullptr);
  if (r != 0) return cu_fail(r, "cuLaunchKernel(psad_peer_wait_kernel)");
  g_launches.fetch_add(1);
  return 0;
}

extern "C" int psad_launch_cache_stats(unsigned long long* hits, unsigned long long* misses) {
  if (hits) *hits = g_cache_hits.load();
  if (misses) *misses = g_cache_misses.load();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// NCCL ghost-layer exchange
typedef struct ncclComm* ncclComm_t;
struct NcclUniqueId { char internal[128]; };
struct Nccl {
  void* lib = nullptr;
  int (*ncclGetUniqueId)(NcclUniqueId*);
  int (*ncclCommInitRank)(ncclComm_t*, int, NcclUniqueId, int);
  int (*ncclCommDestroy)(ncclComm_t);
  int (*ncclGroupStart)();
  int (*ncclGroupEnd)();
  int (*ncclSend)(const void*, size_t, int, int, ncclComm_t, CUstream);
  int (*ncclRecv)(void*, size_t, int, int, ncclComm_t, CUstream);
  const char* (*ncclGetErrorString)(int);
};
static Nccl g_nccl;
static std::once_flag g_nccl_once;
static std::string g_nccl_err;

static void load_nccl() {
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  void* lib = nullptr;
  for (const char* n : names) { lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (lib) break; }
  if (!lib) { g_nccl_err = std::string("cannot load libnccl.so.2: ") + dlerror(); return; }
  Nccl n; n.lib = lib; std::string e;
  bool ok = sym(lib, "ncclGetUniqueId", n.ncclGetUniqueId, e) && sym(lib, "ncclCommInitRank", n.ncclCommInitRank, e) &&
            sym(lib, "ncclCommDestroy", n.ncclCommDestroy, e) && sym(lib, "ncclGroupStart", n.ncclGroupStart, e) &&
            sym(lib, "ncclGroupEnd", n.ncclGroupEnd, e) && sym(lib, "ncclSend", n.ncclSend, e) && sym(lib, "ncclRecv", n.ncclRecv, e) &&
            sym(lib, "ncclGetErrorString", n.ncclGetErrorString, e);
  if (!ok) { g_nccl_err = e; return; }
  g_nccl = n;
}
static int need_nccl() {
  std::call_once(g_nccl_once, load_nccl);
  if (!g_nccl.lib) return fail(PSAD_ERR_NO_DRIVER, "%s", g_nccl_err.c_str());
  return 0;
}
#define NCCL_CHECK(call) do { int _r = (call); if (_r != 0) return fail(PSAD_ERR_NCCL, "%s failed: %s", #call, g_nccl.ncclGetErrorString(_r)); } while (0)

extern "C" int psad_nccl_unique_id(void* unique_id_128) {
  if (!unique_id_128) return fail(PSAD_ERR_INVALID, "null id");
  if (int rc = need_nccl()) return rc;
  NcclUniqueId id;
  NCCL_CHECK(g_nccl.ncclGetUniqueId(&id));
  memcpy(unique_id_128, &id, sizeof(id));
  return 0;
}

extern "C" int psad_nccl_comm_create(const void* unique_id_128, int rank, int world_size, void** comm) {
  if (!unique_id_128 || !comm) return fail(PSAD_ERR_INVALID, "null argument");
  if (int rc = need_nccl()) return rc;
  NcclUniqueId id;
  memcpy(&id, unique_id_128, sizeof(id));
  ncclComm_t c;
  NCCL_CHECK(g_nccl.ncclCommInitRank(&c, world_size, id, rank));
  *comm = c;
  return 0;
}

extern "C" int psad_nccl_comm_destroy(void* comm) {
  if (!comm) return 0;
  if (int rc = need_nccl()) return rc;
  NCCL_CHECK(g_nccl.ncclCommDestroy((ncclComm_t)comm));
  return 0;
}

extern "C" int psad_halo_exchange(void* comm, const void* lo_send, void* lo_recv, const void* hi_send, void* hi_recv,
                                  size_t bytes, int lo_rank, int hi_rank, void* stream) {
  if (!comm) return fail(PSAD_ERR_INVALID, "null communicator");
  if (int rc = need_nccl()) return rc;
  if (bytes == 0 || (lo_rank < 0 && hi_rank < 0)) return 0;
  NvtxRange nvtx("psad_halo_exchange");
  ncclComm_t c = (ncclComm_t)comm;
  CUstream s = (CUstream)stream;
  NCCL_CHECK(g_nccl.ncclGroupStart());
  int rc = 0;
  // ncclInt8 == ncclChar == 0: counts are bytes
  if (lo_rank >= 0 && lo_rank == hi_rank) {
    // two ranks on a periodic domain: both neighbours are the same peer.  Sends and receives between one pair of ranks
    // match in issue order, so the receives are posted in the order the peer sends: its first planes (our upper ghost
    // planes), then its last planes (our lower ghost planes).
    if (!rc) rc = g_nccl.ncclSend(lo_send, bytes, 0, lo_rank, c, s);
    if (!rc) rc = g_nccl.ncclSend(hi_send, bytes, 0, hi_rank, c, s);
    if (!rc) rc = g_nccl.ncclRecv(hi_recv, bytes, 0, hi_rank, c, s);
    if (!rc) rc = g_nccl.ncclRecv(lo_recv, bytes, 0, lo_rank, c, s);
  } else {
    if (lo_rank >= 0) {
      if (!rc) rc = g_nccl.ncclSend(lo_send, bytes, 0, lo_rank, c, s);
      if (!rc) rc = g_nccl.ncclRecv(lo_recv, bytes, 0, lo_rank, c, s);
    }
    if (hi_rank >= 0) {
      if (!rc) rc = g_nccl.ncclSend(hi_send, bytes, 0, hi_rank, c, s);
      if (!rc) rc = g_nccl.ncclRecv(hi_recv, bytes, 0, hi_rank, c, s);
    }
  }
  int rc2 = g_nccl.ncclGroupEnd();
  if (rc) return fail(PSAD_ERR_NCCL, "ncclSend/ncclRecv failed: %s", g_nccl.ncclGetErrorString(rc));
  if (rc2) return fail(PSAD_ERR_NCCL, "ncclGroupEnd failed: %s", g_nccl.ncclGetErrorString(rc2));
  return 0;
}
