// Library services of the crop2seg_b200 C ABI: error text, launch accounting, ABI version; tensor maps and SM counts for the
// kernels.
#include <atomic>
#include <cstring>

#include "c2s_sm100.cuh"

namespace c2s {

namespace {
thread_local char g_error[512] = "";
// process-wide (autograd runs backward kernels on its own thread); diagnostics only
char g_kernel[128] = "";
char g_ltae_kernel[128] = "";
std::atomic<int64_t> g_launches{0};
std::atomic<int> g_options[4] = {{0}, {0}, {0}, {0}};
}  // namespace

int option(int which) { return (which >= 0 && which < 4) ? g_options[which].load(std::memory_order_relaxed) : 0; }

// cudaFuncSetAttribute is a per-device setting: `done` holds one flag per device ordinal for one kernel.
int set_max_dynamic_smem(const void* func, int bytes, std::atomic<unsigned long long>* done) {
  int dev = 0;
  C2S_CUDA(cudaGetDevice(&dev));
  const unsigned long long bit = 1ull << (dev & 63);
  if (done->load(std::memory_order_acquire) & bit) return C2S_OK;
  cudaFuncAttributes fa;
  C2S_CUDA(cudaFuncGetAttributes(&fa, func));
  const int room = 232448 - static_cast<int>(fa.sharedSizeBytes);  // 227 KB per CTA, static part included
  C2S_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes < room ? bytes : room));
  done->fetch_or(bit, std::memory_order_release);
  return C2S_OK;
}

int encode_tensor_map(CUtensorMap* map, CUtensorMapDataType dtype, cuuint32_t rank, const void* base, const cuuint64_t* dims,
                      const cuuint64_t* strides, const cuuint32_t* box, CUtensorMapSwizzle swizzle,
                      CUtensorMapL2promotion l2_promotion, const char* what) {
  using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                     CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  // the driver entry point, looked up once (the library does not link libcuda); static initialisation is thread-safe
  static const EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      return reinterpret_cast<EncodeTiledFn>(p);
    return nullptr;
  }();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return C2S_ERR_CUDA;
  }
  const cuuint32_t elem_strides[5] = {1, 1, 1, 1, 1};
  const CUresult r = fn(map, dtype, rank, const_cast<void*>(base), dims, strides, box, elem_strides,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, l2_promotion, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (%s) failed with CUresult %d", what, static_cast<int>(r));
    return C2S_ERR_CUDA;
  }
  return C2S_OK;
}

int sm_count() {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
    sms = 148;
  return sms;
}

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

void note_launch(const char* kernel_name) {
  ++g_launches;
  strncpy(g_kernel, kernel_name, sizeof(g_kernel) - 1);
  g_kernel[sizeof(g_kernel) - 1] = '\0';
  if (strncmp(kernel_name, "ltae_forward", 12) == 0) {
    strncpy(g_ltae_kernel, kernel_name, sizeof(g_ltae_kernel) - 1);
    g_ltae_kernel[sizeof(g_ltae_kernel) - 1] = '\0';
  }
}

int check_device() {
  int dev = 0;
  cudaError_t err = cudaGetDevice(&dev);
  if (err != cudaSuccess) {
    set_error("cudaGetDevice failed: %s", cudaGetErrorString(err));
    return C2S_ERR_NO_DEVICE;
  }
  // one attribute query per device, cached (re-entrant: worst case two threads write the same value)
  static int cached_major[64] = {0};
  if (dev < 64 && cached_major[dev] == 0) {
    int major = 0;
    err = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (err != cudaSuccess) {
      set_error("cudaDeviceGetAttribute failed: %s", cudaGetErrorString(err));
      return C2S_ERR_NO_DEVICE;
    }
    cached_major[dev] = major;
  }
  if (dev < 64 && cached_major[dev] != 10) {
    set_error("crop2seg_b200 is built for sm_100a only; device %d has compute capability major %d",
              dev, cached_major[dev]);
    return C2S_ERR_NO_DEVICE;
  }
  return C2S_OK;
}

}  // namespace c2s

extern "C" {

int c2s_abi_version(void) { return C2S_ABI_VERSION; }

const char* c2s_last_error(void) { return c2s::g_error; }

int64_t c2s_launch_count(void) { return c2s::g_launches.load(); }

void c2s_reset_launch_count(void) { c2s::g_launches.store(0); }

int c2s_set_option(int option, int value) {
  const int max_value[4] = {C2S_LTAE_KERNEL_TEAM, 1, 1, 1};
  if (option < 0 || option >= 4 || value < 0 || value > max_value[option]) {
    c2s::set_error("c2s_set_option: unknown option %d / value %d", option, value);
    return C2S_ERR_BAD_ARGUMENT;
  }
  c2s::g_options[option].store(value);
  return C2S_OK;
}

int c2s_get_option(int option) { return (option >= 0 && option < 4) ? c2s::g_options[option].load() : -1; }

const char* c2s_last_kernel(void) { return c2s::g_kernel; }
const char* c2s_last_ltae_kernel(void) { return c2s::g_ltae_kernel; }

}  // extern "C"
