// Library-level C-ABI entry points and host helpers (errors, TMA descriptor encoding).
#include "host.h"

#include <stdlib.h>

#include <atomic>
#include <map>
#include <mutex>
#include <utility>

namespace xclip {

static thread_local char g_err[1024] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn g_encode = nullptr;
static int g_sms = 0;
static std::mutex g_init_mu;
static bool g_inited = false;

static int do_init() {
  std::lock_guard<std::mutex> lk(g_init_mu);
  if (g_inited) return XCLIP_OK;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess)
    return fail(XCLIP_ERR_CUDA, "cudaGetDevice failed: %s", cudaGetErrorString(e));
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess)
    return fail(XCLIP_ERR_CUDA, "cudaGetDeviceProperties failed: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(XCLIP_ERR_UNSUPPORTED,
                "x_clip_b200 needs an sm_100 (B200) device; device %d is sm_%d%d - there is no "
                "fallback path",
                dev, prop.major, prop.minor);
  g_sms = prop.multiProcessorCount;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || fn == nullptr)
    return fail(XCLIP_ERR_CUDA, "cannot resolve cuTensorMapEncodeTiled (%s)",
                cudaGetErrorString(e));
  g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  g_inited = true;
  return XCLIP_OK;
}

int num_sms() { return g_sms; }

int ensure_dynamic_smem(const void* kernel, int bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, int> done;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return fail(XCLIP_ERR_CUDA, "cudaGetDevice failed: %s", cudaGetErrorString(e));
  std::lock_guard<std::mutex> lk(mu);
  int& cur = done[std::make_pair(dev, kernel)];
  if (cur >= bytes) return XCLIP_OK;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess)
    return fail(XCLIP_ERR_CUDA, "cudaFuncSetAttribute(%d B dynamic smem) failed: %s", bytes,
                cudaGetErrorString(e));
  cur = bytes;
  return XCLIP_OK;
}

int encode_2d_bf16(CUtensorMap* out, const void* ptr, uint64_t inner, uint64_t outer,
                   uint64_t outer_stride_elems, uint32_t box_inner, uint32_t box_outer) {
  if (!g_inited) {
    int rc = do_init();
    if (rc) return rc;
  }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {outer_stride_elems * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims,
                        strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(XCLIP_ERR_CUDA,
                "cuTensorMapEncodeTiled(2d) failed: CUresult %d (ptr=%p inner=%llu outer=%llu "
                "stride=%llu box=%ux%u)",
                (int)r, ptr, (unsigned long long)inner, (unsigned long long)outer,
                (unsigned long long)outer_stride_elems, box_inner, box_outer);
  return XCLIP_OK;
}

int encode_3d_bf16(CUtensorMap* out, const void* ptr, uint64_t inner, uint64_t mid,
                   uint64_t outer, uint64_t mid_stride_elems, uint64_t outer_stride_elems,
                   uint32_t box_inner, uint32_t box_mid) {
  if (!g_inited) {
    int rc = do_init();
    if (rc) return rc;
  }
  cuuint64_t dims[3] = {inner, mid, outer};
  cuuint64_t strides[2] = {mid_stride_elems * 2, outer_stride_elems * 2};
  cuuint32_t box[3] = {box_inner, box_mid, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = g_encode(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims,
                        strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(XCLIP_ERR_CUDA,
                "cuTensorMapEncodeTiled(3d) failed: CUresult %d (ptr=%p dims=%llu,%llu,%llu)",
                (int)r, ptr, (unsigned long long)inner, (unsigned long long)mid,
                (unsigned long long)outer);
  return XCLIP_OK;
}

}  // namespace xclip

extern "C" {

int xclip_tune_set(int, int) { return -1; }

int xclip_abi_version(void) { return 2; }

const char* xclip_last_error(void) { return xclip::g_err; }

int xclip_init(void) { return xclip::do_init(); }

long long xclip_launch_count(void) { return xclip::g_launches.load(); }

void xclip_launch_count_reset(void) { xclip::g_launches.store(0); }

}  // extern "C"
