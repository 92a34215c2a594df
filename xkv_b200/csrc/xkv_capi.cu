// xkv_b200 — C-ABI plumbing: error reporting, launch accounting, TMA tensor-map encoding.
#include <cudaTypedefs.h>

#include "xkv_host.h"

namespace xkv {

std::atomic<long long> g_launch_count{0};

char* error_buffer() {
  static thread_local char buf[1024] = {0};
  return buf;
}

int set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(error_buffer(), 1024, fmt, ap);
  va_end(ap);
  return 1;
}

int device_sm_count() {
  static PerDevice<int> sms;
  int& n = sms();
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        n <= 0)
      n = 148;
  }
  return n;
}

// cuTensorMapEncodeTiled is a driver-API symbol. It is resolved at run time through the runtime's
// driver entry-point query so the library has no link-time dependency on libcuda.so and still loads
// (for symbol checks) on a machine without a GPU driver.
static PFN_cuTensorMapEncodeTiled_v12000 tensor_map_encoder() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = []() -> PFN_cuTensorMapEncodeTiled_v12000 {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess) return nullptr;
    if (q != cudaDriverEntryPointSuccess) return nullptr;
    return reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }();
  return fn;
}

int encode_tmap_2d_bf16(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t ld_elems,
                        uint32_t box_inner, uint32_t box_outer) {
  auto enc = tensor_map_encoder();
  XKV_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
  cuuint64_t gdim[2] = {inner, outer};
  cuuint64_t gstride[1] = {ld_elems * 2};  // bytes, dimension 1
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estride[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estride,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  XKV_REQUIRE(r == CUDA_SUCCESS,
              "cuTensorMapEncodeTiled failed (%d): base=%p inner=%llu outer=%llu ld=%llu box=%ux%u", static_cast<int>(r),
              base, static_cast<unsigned long long>(inner), static_cast<unsigned long long>(outer),
              static_cast<unsigned long long>(ld_elems), box_inner, box_outer);
  return 0;
}

int encode_tmap_3d_bf16(CUtensorMap* map, const void* base, const uint64_t dims[3], const uint64_t strides_elems[2],
                        const uint32_t box[3]) {
  auto enc = tensor_map_encoder();
  XKV_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
  cuuint64_t gdim[3] = {dims[0], dims[1], dims[2]};
  cuuint64_t gstride[2] = {strides_elems[0] * 2, strides_elems[1] * 2};   // bytes, dimensions 1 and 2
  cuuint32_t bx[3] = {box[0], box[1], box[2]};
  cuuint32_t estride[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), gdim, gstride, bx, estride,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  XKV_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d): base=%p dims=%llux%llux%llu strides=%llu,%llu",
              static_cast<int>(r), base, static_cast<unsigned long long>(dims[0]), static_cast<unsigned long long>(dims[1]),
              static_cast<unsigned long long>(dims[2]), static_cast<unsigned long long>(strides_elems[0]),
              static_cast<unsigned long long>(strides_elems[1]));
  return 0;
}

}  // namespace xkv

extern "C" const char* xkv_last_error(void) { return xkv::error_buffer(); }
extern "C" int xkv_version(void) { return 203; }
extern "C" int64_t xkv_launch_count(void) { return xkv::g_launch_count.load(); }
