// Library-level pieces of the C ABI: error text, device check, deterministic mode, tensor-map encoding.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"
#include "../../include/roomslam_b200.h"

namespace rs {

static thread_local char g_error[1024] = "";
static unsigned long long g_launches = 0;
static int g_deterministic = 0;

bool deterministic() { return __atomic_load_n(&g_deterministic, __ATOMIC_RELAXED) != 0; }

void count_launch(int n) { __atomic_fetch_add(&g_launches, (unsigned long long)n, __ATOMIC_RELAXED); }

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

int check_device_sm100() {
    static thread_local int cached_dev = -1;
    static thread_local int cached_ok = 0;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        set_error("no CUDA device: %s (roomslam_b200 has no CPU fallback)", cudaGetErrorString(e));
        return 3;
    }
    if (dev != cached_dev) {
        int major = 0, minor = 0;
        cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
        cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
        cached_dev = dev;
        cached_ok = (major == 10 && minor == 0);
        if (!cached_ok) set_error("device %d is sm_%d%d; roomslam_b200 kernels are built for sm_100a only", dev, major, minor);
    }
    if (!cached_ok) {
        if (g_error[0] == 0) set_error("current device is not sm_100");
        return 3;
    }
    return 0;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_tmap_2d(CUtensorMap* out, const void* base, CUtensorMapDataType dtype, uint32_t elem_bytes, uint64_t inner,
                 uint64_t outer, uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_outer,
                 CUtensorMapSwizzle swizzle) {
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
            set_error("cuTensorMapEncodeTiled entry point unavailable: %s", cudaGetErrorString(e));
            return 2;
        }
        encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    (void)elem_bytes;
    cuuint64_t dims[2] = {inner, outer};
    cuuint64_t strides[1] = {row_stride_bytes};
    cuuint32_t box[2] = {box_inner, box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(out, dtype, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (inner=%llu outer=%llu stride=%llu box=%ux%u)", (int)r,
                  (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)row_stride_bytes, box_inner,
                  box_outer);
        return 2;
    }
    return 0;
}

}  // namespace rs

extern "C" const char* rs_last_error(void) { return rs::g_error; }
extern "C" int rs_abi_version(void) { return 2; }
extern "C" int64_t rs_launch_count(void) { return (int64_t)__atomic_load_n(&rs::g_launches, __ATOMIC_RELAXED); }
extern "C" int rs_device_ok(void) { return rs::check_device_sm100() == 0 ? 1 : 0; }
extern "C" int rs_set_deterministic(int on) {
    __atomic_store_n(&rs::g_deterministic, on ? 1 : 0, __ATOMIC_RELAXED);
    return 0;
}
extern "C" int rs_deterministic(void) { return rs::deterministic() ? 1 : 0; }
