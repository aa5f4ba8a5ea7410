#include "common.h"

#include <stdarg.h>
#include <string.h>

#include <atomic>

namespace ofx {

static thread_local char g_err[512] = "";

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

const char* last_error() { return g_err; }

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
long long launches() { return g_launches.load(std::memory_order_relaxed); }

static int g_sm_count[DeviceOnce::kMaxDevices] = {};

int require_sm100() {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(OFX_E_ARCH, "no CUDA device: %s", cudaGetErrorString(e));
    }
    return ofx_device_ok(dev);
}

int sm_count() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= DeviceOnce::kMaxDevices) return 148;
    const int cached = __atomic_load_n(&g_sm_count[dev], __ATOMIC_RELAXED);
    if (cached > 0) return cached;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    __atomic_store_n(&g_sm_count[dev], n, __ATOMIC_RELAXED);
    return n;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// libcuda is not linked (the library must load on hosts without a driver, where only the
// symbol table is inspected); the encoder is resolved through the runtime at first use.
static EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) ==
                cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

int make_tmap_bf16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                   uint32_t box_rows) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail(OFX_E_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * 2};  // bytes, dim 1
    cuuint32_t box[2] = {64, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims,
                     strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(OFX_E_CUDA, "cuTensorMapEncodeTiled failed (%d): rows=%llu cols=%llu ld=%llu",
                    static_cast<int>(r), (unsigned long long)rows, (unsigned long long)cols,
                    (unsigned long long)ld);
    return OFX_OK;
}

// 2-D fp32 tensor map: box = box_rows x 32 elements (128 B), 128-byte swizzle
int make_tmap_f32(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                  uint32_t box_rows) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail(OFX_E_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * 4};
    cuuint32_t box[2] = {32, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(OFX_E_CUDA, "cuTensorMapEncodeTiled (fp32) failed (%d): rows=%llu cols=%llu ld=%llu",
                    static_cast<int>(r), (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld);
    return OFX_OK;
}

}  // namespace ofx

extern "C" {

int ofx_version(void) { return OFX_VERSION; }

const char* ofx_last_error(void) { return ofx::last_error(); }

int64_t ofx_launch_count(void) { return ofx::launches(); }

int ofx_device_ok(int device) {
    int major = 0, n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || device < 0 || device >= n) {
        cudaGetLastError();
        return ofx::fail(OFX_E_ARCH, "CUDA device %d not available (%s)", device,
                         e != cudaSuccess ? cudaGetErrorString(e) : "out of range");
    }
    e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
    if (e != cudaSuccess) return ofx::fail(OFX_E_CUDA, "%s", cudaGetErrorString(e));
    if (major != 10)
        return ofx::fail(OFX_E_ARCH, "device %d has compute capability %d.x; libofx needs sm_100a", device,
                         major);
    return OFX_OK;
}
}
