// Host-side helpers shared by all translation units of libofx.so: error convention,
// TMA tensor-map creation, launch helpers.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/ofx.h"

namespace ofx {

// thread-local last-error string returned by ofx_last_error()
void set_error(const char* fmt, ...);
int fail(int code, const char* fmt, ...);
const char* last_error();

#define OFX_CUDA(expr)                                                                        \
    do {                                                                                      \
        cudaError_t e__ = (expr);                                                             \
        if (e__ != cudaSuccess)                                                               \
            return ::ofx::fail(OFX_E_CUDA, "%s failed: %s (%s:%d)", #expr,                    \
                               cudaGetErrorString(e__), __FILE__, __LINE__);                  \
    } while (0)

#define OFX_TRY(expr)              \
    do {                           \
        int rc__ = (expr);         \
        if (rc__ != OFX_OK) return rc__; \
    } while (0)

// every kernel launch of the library goes through this: error check + launch counter
// (ofx_launch_count, read by bench.py for its gpu_launches claim)
void count_launch();
long long launches();
#define OFX_LAUNCH_CHECK()            \
    do {                              \
        ::ofx::count_launch();        \
        OFX_CUDA(cudaGetLastError()); \
    } while (0)

// Requires a device of compute capability 10.x (the kernels are sm_100a-only).
int require_sm100();
int sm_count();      // of the CURRENT device (cached per device)

// "Done once per DEVICE" flag for per-device function attributes (the dynamic shared-memory opt-in of
// cudaFuncSetAttribute is per device: a process-wide `static bool` left every kernel above 48 KB unlaunchable
// on the second GPU of a process).  need() is true the first time it is called with a given current device;
// a race between host threads only sets the attribute twice.
struct DeviceOnce {
    static constexpr int kMaxDevices = 64;
    unsigned char done[kMaxDevices] = {};
    bool need() {
        int dev = -1;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return true;
        if (__atomic_load_n(&done[dev], __ATOMIC_RELAXED)) return false;
        __atomic_store_n(&done[dev], static_cast<unsigned char>(1), __ATOMIC_RELAXED);
        return true;
    }
};

// 2-D bf16 tensor map: `rows` x `cols` elements, row pitch `ld` elements, box = box_rows x 64
// elements (128 B) with the 128-byte swizzle the UMMA descriptors expect; OOB reads give zeros.
// TMA moves the 2-byte elements without interpreting them (OOB_FILL_NONE writes zero bits), so the
// same map carries fp16 rows.
int make_tmap_bf16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                   uint32_t box_rows);

// 2-D fp32 tensor map, box = box_rows x 32 elements (128 B), 128-byte swizzle
int make_tmap_f32(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                  uint32_t box_rows);

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace ofx
