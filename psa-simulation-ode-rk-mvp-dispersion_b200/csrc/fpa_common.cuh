// fpa_common.cuh -- shared host/device helpers of libfpa_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/fpa_b200.h"

namespace fpa {

// ----------------------------------------------------------------- error plumbing
void set_error(const char* fmt, ...);
int  cuda_fail(cudaError_t e, const char* what);

#define FPA_CUDA(call)                                              \
    do {                                                            \
        cudaError_t e__ = (call);                                   \
        if (e__ != cudaSuccess) return ::fpa::cuda_fail(e__, #call); \
    } while (0)

#define FPA_REQUIRE(cond, ...)                    \
    do {                                          \
        if (!(cond)) {                            \
            ::fpa::set_error(__VA_ARGS__);        \
            return FPA_ERR_INVALID;               \
        }                                         \
    } while (0)

// FPA_ERR_INVALID unless `ptr` (NULL passes) is 16-byte aligned.  The kernels move complex128 values and rows of
// maxima with 16-byte vector accesses, which fault on an address that is only 8-byte aligned.  For the device
// pointers of the _dev entries, checked by the launchers; the host entries stage such arrays instead.
#define FPA_REQUIRE_ALIGNED16(ptr, name)                                                           \
    FPA_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "%s must be 16-byte aligned (got %p)", \
                name, (const void*)(ptr))

// The same for the arrays the kernels store one double at a time (the transfer kernels' jac).
#define FPA_REQUIRE_ALIGNED8(ptr, name)                                                          \
    FPA_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 7) == 0, "%s must be 8-byte aligned (got %p)", \
                name, (const void*)(ptr))

// Selects `device` (must exist) -- there is no CPU fallback anywhere in this library.
int use_device(int device);

// Grow-only device workspace, one per (host thread, device, slot).
// Returned pointer stays valid until a later call asks the same slot for more bytes.
int workspace(int device, int slot, size_t bytes, void** out);

// ----------------------------------------------------------------- device helpers
__device__ __forceinline__ bool nonfinite(double v) {
    // exponent field all ones <=> Inf or NaN; integer test keeps the FP64 pipe free
    return (__double2hiint(v) & 0x7ff00000) == 0x7ff00000;
}

__device__ __forceinline__ double qnan() { return __longlong_as_double(0x7ff8000000000000LL); }

// 16-byte streaming store of one complex128
__device__ __forceinline__ void store_c128(double* p, double re, double im) {
    *reinterpret_cast<double2*>(p) = make_double2(re, im);
}

// 32-byte store of two complex128 (sm_100 256-bit vector store: one full 32 B sector per thread).
// p must be 32-byte aligned.
__device__ __forceinline__ void store_2c128(double* p, double a, double b, double c, double d) {
    asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

}  // namespace fpa
