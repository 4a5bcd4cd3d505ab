// Shared helpers for the gnnml3_b200 C-ABI library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include <mutex>

#include "../../include/gnnml3_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "gnnml3_b200 is written for sm_100a (B200) only"
#endif

namespace gnnml3 {

// thread-local last-error string (the autograd engine calls backward from its own thread)
char* err_buf();
int set_err(int code, const char* fmt, ...);
void count_launch(int n);

#define GNNML3_REQUIRE(cond, ...)                                        \
    do {                                                                 \
        if (!(cond)) return ::gnnml3::set_err(GNNML3_ERR_INVALID, __VA_ARGS__); \
    } while (0)

#define GNNML3_CUDA(expr)                                                                          \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return ::gnnml3::set_err(GNNML3_ERR_CUDA, "%s:%d: %s -> %s", __FILE__, __LINE__, #expr, \
                                     cudaGetErrorString(_e));                                      \
    } while (0)

#define GNNML3_LAUNCH_CHECK()           \
    do {                              \
        ::gnnml3::count_launch(1);    \
        GNNML3_CUDA(cudaGetLastError()); \
    } while (0)

static inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline bool prec_valid(int prec) {
    return prec == GNNML3_PREC_3XTF32 || prec == GNNML3_PREC_TF32 || prec == GNNML3_PREC_BF16;
}

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

// cudaFuncSetAttribute is per device: `flags` is a per-kernel static array, true once the attribute was set on the current
// device (a process normally drives one GPU, but nothing here assumes it).  Thread-safe (the autograd engine calls backward
// from its own thread): the first caller on a device gets a guard that holds the library's configuration mutex until the
// attribute calls in the `if` body are done, and only then publishes the flag; later callers take the lock-free path.
//     if (auto once = first_use_on_device(configured)) GNNML3_CUDA(cudaFuncSetAttribute(...));
std::mutex& config_mutex();      // runtime.cu
struct DeviceOnce {
    bool* flag;
    std::unique_lock<std::mutex> lock;
    explicit operator bool() const { return flag != nullptr; }
    ~DeviceOnce() {
        if (flag) __atomic_store_n(flag, true, __ATOMIC_RELEASE);
    }
};
static inline DeviceOnce first_use_on_device(bool (&flags)[64]) {
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    if (__atomic_load_n(&flags[dev], __ATOMIC_ACQUIRE)) return DeviceOnce{nullptr, {}};
    std::unique_lock<std::mutex> lk(config_mutex());
    if (flags[dev]) return DeviceOnce{nullptr, {}};
    return DeviceOnce{&flags[dev], std::move(lk)};
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float2 ldg2(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }

// streaming 128-bit store that does not pollute L1 (outputs are written once)
__device__ __forceinline__ void st_na4(float* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}

// tanh via one ex2.approx and one rcp.approx: 1 - 2 / (e^{2x} + 1), evaluated on |x| and mirrored.
// Absolute error <= ~2e-7 over the whole range (the FP32 parity bar is 1e-5 relative to the tensor's scale);
// ~6 instructions instead of the ~25 of tanhf -- the edge MLP evaluates 4K tanh per edge.
__device__ __forceinline__ float tanh_fast(float x) {
    const float e = __expf(2.0f * fabsf(x));
    const float r = 1.0f - __fdividef(2.0f, e + 1.0f);
    return copysignf(r, x);
}

// Same function without the |x| / copysign mirror: e^{2x} = inf gives 1 - 0, e^{2x} = 0 gives 1 - 2; five instructions
// (FMUL, MUFU.EX2, FADD, MUFU.RCP, FFMA).  Same absolute error bound.
__device__ __forceinline__ float tanh_fast5(float x) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.885390081777927f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
}

}  // namespace gnnml3
