// Shared helpers for libsglm_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <stdio.h>
#include <string.h>

#include "../../include/sglm_b200.h"

namespace sglm {

// Thread-local last error text (sglm_last_error()).
char *last_error_buf();
int fail(int code, const char *fmt, ...);

#define SGLM_CHECK_ARG(cond, code, ...)                    \
    do {                                                   \
        if (!(cond)) return ::sglm::fail((code), __VA_ARGS__); \
    } while (0)

#define SGLM_CUDA_OK(expr)                                                              \
    do {                                                                                \
        cudaError_t _e = (expr);                                                        \
        if (_e != cudaSuccess)                                                          \
            return ::sglm::fail(SGLM_E_CUDA, "%s failed: %s (%s:%d)", #expr,            \
                                cudaGetErrorString(_e), __FILE__, __LINE__);            \
    } while (0)

#define SGLM_LAUNCH_OK(name)                                                            \
    do {                                                                                \
        cudaError_t _e = cudaGetLastError();                                            \
        if (_e != cudaSuccess)                                                          \
            return ::sglm::fail(SGLM_E_CUDA, "launch of %s failed: %s", (name),         \
                                cudaGetErrorString(_e));                                \
    } while (0)

inline int sm_count() {
    int dev = 0, n = 148;
    if (cudaGetDevice(&dev) == cudaSuccess)
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n > 0 ? n : 148;
}

template <typename T>
__host__ __device__ inline T ceil_div(T a, T b) { return (a + b - 1) / b; }

// Tweedie families with log link (the terms of scikit-learn's HalfTweedieLoss), a compile-time parameter of the GLM
// passes: FAM_POISSON (power 1), FAM_GAMMA (power 2: Fisher weight 1), FAM_TWEEDIE (any other power > 1, a runtime
// scalar; mu^(1-p) = exp((1-p) eta), one exp more per element).
enum { FAM_POISSON = 0, FAM_GAMMA = 1, FAM_TWEEDIE = 2 };
inline bool glm_power_ok(double power) { return power == 1.0 || power > 1.0; }
inline int glm_family(double power) { return power == 1.0 ? FAM_POISSON : (power == 2.0 ? FAM_GAMMA : FAM_TWEEDIE); }

// Soft-threshold branch select of the coordinate-descent step, (r > l1) ? dpos : ((r < -l1) ? dneg : other), as two
// predicated selects.  Written in PTX because the compiler otherwise turns the nested conditional into a divergent
// branch around the second FMA (BSSY / BRA / BSYNC + a BRA.DIV convergence check before the next shuffle) — on the
// 32-step dependent chain that bounds the heaviest models (ncu source view, profiles/r2_cd_experiments.txt §5).
__device__ __forceinline__ double cd_soft_select(double r, double l1, double dpos, double dneg, double other) {
    double out;
    asm("{\n\t.reg .pred p, q;\n\t"
        "setp.gt.f64 p, %1, %2;\n\t"
        "setp.lt.f64 q, %1, %3;\n\t"
        "selp.f64 %0, %5, %6, q;\n\t"
        "selp.f64 %0, %4, %0, p;\n\t}"
        : "=&d"(out) : "d"(r), "d"(l1), "d"(-l1), "d"(dpos), "d"(dneg), "d"(other));
    return out;
}

// Measurement switches (kernel shape variants, A/B forms) are honoured only when the process was started with
// SGLM_TUNING=1 — read once; a production call never consults the environment.
inline const char *tuning_env(const char *name) {
    static const bool on = [] { const char *v = getenv("SGLM_TUNING"); return v && v[0] == '1'; }();
    return on ? getenv(name) : nullptr;
}

__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

}  // namespace sglm
