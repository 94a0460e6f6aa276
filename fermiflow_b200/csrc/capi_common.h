// Host-side plumbing shared by the translation units of the C ABI (capi.cu, capi_eloc.cu): error reporting,
// option switches, launch counter, device attributes.  Definitions live in capi.cu.
#pragma once
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <algorithm>
#include <atomic>
#include <cuda_runtime.h>

#include "../../include/fermiflow_b200.h"

namespace ffc {

int fail(int code, const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

// "this launcher does not apply, try the next one" -- outside the range of cudaError_t (>= 0) and of the argument /
// capacity errors reported to the caller (-1, -2)
constexpr int FF_FALLBACK = -1000;

// Kernel-path switches: each forces a path the library also picks by itself for some inputs, so that tests can compare
// it with the default path at sizes where both run.  Set explicitly through ff_set_option, process-wide atomics.  The
// library never reads the environment.  0 = default behaviour for every option.
enum Opt {
    OPT_NO_TABLE,            // evaluate every hidden unit instead of the certified Taylor tables
    OPT_FLOW_CTA,            // CTA-synchronous flow sweeps instead of warp-per-walker
    OPT_ELOC_GENERIC,        // generic flow_kernel<MODE_ELOC> instead of the statically specialised eloc kernels
    OPT_SLATER_CTA,          // CTA-cooperative Slater kernel instead of warp-per-walker
    OPT_METROPOLIS_KERNEL,   // 0 auto, 1 registers (thread per walker), 2 warp per walker, 3 thread per walker (shared memory)
    OPT_ADJOINT_CTA,         // CTA-synchronous adjoint sweep
    OPT_PGRAD_DIRECT,        // direct parameter-gradient kernel (every hidden unit) instead of binned Taylor moments
    OPT_COUNT
};
extern std::atomic<int> g_opt[OPT_COUNT];
inline int opt(Opt o) { return g_opt[o].load(std::memory_order_relaxed); }

#define FF_CUDA(call)                                              \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return ffc::cuda_fail(e__, #call); \
    } while (0)

// every kernel launch of the library is counted (ff_launch_count: the "gpu_launches" figure of bench.py)
extern std::atomic<long long> g_launches;
#define FF_LAUNCHED()                                            \
    do {                                                         \
        ffc::g_launches.fetch_add(1, std::memory_order_relaxed); \
        FF_CUDA(cudaGetLastError());                             \
    } while (0)

struct DevInfo { int sms = 0; int smem_optin = 0; int smem_sm = 0; int smem_reserved = 1024; bool ok = false; };
DevInfo dev_info();
int check_model(const ff_model* m);
inline int even(int x) { return (x + 1) & ~1; }

}  // namespace ffc
