// C ABI of fermiflow_b200 (see include/fermiflow_b200.h).  Host-side launch planning only;
// all arithmetic is in the kernels.  The E_loc sweep lives in capi_eloc.cu (separate translation unit).
#define FF_RADIAL_TABLE_KERNELS
#include "capi_flow.h"
#include "ff_adjoint.cuh"
#include "ff_pgrad_binned.cuh"
#include "ff_misc.cuh"
#include "ff_metro_reg.cuh"
#include "ff_observables.cuh"
#include "ff_momentum.cuh"
#include "ff_renyi.cuh"
#include "ff_density_matrix.cuh"

namespace ffc {


thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int cuda_fail(cudaError_t e, const char* what) {
    return fail((int)e, "%s: %s", what, cudaGetErrorString(e));
}

// in the order of enum Opt
const char* const kOptNames[] = {
    "no_table", "no_w_balance", "no_rt_cache", "flow_warp_fill", "flow_cta", "flow_big", "eloc_generic", "slater_cta",
    "metropolis_kernel", "adjoint_cta", "pgrad_direct", "pgrad_tile", "pgrad_fixed_range", "adjoint_no_prefetch", "finale_cta",
    "metropolis_no_split"};
static_assert(sizeof(kOptNames) / sizeof(kOptNames[0]) == OPT_COUNT, "one name per option");
std::atomic<int> g_opt[OPT_COUNT];
std::atomic<long long> g_launches{0};

DevInfo dev_info() {
    static thread_local DevInfo di[16];
    int dev = 0;
    cudaGetDevice(&dev);
    DevInfo& d = di[dev & 15];
    if (!d.ok) {
        cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&d.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        cudaDeviceGetAttribute(&d.smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
        cudaDeviceGetAttribute(&d.smem_reserved, cudaDevAttrReservedSharedMemoryPerBlock, dev);
        d.ok = true;
    }
    return d;
}

int check_model(const ff_model* m) {
    if (!m) return fail(-1, "model is null");
    const int n = m->n_up + m->n_dn;
    if (m->n_up < 0 || m->n_dn < 0 || n < 1) return fail(-1, "bad particle numbers %d/%d", m->n_up, m->n_dn);
    if (n > 200) return fail(-1, "n = %d particles exceeds the supported 200", n);
    if (m->H_eta < 1 || m->H_mu < 0) return fail(-1, "bad hidden sizes");
    if (m->nsteps < 1) return fail(-1, "nsteps must be >= 1");
    if (!m->eta_w1 || !m->eta_b1 || !m->eta_w2) return fail(-1, "eta parameters missing");
    if (m->H_mu > 0 && (!m->mu_w1 || !m->mu_b1 || !m->mu_w2)) return fail(-1, "mu parameters missing");
    return 0;
}

int RadialTables::build(const ff_model* m, cudaStream_t stream, ff::FlowArgs& a) {
    a.rt_eta = nullptr; a.rt_mu = nullptr;
    if (opt(OPT_NO_TABLE)) return 0;
    st = stream;
    {   // keep the stream-ordered pool's memory across synchronisation points (default: trimmed at every sync)
        static thread_local bool pool_ready[16] = {};
        int dev = 0;
        cudaGetDevice(&dev);
        if (!pool_ready[dev & 15]) {
            cudaMemPool_t pool;
            if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
                unsigned long long keep = 64ull << 20;
                cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
            }
            pool_ready[dev & 15] = true;
        }
    }
    const size_t per = ff::radial_table_doubles();
    FF_CUDA(cudaMallocAsync((void**)&buf, 2 * per * sizeof(double), st));
    ff::RadialBuildArgs b{};
    b.w1[0] = m->eta_w1; b.b1[0] = m->eta_b1; b.w2[0] = m->eta_w2; b.H[0] = m->H_eta; b.table[0] = buf;
    b.w1[1] = m->mu_w1; b.b1[1] = m->mu_b1; b.w2[1] = m->mu_w2; b.H[1] = m->H_mu; b.table[1] = m->H_mu > 0 ? buf + per : nullptr;
    ff::radial_table_build_kernel<<<dim3(ff::kRtMaxNodes / 128, 2), 128, 0, st>>>(b);
    FF_LAUNCHED();
    ff::radial_table_check_kernel<<<dim3(1, 2), 128, 0, st>>>(b.table[0], b.table[1]);
    FF_LAUNCHED();
    a.rt_eta = b.table[0]; a.rt_mu = b.table[1];
    return 0;
}

}  // namespace ffc

using namespace ffc;

extern "C" {

int ff_version(void) { return 200; }

long long ff_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int ff_set_option(const char* name, int value) {
    if (!name) return fail(-1, "ff_set_option: null name");
    for (int k = 0; k < OPT_COUNT; ++k)
        if (strcmp(name, kOptNames[k]) == 0) { g_opt[k].store(value, std::memory_order_relaxed); return 0; }
    return fail(-1, "ff_set_option: unknown option '%s'", name);
}
int ff_get_option(const char* name, int* value) {
    if (!name || !value) return fail(-1, "ff_get_option: null argument");
    for (int k = 0; k < OPT_COUNT; ++k)
        if (strcmp(name, kOptNames[k]) == 0) { *value = opt((Opt)k); return 0; }
    return fail(-1, "ff_get_option: unknown option '%s'", name);
}
const char* ff_last_error(void) { return g_err; }

int ff_stash_sizes(const ff_model* m, long long B, long long* ny, long long* nc) {
    if (int e = check_model(m)) return e;
    const long long n = m->n_up + m->n_dn, NS = 4LL * m->nsteps;
    const long long P = n * (n - 1) / 2 + (m->H_mu > 0 ? n : 0);
    if (ny) *ny = B * NS * 2 * n;
    if (nc) *nc = B * NS * P * 3;
    return 0;
}

int ff_cnf_generate(const ff_model* m, const double* z, long long B, int reverse, double* x, void* stream) {
    if (int e = check_model(m)) return e;
    if (B < 0 || (B > 0 && (!z || !x))) return fail(-1, "ff_cnf_generate: null buffer");
    ff::FlowArgs a{};
    int threads; size_t smem;
    if (int e = plan_flow(ff::MODE_V, m, a, threads, smem)) return e;
    a.ta = reverse ? m->t1 : m->t0; a.tb = reverse ? m->t0 : m->t1;
    a.B = B; a.x_in = z; a.y_out = x;
    RadialTables rt;
    if (int e = rt.build(m, (cudaStream_t)stream, a)) return e;
    return launch_flow<ff::MODE_V>(a, threads, smem, (cudaStream_t)stream);
}

int ff_cnf_delta_logp(const ff_model* m, const double* x, long long B, double* z, double* delta_logp,
                      double* stash_y, double* stash_c, void* stream) {
    if (int e = check_model(m)) return e;
    if (B < 0 || (B > 0 && !x)) return fail(-1, "ff_cnf_delta_logp: null input");
    const bool stash = stash_y != nullptr;
    if (stash_c && !stash_y) return fail(-1, "ff_cnf_delta_logp: stash_c needs stash_y");
    ff::FlowArgs a{};
    int threads; size_t smem;
    const int mode = stash ? ff::MODE_STASH : ff::MODE_DIV;
    if (int e = plan_flow(mode, m, a, threads, smem)) return e;
    a.ta = m->t1; a.tb = m->t0;
    a.B = B; a.x_in = x; a.y_out = z; a.delta_out = delta_logp;
    a.stash_y = stash_y; a.stash_c = stash_c;
    RadialTables rt;
    if (int e = rt.build(m, (cudaStream_t)stream, a)) return e;
    return stash ? launch_flow<ff::MODE_STASH>(a, threads, smem, (cudaStream_t)stream)
                 : launch_flow<ff::MODE_DIV>(a, threads, smem, (cudaStream_t)stream);
}

#include "capi_rest.inc"
#ifdef FF_PG_TIMING
extern "C" int ff_debug_pg_cycles(unsigned long long* out, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, ff::g_pg_cyc, sizeof(unsigned long long) * 160);
    cudaMemcpyFromSymbol(out + 160, ff::g_pg_maxbin, sizeof(unsigned long long) * 4);
    if (reset) { unsigned long long z[160] = {}; cudaMemcpyToSymbol(ff::g_pg_cyc, z, sizeof z); cudaMemcpyToSymbol(ff::g_pg_maxbin, z, 32); }
    return 0;
}
#endif

}  // extern "C"
