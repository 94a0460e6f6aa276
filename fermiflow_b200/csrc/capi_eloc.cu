// C ABI, E_loc sweep (ff_eloc): statically specialised kernels for the particle numbers of the BASELINE.json configs,
// generic flow_kernel<MODE_ELOC> otherwise.  Separate translation unit (the kernels dominate the build time).
#include "capi_flow.h"
#include "ff_eloc5.cuh"

using namespace ffc;

namespace {

// Finale from the final states in global memory (fin: `stride` doubles per walker): one warp per walker
// (ff_finale.cuh).  eloc5_kernel runs for N = 6 ... 20, i.e. NB8 = ceil(2 N / 8) = 2 ... 5.
template <int NB8>
int launch_finale_warp(const ff::FlowArgs& a, const double* fin, int stride, cudaStream_t st) {
    const DevInfo di = dev_info();
    const int warps = 4;
    const size_t smem = (size_t)warps * ff::finale_warp_slice(a.n, std::max(a.n_up, a.n - a.n_up)) * 8;
    auto kernel = ff::eloc_finale_warp_kernel<NB8>;
    if ((long long)smem > di.smem_optin) return fail(-2, "E_loc finale: n = %d needs %zu bytes of shared memory", a.n, smem);
    FF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    FF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, 32 * warps, smem));
    if (occ < 1) return fail(-2, "E_loc finale kernel does not fit (n = %d)", a.n);
    const long long grid = std::min<long long>((a.B + warps - 1) / warps, (long long)di.sms * occ);
    kernel<<<(unsigned)grid, 32 * warps, smem, st>>>(a, fin, stride);
    FF_LAUNCHED();
    return 0;
}

int launch_finale(const ff::FlowArgs& a, const double* fin, int stride, cudaStream_t st) {
    switch ((2 * a.n + 7) / 8) {
        case 2: return launch_finale_warp<2>(a, fin, stride, st);
        case 3: return launch_finale_warp<3>(a, fin, stride, st);
        case 4: return launch_finale_warp<4>(a, fin, stride, st);
        case 5: return launch_finale_warp<5>(a, fin, stride, st);
        default: return fail(-2, "E_loc finale: no kernel for n = %d", a.n);
    }
}

// Register-resident sweep (ff_eloc5.cuh eloc5_kernel) + finale kernel.
int launch_eloc_reg(void (*kernel)(const ff::FlowArgs, double*, int*), int threads, size_t smem, int fin_stride, ff::FlowArgs& a, cudaStream_t st) {
    const DevInfo di = dev_info();
    if (a.B < 1) return 0;
    if ((long long)smem > di.smem_optin) return FF_FALLBACK;
    // final states of the sweep for the finale kernel: stream-ordered allocation from the device's default pool, which is
    // told once to keep what it has instead of returning it to the driver at every synchronisation (0.9 GB at 65536
    // walkers: re-mapping it costs ~10 ms per call)
    {
        static thread_local bool pool_set[16] = {};
        int dev = 0;
        FF_CUDA(cudaGetDevice(&dev));
        if (dev < 16 && !pool_set[dev]) {
            cudaMemPool_t pool;
            FF_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
            unsigned long long keep = ~0ull;
            FF_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
            pool_set[dev] = true;
        }
    }
    double* fin = nullptr;
    // (+ 1 KB behind the final states: per-SM counters by which the co-resident CTAs of eloc5_kernel tell themselves apart)
    const size_t fin_bytes = (size_t)a.B * fin_stride * sizeof(double);
    FF_CUDA(cudaMallocAsync((void**)&fin, fin_bytes + 1024, st));
    FF_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(fin) + fin_bytes, 0, 1024, st));
    int* const sm_count = reinterpret_cast<int*>(reinterpret_cast<char*>(fin) + fin_bytes);
    struct Release { double* p; cudaStream_t s; ~Release() { cudaFreeAsync(p, s); } } release{fin, st};
    FF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // as many walkers per SM as registers and shared memory allow (two at N = 20, more for smaller blocks); what is left of
    // the 256 KB stays L1 (the tails of the Taylor tables of the radial functions live there)
    FF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    int occ = 0;
    FF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem));
    if (occ < 1) return FF_FALLBACK;
    const int carve = (int)std::min<long long>(100, ((long long)occ * ((long long)smem + di.smem_reserved) * 100 + di.smem_sm - 1) / di.smem_sm);
    FF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
    const long long grid = std::min<long long>(a.B, (long long)di.sms * occ);
    kernel<<<(unsigned)grid, threads, smem, st>>>(a, fin, sm_count);
    FF_LAUNCHED();
    return launch_finale(a, fin, fin_stride, st);
}
template <int SN, int SMU>
int launch_eloc5(ff::FlowArgs& a, cudaStream_t st) {
    constexpr ff::Eloc5Geom g = ff::eloc5_geom(SN, SMU != 0);
    // two CTAs per SM with the whole shared-memory carve-out: what the walker block leaves of a CTA's half mirrors the
    // head of the eta table (ff::kRtPitch doubles per node)
    const DevInfo di = dev_info();
    const long long half = std::min<long long>(di.smem_sm / 2 - di.smem_reserved, di.smem_optin);
    const long long room = half - (long long)g.total * 8;
    // (at most 256 rows: small walker blocks leave the shared memory to more resident CTAs instead)
    a.rt_cache_nodes = (a.rt_eta != nullptr && room > 0) ? (int)std::min<long long>(room / (8 * ff::kRtPitch), 256) : 0;
    size_t smem = (size_t)(g.total + a.rt_cache_nodes * ff::kRtPitch) * 8;
#ifdef FF_DEV_ONE_CTA
    smem = std::max<size_t>(smem, (size_t)di.smem_sm / 2 + 4096);          // (dev experiment: one resident CTA per SM)
#endif
    return launch_eloc_reg(ff::eloc5_kernel<SN, SMU>, g.threads, smem, g.fin_stride, a, st);
}

// Statically specialised E_loc sweep (ff_eloc5.cuh) for the particle numbers it is instantiated for; anything else, or
// "eloc_generic", runs the generic flow_kernel<MODE_ELOC>.  Without the Taylor tables ("no_table") every item of the
// static sweep takes its direct-evaluation path.
int try_eloc_static(ff::FlowArgs& a, cudaStream_t st) {
    if (opt(OPT_ELOC_GENERIC)) return FF_FALLBACK;
    if (a.H_mu > 0) {
        switch (a.n) {       // one walker per CTA; below 6 particles the generic sweep packs several walkers into a CTA
            case 20: return launch_eloc5<20, 1>(a, st);
            case 19: return launch_eloc5<19, 1>(a, st);
            case 18: return launch_eloc5<18, 1>(a, st);
            case 17: return launch_eloc5<17, 1>(a, st);
            case 16: return launch_eloc5<16, 1>(a, st);
            case 15: return launch_eloc5<15, 1>(a, st);
            case 14: return launch_eloc5<14, 1>(a, st);
            case 13: return launch_eloc5<13, 1>(a, st);
            case 12: return launch_eloc5<12, 1>(a, st);
            case 11: return launch_eloc5<11, 1>(a, st);
            case 10: return launch_eloc5<10, 1>(a, st);
            case 9: return launch_eloc5<9, 1>(a, st);
            case 8: return launch_eloc5<8, 1>(a, st);
            case 7: return launch_eloc5<7, 1>(a, st);
            case 6: return launch_eloc5<6, 1>(a, st);
            default: return FF_FALLBACK;
        }
    }
    switch (a.n) {           // reference drivers' --nomu: no one-body backflow
        case 20: return launch_eloc5<20, 0>(a, st);
        case 12: return launch_eloc5<12, 0>(a, st);
        case 6: return launch_eloc5<6, 0>(a, st);
        default: return FF_FALLBACK;
    }
}

}  // namespace

extern "C" {

#ifdef FF_E5_TIMING
int ff_debug_e5_cycles(unsigned long long* out, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, ff::g_e5_cyc, sizeof(unsigned long long) * 64);
    if (reset) { unsigned long long z[64] = {}; cudaMemcpyToSymbol(ff::g_e5_cyc, z, sizeof z); }
    return 0;
}
#endif

int ff_eloc(const ff_model* m, const double* x, long long B, const int* orb, const int* walker_state,
            double Z, int harmonic, double* z, double* delta_logp, double* logp, double* grad,
            double* lap, double* kinetic, double* potential, double* eloc,
            double* stash_y, double* stash_c, void* stream) {
    if (int e = check_model(m)) return e;
    if (B < 0 || (B > 0 && (!x || !orb))) return fail(-1, "ff_eloc: null input");
    if (stash_c && !stash_y) return fail(-1, "ff_eloc: stash_c needs stash_y");
    ff::FlowArgs a{};
    int threads; size_t smem;
    bool jglobal = false;
    if (int e = plan_flow(ff::MODE_ELOC, m, a, threads, smem, jglobal)) return e;
    a.ta = m->t1; a.tb = m->t0;
    a.B = B; a.x_in = x; a.y_out = z; a.delta_out = delta_logp;
    a.stash_y = stash_y; a.stash_c = stash_c;
    a.orb = orb; a.walker_state = walker_state; a.Z = Z; a.harmonic = harmonic;
    a.logp = logp; a.grad = grad; a.lap = lap; a.kin = kinetic; a.pot = potential; a.eloc = eloc;
    RadialTables rt;
    if (int e = rt.build(m, (cudaStream_t)stream, a)) return e;
    {
        ff::FlowArgs a2 = a;
        const int r = try_eloc_static(a2, (cudaStream_t)stream);
        if (r != FF_FALLBACK) return r;
    }
    // particle numbers beyond the shared-memory budget (n > 26): RK partials of J in a stream-ordered global scratch,
    // one slot per walker of every CTA the device can hold
    struct Scratch { double* p = nullptr; cudaStream_t s = nullptr; ~Scratch() { if (p) cudaFreeAsync(p, s); } } scratch;
    if (jglobal) {
        const DevInfo di = dev_info();
        const long long ctas = (long long)di.sms * std::max<long long>(1, (long long)di.smem_sm / (long long)smem);
        scratch.s = (cudaStream_t)stream;
        FF_CUDA(cudaMallocAsync((void**)&scratch.p, (size_t)ctas * a.W * 4 * a.D * a.D * sizeof(double), scratch.s));
        a.jpart = scratch.p;
    }
    return launch_flow<ff::MODE_ELOC>(a, threads, smem, (cudaStream_t)stream);
}

}  // extern "C"
