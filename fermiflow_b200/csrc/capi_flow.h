// Launch planning of the flow sweeps (generate / delta_logp / generic E_loc), shared by capi.cu and capi_eloc.cu.
#pragma once
#include "capi_common.h"
#include "ff_flow.cuh"
#include "ff_flow_warp.cuh"

namespace ffc {

// Certified Taylor tables of the radial functions for one sweep launch (ff_radial_table.cuh): built from
// the current parameters on the launch stream, released stream-ordered after the sweep (definition: capi.cu).
// Option "no_table" keeps the direct evaluation of every hidden unit.
struct RadialTables {
    double* buf = nullptr;
    cudaStream_t st = nullptr;
    int build(const ff_model* m, cudaStream_t stream, ff::FlowArgs& a);
    ~RadialTables() { if (buf) cudaFreeAsync(buf, st); }
};

// Fills the geometry fields of FlowArgs and returns threads / dynamic smem bytes.
inline int plan_flow(int mode, const ff_model* m, ff::FlowArgs& a, int& threads, size_t& smem, bool& jglobal);
inline int plan_flow(int mode, const ff_model* m, ff::FlowArgs& a, int& threads, size_t& smem) {
    bool jglobal = false;
    return plan_flow(mode, m, a, threads, smem, jglobal);
}
inline int plan_flow(int mode, const ff_model* m, ff::FlowArgs& a, int& threads, size_t& smem, bool& jglobal) {
    jglobal = false;
    const DevInfo di = dev_info();
    const int n = m->n_up + m->n_dn;
    a.n = n; a.n_up = m->n_up; a.H_eta = m->H_eta; a.H_mu = m->H_mu;
    a.eta_w1 = m->eta_w1; a.eta_b1 = m->eta_b1; a.eta_w2 = m->eta_w2;
    a.mu_w1 = m->mu_w1; a.mu_b1 = m->mu_b1; a.mu_w2 = m->mu_w2;
    a.nsteps = m->nsteps;
    const bool eloc = mode == ff::MODE_ELOC;
    ff::FlowGeom g = ff::flow_geom(mode, n, m->H_mu > 0);
    const int fin_need = eloc ? ff::slater_scratch_size(m->n_up, m->n_dn) + 2 * g.D + n * n + g.NP + 8 : 0;
    a.jpart = nullptr;
    if (eloc) {
        // a walker whose blocks do not fit in shared memory keeps the RK partials of J in global memory (the caller
        // allocates FlowArgs::jpart when jglobal comes back set)
        int common0 = ff::kTabDoubles + 6 * (((m->H_eta + 3) & ~3) + ((m->H_mu + 3) & ~3));
        common0 = even(common0) + 2 * ((g.NP + 7) / 8) + 2;
        if ((long long)di.smem_optin / 8 - common0 < g.wstride) { g = ff::flow_geom(mode, n, m->H_mu > 0, true, even(fin_need)); jglobal = true; }
    }
    a.D = g.D; a.NP = g.NP; a.P = g.P; a.DP = g.DP; a.NV = g.NV; a.NSV = g.NSV; a.NPAR = g.NPAR; a.grec = g.grec;
    a.off_G = g.off_G; a.off_AM = g.off_AM; a.off_u = g.off_u; a.off_kLx = g.off_kLx; a.off_part = g.off_part;
    a.off_x0 = g.off_x0; a.off_sl = g.off_sl; a.wstride = g.wstride;
    if (a.P < 1) return fail(-1, "a single particle without one-body backflow has no velocity field");
    if (eloc) {
        if (fin_need > g.off_G - g.NSV) return fail(-2, "internal: finale scratch does not fit");
    }
    int common = ff::kTabDoubles + 6 * (((m->H_eta + 3) & ~3) + ((m->H_mu + 3) & ~3));
    common = even(common) + 2 * ((a.NP + 7) / 8) + 2;
    // E_loc sweep: aim for two resident CTAs per SM (their FP64-bound and shared-memory-bound
    // phases overlap), fall back to one large CTA when a walker does not fit in half an SM.
    long long budget = (long long)di.smem_optin / 8 - common;
    int target_threads = eloc ? 512 : 256;
    if (eloc) {
        const long long half = ((long long)di.smem_sm / 2 - di.smem_reserved) / 8 - common;
        if (half >= a.wstride && a.P <= 256) { budget = half; target_threads = 256; }
    }
    int W = (int)(budget / a.wstride);
    if (W > target_threads / a.P) W = target_threads / a.P;
    if (a.P > 512) return fail(-2, "n = %d needs %d threads per walker (> 512)", n, a.P);
    if (W < 1) {
        if (budget / a.wstride < 1)
            return fail(-2, "n = %d needs %lld bytes of shared memory per walker, device allows %d",
                        n, (long long)(a.wstride + common) * 8, di.smem_optin);
        W = 1;
    }
    a.W = W;
    threads = ((W * a.P + 31) / 32) * 32;
    if (threads < 64) threads = 64;
    // helper warp: its Gram matrix overlaps the MLP loop of the item warps (direct evaluation only; with the
    // Taylor tables the item phase is short and every warp shares the Gram matrix)
    if (eloc && threads + 32 <= 256 && opt(OPT_NO_TABLE)) threads += 32;
    smem = (size_t)(common + (long long)W * a.wstride) * 8;
    return 0;
}

template <class K>
int launch_flow_kernel(K kernel, ff::FlowArgs& a, int threads, size_t smem, cudaStream_t st) {
    const DevInfo di = dev_info();
    FF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    FF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    int occ = 0;
    FF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem));
    if (occ < 1) return fail(-2, "flow kernel does not fit on an SM (threads %d, smem %zu)", threads, smem);
    long long nb = (a.B + a.W - 1) / a.W;
    long long grid = (long long)di.sms * occ;
    if (a.W > 1 && a.B > 0) {
        // several walkers per CTA (small n): spread them evenly over the rounds the resident CTAs need anyway --
        // 8000 walkers at W = 26 are 308 tasks for 296 CTAs (two rounds, the second almost empty); W = 14 gives 572
        // tasks, two full rounds of half the length.  threads / smem were sized for the larger W and stay valid.
        const long long rounds = (nb + grid - 1) / grid;
        const long long Wb = (a.B + rounds * grid - 1) / (rounds * grid);
        if (Wb < a.W) { a.W = (int)std::max<long long>(1, Wb); nb = (a.B + a.W - 1) / a.W; }
    }
    if (grid > nb) grid = nb;
    if (grid < 1) return 0;
    kernel<<<(unsigned)grid, threads, smem, st>>>(a);
    FF_LAUNCHED();
    return 0;
}

// One-warp-per-walker sweeps (ff_flow_warp.cuh) when the pair items fill the lanes well.
template <int MODE>
int launch_flow_warp(ff::FlowArgs& a, cudaStream_t st) {
    const DevInfo di = dev_info();
    const ff::WarpFlowGeom wg = ff::warp_flow_geom(MODE, a.n, a.P);
    const int warps = 8;
    int common = ff::kTabDoubles + 6 * (((a.H_eta + 3) & ~3) + ((a.H_mu + 3) & ~3));
    common = even(common) + 2 * ((a.NP + 7) / 8) + 2;
    size_t smem = (size_t)(common + (long long)warps * wg.slice) * 8;
    if (smem > (size_t)di.smem_optin) return FF_FALLBACK;
    {   // spare shared memory at FF_WARP_MINB CTAs per SM mirrors the head of the eta Taylor table
        const long long room = (long long)di.smem_sm / FF_WARP_MINB - di.smem_reserved - (long long)smem - 64;
        a.rt_cache_nodes = (a.rt_eta != nullptr && room > 0) ? (int)std::min<long long>(room / (8 * ff::kRtCoef), 2048) : 0;
        smem += (size_t)a.rt_cache_nodes * 8 * ff::kRtCoef;
    }
    auto kernel = ff::flow_warp_kernel<MODE>;
    FF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    FF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    int occ = 0;
    FF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, 32 * warps, smem));
    if (occ < 1) return FF_FALLBACK;
    long long grid = std::min<long long>((a.B + warps - 1) / warps, (long long)di.sms * occ);
    if (grid < 1) return 0;
    kernel<<<(unsigned)grid, 32 * warps, smem, st>>>(a);
    FF_LAUNCHED();
    return 0;
}

template <int MODE>
int launch_flow(ff::FlowArgs& a, int threads, size_t smem, cudaStream_t st) {
    if constexpr (MODE != ff::MODE_ELOC) {
        // lane efficiency of the warp-per-walker layout: NP pair items over ceil(NP / 32) rounds
        const int rounds = (a.NP + 31) / 32;
        // measured (scripts/dev_gen_time_n.py, 65536 walkers): N = 12 (66 pairs, 69 % of three rounds) 7.0 ms CTA-synchronous
        // against 5.7 ms warp-per-walker; N = 9 (36 pairs, 56 %) 4.3 against 4.9 ms; N = 6 (15 pairs, 47 %) 2.0 against 3.8 ms
        constexpr int min_fill = 60;      // per cent of the lanes
        if (a.NP > 0 && a.n <= 255 && 100 * a.NP >= min_fill * 32 * rounds && !opt(OPT_FLOW_CTA)) {
            const int r = launch_flow_warp<MODE>(a, st);
            if (r != FF_FALLBACK) return r;
        }
        if (threads <= 256) return launch_flow_kernel(ff::flow_kernel_small<MODE>, a, threads, smem, st);
    }
    return launch_flow_kernel(ff::flow_kernel<MODE>, a, threads, smem, st);
}


}  // namespace ffc
