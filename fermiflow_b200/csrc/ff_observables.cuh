// Histograms of sampled walkers x [B][n][2] for the spin-resolved one-body density, radial density, pair-separation
// distribution and rotated-frame pair density (ff_observables, include/fermiflow_b200.h has the layout of the counts).
//
// Binning rule, shared bit for bit with the torch restatement in the tests: with s = nbins / (hi - lo) computed on the
// host in double, an item of value v goes to bin k = floor((v - lo) * s); k < 0, k >= nbins or a non-finite v sends it
// to the section's per-channel outside counter, and so does a reference particle at |r_i| == 0 in the rotated section.
// nvcc contracts a*b + c into an FMA by default and the torch restatement rounds every product, so every product that
// feeds a sum or difference is written with __dmul_rn / __dadd_rn / __dsub_rn (the intrinsics are never contracted);
// sqrt and / are IEEE round-to-nearest already.
//
// Each CTA keeps private unsigned int bins in shared memory (integer shared atomics are native on sm_100a, fp64 ones
// are CAS loops: scripts/ubench/smem_atomics.cu) and adds its non-zero bins to the global 64-bit counts before any
// private bin could exceed 2^32 - 1.  Integer counts make the result independent of the order of execution.
#pragma once
#include "ff_common.cuh"

namespace ff {

enum ObsSection { OBS_DENSITY = 0, OBS_RADIAL = 1, OBS_SEPARATION = 2, OBS_ROTATED = 3, OBS_SECTIONS = 4 };

struct ObsArgs {
    const double* x;
    long long B;
    int n, n_up;
    int mask;                       // sections of this launch (bit OBS_*)
    int nb[OBS_SECTIONS];           // bins per channel and axis: n_xy, n_r, n_r, n_rot
    double lo[OBS_SECTIONS];        // lower edge: -extent, 0, 0, -extent
    double s[OBS_SECTIONS];         // nbins / (hi - lo)
    long long goff[OBS_SECTIONS];   // first bin of the section in counts
    long long outside_off;          // first of the 9 outside counters in counts
    int soff[OBS_SECTIONS];         // first bin of the section in shared memory (sections of this launch)
    int sbins;                      // bins of this launch in shared memory; the 9 outside counters follow
    unsigned items;                 // items per walker of this launch
    int first[OBS_SECTIONS + 1];    // item ranges of the sections inside a walker (empty for sections not launched)
    long long chunk;                // walkers per flush (items * chunk + blockDim <= 2^32 - 1)
    unsigned long long* counts;
};

constexpr int kObsOutside = 9;
// first outside counter of each section: density up, down | radial up, down | separation uu, dd, ud | rotated same, opposite
__device__ constexpr int kObsOutsideFirst[OBS_SECTIONS] = {0, 2, 4, 7};
constexpr int kObsThreads = 256;

// bin of v in [lo, lo + nb / s), -1 outside (NaN and +-inf included: the comparisons are false)
__device__ __forceinline__ int obs_bin(double v, double lo, double s, int nb) {
    const double f = floor(__dmul_rn(__dsub_rn(v, lo), s));
    return (f >= 0.0 && f < (double)nb) ? (int)f : -1;
}

__device__ __forceinline__ double obs_norm(double x, double y) { return sqrt(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y))); }

// unordered pair p of n particles (row-major over i < j)
__device__ __forceinline__ void obs_pair(int p, int n, int& i, int& j) {
    const double b = 2.0 * n - 1.0;
    int r = (int)floor(0.5 * (b - sqrt(b * b - 8.0 * p)));
    r = max(0, min(r, n - 2));
    while (r > 0 && r * (2 * n - r - 1) / 2 > p) --r;
    while ((r + 1) * (2 * n - r - 2) / 2 <= p) ++r;
    i = r;
    j = p - r * (2 * n - r - 1) / 2 + r + 1;
}

__global__ void __launch_bounds__(kObsThreads) observables_kernel(const ObsArgs a) {
    extern __shared__ __align__(16) unsigned obs_smem[];
    const int nsh = a.sbins + kObsOutside;
    unsigned* out = obs_smem + a.sbins;
    for (int k = threadIdx.x; k < nsh; k += blockDim.x) obs_smem[k] = 0u;
    const int n = a.n, n_up = a.n_up;
    const long long nchunks = (a.B + a.chunk - 1) / a.chunk;
    for (long long c = blockIdx.x; c < nchunks; c += gridDim.x) {
        __syncthreads();
        const long long w0 = c * a.chunk;
        const long long nw = min(a.chunk, a.B - w0);
        const unsigned total = (unsigned)nw * a.items;
        const double* xc = a.x + w0 * 2 * n;
        for (unsigned t = threadIdx.x; t < total; t += blockDim.x) {
            const unsigned w = t / a.items;
            const int it = (int)(t - w * a.items);
            const double* xw = xc + (size_t)w * 2 * n;
            if (it < a.first[OBS_RADIAL]) {                                    // one-body density
                const int i = it - a.first[OBS_DENSITY], ch = i >= n_up;
                const double2 r = make_double2(xw[2 * i], xw[2 * i + 1]);
                const int nb = a.nb[OBS_DENSITY];
                const int kx = obs_bin(r.x, a.lo[OBS_DENSITY], a.s[OBS_DENSITY], nb);
                const int ky = obs_bin(r.y, a.lo[OBS_DENSITY], a.s[OBS_DENSITY], nb);
                if (kx < 0 || ky < 0) atomicAdd(out + kObsOutsideFirst[OBS_DENSITY] + ch, 1u);
                else atomicAdd(obs_smem + a.soff[OBS_DENSITY] + (ch * nb + kx) * nb + ky, 1u);
            } else if (it < a.first[OBS_SEPARATION]) {                         // radial density
                const int i = it - a.first[OBS_RADIAL], ch = i >= n_up;
                const double2 r = make_double2(xw[2 * i], xw[2 * i + 1]);
                const int nb = a.nb[OBS_RADIAL];
                const int k = obs_bin(obs_norm(r.x, r.y), a.lo[OBS_RADIAL], a.s[OBS_RADIAL], nb);
                if (k < 0) atomicAdd(out + kObsOutsideFirst[OBS_RADIAL] + ch, 1u);
                else atomicAdd(obs_smem + a.soff[OBS_RADIAL] + ch * nb + k, 1u);
            } else if (it < a.first[OBS_ROTATED]) {                            // pair separation, i < j
                int i, j;
                obs_pair(it - a.first[OBS_SEPARATION], n, i, j);
                const int ch = (i < n_up) == (j < n_up) ? (i < n_up ? 0 : 1) : 2;
                const double2 ri = make_double2(xw[2 * i], xw[2 * i + 1]);
                const double2 rj = make_double2(xw[2 * j], xw[2 * j + 1]);
                const int nb = a.nb[OBS_SEPARATION];
                const int k = obs_bin(obs_norm(__dsub_rn(ri.x, rj.x), __dsub_rn(ri.y, rj.y)), a.lo[OBS_SEPARATION],
                                      a.s[OBS_SEPARATION], nb);
                if (k < 0) atomicAdd(out + kObsOutsideFirst[OBS_SEPARATION] + ch, 1u);
                else atomicAdd(obs_smem + a.soff[OBS_SEPARATION] + ch * nb + k, 1u);
            } else {                                                           // rotated frame, i != j
                const int q = it - a.first[OBS_ROTATED];
                const int i = q / (n - 1), jj = q - i * (n - 1), j = jj + (jj >= i);
                const int ch = (i < n_up) != (j < n_up);
                const double2 ri = make_double2(xw[2 * i], xw[2 * i + 1]);
                const double2 rj = make_double2(xw[2 * j], xw[2 * j + 1]);
                const double ni = obs_norm(ri.x, ri.y);
                const double u = __dadd_rn(__dmul_rn(ri.x, rj.x), __dmul_rn(ri.y, rj.y)) / ni;
                const double v = __dsub_rn(__dmul_rn(ri.x, rj.y), __dmul_rn(ri.y, rj.x)) / ni;
                const int nb = a.nb[OBS_ROTATED];
                const int ku = obs_bin(u, a.lo[OBS_ROTATED], a.s[OBS_ROTATED], nb);
                const int kv = obs_bin(v, a.lo[OBS_ROTATED], a.s[OBS_ROTATED], nb);
                if (ni == 0.0 || ku < 0 || kv < 0) atomicAdd(out + kObsOutsideFirst[OBS_ROTATED] + ch, 1u);
                else atomicAdd(obs_smem + a.soff[OBS_ROTATED] + (ch * nb + ku) * nb + kv, 1u);
            }
        }
        // flush: a chunk holds at most (2^32 - 1 - blockDim) / items walkers, so no private bin can wrap
        __syncthreads();
        for (int s = 0; s < OBS_SECTIONS; ++s) {
            if (!(a.mask >> s & 1)) continue;
            const int nch = s == OBS_SEPARATION ? 3 : 2;
            const int bins = nch * ((s == OBS_DENSITY || s == OBS_ROTATED) ? a.nb[s] * a.nb[s] : a.nb[s]);
            for (int k = threadIdx.x; k < bins; k += blockDim.x) {
                const unsigned v = obs_smem[a.soff[s] + k];
                if (v) { atomicAdd(a.counts + a.goff[s] + k, (unsigned long long)v); obs_smem[a.soff[s] + k] = 0u; }
            }
            if (threadIdx.x < nch) {
                const int o = kObsOutsideFirst[s] + threadIdx.x;
                const unsigned v = out[o];
                if (v) { atomicAdd(a.counts + a.outside_off + o, (unsigned long long)v); out[o] = 0u; }
            }
        }
    }
}

}  // namespace ff
