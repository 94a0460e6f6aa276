// Replica swap ratios of spatial regions and their deterministic reduction by particle-number sector
// (ff_swap_ratio, ff_swap_accumulate; include/fermiflow_b200.h has the definitions and the layout of the sums).
//
// A pair p holds two walkers x = x_{pairs[p][0]} and y = x_{pairs[p][1]}.  For region q, x' is x with its particles
// inside A_q replaced by those of y, slot by slot within each spin block (the k-th A-particle of x, in increasing
// particle index, takes the position of the k-th A-particle of y), and y' the reverse; the pair ratio is
//   rho = psi(x') psi(y') / (psi(x) psi(y)),
// 0 when the two replicas have different (n_A_up, n_A_dn).  ff_swap_ratio evaluates C = 2 P (Q + 1) configurations
// -- slot 0 of each side is the walker itself, slot q + 1 its swapped configuration for region q (a plain copy when the
// sectors differ) -- with the flow sweep and the SIGN Slater kernels, as ff_wavefunction_ratio does:
//   renyi_configs_kernel   one thread per slot: the configuration, its occupation row and (slots q + 1) the packed sector
//                          a (n_dn + 1) + b of its side for region q
//   renyi_ratio_kernel     rho from one exponential of the combined exponent, times the four signs
// Membership is decided with every product and sum rounded separately (x x + y y < a a, or x < a): a torch
// restatement reproduces the sectors bit for bit.
//
// ff_swap_accumulate sums the P Q records into [Q][n_sec] cells.  Fixed summation order, no floating-point atomics:
//   renyi_partial_kernel   CTA g takes pairs [g chunk, (g + 1) chunk) in tiles of kRenyiTile pairs; each thread owns
//                          fixed cells (q, sector) or (q, skipped), adds the tile's records in order and the tile sum to
//                          its cells in the CTA's partial row
//   reduce_partial_rows_kernel (ff_misc.cuh)  sums[i] += sum over g = 0, 1, ... of partial[g][i], in CTA order
// The grid depends only on P, Q, n_sec and the device: two calls on the same inputs give bit-identical sums.
#pragma once
#include "ff_common.cuh"

namespace ff {

constexpr int kRenyiMaxQ = 32;

struct RenyiArgs {
    const double* x;            // [B][n][2]
    long long B, P;
    int n, n_up, n_dn, Q, kind; // kind 0: disks |r| < a_q, 1: half-planes x < a_q
    double a[kRenyiMaxQ];
    const int* pairs;           // [P][2]
    const int* walker_state;    // [B] or null
    double* xc;                 // [P][2][Q+1][n][2]
    int* row;                   // [P][2][Q+1] occupation row per configuration (null without walker_state)
    int* sector;                // [P][2][Q]
};

__device__ __forceinline__ bool renyi_inside(int kind, double a, double rx, double ry) {
    return kind == 0 ? __dadd_rn(__dmul_rn(rx, rx), __dmul_rn(ry, ry)) < __dmul_rn(a, a) : rx < a;
}

__global__ void __launch_bounds__(256) renyi_configs_kernel(const RenyiArgs a) {
    const int n = a.n, Q1 = a.Q + 1;
    const long long total = a.P * 2 * Q1;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < total; c += (long long)gridDim.x * blockDim.x) {
        const long long ps = c / Q1;            // pair p = ps / 2, side s = ps % 2
        const int j = (int)(c - ps * Q1);
        const long long p = ps >> 1;
        const int s = (int)(ps & 1);
        const long long w = a.pairs[2 * p + s], v = a.pairs[2 * p + 1 - s];
        const bool ok = w >= 0 && w < a.B && v >= 0 && v < a.B;
        // a pair with a walker index outside [0, B) evaluates walker 0 in every slot (finite, never read out of bounds)
        const double* xw = a.x + (ok ? w : 0) * 2 * n;
        const double* xv = a.x + (ok ? v : 0) * 2 * n;
        double* out = a.xc + c * 2 * n;
        if (a.row) a.row[c] = a.walker_state[ok ? w : 0];
        if (j == 0 || !ok) {
            for (int i = 0; i < 2 * n; ++i) out[i] = xw[i];
            if (j > 0) a.sector[ps * a.Q + j - 1] = -1;
            continue;
        }
        const int q = j - 1, kind = a.kind;
        const double rad = a.a[q];
        int wu = 0, wd = 0, vu = 0, vd = 0;                 // A-particles per spin of w and v
        for (int i = 0; i < n; ++i) {
            const int iw = renyi_inside(kind, rad, xw[2 * i], xw[2 * i + 1]);
            const int iv = renyi_inside(kind, rad, xv[2 * i], xv[2 * i + 1]);
            if (i < a.n_up) { wu += iw; vu += iv; } else { wd += iw; vd += iv; }
        }
        a.sector[ps * a.Q + q] = wu * (a.n_dn + 1) + wd;
        if (wu != vu || wd != vd) {                         // no swapped configuration: a copy, evaluated but unused
            for (int i = 0; i < 2 * n; ++i) out[i] = xw[i];
            continue;
        }
        for (int sp = 0; sp < 2; ++sp) {
            const int i0 = sp ? a.n_up : 0, i1 = sp ? n : a.n_up;
            int k = i0;                                     // the next A-particle of v in this spin block
            for (int i = i0; i < i1; ++i) {
                double rx = xw[2 * i], ry = xw[2 * i + 1];
                if (renyi_inside(kind, rad, rx, ry)) {
                    while (!renyi_inside(kind, rad, xv[2 * k], xv[2 * k + 1])) ++k;
                    rx = xv[2 * k]; ry = xv[2 * k + 1];
                    ++k;
                }
                out[2 * i] = rx;
                out[2 * i + 1] = ry;
            }
        }
    }
}

// ratio[p][q] from log p = lp0 - dl and the signs of slots (p, s, 0) and (p, s, q + 1): NaN for a pair with a walker
// index outside [0, B) (sector -1), 0 for different sectors, exactly 1 for a region that holds no particle of either
// replica (x' = x, y' = y)
__global__ void __launch_bounds__(256) renyi_ratio_kernel(long long P, int Q, const int* sector, const double* lp0,
                                                          const double* dl, const double* sgn, double* ratio) {
    const long long R = P * Q;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (long long)gridDim.x * blockDim.x) {
        const long long p = r / Q;
        const int q = (int)(r - p * Q);
        const int s0 = sector[(2 * p) * Q + q], s1 = sector[(2 * p + 1) * Q + q];
        double v;
        if (s0 < 0) v = __longlong_as_double(0x7ff8000000000000LL);
        else if (s0 != s1) v = 0.0;
        else if (s0 == 0) v = 1.0;
        else {
            const long long x0 = (2 * p) * (Q + 1), y0 = x0 + Q + 1, x1 = x0 + q + 1, y1 = y0 + q + 1;
            const double e = ((lp0[x1] - dl[x1]) + (lp0[y1] - dl[y1])) - ((lp0[x0] - dl[x0]) + (lp0[y0] - dl[y0]));
            v = (sgn[x1] * sgn[y1]) * (sgn[x0] * sgn[y0]) * exp(0.5 * e);
        }
        ratio[r] = v;
    }
}

constexpr int kRenyiThreads = 256;
constexpr int kRenyiTile = 64;                  // pairs per shared-memory tile: kRenyiTile * Q * 16 bytes <= 32 KB

struct RenyiAccArgs {
    const double* ratio;        // [P][Q]
    const int* sector;          // [P][2][Q]
    long long P;
    int Q, n_sec;
    long long n_sums;           // 3 Q n_sec + Q + 1
    long long chunk;            // pairs per CTA
    double* partial;            // [gridDim.x][n_sums]
};

__global__ void __launch_bounds__(kRenyiThreads) renyi_partial_kernel(const RenyiAccArgs a) {
    extern __shared__ __align__(16) double renyi_smem[];
    const int Q = a.Q, ns = a.n_sec, units = Q * (ns + 1);
    double* rt = renyi_smem;                                    // [kRenyiTile][Q] ratio
    int* st = reinterpret_cast<int*>(rt + kRenyiTile * Q);      // [kRenyiTile][2][Q] sectors
    const long long cells = (long long)Q * ns;
    double* part = a.partial + (long long)blockIdx.x * a.n_sums;
    const long long p0 = (long long)blockIdx.x * a.chunk, p1 = min(a.P, p0 + a.chunk);
    // unit u: q = u / (n_sec + 1), k = u % (n_sec + 1); k < n_sec owns cell (q, k) of the three [Q][n_sec] sections,
    // k = n_sec the skipped counter of q
    for (int u = threadIdx.x; u < units; u += blockDim.x) {
        const int q = u / (ns + 1), k = u - q * (ns + 1);
        if (k < ns) { const long long o = (long long)q * ns + k; part[o] = 0.0; part[cells + o] = 0.0; part[2 * cells + o] = 0.0; }
        else part[3 * cells + q] = 0.0;
    }
    if (threadIdx.x == 0) part[3 * cells + Q] = (double)max(0LL, p1 - p0);
    for (long long t0 = p0; t0 < p1; t0 += kRenyiTile) {
        const int nt = (int)min((long long)kRenyiTile, p1 - t0);
        __syncthreads();                                        // the previous tile is consumed
        for (int e = threadIdx.x; e < nt * Q; e += blockDim.x) rt[e] = a.ratio[t0 * Q + e];
        for (int e = threadIdx.x; e < 2 * nt * Q; e += blockDim.x) st[e] = a.sector[t0 * 2 * Q + e];
        __syncthreads();
        for (int u = threadIdx.x; u < units; u += blockDim.x) {
            const int q = u / (ns + 1), k = u - q * (ns + 1);
            if (k < ns) {
                double sr = 0.0, rep = 0.0, mat = 0.0;
                for (int r = 0; r < nt; ++r) {
                    const int s0 = st[(2 * r) * Q + q], s1 = st[(2 * r + 1) * Q + q];
                    if ((unsigned)s0 >= (unsigned)ns || (unsigned)s1 >= (unsigned)ns) continue;
                    rep += (s0 == k) + (s1 == k);
                    if (s0 == k && s1 == k) { mat += 1.0; sr += rt[r * Q + q]; }
                }
                const long long o = (long long)q * ns + k;
                part[o] += sr;
                part[cells + o] += rep;
                part[2 * cells + o] += mat;
            } else {
                double sk = 0.0;
                for (int r = 0; r < nt; ++r) {
                    const int s0 = st[(2 * r) * Q + q], s1 = st[(2 * r + 1) * Q + q];
                    sk += (unsigned)s0 >= (unsigned)ns || (unsigned)s1 >= (unsigned)ns;
                }
                part[3 * cells + q] += sk;
            }
        }
    }
}

}  // namespace ff
