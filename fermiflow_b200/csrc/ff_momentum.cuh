// Signed wave-function ratios of one-particle moves and their reduction onto a momentum grid
// (ff_wavefunction_ratio, ff_momentum_accumulate; include/fermiflow_b200.h has the definitions and the layout of the sums).
//
// psi(x) = sign(det Phi_up(z) det Phi_dn(z)) exp(log p(x) / 2), z = flow^-1(x): the flow's Jacobian determinant is
// positive, so the sign comes from the Slater determinants alone.  A record (b, m) moves particle i = particle[b][m] of
// walker b by s = disp[b][m]; its ratio is rho = psi(x_b with r_i -> r_i + s) / psi(x_b).  ff_wavefunction_ratio
// evaluates B (M + 1) configurations -- slot 0 of each walker is x itself, so psi(x) and psi(x') come from the same
// launches -- with the existing flow sweep (MODE_DIV) and the SIGN instantiations of the Slater kernels:
//   wfr_configs_kernel   x -> [B][M+1][n][2] configurations and one occupation row per configuration
//   wfr_ratio_kernel     rho = sgn' sgn0 exp(((lp0' - dl') - (lp0 - dl)) / 2); NaN for a particle outside [0, n)
//
// ff_momentum_accumulate sums, per spin channel c = (i >= n_up), rho cos(k.s) on a square k grid, rho J0(k |s|) on a
// radial k grid, and rho and the record count in |s| bins.  Fixed summation order, no floating-point atomics:
//   momentum_partial_kernel  CTA g takes records [g chunk, (g + 1) chunk) in tiles of `tile` records.  Per tile the
//                            CTA tabulates rho cos / sin(kx_a s_x), cos / sin(ky_b s_y) (2 n_k sincos per record) and
//                            rho J0(k_j |s|) in shared memory; then each thread owns a fixed set of output "units"
//                            (a k cell, a radial point, an |s| bin, ...) for both channels, sums the tile's records in
//                            order and adds the tile sum to its units in the CTA's partial row.
//   reduce_partial_rows_kernel (ff_misc.cuh)  sums[q] += sum over g = 0, 1, ... of partial[g][q], in CTA order.
// The grid (and so the rounding) depends only on R, the grid sizes and the device: two calls on the same inputs give
// bit-identical sums.
#pragma once
#include "ff_common.cuh"

namespace ff {

struct WfrArgs {
    const double* x;            // [B][n][2]
    long long B;
    int n, M;
    const int* particle;        // [B][M]
    const double* disp;         // [B][M][2]
    const int* walker_state;    // [B] or null
    double* xc;                 // [B][M+1][n][2]
    int* row;                   // [B][M+1] occupation row per configuration (null without walker_state)
};

__global__ void __launch_bounds__(256) wfr_configs_kernel(const WfrArgs a) {
    const int n = a.n, M1 = a.M + 1;
    const long long total = a.B * M1 * n;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const long long c = t / n;
        const int i = (int)(t - c * n);
        const long long b = c / M1;
        const int m = (int)(c - b * M1);
        double rx = a.x[(b * n + i) * 2], ry = a.x[(b * n + i) * 2 + 1];
        if (m > 0) {
            const long long rec = b * a.M + m - 1;
            if (a.particle[rec] == i) { rx += a.disp[2 * rec]; ry += a.disp[2 * rec + 1]; }
        }
        a.xc[2 * t] = rx;
        a.xc[2 * t + 1] = ry;
        if (i == 0 && a.row) a.row[c] = a.walker_state[b];
    }
}

__global__ void __launch_bounds__(256) wfr_ratio_kernel(long long B, int n, int M, const int* particle, const double* lp0,
                                                        const double* dl, const double* sgn, double* ratio) {
    const long long R = B * M;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (long long)gridDim.x * blockDim.x) {
        const long long b = r / M;
        const long long c0 = b * (M + 1), c1 = c0 + (r - b * M) + 1;
        const int i = particle[r];
        double v = __longlong_as_double(0x7ff8000000000000LL);            // NaN: no such particle
        if (i >= 0 && i < n) v = sgn[c1] * sgn[c0] * exp(0.5 * ((lp0[c1] - dl[c1]) - (lp0[c0] - dl[c0])));
        ratio[r] = v;
    }
}

constexpr int kMomThreads = 256;
constexpr int kMomMaxTile = 32;

struct MomArgs {
    const double* ratio;        // [R]
    const int* particle;        // [R]
    const double* disp;         // [R][2]
    long long R;
    int n_up;
    int n_k, n_kr, n_s;
    double k_lo, dk;            // square grid: k_a = k_lo + (a + 1/2) dk
    double dkr;                 // radial points: k_j = (j + 1/2) dkr
    double s_scale;             // n_s / s_max: |s| bin = floor(|s| s_scale)
    int units;                  // n_k^2 + n_kr + 2 n_s + 1; unit u has one output per channel
    long long n_sums;           // 2 units
    int tile;                   // records per shared-memory tile (<= kMomMaxTile)
    long long chunk;            // records per CTA
    double* partial;            // [gridDim.x][n_sums]
};

// offsets of the two outputs of unit u in the layout of the sums (channel 0: out0, channel 1: out0 + stride)
__device__ __forceinline__ void mom_unit(const MomArgs& a, int u, int& kind, int& idx, long long& out0, long long& stride) {
    const int g2 = a.n_k * a.n_k;
    if (u < g2) { kind = 0; idx = u; out0 = u; stride = g2; return; }
    u -= g2;
    long long off = 2LL * g2;
    if (u < a.n_kr) { kind = 1; idx = u; out0 = off + u; stride = a.n_kr; return; }
    u -= a.n_kr; off += 2LL * a.n_kr;
    if (u < a.n_s) { kind = 2; idx = u; out0 = off + u; stride = a.n_s; return; }
    u -= a.n_s; off += 2LL * a.n_s;
    if (u < a.n_s) { kind = 3; idx = u; out0 = off + u; stride = a.n_s; return; }
    off += 2LL * a.n_s;
    kind = 4; idx = 0; out0 = off; stride = 1;
}

__global__ void __launch_bounds__(kMomThreads) momentum_partial_kernel(const MomArgs a) {
    extern __shared__ __align__(16) double mom_smem[];
    const int tid = threadIdx.x, T = blockDim.x, TL = a.tile, nk = a.n_k, nkr = a.n_kr;
    double2* px = reinterpret_cast<double2*>(mom_smem);        // [TL][n_k] (rho cos(kx sx), rho sin(kx sx))
    double2* py = px + TL * nk;                                 // [TL][n_k] (cos(ky sy), sin(ky sy))
    double* jr = reinterpret_cast<double*>(py + TL * nk);       // [TL][n_kr] rho J0(k_j |s|)
    double* rho = jr + TL * nkr;                                // [TL]
    double* sabs = rho + TL;                                    // [TL]
    int* bin = reinterpret_cast<int*>(sabs + TL);               // [TL] |s| bin, -1 outside [0, s_max)
    int* ch = bin + TL;                                         // [TL] channel
    double* part = a.partial + (long long)blockIdx.x * a.n_sums;
    for (int u = tid; u < a.units; u += T) {                    // each thread zeroes the outputs it owns
        int kind, idx; long long o, st;
        mom_unit(a, u, kind, idx, o, st);
        part[o] = 0.0;
        part[o + st] = 0.0;
    }
    const long long r0 = (long long)blockIdx.x * a.chunk, r1 = min(a.R, r0 + a.chunk);
    for (long long t0 = r0; t0 < r1; t0 += TL) {
        const int nt = (int)min((long long)TL, r1 - t0);
        __syncthreads();                                        // the previous tile is consumed
        for (int r = tid; r < nt; r += T) {
            const long long g = t0 + r;
            const double sx = a.disp[2 * g], sy = a.disp[2 * g + 1];
            const double s = sqrt(__dadd_rn(__dmul_rn(sx, sx), __dmul_rn(sy, sy)));
            const double f = floor(__dmul_rn(s, a.s_scale));
            rho[r] = a.ratio[g];
            sabs[r] = s;
            bin[r] = (f >= 0.0 && f < (double)a.n_s) ? (int)f : -1;
            ch[r] = a.particle[g] >= a.n_up;
        }
        __syncthreads();
        for (int e = tid; e < nt * nk; e += T) {
            const int r = e / nk, k = e - r * nk;
            const long long g = t0 + r;
            const double kk = a.k_lo + (k + 0.5) * a.dk;
            double sn, cs;
            sincos(kk * a.disp[2 * g], &sn, &cs);
            px[e] = make_double2(rho[r] * cs, rho[r] * sn);
            sincos(kk * a.disp[2 * g + 1], &sn, &cs);
            py[e] = make_double2(cs, sn);
        }
        for (int e = tid; e < nt * nkr; e += T) {
            const int r = e / nkr, j = e - r * nkr;
            jr[e] = rho[r] * j0((j + 0.5) * a.dkr * sabs[r]);
        }
        __syncthreads();
        for (int u = tid; u < a.units; u += T) {
            int kind, idx; long long o, st;
            mom_unit(a, u, kind, idx, o, st);
            double s0 = 0.0, s1 = 0.0;
            if (kind == 0) {                                    // rho cos(k.s) = rho (cx cy - sx sy)
                const int ia = idx / nk, ib = idx - ia * nk;
                for (int r = 0; r < nt; ++r) {
                    const double2 X = px[r * nk + ia], Y = py[r * nk + ib];
                    const double v = fma(X.x, Y.x, -X.y * Y.y);
                    if (ch[r]) s1 += v; else s0 += v;
                }
            } else if (kind == 1) {                             // rho J0(k |s|)
                for (int r = 0; r < nt; ++r) {
                    const double v = jr[r * nkr + idx];
                    if (ch[r]) s1 += v; else s0 += v;
                }
            } else if (kind == 2) {                             // rho in |s| bin idx
                for (int r = 0; r < nt; ++r)
                    if (bin[r] == idx) { if (ch[r]) s1 += rho[r]; else s0 += rho[r]; }
            } else if (kind == 3) {                             // records in |s| bin idx
                for (int r = 0; r < nt; ++r)
                    if (bin[r] == idx) { if (ch[r]) s1 += 1.0; else s0 += 1.0; }
            } else {                                            // records per channel
                for (int r = 0; r < nt; ++r) { if (ch[r]) s1 += 1.0; else s0 += 1.0; }
            }
            part[o] += s0;
            part[o + st] += s1;
        }
    }
}

}  // namespace ff
