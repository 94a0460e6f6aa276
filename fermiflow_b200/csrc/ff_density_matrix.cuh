// One-body density matrix in the HO2D orbital basis from one-particle-move records (ff_density_matrix_accumulate;
// include/fermiflow_b200.h has the estimator and the layout of the sums).
//
// A record r = b M + m moves particle i = particle[r] of walker b from r_i = x[b][i] to r' = r_i + disp[r] and carries
// a weight w[r] (the estimator passes psi(x with r_i -> r') / psi(x) / q(r')).  Per spin channel c = (i >= n_up):
//   S^c_ab = sum over the records of c of 1/2 [phi_a(r_i) phi_b(r') + phi_b(r_i) phi_a(r')] w,   a, b < K.
// r' is formed with one rounded add per coordinate, as wfr_configs_kernel forms the moved configuration, so for a
// Slater determinant sum_{i in c} phi_a(r_i) ratio_i = phi_a(r') holds to rounding for every occupied a.
// Fixed summation order, no floating-point atomics:
//   density_matrix_partial_kernel  CTA g takes records [g chunk, (g + 1) chunk) in tiles of kDmTile records.  Per tile
//                                  the CTA tabulates in shared memory phi_0 ... phi_{K-1} at r_i and w/2 phi at r'
//                                  (hermite_values and the c_orb_nx / c_orb_ny tables) and the channel; each thread
//                                  owns up to kDmUnits "units" -- a cell a <= b (both channels), the records per
//                                  channel, the skipped records -- and sums every record of its chunk in order in
//                                  registers; at the end it writes both triangles of its cells to the CTA's partial row.
//   reduce_partial_rows_kernel (ff_misc.cuh)  sums[q] += sum over g = 0, 1, ... of partial[g][q], in CTA order.
// A record whose particle index lies outside [0, n) reads neither x nor w; it only counts as skipped.
#pragma once
#include "ff_common.cuh"

namespace ff {

constexpr int kDmThreads = 256;
constexpr int kDmTile = 32;
constexpr int kDmUnits = 3;                                     // units per thread
// shared memory of one tile: phi at r_i and r' (2 K), the 1D tables (32), positions (4) and w/2 per record, channels
__host__ __device__ constexpr long long dm_smem_bytes(int K) { return (long long)kDmTile * ((2LL * K + 37) * 8 + 4); }
static_assert(kMaxOrb * (kMaxOrb + 1) / 2 + 2 <= kDmUnits * kDmThreads, "every unit has a thread");

struct DmArgs {
    const double* x;            // [B][n][2]
    const int* particle;        // [R]
    const double* disp;         // [R][2]
    const double* w;            // [R]
    long long R;
    int n, n_up, M, K;
    long long chunk;            // records per CTA
    long long n_sums;           // 2 K^2 + 3
    double* partial;            // [gridDim.x][n_sums]
};

__global__ void __launch_bounds__(kDmThreads) density_matrix_partial_kernel(const DmArgs a) {
    extern __shared__ __align__(16) double dm_smem[];
    const int tid = threadIdx.x, K = a.K;
    double* u_s = dm_smem;                                      // [kDmTile][K] phi_a(r_i)
    double* v_s = u_s + kDmTile * K;                            // [kDmTile][K] w/2 phi_a(r')
    double* h_s = v_s + kDmTile * K;                            // [kDmTile][4][8] 1D oscillator functions of x_i, y_i, x', y'
    double* pos_s = h_s + kDmTile * 32;                         // [kDmTile][4] x_i, y_i, x', y'
    double* hw_s = pos_s + kDmTile * 4;                         // [kDmTile] w / 2
    int* ch_s = reinterpret_cast<int*>(hw_s + kDmTile);         // [kDmTile] channel, -1: skipped
    const int cells = K * (K + 1) / 2, units = cells + 2;
    // unit -> cell (ua <= ub) of the upper triangle, row by row; units cells and cells + 1 are the counters
    int ua[kDmUnits], ub[kDmUnits];
#pragma unroll
    for (int j = 0; j < kDmUnits; ++j) {
        int u = tid + j * kDmThreads, r = 0;
        if (u < cells) {
            while (u >= K - r) { u -= K - r; ++r; }
            ua[j] = r; ub[j] = r + u;
        } else {
            ua[j] = ub[j] = 0;
        }
    }
    double s0[kDmUnits], s1[kDmUnits];
#pragma unroll
    for (int j = 0; j < kDmUnits; ++j) s0[j] = s1[j] = 0.0;
    const double inv_sqrt_pi = 0.56418958354775628695;
    const long long r0 = (long long)blockIdx.x * a.chunk, r1 = min(a.R, r0 + a.chunk);
    for (long long t0 = r0; t0 < r1; t0 += kDmTile) {
        const int nt = (int)min((long long)kDmTile, r1 - t0);
        __syncthreads();                                        // the previous tile is consumed
        if (tid < nt) {
            const long long g = t0 + tid;
            const int i = a.particle[g];
            const bool ok = i >= 0 && i < a.n;
            ch_s[tid] = ok ? (i >= a.n_up) : -1;
            if (ok) {
                const long long b = g / a.M;
                const double rx = a.x[(b * a.n + i) * 2], ry = a.x[(b * a.n + i) * 2 + 1];
                pos_s[4 * tid] = rx;
                pos_s[4 * tid + 1] = ry;
                pos_s[4 * tid + 2] = __dadd_rn(rx, a.disp[2 * g]);
                pos_s[4 * tid + 3] = __dadd_rn(ry, a.disp[2 * g + 1]);
                hw_s[tid] = 0.5 * a.w[g];
            } else {
                pos_s[4 * tid] = pos_s[4 * tid + 1] = pos_s[4 * tid + 2] = pos_s[4 * tid + 3] = 0.0;
                hw_s[tid] = 0.0;
            }
        }
        __syncthreads();
        for (int e = tid; e < nt * 4; e += kDmThreads) {
            double v[8];
            hermite_values(pos_s[e], v);
#pragma unroll
            for (int q = 0; q < 8; ++q) h_s[8 * e + q] = v[q];
        }
        __syncthreads();
        for (int e = tid; e < nt * K; e += kDmThreads) {
            const int r = e / K, k = e - r * K;
            const int nx = c_orb_nx[k], ny = c_orb_ny[k];
            const double* h = h_s + 32 * r;
            u_s[e] = inv_sqrt_pi * h[nx] * h[8 + ny];
            v_s[e] = hw_s[r] * (inv_sqrt_pi * h[16 + nx] * h[24 + ny]);
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kDmUnits; ++j) {
            const int u = tid + j * kDmThreads;
            if (u < cells) {
                const int ia = ua[j], ib = ub[j];
                for (int r = 0; r < nt; ++r) {
                    const int c = ch_s[r];
                    const double* U = u_s + r * K;
                    const double* V = v_s + r * K;
                    const double t = fma(U[ia], V[ib], U[ib] * V[ia]);
                    if (c == 1) s1[j] += t; else if (c == 0) s0[j] += t;
                }
            } else if (u == cells) {                            // records per channel
                for (int r = 0; r < nt; ++r) { const int c = ch_s[r]; if (c == 1) s1[j] += 1.0; else if (c == 0) s0[j] += 1.0; }
            } else if (u == cells + 1) {                        // skipped records
                for (int r = 0; r < nt; ++r) if (ch_s[r] < 0) s0[j] += 1.0;
            }
        }
    }
    double* part = a.partial + (long long)blockIdx.x * a.n_sums;
    const long long KK = (long long)K * K;
#pragma unroll
    for (int j = 0; j < kDmUnits; ++j) {
        const int u = tid + j * kDmThreads;
        if (u < cells) {
            const int ia = ua[j], ib = ub[j];
            part[ia * K + ib] = s0[j];
            part[ib * K + ia] = s0[j];
            part[KK + ia * K + ib] = s1[j];
            part[KK + ib * K + ia] = s1[j];
        } else if (u == cells) {
            part[2 * KK] = s0[j];
            part[2 * KK + 1] = s1[j];
        } else if (u < units) {
            part[2 * KK + 2] = s0[j];
        }
    }
}

}  // namespace ff
