// Slater determinants over HO2D orbitals, cooperatively by all threads of a CTA for W
// walkers at once (CTA-wide flattened loops separated by __syncthreads()).
//
// Replaces slater.py:4-68 LogAbsSlaterDet (forward: log|det|; backward: Jacobi's formula
// d log|det| = tr(Phi^-1 dPhi)) and its MultStates variant (slater.py:70-156): the
// occupation is a per-walker row of orbital ids.  Second derivatives come from
//   H_{ia,jb} = delta_ij C^{ab}_i - B^a_ij B^b_ji,
//   B^a = (d_a Phi) Phi^-1,  C^{ab}_i = sum_k d_a d_b phi_k(r_i) Phi^-1_{ki}.
#pragma once
#include "ff_common.cuh"

namespace ff {

// A team is the set of threads that runs a cooperative routine: the whole CTA (CtaTeam) or a
// subset of its warps synchronising on a named barrier (SubTeam; warp-specialised kernels).
struct CtaTeam {
    __device__ __forceinline__ int tid() const { return threadIdx.x; }
    __device__ __forceinline__ int size() const { return blockDim.x; }
    __device__ __forceinline__ void sync() const { __syncthreads(); }
};
struct SubTeam {
    int t, T, bar;          // index inside the team, team size (multiple of 32), barrier id (1..15)
    __device__ __forceinline__ int tid() const { return t; }
    __device__ __forceinline__ int size() const { return T; }
    __device__ __forceinline__ void sync() const { asm volatile("bar.sync %0, %1;" ::"r"(bar), "r"(T) : "memory"); }
};

// scratch layout of one spin block with ns particles (doubles)
struct SlBlk {
    int ns, i0, base;
    __device__ __forceinline__ int aug() const { return base; }                       // ns x 2ns
    __device__ __forceinline__ int dx() const { return base + 2 * ns * ns; }
    __device__ __forceinline__ int dy() const { return base + 3 * ns * ns; }
    __device__ __forceinline__ int dxx() const { return base + 4 * ns * ns; }
    __device__ __forceinline__ int dxy() const { return base + 5 * ns * ns; }
    __device__ __forceinline__ int dyy() const { return base + 6 * ns * ns; }
    __device__ __forceinline__ int bx() const { return base + 7 * ns * ns; }
    __device__ __forceinline__ int by() const { return base + 8 * ns * ns; }
    __device__ __forceinline__ int cc() const { return base + 9 * ns * ns; }          // ns x 3
    __device__ __forceinline__ int col() const { return base + 9 * ns * ns + 3 * ns; } // ns
    __device__ __forceinline__ int misc() const { return base + 9 * ns * ns + 4 * ns; } // 4
};
__host__ __device__ __forceinline__ int slater_blk_size(int ns) { return 9 * ns * ns + 4 * ns + 4; }
__host__ __device__ __forceinline__ int slater_scratch_size(int n_up, int n_dn) {
    return slater_blk_size(n_up) + slater_blk_size(n_dn);
}
__device__ __forceinline__ SlBlk slater_blk(int s, int n, int n_up) {
    SlBlk b;
    b.ns = s ? n - n_up : n_up;
    b.i0 = s ? n_up : 0;
    b.base = s ? slater_blk_size(n_up) : 0;
    return b;
}

// Builds Phi and its derivatives, inverts Phi (Gauss-Jordan, partial pivoting), forms
// B^x, B^y, C.  On return, for spin block s of walker w (scratch pointer S = sptr(w)):
//   S[blk.misc()+2] = log|det Phi|, S[blk.aug() + i*2ns + ns + j] = Phi^-1[i][j].
// All threads of the CTA must call it.  DERIV = false stops after log|det|.  SIGN = true also leaves
// S[blk.misc()+3] = sign(det Phi) of each non-empty block: the product of the pivot signs, negated once per row
// swap p != k.  Without SIGN the slot is not touched and the generated code is that of the sign-free routine.
template <bool DERIV, bool SIGN = false, class ZPtr, class SPtr, class OrbPtr, class Team = CtaTeam>
__device__ void slater_team(int W, int n, int n_up, ZPtr zptr, SPtr sptr, OrbPtr orbptr, Team team = Team()) {
    const int tid = team.tid(), T = team.size();
    const double inv_sqrt_pi = 0.56418958354775628695;
    // ---- F1: matrices ------------------------------------------------------------------
    for (int s = 0; s < 2; ++s) {
        const SlBlk blk = slater_blk(s, n, n_up);
        const int ns = blk.ns;
        if (ns == 0) continue;
        for (int g = tid; g < W * ns * ns; g += T) {
            int w = g / (ns * ns), rem = g - w * ns * ns;
            int i = rem / ns, k = rem - i * ns;
            const double* z = zptr(w) + 2 * (blk.i0 + i);
            const int id = orbptr(w)[blk.i0 + k];
            const int nx = c_orb_nx[id], ny = c_orb_ny[id];
            const Herm1D hx = hermite_1d(z[0], nx), hy = hermite_1d(z[1], ny);
            const double vx = hx.v, vx1 = hx.d1, vx2 = hx.d2, vy = hy.v, vy1 = hy.d1, vy2 = hy.d2;
            double* S = sptr(w);
            S[blk.aug() + i * 2 * ns + k] = inv_sqrt_pi * vx * vy;
            S[blk.aug() + i * 2 * ns + ns + k] = (i == k) ? 1.0 : 0.0;
            if (DERIV) {
                S[blk.dx() + i * ns + k] = inv_sqrt_pi * vx1 * vy;
                S[blk.dy() + i * ns + k] = inv_sqrt_pi * vx * vy1;
                S[blk.dxx() + i * ns + k] = inv_sqrt_pi * vx2 * vy;
                S[blk.dxy() + i * ns + k] = inv_sqrt_pi * vx1 * vy1;
                S[blk.dyy() + i * ns + k] = inv_sqrt_pi * vx * vy2;
            }
        }
        for (int w = tid; w < W; w += T) {
            sptr(w)[blk.misc() + 2] = 0.0;
            if (SIGN) sptr(w)[blk.misc() + 3] = 1.0;
        }
    }
    team.sync();
    // ---- F2: Gauss-Jordan on [Phi | I] ---------------------------------------------------
    const int nmax = max(n_up, n - n_up);
    for (int k = 0; k < nmax; ++k) {
        for (int g = tid; g < 2 * W; g += T) {          // pivot search, one thread per block
            int s = g / W, w = g - s * W;
            const SlBlk blk = slater_blk(s, n, n_up);
            const int ns = blk.ns;
            if (k >= ns) continue;
            double* S = sptr(w);
            const double* A = S + blk.aug();
            int p = k; double best = fabs(A[k * 2 * ns + k]);
            for (int r = k + 1; r < ns; ++r) {
                double v = fabs(A[r * 2 * ns + k]);
                if (v > best) { best = v; p = r; }
            }
            S[blk.misc() + 0] = (double)p;
            S[blk.misc() + 1] = A[p * 2 * ns + k];
            S[blk.misc() + 2] += log(best);
            if (SIGN) {
                const double sg = (A[p * 2 * ns + k] < 0.0) != (p != k) ? -1.0 : 1.0;
                S[blk.misc() + 3] *= sg;
            }
        }
        team.sync();
        for (int s = 0; s < 2; ++s) {                    // swap rows k <-> p, scale row k
            const SlBlk blk = slater_blk(s, n, n_up);
            const int ns = blk.ns;
            if (k >= ns) continue;
            for (int g = tid; g < W * 2 * ns; g += T) {
                int w = g / (2 * ns), c = g - w * 2 * ns;
                double* S = sptr(w);
                double* A = S + blk.aug();
                const int p = (int)S[blk.misc() + 0];
                const double ipv = 1.0 / S[blk.misc() + 1];
                const double vk = A[k * 2 * ns + c], vp = A[p * 2 * ns + c];
                A[p * 2 * ns + c] = vk;
                A[k * 2 * ns + c] = vp * ipv;
            }
        }
        team.sync();
        for (int s = 0; s < 2; ++s) {                    // save multipliers (column k)
            const SlBlk blk = slater_blk(s, n, n_up);
            const int ns = blk.ns;
            if (k >= ns) continue;
            for (int g = tid; g < W * ns; g += T) {
                int w = g / ns, r = g - w * ns;
                double* S = sptr(w);
                S[blk.col() + r] = (r == k) ? 0.0 : S[blk.aug() + r * 2 * ns + k];
            }
        }
        team.sync();
        for (int s = 0; s < 2; ++s) {                    // eliminate
            const SlBlk blk = slater_blk(s, n, n_up);
            const int ns = blk.ns;
            if (k >= ns) continue;
            for (int g = tid; g < W * ns * 2 * ns; g += T) {
                int w = g / (2 * ns * ns), rem = g - w * 2 * ns * ns;
                int r = rem / (2 * ns), c = rem - r * 2 * ns;
                double* S = sptr(w);
                double* A = S + blk.aug();
                A[r * 2 * ns + c] = fma(-S[blk.col() + r], A[k * 2 * ns + c], A[r * 2 * ns + c]);
            }
        }
        team.sync();
    }
    if (!DERIV) return;
    // ---- F3: B^x, B^y, C ---------------------------------------------------------------
    for (int s = 0; s < 2; ++s) {
        const SlBlk blk = slater_blk(s, n, n_up);
        const int ns = blk.ns;
        if (ns == 0) continue;
        for (int g = tid; g < W * ns * ns; g += T) {
            int w = g / (ns * ns), rem = g - w * ns * ns;
            int i = rem / ns, j = rem - i * ns;
            double* S = sptr(w);
            const double* inv = S + blk.aug() + ns;
            double bx = 0, by = 0;
            for (int k = 0; k < ns; ++k) {
                const double iv = inv[k * 2 * ns + j];
                bx = fma(S[blk.dx() + i * ns + k], iv, bx);
                by = fma(S[blk.dy() + i * ns + k], iv, by);
            }
            S[blk.bx() + i * ns + j] = bx;
            S[blk.by() + i * ns + j] = by;
            if (j < 3) {
                const int o = (j == 0) ? blk.dxx() : (j == 1) ? blk.dxy() : blk.dyy();
                double c = 0;
                for (int k = 0; k < ns; ++k) c = fma(S[o + i * ns + k], inv[k * 2 * ns + i], c);
                S[blk.cc() + 3 * i + j] = c;
            }
        }
        if (ns < 3) {       // C needs three entries per particle even when ns < 3
            for (int g = tid; g < W * ns * 3; g += T) {
                int w = g / (ns * 3), rem = g - w * ns * 3;
                int i = rem / 3, j = rem - 3 * i;
                double* S = sptr(w);
                const double* inv = S + blk.aug() + ns;
                const int o = (j == 0) ? blk.dxx() : (j == 1) ? blk.dxy() : blk.dyy();
                double c = 0;
                for (int k = 0; k < ns; ++k) c = fma(S[o + i * ns + k], inv[k * 2 * ns + i], c);
                S[blk.cc() + 3 * i + j] = c;
            }
        }
    }
    team.sync();
}

}  // namespace ff
