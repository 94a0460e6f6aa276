// Base-distribution end of the register-resident E_loc sweep (eloc5_kernel), ONE WARP PER WALKER (eloc_finale_warp_kernel).
//
// Input: the final state of the forward-mode sweep in global memory (eloc5_kernel): y = z = flow^-1(x),
// L_b = sum_a d2y_b / dx_a^2, gDelta, Delta, lapDelta and J = dy/dx (row-major).  At z the kernel evaluates
//     log p0 = 2 (log|det Phi_up| + log|det Phi_dn|)                                          (base_dist.py:48-56)
//     g0 = 2 B^a_ii,   H0_{ia,jb} = 2 (delta_ij C^{ab}_i - B^a_ij B^b_ji)                     (Jacobi's formula; slater.py:4-156)
// with B^a = (d_a Phi) Phi^-1, C^{ab}_i = sum_k d_a d_b phi_k(r_i) Phi^-1_ki, and assembles (utils.py:44-65, VMC.py:48-55)
//     log p = log p0 - Delta,   grad = J^T g0 - gDelta,   lap = <H0, J J^T> + g0.L - lapDelta,
//     E_loc = -1/4 lap - 1/8 |grad|^2 + Z sum 1/r_ij + 1/2 sum r^2.
// The Slater part is the warp-synchronous Gauss-Jordan of slater_hvp_warp_kernel (lanes = columns of [Phi | I], pivot by
// shuffles, no CTA barrier).  M = J J^T never touches shared memory: the warp forms the upper block triangle on the tensor
// cores with the operand fragments straight from global memory (every 8 x 4 fragment is eight full 32-byte sectors; the A
// and the B operand of a block are the same kind of fragment) and contracts each accumulator element with H0 in place.
// A CTA-synchronous finale on the same final states (eloc_finale, ff_flow.cuh, which ends the generic sweep) spent 5.7 ms
// per 65536 walkers at N = 20 between its barriers.
#pragma once
#include "ff_flow.cuh"

namespace ff {

__host__ __device__ inline int finale_warp_slice(int n, int nmax) {      // doubles of shared memory per warp
    // [Phi | I] ns x (2 ns + 1) | 1D table ns x 49 | B^x, B^y of BOTH spin blocks n x (nmax + 1) each | C n x 3 | g0 2n
    return ff_even(nmax * (2 * nmax + 1) + nmax * kHermStride + 2 * n * (nmax + 1) + 3 * n + 2 * n + 2);
}

// NB8 = ceil(2 n / 8) row blocks of J
template <int NB8>
__global__ void __launch_bounds__(128) eloc_finale_warp_kernel(const FlowArgs a, const double* __restrict__ fin, int fin_stride) {
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const int g8 = lane >> 2, t4 = lane & 3;
    const int n = a.n, D = 2 * n, n_up = a.n_up;
    const int nmax = max(n_up, n - n_up), LB = nmax + 1;
    double* A = smem + (size_t)warp * finale_warp_slice(n, nmax);       // [ns][2 ns + 1]
    double* Ht = A + nmax * (2 * nmax + 1);                              // [ns][kHermStride]
    double* Bx = Ht + nmax * kHermStride;                                // [n][LB]: row = global particle, column = particle inside its spin block
    double* By = Bx + n * LB;
    double* Cc = By + n * LB;                                            // [n][3]: C^xx, C^xy, C^yy
    double* g0 = Cc + 3 * n;                                             // [2 n]
    const double inv_sqrt_pi = 0.56418958354775628695;
    const int oL = D, oG = 2 * D, oS = 3 * D, oJ = 3 * D + 2;
    constexpr int NTRI = NB8 * (NB8 + 1) / 2;
    const long long wstride = (long long)gridDim.x * nwarp;
    for (long long b = (long long)blockIdx.x * nwarp + warp; b < a.B; b += wstride) {
        const double* F = fin + (size_t)b * fin_stride;
        const int* orb = a.orb + (size_t)(a.walker_state ? a.walker_state[b] : 0) * n;
        // ---- M = J J^T (upper block triangle) on the tensor cores, fragments from global memory ----------------------
        double acc[NTRI][2];
#pragma unroll
        for (int q = 0; q < NTRI; ++q) { acc[q][0] = 0.0; acc[q][1] = 0.0; }
        {
            const double* Jf = F + oJ + t4;
            const int ksteps = (D + 3) >> 2;
            double fc[NB8], fn[NB8];
#pragma unroll
            for (int c = 0; c < NB8; ++c) { const int r = 8 * c + g8; fc[c] = (r < D && t4 < D) ? __ldg(Jf + (size_t)r * D) : 0.0; }
            for (int k = 0; k < ksteps; ++k) {
                if (k + 1 < ksteps) {
#pragma unroll
                    for (int c = 0; c < NB8; ++c) {
                        const int r = 8 * c + g8, col = 4 * (k + 1) + t4;
                        fn[c] = (r < D && col < D) ? __ldg(Jf + (size_t)r * D + 4 * (k + 1)) : 0.0;
                    }
                }
                int q = 0;
#pragma unroll
                for (int rb = 0; rb < NB8; ++rb)
#pragma unroll
                    for (int cb = rb; cb < NB8; ++cb, ++q) dmma_m8n8k4(acc[q][0], acc[q][1], fc[rb], fc[cb]);
#pragma unroll
                for (int c = 0; c < NB8; ++c) fc[c] = fn[c];
            }
        }
        // ---- Slater matrices at z: Phi^-1, log|det|, B^x, B^y, C ----------------------------------------------------------
        double logdet = 0.0;
        for (int s = 0; s < 2; ++s) {
            const int ns = s ? n - n_up : n_up, i0 = s ? n_up : 0;
            if (ns == 0) continue;
            const int LD = 2 * ns + 1;
            for (int e = lane; e < 2 * ns; e += 32) {                   // 1D oscillator functions (orbitals.py:66-90)
                const int i = e >> 1, c = e & 1;
                const double x = F[2 * (i0 + i) + c];
                const double g = exp(-0.5 * x * x);
                double* t = Ht + i * kHermStride + c * 24;
                double hm = 0.0, hh = 1.0;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    t[3 * k] = hh * g;
                    t[3 * k + 1] = (c_herm_d1[k] * hm - x * hh) * g;
                    t[3 * k + 2] = (x * x - (2.0 * k + 1.0)) * hh * g;
                    const double hn = c_herm_up[k] * x * hh - c_herm_dn[k] * hm;
                    hm = hh; hh = hn;
                }
            }
            __syncwarp();
            for (int e = lane; e < ns * ns; e += 32) {                  // [Phi | I]
                const int i = e / ns, k = e - i * ns;
                const int id = orb[i0 + k];
                const double* t = Ht + i * kHermStride;
                A[i * LD + k] = inv_sqrt_pi * t[3 * c_orb_nx[id]] * t[24 + 3 * c_orb_ny[id]];
                A[i * LD + ns + k] = (i == k) ? 1.0 : 0.0;
            }
            __syncwarp();
            for (int k = 0; k < ns; ++k) {                              // Gauss-Jordan, partial pivoting
                double best = -1.0;
                int p = k;
                for (int r = k + lane; r < ns; r += 32) {
                    const double v = fabs(A[r * LD + k]);
                    if (v > best) { best = v; p = r; }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                    const int op = __shfl_xor_sync(0xffffffffu, p, o);
                    if (ob > best || (ob == best && op < p)) { best = ob; p = op; }
                }
                logdet += log(best);
                const double ipv = 1.0 / A[p * LD + k];
                __syncwarp();
                for (int c = lane; c < 2 * ns; c += 32) {               // swap rows k <-> p, scale row k
                    const double vk = A[k * LD + c], vp = A[p * LD + c];
                    A[p * LD + c] = vk;
                    A[k * LD + c] = vp * ipv;
                }
                __syncwarp();
                for (int c = lane; c < 2 * ns; c += 32) {               // eliminate column k from every other row
                    if (c == k) continue;
                    const double akc = A[k * LD + c];
                    for (int r = 0; r < ns; ++r)
                        if (r != k) A[r * LD + c] = fma(-A[r * LD + k], akc, A[r * LD + c]);
                }
                __syncwarp();
            }
            for (int e = lane; e < ns * ns; e += 32) {                  // B^x, B^y
                const int i = e / ns, j = e - i * ns;
                const double* t = Ht + i * kHermStride;
                double bx = 0.0, by = 0.0;
                for (int k = 0; k < ns; ++k) {
                    const int id = orb[i0 + k];
                    const double* tx = t + 3 * c_orb_nx[id];
                    const double* ty = t + 24 + 3 * c_orb_ny[id];
                    const double iv = inv_sqrt_pi * A[k * LD + ns + j];
                    bx = fma(tx[1] * ty[0], iv, bx);
                    by = fma(tx[0] * ty[1], iv, by);
                }
                Bx[(i0 + i) * LB + j] = bx;
                By[(i0 + i) * LB + j] = by;
            }
            for (int i = lane; i < ns; i += 32) {                       // C^xx, C^xy, C^yy
                const double* t = Ht + i * kHermStride;
                double cxx = 0.0, cxy = 0.0, cyy = 0.0;
                for (int k = 0; k < ns; ++k) {
                    const int id = orb[i0 + k];
                    const double* tx = t + 3 * c_orb_nx[id];
                    const double* ty = t + 24 + 3 * c_orb_ny[id];
                    const double iv = inv_sqrt_pi * A[k * LD + ns + i];
                    cxx = fma(tx[2] * ty[0], iv, cxx);
                    cxy = fma(tx[1] * ty[1], iv, cxy);
                    cyy = fma(tx[0] * ty[2], iv, cyy);
                }
                Cc[3 * (i0 + i)] = cxx; Cc[3 * (i0 + i) + 1] = cxy; Cc[3 * (i0 + i) + 2] = cyy;
            }
            __syncwarp();
        }
        for (int i = lane; i < n; i += 32) {                            // g0 = 2 B^a_ii
            const int il = i < n_up ? i : i - n_up;
            g0[2 * i] = 2.0 * Bx[i * LB + il];
            g0[2 * i + 1] = 2.0 * By[i * LB + il];
        }
        __syncwarp();
        // ---- <H0 / 2, M>: every accumulator element against its Hessian entry -------------------------------------------
        double lap0 = 0.0;
        {
            int q = 0;
#pragma unroll
            for (int rb = 0; rb < NB8; ++rb)
#pragma unroll
                for (int cb = rb; cb < NB8; ++cb, ++q) {
                    const int p = 8 * rb + g8, qc = 8 * cb + 2 * t4;        // M[p][qc], M[p][qc + 1]
                    if (p < D && qc < D) {
                        const int i = p >> 1, al = p & 1, j = qc >> 1;
                        if ((i < n_up) == (j < n_up)) {
                            const int il = i < n_up ? i : i - n_up, jl = j < n_up ? j : j - n_up;
                            const double ba = (al ? By : Bx)[i * LB + jl];                    // B^al_ij
                            double h0 = -ba * Bx[j * LB + il], h1 = -ba * By[j * LB + il];    // - B^al_ij B^be_ji, be = x, y
                            if (i == j) { h0 += Cc[3 * i + al]; h1 += Cc[3 * i + al + 1]; }    // C^{al x}, C^{al y}
                            const double w = rb == cb ? 1.0 : 2.0;                            // the lower triangle of blocks by symmetry
                            lap0 = fma(w * h0, acc[q][0], lap0);
                            lap0 = fma(w * h1, acc[q][1], lap0);
                        }
                    }
                }
        }
        // ---- grad = J^T g0 - gDelta, |grad|^2, g0.L, potentials at the original coordinates --------------------------------
        double g2 = 0.0, gl = 0.0, vh = 0.0, vc = 0.0;
        for (int c = lane; c < D; c += 32) {
            double s0 = 0.0, s1 = 0.0;
            const double* Jc = F + oJ + c;
            int r = 0;
            for (; r + 2 <= D; r += 2) {
                s0 = fma(g0[r], __ldg(Jc + (size_t)r * D), s0);
                s1 = fma(g0[r + 1], __ldg(Jc + (size_t)(r + 1) * D), s1);
            }
            if (r < D) s0 = fma(g0[r], __ldg(Jc + (size_t)r * D), s0);
            const double gc = (s0 + s1) - F[oG + c];
            if (a.grad) a.grad[b * D + c] = gc;
            g2 = fma(gc, gc, g2);
            gl = fma(g0[c], F[oL + c], gl);
            const double xc = a.x_in[b * D + c];
            vh = fma(xc, xc, vh);
        }
        {
            const double* x0 = a.x_in + b * D;
            int i = 0, j = 0;                                           // pair index p -> (i, j), advanced incrementally
            const int NP = n * (n - 1) / 2;
            for (int p = 0, pl = lane; pl < NP; pl += 32) {
                while (p + (n - 1 - i) <= pl) { p += n - 1 - i; ++i; }
                j = i + 1 + (pl - p);
                const double dx = x0[2 * i] - x0[2 * j], dy = x0[2 * i + 1] - x0[2 * j + 1];
                vc += a.Z * rsqrt(fma(dx, dx, dy * dy));
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lap0 += __shfl_xor_sync(0xffffffffu, lap0, o);
            g2 += __shfl_xor_sync(0xffffffffu, g2, o);
            gl += __shfl_xor_sync(0xffffffffu, gl, o);
            vh += __shfl_xor_sync(0xffffffffu, vh, o);
            vc += __shfl_xor_sync(0xffffffffu, vc, o);
        }
        if (lane == 0) {
            const double lp = 2.0 * logdet - F[oS];
            const double lap = 2.0 * lap0 + gl - F[oS + 1];
            const double kin = -0.25 * lap - 0.125 * g2;
            const double pot = vc + (a.harmonic ? 0.5 * vh : 0.0);
            if (a.logp) a.logp[b] = lp;
            if (a.lap) a.lap[b] = lap;
            if (a.kin) a.kin[b] = kin;
            if (a.pot) a.pot[b] = pot;
            if (a.eloc) a.eloc[b] = kin + pot;
        }
        __syncwarp();
    }
}

}  // namespace ff
