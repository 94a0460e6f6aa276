// Stand-alone stages of the path: backflow evaluation, Slater log|det| with derivatives,
// the Metropolis sampler of the free-fermion base distribution, potentials, Boltzmann
// occupation sampling, the ordered reduction of per-CTA partial sums and an FP64 throughput probe.
#pragma once
#include "ff_common.cuh"
#include "ff_slater.cuh"

namespace ff {

// ---------------------------------------------------------------------------------------
// Backflow.forward / Backflow.divergence (equivariant_funs.py:80-102) at given x.
// One CTA handles W walkers, one thread per (walker, pair | particle) item.
// ---------------------------------------------------------------------------------------
struct BackflowArgs {
    int n, H_eta, H_mu;
    const double *eta_w1, *eta_b1, *eta_w2, *mu_w1, *mu_b1, *mu_w2;
    long long B;
    const double* x;
    double* v;      // nullable
    double* div;    // nullable
    int W, P, NP;
};

__global__ void __launch_bounds__(512) backflow_kernel(const BackflowArgs a) {
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, T = blockDim.x;
    const int n = a.n, D = 2 * n, P = a.P, NP = a.NP, W = a.W;
    const bool has_mu = a.H_mu > 0;
    double* tab = smem;
    double* coef_eta = tab + kTabDoubles;
    double* coef_mu = coef_eta + 6 * ((a.H_eta + 3) & ~3);
    double* wb = coef_mu + 6 * ((a.H_mu + 3) & ~3);
    const int wstride = D + 3 * P;          // x[D], G[P][3] (vx, vy, q)
    fill_exp_table(tab);
    const double* tabl = tab + (tid & 15);
    load_mlp_coef(coef_eta, a.eta_w1, a.eta_b1, a.eta_w2, a.H_eta);
    if (has_mu) load_mlp_coef(coef_mu, a.mu_w1, a.mu_b1, a.mu_w2, a.H_mu);
    const int it_w = tid / P, it_p = tid - it_w * P;
    for (long long base = (long long)blockIdx.x * W; base < a.B; base += (long long)gridDim.x * W) {
        __syncthreads();
        for (int g = tid; g < W * D; g += T) {
            int w = g / D, e = g - w * D;
            long long b = base + w;
            (wb + (size_t)w * wstride)[e] = (b < a.B) ? a.x[b * D + e] : (double)(e >> 1) + 0.37 * (e & 1);
        }
        __syncthreads();
        if (it_w < W) {
            const double* x = wb + (size_t)it_w * wstride;
            double* G = wb + (size_t)it_w * wstride + D + 3 * it_p;
            double rx, ry;
            const bool pair = it_p < NP;
            if (pair) {
                int i = 0, rem = it_p;
                while (rem >= n - 1 - i) { rem -= n - 1 - i; ++i; }
                const int j = i + 1 + rem;
                rx = x[2 * i] - x[2 * j]; ry = x[2 * i + 1] - x[2 * j + 1];
            } else { const int i = it_p - NP; rx = x[2 * i]; ry = x[2 * i + 1]; }
            const double d = sqrt(fma(rx, rx, ry * ry));
            double f[4];
            radial_mlp<1>(pair ? coef_eta : coef_mu, pair ? a.H_eta : a.H_mu, d, tabl, f);
            G[0] = f[0] * rx; G[1] = f[0] * ry;
            G[2] = (pair ? 2.0 : 1.0) * fma(f[1], d, 2.0 * f[0]);
        }
        __syncthreads();
        for (int g = tid; g < W * D; g += T) {
            int w = g / D, e = g - w * D, i = e >> 1, c = e & 1;
            long long b = base + w;
            const double* G = wb + (size_t)w * wstride + D;
            double acc = 0.0;
            for (int j = 0; j < i; ++j) acc -= G[3 * pair_index(j, i, n) + c];
            for (int j = i + 1; j < n; ++j) acc += G[3 * pair_index(i, j, n) + c];
            if (has_mu) acc += G[3 * (NP + i) + c];
            if (b < a.B && a.v) a.v[b * D + e] = acc;
        }
        for (int w = tid; w < W; w += T) {
            long long b = base + w;
            const double* G = wb + (size_t)w * wstride + D;
            double acc = 0.0;
            for (int p = 0; p < P; ++p) acc += G[3 * p + 2];
            if (b < a.B && a.div) a.div[b] = acc;
        }
    }
}

// ---------------------------------------------------------------------------------------
// log|det|, gradient and Laplacian of one or two spin blocks (slater.py, base_dist.py:48).
// scale = 1 for LogAbsSlaterDet, 2 for FreeFermion.log_prob.
// ---------------------------------------------------------------------------------------
struct SlaterArgs {
    int n, n_up;
    long long B;
    const double* x;
    const int* orb;
    const int* walker_state;
    double scale;
    double *logabs, *grad, *lap;
    int W, wstride;       // doubles per walker: D + scratch + n*n
    double* sign;         // [B] sign(det Phi_up det Phi_dn), written by the SIGN instantiations only (+1 for an empty block)
};

template <bool SIGN>
__device__ __forceinline__ void slater_cta_body(const SlaterArgs& a) {
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, T = blockDim.x;
    const int n = a.n, D = 2 * n, W = a.W;
    const int slsz = slater_scratch_size(a.n_up, n - a.n_up);
    auto xw = [&](int w) { return smem + (size_t)w * a.wstride; };
    auto scr = [&](int w) { return xw(w) + D; };
    auto red = [&](int w) { return xw(w) + D + slsz; };
    const bool deriv = a.grad != nullptr || a.lap != nullptr;
    for (long long base = (long long)blockIdx.x * W; base < a.B; base += (long long)gridDim.x * W) {
        __syncthreads();
        for (int g = tid; g < W * D; g += T) {
            int w = g / D, e = g - w * D;
            long long b = base + w;
            xw(w)[e] = (b < a.B) ? a.x[b * D + e] : (double)(e >> 1) + 0.37 * (e & 1);
        }
        __syncthreads();
        auto orbp = [&](int w) { long long b = base + w; int row = (a.walker_state && b < a.B) ? a.walker_state[b] : 0;
                                 return a.orb + (size_t)row * n; };
        if (deriv) slater_team<true, SIGN>(W, n, a.n_up, [&](int w) { return (const double*)xw(w); }, scr, orbp);
        else slater_team<false, SIGN>(W, n, a.n_up, [&](int w) { return (const double*)xw(w); }, scr, orbp);
        if (deriv) {
            for (int g = tid; g < W * n * n; g += T) {
                int w = g / (n * n), rem = g - w * n * n;
                int I = rem / n, J = rem - I * n;
                const int sI = I >= a.n_up, sJ = J >= a.n_up;
                double t = 0.0;
                if (sI == sJ) {
                    const SlBlk blk = slater_blk(sI, n, a.n_up);
                    const int ns = blk.ns, i = I - blk.i0, j = J - blk.i0;
                    const double* S = scr(w);
                    if (i == j) {      // Laplacian = trace of H: C^{xx}_i + C^{yy}_i - (B^x_ii)^2 - (B^y_ii)^2
                        const double gx = S[blk.bx() + i * ns + i], gy = S[blk.by() + i * ns + i];
                        t = S[blk.cc() + 3 * i] + S[blk.cc() + 3 * i + 2] - gx * gx - gy * gy;
                        long long b = base + w;
                        if (b < a.B && a.grad) {
                            a.grad[b * D + 2 * I] = a.scale * S[blk.bx() + i * ns + i];
                            a.grad[b * D + 2 * I + 1] = a.scale * S[blk.by() + i * ns + i];
                        }
                    }
                }
                red(w)[rem] = t;
            }
            __syncthreads();
        }
        for (int w = tid; w < W; w += T) {
            long long b = base + w;
            if (b >= a.B) continue;
            const double* S = scr(w);
            const SlBlk bu = slater_blk(0, n, a.n_up), bd = slater_blk(1, n, a.n_up);
            double ld = 0.0;
            if (bu.ns) ld += S[bu.misc() + 2];
            if (bd.ns) ld += S[bd.misc() + 2];
            if (a.logabs) a.logabs[b] = a.scale * ld;
            if (a.lap) {
                double acc = 0.0;
                for (int k = 0; k < n * n; ++k) acc += red(w)[k];
                a.lap[b] = a.scale * acc;
            }
            if (SIGN && a.sign) a.sign[b] = (bu.ns ? S[bu.misc() + 3] : 1.0) * (bd.ns ? S[bd.misc() + 3] : 1.0);
        }
    }
}

__global__ void __launch_bounds__(256) slater_kernel(const SlaterArgs a) { slater_cta_body<false>(a); }
// the same, also writing SlaterArgs::sign (ff_wavefunction_ratio)
__global__ void __launch_bounds__(256) slater_sign_kernel(const SlaterArgs a) { slater_cta_body<true>(a); }

// ---------------------------------------------------------------------------------------
// The same with ONE WARP PER WALKER (spin blocks of at most 16 particles): no CTA barrier.
//   1. lanes = (particle, coordinate): all eight 1D oscillator functions psi_a, psi_a', psi_a''
//      by the three-term recursion with tabulated square roots                    (orbitals.py:66-90)
//   2. Phi_ik = psi_nx(k)(x_i) psi_ny(k)(y_i) / sqrt(pi) into [Phi | I]; lanes = columns of the
//      augmented matrix run Gauss-Jordan with partial pivoting (warp arg-max by shuffles)
//   3. lanes = particles: B^x_ii, B^y_ii, C^xx_i, C^yy_i = sum_k d Phi_ik Phi^-1_ki from the 1D
//      table; gradient 2 B (Jacobi's formula), Laplacian sum_i C^xx + C^yy - B^x^2 - B^y^2.
// Replaces slater.py:4-68 / 70-156 forward + backward and the 2N autograd passes of
// utils.py:44-65 for f = FreeFermion.log_prob.
// ---------------------------------------------------------------------------------------
constexpr int kSlaterWarpMax = 16;          // particles per spin block
__host__ __device__ inline int slater_warp_slice(int nmax) {      // doubles of shared memory per warp
    return ff_even(nmax * (2 * nmax + 1) + nmax * kHermStride + 2);
}

template <bool SIGN>
__device__ __forceinline__ void slater_warp_body(const SlaterArgs& a) {
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const int n = a.n, D = 2 * n;
    const int nmax = max(a.n_up, n - a.n_up);
    double* A = smem + (size_t)warp * slater_warp_slice(nmax);        // [ns][2 ns + 1]
    double* Ht = A + nmax * (2 * nmax + 1);                            // [ns][kHermStride]: (coord, order, deriv)
    const double inv_sqrt_pi = 0.56418958354775628695;
    const bool deriv = a.grad != nullptr || a.lap != nullptr;
    const long long wstride = (long long)gridDim.x * nwarp;
    for (long long b = (long long)blockIdx.x * nwarp + warp; b < a.B; b += wstride) {
        const int* orb = a.orb + (size_t)(a.walker_state ? a.walker_state[b] : 0) * n;
        double logdet = 0.0, lap = 0.0, sgn = 1.0;
        for (int s = 0; s < 2; ++s) {
            const int ns = s ? n - a.n_up : a.n_up, i0 = s ? a.n_up : 0;
            if (ns == 0) continue;
            const int LD = 2 * ns + 1;
            // ---- 1. 1D oscillator functions --------------------------------------------------
            for (int e = lane; e < 2 * ns; e += 32) {
                const int i = e >> 1, c = e & 1;
                const double x = a.x[b * D + 2 * (i0 + i) + c];
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
            // ---- 2. [Phi | I], Gauss-Jordan ----------------------------------------------------
            for (int e = lane; e < ns * ns; e += 32) {
                const int i = e / ns, k = e - i * ns;
                const int id = orb[i0 + k];
                const double* t = Ht + i * kHermStride;
                A[i * LD + k] = inv_sqrt_pi * t[3 * c_orb_nx[id]] * t[24 + 3 * c_orb_ny[id]];
                A[i * LD + ns + k] = (i == k) ? 1.0 : 0.0;
            }
            __syncwarp();
            for (int k = 0; k < ns; ++k) {
                // pivot: arg-max of |A[r][k]|, r >= k (lane = row)
                double best = (lane >= k && lane < ns) ? fabs(A[lane * LD + k]) : -1.0;
                int p = lane;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                    const int op = __shfl_xor_sync(0xffffffffu, p, o);
                    if (ob > best || (ob == best && op < p)) { best = ob; p = op; }
                }
                logdet += log(best);
                if (SIGN && ((A[p * LD + k] < 0.0) != (p != k))) sgn = -sgn;     // pivot sign, row swap
                const double ipv = 1.0 / A[p * LD + k];
                __syncwarp();
                if (lane < 2 * ns) {                       // lane = column: swap rows k <-> p, scale row k
                    const double vk = A[k * LD + lane], vp = A[p * LD + lane];
                    A[p * LD + lane] = vk;
                    A[k * LD + lane] = vp * ipv;
                }
                __syncwarp();
                if (lane < 2 * ns && lane != k) {          // eliminate column k from every other row
                    const double akc = A[k * LD + lane];
                    for (int r = 0; r < ns; ++r)
                        if (r != k) A[r * LD + lane] = fma(-A[r * LD + k], akc, A[r * LD + lane]);
                }
                __syncwarp();
            }
            // ---- 3. gradient and Laplacian (lane = particle) -----------------------------------
            if (deriv) {
                for (int i = lane; i - lane < ns; i += 32) {
                    double li = 0.0;
                    if (i < ns) {
                        const double* t = Ht + i * kHermStride;
                        double gx = 0.0, gy = 0.0, cxx = 0.0, cyy = 0.0;
                        for (int k = 0; k < ns; ++k) {
                            const int id = orb[i0 + k];
                            const double* tx = t + 3 * c_orb_nx[id];
                            const double* ty = t + 24 + 3 * c_orb_ny[id];
                            const double iv = inv_sqrt_pi * A[k * LD + ns + i];
                            gx = fma(tx[1] * ty[0], iv, gx);
                            gy = fma(tx[0] * ty[1], iv, gy);
                            cxx = fma(tx[2] * ty[0], iv, cxx);
                            cyy = fma(tx[0] * ty[2], iv, cyy);
                        }
                        li = cxx + cyy - gx * gx - gy * gy;
                        if (a.grad) *reinterpret_cast<double2*>(a.grad + b * D + 2 * (i0 + i)) = make_double2(a.scale * gx, a.scale * gy);
                    }
                    lap += li;
                }
            }
            __syncwarp();
        }
        if (a.lap) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) lap += __shfl_xor_sync(0xffffffffu, lap, o);
        }
        if (lane == 0) {
            if (a.logabs) a.logabs[b] = a.scale * logdet;
            if (a.lap) a.lap[b] = a.scale * lap;
            if (SIGN && a.sign) a.sign[b] = sgn;
        }
    }
}

__global__ void __launch_bounds__(256) slater_warp_kernel(const SlaterArgs a) { slater_warp_body<false>(a); }
// the same, also writing SlaterArgs::sign (ff_wavefunction_ratio)
__global__ void __launch_bounds__(256) slater_warp_sign_kernel(const SlaterArgs a) { slater_warp_body<true>(a); }

// ---------------------------------------------------------------------------------------
// Hessian-vector product of scale * (log|det Phi_up| + log|det Phi_dn|): the double backward of
// LogAbsSlaterDet / LogAbsSlaterDetMultStates (slater.py:40-60, 120-156 build their backward with
// differentiable torch ops so that utils.py:44-65 can differentiate it again).  One warp per walker, any spin
// block up to kMaxOrb particles (lane-strided loops):
//   H_{ia,jb} = delta_ij C^{ab}_i - B^a_ij B^b_ji,   B^a = (d_a Phi) Phi^-1,   C^{ab}_i = sum_k d_a d_b phi_k(r_i) Phi^-1_ki
//   (H v)_{ia} = sum_b C^{ab}_i v_ib - sum_j B^a_ij U_ji,      U_ji = sum_b B^b_ji v_jb.
// ---------------------------------------------------------------------------------------
struct SlaterHvpArgs {
    int n, n_up;
    long long B;
    const double* x;
    const int* orb;
    const int* walker_state;
    double scale;
    const double* v;      // [B][n][2]
    double* hv;           // [B][n][2]
};
__host__ __device__ inline int slater_hvp_slice(int nmax) {      // doubles of shared memory per warp
    return ff_even(nmax * (2 * nmax + 1) + nmax * kHermStride + 3 * nmax * (nmax + 1) + 2);
}

__global__ void __launch_bounds__(128) slater_hvp_warp_kernel(const SlaterHvpArgs a) {
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const int n = a.n, D = 2 * n;
    const int nmax = max(a.n_up, n - a.n_up);
    double* A = smem + (size_t)warp * slater_hvp_slice(nmax);          // [ns][2 ns + 1]
    double* Ht = A + nmax * (2 * nmax + 1);                             // [ns][kHermStride]
    double* Bx = Ht + nmax * kHermStride;                               // [ns][ns + 1]
    double* By = Bx + nmax * (nmax + 1);
    double* U = By + nmax * (nmax + 1);
    const double inv_sqrt_pi = 0.56418958354775628695;
    const long long wstride = (long long)gridDim.x * nwarp;
    for (long long b = (long long)blockIdx.x * nwarp + warp; b < a.B; b += wstride) {
        const int* orb = a.orb + (size_t)(a.walker_state ? a.walker_state[b] : 0) * n;
        for (int s = 0; s < 2; ++s) {
            const int ns = s ? n - a.n_up : a.n_up, i0 = s ? a.n_up : 0;
            if (ns == 0) continue;
            const int LD = 2 * ns + 1, LB = ns + 1;
            for (int e = lane; e < 2 * ns; e += 32) {                   // 1D oscillator functions (orbitals.py:66-90)
                const int i = e >> 1, c = e & 1;
                const double x = a.x[b * D + 2 * (i0 + i) + c];
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
                Bx[i * LB + j] = bx;
                By[i * LB + j] = by;
            }
            __syncwarp();
            const double* vv = a.v + b * D + 2 * i0;
            for (int e = lane; e < ns * ns; e += 32) {                  // U_ji = v_jx B^x_ji + v_jy B^y_ji
                const int j = e / ns, i = e - j * ns;
                U[j * LB + i] = fma(vv[2 * j], Bx[j * LB + i], vv[2 * j + 1] * By[j * LB + i]);
            }
            __syncwarp();
            for (int i = lane; i < ns; i += 32) {
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
                double hx = fma(cxx, vv[2 * i], cxy * vv[2 * i + 1]);
                double hy = fma(cxy, vv[2 * i], cyy * vv[2 * i + 1]);
                for (int j = 0; j < ns; ++j) {
                    const double u = U[j * LB + i];
                    hx = fma(-Bx[i * LB + j], u, hx);
                    hy = fma(-By[i * LB + j], u, hy);
                }
                *reinterpret_cast<double2*>(a.hv + b * D + 2 * (i0 + i)) = make_double2(a.scale * hx, a.scale * hy);
            }
            __syncwarp();
        }
    }
}

// ---------------------------------------------------------------------------------------
// Metropolis sampling of |Psi_0|^2 (base_dist.py:58-70, 103-134), one thread per walker.
// Per-thread matrices live in shared memory, element e of thread t at sm[e * T + t].
// ---------------------------------------------------------------------------------------
struct MetroArgs {
    long long B;
    int n, n_up;
    const int* orb;
    const int* walker_state;
    int steps;
    double tau;
    unsigned long long seed;
    long long walker_offset;
    const double *x0, *normals, *uniforms;     // parity mode when non-null
    double* x;
    int* accept_count;
    double* gscratch;       // global fallback for the matrices when shared memory is too small
    int use_global;
};

// log|det Phi| of one spin block via LU with partial pivoting; X points at the coordinates
// (interleaved with stride T), A is the ns x ns work matrix (interleaved with stride sa).
__device__ __forceinline__ double metro_logdet(const double* X, int xs, int i0, int ns, const int* orb,
                                               double* A, size_t sa) {
    const double inv_sqrt_pi = 0.56418958354775628695;
    for (int r = 0; r < ns; ++r) {
        double hxv[8], hyv[8];
        hermite_values(X[(size_t)(2 * (i0 + r)) * xs], hxv);
        hermite_values(X[(size_t)(2 * (i0 + r) + 1) * xs], hyv);
        for (int c = 0; c < ns; ++c) {
            const int id = orb[i0 + c];
            const int nx = c_orb_nx[id], ny = c_orb_ny[id];
            double vx = 0, vy = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) { if (q == nx) vx = hxv[q]; if (q == ny) vy = hyv[q]; }
            A[(size_t)(r * ns + c) * sa] = inv_sqrt_pi * vx * vy;
        }
    }
    // log|det| = log(prod of pivot mantissas) + (sum of pivot exponents) ln 2: one log per block instead of one per pivot
    double prod = 1.0; int esum = 0;
    for (int k = 0; k < ns; ++k) {
        int p = k; double best = fabs(A[(size_t)(k * ns + k) * sa]);
        for (int r = k + 1; r < ns; ++r) {
            const double v = fabs(A[(size_t)(r * ns + k) * sa]);
            if (v > best) { best = v; p = r; }
        }
        if (p != k) {
            for (int c = k; c < ns; ++c) {
                const double t = A[(size_t)(k * ns + c) * sa];
                A[(size_t)(k * ns + c) * sa] = A[(size_t)(p * ns + c) * sa];
                A[(size_t)(p * ns + c) * sa] = t;
            }
        }
        { int e; prod *= frexp(best, &e); esum += e; }
        const double ipv = 1.0 / A[(size_t)(k * ns + k) * sa];
        for (int r = k + 1; r < ns; ++r) {
            const double l = A[(size_t)(r * ns + k) * sa] * ipv;
            for (int c = k + 1; c < ns; ++c)
                A[(size_t)(r * ns + c) * sa] = fma(-l, A[(size_t)(k * ns + c) * sa], A[(size_t)(r * ns + c) * sa]);
        }
    }
    return log(prod) + esum * 0.69314718055994530942;
}

__global__ void __launch_bounds__(128) metropolis_kernel(const MetroArgs a) {
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, T = blockDim.x;
    const long long b = (long long)blockIdx.x * T + tid;
    const int n = a.n, D = 2 * n, n_up = a.n_up, n_dn = n - n_up;
    const int nsm = max(n_up, n_dn);
    double* X = smem + tid;                        // current, D entries, stride T
    double* Y = smem + (size_t)D * T + tid;        // proposal
    double* A; size_t sa;
    if (a.use_global) { A = a.gscratch + b; sa = (size_t)gridDim.x * T; }
    else { A = smem + (size_t)2 * D * T + tid; sa = T; }
    (void)nsm;
    if (b >= a.B) return;
    const int* orb = a.orb + (size_t)((a.walker_state ? a.walker_state[b] : 0)) * n;
    const unsigned long long wid = (unsigned long long)(b + a.walker_offset);
    const uint2 key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32));
    auto normal_pair = [&](uint32_t step, uint32_t slot, double& g0, double& g1) {
        uint4 r = philox4x32_10(make_uint4((uint32_t)wid, (uint32_t)(wid >> 32), step, slot), key);
        const double u1 = u01_53(r.x, r.y), u2 = u01_53(r.z, r.w);
        const double rad = sqrt(-2.0 * log(u1));
        double sn, cs;
        sincospi(2.0 * u2, &sn, &cs);
        g0 = rad * cs; g1 = rad * sn;
    };
    for (int i = 0; i < n; ++i) {
        double g0, g1;
        if (a.x0) { g0 = a.x0[b * D + 2 * i]; g1 = a.x0[b * D + 2 * i + 1]; }
        else normal_pair(0u, (uint32_t)i, g0, g1);
        X[(size_t)(2 * i) * T] = g0; X[(size_t)(2 * i + 1) * T] = g1;
    }
    double logp = 2.0 * ((n_up ? metro_logdet(X, T, 0, n_up, orb, A, sa) : 0.0) +
                         (n_dn ? metro_logdet(X, T, n_up, n_dn, orb, A, sa) : 0.0));
    int acc = 0;
    for (int s = 0; s < a.steps; ++s) {
        for (int i = 0; i < n; ++i) {
            double g0, g1;
            if (a.normals) {
                const double* e = a.normals + ((size_t)s * a.B + b) * D + 2 * i;
                g0 = e[0]; g1 = e[1];
            } else normal_pair((uint32_t)(s + 1), (uint32_t)i, g0, g1);
            Y[(size_t)(2 * i) * T] = fma(a.tau, g0, X[(size_t)(2 * i) * T]);
            Y[(size_t)(2 * i + 1) * T] = fma(a.tau, g1, X[(size_t)(2 * i + 1) * T]);
        }
        const double nlogp = 2.0 * ((n_up ? metro_logdet(Y, T, 0, n_up, orb, A, sa) : 0.0) +
                                    (n_dn ? metro_logdet(Y, T, n_up, n_dn, orb, A, sa) : 0.0));
        double u;
        if (a.uniforms) u = a.uniforms[(size_t)s * a.B + b];
        else {
            uint4 r = philox4x32_10(make_uint4((uint32_t)wid, (uint32_t)(wid >> 32), (uint32_t)(s + 1), 0xFFFFFFFFu), key);
            u = u01_53(r.x, r.y);
        }
        if (u < exp(nlogp - logp)) {
            for (int e = 0; e < D; ++e) X[(size_t)e * T] = Y[(size_t)e * T];
            logp = nlogp;
            ++acc;
        }
    }
    for (int e = 0; e < D; ++e) a.x[b * D + e] = X[(size_t)e * T];
    if (a.accept_count) a.accept_count[b] = acc;
}

// ---------------------------------------------------------------------------------------
// Metropolis sampling with ONE WARP PER WALKER (spin blocks of at most 16 particles).
// Same chain as metropolis_kernel -- same Philox counters, same proposal, the same LU arithmetic
// element by element, hence bit-identical samples -- but the n Box-Muller pairs of a move are drawn
// by n lanes at once, the 1D oscillator values come from a per-particle table and the two spin
// blocks are factorised side by side: lanes 0-15 own the columns of Phi_up, lanes 16-31 those of
// Phi_down, pivots are found with 16-wide shuffles.
// ---------------------------------------------------------------------------------------
constexpr int kMetroHerm = 17;       // doubles per particle in the value table (2 x 8, odd stride)
__host__ __device__ inline int metro_warp_slice(int n, int nmax) {
    return ff_even(2 * 2 * n + n * kMetroHerm + 2 * nmax * (nmax + 1) + 2);
}

__global__ void __launch_bounds__(256) metropolis_warp_kernel(const MetroArgs a) {
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const int n = a.n, D = 2 * n, n_up = a.n_up, n_dn = n - n_up;
    const int nmax = max(n_up, n_dn), LD = nmax + 1;
    double* X = smem + (size_t)warp * metro_warp_slice(n, nmax);
    double* Y = X + D;
    double* Ht = Y + D;                       // [n][kMetroHerm]
    double* A0 = Ht + n * kMetroHerm;         // two blocks of nmax x LD
    const double inv_sqrt_pi = 0.56418958354775628695;
    const uint2 key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32));
    const int half = lane >> 4, hl = lane & 15;            // spin block / column of this lane
    const int ns = half ? n_dn : n_up, i0 = half ? n_up : 0;
    double* A = A0 + half * nmax * LD;
    const long long wstride = (long long)gridDim.x * nwarp;

    for (long long b = (long long)blockIdx.x * nwarp + warp; b < a.B; b += wstride) {
        const int* orb = a.orb + (size_t)(a.walker_state ? a.walker_state[b] : 0) * n;
        const unsigned long long wid = (unsigned long long)(b + a.walker_offset);
        auto normal_pair = [&](uint32_t step, uint32_t slot, double& g0, double& g1) {
            uint4 r = philox4x32_10(make_uint4((uint32_t)wid, (uint32_t)(wid >> 32), step, slot), key);
            const double u1 = u01_53(r.x, r.y), u2 = u01_53(r.z, r.w);
            const double rad = sqrt(-2.0 * log(u1));
            double sn, cs;
            sincospi(2.0 * u2, &sn, &cs);
            g0 = rad * cs; g1 = rad * sn;
        };
        // log|Psi_0|^2 of the configuration in Z (both spin blocks at once)
        auto logprob = [&](const double* Z) -> double {
            for (int e = lane; e < D; e += 32) {                       // 1D oscillator values
                double v[8];
                hermite_values(Z[e], v);
                double* t = Ht + (e >> 1) * kMetroHerm + (e & 1) * 8;
#pragma unroll
                for (int q = 0; q < 8; ++q) t[q] = v[q];
            }
            __syncwarp();
            if (hl < ns) {                                             // lane = (block, column c): Phi[r][c]
                const int id = orb[i0 + hl];
                const int nx = c_orb_nx[id], ny = c_orb_ny[id];
                for (int r = 0; r < ns; ++r) {
                    const double* t = Ht + (i0 + r) * kMetroHerm;
                    A[r * LD + hl] = inv_sqrt_pi * t[nx] * t[8 + ny];
                }
            }
            __syncwarp();
            double prod = 1.0; int esum = 0;                          // same mantissa / exponent accumulation as metro_logdet
            for (int k = 0; k < nmax; ++k) {
                const bool on = k < ns;                                // this half still has pivots to do
                // pivot: first maximum of |A[r][k]|, r >= k, lane hl = row
                double best = (on && hl >= k && hl < ns) ? fabs(A[hl * LD + k]) : -1.0;
                int p = hl;
#pragma unroll
                for (int o = 8; o > 0; o >>= 1) {
                    const double ob = __shfl_xor_sync(0xffffffffu, best, o, 16);
                    const int op = __shfl_xor_sync(0xffffffffu, p, o, 16);
                    if (ob > best || (ob == best && op < p)) { best = ob; p = op; }
                }
                __syncwarp();
                if (on) {
                    if (p != k && hl >= k && hl < ns) {                // swap rows k <-> p, columns c >= k
                        const double t = A[k * LD + hl];
                        A[k * LD + hl] = A[p * LD + hl];
                        A[p * LD + hl] = t;
                    }
                    { int e; prod *= frexp(best, &e); esum += e; }
                }
                __syncwarp();
                if (on && hl > k && hl < ns) {                         // eliminate below the pivot, columns c > k
                    const double ipv = 1.0 / A[k * LD + k];
                    const double akc = A[k * LD + hl];
                    for (int r = k + 1; r < ns; ++r) {
                        const double l = A[r * LD + k] * ipv;
                        A[r * LD + hl] = fma(-l, akc, A[r * LD + hl]);
                    }
                }
                __syncwarp();
            }
            const double ld = log(prod) + esum * 0.69314718055994530942;
            const double lu = __shfl_sync(0xffffffffu, ld, 0), ldn = __shfl_sync(0xffffffffu, ld, 16);
            return 2.0 * ((n_up ? lu : 0.0) + (n_dn ? ldn : 0.0));
        };

        for (int i = lane; i < n; i += 32) {
            double g0, g1;
            if (a.x0) { g0 = a.x0[b * D + 2 * i]; g1 = a.x0[b * D + 2 * i + 1]; }
            else normal_pair(0u, (uint32_t)i, g0, g1);
            X[2 * i] = g0; X[2 * i + 1] = g1;
        }
        __syncwarp();
        double logp = logprob(X);
        int acc = 0;
        for (int s = 0; s < a.steps; ++s) {
            for (int i = lane; i < n; i += 32) {
                double g0, g1;
                if (a.normals) {
                    const double* e = a.normals + ((size_t)s * a.B + b) * D + 2 * i;
                    g0 = e[0]; g1 = e[1];
                } else normal_pair((uint32_t)(s + 1), (uint32_t)i, g0, g1);
                Y[2 * i] = fma(a.tau, g0, X[2 * i]);
                Y[2 * i + 1] = fma(a.tau, g1, X[2 * i + 1]);
            }
            __syncwarp();
            const double nlogp = logprob(Y);
            double u = 0.0;
            if (lane == 0) {
                if (a.uniforms) u = a.uniforms[(size_t)s * a.B + b];
                else {
                    uint4 r = philox4x32_10(make_uint4((uint32_t)wid, (uint32_t)(wid >> 32), (uint32_t)(s + 1), 0xFFFFFFFFu), key);
                    u = u01_53(r.x, r.y);
                }
            }
            u = __shfl_sync(0xffffffffu, u, 0);
            if (u < exp(nlogp - logp)) {                               // warp-uniform decision
                for (int e = lane; e < D; e += 32) X[e] = Y[e];
                logp = nlogp;
                ++acc;
            }
            __syncwarp();
        }
        for (int e = lane; e < D; e += 32) a.x[b * D + e] = X[e];
        if (a.accept_count && lane == 0) a.accept_count[b] = acc;
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------
// potentials.py: 1/2 sum r^2 and Z sum_{i<j} 1/r_ij, one thread per walker.
// ---------------------------------------------------------------------------------------
__global__ void potential_kernel(const double* x, long long B, int n, double Z, int harmonic, double* V) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double* p = x + b * 2 * n;
    double vh = 0.0, vc = 0.0;
    for (int i = 0; i < n; ++i) {
        const double xi = p[2 * i], yi = p[2 * i + 1];
        vh = fma(xi, xi, fma(yi, yi, vh));
        for (int j = i + 1; j < n; ++j) {
            const double dx = xi - p[2 * j], dy = yi - p[2 * j + 1];
            vc += 1.0 / sqrt(fma(dx, dx, dy * dy));
        }
    }
    V[b] = Z * vc + (harmonic ? 0.5 * vh : 0.0);
}

// ---------------------------------------------------------------------------------------
// Boltzmann / categorical occupation sampling (VMC.py:94-97) by inverse CDF.
// ---------------------------------------------------------------------------------------
__global__ void occupation_cdf_kernel(const double* logits, int S, double* cdf, int* counts) {
    // single thread: S is the number of many-body states (tens to a few thousand); the
    // sequential sum is the definition the oracle mirrors (softmax -> cumsum -> normalise).
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        double mx = logits[0];
        for (int s = 1; s < S; ++s) mx = fmax(mx, logits[s]);
        double tot = 0.0;
        for (int s = 0; s < S; ++s) tot += exp(logits[s] - mx);
        double run = 0.0;
        for (int s = 0; s < S; ++s) { run += exp(logits[s] - mx) / tot; cdf[s] = run; }
        const double last = cdf[S - 1];
        for (int s = 0; s < S; ++s) cdf[s] /= last;
    }
    for (int s = threadIdx.x; s < S; s += blockDim.x) counts[s] = 0;
}
__global__ void occupation_search_kernel(const double* cdf, int S, const double* u, long long B, int* counts) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double ub = u[b];
    int lo = 0, hi = S;              // first index with cdf[idx] >= u  (torch.searchsorted, right=False)
    while (lo < hi) { int mid = (lo + hi) >> 1; if (cdf[mid] < ub) lo = mid + 1; else hi = mid; }
    if (lo > S - 1) lo = S - 1;
    atomicAdd(&counts[lo], 1);
}
// sorted state list: walker b gets the state s with prefix[s] <= b < prefix[s+1]
__global__ void occupation_fill_kernel(const int* counts, int S, long long B, int* state) {
    __shared__ long long start;
    for (int s = blockIdx.x; s < S; s += gridDim.x) {
        if (threadIdx.x == 0) { long long acc = 0; for (int q = 0; q < s; ++q) acc += counts[q]; start = acc; }
        __syncthreads();
        const long long st = start; const int c = counts[s];
        for (int k = threadIdx.x; k < c; k += blockDim.x) if (st + k < B) state[st + k] = s;
        __syncthreads();
    }
}

// sums[q] += sum over p = 0, 1, ... of partial[p][q], in row order: the fixed-order second stage of the estimators'
// partial-sum kernels (ff_momentum_accumulate, ff_swap_accumulate, ff_density_matrix_accumulate), one row per CTA
__global__ void __launch_bounds__(256) reduce_partial_rows_kernel(const double* partial, int parts, long long n_sums, double* sums) {
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n_sums; q += (long long)gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int p = 0; p < parts; ++p) s += partial[(long long)p * n_sums + q];
        sums[q] += s;
    }
}

// Dependent-chain DFMA throughput probe: 8 independent chains per thread.
__global__ void __launch_bounds__(256) fp64_peak_kernel(int iters, double seed, double* sink) {
    double a0 = seed, a1 = seed + 1, a2 = seed + 2, a3 = seed + 3, a4 = seed + 4, a5 = seed + 5, a6 = seed + 6, a7 = seed + 7;
    const double m = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
        }
    }
    double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 123.456) sink[0] = s;
}


// DMMA (mma.sync m8n8k4 f64) throughput probe: 4 independent accumulator tiles per warp.
__global__ void __launch_bounds__(256) dmma_peak_kernel(int iters, double seed, double* sink) {
    double c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const double a = seed + threadIdx.x * 1e-9, b = 1.0000001;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            dmma_m8n8k4(c[0], c[1], a, b); dmma_m8n8k4(c[2], c[3], a, b);
            dmma_m8n8k4(c[4], c[5], a, b); dmma_m8n8k4(c[6], c[7], a, b);
        }
    }
    double s = c[0] + c[1] + c[2] + c[3] + c[4] + c[5] + c[6] + c[7];
    if (s == 123.456) sink[0] = s;
}

}  // namespace ff
