// E_loc sweep, register-resident Jacobian with specialised warps (eloc5_kernel).
//
// Same mathematics as flow_body<MODE_ELOC> (ff_flow.cuh; replaces utils.py:44-65 y_grad_laplacian + VMC.py:41-55 on
// top of flow.py:42-56 / equivariant_funs.py:17-102): the forward-mode state (y, J, L, gDelta, Delta, lapDelta) of ONE
// walker per CTA is integrated with the 3/8-rule RK4 (torchdiffeq rk4_alt_step_func).  The kernel writes the final
// state to global memory (fin_stride doubles per walker); the base-distribution end of the sweep (Slater matrices,
// <H0, J J^T>, E_loc) runs from there in a separate kernel at full occupancy (ff_finale.cuh).
//
//   * The Jacobian is carried TRANSPOSED, K = J^T, and its derivative is K' = K A (A = dv/dy is symmetric).
//     Owner warp cb < NB owns the 8 rows [8 cb, 8 cb + 8) of K in the accumulator layout of mma.m8n8k4 (lane (g, t) holds
//     K[8 cb + g][8 rb + 2 t + e], rb < NB, e < 2).  The contraction index of a matrix product may be permuted freely,
//     so those registers ARE the A operand of the next product: k-step (rb, e) pairs K[.][8 rb + 2 t + e] with row
//     8 rb + 2 t + e of A.  K never leaves the registers of its owner except as the shared copy the Gram matrix is
//     formed from; its RK partials are in shared memory (see "RK in the accumulators" below).
//   * A is stored with the rows of every block of 8 in the order 0 2 4 6 1 3 5 7 (a_row), which makes the owners'
//     B-operand loads (rows 2 t + e of a block) bank-conflict free at the row pitch D8 + 4.
//   * The CTA has NB owner warps and WW = ceil(P / 32) "worker" warps (N = 20: 5 + 7 = 384 threads at 80 registers,
//     two CTAs = 24 warps per SM).  Owners never evaluate items, workers never hold K: neither side
//     carries the other's registers.
//   * Per RK stage both kinds of warps have work in both phases, and they hand data over point to point (named barriers,
//     see below) instead of meeting at CTA-wide barriers:
//       phase 1   workers: finish the items of the stage from (r and the radial functions) kept in registers -- matrices R_c of the
//                 per-particle sums, off-diagonal blocks of A = dv/dy (stored with the step factor of the sub-stage), stash.
//                 owners: M = K^T K on the tensor cores from the shared copy of K.
//       phase 2   owners: row sums (k_y: y advances; u, rho, diagonal of A), K A on the tensor cores with the RK combination
//                 of the earlier sub-stages as the initial value of the accumulators, K u, shared copy of the new K.
//                 workers: contractions of their items with M plus the items' share of A L, per-particle sums of those (L
//                 advances), Delta / lapDelta as per-particle shares -- and then the radial functions (certified Taylor
//                 tables) of the NEXT stage at the y the owners have just advanced: the long-latency table look-up
//                 overlaps the owners' tensor-core work.
//   * Nothing lags: M of stage s is formed in phase 1 of stage s and consumed in its phase 2.
#pragma once
#include "ff_finale.cuh"

namespace ff {

// One RK sub-stage of the two-partial 3/8 rule for a scalar element.
__device__ __forceinline__ double rk_elem(int sub, double s, double hk, double& B, double& C) {
    if (sub == 0) { B = fma(hk, -1.0 / 3.0, s); C = fma(hk, 0.125, s); return fma(hk, 1.0 / 3.0, s); }
    if (sub == 1) { const double b = B; B = (2.0 * s - b) - hk; C = fma(hk, 0.375, C); return b + hk; }
    if (sub == 2) { C = fma(hk, 0.375, C); return B + hk; }
    return fma(hk, 0.125, C);
}

// Ordered shared-memory load / tensor-core product (volatile asm keeps the program order): ptxas otherwise sinks
// every operand load right in front of its DMMA and each product waits ~30 cycles for its own LDS.
__device__ __forceinline__ double lds_ordered(const double* p) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"((unsigned)__cvta_generic_to_shared(p)));
    return v;
}
__device__ __forceinline__ void dmma_ordered(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// physical row of A that holds logical row r: rows of each block of 8 in the order 0 2 4 6 1 3 5 7
__host__ __device__ constexpr int a_row(int r) { return (r & ~7) | ((r & 1) << 2) | ((r & 7) >> 1); }

__device__ __forceinline__ void named_bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

// Direct evaluation of f(d) = sum_h w2_h sigmoid(w1_h d + b1_h) and three derivatives from the parameters in global
// memory (MLP.py:30-45): only for items the certified table does not cover (d beyond its range, invalid table).
__device__ __noinline__ void radial_direct_global(const double* __restrict__ w1, const double* __restrict__ b1,
                                                  const double* __restrict__ w2, int H, double d, double* f) {
    double f0 = 0.0, f1 = 0.0, f2 = 0.0, f3 = 0.0;
    for (int h = 0; h < H; ++h) {
        const double w = __ldg(w1 + h), c = __ldg(w2 + h);
        const double s0 = 1.0 / (1.0 + exp(-fma(w, d, __ldg(b1 + h))));
        const double s1 = fma(-s0, s0, s0);
        const double s2 = s1 * fma(-2.0, s0, 1.0);
        const double s3 = s1 * fma(-6.0, s1, 1.0);
        double cw = c;
        f0 = fma(cw, s0, f0); cw *= w;
        f1 = fma(cw, s1, f1); cw *= w;
        f2 = fma(cw, s2, f2); cw *= w;
        f3 = fma(cw, s3, f3);
    }
    f[0] = f0; f[1] = f1; f[2] = f2; f[3] = f3;
}

// Per-particle sum of component c < 3 of the three-component records G2[p][3] of the M-contractions.  Partner slot
// k < i is pair (k, i) at record K_k + i (K_k a compile-time constant), slot k >= i is pair (i, k + 1) at record
// U_i + k + 1.  Components 0, 1 change sign with the orientation of the pair, component 2 holds the pair total (halved
// here); the one-body item of the particle is added last.
template <int SN, int SMU>
__device__ __forceinline__ double gather3(const double* __restrict__ G2, int i, int c) {
    constexpr int n = SN, NP = SN * (SN - 1) / 2;
    const double* pL = G2 + 3 * i + c;                                             // + 3 * (K_k - k - 1)
    const double* pU = G2 + 3 * (i * (2 * n - i - 1) / 2 - i - 1) + c;             // + 3 * (k + 1)
    double lo0 = 0.0, lo1 = 0.0, up0 = 0.0, up1 = 0.0;
#pragma unroll
    for (int k = 0; k < n - 1; ++k) {
        if (k < i) { const double v = pL[3 * (k * (2 * n - k - 1) / 2 - k - 1)]; if (k & 1) lo1 += v; else lo0 += v; }
        else { const double v = pU[3 * (k + 1)]; if (k & 1) up1 += v; else up0 += v; }
    }
    const double lo = lo0 + lo1, up = up0 + up1;
    double acc = c < 2 ? up - lo : 0.5 * (up + lo);
    if (SMU != 0) acc += G2[3 * (NP + i) + c];
    return acc;
}

// Opaque copy of a lane-dependent index, taken once per RK stage: everything derived from it (dozens of shared-memory
// addresses of the gathers, the contractions and the tensor-core fragments) is then recomputed inside the stage with
// a handful of integer instructions instead of being hoisted out of the stage loop, where those loop invariants filled
// the register file and spilled to local memory (first version: 120 M local loads per 9472 walkers).
__device__ __forceinline__ int stage_local(int v) { asm volatile("" : "+r"(v)); return v; }

struct Eloc5Geom {
    int n, D, D8, DP, NP, P, NB, ntri, MAT, RP, RMAT;
    int threads, OW, WW, G0, GWN;
    int oKs, oA, oM, oR1, oG2, oKB, oKC, oY, oYB, oYC, oL0, oL1, oLB, oLC, oU, oKLx, oP1, oP2, oScal, total;   // the mirror of the eta table starts at `total`
    int fin_stride;
};
__host__ __device__ constexpr Eloc5Geom eloc5_geom(int n, bool has_mu) {
    Eloc5Geom g{};
    g.n = n; g.D = 2 * n; g.D8 = (g.D + 7) & ~7; g.DP = g.D8 + 4;
    g.NP = n * (n - 1) / 2; g.P = g.NP + (has_mu ? n : 0);
    g.NB = g.D8 / 8; g.ntri = g.NB * (g.NB + 1) / 2; g.MAT = g.D8 * g.DP;
    g.OW = g.NB; g.WW = (g.P + 31) / 32; g.threads = 32 * (g.OW + g.WW);
    // owner warps that form the Gram matrix in phase 1 (all of them)
    g.G0 = 0; g.GWN = g.NB < g.ntri ? g.NB : g.ntri;
    g.RP = n | 1; g.RMAT = n * g.RP;
    int off = 0;
    g.oKs = off; off += g.MAT;
    g.oA = off; off += g.MAT;
    g.oM = off; off += g.MAT;
    g.oR1 = off; off = ff_even(off + 5 * g.RMAT);
    g.oG2 = off; off = ff_even(off + 3 * g.P);
    g.oKB = off; off += 2 * g.NB * 32 * g.OW; g.oKC = off; off += 2 * g.NB * 32 * g.OW;
    g.oY = off; off += g.D8; g.oYB = off; off += g.D8; g.oYC = off; off += g.D8;
    g.oL0 = off; off += g.D8; g.oL1 = off; off += g.D8; g.oLB = off; off += g.D8; g.oLC = off; off += g.D8;
    g.oU = off; off += g.D8; g.oKLx = off; off += g.D8;
    g.oP1 = off; off += ff_even(n); g.oP2 = off; off += ff_even(n);
    g.oScal = off; off += 8;           // Delta, B, C, lapDelta, B, C
    g.total = ff_even(off);
    g.fin_stride = 3 * g.D + 2 + g.D * g.D;
    return g;
}
__host__ __device__ constexpr bool eloc5_supported(int n, bool has_mu) {
    const Eloc5Geom g = eloc5_geom(n, has_mu);
    return g.NB >= 1 && g.NB <= 5 && 8 * n <= 32 * g.OW && 3 * n <= 32 * g.WW && g.D <= 32 * g.WW && n <= 32 &&
           (g.ntri + g.GWN - 1) / g.GWN <= 5 && g.threads <= 384;
}

// Blocks of the upper block triangle of M = K^T K that Gram warp W of MW forms.  NB = 5, MW = 5: three blocks each, chosen
// so that a warp needs only 2 or 3 distinct operand fragments per k-step (14 fetches per k-step in total for 15 products).
struct GramList { int nb; int rb[5]; int cb[5]; unsigned mask; };
__host__ __device__ constexpr GramList gram_list(int NB, int MW, int W) {
    GramList L{};
    if (NB == 5 && MW == 5) {
        const int blocks[5][3][2] = {{{0, 0}, {0, 1}, {0, 2}}, {{0, 3}, {0, 4}, {3, 4}}, {{1, 1}, {1, 2}, {2, 2}},
                                     {{1, 3}, {1, 4}, {3, 3}}, {{2, 3}, {2, 4}, {4, 4}}};
        for (int t = 0; t < 3; ++t) { L.rb[t] = blocks[W][t][0]; L.cb[t] = blocks[W][t][1]; }
        L.nb = 3;
    } else {
        int blk = 0;
        for (int r = 0; r < NB; ++r)
            for (int c = r; c < NB; ++c, ++blk)
                if (blk % MW == W && L.nb < 5) { L.rb[L.nb] = r; L.cb[L.nb] = c; ++L.nb; }
    }
    for (int q = 0; q < L.nb; ++q) L.mask |= (1u << L.rb[q]) | (1u << L.cb[q]);
    return L;
}
// M = K^T K from the shared copy of K (row-major): the A and the B operand of block (rb, cb) at k-step k are the SAME kind
// of fragment, Ks[4 k + t][8 c + g] with c = rb or cb, so a warp fetches each column-block fragment it needs once per k-step
// (shared-memory bandwidth, not the tensor pipe, bounds this kernel).
template <int SN, int SMU, int W>
__device__ __forceinline__ void phase_gram5w(double* M, const double* Ks, int lane) {
    constexpr Eloc5Geom G_ = eloc5_geom(SN, SMU != 0);
    constexpr int D8 = G_.D8, DP = G_.DP, NB = G_.NB, KS = D8 / 4;
    constexpr GramList GL = gram_list(G_.NB, G_.GWN, W);
    const int g8 = lane >> 2, t4 = lane & 3;
    const double* base = Ks + t4 * DP + g8;
    double acc[GL.nb > 0 ? GL.nb : 1][2];
#pragma unroll
    for (int q = 0; q < GL.nb; ++q) { acc[q][0] = 0.0; acc[q][1] = 0.0; }
    double fc[NB], fn[NB];
#pragma unroll
    for (int c = 0; c < NB; ++c) { fc[c] = 0.0; fn[c] = 0.0; if ((GL.mask >> c) & 1u) fc[c] = lds_ordered(base + 8 * c); }
#pragma unroll
    for (int k = 0; k < KS; ++k) {
        if (k + 1 < KS) {
#pragma unroll
            for (int c = 0; c < NB; ++c) if ((GL.mask >> c) & 1u) fn[c] = lds_ordered(base + 8 * c + 4 * (k + 1) * DP);
        }
#pragma unroll
        for (int q = 0; q < GL.nb; ++q) dmma_ordered(acc[q][0], acc[q][1], fc[GL.rb[q]], fc[GL.cb[q]]);
#pragma unroll
        for (int c = 0; c < NB; ++c) fc[c] = fn[c];
    }
#pragma unroll
    for (int q = 0; q < GL.nb; ++q)
        *reinterpret_cast<double2*>(M + (8 * GL.rb[q] + g8) * DP + 8 * GL.cb[q] + 2 * t4) = make_double2(acc[q][0], acc[q][1]);
}
template <int SN, int SMU, int W = 0>
__device__ __forceinline__ void phase_gram5(double* M, const double* Ks, int mwarp, int lane) {
    constexpr Eloc5Geom G_ = eloc5_geom(SN, SMU != 0);
    if constexpr (W < G_.GWN) {
        if (mwarp == W) phase_gram5w<SN, SMU, W>(M, Ks, lane);
        else phase_gram5<SN, SMU, W + 1>(M, Ks, mwarp, lane);
    }
}

// Radial function and three derivatives from the certified Taylor table: nodes below `ncache` from the mirror in shared
// memory (rows of kRtPitch doubles: the 16-byte chunks of eight different rows fall into different bank groups), the
// others through L1.  One row = 96 bytes per item, different for every lane: from global memory that is up to 32 cache
// lines per warp instruction, 29 % of the L1 / shared-memory data-pipe traffic of the sweep before the mirror.
constexpr int kRtPitch = 14;
__device__ __forceinline__ bool radial_eval_mirror(const RtHeader& T, const double* __restrict__ cache, int ncache, double d, double (&f)[4]) {
    const double kf = rint(d * T.inv_delta);
    if (T.coef == nullptr || !(kf < (double)T.n_nodes) || !(kf >= 0.0)) return false;
    const double t = fma(-kf, T.delta, d);
    const int k = (int)kf;
    double c[kRtCoef];
    if (k < ncache) {
        const double2* c2 = reinterpret_cast<const double2*>(cache + k * kRtPitch);
#pragma unroll
        for (int q = 0; q < kRtCoef / 2; ++q) { const double2 v = c2[q]; c[2 * q] = v.x; c[2 * q + 1] = v.y; }
    } else {
        const double2* c2 = reinterpret_cast<const double2*>(T.coef + (size_t)k * kRtCoef);
#pragma unroll
        for (int q = 0; q < kRtCoef / 2; ++q) { const double2 v = __ldg(c2 + q); c[2 * q] = v.x; c[2 * q + 1] = v.y; }
    }
    radial_horner<3>(c, t, f);
    return true;
}

// Design notes (each was a compile-time switch while it was being measured; profiles/README.md has the numbers).
// RK in the accumulators: the RK combination of K enters K' = K A as the INITIAL VALUE of the tensor-core accumulators and the
// workers store A already multiplied by the stage's step factor: the new K leaves the DMMA chain finished, with
// 0 - 2 scalar FP64 instructions per element and stage instead of 2 - 5 (rk_elem).  With K_s the input of sub-stage s of
// the 3/8 rule and A_s' = h c_s A_s, c = (1/3, 1, 1, 1/8):
//   K_1 = K_0 + K_0 A_0'          K_2 = (2 K_0 - K_1) + K_1 A_1'          K_3 = (2 K_1 - K_2) + K_2 A_2'
//   K_new = (6 K_2 - K_0) / 8 + 3/8 K_3 + K_3 A_3'
// (same polynomial in h k_1 .. h k_4 as rk_elem).  Buffer KB holds K_0, then -K_0 / 8, then (6 K_2 - K_0) / 8; KC holds K_1.
// A L from the items instead of from the assembled matrix: (A L)_i = sum_j A_ij (L_j - L_i) + (one-body
// block) L_i, and the pair term changes sign with the orientation of the pair exactly like components 0, 1 of the
// contraction records, so every item lane adds its 2-vector to those and the per-particle sums deliver k_L complete
// (11 FP64 instructions per item lane instead of D-term chains on D lanes; as one more row operand of the tensor-core
// product it cost its full pipe time, +3 ms).
// Hand-overs: the two CTA-wide barriers of a stage became point-to-point hand-overs between the owner and the worker group
// (named barriers with bar.arrive on the producing and bar.sync on the consuming side, each with all NT threads of the CTA
// as participants), so that neither group waits for the other at a place where it needs nothing from it:
//   5  items of the stage in place (A off-diagonal, R matrices)      workers arrive, owners sync before their row sums
//   2  row sums in place (y, u, rho)                                 owners arrive,  workers sync before scalars / next radial functions
//   6  K A done: A may be overwritten                                owners arrive,  workers sync before the items of the next stage
//   7  M = K^T K of the stage in place                               owners arrive,  workers sync before the contraction
//   8  contraction done: M may be overwritten                        workers arrive, owners sync before the next Gram matrix
// (1: owners only, 3: workers only, 4: whole CTA at the walker boundaries.)  Every hand-over alternates strictly: the
// producer of one is the consumer of another further round the cycle, so no barrier is armed twice before it completes.
#ifndef FF_E5_ROT
#define FF_E5_ROT 2          // warps by which every other CTA of an SM shifts its roles (0: off)
#endif

#ifdef FF_E5_TIMING
__device__ unsigned long long g_e5_cyc[4][16];
#define E5T(seg) do { if (obs >= 0 && (tid0 & 31) == 0) { const long long t_ = clock64(); atomicAdd(&g_e5_cyc[obs][seg], (unsigned long long)(t_ - tprev)); tprev = t_; } } while (0)
#else
#define E5T(seg) do { } while (0)
#endif

template <int SN, int SMU>
__global__ void __launch_bounds__(eloc5_geom(SN, SMU != 0).threads, 2) eloc5_kernel(const FlowArgs a, double* __restrict__ fin, int* __restrict__ sm_count) {
    extern __shared__ __align__(16) double smem[];
    constexpr Eloc5Geom G_ = eloc5_geom(SN, SMU != 0);
    constexpr int n = G_.n, D = G_.D, DP = G_.DP, NP = G_.NP, P = G_.P, NB = G_.NB;
    constexpr int NT = G_.threads, OW = G_.OW, WW = G_.WW, NOWN = 32 * OW, NWRK = 32 * WW;
    constexpr int RP = G_.RP, RMAT = G_.RMAT;
    constexpr int kScalWarp = WW >= 3 ? 2 : WW - 1;       // worker warp that carries Delta and lapDelta
    static_assert(eloc5_supported(SN, SMU != 0), "eloc5_kernel: particle number not supported");
    double* const S = smem;
    const double h = (a.tb - a.ta) / a.nsteps;
    const int NS = 4 * a.nsteps;

    // Roles by ROTATED warp index: the NB owner warps of a CTA sit on NB consecutive warp slots, i.e. with NB = 5 two of them
    // on the same scheduler (warp slot mod 4), and the co-resident CTA, with the same warp-slot alignment, puts its pair on
    // that scheduler too: four tensor-core streams on one scheduler, two on each of the others.  The CTAs of an SM count
    // themselves (an atomic on a per-SM counter behind the final-state buffer) and every other one shifts its roles by
    // FF_E5_ROT = 2 warps: 3 + 2 + 3 + 2 streams (62.7 against 63.4 ms; shifts by 4 and 8 warps measure like none, 6 like
    // 2 -- and ODD shifts, which put the pair on scheduler 1 or 3, 66.3 ms: the placement of the worker warps with the
    // per-particle sums and the one-body lanes moves with them).
    int rot = 0;
#if FF_E5_ROT
    if (NB == 5 && sm_count != nullptr) {
        int* const flag = reinterpret_cast<int*>(S);
        if (threadIdx.x == 0) {
            unsigned smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            *flag = (atomicAdd(sm_count + (smid & 255u), 1) & 1) * FF_E5_ROT;
        }
        __syncthreads();
        rot = *flag;
        __syncthreads();
    }
#endif
    const int tid0 = ((int)threadIdx.x + NT - 32 * rot) % NT;
    const bool owner0 = tid0 < NOWN;

    for (int e = tid0; e < G_.total; e += NT) S[e] = 0.0;                             // zero padding of the matrices and vectors, once
    // mirror of the head of the eta table (a.rt_cache_nodes rows fit behind the walker block)
    double* const rt_cache = S + G_.total;
    int ncache = 0;
    {
        const RtHeader he = rt_load_header(a.rt_eta);
        if (he.coef != nullptr) ncache = min(a.rt_cache_nodes, he.n_nodes);
        for (int e = tid0; e < ncache * kRtCoef; e += NT) {
            const int k = e / kRtCoef, q = e - k * kRtCoef;
            rt_cache[k * kRtPitch + q] = he.coef[e];
        }
    }
    __syncthreads();

    // Owners and workers run their own stage loops (the register allocation is the larger of the two, not their sum);
    // the CTA-wide barriers inside are named barrier 4 with all NT threads, reached from both loops (barrier 0 is left to
    // __syncthreads, which every thread has to execute at the same place).
    if (owner0) {
        for (long long b = blockIdx.x; b < a.B; b += gridDim.x) {
            // ---- initial state: K = 1 (registers and shared copy), gDelta = 0; y = x -------------------------------
            double Kr[NB][2];
            double gd = 0.0, gdB = 0.0, gdC = 0.0;
            {
                const int warp = tid0 >> 5, g8 = (tid0 >> 2) & 7, t4 = tid0 & 3;
#pragma unroll
                for (int rb = 0; rb < NB; ++rb) {
#pragma unroll
                    for (int e = 0; e < 2; ++e)
                        Kr[rb][e] = (8 * warp + g8 == 8 * rb + 2 * t4 + e && 8 * warp + g8 < D) ? 1.0 : 0.0;
                    *reinterpret_cast<double2*>(S + G_.oKs + (8 * warp + g8) * DP + 8 * rb + 2 * t4) = make_double2(Kr[rb][0], Kr[rb][1]);
                }
            }
            for (int e = tid0; e < D; e += NOWN) {
                S[G_.oY + e] = a.x_in[b * D + e];
                S[G_.oL0 + e] = 0.0; S[G_.oL1 + e] = 0.0; S[G_.oLB + e] = 0.0; S[G_.oLC + e] = 0.0; S[G_.oYB + e] = 0.0; S[G_.oYC + e] = 0.0;
            }
            if (tid0 < 8) S[G_.oScal + tid0] = 0.0;
            named_bar_sync(4, NT);
            named_bar_sync(4, NT);                       // (the workers evaluate the radial functions of stage 0)
            named_bar_arrive(6, NT);                     // A is free for the items of stage 0
#ifdef FF_E5_TIMING
            const int obs = (tid0 >> 5) == 0 ? 0 : (tid0 >> 5) == 1 ? 1 : -1;
            long long tprev = clock64();
#endif
            for (int stage = 0; stage < NS; ++stage) {
                const int sub = stage & 3;
                E5T(15);
                const int tid = stage_local(tid0);          // lane indices of this stage (see stage_local)
                const int warp = tid >> 5, g8 = (tid >> 2) & 7, t4 = tid & 3;
                double* const Ks = S + G_.oKs;
                double* const A = S + G_.oA;
                double* const R1 = S + G_.oR1;
                double* const Y = S + G_.oY;
                double* const U = S + G_.oU;
                // ======== phase 1: M = K^T K of this stage ==========================================================
                named_bar_sync(8, NT);                // the workers are done with the previous M
                if (warp >= G_.G0 && warp < G_.G0 + G_.GWN) phase_gram5<SN, SMU>(S + G_.oM, Ks, warp - G_.G0, tid & 31);
                E5T(0);
                named_bar_arrive(7, NT);              // M of this stage is in place
                named_bar_sync(5, NT);                // the items of this stage are in place
                E5T(1);
                // ======== phase 2 ===================================================================================
                // ---- per-particle sums of this stage: k_y (y advances here), u, rho, diagonal of A -----------------
                // output of this lane: row sum c8 = tid / n of particle i = tid % n: matrices 0..4 (k_y, u, rho) or,
                // c8 = 5, 6, 7, the diagonal block (0,0), (0,1), (1,1) of A = minus the sum of the off-diagonal blocks
                // of its rows (the slot of the diagonal block itself holds minus the one-body part)
                {
                    const int c8 = tid / n, g1_i = tid - c8 * n;
                    if (c8 < 8) {
                        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
                        if (c8 < 5) {
                            const double* R = R1 + c8 * RMAT + g1_i * RP;
#pragma unroll
                            for (int k = 0; k < n; ++k) {
                                const double v = R[k];
                                if ((k & 3) == 0) s0 += v; else if ((k & 3) == 1) s1 += v; else if ((k & 3) == 2) s2 += v; else s3 += v;
                            }
                        } else {
                            // A is symmetric: block (al, be) of particle i is read down columns 2 i + al (consecutive
                            // lanes: stride 2), rows 2 k + be (physical row a_row(2 k) + 4 be)
                            const double* Ac = A + (c8 >= 6 ? 4 * DP : 0) + 2 * g1_i + (c8 == 7 ? 1 : 0);
#pragma unroll
                            for (int k = 0; k < n; ++k) {
                                const double v = (SMU != 0 || k != g1_i) ? Ac[a_row(2 * k) * DP] : 0.0;
                                if ((k & 3) == 0) s0 -= v; else if ((k & 3) == 1) s1 -= v; else if ((k & 3) == 2) s2 -= v; else s3 -= v;
                            }
                        }
                        const double acc = (s0 + s1) + (s2 + s3);
                        if (c8 < 2) {
                            const int m = 2 * g1_i + c8;
                            Y[m] = rk_elem(sub, Y[m], h * acc, S[G_.oYB + m], S[G_.oYC + m]);
                        } else if (c8 < 4) U[2 * g1_i + c8 - 2] = acc;
                        else if (c8 == 4) S[G_.oP1 + g1_i] = acc;
                        else if (c8 == 5) A[a_row(2 * g1_i) * DP + 2 * g1_i] = acc;
                        else if (c8 == 6) { A[a_row(2 * g1_i) * DP + 2 * g1_i + 1] = acc; A[a_row(2 * g1_i + 1) * DP + 2 * g1_i] = acc; }
                        else A[a_row(2 * g1_i + 1) * DP + 2 * g1_i + 1] = acc;
                    }
                }
                E5T(2);
                named_bar_sync(1, NOWN);              // A, u, y complete (owner warps)
                named_bar_arrive(2, NT);              // ... and visible to the workers when they get there
                E5T(3);
                // ---- K' = K A on the tensor cores, k-step (rb, e): A operand = own registers -----------------------
                double acc[NB][2];
                {   // accumulators start from the RK combination of the earlier sub-stages (see "RK in the accumulators" above)
                    double2* const PB = reinterpret_cast<double2*>(S + G_.oKB) + tid;
                    double2* const PC = reinterpret_cast<double2*>(S + G_.oKC) + tid;
#pragma unroll
                    for (int rn = 0; rn < NB; ++rn) {
                        const double k0 = Kr[rn][0], k1 = Kr[rn][1];
                        if (sub == 0) {
                            PB[rn * NOWN] = make_double2(k0, k1);
                            acc[rn][0] = k0; acc[rn][1] = k1;
                        } else if (sub == 1) {
                            const double2 Bv = PB[rn * NOWN];
                            acc[rn][0] = fma(2.0, Bv.x, -k0); acc[rn][1] = fma(2.0, Bv.y, -k1);
                            PB[rn * NOWN] = make_double2(-0.125 * Bv.x, -0.125 * Bv.y);
                            PC[rn * NOWN] = make_double2(k0, k1);
                        } else if (sub == 2) {
                            const double2 Bv = PB[rn * NOWN], Cv = PC[rn * NOWN];
                            acc[rn][0] = fma(2.0, Cv.x, -k0); acc[rn][1] = fma(2.0, Cv.y, -k1);
                            PB[rn * NOWN] = make_double2(fma(0.75, k0, Bv.x), fma(0.75, k1, Bv.y));
                        } else {
                            const double2 Bv = PB[rn * NOWN];
                            acc[rn][0] = fma(0.375, k0, Bv.x); acc[rn][1] = fma(0.375, k1, Bv.y);
                        }
                    }
                }
                // ---- K u (for gDelta' = -u^T J): row sums over the quad, from the K at the stage input ------------------
                double ku = 0.0;
                {
                    double ku1 = 0.0;
#pragma unroll
                    for (int rb = 0; rb < NB; ++rb) {
                        const double2 uv = *reinterpret_cast<const double2*>(U + 8 * rb + 2 * t4);
                        ku = fma(Kr[rb][0], uv.x, ku);
                        ku1 = fma(Kr[rb][1], uv.y, ku1);
                    }
                    ku += ku1;
                }
                {
                    const double* Ab = A + t4 * DP + g8;
                    double bn[NB], bc[NB];
#pragma unroll
                    for (int rn = 0; rn < NB; ++rn) bc[rn] = lds_ordered(Ab + 8 * rn);
#pragma unroll
                    for (int ks = 0; ks < 2 * NB; ++ks) {
                        const int rb = ks >> 1, e = ks & 1;
                        if (ks + 1 < 2 * NB) {
                            const int rb1 = (ks + 1) >> 1, e1 = (ks + 1) & 1;
#pragma unroll
                            for (int rn = 0; rn < NB; ++rn) bn[rn] = lds_ordered(Ab + (8 * rb1 + 4 * e1) * DP + 8 * rn);
                        }
#pragma unroll
                        for (int rn = 0; rn < NB; ++rn) dmma_ordered(acc[rn][0], acc[rn][1], Kr[rb][e], bc[rn]);
#pragma unroll
                        for (int rn = 0; rn < NB; ++rn) bc[rn] = bn[rn];
                    }
                }
                E5T(4);
                if (stage + 1 < NS) named_bar_arrive(6, NT);       // A may be overwritten by the items of the next stage
                // ---- the accumulators ARE the new K; shared copy for the Gram matrix of the next stage -----------------
                ku += __shfl_xor_sync(0xffffffffu, ku, 1);
                ku += __shfl_xor_sync(0xffffffffu, ku, 2);
#pragma unroll
                for (int rn = 0; rn < NB; ++rn) {
                    Kr[rn][0] = acc[rn][0]; Kr[rn][1] = acc[rn][1];
                    *reinterpret_cast<double2*>(Ks + (8 * warp + g8) * DP + 8 * rn + 2 * t4) = make_double2(Kr[rn][0], Kr[rn][1]);
                }
                gd = rk_elem(sub, gd, -h * ku, gdB, gdC);
                E5T(5);
                named_bar_sync(1, NOWN);              // the shared copy of the new K is complete (owners only)
                E5T(7);
            }
            // ---- final state to global memory: gDelta, J = K^T row-major (the workers write the vectors) -----------
            {
                double* F = fin + (size_t)b * G_.fin_stride;
                const int warp = tid0 >> 5, g8 = (tid0 >> 2) & 7, t4 = tid0 & 3;
                const int c = 8 * warp + g8;
                if (c < D) {
                    if (t4 == 0) F[2 * D + c] = gd;
#pragma unroll
                    for (int rb = 0; rb < NB; ++rb)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int r = 8 * rb + 2 * t4 + e;
                            if (r < D) F[3 * D + 2 + r * D + c] = Kr[rb][e];
                        }
                }
            }
            named_bar_sync(4, NT);
        }
    } else {
        // item of this worker lane (one item per lane: P <= NWRK)
        int it_i0 = 0, it_j0 = 0;
        {
            const int p0 = tid0 - NOWN < P ? tid0 - NOWN : 0;
            if (p0 < NP) {
                int i = 0, rem = p0;
                while (rem >= n - 1 - i) { rem -= n - 1 - i; ++i; }
                it_i0 = i; it_j0 = i + 1 + rem;
            } else { it_i0 = p0 - NP; it_j0 = it_i0; }
        }
        for (long long b = blockIdx.x; b < a.B; b += gridDim.x) {
            // the item of the coming stage: r, d, 1/d and the radial function with three derivatives
            double rx = 0.0, ry = 0.0, dd = 1.0, inv_d = 1.0, f0 = 0.0, f1 = 0.0, f2 = 0.0, f3 = 0.0;
            double sDl = 0.0, sDlB = 0.0, sDlC = 0.0, sLd = 0.0, sLdB = 0.0, sLdC = 0.0;     // shares of Delta, lapDelta (lanes wl < n)
            named_bar_sync(4, NT);                       // (the owners have set the initial state)
#ifdef FF_E5_TIMING
            const int obs = (tid0 >> 5) == OW ? 2 : (tid0 >> 5) == OW + WW - 1 ? 3 : -1;
            long long tprev = clock64();
#endif
            for (int stage = -1; stage < NS; ++stage) {
                const int sub = stage & 3;
                E5T(15);
                const int tid = stage_local(tid0);          // lane indices of this stage (see stage_local)
                const int warp = tid >> 5;
                const int wl = tid - NOWN;                  // index inside the worker group
                const bool it_valid = wl < P;
                const int it_p = it_valid ? wl : 0;
                const bool it_pair = it_p < NP;
                const int it_i = stage_local(it_i0), it_j = stage_local(it_j0);
                double* const A = S + G_.oA;
                double* const M = S + G_.oM;
                double* const R1 = S + G_.oR1;
                double* const Y = S + G_.oY;
                double* const U = S + G_.oU;
                double* const Lc = S + ((stage & 1) ? G_.oL1 : G_.oL0);          // L at the stage input
                double* const Ln = S + ((stage & 1) ? G_.oL0 : G_.oL1);
                if (stage >= 0) {
                    // ======== phase 1: the items of this stage from r and the radial functions ======================
                    double ca = 0.0, cb_ = 0.0, ccq = 0.0, ceq = 0.0, a00 = 0.0, a01 = 0.0, a11 = 0.0;
                    if (a.stash_y != nullptr && wl < D) a.stash_y[(b * NS + stage) * D + wl] = Y[wl];
                    if (it_valid) {
                        if (a.stash_c != nullptr) {
                            double* sc = a.stash_c + ((b * NS + stage) * P + it_p) * 3;
                            sc[0] = f0; sc[1] = f1; sc[2] = f2;
                        }
                        const double mult = it_pair ? 2.0 : 1.0;
                        const double inv_d2 = inv_d * inv_d;
                        ca = f1 * inv_d;
                        cb_ = (f2 - ca) * inv_d2;
                        const double q1 = mult * fma(f2, dd, 3.0 * f1);
                        const double q2 = mult * fma(f3, dd, 4.0 * f2);
                        ccq = q1 * inv_d;
                        ceq = (q2 - ccq) * inv_d2;
                        // A is stored multiplied by the step factor h c_sub of this sub-stage (see "RK in the accumulators")
                        const double hs = sub == 0 ? h * (1.0 / 3.0) : sub == 3 ? h * 0.125 : h;
                        const double caS = hs * ca, f0S = hs * f0;
                        a00 = fma(caS * rx, rx, f0S); a01 = caS * rx * ry; a11 = fma(caS * ry, ry, f0S);
                        const double v0 = f0 * rx, v1 = f0 * ry, v2 = ccq * rx, v3 = ccq * ry, v4 = fma(f1, dd, 2.0 * f0);
                        if (it_pair) {          // both orientations of the pair; off-diagonal blocks of A (row-permuted storage)
                            double* const Rij = R1 + it_i * RP + it_j;
                            double* const Rji = R1 + it_j * RP + it_i;
                            Rij[0] = v0; Rji[0] = -v0;
                            Rij[RMAT] = v1; Rji[RMAT] = -v1;
                            Rij[2 * RMAT] = v2; Rji[2 * RMAT] = -v2;
                            Rij[3 * RMAT] = v3; Rji[3 * RMAT] = -v3;
                            Rij[4 * RMAT] = v4; Rji[4 * RMAT] = v4;
                        } else {                // one-body item: diagonal of the matrices
                            double* const Rii = R1 + it_i * (RP + 1);
                            Rii[0] = v0; Rii[RMAT] = v1; Rii[2 * RMAT] = v2; Rii[3 * RMAT] = v3; Rii[4 * RMAT] = v4;
                        }
                    }
                    // (the R matrices were free since the owners' row sums; only the blocks of A have to wait for the owners' K A)
                    named_bar_sync(6, NT);            // the owners are done with the previous A
                    E5T(6);
                    if (it_valid) {
                        const int i2 = 2 * it_i, j2 = 2 * it_j;
                        if (it_pair) {          // off-diagonal blocks of A (row-permuted storage), both orientations
                            *reinterpret_cast<double2*>(A + a_row(i2) * DP + j2) = make_double2(-a00, -a01);
                            *reinterpret_cast<double2*>(A + a_row(i2 + 1) * DP + j2) = make_double2(-a01, -a11);
                            *reinterpret_cast<double2*>(A + a_row(j2) * DP + i2) = make_double2(-a00, -a01);
                            *reinterpret_cast<double2*>(A + a_row(j2 + 1) * DP + i2) = make_double2(-a01, -a11);
                        } else {                // one-body item: minus its block in the diagonal slot of A
                            *reinterpret_cast<double2*>(A + a_row(i2) * DP + i2) = make_double2(-a00, -a01);
                            *reinterpret_cast<double2*>(A + a_row(i2 + 1) * DP + i2) = make_double2(-a01, -a11);
                        }
                    }
                    E5T(0);
                    named_bar_arrive(5, NT);          // the items of this stage are in place
                    named_bar_sync(7, NT);            // M of this stage is in place
                    E5T(1);
                    // ======== phase 2 ===============================================================================
                    // ---- contraction of this lane's item with M = J J^T --------------------------------------------
                    if (it_valid) {
                        const int i2 = 2 * it_i, j2 = 2 * it_j;
                        double w00, w01, w11;
                        if (it_pair) {
                            const double2 mii0 = *reinterpret_cast<const double2*>(M + i2 * DP + i2);
                            const double mii1 = M[(i2 + 1) * DP + i2 + 1];
                            const double2 mjj0 = *reinterpret_cast<const double2*>(M + j2 * DP + j2);
                            const double mjj1 = M[(j2 + 1) * DP + j2 + 1];
                            const double2 mij0 = *reinterpret_cast<const double2*>(M + i2 * DP + j2);
                            const double2 mij1 = *reinterpret_cast<const double2*>(M + (i2 + 1) * DP + j2);
                            w00 = mii0.x + mjj0.x - 2.0 * mij0.x;
                            w11 = mii1 + mjj1 - 2.0 * mij1.y;
                            w01 = mii0.y + mjj0.y - mij0.y - mij1.x;
                        } else {
                            const double2 mii0 = *reinterpret_cast<const double2*>(M + i2 * DP + i2);
                            w00 = mii0.x; w01 = mii0.y; w11 = M[(i2 + 1) * DP + i2 + 1];
                        }
                        const double wrx = fma(w00, rx, w01 * ry), wry = fma(w01, rx, w11 * ry);
                        const double trw = w00 + w11, rwr = fma(rx, wrx, ry * wry);
                        double* const G2 = S + G_.oG2 + 3 * it_p;
                        double dLx, dLy;
                        {
                            const double2 li = *reinterpret_cast<const double2*>(Lc + i2);
                            dLx = li.x; dLy = li.y;
                            if (it_pair) { const double2 lj = *reinterpret_cast<const double2*>(Lc + j2); dLx -= lj.x; dLy -= lj.y; }
                        }
                        const double tl = ca * fma(rx, dLx, ry * dLy);
                        G2[0] = fma(ca, fma(2.0, wrx, trw * rx), cb_ * rwr * rx) + fma(f0, dLx, tl * rx);
                        G2[1] = fma(ca, fma(2.0, wry, trw * ry), cb_ * rwr * ry) + fma(f0, dLy, tl * ry);
                        G2[2] = fma(ccq, trw, ceq * rwr);
                    }
                    E5T(2);
                    if (stage + 1 < NS) named_bar_arrive(8, NT);    // M may be overwritten by the next Gram matrix
                    named_bar_sync(3, NWRK);
                    // ---- per-particle sums of the contractions: lane (particle wl / 3, component wl % 3) -----------
                    {
                        // (two lanes per sum, each with the partners of one parity, measured slower: 1890 against 1360 cycles)
                        const int g2_i = wl / 3, g2_k = wl - 3 * g2_i;
                        if (g2_i < n) {
                            const double acc = gather3<SN, SMU>(S + G_.oG2, g2_i, g2_k);
                            // components 0, 1 are k_L = A L + (d2v : M) complete (see "A L from the items"): L advances here
                            if (g2_k < 2) {
                                const int m = 2 * g2_i + g2_k;
                                Ln[m] = rk_elem(sub, Lc[m], h * acc, S[G_.oLB + m], S[G_.oLC + m]);
                            } else S[G_.oP2 + g2_i] = acc;
                        }
                    }
                    E5T(3);
                    named_bar_sync(2, NT);                // the owners' sums of this stage are in place: y, A, u, rho
                    E5T(4);
                    // (L' = A L + (d2v : M) came out of the per-particle sums above)
                    // Delta' = -rho, lapDelta' = -(sum_i part2_i + u.L): the RK combination is linear, so lane i < n carries
                    // the share of particle i through all stages in registers and the shares meet once, after the sweep
                    // (a per-stage warp reduction was a 25-deep FP64 chain on the critical path of the workers)
                    // (on worker warp kScalWarp: the first warps carry the per-particle sums)
                    if (const int sl = wl - 32 * kScalWarp; sl >= 0 && sl < n) {
                        const double rho = S[G_.oP1 + sl];
                        const double2 uv = *reinterpret_cast<const double2*>(U + 2 * sl), lv = *reinterpret_cast<const double2*>(Lc + 2 * sl);
                        const double lp = fma(uv.x, lv.x, fma(uv.y, lv.y, S[G_.oP2 + sl]));
                        sDl = rk_elem(sub, sDl, -h * rho, sDlB, sDlC);
                        sLd = rk_elem(sub, sLd, -h * lp, sLdB, sLdC);
                    }
                    E5T(5);
                }
                // ---- radial functions of the next stage at the y just advanced (none after the last stage) ---------
                if (stage + 1 < NS && it_valid) {
                    if (it_pair) {
                        const double2 yi = *reinterpret_cast<const double2*>(Y + 2 * it_i), yj = *reinterpret_cast<const double2*>(Y + 2 * it_j);
                        rx = yi.x - yj.x; ry = yi.y - yj.y;
                    } else {
                        const double2 yi = *reinterpret_cast<const double2*>(Y + 2 * it_i);
                        rx = yi.x; ry = yi.y;
                    }
                    const RtHeader my_rt = rt_load_header(it_pair ? a.rt_eta : a.rt_mu);
                    const double d2 = fma(rx, rx, ry * ry);
                    inv_d = rsqrt(d2);
                    dd = d2 * inv_d;
                    double f[4];
                    if (radial_eval_mirror(my_rt, rt_cache, it_pair ? ncache : 0, dd, f)) {
                        f0 = f[0]; f1 = f[1]; f2 = f[2]; f3 = f[3];
                    } else {            // (its own array: the out-of-line call would pin f to the stack frame on the table path too)
                        double g[4];
                        radial_direct_global(it_pair ? a.eta_w1 : a.mu_w1, it_pair ? a.eta_b1 : a.mu_b1,
                                             it_pair ? a.eta_w2 : a.mu_w2, it_pair ? a.H_eta : a.H_mu, dd, g);
                        f0 = g[0]; f1 = g[1]; f2 = g[2]; f3 = g[3];
                    }
                }
                E5T(7);
                if (stage < 0) {
                    named_bar_sync(4, NT);            // (second barrier of the walker start: the owners wait for stage 0's radial functions)
                    named_bar_arrive(8, NT);          // M is free for the Gram matrix of stage 0
                }
            }
            // ---- final state to global memory: y, L, (Delta, lapDelta) ----------------------------------------------
            {
                double* F = fin + (size_t)b * G_.fin_stride;
                const int wl = tid0 - NOWN;
                for (int e = wl; e < D; e += NWRK) {
                    F[e] = S[G_.oY + e]; F[D + e] = S[G_.oL0 + e];       // NS is even: L ends in buffer 0
                    if (a.y_out) a.y_out[b * D + e] = S[G_.oY + e];
                }
                if ((tid0 >> 5) == OW + kScalWarp) {          // the per-particle shares of Delta and lapDelta (n <= 32 lanes of this warp)
                    const int sl = wl - 32 * kScalWarp;
                    double dl = sl < n ? sDl : 0.0, ld = sl < n ? sLd : 0.0;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        dl += __shfl_xor_sync(0xffffffffu, dl, o);
                        ld += __shfl_xor_sync(0xffffffffu, ld, o);
                    }
                    if (sl == 0) {
                        F[3 * D] = dl; F[3 * D + 1] = ld;
                        if (a.delta_out) a.delta_out[b] = dl;
                    }
                }
            }
            named_bar_sync(4, NT);
        }
    }
}

}  // namespace ff
