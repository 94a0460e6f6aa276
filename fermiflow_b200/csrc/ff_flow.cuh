// Fixed-step (3/8-rule RK4) continuous normalizing flow of fermion coordinates, with
// optional divergence integral, adjoint stash, and the forward-mode (Jacobian + Laplacian)
// propagation that yields grad/laplacian of log p and the local energy in ONE sweep.
//
// Replaces, for dim = 2 and D_in = 1 MLPs:
//   flow.py:42-56 CNF.generate / CNF.delta_logp (via NeuralODE/nnModule.py:151 solve_ivp),
//   equivariant_funs.py:17-102 Backflow forward / divergence,
//   utils.py:44-65 y_grad_laplacian (2N nested autograd passes -> forward-mode here),
//   VMC.py:41-55 GSVMC.forward's kinetic + potential energy.
#pragma once
#include "ff_common.cuh"
#include "ff_slater.cuh"
#include "ff_radial_table.cuh"

namespace ff {

#ifdef FF_PHASE_TIMING
static __device__ unsigned long long g_phase_cycles[16];
#define FF_TICK(k) do { if (MODE == MODE_ELOC && tid == 0) { long long now_ = clock64(); tacc[k] += now_ - tlast; tlast = now_; } } while (0)
#else
#define FF_TICK(k) do {} while (0)
#endif

enum FlowMode { MODE_V = 0, MODE_DIV = 1, MODE_STASH = 2, MODE_ELOC = 3 };

struct FlowArgs {
    // model
    int n, n_up, H_eta, H_mu;
    const double *eta_w1, *eta_b1, *eta_w2, *mu_w1, *mu_b1, *mu_w2;
    const double *rt_eta, *rt_mu;   // certified Taylor tables of eta / mu (ff_radial_table.cuh), nullable
    int rt_cache_nodes;             // nodes of the eta table a kernel may mirror in shared memory behind its walker block
    double ta, tb;          // integrate from ta to tb
    int nsteps;
    // batch
    long long B;
    const double* x_in;     // [B][n][2]
    double* y_out;          // [B][n][2]   end point of the flow
    double* delta_out;      // [B]         integral of -div v  (MODE >= DIV)
    // adjoint stash (MODE >= STASH, nullable)
    double* stash_y;        // [B][4*nsteps][D]
    double* stash_c;        // [B][4*nsteps][P][3]   eta, eta', eta'' (or mu...) per item
    // MODE_ELOC
    const int* orb;         // occupation table, rows of n orbital ids (up block then down)
    const int* walker_state;// [B] row of `orb` per walker, or null (row 0 for everybody)
    double Z;               // Coulomb strength
    int harmonic;           // add 1/2 r^2
    double *logp, *grad, *lap, *kin, *pot, *eloc;
    // launch geometry (host-computed)
    int W;                  // walkers per CTA
    int P, NP;              // items per walker (pairs + singles), pairs
    int D, DP;              // 2n, padded row length of J
    int NSV;                // doubles of the stage-input state block: NV + D8*DP (E_loc) or NV
    int NV;                 // vector part: y, L, gDelta, Delta, lapDelta (E_loc: 3D+2) or y(+Delta)
    int NPAR;               // doubles of each RK partial / derivative block: NV + D*D (E_loc) or NV
    int wstride;            // shared doubles per walker
    int grec;               // doubles per item record (kGRec for MODE_ELOC, 3 otherwise: vx, vy, q)
    int off_G, off_AM, off_u, off_kLx, off_part, off_x0, off_sl;   // offsets inside a walker block
    // generic E_loc sweep for particle numbers whose Jacobian blocks do not all fit in shared memory (n > 26): the three RK
    // partials of J and its stage derivative live in global memory instead, 4 D^2 doubles per resident walker (L2 resident)
    double* jpart;
};

// State vector layout (MODE_ELOC): [y:D][L:D][gD:D][Delta, lapDelta][J: D x DP]
// otherwise:                        [y:D][Delta]

// Walker-block geometry of the CTA-synchronous sweeps, planned on the host (capi_flow.h plan_flow) into FlowArgs.
struct FlowGeom {
    int D, DP, NP, P, NV, NSV, NPAR, grec;
    int off_G, off_AM, off_u, off_kLx, off_part, off_x0, off_sl, wstride;
};
__host__ __device__ constexpr int ff_even(int x) { return (x + 1) & ~1; }
inline FlowGeom flow_geom(int mode, int n, bool has_mu, bool jglobal = false, int scratch_min = 0) {
    FlowGeom g{};
    const bool eloc = mode == MODE_ELOC;
    g.D = 2 * n;
    const int D8 = (g.D + 7) & ~7;
    g.NP = n * (n - 1) / 2; g.P = g.NP + (has_mu ? n : 0);
    g.DP = eloc ? D8 + 4 : g.D;                   // DP mod 16 in {4, 12}: conflict-free DMMA fragments
    g.NV = eloc ? 3 * g.D + 2 : g.D + (mode >= MODE_DIV ? 1 : 0);
    g.NSV = eloc ? ff_even(g.NV + D8 * g.DP) : g.NV;
    // (jglobal: the J parts of the RK partials are in FlowArgs::jpart; the area still holds the scratch of the finale)
    g.NPAR = eloc ? (jglobal ? ff_even(g.NV) : ff_even(g.NV + g.D * g.D)) : g.NV;
    g.grec = eloc ? kGRec : 3;
    int off = ff_even(g.NSV + (jglobal && 4 * g.NPAR < scratch_min ? scratch_min : 4 * g.NPAR));
    g.off_G = off; off = ff_even(off + g.P * g.grec);
    g.off_AM = off; if (eloc) off = ff_even(off + D8 * g.DP);
    g.off_u = off; if (eloc) off += g.D;
    g.off_kLx = off; if (eloc) off += g.D;
    g.off_part = off; off = ff_even(off + 2 * n);
    g.off_x0 = off; if (eloc) off += g.D;
    g.off_sl = g.NSV;
    g.wstride = ff_even(off);
    return g;
}

// ---- FP64 tensor-core (DMMA m8n8k4) building blocks --------------------------------------
// A dependent DMMA chain issues only every ~150 cycles, so every warp task below carries
// up to 2*CH independent accumulators (CH column blocks x two interleaved halves of K).
constexpr int kCH = 5;

// C[c] (8x8 each, c < nch) = A(8 x K) * B_c(K x 8).  Lane (g = lane/4, t = lane%4):
//   a_of(k)    -> A[g][k + t]          (the caller bakes g, t into the functor)
//   b_of(c, k) -> B_c[k + t][g]
// K is a multiple of 4.  Results: acc[c][0..1] = C_c[g][2t, 2t+1].
template <class AF, class BF>
__device__ __forceinline__ void dmma_chunk(int K, int nch, AF a_of, BF b_of, double (&acc)[kCH][2]) {
    double e[kCH][2], o[kCH][2];
#pragma unroll
    for (int c = 0; c < kCH; ++c) { e[c][0] = e[c][1] = o[c][0] = o[c][1] = 0.0; }
    int k = 0;
    for (; k + 8 <= K; k += 8) {
        const double a0 = a_of(k), a1 = a_of(k + 4);
#pragma unroll
        for (int c = 0; c < kCH; ++c)
            if (c < nch) {
                dmma_m8n8k4(e[c][0], e[c][1], a0, b_of(c, k));
                dmma_m8n8k4(o[c][0], o[c][1], a1, b_of(c, k + 4));
            }
    }
    if (k < K) {
        const double a0 = a_of(k);
#pragma unroll
        for (int c = 0; c < kCH; ++c)
            if (c < nch) dmma_m8n8k4(e[c][0], e[c][1], a0, b_of(c, k));
    }
#pragma unroll
    for (int c = 0; c < kCH; ++c) { acc[c][0] = e[c][0] + o[c][0]; acc[c][1] = e[c][1] + o[c][1]; }
}

// Same with an individual A operand per chain: a_of(c, k) -> A_c[g][k + t].
template <class AF, class BF>
__device__ __forceinline__ void dmma_chunk_ab(int K, int nch, AF a_of, BF b_of, double (&acc)[kCH][2]) {
    double e[kCH][2], o[kCH][2];
#pragma unroll
    for (int c = 0; c < kCH; ++c) { e[c][0] = e[c][1] = o[c][0] = o[c][1] = 0.0; }
    int k = 0;
    for (; k + 8 <= K; k += 8) {
#pragma unroll
        for (int c = 0; c < kCH; ++c)
            if (c < nch) {
                dmma_m8n8k4(e[c][0], e[c][1], a_of(c, k), b_of(c, k));
                dmma_m8n8k4(o[c][0], o[c][1], a_of(c, k + 4), b_of(c, k + 4));
            }
    }
    if (k < K) {
#pragma unroll
        for (int c = 0; c < kCH; ++c)
            if (c < nch) dmma_m8n8k4(e[c][0], e[c][1], a_of(c, k), b_of(c, k));
    }
#pragma unroll
    for (int c = 0; c < kCH; ++c) { acc[c][0] = e[c][0] + o[c][0]; acc[c][1] = e[c][1] + o[c][1]; }
}

// Gram matrix M = J J^T (upper block triangle of 8x8 blocks) of every walker.  The
// W * NB(NB+1)/2 blocks are dealt out evenly: each warp owns a contiguous run of blocks for
// the whole kernel (GramPlan, computed once) and works on up to kCH of them at once.
// J: [D8][DP], rows >= D zero.
struct GramPlan {
    int nch;                 // blocks of this warp handled by the fast path (<= kCH)
    int first, last;         // run of blocks of this warp
    int oA[kCH], oB[kCH], oM[kCH];   // shared-memory offsets (doubles, relative to wbase)
};

__device__ __forceinline__ void gram_block_offsets(int blk, int W, int D8, int DP, int wstride, int oJ, int off_AM,
                                                   int g, int t, int& oA, int& oB, int& oM) {
    const int NB = D8 >> 3, ntri = NB * (NB + 1) / 2;
    const int w = blk / ntri;
    int rem = blk - w * ntri, rb = 0;
    while (rem >= NB - rb) { rem -= NB - rb; ++rb; }
    const int cb = rb + rem;
    oA = w * wstride + oJ + (8 * rb + g) * DP + t;
    oB = w * wstride + oJ + (8 * cb + g) * DP + t;
    oM = w * wstride + off_AM + (8 * rb + g) * DP + 8 * cb + 2 * t;
}

// Blocks are dealt to the warps [warp0, warp0 + nwarp) only (helper warps when present).
__device__ __forceinline__ GramPlan gram_plan(int W, int D8, int DP, int wstride, int oJ, int off_AM,
                                              int warp0 = 0, int nwarp = -1) {
    const int lane = threadIdx.x & 31;
    if (nwarp < 0) nwarp = blockDim.x >> 5;
    const int warp = (int)(threadIdx.x >> 5) - warp0;
    const int g = lane >> 2, t = lane & 3, NB = D8 >> 3, total = W * NB * (NB + 1) / 2;
    const int per = (total + nwarp - 1) / nwarp;
    GramPlan p;
    if (warp < 0 || warp >= nwarp) { p.first = p.last = p.nch = 0; for (int c = 0; c < kCH; ++c) p.oA[c] = p.oB[c] = p.oM[c] = 0; return p; }
    p.first = min(total, warp * per);
    p.last = min(total, p.first + per);
    p.nch = min(kCH, p.last - p.first);
#pragma unroll
    for (int c = 0; c < kCH; ++c)
        gram_block_offsets(min(p.first + c, total - 1), W, D8, DP, wstride, oJ, off_AM, g, t, p.oA[c], p.oB[c], p.oM[c]);
    return p;
}

__device__ __forceinline__ void gram_run(const GramPlan& p, int W, int D8, int DP, double* wbase, int wstride,
                                         int oJ, int off_AM) {
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    double acc[kCH][2];
    if (p.nch > 0) {
        dmma_chunk_ab(D8, p.nch, [&](int c, int k) { return wbase[p.oA[c] + k]; },
                      [&](int c, int k) { return wbase[p.oB[c] + k]; }, acc);
#pragma unroll
        for (int c = 0; c < kCH; ++c)
            if (c < p.nch) *reinterpret_cast<double2*>(wbase + p.oM[c]) = make_double2(acc[c][0], acc[c][1]);
    }
    for (int b0 = p.first + kCH; b0 < p.last; b0 += kCH) {       // more than kCH blocks per warp: generic path
        const int nch = min(kCH, p.last - b0);
        int oA[kCH], oB[kCH], oM[kCH];
#pragma unroll
        for (int c = 0; c < kCH; ++c)
            gram_block_offsets(min(b0 + c, p.last - 1), W, D8, DP, wstride, oJ, off_AM, g, t, oA[c], oB[c], oM[c]);
        dmma_chunk_ab(D8, nch, [&](int c, int k) { return wbase[oA[c] + k]; },
                      [&](int c, int k) { return wbase[oB[c] + k]; }, acc);
#pragma unroll
        for (int c = 0; c < kCH; ++c)
            if (c < nch) *reinterpret_cast<double2*>(wbase + oM[c]) = make_double2(acc[c][0], acc[c][1]);
    }
}

// Base-distribution end of the E_loc sweep (MODE_ELOC): at z = flow^-1(x) evaluate
// log p0 = 2 (log|det_up| + log|det_dn|) (base_dist.py:48-56) with gradient g0 and the
// Hessian contraction <H0, J J^T>, then assemble
//   log p = log p0 - Delta,  grad = J^T g0 - gDelta,  lap = <H0, JJ^T> + g0.L - lapDelta,
//   E_loc = -1/4 lap - 1/8 |grad|^2 + V(x)                       (VMC.py:48-55).
template <class Team = CtaTeam>
__device__ void eloc_finale(const FlowArgs& a, long long base, double* wbase,
                            const unsigned char* pair_i, const unsigned char* pair_j, Team team = Team(),
                            int team_warp0 = 0) {
    const int tid = team.tid(), T = team.size();
    const int n = a.n, D = a.D, DP = a.DP, W = a.W, NP = a.NP;
    const int oL = D, oG = 2 * D, oS = 3 * D, oJ = 3 * D + 2;
    auto S_in = [&](int w) { return wbase + (size_t)w * a.wstride; };
    auto scr = [&](int w) { return S_in(w) + a.off_sl; };
    const int slsz = slater_scratch_size(a.n_up, n - a.n_up);
    // scratch tail: g0[D], red[n*n + NP + 8]
    auto g0p = [&](int w) { return scr(w) + slsz; };
    auto red = [&](int w) { return scr(w) + slsz + D; };

    slater_team<true>(W, n, a.n_up,
        [&](int w) { return (const double*)S_in(w); }, scr,
        [&](int w) { long long b = base + w; int row = (a.walker_state && b < a.B) ? a.walker_state[b] : 0;
                     return a.orb + (size_t)row * n; }, team);

    // M = J J^T at the end point (upper block triangle), into the AM buffer
    {
        const GramPlan gp = gram_plan(W, (D + 7) & ~7, DP, a.wstride, oJ, a.off_AM, team_warp0, T >> 5);
        gram_run(gp, W, (D + 7) & ~7, DP, wbase, a.wstride, oJ, a.off_AM);
    }
    // g0 and the per-(i,j) Hessian contraction terms
    for (int s = 0; s < 2; ++s) {
        const SlBlk blk = slater_blk(s, n, a.n_up);
        const int ns = blk.ns;
        for (int g = tid; g < W * ns; g += T) {
            int w = g / ns, i = g - w * ns;
            const double* S = scr(w);
            g0p(w)[2 * (blk.i0 + i)] = 2.0 * S[blk.bx() + i * ns + i];
            g0p(w)[2 * (blk.i0 + i) + 1] = 2.0 * S[blk.by() + i * ns + i];
        }
    }
    team.sync();
    for (int g = tid; g < W * n * n; g += T) {
        int w = g / (n * n), rem = g - w * n * n;
        int I = rem / n, Jp = rem - I * n;
        const int sI = I >= a.n_up, sJ = Jp >= a.n_up;
        double t = 0.0;
        if (sI == sJ) {
            const SlBlk blk = slater_blk(sI, n, a.n_up);
            const int ns = blk.ns, i = I - blk.i0, j = Jp - blk.i0;
            const double* S = scr(w);
            const double* M = S_in(w) + a.off_AM;
            const double bxij = S[blk.bx() + i * ns + j], byij = S[blk.by() + i * ns + j];
            const double bxji = S[blk.bx() + j * ns + i], byji = S[blk.by() + j * ns + i];
            double m00, m01, m10, m11;       // M[(2I+a)][(2J+b)]
            if (I <= Jp) {
                m00 = M[(2 * I) * DP + 2 * Jp]; m01 = M[(2 * I) * DP + 2 * Jp + 1];
                m10 = M[(2 * I + 1) * DP + 2 * Jp]; m11 = M[(2 * I + 1) * DP + 2 * Jp + 1];
            } else {
                m00 = M[(2 * Jp) * DP + 2 * I]; m10 = M[(2 * Jp) * DP + 2 * I + 1];
                m01 = M[(2 * Jp + 1) * DP + 2 * I]; m11 = M[(2 * Jp + 1) * DP + 2 * I + 1];
            }
            t = -(bxij * bxji * m00 + bxij * byji * m01 + byij * bxji * m10 + byij * byji * m11);
            if (I == Jp) {
                const double* C = S + blk.cc() + 3 * i;
                t += C[0] * m00 + 2.0 * C[1] * m01 + C[2] * m11;
            }
        }
        red(w)[rem] = t;
    }
    // Coulomb terms at the original coordinates
    for (int g = tid; g < W * NP; g += T) {
        int w = g / NP, p = g - w * NP;
        const double* x0 = S_in(w) + a.off_x0;
        const int i = pair_i[p], j = pair_j[p];
        const double dx = x0[2 * i] - x0[2 * j], dy = x0[2 * i + 1] - x0[2 * j + 1];
        red(w)[n * n + p] = a.Z / sqrt(fma(dx, dx, dy * dy));
    }
    team.sync();
    // grad[c] = sum_r g0[r] J[r][c] - gDelta[c]   (kept in the KK area is dead: write to P3 slot 0..D)
    for (int g = tid; g < W * D; g += T) {
        int w = g / D, c = g - w * D;
        const double* J = S_in(w) + oJ + c;
        const double* g0 = g0p(w);
        double acc = -S_in(w)[oG + c];
        for (int r = 0; r < D; ++r) acc = fma(g0[r], J[r * DP], acc);
        red(w)[n * n + NP + 8 + c] = acc;
        long long b = base + w;
        if (b < a.B && a.grad) a.grad[b * D + c] = acc;
    }
    team.sync();
    for (int w = tid; w < W; w += T) {
        long long b = base + w;
        if (b >= a.B) continue;
        const double* Sw = S_in(w);
        const double* S = scr(w);
        double lap0 = 0.0, vc = 0.0, g2 = 0.0, gl = 0.0, vh = 0.0;
        const double* r = red(w);
        for (int k = 0; k < n * n; ++k) lap0 += r[k];
        for (int k = 0; k < NP; ++k) vc += r[n * n + k];
        for (int k = 0; k < D; ++k) {
            const double gk = r[n * n + NP + 8 + k];
            g2 = fma(gk, gk, g2);
            gl = fma(g0p(w)[k], Sw[oL + k], gl);
            const double xk = (Sw + a.off_x0)[k];
            vh = fma(xk, xk, vh);
        }
        const SlBlk bu = slater_blk(0, n, a.n_up), bd = slater_blk(1, n, a.n_up);
        double ld = 0.0;
        if (bu.ns) ld += S[bu.misc() + 2];
        if (bd.ns) ld += S[bd.misc() + 2];
        const double lp = 2.0 * ld - Sw[oS];
        const double lap = 2.0 * lap0 + gl - Sw[oS + 1];
        const double kin = -0.25 * lap - 0.125 * g2;
        const double pot = vc + (a.harmonic ? 0.5 * vh : 0.0);
        if (a.logp) a.logp[b] = lp;
        if (a.lap) a.lap[b] = lap;
        if (a.kin) a.kin[b] = kin;
        if (a.pot) a.pot[b] = pot;
        if (a.eloc) a.eloc[b] = kin + pot;
    }
    team.sync();
}

// One sweep of W walkers per CTA with the run-time geometry of FlowArgs (plan_flow).
template <int MODE>
__device__ __forceinline__ void flow_body(const FlowArgs& a) {
    extern __shared__ __align__(16) double smem[];
    // one extra "helper" warp (when the launch provides it) computes the Gram matrix while the
    // item warps are still in the MLP loop
    const int tid = threadIdx.x, T = blockDim.x;
    const int n = a.n, D = a.D, DP = a.DP, P = a.P, NP = a.NP, W = a.W, NSV = a.NSV;
    const int off_G = a.off_G, off_AM = a.off_AM, off_u = a.off_u, off_kLx = a.off_kLx, off_part = a.off_part, off_x0 = a.off_x0;
    const int D8 = (D + 7) & ~7;
    (void)DP; (void)D8; (void)off_AM; (void)off_u; (void)off_kLx; (void)off_x0;
    const bool has_mu = a.H_mu > 0;
    const int warp = tid >> 5, lane = tid & 31, nwarp = T >> 5;

    // ---- shared carve-up -------------------------------------------------------------
    double* tab = smem;                               // kTabDoubles
    double* coef_eta = tab + kTabDoubles;             // 6 * even(H_eta)
    double* coef_mu = coef_eta + 6 * ((a.H_eta + 3) & ~3);
    int cbase = kTabDoubles + 6 * (((a.H_eta + 3) & ~3) + ((a.H_mu + 3) & ~3));
    unsigned char* pair_i = reinterpret_cast<unsigned char*>(smem + cbase);   // NP each
    unsigned char* pair_j = pair_i + ((NP + 7) & ~7);
    double* wbase = smem + cbase + 2 * ((NP + 7) / 8);
    if ((wbase - smem) & 1) wbase += 1;
    const int wstride = a.wstride;

    fill_exp_table(tab);
    const double* tabl = tab + (tid & 15);
    load_mlp_coef(coef_eta, a.eta_w1, a.eta_b1, a.eta_w2, a.H_eta);
    if (has_mu) load_mlp_coef(coef_mu, a.mu_w1, a.mu_b1, a.mu_w2, a.H_mu);
    for (int p = tid; p < NP; p += T) {
        int i = 0, rem = p;
        while (rem >= n - 1 - i) { rem -= n - 1 - i; ++i; }
        pair_i[p] = (unsigned char)i;
        pair_j[p] = (unsigned char)(i + 1 + rem);
    }

    const double h = (a.tb - a.ta) / a.nsteps;
    const int NS = 4 * a.nsteps;
    constexpr int oY = 0;
    const int oL = D, oG = 2 * D, oS = 3 * D, oJ = 3 * D + 2;       // ELOC offsets
    const int oDelta = (MODE == MODE_ELOC) ? oS : D;
    const int NV = a.NV, NPAR = a.NPAR;
    const int oP3 = NSV, oP4 = NSV + NPAR, oPO = NSV + 2 * NPAR, oK = NSV + 3 * NPAR;
    // J part (D x D, unpadded) of RK block `which` (0: P3, 1: P4, 2: PO, 3: stage derivative) of walker w of this CTA
    double* const jglob = (MODE == MODE_ELOC) ? a.jpart : nullptr;
    auto jblock = [&](double* Sw, int w, int which) -> double* {
        return jglob ? jglob + (((size_t)blockIdx.x * W + w) * 4 + which) * (size_t)(D * D) : Sw + NSV + which * NPAR + NV;
    };

    GramPlan gplan;
    const int item_warps = (W * P + 31) >> 5;
    const int helper_warps = (MODE == MODE_ELOC) ? nwarp - item_warps : 0;
    if (MODE == MODE_ELOC) gplan = helper_warps > 0 ? gram_plan(W, D8, DP, wstride, oJ, off_AM, item_warps, helper_warps)
                                                    : gram_plan(W, D8, DP, wstride, oJ, off_AM);

    // item owned by this thread
    const int it_w = tid / P, it_p = tid - it_w * P;
    const bool it_valid = it_w < W;
    const bool it_pair = it_p < NP;
    double* const myS = wbase + (size_t)(it_valid ? it_w : 0) * wstride;
    int it_i = 0, it_j = 0;
    const RtHeader my_rt = rt_load_header(it_pair ? a.rt_eta : a.rt_mu);     // Taylor table of this thread's radial function

    for (long long base = (long long)blockIdx.x * W; base < a.B; base += (long long)gridDim.x * W) {
        __syncthreads();
        if (it_valid) {
            if (it_pair) { it_i = pair_i[it_p]; it_j = pair_j[it_p]; }
            else { it_i = it_p - NP; it_j = it_i; }
        }
        // ---- load walkers, initialise state -------------------------------------------
        for (int w = 0; w < W; ++w) {
            double* Sw = wbase + (size_t)w * wstride;
            const long long b = base + w;
            for (int e = tid; e < NSV; e += T) {
                double v = 0.0;
                if (e < D) {
                    // padding walkers get a harmless, well separated configuration
                    v = (b < a.B) ? a.x_in[b * D + e] : (double)(e >> 1) + 0.37 * (e & 1);
                    if (MODE == MODE_ELOC) (Sw + off_x0)[e] = v;
                } else if (MODE == MODE_ELOC && e >= oJ) {
                    const int r = (e - oJ) / DP, c = (e - oJ) - r * DP;
                    v = (r == c && r < D) ? 1.0 : 0.0;
                }
                Sw[e] = v;
            }
            if (MODE == MODE_ELOC)
                for (int e = tid; e < D8 * DP; e += T) (Sw + off_AM)[e] = 0.0;
        }
        __syncthreads();

#ifdef FF_PHASE_TIMING
        long long tacc[16] = {0}; long long tlast = clock64();
#endif
        for (int stage = 0; stage < NS; ++stage) {
            const int sub = stage & 3;
            FF_TICK(0);
            // ======== S0: per-item radial functions (+ Gram matrix for ELOC) ==============
            double rx = 0, ry = 0, ca = 0, cb = 0, ccq = 0, ceq = 0, cf = 0;
            if (it_valid) {
                const double* y = myS + oY;
                if (it_pair) { rx = y[2 * it_i] - y[2 * it_j]; ry = y[2 * it_i + 1] - y[2 * it_j + 1]; }
                else { rx = y[2 * it_i]; ry = y[2 * it_i + 1]; }
                const double d2 = fma(rx, rx, ry * ry);
                const double d = sqrt(d2);
                double f[4];
                constexpr int ORD = (MODE == MODE_V) ? 0 : (MODE == MODE_DIV) ? 1 : (MODE == MODE_STASH) ? 2 : 3;
                // one call for both item kinds: no divergence between pair and single lanes
                if (!radial_table_eval<ORD>(my_rt, d, f))
                    radial_mlp<ORD>(it_pair ? coef_eta : coef_mu, it_pair ? a.H_eta : a.H_mu, d, tabl, f);
                constexpr int GR = (MODE == MODE_ELOC) ? kGRec : 3;
                constexpr int GQ = (MODE == MODE_ELOC) ? 6 : 2;
                double* G = myS + off_G + it_p * GR;
                cf = f[0];
                G[0] = cf * rx;
                G[1] = cf * ry;
                if (MODE >= MODE_DIV) {
                    const double mult = it_pair ? 2.0 : 1.0;
                    G[GQ] = mult * fma(f[1], d, 2.0 * f[0]);                // q
                }
                if (MODE >= MODE_STASH && a.stash_c != nullptr) {
                    long long b = base + it_w;
                    if (b < a.B) {
                        double* sc = a.stash_c + ((b * NS + stage) * P + it_p) * 3;
                        sc[0] = f[0]; sc[1] = f[1]; sc[2] = f[2];
                    }
                }
                if (MODE == MODE_ELOC) {
                    const double mult = it_pair ? 2.0 : 1.0;
                    const double inv_d = 1.0 / d, inv_d2 = inv_d * inv_d;
                    ca = f[1] * inv_d;                                       // f'/d
                    cb = (f[2] - ca) * inv_d2;                               // (f'' - f'/d)/d^2
                    const double q1 = mult * fma(f[2], d, 3.0 * f[1]);       // q'
                    const double q2 = mult * fma(f[3], d, 4.0 * f[2]);       // q''
                    ccq = q1 * inv_d;
                    ceq = (q2 - ccq) * inv_d2;
                    G[2] = ccq * rx;
                    G[3] = ccq * ry;
                    G[8] = fma(ca * rx, rx, cf);
                    G[9] = ca * rx * ry;
                    G[10] = fma(ca * ry, ry, cf);
                }
            }
            if (MODE >= MODE_STASH && a.stash_y != nullptr) {
                for (int q = tid; q < W * D; q += T) {              // flat over (walker, element): small n keeps every lane busy
                    const int w = q / D, e = q - w * D;
                    const long long b = base + w;
                    if (b < a.B) a.stash_y[(b * NS + stage) * D + e] = (wbase + (size_t)w * wstride)[e];
                }
            }
            FF_TICK(1);
            if (MODE == MODE_ELOC) {
                gram_run(gplan, W, D8, DP, wbase, wstride, oJ, off_AM);
                FF_TICK(2);
                __syncthreads();
                FF_TICK(3);
                // ======== S1: second-derivative contractions per item ====================
                if (it_valid) {
                    const double* M = myS + off_AM;
                    const int i2 = 2 * it_i, j2 = 2 * it_j;
                    double w00, w01, w11;
                    if (it_pair) {
                        w00 = M[i2 * DP + i2] + M[j2 * DP + j2] - 2.0 * M[i2 * DP + j2];
                        w11 = M[(i2 + 1) * DP + i2 + 1] + M[(j2 + 1) * DP + j2 + 1] - 2.0 * M[(i2 + 1) * DP + j2 + 1];
                        w01 = M[i2 * DP + i2 + 1] + M[j2 * DP + j2 + 1] - M[i2 * DP + j2 + 1] - M[(i2 + 1) * DP + j2];
                    } else {
                        w00 = M[i2 * DP + i2]; w01 = M[i2 * DP + i2 + 1]; w11 = M[(i2 + 1) * DP + i2 + 1];
                    }
                    const double wrx = fma(w00, rx, w01 * ry), wry = fma(w01, rx, w11 * ry);
                    const double trw = w00 + w11, rwr = fma(rx, wrx, ry * wry);
                    double* G = myS + off_G + it_p * kGRec;
                    G[4] = fma(ca, fma(2.0, wrx, trw * rx), cb * rwr * rx);
                    G[5] = fma(ca, fma(2.0, wry, trw * ry), cb * rwr * ry);
                    G[7] = fma(ccq, trw, ceq * rwr);
                }
            }
            FF_TICK(4);
            __syncthreads();
            FF_TICK(5);
            // ======== S2: gather per particle, build Jacobian matrix ======================
            {
                constexpr int GRg = (MODE == MODE_ELOC) ? kGRec : 3;      // record stride
                constexpr int NC = (MODE == MODE_ELOC) ? kGRec : (MODE >= MODE_DIV ? 3 : 2);
                for (int gg = tid; gg < W * n * NC; gg += T) {           // flat over (walker, particle, quantity)
                    const int w = gg / (n * NC);
                    const int g = gg - w * (n * NC);
                    double* Sw = wbase + (size_t)w * wstride;
                    const double* G = Sw + off_G;
                    {
                        const int i = g / NC, cc = g - i * NC;
                        const int c = (MODE == MODE_ELOC) ? cc : (cc == 2 ? 6 : cc);   // logical quantity
                        const int gc = cc;                                             // column in the record
                        double accm = 0.0, accp = 0.0, accm2 = 0.0, accp2 = 0.0;
                        {   // pairs (j, i), j < i : stored with r = y_j - y_i
                            int idx = i - 1;                       // pair_index(0, i)
                            int j = 0;
                            for (; j + 2 <= i; j += 2) {
                                const int idx2 = idx + n - j - 2;
                                const double v0 = G[idx * GRg + gc], v1 = G[idx2 * GRg + gc];
                                accm += v0; accm2 += v1;
                                idx = idx2 + n - j - 3;
                            }
                            if (j < i) accm += G[idx * GRg + gc];
                        }
                        {   // pairs (i, j), j > i : consecutive
                            const double* Gi = G + pair_index(i, i + 1, n) * GRg + gc;
                            int j = i + 1;
                            for (; j + 4 <= n; j += 4) {
                                const double v0 = Gi[0], v1 = Gi[GRg], v2 = Gi[2 * GRg], v3 = Gi[3 * GRg];
                                accp += v0; accp2 += v1; accp += v2; accp2 += v3;
                                Gi += 4 * GRg;
                            }
                            for (; j < n; ++j) { accp += *Gi; Gi += GRg; }
                        }
                        accm += accm2; accp += accp2;
                        double acc = (c < 6) ? accp - accm : accp + accm;
                        if (c == 6 || c == 7) acc *= 0.5;
                        if (has_mu) acc += G[(NP + i) * GRg + gc];
                        if (c < 2) (Sw + oK)[oY + 2 * i + c] = acc;
                        else if (c < 4) (Sw + off_u)[2 * i + c - 2] = acc;
                        else if (c < 6) (Sw + off_kLx)[2 * i + c - 4] = acc;
                        else if (c < 8) (Sw + off_part)[(c - 6) * n + i] = acc;
                        else {
                            double* A = Sw + off_AM;
                            if (c == 8) A[(2 * i) * DP + 2 * i] = acc;
                            else if (c == 9) { A[(2 * i) * DP + 2 * i + 1] = acc; A[(2 * i + 1) * DP + 2 * i] = acc; }
                            else A[(2 * i + 1) * DP + 2 * i + 1] = acc;
                        }
                    }
                }
                if (MODE == MODE_ELOC && it_valid && it_pair) {
                    double* A = myS + off_AM;
                    const double a00 = -fma(ca * rx, rx, cf), a01 = -(ca * rx * ry), a11 = -fma(ca * ry, ry, cf);
                    const int i2 = 2 * it_i, j2 = 2 * it_j;
                    A[i2 * DP + j2] = a00; A[i2 * DP + j2 + 1] = a01;
                    A[(i2 + 1) * DP + j2] = a01; A[(i2 + 1) * DP + j2 + 1] = a11;
                    A[j2 * DP + i2] = a00; A[j2 * DP + i2 + 1] = a01;
                    A[(j2 + 1) * DP + i2] = a01; A[(j2 + 1) * DP + i2 + 1] = a11;
                }
            }
            FF_TICK(6);
            __syncthreads();
            FF_TICK(7);
            // ======== S3: derivative of the whole state ===================================
            if (MODE == MODE_ELOC) {
                // K.J = A J on the FP64 tensor cores: one warp task per block row (chunks of kCH
                // column blocks).  The two small products K.L = A L + kLx and K.gD = -(u^T J) run
                // as plain DFMA dot products on the last two warps, which have no row task at N=20.
                {
                    const int g = lane >> 2, t = lane & 3, NB = D8 >> 3;
                    const int nchunk = (NB + kCH - 1) / kCH;
                    const int tpw = NB * nchunk;
                    for (int task = warp; task < W * tpw; task += nwarp) {
                        const int w = task / tpw;
                        const int rem = task - w * tpw;
                        double* Sw = wbase + (size_t)w * wstride;
                        double acc[kCH][2];
                        const int rb = rem / nchunk, ch = rem - rb * nchunk;
                        const int cb0 = ch * kCH, nch = min(kCH, NB - cb0);
                        const double* Ap = Sw + off_AM + (8 * rb + g) * DP + t;      // A[row][k]
                        const double* Bp = Sw + oJ + t * DP + 8 * cb0 + g;             // J[k][col]
                        dmma_chunk(D8, nch, [&](int k) { return Ap[k]; },
                                   [&](int c, int k) { return Bp[k * DP + 8 * c]; }, acc);
                        // derivative block keeps J unpadded: [D][D]
                        double* K = jblock(Sw, w, 3) + (8 * rb + g) * D + 8 * cb0 + 2 * t;
                        if (8 * rb + g < D) {
#pragma unroll
                            for (int c = 0; c < kCH; ++c)
                                if (c < nch && 8 * (cb0 + c) + 2 * t < D)
                                    *reinterpret_cast<double2*>(K + 8 * c) = make_double2(acc[c][0], acc[c][1]);
                        }
                    }
                    const int vt = T - 1 - tid;                 // 0 .. 63 on the last two warps
                    if (vt < 64) {
                        for (int q = vt; q < W * 2 * D; q += 64) {
                            const int w = q / (2 * D), e = q - w * 2 * D;
                            double* Sw = wbase + (size_t)w * wstride;
                            double acc0 = 0.0, acc1 = 0.0;
                            if (e < D) {
                                const double* A = Sw + off_AM + e * DP;
                                const double* L = Sw + oL;
                                for (int k = 0; k < D; k += 2) {
                                    const double2 av = *reinterpret_cast<const double2*>(A + k);
                                    const double2 lv = *reinterpret_cast<const double2*>(L + k);
                                    acc0 = fma(av.x, lv.x, acc0); acc1 = fma(av.y, lv.y, acc1);
                                }
                                (Sw + oK)[oL + e] = acc0 + acc1 + (Sw + off_kLx)[e];
                            } else {
                                const int c = e - D;
                                const double* u = Sw + off_u;
                                const double* J = Sw + oJ + c;
                                for (int k = 0; k < D; k += 2) {
                                    acc0 = fma(u[k], J[k * DP], acc0);
                                    acc1 = fma(u[k + 1], J[(k + 1) * DP], acc1);
                                }
                                (Sw + oK)[oG + c] = -(acc0 + acc1);
                            }
                        }
                    }
                }
                FF_TICK(8);
                // scalar rates: one warp per walker, shuffle reductions
                for (int w = nwarp - 1 - warp; w < W && w >= 0; w += nwarp) {
                    double* Sw = wbase + (size_t)w * wstride;
                    const double* part = Sw + off_part;
                    const double* u = Sw + off_u; const double* L = Sw + oL;
                    double rho = 0.0, lp = 0.0;
                    for (int i = lane; i < n; i += 32) { rho += part[i]; lp += part[n + i]; }
                    for (int k = lane; k < D; k += 32) lp = fma(u[k], L[k], lp);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        rho += __shfl_xor_sync(0xffffffffu, rho, o);
                        lp += __shfl_xor_sync(0xffffffffu, lp, o);
                    }
                    if (lane == 0) { (Sw + oK)[oS] = -rho; (Sw + oK)[oS + 1] = -lp; }
                }
            } else if (MODE >= MODE_DIV) {
                for (int w = tid; w < W; w += T) {
                    double* Sw = wbase + (size_t)w * wstride;
                    const double* part = Sw + off_part;
                    double rho = 0.0;
                    for (int i = 0; i < n; ++i) rho += part[i];
                    (Sw + oK)[oDelta] = -rho;
                }
            }
            FF_TICK(9);
            __syncthreads();
            FF_TICK(10);
            // ======== S4: 3/8-rule RK4 bookkeeping (torchdiffeq rk4_alt_step_func) ========
            {
                // element e of the state block <-> element pe of the partial / derivative blocks
                auto upd = [&](double* s, double* p3, double* p4, double* po, const double* kk) {
                    const double k = *kk * h;
                    if (sub == 0) {
                        const double y0 = *s;
                        *p3 = fma(k, -1.0 / 3.0, y0); *p4 = y0 + k; *po = fma(k, 0.125, y0);
                        *s = fma(k, 1.0 / 3.0, y0);
                    } else if (sub == 1) {
                        *s = *p3 + k; *p4 -= k; *po = fma(k, 0.375, *po);
                    } else if (sub == 2) {
                        *s = *p4 + k; *po = fma(k, 0.375, *po);
                    } else {
                        *s = fma(k, 0.125, *po);
                    }
                };
                // flat over (walker, element): with many small walkers per CTA every lane stays busy
                for (int q = tid; q < W * NV; q += T) {
                    const int w = q / NV, e = q - w * NV;
                    double* Sw = wbase + (size_t)w * wstride;
                    upd(Sw + e, Sw + oP3 + e, Sw + oP4 + e, Sw + oPO + e, Sw + oK + e);
                }
                if (MODE == MODE_ELOC) {
                    // J: state rows have stride DP, partial rows stride D
                    const int hD = D >> 1;
                    auto updJ = [&](double* Sw, int w, int r, int c) {
                        double2* s2 = reinterpret_cast<double2*>(Sw + NV + r * DP + c);
                        const int pe = r * D + c;
                        double2* p3 = reinterpret_cast<double2*>(jblock(Sw, w, 0) + pe);
                        double2* p4 = reinterpret_cast<double2*>(jblock(Sw, w, 1) + pe);
                        double2* po = reinterpret_cast<double2*>(jblock(Sw, w, 2) + pe);
                        double2 k = *reinterpret_cast<const double2*>(jblock(Sw, w, 3) + pe);
                        k.x *= h; k.y *= h;
                        if (sub == 0) {
                            const double2 y0 = *s2;
                            *p3 = make_double2(fma(k.x, -1.0 / 3.0, y0.x), fma(k.y, -1.0 / 3.0, y0.y));
                            *p4 = make_double2(y0.x + k.x, y0.y + k.y);
                            *po = make_double2(fma(k.x, 0.125, y0.x), fma(k.y, 0.125, y0.y));
                            *s2 = make_double2(fma(k.x, 1.0 / 3.0, y0.x), fma(k.y, 1.0 / 3.0, y0.y));
                        } else if (sub == 1) {
                            const double2 a3 = *p3, a4 = *p4, ao = *po;
                            *s2 = make_double2(a3.x + k.x, a3.y + k.y);
                            *p4 = make_double2(a4.x - k.x, a4.y - k.y);
                            *po = make_double2(fma(k.x, 0.375, ao.x), fma(k.y, 0.375, ao.y));
                        } else if (sub == 2) {
                            const double2 a4 = *p4, ao = *po;
                            *s2 = make_double2(a4.x + k.x, a4.y + k.y);
                            *po = make_double2(fma(k.x, 0.375, ao.x), fma(k.y, 0.375, ao.y));
                        } else {
                            const double2 ao = *po;
                            *s2 = make_double2(fma(k.x, 0.125, ao.x), fma(k.y, 0.125, ao.y));
                        }
                    };
                    if (hD >= 16) {
                        // one (walker, row) per warp trip, two columns per lane (no integer division in the inner loop)
                        for (int wr = warp; wr < W * D; wr += nwarp) {
                            const int w = wr / D, r = wr - w * D;
                            double* Sw = wbase + (size_t)w * wstride;
                            for (int c2 = lane; c2 < hD; c2 += 32) updJ(Sw, w, r, 2 * c2);
                        }
                    } else {
                        // short rows (small n, many walkers per CTA): flat over (walker, row, column pair)
                        const int per = D * hD;
                        for (int q = tid; q < W * per; q += T) {
                            const int w = q / per, rc = q - w * per;
                            const int r = rc / hD, c2 = rc - r * hD;
                            updJ(wbase + (size_t)w * wstride, w, r, 2 * c2);
                        }
                    }
                }
            }
            FF_TICK(11);
            __syncthreads();
            FF_TICK(12);
        }   // stages
#ifdef FF_PHASE_TIMING
        if (MODE == MODE_ELOC && tid == 0) for (int k = 0; k < 16; ++k) atomicAdd(&g_phase_cycles[k], (unsigned long long)tacc[k]);
#endif

        // ---- outputs ----------------------------------------------------------------------
        for (int w = 0; w < W; ++w) {
            const long long b = base + w;
            const double* Sw = wbase + (size_t)w * wstride;
            if (b < a.B) {
                if (a.y_out) for (int e = tid; e < D; e += T) a.y_out[b * D + e] = Sw[e];
                if (MODE >= MODE_DIV && a.delta_out && tid == 0) a.delta_out[b] = Sw[oDelta];
            }
        }
        if (MODE == MODE_ELOC) eloc_finale(a, base, wbase, pair_i, pair_j);
    }
}

template <int MODE>
__global__ void __launch_bounds__(512, 1) flow_kernel(const FlowArgs a) { flow_body<MODE>(a); }

// Same body for CTAs of at most 256 threads, capped at 64 registers: four CTAs (32 warps) per SM
// keep the FP64 pipe fed across the per-stage barriers of the value / divergence sweeps.
template <int MODE>
__global__ void __launch_bounds__(256, 4) flow_kernel_small(const FlowArgs a) { flow_body<MODE>(a); }


}  // namespace ff
