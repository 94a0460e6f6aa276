// Certified piecewise-Taylor tables of the radial backflow functions eta(d), mu(d).
//
// The velocity field only ever evaluates f(d) = sum_h w2_h sigmoid(w1_h d + b1_h) (MLP.py:30-45 with
// D_in = 1) and its d-derivatives at scalar distances.  f is analytic with its nearest singularity at
// imaginary distance pi / max|w1| from the real axis, so a degree-11 Taylor polynomial around nodes
// spaced delta = 0.15 / max|w1| reproduces f, f', f'', f''' to ~1e-15 .. 3e-14 relative (the rounding
// level of the direct sum): 44 FMAs per item instead of ~25 FP64 instructions per item AND hidden unit.
//
//   build    : every sweep launch rebuilds the tables from the current parameters (one tiny kernel):
//              c[k][m] = sum_h w2_h w1_h^m sigma^(m)(w1_h d_k + b1_h) / m!,  sigma^(m) = P_m(sigma) with the
//              integer polynomials P_0 = s, P_{m+1} = P_m' s (1 - s)
//   certify  : at every interval mid-point the expansions around the two neighbouring nodes must agree
//              (f and f''' within 1e-12 of their scale), otherwise the table is marked invalid
//   evaluate : k = rint(d / delta); anything outside the table, or an invalid table, falls back to the
//              direct evaluation (radial_mlp*), lane by lane.
// The parameter gradient (pgrad_kernel) needs the individual hidden units and keeps the direct sigmoids.
#pragma once
#include "ff_common.cuh"

namespace ff {

constexpr int kRtDeg = 11;                 // Taylor degree
constexpr int kRtCoef = kRtDeg + 1;        // doubles per node (96 bytes)
constexpr int kRtMaxNodes = 8192;          // capacity per function
constexpr int kRtHeader = 8;               // doubles: inv_delta, delta, n_nodes, valid, max|w1|, check, -, -
constexpr double kRtSpacing = 0.15;        // delta * max|w1|
constexpr double kRtDmax = 24.0;           // tabulated range of d
constexpr double kRtMaxDelta = 0.125;
__host__ __device__ constexpr size_t radial_table_doubles() { return kRtHeader + (size_t)kRtMaxNodes * kRtCoef; }

// P_m(s), m = 0..11, lowest power first; P_m starts at c_sigpoly_off[m] and has m + 2 coefficients
static __constant__ double c_sigpoly[90] = {
    0.0, 1.0, 0.0, 1.0, -1.0, 0.0, 1.0, -3.0, 2.0, 0.0, 1.0, -7.0, 12.0, -6.0, 0.0, 1.0, -15.0, 50.0, -60.0,
    24.0, 0.0, 1.0, -31.0, 180.0, -390.0, 360.0, -120.0, 0.0, 1.0, -63.0, 602.0, -2100.0, 3360.0, -2520.0,
    720.0, 0.0, 1.0, -127.0, 1932.0, -10206.0, 25200.0, -31920.0, 20160.0, -5040.0, 0.0, 1.0, -255.0, 6050.0,
    -46620.0, 166824.0, -317520.0, 332640.0, -181440.0, 40320.0, 0.0, 1.0, -511.0, 18660.0, -204630.0, 1020600.0,
    -2739240.0, 4233600.0, -3780000.0, 1814400.0, -362880.0, 0.0, 1.0, -1023.0, 57002.0, -874500.0, 5921520.0,
    -21538440.0, 46070640.0, -59875200.0, 46569600.0, -19958400.0, 3628800.0, 0.0, 1.0, -2047.0, 173052.0,
    -3669006.0, 33105600.0, -158838240.0, 451725120.0, -801496080.0, 898128000.0, -618710400.0, 239500800.0,
    -39916800.0};
static __constant__ int c_sigpoly_off[12] = {0, 2, 5, 9, 14, 20, 27, 35, 44, 54, 65, 77};
static __constant__ double c_inv_fact[12] = {1.0, 1.0, 0.5, 0.16666666666666666, 0.041666666666666664, 0.008333333333333333,
                                      0.001388888888888889, 0.0001984126984126984, 2.48015873015873e-05,
                                      2.7557319223985893e-06, 2.755731922398589e-07, 2.505210838544172e-08};

// grid: enough CTAs of 128 threads to cover kRtMaxNodes; tables[0] = eta, tables[1] = mu (H_mu may be 0)
struct RadialBuildArgs {
    const double *w1[2], *b1[2], *w2[2];
    int H[2];
    double* table[2];
};

#ifdef FF_RADIAL_TABLE_KERNELS      // the two kernels are instantiated by exactly one translation unit (capi.cu)
__global__ void __launch_bounds__(128) radial_table_build_kernel(const RadialBuildArgs a) {
    __shared__ double tab[kTabDoubles];
    __shared__ double red[128];
    fill_exp_table(tab);
    const int f = blockIdx.y;
    const int H = a.H[f];
    double* T = a.table[f];
    if (H <= 0 || T == nullptr) return;
    // max |w1| (every CTA recomputes it: a few dozen numbers)
    double wm = 0.0;
    for (int h = threadIdx.x; h < H; h += blockDim.x) wm = fmax(wm, fabs(a.w1[f][h]));
    red[threadIdx.x] = wm;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] = fmax(red[threadIdx.x], red[threadIdx.x + o]); __syncthreads(); }
    wm = red[0];
    const double delta = fmin(kRtMaxDelta, kRtSpacing / fmax(wm, 1e-300));
    const double nn = ceil(kRtDmax / delta) + 2.0;
    const bool fits = nn <= (double)kRtMaxNodes && isfinite(wm);
    const int n_nodes = fits ? (int)nn : 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        T[0] = 1.0 / delta; T[1] = delta; T[2] = (double)n_nodes; T[3] = fits ? 1.0 : 0.0; T[4] = wm; T[5] = 0.0;
    }
    const double* tabl = tab + (threadIdx.x & 15);
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_nodes; k += gridDim.x * blockDim.x) {
        const double d = k * delta;
        double c[kRtCoef];
#pragma unroll
        for (int m = 0; m < kRtCoef; ++m) c[m] = 0.0;
        for (int h = 0; h < H; ++h) {
            const double w = a.w1[f][h];
            const double s = sigmoid_fast(fma(w, d, a.b1[f][h]), tabl);
            double wp = a.w2[f][h];                       // w2 w1^m
#pragma unroll
            for (int m = 0; m < kRtCoef; ++m) {
                const double* p = c_sigpoly + c_sigpoly_off[m];
                double v = p[m + 1];
#pragma unroll
                for (int q = m; q >= 0; --q) v = fma(v, s, p[q]);
                c[m] = fma(wp * c_inv_fact[m], v, c[m]);
                wp *= w;
            }
        }
        double* o = T + kRtHeader + (size_t)k * kRtCoef;
#pragma unroll
        for (int m = 0; m < kRtCoef; ++m) o[m] = c[m];
    }
}

#endif

// The first ORD + 1 of f, f', f'', f''' of the expansion with coefficients c at offset t: Horner in four running sums.
// The sums of the derivatives start at zero, so their first steps are copies (fma(0, t, p) = p: 6 of the 44 instructions
// at ORD 3, the same values bit for bit).  The node spacing (|t| <= 0.075 / max|w1|) is set by the third derivative: the
// relative size of the term of degree m is 0.0239^m in f and m 0.0239^(m-1) in f', so the value-only sweeps stop at
// degree kRtDeg - 2 (first dropped term 6e-17 of the scale of f) and the value + derivative sweeps at kRtDeg - 1
// (7e-16 of the scale of f'); their top coefficients are never loaded.
template <int ORD>
__device__ __forceinline__ void radial_horner(const double (&c)[kRtCoef], double t, double (&f)[4]) {
    constexpr int TOP = kRtDeg - (ORD == 0 ? 2 : ORD == 1 ? 1 : 0);
    double p0 = c[TOP], p1 = 0.0, p2 = 0.0, p3 = 0.0;
#pragma unroll
    for (int m = TOP - 1; m >= 0; --m) {
        const int it = TOP - 1 - m;
        if (ORD >= 3) p3 = it >= 3 ? fma(p3, t, p2) : p2;
        if (ORD >= 2) p2 = it >= 2 ? fma(p2, t, p1) : p1;
        if (ORD >= 1) p1 = it >= 1 ? fma(p1, t, p0) : p0;
        p0 = fma(p0, t, c[m]);
    }
    f[0] = p0; f[1] = p1; f[2] = 2.0 * p2; f[3] = 6.0 * p3;
}

// f, f', f'', f''' of the expansion around node k at offset t
__device__ __forceinline__ void radial_taylor(const double* __restrict__ c, double t, double (&f)[4]) {
    double p0 = c[kRtDeg], p1 = 0.0, p2 = 0.0, p3 = 0.0;
#pragma unroll
    for (int m = kRtDeg - 1; m >= 0; --m) {
        p3 = fma(p3, t, p2); p2 = fma(p2, t, p1); p1 = fma(p1, t, p0); p0 = fma(p0, t, c[m]);
    }
    f[0] = p0; f[1] = p1; f[2] = 2.0 * p2; f[3] = 6.0 * p3;
}

// Certification: neighbouring expansions must agree at the interval mid-points.
#ifdef FF_RADIAL_TABLE_KERNELS
__global__ void __launch_bounds__(128) radial_table_check_kernel(double* T0, double* T1) {
    double* T = blockIdx.y ? T1 : T0;
    if (T == nullptr) return;
    const int n_nodes = (int)T[2];
    if (n_nodes < 2) return;
    const double delta = T[1];
    __shared__ double rs[128], re[128];
    double scale0 = 0.0, scale3 = 0.0, err0 = 0.0, err3 = 0.0;
    for (int k = threadIdx.x; k < n_nodes - 1; k += blockDim.x) {
        double fa[4], fb[4];
        radial_taylor(T + kRtHeader + (size_t)k * kRtCoef, 0.5 * delta, fa);
        radial_taylor(T + kRtHeader + (size_t)(k + 1) * kRtCoef, -0.5 * delta, fb);
        scale0 = fmax(scale0, fabs(fa[0])); scale3 = fmax(scale3, fabs(fa[3]));
        err0 = fmax(err0, fabs(fa[0] - fb[0])); err3 = fmax(err3, fabs(fa[3] - fb[3]));
    }
    // reduce the four numbers (two passes through shared memory)
    auto block_max = [&](double v) {
        rs[threadIdx.x] = v; __syncthreads();
        for (int o = 64; o > 0; o >>= 1) { if (threadIdx.x < o) rs[threadIdx.x] = fmax(rs[threadIdx.x], rs[threadIdx.x + o]); __syncthreads(); }
        const double r = rs[0]; __syncthreads(); return r;
    };
    (void)re;
    scale0 = block_max(scale0); scale3 = block_max(scale3); err0 = block_max(err0); err3 = block_max(err3);
    if (threadIdx.x == 0) {
        const bool ok = err0 <= 1e-12 * scale0 + 1e-300 && err3 <= 1e-11 * scale3 + 1e-300 && isfinite(err0) && isfinite(err3);
        T[5] = fmax(err0 / fmax(scale0, 1e-300), err3 / fmax(scale3, 1e-300));
        if (!ok) T[3] = 0.0;
    }
}

#endif

// Table header in registers (loop invariant of a sweep: load it once per thread).
struct RtHeader {
    double inv_delta, delta;
    const double* coef;        // nullptr: no usable table -> direct evaluation
    int n_nodes;
};
__device__ __forceinline__ RtHeader rt_load_header(const double* __restrict__ T) {
    RtHeader h;
    h.inv_delta = 0.0; h.delta = 0.0; h.coef = nullptr; h.n_nodes = 0;
    if (T != nullptr && __ldg(T + 3) != 0.0) {
        h.inv_delta = __ldg(T); h.delta = __ldg(T + 1); h.n_nodes = (int)__ldg(T + 2); h.coef = T + kRtHeader;
    }
    return h;
}

// Table look-up.  Returns false when d is outside the table or the table is invalid / absent.
template <int ORD>
__device__ __forceinline__ bool radial_table_eval(const RtHeader& T, double d, double (&f)[4]) {
    const double kf = rint(d * T.inv_delta);
    if (T.coef == nullptr || !(kf < (double)T.n_nodes) || !(kf >= 0.0)) return false;
    const double t = fma(-kf, T.delta, d);
    const double2* c2 = reinterpret_cast<const double2*>(T.coef + (size_t)(int)kf * kRtCoef);
    double c[kRtCoef];
#pragma unroll
    for (int q = 0; q < kRtCoef / 2; ++q) { const double2 v = __ldg(c2 + q); c[2 * q] = v.x; c[2 * q + 1] = v.y; }
    radial_horner<ORD>(c, t, f);
    return true;
}
// The same with the first `ncache` nodes of the table mirrored in shared memory, COEFFICIENT-MAJOR
// (cache[q * ncache + k]): lanes that look up different nodes read
// neighbouring words of one coefficient row instead of rows 96 bytes apart (4 bank groups) -- for kernels whose lanes
// all look up at once (one warp per walker).
template <int ORD>
__device__ __forceinline__ bool radial_table_eval_cached_t(const RtHeader& T, const double* cache, int ncache, double d, double (&f)[4]) {
    const double kf = rint(d * T.inv_delta);
    if (T.coef == nullptr || !(kf < (double)T.n_nodes) || !(kf >= 0.0)) return false;
    const double t = fma(-kf, T.delta, d);
    const int k = (int)kf;
    double c[kRtCoef];
    if (k < ncache) {
#pragma unroll
        for (int q = 0; q < kRtCoef; ++q) c[q] = cache[q * ncache + k];
    } else {
        const double2* c2 = reinterpret_cast<const double2*>(T.coef + (size_t)k * kRtCoef);
#pragma unroll
        for (int q = 0; q < kRtCoef / 2; ++q) { const double2 v = __ldg(c2 + q); c[2 * q] = v.x; c[2 * q + 1] = v.y; }
    }
    radial_horner<ORD>(c, t, f);
    return true;
}
template <int ORD>
__device__ __forceinline__ bool radial_table_eval(const double* __restrict__ T, double d, double (&f)[4]) {
    return radial_table_eval<ORD>(rt_load_header(T), d, f);
}

}  // namespace ff
