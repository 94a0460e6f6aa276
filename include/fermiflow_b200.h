/* fermiflow_b200 -- C ABI of the B200-native FermiFlow VMC hot path.
 *
 * Every entry point takes plain pointers and sizes.  Unless a parameter name ends in
 * `_host`, pointers are DEVICE pointers to float64 (or int32 where stated), C-contiguous,
 * 16-byte aligned.  `stream` is a cudaStream_t passed as void* (NULL = default stream).
 * All functions return 0 on success, a negative value for an argument / capacity error
 * and a positive cudaError_t otherwise; ff_last_error() describes the last failure on
 * the calling thread.  Nothing here falls back to the CPU.
 *
 * Each function names the reference interface (file:line in buwantaiji/FermiFlow) it
 * replaces; INTEGRATION.md shows the Python-side binding.
 */
#ifndef FERMIFLOW_B200_H
#define FERMIFLOW_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* Backflow velocity field (src/equivariant_funs.py:4-102) with its two radial MLPs
 * (src/MLP.py:4-45, D_in = 1, one sigmoid hidden layer, scalar output, fc2 without bias)
 * and the ODE grid of the flow (src/flow.py:6-40 CNF(v, t_span); fixed-step 3/8-rule RK4
 * = torchdiffeq odeint(method="rk4") in place of the adaptive default). */
typedef struct ff_model {
    int n_up, n_dn;               /* particles per spin; coordinates are [n_up+n_dn][2]   */
    int H_eta, H_mu;              /* hidden units; H_mu = 0: no one-body backflow (mu=None) */
    const double *eta_w1, *eta_b1, *eta_w2;   /* fc1.weight[:,0], fc1.bias, fc2.weight[0,:] */
    const double *mu_w1, *mu_b1, *mu_w2;
    double t0, t1;                /* t_span                                                */
    int nsteps;                   /* RK4 steps across t_span                               */
} ff_model;

int ff_version(void);
const char* ff_last_error(void);

/* Kernel-variant switches for tests and A/B timing (no reference counterpart; the library never reads the
 * environment).  Process-wide, thread-safe; 0 restores the default.  Names: no_table, no_w_balance, no_rt_cache,
 * flow_warp_fill, flow_cta, flow_big, eloc_generic, slater_cta, metropolis_kernel (0 auto, 1 registers, 2 warp per
 * walker, 3 thread per walker), adjoint_cta, pgrad_direct, pgrad_tile, pgrad_fixed_range, adjoint_no_prefetch,
 * finale_cta, metropolis_no_split (INTEGRATION.md has the table).  Unknown name: -1. */
/* Number of CUDA kernels this library has launched in the process so far (bench.py reports the difference over its
 * timed region as "gpu_launches"). */
long long ff_launch_count(void);

int ff_set_option(const char* name, int value);
int ff_get_option(const char* name, int* value);

/* Backflow.forward / Backflow.divergence (equivariant_funs.py:80-102).
 * x [B][n][2] -> v [B][n][2] (nullable), div [B] (nullable). */
int ff_backflow(const ff_model* m, const double* x, long long B, double* v, double* div, void* stream);

/* CNF.generate (flow.py:42-50): x = flow_{t0->t1}(z).  reverse != 0 runs t1->t0. */
int ff_cnf_generate(const ff_model* m, const double* z, long long B, int reverse, double* x, void* stream);

/* CNF.delta_logp (flow.py:52-56): (z, delta_logp) = integral over t1->t0 of (v, -div v)
 * starting from (x, 0).  stash_y / stash_c (nullable, sizes from ff_stash_sizes) keep what
 * ff_logp_backward needs (the role of ctx.save_for_backward in NeuralODE/nnModule.py:73):
 * stash_y = the stage inputs (8 bytes x 2n per walker and RK stage), stash_c = the radial functions
 * (f, f', f'') per item.  stash_c is optional: without it ff_logp_backward recomputes them from the
 * stage inputs (16x less memory: 1.3 GB instead of 22 GB for 65536 walkers at n = 20, at the price of a
 * slower backward sweep: 45 ms instead of 16 ms at that size). */
int ff_cnf_delta_logp(const ff_model* m, const double* x, long long B, double* z, double* delta_logp,
                      double* stash_y, double* stash_c, void* stream);

/* number of float64 elements of the two stash arrays for B walkers */
int ff_stash_sizes(const ff_model* m, long long B, long long* n_stash_y, long long* n_stash_c);

/* LogAbsSlaterDet / LogAbsSlaterDetMultStates (slater.py:4-68, 70-156) for ONE spin block
 * of n particles: log|det phi_{orb[k]}(r_i)|, its gradient [B][n][2] (Jacobi's formula,
 * slater.py:40-60) and its Laplacian [B] (both nullable).  orb: int32 rows of n HO2D
 * orbital ids (orbitals.py:89 ordering); walker_state (int32 [B], nullable) selects the
 * row per walker, otherwise row 0 is used for every walker. */
int ff_slater_logabsdet(const double* x, long long B, int n, const int* orb, const int* walker_state,
                        double* logabsdet, double* grad, double* lap, void* stream);

/* FreeFermion.log_prob / log_prob_multstates (base_dist.py:48-56, 72-101):
 * 2 (log|det_up| + log|det_dn|), optional gradient. */
int ff_free_fermion_logp(const double* x, long long B, int n_up, int n_dn, const int* orb,
                         const int* walker_state, double* logp, double* grad, void* stream);

/* The same with the exact Laplacian (sum over all coordinates of d^2 log p0 / dx^2) from Jacobi's
 * formula -- what utils.py:44-65 y_grad_laplacian returns for f = FreeFermion.log_prob with
 * 1 + 2N autograd passes (BASELINE.json config "kernel microbench: batched log|det| + exact
 * Laplacian").  logp, grad, lap nullable. */
int ff_free_fermion_logp_lap(const double* x, long long B, int n_up, int n_dn, const int* orb,
                             const int* walker_state, double* logp, double* grad, double* lap, void* stream);

/* Double backward of LogAbsSlaterDet / LogAbsSlaterDetMultStates / FreeFermion.log_prob (slater.py:40-60 and
 * 120-156 assemble the gradient from differentiable torch ops precisely so that utils.py:44-65 y_grad_laplacian can
 * differentiate it again; reference tests/test_slater.py:65-127): hv = scale * Hessian(log|det Phi_up| +
 * log|det Phi_dn|) v per walker, v and hv [B][n_up+n_dn][2].  One spin block: n_dn = 0. */
int ff_slater_hvp(const double* x, long long B, int n_up, int n_dn, const int* orb, const int* walker_state,
                  double scale, const double* v, double* hv, void* stream);

/* FreeFermion.sample / sample_multstates (base_dist.py:58-70, 103-134): Metropolis chain of
 * `steps` whole-configuration moves x' = x + tau N(0,1), started from x ~ N(0,1).
 * Random numbers: Philox4x32-10 keyed by `seed` (counter = walker, step, particle), or,
 * when normals_/uniforms_ are non-null, read from x0 [B][n][2], normals [steps][B][n][2],
 * uniforms [steps][B] (parity tests).  Writes x [B][n][2]; accept_count [B] int32 nullable. */
int ff_metropolis(long long B, int n_up, int n_dn, const int* orb, const int* walker_state,
                  int steps, double tau, unsigned long long seed, long long walker_offset,
                  const double* x0, const double* normals, const double* uniforms,
                  double* x, int* accept_count, void* stream);

/* The E_loc sweep of GSVMC.forward / BetaVMC.forward (VMC.py:41-55, 124-145): for given x
 * returns z, delta_logp, log p(x), grad_x log p [B][n][2], laplacian_x log p, kinetic,
 * potential (Z sum 1/r_ij + harmonic/2 sum r^2; potentials.py) and E_loc, replacing
 * utils.py:44 y_grad_laplacian by one forward-mode sweep.  All outputs nullable. */
int ff_eloc(const ff_model* m, const double* x, long long B, const int* orb, const int* walker_state,
            double Z, int harmonic, double* z, double* delta_logp, double* logp, double* grad,
            double* lap, double* kinetic, double* potential, double* eloc,
            double* stash_y, double* stash_c, void* stream);

/* Backward of log p = log p0(z) - delta_logp through the flow (the adjoint solve of
 * NeuralODE/nnModule.py:78-103): given upstream gbar_z [B][n][2] and gbar_delta [B] it
 * returns grad_x [B][n][2] (nullable) and ACCUMULATES the parameter gradients into
 * g_eta_* / g_mu_* (same shapes as the parameters).  work: ff_backward_work_size doubles; stash_y and work 16-byte aligned.
 * stash_c may be null (see ff_cnf_delta_logp). */
int ff_logp_backward(const ff_model* m, long long B, const double* stash_y, const double* stash_c,
                     const double* gbar_z, const double* gbar_delta, double* grad_x,
                     double* g_eta_w1, double* g_eta_b1, double* g_eta_w2,
                     double* g_mu_w1, double* g_mu_b1, double* g_mu_w2,
                     double* work, void* stream);
int ff_backward_work_size(const ff_model* m, long long B, long long* n_work);

/* HO.V + CoulombPairPotential.V (potentials.py:13-14, 23-46). */
int ff_potential(const double* x, long long B, int n, double Z, int harmonic, double* V, void* stream);

/* Categorical(logits).sample + sort (VMC.py:94-97) as inverse-CDF on supplied uniforms:
 * state[b] = first s with cdf[s] >= u[b]; counts [S] int32 is the histogram that the
 * reference keeps as state_indices_collection.  cdf_work: S doubles. */
int ff_occupation_sample(const double* logits, int S, const double* uniforms, long long B,
                         int* state, int* counts, double* cdf_work, void* stream);

/* Histograms of sampled walkers for the one-body density and the pair correlations (no reference counterpart: the
 * reference reports energies only).  x [B][n_up+n_dn][2], particle i < n_up spin-up; 8-byte alignment suffices.
 * Four sections, each switched off by 0 bins:
 *   density     particles i on the square grid [-extent, extent)^2, n_xy x n_xy cells, channels up, down
 *   radial      |r_i| over [0, r_max), n_r bins, channels up, down
 *   separation  |r_i - r_j| of the pairs i < j over [0, r_max), n_r bins, channels up-up, down-down, up-down
 *   rotated     ordered pairs i != j in the frame rotated so that particle i lies on the +x axis,
 *               u = (x_i x_j + y_i y_j) / |r_i|, w = (x_i y_j - y_i x_j) / |r_i|, on [-extent, extent)^2 with
 *               n_rot x n_rot cells, channels same spin, opposite spin
 * Binning rule: s = nbins / (hi - lo) in double, bin k = floor((v - lo) * s) with every product and sum rounded
 * separately (no FMA); k < 0, k >= nbins, a non-finite v and, in the rotated section, |r_i| == 0 count in the
 * section's per-channel outside counter instead.
 * Layout of counts (n_counts = 2 n_xy^2 + 2 n_r + 3 n_r + 2 n_rot^2 + 9):
 *   [2][n_xy][n_xy] density (index [ch][ix][iy]), [2][n_r] radial, [3][n_r] separation, [2][n_rot][n_rot] rotated
 *   (index [ch][iu][iw]), then the 9 outside counters in the same order: density up, down, radial up, down,
 *   separation up-up, down-down, up-down, rotated same, opposite.
 * ACCUMULATES into counts (the caller zeroes them); the counts are exact integers, independent of the order of
 * execution.  B == 0 is a no-op.  -1 for bad particle numbers, B < 0, null pointers with B > 0, a non-positive extent
 * or r_max of an enabled section, negative bin counts, n_counts not equal to the layout size, or (B > 0) a section
 * whose bins do not fit in the shared memory of one block (a 128 x 128 density takes 128 KB and fits; sections that do
 * not fit together are counted by one launch each). */
typedef struct ff_obs_grid {
    double extent; int n_xy; int n_rot;     /* square grids over [-extent, extent)^2; 0 cells: section off */
    double r_max;  int n_r;                 /* radial and separation bins over [0, r_max); 0: off          */
} ff_obs_grid;
int ff_observables(const double* x, long long B, int n_up, int n_dn, const ff_obs_grid* g,
                   unsigned long long* counts, long long n_counts, void* stream);

/* Raw FP64 FMA throughput of the device (roofline denominator): runs `iters` dependent
 * DFMA chains on every SM and returns the achieved FLOP/s in *flops_host. */
int ff_fp64_peak(int iters, double* flops_host, void* stream);
/* Same for the FP64 tensor-core path (mma.sync m8n8k4 f64, "DMMA"). */
int ff_fp64_mma_peak(int iters, double* flops_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif
