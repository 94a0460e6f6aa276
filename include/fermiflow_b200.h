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

/* Kernel-path switches: each forces a path the library also picks by itself for some inputs, so that tests can
 * compare it with the default one (no reference counterpart; the library never reads the environment).  Process-wide,
 * thread-safe; 0 restores the default.  Names: no_table, flow_cta, eloc_generic, slater_cta, metropolis_kernel (0 auto,
 * 1 registers, 2 warp per walker, 3 thread per walker), adjoint_cta, pgrad_direct (INTEGRATION.md has the table).
 * Unknown name: -1. */
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

/* Signed wave-function ratios of one-particle moves (no reference counterpart; the off-diagonal observables below need
 * the wave function with its sign at configurations that were not sampled):
 *   psi(x) = sign(det Phi_up(z) det Phi_dn(z)) exp(log p(x) / 2),   z = flow^-1(x)
 * (the flow's Jacobian determinant is positive, so the sign comes from the Slater determinants alone).  A record is one
 * walker b, one particle i = particle[b][m] (int32 [B][M]) and one displacement s = disp[b][m] ([B][M][2]); its ratio is
 *   ratio[b][m] = psi(x_b with r_i -> r_i + s) / psi(x_b).
 * orb and walker_state as in ff_eloc (walker_state nullable: row 0 for every walker).  The call evaluates B (M + 1)
 * configurations with the flow sweep of ff_cnf_delta_logp and the Slater kernels; slot 0 of each walker is x itself, so
 * a record with s = 0 gives 1 to rounding.  A particle index outside [0, n) gives a NaN ratio for that record (nothing
 * synchronises the host to check it).  work: ff_wavefunction_ratio_work_size doubles, 8-byte alignment suffices for
 * every buffer.  -1 for bad particle numbers (check as ff_cnf_delta_logp, at most 36 per spin), B or M < 1 and null
 * buffers. */
int ff_wavefunction_ratio_work_size(const ff_model* m, long long B, int M, long long* n_work);
int ff_wavefunction_ratio(const ff_model* m, const double* x, long long B, const int* orb, const int* walker_state,
                          int M, const int* particle /* int32 [B][M] */, const double* disp /* [B][M][2] */,
                          double* ratio /* [B][M] */, double* work, void* stream);

/* Momentum distribution and one-body coherence from R records (ratio [R], particle int32 [R], disp [R][2], for example
 * the B M records of ff_wavefunction_ratio).  A record's channel is c = (particle >= n_up).  Three sections, each
 * switched off by 0 bins:
 *   momentum  sum of ratio cos(k.s) at the n_k x n_k cell centres k = (kx_a, ky_b) of [-k_max, k_max)^2,
 *             kx_a = -k_max + (a + 1/2) 2 k_max / n_k
 *   radial    sum of ratio J0(k_j |s|) at k_j = (j + 1/2) k_max / n_kr (the direction average of cos(k.s))
 *   coherence sum of ratio and number of records per |s| bin over [0, s_max): bin floor(|s| n_s / s_max), |s| with every
 *             product and sum rounded separately; records with |s| >= s_max are in no bin
 * With particles drawn uniformly from all n and s uniformly in the disk |s| < s_max, M records per walker and W walkers,
 *   n_c(k) ~= n s_max^2 / (4 pi M W) sum over the records of channel c of ratio cos(k.s)
 * (normalised to the integral of n_c(k) d^2k = n_c), and g_c(|s|) = sum of ratio / records in the bin of |s|.
 * Layout of sums (n_sums = 2 n_k^2 + 2 n_kr + 4 n_s + 2):
 *   [2][n_k][n_k] sum ratio cos(k.s) (index [c][a][b]), [2][n_kr] sum ratio J0(k|s|), [2][n_s] sum ratio,
 *   [2][n_s] records (doubles, exact below 2^53), [2] records per channel.
 * ACCUMULATES into sums (the caller zeroes them).  Fixed summation order without floating-point atomics: two calls on
 * the same inputs give bit-identical sums.  A non-finite ratio propagates into the sums of its channel.  Scratch comes
 * from the stream-ordered allocator.  -1 for n_up < 0, R < 1, null pointers, a non-positive or non-finite k_max / s_max
 * of an enabled section, negative bin counts, n_sums not equal to the layout size, or a grid whose per-record tables
 * (4 n_k + n_kr + 3 doubles) do not fit in the shared memory of one block. */
typedef struct ff_mom_grid {
    double k_max; int n_k;    /* n_k x n_k cell centres of [-k_max, k_max)^2; 0: off                  */
    int n_kr;                 /* radial points k_j = (j + 1/2) k_max / n_kr (J0 average); 0: off       */
    double s_max; int n_s;    /* |s| bins over [0, s_max) for g(s): ratio sums and record counts; 0: off */
} ff_mom_grid;
int ff_momentum_accumulate(const double* ratio, const int* particle, const double* disp, long long R, int n_up,
                           const ff_mom_grid* g, double* sums, long long n_sums, void* stream);

/* One-body density matrix in the first K HO2D orbitals phi_0 ... phi_{K-1} (orbitals.py:89 order, shells 0 ... 7,
 * phi_a(r) = pi^-1/2 exp(-r^2/2) h_nx(x) h_ny(y)), per spin channel c:
 *   D^c_ab = integral of phi_a(r) rho1_c(r, r') phi_b(r') dr dr'.
 * Records r = b M + m as in ff_wavefunction_ratio: walker b of x [B][n_up+n_dn][2], particle i = particle[b][m]
 * (int32 [B][M]), displacement disp[b][m] ([B][M][2]) and weight w[b][m] ([B][M]).  The moved position is
 * r' = r_i + disp with one rounded add per coordinate, the position ff_wavefunction_ratio moves the particle to.  A
 * record's channel is c = (i >= n_up).  With particles drawn uniformly from all n, r' drawn from a density q(r') and
 * w = ratio / q(r'), ratio = psi(x with r_i -> r') / psi(x) of ff_wavefunction_ratio,
 *   D^c_ab ~= n / (M W) sum over the records of channel c of 1/2 [phi_a(r_i) phi_b(r') + phi_b(r_i) phi_a(r')] w
 * over W walkers; the kernel knows nothing about q and sums whatever w it is given.  Layout of sums
 * (n_sums = 2 K^2 + 3):
 *   [2][K][K] the symmetrised sums above (index [c][a][b], both triangles written, so the matrices are exactly
 *   symmetric), [2] records per channel, [1] skipped records
 * (counts as doubles, exact below 2^53).  A record whose particle index lies outside [0, n) is skipped: neither x nor
 * w is read for it (nothing synchronises the host to check the indices).  ACCUMULATES into sums (the caller zeroes
 * them).  Fixed summation order without floating-point atomics: two calls on the same inputs give bit-identical sums.
 * A non-finite w propagates into the sums of its channel.  Scratch comes from the stream-ordered allocator; 8-byte
 * alignment suffices for every buffer.  -1 for bad particle numbers (n_up, n_dn >= 0, at most 36 each, n >= 1), B or
 * M < 1, K = n_orb outside [1, 36], n_sums not equal to the layout size, null buffers, and a tile of records whose
 * tables (32 (2 K + 37) doubles) do not fit in the shared memory of one block. */
int ff_density_matrix_accumulate(const double* x, long long B, int n_up, int n_dn, int M,
                                 const int* particle /* int32 [B][M] */, const double* disp /* [B][M][2] */,
                                 const double* w /* [B][M] */, int n_orb, double* sums, long long n_sums, void* stream);

/* Replica swap ratios of spatial regions, for the second Renyi entropy (no reference counterpart):
 *   exp(-S2(A)) = Tr rho_A^2 = < psi(x') psi(y') / (psi(x) psi(y)) >,   x, y independent draws from rho,
 * with psi(x) = sign(det Phi_up(z) det Phi_dn(z)) exp(log p(x) / 2) as in ff_wavefunction_ratio.  Pair p is the two
 * walkers x = x_{pairs[p][0]} and y = x_{pairs[p][1]} (pairs int32 [P][2]; the caller chooses the pairing, and the
 * pairs should be independent: ff_occupation_sample returns sorted states, so neighbouring walkers of BetaVMC are not).
 * Regions (ff_swap_regions, all of one kind, 1 <= Q <= 32): kind 0 the disks |r| < a_q about the trap centre, decided
 * as x*x + y*y < a_q*a_q; kind 1 the half-planes x < a_q; every product and sum is rounded separately (no FMA).
 * For region q, x' is x with its particles inside A_q replaced by those of y, slot by slot within each spin block: the
 * k-th A-particle of x, in increasing particle index, takes the position of the k-th A-particle of y; y' is the
 * reverse.  Another pairing of the A-particles permutes x' and y' by pi and pi^-1, so the product of the two signs
 * does not change.  Each configuration is evaluated with the occupation row of its own walker (orb and walker_state as
 * in ff_eloc; walker_state nullable: row 0 for every walker), so for BetaVMC the records estimate Tr rho_A^2 of the
 * mixed state.  Outputs:
 *   sector[p][s][q]  n_A_up (n_dn + 1) + n_A_dn of side s (int32 [P][2][Q])
 *   ratio[p][q]      the pair ratio; exactly 0 when the two sides' sectors differ (the swapped configurations do not
 *                    exist), exactly 1 when region q holds no particle of either side (x' = x, y' = y)
 * A walker index outside [0, B) gives a NaN ratio and sector -1 on both sides for every region of that pair (nothing
 * synchronises the host to check it, and nothing is read out of bounds).  The call evaluates 2 P (Q + 1)
 * configurations with the flow sweep of ff_cnf_delta_logp and the SIGN Slater kernels.  work:
 * ff_swap_ratio_work_size doubles, 8-byte alignment suffices for every buffer.  -1 for bad particle numbers (check as
 * ff_cnf_delta_logp, at most 36 per spin), B or P < 1, null regions, Q outside [1, 32], a kind other than 0 or 1, a
 * null or non-finite a_q, a negative radius, and null buffers. */
typedef struct ff_swap_regions {
    int kind;                 /* 0: disks |r| < a_q, 1: half-planes x < a_q  */
    int Q;                    /* number of regions, 1 ... 32                 */
    const double* a;          /* HOST [Q]: radii (>= 0) or half-plane edges  */
} ff_swap_regions;
int ff_swap_ratio_work_size(const ff_model* m, long long P, int Q, long long* n_work);
int ff_swap_ratio(const ff_model* m, const double* x, long long B, const int* orb, const int* walker_state,
                  long long P, const int* pairs /* int32 [P][2] */, const ff_swap_regions* reg,
                  double* ratio /* [P][Q] */, int* sector /* int32 [P][2][Q] */, double* work, void* stream);

/* Sector-resolved sums of P Q swap records (ratio [P][Q], sector int32 [P][2][Q], as ff_swap_ratio writes them), with
 * n_sec = (n_up + 1)(n_dn + 1) sectors k = a (n_dn + 1) + b.  A record (p, q) whose two sectors both lie in
 * [0, n_sec) counts both replicas in their sectors, and when the sectors are equal it is a matched pair of that
 * sector and adds its ratio; any other record is skipped.  Layout of sums (n_sums = 3 Q n_sec + Q + 1):
 *   [Q][n_sec] sum of the ratios of the matched pairs,   [Q][n_sec] replicas (both sides counted),
 *   [Q][n_sec] matched pairs,   [Q] skipped records,   [1] pairs P
 * (counts as doubles, exact below 2^53).  With W pairs in all: Tr rho_A^2 ~= sum over the sectors of the ratio sums / W,
 * P(a, b) ~= replicas / (2 W), Tr rho_{A,ab}^2 ~= ratio sum of (a, b) / W and S2(a, b) = -ln(Tr rho_ab^2 / P(a, b)^2).
 * ACCUMULATES into sums (the caller zeroes them).  Fixed summation order without floating-point atomics: two calls on
 * the same inputs give bit-identical sums.  A non-finite ratio of a matched record propagates into its cell.  Scratch
 * comes from the stream-ordered allocator.  -1 for bad particle numbers (n_up, n_dn >= 0, at most 36 each, n >= 1),
 * P < 1, Q outside [1, 32], n_sums not equal to the layout size, and null buffers. */
int ff_swap_accumulate(const double* ratio, const int* sector, long long P, int Q, int n_up, int n_dn,
                       double* sums, long long n_sums, void* stream);

/* Raw FP64 FMA throughput of the device (roofline denominator): runs `iters` dependent
 * DFMA chains on every SM and returns the achieved FLOP/s in *flops_host. */
int ff_fp64_peak(int iters, double* flops_host, void* stream);
/* Same for the FP64 tensor-core path (mma.sync m8n8k4 f64, "DMMA"). */
int ff_fp64_mma_peak(int iters, double* flops_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif
