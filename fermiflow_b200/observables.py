"""Spin-resolved one-body density and pair correlations of sampled walkers (C ABI ff_observables), the momentum
distribution and one-body coherence from signed wave-function ratios (C ABI ff_wavefunction_ratio,
ff_momentum_accumulate), the second Rényi entropy of spatial regions from replica swap ratios (C ABI ff_swap_ratio,
ff_swap_accumulate), and the one-body density matrix in the oscillator basis with its natural-orbital occupations
(C ABI ff_wavefunction_ratio, ff_density_matrix_accumulate).

    est = DensityEstimator(n_up, n_dn, extent=6.0)
    with torch.no_grad():
        for _ in range(16):
            _, x = model.sample((65536,))
            est.accumulate(x)
    est.allreduce()
    est.save("density.npz")

The histograms are accumulated on the device; accumulate() never waits for the GPU.  Each call is one batch of
independent walkers, and the standard errors are batch means over calls: `model.sample` starts fresh Markov chains at
every call, so the batches are independent.  The estimates are meant for fixed parameters, for example after training;
walkers drawn while the parameters change average over the parameters too.
"""
import ctypes as C
import math

import numpy as np
import torch
import torch.distributed as dist

from . import _lib as L
from .orbitals import HO2D

# sections of the count vector (include/fermiflow_b200.h ff_observables): name, channels, square grid
_SECTIONS = (("density", 2, True), ("radial", 2, False), ("separation", 3, False), ("rotated", 2, True))
_OUTSIDE = 9


def _layout(sections):
    """({name: (offset, shape)}, length) of the sections ((name, shape), ...) laid out one after the other."""
    out, off = {}, 0
    for name, shape in sections:
        out[name] = (off, shape)
        off += math.prod(shape)
    return out, off


def count_layout(n_xy, n_r, n_rot):
    """{section: (offset, shape)} of the count vector and the offset of the 9 outside counters; the order is the one
    include/fermiflow_b200.h documents for ff_observables."""
    nb = dict(density=n_xy, radial=n_r, separation=n_r, rotated=n_rot)
    return _layout((name, (nch, nb[name], nb[name]) if square else (nch, nb[name])) for name, nch, square in _SECTIONS)


def observables(x, n_up, n_dn, extent, n_xy, r_max, n_r, n_rot, counts):
    """ff_observables on CUDA float64 x [B, n, 2]: ADDS the histograms to counts (int64, the layout of count_layout)."""
    if x.dim() != 3 or x.shape[-1] != 2 or x.shape[1] != n_up + n_dn:
        raise ValueError("x must be [B, %d, 2], got %s" % (n_up + n_dn, tuple(x.shape)))
    g = L.FFObsGrid(float(extent), int(n_xy), int(n_rot), float(r_max), int(n_r))
    L.check(L.lib().ff_observables(L.ptr(x), x.shape[0], n_up, n_dn, C.byref(g), L.ptr(counts, torch.int64),
                                   counts.numel(), L.stream()))
    return counts


class _BatchMeans:
    """Running sums of per-batch vectors v_k (each a sum over the W_k walkers of batch k) for batch-means errors:
    [sum v_k, sum v_k² / W_k, extra sums, sum W_k, calls] in one float64 vector on `device`, so that ranks merge with
    one all-reduce."""

    def __init__(self, n_up, n_dn):
        if n_up < 0 or n_dn < 0 or n_up + n_dn < 1:
            raise ValueError("bad particle numbers %d/%d" % (n_up, n_dn))
        self.n_up, self.n_dn = int(n_up), int(n_dn)
        self._buf = None

    @staticmethod
    def _check_moves(moves):
        if moves < 1:
            raise ValueError("moves must be at least 1, got %d" % moves)
        return int(moves)

    def _check_walkers(self, x):
        n = self.n_up + self.n_dn
        if x.dim() != 3 or x.shape[-1] != 2 or x.shape[1] != n:
            raise ValueError("x must be [B, %d, 2], got %s" % (n, tuple(x.shape)))
        if not x.is_cuda:
            raise RuntimeError("%s needs CUDA walkers (got %s); no CPU fallback" % (type(self).__name__, x.device))

    def _zeroed_sums(self, n, device, dtype=torch.float64):
        """The buffer for the sums of one batch on `device`, zeroed; allocated again only when the device changes."""
        if self._buf is None or self._buf.device != device:
            self._buf = torch.empty(n, dtype=dtype, device=device)
        return self._buf.zero_()

    def _section(self, t, name):
        """Section `name` of self.layout in the vector t, in its shape."""
        off, shape = self.layout[name]
        return t[off:off + math.prod(shape)].reshape(shape)

    @staticmethod
    def _stderr(var, calls):
        """sqrt(var), NaN with fewer than two calls."""
        return torch.where(calls >= 2, var.sqrt(), torch.full_like(var, float("nan")))

    def _init_state(self, n_values, device, n_extra=0):
        """`n_extra` further running sums (after the squares, before the walker and call counts) for an estimator's
        own second moments; they travel in the same all-reduce."""
        self.device = torch.device(device)
        self._n_values = int(n_values)
        self.state = torch.zeros(2 * self._n_values + int(n_extra) + 2, dtype=torch.float64, device=self.device)

    def _merge(self, values, walkers):
        """Add one batch of `walkers` walkers whose values summed to `values` (plain torch)."""
        if walkers <= 0:
            return
        v = values.to(self.state.device, torch.float64)
        nv = self._n_values
        self.state[:nv] += v
        self.state[nv:2 * nv].addcmul_(v, v, value=1.0 / walkers)
        self.state[-2] += float(walkers)
        self.state[-1] += 1.0

    def allreduce(self):
        """Sum the state over the ranks of torch.distributed (NCCL for CUDA state, gloo for CPU state); a no-op on one
        rank.  Every rank must call it, as with VMC's allreduce_gradients, and then holds the merged state."""
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(self.state)

    def _per_walker(self):
        """(mean per walker, its standard error, walkers, calls, sum v_k² / W_k) as device tensors.  Batch means
        m_k = v_k / W_k weighted by W_k: var(mean) = Σ W_k (m_k − mean)² / ((K − 1) W); NaN below two calls."""
        nv = self._n_values
        s1, s2 = self.state[:nv], self.state[nv:2 * nv]
        W, K = self.state[-2], self.state[-1]
        mean = s1 / W
        return mean, self._stderr((s2 - W * mean * mean).clamp_min(0.0) / ((K - 1.0) * W), K), W, K, s2

    def save(self, path):
        """np.savez of result()."""
        np.savez(path, **self.result())


class DensityEstimator(_BatchMeans):
    """Spin-resolved one-body density, radial density, pair-separation distribution and rotated-frame pair density
    of walkers [B, n_up + n_dn, 2] (particle i < n_up is spin-up).

    Grids: density and rotated density on [-extent, extent)^2 with n_xy^2 and n_rot^2 cells of side
    Δ = 2 extent / n_xy (Δ_rot = 2 extent / n_rot); radial density and separation over [0, r_max) (r_max defaults to
    extent) in n_r bins of edges r_k; 0 bins switch a section off.  In the frame of the rotated density, the reference
    particle i lies on the +x axis: u = r_i · r_j / |r_i|, w = (r_i × r_j) / |r_i|.

    result() normalises per walker (W walkers in all):
      density[s][ix][iy]   particles of spin s per unit area:      Σ density[s] Δ² + outside[s] / W = n_s
      radial[s][k]         the same, averaged over annulus k:      Σ radial[s][k] π (r_{k+1}² − r_k²) + outside / W = n_s
      separation[c][k]     pairs of channel c (↑↑, ↓↓, ↑↓) per unit area of separation:
                           Σ separation[c][k] π (r_{k+1}² − r_k²) + outside[c] / W = pairs of c
                           (n_↑(n_↑−1)/2, n_↓(n_↓−1)/2, n_↑ n_↓)
      rotated[c][iu][iw]   particles of channel c (same, opposite spin) per unit area per reference particle:
                           Σ rotated[c] Δ_rot² + outside[c] / (n W) = ordered pairs of c / n
    outside_fraction[9] is each outside counter over the items of its channel (NaN for a channel without items), in the
    order of include/fermiflow_b200.h.  Each array comes with `<name>_err`, the standard error from batch means over
    the calls of accumulate(), weighted by each call's walker count (NaN with fewer than two calls).

    The state is kept in float64 on `device`: counts are exact below 2^53 per bin.
    """

    def __init__(self, n_up, n_dn, extent, n_xy=64, r_max=None, n_r=128, n_rot=64, device=torch.device("cuda")):
        super().__init__(n_up, n_dn)
        self.extent = float(extent)
        self.r_max = float(extent if r_max is None else r_max)
        self.n_xy, self.n_r, self.n_rot = int(n_xy), int(n_r), int(n_rot)
        self.layout, self.n_bins = count_layout(self.n_xy, self.n_r, self.n_rot)
        self.n_counts = self.n_bins + _OUTSIDE
        # [sum of counts, sum over calls of counts² / walkers, walkers, calls]: one vector, one all-reduce
        self._init_state(self.n_counts, device)

    def accumulate(self, x):
        """Add one batch of independent walkers x (CUDA float64 [B, n_up + n_dn, 2]); no host synchronisation."""
        counts = self._zeroed_sums(self.n_counts, x.device, torch.int64)
        observables(x, self.n_up, self.n_dn, self.extent, self.n_xy, self.r_max, self.n_r, self.n_rot, counts)
        self._add_batch(counts, x.shape[0])

    def _add_batch(self, counts, walkers):
        """Merge the counts of one batch of `walkers` walkers into the running sums (plain torch)."""
        self._merge(counts, walkers)

    def result(self):
        """dict of float64 numpy arrays (see the class docstring)."""
        mean, err, W, K, _ = self._per_walker()
        nu, nd = self.n_up, self.n_dn
        n = nu + nd
        f64 = dict(dtype=torch.float64, device=self.state.device)
        dxy = 2 * self.extent / self.n_xy if self.n_xy else 0.0
        drot = 2 * self.extent / self.n_rot if self.n_rot else 0.0
        r_edges = torch.linspace(0.0, self.r_max, self.n_r + 1, **f64)
        annulus = math.pi * (r_edges[1:] ** 2 - r_edges[:-1] ** 2)
        per_bin = dict(density=torch.full((), dxy * dxy, **f64), radial=annulus, separation=annulus,
                       rotated=torch.full((), drot * drot * n, **f64))
        out = {}
        for name, _, _ in _SECTIONS:
            norm = per_bin[name]
            out[name], out[name + "_err"] = self._section(mean, name) / norm, self._section(err, name) / norm
        items = torch.tensor([nu, nd, nu, nd, nu * (nu - 1) / 2, nd * (nd - 1) / 2, nu * nd,
                              nu * (nu - 1) + nd * (nd - 1), 2 * nu * nd], **f64)
        out["outside_fraction"] = mean[self.n_bins:] / items
        out["outside_fraction_err"] = err[self.n_bins:] / items
        out["xy_edges"] = torch.linspace(-self.extent, self.extent, self.n_xy + 1, **f64)
        out["rot_edges"] = torch.linspace(-self.extent, self.extent, self.n_rot + 1, **f64)
        out["r_edges"] = r_edges
        out["walkers"], out["calls"] = W, K
        out["n_up"], out["n_dn"] = torch.tensor(float(nu), **f64), torch.tensor(float(nd), **f64)
        return {k: v.cpu().numpy() for k, v in out.items()}


    def _summary(self, res, path):
        return ("density: %d walkers saved to %s; outside the density grid: up %.3g, down %.3g (fraction of particles)"
                % (res["walkers"], path, res["outside_fraction"][0], res["outside_fraction"][1]))


def sums_layout(n_k, n_kr, n_s):
    """{section: (offset, shape)} of the sums of ff_momentum_accumulate (include/fermiflow_b200.h) and their length."""
    return _layout((("momentum", (2, n_k, n_k)), ("radial", (2, n_kr)), ("ratio", (2, n_s)), ("records", (2, n_s)),
                    ("channel", (2,))))


def momentum_accumulate(ratio, particle, disp, n_up, k_max, n_k, n_kr, s_max, n_s, sums):
    """ff_momentum_accumulate on CUDA records (ratio float64 [R], particle int32 [R], disp float64 [R, 2]): ADDS the
    sums to `sums` (float64, the layout of sums_layout)."""
    g = L.FFMomGrid(float(k_max), int(n_k), int(n_kr), float(s_max), int(n_s))
    R = ratio.numel()
    L.check(L.lib().ff_momentum_accumulate(L.ptr(ratio.reshape(-1)), L.ptr(particle.reshape(-1), torch.int32),
                                           L.ptr(disp.reshape(-1, 2)), R, int(n_up), C.byref(g), L.ptr(sums),
                                           sums.numel(), L.stream()))
    return sums


class MomentumEstimator(_BatchMeans):
    """Spin-resolved momentum distribution n_c(k) and one-body coherence g_c(|s|) of a VMC model (GSVMC or BetaVMC)
    from signed wave-function ratios.  A record is one walker x ~ |ψ|², one particle i drawn uniformly from all n and
    one displacement s drawn uniformly in the disk |s| < s_max; its ratio is ρ = ψ(x with r_i → r_i + s) / ψ(x)
    (model.wavefunction_ratio, sign included) and its channel c = (i ≥ n_up).  With `moves` = M records per walker
    and W walkers in all:

      n_c(k) = (2π)⁻² ∫ d²s cos(k·s) Σ_{i∈c} ⟨ρ_i(s)⟩  ≈  n s_max² / (4π M W) Σ_records 1{c} ρ cos(k·s)

    normalised to ∫ n_c(k) d²k = n_c (up to the part of ⟨ρ_i(s)⟩ beyond s_max).  ρ is real and even in s because ψ is
    real, so the cosine carries all of it.  The radial n_c(|k|) is the same sum with J0(|k| |s|) in place of the
    cosine.  The one-body coherence g_c(|s|) = (1 / n_c) ∫ d²r ρ1_c(r, r + s), averaged over directions, is the mean
    of ρ over the records of channel c whose |s| falls in the annulus; g_c(0) = 1.  For BetaVMC each walker uses its
    own occupation row, and the same formulas give the quantities of the mixed state.

    result() returns float64 numpy arrays:
      momentum [2][n_k][n_k]      n_c at the cell centres of [-k_max, k_max)², index [c][ix][iy] (k_edges)
      momentum_radial [2][n_kr]   n_c(|k|) at k_radial = (j + 1/2) k_max / n_kr
      coherence [2][n_s]          g_c in the |s| bins s_edges over [0, s_max) (NaN for a bin without records)
    each with `<name>_err` (batch means over the calls of accumulate(), weighted by each call's walker count; NaN with
    fewer than two calls), and k_edges, k_radial, s_edges, walkers, calls, moves, n_up, n_dn.
    """

    def __init__(self, n_up, n_dn, k_max=4.0, n_k=64, n_kr=128, s_max=8.0, n_s=64, moves=8,
                 device=torch.device("cuda")):
        super().__init__(n_up, n_dn)
        self.moves = self._check_moves(moves)
        if not (k_max > 0 and math.isfinite(k_max) and s_max > 0 and math.isfinite(s_max)):
            raise ValueError("k_max and s_max must be positive and finite, got %r and %r" % (k_max, s_max))
        if min(n_k, n_kr, n_s) < 0:
            raise ValueError("negative bin count (n_k %d, n_kr %d, n_s %d)" % (n_k, n_kr, n_s))
        self.k_max, self.s_max = float(k_max), float(s_max)
        self.n_k, self.n_kr, self.n_s = int(n_k), int(n_kr), int(n_s)
        self.layout, self.n_sums = sums_layout(self.n_k, self.n_kr, self.n_s)
        # the sums, then ratio sum + record count per |s| bin: its squares give the cross moment the error of the
        # coherence (a ratio of two means) needs
        self._init_state(self.n_sums + 2 * self.n_s, device)

    def accumulate(self, model, x, generator=None):
        """Add one batch of independent walkers x (CUDA float64 [B, n_up + n_dn, 2], drawn by model.sample at the
        current parameters): `moves` records per walker, drawn on the device (torch.randint / torch.rand with
        `generator`); no host synchronisation."""
        self._check_walkers(x)
        B, M, dev = x.shape[0], self.moves, x.device
        particle = torch.randint(0, self.n_up + self.n_dn, (B, M), device=dev, dtype=torch.int32, generator=generator)
        u = torch.rand(B, M, 2, device=dev, dtype=torch.float64, generator=generator)
        r = self.s_max * u[..., 0].sqrt()
        phi = (2 * math.pi) * u[..., 1]
        disp = torch.stack((r * phi.cos(), r * phi.sin()), -1)
        ratio = model.wavefunction_ratio(x, particle, disp)
        sums = self._zeroed_sums(self.n_sums, dev)
        momentum_accumulate(ratio, particle, disp, self.n_up, self.k_max, self.n_k, self.n_kr, self.s_max, self.n_s,
                            sums)
        self._add_batch(sums, B)

    def _add_batch(self, sums, walkers):
        """Merge the sums of one batch of `walkers` walkers into the running state (plain torch)."""
        both = self._section(sums, "ratio") + self._section(sums, "records")
        self._merge(torch.cat((sums, both.reshape(-1))), walkers)

    def result(self):
        """dict of float64 numpy arrays (see the class docstring)."""
        mean, err, W, K, s2 = self._per_walker()
        nu, nd = self.n_up, self.n_dn
        f64 = dict(dtype=torch.float64, device=self.state.device)
        norm = (nu + nd) * self.s_max ** 2 / (4 * math.pi * self.moves)
        out = {}
        sect = self._section
        out["momentum"], out["momentum_err"] = norm * sect(mean, "momentum"), norm * sect(err, "momentum")
        out["momentum_radial"], out["momentum_radial_err"] = norm * sect(mean, "radial"), norm * sect(err, "radial")
        # coherence g = S / N per bin (S, N: ratio sum and records per walker); delta method over the batch means:
        # var(g) = Σ W_k (s_k − g n_k)² / ((K − 1) W N²), with Σ S_k N_k / W_k from the squares of S_k + N_k
        S, N = sect(mean, "ratio"), sect(mean, "records")
        g = S / N
        qS, qN = sect(s2, "ratio"), sect(s2, "records")
        cross = 0.5 * (s2[self.n_sums:].reshape(S.shape) - qS - qN)
        dev2 = qS - 2 * g * cross + g * g * qN                          # Σ W_k (s_k − g n_k)², Σ W_k (s_k − g n_k) = 0
        out["coherence"] = g
        out["coherence_err"] = self._stderr(dev2.clamp_min(0.0) / ((K - 1.0) * W * N * N), K)
        out["k_edges"] = torch.linspace(-self.k_max, self.k_max, self.n_k + 1, **f64)
        out["k_radial"] = (torch.arange(self.n_kr, **f64) + 0.5) * (self.k_max / max(self.n_kr, 1))
        out["s_edges"] = torch.linspace(0.0, self.s_max, self.n_s + 1, **f64)
        out["walkers"], out["calls"] = W, K
        out["moves"] = torch.tensor(float(self.moves), **f64)
        out["n_up"], out["n_dn"] = torch.tensor(float(nu), **f64), torch.tensor(float(nd), **f64)
        return {k: v.cpu().numpy() for k, v in out.items()}

    def _summary(self, res, path):
        dk = 2 * self.k_max / self.n_k
        return ("momentum: %d walkers saved to %s; integral of n(k) over the grid: up %.4g, down %.4g"
                % (res["walkers"], path, res["momentum"][0].sum() * dk * dk, res["momentum"][1].sum() * dk * dk))


def swap_layout(Q, n_up, n_dn):
    """{section: (offset, shape)} of the sums of ff_swap_accumulate (include/fermiflow_b200.h) and their length."""
    sec = (Q, n_up + 1, n_dn + 1)
    return _layout((("ratio", sec), ("replicas", sec), ("matched", sec), ("skipped", (Q,)), ("pairs", (1,))))


def swap_accumulate(ratio, sector, n_up, n_dn, sums):
    """ff_swap_accumulate on CUDA records (ratio float64 [P, Q], sector int32 [P, 2, Q]): ADDS the sums to `sums`
    (float64, the layout of swap_layout)."""
    P, Q = ratio.shape
    ratio, sector = ratio.contiguous(), sector.contiguous()
    L.check(L.lib().ff_swap_accumulate(L.ptr(ratio), L.ptr(sector, torch.int32), P, Q, int(n_up), int(n_dn),
                                       L.ptr(sums), sums.numel(), L.stream()))
    return sums


class RenyiEstimator(_BatchMeans):
    """Second Rényi entropy S2(A) = −ln Tr ρ_A² of spatial regions A of a VMC model (GSVMC or BetaVMC), from the
    replica swap estimator (Hastings et al. 2010; for fermions McMinis & Tubman 2013):

      Tr ρ_A² = ⟨ ψ(x′) ψ(y′) / (ψ(x) ψ(y)) ⟩,   x, y independent draws from ρ,

    x′ being x with its particles inside A replaced by those of y (slot by slot within each spin block) and y′ the
    reverse; a pair whose replicas hold different numbers (n_A↑, n_A↓) contributes exactly 0.  The regions are all of
    one `kind`: "disk" |r| < a_q about the trap centre or "halfplane" x < a_q, one per entry of `a` (1 to 32).  Each
    call of accumulate() pairs the walkers by a random permutation on the device (the last walker is dropped when B is
    odd).  The pairing must be random: BetaVMC samples its walkers' states sorted, so neighbouring walkers are
    correlated, and pairing them would bias Tr ρ² towards Σ_s p_s Tr ρ_s².  For BetaVMC each replica uses its own
    occupation row, and the estimate is Tr ρ_A² of the mixed state ρ = Σ_s p_s |ψ_s⟩⟨ψ_s|.

    ρ_A is block diagonal in (a, b) = (n_A↑, n_A↓), so the same records resolve the sectors: P(a, b) is the fraction of
    replicas in the sector, Tr ρ_{A,ab}² the sum of the ratios of the pairs in that sector over all pairs
    (Σ_ab Tr ρ_ab² = Tr ρ_A²) and S2(a, b) = −ln(Tr ρ_ab² / P(a, b)²) the entropy of the normalised block.

    Limit: the mean ratio is e^{−S2} while each record is of order one, so the relative error grows as e^{S2} / √pairs;
    regions with S2 ≳ 4 need far more samples than the default driver draws.  Swapping incrementally growing regions
    (the ratio trick) would remove this, and is not done here.

    result() returns float64 numpy arrays:
      swap [Q]                              Tr ρ_A² per region
      S2 [Q]                                −ln swap; its error swap_err / swap (NaN where swap ≤ 0)
      sector_prob [Q][n_up + 1][n_dn + 1]   P(a, b)
      sector_swap [Q][n_up + 1][n_dn + 1]   Tr ρ_{A,ab}²
      S2_sector [Q][n_up + 1][n_dn + 1]     S2(a, b) (NaN for an empty sector or a non-positive sector_swap)
    each with `<name>_err` (batch means over the calls of accumulate(), weighted by each call's pair count; NaN with
    fewer than two calls), and a, kind, pairs, calls, n_up, n_dn.
    """

    def __init__(self, n_up, n_dn, a=(0.5, 1.0, 1.5, 2.0, 2.5, 3.0), kind="disk", device=torch.device("cuda")):
        super().__init__(n_up, n_dn)
        if kind not in ("disk", "halfplane"):
            raise ValueError("kind must be 'disk' or 'halfplane', got %r" % (kind,))
        a = tuple(float(v) for v in a)
        if not 1 <= len(a) <= 32:
            raise ValueError("between 1 and 32 regions, got %d" % len(a))
        if not all(math.isfinite(v) for v in a) or (kind == "disk" and min(a) < 0):
            raise ValueError("region parameters must be finite (and radii non-negative), got %r" % (a,))
        self.a, self.kind, self.Q = a, kind, len(a)
        self.layout, self.n_sums = swap_layout(self.Q, self.n_up, self.n_dn)
        self._n_cells = self.Q * (self.n_up + 1) * (self.n_dn + 1)
        # the sums, then the ratio sum per region (its error) and ratio sum + replicas per sector (the cross moment
        # the error of S2_sector needs)
        self._init_state(self.n_sums + self.Q + self._n_cells, device)

    def accumulate(self, model, x, generator=None):
        """Add one batch of independent walkers x (CUDA float64 [B, n_up + n_dn, 2], B ≥ 2, drawn by model.sample at
        the current parameters): B // 2 pairs from torch.randperm with `generator`; no host synchronisation."""
        self._check_walkers(x)
        B, dev = x.shape[0], x.device
        if B < 2:
            raise ValueError("at least two walkers are needed for one pair, got %d" % B)
        P = B // 2
        pairs = torch.randperm(B, device=dev, generator=generator)[:2 * P].view(P, 2)
        ratio, sector = model.swap_ratio(x, pairs, self.a, self.kind)
        sums = self._zeroed_sums(self.n_sums, dev)
        swap_accumulate(ratio, sector, self.n_up, self.n_dn, sums)
        self._add_batch(sums, P)

    def _add_batch(self, sums, pairs):
        """Merge the sums of one batch of `pairs` pairs into the running state (plain torch)."""
        T = self._section(sums, "ratio")
        per_region = T.reshape(self.Q, -1).sum(1)
        self._merge(torch.cat((sums, per_region, (T + self._section(sums, "replicas")).reshape(-1))), pairs)

    def result(self):
        """dict of float64 numpy arrays, and `kind` as a string array (see the class docstring)."""
        mean, err, W, K, s2 = self._per_walker()
        f64 = dict(dtype=torch.float64, device=self.state.device)
        nan = torch.tensor(float("nan"), **f64)
        ns, Q = self.n_sums, self.Q
        sect = self._section
        out = {}
        swap, swap_err = mean[ns:ns + Q], err[ns:ns + Q]
        ok = swap > 0
        out["swap"], out["swap_err"] = swap, swap_err
        out["S2"] = torch.where(ok, -swap.clamp_min(1e-300).log(), nan)
        out["S2_err"] = torch.where(ok, swap_err / swap, nan)
        T, R = sect(mean, "ratio"), sect(mean, "replicas")              # per pair: ratio sum, replicas
        out["sector_prob"], out["sector_prob_err"] = 0.5 * R, 0.5 * sect(err, "replicas")
        out["sector_swap"], out["sector_swap_err"] = T, sect(err, "ratio")
        # S2(a, b) = −ln T + 2 ln R + const; delta method over the batch means with the cross moment
        # Σ T_k R_k / W_k taken from the squares of T_k + R_k
        good = (T > 0) & (R > 0)
        Tg, Rg = torch.where(good, T, 1.0), torch.where(good, R, 1.0)
        qT, qR = sect(s2, "ratio") - W * T * T, sect(s2, "replicas") - W * R * R
        cross = 0.5 * (s2[ns + Q:].reshape(T.shape) - sect(s2, "ratio") - sect(s2, "replicas")) - W * T * R
        dev2 = qT / (Tg * Tg) + 4 * qR / (Rg * Rg) - 4 * cross / (Tg * Rg)
        var = dev2.clamp_min(0.0) / ((K - 1.0) * W)
        out["S2_sector"] = torch.where(good, -(Tg / (0.25 * Rg * Rg)).log(), nan)
        out["S2_sector_err"] = torch.where(good & (K >= 2), var.sqrt(), nan)
        out["a"] = torch.tensor(self.a, **f64)
        out["pairs"], out["calls"] = W, K
        out["n_up"], out["n_dn"] = torch.tensor(float(self.n_up), **f64), torch.tensor(float(self.n_dn), **f64)
        res = {k: v.cpu().numpy() for k, v in out.items()}
        res["kind"] = np.array(self.kind)
        return res

    def _summary(self, res, path):
        return "renyi: %d pairs saved to %s; S2 per %s: %s" % (res["pairs"], path, self.kind, ", ".join(
            "%g: %.4g +- %.2g" % (v, s, e) for v, s, e in zip(self.a, res["S2"], res["S2_err"])))


def density_matrix_layout(K):
    """{section: (offset, shape)} of the sums of ff_density_matrix_accumulate (include/fermiflow_b200.h) for K orbitals
    and their length 2 K² + 3."""
    return _layout((("matrix", (2, K, K)), ("records", (2,)), ("skipped", (1,))))


def density_matrix_accumulate(x, particle, disp, w, n_up, n_dn, n_orb, sums):
    """ff_density_matrix_accumulate on CUDA walkers x (float64 [B, n_up + n_dn, 2]) and records (particle int32 [B, M],
    disp float64 [B, M, 2], w float64 [B, M]): ADDS the sums to `sums` (float64, the layout of density_matrix_layout)."""
    if particle.dim() != 2:
        raise ValueError("particle must be [B, M], got %s" % (tuple(particle.shape),))
    B, M = particle.shape
    if x.dim() != 3 or tuple(x.shape) != (B, n_up + n_dn, 2) or tuple(disp.shape) != (B, M, 2) \
            or tuple(w.shape) != (B, M):
        raise ValueError("x must be [%d, %d, 2], disp [%d, %d, 2] and w [%d, %d], got %s, %s and %s"
                         % (B, n_up + n_dn, B, M, B, M, tuple(x.shape), tuple(disp.shape), tuple(w.shape)))
    L.check(L.lib().ff_density_matrix_accumulate(L.ptr(x), B, int(n_up), int(n_dn), M, L.ptr(particle, torch.int32),
                                                 L.ptr(disp), L.ptr(w), int(n_orb), L.ptr(sums), sums.numel(),
                                                 L.stream()))
    return sums


class DensityMatrixEstimator(_BatchMeans):
    """Spin-resolved one-body density matrix of a VMC model (GSVMC or BetaVMC) in the first K = (shells + 1)(shells + 2)
    / 2 HO2D orbitals, D^c_ab = ∫∫ φ_a(r) ρ1_c(r, r′) φ_b(r′) dr dr′, and its spectrum, the natural-orbital occupations.
    A Slater determinant has occupations of exactly 1 and 0; correlation and Wigner localisation spread them out.

    A record is one walker x ~ |ψ|², one particle i drawn uniformly from all n and one point r′ drawn from the Gaussian
    q(r′) = exp(−|r′|² / 2σ²) / (2πσ²) about the trap centre; its ratio is ρ = ψ(x with r_i → r′) / ψ(x)
    (model.wavefunction_ratio, sign included) and its channel c = (i ≥ n_up).  With `moves` = M records per walker and
    W walkers in all:

      D^c_ab ≈ n / (M W) Σ_{records of c} ½ [φ_a(r_i) φ_b(r′) + φ_b(r_i) φ_a(r′)] ρ / q(r′)

    ψ(…r′…) φ_b(r′) decays like exp(−|r′|²), so the weight's second moment ∫ (ψ φ_b)² / q is finite only for σ > 1/2.
    σ = 1.5 is the default: it keeps that margin, and the Gaussian still reaches r′ ≈ 4, where the shell-7 orbitals
    and the outer particles of the dot have their weight.  A narrower q samples them rarely with large weights; a wider
    one spends records where ψ is negligible.  On a B200, with the benchmark's random flow at N = 20 and 12 + 0 and
    4 batches of 65536 walkers (scripts/dev_natural_orbitals_timing.py), σ = 1.5 gave the smallest error of the trace
    among σ = 1, 1.5, 2 and 3: 0.022 and 0.029 against 0.18 and 0.097 at σ = 1 and 0.068 and 0.041 at σ = 2.  The
    estimate is unbiased for every σ > 1/2.

    Tr D^c = Tr(P ρ1_c) ≤ n_c, P the projector onto the basis; it equals n_c only when ρ1 lies in the span of the K
    orbitals, so `trace` is the basis coverage.  For BetaVMC each walker uses its own occupation row, and the estimate is
    D of the mixed state.

    Errors are batch means over the calls of accumulate(), weighted by each call's walker count (NaN with fewer than
    two calls).  The occupation errors use the first-order delta method, λ_k = v_kᵀ D v_k with the eigenvector v_k
    held fixed, and the covariance of the K(K + 1)/2 independent entries of D across batches, kept in the state
    (about 7 MB at K = 36), so that allreduce() stays one all-reduce.  Two limits: near-degenerate occupations (for
    example symmetry partners in a circular dot) have only first-order individual errors, since their eigenvectors mix
    from batch to batch, while their sum is robust; and the eigenvalues of a noisy matrix are biased at O(error²) (the
    largest pushed up, the smallest down).

    result() returns float64 numpy arrays:
      density_matrix [2][K][K]      D^c (+ _err, per entry)
      trace [2]                     Tr D^c (+ _err)
      occupations [2][K]            eigenvalues of D^c in descending order (+ _err)
      natural_orbitals [2][K][K]    columns: the eigenvectors in the HO2D basis, largest component positive
      shell_weight [2][K][shells+1] squared coefficients of natural orbital k summed per oscillator shell nx + ny
      orbital_quanta [K][2]         (nx, ny) of the basis orbitals
    and walkers, calls, moves, sigma, n_up, n_dn.
    """

    def __init__(self, n_up, n_dn, shells=7, sigma=1.5, moves=8, device=torch.device("cuda")):
        super().__init__(n_up, n_dn)
        if not 0 <= shells <= 7:
            raise ValueError("shells must be in [0, 7] (HO2D has 36 orbitals), got %d" % shells)
        if not (math.isfinite(sigma) and sigma > 0.5):
            raise ValueError("sigma must be finite and above 1/2 (the weights' variance is infinite below), got %r"
                             % (sigma,))
        self.moves = self._check_moves(moves)
        self.shells, self.sigma = int(shells), float(sigma)
        self.K = K = (self.shells + 1) * (self.shells + 2) // 2
        self.layout, self.n_sums = density_matrix_layout(K)
        self._tri = torch.triu_indices(K, K)                            # the independent entries a <= b
        self._P = self._tri.shape[1]
        self._tri_dev = self._tri.to(device)
        # the sums, then Σ_batches m m^T / W of the independent entries m of each channel (the covariance of D)
        self._init_state(self.n_sums, device, n_extra=2 * self._P * self._P)

    def accumulate(self, model, x, generator=None):
        """Add one batch of independent walkers x (CUDA float64 [B, n_up + n_dn, 2], drawn by model.sample at the
        current parameters): `moves` records per walker, drawn on the device (torch.randint / torch.randn with
        `generator`); no host synchronisation."""
        self._check_walkers(x)
        x = x.detach().contiguous()
        B, M, dev = x.shape[0], self.moves, x.device
        particle = torch.randint(0, self.n_up + self.n_dn, (B, M), device=dev, dtype=torch.int32, generator=generator)
        rp = self.sigma * torch.randn(B, M, 2, device=dev, dtype=torch.float64, generator=generator)
        disp = rp - torch.gather(x, 1, particle.long()[..., None].expand(B, M, 2))
        ratio = model.wavefunction_ratio(x, particle, disp)
        s2 = self.sigma ** 2
        w = ratio * ((2 * math.pi * s2) * torch.exp((rp * rp).sum(-1) / (2 * s2)))           # ρ / q(r′)
        sums = self._zeroed_sums(self.n_sums, dev)
        density_matrix_accumulate(x, particle, disp, w, self.n_up, self.n_dn, self.K, sums)
        self._add_batch(sums, B)

    def _add_batch(self, sums, walkers):
        """Merge the sums of one batch of `walkers` walkers into the running state (plain torch)."""
        if walkers <= 0:
            return
        v = sums.to(self.state.device, torch.float64)
        self._merge(v, walkers)
        K, P = self.K, self._P
        m = v[:2 * K * K].view(2, K, K)[:, self._tri_dev[0], self._tri_dev[1]]              # [2, P]
        o = 2 * self._n_values
        self.state[o:o + 2 * P * P].view(2, P, P).baddbmm_(m[:, :, None], m[:, None, :], alpha=1.0 / walkers)

    def result(self):
        """dict of float64 numpy arrays (see the class docstring)."""
        mean, err, W, Kc, _ = self._per_walker()
        K, P = self.K, self._P
        norm = (self.n_up + self.n_dn) / self.moves
        m = mean[:2 * K * K].view(2, K, K)
        o = 2 * self._n_values
        mt = m[:, self._tri_dev[0], self._tri_dev[1]]
        # covariance of the mean of the independent entries of D, from the batch means as in _per_walker
        cov = (self.state[o:o + 2 * P * P].view(2, P, P) - W * mt[:, :, None] * mt[:, None, :]) \
            * (norm * norm / ((Kc - 1.0) * W))
        D, D_err, cov, W, Kc = (t.cpu() for t in (norm * m, norm * err[:2 * K * K].view(2, K, K), cov, W, Kc))
        ta, tb = self._tri
        diag = (ta == tb).to(torch.float64)
        evals, evecs = torch.linalg.eigh(D)
        occ, V = evals.flip(-1), evecs.flip(-1)
        big = V.abs().argmax(-2, keepdim=True)
        V = V * torch.where(torch.gather(V, -2, big) < 0, -1.0, 1.0)
        G = V[:, ta, :] * V[:, tb, :] * (2.0 - diag)[None, :, None]                         # dλ_k / dD_ab, [2, P, K]

        def sd(var):
            return self._stderr(var.clamp_min(0.0), Kc)

        quanta = torch.tensor([(orb.nx, orb.ny) for orb in HO2D().orbitals[:K]], dtype=torch.float64)
        shell = torch.nn.functional.one_hot(quanta.sum(1).long(), self.shells + 1).to(torch.float64)   # [K, shells+1]
        out = dict(density_matrix=D, density_matrix_err=D_err,
                   trace=D.diagonal(dim1=1, dim2=2).sum(-1), trace_err=sd(torch.einsum("p,cpq,q->c", diag, cov, diag)),
                   occupations=occ, occupations_err=sd(torch.einsum("cpk,cpq,cqk->ck", G, cov, G)),
                   natural_orbitals=V, shell_weight=torch.einsum("cak,as->cks", V * V, shell), orbital_quanta=quanta,
                   walkers=W, calls=Kc)
        f64 = dict(dtype=torch.float64)
        out["moves"], out["sigma"] = torch.tensor(float(self.moves), **f64), torch.tensor(self.sigma, **f64)
        out["n_up"], out["n_dn"] = torch.tensor(float(self.n_up), **f64), torch.tensor(float(self.n_dn), **f64)
        return {k: v.numpy() for k, v in out.items()}

    def _summary(self, res, path):
        lines = []
        for c, (name, nc) in enumerate((("up", self.n_up), ("down", self.n_dn))):
            lead = ", ".join("%.4f +- %.2g" % (v, e) for v, e in
                             list(zip(res["occupations"][c], res["occupations_err"][c]))[:min(nc + 2, self.K)])
            lines.append("%s: trace %.4f +- %.2g of %d, leading occupations %s"
                         % (name, res["trace"][c], res["trace_err"][c], nc, lead))
        return "natural orbitals: %d walkers, %d orbitals saved to %s; %s" % (res["walkers"], self.K, path,
                                                                             "; ".join(lines))


def add_driver_options(p):
    """The estimator options of the drivers (FermionHO2D, BetaFermionHO2D) on the argparse parser p."""
    p.add_argument("--density", metavar="FILE", help="after training, save the density and pair correlations of "
                   "freshly sampled walkers to FILE (.npz, fermiflow_b200.observables.DensityEstimator)")
    p.add_argument("--density-batches", type=int, default=16, help="batches of --batch walkers for --density")
    p.add_argument("--density-extent", type=float, default=6.0, help="half-width of the density grids")
    p.add_argument("--momentum", metavar="FILE", help="after training, save the momentum distribution and one-body "
                   "coherence of freshly sampled walkers to FILE (.npz, fermiflow_b200.observables.MomentumEstimator)")
    p.add_argument("--momentum-batches", type=int, default=16, help="batches of --batch walkers for --momentum")
    p.add_argument("--momentum-kmax", type=float, default=4.0, help="half-width of the momentum grid")
    p.add_argument("--renyi", metavar="FILE", help="after training, save the second Renyi entropy of spatial regions, "
                   "from replica swaps of freshly sampled walkers, to FILE (.npz, fermiflow_b200.observables.RenyiEstimator)")
    p.add_argument("--renyi-batches", type=int, default=16, help="batches of --batch walkers for --renyi")
    p.add_argument("--renyi-a", type=lambda s: [float(v) for v in s.split(",")], default=[0.5, 1.0, 1.5, 2.0, 2.5, 3.0],
                   help="comma-separated region parameters for --renyi: disk radii or half-plane edges x < a")
    p.add_argument("--renyi-kind", choices=("disk", "halfplane"), default="disk", help="region kind for --renyi")
    p.add_argument("--natural-orbitals", metavar="FILE", help="after training, save the one-body density matrix in the "
                   "HO2D basis and its natural-orbital occupations, from one-particle moves of freshly sampled walkers, to "
                   "FILE (.npz, fermiflow_b200.observables.DensityMatrixEstimator)")
    p.add_argument("--natural-orbitals-batches", type=int, default=16,
                   help="batches of --batch walkers for --natural-orbitals")
    p.add_argument("--natural-orbitals-shells", type=int, default=7,
                   help="oscillator shells 0 ... S of the basis for --natural-orbitals ((S + 1)(S + 2) / 2 orbitals)")


# per option of add_driver_options: its destination, the estimator made from the parsed arguments, and whether the
# estimator's accumulate() takes the model
_DRIVER_ESTIMATORS = (
    ("density", lambda a, dev: DensityEstimator(a.nup, a.ndown, a.density_extent, device=dev), False),
    ("momentum", lambda a, dev: MomentumEstimator(a.nup, a.ndown, k_max=a.momentum_kmax, device=dev), True),
    ("renyi", lambda a, dev: RenyiEstimator(a.nup, a.ndown, a=a.renyi_a, kind=a.renyi_kind, device=dev), True),
    ("natural_orbitals",
     lambda a, dev: DensityMatrixEstimator(a.nup, a.ndown, shells=a.natural_orbitals_shells, device=dev), True),
)


def run_driver_options(model, args):
    """After training, for each estimator option of add_driver_options that names a file: its --X-batches batches of
    --batch walkers from model.sample at the current parameters, merged over ranks; rank 0 saves the estimate to the
    file and prints one summary line."""
    for name, make, takes_model in _DRIVER_ESTIMATORS:
        path = getattr(args, name)
        if not path:
            continue
        est = make(args, next(model.parameters()).device)
        with torch.no_grad():
            for _ in range(getattr(args, name + "_batches")):
                _, x = model.sample((args.batch,))
                est.accumulate(*((model, x) if takes_model else (x,)))
        est.allreduce()
        if not (dist.is_available() and dist.is_initialized()) or dist.get_rank() == 0:
            est.save(path)
            print(est._summary(est.result(), path))
