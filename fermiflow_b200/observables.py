"""Spin-resolved one-body density and pair correlations of sampled walkers (C ABI ff_observables).

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

# sections of the count vector (include/fermiflow_b200.h ff_observables): name, channels, square grid
_SECTIONS = (("density", 2, True), ("radial", 2, False), ("separation", 3, False), ("rotated", 2, True))
_OUTSIDE = 9


def count_layout(n_xy, n_r, n_rot):
    """{section: (offset, shape)} of the count vector and the offset of the 9 outside counters; the order is the one
    include/fermiflow_b200.h documents for ff_observables."""
    nb = dict(density=n_xy, radial=n_r, separation=n_r, rotated=n_rot)
    out, off = {}, 0
    for name, nch, square in _SECTIONS:
        shape = (nch, nb[name], nb[name]) if square else (nch, nb[name])
        out[name] = (off, shape)
        off += math.prod(shape)
    return out, off


def observables(x, n_up, n_dn, extent, n_xy, r_max, n_r, n_rot, counts):
    """ff_observables on CUDA float64 x [B, n, 2]: ADDS the histograms to counts (int64, the layout of count_layout)."""
    if x.dim() != 3 or x.shape[-1] != 2 or x.shape[1] != n_up + n_dn:
        raise ValueError("x must be [B, %d, 2], got %s" % (n_up + n_dn, tuple(x.shape)))
    g = L.FFObsGrid(float(extent), int(n_xy), int(n_rot), float(r_max), int(n_r))
    L.check(L.lib().ff_observables(L.ptr(x), x.shape[0], n_up, n_dn, C.byref(g), L.ptr(counts, torch.int64),
                                   counts.numel(), L.stream()))
    return counts


class DensityEstimator:
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
        if n_up < 0 or n_dn < 0 or n_up + n_dn < 1:
            raise ValueError("bad particle numbers %d/%d" % (n_up, n_dn))
        self.n_up, self.n_dn = int(n_up), int(n_dn)
        self.extent = float(extent)
        self.r_max = float(extent if r_max is None else r_max)
        self.n_xy, self.n_r, self.n_rot = int(n_xy), int(n_r), int(n_rot)
        self.device = torch.device(device)
        self.layout, self.n_bins = count_layout(self.n_xy, self.n_r, self.n_rot)
        self.n_counts = self.n_bins + _OUTSIDE
        # [sum of counts, sum over calls of counts² / walkers, walkers, calls]: one vector, one all-reduce
        self.state = torch.zeros(2 * self.n_counts + 2, dtype=torch.float64, device=self.device)
        self._buf = None

    def accumulate(self, x):
        """Add one batch of independent walkers x (CUDA float64 [B, n_up + n_dn, 2]); no host synchronisation."""
        if self._buf is None or self._buf.device != x.device:
            self._buf = torch.empty(self.n_counts, dtype=torch.int64, device=x.device)
        self._buf.zero_()
        observables(x, self.n_up, self.n_dn, self.extent, self.n_xy, self.r_max, self.n_r, self.n_rot, self._buf)
        self._add_batch(self._buf, x.shape[0])

    def _add_batch(self, counts, walkers):
        """Merge the counts of one batch of `walkers` walkers into the running sums (plain torch)."""
        if walkers <= 0:
            return
        c = counts.to(self.state.device, torch.float64)
        nc = self.n_counts
        self.state[:nc] += c
        self.state[nc:2 * nc].addcmul_(c, c, value=1.0 / walkers)
        self.state[-2] += float(walkers)
        self.state[-1] += 1.0

    def allreduce(self):
        """Sum the state over the ranks of torch.distributed (NCCL for CUDA state, gloo for CPU state); a no-op on one
        rank.  Every rank must call it, as with VMC's allreduce_gradients, and then holds the merged state."""
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(self.state)

    def result(self):
        """dict of float64 numpy arrays (see the class docstring)."""
        nc = self.n_counts
        s1, s2 = self.state[:nc], self.state[nc:2 * nc]
        W, K = self.state[-2], self.state[-1]
        mean = s1 / W
        # batch means m_k = c_k / B_k weighted by B_k: var(mean) = Σ B_k (m_k − mean)² / ((K − 1) W)
        var = (s2 - W * mean * mean).clamp_min(0.0) / ((K - 1.0) * W)
        err = torch.where(K >= 2, var.sqrt(), torch.full_like(var, float("nan")))
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
        for name, nch, _ in _SECTIONS:
            off, shape = self.layout[name]
            m, e = (t[off:off + math.prod(shape)].reshape(shape) for t in (mean, err))
            norm = per_bin[name]
            out[name], out[name + "_err"] = m / norm, e / norm
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

    def save(self, path):
        """np.savez of result()."""
        np.savez(path, **self.result())


def sample_density(model, n_up, n_dn, batch, batches, extent, path):
    """The --density option of the drivers: `batches` batches of `batch` walkers from model.sample at the current
    parameters, merged over ranks and saved to `path` by rank 0."""
    est = DensityEstimator(n_up, n_dn, extent, device=next(model.parameters()).device)
    with torch.no_grad():
        for _ in range(batches):
            _, x = model.sample((batch,))
            est.accumulate(x)
    est.allreduce()
    if not (dist.is_available() and dist.is_initialized()) or dist.get_rank() == 0:
        est.save(path)
        res = est.result()
        print("density: %d walkers saved to %s; outside the density grid: up %.3g, down %.3g (fraction of particles)"
              % (res["walkers"], path, res["outside_fraction"][0], res["outside_fraction"][1]))
    return est
