"""Variational Monte Carlo drivers -- mirror of reference src/VMC.py (GSVMC, BetaVMC).

forward(batch) does what the reference does per iteration -- sample walkers, local energy,
and a scalar whose backward() leaves the energy gradient in the parameters' .grad -- but
as three fused CUDA stages:
  1. Metropolis sampling of the base state + flow z -> x     (ff_metropolis, ff_cnf_generate)
  2. one forward-mode sweep x -> z giving log p, its gradient and Laplacian, E_loc, and
     the stash of stage inputs                                (ff_eloc)
  3. on backward(): the exact reverse sweep + parameter-gradient reduction
                                                              (ff_logp_backward)
Walkers are independent Markov chains: under torch.distributed each rank works on its own
`batch` walkers and only the energy moments and the few-KB parameter gradient are
all-reduced (allreduce_gradients()).
"""
import ctypes as C
from collections import Counter

import torch
import torch.distributed as dist

from . import _lib as L
from .base_dist import _FreeFermionLogp, _state_table
from .flow import _backward_through_flow, _flat_params
from .orbitals import orbital_indices
from .potentials import HO, CoulombPairPotential
from .utils import eloc_sweep


def _potential_flags(pair_potential, sp_potential):
    """(Z, harmonic) for the fused sweep: the reference's CoulombPairPotential and HO are evaluated inside it
    (VMC.py:27-28 accepts any object with V(x); others are added by _add_external_potentials)."""
    for name, pot in (("pair_potential", pair_potential), ("sp_potential", sp_potential)):
        if not (pot is None and name == "sp_potential") and not callable(getattr(pot, "V", None)):
            raise TypeError("%s must provide V(x) (reference VMC.py:52-55), got %r" % (name, type(pot).__name__))
    Z = float(pair_potential.Z) if type(pair_potential) is CoulombPairPotential else 0.0
    return Z, type(sp_potential) is HO


def _add_external_potentials(owner, res, x):
    """Potentials the fused sweep does not know (any object with V(x) other than CoulombPairPotential / HO,
    VMC.py:52-55): evaluated by their own V on the device and added to the potential and the local energy."""
    extra = None
    if type(owner.pair_potential) is not CoulombPairPotential:
        extra = owner.pair_potential.V(x.detach())
    if owner.sp_potential is not None and type(owner.sp_potential) is not HO:
        v = owner.sp_potential.V(x.detach())
        extra = v if extra is None else extra + v
    if extra is not None:
        res.potential = res.potential + extra
        res.eloc = res.eloc + extra
    return res


class _LogpFromSweep(torch.autograd.Function):
    """log p(x; theta) of an E_loc sweep as a differentiable function of the flow
    parameters: backward = ff_logp_backward seeded with d log p0/dz and -1."""

    @staticmethod
    def forward(ctx, owner, res, orb, walker_state, n_up, n_dn, *params):
        ctx.owner, ctx.res, ctx.orb, ctx.ws, ctx.nud = owner, res, orb, walker_state, (n_up, n_dn)
        return res.logp.clone()

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        res = ctx.res
        if res.stash is None:
            raise RuntimeError("the adjoint stash of this sweep was released by an earlier backward(): "
                               "run the forward pass again (retain_graph is not supported on the fused path)")
        B = g.shape[0]
        z = res.z.detach().requires_grad_(True)
        with torch.enable_grad():
            lp0 = _FreeFermionLogp.apply(z, ctx.orb, ctx.ws, *ctx.nud)
        g0, = torch.autograd.grad(lp0, z, grad_outputs=g.contiguous())
        _, gparams = _backward_through_flow(ctx.owner.cnf, res.model, res.stash, B, g0, -g, False)
        res.stash = None            # 22 GB at 65536 walkers, N = 20: free it now, not when the graph dies
        return (None, None, None, None, None, None, *gparams)


def _ratio_setup(cnf, x, n_up, work_size, rows, cols):
    """The start of both ratio entry points: x [B, n, 2] checked, detached and contiguous, the model struct of cnf for
    its n particles, and the work buffer that work_size (ff_wavefunction_ratio_work_size or ff_swap_ratio_work_size)
    asks for `rows` x `cols` records."""
    x = x.detach().contiguous()
    if x.dim() != 3 or x.shape[-1] != 2:
        raise ValueError("x must be [B, n, 2], got %s" % (tuple(x.shape),))
    model = cnf._model(x.shape[1], n_up=n_up)
    nw = C.c_longlong()
    L.check(work_size(C.byref(model), rows, cols, C.byref(nw)))
    return x, model, torch.empty(nw.value, dtype=torch.float64, device=x.device)


def _wavefunction_ratio(cnf, x, orb, walker_state, n_up, particle, disp):
    """psi(x_b with r_i -> r_i + s) / psi(x_b) for every record (b, m), i = particle[b, m], s = disp[b, m], with the
    sign of the Slater determinants (C ABI ff_wavefunction_ratio).  x [B, n, 2], particle integer [B, M], disp
    [B, M, 2], all on the device; returns ratio [B, M].  A particle index outside [0, n) gives NaN."""
    B = x.shape[0]
    if particle.dim() != 2 or particle.shape[0] != B or tuple(disp.shape) != (B, particle.shape[1], 2):
        raise ValueError("particle must be [B, M] and disp [B, M, 2] for B = %d walkers, got %s and %s"
                         % (B, tuple(particle.shape), tuple(disp.shape)))
    M = particle.shape[1]
    p32 = particle.to(torch.int32).contiguous()
    disp = disp.detach().contiguous()
    x, model, work = _ratio_setup(cnf, x, n_up, L.lib().ff_wavefunction_ratio_work_size, B, M)
    ratio = torch.empty(B, M, dtype=torch.float64, device=x.device)
    L.check(L.lib().ff_wavefunction_ratio(C.byref(model), L.ptr(x), B, L.ptr(orb, torch.int32),
                                          L.ptr(walker_state, torch.int32) if walker_state is not None else None,
                                          M, L.ptr(p32, torch.int32), L.ptr(disp), L.ptr(ratio), L.ptr(work), L.stream()))
    return ratio


_REGION_KINDS = {"disk": 0, "halfplane": 1}


def _swap_ratio(cnf, x, orb, walker_state, n_up, pairs, a, kind):
    """psi(x') psi(y') / (psi(x) psi(y)) for every pair p (x = x[pairs[p, 0]], y = x[pairs[p, 1]]) and region q, x'
    and y' the two walkers with their particles in region q swapped (C ABI ff_swap_ratio).  x [B, n, 2] and pairs
    integer [P, 2] on the device, a: Q region parameters (disk radii or half-plane edges), kind "disk" or "halfplane";
    returns ratio [P, Q] and sector int32 [P, 2, Q].  A walker index outside [0, B) gives NaN and sector -1."""
    if pairs.dim() != 2 or pairs.shape[1] != 2:
        raise ValueError("pairs must be [P, 2], got %s" % (tuple(pairs.shape),))
    if kind not in _REGION_KINDS:
        raise ValueError("kind must be one of %s, got %r" % (sorted(_REGION_KINDS), kind))
    P = pairs.shape[0]
    av = (C.c_double * len(a))(*[float(v) for v in a])
    reg = L.FFSwapRegions(_REGION_KINDS[kind], len(a), av)
    p32 = pairs.to(torch.int32).contiguous()
    x, model, work = _ratio_setup(cnf, x, n_up, L.lib().ff_swap_ratio_work_size, P, len(a))
    ratio = torch.empty(P, len(a), dtype=torch.float64, device=x.device)
    sector = torch.empty(P, 2, len(a), dtype=torch.int32, device=x.device)
    L.check(L.lib().ff_swap_ratio(C.byref(model), L.ptr(x), x.shape[0], L.ptr(orb, torch.int32),
                                  L.ptr(walker_state, torch.int32) if walker_state is not None else None,
                                  P, L.ptr(p32, torch.int32), C.byref(reg), L.ptr(ratio), L.ptr(sector, torch.int32),
                                  L.ptr(work), L.stream()))
    return ratio, sector


def _multi_rank():
    return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1


def _moments(*vs):
    """[sum v, sum v^2] of each vector plus the local count, as ONE device vector (no host synchronisation)."""
    v0 = vs[0]
    parts = []
    for v in vs:
        parts += [v.sum(), (v * v).sum()]
    parts.append(torch.full((), float(v0.numel()), device=v0.device, dtype=v0.dtype))      # (a fill kernel, not a host-to-device copy)
    return torch.stack(parts)


def _mean_std(tot, tot2, cnt):
    """mean and unbiased standard deviation from the (all-reduced) sums -- device tensors."""
    mean = tot / cnt
    var = (tot2 - cnt * mean * mean).clamp_min(0.0) / (cnt - 1.0).clamp_min(1.0)
    return mean, var.sqrt()


def _global_mean_std(v):
    """mean and unbiased std of v over all ranks (3-number all-reduce) as Python floats, and the global count."""
    s = _moments(v)
    if _multi_rank():
        dist.all_reduce(s)
    mean, std = _mean_std(s[0], s[1], s[2])
    return mean.item(), std.item(), s[2].item()


class _VMCBase(torch.nn.Module):
    """Observables (E, E_std, ...) are kept as device scalars and copied to the host, all in one transfer, the first
    time one of them is read: forward() itself never waits for the GPU, so the backward pass and the optimiser step
    are queued behind the sweep without a gap (the reference calls .item() inside forward, VMC.py:56)."""

    _OBSERVABLES = ()

    def _set_observables(self, **dev):
        self._obs_dev, self._obs_host = dev, None

    def observables_device(self):
        """The observables of the last forward() as one device vector, in the order of their definition (no
        host synchronisation)."""
        return torch.stack([v.reshape(()) for v in self._obs_dev.values()])

    def _observable(self, name):
        if self._obs_host is None:
            keys = list(self._obs_dev)
            self._obs_host = dict(zip(keys, torch.stack([self._obs_dev[k].reshape(()) for k in keys]).tolist()))
        return self._obs_host[name]

    def allreduce_gradients(self):
        """Sum the parameter gradients over ranks (call between backward() and step())."""
        if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
            return
        grads = [p.grad for p in self.parameters() if p.grad is not None]
        if not grads:
            return
        flat = torch.cat([g.reshape(-1) for g in grads])
        dist.all_reduce(flat)
        o = 0
        for g in grads:
            g.copy_(flat[o:o + g.numel()].view_as(g))
            o += g.numel()


def _observable_property(name):
    return property(lambda self: self._observable(name))


class GSVMC(_VMCBase):
    """Ground-state VMC (VMC.py:4-61)."""

    E, E_std = _observable_property("E"), _observable_property("E_std")

    def __init__(self, nup, ndown, orbitals, basedist, cnf, pair_potential, sp_potential=None):
        super().__init__()
        self.orbitals_up, self.orbitals_down = orbitals.orbitals[:nup], orbitals.orbitals[:ndown]
        self.nup, self.ndown = nup, ndown
        self.basedist = basedist
        self.cnf = cnf
        self.pair_potential = pair_potential
        self.sp_potential = sp_potential
        self._Z, self._harmonic = _potential_flags(pair_potential, sp_potential)

    def _orb(self, device):
        return orbital_indices(tuple(self.orbitals_up) + tuple(self.orbitals_down), device)

    def sample(self, sample_shape):                                   # VMC.py:31-34
        z = self.basedist.sample(self.orbitals_up, self.orbitals_down, sample_shape)
        x = self.cnf.generate(z)
        return z, x

    def logp(self, x, params_require_grad=False):                     # VMC.py:36-39
        z, delta_logp = self.cnf.delta_logp(x, params_require_grad=params_require_grad)
        return self.basedist.log_prob(self.orbitals_up, self.orbitals_down, z) - delta_logp

    def local_energy(self, x, stash=False):
        """log p, grad, laplacian, kinetic, potential, E_loc at x (VMC.py:44-55)."""
        res = eloc_sweep(self.cnf, x, self._orb(x.device), None, self.nup, self._Z, self._harmonic, stash=stash)
        return _add_external_potentials(self, res, x)

    def wavefunction_ratio(self, x, particle, disp):
        """psi(x with r_i -> r_i + s) / psi(x) per record, sign included: x [B, n, 2], particle [B, M] (i),
        disp [B, M, 2] (s) -> ratio [B, M] (fermiflow_b200.observables.MomentumEstimator uses it)."""
        return _wavefunction_ratio(self.cnf, x, self._orb(x.device), None, self.nup, particle, disp)

    def swap_ratio(self, x, pairs, a, kind="disk"):
        """Replica swap ratios psi(x') psi(y') / (psi(x) psi(y)) of the walker pairs [P, 2] for the regions a (disk
        radii or half-plane edges, Q of them): x [B, n, 2] -> ratio [P, Q], sector int32 [P, 2, Q]
        (fermiflow_b200.observables.RenyiEstimator uses it)."""
        return _swap_ratio(self.cnf, x, self._orb(x.device), None, self.nup, pairs, a, kind)

    def forward(self, batch):                                         # VMC.py:41-61
        _, x = self.sample((batch,))
        res = self.local_energy(x, stash=True)
        Eloc = res.eloc
        s = _moments(Eloc)
        if _multi_rank():
            dist.all_reduce(s)
        nglobal = s[2]
        E, E_std = _mean_std(s[0], s[1], nglobal)
        self._set_observables(E=E, E_std=E_std)
        self.last = res.without_stash()
        logp_full = _LogpFromSweep.apply(self, res, self._orb(x.device), None, self.nup, self.ndown,
                                         *_flat_params(self.cnf.v))
        # sum / global count == mean over all ranks once the gradients are all-reduced
        gradE = (logp_full * (Eloc - E)).sum() / nglobal
        return gradE


def _beta_estimators(Eloc, sl, log_state_weights, beta, local_cnt):
    """VMC.py:139-171 on this rank's walkers (sl: sorted state index per walker, local_cnt: walkers per state).
    Returns the observables (device scalars), the global walker count, gradF_phi (VMC.py:162, scalar with graph to
    log_state_weights) and the per-walker mean of E_loc over all walkers of the same state (VMC.py:164-168)."""
    NS = log_state_weights.shape[0]
    logp_all = torch.log_softmax(log_state_weights, dim=0)
    logp_states = logp_all.detach()[sl]
    Floc = Eloc + logp_states / beta
    # every cross-rank quantity of the iteration in ONE all-reduce: moments of E_loc, F_loc and log p(state),
    # and per state the sum of E_loc and the number of walkers
    zeros = torch.zeros(NS, dtype=Eloc.dtype, device=Eloc.device)
    red = torch.cat([_moments(Eloc, Floc, logp_states), zeros.index_add(0, sl, Eloc), local_cnt])
    if _multi_rank():
        dist.all_reduce(red)
    nglobal = red[6]
    E, E_std = _mean_std(red[0], red[1], nglobal)
    F, F_std = _mean_std(red[2], red[3], nglobal)
    lpa = logp_all.detach()
    obs = dict(E=E, E_std=E_std, F=F, F_std=F_std, S=-red[4] / nglobal, S_analytical=-(lpa * lpa.exp()).sum(),
               logp_states_all=lpa)
    ssum, cnt = red[7:7 + NS], red[7 + NS:7 + 2 * NS]
    # sum_w logp_all[state_w] (Floc_w - F) = sum_s logp_all[s] (sum_{w in s} Floc_w - F count_s): autograd never
    # sees a batch-fold duplicated gather; as everywhere, local sums / the global walker count become the global
    # mean once the gradients are all-reduced
    wstate = zeros.index_add(0, sl, Floc) - F * local_cnt
    gradF_phi = (logp_all * wstate).sum() / nglobal
    Eloc_x_mean = (ssum / cnt.clamp_min(1.0))[sl]
    return obs, nglobal, gradF_phi, Eloc_x_mean


class BetaVMC(_VMCBase):
    """Finite-temperature VMC (VMC.py:63-171)."""

    E, E_std = _observable_property("E"), _observable_property("E_std")
    F, F_std = _observable_property("F"), _observable_property("F_std")
    S, S_analytical = _observable_property("S"), _observable_property("S_analytical")

    def __init__(self, beta, nup, ndown, deltaE, boltzmann, orbitals, basedist, cnf,
                 pair_potential, sp_potential=None):
        super().__init__()
        self.beta = beta
        self.nup, self.ndown = nup, ndown
        self.states, self.Es_original = orbitals.fermion_states(nup, ndown, deltaE)
        self.Es_original = torch.tensor(self.Es_original, dtype=torch.float64)
        self.Nstates = len(self.states)
        self.log_state_weights = torch.nn.Parameter(
            -self.beta * (self.Es_original - self.Es_original[0])
            if boltzmann else torch.randn(self.Nstates, dtype=torch.float64))
        self.basedist = basedist
        self.cnf = cnf
        self.pair_potential = pair_potential
        self.sp_potential = sp_potential
        self._Z, self._harmonic = _potential_flags(pair_potential, sp_potential)
        self._table = None

    def _state_table(self, device):
        if self._table is None or self._table.device != device:
            self._table = _state_table(self.states, device)
        return self._table

    @property
    def state_indices_collection(self):
        """Counter {state index: multiplicity} of the last sample (VMC.py:97)."""
        return Counter({int(s): int(c) for s, c in enumerate(self.state_counts.tolist()) if c})

    def sample_states(self, batch, uniforms=None):
        """Occupation sampling (VMC.py:94-97): sorted state index per walker."""
        dev = self.log_state_weights.device
        u = torch.rand(batch, dtype=torch.float64, device=dev) if uniforms is None else uniforms.contiguous()
        state = torch.empty(batch, dtype=torch.int32, device=dev)
        counts = torch.empty(self.Nstates, dtype=torch.int32, device=dev)
        work = torch.empty(self.Nstates, dtype=torch.float64, device=dev)
        L.check(L.lib().ff_occupation_sample(L.ptr(self.log_state_weights.detach().contiguous()), self.Nstates,
                                             L.ptr(u), batch, L.ptr(state, torch.int32),
                                             L.ptr(counts, torch.int32), L.ptr(work), L.stream()))
        self.state_indices, self.state_counts = state, counts
        return state

    def sample(self, sample_shape, nframes=None):                      # VMC.py:89-108
        batch = int(sample_shape[0])
        state = self.sample_states(batch)
        z = self.basedist.sample_multstates(self._state_table(state.device), state, sample_shape)
        x = self.cnf.generate(z, nframes=nframes)
        return z, x

    def logp(self, x, params_require_grad=False):                      # VMC.py:110-118
        z, delta_logp = self.cnf.delta_logp(x, params_require_grad=params_require_grad)
        log_prob_z = _FreeFermionLogp.apply(z, self._state_table(x.device), self.state_indices, self.nup, self.ndown)
        return log_prob_z - delta_logp

    def _walker_state(self, x, walker_state):
        """int32 occupation row per walker of x: walker_state, or by default the state_indices of the last sample()."""
        ws = getattr(self, "state_indices", None) if walker_state is None else walker_state
        if ws is None or ws.shape != (x.shape[0],):
            raise ValueError("walker_state must hold one state index per walker (%d), got %s"
                             % (x.shape[0], None if ws is None else tuple(ws.shape)))
        return ws.to(torch.int32).contiguous()

    def wavefunction_ratio(self, x, particle, disp, walker_state=None):
        """GSVMC.wavefunction_ratio with each walker's own occupation row: walker_state (int [B]) defaults to the
        state_indices of the last sample()."""
        return _wavefunction_ratio(self.cnf, x, self._state_table(x.device), self._walker_state(x, walker_state),
                                   self.nup, particle, disp)

    def swap_ratio(self, x, pairs, a, kind="disk", walker_state=None):
        """GSVMC.swap_ratio with each walker's own occupation row (the two sides of a pair may sit in different
        states): walker_state (int [B]) defaults to the state_indices of the last sample()."""
        return _swap_ratio(self.cnf, x, self._state_table(x.device), self._walker_state(x, walker_state), self.nup,
                           pairs, a, kind)

    def forward(self, batch):                                          # VMC.py:120-171
        _, x = self.sample((batch,))
        table, state = self._state_table(x.device), self.state_indices
        res = _add_external_potentials(self, eloc_sweep(self.cnf, x, table, state, self.nup, self._Z, self._harmonic, stash=True), x)
        self.last = res.without_stash()
        Eloc = res.eloc
        obs, nglobal, gradF_phi, Eloc_x_mean = _beta_estimators(Eloc, state.long(), self.log_state_weights, self.beta,
                                                                self.state_counts.to(Eloc.dtype))
        self.logp_states_all = obs.pop("logp_states_all")
        self._set_observables(**obs)
        logp_full = _LogpFromSweep.apply(self, res, table, state, self.nup, self.ndown, *_flat_params(self.cnf.v))
        gradF_theta = (logp_full * (Eloc - Eloc_x_mean)).sum() / nglobal
        return gradF_phi, gradF_theta
