"""GPU tests of the signed wave-function ratios (C ABI ff_wavefunction_ratio, GSVMC / BetaVMC.wavefunction_ratio) and of
the momentum estimators (ff_momentum_accumulate, fermiflow_b200.observables.MomentumEstimator): ratios against the fp64
oracle, accumulation against a torch restatement (J0 from scipy), the exact free-fermion momentum distribution and coherence, and the
--momentum option of the ground-state driver."""
import ctypes
import math
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
torch.set_default_dtype(torch.float64)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _rand_mlp(H, seed, scale, dev):
    from fermiflow_b200 import MLP
    gen = torch.Generator().manual_seed(seed)
    m = MLP(1, H)
    with torch.no_grad():
        m.fc1.weight.copy_(torch.randn(H, 1, generator=gen))
        m.fc1.bias.copy_(torch.randn(H, generator=gen))
        m.fc2.weight.copy_(scale * torch.randn(1, H, generator=gen))
    return m.to(dev)


def _cnf(dev, nsteps=8, H=50, zero=False):
    from fermiflow_b200 import MLP, Backflow, CNF
    if zero:
        eta, mu = MLP(1, 8), MLP(1, 8)
        eta.init_zeros(); mu.init_zeros()
        eta, mu = eta.to(dev), mu.to(dev)
    else:
        eta, mu = _rand_mlp(H, 21, 0.02, dev), _rand_mlp(H, 22, 0.02, dev)
    return CNF(Backflow(eta, mu=mu), (0.0, 1.0), nsteps=nsteps)


def _gs_model(dev, nup, ndn, zero=False):
    from fermiflow_b200 import HO2D, FreeFermion, GSVMC, HO, CoulombPairPotential
    return GSVMC(nup, ndn, HO2D(), FreeFermion(dev), _cnf(dev, zero=zero), CoulombPairPotential(2.0),
                 sp_potential=HO()).to(dev)


def _beta_model(dev, nup, ndn, zero=False):
    from fermiflow_b200 import HO2D, FreeFermion, BetaVMC, HO, CoulombPairPotential
    return BetaVMC(0.5, nup, ndn, 2.0, True, HO2D(), FreeFermion(dev), _cnf(dev, zero=zero), CoulombPairPotential(2.0),
                   sp_potential=HO()).to(dev)


def _records(B, M, n, smax, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    particle = torch.randint(0, n, (B, M), device=dev, generator=g, dtype=torch.int32)
    u = torch.rand(B, M, 2, device=dev, generator=g)
    r, phi = smax * u[..., 0].sqrt(), 2 * math.pi * u[..., 1]
    return particle, torch.stack((r * phi.cos(), r * phi.sin()), -1)


# ---- oracle: the flow and the Slater determinants in fp64 torch on the CPU ---------------------------------------

def _slater_sign_log(z, rows, nup):
    """sign, log|det| and the smallest relative singular value of each spin block at z [C, n, 2]; rows [C, n]."""
    from oracle import fermiflow_oracle as O
    allv = torch.stack([O.ho2d_orbital(k, z) for k in range(len(O.HO2D_QUANTA))], -1)          # [C, n, 36]
    sign = torch.ones(z.shape[0])
    logabs = torch.zeros(z.shape[0])
    rel = torch.ones(z.shape[0])
    for lo, hi in ((0, nup), (nup, z.shape[1])):
        if hi == lo:
            continue
        D = torch.gather(allv[:, lo:hi, :], 2, rows[:, None, lo:hi].expand(-1, hi - lo, -1))
        s, la = torch.linalg.slogdet(D)
        sv = torch.linalg.svdvals(D)
        sign, logabs = sign * s, logabs + la
        rel = torch.minimum(rel, sv[:, -1] / sv[:, 0])
    return sign, logabs, rel


def _oracle_ratio(cnf, x, particle, disp, rows, nup):
    """ratio [B, M] and the node measure (smallest relative singular value at x or x') of every record."""
    from oracle import fermiflow_oracle as O
    x, particle, disp, rows = x.cpu(), particle.long().cpu(), disp.cpu(), rows.long().cpu()
    B, n, _ = x.shape
    M = particle.shape[1]
    xc = x[:, None].repeat(1, M + 1, 1, 1)
    for b in range(B):
        for m in range(M):
            xc[b, m + 1, particle[b, m]] += disp[b, m]
    pe = tuple(t.cpu() for t in cnf.v.eta.kernel_params())
    pm = tuple(t.cpu() for t in cnf.v.mu.kernel_params())
    z, dl = O.cnf_delta_logp(xc.reshape(-1, n, 2), pe, pm, cnf.t_span, cnf.nsteps)
    sign, logabs, rel = _slater_sign_log(z, rows.repeat_interleave(M + 1, 0), nup)
    lp = (2 * logabs - dl).reshape(B, M + 1)
    sign, rel = sign.reshape(B, M + 1), rel.reshape(B, M + 1)
    ratio = sign[:, 1:] * sign[:, :1] * torch.exp(0.5 * (lp[:, 1:] - lp[:, :1]))
    return ratio, torch.minimum(rel[:, 1:], rel[:, :1])


def _check_parity(got, ref, near):
    got = got.cpu()
    assert torch.isfinite(got).all()
    rel = (got.abs() - ref.abs()).abs() / ref.abs()
    assert rel.max() <= 1e-10, float(rel.max())
    far = near > 1e-8
    assert far.float().mean() > 0.8
    assert torch.equal(torch.sign(got)[far], torch.sign(ref)[far])
    assert (ref < 0).float().mean() >= 0.1, float((ref < 0).float().mean())


@pytest.mark.parametrize("nup,ndn", [(3, 3), (7, 6), (10, 10), (12, 0), (18, 0)])
def test_ratio_parity_oracle(dev, nup, ndn):
    """Ratios against the fp64 oracle (flow x -> z and slogdet); 18 + 0 takes the CTA Slater path."""
    model = _gs_model(dev, nup, ndn)
    B, M = 8, 4
    _, x = model.sample((B,))
    particle, disp = _records(B, M, nup + ndn, 2.5, dev, seed=nup * 31 + ndn)
    got = model.wavefunction_ratio(x, particle, disp)
    assert got.shape == (B, M)
    rows = model._orb(dev)[None].expand(B, -1)
    ref, near = _oracle_ratio(model.cnf, x, particle, disp, rows, nup)
    _check_parity(got, ref, near)


def test_ratio_parity_beta_vmc(dev):
    """BetaVMC: each walker's own occupation row (a spin-polarised mixture of several states)."""
    model = _beta_model(dev, 6, 0)
    B, M = 24, 4
    _, x = model.sample((B,))
    ws = model.state_indices
    assert len(set(ws.tolist())) >= 3
    particle, disp = _records(B, M, 6, 2.5, dev, seed=5)
    got = model.wavefunction_ratio(x, particle, disp)
    rows = model._state_table(dev)[ws.long()]
    ref, near = _oracle_ratio(model.cnf, x, particle, disp, rows, 6)
    _check_parity(got, ref, near)
    # explicit walker_state equals the default, and its length is checked
    assert torch.equal(model.wavefunction_ratio(x, particle, disp, walker_state=ws), got)
    with pytest.raises(ValueError):
        model.wavefunction_ratio(x, particle, disp, walker_state=ws[:-1])


@pytest.mark.parametrize("nup,ndn", [(3, 3), (10, 10), (12, 0)])
def test_zero_displacement_and_cta_slater(dev, nup, ndn):
    """s = 0 gives 1 to rounding (bit-exact where a walker's sweep does not depend on its slot); the CTA Slater
    kernel (option slater_cta) gives the signs of the warp kernel and ratios within 1e-12."""
    from fermiflow_b200 import _lib as L
    model = _gs_model(dev, nup, ndn)
    B, M = 64, 6
    _, x = model.sample((B,))
    particle, disp = _records(B, M, nup + ndn, 2.5, dev, seed=11)
    disp[:, ::2] = 0.0
    got = model.wavefunction_ratio(x, particle, disp)
    zero = got[:, ::2]
    assert (zero - 1).abs().max() <= 1e-13, float((zero - 1).abs().max())
    print("n = %d + %d: %d of %d zero-displacement ratios are exactly 1.0"
          % (nup, ndn, int((zero == 1.0).sum()), zero.numel()))
    with L.options(slater_cta=1):
        cta = model.wavefunction_ratio(x, particle, disp)
    assert torch.equal(torch.sign(cta), torch.sign(got))
    assert ((cta - got).abs() / got.abs()).max() <= 1e-12


def test_out_of_range_particle_gives_nan(dev):
    model = _gs_model(dev, 3, 2)
    B, M = 16, 3
    _, x = model.sample((B,))
    particle, disp = _records(B, M, 5, 2.0, dev, seed=2)
    particle[0, 1], particle[3, 0], particle[7, 2] = -1, 5, 1 << 20
    got = model.wavefunction_ratio(x, particle, disp)
    bad = torch.zeros(B, M, dtype=torch.bool, device=dev)
    bad[0, 1] = bad[3, 0] = bad[7, 2] = True
    assert torch.isnan(got[bad]).all() and torch.isfinite(got[~bad]).all()


# ---- accumulation against a torch restatement -------------------------------------------------------------------

def _acc(ratio, particle, disp, n_up, grid, sums=None):
    from fermiflow_b200.observables import momentum_accumulate, sums_layout
    if sums is None:
        sums = torch.zeros(sums_layout(grid["n_k"], grid["n_kr"], grid["n_s"])[1], device=ratio.device)
    return momentum_accumulate(ratio, particle, disp, n_up, sums=sums, **grid)


def _j0(x):
    """J0 from scipy (Cephes, double precision).  torch.special.bessel_j0 is not accurate enough for a 1e-12 comparison:
    against scipy.special.j0 it is off by up to 4e-7 near x = 5."""
    from scipy.special import j0
    return torch.from_numpy(j0(x.cpu().numpy())).to(x.device)


def _acc_ref(ratio, particle, disp, n_up, k_max, n_k, n_kr, s_max, n_s):
    ch = (particle.long() >= n_up).long()
    sx, sy = disp[:, 0], disp[:, 1]
    kk = -k_max + (torch.arange(n_k, device=ratio.device) + 0.5) * (2 * k_max / max(n_k, 1))
    ph = kk[None, :, None] * sx[:, None, None] + kk[None, None, :] * sy[:, None, None]          # [R, n_k, n_k]
    w = torch.stack([ratio * (ch == c) for c in (0, 1)], 1)                                   # [R, 2]
    grid = torch.einsum("rc,rab->cab", w, torch.cos(ph))
    s = (sx * sx + sy * sy).sqrt()
    kr = (torch.arange(n_kr, device=ratio.device) + 0.5) * (k_max / max(n_kr, 1))
    radial = torch.einsum("rc,rj->cj", w, _j0(kr[None, :] * s[:, None]))
    f = (s * (n_s / s_max)).floor()
    ok = (f >= 0) & (f < n_s)
    key = (ch * n_s + f.long().clamp(0, n_s - 1))[ok]
    rsum = torch.zeros(2 * n_s, device=ratio.device).index_add_(0, key, ratio[ok])
    cnt = torch.bincount(key, minlength=2 * n_s).double()
    per = torch.bincount(ch, minlength=2).double()
    return torch.cat([grid.reshape(-1), radial.reshape(-1), rsum, cnt, per])


GRID = dict(k_max=3.0, n_k=16, n_kr=24, s_max=2.5, n_s=10)


def _check_sums(got, ref, ratio, grid):
    """|got - ref| <= 1e-12 sum |ratio| per entry; 5e-12 in the radial section, the absolute error bound of CUDA's
    double j0 for arguments of 8 and more (CUDA Math API), where the kernel's J0 values come from."""
    from fermiflow_b200.observables import sums_layout
    lay, _ = sums_layout(grid["n_k"], grid["n_kr"], grid["n_s"])
    tol = torch.full_like(ref, 1e-12 * float(ratio.abs().sum()))
    o, shape = lay["radial"]
    tol[o:o + math.prod(shape)] *= 5
    bad = (got - ref).abs() > tol
    assert not bad.any(), [(int(i), float(got[i]), float(ref[i])) for i in bad.nonzero()[:8, 0]]


@pytest.mark.parametrize("R", [1, 37, 5000, 70001])
def test_accumulate_equals_torch(dev, R):
    g = torch.Generator(device=dev).manual_seed(R)
    ratio = torch.randn(R, device=dev, generator=g) * 3
    particle = torch.randint(0, 7, (R,), device=dev, generator=g, dtype=torch.int32)
    disp = (torch.rand(R, 2, device=dev, generator=g) * 2 - 1) * 3.0         # some |s| beyond s_max
    got = _acc(ratio, particle, disp, 4, GRID)
    ref = _acc_ref(ratio, particle, disp, 4, **GRID)
    _check_sums(got, ref, ratio, GRID)
    from fermiflow_b200.observables import sums_layout
    lay, _ = sums_layout(GRID["n_k"], GRID["n_kr"], GRID["n_s"])
    o = lay["records"][0]
    assert torch.equal(got[o:], ref[o:])                                        # counts exactly
    # two calls: bit-identical; a second call adds
    assert torch.equal(_acc(ratio, particle, disp, 4, GRID), got)
    twice = _acc(ratio, particle, disp, 4, GRID, sums=got.clone())
    assert torch.equal(twice[o:], 2 * got[o:])


def test_accumulate_sections_off_nan_and_bad_n_sums(dev):
    from fermiflow_b200 import _lib as L
    R = 999
    g = torch.Generator(device=dev).manual_seed(1)
    ratio = torch.randn(R, device=dev, generator=g)
    particle = torch.randint(0, 4, (R,), device=dev, generator=g, dtype=torch.int32)
    disp = torch.rand(R, 2, device=dev, generator=g) * 2
    for grid in (dict(k_max=2.0, n_k=0, n_kr=8, s_max=2.0, n_s=0), dict(k_max=2.0, n_k=8, n_kr=0, s_max=2.0, n_s=5)):
        _check_sums(_acc(ratio, particle, disp, 2, grid), _acc_ref(ratio, particle, disp, 2, **grid), ratio, grid)
    # a non-finite ratio propagates into its channel
    r2 = ratio.clone()
    r2[10] = float("nan")
    c = int(particle[10] >= 2)
    got = _acc(r2, particle, disp, 2, GRID)
    n2 = GRID["n_k"] ** 2
    assert torch.isnan(got[c * n2:(c + 1) * n2]).all() and torch.isfinite(got[(1 - c) * n2:(2 - c) * n2]).all()
    # wrong n_sums: -1, sums untouched
    sums = torch.full((100,), 7.0, device=dev)
    gr = L.FFMomGrid(2.0, 4, 5, 2.0, 6)
    rc = L.lib().ff_momentum_accumulate(L.ptr(ratio), L.ptr(particle, torch.int32), L.ptr(disp), R, 2,
                                        ctypes.byref(gr), L.ptr(sums), 99, L.stream())
    assert rc == -1 and b"n_sums" in L.lib().ff_last_error()
    assert torch.equal(sums, torch.full((100,), 7.0, device=dev))


# ---- exact free-fermion identities -------------------------------------------------------------------------------

def _f1d(n, s):
    """integral of psi_n(x) psi_n(x + s) dx = exp(-s^2 / 4) L_n(s^2 / 2)."""
    from scipy.special import eval_laguerre
    return np.exp(-s * s / 4) * eval_laguerre(n, s * s / 2)


def _free_reference(res, occ_weights):
    """Exact n_c(k) at the cell centres, its direction average at k_radial and the annulus averages of g_c(s) for
    occupations {channel: [(weight, [orbital ids])]}."""
    from oracle import fermiflow_oracle as O
    ke = res["k_edges"]
    kc = 0.5 * (ke[1:] + ke[:-1])
    KX, KY = np.meshgrid(kc, kc, indexing="ij")
    th = 2 * np.pi * (np.arange(64) + 0.5) / 64
    se = res["s_edges"]
    gx, gw = np.polynomial.legendre.leggauss(12)
    ra, rb = se[:-1], se[1:]
    rn = 0.5 * (rb - ra)[:, None] * gx[None, :] + 0.5 * (ra + rb)[:, None]                    # [n_s, 12]

    def phi2(k, X, Y):
        return O.ho2d_orbital(k, torch.from_numpy(np.stack([X, Y], -1))).numpy() ** 2

    out = {}
    for c, occ in occ_weights.items():
        nc = len(occ[0][1])
        grid = sum(w * sum(phi2(k, KX, KY) for k in ids) for w, ids in occ)
        KR = res["k_radial"][:, None]
        radial = sum(w * sum(phi2(k, KR * np.cos(th), KR * np.sin(th)) for k in ids) for w, ids in occ).mean(1)
        SX, SY = rn[..., None] * np.cos(th), rn[..., None] * np.sin(th)
        G = sum(w * sum(_f1d(O.HO2D_QUANTA[k][0], SX) * _f1d(O.HO2D_QUANTA[k][1], SY) for k in ids)
                for w, ids in occ).mean(-1) / nc                                                 # [n_s, 12]
        ann = (G * rn * (0.5 * (rb - ra))[:, None] * gw[None, :]).sum(1) * 2 / (rb ** 2 - ra ** 2)
        out[c] = (grid, radial, ann)
    return out


def _check_free(res, ref):
    for c, (grid, radial, ann) in ref.items():
        big = grid > 0.05 * grid.max()
        assert big.sum() >= 20
        z = np.abs(res["momentum"][c] - grid)[big] / res["momentum_err"][c][big]
        assert z.max() < 5, (c, z.max())
        okr = radial > 0.05 * radial.max()
        z = np.abs(res["momentum_radial"][c] - radial)[okr] / res["momentum_radial_err"][c][okr]
        assert z.max() < 5, (c, z.max())
        z = np.abs(res["coherence"][c] - ann) / res["coherence_err"][c]
        assert z.max() < 5, (c, z.max())


def test_free_fermion_momentum_and_coherence(dev):
    """Identity flow, 3 + 3 free fermions: n_c(k) = sum over occupied orbitals of phi_a(k)^2 (HO eigenfunctions are
    their own Fourier transforms) and g_c(s) from the 1D overlaps, within 5 standard errors."""
    from fermiflow_b200 import FreeFermion, HO2D, MomentumEstimator
    occ = HO2D().orbitals[:3]
    model = _gs_model(dev, 3, 3, zero=True)
    ff = FreeFermion(dev)
    est = MomentumEstimator(3, 3, k_max=3.0, n_k=12, n_kr=16, s_max=6.0, n_s=12, device=dev)
    gen = torch.Generator(device=dev).manual_seed(7)
    for _ in range(16):
        est.accumulate(model, ff.sample(occ, occ, (65536,), equilibrim_steps=2000), generator=gen)
    res = est.result()
    assert res["walkers"] == 16 * 65536 and res["calls"] == 16 and res["moves"] == 8
    ids = [0, 1, 2]
    _check_free(res, _free_reference(res, {0: [(1.0, ids)], 1: [(1.0, ids)]}))


def test_free_fermion_beta_mixture(dev):
    """Identity flow, BetaVMC with four occupation rows of 4 + 0 particles spread over the walkers: the estimates are
    the state-weighted averages of the single-state quantities."""
    from fermiflow_b200 import FreeFermion, MomentumEstimator
    model = _beta_model(dev, 4, 0, zero=True)
    table = model._state_table(dev)
    S = min(4, table.shape[0])
    assert S >= 3
    ff = FreeFermion(dev)
    est = MomentumEstimator(4, 0, k_max=3.0, n_k=12, n_kr=16, s_max=6.0, n_s=12, device=dev)
    B = 65536
    ws = (torch.arange(B, device=dev) % S).to(torch.int32)
    model.state_indices = ws
    for _ in range(16):
        est.accumulate(model, ff.sample_multstates(table, ws, (B,), equilibrim_steps=2000))
    res = est.result()
    rows = table[:S].cpu().tolist()
    _check_free(res, _free_reference(res, {0: [(1.0 / S, r) for r in rows]}))
    assert np.isnan(res["coherence"][1]).all() and (res["momentum"][1] == 0).all()


def test_ground_state_driver_writes_momentum(dev, tmp_path):
    from fermiflow_b200 import FermionHO2D
    path = os.path.join(str(tmp_path), "mom.npz")
    hist = FermionHO2D.main(["--nup", "2", "--ndown", "1", "--Z", "2.0", "--batch", "4096", "--iternum", "3",
                             "--nsteps", "4", "--Deta", "8", "--Dmu", "8", "--momentum", path, "--momentum-batches", "16"])
    assert len(hist) == 3
    res = dict(np.load(path))
    for k in ("momentum", "momentum_err", "momentum_radial", "momentum_radial_err", "coherence", "coherence_err",
              "k_edges", "k_radial", "s_edges", "walkers", "calls", "moves", "n_up", "n_dn"):
        assert k in res, k
    assert res["walkers"] == 16 * 4096 and res["calls"] == 16 and res["momentum"].shape == (2, 64, 64)
    dk = np.diff(res["k_edges"])[0]
    for c, nc in enumerate((2, 1)):
        # the grid sum weighs each record by a Dirichlet kernel of |s|: about 0.075 standard error at this size
        assert abs(res["momentum"][c].sum() * dk * dk - nc) < 0.4
        assert abs(res["coherence"][c][0] - 1) < 0.1
