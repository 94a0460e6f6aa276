"""GPU tests of the one-body density matrix in the HO2D basis (C ABI ff_density_matrix_accumulate,
fermiflow_b200.observables.DensityMatrixEstimator): the accumulation against a torch restatement, the determinant
identity that makes the occupied block exact walker by walker, the occupations of free fermions and of a BetaVMC
mixture, an interacting flow at two proposal widths, and the --natural-orbitals option of both drivers."""
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


def _cnf(dev, zero):
    from fermiflow_b200 import MLP, Backflow, CNF
    if zero:
        eta, mu = MLP(1, 8), MLP(1, 8)
        eta.init_zeros(); mu.init_zeros()
        eta, mu = eta.to(dev), mu.to(dev)
    else:
        eta, mu = _rand_mlp(50, 21, 0.02, dev), _rand_mlp(50, 22, 0.02, dev)
    return CNF(Backflow(eta, mu=mu), (0.0, 1.0), nsteps=8)


def _gs_model(dev, nup, ndn, zero):
    from fermiflow_b200 import HO2D, FreeFermion, GSVMC, HO, CoulombPairPotential
    return GSVMC(nup, ndn, HO2D(), FreeFermion(dev), _cnf(dev, zero), CoulombPairPotential(2.0),
                 sp_potential=HO()).to(dev)


def _walkers(model, B, dev):
    """B walkers from |psi|^2: well-equilibrated base samples z (2000 Metropolis steps) carried through the flow."""
    from fermiflow_b200 import FreeFermion
    z = FreeFermion(dev).sample(model.orbitals_up, model.orbitals_down, (B,), equilibrim_steps=2000)
    with torch.no_grad():
        return model.cnf.generate(z)


def _orbitals(pos, K):
    from oracle import fermiflow_oracle as O
    return torch.stack([O.ho2d_orbital(k, pos) for k in range(K)], -1)


# ---- accumulation against a torch restatement -------------------------------------------------------------------

def _acc(x, particle, disp, w, n_up, n_dn, K):
    from fermiflow_b200.observables import density_matrix_accumulate, density_matrix_layout
    sums = torch.zeros(density_matrix_layout(K)[1], device=x.device)
    return density_matrix_accumulate(x, particle, disp, w, n_up, n_dn, K, sums)


def _acc_ref(x, particle, disp, w, n_up, K):
    """(sums, sum of |terms| per entry) in the layout of ff_density_matrix_accumulate."""
    B, M = particle.shape
    n = x.shape[1]
    p, d, w = particle.reshape(-1).long(), disp.reshape(-1, 2), w.reshape(-1)
    b = torch.arange(B * M, device=x.device) // M
    ok = (p >= 0) & (p < n)
    ri = x[b[ok], p[ok]]
    U, V = _orbitals(ri, K), _orbitals(ri + d[ok], K) * w[ok, None]
    ch = (p[ok] >= n_up)
    mats, mags = [], []
    for c in (0, 1):
        u, v = U[ch == c], V[ch == c]
        mats.append(0.5 * (u.T @ v + v.T @ u))
        mags.append(0.5 * (u.abs().T @ v.abs() + v.abs().T @ u.abs()))
    counts = torch.stack([(ch == 0).sum(), (ch == 1).sum(), (~ok).sum()]).double()
    return torch.cat([torch.stack(mats).reshape(-1), counts]), torch.cat([torch.stack(mags).reshape(-1), counts])


@pytest.mark.parametrize("K,B,M", [(1, 1, 1), (6, 37, 3), (21, 5000, 2), (36, 10001, 7)])
def test_accumulate_equals_torch(dev, K, B, M):
    """Both channels, several CTAs and a ragged last tile (R = 70007 at K = 36), invalid particle indices skipped and
    counted (their w is NaN, so reading it would show), agreement to 1e-12 of sum |terms|, two calls bit-identical."""
    n_up, n_dn = 4, 3
    g = torch.Generator(device=dev).manual_seed(K * 1000 + B)
    x = 1.3 * torch.randn(B, n_up + n_dn, 2, device=dev, generator=g)
    particle = torch.randint(0, n_up + n_dn, (B, M), device=dev, generator=g, dtype=torch.int32)
    disp = 1.5 * torch.randn(B, M, 2, device=dev, generator=g)
    w = torch.randn(B, M, device=dev, generator=g) * 4
    if B * M > 3:
        flat = particle.view(-1)
        bad = torch.tensor([1, B * M // 2, B * M - 1], device=dev)
        flat[bad] = torch.tensor([-1, n_up + n_dn, 1 << 20], device=dev, dtype=torch.int32)
        w.view(-1)[bad] = float("nan")
    got = _acc(x, particle, disp, w, n_up, n_dn, K)
    ref, mag = _acc_ref(x, particle, disp, w, n_up, K)
    assert torch.isfinite(got).all()
    bad = (got - ref).abs() > 1e-12 * mag
    assert not bad.any(), [(int(i), float(got[i]), float(ref[i])) for i in bad.nonzero()[:8, 0]]
    assert torch.equal(got[-3:], ref[-3:])                                    # counts exactly
    if B * M > 3:
        assert float(got[-1]) == 3.0
    mat = got[:2 * K * K].view(2, K, K)
    assert torch.equal(mat, mat.transpose(1, 2))
    assert torch.equal(_acc(x, particle, disp, w, n_up, n_dn, K), got)
    from fermiflow_b200.observables import density_matrix_accumulate
    twice = density_matrix_accumulate(x, particle, disp, w, n_up, n_dn, K, got.clone())
    assert torch.equal(twice[-3:], 2 * got[-3:])


# ---- determinant identity ----------------------------------------------------------------------------------------

def _slater_rel_sv(x, model):
    """Smallest relative singular value of the two spin blocks of Phi at x [B, n, 2]."""
    rows = model._orb(x.device).long()
    allv = _orbitals(x, 36)
    rel = torch.ones(x.shape[0], device=x.device)
    for lo, hi in ((0, model.nup), (model.nup, model.nup + model.ndown)):
        if hi > lo:
            sv = torch.linalg.svdvals(allv[:, lo:hi][..., rows[lo:hi]])
            rel = torch.minimum(rel, sv[:, -1] / sv[:, 0])
    return rel


@pytest.mark.parametrize("nup,ndn", [(3, 3), (6, 6), (4, 2), (10, 10)])
def test_determinant_identity_exact(dev, nup, ndn):
    """Identity flow, psi = det Phi_up det Phi_dn.  Every particle of a walker moves to one shared r' (M = n records);
    then sum_{i in c} phi_a(r_i) psi(r_i -> r') / psi = phi_a(r') for every occupied a, and the occupied x occupied
    block of the sums is exactly sum over walkers of phi_a(r') phi_b(r') / q(r').  Walkers whose Slater matrices are
    ill-conditioned are given an invalid particle index, which the kernel skips."""
    from fermiflow_b200.observables import density_matrix_accumulate, density_matrix_layout
    model = _gs_model(dev, nup, ndn, zero=True)
    n, B, sigma = nup + ndn, 512, 1.5
    x = _walkers(model, B, dev)
    g = torch.Generator(device=dev).manual_seed(nup * 17 + ndn)
    rp = sigma * torch.randn(B, 1, 2, device=dev, generator=g)
    particle = torch.arange(n, device=dev, dtype=torch.int32).expand(B, n).contiguous()
    disp = (rp - x).contiguous()
    ratio = model.wavefunction_ratio(x, particle, disp)
    qv = torch.exp(-(rp * rp).sum(-1) / (2 * sigma ** 2)) / (2 * math.pi * sigma ** 2)        # [B, 1]
    w = ratio / qv
    keep = _slater_rel_sv(x, model) > 1e-3
    assert keep.float().mean() > 0.9
    particle = torch.where(keep[:, None], particle, torch.full_like(particle, -1))
    K = 36
    sums = density_matrix_accumulate(x, particle, disp, w, nup, ndn, K,
                                     torch.zeros(density_matrix_layout(K)[1], device=dev))
    assert float(sums[-1]) == n * int((~keep).sum())
    D = sums[:2 * K * K].view(2, K, K)
    _, mag = _acc_ref(x, particle, disp, w, nup, K)
    mag = mag[:2 * K * K].view(2, K, K)
    phi = _orbitals(rp[keep, 0], K) / qv[keep, 0].sqrt()[:, None]                               # [kept, K]
    exact = phi.T @ phi
    rows = model._orb(dev).long().tolist()
    worst = 0.0
    for c, occ in ((0, rows[:nup]), (1, rows[nup:])):
        if not occ:
            continue
        o = torch.tensor(occ, device=dev)
        got, ref, scale = D[c][o][:, o], exact[o][:, o], mag[c][o][:, o]
        err = ((got - ref).abs() / scale).max()
        worst = max(worst, float(err))
        assert err <= 1e-10, (c, float(err))
        assert float(((got - ref).abs() / ref.abs().max()).max()) <= 1e-10
    print("%d + %d: occupied block matches to %.2e of sum |terms|" % (nup, ndn, worst))


# ---- estimator ---------------------------------------------------------------------------------------------------

def _estimate(model, walkers, batches, seed, dev, **kw):
    from fermiflow_b200 import DensityMatrixEstimator
    est = DensityMatrixEstimator(model.nup, model.ndown, device=dev, **kw)
    gen = torch.Generator(device=dev).manual_seed(seed)
    for _ in range(batches):
        est.accumulate(model, walkers(), generator=gen)
    return est.result()


# The noisy eigenvalues of an m-fold degenerate block spread over about sqrt(2 m) of their first-order errors, so the
# tests that check single occupations against their errors use small bases (m <= 6).  The weights rho / q have an
# infinite fourth moment (a walker near a node of psi gives rho ~ 1 / psi(x)), so the batch-means errors themselves
# scatter: 32 batches keep them steady, and the checks that take the maximum over every entry of D use 6 errors
# (ENTRY_Z); single occupations and traces use 5.
ENTRY_Z = 6

@pytest.mark.parametrize("nup,ndn,shells", [(3, 3, 2), (6, 0, 3)])
def test_determinant_occupations(dev, nup, ndn, shells):
    """Identity flow: occupations 1 for the n_c occupied orbitals and 0 for the rest and the trace n_c, within 5
    standard errors, and every entry of D equal to the projector on the occupied orbitals within ENTRY_Z."""
    model = _gs_model(dev, nup, ndn, zero=True)
    res = _estimate(model, lambda: _walkers(model, 65536, dev), 32, 5, dev, shells=shells)
    K = (shells + 1) * (shells + 2) // 2
    assert res["walkers"] == 32 * 65536 and res["calls"] == 32 and res["density_matrix"].shape == (2, K, K)
    for c, nc in enumerate((nup, ndn)):
        if nc == 0:
            assert (res["density_matrix"][c] == 0).all() and (res["occupations"][c] == 0).all()
            assert res["trace"][c] == 0
            continue
        exact = np.diag([1.0] * nc + [0.0] * (K - nc))
        z = np.abs(res["density_matrix"][c] - exact) / res["density_matrix_err"][c]
        assert z.max() < ENTRY_Z, (c, z.max())
        want = np.array([1.0] * nc + [0.0] * (K - nc))
        z = np.abs(res["occupations"][c] - want) / res["occupations_err"][c]
        assert z.max() < 5, (c, z.max(), res["occupations"][c], res["occupations_err"][c])
        assert abs(res["trace"][c] - nc) < 5 * res["trace_err"][c], (res["trace"][c], res["trace_err"][c])
        # the leading natural orbitals lie in the occupied shells
        top = int(res["orbital_quanta"][:nc].sum(1).max()) + 1
        assert (res["shell_weight"][c][:nc, :top].sum(-1) > 0.99).all()
        print("%d + %d, channel %d: occupations %s +- %s" % (nup, ndn, c, np.round(res["occupations"][c], 4),
                                                            np.round(res["occupations_err"][c], 4)))


def test_interacting_flow(dev):
    """Random backflow, Z = 2, 3 + 3: sigma = 1.0 and sigma = 2.0 agree within errors (the estimate does not depend on
    the proposal) and D_up = D_dn, entry by entry within ENTRY_Z errors; occupations in [-5 err, 1 + 5 err] and the
    trace at most n_c + 5 err.
    The two channels share the walkers and the split of the records between them, so their errors are correlated;
    err_up + err_dn bounds the error of their difference whatever the correlation."""
    model = _gs_model(dev, 3, 3, zero=False)
    res = [_estimate(model, lambda: _walkers(model, 65536, dev), 32, 11 + k, dev, shells=3, sigma=s)
           for k, s in enumerate((1.0, 2.0))]
    a, b = res
    z = np.abs(a["density_matrix"] - b["density_matrix"]) / np.hypot(a["density_matrix_err"], b["density_matrix_err"])
    assert z.max() < ENTRY_Z, z.max()
    for r in res:
        D, E = r["density_matrix"], r["density_matrix_err"]
        z = np.abs(D[0] - D[1]) / (E[0] + E[1])
        assert z.max() < ENTRY_Z, (r["sigma"], z.max(), np.unravel_index(z.argmax(), z.shape))
        occ, err = r["occupations"], r["occupations_err"]
        assert (occ >= -5 * err).all() and (occ <= 1 + 5 * err).all(), (occ, err)
        assert (r["trace"] <= 3 + 5 * r["trace_err"]).all(), (r["trace"], r["trace_err"])
        print("sigma %.1f: trace %s +- %s, occupations %s, median entry error %.3g"
              % (r["sigma"], r["trace"], r["trace_err"], np.round(occ[0], 4), np.median(E)))


def test_beta_vmc_mixture(dev):
    """Identity flow, BetaVMC at 6 + 0: D = sum_s p_s (projector on the occupied orbitals of state s) with p_s the
    softmax of log_state_weights, entry by entry within ENTRY_Z standard errors."""
    from fermiflow_b200 import HO2D, FreeFermion, BetaVMC, HO, CoulombPairPotential
    model = BetaVMC(0.5, 6, 0, 2.0, True, HO2D(), FreeFermion(dev), _cnf(dev, True), CoulombPairPotential(2.0),
                    sp_potential=HO()).to(dev)
    table = model._state_table(dev)
    assert table.shape[0] >= 3 and int(table.max()) < 36
    ff = FreeFermion(dev)

    def walkers():
        ws = model.sample_states(65536)
        return ff.sample_multstates(table, ws, (65536,), equilibrim_steps=2000)

    res = _estimate(model, walkers, 16, 3, dev, shells=7)
    p = torch.softmax(model.log_state_weights.detach(), 0).cpu()
    exact = torch.zeros(36, 36)
    for s, row in enumerate(table.cpu().tolist()):
        exact[row, row] += p[s]
    z = np.abs(res["density_matrix"][0] - exact.numpy()) / res["density_matrix_err"][0]
    assert z.max() < ENTRY_Z, z.max()
    assert (res["density_matrix"][1] == 0).all()
    assert abs(res["trace"][0] - 6) < 5 * res["trace_err"][0]
    print("BetaVMC 6 + 0: %d states, leading occupations %s" % (table.shape[0], np.round(res["occupations"][0][:8], 4)))


# ---- drivers ----------------------------------------------------------------------------------------------------

_KEYS = ("density_matrix", "density_matrix_err", "trace", "trace_err", "occupations", "occupations_err",
         "natural_orbitals", "shell_weight", "orbital_quanta", "walkers", "calls", "moves", "sigma", "n_up", "n_dn")


@pytest.mark.parametrize("driver,particles,nc", [("FermionHO2D", ["--nup", "2", "--ndown", "1"], (2, 1)),
                                                ("BetaFermionHO2D", ["--nup", "3", "--deltaE", "2.0", "--boltzmann"], (3, 0))])
def test_driver_writes_natural_orbitals(dev, tmp_path, driver, particles, nc):
    import importlib
    mod = importlib.import_module("fermiflow_b200." + driver)
    path = os.path.join(str(tmp_path), "no.npz")
    argv = particles + ["--Z", "2.0", "--batch", "4096", "--iternum", "3", "--nsteps", "4", "--Deta", "8", "--Dmu", "8",
                        "--natural-orbitals", path, "--natural-orbitals-batches", "4", "--natural-orbitals-shells", "3"]
    hist = mod.main(argv)
    assert len(hist) == 3
    res = dict(np.load(path))
    assert sorted(res) == sorted(_KEYS)
    assert res["walkers"] == 4 * 4096 and res["calls"] == 4 and res["moves"] == 8 and res["sigma"] == 1.5
    assert res["density_matrix"].shape == (2, 10, 10) and res["shell_weight"].shape == (2, 10, 4)
    assert np.isfinite(res["occupations"]).all() and np.isfinite(res["occupations_err"]).all()
    for c in (0, 1):
        assert abs(res["trace"][c] - nc[c]) < 0.2
