"""GPU tests of the replica swap ratios (C ABI ff_swap_ratio, GSVMC / BetaVMC.swap_ratio) and of the Rényi estimator
(ff_swap_accumulate, fermiflow_b200.observables.RenyiEstimator): ratios against the fp64 oracle with the swapped
configurations built by a torch restatement, identities that hold for any flow, the accumulation against a torch
restatement, the exact free-fermion Tr ρ_A² and its sectors, the purity of a mixed state with sorted walker states,
and the --renyi option of the ground-state driver."""
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


def _pairs(B, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    return torch.randperm(B, device=dev, generator=g)[:2 * (B // 2)].view(-1, 2).to(torch.int32)


# ---- torch restatement of the swapped configurations, and the fp64 oracle ---------------------------------------

def _inside(r, a, kind):
    """membership with every product and sum rounded separately, as the kernel decides it (CPU float64)."""
    if kind == "disk":
        return r[..., 0] * r[..., 0] + r[..., 1] * r[..., 1] < a * a
    return r[..., 0] < a


def _swap_ref(x, pairs, a, kind, nup):
    """sector [P, 2, Q] and {(p, q): (x', y')} for the matched records: the k-th A-particle of one side, in increasing
    particle index within its spin block, takes the position of the k-th A-particle of the other side."""
    x, pairs = x.cpu(), pairs.long().cpu()
    n = x.shape[1]
    xs = x[pairs]                                                              # [P, 2, n, 2]
    ins = torch.stack([_inside(xs, float(aq), kind) for aq in a], -1)           # [P, 2, n, Q]
    sector = (ins[:, :, :nup].sum(2) * (n - nup + 1) + ins[:, :, nup:].sum(2)).to(torch.int32)
    swapped = {}
    for p in range(pairs.shape[0]):
        for q in range(len(a)):
            if sector[p, 0, q] != sector[p, 1, q]:
                continue
            out = []
            for s in (0, 1):
                w, v = xs[p, s].clone(), xs[p, 1 - s]
                for lo, hi in ((0, nup), (nup, n)):
                    iw = torch.tensor([i for i in range(lo, hi) if ins[p, s, i, q]], dtype=torch.long)
                    iv = torch.tensor([i for i in range(lo, hi) if ins[p, 1 - s, i, q]], dtype=torch.long)
                    w[iw] = v[iv]
                out.append(w)
            swapped[(p, q)] = out
    return sector, swapped


def _slater_sign_log(z, rows, nup):
    """sign, log|det| and the smallest relative singular value of each spin block at z [C, n, 2]; rows [C, n]."""
    from oracle import fermiflow_oracle as O
    allv = torch.stack([O.ho2d_orbital(k, z) for k in range(len(O.HO2D_QUANTA))], -1)
    sign, logabs, rel = torch.ones(z.shape[0]), torch.zeros(z.shape[0]), torch.ones(z.shape[0])
    for lo, hi in ((0, nup), (nup, z.shape[1])):
        if hi == lo:
            continue
        D = torch.gather(allv[:, lo:hi, :], 2, rows[:, None, lo:hi].expand(-1, hi - lo, -1))
        s, la = torch.linalg.slogdet(D)
        sv = torch.linalg.svdvals(D)
        sign, logabs = sign * s, logabs + la
        rel = torch.minimum(rel, sv[:, -1] / sv[:, 0])
    return sign, logabs, rel


def _oracle_swap(cnf, x, pairs, a, kind, rows, nup):
    """ratio [P, Q], sector [P, 2, Q] and the node measure of every record (fp64 flow and slogdet on the CPU)."""
    from oracle import fermiflow_oracle as O
    sector, swapped = _swap_ref(x, pairs, a, kind, nup)
    x, pairs, rows = x.cpu(), pairs.long().cpu(), rows.long().cpu()
    P, n, Q = pairs.shape[0], x.shape[1], len(a)
    keys = sorted(swapped)
    conf = [x[pairs.reshape(-1)]] + [torch.stack(swapped[k]) for k in keys]
    crow = [rows[pairs.reshape(-1)]] + [rows[pairs[p]] for p, _ in keys]
    X, Rw = torch.cat(conf), torch.cat(crow)
    pe = tuple(t.cpu() for t in cnf.v.eta.kernel_params())
    pm = tuple(t.cpu() for t in cnf.v.mu.kernel_params())
    z, dl = O.cnf_delta_logp(X, pe, pm, cnf.t_span, cnf.nsteps)
    sign, logabs, rel = _slater_sign_log(z, Rw, nup)
    lp = 2 * logabs - dl
    ratio = torch.zeros(P, Q)
    near = torch.ones(P, Q)
    for j, (p, q) in enumerate(keys):
        b0, b1, s0, s1 = 2 * p, 2 * p + 1, 2 * P + 2 * j, 2 * P + 2 * j + 1
        e = (lp[s0] + lp[s1]) - (lp[b0] + lp[b1])
        ratio[p, q] = sign[s0] * sign[s1] * sign[b0] * sign[b1] * torch.exp(0.5 * e)
        near[p, q] = min(rel[b0], rel[b1], rel[s0], rel[s1])
    return ratio, sector, near


def _regions(x, kind, fracs):
    """region parameters holding about fracs of the particles: quantiles of |r| (disks) or x (half-planes)."""
    v = x[..., 0] if kind == "halfplane" else (x * x).sum(-1).sqrt()
    return [float(t) for t in torch.quantile(v.reshape(-1).cpu(), torch.tensor(fracs))]


def _check_parity(model, x, pairs, rows, nup, n, swap=None):
    """ratios and sectors of swap (default model.swap_ratio) against the oracle for disks and half-planes; returns the
    oracle ratios of the records that swap at least one particle."""
    swap = model.swap_ratio if swap is None else swap
    fracs = [min(0.5, f / n) for f in (1.5, 2.5, 4.0)]
    pooled = []
    for kind in ("disk", "halfplane"):
        a = _regions(x, kind, fracs)
        got, gsec = swap(x, pairs, a, kind)
        assert got.shape == (pairs.shape[0], 3) and gsec.shape == (pairs.shape[0], 2, 3) and gsec.dtype == torch.int32
        ref, rsec, near = _oracle_swap(model.cnf, x, pairs, a, kind, rows, nup)
        got, gsec = got.cpu(), gsec.cpu()
        assert torch.equal(gsec, rsec)
        matched = rsec[:, 0] == rsec[:, 1]
        assert (got[~matched] == 0).all()                               # exactly 0, not merely small
        assert (got[matched & (rsec[:, 0] == 0)] == 1).all()
        live = matched & (rsec[:, 0] > 0)
        g, r, nr = got[live], ref[live], near[live]
        assert torch.isfinite(g).all()
        rel = (g.abs() - r.abs()).abs() / r.abs()
        assert rel.max() <= 1e-10, (kind, float(rel.max()))
        far = nr > 1e-8
        assert torch.equal(torch.sign(g)[far], torch.sign(r)[far])
        pooled.append(r)
    r = torch.cat(pooled)
    assert r.numel() >= 12, r.numel()
    assert (r < 0).float().mean() >= 0.1, float((r < 0).float().mean())
    return r


@pytest.mark.parametrize("nup,ndn", [(3, 3), (7, 6), (10, 10), (12, 0), (18, 0)])
def test_swap_ratio_parity_oracle(dev, nup, ndn):
    """Ratios against the fp64 oracle, sectors equal to the restatement, mismatched pairs exactly 0; 18 + 0 takes the
    CTA Slater path."""
    model = _gs_model(dev, nup, ndn)
    B = 48
    _, x = model.sample((B,))
    pairs = _pairs(B, dev, seed=nup * 31 + ndn)
    rows = model._orb(dev)[None].expand(B, -1)
    _check_parity(model, x, pairs, rows, nup, nup + ndn)


@pytest.mark.parametrize("nup,ndn", [(6, 0), (3, 2)])
def test_swap_ratio_parity_beta_vmc(dev, nup, ndn):
    """Occupation mixtures: each replica is evaluated with its own occupation row, and the two sides of a pair sit in
    different states.  6 + 0 goes through BetaVMC.swap_ratio.  BetaVMC builds spin-polarised states only, so 3 + 2
    passes a hand-made table of four spinful rows, sorted over the walkers, to the helper both models share."""
    B = 48
    if ndn == 0:
        model = _beta_model(dev, nup, ndn)
        _, x = model.sample((B,))
        ws = model.state_indices
        table, swap = model._state_table(dev), None
    else:
        from fermiflow_b200 import HO2D
        from fermiflow_b200.base_dist import _state_table
        from fermiflow_b200.VMC import _swap_ratio
        model = _gs_model(dev, nup, ndn)
        _, x = model.sample((B,))
        o = HO2D().orbitals
        table = _state_table([((o[0], o[1], o[2]), (o[0], o[1])), ((o[0], o[1], o[3]), (o[0], o[2])),
                              ((o[0], o[2], o[4]), (o[0], o[1])), ((o[1], o[2], o[3]), (o[0], o[3]))], dev)
        ws = (torch.arange(B, device=dev) * 4 // B).to(torch.int32)

        def swap(x, pairs, a, kind):
            return _swap_ratio(model.cnf, x, table, ws, nup, pairs, a, kind)
    assert len(set(ws.tolist())) >= 2
    pairs = _pairs(B, dev, seed=3 + nup)
    assert (ws[pairs[:, 0].long()] != ws[pairs[:, 1].long()]).any()
    rows = table[ws.long()]
    _check_parity(model, x, pairs, rows, nup, nup + ndn, swap=swap)
    if ndn == 0:
        a = [0.8, 1.5]
        got = model.swap_ratio(x, pairs, a)
        assert all(torch.equal(u, v) for u, v in zip(model.swap_ratio(x, pairs, a, walker_state=ws), got))
        with pytest.raises(ValueError):
            model.swap_ratio(x, pairs, a, walker_state=ws[:-1])


@pytest.mark.parametrize("nup,ndn", [(3, 3), (10, 10), (12, 0)])
def test_swap_identities(dev, nup, ndn):
    """Any flow: empty regions give exactly 1 and sector 0; the whole plane swaps the walkers (ratio 1 to 1e-12,
    sector (n_up, n_dn)); a walker index outside [0, B) gives NaN and sector -1 for that pair only."""
    model = _gs_model(dev, nup, ndn)
    B = 256
    _, x = model.sample((B,))
    pairs = _pairs(B, dev, seed=17)
    for a, kind in (([0.0, 0.0], "disk"), ([-1e3], "halfplane")):
        r, s = model.swap_ratio(x, pairs, a, kind)
        assert (r == 1.0).all() and (s == 0).all()
    r, s = model.swap_ratio(x, pairs, [1e3], "disk")
    assert (r - 1).abs().max() <= 1e-12, float((r - 1).abs().max())
    assert (s == nup * (ndn + 1) + ndn).all()
    r, s = model.swap_ratio(x, pairs, [1e3], "halfplane")
    assert (r - 1).abs().max() <= 1e-12 and (s == nup * (ndn + 1) + ndn).all()
    bad = pairs.clone()
    bad[0, 1], bad[5, 0], bad[9, 1] = -1, B, 1 << 30
    a = [0.0, 1.0, 1e3]
    r, s = model.swap_ratio(x, bad, a)
    r0, s0 = model.swap_ratio(x, pairs, a)
    hit = torch.zeros(pairs.shape[0], dtype=torch.bool, device=dev)
    hit[[0, 5, 9]] = True
    assert torch.isnan(r[hit]).all() and (s[hit] == -1).all()
    assert torch.isfinite(r[~hit]).all() and torch.equal(s[~hit], s0[~hit])


# ---- accumulation against a torch restatement -------------------------------------------------------------------

def _acc_ref(ratio, sector, n_up, n_dn):
    P, Q = ratio.shape
    ns = (n_up + 1) * (n_dn + 1)
    ratio, sector = ratio.cpu(), sector.long().cpu()
    s0, s1 = sector[:, 0], sector[:, 1]
    ok = (s0 >= 0) & (s0 < ns) & (s1 >= 0) & (s1 < ns)
    cell = torch.arange(Q)[None] * ns
    rep = torch.zeros(Q * ns)
    rep.index_add_(0, (cell + s0)[ok], torch.ones(int(ok.sum())))
    rep.index_add_(0, (cell + s1)[ok], torch.ones(int(ok.sum())))
    m = ok & (s0 == s1)
    rsum = torch.zeros(Q * ns).index_add_(0, (cell + s0)[m], ratio[m])
    mat = torch.zeros(Q * ns).index_add_(0, (cell + s0)[m], torch.ones(int(m.sum())))
    absum = torch.zeros(Q * ns).index_add_(0, (cell + s0)[m], ratio[m].abs())
    return torch.cat([rsum, rep, mat, (~ok).sum(0).double(), torch.tensor([float(P)])]), absum


@pytest.mark.parametrize("Q", [1, 32])
@pytest.mark.parametrize("P", [1, 37, 5000, 70001])
def test_accumulate_equals_torch(dev, P, Q):
    from fermiflow_b200.observables import swap_accumulate, swap_layout
    n_up, n_dn = 3, 2
    ns = (n_up + 1) * (n_dn + 1)
    g = torch.Generator(device=dev).manual_seed(P * 7 + Q)
    ratio = torch.randn(P, Q, device=dev, generator=g) * 3
    s0 = torch.randint(-2, ns + 2, (P, Q), device=dev, generator=g)            # some sectors outside [0, n_sec)
    other = torch.randint(-1, ns + 1, (P, Q), device=dev, generator=g)
    same = torch.rand(P, Q, device=dev, generator=g) < 0.5
    sector = torch.stack((s0, torch.where(same, s0, other)), 1).to(torch.int32)
    lay, n_sums = swap_layout(Q, n_up, n_dn)
    got = swap_accumulate(ratio, sector, n_up, n_dn, torch.zeros(n_sums, device=dev))
    ref, absum = _acc_ref(ratio, sector, n_up, n_dn)
    got_c = got.cpu()
    k = Q * ns
    assert torch.equal(got_c[k:], ref[k:])                                     # counts exactly
    assert ((got_c[:k] - ref[:k]).abs() <= 1e-12 * absum.clamp_min(1e-300)).all()
    # two calls: bit-identical; a second call adds
    assert torch.equal(swap_accumulate(ratio, sector, n_up, n_dn, torch.zeros(n_sums, device=dev)), got)
    twice = swap_accumulate(ratio, sector, n_up, n_dn, got.clone())
    assert torch.equal(twice[k:], 2 * got[k:])


# ---- exact free-fermion values -----------------------------------------------------------------------------------

def _overlap(ids, a, kind):
    """O_kl = ∫_A φ_k φ_l of the HO2D orbitals ids: polar Gauss-Legendre on a disk, a 1D integral in x on a
    half-plane (the y factors are orthonormal)."""
    from oracle import fermiflow_oracle as O
    if kind == "disk":
        gx, gw = np.polynomial.legendre.leggauss(64)
        r, wr = 0.5 * a * (gx + 1), 0.5 * a * gw
        th = 2 * np.pi * (np.arange(128) + 0.5) / 128
        pts = torch.from_numpy(np.stack([r[:, None] * np.cos(th), r[:, None] * np.sin(th)], -1))
        phi = np.stack([O.ho2d_orbital(k, pts).numpy() for k in ids])          # [m, 64, 128]
        w = (wr * r)[:, None] * (2 * np.pi / 128)
        return np.einsum("kij,lij,ij->kl", phi, phi, w)
    lo = -12.0
    gx, gw = np.polynomial.legendre.leggauss(200)
    xs, w = lo + 0.5 * (a - lo) * (gx + 1), 0.5 * (a - lo) * gw
    t = torch.from_numpy(xs)

    def psi(nq):
        return (math.pi ** -0.25 * torch.exp(-0.5 * t * t) * O.hermite_fn(nq, t)).numpy()

    q = [O.HO2D_QUANTA[k] for k in ids]
    return np.array([[(psi(qk[0]) * psi(ql[0]) * w).sum() if qk[1] == ql[1] else 0.0 for ql in q] for qk in q])


def _free_exact(ids_up, ids_dn, a, kind):
    """Tr ρ_A², P(a, b) and Tr ρ_ab² of free fermions from the eigenvalues λ of the overlap matrices:
    Π(1 − λ + λ t) and Π((1 − λ)² + λ² t) generate P and Tr ρ² by particle number."""
    polys = []
    for ids in (ids_up, ids_dn):
        lam = np.linalg.eigvalsh(_overlap(ids, a, kind)) if ids else np.zeros(0)
        p, s = np.ones(1), np.ones(1)
        for v in lam:
            p = np.polynomial.polynomial.polymul(p, [1 - v, v])
            s = np.polynomial.polynomial.polymul(s, [(1 - v) ** 2, v * v])
        polys.append((p, s))
    (pu, su), (pd, sd) = polys
    return su.sum() * sd.sum(), np.outer(pu, pd), np.outer(su, sd)


def _check_free(res, ids_up, ids_dn):
    for q, (a, kind) in enumerate(zip(res["a"], [str(res["kind"])] * len(res["a"]))):
        swap, prob, ss = _free_exact(ids_up, ids_dn, float(a), kind)
        z = abs(res["swap"][q] - swap) / res["swap_err"][q]
        assert z < 5, (kind, a, res["swap"][q], swap, z)
        big = prob > 0.01
        assert big.any()
        z = np.abs(res["sector_prob"][q] - prob)[big] / res["sector_prob_err"][q][big]
        assert z.max() < 5, (kind, a, z.max())
        z = np.abs(res["sector_swap"][q] - ss)[big] / res["sector_swap_err"][q][big]
        assert z.max() < 5, (kind, a, z.max())
        print("%s a = %g: swap %.5g +- %.2g (exact %.5g), S2 %.4g" % (kind, a, res["swap"][q], res["swap_err"][q], swap,
                                                                     -math.log(swap)))


@pytest.mark.parametrize("nup,a,kind", [(3, (0.5, 1.0, 1.5, 2.5), "disk"), (3, (-1.0, -0.3), "halfplane"),
                                        (6, (0.6, 1.0), "disk")])
def test_free_fermion_renyi(dev, nup, a, kind):
    """Identity flow, nup + nup free fermions in the lowest HO2D orbitals: Tr ρ_A², P(a, b) and Tr ρ_ab² within 5
    standard errors of the values from the overlap eigenvalues."""
    from fermiflow_b200 import FreeFermion, HO2D, RenyiEstimator
    occ = HO2D().orbitals[:nup]
    model = _gs_model(dev, nup, nup, zero=True)
    ff = FreeFermion(dev)
    est = RenyiEstimator(nup, nup, a=a, kind=kind, device=dev)
    gen = torch.Generator(device=dev).manual_seed(11 + nup)
    for _ in range(24):
        est.accumulate(model, ff.sample(occ, occ, (65536,), equilibrim_steps=2000), generator=gen)
    res = est.result()
    assert res["pairs"] == 24 * 32768 and res["calls"] == 24
    assert res["sector_prob"].shape == (len(a), nup + 1, nup + 1)
    np.testing.assert_allclose(res["sector_prob"].sum((1, 2)), 1.0, rtol=1e-12)
    np.testing.assert_allclose(res["sector_swap"].sum((1, 2)), res["swap"], rtol=1e-10, atol=1e-14)
    ids = list(range(nup))
    _check_free(res, ids, ids)


def test_mixed_state_purity_with_sorted_states(dev):
    """BetaVMC, identity flow, walker states SORTED over S = 4 rows (as ff_occupation_sample returns them): the
    whole-plane swap estimates the purity Σ p_s² = 1/4 only because the estimator pairs the walkers at random
    (pairing neighbours would give about 1)."""
    from fermiflow_b200 import FreeFermion, RenyiEstimator
    model = _beta_model(dev, 4, 0, zero=True)
    table = model._state_table(dev)
    S = 4
    assert table.shape[0] >= S
    ff = FreeFermion(dev)
    B = 65536
    ws = (torch.arange(B, device=dev) * S // B).to(torch.int32)
    model.state_indices = ws
    est = RenyiEstimator(4, 0, a=(1e3,), device=dev)
    for _ in range(16):
        est.accumulate(model, ff.sample_multstates(table, ws, (B,), equilibrim_steps=2000))
    res = est.result()
    z = abs(res["swap"][0] - 0.25) / res["swap_err"][0]
    print("purity: %.5g +- %.2g (exact 0.25)" % (res["swap"][0], res["swap_err"][0]))
    assert z < 5, (res["swap"][0], res["swap_err"][0])
    assert res["sector_prob"][0, 4, 0] == 1.0


def test_ground_state_driver_writes_renyi(dev, tmp_path):
    from fermiflow_b200 import FermionHO2D
    path = os.path.join(str(tmp_path), "renyi.npz")
    hist = FermionHO2D.main(["--nup", "2", "--ndown", "1", "--Z", "2.0", "--batch", "4096", "--iternum", "3",
                             "--nsteps", "4", "--Deta", "8", "--Dmu", "8", "--renyi", path, "--renyi-batches", "8",
                             "--renyi-a", "0.5,1.0,2.0"])
    assert len(hist) == 3
    res = dict(np.load(path))
    for k in ("swap", "swap_err", "S2", "S2_err", "sector_prob", "sector_prob_err", "sector_swap", "sector_swap_err",
              "S2_sector", "S2_sector_err", "a", "kind", "pairs", "calls", "n_up", "n_dn"):
        assert k in res, k
    assert res["pairs"] == 8 * 2048 and res["calls"] == 8 and str(res["kind"]) == "disk"
    assert res["sector_prob"].shape == (3, 3, 2) and np.allclose(res["a"], [0.5, 1.0, 2.0])
    assert np.isfinite(res["S2"][:2]).all() and np.isfinite(res["S2_err"][:2]).all()
    assert (res["S2"][:2] > 0).all() and res["S2"][0] < res["S2"][1]
