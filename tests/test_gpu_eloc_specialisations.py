"""Every compiled specialisation of the register-resident E_loc sweep (eloc5_kernel<N, MU>, ff_eloc5.cuh).

try_eloc_static (capi_eloc.cu) dispatches to eloc5_kernel<N, 1> for N = 6 ... 20 and to eloc5_kernel<N, 0> (no one-body
backflow, the reference drivers' --nomu) for N = 6, 12 and 20.  Each instantiation has its own geometry (row blocks,
worker warps, Gram work split, shared-memory layout, size of the table mirror; rotated warp roles of every other
co-resident CTA at five row blocks, N = 17 ... 20), so each one is tested on its own:
  * dispatch: the default path launches the sweep and a separate finale, one kernel more than the generic
    flow_kernel<MODE_ELOC> -- so every test below is provably about eloc5_kernel, and a silent fallback fails here;
  * the fp64 oracle: log p, its gradient and Laplacian, E_loc and the parameter gradient through the stash;
  * the generic kernel over spin splits and batch sizes (several walkers per CTA, two CTAs per SM) with one walker
    beyond the Taylor tables, and the kernel variants (no tables, no table mirror, CTA-synchronous finale);
  * excited occupations with orbitals of the highest shell, one row per walker, through the eloc5 finale."""
import pytest
import torch

pytestmark = pytest.mark.gpu

torch.set_default_dtype(torch.float64)
RTOL = 1e-10

# (N, one-body MLP) pairs with an eloc5_kernel instantiation (capi_eloc.cu try_eloc_static) ...
ELOC5 = [(n, True) for n in range(6, 21)] + [(6, False), (12, False), (20, False)]
# ... and neighbours without one, which run the generic flow_kernel<MODE_ELOC>
GENERIC = [(5, True), (21, True), (13, False)]


def _nid(n, mu):
    return "N%d" % n + ("" if mu else "-nomu")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def O():
    from oracle import fermiflow_oracle
    return fermiflow_oracle


def close(a, b, rtol=RTOL, atol=0.0):
    """max |a - b| <= atol + rtol max |b|, evaluated on the device of a (the stashes of a large batch are hundreds of MB)."""
    a = torch.as_tensor(a).detach()
    b = torch.as_tensor(b).detach().to(a.device)
    assert a.shape == b.shape, (a.shape, b.shape)
    err = float((a - b).abs().max()) if a.numel() else 0.0
    ref = float(b.abs().max()) if b.numel() else 0.0
    assert err <= atol + rtol * ref, (err, ref)


def rand_mlp(H, seed, scale, dev):
    from fermiflow_b200 import MLP
    gen = torch.Generator().manual_seed(seed)
    m = MLP(1, H)
    with torch.no_grad():
        m.fc1.weight.copy_(torch.randn(H, 1, generator=gen))
        m.fc1.bias.copy_(torch.randn(H, generator=gen))
        m.fc2.weight.copy_(scale * torch.randn(1, H, generator=gen))
    return m.to(dev)


def cpu_params(m):
    return tuple(t.cpu() for t in m.kernel_params())


def _model(dev, nup, ndn, H, Hm, scale, S):
    """GSVMC with random radial MLPs (eta: H hidden units, mu: Hm, none if Hm = 0); returns (model, eta, mu)."""
    from fermiflow_b200 import Backflow, CNF, HO2D, FreeFermion, GSVMC, HO, CoulombPairPotential
    eta = rand_mlp(H, 1, scale, dev)
    mu = rand_mlp(Hm, 2, scale, dev) if Hm else None
    cnf = CNF(Backflow(eta, mu=mu), (0.0, 1.0), nsteps=S)
    model = GSVMC(nup, ndn, HO2D(), FreeFermion(dev), cnf, CoulombPairPotential(2.0), sp_potential=HO()).to(dev)
    return model, eta, mu


def _launches(fn):
    from fermiflow_b200 import _lib as L
    c0 = L.lib().ff_launch_count()
    fn()
    return L.lib().ff_launch_count() - c0


# ---------------------------------------------------------------------------------------
DISPATCH = [(n, mu, True) for n, mu in ELOC5] + [(n, mu, False) for n, mu in GENERIC]


@pytest.mark.parametrize("n,mu,static", DISPATCH, ids=[_nid(n, mu) + ("-eloc5" if s else "-generic") for n, mu, s in DISPATCH])
def test_dispatch_runs_eloc5_where_instantiated(dev, n, mu, static):
    """One local_energy call launches the two kernels of the radial tables (build, check) and then either eloc5_kernel
    and its finale (4) or the generic flow_kernel<MODE_ELOC>, which does the finale inside its one launch (3).  The
    default path must take the first where an instantiation exists and the second elsewhere; option eloc_generic
    always takes the second.  A dispatch change or a silent fall-back (shared memory, occupancy) fails here."""
    from fermiflow_b200 import _lib as L
    model, _, _ = _model(dev, (n + 1) // 2, n // 2, 8, 6 if mu else 0, 0.05, 2)
    x = 0.9 * torch.randn(2, n, 2, device=dev)
    with L.options(eloc_generic=1):
        generic = _launches(lambda: model.local_energy(x))
    default = _launches(lambda: model.local_energy(x))
    assert (default, generic) == ((4, 3) if static else (3, 3)), (_nid(n, mu), default, generic)


# ---------------------------------------------------------------------------------------
def _eloc_and_gradients_vs_oracle(dev, O, nup, ndn, H, Hm, S, B):
    """E_loc sweep and the parameter gradient through its stash (_LogpFromSweep, as GSVMC.forward) against the oracle."""
    from fermiflow_b200.VMC import _LogpFromSweep
    from fermiflow_b200.flow import _flat_params
    n = nup + ndn
    ts = (0.0, 1.0)
    model, eta, mu = _model(dev, nup, ndn, H, Hm, 0.05, S)
    cnf = model.cnf
    gen = torch.Generator().manual_seed(5)
    z0 = 0.9 * torch.randn(B, n, 2, generator=gen)
    w = torch.randn(B, generator=gen) / B
    eta_c, mu_c = cpu_params(eta), (cpu_params(mu) if mu is not None else None)
    up, dn = list(range(nup)), list(range(ndn))

    x = cnf.generate(z0.to(dev))
    x_ref = O.cnf_generate(z0, eta_c, mu_c, ts, S)
    close(x, x_ref, 1e-12)
    r = model.local_energy(x, stash=True)
    ref = O.local_energy(x_ref, up, dn, eta_c, mu_c, ts, S, 2.0)
    for k in ("logp", "grad", "lap", "kinetic", "potential", "eloc"):
        try:
            close(getattr(r, k), ref[k])
        except AssertionError as e:
            raise AssertionError("%s: %s" % (k, e)) from None

    gref = O.weighted_logp_param_grad(x_ref, w, up, dn, eta_c, mu_c, ts, S)
    names = [eta.fc1.weight, eta.fc1.bias, eta.fc2.weight] + ([mu.fc1.weight, mu.fc1.bias, mu.fc2.weight] if mu else [])
    lp = _LogpFromSweep.apply(model, r, model._orb(dev), None, nup, ndn, *_flat_params(cnf.v))
    (lp * w.to(dev)).sum().backward()
    for p, gr in zip(names, gref):
        close(p.grad.reshape(-1), gr.reshape(-1), 1e-9, 1e-13)


@pytest.mark.parametrize("n,mu", ELOC5, ids=[_nid(*p) for p in ELOC5])
def test_eloc5_vs_oracle(dev, O, n, mu):
    """Every instantiation against the fp64 oracle (balanced split, 3 walkers, 3 RK4 steps) at the 1e-10 of the
    north star, and the parameter gradient of the backward sweep fed by eloc5_kernel's stash at 1e-9."""
    _eloc_and_gradients_vs_oracle(dev, O, (n + 1) // 2, n // 2, 12, 10 if mu else 0, 3, 3)


# ---------------------------------------------------------------------------------------
def _splits(n):
    out = []
    for s in (((n + 1) // 2, n // 2), (n, 0), (n - 1, 1), (n // 2, (n + 1) // 2)):
        if s not in out:
            out.append(s)
    return out


SPLITS = [(nup, ndn, mu) for n, mu in ELOC5 for nup, ndn in _splits(n)]
OUTPUTS = ("z", "delta_logp", "logp", "grad", "lap", "kinetic", "potential", "eloc")


def _variant_model(dev, nup, ndn, mu):
    """The benchmark's MLP width (50 hidden units), 4 RK4 steps, radial functions positive at large distances: the
    inverse flow then pulls a far particle of x in, so that its z stays where the Gaussian orbitals are representable
    (with the opposite sign it moves out by N f r: z ~ 160 for N = 20 and log p = -inf)."""
    model, eta, mu_ = _model(dev, nup, ndn, 50, 50 if mu else 0, 0.02, 4)
    with torch.no_grad():
        for m in (eta, mu_):
            if m is not None and float((m.fc2.weight[0] * (m.fc1.weight[:, 0] > 0)).sum()) < 0:
                m.fc2.weight.neg_()
    return model


def _walkers(model, large):
    """B = 1, or 16 walkers per SM + 37 (every CTA loops over several walkers; two resident CTAs per SM at five row
    blocks, so half of them run the rotated warp roles) with one particle of one walker moved 27 beyond the others in
    x: its pair distances lie beyond the Taylor tables (direct evaluation).  Returns x and the groups of walkers
    compared separately (the far walker's values are several times larger than the others')."""
    B = 16 * torch.cuda.get_device_properties(0).multi_processor_count + 37 if large else 1
    _, x = model.sample((B,))
    if not large:
        return x, {"walker": slice(None)}
    far = B // 2
    x = x.clone()
    x[far, 0, 0] = x[far, 1:, 0].max() + 27.0
    rest = torch.ones(B, dtype=torch.bool, device=x.device)
    rest[far] = False
    return x, {"walkers": rest, "far walker": slice(far, far + 1)}


def _agree(r, ref, groups, what):
    B = ref.logp.shape[0]
    for name, rows in groups.items():
        for k in OUTPUTS + ("stash.y", "stash.c"):
            try:
                if k.startswith("stash"):
                    a, b = (getattr(t.stash, k[6:]).view(B, -1)[rows] for t in (r, ref))
                    close(a, b, *((1e-13,) if k == "stash.y" else (1e-12, 1e-14)))
                else:
                    assert torch.isfinite(getattr(ref, k)[rows]).all(), "non-finite reference"
                    close(getattr(r, k)[rows], getattr(ref, k)[rows], 1e-11, 1e-12)
            except AssertionError as e:
                raise AssertionError("%s, %s, %s: %s" % (what, name, k, e)) from None


@pytest.mark.parametrize("large", [False, True], ids=["B1", "Bmany"])
@pytest.mark.parametrize("nup,ndn,mu", SPLITS, ids=["%d+%d%s" % (u, d, "" if m else "-nomu") for u, d, m in SPLITS])
def test_eloc5_matches_generic(dev, nup, ndn, mu, large):
    """eloc5_kernel against the generic flow_kernel<MODE_ELOC> (option eloc_generic) at every instantiation, for the
    spin splits (ceil(N/2), floor(N/2)), (N, 0), (N - 1, 1) and (floor(N/2), ceil(N/2)): every output and the stash."""
    from fermiflow_b200 import _lib as L
    model = _variant_model(dev, nup, ndn, mu)
    x, groups = _walkers(model, large)
    with L.options(eloc_generic=1):
        ref = model.local_energy(x, stash=True)
    r = model.local_energy(x, stash=True)
    _agree(r, ref, groups, "eloc5 against generic")


@pytest.mark.parametrize("n,mu", ELOC5, ids=[_nid(*p) for p in ELOC5])
def test_eloc5_generic_and_direct_paths_agree(dev, n, mu):
    """The kernel variants at every instantiation (balanced split, the large batch with the far walker): eloc5_kernel
    with the Taylor tables (default) against the generic kernel with and without tables and eloc5_kernel evaluating
    every hidden unit (no_table)."""
    from fermiflow_b200 import _lib as L
    model = _variant_model(dev, (n + 1) // 2, n // 2, mu)
    x, groups = _walkers(model, True)
    r0 = model.local_energy(x, stash=True)
    for env in (dict(eloc_generic=1), dict(eloc_generic=1, no_table=1), dict(no_table=1)):
        with L.options(**env):
            r = model.local_energy(x, stash=True)
        _agree(r, r0, groups, str(env))


# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("nup,ndn", [(5, 3), (8, 0)])
def test_eloc5_warp_finale_excited_high_shell_occupations(dev, O, nup, ndn):
    """eloc5_kernel<8, 1> with a hand-made int32 occupation table and one row per walker (walker_state), passed to the
    sweep helper GSVMC.local_energy calls: orbitals up to index 35, i.e. nx or ny = 7, the top of the 8-entry Hermite
    recursion of the finale (eloc_finale_warp_kernel).  Against the oracle with the same occupation rows."""
    from fermiflow_b200.utils import eloc_sweep
    n, S, B = nup + ndn, 3, 12
    rows = {(5, 3): [(0, 1, 2, 3, 4, 0, 1, 2),
                     (0, 7, 20, 28, 35, 1, 27, 35),            # 28: (nx, ny) = (0, 7), 35: (7, 0), 27: (6, 0)
                     (3, 14, 29, 34, 35, 28, 31, 33),
                     (1, 2, 5, 9, 30, 0, 4, 32)],
            (8, 0): [(0, 1, 2, 3, 4, 5, 6, 7),
                     (0, 2, 7, 20, 28, 31, 34, 35),
                     (1, 4, 12, 21, 27, 28, 29, 35),
                     (3, 5, 8, 16, 24, 30, 32, 33)]}[(nup, ndn)]
    table = torch.tensor(rows, dtype=torch.int32, device=dev)
    model, eta, mu = _model(dev, nup, ndn, 12, 10, 0.05, S)
    gen = torch.Generator().manual_seed(9)
    ws = torch.randperm(B, generator=gen) % len(rows)
    assert set(ws.tolist()) == set(range(len(rows)))
    ws = ws.to(torch.int32).to(dev)
    x = model.cnf.generate(1.3 * torch.randn(B, n, 2, generator=gen).to(dev))
    occ = table[ws.long()].cpu().long()                                  # (B, n) HO2D orbital ids per walker
    ref = O.local_energy(x.cpu(), occ[:, :nup], occ[:, nup:], cpu_params(eta), cpu_params(mu), (0.0, 1.0), S, 2.0)
    r = eloc_sweep(model.cnf, x, table, ws, nup, model._Z, model._harmonic)
    for k in ("logp", "grad", "lap", "kinetic", "potential", "eloc"):
        try:
            close(getattr(r, k), ref[k])
        except AssertionError as e:
            raise AssertionError("%s: %s" % (k, e)) from None
