"""GPU tests of the walker histograms (C ABI ff_observables, fermiflow_b200.observables.DensityEstimator): exact counts
against a torch restatement of the binning rule, edge cases, accumulation beyond 2^32 in one bin, the free-fermion
density, and the --density option of the ground-state driver."""
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


# ---- oracle: the binning rule of include/fermiflow_b200.h restated in torch, same operation order ----------------

def _bin(v, lo, s, nb):
    f = ((v - lo) * s).floor()
    ok = (f >= 0) & (f < nb)
    return torch.where(ok, f, torch.zeros_like(f)).long(), ok


def _hist(key, ok, ch, nch, cells):
    """(bins [nch * cells], outside [nch]) from flat in-channel bin keys; a section with 0 bins counts nothing."""
    if cells == 0:
        return key.new_zeros(0), key.new_zeros(nch)
    bins = torch.bincount((ch * cells + key)[ok], minlength=nch * cells)
    outside = torch.bincount(ch[~ok], minlength=nch)
    return bins, outside


def _oracle_chunk(x, n_up, extent, n_xy, r_max, n_r, n_rot):
    dev = x.device
    B, n, _ = x.shape
    spin = (torch.arange(n, device=dev) >= n_up).long()
    parts, outs = [], []
    # density
    sx = n_xy / (2.0 * extent)
    kx, okx = _bin(x[..., 0], -extent, sx, n_xy)
    ky, oky = _bin(x[..., 1], -extent, sx, n_xy)
    b, o = _hist(kx * n_xy + ky, okx & oky, spin.expand(B, n), 2, n_xy * n_xy)
    parts.append(b); outs.append(o)
    # radial
    sr = n_r / r_max if n_r else 0.0
    r = (x[..., 0] * x[..., 0] + x[..., 1] * x[..., 1]).sqrt()
    k, ok = _bin(r, 0.0, sr, n_r)
    b, o = _hist(k, ok, spin.expand(B, n), 2, n_r)
    parts.append(b); outs.append(o)
    # separation, i < j
    i, j = torch.triu_indices(n, n, 1, device=dev)
    dx = x[:, i, 0] - x[:, j, 0]
    dy = x[:, i, 1] - x[:, j, 1]
    d = (dx * dx + dy * dy).sqrt()
    ch = torch.where(spin[i] == spin[j], spin[i], torch.full_like(spin[i], 2))
    k, ok = _bin(d, 0.0, sr, n_r)
    b, o = _hist(k, ok, ch.expand(B, -1), 3, n_r)
    parts.append(b); outs.append(o)
    # rotated frame, i != j
    ii, jj = torch.meshgrid(torch.arange(n, device=dev), torch.arange(n, device=dev), indexing="ij")
    m = ii != jj
    i, j = ii[m], jj[m]
    xi, yi, xj, yj = x[:, i, 0], x[:, i, 1], x[:, j, 0], x[:, j, 1]
    ni = (xi * xi + yi * yi).sqrt()
    u = (xi * xj + yi * yj) / ni
    w = (xi * yj - yi * xj) / ni
    sq = n_rot / (2.0 * extent)
    ku, oku = _bin(u, -extent, sq, n_rot)
    kw, okw = _bin(w, -extent, sq, n_rot)
    ch = (spin[i] != spin[j]).long()
    b, o = _hist(ku * n_rot + kw, oku & okw & (ni != 0), ch.expand(B, -1), 2, n_rot * n_rot)
    parts.append(b); outs.append(o)
    return torch.cat(parts + outs)


def oracle(x, n_up, extent, n_xy, r_max, n_r, n_rot, chunk=4096):
    tot = None
    for c in range(0, x.shape[0], chunk):
        h = _oracle_chunk(x[c:c + chunk], n_up, extent, n_xy, r_max, n_r, n_rot)
        tot = h if tot is None else tot + h
    if tot is None:
        tot = _oracle_chunk(x[:0], n_up, extent, n_xy, r_max, n_r, n_rot)
    return tot


def counts_of(x, n_up, n_dn, extent, n_xy, r_max, n_r, n_rot, into=None):
    from fermiflow_b200.observables import count_layout, observables
    if into is None:
        _, nb = count_layout(n_xy, n_r, n_rot)
        into = torch.zeros(nb + 9, dtype=torch.int64, device=x.device)
    return observables(x, n_up, n_dn, extent, n_xy, r_max, n_r, n_rot, into)


def _walkers(B, n, dev, seed, scale=1.3):
    """Gaussian walkers, wide enough that some fall outside both grids (extent 2.5 and r_max 2.0 below)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    return scale * torch.randn(B, n, 2, device=dev, generator=g)


GRID = dict(extent=2.5, n_xy=16, r_max=2.0, n_r=24, n_rot=20)


@pytest.mark.parametrize("n_up,n_dn", [(3, 3), (2, 1), (12, 0), (1, 0), (10, 10)])
@pytest.mark.parametrize("B", [1, 7, 1000, 65536])
def test_counts_equal_oracle(dev, n_up, n_dn, B):
    x = _walkers(B, n_up + n_dn, dev, seed=B + 31 * n_up + n_dn)
    got = counts_of(x, n_up, n_dn, **GRID)
    ref = oracle(x if B > 256 else x.cpu(), n_up, **GRID).to(dev)
    assert torch.equal(got, ref)
    outside = got[-9:]
    if B >= 1000:                                                      # walkers beyond both grids occur
        assert outside[0] > 0 and outside[2] > 0
        assert n_up + n_dn == 1 or outside[-2:].sum() > 0


def test_sections_too_big_for_one_launch(dev):
    """128 x 128 density and rotated grids are 128 KB each: one launch per section."""
    from fermiflow_b200 import _lib as L
    before = L.lib().ff_launch_count()
    x = _walkers(4096, 6, dev, seed=3)
    grid = dict(extent=3.0, n_xy=128, r_max=3.0, n_r=64, n_rot=128)
    got = counts_of(x, 3, 3, **grid)
    assert L.lib().ff_launch_count() - before == 4
    assert torch.equal(got, oracle(x, 3, **grid))
    before = L.lib().ff_launch_count()
    counts_of(x, 3, 3, **GRID)
    assert L.lib().ff_launch_count() - before == 1


def test_sections_switched_off(dev):
    x = _walkers(500, 5, dev, seed=4)
    for grid in (dict(extent=2.5, n_xy=0, r_max=2.0, n_r=24, n_rot=20), dict(extent=2.5, n_xy=16, r_max=2.0, n_r=0, n_rot=0),
                 dict(extent=2.5, n_xy=0, r_max=2.0, n_r=24, n_rot=0)):
        assert torch.equal(counts_of(x, 2, 3, **grid), oracle(x, 2, **grid))


def test_edges_nonfinite_and_origin(dev):
    """Coordinates on bin edges, at +extent and r_max (outside), at -extent (bin 0); NaN and +-inf; a particle at the
    origin (outside of the rotated section as a reference particle)."""
    e, r_max = 2.0, 1.5
    grid = dict(extent=e, n_xy=8, r_max=r_max, n_r=6, n_rot=8)
    pts = [(-e, -e), (e, 0.0), (0.0, e), (-e, 0.5), (0.5, 0.25), (r_max, 0.0), (0.0, -r_max), (0.0, 0.0),
           (float("nan"), 0.0), (0.0, float("inf")), (float("-inf"), 1.0), (1.0, 1.0), (-0.5, 0.75), (0.25, -1.75)]
    g = torch.Generator().manual_seed(11)
    rows = []
    for _ in range(64):
        idx = torch.randint(len(pts), (4,), generator=g)
        rows.append([pts[int(k)] for k in idx])
    x = torch.tensor(rows).to(dev)
    got = counts_of(x, 2, 2, **grid)
    ref = oracle(x.cpu(), 2, **grid).to(dev)
    assert torch.equal(got, ref)
    # the rule itself on one walker: -extent is bin 0, +extent is outside, the origin is outside as a reference
    one = torch.tensor([[[-e, -e], [e, 0.0]]], device=dev)
    c = counts_of(one, 2, 0, **grid)
    assert int(c[0]) == 1 and int(c[-9]) == 1
    origin = torch.tensor([[[0.0, 0.0], [0.5, 0.5]]], device=dev)
    c = counts_of(origin, 1, 1, **grid)
    assert int(c[-1]) == 1                                         # (origin -> other) is outside, the reverse is not


def test_accumulation_determinism_and_empty_batch(dev):
    x = _walkers(20000, 6, dev, seed=5)
    whole = counts_of(x, 3, 3, **GRID)
    acc = counts_of(x[:7001], 3, 3, **GRID)
    counts_of(x[7001:], 3, 3, **GRID, into=acc)
    assert torch.equal(acc, whole)
    assert torch.equal(counts_of(x, 3, 3, **GRID), whole)
    before = whole.clone()
    counts_of(x[:0], 3, 3, **GRID, into=whole)
    assert torch.equal(whole, before)


def test_one_bin_beyond_2_to_32(dev):
    """About 11.4 M identical spin-polarised walkers, every particle at (1, 0): 380 ordered pairs per walker fall in one
    same-spin rotated bin, 380 B > 2^32 in all."""
    B, n = 11_400_000, 20
    grid = dict(extent=2.0, n_xy=4, r_max=2.0, n_r=4, n_rot=4)
    x = torch.zeros(B, n, 2, device=dev)
    x[..., 0] = 1.0
    got = counts_of(x, n, 0, **grid).cpu()
    del x
    assert 380 * B > 2 ** 32
    expect = torch.zeros_like(got)
    expect[(0 * 4 + 3) * 4 + 2] = n * B                  # density: x bin floor(3 * 1) = 3, y bin 2
    expect[32 + 2] = n * B                               # radial: r = 1 -> bin 2
    expect[32 + 8 + 0] = 190 * B                         # separation up-up: d = 0 -> bin 0
    expect[32 + 8 + 12 + (3 * 4 + 2)] = 380 * B          # rotated same spin: u = 1, w = 0
    assert torch.equal(got, expect)


def test_free_fermion_density_and_integral_identities(dev):
    """3 + 3 free fermions: the radial and 2D densities equal sum_k |phi_k|^2 of the occupied HO2D orbitals within 5
    standard errors; the normalisation identities hold to rounding; same-spin pairs show the Pauli hole."""
    from fermiflow_b200 import FreeFermion, HO2D, DensityEstimator
    ho = HO2D()
    occ = ho.orbitals[:3]
    ff = FreeFermion(dev)
    est = DensityEstimator(3, 3, extent=3.0, n_xy=12, r_max=3.0, n_r=24, n_rot=16, device=dev)
    for _ in range(16):
        est.accumulate(ff.sample(occ, occ, (65536,), equilibrim_steps=2000))
    res = est.result()
    assert res["walkers"] == 16 * 65536 and res["calls"] == 16

    # exact cell and annulus averages of sum_k |phi_k|^2 by Gauss-Legendre quadrature (orbitals.py's normalisation)
    gx, gw = np.polynomial.legendre.leggauss(16)

    def rho(pts):
        return sum(o(pts) ** 2 for o in occ)

    edges = res["xy_edges"]
    a, b = edges[:-1], edges[1:]
    nodes = (0.5 * (b - a)[:, None] * gx[None, :] + 0.5 * (a + b)[:, None]).reshape(-1)     # [12 * 16]
    X, Y = np.meshgrid(nodes, nodes, indexing="ij")
    vals = rho(torch.from_numpy(np.stack([X, Y], -1))).numpy().reshape(12, 16, 12, 16)
    cell = np.einsum("iajb,a,b->ij", vals, gw, gw) / 4.0                                       # mean over the cell
    re = res["r_edges"]
    ra, rb = re[:-1], re[1:]
    rn = 0.5 * (rb - ra)[:, None] * gx[None, :] + 0.5 * (ra + rb)[:, None]
    ring = rho(torch.from_numpy(np.stack([rn, np.zeros_like(rn)], -1))).numpy()            # radially symmetric
    annulus = (ring * 2 * np.pi * rn * (0.5 * (rb - ra))[:, None] * gw[None, :]).sum(1) / (np.pi * (rb ** 2 - ra ** 2))

    for s in range(2):
        d, e = res["density"][s], res["density_err"][s]
        big = cell * (6.0 / 12) ** 2 * 65536 > 200                      # cells with enough walkers per call
        assert big.sum() > 60
        z = np.abs(d - cell)[big] / e[big]
        assert z.max() < 5, z.max()
        z = np.abs(res["radial"][s] - annulus) / res["radial_err"][s]
        assert z[annulus * np.pi * (rb ** 2 - ra ** 2) * 65536 > 200].max() < 5

    W = res["walkers"]
    dxy, drot = 6.0 / 12, 6.0 / 16
    ring_area = np.pi * (rb ** 2 - ra ** 2)
    out = res["outside_fraction"]
    items = np.array([3, 3, 3, 3, 3, 3, 9, 12, 18], dtype=float)
    for s in range(2):
        assert math.isclose(res["density"][s].sum() * dxy ** 2 + out[s] * items[s], 3.0, rel_tol=1e-12)
        assert math.isclose((res["radial"][s] * ring_area).sum() + out[2 + s] * items[2 + s], 3.0, rel_tol=1e-12)
    for c, pairs in enumerate((3, 3, 9)):
        assert math.isclose((res["separation"][c] * ring_area).sum() + out[4 + c] * items[4 + c], pairs, rel_tol=1e-12)
    for c, pairs in enumerate((12, 18)):
        assert math.isclose(res["rotated"][c].sum() * drot ** 2 + out[7 + c] * items[7 + c] / 6, pairs / 6, rel_tol=1e-12)
    assert W == 16 * 65536
    sep = res["separation"]
    assert sep[0][0] < 0.1 * sep[2][0] and sep[1][0] < 0.1 * sep[2][0]


def test_estimator_argument_errors(dev):
    from fermiflow_b200 import DensityEstimator
    est = DensityEstimator(2, 1, extent=2.0, device=dev)
    x = torch.randn(8, 3, 2, device=dev)
    with pytest.raises(RuntimeError, match="CUDA"):
        est.accumulate(x.cpu())
    with pytest.raises(TypeError):
        est.accumulate(x.float())
    with pytest.raises(ValueError):
        est.accumulate(torch.randn(8, 4, 2, device=dev))
    assert est.result()["calls"] == 0


def test_section_beyond_shared_memory_rejected(dev):
    from fermiflow_b200 import _lib as L
    from fermiflow_b200.observables import count_layout
    x = torch.randn(4, 2, 2, device=dev)
    _, nb = count_layout(256, 0, 0)
    counts = torch.zeros(nb + 9, dtype=torch.int64, device=dev)
    g = L.FFObsGrid(2.0, 256, 0, 2.0, 0)
    import ctypes
    assert L.lib().ff_observables(L.ptr(x), 4, 1, 1, ctypes.byref(g), L.ptr(counts, torch.int64), nb + 9, L.stream()) == -1
    assert b"shared memory" in L.lib().ff_last_error()
    assert int(counts.abs().sum()) == 0


def test_ground_state_driver_writes_density(dev, tmp_path):
    from fermiflow_b200 import FermionHO2D
    path = os.path.join(str(tmp_path), "dens.npz")
    hist = FermionHO2D.main(["--nup", "2", "--ndown", "1", "--Z", "2.0", "--batch", "4096", "--iternum", "5",
                             "--nsteps", "4", "--Deta", "8", "--Dmu", "8", "--density", path, "--density-batches", "4"])
    assert len(hist) == 5 and all(len(h) == 2 for h in hist)
    res = dict(np.load(path))
    for k in ("density", "density_err", "radial", "radial_err", "separation", "separation_err", "rotated",
              "rotated_err", "outside_fraction", "xy_edges", "r_edges", "rot_edges", "walkers", "calls"):
        assert k in res, k
    assert res["walkers"] == 4 * 4096 and res["calls"] == 4
    dxy = np.diff(res["xy_edges"])[0]
    for s, ns in enumerate((2, 1)):
        total = res["density"][s].sum() * dxy ** 2 + res["outside_fraction"][s] * ns
        assert math.isclose(total, ns, rel_tol=1e-12)
