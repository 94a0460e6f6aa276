"""CPU-only checks of the walker histograms: argument errors of the C ABI ff_observables, and the two-rank gloo merge
of DensityEstimator state (fermiflow_b200.observables)."""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

torch.set_default_dtype(torch.float64)


def _call(B, n_up, n_dn, grid, n_counts, x=None, counts=None):
    from fermiflow_b200 import _lib as L
    g = L.FFObsGrid(*grid)
    return L.lib().ff_observables(x, B, n_up, n_dn, ctypes.byref(g), counts, n_counts, None)


def test_c_abi_argument_errors():
    """Every -1 case of ff_observables that needs no device sets ff_last_error; B == 0 is a no-op."""
    from fermiflow_b200 import _lib as L
    from fermiflow_b200.observables import count_layout
    ok = (2.0, 4, 3, 1.5, 5)                                   # extent, n_xy, n_rot, r_max, n_r
    n_ok = count_layout(4, 5, 3)[1] + 9
    assert n_ok == 2 * 16 + 2 * 5 + 3 * 5 + 2 * 9 + 9
    fake = ctypes.c_void_p(0x1000)
    cases = [
        (dict(B=1, n_up=-1, n_dn=2, grid=ok, n_counts=n_ok, x=fake, counts=fake), b"particle"),
        (dict(B=1, n_up=1, n_dn=-1, grid=ok, n_counts=n_ok, x=fake, counts=fake), b"particle"),
        (dict(B=1, n_up=0, n_dn=0, grid=ok, n_counts=n_ok, x=fake, counts=fake), b"particle"),
        (dict(B=-1, n_up=1, n_dn=1, grid=ok, n_counts=n_ok), b"walker"),
        (dict(B=3, n_up=1, n_dn=1, grid=ok, n_counts=n_ok, counts=fake), b"null"),
        (dict(B=3, n_up=1, n_dn=1, grid=ok, n_counts=n_ok, x=fake), b"null"),
        (dict(B=0, n_up=1, n_dn=1, grid=(0.0, 4, 3, 1.5, 5), n_counts=n_ok), b"extent"),
        (dict(B=0, n_up=1, n_dn=1, grid=(-1.0, 0, 3, 1.5, 5), n_counts=count_layout(0, 5, 3)[1] + 9), b"extent"),
        (dict(B=0, n_up=1, n_dn=1, grid=(float("nan"), 4, 0, 1.5, 5), n_counts=count_layout(4, 5, 0)[1] + 9), b"extent"),
        (dict(B=0, n_up=1, n_dn=1, grid=(2.0, 4, 3, 0.0, 5), n_counts=n_ok), b"r_max"),
        (dict(B=0, n_up=1, n_dn=1, grid=(2.0, -4, 3, 1.5, 5), n_counts=n_ok), b"negative"),
        (dict(B=0, n_up=1, n_dn=1, grid=(2.0, 4, 3, 1.5, -1), n_counts=n_ok), b"negative"),
        (dict(B=0, n_up=1, n_dn=1, grid=ok, n_counts=n_ok - 1), b"n_counts"),
        (dict(B=0, n_up=1, n_dn=1, grid=ok, n_counts=n_ok + 1), b"n_counts"),
    ]
    for kw, msg in cases:
        assert _call(**kw) == -1, kw
        assert msg in L.lib().ff_last_error(), (kw, L.lib().ff_last_error())
    assert _call(0, 1, 1, ok, n_ok) == 0
    # sections that are off need no valid extent / r_max
    assert _call(0, 1, 1, (0.0, 0, 0, 0.0, 0), 9) == 0
    assert _call(0, 2, 0, (0.0, 0, 0, 1.0, 5), count_layout(0, 5, 0)[1] + 9) == 0


def test_estimator_rejects_cpu_walkers():
    from fermiflow_b200 import DensityEstimator
    est = DensityEstimator(1, 1, extent=2.0, device="cpu")
    with pytest.raises(RuntimeError, match="CUDA"):
        est.accumulate(torch.randn(4, 2, 2))


def _batches(seed, n_counts):
    """Four batches of integer counts with their walker counts (the merge does not look at how they were binned)."""
    g = torch.Generator().manual_seed(seed)
    return [(torch.randint(0, 1000, (n_counts,), generator=g), int(w)) for w in (300, 512, 77, 1024)]


_GRID = dict(n_up=2, n_dn=1, extent=2.0, n_xy=4, r_max=1.5, n_r=5, n_rot=3)


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from fermiflow_b200 import DensityEstimator
    est = DensityEstimator(**_GRID, device="cpu")
    for k, (c, w) in enumerate(_batches(7, est.n_counts)):
        if k % world == rank:
            est._add_batch(c, w)
    est.allreduce()
    if rank == 0:
        # numpy copies travel by value; a torch tensor in the queue would be fetched from this process, which may have
        # exited by then
        out.put(est.result())
    dist.destroy_process_group()


def test_estimator_allreduce_gloo():
    """Two ranks merge their estimator state with one all-reduce: the result equals one estimator fed every batch."""
    from fermiflow_b200 import DensityEstimator
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    merged = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
    ref = DensityEstimator(**_GRID, device="cpu")
    for c, w in _batches(7, ref.n_counts):
        ref._add_batch(c, w)
    single = ref.result()
    assert sorted(merged) == sorted(single)
    assert merged["walkers"] == 300 + 512 + 77 + 1024 and merged["calls"] == 4
    for k in single:
        np.testing.assert_allclose(merged[k], single[k], rtol=1e-13, atol=0, equal_nan=True, err_msg=k)
    assert np.isfinite(single["density_err"]).all()


def test_estimator_normalisation_identities_host():
    """The integral identities of the DensityEstimator docstring on counts built by hand; errors are NaN below two
    calls."""
    from fermiflow_b200 import DensityEstimator
    est = DensityEstimator(**_GRID, device="cpu")
    lay = est.layout
    W = 10
    c = torch.zeros(est.n_counts, dtype=torch.int64)
    per = dict(density=(2, 1), radial=(2, 1), separation=(1, 0, 2), rotated=(2, 4))   # items per walker and channel
    outside = torch.tensor([3, 0, 5, 2, 1, 0, 4, 6, 7])
    o = 0
    for name in ("density", "radial", "separation", "rotated"):
        off, shape = lay[name]
        cells = int(np.prod(shape[1:]))
        for ch, items in enumerate(per[name]):
            total = items * W - int(outside[o])
            c[off + ch * cells + (ch % cells)] = total
            o += 1
    c[-9:] = outside
    est._add_batch(c, W)
    res = est.result()
    assert np.isnan(res["density_err"]).all()
    dxy, drot = 4.0 / 4, 4.0 / 3
    r = res["r_edges"]
    ring = np.pi * (r[1:] ** 2 - r[:-1] ** 2)
    out = res["outside_fraction"]
    for s, ns in enumerate((2, 1)):
        assert np.isclose(res["density"][s].sum() * dxy ** 2 + out[s] * ns, ns, rtol=1e-13)
        assert np.isclose((res["radial"][s] * ring).sum() + out[2 + s] * ns, ns, rtol=1e-13)
    for ch, pairs in enumerate((1, 0, 2)):
        assert np.isclose((res["separation"][ch] * ring).sum() + (out[4 + ch] * pairs if pairs else 0), pairs, rtol=1e-13)
    assert np.isnan(out[5])                                              # no down-down pairs
    for ch, pairs in enumerate((2, 4)):
        assert np.isclose(res["rotated"][ch].sum() * drot ** 2 + out[7 + ch] * pairs / 3, pairs / 3, rtol=1e-13)
