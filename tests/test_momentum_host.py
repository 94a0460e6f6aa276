"""CPU-only checks of the momentum estimators: argument errors of the C ABI ff_wavefunction_ratio(_work_size) and
ff_momentum_accumulate, and the two-rank gloo merge of MomentumEstimator state (fermiflow_b200.observables)."""
import ctypes
import math
import os

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

torch.set_default_dtype(torch.float64)

FAKE = ctypes.c_void_p(0x1000)


def _model(n_up=2, n_dn=1):
    from fermiflow_b200 import _lib as L
    m = L.FFModel()
    m.n_up, m.n_dn, m.H_eta, m.H_mu = n_up, n_dn, 4, 4
    m.eta_w1 = m.eta_b1 = m.eta_w2 = m.mu_w1 = m.mu_b1 = m.mu_w2 = FAKE
    m.t0, m.t1, m.nsteps = 0.0, 1.0, 2
    return m


def test_ratio_argument_errors():
    """Every -1 case of ff_wavefunction_ratio and its work size sets ff_last_error; nothing reaches the device."""
    from fermiflow_b200 import _lib as L
    lib = L.lib()
    nw = ctypes.c_longlong(-7)
    assert lib.ff_wavefunction_ratio_work_size(ctypes.byref(_model()), 5, 3, ctypes.byref(nw)) == 0
    C = 5 * 4
    assert nw.value == C * (4 * 3 + 3) + (C + 1) // 2
    ws_cases = [
        ((None, 5, 3, ctypes.byref(nw)), b"model is null"),
        ((ctypes.byref(_model(-1, 2)), 5, 3, ctypes.byref(nw)), b"particle"),
        ((ctypes.byref(_model()), 0, 3, ctypes.byref(nw)), b"at least 1"),
        ((ctypes.byref(_model()), 5, 0, ctypes.byref(nw)), b"at least 1"),
        ((ctypes.byref(_model()), 5, 3, None), b"null"),
    ]
    for args, msg in ws_cases:
        assert lib.ff_wavefunction_ratio_work_size(*args) == -1, args
        assert msg in lib.ff_last_error(), (args, lib.ff_last_error())

    def call(m=None, B=4, M=2, x=FAKE, orb=FAKE, ws=None, particle=FAKE, disp=FAKE, ratio=FAKE, work=FAKE):
        m = _model() if m is None else m
        return lib.ff_wavefunction_ratio(ctypes.byref(m) if m != "null" else None, x, B, orb, ws, M, particle, disp,
                                         ratio, work, None)

    cases = [
        (dict(m="null"), b"model is null"),
        (dict(m=_model(-1, 2)), b"particle"),
        (dict(m=_model(0, 0)), b"particle"),
        (dict(m=_model(37, 0)), b"particle"),
        (dict(m=_model(3, 37)), b"particle"),
        (dict(B=0), b"at least 1"),
        (dict(B=-3), b"at least 1"),
        (dict(M=0), b"at least 1"),
        (dict(x=None), b"null"),
        (dict(orb=None), b"null"),
        (dict(particle=None), b"null"),
        (dict(disp=None), b"null"),
        (dict(ratio=None), b"null"),
        (dict(work=None), b"null"),
    ]
    for kw, msg in cases:
        assert call(**kw) == -1, kw
        assert msg in lib.ff_last_error(), (kw, lib.ff_last_error())


def _acc(R=3, n_up=1, grid=(2.0, 4, 5, 3.0, 6), n_sums=None, ratio=FAKE, particle=FAKE, disp=FAKE, sums=FAKE,
         null_grid=False):
    from fermiflow_b200 import _lib as L
    from fermiflow_b200.observables import sums_layout
    g = L.FFMomGrid(*grid)
    if n_sums is None:
        n_sums = sums_layout(grid[1], grid[2], grid[4])[1]
    return L.lib().ff_momentum_accumulate(ratio, particle, disp, R, n_up, None if null_grid else ctypes.byref(g),
                                          sums, n_sums, None)


def test_accumulate_argument_errors():
    """Every -1 case of ff_momentum_accumulate sets ff_last_error; sections that are off need no valid k_max / s_max."""
    from fermiflow_b200 import _lib as L
    from fermiflow_b200.observables import sums_layout
    n_ok = sums_layout(4, 5, 6)[1]
    assert n_ok == 2 * 16 + 2 * 5 + 4 * 6 + 2
    nan = float("nan")
    cases = [
        (dict(n_up=-1), b"particle"),
        (dict(null_grid=True), b"null grid"),
        (dict(grid=(2.0, -4, 5, 3.0, 6), n_sums=n_ok), b"negative"),
        (dict(grid=(2.0, 4, -5, 3.0, 6), n_sums=n_ok), b"negative"),
        (dict(grid=(2.0, 4, 5, 3.0, -6), n_sums=n_ok), b"negative"),
        (dict(grid=(0.0, 4, 5, 3.0, 6)), b"k_max"),
        (dict(grid=(-1.0, 4, 0, 3.0, 6)), b"k_max"),
        (dict(grid=(nan, 0, 5, 3.0, 6)), b"k_max"),
        (dict(grid=(float("inf"), 4, 5, 3.0, 6)), b"k_max"),
        (dict(grid=(2.0, 4, 5, 0.0, 6)), b"s_max"),
        (dict(grid=(2.0, 4, 5, nan, 6)), b"s_max"),
        (dict(n_sums=n_ok - 1), b"n_sums"),
        (dict(n_sums=n_ok + 1), b"n_sums"),
        (dict(R=0), b"R = 0"),
        (dict(R=-2), b"R = -2"),
        (dict(ratio=None), b"null"),
        (dict(particle=None), b"null"),
        (dict(disp=None), b"null"),
        (dict(sums=None), b"null"),
    ]
    for kw, msg in cases:
        assert _acc(**kw) == -1, kw
        assert msg in L.lib().ff_last_error(), (kw, L.lib().ff_last_error())
    # sections that are off: the grid check passes and the call stops at the walker count
    for grid in ((0.0, 0, 0, 3.0, 6), (2.0, 4, 5, -1.0, 0), (nan, 0, 0, nan, 0)):
        assert _acc(R=0, grid=grid) == -1
        assert b"R = 0" in L.lib().ff_last_error(), grid


def test_estimator_argument_errors_host():
    from fermiflow_b200 import MomentumEstimator
    for kw in (dict(n_up=-1, n_dn=1), dict(n_up=0, n_dn=0), dict(n_up=1, n_dn=1, moves=0),
               dict(n_up=1, n_dn=1, k_max=0.0), dict(n_up=1, n_dn=1, s_max=float("nan")), dict(n_up=1, n_dn=1, n_k=-1)):
        with pytest.raises(ValueError):
            MomentumEstimator(device="cpu", **kw)
    est = MomentumEstimator(2, 1, device="cpu")
    with pytest.raises(RuntimeError, match="CUDA"):
        est.accumulate(None, torch.randn(4, 3, 2))
    with pytest.raises(ValueError):
        est.accumulate(None, torch.randn(4, 2, 2))


_GRID = dict(n_up=2, n_dn=1, k_max=3.0, n_k=4, n_kr=5, s_max=2.0, n_s=3, moves=4)


def _batches(seed, n_sums, n_s):
    """Four batches of sums with their walker counts; the record counts are non-negative integers."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for w in (300, 512, 77, 1024):
        s = torch.randn(n_sums, generator=g) * 50
        s[-2 - 2 * n_s:] = torch.randint(1, 1000, (2 + 2 * n_s,), generator=g).double()
        out.append((s, int(w)))
    return out


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from fermiflow_b200 import MomentumEstimator
    est = MomentumEstimator(**_GRID, device="cpu")
    for k, (s, w) in enumerate(_batches(9, est.n_sums, est.n_s)):
        if k % world == rank:
            est._add_batch(s, w)
    est.allreduce()
    if rank == 0:
        out.put(est.result())                 # numpy arrays travel by value
    dist.destroy_process_group()


def test_momentum_estimator_allreduce_gloo():
    """Two ranks merge their MomentumEstimator state with one all-reduce: the result equals one estimator fed every
    batch."""
    from fermiflow_b200 import MomentumEstimator
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 35600 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    merged = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
    ref = MomentumEstimator(**_GRID, device="cpu")
    for s, w in _batches(9, ref.n_sums, ref.n_s):
        ref._add_batch(s, w)
    single = ref.result()
    assert sorted(merged) == sorted(single)
    for k in ("momentum", "momentum_err", "momentum_radial", "momentum_radial_err", "coherence", "coherence_err",
              "k_edges", "k_radial", "s_edges", "walkers", "calls", "moves", "n_up", "n_dn"):
        assert k in single, k
    assert merged["walkers"] == 300 + 512 + 77 + 1024 and merged["calls"] == 4
    for k in single:
        np.testing.assert_allclose(merged[k], single[k], rtol=1e-12, atol=0, equal_nan=True, err_msg=k)
    assert np.isfinite(single["momentum_err"]).all() and np.isfinite(single["coherence_err"]).all()


def test_momentum_estimator_normalisation_host():
    """result() on sums built by hand: the momentum normalisation n s_max² / (4π M W), the coherence as ratio sum over
    records, and its batch-means error against a direct computation of the delta method."""
    from fermiflow_b200 import MomentumEstimator
    est = MomentumEstimator(**_GRID, device="cpu")
    lay = est.layout
    batches = _batches(3, est.n_sums, est.n_s)
    for s, w in batches:
        est._add_batch(s, w)
    res = est.result()
    W = sum(w for _, w in batches)
    tot = sum(s for s, _ in batches)
    norm = 3 * 2.0 ** 2 / (4 * math.pi * 4)
    off, shape = lay["momentum"]
    np.testing.assert_allclose(res["momentum"], norm * tot[off:off + 32].reshape(shape).numpy() / W, rtol=1e-13)
    o1, o2 = lay["ratio"][0], lay["records"][0]
    S, N = tot[o1:o1 + 6], tot[o2:o2 + 6]
    g = (S / N).reshape(2, 3).numpy()
    np.testing.assert_allclose(res["coherence"], g, rtol=1e-13)
    # delta method written out over the batches
    dev = sum(w * ((s[o1:o1 + 6] / w) - torch.from_numpy(g.reshape(-1)) * (s[o2:o2 + 6] / w)) ** 2 for s, w in batches)
    err = (dev / (3 * W * (N / W) ** 2)).sqrt().reshape(2, 3).numpy()
    np.testing.assert_allclose(res["coherence_err"], err, rtol=1e-9)
    assert np.allclose(res["k_radial"], (np.arange(5) + 0.5) * 3.0 / 5)
    assert res["moves"] == 4 and res["n_up"] == 2 and res["n_dn"] == 1
