"""CPU-only checks of the Rényi estimator: argument errors of the C ABI ff_swap_ratio(_work_size) and
ff_swap_accumulate, the normalisation of RenyiEstimator.result() on sums built by hand, and the two-rank gloo merge of
its state (fermiflow_b200.observables)."""
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


def _regions(a, kind=0, Q=None):
    from fermiflow_b200 import _lib as L
    arr = (ctypes.c_double * max(len(a), 1))(*a)
    return L.FFSwapRegions(kind, len(a) if Q is None else Q, arr), arr


def test_swap_ratio_argument_errors():
    """Every -1 case of ff_swap_ratio and its work size sets ff_last_error; nothing reaches the device (every pointer
    but the host region parameters is a fake)."""
    from fermiflow_b200 import _lib as L
    lib = L.lib()
    nw = ctypes.c_longlong(-7)
    assert lib.ff_swap_ratio_work_size(ctypes.byref(_model()), 5, 3, ctypes.byref(nw)) == 0
    C = 2 * 5 * 4
    assert nw.value == C * (4 * 3 + 3) + (C + 1) // 2
    ws_cases = [
        ((None, 5, 3, ctypes.byref(nw)), b"model is null"),
        ((ctypes.byref(_model(-1, 2)), 5, 3, ctypes.byref(nw)), b"particle"),
        ((ctypes.byref(_model()), 0, 3, ctypes.byref(nw)), b"P = 0"),
        ((ctypes.byref(_model()), 5, 0, ctypes.byref(nw)), b"Q = 0"),
        ((ctypes.byref(_model()), 5, 33, ctypes.byref(nw)), b"Q = 33"),
        ((ctypes.byref(_model()), 5, 3, None), b"null"),
    ]
    for args, msg in ws_cases:
        assert lib.ff_swap_ratio_work_size(*args) == -1, args
        assert msg in lib.ff_last_error(), (args, lib.ff_last_error())

    def call(m=None, B=4, P=2, x=FAKE, orb=FAKE, ws=None, pairs=FAKE, reg="ok", ratio=FAKE, sector=FAKE, work=FAKE):
        m = _model() if m is None else m
        keep = None
        if reg == "ok":
            reg, keep = _regions([0.5, 1.0])
        return lib.ff_swap_ratio(ctypes.byref(m) if m != "null" else None, x, B, orb, ws, P, pairs,
                                 ctypes.byref(reg) if reg is not None else None, ratio, sector, work, None), keep

    nan, inf = float("nan"), float("inf")
    cases = [
        (dict(m="null"), b"model is null"),
        (dict(m=_model(-1, 2)), b"particle"),
        (dict(m=_model(0, 0)), b"particle"),
        (dict(m=_model(37, 0)), b"particle"),
        (dict(m=_model(3, 37)), b"particle"),
        (dict(B=0), b"at least 1"),
        (dict(B=-3), b"at least 1"),
        (dict(P=0), b"at least 1"),
        (dict(P=-1), b"at least 1"),
        (dict(reg=None), b"null regions"),
        (dict(reg=_regions([], Q=0)[0]), b"Q = 0"),
        (dict(reg=_regions([1.0] * 33)[0]), b"Q = 33"),
        (dict(reg=_regions([1.0], Q=-2)[0]), b"Q = -2"),
        (dict(reg=_regions([1.0], kind=2)[0]), b"kind 2"),
        (dict(reg=_regions([1.0], kind=-1)[0]), b"kind -1"),
        (dict(reg=_regions([0.5, nan])[0]), b"not finite"),
        (dict(reg=_regions([inf])[0]), b"not finite"),
        (dict(reg=_regions([-inf], kind=1)[0]), b"not finite"),
        (dict(reg=_regions([1.0, -0.5])[0]), b"negative radius"),
        (dict(x=None), b"null buffer"),
        (dict(orb=None), b"null buffer"),
        (dict(pairs=None), b"null buffer"),
        (dict(ratio=None), b"null buffer"),
        (dict(sector=None), b"null buffer"),
        (dict(work=None), b"null buffer"),
    ]
    from fermiflow_b200 import _lib as L2
    null_a = L2.FFSwapRegions(0, 2, None)
    cases.append((dict(reg=null_a), b"null region parameters"))
    for kw, msg in cases:
        rc, _ = call(**kw)
        assert rc == -1, kw
        assert msg in lib.ff_last_error(), (kw, lib.ff_last_error())


def test_swap_accumulate_argument_errors():
    from fermiflow_b200 import _lib as L
    from fermiflow_b200.observables import swap_layout
    n_ok = swap_layout(3, 2, 1)[1]
    assert n_ok == 3 * 3 * 6 + 3 + 1

    def acc(P=5, Q=3, n_up=2, n_dn=1, n_sums=n_ok, ratio=FAKE, sector=FAKE, sums=FAKE):
        return L.lib().ff_swap_accumulate(ratio, sector, P, Q, n_up, n_dn, sums, n_sums, None)

    cases = [
        (dict(n_up=-1), b"particle"),
        (dict(n_dn=-1), b"particle"),
        (dict(n_up=0, n_dn=0), b"particle"),
        (dict(n_up=37), b"particle"),
        (dict(P=0), b"P = 0"),
        (dict(P=-4), b"P = -4"),
        (dict(Q=0), b"Q = 0"),
        (dict(Q=33), b"Q = 33"),
        (dict(n_sums=n_ok - 1), b"n_sums"),
        (dict(n_sums=n_ok + 1), b"n_sums"),
        (dict(ratio=None), b"null"),
        (dict(sector=None), b"null"),
        (dict(sums=None), b"null"),
    ]
    for kw, msg in cases:
        assert acc(**kw) == -1, kw
        assert msg in L.lib().ff_last_error(), (kw, L.lib().ff_last_error())


def test_estimator_argument_errors_host():
    from fermiflow_b200 import RenyiEstimator
    for kw in (dict(n_up=-1, n_dn=1), dict(n_up=0, n_dn=0), dict(n_up=1, n_dn=1, kind="square"),
               dict(n_up=1, n_dn=1, a=()), dict(n_up=1, n_dn=1, a=[1.0] * 33), dict(n_up=1, n_dn=1, a=(1.0, -1.0)),
               dict(n_up=1, n_dn=1, a=(float("nan"),), kind="halfplane")):
        with pytest.raises(ValueError):
            RenyiEstimator(device="cpu", **kw)
    RenyiEstimator(1, 1, a=(-2.0, 0.0), kind="halfplane", device="cpu")
    est = RenyiEstimator(2, 1, device="cpu")
    with pytest.raises(RuntimeError, match="CUDA"):
        est.accumulate(None, torch.randn(4, 3, 2))
    with pytest.raises(ValueError):
        est.accumulate(None, torch.randn(4, 2, 2))


_ARGS = dict(n_up=2, n_dn=1, a=(0.7, 1.4, 2.1), kind="disk")


def _batches(seed, est):
    """Four batches of sums with their pair counts: every pair in a sector, half of them matched with ratios of mixed
    sign, so that the sector sums, replica counts and ratio sums vary from batch to batch."""
    g = torch.Generator().manual_seed(seed)
    lay = est.layout
    out = []
    for P in (300, 512, 77, 1024):
        s = torch.zeros(est.n_sums)
        for name in ("ratio", "replicas", "matched"):
            o, sh = lay[name]
            k = math.prod(sh)
            if name == "ratio":
                s[o:o + k] = torch.rand(k, generator=g) * P * 0.3 + (torch.rand(k, generator=g) - 0.7) * 5
            else:
                s[o:o + k] = torch.randint(1, P, (k,), generator=g).double()
        o1, o2, o3 = lay["ratio"][0], lay["replicas"][0], lay["matched"][0]
        s[o1] = -0.1 * P                                  # a negative sector sum: S2_sector NaN
        s[o1 + 5] = s[o2 + 5] = s[o3 + 5] = 0.0           # an empty sector: S2_sector NaN
        s[lay["skipped"][0]:lay["skipped"][0] + est.Q] = torch.randint(0, 3, (est.Q,), generator=g).double()
        s[lay["pairs"][0]] = P
        out.append((s, P))
    return out


def test_renyi_estimator_normalisation_host():
    """result() on sums built by hand: swap as the ratio sum over pairs, S2 = -ln swap, the sector probabilities as
    replicas over 2 pairs, and the batch-means errors of swap and S2_sector against a direct computation."""
    from fermiflow_b200 import RenyiEstimator
    est = RenyiEstimator(**_ARGS, device="cpu")
    batches = _batches(3, est)
    for s, P in batches:
        est._add_batch(s, P)
    res = est.result()
    W, K = sum(P for _, P in batches), len(batches)
    Q, shape = est.Q, (3, 3, 2)
    o1, o2 = est.layout["ratio"][0], est.layout["replicas"][0]
    k = math.prod(shape)

    def per_batch(o):
        return [(s[o:o + k].reshape(shape), P) for s, P in batches]

    T = sum(t for t, _ in per_batch(o1)) / W
    R = sum(r for r, _ in per_batch(o2)) / W
    swap = T.sum((1, 2))
    np.testing.assert_allclose(res["swap"], swap.numpy(), rtol=1e-13)
    np.testing.assert_allclose(res["S2"], -np.log(swap.numpy()), rtol=1e-13)
    np.testing.assert_allclose(res["sector_prob"], 0.5 * R.numpy(), rtol=1e-13)
    np.testing.assert_allclose(res["sector_prob"].sum((1, 2)), 0.5 * sum(s[o2:o2 + k].reshape(Q, -1).sum(1)
                                                                          for s, _ in batches).numpy() / W, rtol=1e-13)
    np.testing.assert_allclose(res["sector_swap"], T.numpy(), rtol=1e-13)
    # batch means written out
    sw = [(t.sum((1, 2)) / P, P) for t, P in per_batch(o1)]
    err = (sum(P * (m - swap) ** 2 for m, P in sw) / ((K - 1) * W)).sqrt()
    np.testing.assert_allclose(res["swap_err"], err.numpy(), rtol=1e-9)
    np.testing.assert_allclose(res["S2_err"], (err / swap).numpy(), rtol=1e-9)
    good = (T > 0) & (R > 0)
    assert good.any() and (~good).any()
    S2s = -torch.log(T / (0.25 * R * R))
    np.testing.assert_allclose(res["S2_sector"][good.numpy()], S2s[good].numpy(), rtol=1e-12)
    assert np.isnan(res["S2_sector"][~good.numpy()]).all()
    # delta method: S2(a, b) = -ln t + 2 ln r + ln 4, derivatives -1/t and 2/r at the batch means
    dev = sum(P * (-(t / P - T) / T + 2 * (r / P - R) / R) ** 2
              for (t, P), (r, _) in zip(per_batch(o1), per_batch(o2)))
    e2 = (dev / ((K - 1) * W)).sqrt()
    np.testing.assert_allclose(res["S2_sector_err"][good.numpy()], e2[good].numpy(), rtol=1e-8)
    assert res["pairs"] == W and res["calls"] == K and str(res["kind"]) == "disk"
    assert np.allclose(res["a"], _ARGS["a"]) and res["n_up"] == 2 and res["n_dn"] == 1


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from fermiflow_b200 import RenyiEstimator
    est = RenyiEstimator(**_ARGS, device="cpu")
    for k, (s, P) in enumerate(_batches(9, est)):
        if k % world == rank:
            est._add_batch(s, P)
    est.allreduce()
    if rank == 0:
        out.put(est.result())                 # numpy arrays travel by value
    dist.destroy_process_group()


def test_renyi_estimator_allreduce_gloo():
    """Two ranks merge their RenyiEstimator state with one all-reduce: the result equals one estimator fed every
    batch."""
    from fermiflow_b200 import RenyiEstimator
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 37600 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    merged = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
    ref = RenyiEstimator(**_ARGS, device="cpu")
    for s, P in _batches(9, ref):
        ref._add_batch(s, P)
    single = ref.result()
    assert sorted(merged) == sorted(single)
    for k in ("swap", "swap_err", "S2", "S2_err", "sector_prob", "sector_prob_err", "sector_swap", "sector_swap_err",
              "S2_sector", "S2_sector_err", "a", "kind", "pairs", "calls", "n_up", "n_dn"):
        assert k in single, k
    assert merged["pairs"] == 300 + 512 + 77 + 1024 and merged["calls"] == 4
    for k in single:
        if k == "kind":
            assert str(merged[k]) == str(single[k])
            continue
        np.testing.assert_allclose(merged[k], single[k], rtol=1e-12, atol=0, equal_nan=True, err_msg=k)
    assert np.isfinite(single["swap_err"]).all() and np.isfinite(single["sector_prob_err"]).all()
