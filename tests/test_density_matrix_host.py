"""CPU-only checks of the one-body density-matrix estimator: argument errors of the C ABI ff_density_matrix_accumulate,
the layout of its sums, the occupation errors of DensityMatrixEstimator.result() on sums built by hand, and the two-rank
gloo merge of its state (fermiflow_b200.observables)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

torch.set_default_dtype(torch.float64)

FAKE = ctypes.c_void_p(0x1000)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_density_matrix_accumulate_argument_errors():
    """Every -1 case sets ff_last_error; nothing reaches the device (every pointer is a fake)."""
    from fermiflow_b200 import _lib as L
    from fermiflow_b200.observables import density_matrix_layout
    K = 10
    n_ok = density_matrix_layout(K)[1]

    def acc(B=4, n_up=2, n_dn=1, M=3, n_orb=K, n_sums=n_ok, x=FAKE, particle=FAKE, disp=FAKE, w=FAKE, sums=FAKE):
        return L.lib().ff_density_matrix_accumulate(x, B, n_up, n_dn, M, particle, disp, w, n_orb, sums, n_sums, None)

    cases = [
        (dict(n_up=-1), b"particle"),
        (dict(n_dn=-1), b"particle"),
        (dict(n_up=0, n_dn=0), b"particle"),
        (dict(n_up=37), b"particle"),
        (dict(n_dn=37), b"particle"),
        (dict(B=0), b"at least 1"),
        (dict(B=-2), b"at least 1"),
        (dict(M=0), b"at least 1"),
        (dict(M=-1), b"at least 1"),
        (dict(n_orb=0), b"K = 0"),
        (dict(n_orb=37), b"K = 37"),
        (dict(n_orb=-3), b"K = -3"),
        (dict(n_sums=n_ok - 1), b"n_sums"),
        (dict(n_sums=n_ok + 1), b"n_sums"),
        (dict(n_orb=K + 1), b"n_sums"),
        (dict(x=None), b"null"),
        (dict(particle=None), b"null"),
        (dict(disp=None), b"null"),
        (dict(w=None), b"null"),
        (dict(sums=None), b"null"),
    ]
    for kw, msg in cases:
        assert acc(**kw) == -1, kw
        assert msg in L.lib().ff_last_error(), (kw, L.lib().ff_last_error())


def test_density_matrix_layout_matches_header():
    from fermiflow_b200.observables import density_matrix_layout
    with open(os.path.join(ROOT, "include", "fermiflow_b200.h")) as f:
        header = f.read()
    assert "(n_sums = 2 K^2 + 3)" in header
    assert re.search(r"\[2\]\[K\]\[K\] the symmetrised sums.*\[2\] records per channel, \[1\] skipped records", header,
                     re.S)
    for K in (1, 6, 21, 36):
        lay, n = density_matrix_layout(K)
        assert n == 2 * K * K + 3
        assert lay == {"matrix": (0, (2, K, K)), "records": (2 * K * K, (2,)), "skipped": (2 * K * K + 2, (1,))}


def test_estimator_argument_errors_host():
    from fermiflow_b200 import DensityMatrixEstimator
    for kw in (dict(n_up=-1, n_dn=1), dict(n_up=0, n_dn=0), dict(n_up=1, n_dn=1, shells=8),
               dict(n_up=1, n_dn=1, shells=-1), dict(n_up=1, n_dn=1, sigma=0.5), dict(n_up=1, n_dn=1, sigma=float("inf")),
               dict(n_up=1, n_dn=1, moves=0)):
        with pytest.raises(ValueError):
            DensityMatrixEstimator(device="cpu", **kw)
    est = DensityMatrixEstimator(2, 1, device="cpu")
    assert est.K == 36 and est.n_sums == 2 * 36 * 36 + 3
    assert est.state.numel() == 2 * est.n_sums + 2 * 666 * 666 + 2
    with pytest.raises(RuntimeError, match="CUDA"):
        est.accumulate(None, torch.randn(4, 3, 2))
    with pytest.raises(ValueError):
        est.accumulate(None, torch.randn(4, 2, 2))


_ARGS = dict(n_up=3, n_dn=2, shells=3, sigma=1.5, moves=4)


def _batches(seed, est):
    """Five batches of sums with their walker counts: symmetric matrices with distinct eigenvalues around a fixed
    D, different in each batch, and the record counters."""
    g = torch.Generator().manual_seed(seed)
    K = est.K
    base = torch.randn(2, K, K, generator=g)
    base = base @ base.transpose(1, 2) / K
    out = []
    for W in (300, 512, 77, 1024, 640):
        noise = torch.randn(2, K, K, generator=g) * 0.3
        S = W * (base + 0.5 * (noise + noise.transpose(1, 2)))
        s = torch.zeros(est.n_sums)
        s[:2 * K * K] = S.reshape(-1)
        s[2 * K * K:2 * K * K + 2] = torch.tensor([W * 3.0, W * 1.0])
        s[-1] = float(W % 3)
        out.append((s, W))
    return out


def test_density_matrix_result_host():
    """result() on sums built by hand: D as n / M times the sums per walker, the trace and the occupations with their
    batch-means errors recomputed from the per-batch matrices (v_k^T D_b v_k with the eigenvectors v_k of D), the
    eigen-decomposition and the shell weights."""
    from fermiflow_b200 import DensityMatrixEstimator
    est = DensityMatrixEstimator(**_ARGS, device="cpu")
    batches = _batches(3, est)
    for s, W in batches:
        est._add_batch(s, W)
    res = est.result()
    K, norm = est.K, 5 / 4
    Wt, nb = sum(W for _, W in batches), len(batches)
    Db = [(norm * s[:2 * K * K].reshape(2, K, K) / W, W) for s, W in batches]
    D = sum(W * d for d, W in Db) / Wt
    np.testing.assert_allclose(res["density_matrix"], D.numpy(), rtol=1e-12, atol=1e-14)
    assert np.array_equal(res["density_matrix"], res["density_matrix"].transpose(0, 2, 1))

    def spread(vals):                                   # batch-means error of per-batch values [nb, ...]
        m = sum(W * v for (_, W), v in zip(Db, vals)) / Wt
        return (sum(W * (v - m) ** 2 for (_, W), v in zip(Db, vals)) / ((nb - 1) * Wt)).sqrt()

    np.testing.assert_allclose(res["density_matrix_err"], spread([d for d, _ in Db]).numpy(), rtol=1e-9)
    np.testing.assert_allclose(res["trace"], D.diagonal(dim1=1, dim2=2).sum(-1).numpy(), rtol=1e-12)
    np.testing.assert_allclose(res["trace_err"], spread([d.diagonal(dim1=1, dim2=2).sum(-1) for d, _ in Db]).numpy(),
                               rtol=1e-9)
    V, occ = torch.from_numpy(res["natural_orbitals"]), torch.from_numpy(res["occupations"])
    assert (np.diff(res["occupations"], axis=1) <= 0).all()
    np.testing.assert_allclose((V.transpose(1, 2) @ V).numpy(), np.broadcast_to(np.eye(K), (2, K, K)), atol=1e-12)
    np.testing.assert_allclose((D @ V).numpy(), (V * occ[:, None, :]).numpy(), atol=1e-12)
    big = V.abs().argmax(1)
    assert (torch.gather(V, 1, big[:, None, :]) > 0).all()
    lam = [torch.einsum("cak,cab,cbk->ck", V, d, V) for d, _ in Db]
    np.testing.assert_allclose(res["occupations_err"], spread(lam).numpy(), rtol=1e-8)
    assert np.isfinite(res["occupations_err"]).all() and (res["occupations_err"] > 0).all()
    # shell weights: squared coefficients per shell nx + ny, summing to 1 per natural orbital
    q = res["orbital_quanta"]
    assert q.shape == (K, 2) and [tuple(r) for r in q[:6]] == [(0, 0), (0, 1), (1, 0), (0, 2), (1, 1), (2, 0)]
    sw = res["shell_weight"]
    assert sw.shape == (2, K, 4)
    np.testing.assert_allclose(sw.sum(-1), 1.0, rtol=1e-12)
    shell = q.sum(1)
    np.testing.assert_allclose(sw[1, :, 2], (V[1] ** 2)[shell == 2].sum(0).numpy(), rtol=1e-12)
    assert res["walkers"] == Wt and res["calls"] == nb and res["moves"] == 4 and res["sigma"] == 1.5
    assert res["n_up"] == 3 and res["n_dn"] == 2
    # one call: no errors
    one = DensityMatrixEstimator(**_ARGS, device="cpu")
    one._add_batch(*batches[0])
    r1 = one.result()
    assert np.isnan(r1["occupations_err"]).all() and np.isnan(r1["trace_err"]).all()


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from fermiflow_b200 import DensityMatrixEstimator
    est = DensityMatrixEstimator(**_ARGS, device="cpu")
    for k, (s, W) in enumerate(_batches(9, est)):
        if k % world == rank:
            est._add_batch(s, W)
    est.allreduce()
    if rank == 0:
        out.put(est.result())                 # numpy arrays travel by value
    dist.destroy_process_group()


def test_density_matrix_allreduce_gloo():
    """Two ranks merge their DensityMatrixEstimator state, second moments included, with one all-reduce: the result
    equals one estimator fed every batch."""
    from fermiflow_b200 import DensityMatrixEstimator
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 39600 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    merged = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
    ref = DensityMatrixEstimator(**_ARGS, device="cpu")
    for s, W in _batches(9, ref):
        ref._add_batch(s, W)
    single = ref.result()
    keys = ("density_matrix", "density_matrix_err", "trace", "trace_err", "occupations", "occupations_err",
            "natural_orbitals", "shell_weight", "orbital_quanta", "walkers", "calls", "moves", "sigma", "n_up", "n_dn")
    assert sorted(merged) == sorted(single) == sorted(keys)
    assert merged["walkers"] == 300 + 512 + 77 + 1024 + 640 and merged["calls"] == 5
    for k in keys:
        np.testing.assert_allclose(merged[k], single[k], rtol=1e-9, atol=1e-12, err_msg=k)
    assert np.isfinite(single["occupations_err"]).all()
