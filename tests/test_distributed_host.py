"""world_size-2 gloo test of the only cross-rank step of the path: all-reduce of the energy
moments and of the parameter gradient (fermiflow_b200.VMC)."""
import os

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

torch.set_default_dtype(torch.float64)


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from fermiflow_b200.VMC import _global_mean_std, _VMCBase
    g = torch.Generator().manual_seed(5)
    full = torch.randn(64, generator=g)
    mine = full[rank::world].clone()
    mean, std, cnt = _global_mean_std(mine)

    class M(_VMCBase):
        def __init__(self):
            super().__init__()
            self.a = torch.nn.Parameter(torch.zeros(3))
            self.b = torch.nn.Parameter(torch.zeros(2, 2))
    m = M()
    m.a.grad = torch.full((3,), float(rank + 1))
    m.b.grad = torch.full((2, 2), float(10 * (rank + 1)))
    m.allreduce_gradients()
    if rank == 0:
        out.put((mean, std, cnt, float(full.mean()), float(full.std()), m.a.grad.tolist(), m.b.grad.tolist()))
    dist.destroy_process_group()


def test_moments_and_gradient_allreduce_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
    mean, std, cnt, fmean, fstd, ga, gb = res
    assert cnt == 64
    assert abs(mean - fmean) < 1e-14 and abs(std - fstd) < 1e-13
    assert ga == [3.0, 3.0, 3.0] and gb == [[30.0, 30.0], [30.0, 30.0]]


def _beta_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from fermiflow_b200.VMC import _beta_estimators
    g = torch.Generator().manual_seed(9)
    NS, B, beta = 5, 40, 1.7
    lw_full = torch.randn(NS, generator=g)
    E_full = 10 + torch.randn(B, generator=g)
    st_full = torch.randint(NS, (B,), generator=g)
    mine = slice(rank * B // world, (rank + 1) * B // world)          # each rank: its own walkers, states sorted locally
    st, order = torch.sort(st_full[mine])
    E = E_full[mine][order]
    lw = lw_full.clone().requires_grad_(True)
    cnt = torch.bincount(st, minlength=NS).to(torch.float64)
    obs, nglobal, gphi, xmean = _beta_estimators(E, st, lw, beta, cnt)
    gphi.backward()
    grad = lw.grad.clone()
    dist.all_reduce(grad)
    w = (E - xmean) / nglobal
    gathered = [torch.zeros(B // world) for _ in range(world)]
    gathered_E = [torch.zeros(B // world) for _ in range(world)]
    gathered_s = [torch.zeros(B // world, dtype=torch.long) for _ in range(world)]
    dist.all_gather(gathered, w); dist.all_gather(gathered_E, E); dist.all_gather(gathered_s, st)
    if rank == 0:
        # numpy copies travel by value; a torch tensor in the queue would be fetched from this process, which may have
        # exited by then
        out.put(({k: float(v) for k, v in obs.items() if k != "logp_states_all"}, float(nglobal), grad.numpy(),
                 torch.cat(gathered).numpy(), torch.cat(gathered_E).numpy(), torch.cat(gathered_s).numpy(),
                 lw_full.numpy(), beta))
    dist.destroy_process_group()


def test_finite_temperature_estimators_allreduce_gloo():
    """BetaVMC's estimators (one fused all-reduce; VMC.py:139-171) on two ranks against the oracle's restatement of
    those lines on the union of the walkers."""
    from oracle import fermiflow_oracle as O
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    procs = [ctx.Process(target=_beta_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    obs, nglobal, grad, w, E, st, lw_full, beta = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
    grad, w, E, st, lw_full = (torch.from_numpy(a) for a in (grad, w, E, st, lw_full))
    assert nglobal == 40
    lw = lw_full.clone().requires_grad_(True)
    ref = O.beta_vmc_estimators(E, st, lw, beta)
    for k in ("E", "E_std", "F", "F_std", "S", "S_analytical"):
        assert abs(obs[k] - ref[k]) < 1e-12 * max(1.0, abs(ref[k])), (k, obs[k], ref[k])
    ref["gradF_phi"].backward()
    assert torch.allclose(grad, lw.grad, rtol=1e-12, atol=1e-14)
    assert torch.allclose(w, ref["theta_weights"], rtol=1e-12, atol=1e-15)
