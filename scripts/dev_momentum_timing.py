"""Time of ff_wavefunction_ratio (split into the flow sweep over the B (M + 1) configurations and the rest: building the
configurations, the Slater determinants with their signs, the ratios) and of ff_momentum_accumulate with the default
MomentumEstimator grid (n_k = 64, n_kr = 128, n_s = 64, k_max = 4, s_max = 8), at 65536 walkers and M = 8 records per
walker, for N = 20 (10 + 10) and N = 12 (12 + 0).  The sums are checked against a torch restatement (cos, scipy's j0,
bincount; chunked over the records; tolerance 1e-12 sum |ratio| per entry, 5e-12 for the J0 section, the absolute
error bound of CUDA's double j0 for arguments of 8 and more), and the VMC step time of the same model is printed for
scale.  CUDA events after warm-up; one JSON line per particle number, with the device name and power limit."""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from scipy.special import j0  # noqa: E402

import bench  # noqa: E402
from fermiflow_b200.observables import momentum_accumulate, sums_layout  # noqa: E402

torch.set_default_dtype(torch.float64)


def timed(f, reps):
    """min over reps of the CUDA-event time of f() in ms, after one warm-up call."""
    f()
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        f()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def torch_sums(ratio, particle, disp, n_up, k_max, n_k, n_kr, s_max, n_s, chunk=8192):
    """The layout of ff_momentum_accumulate restated in torch: cos(k.s), J0 (scipy: torch.special.bessel_j0 is off by up
    to 4e-7 near x = 5) and the |s| bins."""
    dev = ratio.device
    kk = -k_max + (torch.arange(n_k, device=dev) + 0.5) * (2 * k_max / n_k)
    kr = (torch.arange(n_kr, device=dev) + 0.5) * (k_max / n_kr)
    grid = torch.zeros(2, n_k, n_k, device=dev)
    radial = torch.zeros(2, n_kr, device=dev)
    rsum = torch.zeros(2 * n_s, device=dev)
    cnt = torch.zeros(2 * n_s, device=dev)
    per = torch.zeros(2, device=dev)
    for c0 in range(0, ratio.numel(), chunk):
        r, p, d = ratio[c0:c0 + chunk], particle[c0:c0 + chunk], disp[c0:c0 + chunk]
        ch = (p.long() >= n_up).long()
        w = torch.stack([r * (ch == c) for c in (0, 1)], 1)
        ph = kk[None, :, None] * d[:, 0, None, None] + kk[None, None, :] * d[:, 1, None, None]
        grid += torch.einsum("rc,rab->cab", w, torch.cos(ph))
        s = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]).sqrt()
        radial += torch.einsum("rc,rj->cj", w, torch.from_numpy(j0((kr[None, :] * s[:, None]).cpu().numpy())).to(dev))
        f = (s * (n_s / s_max)).floor()
        ok = (f >= 0) & (f < n_s)
        key = (ch * n_s + f.long().clamp(0, n_s - 1))[ok]
        rsum.index_add_(0, key, r[ok])
        cnt += torch.bincount(key, minlength=2 * n_s).double()
        per += torch.bincount(ch, minlength=2).double()
    return torch.cat([grid.reshape(-1), radial.reshape(-1), rsum, cnt, per])


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--walkers", type=int, default=65536)
    p.add_argument("--moves", type=int, default=8)
    p.add_argument("--reps", type=int, default=5)
    p.add_argument("--vmc-steps", type=int, default=3)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip()
    grid = dict(k_max=4.0, n_k=64, n_kr=128, s_max=8.0, n_s=64)
    _, n_sums = sums_layout(grid["n_k"], grid["n_kr"], grid["n_s"])
    failed = False
    for nup, ndown in ((10, 10), (12, 0)):
        n, B, M = nup + ndown, args.walkers, args.moves
        model = bench.build_model(argparse.Namespace(hidden=50, ode_steps=16, nup=nup, ndown=ndown, Z=2.0), dev)
        g = torch.Generator(device=dev).manual_seed(1)
        with torch.no_grad():
            _, x = model.sample((B,))
        particle = torch.randint(0, n, (B, M), device=dev, dtype=torch.int32, generator=g)
        u = torch.rand(B, M, 2, device=dev, generator=g)
        r, phi = grid["s_max"] * u[..., 0].sqrt(), 2 * math.pi * u[..., 1]
        disp = torch.stack((r * phi.cos(), r * phi.sin()), -1)
        out = {}

        def ratio():
            out["ratio"] = model.wavefunction_ratio(x, particle, disp)

        t_ratio = timed(ratio, args.reps)
        # the flow sweep alone on B (M + 1) configurations of the same size
        xc = x[:, None].expand(B, M + 1, n, 2).reshape(-1, n, 2).contiguous()
        del out["ratio"]
        with torch.no_grad():
            t_flow = timed(lambda: model.cnf.delta_logp(xc), args.reps)
        del xc
        ratio()
        rho = out["ratio"]
        sums = torch.zeros(n_sums, device=dev)

        def acc():
            sums.zero_()
            momentum_accumulate(rho, particle, disp, nup, sums=sums, **grid)

        t_acc = timed(acc, args.reps)
        ref = torch_sums(rho.reshape(-1), particle.reshape(-1), disp.reshape(-1, 2), nup, **grid)
        tol = 1e-12 * float(rho.abs().sum())
        lay, _ = sums_layout(grid["n_k"], grid["n_kr"], grid["n_s"])
        scale = torch.ones_like(ref)
        o = lay["radial"][0]
        scale[o:o + 2 * grid["n_kr"]] = 5.0
        err = float(((sums - ref).abs() / scale).max())

        def step():
            model(B).backward()

        t_step = timed(step, args.vmc_steps)
        new = t_ratio - t_flow + t_acc
        print(json.dumps(dict(n_up=nup, n_dn=ndown, walkers=B, moves=M, grid=grid,
                              wavefunction_ratio_ms=round(t_ratio, 2), flow_sweep_ms=round(t_flow, 2),
                              ratio_rest_ms=round(t_ratio - t_flow, 3), momentum_accumulate_ms=round(t_acc, 3),
                              new_kernels_share_of_flow=round(new / t_flow, 4),
                              torch_max_abs_diff=err, torch_tolerance=tol, sums_agree=err <= tol,
                              negative_ratio_fraction=round(float((rho < 0).double().mean()), 4),
                              vmc_step_ms=round(t_step, 2),
                              device=torch.cuda.get_device_name(dev), power_limit=power)))
        failed = failed or not err <= tol
        del model, x, rho, out, ref
        torch.cuda.empty_cache()
    if failed:
        raise SystemExit("sums differ from the torch restatement")


if __name__ == "__main__":
    main()
