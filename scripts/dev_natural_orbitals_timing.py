"""Time of ff_wavefunction_ratio and of ff_density_matrix_accumulate with the full basis (K = 36, shells 0 ... 7), at
65536 walkers and M = 8 records per walker, for N = 20 (10 + 10) and N = 12 (12 + 0).  The records are those of
DensityMatrixEstimator: particles drawn uniformly, r' from the Gaussian of width sigma = 1.5, w = ratio / q(r').  The sums
are checked against a torch restatement (the oracle's orbitals, chunked over the records; tolerance 1e-12 of sum |terms|
per entry, counts exactly).  A short scan of the proposal width prints, for sigma = 1.0, 1.5, 2.0 and 3.0, the median
relative error of the diagonal of D and the error of the trace from 4 batches, so that the default can be judged.  CUDA
events after warm-up; one JSON line per particle number, with the device name and power limit."""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from fermiflow_b200 import DensityMatrixEstimator  # noqa: E402
from fermiflow_b200.observables import density_matrix_accumulate, density_matrix_layout  # noqa: E402
from oracle import fermiflow_oracle as O  # noqa: E402

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


def torch_sums(x, particle, disp, w, n_up, K, chunk=16384):
    """(sums, sum of |terms|) in the layout of ff_density_matrix_accumulate, restated with the oracle's orbitals."""
    B, M = particle.shape
    n = x.shape[1]
    mats = torch.zeros(2, K, K, device=x.device)
    mags = torch.zeros(2, K, K, device=x.device)
    counts = torch.zeros(3, device=x.device)
    p_all, d_all, w_all = particle.reshape(-1).long(), disp.reshape(-1, 2), w.reshape(-1)
    for c0 in range(0, B * M, chunk):
        p, d, ww = p_all[c0:c0 + chunk], d_all[c0:c0 + chunk], w_all[c0:c0 + chunk]
        b = (torch.arange(c0, c0 + p.numel(), device=x.device) // M)
        ok = (p >= 0) & (p < n)
        ri = x[b[ok], p[ok]]
        U = torch.stack([O.ho2d_orbital(k, ri) for k in range(K)], -1)
        V = torch.stack([O.ho2d_orbital(k, ri + d[ok]) for k in range(K)], -1) * ww[ok, None]
        ch = p[ok] >= n_up
        for c in (0, 1):
            u, v = U[ch == c], V[ch == c]
            mats[c] += 0.5 * (u.T @ v + v.T @ u)
            mags[c] += 0.5 * (u.abs().T @ v.abs() + v.abs().T @ u.abs())
            counts[c] += float((ch == c).sum())
        counts[2] += float((~ok).sum())
    return torch.cat([mats.reshape(-1), counts]), torch.cat([mags.reshape(-1), counts])


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--walkers", type=int, default=65536)
    p.add_argument("--moves", type=int, default=8)
    p.add_argument("--reps", type=int, default=5)
    p.add_argument("--scan-batches", type=int, default=4)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip()
    K, sigma = 36, 1.5
    _, n_sums = density_matrix_layout(K)
    failed = False
    for nup, ndown in ((10, 10), (12, 0)):
        n, B, M = nup + ndown, args.walkers, args.moves
        model = bench.build_model(argparse.Namespace(hidden=50, ode_steps=16, nup=nup, ndown=ndown, Z=2.0), dev)
        g = torch.Generator(device=dev).manual_seed(1)
        with torch.no_grad():
            _, x = model.sample((B,))
        particle = torch.randint(0, n, (B, M), device=dev, dtype=torch.int32, generator=g)
        rp = sigma * torch.randn(B, M, 2, device=dev, generator=g)
        disp = rp - torch.gather(x, 1, particle.long()[..., None].expand(B, M, 2))
        out = {}

        def ratio():
            out["ratio"] = model.wavefunction_ratio(x, particle, disp)

        t_ratio = timed(ratio, args.reps)
        w = out["ratio"] * ((2 * math.pi * sigma ** 2) * torch.exp((rp * rp).sum(-1) / (2 * sigma ** 2)))
        sums = torch.zeros(n_sums, device=dev)

        def acc():
            sums.zero_()
            density_matrix_accumulate(x, particle, disp, w, nup, ndown, K, sums)

        t_acc = timed(acc, args.reps)
        ref, mag = torch_sums(x, particle, disp, w, nup, K)
        err = float(((sums - ref).abs() / mag.clamp_min(1e-300)).max())
        counts_equal = bool(torch.equal(sums[-3:], ref[-3:]))
        ok = err <= 1e-12 and counts_equal
        scan = {}
        for s in (1.0, 1.5, 2.0, 3.0):
            est = DensityMatrixEstimator(nup, ndown, shells=7, sigma=s, moves=M, device=dev)
            gen = torch.Generator(device=dev).manual_seed(7)
            for _ in range(args.scan_batches):
                with torch.no_grad():
                    _, xs = model.sample((B,))
                est.accumulate(model, xs, generator=gen)
            r = est.result()
            d, e = np.diagonal(r["density_matrix"][0]), np.diagonal(r["density_matrix_err"][0])
            scan[str(s)] = dict(median_rel_err_diag=float(np.median(e / np.abs(d))),
                                trace=round(float(r["trace"][0]), 5), trace_err=float(r["trace_err"][0]),
                                leading_occupations=[round(float(v), 4) for v in r["occupations"][0][:nup + 2]])
        print(json.dumps(dict(n_up=nup, n_dn=ndown, walkers=B, moves=M, K=K, sigma=sigma,
                              wavefunction_ratio_ms=round(t_ratio, 2), density_matrix_accumulate_ms=round(t_acc, 3),
                              accumulate_share_of_ratio=round(t_acc / t_ratio, 5),
                              gfma_per_call=round(B * M * (K * (K + 1) // 2) * 2 / 1e9, 3),
                              torch_max_rel_diff=err, counts_equal=counts_equal, sums_agree=ok,
                              sigma_scan=scan, device=torch.cuda.get_device_name(dev), power_limit=power)))
        failed = failed or not ok
        del model, x, out, w, ref, mag
        torch.cuda.empty_cache()
    if failed:
        raise SystemExit("sums differ from the torch restatement")


if __name__ == "__main__":
    main()
