"""Time of ff_swap_ratio (split into the flow sweep over the 2 P (Q + 1) configurations and the rest: building the
swapped configurations, the Slater determinants with their signs, the pair ratios) and of ff_swap_accumulate, at 65536
walkers randomly paired (P = 32768) and Q = 8 disks of radii 0.5 ... 4, for N = 20 (10 + 10) and N = 12 (12 + 0).  The
sums are checked against a torch restatement (index_add; counts exactly, ratio sums to 1e-12 of the sum of |ratio|
per cell), and the VMC step time of the same model is printed for scale.  CUDA events after warm-up; one JSON line
per particle number, with the device name and power limit."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from fermiflow_b200.observables import swap_accumulate, swap_layout  # noqa: E402

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


def torch_sums(ratio, sector, n_up, n_dn):
    """The layout of ff_swap_accumulate restated in torch, and the sum of |ratio| per cell."""
    P, Q = ratio.shape
    ns = (n_up + 1) * (n_dn + 1)
    dev = ratio.device
    s0, s1 = sector[:, 0].long(), sector[:, 1].long()
    ok = (s0 >= 0) & (s0 < ns) & (s1 >= 0) & (s1 < ns)
    cell = torch.arange(Q, device=dev)[None] * ns
    one = torch.ones(P, Q, device=dev)
    rep = torch.zeros(Q * ns, device=dev).index_add_(0, (cell + s0)[ok], one[ok]).index_add_(0, (cell + s1)[ok], one[ok])
    m = ok & (s0 == s1)
    rsum = torch.zeros(Q * ns, device=dev).index_add_(0, (cell + s0)[m], ratio[m])
    mat = torch.zeros(Q * ns, device=dev).index_add_(0, (cell + s0)[m], one[m])
    absum = torch.zeros(Q * ns, device=dev).index_add_(0, (cell + s0)[m], ratio[m].abs())
    return torch.cat([rsum, rep, mat, (~ok).sum(0).double(), torch.tensor([float(P)], device=dev)]), absum


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--walkers", type=int, default=65536)
    p.add_argument("--regions", type=int, default=8)
    p.add_argument("--reps", type=int, default=5)
    p.add_argument("--vmc-steps", type=int, default=3)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip()
    a = [0.5 * (q + 1) for q in range(args.regions)]
    failed = False
    for nup, ndown in ((10, 10), (12, 0)):
        n, B, Q = nup + ndown, args.walkers, len(a)
        model = bench.build_model(argparse.Namespace(hidden=50, ode_steps=16, nup=nup, ndown=ndown, Z=2.0), dev)
        g = torch.Generator(device=dev).manual_seed(1)
        with torch.no_grad():
            _, x = model.sample((B,))
        P = B // 2
        pairs = torch.randperm(B, device=dev, generator=g)[:2 * P].view(P, 2)
        out = {}

        def swap():
            out["r"] = model.swap_ratio(x, pairs, a)

        t_swap = timed(swap, args.reps)
        del out["r"]
        # the flow sweep alone on 2 P (Q + 1) configurations of the same size
        xc = x[pairs.reshape(-1).long()][:, None].expand(2 * P, Q + 1, n, 2).reshape(-1, n, 2).contiguous()
        with torch.no_grad():
            t_flow = timed(lambda: model.cnf.delta_logp(xc), args.reps)
        del xc
        swap()
        ratio, sector = out["r"]
        lay, n_sums = swap_layout(Q, nup, ndown)
        sums = torch.zeros(n_sums, device=dev)

        def acc():
            sums.zero_()
            swap_accumulate(ratio, sector, nup, ndown, sums)

        t_acc = timed(acc, args.reps)
        ref, absum = torch_sums(ratio, sector, nup, ndown)
        k = lay["replicas"][0]
        counts_equal = bool(torch.equal(sums[k:], ref[k:]))
        err = float(((sums[:k] - ref[:k]).abs() - 1e-12 * absum).max())
        ok = counts_equal and err <= 0

        def step():
            model(B).backward()

        t_step = timed(step, args.vmc_steps)
        new = t_swap - t_flow + t_acc
        swap_est = (sums[:k].reshape(Q, -1).sum(1) / P).tolist()
        print(json.dumps(dict(n_up=nup, n_dn=ndown, walkers=B, pairs=P, radii=a,
                              swap_ratio_ms=round(t_swap, 2), flow_sweep_ms=round(t_flow, 2),
                              swap_rest_ms=round(t_swap - t_flow, 3), swap_accumulate_ms=round(t_acc, 3),
                              new_kernels_share_of_flow=round(new / t_flow, 4),
                              counts_equal=counts_equal, sums_agree=ok,
                              swap_estimate=[round(v, 5) for v in swap_est],
                              negative_ratio_fraction=round(float((ratio < 0).double().mean()), 4),
                              vmc_step_ms=round(t_step, 2),
                              device=torch.cuda.get_device_name(dev), power_limit=power)))
        failed = failed or not ok
        del model, x, ratio, sector, out, ref
        torch.cuda.empty_cache()
    if failed:
        raise SystemExit("sums differ from the torch restatement")


if __name__ == "__main__":
    main()
