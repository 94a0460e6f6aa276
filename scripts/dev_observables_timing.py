"""Time of ff_observables (all four sections: n_xy = n_rot = 64, n_r = 128, extent = r_max = 6) at 65536 walkers for
N = 20 (10 + 10) and N = 12 (12 + 0), against the same counts formed with torch (bincount over the materialised pair
tensors: the oracle of tests/test_gpu_observables.py), checked equal, and the VMC step time of the same model for scale.
CUDA events after warm-up; prints one JSON line per particle number, with the device name and power limit."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

import bench  # noqa: E402
from fermiflow_b200.observables import count_layout, observables  # noqa: E402
from test_gpu_observables import oracle  # noqa: E402

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


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--walkers", type=int, default=65536)
    p.add_argument("--reps", type=int, default=20)
    p.add_argument("--vmc-steps", type=int, default=3)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip()
    grid = dict(extent=6.0, n_xy=64, r_max=6.0, n_r=128, n_rot=64)
    _, nb = count_layout(grid["n_xy"], grid["n_r"], grid["n_rot"])
    for nup, ndown in ((10, 10), (12, 0)):
        n, B = nup + ndown, args.walkers
        model = bench.build_model(argparse.Namespace(hidden=50, ode_steps=16, nup=nup, ndown=ndown, Z=2.0), dev)
        with torch.no_grad():
            _, x = model.sample((B,))
        counts = torch.zeros(nb + 9, dtype=torch.int64, device=dev)

        def kernel():
            counts.zero_()
            observables(x, nup, ndown, grid["extent"], grid["n_xy"], grid["r_max"], grid["n_r"], grid["n_rot"], counts)

        t_kernel = timed(kernel, args.reps)
        ref = {}

        def torch_counts():
            ref["c"] = oracle(x, nup, chunk=B, **grid)

        t_torch = timed(torch_counts, max(2, args.reps // 5))
        kernel()
        equal = bool(torch.equal(counts, ref["c"]))

        def step():
            model(B).backward()

        t_step = timed(step, args.vmc_steps)
        items = 2 * n + n * (n - 1) // 2 + n * (n - 1)
        print(json.dumps(dict(n_up=nup, n_dn=ndown, walkers=B, items_per_walker=items, grid=grid,
                              observables_ms=round(t_kernel, 4), torch_bincount_ms=round(t_torch, 3),
                              counts_equal=equal, vmc_step_ms=round(t_step, 2),
                              G_items_per_s=round(items * B / (t_kernel * 1e-3) / 1e9, 2),
                              device=torch.cuda.get_device_name(dev), power_limit=power)))
        if not equal:
            raise SystemExit("counts differ from the torch restatement")
        del model, x, ref
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
