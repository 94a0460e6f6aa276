#!/usr/bin/env python
"""bench.py -- VMC walker-updates/s (sample + E_loc + grad) on the N = 20 ground-state quantum dot.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" is one VMC iteration of reference src/FermionHO2D.py's loop body on `--walkers`
walkers per GPU: Metropolis sampling of the base state, flow z -> x, local energy (log p,
its gradient and Laplacian), energy gradient w.r.t. the flow parameters, all-reduce of the
energy moments and the gradient, Adam update.  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

torch.set_default_dtype(torch.float64)

METRIC = "VMC walker-updates/s (sample+E_loc+grad) N=20"
UNIT = "walker-updates/s"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--walkers", type=int, default=65536,
                   help="walkers of the whole job (strong scaling: split over the GPUs) / per GPU (weak scaling)")
    p.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                   help="strong (BASELINE configs[2]: 65536 walkers sharded over 1/2/4/8 GPUs) or weak (--walkers per GPU)")
    p.add_argument("--nup", type=int, default=10)
    p.add_argument("--ndown", type=int, default=10)
    p.add_argument("--hidden", type=int, default=50, help="Deta = Dmu (reference default 50)")
    p.add_argument("--Z", type=float, default=2.0)
    p.add_argument("--ode-steps", type=int, default=16, help="RK4 steps across t_span")
    p.add_argument("--ref-walkers", type=int, default=32,
                   help="walkers per step of the CPU reference arm (a second, 4x smaller batch is timed beside it so "
                        "that the saturation of the CPU throughput with the batch is visible)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--config", default="n20", choices=["n20", "readme_finiteT", "strong_coupling", "slater_sweep"],
                   help="n20 (default; BASELINE configs[2], the configuration the metric is quoted on) | readme_finiteT "
                        "(configs[1]: beta 10, 3 up, Z 2, deltaE 2, Boltzmann sampler, 8000 walkers) | strong_coupling "
                        "(configs[3]: Z 8, N 12, 32 RK4 steps, finite T) | slater_sweep (configs[4]: log|det| + gradient + "
                        "Laplacian, N = 6..30, 1e6 walkers).  The extra configurations print the same JSON shape; the driver "
                        "runs the default only.")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write what the last one computed as DIR/<name>.npy (n20, --impl ours; "
                        "rank 0's walkers, a seeded sample of them when they exceed 60 MB)")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.config != "n20"):
        p.error("--dump-outputs covers the n20 configuration of --impl ours")
    return a


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [s.strip() for s in out.strip().split(",")]
                if len(f) >= 6:
                    self.rows.append(f)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        mhz = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None,
                "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None, "reasons": reasons}


def flops_per_walker_eloc(n, H_eta, H_mu, ode_steps, tables=True):
    """FP64 flop count of one E_loc sweep per walker (DESIGN.md, kernel `ff_eloc`).
    Per RK stage: radial functions of the P items + Jacobian GEMM 2 D^3 + Gram matrix 4 n (n+1) D +
    K u 2 D^2 + per-particle sums 22 n (n-1) + RK combinations 3 D^2.
    tables=True  (what the kernel executes): certified degree-11 Taylor tables, 76 flop (Horner for f and its three
                 derivatives without the zero steps) + 70 flop of geometry + 22 flop (the item's share of A L) per item;
                 the RK combination of K is the initial value of the tensor-core accumulators (1.25 FMA per element);
    tables=False (reference formulation, option no_table): 43 flop per item AND hidden unit (sigmoid 21,
                 pre-activation 2, three derivative factors 8, four accumulations 8, geometry amortised), A L as a
                 matrix-vector product, two-partial RK update."""
    D, NP = 2 * n, n * (n - 1) // 2
    P = NP + (n if H_mu else 0)
    if tables:
        per_stage = (76 + 70 + 22) * P + 2 * D ** 3 + 4 * n * (n + 1) * D + 2 * D * D + 22 * n * (n - 1) + 3 * D * D
    else:
        per_stage = 43 * (NP * H_eta + n * H_mu) + 2 * D ** 3 + 4 * n * (n + 1) * D + 4 * D * D + 22 * n * (n - 1) + 6 * D * D
    return 4 * ode_steps * per_stage


def hbm_bytes_per_walker_eloc(n, has_mu, ode_steps):
    """coordinates in, adjoint stash out (stage inputs + three radial values per item), results out, and the final
    state of the sweep (y, L, gDelta, Delta, lapDelta, J) written once and read once by the finale kernel"""
    D, P = 2 * n, n * (n - 1) // 2 + (n if has_mu else 0)
    return 8 * (D + 4 * ode_steps * (D + 3 * P) + 2 * D + 6 + 2 * (3 * D + 2 + D * D))


def build_model(args, dev):
    from fermiflow_b200 import MLP, Backflow, CNF, HO2D, FreeFermion, GSVMC, HO, CoulombPairPotential
    eta, mu = MLP(1, args.hidden), MLP(1, args.hidden)
    # random-init weights of the reference architecture (FermionHO2D.py uses zeros, which
    # would make the flow trivial; a 1e-2-scale Gaussian keeps every code path live)
    g = torch.Generator().manual_seed(42)
    with torch.no_grad():
        for m in (eta, mu):
            m.fc1.weight.copy_(torch.randn(m.fc1.weight.shape, generator=g))
            m.fc1.bias.copy_(torch.randn(m.fc1.bias.shape, generator=g))
            m.fc2.weight.copy_(1e-2 * torch.randn(m.fc2.weight.shape, generator=g))
    cnf = CNF(Backflow(eta, mu=mu), (0.0, 1.0), nsteps=args.ode_steps)
    model = GSVMC(args.nup, args.ndown, HO2D(), FreeFermion(dev), cnf, CoulombPairPotential(args.Z), sp_potential=HO())
    return model.to(dev)


DUMP_BYTES = 60 << 20


def dump_outputs(out_dir, model):
    """What a caller of one VMC iteration receives, as float64 .npy files: the per-walker results of the E_loc sweep
    (model.last), the energy estimate, the parameter gradients and the parameters after the optimiser step.  Runs of
    the same arguments see the same inputs, so two builds can be compared file by file."""
    import numpy as np
    last = model.last
    per_walker = {k: getattr(last, k) for k in ("z", "delta_logp", "logp", "grad", "lap", "kinetic", "potential", "eloc")}
    B = last.eloc.shape[0]
    row_bytes = sum(t[0].numel() * 8 for t in per_walker.values())
    rows = None
    if B * row_bytes > DUMP_BYTES:
        keep = DUMP_BYTES // row_bytes
        rows = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:keep].sort().values.to(last.eloc.device)
    arrays = {"walker_" + k: t if rows is None else t[rows] for k, t in per_walker.items()}
    arrays["energy"] = model.observables_device()             # E, E_std
    for name, p in model.named_parameters():
        arrays["param." + name] = p.detach()
        arrays["param_grad." + name] = p.grad
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().to("cpu", torch.float64).numpy())


def run_ours(args):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL writes its version banner and debug lines (NCCL_DEBUG >= VERSION) to stdout by default, before the
        # JSON line: send them to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":      # NCCL honours the file only above VERSION
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    from fermiflow_b200 import _lib as L
    import ctypes as C

    model = build_model(args, dev)
    model.basedist.manual_seed(1000)          # FreeFermion offsets the Philox walker index by rank * B
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    B = args.walkers // world if args.scaling == "strong" else args.walkers      # walkers of this rank
    params = list(model.parameters())
    nparam = sum(p.numel() for p in params)

    # kernel-level timing of the dominant kernel (ff_eloc) with CUDA events on the launch stream
    from fermiflow_b200 import utils as U
    eloc_events = []
    orig_sweep = U.eloc_sweep

    def timed_sweep(*a, **k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = orig_sweep(*a, **k)
        e1.record()
        eloc_events.append((e0, e1))
        return r
    import fermiflow_b200.VMC as V
    V.eloc_sweep = timed_sweep

    def step():
        gradE = model(B)
        opt.zero_grad(set_to_none=True)
        gradE.backward()
        model.allreduce_gradients()
        opt.step()
        return model.E

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    # FP64 roofline denominator, measured on this device (MEASURED_PEAKS.json has no fp64 entry)
    peak = C.c_double()
    L.check(L.lib().ff_fp64_peak(20000, C.byref(peak), None))
    eloc_events.clear()
    launches0 = L.lib().ff_launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    E = None
    for _ in range(args.steps):
        E = step()
    t1.record()
    barrier()
    launches = L.lib().ff_launch_count() - launches0
    ms = t0.elapsed_time(t1)
    eloc_ms = sum(a.elapsed_time(b) for a, b in eloc_events) / max(len(eloc_events), 1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model)

    # end-to-end through the public API with HOST buffers: parameters come from pinned host
    # memory every step, energy moments and the gradient go back to the host.
    host_params = torch.cat([p.detach().reshape(-1) for p in params]).cpu().pin_memory()
    host_out = torch.empty(nparam + 2, dtype=torch.float64).pin_memory()
    dev_params = torch.empty(nparam, device=dev)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        dev_params.copy_(host_params, non_blocking=True)
        o = 0
        with torch.no_grad():
            for p in params:
                p.copy_(dev_params[o:o + p.numel()].view_as(p))
                o += p.numel()
        gradE = model(B)
        opt.zero_grad(set_to_none=True)
        gradE.backward()
        model.allreduce_gradients()
        flat = torch.cat([p.grad.reshape(-1) for p in params] + [model.observables_device()])
        host_out.copy_(flat, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # per-stage breakdown of one step (outside the timed regions; CUDA events on the launch stream)
    def ev_time(f):
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(); r = f(); a1.record(); torch.cuda.synchronize()
        return a0.elapsed_time(a1), r
    bd = {}
    bd["metropolis_ms"], z = ev_time(lambda: model.basedist.sample(model.orbitals_up, model.orbitals_down, (B,)))
    bd["flow_generate_ms"], x = ev_time(lambda: model.cnf.generate(z))
    del z, x
    bd["eloc_sweep_ms"] = eloc_ms
    t_fwd, gradE = ev_time(lambda: model(B))
    opt.zero_grad(set_to_none=True)
    bd["backward_ms"], _ = ev_time(lambda: gradE.backward())
    bd["forward_total_ms"] = t_fwd
    del gradE

    tms = torch.tensor([ms, e2e_ms], device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms, e2e_ms = tms.tolist()
    total_walkers = B * world * args.steps
    value = total_walkers / (ms * 1e-3)
    n = args.nup + args.ndown
    tables_on = L.get_option("no_table") == 0
    fl = flops_per_walker_eloc(n, args.hidden, args.hidden, args.ode_steps, tables=tables_on) * B
    by = hbm_bytes_per_walker_eloc(n, True, args.ode_steps) * B
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "ground-state 2D quantum dot N=%d (%d up/%d down), %d walkers in total (%d per GPU), Z=%.1f, "
                               "Deta=Dmu=%d, %d RK4 steps" % (n, args.nup, args.ndown, B * world, B, args.Z, args.hidden, args.ode_steps),
                   "walkers_total": B * world, "walkers_per_gpu": B, "ode_steps": args.ode_steps,
                   "l2_policy": "inputs larger than L2 (per step: 21 MB coordinates, >20 GB stash streamed)",
                   "parallelism": "walkers sharded, dp%d" % world},
        "e2e": {"value": total_walkers / (e2e_ms * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": nparam * 8, "d2h_bytes_per_step": (nparam + 2) * 8},
        "gpu_launches": int(launches),     # counted by the library (ff_launch_count) over the timed steps of this rank
        "clocks": sampler.summary(),
        "breakdown_ms": {k: round(v, 2) for k, v in bd.items()},
        "roofline": {"bound": "fp64", "kernel": "ff_eloc: ff::eloc5_kernel<20,1> (E_loc sweep, 97 % of the call) + ff::eloc_finale_warp_kernel + table build", "achieved": fl / (eloc_ms * 1e-3) / 1e12,
                     "peak": peak.value / 1e12, "unit": "TFLOP/s", "frac": fl / (eloc_ms * 1e-3) / peak.value,
                     "peak_source": "ff_fp64_peak DFMA microbenchmark on this device (MEASURED_PEAKS.json has no fp64 entry)",
                     "flops_counted": "executed formulation (radial functions from certified Taylor tables)" if tables_on
                                      else "reference formulation (every hidden unit evaluated)",
                     # ncu --set full (profiles/r02_eloc5_ncu_full.md, r02_finale_ncu_full.md): sweep 3.324 GB written + 0.004 GB
                     # read, finale 0.134 GB read + 0.005 GB written for 9472 walkers
                     "traffic": 3.4663e9 / 9472 * B if (n == 20 and args.hidden == 50 and args.ode_steps == 16) else None,
                     "traffic_source": "ncu dram__bytes_read+write, 9472-walker capture scaled per walker",
                     "kernel_ms": eloc_ms,
                     "hbm": {"achieved": by / (eloc_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": by / (eloc_ms * 1e-3) / 1e9 / hbm_peak}},
        "energy": E,
    }
    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(args, budget_s=40.0)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


FINITE_T = {   # BASELINE.json configs[1] and configs[3] (reference: src/BetaFermionHO2D.py command lines)
    "readme_finiteT": dict(beta=10.0, nup=3, ndown=0, Z=2.0, deltaE=2.0, nsteps=16, batch=8000,
                           what="README finite-T run (--beta 10.0 --nup 3 --Z 2.0 --deltaE 2.0 --boltzmann)"),
    "strong_coupling": dict(beta=2.0, nup=12, ndown=0, Z=8.0, deltaE=2.0, nsteps=32, batch=8000,
                            what="strong-coupling Wigner-molecule regime (--beta 2.0 --nup 12 --Z 8.0 --deltaE 2.0 --boltzmann, 32 RK4 steps)"),
}


def run_config(args):
    """The other BASELINE configurations on one GPU, same JSON shape as the default line (device-timed value, end-to-end
    value through host buffers, roofline of the dominant kernel, CPU baseline of the reference algorithm)."""
    import ctypes as C
    from fermiflow_b200 import _lib as L
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    peak = C.c_double()
    L.check(L.lib().ff_fp64_peak(20000, C.byref(peak), None))
    sampler = ClockSampler(0)
    if args.config == "slater_sweep":
        return run_slater_sweep(args, dev, peak.value, sampler)
    from fermiflow_b200 import MLP, Backflow, CNF, HO2D, FreeFermion, BetaVMC, HO, CoulombPairPotential
    from fermiflow_b200 import utils as U
    import fermiflow_b200.VMC as V
    cfg = FINITE_T[args.config]
    n = cfg["nup"] + cfg["ndown"]
    g = torch.Generator().manual_seed(42)
    eta, mu = MLP(1, args.hidden), MLP(1, args.hidden)
    with torch.no_grad():
        for m in (eta, mu):
            m.fc1.weight.copy_(torch.randn(m.fc1.weight.shape, generator=g))
            m.fc1.bias.copy_(torch.randn(m.fc1.bias.shape, generator=g))
            m.fc2.weight.copy_(1e-2 * torch.randn(m.fc2.weight.shape, generator=g))
    cnf = CNF(Backflow(eta, mu=mu), (0.0, 1.0), nsteps=cfg["nsteps"])
    model = BetaVMC(cfg["beta"], cfg["nup"], cfg["ndown"], cfg["deltaE"], True, HO2D(), FreeFermion(dev), cnf,
                    CoulombPairPotential(cfg["Z"]), sp_potential=HO()).to(dev)
    model.basedist.manual_seed(1000)
    opt = torch.optim.Adam(model.parameters(), lr=1e-2)
    B = cfg["batch"]
    params = list(model.parameters())
    nparam = sum(p.numel() for p in params)
    eloc_events = []
    orig_sweep = U.eloc_sweep

    def timed_sweep(*a, **k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); r = orig_sweep(*a, **k); e1.record()
        eloc_events.append((e0, e1))
        return r
    V.eloc_sweep = timed_sweep

    def step():
        gphi, gtheta = model(B)
        opt.zero_grad(set_to_none=True)
        gphi.backward(); gtheta.backward()
        opt.step()

    steps, warmup = max(args.steps, 20), max(args.warmup, 5)
    for _ in range(warmup):
        step()
    # the cost of an iteration depends on the state of the optimisation (node ranges of the binned gradient, records
    # beyond them): both timed loops start from this snapshot and see the same sequence of iterations
    import copy
    snap = (copy.deepcopy(model.state_dict()), copy.deepcopy(opt.state_dict()))
    eloc_events.clear()
    launches0 = L.lib().ff_launch_count()
    sampler.start()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        step()
    t1.record(); torch.cuda.synchronize()
    ms = t0.elapsed_time(t1)
    launches = L.lib().ff_launch_count() - launches0
    eloc_ms = sum(a.elapsed_time(b) for a, b in eloc_events) / max(len(eloc_events), 1)
    model.load_state_dict(snap[0]); opt.load_state_dict(snap[1])
    host_params = torch.cat([p.detach().reshape(-1) for p in params]).cpu().pin_memory()
    host_out = torch.empty(nparam + 5, dtype=torch.float64).pin_memory()
    dev_params = torch.empty(nparam, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        dev_params.copy_(host_params, non_blocking=True)
        o = 0
        with torch.no_grad():
            for p in params:
                p.copy_(dev_params[o:o + p.numel()].view_as(p)); o += p.numel()
        gphi, gtheta = model(B)
        opt.zero_grad(set_to_none=True)
        gphi.backward(); gtheta.backward()
        opt.step()                        # the optimisation goes on as in the device-timed loop (the cost of a step depends on the state)
        obs = torch.stack([getattr(model, "_obs_dev")[k].reshape(()) for k in ("E", "E_std", "F", "F_std", "S")])
        host_out.copy_(torch.cat([p.grad.reshape(-1) for p in params] + [obs]), non_blocking=True)
        host_params.copy_(torch.cat([p.detach().reshape(-1) for p in params]), non_blocking=True)     # next step's input
        torch.cuda.current_stream().synchronize()
    e1.record(); torch.cuda.synchronize()
    e2e_ms = e0.elapsed_time(e1)
    sampler.stop_flag = True; sampler.join(timeout=2)
    fl = flops_per_walker_eloc(n, args.hidden, args.hidden, cfg["nsteps"], tables=L.get_option("no_table") == 0) * B
    line = {
        "metric": "VMC walker-updates/s (sample+E_loc+grad), " + args.config, "value": B * steps / (ms * 1e-3), "unit": UNIT,
        "n_gpus": 1, "steps": steps, "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s: N=%d, %d many-body states, %d walkers per iteration, Deta=Dmu=%d, %d RK4 steps" % (
            cfg["what"], n, model.Nstates, B, args.hidden, cfg["nsteps"]), "walkers_total": B, "ode_steps": cfg["nsteps"],
            "l2_policy": "inputs smaller than L2 (8000 walkers); every iteration writes and reads its own adjoint stash (%.2f GB)" % (
                hbm_bytes_per_walker_eloc(n, True, cfg["nsteps"]) * B / 1e9)},
        "e2e": {"value": B * steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": nparam * 8, "d2h_bytes_per_step": (2 * nparam + 5) * 8},
        "gpu_launches": int(launches), "clocks": sampler.summary(),
        "roofline": {"bound": "fp64", "kernel": "ff_eloc (E_loc sweep of the %d-particle block)" % n, "achieved": fl / (eloc_ms * 1e-3) / 1e12,
                     "peak": peak.value / 1e12, "unit": "TFLOP/s", "frac": fl / (eloc_ms * 1e-3) / peak.value,
                     "peak_source": "ff_fp64_peak DFMA microbenchmark on this device", "traffic": None, "kernel_ms": eloc_ms},
        "F": model.F, "F_std": model.F_std, "E": model.E, "S": model.S,
    }
    if not args.no_cpu_baseline:
        # the reference algorithm at the same particle number on the host cores (ground-state occupation for every walker:
        # the per-walker cost of the multi-state Slater determinant is the same)
        from oracle import reference_port as R
        torch.set_num_threads(os.cpu_count() or 1)
        R.time_vmc_iteration(cfg["nup"], cfg["ndown"], args.hidden, cfg["Z"], 1, seed=1, equil=2)
        w = 16 if n > 6 else 64
        t = R.time_vmc_iteration(cfg["nup"], cfg["ndown"], args.hidden, cfg["Z"], w, seed=7)
        line["cpu_baseline"] = {"value": w / t, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "ref_walkers": w,
                                "sample": "1 VMC iteration of %d walkers of the %s (ground-state occupation for every walker)" % (w, _ref_note(n))}
    print(json.dumps(line))


def run_slater_sweep(args, dev, peak, sampler):
    """BASELINE configs[4]: batched log|det| + gradient + exact Laplacian of the free-fermion state, N = 6..30 (N/2 up, N/2
    down), 1e6 walkers, against the reference's autograd path (slogdet + 1 + 2N nested passes, utils.py:44-65) on the host."""
    from fermiflow_b200 import HO2D, FreeFermion, _lib as L
    from oracle import fermiflow_oracle as O
    B, cpu_walkers = 1000000, 4096
    ho, ffm = HO2D(), FreeFermion(dev)
    torch.set_num_threads(os.cpu_count() or 1)
    rows = []
    sampler.start()
    launches0 = L.lib().ff_launch_count()
    for N in range(6, 31, 2):
        nup = N // 2
        up, dn = ho.orbitals[:nup], ho.orbitals[:N - nup]
        x = 1.2 * torch.randn(B, N, 2, device=dev)
        xh = x.cpu().pin_memory()
        for _ in range(3):
            ffm.log_prob_grad_laplacian(up, dn, x)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ts = []
        for _ in range(5):
            e0.record(); logp, grad, lap = ffm.log_prob_grad_laplacian(up, dn, x); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ms = sorted(ts)[len(ts) // 2]
        # end to end: coordinates from pinned host memory, log p / gradient / Laplacian back to the host
        out_h = [torch.empty_like(t, device="cpu").pin_memory() for t in (logp, grad, lap)]
        te = []
        for _ in range(3):
            e0.record()
            xd = xh.to(dev, non_blocking=True)
            res = ffm.log_prob_grad_laplacian(up, dn, xd)
            for o, r in zip(out_h, res):
                o.copy_(r, non_blocking=True)
            e1.record(); torch.cuda.synchronize()
            te.append(e0.elapsed_time(e1))
        e2e_ms = sorted(te)[1]
        row = {"N": N, "gpu_ms": round(ms, 3), "walkers_per_s": B / ms * 1e3, "e2e_walkers_per_s": B / e2e_ms * 1e3}
        if not args.no_cpu_baseline:
            xc = x[:cpu_walkers].cpu()
            O.free_fermion_grad_laplacian(list(range(nup)), list(range(N - nup)), xc[:64])      # warm-up
            t = time.time()
            lp_ref, g_ref, l_ref = O.free_fermion_grad_laplacian(list(range(nup)), list(range(N - nup)), xc)
            tc = time.time() - t
            row["cpu_walkers_per_s"] = cpu_walkers / tc
            row["max_rel_err_vs_oracle"] = max(float((logp[:cpu_walkers].cpu() - lp_ref).abs().max() / lp_ref.abs().max()),
                                               float((grad[:cpu_walkers].cpu() - g_ref).abs().max() / g_ref.abs().max()),
                                               float((lap[:cpu_walkers].cpu() - l_ref).abs().max() / l_ref.abs().max()))
        rows.append(row)
    sampler.stop_flag = True; sampler.join(timeout=2)
    r20 = [r for r in rows if r["N"] == 20][0]
    ns = 10
    # executed flops per walker at N = 20 (two 10 x 10 blocks): Gauss-Jordan on [Phi | I] 2 ns^2 (2 ns) + orbitals and the
    # Jacobi-formula contractions 8 ns^2 + 1D oscillator tables 2 ns * 8 * 10
    fl = 2 * (2 * ns * ns * 2 * ns + 8 * ns * ns + 2 * ns * 80)
    hbm = (20 * 2 + 20 * 2 + 2) * 8.0
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    line = {
        "metric": "batched log|det| + gradient + exact Laplacian, walkers/s at N=20 (sweep N=6..30)", "value": r20["walkers_per_s"],
        "unit": "walkers/s", "n_gpus": 1, "steps": 5, "warmup": 3, "ms_per_step": r20["gpu_ms"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "kernel microbench: free-fermion log|det| + gradient + Laplacian, N = 6..30 (N/2 up, N/2 down), 1e6 walkers",
                   "walkers_total": B, "l2_policy": "inputs larger than L2 from N = 8 on (16 N bytes in, 16 N + 16 out per walker)"},
        "e2e": {"value": r20["e2e_walkers_per_s"], "unit": "walkers/s", "h2d_bytes_per_step": B * 40 * 8, "d2h_bytes_per_step": B * 42 * 8},
        "gpu_launches": int(L.lib().ff_launch_count() - launches0), "clocks": sampler.summary(),
        "roofline": {"bound": "fp64", "kernel": "ff::slater_warp_kernel (one warp per walker)", "achieved": fl * r20["walkers_per_s"] / 1e12,
                     "peak": peak / 1e12, "unit": "TFLOP/s", "frac": fl * r20["walkers_per_s"] / peak, "traffic": None,
                     "peak_source": "ff_fp64_peak DFMA microbenchmark on this device",
                     "hbm": {"achieved": hbm * r20["walkers_per_s"] / 1e9, "peak": peaks.get("hbm_gbs", 6650.0), "unit": "GB/s",
                             "frac": hbm * r20["walkers_per_s"] / 1e9 / peaks.get("hbm_gbs", 6650.0)},
                     "note": "latency / issue bound: shuffle-based pivot search and rank-1 updates of 10 x 21 matrices"},
        "sweep": rows,
    }
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = {"value": r20["cpu_walkers_per_s"], "unit": "walkers/s", "cores": torch.get_num_threads(), "kind": "port",
                                "sample": "%d walkers per N through the reference's path (torch slogdet + 1 + 2N nested autograd passes, "
                                          "oracle/fermiflow_oracle.py free_fermion_grad_laplacian), one warm-up call" % cpu_walkers}
    print(json.dumps(line))


def _ref_note(n):
    return ("reference algorithm ported to torch-CPU (oracle/reference_port.py: dopri5 rtol 1e-6 + continuous adjoint + "
            "2N nested autograd passes, N=%d); /root/reference is plain Python and needs the absent torchdiffeq" % n)


def cpu_baseline(args, budget_s):
    """The reference's own algorithm (adaptive dopri5, adjoint, nested-autograd Laplacian) ported to torch-CPU
    (oracle/reference_port.py): one VMC iteration at two batch sizes, so that the saturation of the CPU throughput
    with the batch is visible (the reference's default batch is 8000, FermionHO2D.py:30; its per-walker cost falls
    with the batch until the BLAS / autograd overheads are amortised)."""
    from oracle import reference_port as R
    torch.set_num_threads(os.cpu_count() or 1)
    n = args.nup + args.ndown
    R.time_vmc_iteration(args.nup, args.ndown, args.hidden, args.Z, 1, seed=1, equil=2)       # warm-up (thread pools, allocator)
    small = max(2, args.ref_walkers // 8)
    t_small = R.time_vmc_iteration(args.nup, args.ndown, args.hidden, args.Z, small, seed=7)
    # second point: as large as the budget allows (cost grows ~ batch^0.6 in this range), at most --ref-walkers / 2
    big = small
    while big * 2 <= max(args.ref_walkers // 2, small) and t_small * (big * 2 / small) ** 0.6 < budget_s:
        big *= 2
    pts = [{"walkers": small, "value": small / t_small, "seconds": round(t_small, 1)}]
    if big > small:
        t_big = R.time_vmc_iteration(args.nup, args.ndown, args.hidden, args.Z, big, seed=8)
        pts.append({"walkers": big, "value": big / t_big, "seconds": round(t_big, 1)})
    best = max(pts, key=lambda q: q["value"])
    return {"value": best["value"], "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "ref_walkers": best["walkers"], "batch_points": pts,
            "sample": "1 VMC iteration of %d walkers (and one of %d) of the %s" % (best["walkers"], pts[0]["walkers"], _ref_note(n))}


def run_reference(args):
    """--impl reference: the reference's CPU path on the host cores, K timed steps of `--ref-walkers` walkers (reduced
    until K steps fit ~8 minutes), plus single steps at other batch sizes as further data points."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from oracle import reference_port as R
    torch.set_num_threads(os.cpu_count() or 1)
    n = args.nup + args.ndown
    for _ in range(max(1, min(args.warmup, 1))):
        R.time_vmc_iteration(args.nup, args.ndown, args.hidden, args.Z, 1, seed=1, equil=2)
    # K timed steps must fit a few minutes: their batch is the largest power-of-two fraction of --ref-walkers for which
    # K steps take at most ~8 minutes (the cost of a step grows ~ batch^0.6 in this range); ONE extra step at --ref-walkers is
    # timed beside them so that the saturation of the CPU throughput with the batch is on record (the reference's default
    # batch is 8000, FermionHO2D.py:30; 32 walkers of N = 20 take ~46 s on 16 threads)
    t_start = time.time()
    small = max(2, args.ref_walkers // 4)
    t_small = R.time_vmc_iteration(args.nup, args.ndown, args.hidden, args.Z, small, seed=5)
    walkers = args.ref_walkers
    while walkers > max(2, small // 2) and args.steps * t_small * (walkers / small) ** 0.6 > 480.0:
        walkers //= 2
    ts = [R.time_vmc_iteration(args.nup, args.ndown, args.hidden, args.Z, walkers, seed=10 + i) for i in range(args.steps)]
    tot = sum(ts)
    value = walkers * args.steps / tot
    pts = [{"walkers": small, "value": small / t_small, "seconds": round(t_small, 1)}]
    if walkers != small:
        pts.append({"walkers": walkers, "value": value, "seconds": round(tot / args.steps, 1)})
    if walkers < args.ref_walkers and time.time() - t_start < 600.0:
        t_big = R.time_vmc_iteration(args.nup, args.ndown, args.hidden, args.Z, args.ref_walkers, seed=99)
        pts.append({"walkers": args.ref_walkers, "value": args.ref_walkers / t_big, "seconds": round(t_big, 1)})
    pts.sort(key=lambda q: q["walkers"])
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "ground-state 2D quantum dot N=%d (%d up/%d down), Z=%.1f, Deta=Dmu=%d; bounded sample of "
                               "%d walkers per step on the host CPU" % (n, args.nup, args.ndown, args.Z, args.hidden, walkers),
                   "ref_walkers": walkers, "cores": torch.get_num_threads()},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                         "ref_walkers": walkers, "batch_points": pts,
                         "sample": "%d VMC iterations of %d walkers (batch_points: single iterations at other batch sizes) of the %s" % (args.steps, walkers, _ref_note(n))},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.config == "n20":
        run_ours(a)
    else:
        run_config(a)
