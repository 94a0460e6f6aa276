"""Ground-state VMC of the 2D quantum dot -- mirror of reference src/FermionHO2D.py.

    python -m fermiflow_b200.FermionHO2D --nup 3 --ndown 3 --Z 2.0 --batch 8000 --iternum 100

Same options as the reference plus --nsteps (fixed RK4 steps of the flow)."""
import argparse
import time

import torch

from .MLP import MLP
from .VMC import GSVMC
from .base_dist import FreeFermion
from .equivariant_funs import Backflow
from .flow import CNF
from .observables import add_driver_options, run_driver_options
from .orbitals import HO2D
from .potentials import HO, CoulombPairPotential


def main(argv=None):
    p = argparse.ArgumentParser(description="Ground-state variational Monte Carlo simulation")
    p.add_argument("--nup", type=int, default=6)
    p.add_argument("--ndown", type=int, default=0)
    p.add_argument("--Z", type=float, default=0.5)
    p.add_argument("--cuda", type=int, default=0)
    p.add_argument("--Deta", type=int, default=50)
    p.add_argument("--nomu", action="store_true")
    p.add_argument("--Dmu", type=int, default=50)
    p.add_argument("--t0", type=float, default=0.0)
    p.add_argument("--t1", type=float, default=1.0)
    p.add_argument("--nsteps", type=int, default=16)
    p.add_argument("--iternum", type=int, default=1000)
    p.add_argument("--batch", type=int, default=8000)
    p.add_argument("--lr", type=float, default=1e-2)
    add_driver_options(p)
    args = p.parse_args(argv)

    device = torch.device("cuda:%d" % args.cuda)
    eta = MLP(1, args.Deta); eta.init_zeros()
    mu = None
    if not args.nomu:
        mu = MLP(1, args.Dmu); mu.init_zeros()
    cnf = CNF(Backflow(eta, mu=mu), (args.t0, args.t1), nsteps=args.nsteps)
    model = GSVMC(args.nup, args.ndown, HO2D(), FreeFermion(device=device), cnf,
                  CoulombPairPotential(args.Z), sp_potential=HO()).to(device)
    print("nup = %d, ndown = %d, Z = %.1f" % (args.nup, args.ndown, args.Z))
    optimizer = torch.optim.Adam(model.parameters(), lr=args.lr)
    print("batch = %d, iternum = %d." % (args.batch, args.iternum))
    history = []
    for i in range(1, args.iternum + 1):
        start = time.time()
        gradE = model(args.batch)
        optimizer.zero_grad()
        gradE.backward()
        model.allreduce_gradients()
        optimizer.step()
        history.append((model.E, model.E_std))
        print("iter: %03d" % i, "E:", model.E, "E_std:", model.E_std,
              "Instant speed (hours per 100 iters):", (time.time() - start) * 100 / 3600)
    run_driver_options(model, args)
    return history


if __name__ == "__main__":
    main()
