"""Finite-temperature VMC of the 2D quantum dot -- mirror of reference src/BetaFermionHO2D.py.

    python -m fermiflow_b200.BetaFermionHO2D --beta 10.0 --nup 3 --Z 2.0 --deltaE 2.0 --boltzmann --iternum 1000
"""
import argparse
import time

import torch

from .MLP import MLP
from .VMC import BetaVMC
from .base_dist import FreeFermion
from .equivariant_funs import Backflow
from .flow import CNF
from .observables import sample_density, sample_momentum, sample_natural_orbitals, sample_renyi
from .orbitals import HO2D
from .potentials import HO, CoulombPairPotential


def main(argv=None):
    p = argparse.ArgumentParser(description="Finite-temperature variational Monte Carlo simulation")
    p.add_argument("--beta", type=float, default=2.0)
    p.add_argument("--nup", type=int, default=6)
    p.add_argument("--ndown", type=int, default=0)
    p.add_argument("--Z", type=float, default=0.5)
    p.add_argument("--deltaE", type=float, default=2.0)
    p.add_argument("--cuda", type=int, default=0)
    p.add_argument("--Deta", type=int, default=50)
    p.add_argument("--nomu", action="store_true")
    p.add_argument("--Dmu", type=int, default=50)
    p.add_argument("--t0", type=float, default=0.0)
    p.add_argument("--t1", type=float, default=1.0)
    p.add_argument("--nsteps", type=int, default=16)
    p.add_argument("--boltzmann", action="store_true")
    p.add_argument("--iternum", type=int, default=1000)
    p.add_argument("--batch", type=int, default=8000)
    p.add_argument("--lr", type=float, default=1e-2)
    p.add_argument("--density", metavar="FILE", help="after training, save the density and pair correlations of "
                   "freshly sampled walkers to FILE (.npz, fermiflow_b200.observables.DensityEstimator)")
    p.add_argument("--density-batches", type=int, default=16, help="batches of --batch walkers for --density")
    p.add_argument("--density-extent", type=float, default=6.0, help="half-width of the density grids")
    p.add_argument("--momentum", metavar="FILE", help="after training, save the momentum distribution and one-body "
                   "coherence of freshly sampled walkers to FILE (.npz, fermiflow_b200.observables.MomentumEstimator)")
    p.add_argument("--momentum-batches", type=int, default=16, help="batches of --batch walkers for --momentum")
    p.add_argument("--momentum-kmax", type=float, default=4.0, help="half-width of the momentum grid")
    p.add_argument("--renyi", metavar="FILE", help="after training, save the second Renyi entropy of spatial regions, "
                   "from replica swaps of freshly sampled walkers, to FILE (.npz, fermiflow_b200.observables.RenyiEstimator)")
    p.add_argument("--renyi-batches", type=int, default=16, help="batches of --batch walkers for --renyi")
    p.add_argument("--renyi-a", type=lambda s: [float(v) for v in s.split(",")], default=[0.5, 1.0, 1.5, 2.0, 2.5, 3.0],
                   help="comma-separated region parameters for --renyi: disk radii or half-plane edges x < a")
    p.add_argument("--renyi-kind", choices=("disk", "halfplane"), default="disk", help="region kind for --renyi")
    p.add_argument("--natural-orbitals", metavar="FILE", help="after training, save the one-body density matrix in the "
                   "HO2D basis and its natural-orbital occupations, from one-particle moves of freshly sampled walkers, to "
                   "FILE (.npz, fermiflow_b200.observables.DensityMatrixEstimator)")
    p.add_argument("--natural-orbitals-batches", type=int, default=16,
                   help="batches of --batch walkers for --natural-orbitals")
    p.add_argument("--natural-orbitals-shells", type=int, default=7,
                   help="oscillator shells 0 ... S of the basis for --natural-orbitals ((S + 1)(S + 2) / 2 orbitals)")
    args = p.parse_args(argv)

    device = torch.device("cuda:%d" % args.cuda)
    eta = MLP(1, args.Deta); eta.init_zeros()
    mu = None
    if not args.nomu:
        mu = MLP(1, args.Dmu); mu.init_zeros()
    cnf = CNF(Backflow(eta, mu=mu), (args.t0, args.t1), nsteps=args.nsteps)
    model = BetaVMC(args.beta, args.nup, args.ndown, args.deltaE, args.boltzmann, HO2D(), FreeFermion(device=device),
                    cnf, CoulombPairPotential(args.Z), sp_potential=HO()).to(device)
    print("beta = %.1f, nup = %d, ndown = %d, Z = %.1f" % (args.beta, args.nup, args.ndown, args.Z))
    print("deltaE = %.1f, total number of states = %d" % (args.deltaE, model.Nstates))
    optimizer = torch.optim.Adam(model.parameters(), lr=args.lr)
    history = []
    for i in range(1, args.iternum + 1):
        start = time.time()
        gradF_phi, gradF_theta = model(args.batch)
        optimizer.zero_grad()
        gradF_phi.backward()
        gradF_theta.backward()
        model.allreduce_gradients()
        optimizer.step()
        history.append((model.F, model.F_std, model.E, model.E_std, model.S))
        print("iter: %03d" % i, "F:", model.F, "F_std:", model.F_std, "E:", model.E, "E_std:", model.E_std,
              "S:", model.S, "S_analytical:", model.S_analytical,
              "Instant speed (hours per 100 iters):", (time.time() - start) * 100 / 3600)
    if args.density:
        sample_density(model, args.nup, args.ndown, args.batch, args.density_batches, args.density_extent, args.density)
    if args.momentum:
        sample_momentum(model, args.nup, args.ndown, args.batch, args.momentum_batches, args.momentum_kmax, args.momentum)
    if args.renyi:
        sample_renyi(model, args.nup, args.ndown, args.batch, args.renyi_batches, args.renyi_a, args.renyi_kind, args.renyi)
    if args.natural_orbitals:
        sample_natural_orbitals(model, args.nup, args.ndown, args.batch, args.natural_orbitals_batches,
                                args.natural_orbitals_shells, args.natural_orbitals)
    return history


if __name__ == "__main__":
    main()
