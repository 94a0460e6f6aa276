"""fermiflow_b200 -- B200-native implementation of FermiFlow's per-walker VMC hot path.

Module names follow the reference's src/ tree so that `from fermiflow_b200.VMC import GSVMC`
replaces `from VMC import GSVMC`."""
from . import _lib  # noqa: F401
from .MLP import MLP  # noqa: F401
from .equivariant_funs import Backflow  # noqa: F401
from .flow import CNF  # noqa: F401
from .orbitals import HO2D  # noqa: F401
from .base_dist import FreeFermion  # noqa: F401
from .potentials import HO, CoulombPairPotential  # noqa: F401
from .slater import LogAbsSlaterDet, LogAbsSlaterDetMultStates  # noqa: F401
from .VMC import GSVMC, BetaVMC  # noqa: F401
from .observables import DensityEstimator, MomentumEstimator, RenyiEstimator  # noqa: F401
