"""CPU-only checks: the C-ABI library loads and exports every symbol include/*.h declares,
the host-side mirror behaves like the reference's host logic, and nothing silently falls
back to the CPU."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
torch.set_default_dtype(torch.float64)


def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "fermiflow_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(ff_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as g
    path = g.build()
    lib = ctypes.CDLL(path)
    names = _declared_symbols()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), "missing symbol " + n
    lib.ff_version.restype = ctypes.c_int
    assert lib.ff_version() >= 100


def test_ctypes_signatures_cover_header():
    from fermiflow_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared_symbols()


def test_no_cpu_fallback():
    from fermiflow_b200 import MLP, Backflow, CNF
    cnf = CNF(Backflow(MLP(1, 4)), (0.0, 1.0), nsteps=2)
    with pytest.raises(RuntimeError, match="CUDA"):
        cnf.generate(torch.randn(2, 3, 2))
    with pytest.raises(RuntimeError, match="CUDA"):
        Backflow(MLP(1, 4))(torch.randn(2, 3, 2))


def test_argument_errors_reported():
    """Error behaviour of the C ABI without touching a device."""
    from fermiflow_b200 import _lib as L
    lib = L.lib()
    assert lib.ff_cnf_generate(None, None, 0, 0, None, None) != 0
    assert b"model" in lib.ff_last_error()
    m = L.FFModel()
    m.n_up, m.n_dn, m.H_eta, m.nsteps = 2, 0, 0, 4
    assert lib.ff_cnf_generate(ctypes.byref(m), None, 0, 0, None, None) != 0
    assert b"hidden" in lib.ff_last_error()
    assert lib.ff_potential(None, 5, 3, 1.0, 1, None, None) != 0


def test_fermion_states_match_reference(golden):
    from fermiflow_b200 import HO2D
    ho, g = HO2D(), golden("states")
    for nup, dE in ((3, 2), (6, 2), (3, 4), (10, 2), (4, 3)):
        states, Es = ho.fermion_states(nup, 0, dE)
        idx = np.array([[o.index for o in up] for up, _ in states])
        assert np.array_equal(idx, g["states_%d_%d" % (nup, dE)])
        assert np.array_equal(np.array(Es), g["Es_%d_%d" % (nup, dE)])
    with pytest.raises(ValueError):
        ho.fermion_states(3, 1, 2)


def test_orbital_callables_match_reference(golden):
    from fermiflow_b200 import HO2D
    g = golden("slater")
    x = torch.from_numpy(g["x_orb"])
    vals = torch.stack([o(x) for o in HO2D().orbitals], -1)
    assert np.abs(vals.numpy() - g["orbitals"]).max() < 1e-13
    assert HO2D().Es == list(g["Es"])


def test_mlp_mirror_matches_reference_mlp(golden):
    """MLP.forward / grad (MLP.py:30-45) and parameter naming (state_dict compatibility)."""
    from fermiflow_b200 import MLP
    m = MLP(1, 7)
    assert sorted(m.state_dict()) == ["fc1.bias", "fc1.weight", "fc2.weight"]
    x = torch.randn(11, 1, requires_grad=True)
    y = m(x)
    gx, = torch.autograd.grad(y.sum(), x)
    assert torch.allclose(gx, m.grad(x))
    m.init_zeros()
    assert float(m(x).abs().max()) == 0.0
    with pytest.raises(ValueError):
        MLP(2, 3).kernel_params()


def test_vmc_potential_objects():
    """Any object with V(x) is a potential (reference VMC.py:27-28, 52-55); one without is refused at construction."""
    from fermiflow_b200 import MLP, Backflow, CNF, HO2D, FreeFermion, GSVMC

    class NoV:
        pass

    class Quartic:
        def V(self, x):
            return (x ** 4).sum(dim=(-2, -1))
    cnf = CNF(Backflow(MLP(1, 4)), (0.0, 1.0))
    with pytest.raises(TypeError):
        GSVMC(2, 0, HO2D(), FreeFermion("cpu"), cnf, NoV())
    with pytest.raises(TypeError):
        GSVMC(2, 0, HO2D(), FreeFermion("cpu"), cnf, Quartic(), sp_potential=NoV())
    model = GSVMC(2, 0, HO2D(), FreeFermion("cpu"), cnf, Quartic())
    assert model._Z == 0.0 and not model._harmonic


REFERENCE_CNF_KEYS = [   # list(CNF(Backflow(MLP(1, H), mu=MLP(1, H)), t_span).state_dict()) of reference src/flow.py:28,37
    "v_wrapper.v.eta.fc1.weight", "v_wrapper.v.eta.fc1.bias", "v_wrapper.v.eta.fc2.weight",
    "v_wrapper.v.mu.fc1.weight", "v_wrapper.v.mu.fc1.bias", "v_wrapper.v.mu.fc2.weight",
    "f.v.eta.fc1.weight", "f.v.eta.fc1.bias", "f.v.eta.fc2.weight",
    "f.v.mu.fc1.weight", "f.v.mu.fc1.bias", "f.v.mu.fc2.weight"]


def test_cnf_state_dict_has_the_reference_layout():
    """A checkpoint of the reference's CNF / GSVMC loads with strict=True and vice versa (flow.py:18-37)."""
    from fermiflow_b200 import MLP, Backflow, CNF, HO2D, FreeFermion, GSVMC, HO, CoulombPairPotential
    cnf = CNF(Backflow(MLP(1, 4), mu=MLP(1, 3)), (0.0, 1.0))
    assert list(cnf.state_dict()) == REFERENCE_CNF_KEYS
    assert len(list(cnf.parameters())) == 6                           # shared parameters are not duplicated
    ref_ckpt = {k: torch.randn_like(v) for k, v in cnf.state_dict().items()}
    for k in list(ref_ckpt):                                          # the reference stores the same tensor twice
        if k.startswith("f.v."):
            ref_ckpt[k] = ref_ckpt["v_wrapper.v." + k[4:]]
    cnf.load_state_dict(ref_ckpt, strict=True)
    assert torch.equal(cnf.v.eta.fc1.weight, ref_ckpt["v_wrapper.v.eta.fc1.weight"])
    assert cnf.v is cnf.v_wrapper.v and cnf.v is cnf.f.v
    model = GSVMC(2, 1, HO2D(), FreeFermion("cpu"), cnf, CoulombPairPotential(2.0), sp_potential=HO())
    assert list(model.state_dict()) == ["cnf." + k for k in REFERENCE_CNF_KEYS]
    # checkpoints written by round-1 builds (`v.eta...`) are remapped
    old = {"v." + k[len("v_wrapper.v."):]: torch.randn_like(v) for k, v in cnf.state_dict().items() if k.startswith("v_wrapper")}
    cnf.load_state_dict(old, strict=True)
    assert torch.equal(cnf.v.mu.fc2.weight, old["v.mu.fc2.weight"])


def test_reference_cnf_checkpoint_round_trip(tmp_path):
    """A checkpoint file as the reference writes it for CNF(Backflow(MLP(1, 5), mu=MLP(1, 4)), t_span) (keys of
    REFERENCE_CNF_KEYS, MLP fc1 with bias and fc2 without, every `f.v.` entry the same tensor as its `v_wrapper.v.`
    twin) loads here with strict=True, and the file saved back has the same keys, shapes, dtypes and sharing, which
    is what the reference's strict load of it checks."""
    from collections import OrderedDict
    from fermiflow_b200 import MLP, Backflow, CNF
    H = {"eta": 5, "mu": 4}
    shapes = {"fc1.weight": lambda h: (h, 1), "fc1.bias": lambda h: (h,), "fc2.weight": lambda h: (1, h)}
    gen = torch.Generator().manual_seed(3)
    ref = OrderedDict()
    for k in REFERENCE_CNF_KEYS:
        if k.startswith("f.v."):
            ref[k] = ref["v_wrapper.v." + k[len("f.v."):]]
        else:
            net, layer = k.split(".")[2], ".".join(k.split(".")[3:])
            ref[k] = torch.randn(shapes[layer](H[net]), generator=gen, dtype=torch.float64)
    a, b = tmp_path / "ref.pt", tmp_path / "ours.pt"
    torch.save(ref, a)
    cnf = CNF(Backflow(MLP(1, 5), mu=MLP(1, 4)), (0.0, 1.0))
    cnf.load_state_dict(torch.load(a), strict=True)
    for k, v in ref.items():
        assert torch.equal(cnf.state_dict()[k], v), k
    torch.save(cnf.state_dict(), b)
    ours = torch.load(b)
    assert list(ours) == REFERENCE_CNF_KEYS
    for k, v in ref.items():
        assert ours[k].shape == v.shape and ours[k].dtype == v.dtype and torch.equal(ours[k], v), k
        if k.startswith("f.v."):
            assert ours[k].data_ptr() == ours["v_wrapper.v." + k[len("f.v."):]].data_ptr(), k


def test_metropolis_seed_and_rank_offset(monkeypatch):
    """FreeFermion draws its default seed from torch's generator and offsets the Philox walker index by rank * B
    (every rank gets its own chains; ADVICE r1)."""
    from fermiflow_b200 import base_dist as BD
    calls = []

    class FakeLib:
        def ff_metropolis(self, B, n_up, n_dn, orb, ws, steps, tau, seed, offset, *rest):
            calls.append((B, seed, offset))
            return 0
    monkeypatch.setattr(BD.L, "lib", lambda: FakeLib())
    monkeypatch.setattr(BD.L, "ptr", lambda t, dtype=None: None)
    monkeypatch.setattr(BD.L, "stream", lambda: None)
    monkeypatch.setattr(BD, "orbital_indices", lambda orbs, dev: None)
    torch.manual_seed(123)
    fd = BD.FreeFermion("cpu")
    fd.sample((0, 1), (0,), (8,))
    fd.sample((0, 1), (0,), (8,))
    assert calls[0][1] == 123 and calls[1][1] != calls[0][1] and calls[0][2] == 0
    monkeypatch.setattr(BD, "_rank_world", lambda: (3, 4))
    fd.manual_seed(7)
    fd.sample((0, 1), (0,), (8,))
    assert calls[2] == (8, 7, 24)
    torch.manual_seed(124)
    assert BD.FreeFermion("cpu").seed is None


def test_orbital_index_vectors_are_cached_per_device():
    """orbital_indices builds its int32 vector once per (occupation, device): the hot path asks for the same vectors at
    every iteration and a fresh torch.tensor(list, device=cuda) is a blocking host-to-device copy."""
    from fermiflow_b200 import HO2D
    from fermiflow_b200.orbitals import orbital_indices
    ho = HO2D()
    a = orbital_indices(tuple(ho.orbitals[:3]) + tuple(ho.orbitals[:2]), "cpu")
    b = orbital_indices(tuple(ho.orbitals[:3]) + tuple(ho.orbitals[:2]), torch.device("cpu"))
    assert a is b and a.dtype == torch.int32 and a.tolist() == [0, 1, 2, 0, 1]
    c = orbital_indices(tuple(ho.orbitals[:3]), "cpu")
    assert c is not a and c.tolist() == [0, 1, 2]
    with pytest.raises(TypeError):
        orbital_indices((lambda x: x,), "cpu")
