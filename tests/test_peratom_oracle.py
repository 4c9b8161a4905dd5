"""CPU: the per-atom reference (tests/peratom_ref.py: per-atom energies and virials of both oracles in the convention of
include/b200mlip.h b2m_compute_peratom) and the per-atom ASE properties of PESCalculator_Dist on a Potential_Dist double."""
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from distmlip_b200.structures import SimpleAtoms, rough_cell, si_diamond
from oracle import chgnet_ref, tensornet_ref
from tests._util import make_model
from tests.peratom_ref import potential_ref_peratom
from tests.test_oracle_tensornet import make_tn

HERE = os.path.dirname(os.path.abspath(__file__))
GPA_PER_EVA3 = 160.21766208
MEAN, STD = 0.7, 1.3


def mixed(atoms, other="O", every=3):
    sym = [other if i % every == 0 else s for i, s in enumerate(atoms.get_chemical_symbols())]
    return SimpleAtoms(sym, atoms.get_positions(), atoms.get_cell())


def refs_for(model):
    return np.linspace(-3.0, -1.0, len(model.element_types))


def run(kind, atoms, **kw):
    """(E, stress GPa, e_i, W_i) of one f64 oracle evaluation with data_mean, data_std and element_refs"""
    m = make_model().double() if kind == "chgnet" else make_tn(seed=3, scale=1.5)
    ref = potential_ref_peratom(m, atoms, data_mean=MEAN, data_std=STD, element_refs=refs_for(m), **kw)
    E, S, ei, W = ref[0], ref[2], ref[-2], ref[-1]
    return float(E), S.numpy(), ei.numpy(), W.numpy()


STRUCTURES = {
    "diamond": lambda: mixed(si_diamond(2, seed=1)),
    "rough": lambda: mixed(rough_cell(80, seed=2)),
}


@pytest.mark.parametrize("kind", ["chgnet", "tensornet"])
@pytest.mark.parametrize("structure", sorted(STRUCTURES))
def test_per_atom_sum_rules(kind, structure):
    atoms = STRUCTURES[structure]()
    E, S, ei, W = run(kind, atoms)
    assert ei.shape == (len(atoms),) and W.shape == (len(atoms), 3, 3)
    assert abs(ei.sum() - E) < 1e-12 * max(1.0, abs(E))
    Ssum = W.sum(0) * GPA_PER_EVA3 / atoms.get_volume()
    assert np.abs(Ssum - S).max() < 1e-10 * np.abs(S).max()
    assert np.abs(W).max() > 0  # a structure with a non-zero virial


@pytest.mark.parametrize("kind", ["chgnet", "tensornet"])
def test_per_atom_reference_leaves_the_oracle_alone(kind):
    """the oracle's own outputs come back unchanged, and the model is left with its class forward_graph"""
    atoms = STRUCTURES["diamond"]()
    make = (lambda: make_model().double()) if kind == "chgnet" else (lambda: make_tn(seed=3, scale=1.5))
    oracle = chgnet_ref if kind == "chgnet" else tensornet_ref
    plain = oracle.potential_ref(make(), atoms, dtype=torch.float64, data_mean=MEAN, data_std=STD)
    m = make()
    per = potential_ref_peratom(m, atoms, data_mean=MEAN, data_std=STD)
    assert len(per) == len(plain) + 2
    for a, b in zip(plain, per[: len(plain)]):
        assert torch.equal(a, b)
    assert "forward_graph" not in m.__dict__


@pytest.mark.parametrize("kind", ["chgnet", "tensornet"])
def test_perfect_diamond_is_uniform(kind):
    """every site of an unperturbed diamond lattice is equivalent under the space group: the split convention must give
    every atom the same energy and the same virial"""
    atoms = si_diamond(2, sigma=0)
    E, _S, ei, W = run(kind, atoms)
    assert np.abs(ei - ei.mean()).max() <= 1e-12 * abs(ei.mean())
    assert np.abs(W - W.mean(0)).max() <= 1e-12 * np.abs(W.mean(0)).max()
    assert np.abs(W.mean(0)).max() > 0


# ------------------------------------------------------------------ ASE surface
try:
    import ase  # noqa: F401
except ImportError:
    sys.path.insert(0, os.path.join(HERE, "stubs"))

import distmlip_b200.implementations.matgl.ase as mase  # noqa: E402
from distmlip_b200.implementations.matgl.pes import Potential_Dist  # noqa: E402


class PerAtomPotential(Potential_Dist):
    """Potential_Dist double with per-atom output: fixed per-atom energies and stresses (GPa) left on last_dist_info,
    totals their sums, the way the engine-backed Potential_Dist hands them over"""

    def __init__(self, n, seed=0):
        rng = np.random.default_rng(seed)
        self.calc_forces = self.calc_stresses = self.calc_per_atom = True
        self.calc_hessian = self.calc_site_wise = False
        self.e_i = rng.normal(-4.0, 0.3, n)
        self.s_i = rng.normal(0.0, 0.5, (n, 3, 3))
        self.last_dist_info = None

    def forward(self, atoms, state_attr=None, tol=1e-8):
        self.last_dist_info = SimpleNamespace(energies=self.e_i.copy(), stresses=self.s_i.copy())
        return (torch.tensor([self.e_i.sum()], dtype=torch.float64), torch.zeros(len(atoms), 3),
                torch.as_tensor(self.s_i.sum(0)), None)


@pytest.mark.parametrize("use_voigt", [False, True])
@pytest.mark.parametrize("stress_unit,weight", [("GPa", 1.0), ("eV/A3", 1.0), ("GPa", 0.5)])
def test_calculator_per_atom_results(use_voigt, stress_unit, weight):
    from ase import Atoms

    n = 10
    pot = PerAtomPotential(n)
    calc = mase.PESCalculator_Dist(potential=pot, stress_unit=stress_unit, stress_weight=weight, use_voigt=use_voigt)
    assert "energies" in calc.implemented_properties and "stresses" in calc.implemented_properties
    atoms = Atoms(["Si"] * n, np.random.default_rng(1).random((n, 3)) * 5.0, np.eye(3) * 6.0)
    calc.calculate(atoms, ["energy", "stress", "energies", "stresses"])
    r = calc.results
    assert r["energies"].shape == (n,)
    assert r["stresses"].shape == ((n, 6) if use_voigt else (n, 3, 3))
    assert abs(r["energies"].sum() - r["energy"]) < 1e-12 * abs(r["energy"])
    assert np.allclose(r["stresses"].sum(0), r["stress"], rtol=1e-6, atol=1e-9)
    factor = weight * (1.0 if stress_unit == "GPa" else 1.0 / GPA_PER_EVA3)
    ref = pot.s_i * factor
    if use_voigt:
        ref = np.stack([ref[:, 0, 0], ref[:, 1, 1], ref[:, 2, 2], (ref[:, 1, 2] + ref[:, 2, 1]) / 2,
                        (ref[:, 0, 2] + ref[:, 2, 0]) / 2, (ref[:, 0, 1] + ref[:, 1, 0]) / 2], axis=1)
    assert np.allclose(r["stresses"], ref, rtol=1e-12, atol=0)


def test_calculator_without_per_atom_output_has_no_per_atom_results():
    from ase import Atoms

    pot = PerAtomPotential(4)
    pot.calc_per_atom = False
    calc = mase.PESCalculator_Dist(potential=pot)
    assert "energies" not in calc.implemented_properties and "stresses" not in calc.implemented_properties
    calc.calculate(Atoms(["Si"] * 4, np.zeros((4, 3)), np.eye(3) * 6.0), ["energy"])
    assert "energies" not in calc.results and "stresses" not in calc.results
