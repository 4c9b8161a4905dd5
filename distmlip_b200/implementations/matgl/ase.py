"""ASE adapters -- thin mirrors of DistMLIP/implementations/matgl/ase.py (PESCalculator_Dist :53-127,
Relaxer :130-223, MolecularDynamics :228-491, TrajectoryObserver from matgl.ext.ase).

ASE / pymatgen are imported lazily: PESCalculator_Dist works on any Atoms-like object (tests use
distmlip_b200.structures.SimpleAtoms); Relaxer and MolecularDynamics need an `ase` package and keep the reference's
keyword arguments, optimizers and eight ensembles (tests run them against tests/stubs/ase, a minimal stand-in, because
ASE is not installed in the build image).
"""
from __future__ import annotations

import numpy as np

from distmlip_b200.implementations.matgl.pes import Potential_Dist

try:  # pragma: no cover - ASE is absent in the build image
    from ase.calculators.calculator import Calculator as _Calculator, all_changes as _all_changes
    _HAVE_ASE = True
except Exception:  # noqa: BLE001
    _HAVE_ASE = False
    _all_changes = ["positions", "numbers", "cell", "pbc", "initial_charges", "initial_magmoms"]

    class _Calculator:  # minimal stand-in with the attributes PESCalculator_Dist touches
        def __init__(self, **kwargs):
            self.results = {}
            self.atoms = None

        def calculate(self, atoms=None, properties=None, system_changes=None):
            self.atoms = atoms


def _voigt6(s):
    """[..., 3, 3] -> [..., 6] (xx, yy, zz, yz, xz, xy)"""
    s = np.asarray(s)
    return np.stack([s[..., 0, 0], s[..., 1, 1], s[..., 2, 2], (s[..., 1, 2] + s[..., 2, 1]) / 2,
                     (s[..., 0, 2] + s[..., 2, 0]) / 2, (s[..., 0, 1] + s[..., 1, 0]) / 2], axis=-1)


class PESCalculator_Dist(_Calculator):
    """Machine Learning Interatomic Potential calculator for ASE."""

    implemented_properties = ("energy", "free_energy", "forces", "stress", "hessian", "magmoms")

    def __init__(self, potential=None, state_attr=None, stress_unit="GPa", stress_weight=1.0, use_voigt=False,
                 **kwargs):
        super().__init__(**kwargs)
        assert isinstance(potential, Potential_Dist), "PESCalculatorDist requires using a Potential_Dist."
        self.potential = potential
        self.compute_stress = potential.calc_stresses
        self.compute_hessian = potential.calc_hessian
        self.compute_magmom = potential.calc_site_wise
        self.compute_per_atom = getattr(potential, "calc_per_atom", False)
        if self.compute_per_atom:  # ASE's per-atom properties, offered when the potential computes them
            self.implemented_properties = type(self).implemented_properties + ("energies", "stresses")
        if stress_unit == "eV/A3":
            conversion_factor = 0.006241509125883258  # GPa -> eV/A^3 (ase.units)
        elif stress_unit == "GPa":
            conversion_factor = 1.0
        else:
            raise ValueError(f"Unsupported stress_unit: {stress_unit}. Must be 'GPa' or 'eV/A3'.")
        self.stress_weight = stress_weight * conversion_factor
        self.state_attr = state_attr
        self.use_voigt = use_voigt
        self.last_count = None

    def calculate(self, atoms, properties=None, system_changes=None):
        """ase.py:80-127."""
        properties = properties or ["energy"]
        system_changes = system_changes or _all_changes
        _Calculator.calculate(self, atoms=atoms, properties=properties, system_changes=system_changes)
        calc_result = self.potential(atoms, self.state_attr)
        self.results.update(
            energy=calc_result[0].detach().cpu().numpy().item(),
            free_energy=calc_result[0].detach().cpu().numpy(),
            forces=calc_result[1].detach().cpu().numpy(),
        )
        if self.compute_stress:
            st = calc_result[2].detach().cpu().numpy()
            self.results.update(stress=(_voigt6(st) if self.use_voigt else st) * self.stress_weight)
        if self.compute_magmom:
            self.results.update(magmoms=calc_result[4].detach().cpu().numpy())
        if self.compute_per_atom:  # ASE's per-atom properties: they sum to `energy` and `stress`
            info = self.potential.last_dist_info
            sts = np.asarray(info.stresses)
            self.results.update(energies=np.asarray(info.energies),
                                stresses=(_voigt6(sts) if self.use_voigt else sts) * self.stress_weight)


class TrajectoryObserver:
    """matgl.ext.ase.TrajectoryObserver look-alike (collections of energies/forces/stresses per step)."""

    def __init__(self, atoms):
        self.atoms = atoms
        self.energies, self.forces, self.stresses = [], [], []
        self.atom_positions, self.cells = [], []

    def __call__(self):
        self.energies.append(float(self.atoms.get_potential_energy()))
        self.forces.append(self.atoms.get_forces())
        self.stresses.append(self.atoms.get_stress())
        self.atom_positions.append(self.atoms.get_positions())
        self.cells.append(self.atoms.get_cell()[:])

    def save(self, filename):
        import pickle

        with open(filename, "wb") as f:
            pickle.dump({"energy": self.energies, "forces": self.forces, "stresses": self.stresses,
                         "atom_positions": self.atom_positions, "cell": self.cells,
                         "atomic_number": self.atoms.get_atomic_numbers()}, f)


_OPTIMIZERS = {"fire": "FIRE", "bfgs": "BFGS", "lbfgs": "LBFGS", "lbfgslinesearch": "LBFGSLineSearch", "mdmin": "MDMin",
               "bfgslinesearch": "BFGSLineSearch"}  # ase.py:40-50 (the two scipy wrappers are looked up by name)


def _require_ase(what):
    try:
        import ase  # noqa: F401
    except Exception as ex:  # noqa: BLE001
        raise ImportError(f"{what} needs ASE (not installed in this image)") from ex


class Relaxer:
    """ase.py:130-223: Relaxer(potential, state_attr, optimizer="FIRE", relax_cell=True, stress_weight=1/160.21766208)."""

    def __init__(self, potential=None, state_attr=None, optimizer="FIRE", relax_cell=True,
                 stress_weight=1 / 160.21766208):
        _require_ase("Relaxer")
        import ase.optimize as opt

        if isinstance(optimizer, str):
            name = _OPTIMIZERS.get(optimizer.lower(), optimizer)
            if not hasattr(opt, name):
                raise KeyError(optimizer)
            optimizer = getattr(opt, name)
        self.optimizer = optimizer
        # ase.py:153-157: the reference passes ONLY stress_weight (GPa -> eV/A^3); stress_unit stays "GPa" (factor 1)
        self.calculator = PESCalculator_Dist(potential=potential, state_attr=state_attr, stress_weight=stress_weight)
        self.relax_cell = relax_cell

    def relax(self, atoms, fmax=0.1, steps=500, traj_file=None, interval=1, verbose=False,
              ase_cellfilter="Frechet", params_asecellfilter=None, **kwargs):
        import contextlib
        import io
        import sys

        try:
            from ase.filters import ExpCellFilter, FrechetCellFilter
        except ImportError:  # older ASE keeps ExpCellFilter under constraints (as the reference imports it)
            from ase.constraints import ExpCellFilter
            from ase.filters import FrechetCellFilter

        adaptor = None
        try:  # pymatgen Structure / Molecule in, Structure out (ase.py:196-197, 220-223) when pymatgen is installed
            from pymatgen.core import Molecule, Structure
            from pymatgen.io.ase import AseAtomsAdaptor

            adaptor = AseAtomsAdaptor()
            if isinstance(atoms, (Structure, Molecule)):
                atoms = adaptor.get_atoms(atoms)
        except ImportError:
            pass
        atoms.set_calculator(self.calculator)
        stream = sys.stdout if verbose else io.StringIO()
        params_asecellfilter = params_asecellfilter or {}
        with contextlib.redirect_stdout(stream):
            obs = TrajectoryObserver(atoms)
            if self.relax_cell:
                atoms = (FrechetCellFilter(atoms, **params_asecellfilter) if ase_cellfilter == "Frechet"
                         else ExpCellFilter(atoms, **params_asecellfilter))
            optimizer = self.optimizer(atoms, **kwargs)
            optimizer.attach(obs, interval=interval)
            optimizer.run(fmax=fmax, steps=steps)
            obs()
        if traj_file is not None:
            obs.save(traj_file)
        if self.relax_cell:
            atoms = atoms.atoms
        return {"final_structure": adaptor.get_structure(atoms) if adaptor is not None else atoms, "trajectory": obs}


class MolecularDynamics:
    """ase.py:228-491: same keyword arguments and the same eight ensembles, delegating to ase.md."""

    def __init__(self, atoms, potential, state_attr=None, stress_weight=1.0, ensemble="nvt", temperature=300,
                 timestep=1.0, pressure=1.01325 * 1e-4, taut=None, taup=None, friction=1.0e-3, andersen_prob=1.0e-2,
                 ttime=25.0, pfactor=75.0**2.0, external_stress=None, compressibility_au=None, trajectory=None,
                 logfile=None, loginterval=1, append_trajectory=False, mask=None):
        _require_ase("MolecularDynamics")
        from ase import units
        from ase.md import Langevin
        from ase.md.andersen import Andersen
        from ase.md.nvtberendsen import NVTBerendsen
        from ase.md.verlet import VelocityVerlet

        try:
            from pymatgen.core import Molecule, Structure
            from pymatgen.io.ase import AseAtomsAdaptor

            if isinstance(atoms, (Structure, Molecule)):
                atoms = AseAtomsAdaptor().get_atoms(atoms)
        except ImportError:
            pass
        self.atoms = atoms
        if isinstance(potential, Potential_Dist):  # ase.py:291-302
            self.atoms.set_calculator(PESCalculator_Dist(potential=potential, state_attr=state_attr,
                                                         stress_unit="eV/A3", stress_weight=stress_weight))
        elif isinstance(potential, _Calculator):
            self.atoms.calc = potential
        else:
            raise Exception(f"Input of type {potential} not supported for potential input.")
        taut = taut if taut is not None else 100 * timestep * units.fs
        taup = taup if taup is not None else 1000 * timestep * units.fs
        mask = mask if mask is not None else np.array([(1, 0, 0), (0, 1, 0), (0, 0, 1)])
        external_stress = external_stress if external_stress is not None else 0.0
        common = dict(trajectory=trajectory, logfile=logfile, loginterval=loginterval,
                      append_trajectory=append_trajectory)
        ens = ensemble.lower()
        if ens == "nvt":
            self.dyn = NVTBerendsen(self.atoms, timestep * units.fs, temperature_K=temperature, taut=taut, **common)
        elif ens == "nve":
            self.dyn = VelocityVerlet(self.atoms, timestep * units.fs, **common)
        elif ens == "nvt_langevin":
            self.dyn = Langevin(self.atoms, timestep * units.fs, temperature_K=temperature, friction=friction, **common)
        elif ens == "nvt_andersen":
            self.dyn = Andersen(self.atoms, timestep * units.fs, temperature_K=temperature,
                                andersen_prob=andersen_prob, **common)
        elif ens == "nvt_bussi":
            from ase.md.bussi import Bussi
            from ase.md.velocitydistribution import MaxwellBoltzmannDistribution

            if np.isclose(self.atoms.get_kinetic_energy(), 0.0, rtol=0, atol=1e-12):
                MaxwellBoltzmannDistribution(self.atoms, temperature_K=temperature)
            self.dyn = Bussi(self.atoms, timestep * units.fs, temperature_K=temperature, taut=taut, **common)
        elif ens == "npt":  # Inhomogeneous_NPTBerendsen: three lattice parameters change independently, angles fixed
            from ase.md.nptberendsen import Inhomogeneous_NPTBerendsen

            self.dyn = Inhomogeneous_NPTBerendsen(self.atoms, timestep * units.fs, temperature_K=temperature,
                                                  pressure_au=pressure, taut=taut, taup=taup,
                                                  compressibility_au=compressibility_au, **common)
        elif ens == "npt_berendsen":
            from ase.md.nptberendsen import NPTBerendsen

            self.dyn = NPTBerendsen(self.atoms, timestep * units.fs, temperature_K=temperature, pressure_au=pressure,
                                    taut=taut, taup=taup, compressibility_au=compressibility_au, **common)
        elif ens == "npt_nose_hoover":
            from ase.md.npt import NPT

            self.upper_triangular_cell()
            self.dyn = NPT(self.atoms, timestep * units.fs, temperature_K=temperature, externalstress=external_stress,
                           ttime=ttime * units.fs, pfactor=pfactor * units.fs, mask=mask, **common)
        else:
            raise ValueError("Ensemble not supported")
        self.trajectory, self.logfile, self.loginterval, self.timestep = trajectory, logfile, loginterval, timestep

    def run(self, steps):
        """ase.py:443-449."""
        self.dyn.run(steps)

    def set_atoms(self, atoms):
        """ase.py:451-461."""
        calculator = self.atoms.calc
        self.atoms = atoms
        self.dyn.atoms = atoms
        self.dyn.atoms.set_calculator(calculator)

    def upper_triangular_cell(self, verbose=False):
        """ase.py:463-491: ASE's Nose-Hoover NPT wants an upper-triangular cell (ASE's canonical cells are lower
        triangular); if the cell is not, rebuild it from its lengths and angles with c along z, b in the yz plane."""
        cell = np.array(self.atoms.get_cell(), dtype=float)
        if np.allclose(cell, np.triu(cell)):
            return
        la, lb, lc = np.linalg.norm(cell, axis=1)
        ang = lambda u, v: np.arccos(np.clip(np.dot(u, v) / (np.linalg.norm(u) * np.linalg.norm(v)), -1.0, 1.0))
        al, be, ga = ang(cell[1], cell[2]), ang(cell[0], cell[2]), ang(cell[0], cell[1])
        # azimuth of a around z once b sits in the yz plane
        cos_phi = np.clip((np.cos(ga) - np.cos(al) * np.cos(be)) / (np.sin(al) * np.sin(be)), -1.0, 1.0)
        sin_phi = np.sqrt(1.0 - cos_phi**2)
        upper = np.array([[la * np.sin(be) * sin_phi, la * np.sin(be) * cos_phi, la * np.cos(be)],
                          [0.0, lb * np.sin(al), lb * np.cos(al)],
                          [0.0, 0.0, lc]])
        self.atoms.set_cell(upper, scale_atoms=True)
        if verbose:
            print("Transformed to upper triangular unit cell.", flush=True)
