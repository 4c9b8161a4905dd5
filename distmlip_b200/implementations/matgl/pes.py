"""Potential_Dist -- drop-in for DistMLIP.implementations.matgl.pes.Potential_Dist (pes.py:13-146).

Same constructor kwargs and call convention: `potential(atoms, state_attr=None, tol=1e-8)` returns
`(energies, forces, stresses(GPa, 3x3), hessian=None[, site_wise])` as torch tensors.  Differences, all
deliberate: one partition is allowed (the reference asserts > 1 GPU, pes.py:40-42); energy, forces and
stress come out of one b2m_compute call (hand-written backward) instead of torch.autograd.backward
(pes.py:122-124); results are CPU tensors (the ASE calculator immediately calls .cpu().numpy()).

`calc_per_atom=True` (not in the reference) also computes per-atom energies and stresses in the same evaluation and leaves
them on `last_dist_info` as `energies` [N] (eV) and `stresses` [N,3,3] (GPa); they sum to the energy and the stress.
The return tuple does not change.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from distmlip_b200.distributed.dist import Distributed


class Potential_Dist:
    """A class representing an interatomic potential."""

    __version__ = 2

    def __init__(self, model=None, num_threads=None, data_mean=0.0, data_std=1.0, element_refs=None,
                 calc_forces=True, calc_stresses=True, calc_hessian=False, calc_site_wise=False, debug_mode=False,
                 calc_repuls=False, zbl_trainable=False, calc_per_atom=False, **kwargs):
        if model is None:
            raise ValueError("model is required")
        self.model = model
        assert getattr(self.model, "dist_enabled", False), "Distributed mode must be enabled"
        assert hasattr(self.model, "gpus"), "Model should have gpus attribute"
        if calc_repuls:
            raise NotImplementedError("ZBL repulsion is not part of the CHGNet / TensorNet paths")
        self.calc_forces = calc_forces
        self.calc_stresses = calc_stresses
        self.calc_hessian = calc_hessian
        self.calc_site_wise = calc_site_wise
        self.calc_per_atom = calc_per_atom
        self.debug_mode = debug_mode
        self.data_mean = float(torch.as_tensor(data_mean).item()) if data_mean is not None else 0.0
        self.data_std = float(torch.as_tensor(data_std).item()) if data_std is not None else 1.0
        if element_refs is not None and hasattr(element_refs, "property_offset"):
            element_refs = np.asarray(element_refs.property_offset, dtype=np.float64)  # matgl AtomRef
        self.element_refs = None if element_refs is None else np.asarray(element_refs, dtype=np.float64)
        if self.calc_hessian:
            print("Warning: turning off calc_hessian as it is not implemented within distributed inference.")
            self.calc_hessian = False
        self.num_threads = num_threads
        self.last_dist_info = None

    def __call__(self, *args, **kwargs):
        return self.forward(*args, **kwargs)

    def forward(self, atoms, state_attr=None, tol=1.0e-8):
        """pes.py:50-146."""
        # kept for signature compatibility; the graph build has no host threads
        _ = self.num_threads if self.num_threads else int(os.environ.get("DISTMLIP_NUM_THREADS", 8))
        lattice_matrix = np.array(atoms.get_cell())
        # `atoms.positions` is ASE's internal array (no copy); it is copied once into the engine's pinned staging buffer
        cart_coords = np.asarray(getattr(atoms, "positions", None) if hasattr(atoms, "positions")
                                 else atoms.get_positions(wrap=False))
        pbc = atoms.get_pbc().astype(np.int64)
        model = self.model
        species = model._species_of(atoms)
        model._want_site = bool(self.calc_site_wise)
        model._want_peratom = bool(self.calc_per_atom)
        model._finalize(self.data_mean, self.data_std, self.element_refs)
        dist_info = Distributed.create_distributed(
            cart_coords=cart_coords, frac_coords=None, lattice_matrix=lattice_matrix,
            num_partitions=model._engine.world, pbc=pbc,
            use_bond_graph=model.use_bond_graph if hasattr(model, "use_bond_graph") else False,  # pes.py:79-80
            cutoff=float(model.cutoff),
            three_body_cutoff=float(model.three_body_cutoff) if hasattr(model, "three_body_cutoff") else 0,
            tol=tol, num_threads=1, engine=model._engine, species=species)
        self.last_dist_info = dist_info
        model_out = model.potential_forward_dist(dist_info, atoms, lattice_matrix, self.calc_stresses,
                                                 self.calc_forces, self.calc_hessian, state_attr)
        if self.debug_mode:
            print("Debug mode true, returning early")
            return model_out[-1]
        _node_types, _positions, _strain, (total_energies, site_wise) = model_out
        forces = torch.as_tensor(dist_info.forces) if self.calc_forces else None
        stresses = torch.as_tensor(dist_info.stress) if self.calc_stresses else None
        hessian = None
        if self.calc_site_wise:
            return total_energies, forces, stresses, hessian, site_wise
        return total_energies, forces, stresses, hessian
