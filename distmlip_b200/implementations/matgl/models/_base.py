"""Shared machinery of the engine-backed `*_Dist` model wrappers (CHGNet_Dist, TensorNet_Dist): the reference's
`from_existing` shallow copy (chgnet.py:551-560, tensornet.py:206-217), the process layout behind
`enable_distributed_mode(gpus)`, species lookup, weight finalisation and the `potential_forward_dist` seam."""
from __future__ import annotations

import numpy as np
import torch

import distmlip_b200
from distmlip_b200 import _lib


class EngineBackedModel:
    """Base of the `*_Dist` wrappers: everything that does not depend on the model family."""

    _has_site = False  # CHGNet's site-wise (magmom) readout

    # ------------------------------------------------------------------ construction
    @classmethod
    def from_existing(cls, model, dtype=distmlip_b200.float_th):
        """chgnet.py:551-560 / tensornet.py:206-217: takes the matgl model (any nn.Module with that attribute tree)."""
        if dtype not in (torch.float, torch.float32):
            raise ValueError("the sm_100a engine computes in fp32 only")
        model.to("cpu")
        dist_model = cls.__new__(cls)
        dist_model.__dict__ = model.__dict__.copy()
        dist_model._state_dict = {k: v.detach().clone().float() for k, v in model.state_dict().items()}
        dist_model.dist_enabled = False
        dist_model.dtype = dtype
        dist_model._engine = None
        return dist_model

    def _attr(self, name, default=None):
        # nn.Module keeps sub-modules/buffers out of __dict__'s top level; plain attributes are there.
        if name in self.__dict__:
            return self.__dict__[name]
        for store in ("_modules", "_parameters", "_buffers"):
            d = self.__dict__.get(store)
            if d is not None and name in d:
                return d[name]
        return default

    def __getattr__(self, name):
        v = self._attr(name, default=AttributeError)
        if v is AttributeError:
            raise AttributeError(name)
        return v

    def _process_layout(self, gpus):
        """(gpus, rank, world, group) for `enable_distributed_mode(gpus)`: a single-process group when one process is
        handed several GPUs (the reference's usage), one rank per GPU under torchrun, a replica for a single GPU."""
        if self.__dict__.get("dist_enabled"):
            raise Exception("Current model already has distributed mode enabled.")
        gpus = list(gpus)
        if any(g == "cpu" for g in gpus):
            raise RuntimeError('"cpu" partitions are not supported: libb200mlip has no CPU fallback')
        if len(gpus) < 1:
            raise ValueError("need at least one GPU")
        rank, world = 0, 1
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            rank, world = torch.distributed.get_rank(), torch.distributed.get_world_size()
        group = False
        if world != len(gpus):
            if len(gpus) == 1:
                rank, world = 0, 1  # replica mode: every process runs its own single-GPU engine
            elif world == 1:
                group = True        # the reference's usage: one process drives every GPU of the list
            else:
                raise RuntimeError(
                    f"enable_distributed_mode({gpus}) inside a {world}-process job: pass one GPU per process "
                    f"(len(gpus) == world) or a single GPU")
        return gpus, rank, world, group

    def _attach_engine(self, eng, gpus, rank, world, group):
        self.gpus = ["cuda:" + str(g) for g in gpus]
        eng.load_state_dict(self._state_dict)
        if group:
            rank, world = 0, 1  # one host process: results need no cross-process reduction
        elif world > 1:
            ids = [_lib.comm_unique_id() if rank == 0 else None]
            torch.distributed.broadcast_object_list(ids, src=0)
            eng.comm_init(ids[0], rank, world)
        self._engine = eng
        self._engine_finalized = False
        self._rank, self._world = rank, world
        self.element_to_index = {elem: idx for idx, elem in enumerate(self._attr("element_types"))}
        self.dist_enabled = True

    # ------------------------------------------------------------------ hot path
    def _species_of(self, atoms):
        """element index per atom (chgnet.py:66-72), vectorised through atomic numbers when the Atoms object has them"""
        if hasattr(atoms, "get_atomic_numbers"):
            z = np.asarray(atoms.numbers) if hasattr(atoms, "numbers") else np.asarray(atoms.get_atomic_numbers())
            cached = self.__dict__.get("_species_cache")
            if cached is not None and cached[0].shape == z.shape and np.array_equal(cached[0], z):
                return cached[1]  # MD / relaxation: the composition does not change between calls
            lut = self.__dict__.get("_z_lut")
            if lut is None:
                from distmlip_b200.structures import Z_OF

                lut = np.full(len(Z_OF) + 1, -1, dtype=np.int32)
                for el, idx in self.element_to_index.items():
                    if el in Z_OF:
                        lut[Z_OF[el]] = idx
                self._z_lut = lut
            sp = lut[z]
            if (sp < 0).any():
                raise KeyError("structure contains an element that is not in model.element_types")
            self._species_cache = (z.copy(), sp)
            return sp
        return np.array([self.element_to_index[s] for s in atoms.get_chemical_symbols()], dtype=np.int32)

    def _finalize(self, data_mean, data_std, element_refs):
        eng = self._engine
        key = (float(data_mean), float(data_std), None if element_refs is None else tuple(np.ravel(element_refs)))
        if self._engine_finalized and key == self._final_key:
            return
        eng.set_scaling(key[0], key[1])
        eng.set_element_refs(None if element_refs is None else np.ravel(element_refs))
        eng.finalize()
        self._engine_finalized, self._final_key = True, key

    def potential_forward_dist(self, dist_info, atoms, lattice_matrix, calc_stresses, calc_forces, calc_hessian,
                               state_attr=None):
        """Seam of chgnet.py:21-30,199-206 / tensornet.py:10-19.  Returns (node_types, positions, strain, (E, site_wise));
        forces / stress of the same evaluation are left on `dist_info` (no autograd graph exists), and so are the
        per-atom energies [N] (eV) and stresses [N,3,3] (GPa, W_i * 160.21766208 / V) when the Potential asks for them."""
        if calc_hessian:
            raise NotImplementedError("Calculating hessians is not implemented for distributed inference.")
        eng = self._engine
        if self.__dict__.get("_want_peratom", False):
            e, f, s, atom_e, atom_w = eng.compute_peratom(forces=calc_forces)
            s = s if calc_stresses else None
            dist_info.energies = atom_e
            dist_info.stresses = atom_w * (160.21766208 / abs(np.linalg.det(np.asarray(lattice_matrix, dtype=float))))
        else:
            e, f, s = eng.compute(forces=calc_forces, stress=calc_stresses)
        dist_info.forces, dist_info.stress = f, s
        node_types = torch.as_tensor(dist_info.species, dtype=distmlip_b200.int_th)
        positions = torch.from_numpy(dist_info.cart)  # zero-copy view (f64); no autograd graph hangs off it here
        strain = torch.zeros(1, 3, 3, dtype=distmlip_b200.float_th)
        # the site-wise readout is only gathered (one more all-reduce) when the Potential asks for it
        want_site = self._has_site and self.__dict__.get("_want_site", True)
        site = torch.as_tensor(eng.sitewise()).reshape(-1, 1) if want_site else None
        return node_types, positions, strain, (torch.tensor([e], dtype=torch.float64), site)

    def dist_forward(self, *args, **kwargs):
        raise NotImplementedError("dist_forward over DGL graphs does not exist here; use potential_forward_dist")

    def predict_structure_dist(self, structure, state_feats=None):
        raise NotImplementedError(
            "Distributed direct property prediction is not yet supported. Please raise an issue or use Potential_Dist")
