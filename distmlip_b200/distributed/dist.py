"""Distributed -- host-side view of the GPU-resident partitioned graph.

Mirror of DistMLIP/distributed/dist.py (class Distributed).  In the reference this object holds the
19 host arrays produced by the C extension for *all* partitions and moves halo rows between GPUs
with cross-device slice assignment (dist.py:323-388).  Here every partition's graph is built and kept on
its GPU by libb200mlip (b2m_set_structure) and the halo exchange happens inside b2m_compute.  The accessors
below expose the same counters with the same optional `partition` argument (dist.py:462-551): in a
single-process group (the reference's setting) any partition can be asked for; under one-process-per-GPU
each rank sees its own.  For tests, the partition content is available in canonical form.
"""
from __future__ import annotations

import numpy as np


class Distributed:
    "Distributed Graph for parallelized MLIP inference (one rank's partition)"

    def __init__(self, engine, species, total_num_nodes, use_bond_graph, num_partitions):
        self.engine = engine
        self.species = species
        self.total_num_nodes = total_num_nodes
        self.use_bond_graph = use_bond_graph
        self.num_partitions = num_partitions
        c = engine.counts()
        self.counts = c
        self.rank = c["rank"]
        self._group = bool(getattr(engine, "group", False))
        self.total_num_edges = None  # global count needs a reduction over ranks; see num_atom_edges
        self.forces = None
        self.stress = None
        self.energies = None  # per-atom energies [N] (eV) and stresses [N,3,3] (GPa) of a calc_per_atom evaluation
        self.stresses = None

    @staticmethod
    def cartesian_to_wrapped_fractional(positions_cartesian, lattice, pbc):
        """dist.py:128-156."""
        if not pbc[0] and not pbc[1] and not pbc[2]:
            return positions_cartesian
        frac = np.linalg.solve(lattice.T, np.transpose(positions_cartesian)).T
        for i, periodic in enumerate(pbc):
            if periodic:
                frac[:, i] %= 1.0
                frac[:, i] %= 1.0
        return frac

    @classmethod
    def create_distributed(cls, cart_coords, frac_coords, lattice_matrix, num_partitions, pbc, cutoff,
                           three_body_cutoff=0, tol=1e-8, use_bond_graph=False, num_threads=1, *, engine=None,
                           species=None):
        """dist.py:158-275.  `engine` (a distmlip_b200._lib.Engine) and `species` are the two extra
        keyword-only arguments: the graph is built on that engine's GPU.  frac_coords / num_threads are
        accepted for signature compatibility (wrapping is recomputed on the device; no host threads)."""
        if engine is None:
            raise RuntimeError("create_distributed needs engine=: the graph lives on the GPU, there is no CPU builder")
        if num_partitions != engine.world:
            raise ValueError(f"num_partitions={num_partitions} but the engine's communicator has {engine.world} ranks")
        cart_coords = np.ascontiguousarray(cart_coords, dtype=float)
        lattice_matrix = np.ascontiguousarray(lattice_matrix, dtype=float)
        if species is None:
            species = np.zeros(len(cart_coords), dtype=np.int32)
        engine.set_structure(cart_coords, lattice_matrix, species, np.asarray(pbc).astype(np.int32), tol)
        obj = cls(engine, np.asarray(species), len(cart_coords), use_bond_graph, num_partitions)
        obj.cart = cart_coords
        return obj

    # ---- counters (dist.py:462-551) ----
    def _c(self, partition):
        """counts of `partition` (None: this rank's partition / partition 0 of a group)"""
        if partition is None or (not self._group and partition == self.rank):
            return self.counts
        if not self._group:
            raise ValueError(f"partition {partition} lives in another process (this rank owns partition {self.rank})")
        if not 0 <= partition < self.num_partitions:
            raise ValueError(f"partition {partition} out of range [0, {self.num_partitions})")
        return self.engine.counts(partition)

    def num_atoms(self, partition=None):
        c = self._c(partition)
        return c["n_own"] + c["n_halo"]

    def num_atom_edges(self, partition=None):
        return self._c(partition)["n_edges"]

    def num_bonds(self, partition=None):
        assert self.use_bond_graph, "num_bonds only works when bond graph is enabled"
        c = self._c(partition)
        return c["n_bond_own"] + c["n_bond_halo"]

    def num_bond_edges(self, partition=None):
        assert self.use_bond_graph, "num_bond_edges only works when bond graph is enabled"
        return self._c(partition)["n_angles"]

    def num_atom_border_nodes(self, partition=None):
        return self._c(partition)["n_halo"]

    def num_bond_border_nodes(self, partition=None):
        assert self.use_bond_graph, "num_bond_border_nodes only works when bond graph is enabled"
        return self._c(partition)["n_bond_halo"]

    def partition_content(self, partition, which):
        """canonical content (b2m_get_partition_info `which`) of any partition of a single-process group"""
        if not self._group:
            if partition != self.rank:
                raise ValueError("only this rank's partition is visible in one-process-per-GPU mode")
            return self.engine.partition_info(which)
        self.engine.set_view(partition)
        try:
            return self.engine.partition_info(which)
        finally:
            self.engine.set_view(0)

    # ---- canonical partition content (tests) ----
    def owned_gids(self):
        return self.engine.partition_info(0)

    def halo_gids(self):
        return self.engine.partition_info(1), self.engine.partition_info(2)

    def edges(self):
        return self.engine.partition_info(3)

    def bonds(self):
        return self.engine.partition_info(4)

    def angles(self):
        return self.engine.partition_info(5)

    def to_lists(self):
        return self.engine.partition_info(6)

    def walls(self):
        return self.engine.partition_info(7)

    def __repr__(self):
        c = self.counts
        val = f"""Distributed:
    Total num atoms: {self.total_num_nodes}
    Bond graph exists: {self.use_bond_graph}\n"""
        parts = range(self.num_partitions) if self._group else [self.rank]
        for p in parts:  # dist.py:704-721 prints every partition; under one process per GPU only this rank's is here
            c = self._c(p)
            val += f"Partition {p} (of {self.num_partitions}):\n"
            val += f"\t# of atom graph nodes: {c['n_own'] + c['n_halo']} ({c['n_halo']} border nodes)\n"
            val += f"\t# of atom graph edges: {c['n_edges']}\n"
            if self.use_bond_graph:
                val += f"\t# of bond graph nodes: {c['n_bond_own'] + c['n_bond_halo']}. ({c['n_bond_halo']} border nodes)\n"
                val += f"\t# of bond graph edges: {c['n_angles']}\n"
        return val
