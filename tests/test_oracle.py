"""CPU tests that pin the oracle (test infrastructure) before anything is checked against it:
  * oracle/graph_ref.py  == committed golden digests generated from the reference's own C code
  * oracle/graph_ref.py  == the full edge set the reference's own C code builds for one cell (stored golden vectors)
  * oracle/manual_ref.py (factorised forward + hand-derived backward) == autograd of chgnet_ref.py
"""
import json
import os

import numpy as np
import pytest
import torch

from tests._util import (digest, golden_cases, make_model, manual_run, oracle_graph, oracle_partition_digests)
from oracle import graph_ref as G
from oracle import manual_ref as M
from oracle.chgnet_ref import potential_ref
from distmlip_b200.structures import si_diamond

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "graph_golden.json")))


@pytest.mark.parametrize("name", sorted(GOLD))
def test_graph_oracle_matches_golden(name):
    atoms, P = golden_cases()[name]
    g = GOLD[name]
    o = G.GraphOracle(atoms.get_positions(), atoms.get_cell(), atoms.get_pbc().astype(np.int64), P, 5.0, 3.0, True,
                      frac_wrapped=atoms.get_scaled_positions(wrap=True))
    assert o.accepts and o.unique_to
    assert digest(np.column_stack([o.i1, o.i2, o.off])) == g["edges"]
    assert digest(np.column_stack([o.i1[o.bond], o.i2[o.bond], o.off[o.bond]])) == g["bond_edges"]
    for p in range(P):
        mine = oracle_partition_digests(o, p)
        assert mine == g["parts"][p], (name, p)


def test_graph_oracle_matches_live_reference():
    """against the full output of the reference's C graph builder for one cell, stored by make_golden.reference_edges"""
    ref = np.load(os.path.join(HERE, "golden", "ref_edges_si_6x6x7_P2.npz"))
    atoms = si_diamond(6, nz=7, seed=11)
    cart, lat, pbc = atoms.get_positions(), atoms.get_cell(), atoms.get_pbc().astype(np.int64)
    o = G.GraphOracle(cart, lat, pbc, 2, 5.0, 3.0, True)
    i1, i2, off = ref["i1"].astype(np.int64), ref["i2"].astype(np.int64), ref["off"].astype(np.int64)
    assert np.array_equal(o.i1, i1) and np.array_equal(o.i2, i2)
    assert np.array_equal(o.off, off)
    assert np.allclose(np.sqrt(o.d2[ref["dist_idx"]]), ref["dist"], atol=1e-12)
    for p in range(2):
        for q in range(2):
            assert np.array_equal(ref[f"to_{p}_{q}"], o.to_list(p, q))
            assert np.array_equal(ref[f"from_{p}_{q}"], o.from_list(p, q))
        m = ref["owner"] == p
        order = np.lexsort((off[m, 2], off[m, 1], off[m, 0], i1[m], i2[m]))
        s, d, of = o.edges_of(p)
        assert np.array_equal(s, i1[m][order]) and np.array_equal(d, i2[m][order])
        assert len(o.angles_of(p)) == ref["n_angles"][p]


def test_reference_rejects_thin_slabs_and_so_does_oracle():
    atoms = si_diamond(4)  # 21.7 A: slab of 10.9 A <= 2 (5 + 3)   (subgraph_creation_utils.c:1512-1529)
    o = G.GraphOracle(atoms.get_positions(), atoms.get_cell(), atoms.get_pbc().astype(np.int64), 2, 5.0, 3.0, True)
    assert not o.accepts


def test_reference_graph_invariants():
    """SURVEY.md 4: invariants probed on the compiled reference, restated on the oracle."""
    atoms = si_diamond(8)
    o = G.GraphOracle(atoms.get_positions(), atoms.get_cell(), atoms.get_pbc().astype(np.int64), 2, 5.0, 3.0, True)
    cart, lat = atoms.get_positions(), atoms.get_cell()
    v = cart[o.i2] + o.off @ lat - cart[o.i1]
    assert np.allclose(np.einsum("ij,ij->i", v, v), o.d2, atol=1e-10)
    fwd = set(zip(o.i1.tolist(), o.i2.tolist(), map(tuple, o.off.tolist())))
    assert all((j, i, (-a, -b, -c)) in fwd for i, j, (a, b, c) in list(fwd)[:2000])  # symmetric edge set
    assert abs(len(o.i1) / len(cart) - 27.99) < 0.1 and abs(o.bond.sum() / len(cart) - 4.0) < 0.05
    for p in range(2):
        assert np.array_equal(o.to_list(p, 1 - p), o.from_list(1 - p, p))


def test_manual_backward_equals_autograd():
    model = make_model().double()
    atoms = si_diamond(2)
    og = oracle_graph(atoms)
    E, F, S, _ = potential_ref(model, atoms, graph=(og["i1"], og["i2"], og["off"], og["bond"]), dtype=torch.float64)
    out = manual_run(model, atoms, og)
    Fm, Sm = M.forces_from_gvec(out["gvec"], og["vec"], og["i1"], og["i2"], len(atoms), atoms.get_volume())
    assert abs(E.item() - out["energy"].item()) < 1e-12
    assert (Fm - F).abs().max().item() < 1e-13 and (Sm - S).abs().max().item() < 1e-13


def test_oracle_physical_sanity():
    """translation invariance and zero net force of the restated model (fp64)."""
    model = make_model().double()
    atoms = si_diamond(2)
    E, F, _, _ = potential_ref(model, atoms, dtype=torch.float64)
    assert F.sum(0).abs().max().item() < 1e-12
    atoms.set_positions(atoms.get_positions() + np.array([0.37, -1.2, 2.9]))
    E2, F2, _, _ = potential_ref(model, atoms, dtype=torch.float64)
    assert abs(E.item() - E2.item()) < 1e-10 and (F - F2).abs().max().item() < 1e-10
