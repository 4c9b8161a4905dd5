"""Generates tests/golden/graph_golden.json and tests/golden/ref_edges_si_6x6x7_P2.npz from the reference's own
C graph builder (oracle/_ref, compiled by oracle/Makefile from a DistMLIP checkout).  With that checkout at hand:

    make -C oracle REF=<DistMLIP checkout> && python tests/golden/make_golden.py

Each case of graph_golden.json stores order-independent integer digests of what get_subgraphs_fast returned
(subgraph_creation_fast.c:403-422); the .npz stores one cell's edge set in full (see reference_edges).  With
them the numpy restatement (oracle/graph_ref.py) and the CUDA graph builder are checked against the reference
wherever the tests run, with or without a DistMLIP checkout.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from distmlip_b200.structures import SimpleAtoms, rough_cell, si_diamond  # noqa: E402
from oracle import graph_ref as G  # noqa: E402

MOD = (1 << 61) - 1


def digest(rows):
    """order-independent digest of integer tuples"""
    rows = np.asarray(rows, dtype=np.int64)
    if rows.size == 0:
        return [0, 0, 0]
    rows = rows.reshape(len(rows), -1)
    acc = np.zeros(len(rows), dtype=object)
    for c in range(rows.shape[1]):
        acc = (acc * 1000003 + (rows[:, c].astype(object) + 7919)) % MOD
    return [int(len(rows)), int(sum(acc) % MOD), int(sum((a * a) % MOD for a in acc) % MOD)]


def cases():
    out = {}
    out["si_8x8x8_P2"] = (si_diamond(8), 2)
    out["si_4x4x12_P3"] = (si_diamond(4, nz=12), 3)
    out["si_4x4x16_P4_seed3"] = (si_diamond(4, nz=16, seed=3), 4)
    a = si_diamond(4, nz=8, seed=5)
    # sheared (triclinic) cell, same fractional coordinates
    lat = a.get_cell()
    lat[2, 0] = 3.0
    lat[1, 0] = 1.5
    frac = a.get_scaled_positions()
    out["si_triclinic_4x4x8_P2"] = (SimpleAtoms(a.get_chemical_symbols(), frac @ lat, lat), 2)
    # unwrapped input: shift a third of the atoms by lattice vectors
    b = si_diamond(4, nz=8, seed=7)
    pos = b.get_positions()
    latb = b.get_cell()
    pos[::3] += latb[0] - 2 * latb[2]
    out["si_unwrapped_4x4x8_P2"] = (SimpleAtoms(b.get_chemical_symbols(), pos, latb), 2)
    out["rough_3000_P2"] = (rough_cell(3000, aspect=(1, 1, 3), seed=1), 2)
    return out


def describe(atoms, P):
    cart, lat, pbc = atoms.get_positions(), atoms.get_cell(), atoms.get_pbc().astype(np.int64)
    frac = atoms.get_scaled_positions(wrap=True)
    t = G.ref_get_subgraphs(cart, frac, lat, pbc, P, 5.0, 3.0, True)
    c = G.canon_from_ref_tuple(t, P)
    d = {"natoms": len(cart), "P": P,
         "edges": digest(np.column_stack([c["i1"], c["i2"], c["off"]])),
         "bond_edges": digest(np.column_stack([c["i1"][c["within"]], c["i2"][c["within"]], c["off"][c["within"]]])),
         "parts": []}
    for p in range(P):
        part = c["parts"][p]
        e = part["edges"]
        own_b = part["ude2edge"][: part["n_bond_owned"]]
        ld, ls = part["line_dst"], part["line_src"]
        de = part["ude2edge"][ld]
        pd = {
            "n_owned": part["n_owned"],
            "owned": digest(np.sort(np.concatenate([part["pure"]] + part["to"]))[:, None]),
            "to": [digest(np.asarray(x)[:, None]) for x in part["to"]],
            "from": [digest(np.asarray(x)[:, None]) for x in part["from"]],
            "edges": digest(np.column_stack(e)),
            "bonds_owned": digest(np.column_stack([c["i1"][own_b], c["i2"][own_b], c["off"][own_b]])),
            "n_bond_halo": part["n_bond_total"] - part["n_bond_owned"],
            "n_angles": int(len(ld)),
            "angle_dst_center": digest(np.column_stack([c["i1"][de], c["i2"][de], c["off"][de], part["center"]])),
        }
        d["parts"].append(pd)
    return d


REF_EDGES = "ref_edges_si_6x6x7_P2.npz"


def reference_edges(n_dist=4096):
    """What tests/test_oracle.py::test_graph_oracle_matches_live_reference compares with, for
    si_diamond(6, nz=7, seed=11) on 2 slabs: the whole edge set in canonical (i1, i2, off) order, the partition
    that owns each edge, the halo lists, the number of angles of each partition, and the distances of a fixed
    seeded sample of n_dist edges (all 56k of them would make the file five times larger)."""
    atoms = si_diamond(6, nz=7, seed=11)
    cart, lat, pbc = atoms.get_positions(), atoms.get_cell(), atoms.get_pbc().astype(np.int64)
    t = G.ref_get_subgraphs(cart, atoms.get_scaled_positions(wrap=True), lat, pbc, 2, 5.0, 3.0, True)
    c = G.canon_from_ref_tuple(t, 2)
    order = np.lexsort((c["off"][:, 2], c["off"][:, 1], c["off"][:, 0], c["i2"], c["i1"]))
    owner = np.full(len(order), -1, dtype=np.int8)
    for p in range(2):
        owner[t[16][p]] = p  # local -> global edge map of partition p
    assert (owner >= 0).all()
    i1, i2, off, owner = c["i1"][order], c["i2"][order], c["off"][order], owner[order]
    dist_idx = np.sort(np.random.default_rng(0).choice(len(order), size=n_dist, replace=False))
    out = {"i1": i1.astype(np.int32), "i2": i2.astype(np.int32), "off": off.astype(np.int8), "owner": owner,
           "dist_idx": dist_idx.astype(np.int32), "dist": c["dist"][order][dist_idx],
           "n_angles": np.array([len(c["parts"][p]["line_src"]) for p in range(2)], dtype=np.int64)}
    for p in range(2):
        for q in range(2):
            out[f"to_{p}_{q}"] = np.asarray(c["parts"][p]["to"][q], dtype=np.int32)
            out[f"from_{p}_{q}"] = np.asarray(c["parts"][p]["from"][q], dtype=np.int32)
        # the owner mask restates the partition's canonically sorted edge list exactly
        m = owner == p
        po = np.lexsort((off[m, 2], off[m, 1], off[m, 0], i1[m], i2[m]))
        s, d, _o = c["parts"][p]["edges"]
        assert np.array_equal(i1[m][po], s) and np.array_equal(i2[m][po], d)
    return out


if __name__ == "__main__":
    here = os.path.dirname(os.path.abspath(__file__))
    res = {k: describe(a, P) for k, (a, P) in cases().items()}
    with open(os.path.join(here, "graph_golden.json"), "w") as f:
        json.dump(res, f, indent=1)
    print({k: (v["natoms"], v["edges"][0]) for k, v in res.items()})
    np.savez_compressed(os.path.join(here, REF_EDGES), **reference_edges())
