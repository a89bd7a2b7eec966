"""Names of every field of a graph / batch object — the data contract of the reference
(torch_m3gnet/data/MaterialGraphKey.py:1-37); the strings are kept verbatim so that user code written
against the reference keeps working: ``graph[MaterialGraphKey.FORCES]`` etc."""

_INPUT = {
    "POS": "pos", "ATOM_TYPES": "atom_types", "NUM_TRIPLET_I": "num_triplet_i",
    "EDGE_INDEX": "edge_index", "EDGE_CELL_SHIFT": "edge_cell_shift", "NUM_TRIPLET_IJ": "num_triplet_ij",
    "TRIPLET_EDGE_INDEX": "triplet_edge_index", "LATTICE": "lattice",
    "NUM_NODES": "num_nodes", "NUM_EDGES": "num_edges", "NUM_TRIPLETS": "num_triplets",
}
_DERIVED = {
    "SCALED_POS": "scaled_pos", "SCALED_LATTICE": "scaled_lattice", "EDGE_DISTANCES": "edge_distances",
    "EDGE_WEIGHTS": "edge_weights", "TRIPLET_ANGLES": "triplet_angles", "ELEMENTAL_ENERGIES": "elemental_energies",
    "NODE_FEATURES": "x", "EDGE_ATTR": "edge_attr",
}
_TARGET = {
    "SCALED_ATOMIC_ENERGIES": "scaled_atomic_energies", "SCALED_TOTAL_ENERGY": "scaled_total_energy",
    "TOTAL_ENERGY": "total_energy", "FORCES": "forces", "STRESSES": "stresses",
}
_BATCH = {"BATCH": "batch"}
# extensions with no reference counterpart
_EXTENSION = {
    # (B,3,3) eV/A^3: sigma = (1/V) dE/d(strain), ASE's stress convention; filled when Gradient.compute_stress is set.
    # Not the reference's STRESSES row (sum_i pos_i (x) F_i / V), which keeps its meaning.
    "CELL_STRESS": "cell_stress",
}

ALL_KEYS = {**_INPUT, **_DERIVED, **_TARGET, **_BATCH, **_EXTENSION}
globals().update(ALL_KEYS)
__all__ = list(ALL_KEYS)
