"""Cell stress of the oracle (``oracle/m3gnet_oracle.py``) by the definition: sigma = (1/V) dE/d(eps) at eps = 0, with
positions and lattice rows deformed as r -> r (I + eps), and the same quantity in bond form, (1/V) sum_e v_e (x) dE/dv_e.
Shared by the CPU and GPU cell-stress tests."""
import contextlib

import torch

from oracle import m3gnet_oracle as O


def volumes(lattice):
    lat = lattice.reshape(-1, 3, 3)
    return torch.abs(torch.linalg.det(lat.double())).to(lat.dtype)


def strained(graph, eps):
    """Copy of an oracle graph with positions and lattices deformed by (I + eps[b]) (eps (B,3,3))."""
    g = dict(graph)
    lat = graph["lattice"].reshape(-1, 3, 3)
    eye = torch.eye(3, dtype=lat.dtype)
    defo = eye + eps
    g["pos"] = torch.einsum("na,nac->nc", graph["pos"], defo[graph["batch"]])
    g["lattice"] = torch.bmm(lat, defo)
    return g


def energy(p, hp, graph, factors=None):
    out = O.forward(p, hp, {k: (v.clone() if torch.is_tensor(v) else v) for k, v in graph.items()}, factors=factors,
                    create_graph=False, with_forces=False)
    return out["total_energy"]


def cell_stress(p, hp, graph, factors=None):
    """(B,3,3): (1/V) dE_b/d(eps_b) by autograd through the strained geometry."""
    B = graph["lattice"].reshape(-1, 3, 3).shape[0]
    eps = torch.zeros((B, 3, 3), dtype=graph["pos"].dtype, requires_grad=True)
    e = O.forward(p, hp, strained(graph, eps), factors=factors, create_graph=False, with_forces=False)["total_energy"]
    (g,) = torch.autograd.grad(e.sum(), eps)
    return g / volumes(graph["lattice"])[:, None, None]


@contextlib.contextmanager
def _capture_bond_vectors(store):
    orig = O.pair_geometry

    def wrapped(*args):
        vec, dist, cos = orig(*args)
        store["vec"] = vec
        return vec, dist, cos

    O.pair_geometry = wrapped
    try:
        yield
    finally:
        O.pair_geometry = orig


def bond_form(p, hp, graph, factors=None):
    """(B,3,3): (1/V) sum_{bonds e of b} v_e (x) dE/dv_e (v in the oracle's scaled lengths; the product does not
    depend on the length unit)."""
    store = {}
    pos = graph["pos"].clone().requires_grad_(True)  # any leaf: the bond vectors must be part of an autograd graph
    g = dict(graph)
    g["pos"] = pos
    with _capture_bond_vectors(store):
        e = O.forward(p, hp, g, factors=factors, create_graph=False, with_forces=False)["total_energy"]
    vec = store["vec"]
    (gv,) = torch.autograd.grad(e.sum(), vec)
    B = graph["lattice"].reshape(-1, 3, 3).shape[0]
    b_e = graph["batch"][graph["edge_index"][0]]
    w = torch.zeros((B, 3, 3), dtype=vec.dtype).index_add_(0, b_e, vec[:, :, None] * gv[:, None, :])
    return w / volumes(graph["lattice"])[:, None, None]


def reference_stresses(p, hp, graph, factors=None):
    """The oracle's ``stresses`` row (sum_i pos_i (x) F_i / V, Voigt xx yy zz yz zx xy), for comparison."""
    out = O.forward(p, hp, {k: (v.clone() if torch.is_tensor(v) else v) for k, v in graph.items()}, factors=factors,
                    create_graph=False)
    return out["stresses"].detach()
