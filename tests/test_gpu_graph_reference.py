"""GPU: the integer graph (bond list, triplet list, plan) bit for bit against numpy at the shapes and edges where the
kernels branch: the cell list's 512-candidate overflow, pairs a few ulps either side of both cut-off tests, large image
reach, empty structures, member counts across the 32 / 64 / 96 / 128 tiers, hand-built triplet lists that are not
canonical, and the scan / CSR primitives across their tile sizes.  Every comparison is ``torch.equal`` on whole
tensors (values, shapes, dtypes, order).  The numpy side is oracle/m3gnet_oracle.py plus tests/graph_reference.py."""
import functools

import numpy as np
import pytest
import torch

from oracle import m3gnet_oracle as O
from tests import graph_reference as R
from tests.util import golden, graph_dict, report, state_dict_of, to_batch

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------
# structures (host only)
# ---------------------------------------------------------------------------------------------------------------------

def _fcc(lat, reps=1, jitter=0.0, seed=0):
    base = np.array([[0, 0, 0], [0, 0.5, 0.5], [0.5, 0, 0.5], [0.5, 0.5, 0]], dtype=np.float64)
    cells = np.stack(np.meshgrid(*[np.arange(reps)] * 3, indexing="ij"), axis=-1).reshape(-1, 3)
    frac = ((cells[:, None, :] + base[None]) / reps).reshape(-1, 3)
    cart = frac @ lat + np.random.default_rng(seed).uniform(-jitter, jitter, size=(len(frac), 3))
    return lat, cart, np.full(len(frac), 29)


def _sphere(k, radius):
    """k points on a sphere (Fibonacci spiral)."""
    i = np.arange(k) + 0.5
    phi = np.arccos(1 - 2 * i / k)
    th = np.pi * (1 + 5 ** 0.5) * i
    return radius * np.stack([np.cos(th) * np.sin(phi), np.sin(th) * np.sin(phi), np.cos(phi)], axis=1)


def _star(k, box=14.0):
    """One centre atom with k member bonds (satellites at 2 A, r3 = 2.5): the centre has the largest member count."""
    centre = np.full(3, box / 2)
    cart = np.concatenate([centre[None], centre + _sphere(k, 2.0)]) if k else centre[None]
    return np.eye(3) * box, cart, np.full(len(cart), 8)


def _accept_threshold(r):
    """Smallest float64 x > 0 along a lattice axis whose bond is rejected: x * x >= r * r + 1e-8 (float64)."""
    x = np.sqrt(r * r + 1e-8)
    while x * x >= r * r + 1e-8:
        x = np.nextafter(x, 0.0)
    while x * x < r * r + 1e-8:
        x = np.nextafter(x, np.inf)
    return x


def _ulps(x, k):
    for _ in range(abs(k)):
        x = np.nextafter(x, np.inf if k > 0 else 0.0)
    return x


def _axis_pair(x, box=12.0):
    """Atoms at the origin and at (x, 0, 0), plus one at (0, 2, 0) so that the origin can head triplets.  All
    coordinates and the lattice are small integers or x itself: every float64 step of the accept test is exact but the
    last, so the outcome is that of x * x against the threshold."""
    cart = np.array([[0.0, 0.0, 0.0], [x, 0.0, 0.0], [0.0, 2.0, 0.0]])
    return np.eye(3) * box, cart, np.array([8, 8, 8])


def _disagreeing_pair(r, box=12.0):
    """Two atoms bonded across the periodic boundary whose two directions round differently: (cart[j] + s a) - cart[i]
    differs in the last bit from -((cart[i] - s a) - cart[j]), and the pair sits on the accept test, so i -> j is a
    bond and j -> i is not (or the reverse).  A third and a fourth atom next to them give each a second member bond."""
    thr = r * r + 1e-8
    for u in np.linspace(0.1, 0.9, 4001):
        xj = box - (np.sqrt(thr) - u)
        for k in range(-40, 41):
            pj = _ulps(xj, k)
            v_ij = (pj - box) - u  # i = 0 at (u, 0, 0), j = 1 at (pj, 0, 0), image -1 seen from i
            v_ji = (u + box) - pj  # image +1 seen from j
            if (v_ij * v_ij < thr) != (v_ji * v_ji < thr):
                cart = np.array([[u, 0.0, 0.0], [pj, 0.0, 0.0], [u, 2.0, 0.0], [pj, 0.0, 2.0]])
                return np.eye(3) * box, cart, np.array([8, 8, 8, 8])
    raise AssertionError("no pair found whose two directions disagree")


def _overflow_box(n=600, box=6.2, seed=5):
    """Uniform random atoms at 2.5 per A^3: with r = 2 the cell list has 3 bins per axis and each atom's 27 bins hold
    all n > 512 atoms, so nbr_kernel falls back to the sweep over the structure."""
    cart = np.random.default_rng(seed).uniform(0, box, size=(n, 3))
    return np.eye(3) * box, cart, np.full(n, 1)


def _boundary_box(L=15.3):
    """3 cell-list bins per axis at r = 5; atoms on fractional 0, 1/3, 2/3 and 1 (bin boundaries and cell faces)."""
    g = np.stack(np.meshgrid(*[np.array([0.0, 1 / 3, 2 / 3])] * 3, indexing="ij"), axis=-1).reshape(-1, 3)
    frac = np.concatenate([g, g + np.array([1.0, 0.5, 0.5]), g + np.array([0.5, 1.0, 1 / 6])])
    lat = np.eye(3) * L
    return lat, frac @ lat, np.full(len(frac), 14)


def _sheared(lat_shear):
    lat, cart, z = _fcc(np.eye(3) * 7.23, reps=2, jitter=0.1, seed=4)
    frac = cart @ np.linalg.inv(lat)
    lat_s = lat @ lat_shear
    return lat_s, frac @ lat_s, z


def _far_outside():
    """Every atom displaced by a different lattice vector of up to +-10 cells."""
    lat, cart, z = _fcc(np.array([[4.24, 0, 0], [0.7, 4.1, 0], [-0.3, 0.5, 4.4]]), reps=1, jitter=0.05, seed=7)
    s = np.random.default_rng(8).integers(-10, 11, size=(len(cart), 3))
    s[0] = [10, -10, 10]
    s[1] = [-10, 10, -10]
    return lat, cart + s @ lat, z


STRUCTURES = {
    # name: (list of structures, cutoff, three-body cutoff)
    "orthorhombic": ([_fcc(np.diag([7.23, 8.0, 6.8]), reps=2, jitter=0.1, seed=1)], 5.0, 4.0),
    "sheared": ([_sheared(np.eye(3) + np.array([[0, 0.6, 0.3], [0, 0, 0.5], [0.4, 0, 0]]))], 5.0, 4.0),
    "far_outside": ([_far_outside()], 5.0, 4.0),
    "bin_boundaries": ([_boundary_box(), _fcc(np.eye(3) * 4.24)], 5.0, 4.0),
    "overflow_mixed": ([_overflow_box(), _fcc(np.eye(3) * 18.075, reps=5, jitter=0.3, seed=11),
                        _fcc(np.eye(3) * 4.24)], 2.0, 2.0),
    "self_images": ([(np.eye(3), np.array([[0, 0, 0], [0.5, 0.5, 0.5], [0.5, 0, 0], [0, 0.5, 0.5]]),
                      np.array([3, 3, 1, 1]))], 5.0, 1.5),
    "isolated": ([(np.eye(3) * 20.0, np.array([[3.0, 4.0, 5.0]]), np.array([6]))], 5.0, 4.0),
    "no_bonds_batch": ([(np.eye(3) * 20.0, np.array([[3.0, 4.0, 5.0]]), np.array([6])),
                        (np.eye(3) * 11.0, np.array([[0.0, 0.0, 0.0]]), np.array([8]))], 5.0, 4.0),
    "no_triplets": ([_fcc(np.eye(3) * 7.23, reps=2, jitter=0.05, seed=2)], 5.0, 1.0),
    "tiers_low": ([_star(k) for k in (0, 1, 2, 31, 32, 33, 64, 65)], 5.0, 2.5),
    "tier_96": ([_star(96)], 5.0, 2.5),
    "tier_97": ([_star(97), _star(3)], 5.0, 2.5),
    "tier_128": ([_star(128)], 5.0, 2.5),
    "tier_129": ([_star(129), _star(2)], 5.0, 2.5),
}


def _accept_edge_structures(r=5.0):
    thr = _accept_threshold(r)
    return [_axis_pair(_ulps(thr, k)) for k in range(-3, 4)]


def _member_edge_structures(r3=4.1):
    f = float(np.float32(r3))
    up = float(np.nextafter(np.float32(r3), np.float32(np.inf)))
    mid = 0.5 * (f + up)  # exact in float64; float32 rounds it to even
    xs = [_ulps(f, k) for k in (-2, -1, 0, 1, 2)] + [_ulps(mid, k) for k in (-1, 0, 1)] + [up]
    return [_axis_pair(x) for x in xs]


STRUCTURES["accept_edge"] = (_accept_edge_structures(), 5.0, 4.1)
STRUCTURES["member_edge"] = (_member_edge_structures(), 5.0, 4.1)
STRUCTURES["disagreeing_directions"] = ([_disagreeing_pair(5.0)], 5.0, 5.0)


# ---------------------------------------------------------------------------------------------------------------------
# references (numpy) and GPU runs
# ---------------------------------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def _reference(name):
    structs, r, r3 = STRUCTURES[name]
    src, dst, img, dist, n_off = [], [], [], [], 0
    for lat, cart, _ in structs:
        s, d, im, di = O.neighbor_list_bruteforce(lat, cart, r)
        src.append(s + n_off)
        dst.append(d + n_off)
        img.append(im)
        dist.append(di)
        n_off += len(cart)
    ei = np.stack([np.concatenate(src), np.concatenate(dst)]).astype(np.int64)
    d32 = np.concatenate(dist).astype(np.float32)
    out = R.triplets_src_grouped(n_off, ei, d32, r3)
    out.update(edge_index=ei, edge_cell_shift=np.concatenate(img).astype(np.int32).reshape(-1, 3), dist=d32, N=n_off)
    return out


def _arrays(structs):
    lat = np.stack([s[0] for s in structs])
    cart = np.concatenate([s[1] for s in structs])
    z = np.concatenate([np.asarray(s[2]) for s in structs])
    return lat, cart, z, [len(s[1]) for s in structs]


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a))


def _equal(name, got, want):
    got = got.cpu()
    want = _t(want) if isinstance(want, np.ndarray) else want
    assert got.dtype == want.dtype, f"{name}: dtype {got.dtype} vs {want.dtype}"
    assert got.shape == want.shape, f"{name}: shape {tuple(got.shape)} vs {tuple(want.shape)}"
    if not torch.equal(got, want):
        bad = (got != want).reshape(-1).nonzero().flatten()
        raise AssertionError(f"{name}: {bad.numel()} entries differ, first at flat index {bad[:5].tolist()}: "
                             f"{got.reshape(-1)[bad[:5]].tolist()} vs {want.reshape(-1)[bad[:5]].tolist()}")


def _no_cell_list(monkeypatch):
    from torch_m3gnet_b200.data.material_graph import Batch

    monkeypatch.setattr(Batch, "_cell_list", staticmethod(lambda *a: (None, None, None, None)))


def _gpu_bonds(structs, r, r3, device):
    """The builder's bond pass (count -> scan -> fill) with its member flags, which the Batch does not keep."""
    from torch_m3gnet_b200.data.material_graph import Batch

    lat, cart, _, sizes = _arrays(structs)
    lat64 = torch.as_tensor(lat).to(device)
    cart64 = torch.as_tensor(cart).to(device)
    atom_ptr = torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)).to(device)
    edge_ptr, E, ei, shift, dist, member = Batch._sweep(lat, lat64, cart64, atom_ptr, len(sizes), int(sum(sizes)), r,
                                                        r3, device)
    return {"edge_ptr": edge_ptr, "edge_index": ei, "edge_cell_shift": shift, "dist": dist, "member": member}


def _check_bonds(got, ref):
    _equal("edge_index", got["edge_index"], ref["edge_index"])
    _equal("edge_cell_shift", got["edge_cell_shift"], ref["edge_cell_shift"])
    _equal("edge distances (float32)", got["dist"], ref["dist"])
    _equal("member flags", got["member"], ref["member"])
    ptr = np.concatenate([[0], np.cumsum(np.bincount(ref["edge_index"][0], minlength=ref["N"]))]).astype(np.int32)
    _equal("edge_ptr", got["edge_ptr"], ptr)


def _check_plan_csr(plan, src, dst, N):
    """in_ptr / in_perm: the stable counting sort of dst."""
    ptr, perm = R.csr_by_key(dst, N)
    _equal("in_ptr", plan.in_ptr, ptr)
    _equal("in_perm", plan.in_perm[:plan.E], perm)
    _equal("src", plan.src, src.astype(np.int32))
    _equal("dst", plan.dst, dst.astype(np.int32))


def _check_graph(b, ref):
    from torch_m3gnet_b200 import _lib

    _equal("edge_index", b["edge_index"], ref["edge_index"])
    _equal("edge_cell_shift", b["edge_cell_shift"], ref["edge_cell_shift"])
    _equal("edge_distances_build", b._private["edge_distances_build"], ref["dist"])
    _equal("triplet_edge_index", b["triplet_edge_index"], ref["triplet_edge_index"])
    _equal("num_triplet_i", b["num_triplet_i"], ref["num_triplet_i"])
    _equal("num_triplet_ij", b["num_triplet_ij"], ref["num_triplet_ij"])
    assert b["num_triplets"] == ref["triplet_edge_index"].shape[1]
    plan = b._plan
    _equal("tri_ptr", plan.tri_ptr, ref["tri_ptr"])
    _equal("tri_e2", plan.tri_e2[:plan.T], ref["tri_e2"])
    _equal("member_edges", plan.member_edges, ref["member_edges"])
    assert plan.max_members == ref["max_members"]
    assert plan.tri_dense == (ref["max_members"] <= _lib.tb_atom_capacity())
    assert plan.tri_moment == (ref["max_members"] <= _lib.tb_mom_capacity())
    _check_plan_csr(plan, ref["edge_index"][0], ref["edge_index"][1], ref["N"])


# ---------------------------------------------------------------------------------------------------------------------
# 1-3. bond list, cut-off edges, triplets and the builder's plan
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("cell_list", [True, False], ids=["cell_list", "sweep"])
@pytest.mark.parametrize("name", sorted(STRUCTURES))
def test_builder_equals_reference(device, monkeypatch, name, cell_list):
    """Bonds (edge_index, images, float32 distances, member flags) against ``neighbor_list_bruteforce``; triplets,
    per-atom / per-bond counts and the seeded plan against the src-grouped restatement.  ``sweep`` runs the same
    structures with the cell list switched off."""
    from torch_m3gnet_b200.data.material_graph import Batch

    structs, r, r3 = STRUCTURES[name]
    ref = _reference(name)
    if not cell_list:
        _no_cell_list(monkeypatch)
    _check_bonds(_gpu_bonds(structs, r, r3, device), ref)
    lat, cart, z, sizes = _arrays(structs)
    b = Batch.from_arrays(lat, cart, z, sizes, r, r3, device=device)
    _check_graph(b, ref)


def test_cases_reach_their_edges(device):
    """The structures above exercise what they are named for (host-side facts about the reference)."""
    from torch_m3gnet_b200 import _lib

    acc = _reference("accept_edge")
    n_bonds = [int((acc["edge_index"][0] == 3 * k).sum()) for k in range(7)]
    assert n_bonds == [2, 2, 2, 1, 1, 1, 1], n_bonds  # the pair bond is accepted up to the threshold, not beyond
    mem = _reference("member_edge")
    pair = mem["member"][(mem["edge_index"][0] % 3 == 0) & (mem["edge_index"][1] % 3 == 1)]
    assert 0 < pair.sum() < pair.size, pair
    si = _reference("self_images")
    assert np.bincount(si["edge_index"][0]).min() > 400  # hundreds of self-image bonds per atom
    assert np.abs(si["edge_cell_shift"]).max() == 5
    far = _reference("far_outside")
    assert np.abs(far["edge_cell_shift"]).max() >= 20
    n3 = _reference("tiers_low")["n3"]
    for k in (0, 1, 2, 31, 32, 33, 64, 65):
        assert k in n3, k
    cap = _lib.tb_atom_capacity()
    assert _reference("tier_96")["max_members"] == cap < _reference("tier_97")["max_members"]
    assert _reference("tier_128")["max_members"] == _lib.tb_mom_capacity() < _reference("tier_129")["max_members"]


def test_candidate_overflow_happens(device):
    """The 27-bin neighbourhood of every atom of the dense box holds more than CAND_MAX = 512 atoms (so nbr_kernel
    sweeps the whole structure), while the 500-atom box of the same batch stays on the bin candidates."""
    from torch_m3gnet_b200.data.material_graph import Batch

    structs, r, _ = STRUCTURES["overflow_mixed"]
    lat, cart, _, sizes = _arrays(structs)
    N = int(sum(sizes))
    atom_ptr = torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)).to(device)
    bins, bin_base, bin_ptr, _ = Batch._cell_list(lat, len(sizes), N, r, torch.as_tensor(lat).to(device),
                                                  torch.as_tensor(cart).to(device), atom_ptr, device)
    nb = bins.cpu().numpy().reshape(-1, 3)
    base = bin_base.cpu().numpy()
    count = np.diff(bin_ptr.cpu().numpy())
    assert nb[0].tolist() == [3, 3, 3] and nb[1].tolist() == [9, 9, 9] and nb[2].tolist() == [0, 0, 0]
    assert count[base[0]:base[1]].sum() == sizes[0] == 600 and count[base[1]:base[2]].sum() == sizes[1]

    def cand27(s):
        c = count[base[s]:base[s + 1]].reshape(*nb[s])
        return sum(np.roll(c, (dx, dy, dz), axis=(0, 1, 2))
                   for dx in (-1, 0, 1) for dy in (-1, 0, 1) for dz in (-1, 0, 1))

    assert cand27(0).min() > 512
    assert cand27(1).max() <= 512


def test_directions_that_disagree_follow_the_src_grouped_rule(device):
    """Bond i -> j accepted, j -> i rejected (the two directions of one pair round differently at the accept test).
    The builder counts member bonds per source atom; the oracle's dst-degree walk (quirk Q6) is unpinned there and
    differs, which this asserts so that the case stays the one it is meant to be."""
    ref = _reference("disagreeing_directions")
    ei = ref["edge_index"]
    pairs = set(map(tuple, ei.T.tolist()))
    assert (1, 0) in pairs and (0, 1) not in pairs
    tri, nti, _ = O.enumerate_triplets(ref["N"], ei, ref["dist"], 5.0)
    assert not np.array_equal(nti, ref["num_triplet_i"])
    assert ref["num_triplet_i"].tolist() == [0, 2, 0, 0]


# ---------------------------------------------------------------------------------------------------------------------
# 4. plans of hand-built triplet lists (GraphPlan.build) and the model on them
# ---------------------------------------------------------------------------------------------------------------------

def _triangle():
    """Three atoms, two member bonds each: six triplets, so one repeated triplet is a large share of the three-body
    term and its gradient."""
    cart = np.array([[2.0, 2.0, 2.0], [4.0, 2.1, 2.0], [2.9, 4.1, 2.3]])
    g = O.build_graph(np.eye(3) * 11.0, cart, [8, 14, 8], 5.0, 4.0)
    g = O.collate([g])
    return g


@functools.lru_cache(maxsize=None)
def _plan_graphs():
    return {"c1": graph_dict(golden("c1_default")), "triangle": _triangle()}


# Bessel normalisation table scale: O(1) on the 32-atom cell as in test_gpu_engine.py; 0.03 on the triangle, where the
# three-body term then carries the forces (one repeated triplet moves them by 25x the force tolerance)
FACTOR_SCALE = {"c1": 1.0, "triangle": 0.03}

VARIANTS = ["canonical", "permuted", "non_symmetric", "duplicated", "row_misses_member", "member_removed",
            "single_member_row", "thinned"]


def _variant_batch(graph, variant, device):
    gd = {k: v.clone() for k, v in _plan_graphs()[graph].items()}
    ei = gd["edge_index"].numpy()
    tri, dense, sym = R.triplet_list_variants(ei[0], gd["triplet_edge_index"].numpy())[variant]
    gd["triplet_edge_index"] = _t(tri.astype(np.int64))
    return gd, to_batch(gd, device), dense, sym


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("graph", ["c1", "triangle"])
def test_plan_of_hand_built_triplet_list(device, graph, variant):
    """GraphPlan.build: the triplet CSR (rows by first bond, ascending), its transpose with multiplicities, the
    symmetry flag, the dense-layout certificate, max_members, member bonds and the dst CSR."""
    from torch_m3gnet_b200 import _lib
    from torch_m3gnet_b200.data.material_graph import GraphPlan

    gd, b, dense, sym = _variant_batch(graph, variant, device)
    ei = gd["edge_index"].numpy()
    e1, e2 = gd["triplet_edge_index"].numpy()
    E, N = ei.shape[1], gd["pos"].shape[0]
    plan = GraphPlan.build(b)
    ptr, cols = R.csr_rows(E, e1, e2)
    _equal("tri_ptr", plan.tri_ptr, ptr)
    _equal("tri_e2", plan.tri_e2[:plan.T], cols)
    want_sym = R.is_symmetric(E, e1, e2)
    want_dense, want_max = R.dense_certificate(ei[0], N, e1, e2)
    if dense is not None:
        assert (want_dense, want_sym) == (dense, sym)
    assert plan.tri_symmetric == want_sym
    tptr, tcols = R.csr_transpose(E, e1, e2)
    _equal("trt_ptr", plan.trt_ptr, tptr)
    _equal("trt_e1", plan.trt_e1[:plan.T], tcols)
    assert plan.max_members == want_max
    assert plan.tri_dense == (want_dense and want_max <= _lib.tb_atom_capacity())
    assert plan.tri_moment == (want_dense and want_max <= _lib.tb_mom_capacity())
    used = (ptr[1:] > ptr[:-1]) | (tptr[1:] > tptr[:-1])
    _equal("member_edges", plan.member_edges, np.nonzero(used)[0].astype(np.int32))
    _check_plan_csr(plan, ei[0], ei[1], N)


def _model(device, sd, fac):
    from torch_m3gnet_b200 import build_model

    model = build_model(5.0, 4.0, 3, 3, 95, 64, 3, device=device)
    model.load_state_dict(sd)
    for i in (6, 8, 10):
        model.model[i].nsb.factors = fac.to(device)  # O(1) table: the three-body adjoint is visible in the forces
    return model


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("graph", ["c1", "triangle"])
def test_model_on_hand_built_triplet_list(device, graph, variant):
    """Energies and forces on the path the plan selects, with the whole-step executor enabled and disabled, against
    the oracle fed the same triplet list (tolerances of test_gpu_engine.py).  With a repeated triplet the forward sums
    it twice, so the adjoint must too: a plan that certified that list as symmetric would reuse its rows as their own
    transpose and count the repeat once."""
    from torch_m3gnet_b200 import engine

    sd = {k: (v * 3 if k.endswith("weight") else v) for k, v in state_dict_of(golden("c1_default")).items()}
    fac = (torch.rand(3, 3, generator=torch.Generator().manual_seed(2)) + 0.5) * FACTOR_SCALE[graph]
    model = _model(device, sd, fac)
    gd, _, _, _ = _variant_batch(graph, variant, device)
    ref = O.forward(sd, O.HyperParams(), {k: v.clone() for k, v in gd.items()}, factors=fac, create_graph=False)
    n = gd["pos"].shape[0]
    old = engine.ENABLED
    try:
        for flag in (True, False):
            engine.ENABLED = flag
            out = model(_variant_batch(graph, variant, device)[1])
            tag = f"{graph}.{variant}.engine={int(flag)}"
            report(tag + ".energy", out["total_energy"], ref["total_energy"], n * 1e-5, 1e-5)
            report(tag + ".forces", out["forces"], ref["forces"], 1e-4, 1e-3)
    finally:
        engine.ENABLED = old


# ---------------------------------------------------------------------------------------------------------------------
# 5. primitives through the C ABI
# ---------------------------------------------------------------------------------------------------------------------

def _i32(a, device):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32)).to(device)


@pytest.mark.parametrize("n", [0, 1, 2047, 2048, 2049, 256 * 2048, 256 * 2048 + 1, 3_000_000])
def test_exclusive_scan(device, n):
    """Across the 2048-element tile and past the 256-tile chunk of the totals pass; out[n] is the total."""
    from torch_m3gnet_b200 import _lib

    x = np.random.default_rng(n).integers(0, 200, size=n).astype(np.int32)
    out = torch.full((n + 1,), -7, dtype=torch.int32, device=device)
    work = torch.full((_lib.scan_work_elems(n),), -7, dtype=torch.int32, device=device)
    _lib.call("exclusive_scan_i32", _i32(x, device), out, n, work)
    _equal(f"scan n={n}", out, np.concatenate([[0], np.cumsum(x, dtype=np.int64)]).astype(np.int32))


@pytest.mark.parametrize("kind", ["skewed", "empty_rows", "one_row", "uniform"])
def test_csr_by_key(device, kind):
    from torch_m3gnet_b200 import _lib

    rng = np.random.default_rng(3)
    n_rows, n = 3000, 20000
    keys = {"skewed": np.where(rng.random(n) < 0.9, 17, rng.integers(0, n_rows, size=n)),
            "empty_rows": rng.integers(0, n_rows // 10, size=n) * 10,
            "one_row": np.full(n, n_rows - 1),
            "uniform": rng.integers(0, n_rows, size=n)}[kind]
    ptr = torch.full((n_rows + 1,), -7, dtype=torch.int32, device=device)
    perm = torch.full((n,), -7, dtype=torch.int32, device=device)
    work = torch.empty(n_rows + 1 + _lib.scan_work_elems(n_rows), dtype=torch.int32, device=device)
    _lib.call("csr_by_key", _i32(keys, device), n, n_rows, ptr, perm, work)
    want_ptr, want_perm = R.csr_by_key(keys, n_rows)
    _equal("row_ptr", ptr, want_ptr)
    _equal("perm", perm, want_perm)


def test_csr_from_sorted_and_check_sorted(device):
    from torch_m3gnet_b200 import _lib

    flags = torch.empty(2, dtype=torch.int32, device=device)
    keys = np.sort(np.random.default_rng(4).integers(0, 50, size=1000)) * 2  # every odd row empty
    step = int(np.nonzero(np.diff(keys[500:]))[0][0]) + 500  # keys[step] < keys[step + 1]: swapping them descends
    descending = keys.copy()
    descending[[step, step + 1]] = keys[[step + 1, step]]
    cases = {
        "sorted": (keys, 100, [1, 1]),
        "empty": (keys[:0], 100, [1, 1]),
        "descending_pair": (descending, 100, [0, 1]),
        "key_too_large": (np.concatenate([keys, [100]]), 100, [1, 0]),
        "negative_key": (np.concatenate([[-1], keys]), 100, [1, 0]),
    }
    for name, (k, n_rows, want) in cases.items():
        _lib.call("check_sorted", _i32(k, device), len(k), n_rows, flags)
        assert flags.tolist() == want, name
    ptr = torch.full((101,), -7, dtype=torch.int32, device=device)
    _lib.call("csr_from_sorted", _i32(keys, device), len(keys), 100, ptr)
    _equal("row_ptr", ptr, np.searchsorted(keys, np.arange(101), side="left").astype(np.int32))
    _lib.call("csr_from_sorted", _i32(keys[:0], device), 0, 100, ptr)
    _equal("row_ptr (no keys)", ptr, np.zeros(101, np.int32))


def test_sort_rows_and_gather(device):
    from torch_m3gnet_b200 import _lib

    rng = np.random.default_rng(5)
    lens = np.concatenate([np.arange(0, 201), rng.integers(0, 201, size=300)])
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    cols = rng.integers(-5, 60, size=int(ptr[-1])).astype(np.int32)  # repeats and negative values
    got = _i32(cols, device)
    _lib.call("sort_rows", _i32(ptr, device), len(lens), got)
    want = np.concatenate([np.sort(cols[ptr[r]:ptr[r + 1]]) for r in range(len(lens))])
    _equal("sorted rows", got, want.astype(np.int32))
    perm = rng.permutation(len(cols)).astype(np.int32)
    out = torch.full((len(cols),), -7, dtype=torch.int32, device=device)
    _lib.call("gather_i32", _i32(cols, device), _i32(perm, device), len(cols), out)
    _equal("gather", out, cols[perm])


@pytest.mark.parametrize("W", [1, 3, 64, 65])
def test_rows_gather_and_scatter_add(device, W):
    from torch_m3gnet_b200 import _lib

    rng = np.random.default_rng(W)
    n_in, n = 700, 500
    src = torch.from_numpy(rng.standard_normal((n_in, W)).astype(np.float32))
    idx = rng.permutation(n_in)[:n].astype(np.int32)  # unique rows, as the halo exchange hands them over
    out = torch.full((n, W), -7.0, device=device)
    _lib.call("rows_gather", src.to(device), _i32(idx, device), n, W, out)
    _equal("rows_gather", out, src[torch.from_numpy(idx).long()])
    add = torch.from_numpy(rng.standard_normal((n, W)).astype(np.float32))
    acc = src.to(device)
    _lib.call("rows_scatter_add", add.to(device), _i32(idx, device), n, W, acc)
    want = src.clone()
    want[torch.from_numpy(idx).long()] += add
    _equal("rows_scatter_add", acc, want)
