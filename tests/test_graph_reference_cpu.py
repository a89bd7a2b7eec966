"""CPU: the numpy restatements of tests/graph_reference.py against the oracle's graph build on the existing fixtures,
and the layout certificate / symmetry test on hand-made positive and negative triplet lists.  The GPU graph tests
(tests/test_gpu_graph_reference.py) compare the kernels with these helpers, so they are checked first."""
import numpy as np
import pytest

from oracle import m3gnet_oracle as O
from tests import graph_reference as R
from tests.util import golden


def _fixtures():
    r_nn = 3.0
    lat_al = r_nn * np.sqrt(2) * np.eye(3)
    fr_al = np.array([[0, 0, 0], [0, 0.5, 0.5], [0.5, 0, 0.5], [0.5, 0.5, 0]])
    g = golden("tio2_default")
    return {
        "fcc_al": (lat_al, fr_al @ lat_al, [13] * 4, r_nn + 1e-4, r_nn + 1e-4),
        "unit_cube": (np.eye(3), np.array([[0, 0, 0], [0.5, 0.5, 0.5], [0.5, 0, 0], [0, 0.5, 0.5]]), [3, 3, 1, 1],
                      1.0, 1.0),
        "cu32": O.fcc_supercell(2, jitter=0.05, seed=0) + (5.0, 4.0),
        "tio2": (g["g.lattice"][0].astype(np.float64), g["g.pos"].astype(np.float64), [22] * 8 + [8] * 24, 5.0, 4.0),
        "mpf3": O.mpf_like_structure(3) + (5.0, 4.0),
    }


FIXTURES = _fixtures()


@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_src_grouped_triplets_equal_the_oracle(name):
    """On graphs whose pairs agree on membership in both directions, the src-grouped rule is the oracle's rule."""
    lat, cart, z, r, r3 = FIXTURES[name]
    g = O.build_graph(lat, cart, z, r, r3)
    ei = g["edge_index"].numpy()
    d32 = g["edge_distances_build"].numpy()
    ref = R.triplets_src_grouped(len(cart), ei, d32, r3)
    assert np.array_equal(ref["triplet_edge_index"], g["triplet_edge_index"].numpy())
    assert np.array_equal(ref["num_triplet_i"], g["num_triplet_i"].numpy())
    assert np.array_equal(ref["num_triplet_ij"], g["num_triplet_ij"].numpy())
    tri = ref["triplet_edge_index"]
    ptr, cols = R.csr_rows(ei.shape[1], tri[0], tri[1])
    assert np.array_equal(ptr, ref["tri_ptr"]) and np.array_equal(cols, ref["tri_e2"])
    # the canonical list is its own transpose and has the dense layout, with the builder's max_members
    assert R.is_symmetric(ei.shape[1], tri[0], tri[1])
    assert R.dense_certificate(ei[0], len(cart), tri[0], tri[1]) == (True, ref["max_members"])
    used = np.nonzero(ptr[1:] > ptr[:-1])[0]
    assert np.array_equal(used, ref["member_edges"])


def test_src_grouped_triplets_differ_from_the_dst_walk_when_directions_disagree():
    """A bond i->j that is a member while j->i is not: the src-grouped rule counts it at i, the oracle's dst walk
    (quirk Q6) at j, so the two lists differ."""
    ei = np.array([[0, 0, 1, 2], [1, 2, 0, 0]])
    d32 = np.array([1.0, 1.0, 2.5, 1.0], dtype=np.float32)  # 0->1 member, 1->0 not
    ref = R.triplets_src_grouped(3, ei, d32, 2.0)
    assert ref["n3"].tolist() == [2, 0, 1]
    assert ref["triplet_edge_index"].tolist() == [[0, 1], [1, 0]]
    tri, nti, _ = O.enumerate_triplets(3, ei, d32, 2.0)
    assert nti.tolist() == [0, 0, 0] and tri.shape == (2, 0)  # dst degrees [1, 1, 1]: no triplets


def test_member_flags_are_the_float32_test():
    r3 = 4.0000001
    d = np.array([np.float32(r3), np.nextafter(np.float32(r3), np.float32(9)), np.float32(3.9)], dtype=np.float32)
    assert R.member_flags(d, r3).tolist() == [1, 0, 1]


def test_csr_by_key_is_a_stable_counting_sort():
    rng = np.random.default_rng(0)
    keys = np.concatenate([np.zeros(50, np.int64), rng.integers(0, 40, size=200), np.full(30, 39)])
    rng.shuffle(keys)
    ptr, perm = R.csr_by_key(keys, 45)
    want = [i for k in range(45) for i in range(len(keys)) if keys[i] == k]
    assert perm.tolist() == want
    assert ptr.tolist() == [sum(keys < k) for k in range(46)]
    assert ptr[41:].tolist() == [len(keys)] * 5  # empty rows at the end


def test_csr_transpose_keeps_multiplicities():
    e1 = np.array([3, 0, 0, 1, 0])
    e2 = np.array([0, 1, 1, 0, 3])
    ptr, cols = R.csr_transpose(4, e1, e2)
    assert ptr.tolist() == [0, 2, 4, 4, 5] and cols.tolist() == [1, 3, 0, 0, 0]
    assert not R.is_symmetric(4, e1, e2)  # (0, 1) twice, (1, 0) once
    assert R.is_symmetric(4, np.array([0, 1, 0, 1]), np.array([1, 0, 1, 0]))


@pytest.mark.parametrize("name", ["cu32", "tio2"])
def test_certificate_on_hand_made_lists(name):
    lat, cart, z, r, r3 = FIXTURES[name]
    g = O.build_graph(lat, cart, z, r, r3)
    ei = g["edge_index"].numpy()
    E = ei.shape[1]
    tri = g["triplet_edge_index"].numpy()
    n3_max = R.triplets_src_grouped(len(cart), ei, g["edge_distances_build"].numpy(), r3)["max_members"]
    variants = R.triplet_list_variants(ei[0], tri)
    for vname, (t, dense, sym) in variants.items():
        got_dense, got_max = R.dense_certificate(ei[0], len(cart), t[0], t[1])
        got_sym = R.is_symmetric(E, t[0], t[1])
        if dense is not None:
            assert (got_dense, got_sym) == (dense, sym), vname
        assert got_max <= n3_max, vname
    assert R.dense_certificate(ei[0], len(cart), tri[0], tri[1])[1] == n3_max
    # the member bond that left its atom's member set lowers that atom's count by one
    t = variants["member_removed"][0]
    atom = ei[0][tri[0, 0]]
    assert (np.unique(t[0][ei[0][t[0]] == atom]).size
            == np.unique(tri[0][ei[0][tri[0]] == atom]).size - 1)
