"""Numpy restatements of the integer graph outputs the GPU builder and ``GraphPlan`` produce, beyond what
``oracle.m3gnet_oracle`` already states (``neighbor_list_bruteforce``, ``verlet_filter``, ``enumerate_triplets``).

Every function here is exact integer work: the GPU tests compare with ``torch.equal``.

* ``triplets_src_grouped``: the builder's triplet rule.  Member counts are taken per SOURCE atom of the member bonds,
  which equals the oracle's dst-degree walk (quirk Q6) whenever both directions of every pair agree on membership.
* ``csr_by_key``: the stable counting sort of ``m3g_csr_by_key`` (``argsort(kind="stable")``).
* ``csr_rows`` / ``csr_transpose``: the plan's triplet CSR (rows by first bond, ascending second bond) and its
  transpose, repeated triplets kept with their multiplicity.
* ``is_symmetric``: the triplet multiset equals its transpose.
* ``dense_certificate``: the canonical per-atom layout test of ``m3g_tri_dense_check`` and its ``max_members``.
"""
import numpy as np


def member_flags(distances_f32, threebody_cutoff):
    """float32 member test of the builder: float(d) <= float(r3)."""
    return (np.asarray(distances_f32, dtype=np.float32) <= np.float32(threebody_cutoff)).astype(np.int32)


def csr_by_key(keys, n_rows):
    """(row_ptr int32 (n_rows + 1), perm int32): positions sorted by key, ties in ascending position."""
    keys = np.asarray(keys, dtype=np.int64)
    perm = np.argsort(keys, kind="stable").astype(np.int32)
    ptr = np.concatenate([[0], np.cumsum(np.bincount(keys, minlength=n_rows))]).astype(np.int32)
    return ptr, perm


def csr_rows(n_rows, rows, cols):
    """(row_ptr, cols) with the entries grouped by ``rows`` and every row sorted ascending; repeats kept."""
    rows = np.asarray(rows, dtype=np.int64)
    cols = np.asarray(cols, dtype=np.int64)
    order = np.lexsort((cols, rows))
    ptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n_rows))]).astype(np.int32)
    return ptr, cols[order].astype(np.int32)


def csr_transpose(n_rows, e1, e2):
    """Rows by second bond, each holding the first bonds ascending: (e1, e2) repeated k times appears k times."""
    return csr_rows(n_rows, e2, e1)


def is_symmetric(n_rows, e1, e2):
    """True iff the multiset of (e1, e2) pairs equals the multiset of (e2, e1) pairs."""
    p, c = csr_rows(n_rows, e1, e2)
    pt, ct = csr_transpose(n_rows, e1, e2)
    return bool(np.array_equal(p, pt) and np.array_equal(c, ct))


def dense_certificate(src, n_atoms, e1, e2):
    """(dense, max_members) of a triplet list over bonds grouped by ``src``.

    A member bond is one whose triplet row is non-empty.  The layout is dense iff, for every atom, the row of each
    member bond holds exactly the atom's other member bonds, ascending, once each.  ``max_members`` is the largest
    number of member bonds of one atom (0 without triplets), whether or not the layout is dense."""
    src = np.asarray(src, dtype=np.int64)
    E = src.shape[0]
    ptr, cols = csr_rows(E, e1, e2)
    used = ptr[1:] > ptr[:-1]
    dense, max_members = True, 0
    for a in range(n_atoms):
        bonds = np.nonzero(src == a)[0]
        members = bonds[used[bonds]]
        if members.size == 0:
            continue
        max_members = max(max_members, int(members.size))
        for m in members:
            if not np.array_equal(cols[ptr[m]:ptr[m + 1]], members[members != m]):
                dense = False
    return dense, max_members


def triplets_src_grouped(num_nodes, edge_index, distances_f32, threebody_cutoff):
    """The builder's triplets (csrc/neighbor.cu triplet_count / triplet_fill) restated.

    For every atom i with member bonds m_0 < m_1 < ... (bonds leaving i whose float32 distance is <= float32(r3)):
    the ordered pairs (m_a, m_b), a != b, ascending in (a, b); atoms ascending.  Returns a dict of int arrays:
    ``triplet_edge_index`` (2, T) int64, ``num_triplet_i`` (N) int64 = n3 (n3 - 1), ``num_triplet_ij`` (E) int32
    = n3 - 1 on member bonds, ``tri_ptr`` (E + 1) int32, ``tri_e2`` (T) int32, ``member`` (E) int32 flags,
    ``member_edges`` int32 (member bonds of atoms with n3 >= 2, ascending), ``n3`` (N) and ``max_members``
    (largest n3 among atoms with n3 >= 2, else 0)."""
    src = np.asarray(edge_index[0], dtype=np.int64)
    E = src.shape[0]
    member = member_flags(distances_f32, threebody_cutoff)
    mem = np.nonzero(member)[0]
    n3 = np.bincount(src[mem], minlength=num_nodes).astype(np.int64)
    e1_parts, e2_parts = [], []
    for i in np.nonzero(n3 >= 2)[0]:
        loc = mem[src[mem] == i]
        a, b = np.meshgrid(loc, loc, indexing="ij")
        keep = a != b
        e1_parts.append(a[keep])
        e2_parts.append(b[keep])
    if e1_parts:
        tri = np.stack([np.concatenate(e1_parts), np.concatenate(e2_parts)]).astype(np.int64)
    else:
        tri = np.zeros((2, 0), dtype=np.int64)
    ntij = np.zeros(E, dtype=np.int32)
    ntij[mem] = n3[src[mem]] - 1
    heads = n3 >= 2
    return {
        "triplet_edge_index": tri,
        "num_triplet_i": n3 * (n3 - 1),
        "num_triplet_ij": ntij,
        "tri_ptr": np.concatenate([[0], np.cumsum(ntij)]).astype(np.int32),
        "tri_e2": tri[1].astype(np.int32),
        "member": member,
        "member_edges": mem[heads[src[mem]]].astype(np.int32),
        "n3": n3,
        "max_members": int(n3[heads].max()) if heads.any() else 0,
    }


def triplet_list_variants(src, tri, seed=0):
    """Hand-built triplet lists derived from a canonical one (``tri`` (2, T) over bonds grouped by ``src``), with the
    layout flags each must get: {name: (list (2, T') int64, dense, symmetric)}.

    ``member`` below is a second member bond of the atom that heads the first triplet."""
    src = np.asarray(src, dtype=np.int64)
    tri = np.asarray(tri, dtype=np.int64)
    T = tri.shape[1]
    e_first = tri[0, 0]
    atom = src[e_first]
    member = int(tri[1, 0])
    bonds_of_atom = src[tri[0]] == atom
    perm = np.random.default_rng(seed).permutation(T)
    return {
        "canonical": (tri, True, True),
        "permuted": (tri[:, perm], True, True),
        # one triplet dropped: its transpose partner stays
        "non_symmetric": (tri[:, 1:], False, False),
        # one triplet twice, its transpose once: every (r, c) has some (c, r), but not as often
        "duplicated": (np.concatenate([tri, tri[:, :1]], axis=1), False, False),
        # the member bond keeps its own row but drops out of the rows of the atom's other members
        "row_misses_member": (tri[:, (tri[1] != member) | (tri[0] == member)], False, False),
        # the member bond leaves the atom's member set entirely: again the full pair matrix of the rest
        "member_removed": (tri[:, (tri[0] != member) & (tri[1] != member)], True, True),
        # of the atom's rows only the first member's stays: a single member bond with a non-empty row
        "single_member_row": (tri[:, ~bonds_of_atom | (tri[0] == e_first)], False, False),
        # every other triplet: neither the pair matrix nor symmetric in general (flags from the helpers)
        "thinned": (tri[:, ::2], None, None),
    }
