"""CPU: BatchPhonon with the numpy restatement (tests/phonon_oracle.py) standing in for the kernels -- an exactly
harmonic spring model against its analytic dispersion, equidistant minimum images against the full supercell Hessian,
an Einstein solid against the closed-form thermal properties, Lennard-Jones fcc -- and the host side: record order,
independence from the working-set budget and from batch neighbours, failure isolation, validation, mesh_qpoints and
the minimum-image table on a skewed cell."""
import itertools

import numpy as np
import pytest
import torch

from tests import phonon_oracle as PO
from tests.test_batch_fire_cpu import BatchLJ
from tests.test_batch_neb_cpu import lj_lattice_constant
from tests.test_cell_stress_cpu import _fcc

A = 3.6                                        # lattice constant of the site models (A)
FCC_PRIM = 0.5 * A * np.array([[0.0, 1.0, 1.0], [1.0, 0.0, 1.0], [1.0, 1.0, 0.0]])
K_SPRING = 1.7                                 # eV/A^2
M1, M2 = 63.546, 12.011


class SiteModel:
    """``compute``'s protocol for crystals whose sites sit on the a/2 grid: u = r - (r rounded to the grid), float64
    forces.  ``kind`` "spring": E = 1/2 sum over bonds k (d^.(u_i - u_j))^2, bonds between sites ``r_bond`` apart
    (every periodic image); "einstein": E = 1/2 k sum |u_i|^2."""

    def __init__(self, kind, r_bond=None, k=K_SPRING, device=torch.device("cpu")):
        self.kind, self.r_bond, self.k, self.device = kind, r_bond, k, device
        self.calls = []
        self._bonds = {}

    def bonds(self, lat, R):
        key = (lat.tobytes(), R.tobytes())
        if key not in self._bonds:
            t = np.stack(np.meshgrid(*[np.arange(-2, 3)] * 3, indexing="ij"), -1).reshape(-1, 3) @ lat
            d = R[None, :, None, :] + t[None, None] - R[:, None, None, :]
            r = np.linalg.norm(d, axis=-1)
            i, j, m = np.nonzero(np.abs(r - self.r_bond) < 1e-6)
            self._bonds[key] = (i, j, d[i, j, m] / self.r_bond)
        return self._bonds[key]

    def forces(self, lat, cart):
        R = np.round(cart / (A / 2)) * (A / 2)
        u = cart - R
        if self.kind == "einstein":
            return -self.k * u
        i, j, dh = self.bonds(lat, R)
        f = -self.k * dh * ((u[i] - u[j]) * dh).sum(axis=1, keepdims=True)
        out = np.zeros_like(u)
        np.add.at(out, i, f)
        return out

    def compute(self, lattices, cart, atomic_numbers, sizes=None, with_stress=False):
        cart = np.asarray(cart, dtype=np.float64).reshape(-1, 3)
        sizes = [len(cart)] if sizes is None else [int(n) for n in sizes]
        lat = np.asarray(lattices, dtype=np.float64).reshape(len(sizes), 3, 3)
        self.calls.append(tuple(sizes))
        ptr = np.concatenate([[0], np.cumsum(sizes)])
        f = np.concatenate([self.forces(lat[b], cart[ptr[b]:ptr[b + 1]]) for b in range(len(sizes))])
        return (torch.zeros(len(sizes), dtype=torch.float64, device=self.device),
                torch.from_numpy(f).to(self.device), torch.zeros((len(sizes), 6), dtype=torch.float64))


@pytest.fixture
def restated(monkeypatch):
    from torch_m3gnet_b200 import phonon

    for name in ("fc_launch", "frequencies_launch", "thermal_launch"):
        monkeypatch.setattr(phonon, name, getattr(PO, name))
    return phonon


def fcc_conventional(a=A):
    lat, cart = _fcc(a)
    return lat, cart, np.full(4, 29)


def rock_salt_conventional(a=A):
    lat, c1 = _fcc(a)
    cart = np.concatenate([c1, c1 + np.array([0.5 * a, 0.0, 0.0])])
    return lat, cart, np.array([29] * 4 + [6] * 4)


def analytic_eigs(lat, cart, masses, r_bond, q_frac, k=K_SPRING):
    """Eigenvalues of the spring model's D(q) in closed form: D = [delta_kk' sum_{bonds of k} k d^d^T
    - sum_{bonds k->k'} k d^d^T exp(i q.d)] / sqrt(m_k m_k') over the bonds of the infinite crystal (for one atom per
    cell this is sum_d k (1 - cos q.d) d^d^T / m)."""
    n = len(cart)
    qc = 2 * np.pi * np.linalg.solve(lat, q_frac)              # Cartesian q: q_c . (f @ lat) = 2 pi q_frac . f
    t = np.stack(np.meshgrid(*[np.arange(-3, 4)] * 3, indexing="ij"), -1).reshape(-1, 3) @ lat
    D = np.zeros((n, 3, n, 3), complex)
    for a in range(n):
        for b in range(n):
            d = cart[b] + t - cart[a]
            for dv in d[np.abs(np.linalg.norm(d, axis=1) - r_bond) < 1e-6]:
                dd = np.outer(dv, dv) / r_bond ** 2 * k
                D[a, :, a, :] += dd / masses[a]
                D[a, :, b, :] -= dd * np.exp(1j * qc @ dv) / np.sqrt(masses[a] * masses[b])
    return np.linalg.eigvalsh(D.reshape(3 * n, 3 * n))


def random_q(count, seed=0):
    return np.random.default_rng(seed).uniform(-0.5, 0.5, (count, 3))


# ---------------------------------------------------------------------------------------------------------------------
# physics
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("variant", ["fcc", "rock_salt"])
def test_spring_model_matches_the_analytic_dispersion(restated, variant):
    if variant == "fcc":
        s, masses, r_bond, reps = fcc_conventional(), {29: M1}, A / np.sqrt(2), (3, 3, 3)
    else:
        s, masses, r_bond, reps = rock_salt_conventional(), {29: M1, 6: M2}, A / 2, (2, 2, 2)
    ph = restated.BatchPhonon(SiteModel("spring", r_bond), [s], reps, masses)
    rec = ph.run()[0]
    assert rec["status"] == "ok" and rec["max_residual_force"] == 0.0
    tables = restated.minimum_images(s[0], s[1], reps)
    nn = np.abs(rec["force_constants"]).reshape(len(s[2]) * len(s[2]) * np.prod(reps), 9).max(axis=1) > 0
    assert (np.diff(tables[0])[nn] == 1).all()                   # every bonded pair has a unique minimum image
    q = random_q(12)
    got = ph.frequencies(q)[0]
    m = np.array([masses[z] for z in s[2]])
    worst = 0.0
    for i in range(len(q)):
        want = analytic_eigs(s[0], s[1], m, r_bond, q[i])
        lam = np.sign(got[i]) * (got[i] / PO.THZ) ** 2
        worst = max(worst, np.abs(lam - want).max() / np.abs(want).max())
    print(f"[phonon-spring] {variant}: max relative eigenvalue error {worst:.2e}")
    assert worst < 1e-9


def supercell_hessian_eigs(calc, lat, cart, masses, h=1e-3):
    """Eigenvalues of the mass-weighted 3N x 3N Hessian of an exactly harmonic calculator (central differences)."""
    x = cart.reshape(-1)
    H = np.empty((x.size, x.size))
    for c in range(x.size):
        d = np.zeros_like(x)
        d[c] = h
        fp = calc.forces(lat, (x + d).reshape(-1, 3)).reshape(-1)
        fm = calc.forces(lat, (x - d).reshape(-1, 3)).reshape(-1)
        H[:, c] = -(fp - fm) / (2 * h)
    w = 1 / np.sqrt(np.repeat(masses, 3))
    return np.linalg.eigvalsh(0.5 * (H + H.T) * np.outer(w, w))


@pytest.mark.parametrize("cell", ["fcc_primitive", "rock_salt_primitive"])
def test_equidistant_images_hermitian_and_supercell_hessian(restated, cell):
    from torch_m3gnet_b200 import phonon

    if cell == "fcc_primitive":
        s, masses, r_bond = (FCC_PRIM, np.zeros((1, 3)), np.array([29])), {29: M1}, A / np.sqrt(2)
    else:
        s, masses, r_bond = (FCC_PRIM, np.array([[0, 0, 0], [A / 2, 0, 0]]), np.array([29, 6])), {29: M1, 6: M2}, A / 2
    reps = (2, 2, 2)
    calc = SiteModel("spring", r_bond)
    ph = restated.BatchPhonon(calc, [s], reps, masses)
    ph.run()
    sv_ptr, _ = phonon.minimum_images(s[0], s[1], reps)
    if cell == "fcc_primitive":
        assert np.diff(sv_ptr).max() > 1                         # equidistant images exist
    st = ph._st
    for q in random_q(6, seed=1):
        D = PO.structure_dynmat(st, 0, q)
        assert np.abs(D - D.conj().T).max() <= 1e-12 * np.linalg.norm(D)
    comm = np.array(list(itertools.product([0.0, 0.5], repeat=3)))
    lam = np.sort(np.concatenate([np.sign(f) * (f / PO.THZ) ** 2 for f in ph.frequencies(comm)[0]]))
    S, pos = phonon.supercell(s[0], s[1], reps)
    m = np.tile([masses[z] for z in s[2]], 8)
    want = supercell_hessian_eigs(calc, S, pos, m)
    err = np.abs(lam - want).max() / np.abs(want).max()
    print(f"[phonon-equidistant] {cell}: max image count {np.diff(sv_ptr).max()}, commensurate vs supercell Hessian "
          f"{err:.2e}")
    assert err < 1e-10


def test_einstein_solid_closed_form(restated):
    kappa = 2.3
    s = fcc_conventional()
    ph = restated.BatchPhonon(SiteModel("einstein", k=kappa), [s], (2, 2, 2), {29: M1}, symmetrize=0)
    ph.run()
    fE = np.sqrt(kappa / M1) * PO.THZ
    f = ph.frequencies(random_q(5))[0]
    np.testing.assert_allclose(f, fE, rtol=1e-12)
    temps = np.array([0.0, 1.0, 50.0, 300.0, 1000.0, 1e6])
    th = ph.thermal_properties(mesh=(3, 2, 2), temperatures=temps)[0]
    e = PO.H_THZ * fE
    n3 = 3 * len(s[2])
    with np.errstate(divide="ignore", over="ignore", invalid="ignore"):
        x = e / (PO.KB * temps)
        F = n3 * (e / 2 + np.where(temps > 0, PO.KB * temps * np.log1p(-np.exp(-x)), 0.0))
        S = n3 * PO.KB * np.where(temps > 0, x / np.expm1(x) - np.log1p(-np.exp(-x)), 0.0)
        C = n3 * PO.KB * np.where(temps > 0, x * x * np.exp(-x) / np.expm1(-x) ** 2, 0.0)
        E = n3 * e * (0.5 + np.where(temps > 0, 1 / np.expm1(x), 0.0))
    for key, want in (("free_energy", F), ("entropy", S), ("heat_capacity", C), ("energy", E)):
        np.testing.assert_allclose(th[key], want, rtol=1e-12, atol=1e-12 * np.abs(want).max(), err_msg=key)
    assert th["heat_capacity"][-1] == pytest.approx(n3 * PO.KB, rel=1e-8)        # Dulong-Petit (1 - x^2/12)
    assert th["free_energy"][0] == th["energy"][0] == pytest.approx(n3 * e / 2, rel=1e-14)
    assert th["n_imaginary"] == 0 and th["min_frequency"] == pytest.approx(fE, rel=1e-12)


def lj_fcc(perm=None):
    a = lj_lattice_constant()
    lat, cart = _fcc(a)
    if perm is not None:
        cart = cart[perm]
    return lat, cart, np.full(4, 18)


def test_lennard_jones_fcc(restated):
    ph = restated.BatchPhonon(BatchLJ(), [lj_fcc(), lj_fcc([2, 0, 3, 1])], (3, 3, 3), {18: 39.948})
    recs = ph.run()
    assert all(r["status"] == "ok" for r in recs)
    gamma = ph.frequencies(np.zeros((1, 3)))
    q = random_q(8, seed=4)
    fq, fmq = ph.frequencies(q), ph.frequencies(-q)
    print(f"[phonon-lj] Gamma acoustic {gamma[0][0, :3]} THz, max |f(q) - f(-q)| "
          f"{np.abs(fq[0] - fmq[0]).max():.2e}, permuted {np.abs(fq[0] - fq[1]).max():.2e} THz, "
          f"residual {recs[0]['max_residual_force']:.2e} eV/A")
    assert np.abs(gamma[0][0, :3]).max() < 1e-3 and gamma[0][0, 3:].min() > 1.0
    np.testing.assert_allclose(fq[0], fmq[0], rtol=0, atol=1e-10 * np.abs(fq[0]).max())
    np.testing.assert_allclose(fq[0], fq[1], rtol=0, atol=1e-6 * np.abs(fq[0]).max())


# ---------------------------------------------------------------------------------------------------------------------
# host logic
# ---------------------------------------------------------------------------------------------------------------------

def ragged_lj():
    """LJ cells of 4, 1 and 8 atoms, jittered, with different supercells."""
    rng = np.random.default_rng(5)
    a = lj_lattice_constant()
    lat, cart = _fcc(a)
    out = [(lat, cart + rng.uniform(-0.03, 0.03, cart.shape), np.full(4, 18))]
    prim = 0.5 * a * np.array([[0.0, 1.0, 1.0], [1.0, 0.0, 1.0], [1.0, 1.0, 0.0]])
    out.append((prim, np.zeros((1, 3)), np.array([18])))
    lat2 = np.diag([a, a, 2 * a])
    c2 = np.concatenate([cart, cart + [0, 0, a]])
    out.append((lat2, c2 + rng.uniform(-0.03, 0.03, c2.shape), np.full(8, 18)))
    return out, [(2, 2, 2), (3, 3, 3), (2, 2, 1)]


def _run(mod, structs, reps, **kw):
    calc = BatchLJ()
    ph = mod.BatchPhonon(calc, structs, reps, {18: 39.948}, **kw)
    return ph, ph.run(), calc


def test_order_budget_and_neighbours(restated):
    structs, reps = ragged_lj()
    ph, ref, calc = _run(restated, structs, reps)
    n = [len(s[2]) for s in structs]
    N = [a * int(np.prod(r)) for a, r in zip(n, reps)]
    assert calc.calls == [tuple(N[b] for b in range(3) for _ in range(6 * n[b] + 1))]
    q = random_q(4, seed=6)
    fref = ph.frequencies(q)
    for budget in (100, 300):
        ph2, got, calc2 = _run(restated, structs, reps, max_atoms=budget)
        assert len(calc2.calls) > 1 and all(sum(c) <= budget or len(c) == 1 for c in calc2.calls)
        for a, b in zip(ref, got):
            assert a["status"] == b["status"]
            assert np.array_equal(a["force_constants"], b["force_constants"])
        for a, b in zip(fref, ph2.frequencies(q)):
            assert np.array_equal(a, b)
    for order in ([2, 0, 1], [1]):                               # other neighbours, other positions
        ph3, got, _ = _run(restated, [structs[i] for i in order], [reps[i] for i in order], max_atoms=150)
        f3 = ph3.frequencies(q)
        for j, i in enumerate(order):
            assert np.array_equal(got[j]["force_constants"], ref[i]["force_constants"])
            assert np.array_equal(f3[j], fref[i])
    for b, r in enumerate(ref):
        assert r["force_constants"].shape == (n[b], N[b], 3, 3)
        np.testing.assert_array_equal(r["supercell_lattice"], structs[b][0] * np.array(reps[b])[:, None])
        assert r["max_residual_force"] > 0
    per = [q[:2], q[1:], q[:1]]
    fper = ph.frequencies(per)
    for b in range(3):
        assert fper[b].shape == (len(per[b]), 3 * n[b])
        assert np.array_equal(fper[b], fref[b][[0, 1] if b == 0 else [1, 2, 3] if b == 1 else [0]])


def test_failure_is_isolated(restated):
    structs, reps = ragged_lj()
    ph, ref, _ = _run(restated, structs, reps)
    lat, cart, z = structs[2]
    cart = cart.copy()
    cart[1] = cart[0] + np.array([1e-6, 0.0, 0.0])               # float32 LJ forces overflow
    bad = [structs[0], structs[1], (lat, cart, z)]
    ph2, got, _ = _run(restated, bad, reps)
    assert got[2]["status"] == "failed" and np.isnan(got[2]["force_constants"]).all()
    assert np.isnan(got[2]["max_residual_force"])
    q = random_q(3, seed=7)
    f_ref, f_got = ph.frequencies(q), ph2.frequencies(q)
    assert np.isnan(f_got[2]).all()
    th_ref = ph.thermal_properties(mesh=(2, 2, 2), temperatures=[0, 300])
    th_got = ph2.thermal_properties(mesh=(2, 2, 2), temperatures=[0, 300])
    assert np.isnan(th_got[2]["free_energy"]).all() and th_got[2]["n_imaginary"] == -1
    for b in (0, 1):
        assert got[b]["status"] == "ok"
        assert np.array_equal(got[b]["force_constants"], ref[b]["force_constants"])
        assert np.array_equal(f_got[b], f_ref[b])
        for k in ("free_energy", "entropy", "heat_capacity", "energy"):
            assert np.array_equal(th_got[b][k], th_ref[b][k])


def test_validation():
    from torch_m3gnet_b200.phonon import MAX_ATOMS, BatchPhonon

    calc = BatchLJ()
    s = lj_fcc()
    m = {18: 39.948}
    big = (np.eye(3) * 20, np.random.default_rng(0).uniform(0, 20, (MAX_ATOMS + 1, 3)), np.full(MAX_ATOMS + 1, 18))
    with pytest.raises(ValueError, match="at most"):
        BatchPhonon(calc, [s, big], (1, 1, 1), m)
    with pytest.raises(ValueError, match="at least 1"):
        BatchPhonon(calc, [s], (2, 0, 2), m)
    with pytest.raises(ValueError, match="integers"):
        BatchPhonon(calc, [s], (2, 1.5, 2), m)
    with pytest.raises(ValueError, match="supercell"):
        BatchPhonon(calc, [s, s], [(2, 2, 2)] * 3, m)
    for h in (0.0, -0.01, np.nan, np.inf):
        with pytest.raises(ValueError, match="displacement"):
            BatchPhonon(calc, [s], (2, 2, 2), m, displacement=h)
    with pytest.raises(ValueError, match="no mass"):
        BatchPhonon(calc, [s], (2, 2, 2), {29: 63.5})
    with pytest.raises(ValueError, match="finite and positive"):
        BatchPhonon(calc, [s], (2, 2, 2), [np.array([1.0, 1.0, -1.0, 1.0])])
    with pytest.raises(ValueError, match="expected 1 arrays"):
        BatchPhonon(calc, [s], (2, 2, 2), [np.ones(4), np.ones(4)])
    with pytest.raises(ValueError, match="symmetrize"):
        BatchPhonon(calc, [s], (2, 2, 2), m, symmetrize=-1)
    with pytest.raises(ValueError, match="max_atoms"):
        BatchPhonon(calc, [s], (2, 2, 2), m, max_atoms=0)
    ph = BatchPhonon(calc, [s, s], [(2, 2, 2), (1, 2, 3)], m)
    assert ph.reps.tolist() == [[2, 2, 2], [1, 2, 3]]
    with pytest.raises(RuntimeError, match="run"):
        ph.frequencies(np.zeros((1, 3)))
    assert BatchPhonon(calc, [], (2, 2, 2), m).run() == []


def test_thermal_validation(restated):
    ph, _, _ = _run(restated, [lj_fcc()], [(1, 1, 1)])
    with pytest.raises(ValueError, match="temperatures"):
        ph.thermal_properties(mesh=(2, 2, 2), temperatures=[-1.0])
    with pytest.raises(ValueError, match="mesh"):
        ph.thermal_properties(mesh=(2, 0, 2))
    with pytest.raises(ValueError, match="qpoints"):
        ph.frequencies([np.zeros((1, 3)), np.zeros((1, 3))])


def test_mesh_qpoints():
    from torch_m3gnet_b200.phonon import mesh_qpoints

    for mesh in ((1, 1, 1), (4, 3, 5), (2, 2, 2)):
        q = mesh_qpoints(mesh)
        assert q.shape == (int(np.prod(mesh)), 3)
        assert (q > -0.5).all() and (q <= 0.5).all()
        assert np.array_equal(q[0], [0.0, 0.0, 0.0])
        idx = np.round(q * np.array(mesh)).astype(int) % np.array(mesh)
        assert len({tuple(i) for i in idx}) == len(q)             # every point of the mesh once
        np.testing.assert_allclose(q * np.array(mesh), np.round(q * np.array(mesh)), atol=1e-12)
    q = mesh_qpoints((4, 3, 5))
    assert np.array_equal(q[1], [0.0, 0.0, 0.2]) and np.array_equal(q[5], [0.0, 1 / 3, 0.0])


def test_minimum_image_table_on_a_skewed_cell():
    from torch_m3gnet_b200.phonon import minimum_images, supercell

    lat = np.array([[3.1, 0.0, 0.0], [1.4, 2.9, 0.0], [-0.8, 0.9, 3.3]])
    cart = np.array([[0.1, 0.2, 0.3], [1.9, 1.1, 1.7], [2.6, -0.4, 3.9]])   # one atom outside the cell
    reps = np.array([2, 3, 2])
    sv_ptr, sv = minimum_images(lat, cart, reps)
    S, pos = supercell(lat, cart, reps)
    n, N = len(cart), len(pos)
    assert sv_ptr.shape == (n * N + 1,) and sv_ptr[-1] == len(sv) and (np.diff(sv_ptr) >= 1).all()
    big = np.stack(np.meshgrid(*[np.arange(-5, 6)] * 3, indexing="ij"), -1).reshape(-1, 3)
    multi = 0
    for k in range(n):
        for j in range(N):
            d = pos[j] + big @ S - cart[k]
            r = np.linalg.norm(d, axis=1)
            want = {tuple(x) for x in np.round((d[r <= r.min() * (1 + 1e-5)] - (cart[j % n] - cart[k]))
                                               @ np.linalg.inv(lat)).astype(int)}
            p = k * N + j
            got = sv[sv_ptr[p]:sv_ptr[p + 1]]
            np.testing.assert_array_equal(got, np.round(got))
            assert {tuple(x) for x in got.astype(int)} == want, (k, j)
            multi += len(got) > 1
    # a cubic cell's half-supercell vectors: equidistant images are all kept
    sv_ptr, sv = minimum_images(np.eye(3) * 2.0, np.zeros((1, 3)), (2, 2, 2))
    assert np.diff(sv_ptr).tolist() == [1, 2, 2, 4, 2, 4, 4, 8]
