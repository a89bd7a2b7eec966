"""CPU: the numpy restatement of the batched NEB step (tests/neb_oracle.py) -- the force projections and every tangent
branch, the Mueller-Brown saddle and a Lennard-Jones vacancy hop found by BatchNEB with the restatement standing in for
the kernel -- and BatchNEB's host side: results in input order, independence from the working-set budget, endpoint
evaluation, failure isolation, limits, validation and interpolation."""
import numpy as np
import pytest
import torch
from scipy.optimize import minimize_scalar, root

from tests import fire_oracle as FO
from tests import neb_oracle as NO
from tests.test_batch_fire_cpu import BatchLJ
from tests.test_cell_stress_cpu import _fcc, lj

# Mueller-Brown (Mueller & Brown 1979): minima near A and B, the saddle between them
MB_A = np.array([-200.0, -100.0, -170.0, 15.0])
MB_a = np.array([-1.0, -1.0, -6.5, 0.7])
MB_b = np.array([0.0, 0.0, 11.0, 0.6])
MB_c = np.array([-10.0, -10.0, -6.5, 0.7])
MB_x0 = np.array([1.0, 0.0, -0.5, -1.0])
MB_y0 = np.array([0.0, 0.5, 1.5, 1.0])
MB_MIN_A, MB_MIN_B = (-0.558, 1.442), (0.623, 0.028)
MB_SCALE, MB_CELL = 0.01, 100.0


def mb(p):
    """Energy 0.01 MB(x, y) + z^2 / 2 (eV) and its gradient at p = (x, y, z)."""
    x, y, z = p
    dx, dy = x - MB_x0, y - MB_y0
    t = MB_A * np.exp(MB_a * dx * dx + MB_b * dx * dy + MB_c * dy * dy)
    gx = (t * (2 * MB_a * dx + MB_b * dy)).sum()
    gy = (t * (MB_b * dx + 2 * MB_c * dy)).sum()
    return MB_SCALE * t.sum() + 0.5 * z * z, np.array([MB_SCALE * gx, MB_SCALE * gy, z])


class BatchMB:
    """``compute``'s protocol for one-atom images on the Mueller-Brown surface, in a large cubic cell; energy and forces
    rounded to float32 as the model's are, returned on ``device``."""

    def __init__(self, device=torch.device("cpu")):
        self.device = device
        self.calls = []

    def compute(self, lattices, cart, atomic_numbers, sizes=None, with_stress=False):
        cart = cart.cpu().numpy() if torch.is_tensor(cart) else np.asarray(cart, dtype=np.float64)
        cart = cart.reshape(-1, 3)
        sizes = [len(cart)] if sizes is None else [int(n) for n in sizes]
        assert all(n == 1 for n in sizes)
        self.calls.append(tuple(sizes))
        with np.errstate(over="ignore", invalid="ignore"):
            ef = [mb(p) for p in cart]
            e32 = np.asarray([e for e, _ in ef]).astype(np.float32)
            f32 = -np.stack([g for _, g in ef]).astype(np.float32)
        return (torch.from_numpy(e32).to(self.device), torch.from_numpy(f32).to(self.device),
                torch.zeros((len(sizes), 6), dtype=torch.float32, device=self.device))


def mb_point(x, y, z=0.0):
    return (np.eye(3) * MB_CELL, np.array([[x, y, z]]), np.array([1]))


def mb_saddle():
    s = root(lambda q: mb((q[0], q[1], 0.0))[1][:2], [-0.82, 0.62], tol=1e-12)
    assert np.abs(mb((s.x[0], s.x[1], 0.0))[1][:2]).max() < 1e-10
    return s.x


def mb_hessian(x, y, h=1e-5):
    H = np.empty((2, 2))
    for k in range(2):
        d = np.zeros(3)
        d[k] = h
        H[:, k] = (mb(np.array([x, y, 0.0]) + d)[1][:2] - mb(np.array([x, y, 0.0]) - d)[1][:2]) / (2 * h)
    return 0.5 * (H + H.T)


def oracle_step(st, forces, energy, climb, fire, fmax, steps):
    """neb.neb_step with the numpy restatement in place of the kernel (CPU tensors)."""
    d = {k: getattr(st, k).numpy().copy() for k in NO.STATE_KEYS}
    NO.neb_step(d, forces.double().numpy(), energy.double().numpy(), st.ends.numpy(), st.e_end.numpy(), st.k.numpy(),
                climb, fire, fmax, steps, st.row_ptr.numpy(), st.image_ptr.numpy(), st.end_ptr.numpy())
    for k, val in d.items():
        getattr(st, k).copy_(torch.from_numpy(val))


@pytest.fixture
def restated(monkeypatch):
    from torch_m3gnet_b200 import neb

    monkeypatch.setattr(neb, "neb_step", oracle_step)
    return neb


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f"), k


# ---------------------------------------------------------------------------------------------------------------------
# the restatement's forces
# ---------------------------------------------------------------------------------------------------------------------

# band energies hitting every tangent branch; the expected (c+, c-) of t = c+ t+ + c- t- per interior image
BRANCH_E = np.array([0.0, 1.0, 2.0, 1.0, 0.5, 0.5, 0.5, 3.0, 3.0, 1.0, 0.0])
BRANCH_C = [(1.0, 0.0),   # 1: rising -> t+
            (1.0, 1.0),   # 2: E_{i+1} = E_{i-1} (a local maximum): dVmin t+ + dVmax t-, both 1
            (0.0, 1.0),   # 3: falling -> t-
            (0.0, 0.5),   # 4: E_{i+1} = E_i < E_{i-1}: dVmin t+ + dVmax t-
            (1.0, 1.0),   # 5: flat triplet -> t+ + t-
            (2.5, 0.0),   # 6: E_{i-1} = E_i < E_{i+1}: dVmax t+ + dVmin t-
            (2.5, 0.0),   # 7: the first of two highest images (the climbing one): dVmax t+ + dVmin t-
            (0.0, 2.0),   # 8: the second: dVmin t+ + dVmax t-
            (0.0, 1.0)]   # 9: falling -> t-


@pytest.mark.parametrize("climb", [False, True])
def test_restatement_forces_and_tangent_branches(climb):
    rng = np.random.default_rng(0)
    M, n, k = len(BRANCH_E) - 2, 5, 0.37
    R = np.cumsum(rng.normal(0, 0.3, (M + 2, n, 3)), axis=0)
    F = rng.normal(0, 1.0, (M, n, 3))
    G, ic, ok = NO.neb_forces(BRANCH_E, R, F, k, climb)
    assert ok and ic == 7                                   # the two-way tie goes to the lower index
    for i in range(1, M + 1):
        t, tp, tm = NO.tangent(BRANCH_E, R, i)
        cp, cm = BRANCH_C[i - 1]
        np.testing.assert_allclose(t, cp * tp + cm * tm, rtol=0, atol=1e-15)
        th = t / np.sqrt((t * t).sum())
        g, f = G[i - 1], F[i - 1]
        g_t, f_t = (g * th).sum(), (f * th).sum()
        if climb and i == ic:
            assert g_t == pytest.approx(-f_t, rel=1e-12, abs=1e-13)
        else:
            spring = k * (np.sqrt((tp * tp).sum()) - np.sqrt((tm * tm).sum()))
            assert g_t == pytest.approx(spring, rel=1e-12, abs=1e-13)
        np.testing.assert_allclose(g - g_t * th, f - f_t * th, rtol=0, atol=1e-13)


def test_restatement_degenerate_band():
    R = np.zeros((3, 2, 3))
    R[2] = 1.0
    R[1] = R[0]                                             # t- = 0, and a falling triplet takes t = t-
    _, _, ok = NO.neb_forces(np.array([1.0, 0.5, 0.0]), R, np.ones((1, 2, 3)), 0.1, False)
    assert not ok
    _, _, ok = NO.neb_forces(np.array([0.0, 0.5, 1.0]), R, np.ones((1, 2, 3)), 0.1, False)
    assert ok                                               # a rising triplet takes t = t+, which is not 0


# ---------------------------------------------------------------------------------------------------------------------
# known saddles
# ---------------------------------------------------------------------------------------------------------------------

def run_mb(neb_mod, calc, fmax=1e-3, steps=1000):
    opt = neb_mod.BatchNEB(calc, [(mb_point(*MB_MIN_A), mb_point(*MB_MIN_B))], n_images=9, climb=True)
    return opt.run(fmax=fmax, steps=steps)[0]


def check_mb_saddle(r):
    s = mb_saddle()
    np.testing.assert_allclose(s, [-0.822002, 0.624313], atol=1e-6)
    p = r["positions"][r["i_climb"], 0]
    err = np.hypot(*(p[:2] - s))
    eig = np.linalg.eigvalsh(mb_hessian(*s))
    print(f"[neb-mb] {r['status']} in {r['n_steps']} steps, climbing image {r['i_climb']} at {p[:2]}, "
          f"|dx| = {err:.2e}, Hessian eigenvalues {eig}, barrier {r['barrier_forward']:.6f} eV")
    assert r["status"] == "converged" and r["fmax"] < 1e-3
    assert err < 5e-4
    assert eig[0] < 0 < eig[1]
    assert r["positions"].shape == (11, 1, 3) and r["energies"].shape == (11,)
    assert r["energies"][r["i_climb"]] == r["energies"].max()


def test_mueller_brown_climbing_image_finds_the_saddle(restated):
    check_mb_saddle(run_mb(restated, BatchMB()))


def lj_lattice_constant():
    _, c1 = _fcc(1.0)
    return minimize_scalar(lambda a: lj(np.eye(3) * a, c1 * a)[0], bounds=(3.0, 4.5), method="bounded",
                           options=dict(xatol=1e-10)).x


def lj_vacancy_hop(fire_relax):
    """(initial, final) of a nearest-neighbour hop into a vacancy of a 2x2x2 fcc LJ cell (31 atoms), both relaxed with
    ``fire_relax(structures) -> [(lattice, cart, numbers)]``."""
    lat, cart = _fcc(lj_lattice_constant(), 2)
    cart = cart[1:]                                         # the vacancy at the origin
    j = int(np.argmin(np.linalg.norm(cart - np.array([0.0, 0.5, 0.5]) * lat[0, 0] / 2, axis=1)))
    z = np.full(len(cart), 18)
    final = cart.copy()
    final[j] = 0.0                                          # the neighbour at (0, a/2, a/2) hops into the vacancy
    return fire_relax([(lat, cart, z), (lat, final, z)])


def fire_relax_restated(structs):
    st, ptr = FO.fresh_state(structs, FO.FIRE_DEFAULTS)
    calc = BatchLJ()
    for _ in range(2000):
        out = calc.compute(st["lattice"], st["pos"], np.concatenate([s[2] for s in structs]), np.diff(ptr))
        FO.fire_step(st, out[1].numpy(), None, out[0].double().numpy(), FO.FIRE_DEFAULTS, 1e-4, 2000, 0.0, ptr)
        if (st["status"] != FO.RUNNING).all():
            break
    assert (st["status"] == FO.CONVERGED).all()
    return [(s[0], st["pos"][ptr[b]:ptr[b + 1]].copy(), s[2]) for b, s in enumerate(structs)]


def check_lj_saddle(r):
    p = r["positions"][r["i_climb"]]
    lat = r["lattice"]
    f_true = np.linalg.norm(lj(lat, p)[1], axis=1).max()
    x0, h = p.reshape(-1), 1e-4
    H = np.empty((x0.size, x0.size))
    for k in range(x0.size):
        d = np.zeros_like(x0)
        d[k] = h
        H[:, k] = -(lj(lat, (x0 + d).reshape(-1, 3))[1] - lj(lat, (x0 - d).reshape(-1, 3))[1]).reshape(-1) / (2 * h)
    eig = np.linalg.eigvalsh(0.5 * (H + H.T))
    E = r["energies"]
    print(f"[neb-lj] {r['status']} in {r['n_steps']} steps, climbing image {r['i_climb']}, true max |F| {f_true:.2e}, "
          f"eigenvalues {eig[:5]}, barrier {r['barrier_forward']:.6f} eV, max |E_i - E_(M+1-i)| "
          f"{np.abs(E - E[::-1]).max():.2e}")
    assert r["status"] == "converged"
    assert f_true < 1e-3
    assert (eig < -0.1).sum() == 1 and (np.abs(eig) < 0.05).sum() == 3 and (eig > 0.1).sum() == eig.size - 4
    assert np.abs(E - E[::-1]).max() < 1e-6
    assert r["i_climb"] == (len(E) - 1) // 2


def test_lj_vacancy_hop_saddle(restated):
    ini, fin = lj_vacancy_hop(fire_relax_restated)
    r = restated.BatchNEB(BatchLJ(), [(ini, fin)], n_images=5, climb=True).run(fmax=1e-3, steps=1000)[0]
    check_lj_saddle(r)


# ---------------------------------------------------------------------------------------------------------------------
# host logic
# ---------------------------------------------------------------------------------------------------------------------

def mb_bands():
    """Five Mueller-Brown bands of 3, 9, 1, 5 and 2 interior images (one atom each) between perturbed minima."""
    rng = np.random.default_rng(1)
    out = []
    for m in (3, 9, 1, 5, 2):
        a = np.array(MB_MIN_A) + rng.uniform(-0.05, 0.05, 2)
        b = np.array(MB_MIN_B) + rng.uniform(-0.05, 0.05, 2)
        out.append(([mb_point(*a, rng.uniform(-0.1, 0.1)), mb_point(*b)], m))
    return out


def _mb_run(neb_mod, calc, fmax=2e-2, steps=60, **kw):
    from torch_m3gnet_b200.neb import interpolate

    bands = [interpolate(*ends, m) for ends, m in mb_bands()]
    return neb_mod.BatchNEB(calc, bands, climb=True, **kw).run(fmax=fmax, steps=steps)


def test_host_logic_order_budget_and_endpoints(restated):
    full_calc = BatchMB()
    full = _mb_run(restated, full_calc)
    M = [m for _, m in mb_bands()]
    assert full_calc.calls[0] == (1,) * 10                  # the endpoints, in one chunk
    assert full_calc.calls[1] == (1,) * sum(M)              # every interior image, in input order
    for budget in (4, 6):
        calc = BatchMB()
        opt = restated.BatchNEB(calc, [b for b in _bands_of_mb()], climb=True, max_atoms=budget)
        small = opt.run(fmax=2e-2, steps=60)
        assert opt.n_endpoint_calls == -(-10 // budget)     # endpoint chunks of at most `budget` atoms
        assert calc.calls[:opt.n_endpoint_calls] == [(1,) * min(budget, 10 - c * budget)
                                                    for c in range(opt.n_endpoint_calls)]
        steps = calc.calls[opt.n_endpoint_calls:]
        assert (1,) * 9 in steps                            # the 9-image band, larger than the budget, ran alone
        assert all(len(c) <= budget or (len(c) in M and len(c) > budget) for c in steps) and opt.n_regroups >= 2
        for a, b in zip(full, small):
            _same(a, b)
    statuses = {r["status"] for r in full}
    for r, m in zip(full, M):
        assert r["positions"].shape == (m + 2, 1, 3) and r["energies"].shape == (m + 2,)
        assert 1 <= r["i_climb"] <= m and r["energies"][r["i_climb"]] == r["energies"][1:-1].max()
        assert r["barrier_forward"] == r["energies"].max() - r["energies"][0]
        assert r["barrier_backward"] == r["energies"].max() - r["energies"][-1]
        np.testing.assert_array_equal(r["lattice"], np.eye(3) * MB_CELL)
    print(f"[neb-host] statuses {[r['status'] for r in full]}, steps {[r['n_steps'] for r in full]}")
    assert "converged" in statuses and "not converged" in statuses


def _bands_of_mb():
    from torch_m3gnet_b200.neb import interpolate

    return [interpolate(*ends, m) for ends, m in mb_bands()]


def lj_bands(count=3, seed=2):
    """Bands of 4-atom fcc LJ cells: 3 interior images between two jittered configurations."""
    from torch_m3gnet_b200.neb import interpolate

    rng = np.random.default_rng(seed)
    lat, cart = _fcc(3.65)
    z = np.full(4, 18)
    return [interpolate((lat, cart + rng.uniform(-0.05, 0.05, cart.shape), z),
                        (lat, cart + rng.uniform(-0.05, 0.05, cart.shape), z), 3) for _ in range(count)]


def test_failure_is_isolated(restated):
    bands = lj_bands()
    ref = restated.BatchNEB(BatchLJ(), bands).run(fmax=1e-3, steps=30)
    bad = [list(b) for b in bands]
    lat, cart, z = bad[1][2]
    cart = cart.copy()
    cart[1] = cart[0] + np.array([1e-6, 0.0, 0.0])          # float32 LJ forces overflow in one image
    bad[1][2] = (lat, cart, z)
    got = restated.BatchNEB(BatchLJ(), bad).run(fmax=1e-3, steps=30)
    assert got[1]["status"] == "failed" and got[1]["n_steps"] == 0 and got[1]["fmax"] == np.inf
    for i in (0, 2):
        _same(ref[i], got[i])
    # a band with a non-finite endpoint energy fails before any step, without entering the working set
    far = [mb_point(-2000.0, 0.0), mb_point(*MB_MIN_A), mb_point(*MB_MIN_B)]
    calc = BatchMB()
    res = restated.BatchNEB(calc, [far, _bands_of_mb()[0]]).run(fmax=2e-2, steps=5)
    assert res[0]["status"] == "failed" and res[0]["n_steps"] == 0 and res[0]["i_climb"] == -1
    assert np.isinf(res[0]["energies"][0]) and np.isnan(res[0]["energies"][1])
    assert calc.calls[0] == (1,) * 4 and all(c == (1,) * 3 for c in calc.calls[1:]) and res[1]["n_steps"] == 5
    # a degenerate tangent: two coincident images on a falling triplet
    a, b = mb_point(-0.3, 0.5), mb_point(0.4, 0.1)
    res = restated.BatchNEB(BatchMB(), [[mb_point(*MB_MIN_A), mb_point(-0.3, 0.5), a, b, mb_point(*MB_MIN_B)]]) \
        .run(fmax=1e-3, steps=5)
    assert res[0]["status"] == "failed" and res[0]["n_steps"] == 0


def test_converged_at_step_zero_and_step_limit(restated):
    r = run_mb(restated, BatchMB(), fmax=1e-2)
    again = restated.BatchNEB(BatchMB(), [[(r["lattice"], p, [1]) for p in r["positions"]]], climb=True) \
        .run(fmax=1e-2, steps=10)[0]
    assert again["status"] == "converged" and again["n_steps"] == 0 and again["fmax"] < 1e-2
    capped = restated.BatchNEB(BatchMB(), _bands_of_mb()).run(fmax=1e-9, steps=3)
    assert all(c["status"] == "not converged" and c["n_steps"] == 3 for c in capped)


def test_validation():
    from torch_m3gnet_b200.neb import MAX_IMAGES, BatchNEB

    a, b = mb_point(*MB_MIN_A), mb_point(*MB_MIN_B)
    calc = BatchMB()
    with pytest.raises(ValueError, match="lattice"):
        BatchNEB(calc, [(a, (np.eye(3) * (MB_CELL + 1e-9), b[1], b[2]))], n_images=3)
    with pytest.raises(ValueError, match="atomic numbers"):
        BatchNEB(calc, [(a, (b[0], b[1], [2]))], n_images=3)
    with pytest.raises(ValueError, match="atomic numbers"):
        BatchNEB(calc, [[a, a, (b[0], np.zeros((2, 3)), [1, 1])]])
    with pytest.raises(ValueError, match="n_images"):
        BatchNEB(calc, [(a, b)], n_images=0)
    with pytest.raises(ValueError, match="n_images"):
        BatchNEB(calc, [(a, b)])
    with pytest.raises(ValueError, match="at most"):
        BatchNEB(calc, [(a, b)], n_images=MAX_IMAGES + 1)
    BatchNEB(calc, [(a, b)], n_images=MAX_IMAGES)
    with pytest.raises(ValueError, match="k must"):
        BatchNEB(calc, [(a, b)], n_images=3, k=-0.1)
    with pytest.raises(ValueError, match="one per band"):
        BatchNEB(calc, [(a, b)], n_images=3, k=[0.1, 0.2])
    with pytest.raises(ValueError, match="at least 3"):
        BatchNEB(calc, [[a]])
    with pytest.raises(ValueError, match="max_atoms"):
        BatchNEB(calc, [(a, b)], n_images=3, max_atoms=0)
    assert list(BatchNEB(calc, [(a, b), (b, a)], n_images=2, k=[0.0, 0.5]).k) == [0.0, 0.5]
    assert BatchNEB(calc, []).run() == []


def test_interpolate():
    from torch_m3gnet_b200.neb import interpolate

    lat = np.array([[4.0, 0.0, 0.0], [1.0, 5.0, 0.0], [0.0, 0.5, 6.0]])
    c0 = np.array([[0.2, 0.3, 0.4], [2.0, 2.0, 2.0]])
    c1 = c0 + np.array([[0.4, 0.0, 0.0], [0.0, 0.0, 0.0]]) + np.array([[0.0, 0.0, 0.0], [1.0, 5.0, 0.0]])
    z = np.array([3, 8])
    images = interpolate((lat, c0, z), (lat, c1, z), 3)
    assert len(images) == 5
    np.testing.assert_array_equal(images[0][1], c0)
    np.testing.assert_allclose(images[4][1], c1, atol=1e-15)
    np.testing.assert_allclose(images[2][1], 0.5 * (c0 + c1), atol=1e-15)
    for im in images:
        np.testing.assert_array_equal(im[0], lat)
        np.testing.assert_array_equal(im[2], z)
    # mic: atom 1 moved by a whole lattice vector (b) -- it stays put; atom 0 moves 0.4 A along x
    m = interpolate((lat, c0, z), (lat, c1, z), 3, mic=True)
    np.testing.assert_allclose(m[4][1], c0 + np.array([[0.4, 0.0, 0.0], [0.0, 0.0, 0.0]]), atol=1e-14)
    np.testing.assert_allclose(m[1][1], c0 + np.array([[0.1, 0.0, 0.0], [0.0, 0.0, 0.0]]), atol=1e-14)
    wrapped = c0 + np.array([[-0.3, 0.0, 0.0], [0.0, 0.0, 0.0]]) + lat[0]   # -0.3 A, seen across the cell
    m = interpolate((lat, c0, z), (lat, wrapped, z), 2, mic=True)
    np.testing.assert_allclose(m[3][1] - c0, [[-0.3, 0.0, 0.0], [0.0, 0.0, 0.0]], atol=1e-14)
    with pytest.raises(ValueError, match="n_images"):
        interpolate((lat, c0, z), (lat, c1, z), 0)
