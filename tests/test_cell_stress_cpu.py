"""CPU: the cell stress sigma = (1/V) dE/d(strain) of the oracle (definition, finite differences, bond form, invariance)
and the variable-cell FIRE on ASE UnitCellFilter coordinates, driven by a periodic Lennard-Jones calculator on the CPU."""
import numpy as np
import pytest
import torch
from scipy.optimize import minimize_scalar

from oracle import m3gnet_oracle as O
from tests import strain_oracle as S
from tests.util import golden, graph_dict, state_dict_of


def _case(name):
    g = golden(name)
    if name == "small_batch":
        rc = float(g["cutoff"])
        hp = O.HyperParams(cutoff=rc, threebody_cutoff=rc, l_max=2, n_max=3, num_types=93, embedding_dim=17,
                           num_blocks=2)
        sd = {k: (v * 2 if k.endswith("weight") else v) for k, v in state_dict_of(g).items()}
        return graph_dict(g), sd, hp, torch.from_numpy(g["factors"])
    c1 = golden("c1_default")
    sd = {k: (v * 3 if k.endswith("weight") else v) for k, v in state_dict_of(c1).items()}
    return graph_dict(g), sd, O.HyperParams(), torch.from_numpy(c1["factors"])


@pytest.mark.parametrize("name", ["c1_default", "tio2_default", "small_batch"])
def test_oracle_cell_stress_is_the_strain_derivative(name):
    """Autograd strain derivative == central differences of the energy under +-1e-3 strain == bond form."""
    torch.set_num_threads(4)
    gd, sd, hp, fac = _case(name)
    sigma = S.cell_stress(sd, hp, gd, fac)
    B = sigma.shape[0]
    vol = S.volumes(gd["lattice"])
    h = 1e-3
    fd = torch.zeros_like(sigma)
    for a in range(3):
        for c in range(3):
            eps = torch.zeros((B, 3, 3))
            eps[:, a, c] = h
            ep = S.energy(sd, hp, S.strained(gd, eps), fac)
            em = S.energy(sd, hp, S.strained(gd, -eps), fac)
            fd[:, a, c] = (ep - em) / (2 * h) / vol
    scale = sigma.abs().max().item()
    err = (fd - sigma).abs().max().item()
    print(f"[stress] {name}: max|sigma|={scale:.3e} eV/A^3, max|fd - sigma|={err:.3e}")
    assert scale > 1e-5
    assert err <= 1e-5 + 1e-2 * scale
    bond = S.bond_form(sd, hp, gd, fac)
    assert (bond - sigma).abs().max().item() <= 1e-7 + 1e-4 * scale
    # symmetric (rotation invariance of E) to float32 rounding
    assert (sigma - sigma.transpose(1, 2)).abs().max().item() <= 1e-3 * scale


def _shifted_copy(gd, atom, image, shift):
    """The same periodic structure with every atom translated by ``shift`` and ``atom`` replaced by its periodic image
    ``image`` (integer lattice vector); the bond image shifts are rewritten so that every bond vector is unchanged."""
    moved = dict(gd)
    lat = gd["lattice"].reshape(-1, 3, 3)[0]
    img = torch.tensor(image)
    pos = gd["pos"] + torch.tensor(shift)
    pos[atom] += img.to(pos.dtype) @ lat
    moved["pos"] = pos
    sh = gd["edge_cell_shift"].clone()
    src, dst = gd["edge_index"][0], gd["edge_index"][1]
    sh[src == atom] += img.to(sh.dtype)
    sh[dst == atom] -= img.to(sh.dtype)
    moved["edge_cell_shift"] = sh
    return moved


def test_oracle_cell_stress_is_translation_invariant_unlike_stresses():
    """sigma depends on bond vectors only; the reference's sum_i pos_i (x) F_i / V changes when an atom is replaced by
    one of its periodic images (the same crystal described from another origin)."""
    torch.set_num_threads(4)
    gd, sd, hp, fac = _case("c1_default")
    moved = _shifted_copy(gd, 0, [1, -1, 0], [1.7, -2.3, 0.9])
    e0, e1 = S.energy(sd, hp, gd, fac), S.energy(sd, hp, moved, fac)
    assert abs(float(e1 - e0)) <= 1e-5 * abs(float(e0))
    s0, s1 = S.cell_stress(sd, hp, gd, fac), S.cell_stress(sd, hp, moved, fac)
    r0, r1 = S.reference_stresses(sd, hp, gd, fac), S.reference_stresses(sd, hp, moved, fac)
    scale = s0.abs().max().item()
    print(f"[stress] translated: |d sigma|={(s1 - s0).abs().max().item():.2e}, "
          f"|d stresses|={(r1 - r0).abs().max().item():.2e}, max|sigma|={scale:.2e}")
    assert (s1 - s0).abs().max().item() <= 1e-3 * scale
    assert (r1 - r0).abs().max().item() > 100 * (s1 - s0).abs().max().item()
    # and it is not the reference's row (Voigt xx, yy, zz, yz, zx, xy)
    voigt = torch.stack([s0[:, 0, 0], s0[:, 1, 1], s0[:, 2, 2], s0[:, 1, 2], s0[:, 2, 0], s0[:, 0, 1]], dim=1)
    assert (voigt - r0).abs().max().item() > 0.1 * scale


# ---------------------------------------------------------------------------------------------------------------------
# Variable-cell FIRE on a periodic Lennard-Jones solid (host logic only: the calculator below runs on the CPU)
# ---------------------------------------------------------------------------------------------------------------------

LJ_EPS, LJ_SIG, LJ_RC = 0.4, 2.3, 5.0


def _lj_phi(r):
    sr6 = (LJ_SIG / r) ** 6
    return 4 * LJ_EPS * (sr6 * sr6 - sr6), 4 * LJ_EPS * (-12 * sr6 * sr6 + 6 * sr6) / r


def lj(lattice, cart):
    """Energy (truncated and shifted at LJ_RC), forces and the bond-form stress (1/V) sum v (x) dE/dv."""
    lattice = np.asarray(lattice, dtype=np.float64).reshape(3, 3)
    cart = np.asarray(cart, dtype=np.float64)
    inv_w = np.linalg.norm(np.linalg.inv(lattice), axis=0)  # 1 / plane spacings
    n_img = np.ceil(LJ_RC * inv_w).astype(int)
    rng = [np.arange(-k, k + 1) for k in n_img]
    imgs = np.stack(np.meshgrid(*rng, indexing="ij"), axis=-1).reshape(-1, 3) @ lattice
    v = cart[None, :, None, :] + imgs[None, None, :, :] - cart[:, None, None, :]  # (i, j, image, 3): r_j + s - r_i
    r = np.linalg.norm(v, axis=-1)
    mask = (r > 1e-9) & (r < LJ_RC)
    rr = np.where(mask, r, 1.0)
    phi, dphi = _lj_phi(rr)
    shift, _ = _lj_phi(LJ_RC)
    phi = np.where(mask, phi - shift, 0.0)
    dphi = np.where(mask, dphi, 0.0)
    energy = 0.5 * phi.sum()
    g = 0.5 * (dphi / rr)[..., None] * v  # dE/dv of every ordered pair (each pair appears twice)
    forces = g.sum(axis=(1, 2)) - g.sum(axis=(0, 2))  # F_i = -dE/dr_i = sum_j g_ij - sum_j g_ji
    vol = abs(np.linalg.det(lattice))
    stress = np.einsum("ijka,ijkc->ac", v, g) / vol
    return energy, forces, stress


class LJCalculator:
    """The ``compute`` protocol of M3GNetCalculator on the CPU (float64 tensors)."""

    device = torch.device("cpu")

    def __init__(self):
        self.calls = 0

    def compute(self, lattices, cart, atomic_numbers, sizes=None, with_stress=False):
        self.calls += 1
        cart = cart.cpu().numpy() if torch.is_tensor(cart) else np.asarray(cart)
        e, f, s = lj(np.asarray(lattices).reshape(3, 3), cart)
        out = (torch.tensor([e], dtype=torch.float64), torch.from_numpy(f), torch.zeros((1, 6), dtype=torch.float64))
        return out + (torch.from_numpy(s)[None],) if with_stress else out


def _fcc(a, reps=1):
    base = np.array([[0, 0, 0], [0, 0.5, 0.5], [0.5, 0, 0.5], [0.5, 0.5, 0]])
    cells = np.stack(np.meshgrid(*[np.arange(reps)] * 3, indexing="ij"), axis=-1).reshape(-1, 3)
    frac = (cells[:, None, :] + base[None]).reshape(-1, 3) / reps
    lat = np.eye(3) * a * reps
    return lat, frac @ lat


def test_lj_stress_is_the_strain_derivative():
    rng = np.random.default_rng(0)
    lat, cart = _fcc(3.6)
    lat = lat @ (np.eye(3) + rng.uniform(-0.03, 0.03, (3, 3)))
    cart = cart + rng.uniform(-0.05, 0.05, cart.shape)
    _, f, s = lj(lat, cart)
    h, vol = 1e-5, abs(np.linalg.det(lat))
    for a in range(3):
        for c in range(3):
            eps = np.zeros((3, 3))
            eps[a, c] = h
            ep = lj(lat @ (np.eye(3) + eps), cart @ (np.eye(3) + eps))[0]
            em = lj(lat @ (np.eye(3) - eps), cart @ (np.eye(3) - eps))[0]
            assert abs((ep - em) / (2 * h) / vol - s[a, c]) < 1e-6 * max(abs(s).max(), 1e-3)
    k = 1
    dp = np.zeros_like(cart)
    dp[k, 2] = h
    fd = (lj(lat, cart + dp)[0] - lj(lat, cart - dp)[0]) / (2 * h)
    assert abs(-fd - f[k, 2]) < 1e-6


def test_generalised_forces_are_minus_the_gradient_of_enthalpy():
    """UnitCellFilter coordinates: -d(E + pV)/d(generalised positions) == the forces Fire relaxes along."""
    from torch_m3gnet_b200.calculator import Fire

    rng = np.random.default_rng(1)
    lat, cart = _fcc(3.6)
    cart = cart + rng.uniform(-0.05, 0.05, cart.shape)
    p = 0.01
    opt = Fire(LJCalculator(), lat, cart, np.full(len(cart), 18), relax_cell=True, pressure=p)
    assert opt.vel.device.type == "cpu" and opt.gen_forces.shape == (len(cart) + 3, 3)
    # move away from D = I so that the cell part of the map is exercised
    x0 = opt._x.clone()
    x0[len(cart):] += torch.from_numpy(rng.uniform(-0.05, 0.05, (3, 3))) * opt.cell_factor
    opt._set_generalised(x0)
    opt._evaluate()
    gen = opt.gen_forces.numpy()

    def enthalpy(x):
        probe = Fire.__new__(Fire)
        probe.__dict__.update(opt.__dict__)
        probe._set_generalised(torch.from_numpy(x))
        e, _, _ = lj(probe.lattice[0], probe.pos.numpy())
        return e + p * abs(np.linalg.det(probe.lattice[0]))

    x = x0.numpy()
    h = 1e-6
    worst = 0.0
    for i in range(x.shape[0]):
        for c in range(3):
            d = np.zeros_like(x)
            d[i, c] = h
            fd = -(enthalpy(x + d) - enthalpy(x - d)) / (2 * h)
            worst = max(worst, abs(fd - gen[i, c]))
    print(f"[ucf] max |generalised force + d(E+pV)/dx| = {worst:.2e}, max |f| = {np.abs(gen).max():.2e}")
    assert worst < 1e-5 * max(np.abs(gen).max(), 1.0)


def test_variable_cell_fire_reaches_the_lj_lattice_constant():
    from torch_m3gnet_b200.calculator import Fire

    _, c1 = _fcc(1.0)
    res = minimize_scalar(lambda a: lj(np.eye(3) * a, c1 * a)[0], bounds=(3.0, 4.5), method="bounded",
                          options=dict(xatol=1e-10))
    a_star = res.x
    lat, cart = _fcc(3.7)
    lat = lat @ np.diag([1.03, 1.0, 0.98])       # tetragonal start
    cart = cart @ np.diag([1.03, 1.0, 0.98])
    calc = LJCalculator()
    opt = Fire(calc, lat, cart, np.full(len(cart), 18), relax_cell=True)
    done = opt.run(fmax=1e-4, steps=2000)
    L = opt.lattice[0]
    print(f"[ucf] a* = {a_star:.6f} A, relaxed cell diag {np.diag(L)}, {opt.n_steps} steps, fmax {opt.fmax():.2e}")
    assert done
    np.testing.assert_allclose(np.diag(L), a_star, rtol=1e-4)
    assert np.abs(L - np.diag(np.diag(L))).max() < 1e-4 * a_star
    # atoms still on their fcc sites of the relaxed cell
    frac = opt.pos.numpy() @ np.linalg.inv(L)
    base = np.array([[0, 0, 0], [0, 0.5, 0.5], [0.5, 0, 0.5], [0.5, 0.5, 0]])
    d = (frac - frac[0]) - base
    assert np.abs(d - np.round(d)).max() < 1e-4
