"""GPU: the NPT step (m3g_langevin_npt_step, csrc/md.cu) against its numpy restatement (tests/npt_oracle.py) on random
ragged state, bitwise equality with the fixed-cell run at zero compressibility, batch independence, the exact volume
distribution of an ideal gas and the exact per-axis distribution with a harmonic axis energy, <P_int> = P0 on a
Lennard-Jones crystal for both couplings, BatchMD(pressure=...) on the model against a fresh evaluation, and the launch
count."""
import types

import numpy as np
import pytest
import torch

from tests import md_oracle as MO
from tests import npt_oracle as NO
from tests.test_batch_fire_cpu import BatchLJ, lj_structures
from tests.test_batch_md_cpu import AR
from tests.test_batch_npt_cpu import _axis_quadrature, block_mean
from tests.test_gpu_batch_md import MD_SIZES, _cu_masses, _random_case

pytestmark = pytest.mark.gpu

SIGMA_NAN, STRAIN = 1, 7          # structures of the random case that fail on a NaN stress and on the strain guard


def _to_device(st, ptr, device):
    ns = types.SimpleNamespace(**{k: torch.as_tensor(np.ascontiguousarray(v)).to(device) for k, v in st.items()})
    ns.atom_ptr = torch.as_tensor(ptr.astype(np.int32)).to(device)
    ns.B = len(ptr) - 1
    return ns


def _random_npt_case(seed=0):
    """test_gpu_batch_md's random ragged case (failures at 5, 6, 8, 9) plus random cells, stresses and barostat
    parameters; structure 1 gets a NaN stress and structure 7 a compressibility that breaks the strain guard."""
    st, ptr, forces, energy = _random_case(MD_SIZES, seed)
    rng = np.random.default_rng(seed + 100)
    B = len(MD_SIZES)
    st["lattice"] = np.eye(3)[None] * rng.uniform(18, 24, (B, 1, 1)) + rng.uniform(-1, 1, (B, 3, 3))
    st["P0"] = rng.uniform(-0.01, 0.01, B)
    st["beta_T"] = rng.uniform(0.5, 5.0, B)
    st["tau_p"] = rng.uniform(200.0, 2000.0, B)
    st["beta_T"][STRAIN] = 1e7
    sigma = rng.normal(0, 0.01, (B, 3, 3)).astype(np.float32)
    sigma[SIGMA_NAN, 2, 0] = np.nan
    return st, ptr, forces, sigma, energy


@pytest.mark.parametrize("coupling", [NO.ISOTROPIC, NO.PER_AXIS])
@pytest.mark.parametrize("advance,slot", [(True, 2), (True, -1), (False, 0)])
def test_npt_kernel_matches_the_restatement(device, coupling, advance, slot):
    from torch_m3gnet_b200 import md

    st, ptr, forces, sigma, energy = _random_npt_case()
    B, W = len(MD_SIZES), NO.obs_width(coupling)
    seed = (1 << 63) + 777
    sw = seed - (1 << 64)
    want = {k: v.copy() for k, v in st.items()}
    obs_want = np.full((3, B, W), np.nan)
    NO.npt_step(want, forces, sigma, energy.astype(np.float64), ptr, 2.0, 0.5, seed, advance, slot, obs_want, coupling,
                0.02)
    outs = []
    for _ in range(2):
        d = _to_device(st, ptr, device)
        obs = torch.full((3, B, W), float("nan"), dtype=torch.float64, device=device)
        md.langevin_npt_step(d, torch.as_tensor(forces).to(device), torch.as_tensor(sigma).to(device),
                             torch.as_tensor(energy).to(device), 2.0, 0.5, sw, advance, slot, obs, coupling, 0.02)
        torch.cuda.synchronize()
        outs.append(({k: getattr(d, k).cpu().numpy() for k in st}, obs.cpu().numpy()))
    (got, obs_got), (again, obs_again) = outs
    for k in st:
        assert np.array_equal(got[k], again[k]), k                 # repeated calls are bitwise equal
    assert np.array_equal(obs_got, obs_again, equal_nan=True)
    failed = [SIGMA_NAN, 5, 6, STRAIN, 8, 9]
    assert np.array_equal(got["status"], want["status"]) and np.array_equal(got["step"], want["step"])
    assert want["status"][failed].tolist() == [MO.FAILED] * 6 and (np.delete(want["status"], failed) == 0).all()
    for k in ("pos", "v", "bath", "lattice"):
        scale = np.abs(want[k]).max()
        np.testing.assert_allclose(got[k], want[k], rtol=1e-12, atol=1e-12 * scale, err_msg=k)
    np.testing.assert_allclose(obs_got, obs_want, rtol=1e-12, atol=1e-15, equal_nan=True)
    for b in failed:                                                # failed: bit-untouched, nothing recorded
        s, t = ptr[b], ptr[b + 1]
        for k in ("pos", "v"):
            assert np.array_equal(got[k][s:t], st[k][s:t]), (b, k)
        assert np.array_equal(got["lattice"][b], st["lattice"][b]) and got["bath"][b] == st["bath"][b]
        assert np.isnan(obs_got[:, b]).all()
    run = np.delete(np.arange(B), failed)
    assert (np.abs(got["lattice"][run] - st["lattice"][run]).max(axis=(1, 2)) > 0).all() == advance
    if slot >= 0:
        assert np.isfinite(obs_got[slot, run]).all()


def test_zero_compressibility_is_the_fixed_cell_run(device):
    """beta_T = 0 makes mu exactly 1: BatchMD(pressure=...) then reproduces BatchMD(pressure=None) bit for bit on a
    calculator whose forces do not depend on with_stress.  (The public argument must be positive, so the test sets
    the stored per-structure values to zero after construction.)"""
    from torch_m3gnet_b200 import BatchMD

    structs = lj_structures(6, seed=30)
    kw = dict(masses={18: AR}, temperature=[60.0 + 30 * i for i in range(6)], friction=0.02, dt=2.0, seed=8)
    ref = BatchMD(BatchLJ(device), structs, **kw).run(60, record_every=5, trajectory_every=20)
    md = BatchMD(BatchLJ(device), structs, pressure=[0.0, 0.01, -0.02, 0.0, 0.005, 0.1], **kw)
    md.compressibility[:] = 0.0
    got = md.run(60, record_every=5, trajectory_every=20)
    for i, s in enumerate(structs):
        assert got[i]["status"] == "completed"
        for k in ref[i]:
            assert np.array_equal(np.asarray(ref[i][k]), np.asarray(got[i][k])), (i, k)
        assert np.array_equal(got[i]["lattice"], s[0]) and (got[i]["lattice_trajectory"] == s[0]).all()


def test_npt_structure_steps_the_same_anywhere_in_the_batch(device):
    from torch_m3gnet_b200 import BatchMD

    structs = lj_structures(7, seed=31)
    kw = dict(masses={18: AR}, temperature=[60.0 + 30 * i for i in range(7)], friction=0.02, dt=2.0, seed=5,
              pressure=[0.001 * i for i in range(7)], barostat_time=500.0, coupling="per_axis")
    full = BatchMD(BatchLJ(device), structs, **kw).run(40, record_every=10, trajectory_every=20)
    for max_atoms in (40, 3):
        other = BatchMD(BatchLJ(device), structs, max_atoms=max_atoms, **kw).run(40, record_every=10,
                                                                                 trajectory_every=20)
        for i in range(len(structs)):
            assert full[i]["status"] == "completed"
            for k in full[i]:
                assert np.array_equal(np.asarray(full[i][k]), np.asarray(other[i][k])), (max_atoms, i, k)


class ZeroCalc:
    """No interactions: zero energy, forces and stress (an ideal gas), or the harmonic axis energy
    E = sum_a kappa / 2 (L_a - L0)^2 of diagonal cells with sigma_aa = kappa (L_a - L0) L_a / V."""

    def __init__(self, device, harmonic=None):
        self.device, self.harmonic = device, harmonic

    def compute(self, lattices, cart, atomic_numbers, sizes=None, with_stress=False):
        B = len(sizes)
        lat = torch.as_tensor(np.asarray(lattices, dtype=np.float64).reshape(B, 3, 3), device=self.device)
        e = torch.zeros(B, dtype=torch.float64, device=self.device)
        sigma = torch.zeros((B, 3, 3), dtype=torch.float64, device=self.device)
        if self.harmonic is not None:
            kappa, L0 = self.harmonic
            diag = torch.diagonal(lat, dim1=1, dim2=2)
            vol = torch.linalg.det(lat).abs()
            e = 0.5 * kappa * ((diag - L0) ** 2).sum(dim=1)
            sigma = torch.diag_embed(kappa * (diag - L0) * diag / vol[:, None])
        out = (e.float(), torch.zeros_like(cart, dtype=torch.float32), torch.zeros((B, 6), device=self.device))
        return out + (sigma.float(),) if with_stress else out


def test_ideal_gas_volume_on_the_device(device):
    """512 ideal-gas structures of 8 atoms (some 4 and 16) at two temperatures and two pressures, isotropic, tau_p =
    100 dt, beta_T P0 = 1: <V> = n kT / P0 per group and var V = n (kT / P0)^2 (pooled in those units)."""
    from torch_m3gnet_b200 import BatchMD

    S = 512
    rng = np.random.default_rng(5)
    n = np.where(np.arange(S) % 16 == 3, 4, np.where(np.arange(S) % 16 == 7, 16, 8))
    grp = np.arange(S) % 4
    T = np.array([300.0, 600.0, 300.0, 600.0])[grp]
    P0 = np.array([0.002, 0.002, 0.006, 0.006])[grp]
    V0 = n * MO.KB * T / P0
    structs = [(np.eye(3) * V0[s] ** (1 / 3), rng.uniform(0, 4, (n[s], 3)), np.full(n[s], 6)) for s in range(S)]
    steps, every, burn = 50000, 5, 5000
    res = BatchMD(ZeroCalc(device), structs, {6: 12.0}, T, friction=0.05, dt=1.0, seed=41, pressure=P0,
                  compressibility=1.0 / P0, barostat_time=100.0, max_step_strain=10.0).run(steps, record_every=every)
    assert all(r["status"] == "completed" for r in res)
    x = np.stack([r["volume"][burn // every:] for r in res], axis=1) / V0          # (frames, S)
    for g in range(4):
        mean, se = block_mean(x[:, grp == g].mean(axis=1))
        print(f"[npt-gpu] ideal gas T={T[g]:.0f} K P0={P0[g]}: <V> / (n kT/P0) = {mean:.4f} +- {se:.4f}")
        assert abs(mean - 1) < 4 * se and abs(mean - 1) < 0.01
    var, var_se = block_mean((((x - 1.0) ** 2) * n).mean(axis=1))
    print(f"[npt-gpu] ideal gas var V / (n (kT/P0)^2) = {var:.4f} +- {var_se:.4f}")
    assert abs(var - 1) < 4 * var_se and abs(var - 1) < 0.015
    # per axis on the same kernel: the harmonic axis energy against the 3-D quadrature (test_batch_npt_cpu's units)
    kT = MO.KB * 300.0
    Pa, kappa, L0 = kT / 8.0, kT, 4.0
    cells = [(np.eye(3) * L0, rng.uniform(0, 4, (8, 3)), np.full(8, 6)) for _ in range(256)]
    res = BatchMD(ZeroCalc(device, (kappa, L0)), cells, {6: 12.0}, 300.0, friction=0.05, dt=1.0, seed=42,
                  pressure=Pa, compressibility=0.5 / Pa, barostat_time=100.0, coupling="per_axis",
                  max_step_strain=10.0).run(30000, record_every=every, trajectory_every=every)
    want_l, want_v, want_var = _axis_quadrature(8, kT, Pa, kappa, L0, 0.05 * L0, 3.0 * L0)
    lt = np.stack([r["lattice_trajectory"][burn // every:] for r in res], axis=1)      # (frames, S, 3, 3)
    vol = np.stack([r["volume"][burn // every:] for r in res], axis=1)
    mean_l, se_l = block_mean(np.diagonal(lt, axis1=2, axis2=3).mean(axis=(1, 2)))
    mean_v, se_v = block_mean(vol.mean(axis=1))
    var_v, _ = block_mean(((vol - want_v) ** 2).mean(axis=1))
    print(f"[npt-gpu] per axis: <L_a> {mean_l:.4f} +- {se_l:.4f} (exact {want_l:.4f}), <V> {mean_v:.3f} +- {se_v:.3f} "
          f"(exact {want_v:.3f}), var V {var_v:.3f} (exact {want_var:.3f})")
    assert abs(mean_l - want_l) < 4 * se_l and abs(mean_l / want_l - 1) < 0.005
    assert abs(mean_v - want_v) < 4 * se_v and abs(mean_v / want_v - 1) < 0.005
    assert abs(var_v / want_var - 1) < 0.02
    assert np.abs(lt - np.eye(3) * np.diagonal(lt, axis1=2, axis2=3)[..., None, :]).max() == 0.0   # never sheared


class TorchLJ:
    """Periodic Lennard-Jones (test_cell_stress_cpu's lj: eps 0.4 eV, sigma 2.3 A, truncated and shifted at 5 A) for
    equal-size structures on the device in float64, minimum image plus the 26 neighbouring images (plane spacings must
    exceed the cutoff): energy, forces and the bond-form stress (1/V) sum v (x) dE/dv."""

    def __init__(self, device):
        from tests.test_cell_stress_cpu import LJ_EPS, LJ_RC, LJ_SIG

        self.device, self.eps, self.sig, self.rc = device, LJ_EPS, LJ_SIG, LJ_RC
        g = torch.arange(-1, 2, dtype=torch.float64)
        self.imgs = torch.stack(torch.meshgrid(g, g, g, indexing="ij"), dim=-1).reshape(-1, 3).to(device)

    def _phi(self, r):
        sr6 = (self.sig / r) ** 6
        return 4 * self.eps * (sr6 * sr6 - sr6), 4 * self.eps * (-12 * sr6 * sr6 + 6 * sr6) / r

    def compute(self, lattices, cart, atomic_numbers, sizes=None, with_stress=False):
        B = len(sizes)
        n = int(sizes[0])
        lat = torch.as_tensor(np.asarray(lattices, dtype=np.float64).reshape(B, 3, 3), device=self.device)
        x = cart.reshape(B, n, 3)
        frac = x @ torch.linalg.inv(lat)
        d = frac[:, None, :, :] - frac[:, :, None, :]                      # (B, i, j, 3): r_j - r_i
        d = d - torch.round(d)
        v = (d[:, :, :, None, :] + self.imgs[None, None, None]) @ lat[:, None, None]   # (B, i, j, 27, 3)
        r = v.norm(dim=-1)
        mask = (r > 1e-9) & (r < self.rc)
        rr = torch.where(mask, r, torch.ones_like(r))
        phi, dphi = self._phi(rr)
        shift, _ = self._phi(torch.tensor(self.rc, dtype=torch.float64))
        phi = torch.where(mask, phi - shift, torch.zeros_like(phi))
        dphi = torch.where(mask, dphi, torch.zeros_like(dphi))
        energy = 0.5 * phi.sum(dim=(1, 2, 3))
        g = 0.5 * (dphi / rr)[..., None] * v
        forces = g.sum(dim=(2, 3)) - g.sum(dim=(1, 3))
        vol = torch.linalg.det(lat).abs()
        stress = torch.einsum("bijka,bijkc->bac", v, g) / vol[:, None, None]
        out = (energy.float(), forces.reshape(-1, 3).float(), torch.zeros((B, 6), device=self.device))
        return out + (stress.float(),) if with_stress else out


def _lj_crystals(count, seed):
    """32-atom fcc LJ cells: even indices cubic, odd ones strained 3 % along z; small jitter."""
    from tests.test_cell_stress_cpu import _fcc

    rng = np.random.default_rng(seed)
    out = []
    for s in range(count):
        lat, cart = _fcc(3.62, 2)
        strain = np.diag([1.0, 1.0, 1.03 if s % 2 else 1.0])
        out.append((lat @ strain, cart @ strain + rng.uniform(-0.02, 0.02, cart.shape), np.full(32, 18)))
    return out


@pytest.mark.parametrize("coupling", ["isotropic", "per_axis"])
def test_lj_mean_pressure_is_exact(device, coupling):
    """At stationarity E[d eps] = 0, so <P_int> = P0 exactly at any dt (per axis <P_a> = P0).  Under per_axis the 3 %
    tetragonal cells become cubic on average; under isotropic they keep their c/a ratio to rounding."""
    from torch_m3gnet_b200 import BatchMD

    S, steps, burn = 64, 4000, 1000
    structs = _lj_crystals(S, seed=7)
    P0 = np.where(np.arange(S) % 4 < 2, 0.0, -0.02)
    res = BatchMD(TorchLJ(device), structs, {18: AR}, 100.0, friction=0.02, dt=2.0, seed=50, pressure=P0,
                  barostat_time=200.0, coupling=coupling).run(steps, record_every=1, trajectory_every=10)
    assert all(r["status"] == "completed" for r in res)
    for p0 in (0.0, -0.02):
        grp = [s for s in range(S) if P0[s] == p0]
        pint = np.stack([res[s]["pressure"][burn:] for s in grp], axis=1).mean(axis=1)
        mean, se = block_mean(pint)
        print(f"[npt-lj] {coupling} P0={p0}: <P_int> = {mean:.6f} +- {se:.6f} eV/A^3")
        assert abs(mean - p0) < 4 * se and se < 2e-3
        if coupling == "per_axis":
            pa = np.stack([res[s]["axis_pressure"][burn:] for s in grp], axis=1).mean(axis=1)
            m3, se3 = block_mean(pa)
            print(f"[npt-lj]   <P_a> = {m3} +- {se3}")
            assert (np.abs(m3 - p0) < 4 * se3).all()
    strained = [s for s in range(S) if s % 2]
    diag = np.stack([np.diagonal(res[s]["lattice_trajectory"][burn // 10:], axis1=1, axis2=2) for s in strained],
                    axis=1)
    if coupling == "per_axis":
        d_xz, se_xz = block_mean(diag[..., 2].mean(axis=1) - diag[..., 0].mean(axis=1))
        d_xy, se_xy = block_mean(diag[..., 1].mean(axis=1) - diag[..., 0].mean(axis=1))
        print(f"[npt-lj] per axis strained cells: <L_z - L_x> = {d_xz:.5f} +- {se_xz:.5f} A, "
              f"<L_y - L_x> = {d_xy:.5f} +- {se_xy:.5f} A (started at {0.03 * structs[1][0][0, 0]:.3f})")
        assert abs(d_xz) < 4 * se_xz and abs(d_xy) < 4 * se_xy
    else:
        for s in strained + [0]:
            L, L0 = res[s]["lattice"], structs[s][0]
            assert L[2, 2] / L[0, 0] == pytest.approx(L0[2, 2] / L0[0, 0], rel=1e-12)
            assert L[1, 1] / L[0, 0] == pytest.approx(L0[1, 1] / L0[0, 0], rel=1e-12)
            assert np.abs(L - np.diag(np.diag(L))).max() == 0.0


def test_model_npt_batch(device):
    """Ragged Cu and multi-species cells at 300 K on the c1_default x3 model, 200 NPT steps: every structure completes
    with finite state, the last frame's energy, forces and stress equal a fresh Batch.from_arrays evaluation at the
    returned positions and lattice, and its recorded V and P_int are |det L| and 2 K / (3 V) - tr(sigma) / 3."""
    from tests.util import golden, state_dict_of
    from torch_m3gnet_b200 import Batch, BatchMD, M3GNetCalculator, build_model, synthetic
    from torch_m3gnet_b200.data import MaterialGraphKey as K

    model = build_model(5.0, 4.0, 3, 3, 95, 64, 3, device=device)
    model.load_state_dict({k: (v * 3 if k.endswith("weight") else v)
                           for k, v in state_dict_of(golden("c1_default")).items()})
    structs = [synthetic.mpf_like_structure(s) for s in range(4)] + [synthetic.fcc_cu_supercell(2, 0.05, s)
                                                                    for s in range(4)]
    sizes = [len(s[2]) for s in structs]
    calc = M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device)
    last = {}
    compute = calc.compute

    def keep_last(*a, **k):
        out = compute(*a, **k)
        last["forces"], last["stress"] = out[1].clone(), out[3].clone()
        return out

    calc.compute = keep_last
    steps = 200
    res = BatchMD(calc, structs, _cu_masses(structs), 300.0, friction=0.01, dt=1.0, seed=19, pressure=0.0,
                  barostat_time=200.0).run(steps, record_every=10)
    lat = np.stack([r["lattice"] for r in res])
    model.compute_stress = True
    try:
        fresh = model(Batch.from_arrays(lat, np.concatenate([r["positions"] for r in res]),
                                        np.concatenate([s[2] for s in structs]), sizes, 5.0, 4.0, device=device))
    finally:
        model.compute_stress = False
    assert torch.equal(fresh["forces"], last["forces"])
    assert torch.equal(fresh[K.CELL_STRESS].reshape(-1, 3, 3), last["stress"].reshape(-1, 3, 3))
    sig = fresh[K.CELL_STRESS].reshape(-1, 3, 3).double().cpu().numpy()
    for i, r in enumerate(res):
        assert r["status"] == "completed" and r["n_steps"] == steps
        assert np.isfinite(r["positions"]).all() and np.isfinite(r["velocities"]).all() and np.isfinite(lat[i]).all()
        assert r["energy"][-1] == float(fresh["total_energy"][i])
        V = abs(np.linalg.det(lat[i]))
        assert r["volume"][-1] == pytest.approx(V, rel=1e-12)
        assert r["pressure"][-1] == pytest.approx(2 * r["kinetic_energy"][-1] / (3 * V) - np.trace(sig[i]) / 3,
                                                  rel=1e-10, abs=1e-12)
        print(f"[npt-model] structure {i} ({sizes[i]} atoms): V {r['volume'][0]:.2f} -> {r['volume'][-1]:.2f} A^3, "
              f"P_int {r['pressure'][-1]:.5f} eV/A^3")


def test_npt_launch_count(device):
    from tests.test_gpu_batch_fire import _verlet_model
    from torch_m3gnet_b200 import BatchMD, M3GNetCalculator, _lib, synthetic

    model = _verlet_model(device)
    calc = M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device)
    inner = []
    compute = calc.compute

    def counted(*a, **k):
        before = _lib.LAUNCHES
        out = compute(*a, **k)
        inner.append(_lib.LAUNCHES - before)
        return out

    calc.compute = counted
    structs = [synthetic.fcc_cu_supercell(2, 0.05, s) for s in range(4)]
    for velocities in (None, [np.zeros((32, 3))] * 4):
        inner.clear()
        md = BatchMD(calc, structs, {29: 63.546}, 300.0, velocities=velocities, pressure=0.0)
        before = _lib.LAUNCHES
        md.run(3)
        assert md.n_iterations == len(inner) == 4
        assert _lib.LAUNCHES - before == sum(inner) + md.n_iterations + (velocities is None)
