"""GPU: the batched Langevin kernels (m3g_langevin_step, m3g_md_maxwell_boltzmann, csrc/md.cu) against their numpy
restatement (tests/md_oracle.py), the device Philox4x64-10 against numpy.random.Philox, batch independence, exact
configurational sampling of a harmonic (Einstein) crystal, BatchMD on the model against VelocityVerlet, and the launch
count."""
import types

import numpy as np
import pytest
import torch

from tests import md_oracle as MO
from tests.test_batch_fire_cpu import BatchLJ, lj_structures
from tests.test_batch_md_cpu import AR, M64, _counter_plus_one, _zero_momentum_velocities
from tests.test_gpu_batch_fire import SIZES, _verlet_model

pytestmark = pytest.mark.gpu

MD_SIZES = [s if s > 1 else 9 for s in SIZES]   # no single-atom structure: [9, 2, 32, 700, 5, 3, 4, 6, 8, 12, 257]


def _i64(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64))


def test_philox_words_match_numpy(device):
    from torch_m3gnet_b200 import _lib

    rng = np.random.default_rng(1)
    ctrs, keys, want = [], [], []
    for t in range(256):
        c = rng.integers(0, M64, 4, dtype=np.uint64)
        k = rng.integers(0, M64, 2, dtype=np.uint64)
        if t % 3 == 0:
            c[0] = np.uint64(M64 - 1 - t % 5)           # counter words near 2^64 (the increment carries)
        if t % 11 == 0:
            c[:3] = np.uint64(M64 - 1)
        if t % 7 == 0:
            k[:] = np.uint64(M64 - 1 - t)
        want.append(np.random.Philox(counter=c, key=k).random_raw(4))
        ctrs.append(_counter_plus_one(c))               # numpy increments its counter before it generates
        keys.append(k)
    ctr, key = _i64(np.stack(ctrs)).to(device), _i64(np.stack(keys)).to(device)
    out = torch.empty((256, 4), dtype=torch.int64, device=device)
    _lib.call("debug_philox4x64", ctr, key, 256, out)
    got = out.cpu().numpy().view(np.uint64)
    assert np.array_equal(got, np.stack(want))
    zero = torch.zeros((1, 4), dtype=torch.int64, device=device)
    _lib.call("debug_philox4x64", zero, zero[:, :2].contiguous(), 1, out)
    assert [int(w) for w in out[0].cpu().numpy().view(np.uint64)] == \
        [0x16554d9eca36314c, 0xdb20fe9d672d0fdc, 0xd7e772cee186176b, 0x7e68b68aec7ba23b]


def _to_device(st, ptr, device):
    ns = types.SimpleNamespace(**{k: torch.as_tensor(np.ascontiguousarray(v)).to(device) for k, v in st.items()})
    ns.atom_ptr = torch.as_tensor(ptr.astype(np.int32)).to(device)
    ns.B = len(ptr) - 1
    return ns


def _random_case(sizes, seed=0):
    """Random ragged state: per-structure T and friction (0 included), structures at their first frame and later ones,
    a failed structure, one with a NaN force, one with a NaN energy and one moving too fast."""
    from torch_m3gnet_b200.calculator import ACC_UNIT

    rng = np.random.default_rng(seed)
    B, N = len(sizes), int(sum(sizes))
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    masses = rng.choice([1.008, 12.011, 63.546, 195.08], N)
    c1 = np.exp(-rng.uniform(0.0, 0.1, B) * 2.0)
    c1[1] = 1.0
    st = dict(pos=rng.uniform(0, 10, (N, 3)), v=rng.normal(0, 0.01, (N, 3)), inv_mass=ACC_UNIT / masses, c1=c1,
              c2=np.sqrt(1.0 - c1 * c1), kT=MO.KB * rng.uniform(10, 2000, B), bath=rng.normal(0, 0.1, B),
              sid=rng.integers(0, 1 << 40, B).astype(np.int64), step=rng.integers(1, 1000, B).astype(np.int32),
              status=np.zeros(B, np.int32))
    st["step"][[0, 3, 7]] = 0
    st["status"][5] = MO.FAILED
    forces = rng.normal(0, 0.5, (N, 3)).astype(np.float32)
    forces[ptr[6] + 1, 2] = np.nan
    energy = rng.normal(-3, 1, B).astype(np.float32)
    energy[8] = np.inf
    st["v"][ptr[9]] = 0.3                                # |v| dt = 0.3 sqrt(3) * 2 > 0.5 A
    return st, ptr, forces, energy


@pytest.mark.parametrize("advance,slot", [(True, 2), (True, -1), (False, 0)])
def test_kernel_matches_the_restatement(device, advance, slot):
    from torch_m3gnet_b200 import md

    st, ptr, forces, energy = _random_case(MD_SIZES)
    B = len(MD_SIZES)
    seed = (1 << 63) + 12345
    sw = seed - (1 << 64)
    want = {k: v.copy() for k, v in st.items()}
    obs_want = np.full((3, B, 4), np.nan)
    MO.langevin_step(want, forces, energy.astype(np.float64), ptr, 2.0, 0.5, seed, advance, slot, obs_want)
    outs = []
    for _ in range(2):
        d = _to_device(st, ptr, device)
        obs = torch.full((3, B, 4), float("nan"), dtype=torch.float64, device=device)
        md.langevin_step(d, torch.as_tensor(forces).to(device), torch.as_tensor(energy).to(device), 2.0, 0.5, sw,
                         advance, slot, obs)
        torch.cuda.synchronize()
        outs.append(({k: getattr(d, k).cpu().numpy() for k in st}, obs.cpu().numpy()))
    (got, obs_got), (again, obs_again) = outs
    for k in st:
        assert np.array_equal(got[k], again[k]), k                 # repeated calls are bitwise equal
    assert np.array_equal(obs_got, obs_again, equal_nan=True)
    assert np.array_equal(got["status"], want["status"]) and np.array_equal(got["step"], want["step"])
    assert want["status"][[5, 6, 8, 9]].tolist() == [MO.FAILED] * 4 and (np.delete(want["status"], [5, 6, 8, 9]) == 0).all()
    for k in ("pos", "v", "bath"):
        scale = np.abs(want[k]).max()
        np.testing.assert_allclose(got[k], want[k], rtol=1e-12, atol=1e-12 * scale, err_msg=k)
    np.testing.assert_allclose(obs_got, obs_want, rtol=1e-12, atol=0, equal_nan=True)
    for b in (5, 6, 8, 9):                                         # failed: bit-untouched, nothing recorded
        s, t = ptr[b], ptr[b + 1]
        for k in ("pos", "v"):
            assert np.array_equal(got[k][s:t], st[k][s:t]), (b, k)
        assert got["bath"][b] == st["bath"][b] and np.isnan(obs_got[:, b]).all()
    moved = np.abs(got["pos"] - st["pos"]).max(axis=1) > 0
    assert moved.any() == advance
    if slot >= 0:
        assert np.isfinite(obs_got[slot, np.delete(np.arange(B), [5, 6, 8, 9])]).all()


def test_maxwell_boltzmann_matches_the_restatement(device):
    from torch_m3gnet_b200 import md

    st, ptr, _, _ = _random_case(MD_SIZES, seed=3)
    want = {k: v.copy() for k, v in st.items()}
    MO.maxwell_boltzmann(want, ptr, 77)
    d = _to_device(st, ptr, device)
    md.maxwell_boltzmann(d, 77)
    got = d.v.cpu().numpy()
    np.testing.assert_allclose(got, want["v"], rtol=1e-12, atol=1e-12 * np.abs(want["v"]).max())
    m = 1.0 / st["inv_mass"]
    for b in range(len(MD_SIZES)):
        s, t = ptr[b], ptr[b + 1]
        p = (m[s:t, None] * got[s:t]).sum(axis=0)
        assert np.abs(p).max() <= 1e-12 * (m[s:t, None] * np.abs(got[s:t])).sum()


def _drive(structs, order, sids, steps, device, seed=9):
    """``steps`` MD steps of the structures ``order`` (stream ids ``sids[i]``) in one batch on a per-structure
    calculator, through md.py's kernels; final state per structure index."""
    from torch_m3gnet_b200 import md

    sub = [structs[i] for i in order]
    temps = [50.0 + 40.0 * i for i in order]
    st, ptr = MO.fresh_state([s[1] for s in sub], [np.full(len(s[2]), AR) for s in sub], temps,
                             [0.01 * (1 + i % 3) for i in order], 2.0, ids=[sids[i] for i in order])
    d = _to_device(st, ptr, device)
    md.maxwell_boltzmann(d, seed)
    calc = BatchLJ(device)
    lat = np.stack([s[0] for s in sub])
    z = np.concatenate([s[2] for s in sub])
    sizes = [len(s[2]) for s in sub]
    obs = torch.zeros((1, len(sub), 4), dtype=torch.float64, device=device)
    for k in range(steps + 1):
        e, f, _ = calc.compute(lat, d.pos, z, sizes)
        md.langevin_step(d, f, e, 2.0, 0.5, seed, k < steps, 0 if k == steps else -1, obs)
    out = {}
    for j, i in enumerate(order):
        sl = slice(ptr[j], ptr[j + 1])
        out[i] = (d.pos[sl].cpu().numpy(), d.v[sl].cpu().numpy(), float(d.bath[j]), obs[0, j].cpu().numpy())
    return out


def test_a_structure_steps_the_same_anywhere_in_the_batch(device):
    from torch_m3gnet_b200 import BatchMD

    structs = lj_structures(7, seed=13)
    sids = [11, 3, 500, 7, 1 << 40, 2, 9]
    runs = [_drive(structs, order, sids, 50, device) for order in ([0, 1, 2, 3, 4, 5, 6], [6, 4, 1, 3, 0, 5, 2],
                                                                    [3, 1], [1, 5, 6])]
    for r in runs[1:]:
        for i in r:
            for a, b in zip(runs[0][i], r[i]):
                assert np.array_equal(a, b), i
    # BatchMD: the working-set budget does not change any structure's trajectory
    kw = dict(masses={18: AR}, temperature=[60.0 + 30 * i for i in range(7)], friction=0.02, dt=2.0, seed=5)
    full = BatchMD(BatchLJ(device), structs, **kw).run(50, record_every=10, trajectory_every=25)
    for max_atoms in (40, 3):
        other = BatchMD(BatchLJ(device), structs, max_atoms=max_atoms, **kw).run(50, record_every=10,
                                                                                 trajectory_every=25)
        for i in range(len(structs)):
            for k in full[i]:
                assert np.array_equal(np.asarray(full[i][k]), np.asarray(other[i][k])), (max_atoms, i, k)


class Einstein:
    """Harmonic (Einstein) crystal on the GPU in torch: every atom tethered to its site, F = -kappa (x - x0)."""

    def __init__(self, x0, kappa, device):
        self.device, self.kappa = device, kappa
        self.x0 = torch.as_tensor(x0).to(device)

    def compute(self, lattices, cart, atomic_numbers, sizes=None, with_stress=False):
        u = cart - self.x0
        e = 0.5 * self.kappa * (u * u).sum(dim=1)
        batch = torch.repeat_interleave(torch.arange(len(sizes), device=self.device),
                                        torch.as_tensor(list(sizes), device=self.device))
        energy = torch.zeros(len(sizes), dtype=e.dtype, device=self.device).index_add_(0, batch, e)
        return energy.float(), (-self.kappa * u).float(), torch.zeros((len(sizes), 6), device=self.device)


def _baoab_stationary(omega, dt, c1, c2):
    """Stationary covariance of (x, v) at full steps of BAOAB on x'' = -omega^2 x with unit kT / m (noise c2 xi)."""
    import scipy.linalg

    h = 0.5 * dt
    Bm = np.array([[1.0, 0.0], [-h * omega ** 2, 1.0]])
    Am = np.array([[1.0, h], [0.0, 1.0]])
    Om = np.array([[1.0, 0.0], [0.0, c1]])
    T = Bm @ Am @ Om @ Am @ Bm
    q = Bm @ Am @ np.array([0.0, c2])
    return scipy.linalg.solve_discrete_lyapunov(T, np.outer(q, q))


def test_einstein_crystal_is_sampled_exactly(device):
    """BAOAB samples the configurations of a harmonic system exactly at any stable dt.  With equal masses in a
    structure the centre-of-mass removal leaves 3n - 3 independent internal modes of frequency sqrt(kappa / m), so
    <u_i^2> = (1 - 1/n) kT / kappa per axis; the mean kinetic temperature is that of BAOAB's full-step velocities
    (the stationary covariance of the step map), and the total momentum stays at the rounding level of the float32
    forces."""
    from torch_m3gnet_b200 import BatchMD
    from torch_m3gnet_b200.calculator import ACC_UNIT

    kappa, n, S, dt, gamma = 4.0, 8, 256, 10.0, 0.02
    masses = [4.0, 16.0, 64.0, 12.0]
    temps = [100.0, 300.0, 1000.0]
    omega_max = np.sqrt(kappa * ACC_UNIT / min(masses))
    assert 0.45 < omega_max * dt / 2.0 < 0.55               # about half the stability limit omega dt < 2
    rng = np.random.default_rng(0)
    structs = [(np.eye(3) * 6.0, rng.uniform(0, 6, (n, 3)), np.full(n, 1 + s % 4)) for s in range(S)]
    T = np.array([temps[s % 3] for s in range(S)])
    mass = np.array([masses[s % 4] for s in range(S)])
    calc = Einstein(np.concatenate([s[1] for s in structs]), kappa, device)
    steps, burn, every = 4000, 200, 2
    # at 1000 K the fastest 4-amu atoms move ~0.9 A in a 10 fs step; the tethered atoms share no neighbour list
    res = BatchMD(calc, structs, {z: masses[z - 1] for z in range(1, 5)}, T, friction=gamma, dt=dt, seed=21,
                  max_step_move=2.0).run(steps, record_every=1, trajectory_every=every)
    c1 = np.exp(-gamma * dt)
    c2 = np.sqrt(1 - c1 * c1)
    nb = 10
    for t in temps:
        group = [s for s in range(S) if T[s] == t]
        assert all(res[s]["status"] == "completed" for s in group)
        # position variance against kT / kappa, over time blocks of the group
        u2 = np.stack([((res[s]["trajectory"][burn // every:] - structs[s][1]) ** 2).mean(axis=(1, 2)) for s in group])
        ratio = u2.mean(axis=0) / ((1 - 1 / n) * MO.KB * t / kappa)
        blocks = ratio[: len(ratio) // nb * nb].reshape(nb, -1).mean(axis=1)
        se = blocks.std(ddof=1) / np.sqrt(nb)
        # kinetic temperature against BAOAB's stationary full-step velocity variance
        want_T = np.array([_baoab_stationary(np.sqrt(kappa * ACC_UNIT / mass[s]), dt, c1, c2)[1, 1] for s in group])
        tk = np.stack([res[s]["temperature"][burn:] / (t * want_T[j]) for j, s in enumerate(group)]).mean(axis=0)
        tblocks = tk[: len(tk) // nb * nb].reshape(nb, -1).mean(axis=1)
        tse = tblocks.std(ddof=1) / np.sqrt(nb)
        print(f"[einstein] T={t:.0f} K: <u^2> / (kT/kappa (1 - 1/n)) = {blocks.mean():.4f} +- {se:.4f}, "
              f"T_kin / T_BAOAB = {tblocks.mean():.4f} +- {tse:.4f} (T_BAOAB / T = {want_T.min():.4f}..{want_T.max():.4f})")
        assert abs(blocks.mean() - 1) < 4 * se and se < 0.02
        assert abs(tblocks.mean() - 1) < 4 * tse and tse < 0.02
    # the last frame's closing half kick adds dt/2 of the float32 force sum (not zero at rounding level) to the momentum
    # the step's centre-of-mass removal left at zero
    for s in range(S):
        v = res[s]["velocities"]
        assert np.abs((mass[s] * v).sum(axis=0)).max() <= 1e-7 * mass[s] * np.abs(v).sum()
    # the exact configurational variance of the step map itself
    assert _baoab_stationary(omega_max, dt, c1, c2)[0, 0] * omega_max ** 2 == pytest.approx(1.0, rel=1e-9)


def _cu_masses(structs):
    return [np.where(s[2] == 29, 63.546, 2.0 * s[2] + 1.0) for s in structs]


def test_model_nve_follows_velocity_verlet(device):
    from torch_m3gnet_b200 import BatchMD, M3GNetCalculator, VelocityVerlet, synthetic

    model = _verlet_model(device)
    lat, cart, z = synthetic.fcc_cu_supercell(2, 0.05, 3)
    v0 = _zero_momentum_velocities(32, 600.0, 2) * np.sqrt(AR / 63.546)
    ref = VelocityVerlet(M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device), lat, cart, z,
                         np.full(32, 63.546), dt=2.0, velocities=v0)
    ref.step(20)
    res = BatchMD(M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device), [(lat, cart, z)], {29: 63.546}, 600.0,
                  friction=0.0, dt=2.0, velocities=[v0]).run(20, record_every=20)
    dx = np.abs(res[0]["positions"] - ref.pos.cpu().numpy()).max()
    dv = np.abs(res[0]["velocities"] - ref.vel.cpu().numpy()).max()
    de = abs(res[0]["energy"][-1] + res[0]["kinetic_energy"][-1] - ref.potential_energy() - ref.kinetic_energy())
    print(f"[batch-md-model] friction 0 vs VelocityVerlet after 20 steps: |dx| {dx:.2e} A, |dv| {dv:.2e} A/fs, "
          f"|dE| {de:.2e} eV, moved {np.abs(res[0]['positions'] - cart).max():.3f} A")
    assert res[0]["status"] == "completed" and dx <= 1e-6 and dv <= 1e-7 and de <= 1e-4
    assert np.abs(res[0]["bath"]).max() < 1e-9


def test_model_langevin_batch(device):
    """Ragged multi-species cells and Cu cells at 300 K: finite, E_pot + E_kin - bath within its bound, and the last
    frame's energy and forces are those of a fresh Batch.from_arrays evaluation at the returned positions."""
    from torch_m3gnet_b200 import Batch, BatchMD, M3GNetCalculator, synthetic

    model = _verlet_model(device)
    structs = [synthetic.mpf_like_structure(s) for s in range(6)] + [synthetic.fcc_cu_supercell(2, 0.05, s)
                                                                    for s in range(4)]
    sizes = [len(s[2]) for s in structs]
    calc = M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device)
    last = {}
    compute = calc.compute

    def keep_last(*a, **k):
        out = compute(*a, **k)
        last["forces"] = out[1].clone()
        return out

    calc.compute = keep_last
    steps = 100
    res = BatchMD(calc, structs, _cu_masses(structs), 300.0, friction=0.01, dt=1.0, seed=17).run(steps,
                                                                                                   record_every=1)
    fresh = model(Batch.from_arrays(np.stack([r["lattice"] for r in res]), np.concatenate([r["positions"] for r in res]),
                                    np.concatenate([s[2] for s in structs]), sizes, 5.0, 4.0, device=device))
    assert torch.equal(fresh["forces"], last["forces"])
    worst = 0.0
    for i, r in enumerate(res):
        assert r["status"] == "completed" and r["n_steps"] == steps and np.isfinite(r["positions"]).all()
        assert r["energy"][-1] == float(fresh["total_energy"][i])
        conserved = r["energy"] + r["kinetic_energy"] - r["bath"]
        drift = np.abs(conserved - conserved[0]).max()
        worst = max(worst, drift / r["kinetic_energy"].std())
        assert drift <= 0.25 * r["kinetic_energy"].std() + 1e-5 * abs(r["energy"][0]), i
    print(f"[batch-md-model] max |E_pot + E_kin - bath drift| / std(E_kin) over {len(res)} structures: {worst:.3f}")


def test_launch_count(device):
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
        md = BatchMD(calc, structs, {29: 63.546}, 300.0, velocities=velocities)
        before = _lib.LAUNCHES
        md.run(3)
        assert md.n_iterations == len(inner) == 4
        assert _lib.LAUNCHES - before == sum(inner) + md.n_iterations + (velocities is None)
