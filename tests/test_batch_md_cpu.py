"""CPU: the numpy restatement of the batched Langevin step (tests/md_oracle.py) -- its Philox4x64-10 against the known
answer and numpy.random.Philox, its friction = 0 limit against calculator.py::VelocityVerlet, the conserved quantity
E_pot + E_kin - bath with the thermostat on -- and the host side of BatchMD (results in input order, independence from
the chunk budget, failure isolation, input validation) with the restatement standing in for the kernels and a periodic
Lennard-Jones calculator on the CPU."""
import numpy as np
import pytest
import torch

from tests import md_oracle as MO
from tests.test_batch_fire_cpu import BatchLJ, lj_structures

AR = 39.948  # amu; the LJ cells of lj_structures are argon-like (Z = 18)
M64 = 1 << 64


def _oracle_step(st, forces, energy, dt, max_step_move, seed, advance, slot, obs):
    """md.langevin_step with the numpy restatement in place of the kernel (CPU tensors)."""
    d = {k: getattr(st, k).numpy().copy() for k in MO.STATE_KEYS}
    o = obs.numpy().copy()
    MO.langevin_step(d, forces.double().numpy(), energy.double().numpy(), st.atom_ptr.numpy(), dt, max_step_move,
                     MO.seed_word(seed), advance, slot, o)
    for k, val in d.items():
        getattr(st, k).copy_(torch.from_numpy(val))
    obs.copy_(torch.from_numpy(o))


def _oracle_mb(st, seed):
    d = {k: getattr(st, k).numpy().copy() for k in MO.STATE_KEYS}
    MO.maxwell_boltzmann(d, st.atom_ptr.numpy(), MO.seed_word(seed))
    st.v.copy_(torch.from_numpy(d["v"]))


@pytest.fixture
def restated(monkeypatch):
    from torch_m3gnet_b200 import md

    monkeypatch.setattr(md, "langevin_step", _oracle_step)
    monkeypatch.setattr(md, "maxwell_boltzmann", _oracle_mb)
    return md


def _counter_plus_one(c):
    v = (sum(int(w) << (64 * i) for i, w in enumerate(c)) + 1) % (1 << 256)
    return np.array([(v >> (64 * i)) % M64 for i in range(4)], dtype=np.uint64)


def test_philox_known_answer_and_numpy():
    words = MO.philox4x64_10(np.zeros(4, np.uint64), np.zeros(2, np.uint64))
    assert [int(w) for w in words] == [0x16554d9eca36314c, 0xdb20fe9d672d0fdc, 0xd7e772cee186176b, 0x7e68b68aec7ba23b]
    rng = np.random.default_rng(0)
    ctrs, keys, want = [], [], []
    for t in range(64):
        c = rng.integers(0, M64, 4, dtype=np.uint64)
        k = rng.integers(0, M64, 2, dtype=np.uint64)
        if t % 4 == 0:
            c[0] = np.uint64(M64 - 1)                   # the increment carries into the next word
        if t % 9 == 0:
            c[:] = np.uint64(M64 - 1)
        # numpy increments its counter before it generates
        want.append(np.random.Philox(counter=c, key=k).random_raw(4))
        ctrs.append(_counter_plus_one(c))
        keys.append(k)
    assert np.array_equal(MO.philox4x64_10(np.stack(ctrs), np.stack(keys)), np.stack(want))


def test_normals_are_standard():
    xi = np.concatenate([MO.normals(4096, s, 7, 0, 12345) for s in range(4)])
    assert np.isfinite(xi).all()
    assert abs(xi.mean()) < 4 / np.sqrt(xi.size) and abs(xi.var() - 1) < 4 * np.sqrt(2 / xi.size)
    u = MO.uniform53(np.array([0, M64 - 1], dtype=np.uint64))
    assert u[0] == 2.0 ** -54 and u[1] == 1.0           # never 0, so the log is finite; 1 - 2^-54 rounds to 1
    # the counter names the structure and the step: other streams give other numbers
    assert not np.array_equal(MO.normals(8, 0, 7, 0, 1), MO.normals(8, 1, 7, 0, 1))
    assert not np.array_equal(MO.normals(8, 0, 7, 0, 1), MO.normals(8, 0, 8, 0, 1))
    assert not np.array_equal(MO.normals(8, 0, 0, 0, 1), MO.normals(8, 0, 0, 1, 1))


def _zero_momentum_velocities(n, T, seed):
    from torch_m3gnet_b200.calculator import ACC_UNIT

    v = np.random.default_rng(seed).normal(0, np.sqrt(MO.KB * T * ACC_UNIT / AR), (n, 3))
    return v - v.mean(axis=0)


def test_nve_limit_follows_velocity_verlet():
    """friction = 0: c1 = 1, c2 = 0, and BAOAB is velocity Verlet.  The restatement also removes the centre-of-mass
    velocity that the float32 force sums give (VelocityVerlet's centre of mass drifts by ~1e-11 A/fs here), so the two
    differ by a rigid translation of a few 1e-9 A and agree to ~1e-14 A once it is taken out."""
    from torch_m3gnet_b200.calculator import VelocityVerlet

    (lat, cart, z), = [s for s in lj_structures(2, seed=7) if len(s[2]) == 32]
    v0 = _zero_momentum_velocities(32, 300.0, 1)
    calc = BatchLJ()
    ref = VelocityVerlet(calc, lat, cart, z, np.full(32, AR), dt=2.0, velocities=v0)
    st, ptr = MO.fresh_state([cart], [np.full(32, AR)], 300.0, 0.0, 2.0)
    st["v"][:] = v0
    assert st["c1"][0] == 1.0 and st["c2"][0] == 0.0
    obs = np.zeros((1, 1, 4))
    worst = rigid = 0.0
    for k in range(200):
        out = calc.compute(lat, st["pos"], z, [32])
        MO.langevin_step(st, out[1].numpy(), out[0].double().numpy(), ptr, 2.0, 0.5, 0, True, -1, obs)
        ref.step()
        d = st["pos"] - ref.pos.numpy()
        worst, rigid = max(worst, np.abs(d - d.mean(axis=0)).max()), max(rigid, np.abs(d).max())
    out = calc.compute(lat, st["pos"], z, [32])
    MO.langevin_step(st, out[1].numpy(), out[0].double().numpy(), ptr, 2.0, 0.5, 0, False, 0, obs)
    print(f"[md-oracle] friction 0 over 200 steps: max |restatement - VelocityVerlet| = {rigid:.2e} A, "
          f"{worst:.2e} A without the centre-of-mass drift")
    assert worst <= 1e-12 and rigid <= 1e-8
    dv = st["v"] - ref.vel.numpy()
    assert np.abs(dv - dv.mean(axis=0)).max() <= 1e-14 and np.abs(dv).max() <= 1e-10
    assert abs(st["bath"][0]) < 1e-12 and st["step"][0] == 200   # only the centre-of-mass removal, at rounding level
    assert obs[0, 0, 1] == pytest.approx(ref.kinetic_energy(), rel=1e-9)
    assert np.abs(st["pos"] - cart).max() > 0.05  # it moved


def test_thermostat_conserves_the_extended_energy():
    """E_pot + E_kin - bath stays constant up to the integration error while the thermostat exchanges energy."""
    structs = [s for s in lj_structures(4, seed=8) if len(s[2]) == 32]
    calc = BatchLJ()
    n = len(structs)
    carts = [s[1] for s in structs]
    st, ptr = MO.fresh_state(carts, [np.full(len(c), AR) for c in carts], 120.0, 0.02, 2.0)
    MO.maxwell_boltzmann(st, ptr, 3)
    steps = 400
    obs = np.zeros((steps + 1, n, 4))
    lat = np.stack([s[0] for s in structs])
    z = np.concatenate([s[2] for s in structs])
    for k in range(steps + 1):
        out = calc.compute(lat, st["pos"], z, [32] * n)
        MO.langevin_step(st, out[1].numpy(), out[0].double().numpy(), ptr, 2.0, 0.5, 3, k < steps, k, obs)
    assert (st["status"] == 0).all()
    e_pot, e_kin, temp, bath = np.moveaxis(obs, -1, 0)
    conserved = e_pot + e_kin - bath
    drift = np.abs(conserved - conserved[0]).max(axis=0)
    spread = e_kin.std(axis=0)
    print(f"[md-oracle] extended-energy drift {drift} eV, E_kin std {spread} eV, bath {bath[-1]} eV")
    assert (np.abs(bath[-1]) > 2 * drift).all()       # the thermostat did exchange energy
    assert (drift < 0.05 * spread).all()


def _run(md, structs, **kw):
    calc = BatchLJ()
    args = dict(masses={18: AR}, temperature=[80.0, 150.0, 300.0, 60.0, 200.0, 100.0][:len(structs)],
                friction=0.02, dt=2.0, seed=2 ** 63 + 5)
    args.update(kw)
    steps = args.pop("steps", 30)
    rec_every = args.pop("record_every", 5)
    traj_every = args.pop("trajectory_every", 10)
    res = md.BatchMD(calc, structs, **args).run(steps, record_every=rec_every, trajectory_every=traj_every)
    return res, calc


KEYS = {"status", "n_steps", "times", "energy", "kinetic_energy", "temperature", "bath", "positions", "velocities",
        "lattice", "trajectory"}


def test_results_in_input_order_and_independent_of_the_budget(restated):
    structs = lj_structures(6, seed=9)                   # sizes [4, 32, 4, 4, 32, 4]
    full, calc_full = _run(restated, structs)
    assert calc_full.calls[0] == tuple(len(s[2]) for s in structs) and len(calc_full.calls) == 31
    small, calc_small = _run(restated, structs, max_atoms=12)
    assert calc_small.calls[0] == (4,) and (4, 4) in calc_small.calls and (32,) in calc_small.calls
    tiny, calc_tiny = _run(restated, structs, max_atoms=3)     # smaller than any structure: one at a time
    assert set(calc_tiny.calls) == {(4,), (32,)} and len(calc_tiny.calls) == 6 * 31
    for i, s in enumerate(structs):
        a = full[i]
        assert a.keys() == KEYS and a["status"] == "completed" and a["n_steps"] == 30
        assert a["positions"].shape == a["velocities"].shape == (len(s[2]), 3)
        assert a["trajectory"].shape == (4, len(s[2]), 3) and np.array_equal(a["trajectory"][0], s[1])
        assert np.array_equal(a["times"], 10.0 * np.arange(7)) and a["energy"].shape == (7,)
        assert np.array_equal(a["lattice"], s[0])
        for other in (small, tiny):
            for k in a:
                assert np.array_equal(np.asarray(a[k]), np.asarray(other[i][k])), (i, k)
    # the noise is keyed to the structure's index in the input list: the same cell at another index moves otherwise
    twin, _ = _run(restated, [structs[1], structs[1]], temperature=150.0)
    assert not np.array_equal(twin[0]["positions"], twin[1]["positions"])
    assert np.array_equal(twin[0]["positions"], _run(restated, [structs[1]], temperature=150.0)[0][0]["positions"])


class PoisonedLJ(BatchLJ):
    """BatchLJ whose forces for atom rows [lo, hi) are NaN from call ``at`` on."""

    def __init__(self, lo, hi, at):
        super().__init__()
        self.lo, self.hi, self.at = lo, hi, at

    def compute(self, *a, **k):
        out = super().compute(*a, **k)
        if len(self.calls) > self.at:
            out[1][self.lo:self.hi] = float("nan")
        return out


def test_a_failed_structure_is_frozen_and_isolated(restated):
    structs = lj_structures(4, seed=10)                  # sizes [4, 32, 4, 4]
    kw = dict(masses=[np.full(len(s[2]), AR) for s in structs], temperature=100.0, dt=2.0, seed=4)
    ref = restated.BatchMD(BatchLJ(), structs, **kw).run(20, record_every=3, trajectory_every=4)
    got = restated.BatchMD(PoisonedLJ(4, 36, 13), structs, **kw).run(20, record_every=3, trajectory_every=4)
    bad = got[1]
    assert bad["status"] == "failed" and bad["n_steps"] == 13
    assert np.array_equal(bad["times"], [0.0, 6.0, 12.0, 18.0, 24.0])    # frames 0, 3, 6, 9, 12 < 13
    for k in ("energy", "kinetic_energy", "temperature", "bath"):
        assert np.array_equal(bad[k], ref[1][k][:5]), k
    assert np.array_equal(bad["trajectory"], ref[1]["trajectory"][:4])  # frames 0, 4, 8, 12
    assert np.isfinite(bad["positions"]).all()
    for i in (0, 2, 3):
        for k in ref[i]:
            assert np.array_equal(np.asarray(ref[i][k]), np.asarray(got[i][k])), (i, k)
    # a structure about to move further than max_step_move in one step fails at frame 0
    hot = restated.BatchMD(BatchLJ(), structs[:1], masses={18: AR}, temperature=0.0, dt=2.0,
                           velocities=[np.full((4, 3), 0.2)], max_step_move=0.5).run(5)
    assert hot[0]["status"] == "failed" and hot[0]["n_steps"] == 0 and hot[0]["energy"].size == 0


def test_maxwell_boltzmann_velocities(restated):
    structs = [s for s in lj_structures(6, seed=11) if len(s[2]) == 32]
    res, _ = _run(restated, structs, steps=0, temperature=500.0, friction=0.0)
    for r in res:
        p = (AR * r["velocities"]).sum(axis=0)
        assert np.abs(p).max() < 1e-12 * AR * np.abs(r["velocities"]).max() * 32
        assert 150.0 < r["temperature"][0] < 1500.0 and r["times"].tolist() == [0.0]


def test_validation():
    from torch_m3gnet_b200 import BatchMD

    structs = lj_structures(2, seed=12)
    m = {18: AR}
    one = (np.eye(3) * 5.0, np.zeros((1, 3)), np.array([18]))
    with pytest.raises(ValueError, match="one atom"):
        BatchMD(BatchLJ(), structs + [one], m, 300.0)
    with pytest.raises(ValueError, match="atomic numbers \\[18\\]"):
        BatchMD(BatchLJ(), structs, {29: 63.5}, 300.0)
    with pytest.raises(ValueError, match="masses"):
        BatchMD(BatchLJ(), structs, [np.full(4, AR)], 300.0)
    with pytest.raises(ValueError, match="masses"):
        BatchMD(BatchLJ(), structs, [np.full(4, AR), np.full(31, AR)], 300.0)
    with pytest.raises(ValueError, match="positive"):
        BatchMD(BatchLJ(), structs, [np.full(4, AR), np.full(32, -1.0)], 300.0)
    with pytest.raises(ValueError, match="temperature"):
        BatchMD(BatchLJ(), structs, m, -1.0)
    with pytest.raises(ValueError, match="temperature"):
        BatchMD(BatchLJ(), structs, m, [300.0, 300.0, 300.0])
    with pytest.raises(ValueError, match="friction"):
        BatchMD(BatchLJ(), structs, m, 300.0, friction=[0.01, -0.01])
    with pytest.raises(ValueError, match="dt"):
        BatchMD(BatchLJ(), structs, m, 300.0, dt=-1.0)
    with pytest.raises(ValueError, match="dt"):
        BatchMD(BatchLJ(), structs, m, 300.0, dt=0.0)
    with pytest.raises(ValueError, match="velocities"):
        BatchMD(BatchLJ(), structs, m, 300.0, velocities=[np.zeros((4, 3))])
    with pytest.raises(ValueError, match="velocities"):
        BatchMD(BatchLJ(), structs, m, 300.0, velocities=[np.zeros((4, 3)), np.full((32, 3), np.nan)])
    with pytest.raises(ValueError, match="seed"):
        BatchMD(BatchLJ(), structs, m, 300.0, seed=-1)
    with pytest.raises(ValueError, match="max_atoms"):
        BatchMD(BatchLJ(), structs, m, 300.0, max_atoms=0)
    with pytest.raises(ValueError, match="steps"):
        BatchMD(BatchLJ(), structs, m, 300.0).run(-1)
