"""CPU: the numpy restatement of the batched FIRE step (tests/fire_oracle.py) against calculator.py::Fire, and the host
side of BatchFire (admission, budget, regroups, results in input order) with the restatement standing in for the
kernel and a periodic Lennard-Jones calculator on the CPU."""
import numpy as np
import pytest
import torch

from tests import fire_oracle as FO
from tests.test_cell_stress_cpu import _fcc, lj


class BatchLJ:
    """``M3GNetCalculator.compute``'s protocol for a ragged batch: float64 LJ per structure (tests/test_cell_stress_cpu
    ``lj``), energy, forces and stress rounded to float32 as the model's are, returned on ``device``."""

    def __init__(self, device=torch.device("cpu")):
        self.device = device
        self.calls = []

    def compute(self, lattices, cart, atomic_numbers, sizes=None, with_stress=False):
        cart = cart.cpu().numpy() if torch.is_tensor(cart) else np.asarray(cart, dtype=np.float64)
        cart = cart.reshape(-1, 3)
        sizes = [len(cart)] if sizes is None else [int(n) for n in sizes]
        lat = np.asarray(lattices, dtype=np.float64).reshape(len(sizes), 3, 3)
        self.calls.append(tuple(sizes))
        ptr = np.concatenate([[0], np.cumsum(sizes)])
        es, fs, ss = [], [], []
        with np.errstate(over="ignore", invalid="ignore"):
            for b in range(len(sizes)):
                e, f, s = lj(lat[b], cart[ptr[b]:ptr[b + 1]])
                es.append(e), fs.append(f), ss.append(s)
            e32 = np.asarray(es).astype(np.float32)
            f32 = np.concatenate(fs).astype(np.float32)
            s32 = np.stack(ss).astype(np.float32)
        out = (torch.from_numpy(e32).to(self.device), torch.from_numpy(f32).to(self.device),
               torch.zeros((len(sizes), 6), dtype=torch.float32, device=self.device))
        return out + (torch.from_numpy(s32).to(self.device),) if with_stress else out


def lj_structures(count, seed=0):
    """Ragged set of strained / jittered fcc LJ cells (4 and 32 atoms)."""
    rng = np.random.default_rng(seed)
    out = []
    for s in range(count):
        lat, cart = _fcc(3.7, 1 + (s % 3 == 1))
        strain = np.eye(3) + np.diag(rng.uniform(-0.03, 0.03, 3))
        cart = cart @ strain + rng.uniform(-0.08, 0.08, cart.shape)
        out.append((lat @ strain, cart, np.full(len(cart), 18)))
    return out


def oracle_step(st, forces, sigma, energy, fire, fmax, steps, pressure):
    """relax.fire_step with the numpy restatement in place of the kernel (CPU tensors)."""
    d = {k: getattr(st, k).numpy().copy() for k in FO.STATE_KEYS if getattr(st, k, None) is not None}
    FO.fire_step(d, forces.double().numpy(), None if sigma is None else sigma.double().numpy(), energy.double().numpy(),
                 fire, fmax, steps, pressure, st.atom_ptr.numpy())
    for k, val in d.items():
        getattr(st, k).copy_(torch.from_numpy(val))


@pytest.mark.parametrize("relax_cell", [False, True])
def test_restatement_follows_fire_for_50_steps(relax_cell):
    from torch_m3gnet_b200.calculator import Fire

    (lat, cart, z), = lj_structures(1, seed=3)
    p = 0.005 if relax_cell else 0.0
    calc = BatchLJ()
    ref = Fire(calc, lat, cart, z, relax_cell=relax_cell, pressure=p)
    st, ptr = FO.fresh_state([(lat, cart, z)], FO.FIRE_DEFAULTS)
    worst = 0.0
    for k in range(50):
        out = calc.compute(st["lattice"], st["pos"], z, [len(z)], with_stress=relax_cell)
        sigma = out[3].double().numpy() if relax_cell else None
        if relax_cell:
            g = FO.generalised_forces(out[1].numpy(), sigma[0], st["L0"][0], st["lattice"][0], st["cell_factor"][0], p)
            np.testing.assert_allclose(g, ref.gen_forces.numpy(), rtol=1e-12, atol=1e-14)
        FO.fire_step(st, out[1].numpy(), sigma, out[0].double().numpy(), FO.FIRE_DEFAULTS, 0.0, 1000, p, ptr)
        ref.step()
        worst = max(worst, np.abs(st["pos"] - ref.pos.numpy()).max(), np.abs(st["lattice"][0] - ref.lattice[0]).max())
        assert st["n_steps"][0] == ref.n_steps and st["n_pos"][0] == ref.n_pos
        assert st["dt"][0] == pytest.approx(ref.dt, rel=1e-14) and st["a"][0] == pytest.approx(ref.a, rel=1e-14)
    print(f"[fire-oracle] relax_cell={relax_cell}: max |restatement - Fire| over 50 steps = {worst:.2e} A")
    assert worst <= 1e-12
    assert np.abs(st["pos"] - cart).max() > 1e-2  # it moved


def test_admission_order_and_budget():
    from torch_m3gnet_b200.relax import admit, should_regroup

    sizes = [4, 32, 4, 108, 4, 4]
    assert admit(sizes, 0, None, 0, 0) == 6
    assert admit(sizes, 0, 40, 0, 0) == 3           # 4 + 32 + 4 = 40 fits, 108 does not
    assert admit(sizes, 3, 40, 0, 0) == 4           # larger than the budget: enters alone into an empty set
    assert admit(sizes, 3, 40, 4, 1) == 3           # ... but not next to anything else
    assert admit(sizes, 4, 40, 36, 2) == 5          # input order, while the atoms fit
    assert admit(sizes, 6, 40, 0, 0) == 6
    assert should_regroup(10, 40, True, False, False) and not should_regroup(9, 40, True, False, False)
    assert should_regroup(1, 40, True, False, True) and not should_regroup(0, 40, False, False, True)
    assert should_regroup(40, 40, True, True, False)


@pytest.mark.parametrize("relax_cell", [False, True])
def test_batch_fire_host_logic_with_the_restatement(monkeypatch, relax_cell):
    """Results in input order and independent of the working-set budget (bitwise), a structure larger than the budget
    relaxed alone, admission in input order, and every structure equal to its own Fire run."""
    from torch_m3gnet_b200 import relax
    from torch_m3gnet_b200.calculator import Fire

    monkeypatch.setattr(relax, "fire_step", oracle_step)
    structs = lj_structures(6, seed=1)
    p = 0.002 if relax_cell else 0.0
    kw = dict(relax_cell=relax_cell, pressure=p)
    full_calc = BatchLJ()
    full = relax.BatchFire(full_calc, structs, **kw).run(fmax=0.02, steps=60)
    assert full_calc.calls[0] == tuple(len(s[2]) for s in structs)
    small_calc = BatchLJ()
    opt = relax.BatchFire(small_calc, structs, max_atoms=20, **kw)
    small = opt.run(fmax=0.02, steps=60)
    sizes = [len(s[2]) for s in structs]                  # [4, 32, 4, 4, 32, 4]
    assert small_calc.calls[0] == (4,)                    # 4 + 32 > 20: the first structure starts alone
    assert max(sum(c) for c in small_calc.calls) <= 32    # the 32-atom cells (> 20) ran alone
    assert any(c == (32,) for c in small_calc.calls) and opt.n_regroups >= 4
    statuses = set()
    for i, (a, b) in enumerate(zip(full, small)):
        assert a.keys() == b.keys() == ({"status", "n_steps", "energy", "fmax", "positions", "lattice"}
                                        | ({"cell_stress"} if relax_cell else set()))
        for k in a:
            assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), (i, k)
        assert a["positions"].shape == (sizes[i], 3)
        ref = Fire(BatchLJ(), *structs[i], relax_cell=relax_cell, pressure=p)
        ok = ref.run(fmax=0.02, steps=60)
        assert a["status"] == ("converged" if ok else "not converged") and a["n_steps"] == ref.n_steps
        assert np.abs(a["positions"] - ref.pos.numpy()).max() < 1e-9
        assert np.abs(a["lattice"] - ref.lattice[0]).max() < 1e-9
        # Fire.fmax() takes the fixed-cell norm in float32 (the forces' dtype); the batched step in float64
        assert a["fmax"] == pytest.approx(ref.fmax(), rel=1e-9 if relax_cell else 1e-6)
        assert a["energy"] == pytest.approx(float(ref.energy[0]), rel=1e-7)
        statuses.add(a["status"])
    print(f"[batch-fire] statuses {statuses}, steps {[r['n_steps'] for r in full]}, regroups {opt.n_regroups}")
    assert "converged" in statuses


def test_failed_structure_leaves_the_batch(monkeypatch):
    from torch_m3gnet_b200 import relax

    monkeypatch.setattr(relax, "fire_step", oracle_step)
    structs = lj_structures(4, seed=2)
    lat, cart, z = structs[2]
    cart = cart.copy()
    cart[1] = cart[0] + np.array([1e-6, 0.0, 0.0])        # float32 LJ forces overflow
    bad = structs[:2] + [(lat, cart, z)] + structs[3:]
    ref = relax.BatchFire(BatchLJ(), structs).run(fmax=0.02, steps=40)
    got = relax.BatchFire(BatchLJ(), bad).run(fmax=0.02, steps=40)
    assert got[2]["status"] == "failed" and got[2]["n_steps"] == 0 and got[2]["fmax"] == np.inf
    for i in (0, 1, 3):
        for k in ref[i]:
            assert np.array_equal(np.asarray(ref[i][k]), np.asarray(got[i][k])), (i, k)
    # converged at step 0, and the step limit
    relaxed = [(r["lattice"], r["positions"], s[2]) for r, s in zip(ref, structs)]
    again = relax.BatchFire(BatchLJ(), relaxed[:1]).run(fmax=0.05, steps=40)
    assert again[0]["status"] == "converged" and again[0]["n_steps"] == 0
    capped = relax.BatchFire(BatchLJ(), structs[:1]).run(fmax=1e-9, steps=3)
    assert capped[0]["status"] == "not converged" and capped[0]["n_steps"] == 3
