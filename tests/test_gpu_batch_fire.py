"""GPU: the batched FIRE step (m3g_fire_step, csrc/relax.cu) against its numpy restatement (tests/fire_oracle.py),
batch independence, BatchFire against sequential Fire on a periodic Lennard-Jones calculator and on the model, the
working-set budget, failure isolation and the launch count."""
import types

import numpy as np
import pytest
import torch

from tests import fire_oracle as FO
from tests.test_batch_fire_cpu import BatchLJ, lj_structures

pytestmark = pytest.mark.gpu

F64_KEYS = ("pos", "v", "x", "xc", "vc", "lattice", "sigma_frame", "dt", "a", "fmax", "e_frame")
I32_KEYS = ("n_pos", "n_steps", "status")
FIRE = dict(FO.FIRE_DEFAULTS)


def _to_device(st, ptr, device):
    ns = types.SimpleNamespace(**{k: torch.as_tensor(np.ascontiguousarray(v)).to(device) for k, v in st.items()})
    ns.atom_ptr = torch.as_tensor(ptr.astype(np.int32)).to(device)
    ns.B = len(ptr) - 1
    return ns


def _kernel(st, ptr, forces, sigma, energy, device, fire=FIRE, fmax=1e-3, steps=50, pressure=0.01):
    from torch_m3gnet_b200 import relax

    d = _to_device(st, ptr, device)
    relax.fire_step(d, torch.as_tensor(forces).to(device), None if sigma is None else torch.as_tensor(sigma).to(device),
                    torch.as_tensor(energy).to(device), fire, fmax, steps, pressure)
    torch.cuda.synchronize()
    return {k: getattr(d, k).cpu().numpy() for k in st}


def _random_case(sizes, relax_cell, seed=0):
    """Random ragged state: both power signs, n_pos above and below n_min, max_move clipping on and off, a structure
    without forces, finished structures, one at its step limit."""
    rng = np.random.default_rng(seed)
    B, N = len(sizes), int(sum(sizes))
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    lat0 = np.stack([np.eye(3) * rng.uniform(4, 12) + rng.uniform(-0.3, 0.3, (3, 3)) for _ in range(B)])
    cf = np.asarray(sizes, dtype=np.float64)
    Dx = np.eye(3)[None] + rng.uniform(-0.02, 0.02, (B, 3, 3))
    forces = rng.normal(0, 0.3, (N, 3)).astype(np.float32)
    v = rng.normal(0, 0.05, (N, 3))
    vc = rng.normal(0, 0.05, (B, 3, 3))
    for b in range(B):
        s, t = ptr[b], ptr[b + 1]
        sign = 1.0 if b % 2 == 0 else -1.0          # power > 0 / <= 0
        v[s:t] = sign * np.abs(v[s:t]) * np.sign(forces[s:t])
        if b % 4 == 1:
            forces[s:t] *= 300.0                    # big steps: the max_move clip
    forces[ptr[4]:ptr[5]] = 0.0                     # no bonds
    sigma = rng.normal(0, 2e-3, (B, 3, 3)).astype(np.float32)
    st = dict(pos=rng.uniform(0, 10, (N, 3)), v=v, x=rng.uniform(0, 10, (N, 3)), xc=cf[:, None, None] * Dx,
              vc=vc, L0=lat0, lattice=np.einsum("bij,bkj->bik", lat0, Dx), sigma_frame=np.zeros((B, 3, 3)),
              dt=rng.uniform(0.05, 0.5, B), a=rng.uniform(0.05, 0.1, B), fmax=np.zeros(B), e_frame=np.zeros(B),
              cell_factor=cf, n_pos=rng.integers(0, 9, B).astype(np.int32),
              n_steps=rng.integers(0, 40, B).astype(np.int32), status=np.zeros(B, np.int32))
    st["status"][6], st["status"][7], st["status"][8] = FO.CONVERGED, FO.NOT_CONVERGED, FO.FAILED
    st["n_steps"][9] = 50                           # at the step limit
    st["dt"][1::4] = 0.5
    st["n_pos"][0], st["n_pos"][2], st["n_pos"][3] = 8, 2, 7
    energy = rng.normal(-3, 1, B).astype(np.float32)
    return st, ptr, forces, (sigma if relax_cell else None), energy


SIZES = [1, 2, 32, 700, 5, 3, 4, 6, 8, 12, 257]


@pytest.mark.parametrize("relax_cell", [False, True])
def test_kernel_matches_the_restatement(device, relax_cell):
    st, ptr, forces, sigma, energy = _random_case(SIZES, relax_cell)
    want = {k: v.copy() for k, v in st.items()}
    FO.fire_step(want, forces.astype(np.float64), None if sigma is None else sigma.astype(np.float64),
                 energy.astype(np.float64), FIRE, 1e-3, 50, 0.01, ptr)
    got = _kernel(st, ptr, forces, sigma, energy, device)
    again = _kernel(st, ptr, forces, sigma, energy, device)
    for k in st:
        assert np.array_equal(got[k], again[k]), k                # repeated calls are bitwise equal
    for k in I32_KEYS:
        assert np.array_equal(got[k], want[k]), (k, got[k], want[k])
    for k in F64_KEYS:
        if not relax_cell and k in ("x", "xc", "vc", "lattice", "sigma_frame"):
            assert np.array_equal(got[k], st[k]), k               # not read nor written without the cell filter
            continue
        scale = max(np.abs(want[k][np.isfinite(want[k])]).max(initial=0.0), 1e-300)
        np.testing.assert_allclose(got[k], want[k], rtol=1e-12, atol=1e-12 * scale, err_msg=k)
    for b in (6, 7, 8):                                           # finished: bit-untouched
        s, t = ptr[b], ptr[b + 1]
        for k in ("pos", "v", "x"):
            assert np.array_equal(got[k][s:t], st[k][s:t]), (b, k)
        for k in ("dt", "a", "n_pos", "n_steps", "status", "fmax", "e_frame", "xc", "vc", "lattice", "sigma_frame"):
            assert np.array_equal(got[k][b], st[k][b]), (b, k)
    status = want["status"]
    assert status[9] == FO.NOT_CONVERGED and (relax_cell or status[4] == FO.CONVERGED)
    # the case covers both power branches (n_pos + 1 after P > 0, 0 otherwise), n_pos > n_min and the clip on and off
    moved = [b for b in range(len(SIZES)) if want["n_steps"][b] > st["n_steps"][b]]
    positive = [b for b in moved if want["n_pos"][b] == st["n_pos"][b] + 1]
    assert positive and len(positive) < len(moved)
    assert any(st["n_pos"][b] > FIRE["n_min"] for b in positive)
    clipped = [b for b in moved if b % 4 == 1]
    for b in clipped:
        s, t = ptr[b], ptr[b + 1]
        key = "x" if relax_cell else "pos"
        dr = np.concatenate([want[key][s:t] - st[key][s:t]] + ([want["xc"][b] - st["xc"][b]] if relax_cell else []))
        assert np.sqrt((dr * dr).sum()) == pytest.approx(FIRE["max_move"], rel=1e-9)
    assert clipped and len(moved) > len(clipped)


@pytest.mark.parametrize("relax_cell", [False, True])
def test_a_structure_steps_the_same_anywhere_in_the_batch(device, relax_cell):
    """The same structure and forces at different batch offsets, next to different neighbours: bitwise equal state."""
    st, ptr, forces, sigma, energy = _random_case(SIZES, relax_cell, seed=4)
    probe = 3                                                       # the 700-atom structure
    results = []
    for order in ([3, 0, 1, 2, 4, 5, 6, 7, 8, 9, 10], [10, 2, 3, 9], [3], [0, 1, 4, 5, 3]):
        sizes = [SIZES[b] for b in order]
        p = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        atom_rows = np.concatenate([np.arange(ptr[b], ptr[b + 1]) for b in order])
        sub = {k: (v[atom_rows] if v.shape[0] == ptr[-1] else v[order]) for k, v in st.items()}
        out = _kernel(sub, p, forces[atom_rows], None if sigma is None else sigma[order], energy[order], device)
        j = order.index(probe)
        sl = slice(p[j], p[j + 1])
        results.append({k: (out[k][sl] if st[k].shape[0] == ptr[-1] else out[k][j]) for k in st})
    for r in results[1:]:
        for k in r:
            assert np.array_equal(r[k], results[0][k]), k


def _compare_with_fire(got, structs, relax_cell, pressure, fmax, steps):
    from torch_m3gnet_b200 import Fire

    worst = 0.0
    for i, s in enumerate(structs):
        ref = Fire(BatchLJ(), *s, relax_cell=relax_cell, pressure=pressure)
        ok = ref.run(fmax=fmax, steps=steps)
        assert got[i]["status"] == ("converged" if ok else "not converged"), i
        assert got[i]["n_steps"] == ref.n_steps, i
        worst = max(worst, np.abs(got[i]["positions"] - ref.pos.numpy()).max(),
                    np.abs(got[i]["lattice"] - ref.lattice[0]).max())
    print(f"[batch-fire-lj] relax_cell={relax_cell}: max |BatchFire - Fire| = {worst:.2e} A, "
          f"steps {[r['n_steps'] for r in got]}")
    assert worst <= 1e-9


@pytest.mark.parametrize("relax_cell", [False, True])
def test_lj_batch_matches_sequential_fire_and_budget(device, relax_cell):
    from torch_m3gnet_b200 import BatchFire

    structs = lj_structures(12, seed=5)
    p = 0.002 if relax_cell else 0.0
    got = BatchFire(BatchLJ(device), structs, relax_cell=relax_cell, pressure=p).run(fmax=0.02, steps=80)
    _compare_with_fire(got, structs, relax_cell, p, 0.02, 80)
    opt = BatchFire(BatchLJ(device), structs, relax_cell=relax_cell, pressure=p, max_atoms=40)
    small = opt.run(fmax=0.02, steps=80)
    assert opt.n_regroups >= 3
    for i in range(len(structs)):
        for k in got[i]:
            assert np.array_equal(np.asarray(got[i][k]), np.asarray(small[i][k])), (i, k)


def test_failure_is_isolated_and_limits(device):
    from torch_m3gnet_b200 import BatchFire

    structs = lj_structures(8, seed=6)
    lat, cart, z = structs[3]
    cart = cart.copy()
    cart[2] = cart[1] + np.array([0.0, 1e-6, 0.0])
    bad = structs[:3] + [(lat, cart, z)] + structs[4:]
    ref = BatchFire(BatchLJ(device), structs).run(fmax=0.02, steps=60)
    got = BatchFire(BatchLJ(device), bad).run(fmax=0.02, steps=60)
    assert got[3]["status"] == "failed" and got[3]["fmax"] == np.inf
    for i in range(len(structs)):
        if i != 3:
            for k in ref[i]:
                assert np.array_equal(np.asarray(ref[i][k]), np.asarray(got[i][k])), (i, k)
    done = [(r["lattice"], r["positions"], s[2]) for r, s in zip(ref, structs) if r["status"] == "converged"]
    again = BatchFire(BatchLJ(device), done).run(fmax=0.05, steps=10)
    assert done and all(r["status"] == "converged" and r["n_steps"] == 0 for r in again)
    capped = BatchFire(BatchLJ(device), structs).run(fmax=1e-9, steps=4)
    assert all(r["status"] == "not converged" and r["n_steps"] == 4 for r in capped)


def _verlet_model(device):
    from torch_m3gnet_b200 import build_model

    torch.manual_seed(11)
    model = build_model(5.0, 4.0, 3, 3, 95, 64, 3, device=device)
    sd = model.state_dict()
    model.load_state_dict({k: (v * 3 if k.endswith("weight") else v) for k, v in sd.items()})
    return model


def test_model_fixed_cell_batch(device):
    """Cu cells and ragged multi-species cells relaxed in one batch: energies and fmax go down, every record is the frame a
    fresh model call computes at the returned positions, and the energies agree with sequential Fire runs.  A fixed
    number of steps (fmax = 0): every structure stops at the same frame, and the trajectories have not yet drifted apart
    beyond the fp32 rounding with which the model's message sums depend on the batch position (DESIGN.md §4.1)."""
    from torch_m3gnet_b200 import Batch, BatchFire, Fire, M3GNetCalculator, synthetic

    model = _verlet_model(device)
    structs = [synthetic.fcc_cu_supercell(2, 0.08, 100 + s) for s in range(16)]
    structs += [synthetic.mpf_like_structure(s) for s in range(3)]
    sizes = [len(s[2]) for s in structs]
    calc = M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device)
    res = BatchFire(calc, structs).run(fmax=0.0, steps=30)
    fresh = model(Batch.from_arrays(np.stack([r["lattice"] for r in res]), np.concatenate([r["positions"] for r in res]),
                                    np.concatenate([s[2] for s in structs]), sizes, 5.0, 4.0, device=device))
    f = fresh["forces"].double()
    ptr = np.concatenate([[0], np.cumsum(sizes)])
    worst = 0.0
    for i, (r, s) in enumerate(zip(res, structs)):
        assert r["status"] == "not converged" and r["n_steps"] == 30
        assert r["energy"] == float(fresh["total_energy"][i])
        assert r["fmax"] == pytest.approx(float(f[ptr[i]:ptr[i + 1]].norm(dim=1).max()), rel=1e-12)
        ref = Fire(M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device), *s)
        e0, f0 = float(ref.energy[0]), ref.fmax()
        ref.run(fmax=0.0, steps=30)
        assert r["energy"] < e0 and r["fmax"] < f0, i
        worst = max(worst, abs(r["energy"] - float(ref.energy[0])) / sizes[i])
    print(f"[batch-fire-model] max |dE|/atom vs sequential Fire after 30 steps {worst:.2e} eV")
    assert worst <= 1e-5


def test_model_variable_cell_batch(device):
    """test_variable_cell_relaxation_of_strained_fcc_cu's assertions for three copies strained along x, y and z, relaxed
    in one batch."""
    from tests.util import golden, state_dict_of
    from torch_m3gnet_b200 import BatchFire, M3GNetCalculator, build_model, synthetic

    model = build_model(5.0, 4.0, 3, 3, 95, 64, 3, device=device)
    model.load_state_dict({k: (v * 3 if k.endswith("weight") else v) for k, v in state_dict_of(golden("c1_default")).items()})
    lat0, cart0, z = synthetic.fcc_cu_supercell(2, 0.0, 0)
    calc = M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device)
    sig = calc.compute(lat0, cart0, z, with_stress=True)[3][0].double().cpu().numpy()
    p = -float(np.trace(sig)) / 3
    strains = [np.diag(np.roll([1.03, 1.0, 1.0], ax)) for ax in range(3)]
    res = BatchFire(calc, [(lat0 @ s, cart0 @ s, z) for s in strains], relax_cell=True, pressure=p).run(fmax=0.05,
                                                                                                     steps=150)
    tet0 = 0.03 * lat0[0, 0]
    for ax, r in enumerate(res):
        L = r["lattice"]
        o1, o2 = (ax + 1) % 3, (ax + 2) % 3
        tet = abs(L[ax, ax] - L[o1, o1])
        frac = r["positions"] @ np.linalg.inv(L)
        dev_sites = frac - cart0 / lat0[0, 0]
        dev_sites -= np.round(dev_sites)
        print(f"[batch-vc-fire] axis {ax}: {r['status']} fmax {r['fmax']:.4f} in {r['n_steps']} steps, "
              f"cell diag {np.diag(L)}")
        assert r["status"] == "converged" and r["fmax"] < 0.05
        assert np.abs(L - np.diag(np.diag(L))).max() < 1e-5
        assert abs(L[o1, o1] - L[o2, o2]) < 1e-5
        assert np.abs(dev_sites).max() < 1e-5
        assert tet < 0.25 * tet0
        assert r["cell_stress"].shape == (3, 3)


def test_launch_count(device):
    from torch_m3gnet_b200 import BatchFire, M3GNetCalculator, _lib, synthetic

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
    for relax_cell in (False, True):
        inner.clear()
        opt = BatchFire(calc, structs, relax_cell=relax_cell)
        before = _lib.LAUNCHES
        opt.run(fmax=0.0, steps=3)
        assert opt.n_iterations == len(inner) == 4
        assert _lib.LAUNCHES - before == sum(inner) + opt.n_iterations * _lib._KERNELS_PER_CALL["fire_step"] == \
            sum(inner) + opt.n_iterations
