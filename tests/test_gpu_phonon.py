"""GPU: the batched phonon kernels (csrc/phonon.cu) against their numpy restatement (tests/phonon_oracle.py) on random
ragged inputs (every unit-cell size 1 .. 32, odd 3n, degenerate spectra, failed structures), bitwise repeatability and
batch independence, the spring model on the device with float32 forces against its analytic dispersion, BatchPhonon on
the model against a fresh evaluation and against central differences of float64 oracle forces, rotation invariance,
the ABI's cap and the launch counts."""
import types
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import phonon_oracle as PO
from tests.test_phonon_cpu import (A, K_SPRING, M1, SiteModel, analytic_eigs, fcc_conventional, random_q,
                                   rock_salt_conventional)

pytestmark = pytest.mark.gpu

NS = [1, 2, 3, 5, 7, 8, 11, 16, 21, 32, 4, 6]          # 3n from 3 to 96, odd 3n for odd n
REPS = [(3, 2, 2), (2, 2, 2), (2, 1, 2), (1, 2, 2), (2, 1, 1), (1, 1, 2), (1, 2, 1), (1, 1, 2), (1, 1, 1),
        (1, 1, 2), (2, 2, 1), (1, 2, 1)]
NAN_STRUCT = 5                                          # gets one non-finite force
POISON = 99                                             # atomic number that makes RandomForces emit a NaN


class RandomForces:
    """``compute``'s protocol with float32 forces drawn from N(0, 1) seeded by the supercell's own positions (so a
    supercell gets the same forces in any chunk); a supercell holding atomic number ``POISON`` gets one NaN."""

    def __init__(self, device):
        self.device = device
        self.calls = []

    def compute(self, lattices, cart, atomic_numbers, sizes=None, with_stress=False):
        cart = np.asarray(cart, dtype=np.float64).reshape(-1, 3)
        z = np.asarray(atomic_numbers).reshape(-1)
        self.calls.append(tuple(sizes))
        out, o = [], 0
        for n in sizes:
            rng = np.random.default_rng(zlib.crc32(cart[o:o + n].tobytes()))
            f = rng.normal(0.0, 1.0, (n, 3)).astype(np.float32)
            if (z[o:o + n] == POISON).any():
                f[min(3, n - 1), 1] = np.nan
            out.append(f)
            o += n
        return (torch.zeros(len(sizes), device=self.device), torch.from_numpy(np.concatenate(out)).to(self.device),
                torch.zeros((len(sizes), 6), device=self.device))


def random_structures(seed=0):
    rng = np.random.default_rng(seed)
    out, masses = [], []
    for i, n in enumerate(NS):
        a = 2.6 * n ** (1 / 3)
        lat = a * (np.eye(3) + rng.uniform(-0.15, 0.15, (3, 3)))
        cart = rng.uniform(0, 1, (n, 3)) @ lat
        z = np.full(n, POISON if i == NAN_STRUCT else 14)
        out.append((lat, cart, z))
        masses.append(rng.uniform(1.0, 200.0, n))
    return out, masses


def _cpu_state(st):
    return types.SimpleNamespace(**{k: (v.cpu() if torch.is_tensor(v) else v) for k, v in vars(st).items()})


def _rel(got, want):
    scale = np.abs(want[np.isfinite(want)]).max(initial=0.0)
    return np.abs(got - want).max() / max(scale, 1e-300)


def test_kernels_match_the_restatement(device, monkeypatch):
    from torch_m3gnet_b200 import phonon

    structs, masses = random_structures()
    dev = phonon.BatchPhonon(RandomForces(device), structs, REPS, masses, symmetrize=2, max_atoms=400)
    recs = dev.run()
    with monkeypatch.context() as m:
        m.setattr(phonon, "fc_launch", PO.fc_launch)
        ref = phonon.BatchPhonon(RandomForces(torch.device("cpu")), structs, REPS, masses, symmetrize=2)
        ref_recs = ref.run()
    worst = dict(fc=0.0, D=0.0, eig=0.0, thermal=0.0)
    # force constants and flags
    for b, (r, w) in enumerate(zip(recs, ref_recs)):
        assert r["status"] == w["status"] == ("failed" if b == NAN_STRUCT else "ok")
        if b == NAN_STRUCT:
            assert np.isnan(r["force_constants"]).all() and np.isnan(r["max_residual_force"])
            continue
        worst["fc"] = max(worst["fc"], _rel(r["force_constants"], w["force_constants"]))
        assert r["max_residual_force"] == w["max_residual_force"]
    # D(q)
    rng = np.random.default_rng(1)
    qs = [rng.uniform(-0.5, 0.5, (1 + b % 3, 3)) for b in range(len(NS))]
    st, st_c = dev._st, _cpu_state(ref._st)
    q_ptr = torch.as_tensor(phonon._cum([len(q) for q in qs], np.int32)).to(device)
    D = phonon.dynmat_launch(st, torch.as_tensor(np.concatenate(qs)).to(device), q_ptr, 3 * max(NS)).cpu().numpy()
    i = 0
    for b, q in enumerate(qs):
        d = 3 * NS[b]
        for qq in q:
            want = PO.structure_dynmat(st_c, b, qq)
            got = D[i]
            i += 1
            assert (got[d:] == 0).all() and (got[:, d:] == 0).all()
            if b == NAN_STRUCT:
                assert np.isnan(got[:d, :d]).all()
                continue
            err = np.abs(got[:d, :d] - want).max() / np.linalg.norm(want)
            worst["D"] = max(worst["D"], err)
    # eigenvalues
    out, _, _ = dev._frequencies(qs)
    eig, sweeps, qst = out.eig.cpu().numpy(), out.sweeps.cpu().numpy(), out.q_status.cpu().numpy()
    o = i = 0
    for b, q in enumerate(qs):
        d = 3 * NS[b]
        for qq in q:
            got = eig[o:o + d]
            if b == NAN_STRUCT:
                assert np.isnan(got).all() and qst[i] == 1
            else:
                Dq = PO.structure_dynmat(st_c, b, qq)
                H = 0.5 * (Dq + Dq.conj().T)
                err = np.abs(got - np.linalg.eigvalsh(H)).max() / np.linalg.norm(H)
                worst["eig"] = max(worst["eig"], err)
                assert qst[i] == 0 and 1 <= sweeps[i] <= 30 and (np.diff(got) >= 0).all()
            o, i = o + d, i + 1
    f_dev = dev.frequencies(qs)
    o = 0
    for b in range(len(NS)):
        d = len(qs[b]) * 3 * NS[b]
        assert np.array_equal(f_dev[b].reshape(-1), PO.to_thz(eig[o:o + d]), equal_nan=True)
        o += d
    # thermal properties, against the restated sums over the kernel's own mesh frequencies
    temps = np.array([0.0, 1.0, 10.0, 300.0, 1000.0])
    th = dev.thermal_properties(mesh=(3, 2, 2), temperatures=temps, cutoff_frequency=0.05)
    fm = dev.frequencies(phonon.mesh_qpoints((3, 2, 2)))
    for b in range(len(NS)):
        if b == NAN_STRUCT:
            assert np.isnan(th[b]["free_energy"]).all() and th[b]["n_imaginary"] == -1
            continue
        values, n_imag, fmin = PO.thermal(fm[b], temps, 0.05)
        for k, key in enumerate(("free_energy", "entropy", "heat_capacity", "energy")):
            worst["thermal"] = max(worst["thermal"], _rel(th[b][key], values[:, k]))
        assert th[b]["n_imaginary"] == n_imag > 0 and th[b]["min_frequency"] == fmin
    print(f"[phonon-kernels] max relative errors {worst}, sweeps {sweeps.min()} .. {sweeps.max()}")
    assert worst["fc"] <= 1e-12 and worst["D"] <= 1e-12 and worst["eig"] <= 1e-11 and worst["thermal"] <= 1e-12


def test_degenerate_spectra(device):
    """A diagonal D (no rotation needed), fcc Gamma triplets and cubic degeneracies of the spring model."""
    from torch_m3gnet_b200.phonon import BatchPhonon

    s_fcc = fcc_conventional()
    s_rs = rock_salt_conventional()
    ph = BatchPhonon(SiteModel("spring", A / np.sqrt(2), device=device), [s_fcc], (2, 2, 2), {29: M1})
    ph.run()
    q = np.array([[0, 0, 0], [0, 0, 0.25], [0.25, 0.25, 0.25], [0.5, 0.5, 0.5], [0.5, 0, 0]])
    out, _, _ = ph._frequencies([q])
    eig = out.eig.cpu().numpy().reshape(len(q), 12)
    st_c = _cpu_state(ph._st)
    worst = 0.0
    for i, qq in enumerate(q):
        Dq = PO.structure_dynmat(st_c, 0, qq)
        worst = max(worst, np.abs(eig[i] - PO.eigenvalues(Dq)).max() / np.linalg.norm(Dq))
    gamma = eig[0]
    assert np.abs(gamma[:3]).max() < 1e-12 * np.abs(gamma).max()
    assert np.ptp(gamma[3:6]) < 1e-6 * gamma.max()                # a triplet at Gamma (float32 forces split it)
    # a diagonal D: Einstein force constants (symmetrize 0), repeated values
    ein = BatchPhonon(SiteModel("einstein", k=2.0, device=device), [s_rs], (1, 1, 1), {29: M1, 6: 12.011},
                      symmetrize=0)
    ein.run()
    out, _, _ = ein._frequencies([random_q(3)])
    lam = out.eig.cpu().numpy().reshape(3, 24)
    assert (out.sweeps.cpu().numpy() == 0).all()
    np.testing.assert_allclose(lam, np.tile(np.repeat([2.0 / M1, 2.0 / 12.011], 12), (3, 1)), rtol=1e-6)
    print(f"[phonon-degenerate] max |dlambda| / ||D||_F {worst:.2e}, Gamma {np.round(gamma, 6)}")
    assert worst <= 1e-11


def test_bitwise_repeat_and_batch_independence(device):
    from torch_m3gnet_b200.phonon import BatchPhonon, mesh_qpoints

    structs, masses = random_structures(seed=3)
    q = random_q(3, seed=2)

    def run(ids, budget):
        ph = BatchPhonon(RandomForces(device), [structs[i] for i in ids], [REPS[i] for i in ids],
                         [masses[i] for i in ids], max_atoms=budget)
        recs = ph.run()
        th = ph.thermal_properties(mesh=(2, 2, 2), temperatures=[0.0, 300.0])
        return recs, ph.frequencies(q), ph.frequencies(mesh_qpoints((2, 2, 2))), th

    probe = 9                                                     # n = 32
    results = []
    for ids, budget in (([probe, 0, 1, 2], None), ([probe, 0, 1, 2], None), ([3, 4, probe], 500), ([probe], 64),
                        ([11, probe, NAN_STRUCT, 7], 300)):
        recs, f, fm, th = run(ids, budget)
        j = ids.index(probe)
        results.append((recs[j]["force_constants"], f[j], fm[j],
                        [th[j][k] for k in ("free_energy", "entropy", "heat_capacity", "energy")]))
    for r in results[1:]:
        assert np.array_equal(r[0], results[0][0]) and np.array_equal(r[1], results[0][1])
        assert np.array_equal(r[2], results[0][2])
        assert all(np.array_equal(a, b) for a, b in zip(r[3], results[0][3]))


def test_spring_model_on_the_device_with_float32_forces(device):
    """Float32 forces: each force component is rounded with relative error <= 2^-24, |F| <= z k h for z bonds, so each
    raw constant is off by <= 2^-24 z k; the acoustic sum puts up to z of those on the self block, and a row of D has
    3 (z + 1) entries per Cartesian column: |dlambda| <= ||dD||_inf <= 3 (2 z) 2^-24 z k / m_min."""
    from torch_m3gnet_b200.phonon import BatchPhonon

    worst_all = []
    for s, masses, r_bond, reps, z in ((fcc_conventional(), {29: M1}, A / np.sqrt(2), (3, 3, 3), 12),
                                       (rock_salt_conventional(), {29: M1, 6: 12.011}, A / 2, (2, 2, 2), 6)):
        ph = BatchPhonon(SiteModel("spring", r_bond, device=device), [s], reps, masses)
        ph.run()
        q = random_q(10, seed=8)
        f = ph.frequencies(q)[0]
        m = np.array([masses[a] for a in s[2]])
        bar = 3 * 2 * z * 2.0 ** -24 * z * K_SPRING / m.min()
        worst = 0.0
        for i in range(len(q)):
            lam = np.sign(f[i]) * (f[i] / PO.THZ) ** 2
            worst = max(worst, np.abs(lam - analytic_eigs(s[0], s[1], m, r_bond, q[i])).max())
        print(f"[phonon-spring-gpu] z={z}: max |dlambda| {worst:.2e} (bar {bar:.2e}) eV/(amu A^2)")
        assert worst <= bar
        worst_all.append(worst)


# ---------------------------------------------------------------------------------------------------------------------
# the model
# ---------------------------------------------------------------------------------------------------------------------

def _c1(device):
    from tests.util import golden, state_dict_of
    from torch_m3gnet_b200 import build_model

    model = build_model(5.0, 4.0, 3, 3, 95, 64, 3, device=device)
    sd = state_dict_of(golden("c1_default"))
    sd = {k: (v * 3 if k.endswith("weight") else v) for k, v in sd.items()}
    model.load_state_dict(sd)
    return model, sd


CU, AL = 29, 13
CU_A = 3.615
MASSES = {CU: 63.546, AL: 26.982}


def model_cells():
    """fcc Cu and L1_2 Cu3Al (conventional cells, 4 atoms)."""
    lat, cart = np.eye(3) * CU_A, np.array([[0, 0, 0], [0, 0.5, 0.5], [0.5, 0, 0.5], [0.5, 0.5, 0]]) * CU_A
    return [(lat, cart, np.full(4, CU)), (lat.copy(), cart.copy(), np.array([AL, CU, CU, CU]))]


def forward64(sd, lat, cart, z):
    """Forces of oracle.forward evaluated in float64 (the one-hot embedding and elemental energies promoted)."""
    from oracle import m3gnet_oracle as O

    hp = O.HyperParams()
    g = O.collate([O.build_graph(lat, cart, z, hp.cutoff, hp.threebody_cutoff)])
    p = {k: v.double() for k, v in sd.items()}
    pos = torch.tensor(np.asarray(cart), dtype=torch.float64, requires_grad=True)
    lattice = torch.tensor(np.asarray(lat), dtype=torch.float64)[None]
    factors = O.bessel_factors(hp.scaled_cutoff, hp.l_max, hp.n_max).double()
    ei, ti = g["edge_index"], g["triplet_edge_index"]
    _, dist, cos = O.pair_geometry(pos / hp.length_scale, lattice / hp.length_scale, g["batch"], ei,
                                   g["edge_cell_shift"], ti)
    x = F.linear(F.one_hot(g["atom_types"], num_classes=hp.num_types).double(), p["model.3.linear.weight"])
    h = O.radial_basis(dist, hp.n_max, hp.scaled_cutoff)
    e = F.silu(F.linear(h.clone(), p["model.5.linear.weight"]))
    tb_idx, cv_idx, ro_idx = O.block_indices(hp)
    for b in range(hp.num_blocks):
        e, _ = O.three_body(p, f"model.{tb_idx[b]}", hp, x, e, dist, cos, ei, ti, factors)
        x, e = O.conv(p, f"model.{cv_idx[b]}", x, e, h, ei)
    elemental = torch.as_tensor(hp.elemental_energies).double()[g["atom_types"]]
    _, _, tot = O.readout(p, f"model.{ro_idx}", x, elemental, g["batch"], 1, hp.energy_scale)
    (gr,) = torch.autograd.grad(tot.sum(), pos)
    return (-gr).numpy()


def test_model_force_constants(device):
    """run() on the model equals the restatement applied to a fresh model evaluation of the same displaced supercells
    in the same chunk layout, and the raw constants of fcc Cu's atom 0 agree with central differences of float64
    oracle forces within max |F_model - F_oracle| / h over those supercells."""
    from torch_m3gnet_b200 import Batch, BatchPhonon, M3GNetCalculator
    from torch_m3gnet_b200.relax import admit

    model, sd = _c1(device)
    calc = M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device)
    cells = model_cells()
    budget = 200
    ph = BatchPhonon(calc, cells, (2, 2, 2), MASSES, max_atoms=budget)
    recs = ph.run()
    jobs = [(b, s) for b in range(2) for s in range(25)]
    sizes = [32] * len(jobs)
    forces, start = [], 0
    while start < len(jobs):
        end = admit(sizes, start, budget, 0, 0)
        sc = [ph._supercell(b, s) for b, s in jobs[start:end]]
        out = model(Batch.from_arrays(np.stack([c[0] for c in sc]), np.concatenate([c[1] for c in sc]),
                                      np.concatenate([c[2] for c in sc]), sizes[start:end], 5.0, 4.0, device=device))
        forces.append(out["forces"].float().cpu().numpy())
        start = end
    assert ph.n_compute_calls == len(forces) > 1
    forces = np.concatenate(forces).reshape(2, 25 * 32, 3)
    for b in range(2):
        want, status, _ = PO.force_constants(forces[b], 4, (2, 2, 2), ph.h, ph.symmetrize)
        assert recs[b]["status"] == "ok" and status == PO.OK
        err = _rel(recs[b]["force_constants"], want)
        print(f"[phonon-model] structure {b}: FC vs restated fresh evaluation {err:.2e}, residual "
              f"{recs[b]['max_residual_force']:.2e} eV/A")
        assert err <= 1e-12
    # raw differences of atom 0 against the float64 oracle
    raw = BatchPhonon(calc, cells[:1], (2, 2, 2), MASSES, symmetrize=0).run()[0]["force_constants"][0]
    f32 = forces[0].reshape(25, 32, 3)
    df, fd = 0.0, np.empty((32, 3, 3))
    for a in range(3):
        f64 = []
        for sign, s in ((1, 1 + 2 * a), (-1, 2 + 2 * a)):
            _, pos, z = ph._supercell(0, s)
            f64.append(forward64(sd, ph._supercell(0, s)[0], pos, z))
            df = max(df, np.abs(f64[-1] - f32[s]).max())
        fd[:, a, :] = -(f64[0] - f64[1]) / (2 * ph.h)
    err = np.abs(raw - fd).max()
    print(f"[phonon-model] raw FC of atom 0 vs float64 oracle differences: {err:.2e} eV/A^2 (bar {df / ph.h:.2e}; "
          f"max |F32 - F64| {df:.2e} eV/A, max |Phi| {np.abs(fd).max():.3f})")
    assert err <= df / ph.h


def test_model_gamma_and_rotation(device):
    from torch_m3gnet_b200 import BatchPhonon, M3GNetCalculator

    model, _ = _c1(device)
    calc = M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device)
    cells = model_cells()
    th = np.random.default_rng(4).normal(size=3)
    ang = np.linalg.norm(th)
    kx = np.array([[0, -th[2], th[1]], [th[2], 0, -th[0]], [-th[1], th[0], 0]]) / ang
    R = np.eye(3) + np.sin(ang) * kx + (1 - np.cos(ang)) * kx @ kx
    rotated = [(lat @ R.T, cart @ R.T, z) for lat, cart, z in cells]
    ph = BatchPhonon(calc, cells + rotated, (2, 2, 2), MASSES)
    assert all(r["status"] == "ok" for r in ph.run())
    gamma = ph.frequencies(np.zeros((1, 3)))
    print(f"[phonon-model] Gamma acoustic |f| {[np.abs(g[0, :3]).max() for g in gamma]} THz, lowest optical "
          f"{[g[0, 3] for g in gamma]} THz")
    for g in gamma:
        assert np.abs(g[0, :3]).max() < 1e-3
    # float32 level: the model's forces carry errors of about EPS_F (6e-7 eV/A against the float64 oracle in
    # test_model_force_constants), so each constant is off by up to EPS_F / h in either run and a row of D (3N entries,
    # masses >= m_min) by 2 x 3N EPS_F / (h m_min)
    eps_f = 1e-6
    bar = 2 * 3 * 32 * eps_f / (ph.h * min(MASSES.values()))
    q = random_q(6, seed=5)
    f = ph.frequencies(q)
    for b in range(2):
        lam, lam_r = (np.sign(x) * (x / PO.THZ) ** 2 for x in (f[b], f[b + 2]))
        err = np.abs(lam - lam_r).max()
        print(f"[phonon-model] structure {b}: rotation changes eigenvalues by {err:.2e} eV/(amu A^2) (bar {bar:.2e}, "
              f"max |lambda| {np.abs(lam).max():.3f})")
        assert err <= bar


def test_abi_cap(device):
    from torch_m3gnet_b200 import _lib
    from torch_m3gnet_b200.phonon import BatchPhonon, MAX_ATOMS

    assert MAX_ATOMS == PO.MAX_ATOMS == 32
    ph = BatchPhonon(RandomForces(device), random_structures()[0][:1], (1, 1, 1), [np.ones(1)])
    ph.run()
    st = ph._st
    q = torch.zeros((1, 3), dtype=torch.float64, device=device)
    q_ptr = torch.tensor([0, 1], dtype=torch.int32, device=device)
    f_ptr = torch.tensor([0, 3], dtype=torch.int64, device=device)
    buf = torch.empty(3, dtype=torch.float64, device=device)
    ibuf = torch.empty(1, dtype=torch.int32, device=device)
    with pytest.raises(RuntimeError, match="atoms per unit cell"):
        _lib.call("phonon_frequencies", st.fc, st.atom_ptr, st.reps, st.pair_ptr, st.sv_ptr, st.sv, st.mass,
                  st.status, q, q_ptr, f_ptr, 1, 1, MAX_ATOMS + 1, 1.0, buf, buf.clone(), ibuf, ibuf.clone())


def test_launch_counts(device):
    from tests.test_gpu_batch_fire import _verlet_model
    from torch_m3gnet_b200 import BatchPhonon, M3GNetCalculator, _lib

    calc = M3GNetCalculator(_verlet_model(device), 5.0, 4.0, skin=0.5, device=device)
    inner = []
    compute = calc.compute

    def counted(*a, **k):
        before = _lib.LAUNCHES
        out = compute(*a, **k)
        inner.append(_lib.LAUNCHES - before)
        return out

    calc.compute = counted
    ph = BatchPhonon(calc, model_cells(), (2, 2, 2), MASSES, max_atoms=300)
    before = _lib.LAUNCHES
    ph.run()
    assert len(inner) == ph.n_compute_calls == 6                  # 50 supercells of 32 atoms, 9 per call
    assert _lib.LAUNCHES - before == sum(inner) + 1
    before = _lib.LAUNCHES
    ph.frequencies(random_q(5))
    assert _lib.LAUNCHES - before == 1
    before = _lib.LAUNCHES
    ph.thermal_properties(mesh=(4, 4, 4), temperatures=[0, 100, 300])
    assert _lib.LAUNCHES - before == 2
