"""CPU: the numpy restatement of the NPT step (tests/npt_oracle.py) -- bit for bit the fixed-cell step
(tests/md_oracle.py) at zero compressibility, the exact volume distribution of an ideal gas, and the exact per-axis
distribution of an ideal gas with a harmonic energy on the axis lengths -- and the host side of BatchMD(pressure=...)
(results in input order, independence from the chunk budget, failures frozen with their cells, input validation, no
stress requested without a pressure) with the restatement standing in for the kernels and a periodic Lennard-Jones
calculator on the CPU."""
import numpy as np
import pytest
import torch

from tests import md_oracle as MO
from tests import npt_oracle as NO
from tests.test_batch_fire_cpu import BatchLJ, lj_structures
from tests.test_batch_md_cpu import AR, _oracle_mb, _oracle_step


def _oracle_npt_step(st, forces, sigma, energy, dt, max_step_move, seed, advance, slot, obs, coupling,
                     max_step_strain):
    """md.langevin_npt_step with the numpy restatement in place of the kernel (CPU tensors)."""
    d = {k: getattr(st, k).numpy().copy() for k in NO.STATE_KEYS}
    o = obs.numpy().copy()
    NO.npt_step(d, forces.double().numpy(), sigma.double().numpy(), energy.double().numpy(), st.atom_ptr.numpy(), dt,
                max_step_move, MO.seed_word(seed), advance, slot, o, coupling, max_step_strain)
    for k, val in d.items():
        getattr(st, k).copy_(torch.from_numpy(val))
    obs.copy_(torch.from_numpy(o))


@pytest.fixture
def restated(monkeypatch):
    from torch_m3gnet_b200 import md

    monkeypatch.setattr(md, "langevin_step", _oracle_step)
    monkeypatch.setattr(md, "langevin_npt_step", _oracle_npt_step)
    monkeypatch.setattr(md, "maxwell_boltzmann", _oracle_mb)
    return md


def block_mean(x, nb=20):
    """Mean of the time series x (frames first) and its standard error from nb contiguous blocks."""
    x = np.asarray(x, dtype=np.float64)
    x = x[: len(x) // nb * nb]
    blocks = x.reshape(nb, -1, *x.shape[1:]).mean(axis=1)
    return blocks.mean(axis=0), blocks.std(axis=0, ddof=1) / np.sqrt(nb)


def test_zero_compressibility_is_the_fixed_cell_step():
    """beta_T = 0: mu = exp(0) = 1, every scaling is a multiplication by 1, and the restatement is md_oracle's step bit
    for bit over 100 steps: positions, velocities, bath, steps, statuses and observables; the cells do not move."""
    structs = lj_structures(5, seed=20)                  # sizes [4, 32, 4, 4, 32]
    calc = BatchLJ()
    carts = [s[1] for s in structs]
    lat = np.stack([s[0] for s in structs])
    z = np.concatenate([s[2] for s in structs])
    sizes = [len(c) for c in carts]
    masses = [np.full(len(c), AR) for c in carts]
    temps = [60.0, 120.0, 200.0, 90.0, 150.0]
    ref, ptr = MO.fresh_state(carts, masses, temps, 0.02, 2.0, ids=[4, 0, 9, 2, 7])
    MO.maxwell_boltzmann(ref, ptr, 5)
    got, _ = NO.fresh_state(carts, lat, masses, temps, 0.02, 2.0, [0.0, 0.01, -0.02, 0.0, 0.003], 0.0, 500.0,
                            ids=[4, 0, 9, 2, 7])
    got["v"][:] = ref["v"]
    steps = 100
    obs_ref, obs_got = np.zeros((steps + 1, 5, 4)), np.zeros((steps + 1, 5, 6))
    for k in range(steps + 1):
        e, f, _, s = calc.compute(lat, ref["pos"], z, sizes, with_stress=True)
        MO.langevin_step(ref, f.numpy(), e.double().numpy(), ptr, 2.0, 0.5, 11, k < steps, k, obs_ref)
        NO.npt_step(got, f.numpy(), s.numpy(), e.double().numpy(), ptr, 2.0, 0.5, 11, k < steps, k, obs_got,
                    NO.ISOTROPIC, 0.01)
        for key in MO.STATE_KEYS:
            assert np.array_equal(got[key], ref[key]), (k, key)
    assert (ref["status"] == 0).all() and (ref["step"] == steps).all()
    assert np.array_equal(obs_got[..., :4], obs_ref)
    assert np.array_equal(got["lattice"], lat)
    assert np.array_equal(obs_got[..., 4], np.broadcast_to(NO.volume(lat), (steps + 1, 5)))


def _ideal_gas(coupling, T, P0, beta_T, sizes, steps, seed, harmonic=None):
    """NPT restatement on structures without interactions (zero forces; zero stress, or the stress of the harmonic axis
    energy E = sum_a kappa / 2 (L_a - L0)^2 on diagonal cells, sigma_aa = kappa (L_a - L0) L_a / V); dt 1 fs,
    tau_p = 100 dt, friction 0.05 / fs.  Per recorded step: (V, L_xx, L_yy, L_zz) per structure."""
    S = len(sizes)
    kT = MO.KB * np.asarray(T)
    V0 = np.asarray(sizes) * kT / np.asarray(P0)
    lats = [np.eye(3) * v ** (1 / 3) for v in V0] if harmonic is None else [np.eye(3) * harmonic[1]] * S
    rng = np.random.default_rng(seed)
    carts = [rng.uniform(0, 4, (n, 3)) for n in sizes]
    st, ptr = NO.fresh_state(carts, lats, [np.full(n, 12.0) for n in sizes], T, 0.05, 1.0, P0, beta_T, 100.0)
    MO.maxwell_boltzmann(st, ptr, seed)
    f, e = np.zeros((int(ptr[-1]), 3)), np.zeros(S)
    obs = np.zeros((1, S, NO.obs_width(coupling)))
    out = np.zeros((steps, S, 4))
    for k in range(steps):
        L = st["lattice"]
        diag = np.stack([L[:, 0, 0], L[:, 1, 1], L[:, 2, 2]], axis=1)
        sig = np.zeros((S, 3, 3))
        if harmonic is not None:
            kappa, L0 = harmonic
            s = kappa * (diag - L0) * diag / NO.volume(L)[:, None]
            sig[:, [0, 1, 2], [0, 1, 2]] = s.astype(np.float32)
        NO.npt_step(st, f, sig, e, ptr, 1.0, 0.5, seed, True, 0, obs, coupling, 10.0)
        out[k, :, 0] = obs[0, :, 4]
        out[k, :, 1:] = diag
    assert (st["status"] == 0).all()
    return out


def test_ideal_gas_volume_is_gamma_distributed():
    """Isotropic stochastic cell rescaling of an ideal gas of n atoms (centre of mass fixed, so n - 1 relative
    positions) samples p(V) ~ V^(n-1) exp(-P0 V / kT): <V> = n kT / P0 and var V = n (kT / P0)^2.  Two groups at
    different temperature, pressure and compressibility (beta_T P0 = 1) share the batch.  Over 1.8e4 steps the block
    standard error of var V is about 1 % here (observed 1.001-1.031 across seeds and masses), so var V is held to 4 of
    them and 4 %; the GPU test, with more structures and steps, holds it tighter."""
    S, n = 256, 8
    grp = np.arange(S) % 2
    T, P0 = np.where(grp == 0, 300.0, 600.0), np.where(grp == 0, 0.002, 0.005)
    out = _ideal_gas(NO.ISOTROPIC, T, P0, 1.0 / P0, [n] * S, 20000, seed=3)[2000:]
    for g in (0, 1):
        scale = n * MO.KB * T[g] / P0[g]
        x = out[:, grp == g, 0] / scale                 # V / <V>_exact
        mean, se = block_mean(x.mean(axis=1))
        var, var_se = block_mean(((x - 1.0) ** 2).mean(axis=1) * n)   # var V / (n (kT/P0)^2), about the exact mean
        print(f"[npt-oracle] ideal gas T={T[g]:.0f} K P0={P0[g]} eV/A^3: <V> / (n kT/P0) = {mean:.4f} +- {se:.4f}, "
              f"var V / (n (kT/P0)^2) = {var:.4f} +- {var_se:.4f}")
        assert abs(mean - 1) < 4 * se and abs(mean - 1) < 0.01
        assert abs(var - 1) < 4 * var_se and abs(var - 1) < 0.04


def _axis_quadrature(n, kT, P0, kappa, L0, lo, hi, m=240):
    """<L_a>, <V> and var V under p(L) ~ prod L_a^(n-1) exp(-(E + P0 V) / kT), E = sum_a kappa / 2 (L_a - L0)^2."""
    g = np.linspace(lo, hi, m)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    V = X * Y * Z
    logw = (n - 1) * np.log(V) - (0.5 * kappa * ((X - L0) ** 2 + (Y - L0) ** 2 + (Z - L0) ** 2) + P0 * V) / kT
    w = np.exp(logw - logw.max())
    w /= w.sum()
    mv = (w * V).sum()
    return (w * X).sum(), mv, (w * V * V).sum() - mv * mv


def test_per_axis_harmonic_cell_matches_quadrature():
    """Per-axis coupling samples p(L_x, L_y, L_z) ~ prod L_a^(n-1) exp(-(E + P0 V) / kT) on diagonal cells.  An ideal
    gas alone has no normalisable per-axis density, so a harmonic energy on the axis lengths holds the shape; in units
    of kT and 2 A: kappa = 4, L0 = 2, P0 = 1, beta_T P0 = 0.5."""
    S, n = 256, 8
    kT = MO.KB * 300.0
    ell = 2.0
    P0, kappa, L0 = kT / ell ** 3, 4 * kT / ell ** 2, 2 * ell
    out = _ideal_gas(NO.PER_AXIS, 300.0, P0, 0.5 / P0, [n] * S, 20000, seed=4, harmonic=(kappa, L0))[2000:]
    want_l, want_v, want_var = _axis_quadrature(n, kT, P0, kappa, L0, 0.05 * L0, 3.0 * L0)
    mean_l, se_l = block_mean(out[:, :, 1:].mean(axis=(1, 2)))
    mean_v, se_v = block_mean(out[:, :, 0].mean(axis=1))
    var_v, se_var = block_mean(((out[:, :, 0] - want_v) ** 2).mean(axis=1))
    print(f"[npt-oracle] per axis: <L_a> {mean_l:.4f} +- {se_l:.4f} (exact {want_l:.4f}), <V> {mean_v:.3f} +- "
          f"{se_v:.3f} (exact {want_v:.3f}), var V {var_v:.3f} +- {se_var:.3f} (exact {want_var:.3f})")
    assert abs(mean_l - want_l) < 4 * se_l and abs(mean_l / want_l - 1) < 0.005
    assert abs(mean_v - want_v) < 4 * se_v and abs(mean_v / want_v - 1) < 0.005
    assert abs(var_v / want_var - 1) < 0.02


class StressLJ(BatchLJ):
    """BatchLJ that records ``with_stress`` of every call; NaN forces for atom rows [lo, hi) or a NaN stress for
    structure ``sigma_nan`` from call ``at`` on."""

    def __init__(self, lo=0, hi=0, at=None, sigma_nan=None):
        super().__init__()
        self.lo, self.hi, self.at, self.sigma_nan = lo, hi, at, sigma_nan
        self.stress_flags = []

    def compute(self, *a, with_stress=False, **k):
        self.stress_flags.append(with_stress)
        out = super().compute(*a, with_stress=with_stress, **k)
        if self.at is not None and len(self.calls) > self.at:
            out[1][self.lo:self.hi] = float("nan")
            if self.sigma_nan is not None and with_stress:
                out[3][self.sigma_nan, 1, 2] = float("nan")
        return out


def _run_npt(md, structs, calc=None, **kw):
    args = dict(masses={18: AR}, temperature=[80.0, 150.0, 300.0, 60.0, 200.0, 100.0][:len(structs)],
                friction=0.02, dt=2.0, seed=2 ** 63 + 9, pressure=[0.0, 0.002, -0.001, 0.01, 0.0, 0.004][:len(structs)],
                barostat_time=1000.0)
    args.update(kw)
    calc = calc or StressLJ()
    res = md.BatchMD(calc, structs, **args).run(30, record_every=5, trajectory_every=10)
    return res, calc


NPT_KEYS = {"status", "n_steps", "times", "energy", "kinetic_energy", "temperature", "bath", "positions", "velocities",
            "lattice", "trajectory", "volume", "pressure", "lattice_trajectory"}


@pytest.mark.parametrize("coupling", ["isotropic", "per_axis"])
def test_npt_results_in_input_order_and_independent_of_the_budget(restated, coupling):
    structs = lj_structures(6, seed=21)                  # sizes [4, 32, 4, 4, 32, 4]
    full, calc = _run_npt(restated, structs, coupling=coupling)
    assert all(calc.stress_flags) and len(calc.calls) == 31
    keys = NPT_KEYS | ({"axis_pressure"} if coupling == "per_axis" else set())
    for max_atoms in (12, 3):
        other, _ = _run_npt(restated, structs, coupling=coupling, max_atoms=max_atoms)
        for i, s in enumerate(structs):
            a = full[i]
            assert a.keys() == keys and a["status"] == "completed" and a["n_steps"] == 30
            for k in a:
                assert np.array_equal(np.asarray(a[k]), np.asarray(other[i][k])), (max_atoms, i, k)
    for i, (s, a) in enumerate(zip(structs, full)):
        lt = a["lattice_trajectory"]
        assert lt.shape == (4, 3, 3) and np.array_equal(lt[0], s[0]) and not np.array_equal(a["lattice"], s[0])
        # frames 0, 10, 20, 30 of the trajectory are recorded frames 0, 2, 4, 6
        assert np.allclose(a["volume"][::2], np.abs(np.linalg.det(lt)), rtol=1e-13, atol=0)
        if coupling == "isotropic":                     # one scale per step: the cell keeps its shape
            nz = np.abs(s[0]) > 1e-9
            ratio = a["lattice"][nz] / s[0][nz]
            assert np.allclose(ratio, ratio[0], rtol=1e-12, atol=0) and np.array_equal(a["lattice"][~nz], s[0][~nz])
        if coupling == "per_axis":
            assert a["axis_pressure"].shape == (7, 3)
            assert np.allclose(a["axis_pressure"].mean(axis=1), a["pressure"], rtol=1e-9, atol=1e-12)


def test_npt_failures_are_frozen_with_their_cells(restated):
    structs = lj_structures(4, seed=22)                  # sizes [4, 32, 4, 4]
    kw = dict(masses=[np.full(len(s[2]), AR) for s in structs], temperature=100.0, dt=2.0, seed=4, pressure=0.001,
              barostat_time=100.0)
    ref = restated.BatchMD(StressLJ(), structs, **kw).run(20, record_every=3, trajectory_every=1)
    # NaN forces on structure 1 from frame 13 on; a NaN stress on structure 3 from frame 13 on
    got = restated.BatchMD(StressLJ(4, 36, 13, sigma_nan=3), structs, **kw).run(20, record_every=3,
                                                                                  trajectory_every=1)
    for b in (1, 3):
        bad = got[b]
        assert bad["status"] == "failed" and bad["n_steps"] == 13
        for k in ("energy", "kinetic_energy", "temperature", "bath", "volume", "pressure"):
            assert np.array_equal(bad[k], ref[b][k][:5]), (b, k)
        assert np.array_equal(bad["trajectory"], ref[b]["trajectory"][:14])
        assert np.array_equal(bad["lattice_trajectory"], ref[b]["lattice_trajectory"][:14])
        assert np.array_equal(bad["lattice"], ref[b]["lattice_trajectory"][13])    # the cell of the frame that failed
        assert np.array_equal(bad["positions"], ref[b]["trajectory"][13])
    for i in (0, 2):
        for k in ref[i]:
            assert np.array_equal(np.asarray(ref[i][k]), np.asarray(got[i][k])), (i, k)
    # the strain guard: a structure whose log-scale step would exceed max_step_strain fails at frame 0, alone
    soft = dict(kw, compressibility=[1.6021766208, 1.6021766208, 30.0, 1.6021766208])
    res = restated.BatchMD(StressLJ(), structs, **soft).run(20, record_every=3, trajectory_every=1)
    assert res[2]["status"] == "failed" and res[2]["n_steps"] == 0 and res[2]["volume"].size == 0
    assert np.array_equal(res[2]["lattice"], structs[2][0]) and np.array_equal(res[2]["positions"], structs[2][1])
    for i in (0, 1, 3):
        for k in ref[i]:
            assert np.array_equal(np.asarray(ref[i][k]), np.asarray(res[i][k])), (i, k)
    # a looser bound lets it run
    loose = restated.BatchMD(StressLJ(), structs[2:3], **dict(soft, masses={18: AR}, compressibility=30.0,
                                                             max_step_strain=0.5)).run(3)
    assert loose[0]["status"] == "completed"


def test_no_stress_is_requested_without_a_pressure(restated):
    structs = lj_structures(3, seed=23)
    calc = StressLJ()
    res = restated.BatchMD(calc, structs, {18: AR}, 100.0, dt=2.0).run(5, trajectory_every=5)
    assert len(calc.stress_flags) == 6 and not any(calc.stress_flags)
    assert {"volume", "pressure", "axis_pressure", "lattice_trajectory"}.isdisjoint(res[0])


def test_npt_validation():
    from torch_m3gnet_b200 import BatchMD

    structs = lj_structures(2, seed=24)
    m = {18: AR}
    with pytest.raises(ValueError, match="pressure"):
        BatchMD(BatchLJ(), structs, m, 300.0, pressure=np.nan)
    with pytest.raises(ValueError, match="pressure"):
        BatchMD(BatchLJ(), structs, m, 300.0, pressure=[0.0, np.inf])
    with pytest.raises(ValueError, match="pressure"):
        BatchMD(BatchLJ(), structs, m, 300.0, pressure=[0.0, 0.0, 0.0])
    with pytest.raises(ValueError, match="compressibility"):
        BatchMD(BatchLJ(), structs, m, 300.0, pressure=0.0, compressibility=0.0)
    with pytest.raises(ValueError, match="compressibility"):
        BatchMD(BatchLJ(), structs, m, 300.0, pressure=0.0, compressibility=[1.0, -1.0])
    with pytest.raises(ValueError, match="barostat_time"):
        BatchMD(BatchLJ(), structs, m, 300.0, pressure=0.0, barostat_time=0.0)
    with pytest.raises(ValueError, match="barostat_time"):
        BatchMD(BatchLJ(), structs, m, 300.0, pressure=0.0, barostat_time=np.nan)
    with pytest.raises(ValueError, match="coupling"):
        BatchMD(BatchLJ(), structs, m, 300.0, pressure=0.0, coupling="anisotropic")
    with pytest.raises(ValueError, match="max_step_strain"):
        BatchMD(BatchLJ(), structs, m, 300.0, pressure=0.0, max_step_strain=0.0)
    with pytest.raises(ValueError, match="max_step_strain"):
        BatchMD(BatchLJ(), structs, m, 300.0, pressure=0.0, max_step_strain=-0.1)
    md = BatchMD(BatchLJ(), structs, m, 300.0, pressure=[-0.01, 0.02])      # negative pressures are allowed
    assert md.pressure.tolist() == [-0.01, 0.02] and md.compressibility[0] == pytest.approx(1.6021766, rel=1e-7)
