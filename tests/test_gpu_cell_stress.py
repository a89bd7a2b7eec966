"""GPU: the cell stress sigma = (1/V) dE/d(strain) (Gradient.compute_stress, key CELL_STRESS, kernel m3g_bond_virial) on
the whole-step executor and the per-operator path, against the oracle's strain derivative, finite differences on the
device, invariances, determinism, CUDA-graph replay, the calculator's ASE stress and the variable-cell FIRE."""
import numpy as np
import pytest
import torch

from oracle import m3gnet_oracle as O
from tests import strain_oracle as S
from torch_m3gnet_b200.data.material_graph import get_plan
from tests.util import golden, graph_dict, report, state_dict_of, to_batch

pytestmark = pytest.mark.gpu

# Parity bar against the oracle (float32 model vs float32 oracle autograd): |d sigma| <= ATOL + RTOL * max|sigma_ref|.
# Observed worst cases are printed as "[stress-parity]" lines.
ATOL, RTOL = 2e-6, 2e-3


def _build(device, name, scale):
    """(model, oracle graph, oracle params, hyper-parameters, oracle factors) of a golden case; weights x scale."""
    from torch_m3gnet_b200 import build_model

    g = golden(name)
    if name == "small_batch":
        rc = float(g["cutoff"])
        hp = O.HyperParams(cutoff=rc, threebody_cutoff=rc, l_max=2, n_max=3, num_types=93, embedding_dim=17,
                           num_blocks=2)
        sd, fac = state_dict_of(g), torch.from_numpy(g["factors"])
    elif name == "max_lr":
        hp = O.HyperParams(l_max=int(g["l_max"]), n_max=int(g["n_max"]), embedding_dim=int(g["dim"]), num_blocks=1)
        sd, fac = state_dict_of(g), torch.from_numpy(g["factors"])
    else:
        c1 = golden("c1_default")
        hp = O.HyperParams()
        sd, fac = state_dict_of(c1), torch.from_numpy(c1["factors"])
    sd = {k: (v * scale if k.endswith("weight") else v) for k, v in sd.items()}
    model = build_model(hp.cutoff, hp.threebody_cutoff, hp.l_max, hp.n_max, hp.num_types, hp.embedding_dim,
                        hp.num_blocks, device=device)
    model.load_state_dict(sd)
    for m in model.model:
        if hasattr(m, "nsb"):
            m.nsb.factors = fac.to(device)
    return model, graph_dict(g), sd, hp, fac


def _sigma(model, batch, keep_graph=False):
    model.compute_stress = True
    model.keep_graph = keep_graph
    try:
        out = model(batch)
    finally:
        model.compute_stress = False
        model.keep_graph = False
    return out["cell_stress"].detach().clone()


CASES = [("c1_default", 1), ("c1_default", 3), ("tio2_default", 3), ("small_batch", 2), ("max_lr", 1)]


@pytest.mark.parametrize("name,scale", CASES)
def test_parity_with_oracle_strain_derivative(device, name, scale):
    from torch_m3gnet_b200 import engine

    model, gd, sd, hp, fac = _build(device, name, scale)
    ref = S.cell_stress(sd, hp, gd, fac)
    b = to_batch(gd, device)
    eng = _sigma(model, b)
    ran_engine = model.step_engine().supports(b, get_plan(b))
    prev = engine.ENABLED
    engine.ENABLED = False
    try:
        per_op = _sigma(model, to_batch(gd, device))
    finally:
        engine.ENABLED = prev
    kept = _sigma(model, to_batch(gd, device), keep_graph=True)
    scale_ref = ref.abs().max().item()
    worst = max((x.cpu().double() - ref.double()).abs().max().item() for x in (eng, per_op, kept))
    print(f"[stress-parity] {name} x{scale}: engine={ran_engine} max|sigma_ref|={scale_ref:.3e} eV/A^3 "
          f"worst |d|={worst:.3e} rel={worst / max(scale_ref, 1e-30):.2e}")
    for tag, x in (("engine", eng), ("per-op", per_op), ("keep_graph", kept)):
        report(f"{name}x{scale}.sigma.{tag}", x, ref, ATOL, RTOL)
    # the two GPU paths run the same kernel on the same bond gradients up to the adjoint's summation order
    report(f"{name}x{scale}.sigma.engine-vs-per-op", eng, per_op, 1e-7, 1e-4)
    # the outputs of the step are those of the step without the stress
    out = model(to_batch(gd, device))
    b2 = to_batch(gd, device)
    model.compute_stress = True
    out2 = model(b2)
    model.compute_stress = False
    for k in ("total_energy", "forces", "stresses"):
        assert torch.equal(out[k], out2[k]), k


def test_finite_differences_on_device(device):
    """Central differences of total_energy under +-1e-3 strain of positions and lattice on a fixed graph (tolerances of
    test_forces_vs_finite_differences: atol 1e-3, rtol 1e-2 on dE/d(eps) in eV)."""
    model, gd, sd, hp, fac = _build(device, "small_batch", 2)
    b = to_batch(gd, device)
    sigma = _sigma(model, b)
    vol = S.volumes(gd["lattice"]).to(device)
    w = sigma * vol[:, None, None]
    h = 1e-3
    B = w.shape[0]
    for a in range(3):
        for c in range(3):
            eps = torch.zeros((B, 3, 3), dtype=torch.float32)
            eps[:, a, c] = h
            ep = model(to_batch(S.strained(gd, eps), device))["total_energy"]
            em = model(to_batch(S.strained(gd, -eps), device))["total_energy"]
            torch.testing.assert_close(w[:, a, c], (ep - em) / (2 * h), atol=1e-3, rtol=1e-2)


def test_symmetric_translation_and_rotation(device):
    model, gd, sd, hp, fac = _build(device, "c1_default", 3)
    b = to_batch(gd, device)
    s0 = _sigma(model, b)
    r0 = b["stresses"].clone()
    scale = s0.abs().max().item()
    asym = (s0 - s0.transpose(1, 2)).abs().max().item()
    print(f"[stress] max|sigma - sigma^T| = {asym:.2e} (max|sigma| {scale:.2e})")
    assert asym <= 1e-4 * scale
    # the same crystal from another origin: all atoms translated, atom 0 replaced by a periodic image
    from tests.test_cell_stress_cpu import _shifted_copy

    moved = _shifted_copy(gd, 0, [1, -1, 0], [1.7, -2.3, 0.9])
    bm = to_batch(moved, device)
    s1 = _sigma(model, bm)
    assert (s1 - s0).abs().max().item() <= 1e-4 * scale
    assert (bm["stresses"] - r0).abs().max().item() > 10 * (s1 - s0).abs().max().item() + 1e-6
    # rotation: positions and lattice rows r -> r R^T  =>  sigma -> R sigma R^T
    q, _ = np.linalg.qr(np.random.default_rng(3).normal(size=(3, 3)))
    R = torch.from_numpy(q).float()
    rot = dict(gd)
    rot["pos"] = gd["pos"] @ R.T
    rot["lattice"] = gd["lattice"] @ R.T
    s2 = _sigma(model, to_batch(rot, device)).cpu()
    want = R @ s0.cpu()[0] @ R.T
    assert (s2[0] - want).abs().max().item() <= 1e-4 * scale


def test_single_atom_bonded_to_its_own_images(device):
    """Zero forces and zero reference stresses, but a finite strain derivative that matches the oracle."""
    from torch_m3gnet_b200 import Batch

    lat = np.array([[2.6, 0, 0], [0.3, 2.7, 0], [0.1, -0.2, 2.9]])
    cart, z = np.array([[0.1, 0.2, 0.3]]), np.array([29])
    model, _, sd, hp, _ = _build(device, "c1_default", 3)
    for m in model.model:  # the oracle's default Bessel table
        if hasattr(m, "nsb"):
            m.nsb.factors = O.bessel_factors(hp.scaled_cutoff, hp.l_max, hp.n_max).to(device)
    b = Batch.from_arrays(lat[None], cart, z, [1], 5.0, 4.0, device=device)
    sigma = _sigma(model, b)
    assert b["forces"].abs().max().item() <= 1e-6 and b["stresses"].abs().max().item() <= 1e-6
    gd = O.collate([O.build_graph(lat, cart, z, 5.0, 4.0)])
    ref = S.cell_stress(sd, hp, gd)
    print(f"[stress] self-images: sigma diag {sigma[0].diagonal().tolist()}, max|ref| {ref.abs().max().item():.3e}")
    assert ref.abs().max().item() > 1e-4
    report("self_images.sigma", sigma, ref, ATOL, RTOL)


def test_bondless_structure_in_ragged_batch(device):
    from torch_m3gnet_b200 import Batch
    from torch_m3gnet_b200.data.structure import Structure

    big = 30.0 * np.eye(3)
    structs = [(big, np.array([[1.0, 2.0, 3.0]]), np.array([6])),
               (big, np.array([[0.0, 0.0, 0.0], [0.0, 0.0, 2.2]]), np.array([8, 1])),
               O.fcc_supercell(2, jitter=0.05, seed=2)]
    model, _, sd, hp, _ = _build(device, "c1_default", 2)
    for m in model.model:
        if hasattr(m, "nsb"):
            m.nsb.factors = O.bessel_factors(hp.scaled_cutoff, hp.l_max, hp.n_max).to(device)
    b = Batch.from_structures([Structure(l, [int(v) for v in zz], c, coords_are_cartesian=True) for l, c, zz in structs],
                              5.0, 4.0, device=device)
    sigma = _sigma(model, b)
    assert sigma[0].abs().max().item() == 0.0
    gd = O.collate([O.build_graph(l, c, zz, 5.0, 4.0) for l, c, zz in structs])
    report("ragged.sigma", sigma, S.cell_stress(sd, hp, gd), ATOL, RTOL)
    lone = Batch.from_structures([Structure(big, [6], np.array([[1.0, 2.0, 3.0]]), coords_are_cartesian=True)], 5.0,
                                 4.0, device=device)
    s1 = _sigma(model, lone)
    assert s1.shape == (1, 3, 3) and s1.abs().max().item() == 0.0


def test_large_cell_spans_many_chunks(device):
    """A 2 048-atom cell (about 90 000 bonds, dozens of 2 048-bond chunks in one structure) next to a small one: the
    two-stage sum equals a float64 sum of the same bond terms."""
    from torch_m3gnet_b200 import Batch, synthetic
    from torch_m3gnet_b200.nn._functions import cell_stress

    la, ca, za = synthetic.fcc_cu_supercell(8, 0.05, 1)
    lb, cb, zb = synthetic.fcc_cu_supercell(2, 0.05, 2)
    b = Batch.from_arrays(np.stack([lb, la]), np.concatenate([cb, ca]), np.concatenate([zb, za]), [len(cb), len(ca)],
                          5.0, 4.0, device=device)
    plan = get_plan(b)
    E = plan.E
    gen = torch.Generator(device="cpu").manual_seed(0)
    vec = torch.randn(E, 3, generator=gen).double()
    r = vec.norm(dim=1, keepdim=True)
    vec4 = torch.cat([vec, r], 1).float()
    g4 = torch.randn(E, 4, generator=gen).float()
    gd = torch.randn(E, generator=gen).float()
    lat = torch.from_numpy(np.stack([lb, la])).float()
    got = cell_stress(vec4.to(device), g4.to(device), gd.to(device), plan, lat.to(device)).cpu().double()
    v4 = vec4.double()
    ge = g4[:, :3].double() + ((g4[:, 3] + gd).double() / v4[:, 3])[:, None] * v4[:, :3]
    ep = plan.edge_ptr.cpu()[plan.atom_ptr.cpu().long()].long()
    want = torch.stack([(v4[s:t, :3, None] * ge[s:t, None, :]).sum(0) for s, t in zip(ep[:-1], ep[1:])])
    want = want / torch.abs(torch.linalg.det(lat.double()))[:, None, None]
    assert E > 30 * 2048
    report("chunks.sigma", got, want, 1e-7, 1e-5)
    assert torch.equal(cell_stress(vec4.to(device), g4.to(device), gd.to(device), plan, lat.to(device)).cpu(),
                       got.float())


def test_determinism_replay_and_calculator(device):
    from torch_m3gnet_b200 import M3GNetCalculator, synthetic
    from torch_m3gnet_b200.calculator import voigt
    from torch_m3gnet_b200.graphed import GraphedStep

    model, gd, sd, hp, fac = _build(device, "c1_default", 3)
    s1, s2 = _sigma(model, to_batch(gd, device)), _sigma(model, to_batch(gd, device))
    assert torch.equal(s1, s2)
    model.compute_stress = True
    try:
        step = GraphedStep(model, to_batch(gd, device))
        out = step()
        assert torch.equal(out["cell_stress"], s1)
        new_pos = to_batch(gd, device)["pos"] + 0.01
        out = step(pos=new_pos)
        b2 = to_batch(gd, device)
        b2["pos"] = new_pos.clone()
        assert torch.equal(out["cell_stress"], model(b2)["cell_stress"])
    finally:
        model.compute_stress = False
    assert "cell_stress" not in GraphedStep(model, to_batch(gd, device)).out

    class Atoms:
        def __init__(self, cell, positions, numbers):
            self.cell, self.positions, self.numbers = cell, positions, numbers

        def get_cell(self):
            return self.cell

        def get_positions(self):
            return self.positions

        def get_atomic_numbers(self):
            return self.numbers

    lat, cart, z = synthetic.fcc_cu_supercell(2, 0.02, 8)
    calc = M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device, stress=True)
    assert "stress" in calc.implemented_properties
    assert "stress" not in M3GNetCalculator(model, 5.0, 4.0, device=device).implemented_properties
    res = calc.calculate(Atoms(lat, cart, z), ("energy", "forces", "stress"))
    from torch_m3gnet_b200 import Batch

    ref = _sigma(model, Batch.from_arrays(lat[None], cart, z, [len(cart)], 5.0, 4.0, device=device))
    np.testing.assert_array_equal(res["stress"], voigt(ref[0].double().cpu().numpy()))
    assert res["stress"].shape == (6,) and model.compute_stress is False
    e, f, s = calc.compute(lat, cart, z)                       # the 3-tuple is unchanged
    e4, f4, s4, sig = calc.compute(lat, cart, z, with_stress=True)
    assert torch.equal(e, e4) and torch.equal(f, f4) and torch.equal(sig, ref)
    replay = M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device, graph_replay=True, replay_after=2,
                              stress=True)
    rng = np.random.default_rng(2)
    for frame in range(6):
        a = calc.calculate(Atoms(lat, cart, z), ("stress",))["stress"].copy()
        r = replay.calculate(Atoms(lat, cart, z), ("stress",))["stress"]
        np.testing.assert_array_equal(a, r)
        cart = cart + rng.normal(0.0, 0.002, size=cart.shape)
    assert replay.n_replays > 0


def test_launch_count_and_domain_refusal(device):
    from torch_m3gnet_b200 import _lib, domain

    model, gd, sd, hp, fac = _build(device, "c1_default", 1)
    eng = model.step_engine()
    b = to_batch(gd, device)
    model(b)  # plan, weight packing
    l0 = _lib.LAUNCHES
    model(b)
    off = _lib.LAUNCHES - l0
    assert off == eng.launches(True)
    l0 = _lib.LAUNCHES
    _sigma(model, b)
    assert _lib.LAUNCHES - l0 == eng.launches(True, stress=True) == off + 2
    model.compute_stress = True
    try:
        with pytest.raises(NotImplementedError):
            domain.evaluate_emulated(model, [])
        with pytest.raises(NotImplementedError):
            domain.evaluate_distributed(model, None)
        with pytest.raises(NotImplementedError):
            domain.DomainStep(model, None)
    finally:
        model.compute_stress = False


def test_variable_cell_relaxation_of_strained_fcc_cu(device):
    """A perfect 32-atom fcc Cu cell under a 3 % tetragonal strain relaxes back toward cubic with Fire(relax_cell=True),
    with the pressure set to -tr(sigma)/3 of the cubic cell so that the cubic cell is stationary.  Weights: c1_default
    x3 with the model's own Bessel table -- E + pV has a minimum there (tetragonal curvature about +590 eV measured on a
    B200), whereas e.g. the seed-11 x2 / x3 weights of the Verlet tests have none near the cubic cell."""
    from torch_m3gnet_b200 import Fire, M3GNetCalculator, build_model, synthetic

    model = build_model(5.0, 4.0, 3, 3, 95, 64, 3, device=device)  # the model's own Bessel table
    model.load_state_dict({k: (v * 3 if k.endswith("weight") else v) for k, v in state_dict_of(golden("c1_default")).items()})
    lat0, cart0, z = synthetic.fcc_cu_supercell(2, 0.0, 0)
    calc = M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device)
    sig = calc.compute(lat0, cart0, z, with_stress=True)[3][0].double().cpu().numpy()
    p = -float(np.trace(sig)) / 3
    strain = np.diag([1.03, 1.0, 1.0])
    opt = Fire(calc, lat0 @ strain, cart0 @ strain, z, relax_cell=True, pressure=p)
    f0 = opt.fmax()
    ok = opt.run(fmax=0.05, steps=150)
    L = opt.lattice[0]
    tet0 = 0.03 * lat0[0, 0]
    tet = abs(L[0, 0] - L[1, 1])
    frac = opt.pos.cpu().numpy() @ np.linalg.inv(L)
    dev_sites = frac - cart0 / lat0[0, 0]
    dev_sites -= np.round(dev_sites)
    print(f"[vc-fire] p={p:.3e} eV/A^3, fmax {f0:.3f} -> {opt.fmax():.4f} eV/A in {opt.n_steps} steps, cell diag "
          f"{np.diag(L)}, |Lxx-Lyy| {tet0:.4f} -> {tet:.4f} A")
    assert ok and opt.fmax() < 0.05
    assert np.abs(L - np.diag(np.diag(L))).max() < 1e-5       # off-diagonal cell terms stay 0
    assert abs(L[1, 1] - L[2, 2]) < 1e-5                       # the two unstrained axes stay equal
    assert np.abs(dev_sites).max() < 1e-5                       # atoms stay on their fcc sites
    assert tet < 0.25 * tet0                                    # back toward cubic
