"""GPU: the batched NEB step (m3g_neb_step, csrc/neb.cu) against its numpy restatement (tests/neb_oracle.py), batch
independence, BatchNEB on device Mueller-Brown and Lennard-Jones calculators against the restatement-driven runs and
their known saddles, model runs against a fresh evaluation, the image cap and the launch count."""
import types

import numpy as np
import pytest
import torch

from tests import fire_oracle as FO
from tests import neb_oracle as NO
from tests.test_batch_fire_cpu import BatchLJ
from tests.test_batch_neb_cpu import (BRANCH_E, MB_MIN_A, MB_MIN_B, BatchMB, check_lj_saddle, check_mb_saddle,
                                      fire_relax_restated, lj_vacancy_hop, mb_point, oracle_step)

pytestmark = pytest.mark.gpu

F64_KEYS = ("pos", "v", "dt", "a", "fmax", "e_frame")
I32_KEYS = ("n_pos", "n_steps", "status", "i_climb")
FIRE = dict(FO.FIRE_DEFAULTS)


def _layout(n, M):
    cum = lambda c: np.concatenate([[0], np.cumsum(c)]).astype(np.int64)  # noqa: E731
    return cum([m * k for m, k in zip(M, n)]), cum(M), cum([2 * k for k in n])


def _kernel(st, inp, device, climb, fmax=1e-3, steps=50):
    from torch_m3gnet_b200 import neb

    d = types.SimpleNamespace(**{k: torch.as_tensor(np.ascontiguousarray(v)).to(device) for k, v in st.items()})
    for k in ("row_ptr", "image_ptr", "end_ptr"):
        setattr(d, k, torch.as_tensor(inp[k].astype(np.int32)).to(device))
    for k in ("ends", "e_end", "k"):
        setattr(d, k, torch.as_tensor(inp[k]).to(device))
    d.M, d.B = list(inp["M"]), len(inp["M"])
    neb.neb_step(d, torch.as_tensor(inp["forces"]).to(device), torch.as_tensor(inp["energy"]).to(device), climb, FIRE,
                 fmax, steps)
    torch.cuda.synchronize()
    return {k: getattr(d, k).cpu().numpy() for k in st}


def _oracle(st, inp, climb, fmax=1e-3, steps=50):
    want = {k: v.copy() for k, v in st.items()}
    NO.neb_step(want, inp["forces"].astype(np.float64), inp["energy"].astype(np.float64), inp["ends"], inp["e_end"],
                inp["k"], climb, FIRE, fmax, steps, inp["row_ptr"], inp["image_ptr"], inp["end_ptr"])
    return want


# (atoms per image, interior images) of the random case's bands
BANDS = [(3, 5), (1, 1), (31, 5), (60, 5), (2, 9), (4, 2), (5, 3), (7, 4), (2, 3), (1, 64), (3, 2), (6, 3), (2, 2),
         (9, 3)]
DEGENERATE, NAN_FORCE, NAN_ENERGY, FINISHED, AT_LIMIT, STRAIGHT = 6, 7, 8, (10, 11, 12), 2, 13


def _random_case(seed=0):
    """Random ragged bands: both power signs, the max_move clip on and off, every tangent branch (band 4 has the
    branch-test energies), a degenerate tangent, a non-finite force and energy, finished bands, one at its step limit
    and a straight, evenly spaced band without forces (converged)."""
    rng = np.random.default_rng(seed)
    n = [b[0] for b in BANDS]
    M = [b[1] for b in BANDS]
    row_ptr, image_ptr, end_ptr = _layout(n, M)
    B = len(BANDS)
    ends = rng.normal(0, 2.0, (end_ptr[-1], 3))
    pos = np.empty((row_ptr[-1], 3))
    for b in range(B):                               # a jittered path between the endpoints
        e = ends[end_ptr[b]:end_ptr[b + 1]].reshape(2, n[b], 3)
        t = np.arange(1, M[b] + 1)[:, None, None] / (M[b] + 1)
        path = (1 - t) * e[0] + t * e[1] + rng.normal(0, 0.1, (M[b], n[b], 3))
        pos[row_ptr[b]:row_ptr[b + 1]] = path.reshape(-1, 3)
    forces = rng.normal(0, 0.3, (row_ptr[-1], 3)).astype(np.float32)
    energy = rng.normal(-3, 1, image_ptr[-1]).astype(np.float32)
    e_end = rng.normal(-3.5, 0.3, (B, 2))
    k = rng.uniform(0.0, 0.5, B)
    energy[image_ptr[4]:image_ptr[5]] = BRANCH_E[1:-1]
    e_end[4] = BRANCH_E[0], BRANCH_E[-1]
    s = DEGENERATE                                   # falling energies and t- = 0 at image 2
    energy[image_ptr[s]:image_ptr[s + 1]] = [-1.0, -2.0, -3.0]
    e_end[s] = 0.0, -4.0
    pos[row_ptr[s] + n[s]:row_ptr[s] + 2 * n[s]] = pos[row_ptr[s]:row_ptr[s] + n[s]]
    forces[row_ptr[NAN_FORCE] + 3, 1] = np.nan
    energy[image_ptr[NAN_ENERGY] + 1] = np.inf
    s = STRAIGHT
    e = ends[end_ptr[s]:end_ptr[s + 1]].reshape(2, n[s], 3)
    t = np.arange(1, M[s] + 1)[:, None, None] / (M[s] + 1)
    pos[row_ptr[s]:row_ptr[s + 1]] = ((1 - t) * e[0] + t * e[1]).reshape(-1, 3)
    forces[row_ptr[s]:row_ptr[s + 1]] = 0.0
    for b in (1, 5):
        forces[row_ptr[b]:row_ptr[b + 1]] *= 300.0  # big steps: the max_move clip
    inp = dict(forces=forces, energy=energy, ends=ends, e_end=e_end, k=k, row_ptr=row_ptr, image_ptr=image_ptr,
               end_ptr=end_ptr, M=M, n=n)
    st = dict(pos=pos, v=np.zeros_like(pos), dt=rng.uniform(0.05, 0.5, B), a=rng.uniform(0.05, 0.1, B),
              fmax=np.zeros(B), n_pos=rng.integers(0, 9, B).astype(np.int32),
              n_steps=rng.integers(0, 40, B).astype(np.int32), status=np.zeros(B, np.int32),
              i_climb=np.zeros(B, np.int32), e_frame=np.zeros(image_ptr[-1]))
    st["status"][list(FINISHED)] = NO.CONVERGED, NO.NOT_CONVERGED, NO.FAILED
    st["n_steps"][AT_LIMIT] = 50
    st["n_pos"][0], st["n_pos"][3] = 8, 7
    st["dt"][[1, 5]] = 0.5
    for b in range(B):                               # velocities along +-G: both power signs
        r0, r1 = row_ptr[b], row_ptr[b + 1]
        E = np.concatenate([[e_end[b][0]], energy[image_ptr[b]:image_ptr[b + 1]].astype(np.float64), [e_end[b][1]]])
        R = np.concatenate([ends[end_ptr[b]:end_ptr[b] + n[b]][None], pos[r0:r1].reshape(M[b], n[b], 3),
                            ends[end_ptr[b] + n[b]:end_ptr[b + 1]][None]])
        with np.errstate(invalid="ignore"):
            G, _, _ = NO.neb_forces(E, R, forces[r0:r1].astype(np.float64).reshape(M[b], n[b], 3), k[b], True)
        sign = 1.0 if b % 2 == 0 else -1.0
        g = np.nan_to_num(G.reshape(-1, 3))
        st["v"][r0:r1] = sign * rng.uniform(0.0, 0.05, (r1 - r0, 3)) * np.sign(g)
    return st, inp


@pytest.mark.parametrize("climb", [False, True])
def test_kernel_matches_the_restatement(device, climb):
    st, inp = _random_case()
    want = _oracle(st, inp, climb)
    got = _kernel(st, inp, device, climb)
    again = _kernel(st, inp, device, climb)
    for k in st:
        assert np.array_equal(got[k], again[k], equal_nan=True), k  # repeated calls are bitwise equal
    for k in I32_KEYS:
        assert np.array_equal(got[k], want[k]), (k, got[k], want[k])
    for k in F64_KEYS:
        scale = max(np.abs(want[k][np.isfinite(want[k])]).max(initial=0.0), 1e-300)
        np.testing.assert_allclose(got[k], want[k], rtol=1e-12, atol=1e-12 * scale, err_msg=k)
    rp, ip = inp["row_ptr"], inp["image_ptr"]
    for b in FINISHED:                                              # finished: bit-untouched
        assert np.array_equal(got["pos"][rp[b]:rp[b + 1]], st["pos"][rp[b]:rp[b + 1]])
        assert np.array_equal(got["v"][rp[b]:rp[b + 1]], st["v"][rp[b]:rp[b + 1]])
        assert np.array_equal(got["e_frame"][ip[b]:ip[b + 1]], st["e_frame"][ip[b]:ip[b + 1]])
        for k in ("dt", "a", "fmax", "n_pos", "n_steps", "status", "i_climb"):
            assert np.array_equal(got[k][b], st[k][b]), (b, k)
    status = want["status"]
    assert status[DEGENERATE] == status[NAN_FORCE] == status[NAN_ENERGY] == NO.FAILED
    assert status[AT_LIMIT] == NO.NOT_CONVERGED and status[STRAIGHT] == NO.CONVERGED
    assert want["i_climb"][4] == 7                                  # the tie in the branch band: the lower index
    moved = [b for b in range(len(BANDS)) if want["n_steps"][b] > st["n_steps"][b]]
    positive = [b for b in moved if want["n_pos"][b] == st["n_pos"][b] + 1]
    assert positive and len(positive) < len(moved)
    assert any(st["n_pos"][b] > FIRE["n_min"] for b in positive)
    for b in (1, 5):                                                # the clip
        dr = want["pos"][rp[b]:rp[b + 1]] - st["pos"][rp[b]:rp[b + 1]]
        assert np.sqrt((dr * dr).sum()) == pytest.approx(FIRE["max_move"], rel=1e-9)
    assert 4 in moved and 3 in moved and BANDS[3][0] * BANDS[3][1] > 256 and 1 in moved


def test_a_band_steps_the_same_anywhere_in_the_batch(device):
    st, inp = _random_case(seed=3)
    probe = 3                                                       # the 300-row band
    results = []
    for order in ([3, 0, 1, 2, 4, 5], [9, 4, 3, 12], [3], [0, 1, 2, 5, 13, 3]):
        n = [inp["n"][b] for b in order]
        M = [inp["M"][b] for b in order]
        row_ptr, image_ptr, end_ptr = _layout(n, M)
        pick = lambda p, x: np.concatenate([x[p[b]:p[b + 1]] for b in order])  # noqa: E731
        sub_inp = dict(forces=pick(inp["row_ptr"], inp["forces"]), energy=pick(inp["image_ptr"], inp["energy"]),
                       ends=pick(inp["end_ptr"], inp["ends"]), e_end=inp["e_end"][order], k=inp["k"][order],
                       row_ptr=row_ptr, image_ptr=image_ptr, end_ptr=end_ptr, M=M, n=n)
        sub = dict(pos=pick(inp["row_ptr"], st["pos"]), v=pick(inp["row_ptr"], st["v"]),
                   e_frame=pick(inp["image_ptr"], st["e_frame"]),
                   **{k: st[k][order] for k in ("dt", "a", "fmax", "n_pos", "n_steps", "status", "i_climb")})
        out = _kernel(sub, sub_inp, device, True)
        j = order.index(probe)
        results.append(dict(pos=out["pos"][row_ptr[j]:row_ptr[j + 1]], v=out["v"][row_ptr[j]:row_ptr[j + 1]],
                            e_frame=out["e_frame"][image_ptr[j]:image_ptr[j + 1]],
                            **{k: out[k][j] for k in ("dt", "a", "fmax", "n_pos", "n_steps", "status", "i_climb")}))
    for r in results[1:]:
        for k in r:
            assert np.array_equal(r[k], results[0][k]), k


def test_image_cap_is_checked_by_the_abi(device):
    from torch_m3gnet_b200 import _lib

    st, inp = _random_case()
    d = {k: torch.as_tensor(np.ascontiguousarray(v)).to(device) for k, v in {**st, **inp}.items()
         if k not in ("M", "n")}
    for k in ("row_ptr", "image_ptr", "end_ptr"):
        d[k] = d[k].to(torch.int32)
    with pytest.raises(RuntimeError, match="interior images"):
        _lib.call("neb_step", d["forces"], d["energy"], d["row_ptr"], d["image_ptr"], d["end_ptr"], len(BANDS),
                  NO.MAX_IMAGES + 1, d["ends"], d["e_end"], d["k"], 1, 1.0, 0.2, 5, 1.1, 0.5, 0.1, 0.99, 1e-3, 50,
                  d["pos"], d["v"], d["dt"], d["a"], d["n_pos"], d["n_steps"], d["status"], d["fmax"], d["i_climb"],
                  d["e_frame"])
    from torch_m3gnet_b200.neb import MAX_IMAGES

    assert MAX_IMAGES == NO.MAX_IMAGES == 64


def _same_run(got, ref, tol=1e-9):
    worst = 0.0
    for a, b in zip(got, ref):
        assert a["status"] == b["status"] and a["n_steps"] == b["n_steps"] and a["i_climb"] == b["i_climb"]
        worst = max(worst, np.abs(a["positions"] - b["positions"]).max())
    assert worst <= tol
    return worst


def test_mueller_brown_on_the_device(device, monkeypatch):
    from torch_m3gnet_b200 import neb

    bands = [(mb_point(*MB_MIN_A), mb_point(*MB_MIN_B))]
    got = neb.BatchNEB(BatchMB(device), bands, n_images=9, climb=True).run(fmax=1e-3, steps=1000)
    with monkeypatch.context() as m:
        m.setattr(neb, "neb_step", oracle_step)
        ref = neb.BatchNEB(BatchMB(), bands, n_images=9, climb=True).run(fmax=1e-3, steps=1000)
    worst = _same_run(got, ref)
    print(f"[neb-mb-gpu] max |kernel - restatement| {worst:.2e} A")
    check_mb_saddle(got[0])


def test_lj_vacancy_hop_on_the_device(device, monkeypatch):
    from torch_m3gnet_b200 import neb

    ini, fin = lj_vacancy_hop(fire_relax_restated)
    got = neb.BatchNEB(BatchLJ(device), [(ini, fin)], n_images=5, climb=True).run(fmax=1e-3, steps=1000)
    with monkeypatch.context() as m:
        m.setattr(neb, "neb_step", oracle_step)
        ref = neb.BatchNEB(BatchLJ(), [(ini, fin)], n_images=5, climb=True).run(fmax=1e-3, steps=1000)
    worst = _same_run(got, ref)
    print(f"[neb-lj-gpu] max |kernel - restatement| {worst:.2e} A")
    check_lj_saddle(got[0])


def _c1_model(device):
    from tests.util import golden, state_dict_of
    from torch_m3gnet_b200 import build_model

    model = build_model(5.0, 4.0, 3, 3, 95, 64, 3, device=device)
    sd = state_dict_of(golden("c1_default"))
    model.load_state_dict({k: (v * 3 if k.endswith("weight") else v) for k, v in sd.items()})
    return model


def _cu_bands(calc):
    """Cu vacancy-hop bands in 2x2x2 (31 atoms) and 3x3x3 (107 atoms) cells, endpoints relaxed with BatchFire, 3, 5
    and 5 interior images."""
    from torch_m3gnet_b200 import BatchFire, synthetic
    from torch_m3gnet_b200.neb import interpolate

    hops = [synthetic.fcc_cu_vacancy_hop(r) for r in (2, 3, 2)]
    structs = [s for h in hops for s in h]
    relaxed = BatchFire(calc, structs).run(fmax=0.02, steps=300)
    assert all(r["status"] == "converged" for r in relaxed)
    ends = [(r["lattice"], r["positions"], s[2]) for r, s in zip(relaxed, structs)]
    return [interpolate(ends[2 * i], ends[2 * i + 1], m) for i, m in enumerate((3, 5, 5))]


@pytest.mark.parametrize("climb", [False, True])
def test_model_bands_match_a_fresh_evaluation(device, climb):
    """Ragged Cu vacancy-hop bands on the model for a fixed 30 steps (fmax = 0, so every band stops at the same frame):
    every record is the frame a fresh model call computes at the returned images in the same layout, its fmax is the
    restatement's NEB force of that evaluation, and the band fmax has fallen.  The barrier of these weights is printed,
    not checked."""
    from torch_m3gnet_b200 import Batch, BatchNEB, M3GNetCalculator

    model = _c1_model(device)
    calc = M3GNetCalculator(model, 5.0, 4.0, skin=0.5, device=device)
    bands = _cu_bands(calc)
    start = BatchNEB(calc, bands, climb=climb).run(fmax=0.0, steps=0)
    res = BatchNEB(calc, bands, climb=climb).run(fmax=0.0, steps=30)
    lat = np.concatenate([np.repeat(r["lattice"][None], len(r["energies"]) - 2, axis=0) for r in res])
    cart = np.concatenate([r["positions"][1:-1].reshape(-1, 3) for r in res])
    z = np.concatenate([np.tile(b[0][2], len(b) - 2) for b in bands])
    sizes = [len(b[0][2]) for b in bands for _ in range(len(b) - 2)]
    fresh = model(Batch.from_arrays(lat, cart, z, sizes, 5.0, 4.0, device=device))
    e = fresh["total_energy"].float().cpu().numpy()
    f = fresh["forces"].float().cpu().numpy().astype(np.float64)
    img = row = 0
    for r, r0, b in zip(res, start, bands):
        m, n = len(b) - 2, len(b[0][2])
        assert r0["status"] == "not converged" and r0["n_steps"] == 0
        assert r["status"] == "not converged" and r["n_steps"] == 30
        assert np.array_equal(r["energies"][1:-1], e[img:img + m].astype(np.float64))
        G, ic, ok = NO.neb_forces(r["energies"], r["positions"], f[row:row + m * n].reshape(m, n, 3), 0.1, climb)
        assert ok and ic == r["i_climb"]
        assert r["fmax"] == pytest.approx(float(np.linalg.norm(G.reshape(-1, 3), axis=1).max()), rel=1e-12)
        print(f"[neb-model] climb={climb} n={n} M={m}: fmax {r0['fmax']:.4f} -> {r['fmax']:.4f} eV/A, barrier "
              f"{r['barrier_forward']:.4f} eV at image {r['i_climb']}, "
              f"E - E_0 {np.round(r['energies'] - r['energies'][0], 4)}")
        assert r["fmax"] < r0["fmax"]
        img, row = img + m, row + m * n


def test_launch_count(device):
    from tests.test_gpu_batch_fire import _verlet_model
    from torch_m3gnet_b200 import BatchNEB, M3GNetCalculator, _lib, synthetic

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
    bands = [synthetic.fcc_cu_vacancy_hop(2) for _ in range(3)]
    opt = BatchNEB(calc, bands, n_images=3, max_atoms=100)
    before = _lib.LAUNCHES
    opt.run(fmax=0.0, steps=3)
    # 6 x 31 endpoint atoms in chunks of <= 100; each 93-atom band runs alone, frames 0 .. 3
    assert opt.n_endpoint_calls == 2 and opt.n_iterations == 3 * 4
    assert len(inner) == opt.n_endpoint_calls + opt.n_iterations
    assert _lib.LAUNCHES - before == sum(inner) + opt.n_iterations * _lib._KERNELS_PER_CALL["neb_step"] == \
        sum(inner) + opt.n_iterations
