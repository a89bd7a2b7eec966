"""CPU: the float64 restatements of the per-step kernels (tests/step_kernels_oracle.py) against oracle/m3gnet_oracle.py
run in float64 with autograd, and the float32 geometry restatement against torch CPU float32 bit for bit.  The GPU
step-kernel reference tests measure the kernels with these restatements, so they are checked first."""
import numpy as np
import pytest
import torch

from oracle import m3gnet_oracle as O
from tests import step_kernels_oracle as S

D = torch.float64


def _readout_params(F, seed):
    g = torch.Generator().manual_seed(seed)
    p = {}
    for br in ("dense", "gate"):
        for i, (o, k) in enumerate(((F, F), (F, F), (1, F))):
            p[f"ro.gated.{br}.{2 * i}.weight"] = torch.randn(o, k, generator=g, dtype=D) / k ** 0.5
            p[f"ro.gated.{br}.{2 * i}.bias"] = 0.5 * torch.randn(o, generator=g, dtype=D)
    return p


def readout_weights(p, prefix="ro"):
    """m3g_readout_* weights from oracle parameters (nn/readout.py::AtomWiseReadout._pack)."""
    w = {}
    for br, s in (("dense", "d"), ("gate", "g")):
        q = f"{prefix}.gated.{br}"
        w[f"W0{s}"], w[f"b0{s}"] = p[f"{q}.0.weight"], p[f"{q}.0.bias"]
        w[f"W1{s}"], w[f"b1{s}"] = p[f"{q}.2.weight"], p[f"{q}.2.bias"]
        w[f"w2{s}"], w[f"b2{s}"] = p[f"{q}.4.weight"].reshape(-1), p[f"{q}.4.bias"]
    return w


def close(a, b, tol=1e-12):
    a, b = a.detach().double(), b.detach().double()
    return a.shape == b.shape and float((a - b).abs().max()) <= tol * max(1.0, float(b.abs().max()))


@pytest.mark.parametrize("F", [1, 17, 64, 100])
def test_readout_and_structure_sum(F):
    g = torch.Generator().manual_seed(F)
    N, B, scale = 37, 5, 1.7
    p = _readout_params(F, F)
    w = readout_weights(p)
    x = torch.randn(N, F, generator=g, dtype=D)
    elemental = torch.randn(N, generator=g, dtype=D)
    batch = torch.sort(torch.randint(0, B - 1, (N,), generator=g)).values  # structure B - 1 has no atoms
    ptr = torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(torch.bincount(batch, minlength=B), 0)])
    x_leaf = x.clone().requires_grad_(True)
    atomic, stot, tot = O.readout(p, "ro", x_leaf, elemental, batch, B, scale)
    assert close(S.readout_fwd(x, w, elemental, scale), atomic)
    s_st, s_t = S.structure_sum(atomic.detach(), ptr, scale)
    assert close(s_st, stot) and close(s_t, tot) and float(s_t[-1]) == 0.0
    ups = {"g_atomic": torch.randn(N, generator=g, dtype=D), "g_scaled_total": torch.randn(B, generator=g, dtype=D),
           "g_total": torch.randn(B, generator=g, dtype=D)}
    for names in (("g_atomic",), ("g_scaled_total",), ("g_total",), ("g_atomic", "g_scaled_total", "g_total")):
        loss = sum(((atomic, stot, tot)[("g_atomic", "g_scaled_total", "g_total").index(n)] * ups[n]).sum()
                   for n in names)
        (want,) = torch.autograd.grad(loss, x_leaf, retain_graph=True)
        got = S.readout_bwd(x, w, *(ups[n] if n in names else None for n in ("g_atomic", "g_scaled_total", "g_total")),
                            batch, scale)
        assert close(got, want), names
    # the envelope bounds the value
    env = S.readout_fwd(x.abs(), S.absolute(w), elemental.abs(), scale)
    assert bool((env >= S.readout_fwd(x, w, elemental, scale).abs() * (1 - 1e-12)).all())


@pytest.mark.parametrize("K,M", [(17, 136), (64, 512), (136, 17), (1, 5)])
def test_linear(K, M):
    g = torch.Generator().manual_seed(K * M)
    n = 23
    x = torch.randn(n, K, generator=g, dtype=D).requires_grad_(True)
    W = torch.randn(M, K, generator=g, dtype=D)
    b = torch.randn(M, generator=g, dtype=D)
    base = torch.randn(n, M, generator=g, dtype=D)
    y = torch.nn.functional.linear(x, W, b)
    assert close(S.linear(x.detach(), W.t(), b), y)
    assert close(S.linear(x.detach(), W.t(), None, base), torch.nn.functional.linear(x, W) + base)
    go = torch.randn(n, M, generator=g, dtype=D)
    (want,) = torch.autograd.grad(y, x, go)
    baseK = torch.randn(n, K, generator=g, dtype=D)
    assert close(S.linear_bwd_input(go, W), want)
    assert close(S.linear_bwd_input(go, W, baseK), want + baseK)


def _radial_consts64(R, rc):
    """the product's float32 constant table (nn/featurizer.py::radial_constants); the oracle forms sinc's argument
    (m+1) pi / rc in float32 as well (an integer tensor times a Python float)"""
    from torch_m3gnet_b200.nn.featurizer import radial_constants

    return radial_constants(R, rc)[0].double()


@pytest.mark.parametrize("R", range(1, 11))
@pytest.mark.parametrize("rc", [5.0, 4.2, 3.0])
def test_radial(R, rc):
    g = torch.Generator().manual_seed(R)
    r = torch.cat([torch.rand(200, generator=g, dtype=D) * rc, torch.tensor([rc, 1e-3, 0.5], dtype=D)])
    consts = _radial_consts64(R, rc)
    r_leaf = r.clone().requires_grad_(True)
    want = O.radial_basis(r_leaf, R, rc)
    assert close(S.radial(r, consts, R), want)
    go = torch.randn(want.shape, generator=g, dtype=D)
    (gw,) = torch.autograd.grad(want, r_leaf, go)
    assert close(S.radial(r, consts, R, go), gw, 1e-9)
    # r = 0: h_m from s(0) = 1, and no gradient
    h0 = S.radial(torch.zeros(1, dtype=D), consts, R)
    assert close(h0, O.radial_basis(torch.zeros(1, dtype=D), R, rc))
    assert float(S.radial(torch.zeros(1, dtype=D), consts, R, torch.ones(1, R, dtype=D))[0]) == 0.0
    env = S.radial(r, consts, R, absolute_=True)
    assert bool((env >= want.detach().abs() * (1 - 1e-12)).all())


@pytest.mark.parametrize("F,R", [(1, 1), (17, 3), (64, 4), (128, 10)])
def test_edge_adjust(F, R):
    g = torch.Generator().manual_seed(F + R)
    h = torch.randn(31, R, generator=g, dtype=D).requires_grad_(True)
    W = torch.randn(F, R, generator=g, dtype=D)
    want = torch.nn.functional.silu(torch.nn.functional.linear(h, W))  # oracle ``forward``: e = SiLU(h W^T)
    assert close(S.edge_adjust_fwd(h.detach(), W.t()), want)
    go = torch.randn(want.shape, generator=g, dtype=D)
    (gw,) = torch.autograd.grad(want, h, go)
    assert close(S.edge_adjust_bwd(h.detach(), W.t(), go), gw)


def _graph(lattice, cart):
    gd = O.collate([O.build_graph(np.asarray(lattice), np.asarray(cart), [29] * len(cart), 3.0, 3.0)])
    return gd


def _structures():
    lat, cart, _ = O.fcc_supercell(1, a=3.615, jitter=0.0)  # collinear bonds: cos = -1 and +1 exactly
    flip = np.diag([1.0, -1.0, 1.0]) @ (lat + np.array([[0, 0.3, 0], [0, 0, 0], [0.2, 0, 0]]))  # det < 0
    lat2, cart2, _ = O.fcc_supercell(1, a=3.7, jitter=0.1, seed=3)
    return [(lat, cart), (flip, cart2 @ np.linalg.inv(lat2) @ flip), (lat2, cart2)]


@pytest.mark.parametrize("which", [0, 1, 2])
def test_geometry_and_angles(which):
    lat, cart = _structures()[which]
    gd = _graph(lat, cart)
    ei, sh, tri = gd["edge_index"], gd["edge_cell_shift"], gd["triplet_edge_index"]
    N, E, T = len(cart), ei.shape[1], tri.shape[1]
    assert T > 0
    pos = torch.tensor(cart, dtype=D).requires_grad_(True)
    L = torch.tensor(lat, dtype=D)[None]
    batch = torch.zeros(N, dtype=torch.long)
    vec, dist, cos = O.pair_geometry(pos, L, batch, ei, sh, tri)
    v, r = S.geometry_fwd(pos.detach(), L, batch, ei[0], ei[1], sh)
    assert close(v, vec) and close(r, dist)
    vec4 = torch.cat([v, r[:, None]], 1)
    c_raw, c = S.angles_fwd(vec4, tri)
    assert close(c, cos)
    passes = (c_raw >= -1) & (c_raw <= 1)
    if which == 0:
        assert bool((c_raw.abs() >= 1 - 1e-15).any()), "the perfect FCC cell has collinear bond pairs"
    g = torch.Generator().manual_seed(which)
    gv, gdist, gc = (torch.randn(t.shape, generator=g, dtype=D) for t in (vec, dist, cos))
    for use in ((1, 1, 1), (1, 0, 0), (0, 1, 0), (0, 0, 1)):
        outs = [o for o, u in zip((vec, dist, cos), use) if u]
        gos = [o for o, u in zip((gv, gdist, gc), use) if u]
        (want,) = torch.autograd.grad(outs, pos, gos, retain_graph=True)
        g_vec4 = torch.cat([gv, torch.zeros(E, 1, dtype=D)], 1) if use[0] else None
        if use[2]:
            g_vec4 = (torch.zeros(E, 4, dtype=D) if g_vec4 is None else g_vec4) + S.angles_bwd(vec4, tri, gc, passes)
        got = S.geometry_bwd(vec4, g_vec4, gdist if use[1] else None, ei[0], ei[1], N)
        assert close(got, want, 1e-10), use
    assert close(S.geometry_bwd(vec4, None, gdist, ei[0], ei[1], N, 2.5),
                 2.5 * S.geometry_bwd(vec4, None, gdist, ei[0], ei[1], N))


@pytest.mark.parametrize("which", [0, 1, 2])
def test_geometry_f32_is_torch_f32_bitwise(which):
    """vec: oracle ``pair_geometry`` in float32; dist: the correctly rounded square root (as __fsqrt_rn) of
    torch.sum(v * v) (torch.linalg.norm, and torch's CPU float32 sqrt, differ from it by an ulp in some distances);
    cos: torch.sum(v1 * v2) / (r1 * r2)."""
    lat, cart = _structures()[which]
    gd = _graph(lat, cart)
    ei, sh, tri = gd["edge_index"], gd["edge_cell_shift"], gd["triplet_edge_index"]
    pos = torch.tensor(cart, dtype=torch.float32)
    L = torch.tensor(lat, dtype=torch.float32)[None]
    batch = torch.zeros(len(cart), dtype=torch.long)
    vec, _, _ = O.pair_geometry(pos, L, batch, ei, sh, tri)
    v, r = S.geometry_f32(pos.numpy(), L.numpy(), batch.numpy(), ei[0].numpy(), ei[1].numpy(), sh.numpy())
    assert np.array_equal(v, vec.numpy())
    assert np.array_equal(r, torch.sqrt(torch.sum(vec * vec, dim=1).double()).float().numpy())
    rt = torch.from_numpy(r)
    want = torch.sum(vec[tri[0]] * vec[tri[1]], dim=1) / (rt[tri[0]] * rt[tri[1]])
    c_raw, c = S.angles_f32(np.concatenate([v, r[:, None]], 1), tri.numpy())
    assert np.array_equal(c_raw, want.numpy())
    assert np.array_equal(c, torch.clamp(want, -1, 1).numpy())


def test_forces_virial():
    """oracle ``forward``: forces = -dE/dpos; stresses = Voigt(sum_i pos (x) F) / |a . (b x c)| per structure"""
    g = torch.Generator().manual_seed(3)
    sizes = [5, 0, 40, 1]
    N = sum(sizes)
    ptr = torch.tensor([0] + list(np.cumsum(sizes)))
    pos, g_pos = torch.randn(N, 3, generator=g, dtype=D), torch.randn(N, 3, generator=g, dtype=D)
    lat = torch.randn(len(sizes), 3, 3, generator=g, dtype=D) + 4 * torch.eye(3, dtype=D)
    lat[2, 0] = -lat[2, 0]
    assert float(torch.linalg.det(lat[2])) < 0
    forces, st = S.forces_virial(pos, g_pos, lat, ptr)
    batch = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes))
    outer = pos[:, :, None] * (-g_pos)[:, None, :]
    s = torch.zeros((len(sizes), 3, 3), dtype=D).index_add_(0, batch, outer)
    vol = torch.abs(torch.sum(lat[:, 0] * torch.linalg.cross(lat[:, 1], lat[:, 2]), dim=1))
    voigt = torch.stack([s[:, 0, 0], s[:, 1, 1], s[:, 2, 2], s[:, 1, 2], s[:, 2, 0], s[:, 0, 1]])
    assert torch.equal(forces, -g_pos)
    assert close(st, torch.transpose(voigt / vol, 0, 1)) and float(st[1].abs().max()) == 0.0


def test_segment_sum_f32_order():
    rng = np.random.default_rng(0)
    deg = np.array([0, 3, 1, 0, 40, 2])
    ptr = np.concatenate([[0], np.cumsum(deg)])
    rows = rng.standard_normal((ptr[-1], 5)).astype(np.float32)
    perm = rng.permutation(ptr[-1])
    got = S.segment_sum_f32(rows, ptr, perm)
    for i in range(len(deg)):
        acc = np.zeros(5, np.float32)
        for p in range(ptr[i], ptr[i + 1]):
            acc = acc + rows[perm[p]]
        assert np.array_equal(got[i], acc)
