"""CPU: the float64 restatement of the conv kernel contract (tests/conv_oracle.py) against the oracle's conv block and
gated MLP, its adjoints against finite differences (torch.autograd.gradcheck), and the mode-2 grouping against a
plain per-atom sum.  The GPU reference tests measure the kernels with this restatement, so it is checked first."""
import pytest
import torch

from oracle import m3gnet_oracle as O
from tests import conv_oracle as C

SMALL_E = (1, 31, 32, 33, 127, 128, 129, 261)


def _oracle_params(F, R, seed):
    """Random oracle parameters of one conv block (prefix "c") with nonzero biases, float64."""
    g = torch.Generator().manual_seed(seed)
    p = {}
    for mlp in ("concat_edge_update", "concat_node_update"):
        for br in ("dense", "gate"):
            p[f"c.{mlp}.{br}.0.weight"] = torch.randn(F, 3 * F, generator=g, dtype=torch.float64) / 4
            p[f"c.{mlp}.{br}.0.bias"] = torch.randn(F, generator=g, dtype=torch.float64) / 2
            p[f"c.{mlp}.{br}.2.weight"] = torch.randn(F, F, generator=g, dtype=torch.float64) / 4
            p[f"c.{mlp}.{br}.2.bias"] = torch.randn(F, generator=g, dtype=torch.float64) / 2
    p["c.edge_linear.weight"] = torch.randn(F, R, generator=g, dtype=torch.float64)
    p["c.node_linear.weight"] = torch.randn(F, R, generator=g, dtype=torch.float64)
    return p


def _split(p, F):
    """The kernels' operands from oracle parameters: P (N-independent weights of the per-atom projection) and the
    per-MLP weight dicts of tests/conv_oracle.py (nn/conv.py::M3GNetConv._pack)."""
    ws, wp, bp = {}, [], []
    for name, mlp, lin in (("edge", "concat_edge_update", "edge_linear"), ("node", "concat_node_update",
                                                                          "node_linear")):
        d0, g0 = p[f"c.{mlp}.dense.0.weight"], p[f"c.{mlp}.gate.0.weight"]
        ws[name] = {"W1e": torch.cat([d0[:, 2 * F:], g0[:, 2 * F:]]), "W2d": p[f"c.{mlp}.dense.2.weight"],
                    "b2d": p[f"c.{mlp}.dense.2.bias"], "W2g": p[f"c.{mlp}.gate.2.weight"],
                    "b2g": p[f"c.{mlp}.gate.2.bias"], "WhT": p[f"c.{lin}.weight"].t()}
        wp += [d0[:, :F], g0[:, :F], d0[:, F:2 * F], g0[:, F:2 * F]]
        bp += [p[f"c.{mlp}.dense.0.bias"], p[f"c.{mlp}.gate.0.bias"], torch.zeros(2 * F, dtype=torch.float64)]
    return ws, torch.cat(wp), torch.cat(bp)


def _inputs(kind, E, F, R, seed):
    src, dst, N = C.graph(kind, E, seed)
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(N, F, generator=g, dtype=torch.float64)
    e = torch.randn(E, F, generator=g, dtype=torch.float64)
    h = torch.rand(E, R, generator=g, dtype=torch.float64)
    return src, dst, N, x, e, h


def _close(a, b, what):
    err = (a - b).abs().max().item() if a.numel() else 0.0
    scale = max(b.abs().max().item() if b.numel() else 0.0, 1e-300)
    assert err <= 1e-12 * scale, f"{what}: max|diff| {err:.3e} vs scale {scale:.3e}"


@pytest.mark.parametrize("kind", C.GRAPH_KINDS)
@pytest.mark.parametrize("F,R", [(8, 1), (16, 3), (64, 4)])
def test_forward_matches_oracle_conv(kind, F, R):
    """mode 0 (edge update), mode 1 + segment sum and mode 2 + segment_sum_parts give the oracle's conv block."""
    E = 261
    p = _oracle_params(F, R, seed=F + R)
    src, dst, N, x, e, h = _inputs(kind, E, F, R, seed=7)
    ws, wp, bp = _split(p, F)
    P = x @ wp.t() + bp
    e2 = C.forward(P, 0, src, dst, e, h, ws["edge"], 0)
    msg = C.forward(P, 4 * F, src, dst, e2, h, ws["node"], 1)
    x2 = C.segment_sum(x, msg, src, N)
    x2_parts = C.segment_sum_parts(x, C.forward(P, 4 * F, src, dst, e2, h, ws["node"], 2), src, N)
    want_x, want_e = O.conv(p, "c", x, e, h, torch.stack([src, dst]))
    _close(e2, want_e, "e2")
    _close(x2, want_x, "x2")
    _close(x2_parts, want_x, "x2 from the mode-2 partial rows")


def test_mlp_out_matches_oracle_gated_mlp():
    F, R, E = 16, 3, 129
    p = _oracle_params(F, R, seed=3)
    src, dst, N, x, e, h = _inputs("poisson", E, F, R, seed=5)
    ws, wp, bp = _split(p, F)
    P = x @ wp.t() + bp
    out = C.mlp_out(C.z1_of(P, 0, src, dst, e, ws["edge"]), h, ws["edge"])
    want = O.gated_mlp(p, "c.concat_edge_update", torch.cat([x[src], x[dst], e], 1), 2) * (h @ ws["edge"]["WhT"])
    _close(out, want, "gated MLP")


class _Mlp(torch.autograd.Function):
    """One gated MLP as a function of (P, e, h) whose backward is conv_oracle.mlp_bwd: mode 0 returns out (E,F),
    mode 1 its per-source-atom sum (N,F), the quantity whose upstream gradient mode 1 indexes by src."""

    @staticmethod
    def forward(ctx, P, e, h, po, src, dst, w, mode, N):
        ctx.save_for_backward(P, e, h)
        ctx.args = (po, src, dst, w, mode, N)
        out = C.mlp_out(C.z1_of(P, po, src, dst, e, w), h, w)
        return out if mode == 0 else C.segment_sum(torch.zeros(N, out.shape[1], dtype=out.dtype), out, src, N)

    @staticmethod
    def backward(ctx, g):
        P, e, h = ctx.saved_tensors
        po, src, dst, w, mode, N = ctx.args
        g_e, g_z1, g_h = C.mlp_bwd(P, po, src, dst, e, h, w, g, None, mode)
        F = e.shape[1]
        g_P = torch.zeros_like(P)
        g_P[:, po:po + 2 * F].index_add_(0, src, g_z1)
        g_P[:, po + 2 * F:po + 4 * F].index_add_(0, dst, g_z1)
        return g_P, g_e, g_h, None, None, None, None, None, None


class _Block(torch.autograd.Function):
    """A whole conv block, (P, e, h) -> (per-atom message sum, e2), whose backward is conv_oracle.block_bwd."""

    @staticmethod
    def forward(ctx, P, e, h, src, dst, ws, N):
        F = e.shape[1]
        e2 = C.forward(P, 0, src, dst, e, h, ws["edge"], 0)
        msg = C.forward(P, 4 * F, src, dst, e2, h, ws["node"], 1)
        ctx.save_for_backward(P, e, e2, h)
        ctx.args = (src, dst, ws, N)
        return C.segment_sum(torch.zeros(N, F, dtype=msg.dtype), msg, src, N), e2

    @staticmethod
    def backward(ctx, g_x2, g_e2):
        P, e, e2, h = ctx.saved_tensors
        src, dst, ws, N = ctx.args
        F = e.shape[1]
        _, g_e, gz_n, gz_e, gh_n, gh_e = C.block_bwd(P, src, dst, e, e2, h, ws["edge"], ws["node"], g_x2, g_e2)
        g_P = torch.zeros_like(P)
        for po, gz in ((0, gz_e), (4 * F, gz_n)):
            g_P[:, po:po + 2 * F].index_add_(0, src, gz)
            g_P[:, po + 2 * F:po + 4 * F].index_add_(0, dst, gz)
        return g_P, g_e, gh_n + gh_e, None, None, None, None


@pytest.mark.parametrize("kind", ["poisson", "one_atom", "self", "single"])
@pytest.mark.parametrize("mode", [0, 1])
def test_mlp_adjoints_gradcheck(kind, mode):
    F, R, E = 4, 2, 9
    src, dst, N, x, e, h = _inputs(kind, E, F, R, seed=11)
    g = torch.Generator().manual_seed(2)
    w = {"W1e": torch.randn(2 * F, F, generator=g, dtype=torch.float64),
         "W2d": torch.randn(F, F, generator=g, dtype=torch.float64),
         "W2g": torch.randn(F, F, generator=g, dtype=torch.float64),
         "b2d": torch.randn(F, generator=g, dtype=torch.float64),
         "b2g": torch.randn(F, generator=g, dtype=torch.float64),
         "WhT": torch.randn(R, F, generator=g, dtype=torch.float64)}
    P = torch.randn(N, 8 * F, generator=g, dtype=torch.float64, requires_grad=True)
    po = 4 * F if mode else 0
    assert torch.autograd.gradcheck(
        lambda P_, e_, h_: _Mlp.apply(P_, e_, h_, po, src, dst, w, mode, N),
        (P, e.requires_grad_(True), h.requires_grad_(True)))


@pytest.mark.parametrize("kind", ["poisson", "deg31", "self"])
def test_block_adjoints_gradcheck(kind):
    F, R, E = 4, 3, 12
    p = _oracle_params(F, R, seed=13)
    ws, _, _ = _split(p, F)
    src, dst, N, x, e, h = _inputs(kind, E, F, R, seed=17)
    P = torch.randn(N, 8 * F, dtype=torch.float64, generator=torch.Generator().manual_seed(4), requires_grad=True)
    assert torch.autograd.gradcheck(lambda P_, e_, h_: _Block.apply(P_, e_, h_, src, dst, ws, N),
                                    (P, e.requires_grad_(True), h.requires_grad_(True)))


def test_mlp_bwd_base_and_chain():
    """g_e_base is added once; block_bwd's ge2 is g_e2 plus the node adjoint and feeds the edge MLP as both its
    upstream gradient and its base."""
    F, R, E = 8, 2, 40
    src, dst, N, x, e, h = _inputs("poisson", E, F, R, seed=19)
    ws, wp, bp = _split(_oracle_params(F, R, seed=23), F)
    P = x @ wp.t() + bp
    g = torch.Generator().manual_seed(29)
    g_up, base = torch.randn(E, F, generator=g, dtype=torch.float64), torch.randn(E, F, generator=g,
                                                                                dtype=torch.float64)
    a = C.mlp_bwd(P, 0, src, dst, e, h, ws["edge"], g_up, None, 0)
    b = C.mlp_bwd(P, 0, src, dst, e, h, ws["edge"], g_up, base, 0)
    _close(b[0], a[0] + base, "g_e with base")
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    e2 = C.forward(P, 0, src, dst, e, h, ws["edge"], 0)
    g_x2 = torch.randn(N, F, generator=g, dtype=torch.float64)
    ge2, g_e, gz_n, gz_e, gh_n, gh_e = C.block_bwd(P, src, dst, e, e2, h, ws["edge"], ws["node"], g_x2, base)
    n = C.mlp_bwd(P, 4 * F, src, dst, e2, h, ws["node"], g_x2, base, 1)
    _close(ge2, n[0], "ge2")
    ed = C.mlp_bwd(P, 0, src, dst, e, h, ws["edge"], ge2, ge2, 0)
    _close(g_e, ed[0], "g_e")


@pytest.mark.parametrize("kind", C.GRAPH_KINDS)
@pytest.mark.parametrize("E", SMALL_E + (1380,))
def test_mode2_grouping_is_the_per_atom_sum(kind, E):
    src, dst, N = C.graph(kind, E, seed=E)
    out = torch.randn(E, 3, dtype=torch.float64, generator=torch.Generator().manual_seed(E))
    part, mask = C.group_rows(out, src)
    base = torch.randn(N, 3, dtype=torch.float64)
    _close(C.segment_sum_parts(base, part, src, N), C.segment_sum(base, out, src, N), "parts vs plain sum")
    # the header's statement, literally: out[i] = base[i] + sum_k part[max(b_i, 32 k)] over the blocks k of atom i
    ptr = C.edge_ptr_of(src, N).tolist()
    for i in range(N):
        b, en = ptr[i], ptr[i + 1]
        rows = [max(b, 32 * k) for k in range(b // 32, (en + 31) // 32)] if en > b else []
        assert all(bool(mask[r]) for r in rows)
        want = base[i] + sum((part[r] for r in rows), torch.zeros(3, dtype=torch.float64))
        assert torch.allclose(C.segment_sum_parts(base, part, src, N)[i], want, rtol=1e-12, atol=1e-12)
    assert int(mask.sum()) == sum(len(range(ptr[i] // 32, (ptr[i + 1] + 31) // 32)) for i in range(N)
                                  if ptr[i + 1] > ptr[i])


@pytest.mark.parametrize("E", SMALL_E + (1380, 2 * 148 * 128 + 1))
def test_graph_generators(E):
    for kind in C.GRAPH_KINDS:
        src, dst, N = C.graph(kind, E, seed=1)
        assert src.numel() == dst.numel() == E, kind
        assert bool((src[1:] >= src[:-1]).all()), kind
        assert int(src.max()) < N and int(dst.max()) < N and int(dst.min()) >= 0, kind
        deg = torch.bincount(src, minlength=N)
        if kind == "single":
            assert bool((deg[:E] == 1).all())
        if kind == "one_atom":
            assert int(deg[0]) == E
        if kind.startswith("deg"):
            d = int(kind[3:])
            assert bool((deg[:E // d] == d).all())
        if kind == "hubs" and E >= 400:
            assert {129, 200} <= set(deg.tolist())
        if kind in ("poisson", "hubs"):
            assert int((deg == 0).sum()) >= 1
        if kind == "self":
            assert bool((dst[::2] == src[::2]).all())


def test_tf32_round_has_zero_lo():
    t = torch.randn(1000)
    r = C.tf32_round(t)
    assert torch.equal(C.tf32_round(r), r)
    assert (r - t).abs().max() <= 2.0 ** -10 * t.abs().max()
    w = C.mlp_weights(3, seed=1, tf32=True)
    for v in w.values():
        assert torch.equal(C.tf32_round(v), v)
