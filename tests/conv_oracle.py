"""The tensor-core gated-MLP contract (include/m3gnet_b200.h, "M3GNetConv" and "Tensor-core path") restated in plain
torch float64, with the arguments of the C ABI: P, po, src, dst, e, h, the (out,in) weights, R, mode.  Also the graph
generators the kernel tests sweep.  Shared by the CPU and GPU conv reference tests.

Weights of one gated MLP, ``w``: dict with W1e (2F,F) = rows [dense | gate] of the e-part of layer 1, W2d, W2g (F,F),
b2d, b2g (F), WhT (R,F) = edge_linear / node_linear weight transposed.  F = 64 on the tensor cores."""
import math

import torch

TILE_ROWS = 32  # mode 2 sums messages per 32-row block and source atom


def _d(t):
    return t.to(torch.float64)


def z1_of(P, po, src, dst, e, w):
    """z1 (E,2F) = P[src][po:po+2F] + P[dst][po+2F:po+4F] + e·W1e^T (dense half, then gate half)."""
    F = e.shape[1]
    src, dst = src.long(), dst.long()
    P = _d(P)
    return P[src, po:po + 2 * F] + P[dst, po + 2 * F:po + 4 * F] + _d(e) @ _d(w["W1e"]).t()


def mlp_out(z1, h, w):
    """out (E,F) = SiLU(z2d)·σ(z2g)·(h·Wh^T) with z2d = SiLU(z1d)·W2d^T + b2d, z2g = SiLU(z1g)·W2g^T + b2g."""
    F = z1.shape[1] // 2
    a1 = torch.nn.functional.silu(z1)
    z2d = a1[:, :F] @ _d(w["W2d"]).t() + _d(w["b2d"])
    z2g = a1[:, F:] @ _d(w["W2g"]).t() + _d(w["b2g"])
    return torch.nn.functional.silu(z2d) * torch.sigmoid(z2g) * (_d(h) @ _d(w["WhT"]))


def partial_rows(src):
    """bool (E): rows where mode 2 stores a partial sum, the first row of each (32-row block, source atom) run."""
    src = src.long()
    E = src.numel()
    first = torch.ones(E, dtype=torch.bool, device=src.device)
    if E > 1:
        first[1:] = src[1:] != src[:-1]
    first[torch.arange(0, E, TILE_ROWS, device=src.device)] = True
    return first


def group_rows(out, src):
    """Mode 2: (E,F), the sum of ``out`` over each (32-row block, source atom) run at the run's first row, 0 at the
    other rows.  Returns (y, mask of partial rows)."""
    mask = partial_rows(src)
    run = torch.cumsum(mask.long(), 0) - 1  # run index of every row
    first = torch.nonzero(mask).flatten()
    sums = torch.zeros((first.numel(), out.shape[1]), dtype=out.dtype, device=out.device).index_add_(0, run, out)
    y = torch.zeros_like(out)
    y[first] = sums
    return y, mask


def forward(P, po, src, dst, e, h, w, mode):
    """y of m3g_conv_tc_fwd / m3g_conv_mlp_fwd.  mode 0: e + out; 1: out; 2: group_rows(out, src)[0]."""
    out = mlp_out(z1_of(P, po, src, dst, e, w), h, w)
    if mode == 0:
        return _d(e) + out
    if mode == 1:
        return out
    if mode == 2:
        return group_rows(out, src)[0]
    raise ValueError(f"mode {mode}")


def segment_sum(base, msg, src, N):
    """m3g_segment_sum_add: base + the rows of msg summed per source atom."""
    return _d(base) + torch.zeros((N, msg.shape[1]), dtype=torch.float64, device=msg.device).index_add_(
        0, src.long(), _d(msg))


def segment_sum_parts(base, part, src, N):
    """m3g_segment_sum_parts: base + the partial rows of a mode-2 forward summed per source atom (other rows of
    ``part`` are never read)."""
    mask = partial_rows(src)
    return _d(base) + torch.zeros((N, part.shape[1]), dtype=torch.float64, device=part.device).index_add_(
        0, src.long()[mask], _d(part)[mask])


def mlp_bwd(P, po, src, dst, e, h, w, g_up, g_e_base, mode):
    """Adjoints of one gated MLP on edges (m3g_conv_mlp_bwd, m3g_conv_tc_bwd, m3g_conv_tc_bwd_saved), by autograd.
    Upstream gradient of ``out``: mode 0: g_up (E,F); mode 1: g_up[src] (g_up is (N,F)).  Returns
    g_e = g_e_base (None = 0) + (d out/d e)^T g_u, g_z1 = dL/dz1 (E,2F), g_h (E,R), all float64."""
    e64 = _d(e).detach().requires_grad_(True)
    h64 = _d(h).detach().requires_grad_(True)
    with torch.enable_grad():
        z1 = z1_of(P, po, src, dst, e64, w)
        out = mlp_out(z1, h64, w)
        g_u = _d(g_up) if mode == 0 else _d(g_up)[src.long()]
        g_e, g_z1, g_h = torch.autograd.grad(out, (e64, z1, h64), grad_outputs=g_u)
    if g_e_base is not None:
        g_e = g_e + _d(g_e_base)
    return g_e, g_z1, g_h


def gh_scale(P, po, src, dst, e, h, w, g_up, mode):
    """(E,R): the float64 magnitude of the terms of g_h = q·Wh with q = g_u·SiLU(z2d)·σ(z2g), i.e. |q|·|Wh|.  A g_h
    entry is a sum of F products that can cancel; its rounding error is set by this scale, not by |g_h|."""
    z1 = z1_of(P, po, src, dst, e, w)
    F = z1.shape[1] // 2
    a1 = torch.nn.functional.silu(z1)
    z2d = a1[:, :F] @ _d(w["W2d"]).t() + _d(w["b2d"])
    z2g = a1[:, F:] @ _d(w["W2g"]).t() + _d(w["b2g"])
    g_u = _d(g_up) if mode == 0 else _d(g_up)[src.long()]
    q = g_u * torch.nn.functional.silu(z2d) * torch.sigmoid(z2g)
    return q.abs() @ _d(w["WhT"]).abs().t()


def block_bwd(P, src, dst, e, e2, h, w_edge, w_node, g_x2, g_e2):
    """m3g_conv_tc_block_bwd: the node MLP adjoint (mode 1, P columns 4F.., input e2, g_up = g_x2, base g_e2), then
    the edge MLP adjoint (mode 0, P columns 0.., input e, g_up = g_e_base = ge2).  Returns
    (ge2, g_e, gz_node, gz_edge, gh_node, gh_edge)."""
    F = e.shape[1]
    ge2, gz_node, gh_node = mlp_bwd(P, 4 * F, src, dst, e2, h, w_node, g_x2, g_e2, 1)
    g_e, gz_edge, gh_edge = mlp_bwd(P, 0, src, dst, e, h, w_edge, ge2, ge2, 0)
    return ge2, g_e, gz_node, gz_edge, gh_node, gh_edge


# ---------------------------------------------------------------------------------------------------------------------
# graphs: sorted src (bonds grouped by source atom, as the kernels require), free dst
GRAPH_KINDS = ("poisson", "single", "one_atom", "deg31", "deg32", "deg33", "hubs", "self")


def degrees(kind, E, gen):
    """Per-atom bond counts summing to exactly E (the last atom is cut short where needed)."""
    if kind == "single":
        return [1] * E
    if kind == "one_atom":
        return [E]
    if kind in ("deg31", "deg32", "deg33"):
        d = int(kind[3:])
        return [d] * (E // d) + ([E % d] if E % d else [])
    out, total, i = [], 0, 0
    while total < E:
        if kind == "hubs":
            d = (129, 3, 200, 0, 17)[i % 5]
        else:  # poisson / self: Poisson(12), every 7th atom without bonds
            d = 0 if i % 7 == 3 else int(torch.poisson(torch.tensor(12.0), generator=gen).item())
        d = min(d, E - total)
        out.append(d)
        total += d
        i += 1
    out.append(0)  # a trailing atom without bonds
    return out


def graph(kind, E, seed=0):
    """(src, dst, N) int64 CPU tensors with E bonds of the given degree pattern; "self" makes every other bond point
    at its own source atom."""
    gen = torch.Generator().manual_seed(seed)
    deg = degrees(kind, E, gen)
    N = max(len(deg), 2)
    src = torch.repeat_interleave(torch.arange(len(deg)), torch.tensor(deg, dtype=torch.long))
    dst = torch.randint(0, N, (E,), generator=gen)
    if kind == "self":
        dst[::2] = src[::2]
    assert src.numel() == E
    return src, dst, N


def edge_ptr_of(src, N):
    counts = torch.bincount(src.long(), minlength=N)
    return torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(counts.cpu(), 0)])


# ---------------------------------------------------------------------------------------------------------------------
# weights and inputs
def _row_scales(rows, gen, offset=0):
    """1 for most rows; every 8th row (a different one in each block of 8) scaled by 2^k, k cycling through -6..6,
    so that every 16-column block of every output has a row far above and far below the others."""
    k = (torch.arange(rows // 8) * 5 + offset) % 13 - 6
    s = torch.ones(rows, dtype=torch.float64)
    s[torch.arange(rows // 8) * 8 + torch.randint(0, 8, (rows // 8,), generator=gen)] = torch.pow(2.0, k.double())
    return s


def tf32_round(t):
    """Truncate float32 values to the 10 explicit mantissa bits of TF32 (their lo split is then exactly zero)."""
    i = t.float().contiguous().view(torch.int32)
    return (i & -8192).view(torch.float32)


def mlp_weights(R, seed, F=64, scaled=True, tf32=False):
    """float32 CPU weights of one gated MLP with nonzero biases; ``scaled``: rows of W1e, W2d, W2g multiplied by
    powers of two 2^-6 .. 2^6."""
    gen = torch.Generator().manual_seed(seed)

    def mat(rows, cols, off):
        W = torch.randn(rows, cols, generator=gen, dtype=torch.float64) / math.sqrt(cols)
        if scaled:
            W = W * _row_scales(rows, gen, off)[:, None]
        return W.float()

    w = {"W1e": mat(2 * F, F, 0), "W2d": mat(F, F, 3), "W2g": mat(F, F, 7),
         "b2d": (0.5 * torch.randn(F, generator=gen)).float(), "b2g": (0.5 * torch.randn(F, generator=gen)).float(),
         "WhT": torch.randn(R, F, generator=gen).float()}
    if tf32:
        w = {k: tf32_round(v) for k, v in w.items()}
    return w


def transposed(w):
    """The (in,out) copies the FMA kernels read."""
    return {"W1eT": w["W1e"].t().contiguous(), "W2dT": w["W2d"].t().contiguous(),
            "W2gT": w["W2g"].t().contiguous()}
