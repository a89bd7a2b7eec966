"""The per-step kernels outside the conv MLPs and the three-body op, restated in plain torch float64 with the
arguments of the C ABI (include/m3gnet_b200.h): readout, structure sums, the per-atom projections, the radial basis,
the edge adjustor, pair geometry and angles, forces and virial.  Shared by the CPU and GPU step-kernel reference tests.
The conv MLP kernels, their segment sums and gathers are restated in tests/conv_oracle.py.

Each function also gives the condition-aware scale the GPU tests normalise errors by, the sum of |terms| of each dot
product: a forward evaluated on the absolute values of all inputs and weights (``absolute``; SiLU and sigmoid at |z|
bound their values at z), an adjoint with ``ops=ABS`` (see ``adjoint``) or ``absolute_=True``.

``geometry_f32`` / ``angles_f32`` restate the float32 rounding order of m3g_geometry_fwd / m3g_angles_fwd in numpy,
so that the kernels' distances, bond vectors and cosines can be checked bit for bit."""
import math

import numpy as np
import torch
import torch.nn.functional as Fn


def _d(t):
    return t.to(torch.float64)


def absolute(d):
    """{k: |v|} of a weight dict (float64)"""
    return {k: _d(v).abs() for k, v in d.items()}


# ---------------------------------------------------------------------------------------------------------------------
# Scales of adjoints.  Evaluating an adjoint on |inputs| moves every activation to |z| >= z, where sigmoid' and SiLU''
# are smaller: a gate's adjoint would vanish from the scale.  The scale of an adjoint is therefore the adjoint taken at
# the true operating point with every local factor replaced by its absolute value (|W|, |other factor|, f'(z) by the
# sum of |terms| it is formed from) and the upstream gradient by its absolute value: the sum of |terms| of each dot
# product of the adjoint.
def _silu_dabs(z):
    """SiLU'(z) = s (1 + z (1 - s)) as the kernels form it, by its sum of |terms| (the two terms cancel at z ~ -1.28)"""
    s = torch.sigmoid(z)
    return s * (1 + z.abs() * (1 - s))


def _sigmoid_dabs(z):
    s = torch.sigmoid(z)
    return s * (1 - s)


class _AbsAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z, f, dabs):
        ctx.save_for_backward(dabs(z))
        return f(z)

    @staticmethod
    def backward(ctx, g):
        return g * ctx.saved_tensors[0], None, None


class _AbsMatmul(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, W):
        ctx.save_for_backward(x.abs(), W.abs())
        return x @ W

    @staticmethod
    def backward(ctx, g):
        xa, Wa = ctx.saved_tensors
        return g @ Wa.t(), xa.t() @ g


class _AbsMul(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b):
        ctx.save_for_backward(a.abs(), b.abs())
        return a * b

    @staticmethod
    def backward(ctx, g):
        aa, ba = ctx.saved_tensors
        return g * ba, g * aa


class Ops:
    """the operations the restatements are written in: plain, or (ABS) with the absolute-value adjoints"""

    def __init__(self, absolute_):
        if absolute_:
            self.silu = lambda z: _AbsAct.apply(z, Fn.silu, _silu_dabs)
            self.sigmoid = lambda z: _AbsAct.apply(z, torch.sigmoid, _sigmoid_dabs)
            self.mm, self.mul = _AbsMatmul.apply, _AbsMul.apply
        else:
            self.silu, self.sigmoid = Fn.silu, torch.sigmoid
            self.mm, self.mul = torch.matmul, torch.mul


PLAIN, ABS = Ops(False), Ops(True)


def adjoint(f, inputs, g_out, ops):
    """(d f / d inputs)^T g_out by autograd (ops = ABS: the scale of that adjoint, with |g_out|)"""
    xs = [_d(x).detach().requires_grad_(True) for x in inputs]
    with torch.enable_grad():
        return torch.autograd.grad(f(*xs, ops), xs, grad_outputs=_d(g_out).abs() if ops is ABS else _d(g_out))


# ---------------------------------------------------------------------------------------------------------------------
# readout: nn/readout.py:39-58, GatedMLP(F -> F -> F -> 1, is_output) of nn/core.py:6-62 (oracle ``readout`` /
# ``gated_mlp``).  Weights as m3g_readout_* takes them: W0d, W1d (F,F) (out,in), b0d, b1d (F), w2d (F), b2d (1), and
# the same for the gate branch.
def readout_eps(x, w, ops=PLAIN):
    """eps (N) = dense(x) * gate(x): SiLU, SiLU, linear on the dense branch; SiLU, SiLU, sigmoid on the gate."""
    x = _d(x)
    d = ops.silu(ops.mm(x, _d(w["W0d"]).t()) + _d(w["b0d"]))
    d = ops.silu(ops.mm(d, _d(w["W1d"]).t()) + _d(w["b1d"]))
    d = ops.mm(d, _d(w["w2d"])[:, None])[:, 0] + _d(w["b2d"])
    g = ops.silu(ops.mm(x, _d(w["W0g"]).t()) + _d(w["b0g"]))
    g = ops.silu(ops.mm(g, _d(w["W1g"]).t()) + _d(w["b1g"]))
    g = ops.sigmoid(ops.mm(g, _d(w["w2g"])[:, None])[:, 0] + _d(w["b2g"]))
    return ops.mul(d, g)


def readout_fwd(x, w, elemental, scale):
    """m3g_readout_fwd: atomic (N) = elemental / scale + eps (oracle ``readout``: scaled atomic energies)."""
    return _d(elemental) / scale + readout_eps(x, w)


def readout_upstream(g_atomic, g_scaled_total, g_total, batch, scale, N, device):
    """The upstream gradient of eps per atom: g_atomic + g_scaled_total[b] + scale * g_total[b] (each optional)."""
    ge = torch.zeros(N, dtype=torch.float64, device=device)
    b = batch.long()
    if g_atomic is not None:
        ge = ge + _d(g_atomic)
    if g_scaled_total is not None:
        ge = ge + _d(g_scaled_total)[b]
    if g_total is not None:
        ge = ge + scale * _d(g_total)[b]
    return ge


def readout_bwd(x, w, g_atomic, g_scaled_total, g_total, batch, scale, ops=PLAIN):
    """m3g_readout_bwd: g_x (N,F) = (d eps / d x)^T ge, by autograd (ops = ABS: its scale; pass |upstreams|)."""
    ge = readout_upstream(g_atomic, g_scaled_total, g_total, batch, scale, x.shape[0], x.device)
    return adjoint(lambda x_, o: readout_eps(x_, w, o), [x], ge, ops)[0]


def conv_mlp_bwd_scale(P, po, src, dst, e, h, w, g_up, mode):
    """Scales of the adjoints (g_e, g_z1, g_h) of tests/conv_oracle.py ``mlp_bwd``: the same gated MLP (``mlp_out``
    after ``z1_of``), its adjoint taken with absolute values (see ``adjoint``)."""
    from tests import conv_oracle as C

    F = e.shape[1]
    g_u = _d(g_up) if mode == 0 else _d(g_up)[src.long()]

    def out(e_, z1_part, h_, ops):
        z1 = z1_part + ops.mm(e_, _d(w["W1e"]).t())
        a1 = ops.silu(z1)
        z2d = ops.mm(a1[:, :F], _d(w["W2d"]).t()) + _d(w["b2d"])
        z2g = ops.mm(a1[:, F:], _d(w["W2g"]).t()) + _d(w["b2g"])
        return ops.mul(ops.mul(ops.silu(z2d), ops.sigmoid(z2g)), ops.mm(h_, _d(w["WhT"])))

    base = C.z1_of(P, po, src, dst, torch.zeros_like(_d(e)), w)  # the gathered projections
    return adjoint(out, [e, base, h], g_u, ABS)


def structure_sum(atomic, atom_ptr, scale):
    """m3g_structure_sum: (scaled total (B), total (B) = scale * scaled total) (oracle ``readout``)."""
    ptr = atom_ptr.long()
    B = ptr.numel() - 1
    b = torch.repeat_interleave(torch.arange(B, device=ptr.device), ptr[1:] - ptr[:-1])
    tot = torch.zeros(B, dtype=torch.float64, device=ptr.device).index_add_(0, b, _d(atomic)[:int(ptr[-1])])
    return tot, scale * tot


# ---------------------------------------------------------------------------------------------------------------------
# per-atom projections: torch.nn.Linear (nn/core.py:30-59), and the split first conv layer of nn/conv.py:63-97
def linear(inp, Wt, bias=None, base=None):
    """m3g_linear_fwd (base = None): out (n,M) = base + in (n,K) Wt (K,M) + bias."""
    out = _d(inp) @ _d(Wt)
    if bias is not None:
        out = out + _d(bias)
    if base is not None:
        out = out + _d(base)
    return out


def linear_bwd_input(g, W, base=None):
    """m3g_linear_bwd_input: out (n,K) = base + g (n,M) W (M,K)."""
    out = _d(g) @ _d(W)
    return out if base is None else out + _d(base)


# ---------------------------------------------------------------------------------------------------------------------
# radial basis: nn/featurizer.py:81-100 (oracle ``radial_basis``).  consts as m3g_radial_* takes them:
# [k_0..k_R | coeff_0..coeff_{R-1} | a_0.. | b_0..], h_m = (f_m + a_m h_{m-1}) / b_m, f_m = coeff_m (s(k_m r) +
# s(k_{m+1} r)) with the normalised sinc s(t) = sin(pi t) / (pi t) (quirk Q2).
def _consts(consts, R):
    c = _d(consts)
    return c[:R + 1], c[R + 1:2 * R + 1], c[2 * R + 1:3 * R + 1], c[3 * R + 1:4 * R + 1]


def _sinc(t, absolute_=False):
    """(s(t), s'(t)); ``absolute_``: the envelopes 1 and (|cos(pi t)| + |s(t)|) / |t| that bound their rounding."""
    zero = t == 0
    ts = torch.where(zero, torch.ones_like(t), t)
    p = math.pi * ts
    s = torch.where(zero, torch.ones_like(t), torch.sin(p) / p)
    c = torch.cos(p)
    if absolute_:
        return torch.ones_like(t), torch.where(zero, torch.zeros_like(t), (c.abs() + s.abs()) / ts.abs())
    return s, torch.where(zero, torch.zeros_like(t), (c - s) / ts)


def radial(dist, consts, R, g_h=None, absolute_=False):
    """m3g_radial_fwd: h (E,R); with g_h, m3g_radial_bwd: g_dist (E) = sum_m g_h[:, m] dh_m/dr.  ``absolute_``: the
    sums of |terms| (|coeff|, |a|, |b|, |g_h| and the sinc envelopes)."""
    k, coeff, a, b = _consts(consts, R)
    r = _d(dist)
    if absolute_:
        coeff, a, b = coeff.abs(), a.abs(), b.abs()
    h, dh = [], []
    s_prev, d_prev = _sinc(k[0] * r, absolute_)
    d_prev = d_prev * k[0].abs() if absolute_ else d_prev * k[0]
    for m in range(R):
        s_next, d_next = _sinc(k[m + 1] * r, absolute_)
        d_next = d_next * (k[m + 1].abs() if absolute_ else k[m + 1])
        f, df = coeff[m] * (s_prev + s_next), coeff[m] * (d_prev + d_next)
        h.append(f if m == 0 else (f + a[m] * h[-1]) / b[m])
        dh.append(df if m == 0 else (df + a[m] * dh[-1]) / b[m])
        s_prev, d_prev = s_next, d_next
    h, dh = torch.stack(h, 1), torch.stack(dh, 1)
    if g_h is None:
        return h
    g = _d(g_h).abs() if absolute_ else _d(g_h)
    return (g * dh).sum(1)


# ---------------------------------------------------------------------------------------------------------------------
# edge adjustor: nn/featurizer.py:128-132 (oracle ``forward``: e = SiLU(h W^T)).  Wt (R,F) = W^T as the kernels take it.
def edge_adjust_fwd(h, Wt, ops=PLAIN):
    """m3g_edge_adjust_fwd: e0 (E,F) = SiLU(h Wt)."""
    return ops.silu(ops.mm(_d(h), _d(Wt)))


def edge_adjust_bwd(h, Wt, g_e0, ops=PLAIN):
    """m3g_edge_adjust_bwd: g_h (E,R) = (g_e0 * SiLU'(h Wt)) Wt^T (ops = ABS: its scale)."""
    return adjoint(lambda h_, o: edge_adjust_fwd(h_, Wt, o), [h], g_e0, ops)[0]


# ---------------------------------------------------------------------------------------------------------------------
# pair geometry: nn/invariant.py:20-59 (oracle ``pair_geometry``).  The bond e = (src i -> dst j, integer image s) has
# v = pos[j] + s . lattice[batch[i]] - pos[i], r = |v|; a triplet (e1, e2) has cos = v1 . v2 / (r1 r2), clamped to
# [-1, 1].  vec4 (E,4) = (v, r) as the kernels keep it.
def geometry_fwd(pos, lattice, batch, src, dst, shift):
    """m3g_geometry_fwd: (vec (E,3), dist (E))."""
    src, dst = src.long(), dst.long()
    L = _d(lattice)[batch.long()[src]]
    v = _d(pos)[dst] + torch.einsum("ea,eac->ec", _d(shift), L) - _d(pos)[src]
    return v, torch.sqrt((v * v).sum(1))


def geometry_bwd(vec4, g_vec4, g_dist, src, dst, N, scale=1.0, absolute_=False):
    """m3g_geometry_bwd: g_pos (N,3) = scale * (sum over bonds into i of g_e - sum over bonds out of i of g_e), with
    g_e = g_vec4.xyz + (g_vec4.w + g_dist) v / r (either gradient may be None).  ``absolute_``: sums of |terms|."""
    v4 = _d(vec4)
    E = v4.shape[0]
    gv = torch.zeros((E, 4), dtype=torch.float64, device=v4.device) if g_vec4 is None else _d(g_vec4)
    gr = gv[:, 3] + (0.0 if g_dist is None else _d(g_dist))
    if absolute_:
        ge = gv[:, :3].abs() + (gv[:, 3].abs() + (0.0 if g_dist is None else _d(g_dist).abs()))[:, None] * \
            v4[:, :3].abs() / v4[:, 3:4]
        sign = 1.0
    else:
        ge = gv[:, :3] + gr[:, None] * v4[:, :3] / v4[:, 3:4]
        sign = -1.0
    out = torch.zeros((N, 3), dtype=torch.float64, device=v4.device)
    out.index_add_(0, dst.long(), ge).index_add_(0, src.long(), sign * ge)
    return abs(scale) * out if absolute_ else scale * out


def angles_fwd(vec4, tri):
    """m3g_angles_fwd: (unclamped cos (T), clamped cos (T))."""
    v4 = _d(vec4)
    a, b = v4[tri[0].long()], v4[tri[1].long()]
    c = (a[:, :3] * b[:, :3]).sum(1) / (a[:, 3] * b[:, 3])
    return c, c.clamp(-1.0, 1.0)


def angles_bwd(vec4, tri, g_cos, passes, absolute_=False):
    """m3g_angles_bwd: g_vec4 (E,4) += the adjoint of cos through the clamp.  ``passes`` (T, bool): where the clamp
    passes the gradient, i.e. where the FORWARD's unclamped cos lies in [-1, 1] (torch.clamp's mask is taken from its
    input).  d cos / d v1 = v2 / (r1 r2), d cos / d r1 = -cos / r1 (r is an independent coordinate of vec4)."""
    v4 = _d(vec4)
    e1, e2 = tri[0].long(), tri[1].long()
    a, b = v4[e1], v4[e2]
    inv = 1.0 / (a[:, 3] * b[:, 3])
    c = (a[:, :3] * b[:, :3]).sum(1) * inv
    g = torch.where(passes, _d(g_cos), torch.zeros_like(inv))
    if absolute_:
        a, b, c, g = a.abs(), b.abs(), c.abs(), g.abs()
    ga = torch.cat([g[:, None] * b[:, :3] * inv[:, None], (-g * c / a[:, 3])[:, None]], 1)
    gb = torch.cat([g[:, None] * a[:, :3] * inv[:, None], (-g * c / b[:, 3])[:, None]], 1)
    if absolute_:
        ga, gb = ga.abs(), gb.abs()
    out = torch.zeros_like(v4)
    return out.index_add_(0, e1, ga).index_add_(0, e2, gb)


# ---------------------------------------------------------------------------------------------------------------------
# forces and virial: nn/gradient.py:40-64 (oracle ``forward``, with_forces)
VOIGT = ((0, 0), (1, 1), (2, 2), (1, 2), (2, 0), (0, 1))  # xx, yy, zz, yz, zx, xy


def det_terms(lattice, absolute_=False):
    """a . (b x c) per structure (B), or its sum of |terms|."""
    L = _d(lattice).reshape(-1, 3, 3)
    if absolute_:
        L = L.abs()
        cx = L[:, 1, 1] * L[:, 2, 2] + L[:, 1, 2] * L[:, 2, 1]
        cy = L[:, 1, 2] * L[:, 2, 0] + L[:, 1, 0] * L[:, 2, 2]
        cz = L[:, 1, 0] * L[:, 2, 1] + L[:, 1, 1] * L[:, 2, 0]
    else:
        cx = L[:, 1, 1] * L[:, 2, 2] - L[:, 1, 2] * L[:, 2, 1]
        cy = L[:, 1, 2] * L[:, 2, 0] - L[:, 1, 0] * L[:, 2, 2]
        cz = L[:, 1, 0] * L[:, 2, 1] - L[:, 1, 1] * L[:, 2, 0]
    return L[:, 0, 0] * cx + L[:, 0, 1] * cy + L[:, 0, 2] * cz


def forces_virial(pos, g_pos, lattice, atom_ptr, absolute_=False):
    """m3g_forces_virial: (forces (N,3) = -g_pos, stresses (B,6) = Voigt of sum_i pos_a F_c / |det lattice|).
    ``absolute_``: the stress's sum of |terms| over |det|, plus |stress| times the determinant's relative scale."""
    ptr = atom_ptr.long()
    B = ptr.numel() - 1
    N = int(ptr[-1])
    p, f = _d(pos)[:N], -_d(g_pos)[:N]
    b = torch.repeat_interleave(torch.arange(B, device=ptr.device), ptr[1:] - ptr[:-1])
    outer = (p.abs()[:, :, None] * f.abs()[:, None, :]) if absolute_ else p[:, :, None] * f[:, None, :]
    s = torch.zeros((B, 3, 3), dtype=torch.float64, device=ptr.device).index_add_(0, b, outer)
    vol = det_terms(lattice).abs()
    st = torch.stack([s[:, a, c] for a, c in VOIGT], 1) / vol[:, None]
    if absolute_:
        plain = forces_virial(pos, g_pos, lattice, atom_ptr)[1]
        st = st + plain.abs() * (det_terms(lattice, True) / vol)[:, None]
    return -_d(g_pos), st


# ---------------------------------------------------------------------------------------------------------------------
# float32 rounding order of m3g_geometry_fwd / m3g_angles_fwd (csrc/geometry.cu: explicit _rn operations, no
# contraction), numpy float32 (IEEE round-to-nearest per operation)
def geometry_f32(pos, lattice, batch, src, dst, shift):
    """(vec (E,3), dist (E)) float32: sh_a = (s0 L0a + s1 L1a) + s2 L2a, v_a = (pos_j,a + sh_a) - pos_i,a,
    r = sqrt((v0 v0 + v1 v1) + v2 v2)."""
    pos = np.asarray(pos, np.float32)
    src, dst = np.asarray(src, np.int64), np.asarray(dst, np.int64)
    L = np.asarray(lattice, np.float32).reshape(-1, 3, 3)[np.asarray(batch, np.int64)[src]]
    s = np.asarray(shift).astype(np.float32)
    sh = (s[:, 0:1] * L[:, 0] + s[:, 1:2] * L[:, 1]) + s[:, 2:3] * L[:, 2]
    v = (pos[dst] + sh) - pos[src]
    r2 = (v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2]
    return v, np.sqrt(r2)


def angles_f32(vec4, tri):
    """(unclamped cos (T), clamped cos (T)) float32: dot = (a0 b0 + a1 b1) + a2 b2, cos = dot / (r_a r_b)."""
    v4 = np.asarray(vec4, np.float32)
    tri = np.asarray(tri, np.int64)
    a, b = v4[tri[0]], v4[tri[1]]
    dot = (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]
    c = dot / (a[:, 3] * b[:, 3])
    return c, np.minimum(np.maximum(c, np.float32(-1)), np.float32(1))


def segment_sum_f32(rows, ptr, perm=None):
    """(N, C) float32: for each i, rows[perm[p]] (perm = None: rows[p]) added one by one for p = ptr[i] .. ptr[i+1]-1,
    from 0 -- the order of m3g_segment_sum_add and of both forms of m3g_conv_gather_gz."""
    rows = np.asarray(rows, np.float32)
    ptr = np.asarray(ptr, np.int64)
    idx = np.arange(rows.shape[0]) if perm is None else np.asarray(perm, np.int64)
    N = ptr.size - 1
    acc = np.zeros((N, rows.shape[1]), np.float32)
    deg = ptr[1:] - ptr[:-1]
    for p in range(int(deg.max(initial=0))):
        live = np.nonzero(deg > p)[0]
        acc[live] = acc[live] + rows[idx[ptr[live] + p]]
    return acc
