"""torch.autograd.Functions over the C-ABI kernels (forward kernels + hand-written adjoint kernels).

Only input gradients that lead back to the atomic positions are produced (forces = -dE/dpos).  Weight gradients
are not produced (the kernels read detached, re-laid-out copies of the parameters), and every ``backward`` is
``once_differentiable``: asking for a double backward (the reference's ``create_graph=True`` training path,
nn/gradient.py:33) raises instead of returning silently wrong gradients.
"""
from __future__ import annotations

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from torch_m3gnet_b200 import _lib
from torch_m3gnet_b200._lib import call


_SM_COUNT = {}


def sm_count(device) -> int:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _SM_COUNT:
        _SM_COUNT[idx] = torch.cuda.get_device_properties(idx).multi_processor_count
    return _SM_COUNT[idx]


def tb_path() -> str:
    from torch_m3gnet_b200.nn import interaction

    return interaction.TB_PATH


def tc_bwd_variant() -> int:
    from torch_m3gnet_b200.nn import conv

    return conv.TC_BWD_VARIANT


def msg_reduce() -> bool:
    from torch_m3gnet_b200.nn import conv

    return conv.MSG_REDUCE


def conv_bwd_fused() -> bool:
    from torch_m3gnet_b200.nn import conv

    return conv.CONV_BWD_FUSED


def conv_path() -> str:
    from torch_m3gnet_b200.nn import conv

    return conv.CONV_PATH


def _c(t):
    return None if t is None else t.contiguous()


def _empty(shape, like, dtype=torch.float32):
    return torch.empty(shape, dtype=dtype, device=like.device)


class ScaleFn(Function):
    """nn/scale.py:24-29: out = in / length_scale."""

    @staticmethod
    def forward(ctx, t, length_scale: float):
        ctx.length_scale = float(length_scale)
        t = t.contiguous()
        out = torch.empty_like(t)
        call("scale_fwd", t, out, t.numel(), ctx.length_scale)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        g = g.contiguous()
        out = torch.empty_like(g)
        call("scale_fwd", g, out, g.numel(), ctx.length_scale)
        return out, None


class GeometryFn(Function):
    """nn/invariant.py:20-59 → (vec4 (E,4) = (v, |v|), distances (E), clamped cos (T))."""

    @staticmethod
    def forward(ctx, pos, lattice, plan, tri_index, strain=None, cell=None):
        """``strain`` (optional, (B,3,3) zeros requiring grad): a handle whose gradient is the cell stress
        sigma = (1/V) dE/d(strain) of ``cell_stress`` (``cell`` = the unscaled lattice, for V); it does not enter the
        forward values."""
        ctx.set_materialize_grads(False)
        pos = pos.contiguous()
        lattice = lattice.contiguous()
        E, T = plan.E, plan.T
        vec4 = _empty((E, 4), pos)
        dist = _empty((E,), pos)
        call("geometry_fwd", pos, lattice, plan.batch, plan.src, plan.dst, plan.shift, E, vec4, dist)
        cos = None
        if tri_index is not None:  # builder batches made without the (2,T) API list carry no TRIPLET_ANGLES output
            cos = _empty((T,), pos)
            tri_index = tri_index.contiguous()
            call("angles_fwd", vec4, tri_index, T, cos)
        ctx.plan = plan
        ctx.tri_index = tri_index
        ctx.cell = None if strain is None else cell.detach().reshape(-1, 3, 3).contiguous()
        ctx.save_for_backward(vec4)
        return vec4, dist, cos

    @staticmethod
    @once_differentiable
    def backward(ctx, g_vec4, g_dist, g_cos):
        (vec4,) = ctx.saved_tensors
        plan = ctx.plan
        g_vec4, g_dist = _c(g_vec4), _c(g_dist)
        if g_cos is not None:
            g_vec4 = torch.zeros_like(vec4) if g_vec4 is None else g_vec4.clone()
            call("angles_bwd", vec4, ctx.tri_index, g_cos.contiguous(), plan.T, g_vec4)
        g_pos = _empty((plan.N, 3), vec4)
        call("geometry_bwd", vec4, g_vec4, g_dist, plan.edge_ptr, plan.in_ptr, plan.in_perm, plan.N, 1.0, g_pos)
        g_strain = None
        if ctx.cell is not None and ctx.needs_input_grad[4]:
            g_strain = cell_stress(vec4, g_vec4, g_dist, plan, ctx.cell)
        return g_pos, None, None, None, g_strain, None


def cell_stress(vec4, g_vec4, g_dist, plan, cell):
    """sigma (B,3,3) = (1/V) sum_{bonds of b} v (x) dE/dv  (m3g_bond_virial): the strain derivative of the energy per
    structure in eV/A^3, from the bond-gradient inputs of m3g_geometry_bwd (g_vec4 / g_dist may be None); ``cell`` is
    the (B,3,3) lattice in A."""
    B = plan.B
    work = torch.empty(max(_lib.bond_virial_work_elems(plan.E, B), 1), dtype=torch.float64, device=vec4.device)
    sigma = torch.empty((B, 3, 3), dtype=torch.float32, device=vec4.device)
    call("bond_virial", vec4, _c(g_vec4), _c(g_dist), plan.edge_ptr, plan.atom_ptr, plan.E, B,
         cell.to(torch.float32).contiguous(), work, sigma)
    return sigma


class RadialFn(Function):
    """nn/featurizer.py:81-100 → edge_weights (E,R)."""

    @staticmethod
    def forward(ctx, dist, consts, R: int):
        dist = dist.contiguous()
        h = _empty((dist.numel(), R), dist)
        call("radial_fwd", dist, consts, dist.numel(), R, h)
        ctx.R = R
        ctx.save_for_backward(dist, consts)
        return h

    @staticmethod
    @once_differentiable
    def backward(ctx, g_h):
        dist, consts = ctx.saved_tensors
        g = torch.empty_like(dist)
        call("radial_bwd", dist, consts, g_h.contiguous(), dist.numel(), ctx.R, g)
        return g, None, None


class EdgeAdjustFn(Function):
    """nn/featurizer.py:128-132 → e0 = SiLU(h W^T)."""

    @staticmethod
    def forward(ctx, h, Wt):
        h = h.contiguous()
        E, R = h.shape
        F = Wt.shape[1]
        e0 = _empty((E, F), h)
        call("edge_adjust_fwd", h, Wt, E, R, F, e0)
        ctx.save_for_backward(h, Wt)
        return e0

    @staticmethod
    @once_differentiable
    def backward(ctx, g_e0):
        h, Wt = ctx.saved_tensors
        E, R = h.shape
        g_h = torch.empty_like(h)
        call("edge_adjust_bwd", h, Wt, g_e0.contiguous(), E, R, Wt.shape[1], g_h)
        return g_h, None


class ThreeBodyFn(Function):
    """nn/interaction.py:187-223 (see csrc/threebody_moment.cu / threebody_atom.cu / threebody.cu for the data flow).

    ``radial`` = (G, dG) from ``m3g_tb_radial`` (block-invariant, computed once per step by the caller) selects the
    O(n3) moment kernels; the dependence of G on the bond length is differentiated inside ``m3g_tb_mom_bwd``."""

    @staticmethod
    def forward(ctx, x, e, vec4, plan, w, L: int, R: int, radial=None):
        x, e, vec4 = x.contiguous(), e.contiguous(), vec4.contiguous()
        N, F = x.shape
        E = plan.E
        D = L * R
        sig = _empty((N, D), x)
        if (F, D) == (64, 9):
            call("tb_sigma64_fwd", x, w["Ws"], w["bs"], N, sm_count(x.device), sig)
        else:
            call("tb_sigma_fwd", x, w["Ws"], w["bs"], N, F, D, sig)
        red = _empty((E, D), x)
        e_out = torch.empty_like(e)
        moment = radial is not None
        fast = (L, R, F) == (3, 3, 64) and tb_path() in ("fast", "atom", "moment")
        atom = fast and tb_path() in ("atom", "moment") and plan.tri_dense and not moment
        bas = None
        if moment:
            G = radial[0]
            from torch_m3gnet_b200.nn import interaction

            if interaction.TB_SPLIT:
                call("tb_mom_red", vec4, G, sig, plan.dst, plan.edge_ptr, plan.tri_ptr, w["r3"], plan.N,
                     plan.max_members, sm_count(x.device), red)
                call("tb_edge_update", red, plan.tri_ptr, w["WdT"], w["WgT"], e, E, sm_count(x.device), e_out)
            else:
                call("tb_mom_fwd", vec4, G, sig, plan.dst, plan.edge_ptr, plan.tri_ptr, w["r3"], w["WdT"], w["WgT"], e,
                     plan.N, plan.max_members, sm_count(x.device), red, e_out)
        else:
            bas = _empty((E, D), x)
            call("tb_edge_basis_fwd", vec4, plan.dst, sig, w["consts"], E, L, R, plan.member_edges, plan.n_members,
                 bas)
            if atom:
                call("tb_atom_fwd", vec4, bas, plan.edge_ptr, plan.tri_ptr, w["r3"], w["WdT"], w["WgT"], e, plan.N,
                     sm_count(x.device), red, e_out)
            elif fast:
                call("tb_reduce_fwd_fast", vec4, bas, plan.tri_ptr, plan.tri_e2, w["r3"], w["WdT"], w["WgT"], e, E,
                     plan.tri_group, sm_count(x.device), red, e_out)
            else:
                call("tb_reduce_fwd", vec4, bas, plan.tri_ptr, plan.tri_e2, w["consts"], w["WdT"], w["WgT"], e, E, L,
                     R, F, plan.tri_group, red, e_out)
        ctx.plan, ctx.w, ctx.L, ctx.R, ctx.F, ctx.fast, ctx.atom = plan, w, L, R, F, fast, atom
        ctx.radial = radial
        if moment:
            ctx.save_for_backward(vec4, sig, red)
        else:
            ctx.save_for_backward(vec4, sig, bas, red)
        return e_out

    @staticmethod
    @once_differentiable
    def backward(ctx, g_e):
        plan, w, L, R, F = ctx.plan, ctx.w, ctx.L, ctx.R, ctx.F
        E, N, D = plan.E, plan.N, L * R
        g_e = g_e.contiguous()
        if ctx.radial is not None:
            vec4, sig, red = ctx.saved_tensors
            G, dG = ctx.radial
            g_vec4 = torch.empty_like(vec4)
            g_sig_e = torch.empty_like(red)
            from torch_m3gnet_b200.nn import interaction

            if interaction.TB_BWD_SPLIT:
                q = torch.empty_like(red)  # rows of non-member bonds are never read
                call("tb_mlp_adj", red, g_e, plan.member_edges, plan.n_members, w["WdT"], w["WgT"],
                     sm_count(vec4.device), q)
                call("tb_mom_bwd_q", vec4, G, dG, sig, plan.dst, q, plan.edge_ptr, plan.tri_ptr, w["r3"], N,
                     plan.max_members, sm_count(vec4.device), 0, g_vec4, g_sig_e)
            else:
                call("tb_mom_bwd", vec4, G, dG, sig, plan.dst, red, g_e, plan.edge_ptr, plan.tri_ptr, w["r3"], w["WdT"],
                     w["WgT"], N, plan.max_members, sm_count(vec4.device), 0, g_vec4, g_sig_e)
            g_x = _empty((N, F), vec4)
            call("tb_sigma64_bwd", g_sig_e, plan.in_ptr, plan.in_perm, sig, w["Ws"], None, N, sm_count(vec4.device), g_x)
            return g_x, g_e, g_vec4, None, None, None, None, None
        vec4, sig, bas, red = ctx.saved_tensors
        g_red = torch.empty_like(red)
        g_vec4 = torch.empty_like(vec4)
        g_bas = torch.empty_like(bas)
        if ctx.atom:
            call("tb_atom_bwd", vec4, bas, red, g_e, plan.edge_ptr, plan.tri_ptr, w["r3"], w["WdT"], w["WgT"], N,
                 sm_count(vec4.device), g_vec4, g_bas)
        elif ctx.fast:
            n_sm = sm_count(vec4.device)
            call("tb_gate_bwd_fast", red, g_e, w["WdT"], w["WgT"], plan.tri_ptr, E, n_sm, g_red)
        else:
            call("tb_gate_bwd", red, g_e, w["WdT"], w["WgT"], plan.tri_ptr, E, D, F, g_red)
        if ctx.atom:
            pass
        elif ctx.fast and plan.tri_symmetric:
            call("tb_reduce_bwd_sym", vec4, bas, g_red, plan.tri_ptr, plan.tri_e2, w["r3"], E, plan.tri_group, n_sm,
                 g_vec4, g_bas)
        else:
            call("tb_reduce_bwd", vec4, bas, g_red, plan.tri_ptr, plan.tri_e2, plan.trt_ptr, plan.trt_e1, w["consts"],
                 E, L, R, plan.tri_group, g_vec4, g_bas)
        g_sig_e = g_red  # reuse the buffer: g_red is dead after tb_reduce_bwd
        g_sig_e.zero_()  # rows of bonds without triplets stay zero (only member bonds are evaluated)
        call("tb_edge_basis_bwd", vec4, plan.dst, sig, g_bas, w["consts"], E, L, R, plan.member_edges, plan.n_members,
             g_vec4, g_sig_e)
        g_x = _empty((N, F), vec4)
        call("tb_sigma_bwd", g_sig_e, plan.in_ptr, plan.in_perm, sig, w["Ws"], None, N, F, D, g_x)
        return g_x, g_e, g_vec4, None, None, None, None, None


class ConvFn(Function):
    """nn/conv.py:63-97 → (x', e')."""

    @staticmethod
    def forward(ctx, x, e, h, plan, w):
        ctx.set_materialize_grads(False)
        x, e, h = x.contiguous(), e.contiguous(), h.contiguous()
        N, F = x.shape
        E, R = plan.E, h.shape[1]
        P = _empty((N, 8 * F), x)
        call("linear_fwd", x, w["WpT"], w["bp"], N, F, 8 * F, P)
        e2 = torch.empty_like(e)
        msg = torch.empty_like(e)
        ed, nd = w["edge"], w["node"]
        path = conv_path()
        save_e = save_n = None
        parts = False
        if N * 8 * F >= 2 ** 32:
            raise ValueError(f"{N} atoms: the per-atom projection table exceeds the kernels' 32-bit row offsets")
        if F == 64 and "wimg" in ed and path in ("tc3", "tc1") and R <= 4:
            passes = 3 if path == "tc3" else 1
            n_sm = sm_count(x.device)
            if tc_bwd_variant() == 4 and R <= 3 and any(ctx.needs_input_grad[:3]):
                # activations for the backward (1 KB per edge and MLP): SiLU'(z1) and the layer-2 pre-activations
                n_save = int(_lib.LIB.load().m3g_conv_tc_save_floats(E))
                save_e, save_n = _empty((n_save,), x), _empty((n_save,), x)
            call("conv_tc_fwd", P, 8 * F, 0, plan.src, plan.dst, e, h, ed["wimg"], ed["b2d"], ed["b2g"], ed["WhT"], E, R,
                 0, passes, n_sm, e2, save_e)
            # mode 2: the messages are reduced per source atom inside the kernel's epilogue; msg holds one partial
            # row per (32-row block, atom)
            call("conv_tc_fwd", P, 8 * F, 4 * F, plan.src, plan.dst, e2, h, nd["wimg"], nd["b2d"], nd["b2g"], nd["WhT"],
                 E, R, 2 if msg_reduce() else 1, passes, n_sm, msg, save_n)
            parts = msg_reduce()
        else:
            call("conv_mlp_fwd", P, 8 * F, 0, plan.src, plan.dst, e, h, ed["W1eT"], ed["W2dT"], ed["b2d"], ed["W2gT"],
                 ed["b2g"], ed["WhT"], E, F, R, 0, e2)
            call("conv_mlp_fwd", P, 8 * F, 4 * F, plan.src, plan.dst, e2, h, nd["W1eT"], nd["W2dT"], nd["b2d"],
                 nd["W2gT"], nd["b2g"], nd["WhT"], E, F, R, 1, msg)
        x2 = torch.empty_like(x)
        call("segment_sum_parts" if parts else "segment_sum_add", x, msg, plan.edge_ptr, N, F, x2)
        ctx.plan, ctx.w = plan, w
        ctx.saved_acts = (save_e, save_n)
        ctx.save_for_backward(x, e, e2, h, P)
        return x2, e2

    @staticmethod
    @once_differentiable
    def backward(ctx, g_x2, g_e2):
        x, e, e2, h, P = ctx.saved_tensors
        plan, w = ctx.plan, ctx.w
        N, F = x.shape
        E, R = plan.E, h.shape[1]
        if g_x2 is None:
            g_x2 = torch.zeros_like(x)
        g_x2, g_e2 = g_x2.contiguous(), _c(g_e2)
        g_h = torch.zeros_like(h)
        nd, ed = w["node"], w["edge"]
        gz_node = _empty((E, 2 * F), x)
        g_e = torch.empty_like(e)
        gz_edge = _empty((E, 2 * F), x)
        path = conv_path()
        save_e, save_n = ctx.saved_acts
        if save_e is not None:
            passes = 3 if path == "tc3" else 1
            n_sm = sm_count(x.device)
            if conv_bwd_fused():
                # g_h = fl(node + edge) rows, as the two launches below leave them
                call("conv_tc_block_bwd", plan.src, h, nd["wimgT"], nd["WhT"], save_n, ed["wimgT"], ed["WhT"], save_e,
                     g_x2, g_e2, E, R, passes, n_sm, g_e, gz_node, gz_edge, g_h, None, 1)
            else:
                ge2 = torch.empty_like(e)
                # g_h: the node launch stores its rows, the edge launch adds to them (no zero fill needed)
                call("conv_tc_bwd_saved", plan.src, h, nd["wimgT"], nd["WhT"], save_n, g_x2, g_e2, E, R, 1, passes, n_sm,
                     ge2, gz_node, g_h, 1)
                call("conv_tc_bwd_saved", plan.src, h, ed["wimgT"], ed["WhT"], save_e, ge2, ge2, E, R, 0, passes, n_sm,
                     g_e, gz_edge, g_h, 0)
            ctx.saved_acts = (None, None)
        elif F == 64 and "wimgT" in ed and path in ("tc3", "tc1") and R <= 3:
            ge2 = torch.empty_like(e)
            passes = 3 if path == "tc3" else 1
            n_sm = sm_count(x.device)
            call("conv_tc_bwd", P, 8 * F, 4 * F, plan.src, plan.dst, e2, h, nd["wimg"], nd["wimgT"], nd["b2d"], nd["b2g"],
                 nd["WhT"], g_x2, g_e2, E, R, 1, passes, n_sm, ge2, gz_node, g_h)
            call("conv_tc_bwd", P, 8 * F, 0, plan.src, plan.dst, e, h, ed["wimg"], ed["wimgT"], ed["b2d"], ed["b2g"],
                 ed["WhT"], ge2, ge2, E, R, 0, passes, n_sm, g_e, gz_edge, g_h)
        else:
            ge2 = torch.empty_like(e)
            call("conv_mlp_bwd", P, 8 * F, 4 * F, plan.src, plan.dst, e2, h, nd["W1eT"], nd["W2dT"], nd["b2d"],
                 nd["W2gT"], nd["b2g"], nd["WhT"], nd["W1e"], nd["W2d"], nd["W2g"], nd["Wh"], g_x2, g_e2, E, F, R, 1,
                 ge2, gz_node, g_h)
            call("conv_mlp_bwd", P, 8 * F, 0, plan.src, plan.dst, e, h, ed["W1eT"], ed["W2dT"], ed["b2d"], ed["W2gT"],
                 ed["b2g"], ed["WhT"], ed["W1e"], ed["W2d"], ed["W2g"], ed["Wh"], ge2, ge2, E, F, R, 0, g_e, gz_edge,
                 g_h)
        gP = _empty((N, 8 * F), x)
        call("conv_gather_gz", gz_edge, plan.edge_ptr, plan.in_ptr, plan.in_perm, N, F, 8 * F, 0, gP)
        call("conv_gather_gz", gz_node, plan.edge_ptr, plan.in_ptr, plan.in_perm, N, F, 8 * F, 4 * F, gP)
        g_x = torch.empty_like(x)
        call("linear_bwd_input", gP, w["Wp"], g_x2, N, F, 8 * F, g_x)
        return g_x, g_e, g_h, None, None


class ReadoutFn(Function):
    """nn/readout.py:39-58 → (scaled atomic energies (N), scaled total (B), total (B))."""

    @staticmethod
    def forward(ctx, x, elemental, plan, w, scale: float):
        ctx.set_materialize_grads(False)
        x = x.contiguous()
        N, F = x.shape
        atomic = _empty((N,), x)
        call("readout_fwd", x, w["W0dT"], w["b0d"], w["W1dT"], w["b1d"], w["w2d"], w["b2d"], w["W0gT"], w["b0g"],
             w["W1gT"], w["b1g"], w["w2g"], w["b2g"], elemental.contiguous(), float(scale), N, F, atomic)
        stot = _empty((plan.B,), x)
        tot = _empty((plan.B,), x)
        call("structure_sum", atomic, plan.atom_ptr, plan.B, float(scale), stot, tot)
        ctx.plan, ctx.w, ctx.scale = plan, w, float(scale)
        ctx.save_for_backward(x)
        return atomic, stot, tot

    @staticmethod
    @once_differentiable
    def backward(ctx, g_atomic, g_stot, g_tot):
        (x,) = ctx.saved_tensors
        plan, w = ctx.plan, ctx.w
        N, F = x.shape
        g_x = torch.empty_like(x)
        call("readout_bwd", x, w["W0dT"], w["b0d"], w["W1dT"], w["b1d"], w["w2d"], w["b2d"], w["W0gT"], w["b0g"],
             w["W1gT"], w["b1g"], w["w2g"], w["b2g"], w["W0d"], w["W1d"], w["W0g"], w["W1g"], _c(g_atomic), _c(g_stot),
             _c(g_tot), plan.batch, ctx.scale, N, F, g_x)
        return g_x, None, None, None, None


class SphericalBesselFn(Function):
    """nn/interaction.py:284-350 (elementwise operator API)."""

    @staticmethod
    def forward(ctx, x, order: int):
        x = x.contiguous()
        out, dout = torch.empty_like(x), torch.empty_like(x)
        call("sph_bessel", x, int(order), x.numel(), out, dout)
        ctx.save_for_backward(dout)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, go):
        (dout,) = ctx.saved_tensors
        return dout * go, None


class LegendreCosFn(Function):
    """nn/interaction.py:353-382 incl. the grad_output-per-level backward (quirk Q3)."""

    @staticmethod
    def forward(ctx, x, order: int):
        x = x.contiguous()
        out = torch.empty_like(x)
        call("legendre", x, int(order), x.numel(), out)
        ctx.order = int(order)
        ctx.save_for_backward(x)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, go):
        (x,) = ctx.saved_tensors
        gx = torch.empty_like(x)
        call("legendre_bwd", x, go.contiguous(), ctx.order, x.numel(), gx)
        return gx, None


class CutoffFn(Function):
    """nn/interaction.py:389-400."""

    @staticmethod
    def forward(ctx, r, rc: float):
        r = r.contiguous()
        out, dout = torch.empty_like(r), torch.empty_like(r)
        call("cutoff", r, float(rc), r.numel(), out, dout)
        ctx.save_for_backward(dout)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, go):
        (dout,) = ctx.saved_tensors
        return dout * go, None


class LinearFn(Function):
    """torch.nn.Linear inside a GatedMLP that is called on its own (reference nn/core.py:30-59): out = in W^T + b."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        x2 = x.contiguous().reshape(-1, x.shape[-1])
        n, K = x2.shape
        M = weight.shape[0]
        wt = weight.detach().t().contiguous()
        out = _empty((n, M), x2)
        call("linear_fwd", x2, wt, None if bias is None else bias.detach().contiguous(), n, K, M, out)
        ctx.save_for_backward(weight.detach().contiguous())
        ctx.shape = x.shape
        return out.reshape(x.shape[:-1] + (M,))

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (w,) = ctx.saved_tensors
        M, K = w.shape
        g2 = g.contiguous().reshape(-1, M)
        out = _empty((g2.shape[0], K), g2)
        call("linear_bwd_input", g2, w, None, g2.shape[0], K, M, out)
        return out.reshape(ctx.shape), None, None


class ActivationFn(Function):
    """torch.nn.SiLU (kind 0) / torch.nn.Sigmoid (kind 1) of nn/core.py:45-59."""

    @staticmethod
    def forward(ctx, x, kind: int):
        x = x.contiguous()
        out = torch.empty_like(x)
        call("act_fwd", x, x.numel(), int(kind), out)
        ctx.kind = int(kind)
        ctx.save_for_backward(x)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        out = torch.empty_like(x)
        call("act_bwd", x, g.contiguous(), x.numel(), ctx.kind, out)
        return out, None


class MulFn(Function):
    """dense(x) * gate(x) (nn/core.py:61-62)."""

    @staticmethod
    def forward(ctx, a, b):
        a, b = a.contiguous(), b.contiguous()
        out = torch.empty_like(a)
        call("mul", a, b, a.numel(), out)
        ctx.save_for_backward(a, b)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        g = g.contiguous()
        ga, gb = torch.empty_like(a), torch.empty_like(b)
        call("mul", g, b, a.numel(), ga)
        call("mul", g, a, a.numel(), gb)
        return ga, gb
