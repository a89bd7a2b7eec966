"""Whole-step executor binding (``m3g_step_run``, csrc/step.cu; struct ``M3GStepDesc`` in include/m3gnet_b200.h).

``Gradient.forward`` (reference nn/gradient.py:25-64) hands the default model shape to ``StepEngine``: the forward
kernels, the hand-written adjoint kernels in reverse order and the force / virial assembly are launched from C in one
call — the same kernels, in the same order and with the same arithmetic as the ``torch.autograd.Function`` path of
``nn/_functions.py``, without ~70 Python / ctypes round trips, without an autograd pass and without the dead gradient
with respect to the atom embedding.  Anything the executor does not cover (other widths or basis sizes, hand-made or
permuted triplet lists, empty batches, ``keep_graph``) stays on the per-operator path.

The sequence is cut into phases (``M3G_PHASE_*``) so that the domain-decomposed evaluation (``domain.py``) can run its
halo exchanges between them.
"""
from __future__ import annotations

import ctypes
import os
from typing import Dict, List, Optional

import torch

from torch_m3gnet_b200 import _lib
from torch_m3gnet_b200.data import MaterialGraphKey as K

MAX_BLOCKS = 8
_fp = ctypes.c_void_p

# set M3G_ENGINE=0 to force the per-operator (autograd) path
ENABLED = os.environ.get("M3G_ENGINE", "1") != "0"
# e0 = SiLU(h Wa^T) formed inside block 0's three-body edge update instead of being stored and read back
FUSE_E0 = os.environ.get("M3G_FUSE_E0", "1") != "0"


class _Block(ctypes.Structure):
    _fields_ = ([(n, _fp) for n in ("Ws", "bs", "WdT", "WgT", "tb_consts", "WpT", "bp", "Wp", "e_wimg", "e_wimgT",
                                     "e_b2d", "e_b2g", "e_WhT", "n_wimg", "n_wimgT", "n_b2d", "n_b2g", "n_WhT", "G",
                                     "dG")]
                + [("radial_owner", ctypes.c_int)]
                + [(n, _fp) for n in ("sig", "red", "x_in", "e_in", "e_tb", "e_out", "x_out", "save_e", "save_n")])


class _Desc(ctypes.Structure):
    _fields_ = ([(n, ctypes.c_int64) for n in ("N", "E", "T", "B")]
                + [(n, ctypes.c_int) for n in ("n_blocks", "n_sm", "passes", "max_members")]
                + [("n_members", ctypes.c_int64)]
                + [(n, ctypes.c_float) for n in ("length_scale", "energy_scale", "r3")]
                + [("num_types", ctypes.c_int)]
                + [(n, _fp) for n in ("batch", "src", "dst", "shift", "types", "edge_ptr", "in_ptr", "in_perm",
                                      "tri_ptr", "atom_ptr", "member_edges", "tri_index", "pos", "lattice", "embed_W",
                                      "atomref_table", "radial_consts", "adjust_Wt", "ro_W0dT", "ro_b0d", "ro_W1dT",
                                      "ro_b1d", "ro_w2d", "ro_b2d", "ro_W0gT", "ro_b0g", "ro_W1gT", "ro_b1g", "ro_w2g",
                                      "ro_b2g", "ro_W0d", "ro_W1d", "ro_W0g", "ro_W1g", "g_total", "scaled_pos",
                                      "scaled_lattice", "elemental", "vec4", "dist", "cos_t", "x0", "h", "e0",
                                      "atomic", "scaled_total", "total", "forces", "stresses", "P", "msg")]
                + [("g_x", _fp * 2), ("g_e", _fp * 2)]
                + [(n, _fp) for n in ("ge2", "gz_edge", "gz_node", "gP", "g_h", "g_hs", "g_sig_e", "g_vec4", "g_dist",
                                      "g_pos")]
                + [(n, ctypes.c_int) for n in ("cur_x", "cur_e", "have_g_e", "msg_reduce", "tb_split",
                                               "tb_bwd_split", "fuse_e0", "fuse_conv_bwd")]
                + [("blocks", _Block * MAX_BLOCKS)])


def phase_tb(b: int) -> int:
    return 1 + 2 * b


def phase_conv(b: int) -> int:
    return 2 + 2 * b


def phase_readout(n: int) -> int:
    return 1 + 2 * n


def phase_conv_bwd(n: int, b: int) -> int:
    return 2 + 2 * n + 2 * (n - 1 - b)


def phase_tb_bwd(n: int, b: int) -> int:
    return 3 + 2 * n + 2 * (n - 1 - b)


def phase_epilogue(n: int) -> int:
    return 2 + 4 * n


def phase_forces(n: int) -> int:
    return 3 + 4 * n


_SIZE_CHECKED = False


def _check_size():
    global _SIZE_CHECKED
    if not _SIZE_CHECKED:
        want = int(_lib.LIB.load().m3g_step_desc_size())
        if ctypes.sizeof(_Desc) != want:
            raise RuntimeError(f"M3GStepDesc binding is out of date: ctypes {ctypes.sizeof(_Desc)} B vs library {want} B")
        _SIZE_CHECKED = True


def _p(t: Optional[torch.Tensor]):
    return None if t is None else (t.data_ptr() or _lib._dummy(t.device).data_ptr())


class StepEngine:
    """Binds one model (the ``Sequential`` inside ``Gradient``) to the C executor.  ``supports(plan)`` says whether a
    batch can take this path; ``run(graph, plan)`` evaluates it and fills the graph's output keys."""

    def __init__(self, model: torch.nn.Module):
        from torch_m3gnet_b200.nn.atom_ref import AtomRef
        from torch_m3gnet_b200.nn.conv import M3GNetConv
        from torch_m3gnet_b200.nn.featurizer import AtomFeaturizer, EdgeAdjustor, EdgeFeaturizer
        from torch_m3gnet_b200.nn.interaction import ThreeBodyInteration
        from torch_m3gnet_b200.nn.invariant import DistanceAndAngle
        from torch_m3gnet_b200.nn.readout import AtomWiseReadout
        from torch_m3gnet_b200.nn.scale import ScaleLength

        self.ok = False
        self._ones: Dict = {}
        mods = list(model) if isinstance(model, torch.nn.Sequential) else None
        if mods is None or len(mods) < 9 or (len(mods) - 7) % 2:
            return
        head = (ScaleLength, AtomRef, DistanceAndAngle, AtomFeaturizer, EdgeFeaturizer, EdgeAdjustor)
        if not all(isinstance(m, t) for m, t in zip(mods[:6], head)) or not isinstance(mods[-1], AtomWiseReadout):
            return
        body = mods[6:-1]
        tbs, cvs = body[0::2], body[1::2]
        if not all(isinstance(m, ThreeBodyInteration) for m in tbs) or not all(isinstance(m, M3GNetConv) for m in cvs):
            return
        n = len(tbs)
        if n < 1 or n > MAX_BLOCKS:
            return
        self.scale, self.atomref, _, self.embed, self.radial, self.adjust = mods[:6]
        self.tbs, self.cvs, self.readout = tbs, cvs, mods[-1]
        self.n_blocks = n
        shape_ok = (self.radial.degree == 3 and self.adjust.num_edge_features == 64 and self.readout.in_features == 64
                    and all((t.l_max, t.n_max, t.num_node_features, t.num_edge_features) == (3, 3, 64, 64) for t in tbs)
                    and all((c.degree, c.num_node_features, c.num_edge_features) == (3, 64, 64) for c in cvs)
                    and len({float(t.threebody_cutoff) for t in tbs}) == 1)
        if not shape_ok:
            return
        self.ok = True
        _check_size()

    # ------------------------------------------------------------------------------------------------
    def supports(self, graph, plan) -> bool:
        from torch_m3gnet_b200.nn import conv as conv_mod
        from torch_m3gnet_b200.nn import interaction

        return (self.ok and ENABLED and plan.N > 0 and plan.E > 0 and plan.T > 0 and plan.tri_moment
                and interaction.TB_PATH == "moment" and conv_mod.CONV_PATH in ("tc3", "tc1")
                and conv_mod.TC_BWD_VARIANT == 4 and graph[K.POS].dtype == torch.float32)

    # ------------------------------------------------------------------------------------------------
    def prepare(self, graph, plan, g_total: Optional[torch.Tensor] = None):
        """Allocate outputs + scratch and fill the descriptor.  Returns (desc, keep) where ``keep`` holds every tensor the
        descriptor points to (outputs by name under keep["out"])."""
        from torch_m3gnet_b200.nn import conv as conv_mod
        from torch_m3gnet_b200.nn import interaction
        from torch_m3gnet_b200.nn._functions import sm_count

        pos = graph[K.POS].detach().contiguous()
        lat = graph[K.LATTICE].detach()
        lat = (lat if lat.dim() == 3 else lat[None]).contiguous()
        dev = pos.device
        N, E, T, B, n = plan.N, plan.E, plan.T, plan.B, self.n_blocks
        if N * 512 >= 2 ** 32:
            raise ValueError(f"{N} atoms: the per-atom projection table exceeds the kernels' 32-bit row offsets")
        f32 = dict(dtype=torch.float32, device=dev)
        tri_index = graph[K.TRIPLET_EDGE_INDEX]
        out = {
            K.SCALED_POS: torch.empty((N, 3), **f32), K.SCALED_LATTICE: torch.empty((B, 3, 3), **f32),
            K.ELEMENTAL_ENERGIES: torch.empty(N, **f32), K.EDGE_DISTANCES: torch.empty(E, **f32),
            K.TRIPLET_ANGLES: torch.empty(T, **f32) if tri_index is not None else None,
            K.EDGE_WEIGHTS: torch.empty((E, 3), **f32), K.NODE_FEATURES: torch.empty((N, 64), **f32),
            K.EDGE_ATTR: torch.empty((E, 64), **f32), K.SCALED_ATOMIC_ENERGIES: torch.empty(N, **f32),
            K.SCALED_TOTAL_ENERGY: torch.empty(B, **f32), K.TOTAL_ENERGY: torch.empty(B, **f32),
            K.FORCES: torch.empty((N, 3), **f32), K.STRESSES: torch.empty((B, 6), **f32),
        }
        n_save = int(_lib.LIB.load().m3g_conv_tc_save_floats(E))
        fuse_bwd = bool(conv_mod.CONV_BWD_FUSED)
        # scratch: one allocation carved by offsets (floats, every piece 16-byte aligned)
        sizes: List = [("vec4", 4 * E), ("x0", 64 * N), ("e0", 64 * E), ("P", 512 * N), ("msg", 64 * E),
                       ("g_x0", 64 * N), ("g_x1", 64 * N), ("g_e0", 64 * E), ("g_e1", 64 * E), ("gz_edge", 128 * E),
                       ("gz_node", 128 * E), ("gP", 512 * N), ("g_h", 3 * E), ("g_hs", (2 * n + 1) * 3 * E),
                       ("g_sig_e", 9 * E), ("g_vec4", 4 * E), ("g_dist", E), ("g_pos", 3 * N)]
        if not fuse_bwd:  # the fused block backward keeps ge2 on chip
            sizes.append(("ge2", 64 * E))
        tables: Dict = {}
        weights = []
        for b in range(n):
            w = self.tbs[b]._packed.get()
            weights.append((w, self.cvs[b]._packed.get()))
            if w["consts_key"] not in tables:
                tables[w["consts_key"]] = b
                sizes += [(f"G{b}", 9 * E), (f"dG{b}", 9 * E)]
            sizes += [(f"sig{b}", 9 * N), (f"red{b}", 9 * E), (f"e_tb{b}", 64 * E), (f"save_e{b}", n_save),
                      (f"save_n{b}", n_save)]
            if b < n - 1:
                sizes += [(f"x{b + 1}", 64 * N), (f"e{b + 1}", 64 * E)]
        off, total = {}, 0
        for name, sz in sizes:
            off[name] = total
            total += (sz + 3) // 4 * 4
        scratch = torch.empty(max(total, 4), **f32)
        base = scratch.data_ptr()

        def at(name):
            return base + 4 * off[name]

        d = _Desc()
        d.N, d.E, d.T, d.B = N, E, T, B
        d.n_blocks, d.n_sm, d.max_members = n, sm_count(dev), int(plan.max_members)
        d.passes = 3 if conv_mod.CONV_PATH == "tc3" else 1
        d.msg_reduce = int(conv_mod.MSG_REDUCE)
        d.tb_split = int(interaction.TB_SPLIT)
        d.tb_bwd_split = int(interaction.TB_BWD_SPLIT)
        d.fuse_e0 = int(interaction.TB_SPLIT and FUSE_E0)
        d.fuse_conv_bwd = int(fuse_bwd)
        d.n_members = int(plan.n_members)
        d.length_scale, d.energy_scale = float(self.scale.length_scale), float(self.readout.scale)
        d.r3 = float(weights[0][0]["r3"])
        d.num_types = int(self.embed.num_types)
        for name in ("batch", "src", "dst", "shift", "types", "edge_ptr", "in_ptr", "in_perm", "tri_ptr", "atom_ptr",
                     "member_edges"):
            setattr(d, name, _p(getattr(plan, name)))
        tri_c = tri_index.contiguous() if tri_index is not None else None
        d.tri_index = _p(tri_c)
        d.pos, d.lattice = _p(pos), _p(lat)
        embed_w = self.embed._packed.get()["W"]
        table = self.atomref.elemental_energies.detach().to(device=dev, dtype=torch.float32).contiguous()
        plan.check_types(int(table.numel()), "the elemental-energy table")
        plan.check_types(int(self.embed.num_types), "the atom embedding (num_types)")
        consts = self.radial._device_consts(dev)
        adjust_wt = self.adjust._packed.get()["Wt"]
        d.embed_W, d.atomref_table, d.radial_consts, d.adjust_Wt = _p(embed_w), _p(table), _p(consts), _p(adjust_wt)
        ro = self.readout._packed.get()
        for key in ("W0dT", "b0d", "W1dT", "b1d", "w2d", "b2d", "W0gT", "b0g", "W1gT", "b1g", "w2g", "b2g", "W0d", "W1d",
                    "W0g", "W1g"):
            setattr(d, "ro_" + key, _p(ro[key]))
        if g_total is None:
            g_total = self._ones.get((dev, B))
            if g_total is None:
                g_total = self._ones[(dev, B)] = torch.ones(B, **f32)
        d.g_total = _p(g_total)
        d.scaled_pos, d.scaled_lattice = _p(out[K.SCALED_POS]), _p(out[K.SCALED_LATTICE])
        d.elemental, d.dist, d.cos_t = _p(out[K.ELEMENTAL_ENERGIES]), _p(out[K.EDGE_DISTANCES]), _p(out[K.TRIPLET_ANGLES])
        d.h = _p(out[K.EDGE_WEIGHTS])
        d.atomic, d.scaled_total, d.total = (_p(out[K.SCALED_ATOMIC_ENERGIES]), _p(out[K.SCALED_TOTAL_ENERGY]),
                                             _p(out[K.TOTAL_ENERGY]))
        d.forces, d.stresses = _p(out[K.FORCES]), _p(out[K.STRESSES])
        for name in ("vec4", "x0", "e0", "P", "msg", "gz_edge", "gz_node", "gP", "g_h", "g_hs", "g_sig_e", "g_vec4",
                     "g_dist", "g_pos"):
            setattr(d, name, at(name))
        d.ge2 = None if fuse_bwd else at("ge2")
        d.g_x[0], d.g_x[1] = at("g_x0"), at("g_x1")
        d.g_e[0], d.g_e[1] = at("g_e0"), at("g_e1")
        x_final, e_final = out[K.NODE_FEATURES].data_ptr(), out[K.EDGE_ATTR].data_ptr()
        for b in range(n):
            tw, cw = weights[b]
            k = d.blocks[b]
            k.Ws, k.bs, k.WdT, k.WgT, k.tb_consts = _p(tw["Ws"]), _p(tw["bs"]), _p(tw["WdT"]), _p(tw["WgT"]), _p(tw["consts"])
            k.WpT, k.bp, k.Wp = _p(cw["WpT"]), _p(cw["bp"]), _p(cw["Wp"])
            ed, nd = cw["edge"], cw["node"]
            k.e_wimg, k.e_wimgT, k.e_b2d, k.e_b2g, k.e_WhT = (_p(ed["wimg"]), _p(ed["wimgT"]), _p(ed["b2d"]),
                                                              _p(ed["b2g"]), _p(ed["WhT"]))
            k.n_wimg, k.n_wimgT, k.n_b2d, k.n_b2g, k.n_WhT = (_p(nd["wimg"]), _p(nd["wimgT"]), _p(nd["b2d"]),
                                                              _p(nd["b2g"]), _p(nd["WhT"]))
            owner = tables[tw["consts_key"]]
            k.G, k.dG, k.radial_owner = at(f"G{owner}"), at(f"dG{owner}"), int(owner == b)
            k.sig, k.red = at(f"sig{b}"), at(f"red{b}")
            k.x_in = at(f"x{b}")
            k.e_in = at(f"e{b}")
            k.e_tb = at(f"e_tb{b}")
            k.e_out = e_final if b == n - 1 else at(f"e{b + 1}")
            k.x_out = x_final if b == n - 1 else at(f"x{b + 1}")
            k.save_e, k.save_n = at(f"save_e{b}"), at(f"save_n{b}")
        keep = {"out": out, "scratch": scratch, "off": off, "weights": (weights, embed_w, table, consts, adjust_wt, ro),
                "inputs": (pos, lat, tri_c, g_total), "plan": plan}
        return d, keep

    @staticmethod
    def run_phases(desc, first: int, last: int, device) -> None:
        lib = _lib.LIB.load()
        index = device.index if device.index is not None else torch.cuda.current_device()
        with torch.cuda.device(index):
            stream = _lib._raw_stream(index)
            rc = lib.m3g_step_run(ctypes.byref(desc), int(first), int(last), stream)
        _lib.CALLS += 1
        if rc != 0:
            raise RuntimeError(f"m3g_step_run failed ({rc}): {lib.m3g_last_error().decode()}")

    def launches(self, with_angles: bool = True, stress: bool = False) -> int:
        """Kernel launches of one full step (for bench.py's gpu_launches): prologue 7 (6 when e0 is formed inside the first three-body edge update; +1 for the cos output) + one
        radial table per distinct constant set, 6 per block forward, 2 for the readout with its adjoint, 7 per block
        backward (3 for block 0, whose node-feature gradient is dead; one less per block when the node and edge MLP
        adjoints run as one launch; +1 per block with the split three-body adjoint), 4 in the epilogue, 2 for forces +
        virial; +2 for the cell stress (m3g_bond_virial) when ``stress`` is set."""
        n = self.n_blocks
        tables = len({t._packed.get()["consts_key"] for t in self.tbs})
        from torch_m3gnet_b200.nn import conv as conv_mod
        from torch_m3gnet_b200.nn import interaction

        return (7 - int(interaction.TB_SPLIT and FUSE_E0) + int(with_angles) + tables + (6 + int(interaction.TB_SPLIT)) * n + 2
                + ((7 - int(conv_mod.CONV_BWD_FUSED)) * n - 4 + int(interaction.TB_BWD_SPLIT) * n) + 4 + 2
                + 2 * int(stress))

    @staticmethod
    def cell_stress(keep) -> torch.Tensor:
        """sigma (B,3,3) from the bond vectors and bond gradients the epilogue fed to m3g_geometry_bwd (still in the
        scratch after the forces phase); volume from the unscaled lattice."""
        from torch_m3gnet_b200.nn._functions import cell_stress

        scratch, off, plan = keep["scratch"], keep["off"], keep["plan"]
        E = plan.E

        def view(name, n):
            return scratch[off[name]:off[name] + n]

        lat = keep["inputs"][1]
        with torch.cuda.device(scratch.device):
            return cell_stress(view("vec4", 4 * E), view("g_vec4", 4 * E), view("g_dist", E), plan, lat)

    def run(self, graph, plan, stress: bool = False):
        desc, keep = self.prepare(graph, plan)
        self.run_phases(desc, 0, phase_forces(self.n_blocks), graph[K.POS].device)
        _lib.LAUNCHES += self.launches(keep["out"][K.TRIPLET_ANGLES] is not None)  # the stress call counts its own
        if stress:
            keep["out"][K.CELL_STRESS] = self.cell_stress(keep)
        for k, v in keep["out"].items():
            graph[k] = v
        # the scratch (activations, adjoints) goes back to the caching allocator here; stream order makes that safe
        return graph
