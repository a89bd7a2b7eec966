from __future__ import annotations

import os

import torch

from torch_m3gnet_b200._lib import call
from torch_m3gnet_b200.data import MaterialGraphKey as K
from torch_m3gnet_b200.data.material_graph import get_plan
from torch_m3gnet_b200.nn._functions import ConvFn
from torch_m3gnet_b200.nn._packing import PackedWeights, c_, module_params, t_
from torch_m3gnet_b200.nn.core import GatedMLP


# "tc3": tcgen05 3xTF32 (fp32-faithful, default for F = 64 on CUDA), "tc1": plain TF32, "fma": generic fp32 kernels
CONV_PATH = os.environ.get("M3G_CONV_PATH", "tc3")
# backward of the tensor-core gated MLPs: 4 = from the activations the forward leaves behind (SiLU'(z1) and the layer-2
# pre-activations, 1 KB per edge and MLP; default); 2 = forward recomputed inside the backward kernel (no extra memory)
TC_BWD_VARIANT = int(os.environ.get("M3G_TC_BWD_VARIANT", "4"))
# True (default): the tensor-core node MLP sums its messages per source atom inside its epilogue (one partial row per
# 32-row block and atom, csrc/conv_tc.cu mode 2): 256 B / bond less HBM traffic and no E x 64 message pass.  The grouping
# of the sum then follows the 32-row blocks of the batch's bond list, so the same structure in another batch position
# agrees to fp32 rounding instead of bit for bit.  False: messages written row by row and summed in ascending bond order.
MSG_REDUCE = os.environ.get("M3G_CONV_MSG_REDUCE", "1") != "0"
# True (default): the backward from saved activations runs the node and the edge MLP adjoint of a block in one launch
# (m3g_conv_tc_block_bwd), keeping dL/de2 on chip instead of a 256 B / bond write and two reads; bitwise the same
# results.  False: two m3g_conv_tc_bwd_saved launches.
CONV_BWD_FUSED = os.environ.get("M3G_CONV_BWD_FUSED", "1") != "0"


def _tc_images(w1e: torch.Tensor, w2d: torch.Tensor, w2g: torch.Tensor) -> torch.Tensor:
    """hi/lo SWIZZLE_128B operand images of the three weight matrices of one gated MLP (csrc/conv_tc.cu)."""
    out = torch.empty(2 * 128 * 64 + 4 * 64 * 64, dtype=torch.float32, device=w1e.device)
    with torch.cuda.device(w1e.device):
        call("tc_pack_b", w1e.contiguous(), 128, 64, out[0:8192], out[8192:16384])
        call("tc_pack_b", w2d.contiguous(), 64, 64, out[16384:20480], out[20480:24576])
        call("tc_pack_b", w2g.contiguous(), 64, 64, out[24576:28672], out[28672:32768])
    return out


def _tc_images_transposed(w1eT: torch.Tensor, w2dT: torch.Tensor, w2gT: torch.Tensor) -> torch.Tensor:
    """Images of the transposed weights for the adjoint GEMMs: [W2d^T, W2g^T, W1e_dense^T, W1e_gate^T] (hi|lo each)."""
    out = torch.empty(8 * 64 * 64, dtype=torch.float32, device=w1eT.device)
    mats = [w2dT, w2gT, w1eT[:, :64], w1eT[:, 64:]]
    with torch.cuda.device(w1eT.device):
        for i, m in enumerate(mats):
            base = i * 8192
            call("tc_pack_b", m.contiguous(), 64, 64, out[base:base + 4096], out[base + 4096:base + 8192])
    return out


class M3GNetConv(torch.nn.Module):
    """Graph convolution block (reference nn/conv.py:12-97): gated-MLP edge update, then gated-MLP messages
    aggregated on the source atom.  Updates EDGE_ATTR and NODE_FEATURES.

    The first layer acts on cat[x_i, x_j, e]; it is split into per-atom projections of x (one small GEMM per
    block) and a per-edge product with e, so the per-edge work is halved (csrc/conv.cu)."""

    def __init__(self, degree: int, num_node_features: int, num_edge_features: int,
                 device: torch.device | None = None):
        super().__init__()
        if num_node_features != num_edge_features:
            raise ValueError("the fused kernels assume node and edge feature widths are equal "
                             "(build_model always sets num_edge_features = embedding_dim)")
        self.degree = degree
        self.num_node_features = num_node_features
        self.num_edge_features = num_edge_features
        self.num_concat_features = 2 * num_node_features + num_edge_features
        self.concat_edge_update = GatedMLP(self.num_concat_features, [num_edge_features, num_edge_features],
                                           device=device)
        self.edge_linear = torch.nn.Linear(degree, num_edge_features, bias=False, device=device)
        self.concat_node_update = GatedMLP(self.num_concat_features, [num_edge_features, num_node_features],
                                           device=device)
        self.node_linear = torch.nn.Linear(degree, num_node_features, bias=False, device=device)
        self._packed = PackedWeights(module_params(self), self._pack)

    def _pack_mlp(self, mlp: GatedMLP, lin: torch.nn.Linear):
        F = self.num_node_features
        d0, d1 = mlp.linears("dense")
        g0, g1 = mlp.linears("gate")
        w1e = torch.cat([d0.weight[:, 2 * F:], g0.weight[:, 2 * F:]], dim=0).detach()  # (2F, F) (out,in)
        packed = {
            "W1e": w1e.contiguous(), "W1eT": w1e.t().contiguous(),
            "W2d": c_(d1.weight), "W2dT": t_(d1.weight), "b2d": c_(d1.bias),
            "W2g": c_(g1.weight), "W2gT": t_(g1.weight), "b2g": c_(g1.bias),
            "Wh": c_(lin.weight), "WhT": t_(lin.weight),
        }
        if F == 64 and w1e.is_cuda:
            packed["wimg"] = _tc_images(packed["W1e"], packed["W2d"], packed["W2g"])
            packed["wimgT"] = _tc_images_transposed(packed["W1eT"], packed["W2dT"], packed["W2gT"])
        return packed, d0, g0

    def _pack(self):
        F = self.num_node_features
        edge, ed0, eg0 = self._pack_mlp(self.concat_edge_update, self.edge_linear)
        node, nd0, ng0 = self._pack_mlp(self.concat_node_update, self.node_linear)
        zeros = torch.zeros(2 * F, dtype=torch.float32, device=ed0.weight.device)
        # per-atom projection: columns [edge: src(dense|gate) dst(dense|gate) | node: same], bias on the src part
        wp = torch.cat([
            ed0.weight[:, :F], eg0.weight[:, :F], ed0.weight[:, F:2 * F], eg0.weight[:, F:2 * F],
            nd0.weight[:, :F], ng0.weight[:, :F], nd0.weight[:, F:2 * F], ng0.weight[:, F:2 * F],
        ], dim=0).detach()  # (8F, F) (out,in)
        bp = torch.cat([ed0.bias, eg0.bias, zeros, nd0.bias, ng0.bias, zeros]).detach()
        return {"edge": edge, "node": node, "Wp": wp.contiguous(), "WpT": wp.t().contiguous(),
                "bp": bp.contiguous()}

    def forward(self, graph):
        plan = get_plan(graph)
        x, e = ConvFn.apply(graph[K.NODE_FEATURES], graph[K.EDGE_ATTR], graph[K.EDGE_WEIGHTS], plan,
                            self._packed.get())
        graph[K.NODE_FEATURES] = x
        graph[K.EDGE_ATTR] = e
        return graph
