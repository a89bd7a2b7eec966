from __future__ import annotations

import torch

from torch_m3gnet_b200.data import MaterialGraphKey as K
from torch_m3gnet_b200.data.material_graph import get_plan
from torch_m3gnet_b200.nn._functions import GeometryFn

PAIR_VEC4 = "_pair_vec4"  # private: (E,4) = (r_ij vector, |r_ij|), consumed by the three-body kernels
# private: (B,3,3) zeros requiring grad, set by Gradient when the cell stress is requested; its gradient is the stress
STRAIN_HANDLE = "_strain_handle"


class DistanceAndAngle(torch.nn.Module):
    """Bond vectors, distances and cos(theta_jik) (reference nn/invariant.py:8-59): supplies EDGE_DISTANCES and
    TRIPLET_ANGLES (the *cosine*, clamped to [-1, 1], in the caller's triplet order).  TRIPLET_ANGLES is an output key
    only (the three-body kernels take their cosines from the bond vectors); it stays None for builder batches created
    with ``want_triplet_index=False``."""

    def forward(self, graph):
        plan = get_plan(graph)
        strain = graph._private.get(STRAIN_HANDLE)
        if strain is None:
            vec4, dist, cos = GeometryFn.apply(graph[K.SCALED_POS], graph[K.SCALED_LATTICE], plan,
                                               graph[K.TRIPLET_EDGE_INDEX])
        else:
            vec4, dist, cos = GeometryFn.apply(graph[K.SCALED_POS], graph[K.SCALED_LATTICE], plan,
                                               graph[K.TRIPLET_EDGE_INDEX], strain, graph[K.LATTICE])
        graph._private[PAIR_VEC4] = vec4
        graph[K.EDGE_DISTANCES] = dist
        graph[K.TRIPLET_ANGLES] = cos
        return graph
