from __future__ import annotations

import torch

from torch_m3gnet_b200._lib import call
from torch_m3gnet_b200.data import MaterialGraphKey as K
from torch_m3gnet_b200.data.material_graph import EdgesNotGrouped, get_plan, regroup_by_source
from torch_m3gnet_b200.nn.invariant import STRAIN_HANDLE

_OUTPUT_KEYS = (K.SCALED_POS, K.SCALED_LATTICE, K.EDGE_DISTANCES, K.TRIPLET_ANGLES, K.EDGE_WEIGHTS,
                K.NODE_FEATURES, K.EDGE_ATTR, K.SCALED_ATOMIC_ENERGIES, K.SCALED_TOTAL_ENERGY, K.TOTAL_ENERGY)


class Gradient(torch.nn.Module):
    """Forces = -dE/dpos and the virial stress (reference nn/gradient.py:11-64).

    The backward pass runs the hand-written adjoint kernels through ``torch.autograd.grad``.  The reference
    keeps the autograd graph (``create_graph=True``) because its training loss differentiates the forces; the
    inference path does not, so by default the outputs are detached after the forces are assembled and the
    saved activations are released (set ``keep_graph = True`` to keep first-order autograd connectivity).

    ``compute_stress = True`` (extension, off by default) also fills ``CELL_STRESS`` (B,3,3) in eV/A^3: the strain
    derivative of the energy sigma = (1/V) dE/d(strain) with positions and lattice rows deformed as r -> r (I + eps),
    ASE's stress convention.  It is one bond-level reduction (m3g_bond_virial) over the bond gradients the force pass
    already forms; ``STRESSES`` keeps the reference's meaning."""

    def __init__(self, model: torch.nn.Module):
        super().__init__()
        self.model = model
        self.keep_graph = False
        self.compute_stress = False
        self._engine = None

    def step_engine(self):
        """The whole-step C executor bound to this model (torch_m3gnet_b200/engine.py), built on first use."""
        if self._engine is None:
            from torch_m3gnet_b200.engine import StepEngine

            object.__setattr__(self, "_engine", StepEngine(self.model))
        return self._engine

    def _forward_regrouped(self, graph):
        """Bonds not grouped by source atom (hand-built graphs; the reference accepts any bond order): evaluate a
        stably regrouped copy and hand every bond-level result back in the caller's order."""
        shadow, rank = regroup_by_source(graph)
        out = self.forward(shadow)
        keys = _OUTPUT_KEYS + (K.ELEMENTAL_ENERGIES, K.FORCES, K.STRESSES)
        if self.compute_stress:
            keys += (K.CELL_STRESS,)
        for k in keys:
            v = out[k]
            if torch.is_tensor(v) and k in (K.EDGE_DISTANCES, K.EDGE_WEIGHTS, K.EDGE_ATTR):
                v = v.index_select(0, rank)
            graph[k] = v
        return graph

    def forward(self, graph):
        pos = graph[K.POS]
        try:
            plan = get_plan(graph)
        except EdgesNotGrouped:
            return self._forward_regrouped(graph)
        if not self.keep_graph:
            engine = self.step_engine()
            if engine.supports(graph, plan):
                # default model shape: forward + hand-written adjoint chain launched from C in one call
                graph = engine.run(graph, plan, stress=self.compute_stress)
                graph._private.clear()
                return graph
        pos.requires_grad_(True)
        strain = None
        if self.compute_stress:
            # a zero strain handle through DistanceAndAngle: GeometryFn.backward returns the stress as its gradient
            strain = torch.zeros((plan.B, 3, 3), dtype=torch.float32, device=pos.device, requires_grad=True)
            graph._private[STRAIN_HANDLE] = strain
        graph = self.model(graph)
        graph._private.pop(STRAIN_HANDLE, None)
        energy = graph[K.TOTAL_ENERGY]
        inputs = (pos,) if strain is None else (pos, strain)
        grads = torch.autograd.grad(energy, inputs, grad_outputs=torch.ones_like(energy), retain_graph=self.keep_graph,
                                    allow_unused=strain is not None)
        g_pos = grads[0]
        pos.requires_grad_(False)
        if strain is not None:
            sigma = grads[1]
            graph[K.CELL_STRESS] = torch.zeros_like(strain) if sigma is None else sigma
        plan = get_plan(graph)
        forces = torch.empty_like(pos)
        stresses = torch.empty((plan.B, 6), dtype=torch.float32, device=pos.device)
        call("forces_virial", pos.detach().contiguous(), g_pos.contiguous(), graph[K.LATTICE].contiguous(),
             plan.atom_ptr, plan.N, plan.B, forces, stresses)
        graph[K.FORCES] = forces
        graph[K.STRESSES] = stresses
        if not self.keep_graph:
            for k in _OUTPUT_KEYS:
                v = graph[k]
                if torch.is_tensor(v):
                    graph[k] = v.detach()
            graph._private.clear()
        return graph
