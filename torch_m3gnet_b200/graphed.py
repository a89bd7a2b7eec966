"""CUDA-graph replay of the energy + forces step for a FIXED graph (SURVEY.md §8(f) rank 2: the inner loop of MD /
relaxation between neighbour-list rebuilds).

For small systems the step is launch-bound: ~60 kernel launches plus the autograd bookkeeping of a 32-atom cell cost
far more host time than GPU time.  ``GraphedStep`` captures one ``model(batch)`` call — forward kernels, the hand-written
adjoint kernels driven by ``torch.autograd.grad``, the force / virial assembly and, when the model's
``compute_stress`` is set, the cell stress (``CELL_STRESS``) — into a CUDA graph and replays it:

    step = GraphedStep(model, batch)          # warm-up + capture (positions / lattice are static buffers)
    out = step()                              # replay with the captured positions
    out = step(pos=new_pos)                   # copy new positions into the static buffer, replay

The neighbour list, triplets and image shifts are those of ``batch``: the caller rebuilds the batch (and the
``GraphedStep``) when atoms have moved further than its skin allows, exactly as with any Verlet list.  Outputs are the
static tensors of the captured call (overwritten by the next replay); clone what must be kept.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from torch_m3gnet_b200.data import MaterialGraphKey as K
from torch_m3gnet_b200.data.material_graph import get_plan

_KEYS = (K.TOTAL_ENERGY, K.FORCES, K.STRESSES, K.SCALED_ATOMIC_ENERGIES, K.SCALED_TOTAL_ENERGY)


class GraphedStep:
    def __init__(self, model: torch.nn.Module, batch, warmup: int = 3):
        pos = batch[K.POS]
        if not pos.is_cuda:
            raise RuntimeError("GraphedStep needs a CUDA batch (there is no CPU path)")
        self.model, self.batch = model, batch
        get_plan(batch)  # integer plan kernels and their host read-backs happen outside the capture
        self._pos = batch[K.POS]
        self._lattice = batch[K.LATTICE]
        side = torch.cuda.Stream(device=pos.device)
        side.wait_stream(torch.cuda.current_stream(pos.device))
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 1)):  # allocator warm-up, weight packing, cudaFuncSetAttribute calls
                model(batch)
        torch.cuda.current_stream(pos.device).wait_stream(side)
        torch.cuda.synchronize(pos.device)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            out = model(batch)
        keys = _KEYS + ((K.CELL_STRESS,) if getattr(model, "compute_stress", False) else ())
        self.out: Dict[str, torch.Tensor] = {k: out[k] for k in keys}
        # the captured launches hold the device addresses of the packed weight images / constant tables that existed
        # at capture time; remember what they were made from so that a later parameter edit is noticed
        self._weights = self._weight_signature()

    def _weight_signature(self):
        sig = []
        for m in self.model.modules():
            packed = getattr(m, "_packed", None)
            if packed is not None:
                sig.append(tuple((p.data_ptr(), p._version, p.device) for p in packed._params()))
            table = getattr(m, "elemental_energies", None)
            if torch.is_tensor(table):
                sig.append((table.data_ptr(), table._version, table.device))
        return tuple(sig)

    def stale(self) -> bool:
        """True when a parameter / constant table the capture depends on was replaced or modified since
        (``load_state_dict``, an optimizer step, an edit of ``nsb.factors`` or ``elemental_energies``)."""
        return self._weight_signature() != self._weights

    @torch.no_grad()
    def __call__(self, pos: Optional[torch.Tensor] = None, lattice: Optional[torch.Tensor] = None):
        if self.stale():
            raise RuntimeError("the model's parameters changed after this GraphedStep was captured: build a new "
                               "GraphedStep (the captured launches still point at the old packed weights)")
        if pos is not None:
            self._pos.copy_(pos)
        if lattice is not None:
            self._lattice.copy_(lattice)
        self.graph.replay()
        return self.out
