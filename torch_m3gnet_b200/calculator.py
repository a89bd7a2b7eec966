"""Trajectory-side callers of the hot path (SURVEY.md §8(f) rank 2): an ASE-style calculator, a velocity-Verlet
driver and a FIRE relaxation that keep coordinates, neighbour candidates and results on the GPU between steps.

The reference has no driver loop of its own (its ``scripts/relax_org.py`` uses the TensorFlow package); a user would
call ``MaterialGraph.from_structure`` + ``model(graph)`` per frame (README usage, torch_m3gnet/data/material_graph.py:
132-165).  ``M3GNetCalculator`` does the same per frame through ``VerletList`` (bit-identical graphs, see
data/verlet.py) and the unchanged model, so every frame's energy / forces / stress are those of a fresh
``Batch.from_arrays`` + ``model(batch)`` call.

``M3GNetCalculator`` follows ASE's calculator protocol by duck typing (``calculate(atoms, properties,
system_changes)``, ``results``, ``get_potential_energy / get_forces``) without importing ase: ``atoms`` only
needs ``get_cell()``, ``get_positions()`` and ``get_atomic_numbers()`` (``numpy`` arrays, Å).
"""
from __future__ import annotations

import contextlib
import os
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from torch_m3gnet_b200.data import MaterialGraphKey as K
from torch_m3gnet_b200.data.verlet import VerletList

# 1 eV / (A amu) in A / fs^2: e [J/eV] * 1e20 [A^2/m^2] / (amu [kg] * 1e30 [fs^2/s^2])  (CODATA 2018) = 9.6485332e-3
ACC_UNIT = 1.602176634e-19 * 1e20 / (1.66053906660e-27 * 1e30)


def stabilise_allocator() -> bool:
    """Round CUDA allocation sizes to 1/16 of a power of two (PyTorch's ``roundup_power2_divisions:16``).

    Along a trajectory the bond and triplet counts change by a fraction of a percent from frame to frame, so every
    bond- or triplet-sized tensor of the step has a new size each time; the caching allocator then keeps calling
    cudaMalloc for blocks that fit nothing later (measured on the 32 000-atom cell: 35-190 ms per step instead of
    15 ms).  With rounded request sizes a handful of block sizes recur.  Process-wide setting; left alone when the
    user already chose an allocator policy through PYTORCH_CUDA_ALLOC_CONF.  Returns whether it was applied."""
    conf = os.environ.get("PYTORCH_CUDA_ALLOC_CONF", "") + os.environ.get("PYTORCH_ALLOC_CONF", "")
    if "roundup_power2_divisions" in conf or "expandable_segments" in conf:
        return False
    setter = getattr(torch._C, "_accelerator_setAllocatorSettings", None)
    if setter is None:
        setter = torch.cuda.memory._set_allocator_settings
    setter("roundup_power2_divisions:16")
    return True


class M3GNetCalculator:
    """Energy (eV), forces (eV/A) and the model's ``stresses`` row (6 components exactly as the reference's
    ``Gradient`` module returns them, nn/gradient.py:39-62 -- same order, sign and units as the reference, not
    re-normalised to ASE's convention) for one structure or a batch; neighbour candidates cached between calls."""

    # "stress" is NOT advertised by default: the model's ``stresses`` row is the reference's origin-dependent
    # sum_i pos_i (x) F_i / V (nn/gradient.py:39-62), whose sign and meaning differ from ASE's +dE/d(strain)/V; it
    # stays available as ``results["m3gnet_stresses"]`` / ``get_reference_stresses``.  ``stress=True`` adds ASE's
    # "stress" from the model's cell stress (Gradient.compute_stress, key CELL_STRESS) to the instance's properties.
    implemented_properties = ("energy", "free_energy", "forces")

    def __init__(self, model: torch.nn.Module, cutoff: float = 5.0, threebody_cutoff: float = 4.0, skin: float = 0.5,
                 device: Optional[torch.device] = None, round_allocations: bool = False, graph_replay: bool = False,
                 replay_after: int = 2, stress: bool = False):
        """``graph_replay=True`` (small systems, relaxations / cold MD): while consecutive frames keep the same bonds,
        images and three-body membership, the step is replayed from a CUDA graph (``GraphedStep``) instead of being
        launched kernel by kernel; outputs are bit-identical to the eager call.  The graph is captured once the bond
        set has been stable for ``replay_after`` frames and dropped when it changes; capturing costs tens of eager steps,
        so the required number of stable frames doubles every time a captured graph had to be dropped.

        ``stress=True``: ``calculate`` also sets ``results["stress"]``, the cell stress sigma = (1/V) dE/d(strain) in
        eV/A^3, in ASE's Voigt order [xx, yy, zz, yz, xz, xy] and sign (pressure = -(xx + yy + zz) / 3)."""
        self.model = model
        self.stress = bool(stress)
        if self.stress:
            self.implemented_properties = type(self).implemented_properties + ("stress",)
        if round_allocations:
            stabilise_allocator()
        self.cutoff, self.threebody_cutoff, self.skin = float(cutoff), float(threebody_cutoff), float(skin)
        self.device = device
        self.results: Dict[str, object] = {}
        self._ase_state = None
        self._list: Optional[VerletList] = None
        self._key = None
        self.graph_replay = bool(graph_replay)
        self.replay_after = max(int(replay_after), 1)
        self._need = self.replay_after  # doubled whenever a captured graph had to be dropped (capture is expensive)
        self._last_frame = None
        self._graphed = None
        self._graphed_stress = False
        self._stable = 0
        self.n_replays = self.n_captures = 0

    @contextlib.contextmanager
    def _stress_mode(self, stress: bool):
        """The model's compute_stress set to ``stress`` for the calls inside (restored afterwards)."""
        prev = getattr(self.model, "compute_stress", False)
        if prev == stress:
            yield
            return
        self.model.compute_stress = stress
        try:
            yield
        finally:
            self.model.compute_stress = prev

    def _eval(self, batch, stress: bool):
        with self._stress_mode(stress):
            return self.model(batch)

    @staticmethod
    def _pick(out, stress: bool, clone: bool = False):
        keys = (K.TOTAL_ENERGY, K.FORCES, K.STRESSES) + ((K.CELL_STRESS,) if stress else ())
        return tuple(out[k].clone() if clone else out[k] for k in keys)

    # ---- array interface: one or several structures, results stay on the device ----
    def compute(self, lattices, cart, atomic_numbers, sizes: Optional[Sequence[int]] = None, with_stress: bool = False):
        """Energy (B,), forces (N,3), stresses (B,6) as CUDA tensors for the frame ``cart`` ((N,3) numpy array or
        float64 CUDA tensor).  The neighbour candidates are reused while composition and lattice are unchanged (a new
        lattice rebuilds them).  ``with_stress=True`` appends the cell stress (B,3,3), eV/A^3 (``CELL_STRESS``)."""
        stress = bool(with_stress)
        z = np.asarray(atomic_numbers, dtype=np.int64).reshape(-1)
        if sizes is None:
            sizes = [z.size]
        lat = np.asarray(lattices, dtype=np.float64).reshape(len(sizes), 3, 3)
        key = (tuple(int(n) for n in sizes), z.tobytes())
        if self._list is None or key != self._key:
            self._list = VerletList(lat, z, sizes, self.cutoff, self.threebody_cutoff, self.skin, device=self.device)
            self._key = key
            self._last_frame, self._graphed, self._stable, self._need = None, None, 0, self.replay_after
        elif not np.array_equal(lat, self._list._lattices_h):
            self._list.set_lattice(lat)
            self._last_frame, self._graphed, self._stable = None, None, 0
        if not self.graph_replay:
            return self._pick(self._eval(self._list.update(cart), stress), stress)
        frame = self._list.filter(cart)
        same = self._last_frame is not None and VerletList.same_bonds(frame, self._last_frame)
        self._last_frame = frame
        if not same:
            if self._graphed is not None:
                self._need = min(2 * self._need, 1 << 20)
            self._graphed, self._stable = None, 0
            return self._pick(self._eval(self._list.assemble(frame), stress), stress)
        self._stable += 1
        if self._graphed is not None and self._graphed_stress != stress:
            self._graphed = None  # captured without (or with) the stress launches: capture again
        if self._graphed is None:
            if self._stable < self._need:
                return self._pick(self._eval(self._list.assemble(frame), stress), stress)
            from torch_m3gnet_b200.graphed import GraphedStep

            with self._stress_mode(stress):
                self._graphed = GraphedStep(self.model, self._list.assemble(frame))
            self._graphed_stress = stress
            self.n_captures += 1
        out = self._graphed(pos=frame[0].to(torch.float32))
        self.n_replays += 1
        # the graph's output buffers are overwritten by the next replay
        return self._pick(out, stress, clone=True)

    @property
    def neighbor_list(self) -> Optional[VerletList]:
        return self._list

    # ---- ASE protocol ----
    def calculate(self, atoms=None, properties=("energy",), system_changes=None):
        if atoms is None:
            raise ValueError("M3GNetCalculator.calculate needs an atoms object")
        unknown = [p for p in properties if p not in self.implemented_properties]
        if unknown:
            raise NotImplementedError(f"properties not implemented: {unknown}")
        cell = np.asarray(atoms.get_cell(), dtype=np.float64).reshape(3, 3)
        pos = np.asarray(atoms.get_positions(), dtype=np.float64)
        numbers = np.asarray(atoms.get_atomic_numbers())
        # unchanged atoms: hand back the cached results (ASE calculators do the same through system_changes); an
        # optimizer asking for energy, then forces, costs one model evaluation
        state = (cell.tobytes(), pos.tobytes(), numbers.tobytes())
        if self.results and self._ase_state == state:
            return self.results
        res = self.compute(cell, pos, numbers, with_stress=self.stress)
        e, f, s = res[:3]
        energy = float(e.reshape(-1)[0].item())
        self.results = {"energy": energy, "free_energy": energy, "forces": f.double().cpu().numpy(),
                        "m3gnet_stresses": s.reshape(-1).double().cpu().numpy()}
        if self.stress:
            self.results["stress"] = voigt(res[3].reshape(3, 3).double().cpu().numpy())
        self._ase_state = state
        return self.results

    def get_potential_energy(self, atoms=None, force_consistent: bool = False):
        return self.calculate(atoms, ("energy",))["energy"]

    def get_forces(self, atoms=None):
        return self.calculate(atoms, ("forces",))["forces"]

    def get_stress(self, atoms=None):
        """ASE's stress (Voigt [xx, yy, zz, yz, xz, xy], eV/A^3); needs ``stress=True``."""
        return self.calculate(atoms, ("stress",))["stress"]

    def get_reference_stresses(self, atoms=None):
        """The reference model's ``stresses`` row (nn/gradient.py:39-62), NOT ASE's stress convention."""
        return self.calculate(atoms, ("energy",))["m3gnet_stresses"]


def voigt(sigma: np.ndarray) -> np.ndarray:
    """(3,3) -> ASE's Voigt order [xx, yy, zz, yz, xz, xy]."""
    return np.array([sigma[0, 0], sigma[1, 1], sigma[2, 2], sigma[1, 2], sigma[0, 2], sigma[0, 1]])


class VelocityVerlet:
    """NVE velocity-Verlet integrator on the GPU (coordinates float64 Å, velocities Å/fs, masses amu, dt fs).

    Per step: one half kick, one drift, one ``calculator.compute`` (Verlet-list filter + model), one half kick; nothing
    but the scalars the caller asks for leaves the device."""

    def __init__(self, calculator: M3GNetCalculator, lattice, cart, atomic_numbers, masses, dt: float = 1.0,
                 velocities=None):
        self.calc = calculator
        self.lattice = np.asarray(lattice, dtype=np.float64).reshape(1, 3, 3)
        self.numbers = np.asarray(atomic_numbers, dtype=np.int64).reshape(-1)
        dev = calculator.device if calculator.device is not None else torch.device("cuda", torch.cuda.current_device())
        self.pos = torch.as_tensor(np.ascontiguousarray(cart, dtype=np.float64)).to(dev).reshape(-1, 3)
        m = torch.as_tensor(np.asarray(masses, dtype=np.float64).reshape(-1)).to(dev)
        if m.numel() != self.pos.size(0):
            raise ValueError("one mass per atom")
        self.mass = m
        self._inv_m = (ACC_UNIT / m).unsqueeze(1)
        self.vel = (torch.zeros_like(self.pos) if velocities is None
                    else torch.as_tensor(np.asarray(velocities, dtype=np.float64)).to(dev).reshape(-1, 3))
        self.dt = float(dt)
        self.energy, self.forces, self.stress = self.calc.compute(self.lattice, self.pos, self.numbers)
        self.n_steps = 0

    def step(self, n: int = 1):
        dt = self.dt
        for _ in range(n):
            self.vel.add_(self.forces.to(torch.float64) * self._inv_m, alpha=0.5 * dt)
            self.pos = self.pos + dt * self.vel  # new tensor: the Verlet list keeps the old one as reference
            self.energy, self.forces, self.stress = self.calc.compute(self.lattice, self.pos, self.numbers)
            self.vel.add_(self.forces.to(torch.float64) * self._inv_m, alpha=0.5 * dt)
            self.n_steps += 1

    def kinetic_energy(self) -> float:
        """eV."""
        return float((0.5 * (self.mass.unsqueeze(1) * self.vel * self.vel).sum() / ACC_UNIT).item())

    def potential_energy(self) -> float:
        return float(self.energy.reshape(-1)[0].item())


class Fire:
    """FIRE structure relaxation (Bitzek et al., PRL 97, 170201) with coordinates, velocities and forces on the
    calculator's device; the usual ASE parameters.  ``run(fmax, steps)`` stops when the largest force row is below fmax
    (eV/A).

    ``relax_cell=False``: fixed cell, max_i |F_i|.  ``relax_cell=True``: positions and cell together on ASE's
    ``UnitCellFilter`` coordinates (restated here; ase is not needed).  With the deformation gradient
    D = solve(L0, L)^T of the current lattice L against the starting one L0, the N + 3 generalised positions are the
    atoms mapped back by D (r D^-T) and ``cell_factor`` * D (default cell_factor = N); the generalised forces are F D for
    the atoms and -V (sigma + p I) D^-T / cell_factor for the cell (sigma = the cell stress of the calculator,
    ``compute(..., with_stress=True)``; p = ``pressure`` in eV/A^3), i.e. minus the gradient of E + pV.  fmax is taken
    over all N + 3 rows.  Every cell change rebuilds the calculator's neighbour candidates."""

    def __init__(self, calculator: M3GNetCalculator, lattice, cart, atomic_numbers, dt: float = 0.1,
                 dt_max: float = 1.0, max_move: float = 0.2, n_min: int = 5, f_inc: float = 1.1, f_dec: float = 0.5,
                 a_start: float = 0.1, f_a: float = 0.99, relax_cell: bool = False, pressure: float = 0.0,
                 cell_factor: Optional[float] = None):
        self.calc = calculator
        self.lattice = np.asarray(lattice, dtype=np.float64).reshape(1, 3, 3)
        self.numbers = np.asarray(atomic_numbers, dtype=np.int64).reshape(-1)
        dev = calculator.device if calculator.device is not None else torch.device("cuda", torch.cuda.current_device())
        self.pos = torch.as_tensor(np.ascontiguousarray(cart, dtype=np.float64)).to(dev).reshape(-1, 3)
        self.dt, self.dt_max, self.max_move = float(dt), float(dt_max), float(max_move)
        self.n_min, self.f_inc, self.f_dec, self.a_start, self.f_a = n_min, f_inc, f_dec, a_start, f_a
        self.a, self.n_pos = a_start, 0
        self.relax_cell = bool(relax_cell)
        self.pressure = float(pressure)
        n = self.pos.size(0)
        self.cell_factor = float(n if cell_factor is None else cell_factor)
        self.lattice0 = self.lattice[0].copy()
        self.cell_stress = None
        if self.relax_cell:
            # generalised positions: atoms without the deformation (D = I at the start) and cell_factor * D
            eye = torch.eye(3, dtype=torch.float64, device=dev)
            self._x = torch.cat([self.pos, self.cell_factor * eye])
        self.vel = torch.zeros((n + 3, 3) if self.relax_cell else (n, 3), dtype=torch.float64, device=dev)
        self._evaluate()
        self.n_steps = 0

    def deform_grad(self) -> np.ndarray:
        return np.linalg.solve(self.lattice0, self.lattice[0]).T

    def _evaluate(self):
        if not self.relax_cell:
            self.energy, self.forces, self.stress = self.calc.compute(self.lattice, self.pos, self.numbers)
            return
        self.energy, self.forces, self.stress, sigma = self.calc.compute(self.lattice, self.pos, self.numbers,
                                                                         with_stress=True)
        self.cell_stress = sigma
        self.gen_forces = self.generalised_forces(self.forces, sigma)

    def generalised_forces(self, forces, sigma) -> torch.Tensor:
        """(N+3, 3): F D for the atoms, -V (sigma + p I) D^-T / cell_factor for the cell (ASE UnitCellFilter)."""
        D = self.deform_grad()
        vol = abs(float(np.linalg.det(self.lattice[0])))
        s = sigma.reshape(3, 3).double().cpu().numpy()
        virial = -vol * (s + self.pressure * np.eye(3))
        cell_f = np.linalg.solve(D, virial.T).T / self.cell_factor
        f = forces.to(torch.float64) @ torch.as_tensor(D, device=forces.device)
        return torch.cat([f, torch.as_tensor(cell_f, dtype=torch.float64, device=f.device)])

    def _set_generalised(self, x: torch.Tensor):
        n = self.pos.size(0)
        self._x = x
        D = (x[n:] / self.cell_factor).cpu().numpy()
        self.lattice = (self.lattice0 @ D.T).reshape(1, 3, 3)
        self.pos = x[:n] @ torch.as_tensor(D.T, dtype=torch.float64, device=x.device)

    def fmax(self) -> float:
        f = self.gen_forces if self.relax_cell else self.forces
        return float(f.norm(dim=1).max().item())

    def step(self):
        f = self.gen_forces if self.relax_cell else self.forces.to(torch.float64)
        power = float((f * self.vel).sum().item())
        if power > 0.0:
            fn = f.norm()
            self.vel = (1.0 - self.a) * self.vel + self.a * self.vel.norm() * f / torch.clamp(fn, min=1e-30)
            if self.n_pos > self.n_min:
                self.dt = min(self.dt * self.f_inc, self.dt_max)
                self.a *= self.f_a
            self.n_pos += 1
        else:
            self.vel.zero_()
            self.a, self.dt, self.n_pos = self.a_start, self.dt * self.f_dec, 0
        self.vel = self.vel + self.dt * f
        dr = self.dt * self.vel
        norm = float(dr.norm().item())
        if norm > self.max_move:
            dr = dr * (self.max_move / norm)
        if self.relax_cell:
            self._set_generalised(self._x + dr)
        else:
            self.pos = self.pos + dr
        self._evaluate()
        self.n_steps += 1

    def run(self, fmax: float = 0.05, steps: int = 200) -> bool:
        for _ in range(steps):
            if self.fmax() < fmax:
                return True
            self.step()
        return self.fmax() < fmax
