"""Batched FIRE relaxation: many structures relaxed at once, each with its own FIRE state, on one calculator.

``Fire`` (calculator.py) relaxes one structure; relaxing S structures with it means S sequential runs, each on a graph
too small to fill the GPU.  ``BatchFire`` keeps a working set of structures in one ragged batch, evaluates them with
one ``calc.compute(..., sizes=...)`` call per step and advances every running structure by one FIRE step with one
kernel launch (``m3g_fire_step``, csrc/relax.cu).  Per structure the step is exactly ``Fire.step`` / ``Fire.run``:
its own ``a``, ``dt`` and ``n_pos``; power, norms, ``max_move`` and fmax over its own rows (N_b, or N_b + 3 with
``relax_cell``).  The kernel reduces each structure's rows in a fixed order that depends only on those rows, so given
the same forces a structure's trajectory is bit-identical whatever else is in the batch.

Working set and regroups: structures enter in input order while their atoms fit ``max_atoms`` (a structure larger
than the budget enters alone; ``None`` = everything in one batch).  A structure that stops (converged, out of steps, or
failed on non-finite forces / stress) keeps the values of the frame at which it stopped and stays frozen in the batch.
The working set is regrouped -- finished structures recorded and removed, queued ones admitted with fresh FIRE state --
when the finished structures hold at least a quarter of its atoms, or when nothing in it is running.  A regroup changes
the calculator's ``sizes`` key and so rebuilds its neighbour candidates; with ``relax_cell`` the candidates are rebuilt
every step anyway (every step changes the cells), so the working set is regrouped as soon as anything finished.  The
policy changes only which structures share a batch, never a structure's own result.
"""
from __future__ import annotations

import time
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from torch_m3gnet_b200 import _lib

RUNNING, CONVERGED, NOT_CONVERGED, FAILED = 0, 1, 2, 3
STATUS_NAMES = {CONVERGED: "converged", NOT_CONVERGED: "not converged", FAILED: "failed"}


def as_arrays(structure):
    """(lattice (3,3) f64, cart (n,3) f64, atomic numbers (n,) int64) of a tuple or a duck-typed atoms object."""
    if hasattr(structure, "get_positions"):
        lat, cart, z = structure.get_cell(), structure.get_positions(), structure.get_atomic_numbers()
    else:
        lat, cart, z = structure
    lat = np.array(lat, dtype=np.float64).reshape(3, 3)
    cart = np.array(cart, dtype=np.float64).reshape(-1, 3)
    z = np.array(z, dtype=np.int64).reshape(-1)
    if z.size != cart.shape[0] or z.size == 0:
        raise ValueError("a structure needs one atomic number per atom and at least one atom")
    return lat, cart, z


def admit(sizes: Sequence[int], start: int, budget: Optional[int], held: int, n_held: int) -> int:
    """Index one past the last queued structure (``sizes[start:]``, input order) that enters a working set already
    holding ``n_held`` structures with ``held`` atoms: structures enter while their atoms fit ``budget`` (None = no
    limit); the first that does not fit stops admission, except that an empty working set always takes one."""
    end = start
    while end < len(sizes):
        if budget is not None and held + sizes[end] > budget and (n_held > 0 or end > start):
            break
        held += sizes[end]
        end += 1
    return end


def should_regroup(finished_atoms: int, atoms: int, any_finished: bool, all_finished: bool, relax_cell: bool) -> bool:
    """Regroup policy (module docstring)."""
    if all_finished:
        return True
    if relax_cell:
        return any_finished
    return 4 * finished_atoms >= atoms


class _State:
    """Working-set state on the device: the arrays m3g_fire_step reads and writes, plus host bookkeeping."""

    def __init__(self, device, relax_cell: bool):
        self.device, self.relax_cell = device, relax_cell
        f64 = dict(dtype=torch.float64, device=device)
        i32 = dict(dtype=torch.int32, device=device)
        self.ids: List[int] = []
        self.sizes: List[int] = []
        self.z = np.zeros(0, dtype=np.int64)
        self.lat_h = np.zeros((0, 3, 3))
        self.pos = torch.zeros((0, 3), **f64)
        self.v = torch.zeros((0, 3), **f64)
        self.x = torch.zeros((0, 3), **f64) if relax_cell else None
        self.atom_tensors = ["pos", "v"] + (["x"] if relax_cell else [])
        for k in ("dt", "a", "fmax", "e_frame", "cell_factor"):
            setattr(self, k, torch.zeros(0, **f64))
        for k in ("n_pos", "n_steps", "status"):
            setattr(self, k, torch.zeros(0, **i32))
        for k in ("L0", "lattice", "xc", "vc", "sigma_frame"):
            setattr(self, k, torch.zeros((0, 3, 3), **f64))
        self.struct_tensors = ["dt", "a", "fmax", "e_frame", "cell_factor", "n_pos", "n_steps", "status", "L0",
                               "lattice", "xc", "vc", "sigma_frame"]
        self.atom_ptr = torch.zeros(1, **i32)

    @property
    def B(self) -> int:
        return len(self.ids)

    @property
    def N(self) -> int:
        return int(sum(self.sizes))

    def keep(self, keep: List[int]):
        """Only the structures at working-set positions ``keep`` (ascending) stay; their state rows are carried over."""
        ptr = np.concatenate([[0], np.cumsum(self.sizes)]).astype(np.int64)
        rows = np.concatenate([np.arange(ptr[b], ptr[b + 1]) for b in keep]) if keep else np.zeros(0, np.int64)
        rows_d = torch.as_tensor(rows).to(self.device)
        keep_d = torch.as_tensor(np.asarray(keep, dtype=np.int64)).to(self.device)
        for k in self.atom_tensors:
            setattr(self, k, getattr(self, k).index_select(0, rows_d))
        for k in self.struct_tensors:
            setattr(self, k, getattr(self, k).index_select(0, keep_d))
        self.ids = [self.ids[b] for b in keep]
        self.sizes = [self.sizes[b] for b in keep]
        self.z = self.z[rows]
        self.lat_h = self.lat_h[keep]
        self.reindex()

    def append(self, ids, structures, fire, cell_factor):
        """Fresh FIRE state for the structures ``ids`` (L0 = their starting lattice, zero velocity, D = I)."""
        dev = self.device
        lats = np.stack([structures[i][0] for i in ids])
        carts = np.concatenate([structures[i][1] for i in ids])
        sizes = [len(structures[i][2]) for i in ids]
        cf = np.asarray([float(n if cell_factor is None else cell_factor) for n in sizes])
        f64 = dict(dtype=torch.float64, device=dev)
        pos = torch.as_tensor(carts).to(dev)
        m = len(ids)
        new = dict(pos=pos, v=torch.zeros_like(pos), x=pos.clone(),
                   dt=torch.full((m,), fire["dt"], **f64), a=torch.full((m,), fire["a_start"], **f64),
                   fmax=torch.zeros(m, **f64), e_frame=torch.zeros(m, **f64), cell_factor=torch.as_tensor(cf).to(dev),
                   n_pos=torch.zeros(m, dtype=torch.int32, device=dev),
                   n_steps=torch.zeros(m, dtype=torch.int32, device=dev),
                   status=torch.zeros(m, dtype=torch.int32, device=dev),
                   L0=torch.as_tensor(lats).to(dev), lattice=torch.as_tensor(lats).to(dev),
                   xc=torch.as_tensor(cf[:, None, None] * np.eye(3)[None]).to(dev), vc=torch.zeros((m, 3, 3), **f64),
                   sigma_frame=torch.zeros((m, 3, 3), **f64))
        for k in self.atom_tensors + self.struct_tensors:
            setattr(self, k, torch.cat([getattr(self, k), new[k]]))
        self.ids += list(ids)
        self.sizes += sizes
        self.z = np.concatenate([self.z] + [structures[i][2] for i in ids])
        self.lat_h = np.concatenate([self.lat_h, lats])
        self.reindex()

    def reindex(self):
        self.atom_ptr = torch.as_tensor(np.concatenate([[0], np.cumsum(self.sizes)]).astype(np.int32)).to(self.device)


def fire_step(st: _State, forces, sigma, energy, fire: Dict[str, float], fmax: float, steps: int, pressure: float):
    """One m3g_fire_step call on the working set ``st`` (forces (N,3), sigma (B,3,3) or None, energy (B) float32)."""
    cell = sigma is not None
    _lib.call("fire_step", forces, sigma, energy, st.atom_ptr, st.B, fire["dt_max"], fire["max_move"],
              int(fire["n_min"]), fire["f_inc"], fire["f_dec"], fire["a_start"], fire["f_a"], float(fmax), int(steps),
              float(pressure), st.cell_factor, st.x if cell else None, st.xc if cell else None, st.v,
              st.vc if cell else None, st.dt, st.a, st.n_pos, st.n_steps, st.status, st.L0 if cell else None,
              st.lattice if cell else None, st.pos, st.fmax, st.e_frame, st.sigma_frame if cell else None)


class BatchFire:
    """FIRE relaxation of many structures at once (module docstring).

    ``structures``: (lattice (3,3), cart (n,3), atomic_numbers (n,)) tuples or atoms objects with ``get_cell`` /
    ``get_positions`` / ``get_atomic_numbers``.  ``calc``: anything with ``M3GNetCalculator.compute``'s protocol,
    ``compute(lattices, cart, numbers, sizes, with_stress)``.  Every FIRE parameter has ``Fire``'s meaning, applied per
    structure; ``cell_factor`` defaults to each structure's atom count; ``pressure`` in eV/A^3.  ``max_atoms`` bounds
    the atoms of the working set (None = all structures in one batch)."""

    def __init__(self, calc, structures, relax_cell: bool = False, pressure: float = 0.0,
                 max_atoms: Optional[int] = None, dt: float = 0.1, dt_max: float = 1.0, max_move: float = 0.2,
                 n_min: int = 5, f_inc: float = 1.1, f_dec: float = 0.5, a_start: float = 0.1, f_a: float = 0.99,
                 cell_factor: Optional[float] = None):
        self.calc = calc
        self.structures = [as_arrays(s) for s in structures]
        self.relax_cell = bool(relax_cell)
        self.pressure = float(pressure)
        if max_atoms is not None and int(max_atoms) < 1:
            raise ValueError("max_atoms must be positive or None")
        self.max_atoms = None if max_atoms is None else int(max_atoms)
        self.cell_factor = None if cell_factor is None else float(cell_factor)
        self.fire = dict(dt=float(dt), dt_max=float(dt_max), max_move=float(max_move), n_min=int(n_min),
                         f_inc=float(f_inc), f_dec=float(f_dec), a_start=float(a_start), f_a=float(f_a))
        dev = getattr(calc, "device", None)
        self.device = dev if dev is not None else torch.device("cuda", torch.cuda.current_device())
        self.n_iterations = self.n_regroups = 0
        self.regroup_seconds = 0.0

    def run(self, fmax: float = 0.05, steps: int = 200) -> List[dict]:
        """Relax every structure; one record per input structure, in input order: ``status`` ("converged", "not
        converged" within ``steps`` steps, or "failed" on non-finite forces / stress), ``n_steps``, ``energy`` (eV),
        ``fmax`` (eV/A, over N_b or N_b + 3 rows), ``positions`` (n,3) float64 A, ``lattice`` (3,3) and, with
        ``relax_cell``, ``cell_stress`` (3,3) eV/A^3 -- all of the frame at which the structure stopped."""
        sizes = [len(s[2]) for s in self.structures]
        results: List[Optional[dict]] = [None] * len(sizes)
        if not sizes:
            return []
        st = _State(self.device, self.relax_cell)
        pin = self.device.type == "cuda"
        nxt = admit(sizes, 0, self.max_atoms, 0, 0)
        st.append(range(0, nxt), self.structures, self.fire, self.cell_factor)
        while st.B:
            out = self.calc.compute(st.lat_h, st.pos, st.z, st.sizes, with_stress=self.relax_cell)
            energy = out[0].reshape(-1).to(torch.float32).contiguous()
            forces = out[1].reshape(-1, 3).to(torch.float32).contiguous()
            sigma = out[3].reshape(-1, 3, 3).to(torch.float32).contiguous() if self.relax_cell else None
            fire_step(st, forces, sigma, energy, self.fire, fmax, steps, self.pressure)
            self.n_iterations += 1
            # the step's one read-back: statuses (and the new cells, which the next compute needs on the host)
            status_h = torch.empty(st.B, dtype=torch.int32, pin_memory=pin)
            status_h.copy_(st.status, non_blocking=pin)
            if self.relax_cell:
                lat_h = torch.empty((st.B, 3, 3), dtype=torch.float64, pin_memory=pin)
                lat_h.copy_(st.lattice, non_blocking=pin)
            if pin:
                torch.cuda.current_stream(self.device).synchronize()
            status = status_h.numpy()
            if self.relax_cell:
                st.lat_h = lat_h.numpy().copy()
            done = status != RUNNING
            fin_atoms = int(np.asarray(st.sizes)[done].sum())
            if not should_regroup(fin_atoms, st.N, bool(done.any()), bool(done.all()), self.relax_cell):
                continue
            t0 = time.perf_counter()
            self._record(st, np.flatnonzero(done), status, results)
            st.keep([int(b) for b in np.flatnonzero(~done)])
            end = admit(sizes, nxt, self.max_atoms, st.N, st.B)
            if end > nxt:
                st.append(range(nxt, end), self.structures, self.fire, self.cell_factor)
                nxt = end
            self.n_regroups += 1
            self.regroup_seconds += time.perf_counter() - t0
        return results

    def _record(self, st: _State, finished, status, results):
        if len(finished) == 0:
            return
        idx = torch.as_tensor(finished).to(self.device)
        host = {k: getattr(st, k).index_select(0, idx).cpu().numpy()
                for k in ("n_steps", "e_frame", "fmax", "lattice", "sigma_frame")}
        pos = st.pos.cpu().numpy()
        ptr = np.concatenate([[0], np.cumsum(st.sizes)])
        for j, b in enumerate(finished):
            rec = dict(status=STATUS_NAMES[int(status[b])], n_steps=int(host["n_steps"][j]),
                       energy=float(host["e_frame"][j]), fmax=float(host["fmax"][j]),
                       positions=pos[ptr[b]:ptr[b + 1]].copy(),
                       lattice=host["lattice"][j].copy() if self.relax_cell else st.lat_h[b].copy())
            if self.relax_cell:
                rec["cell_stress"] = host["sigma_frame"][j].copy()
            results[st.ids[b]] = rec
