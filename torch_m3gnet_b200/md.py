"""Batched Langevin molecular dynamics: many structures sampled at once, each at its own temperature and friction, on
one calculator.

``VelocityVerlet`` (calculator.py) integrates one structure in NVE; sampling S structures with it means S sequential
runs on graphs too small to fill the GPU, and it has no thermostat.  ``BatchMD`` keeps a ragged batch of structures,
evaluates them with one ``calc.compute(..., sizes=...)`` call per step and advances every structure by one BAOAB
Langevin step (Leimkuhler & Matthews 2013) with one kernel launch (``m3g_langevin_step``, csrc/md.cu):

    B: v += dt/2 F(x_k) / m;  A: x += dt/2 v;  O: v = c1 v + c2 sqrt(kB T / m) xi, then the centre-of-mass velocity is
    removed;  A: x += dt/2 v -> x_{k+1};  forces F(x_{k+1});  B: v += dt/2 F(x_{k+1}) / m

with c1 = exp(-friction dt), c2 = sqrt(1 - c1^2) per structure (friction = 0 is NVE velocity Verlet).  The noise xi is
counter-based (Philox4x64-10 keyed by the seed, counter = (atom index in its structure, the structure's index in the
input list, step, 0)) and no generator state is stored, so given the same forces a structure's trajectory is bitwise the
same whatever else shares its batch or chunk.  Removing the centre-of-mass velocity after every O step keeps the
Langevin noise from making the structure drift, so the kinetic temperature counts 3 n - 3 degrees of freedom and a
structure needs at least two atoms.

Constant pressure (``pressure`` set): stochastic cell rescaling (Bernetti & Bussi, J. Chem. Phys. 153, 114107 (2020))
on the same step and launch (``m3g_langevin_npt_step``).  Per structure, with V = |det L|, the pressure
P_int = 2 E_kin / (3 V) - tr(sigma) / 3 of frame k (sigma the cell stress, ASE sign) and, per Cartesian axis,
P_a = 2 K_aa / V - sigma_aa, one Ito Euler-Maruyama step in the log-strain

    d eps = -(beta_T dt / tau_p) (P0 - P) + sqrt(2 kT beta_T dt / (V tau_p)) xi

(one xi per structure in ln V, mu = exp(d eps / 3) on every axis; or one per axis, mu_a = exp(d eps_a)) scales the
positions x_{k+1} and the lattice rows by diag(mu) and the velocities by diag(mu)^-1 after B A O A.  It samples the
isothermal-isobaric ensemble; at stationarity <P_int> = P0 exactly (per axis <P_a> = P0) at any dt.  The per-axis mode
never shears the cell.  ``bath`` keeps its meaning (the thermostat's kinetic energy), so E_pot + E_kin - bath is not
conserved under NPT: the barostat's work is not in it.  The calculator needs the lattices on the host, so every step
copies the device lattices (B,3,3) into pinned memory and synchronises once (``BatchFire(relax_cell=True)`` makes the
same single read-back), and every step rebuilds the calculator's neighbour candidates, since the cell changes.

Failures: a structure whose forces, velocities or energy become non-finite, or whose fastest atom would move more than
``max_step_move`` A in one step, is frozen at that frame (its positions stay finite, so the shared neighbour list stays
sane) and reported as "failed"; nothing else in the batch changes.  Under NPT the same holds for a non-finite stress or
volume, or a log-scale step |ln mu_a| beyond ``max_step_strain``: a collapsing cell would otherwise blow up the
neighbour rebuild the whole batch shares.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import List, Mapping, Optional

import numpy as np
import torch

from torch_m3gnet_b200 import _lib
from torch_m3gnet_b200.calculator import ACC_UNIT
from torch_m3gnet_b200.relax import admit, as_arrays

KB = 8.617333262e-5  # eV/K
GPA = 160.21766208  # GPa per eV/A^3
RUNNING, FAILED = 0, 1
COUPLINGS = {"isotropic": 0, "per_axis": 1}
_SIGNS = {"non-negative": lambda a: a >= 0, "positive": lambda a: a > 0, "any sign": lambda a: np.ones_like(a, bool)}


def _per_structure(value, count: int, name: str, sign: str = "non-negative") -> np.ndarray:
    """A scalar or one value per structure, as a float64 array of ``count`` finite values of ``sign`` ("non-negative",
    "positive" or "any sign")."""
    arr = np.asarray(value, dtype=np.float64)
    arr = np.full(count, float(arr)) if arr.ndim == 0 else arr.reshape(-1)
    if arr.size != count:
        raise ValueError(f"{name}: expected a scalar or {count} values, got {arr.size}")
    if not (np.isfinite(arr).all() and _SIGNS[sign](arr).all()):
        raise ValueError(f"{name} must be finite" + ("" if sign == "any sign" else f" and {sign}"))
    return arr


def _masses(masses, structures) -> List[np.ndarray]:
    if isinstance(masses, Mapping):
        table = {int(z): float(m) for z, m in masses.items()}
        missing = sorted({int(z) for s in structures for z in s[2]} - set(table))
        if missing:
            raise ValueError(f"masses: no mass given for atomic numbers {missing}")
        out = [np.asarray([table[int(z)] for z in s[2]], dtype=np.float64) for s in structures]
    else:
        out = [np.asarray(m, dtype=np.float64).reshape(-1) for m in masses]
        if len(out) != len(structures):
            raise ValueError(f"masses: expected {len(structures)} arrays, got {len(out)}")
        for i, (m, s) in enumerate(zip(out, structures)):
            if m.size != len(s[2]):
                raise ValueError(f"masses[{i}]: expected {len(s[2])} values, got {m.size}")
    for m in out:
        if not (np.isfinite(m).all() and (m > 0).all()):
            raise ValueError("masses must be finite and positive")
    return out


def langevin_step(st, forces, energy, dt: float, max_step_move: float, seed: int, advance: bool, slot: int, obs):
    """One m3g_langevin_step call on the chunk ``st`` (forces (N,3), energy (B) float32)."""
    _lib.call("langevin_step", forces, energy, st.atom_ptr, st.B, dt, max_step_move, seed, int(advance), int(slot),
              st.inv_mass, st.c1, st.c2, st.kT, st.sid, st.pos, st.v, st.step, st.status, st.bath, obs)


def langevin_npt_step(st, forces, sigma, energy, dt: float, max_step_move: float, seed: int, advance: bool, slot: int,
                      obs, coupling: int, max_step_strain: float):
    """One m3g_langevin_npt_step call on the chunk ``st`` (forces (N,3), sigma (B,3,3), energy (B) float32)."""
    _lib.call("langevin_npt_step", forces, energy, st.atom_ptr, st.B, dt, max_step_move, seed, int(advance), int(slot),
              st.inv_mass, st.c1, st.c2, st.kT, st.sid, st.pos, st.v, st.step, st.status, st.bath, obs, sigma,
              st.lattice, st.P0, st.beta_T, st.tau_p, int(coupling), float(max_step_strain))


def maxwell_boltzmann(st, seed: int):
    """One m3g_md_maxwell_boltzmann call: st.v drawn at each structure's temperature."""
    _lib.call("md_maxwell_boltzmann", st.atom_ptr, st.B, seed, st.inv_mass, st.kT, st.sid, st.v)


class BatchMD:
    """Langevin (NVT) or, with ``friction=0``, NVE dynamics of many structures at once, and with ``pressure`` NPT
    (module docstring).

    ``structures``: (lattice (3,3), cart (n,3), atomic_numbers (n,)) tuples or atoms objects with ``get_cell`` /
    ``get_positions`` / ``get_atomic_numbers``; cells are fixed unless ``pressure`` is set.  ``calc``: anything with
    ``M3GNetCalculator.compute``'s protocol, ``compute(lattices, cart, numbers, sizes, with_stress)``.  ``masses``: one (n,) array per structure (amu) or a
    ``{atomic number: amu}`` mapping.  ``temperature`` (K) and ``friction`` (1/fs): scalars or one value per structure.
    ``dt`` in fs.  ``velocities``: None (Maxwell-Boltzmann at each structure's temperature, centre of mass at rest, not
    rescaled) or one (n,3) array per structure in A/fs.  ``seed``: 0 <= seed < 2**64.  ``max_atoms`` splits the
    structures, in input order, into chunks of at most that many atoms (a larger structure runs alone); chunks run one
    after another, and every structure runs all steps.  ``max_step_move`` (A): a structure whose fastest atom would move
    further in one step fails.

    Constant pressure: ``pressure`` None (fixed cells; no stress is requested) or the target P0 in eV/A^3, a scalar or
    one value per structure (any sign).  ``compressibility`` beta_T (A^3/eV; default 1 / (100 GPa)) and
    ``barostat_time`` tau_p (fs): positive scalars or one per structure.  ``coupling``: "isotropic" (the cell keeps its
    shape) or "per_axis" (each Cartesian axis has its own scale and pressure; never shears).  ``max_step_strain``: a
    structure whose log-scale step on an axis would exceed it fails.

    To continue a run, build a new ``BatchMD`` from the returned ``positions`` and ``velocities`` (and, under NPT,
    ``lattice``) with a new ``seed``: the noise of step k is keyed to the seed and k, so reusing the seed would replay the
    noise of the first run."""

    def __init__(self, calc, structures, masses, temperature, friction=0.01, dt: float = 1.0, velocities=None,
                 seed: int = 0, max_atoms: Optional[int] = None, max_step_move: float = 0.5, pressure=None,
                 compressibility=GPA / 100.0, barostat_time=1000.0, coupling: str = "isotropic",
                 max_step_strain: float = 0.01):
        self.calc = calc
        self.structures = [as_arrays(s) for s in structures]
        S = len(self.structures)
        for i, s in enumerate(self.structures):
            if len(s[2]) < 2:
                raise ValueError(f"structure {i} has one atom: no internal degrees of freedom to thermostat")
        self.masses = _masses(masses, self.structures)
        self.temperature = _per_structure(temperature, S, "temperature")
        self.friction = _per_structure(friction, S, "friction")
        self.dt = float(dt)
        if not (np.isfinite(self.dt) and self.dt > 0):
            raise ValueError("dt must be positive")
        self.max_step_move = float(max_step_move)
        if not self.max_step_move > 0:
            raise ValueError("max_step_move must be positive")
        if max_atoms is not None and int(max_atoms) < 1:
            raise ValueError("max_atoms must be positive or None")
        self.max_atoms = None if max_atoms is None else int(max_atoms)
        if not 0 <= int(seed) < 1 << 64:
            raise ValueError("seed must be in [0, 2**64)")
        self.seed = int(seed)
        if velocities is not None:
            velocities = [np.asarray(v, dtype=np.float64).reshape(-1, 3) for v in velocities]
            if len(velocities) != S or any(len(v) != len(s[2]) for v, s in zip(velocities, self.structures)):
                raise ValueError("velocities: one (n,3) array per structure")
            if not all(np.isfinite(v).all() for v in velocities):
                raise ValueError("velocities must be finite")
        self.velocities = velocities
        self.pressure = None if pressure is None else _per_structure(pressure, S, "pressure", "any sign")
        self.compressibility = _per_structure(compressibility, S, "compressibility", "positive")
        self.barostat_time = _per_structure(barostat_time, S, "barostat_time", "positive")
        if coupling not in COUPLINGS:
            raise ValueError(f"coupling must be one of {sorted(COUPLINGS)}, got {coupling!r}")
        self.coupling = coupling
        self.max_step_strain = float(max_step_strain)
        if not self.max_step_strain > 0:
            raise ValueError("max_step_strain must be positive")
        dev = getattr(calc, "device", None)
        self.device = dev if dev is not None else torch.device("cuda", torch.cuda.current_device())
        self.n_iterations = 0

    def run(self, steps: int, record_every: int = 10, trajectory_every: Optional[int] = None) -> List[dict]:
        """Run ``steps`` MD steps.  One record per input structure, in input order: ``status`` ("completed" or
        "failed"), ``n_steps`` (steps completed; a failed structure stopped at frame n_steps), ``times`` (fs) and
        ``energy`` (potential, eV), ``kinetic_energy`` (eV), ``temperature`` (K, over 3 n - 3 degrees of freedom) and
        ``bath`` (eV: the kinetic energy the thermostat added; energy + kinetic_energy - bath is conserved up to the
        integration error) at every ``record_every``-th frame from frame 0 (for a failed structure, the frames before
        it failed); ``positions`` and ``velocities`` of the last frame, ``lattice``; with ``trajectory_every``,
        ``trajectory`` (n_frames, n, 3) of every ``trajectory_every``-th frame from frame 0.  With ``pressure`` the
        recorded frames also give ``volume`` (A^3) and ``pressure`` (P_int, eV/A^3), with "per_axis"
        ``axis_pressure`` (n_frames, 3); ``lattice`` is the last frame's cell, and with ``trajectory_every``
        ``lattice_trajectory`` (n_frames, 3, 3) holds the cells of the trajectory's frames."""
        steps, record_every = int(steps), int(record_every)
        if steps < 0 or record_every < 1 or (trajectory_every is not None and int(trajectory_every) < 1):
            raise ValueError("steps must be >= 0, record_every and trajectory_every >= 1")
        sizes = [len(s[2]) for s in self.structures]
        results: List[Optional[dict]] = [None] * len(sizes)
        start = 0
        while start < len(sizes):
            end = admit(sizes, start, self.max_atoms, 0, 0)
            self._run_chunk(list(range(start, end)), steps, record_every,
                            None if trajectory_every is None else int(trajectory_every), results)
            start = end
        return results

    def _run_chunk(self, ids, steps, record_every, trajectory_every, results):
        dev = self.device
        pin = dev.type == "cuda"
        f64 = dict(dtype=torch.float64, device=dev)
        i32 = dict(dtype=torch.int32, device=dev)
        sizes = [len(self.structures[i][2]) for i in ids]
        B, N = len(ids), int(sum(sizes))
        npt = self.pressure is not None
        lat_h = np.stack([self.structures[i][0] for i in ids]).astype(np.float64)
        z = np.concatenate([self.structures[i][2] for i in ids])
        gamma = self.friction[ids]
        c1 = np.exp(-gamma * self.dt)
        st = SimpleNamespace(
            B=B, atom_ptr=torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)).to(dev),
            pos=torch.as_tensor(np.concatenate([self.structures[i][1] for i in ids])).to(dev),
            inv_mass=torch.as_tensor(ACC_UNIT / np.concatenate([self.masses[i] for i in ids])).to(dev),
            c1=torch.as_tensor(c1).to(dev), c2=torch.as_tensor(np.sqrt(1.0 - c1 * c1)).to(dev),
            kT=torch.as_tensor(KB * self.temperature[ids]).to(dev),
            sid=torch.as_tensor(np.asarray(ids, dtype=np.int64)).to(dev),
            step=torch.zeros(B, **i32), status=torch.zeros(B, **i32), bath=torch.zeros(B, **f64))
        if npt:
            st.lattice = torch.as_tensor(lat_h).to(dev)
            st.P0 = torch.as_tensor(self.pressure[ids]).to(dev)
            st.beta_T = torch.as_tensor(self.compressibility[ids]).to(dev)
            st.tau_p = torch.as_tensor(self.barostat_time[ids]).to(dev)
            lat_pin = torch.empty((B, 3, 3), dtype=torch.float64, pin_memory=pin)
        seed = self.seed - (1 << 64) if self.seed >= 1 << 63 else self.seed  # the ABI's int64, read back as uint64
        if self.velocities is None:
            st.v = torch.empty((N, 3), **f64)
            maxwell_boltzmann(st, seed)
        else:
            st.v = torch.as_tensor(np.concatenate([self.velocities[i] for i in ids])).to(dev)
        n_slots = steps // record_every + 1
        width = 4 if not npt else 6 if self.coupling == "isotropic" else 9
        obs = torch.full((n_slots, B, width), float("nan"), **f64)
        traj = lat_traj = None
        if trajectory_every is not None:
            traj = torch.empty((steps // trajectory_every + 1, N, 3), dtype=torch.float64, pin_memory=pin)
            if npt:
                lat_traj = np.empty((steps // trajectory_every + 1, B, 3, 3))
        for k in range(steps + 1):
            if traj is not None and k % trajectory_every == 0:
                traj[k // trajectory_every].copy_(st.pos, non_blocking=pin)
                if lat_traj is not None:
                    lat_traj[k // trajectory_every] = lat_h
            slot = k // record_every if k % record_every == 0 else -1
            out = self.calc.compute(lat_h, st.pos, z, sizes, with_stress=True) if npt else \
                self.calc.compute(lat_h, st.pos, z, sizes)
            energy = out[0].reshape(-1).to(torch.float32).contiguous()
            forces = out[1].reshape(-1, 3).to(torch.float32).contiguous()
            if npt:
                sigma = out[3].reshape(-1, 3, 3).to(torch.float32).contiguous()
                langevin_npt_step(st, forces, sigma, energy, self.dt, self.max_step_move, seed, k < steps, slot, obs,
                                  COUPLINGS[self.coupling], self.max_step_strain)
            else:
                langevin_step(st, forces, energy, self.dt, self.max_step_move, seed, k < steps, slot, obs)
            self.n_iterations += 1
            if npt and k < steps:
                # the step's one read-back: the new cells, which the next compute needs on the host
                lat_pin.copy_(st.lattice, non_blocking=pin)
                if pin:
                    torch.cuda.current_stream(dev).synchronize()
                lat_h = lat_pin.numpy().copy()
        # the chunk's one read-back
        if pin:
            torch.cuda.current_stream(dev).synchronize()
        obs_h, pos, v = obs.cpu().numpy(), st.pos.cpu().numpy(), st.v.cpu().numpy()
        status, n_steps = st.status.cpu().numpy(), st.step.cpu().numpy()
        traj_h = traj.numpy() if traj is not None else None
        ptr = np.concatenate([[0], np.cumsum(sizes)])
        times = self.dt * record_every * np.arange(n_slots)
        for j, i in enumerate(ids):
            failed = int(status[j]) == FAILED
            ns = int(n_steps[j])
            m = -(-ns // record_every) if failed else n_slots  # frames recorded before frame ns failed
            rows = slice(ptr[j], ptr[j + 1])
            rec = dict(status="failed" if failed else "completed", n_steps=ns, times=times[:m].copy(),
                       energy=obs_h[:m, j, 0].copy(), kinetic_energy=obs_h[:m, j, 1].copy(),
                       temperature=obs_h[:m, j, 2].copy(), bath=obs_h[:m, j, 3].copy(),
                       positions=pos[rows].copy(), velocities=v[rows].copy(), lattice=lat_h[j].copy())
            if npt:
                rec["volume"], rec["pressure"] = obs_h[:m, j, 4].copy(), obs_h[:m, j, 5].copy()
                if width == 9:
                    rec["axis_pressure"] = obs_h[:m, j, 6:9].copy()
            if traj_h is not None:
                last = ns // trajectory_every + 1 if failed else traj_h.shape[0]
                rec["trajectory"] = traj_h[:last, rows].copy()
                if lat_traj is not None:
                    rec["lattice_trajectory"] = lat_traj[:last, j].copy()
            results[i] = rec
