"""Batched harmonic phonons: finite-displacement force constants, phonon frequencies and harmonic thermal properties of
many structures at once, on one calculator.

Per structure (a unit cell of n atoms and a diagonal supercell of L = n1 n2 n3 cells, N = n L atoms) the supercell's
atom j = l n + k is atom k of the unit cell translated by cell l = (i1, i2, i3) (lexicographic), positions taken as
given.  Atom k of cell 0 is moved by +h and by -h along x, y and z; with the undisplaced supercell that is 6 n + 1
supercells per structure, evaluated structure-major (undisplaced, then (k, alpha, +h), (k, alpha, -h) for k = 0 .. n-1
and alpha = x, y, z) by ragged ``calc.compute(..., sizes=...)`` calls in chunks of at most ``max_atoms`` atoms
(``relax.admit``: a structure's set may span chunks; a supercell larger than the budget runs alone).  The forces land
in one device buffer, and one launch of ``m3g_phonon_force_constants`` (csrc/phonon.cu) turns every structure's rows
into force constants Phi(0k alpha; j beta) (phonopy's compact layout, eV/A^2): central differences, then ``symmetrize``
rounds of the index-permuted transpose average and the acoustic sum rule, in the order of ASE's
``Phonons.read(symmetrize=k, acoustic=True)``.

Frequencies at q-points (fractional coordinates of the unit cell's reciprocal lattice) come from one launch of
``m3g_phonon_frequencies``: per (structure, q) it builds the dynamical matrix D(q) from the force constants and the
minimum-image table below, takes its Hermitian part and finds its eigenvalues by a cyclic complex Jacobi method.
``thermal_properties`` adds one launch of ``m3g_phonon_thermal`` on a Gamma-centred mesh.  Everything on the device is
float64 and reduced in a fixed order that depends only on the structure's own data, so a structure's results are bitwise
the same whatever else is in the batch.

Minimum images: for each pair (k, j) the supercell translations T that make |r_j + T - r_k| minimal (5^3 supercell
images around the wrapped difference; lengths within a relative 1e-5 count as equal) are averaged in D(q).  They are
stored as the lattice translation from cell 0 to the image's cell, in unit-cell fractional coordinates (integers), in a
CSR table built once per structure on the host (numpy, vectorised).  DESIGN.md §8 gives the equations.
"""
from __future__ import annotations

import math
import time
from types import SimpleNamespace
from typing import List, Optional

import numpy as np
import torch

from torch_m3gnet_b200 import _lib
from torch_m3gnet_b200.md import _masses
from torch_m3gnet_b200.relax import admit, as_arrays

MAX_ATOMS = 32  # atoms per unit cell: M3G_PHONON_MAX_ATOMS (include/m3gnet_b200.h), so 3n <= 96
OK, FAILED = 0, 1
STATUS_NAMES = {OK: "ok", FAILED: "failed"}

# CODATA 2018 (SI exact values for e, h and k_B)
_EV = 1.602176634e-19         # J
_AMU = 1.66053906660e-27      # kg
_ANGSTROM = 1e-10             # m
_PLANCK = 6.62607015e-34      # J s
_BOLTZMANN = 1.380649e-23     # J/K
THZ = math.sqrt(_EV / (_AMU * _ANGSTROM ** 2)) / (2.0 * math.pi) / 1e12  # THz per sqrt(eV / (amu A^2)), ~15.6333
H_THZ = _PLANCK * 1e12 / _EV  # eV per THz (h f)
KB = _BOLTZMANN / _EV         # eV/K
IMAGE_RTOL = 1e-5             # minimum images: lengths within this relative tolerance are equidistant


def mesh_qpoints(mesh) -> np.ndarray:
    """(m1 m2 m3, 3) Gamma-centred mesh in fractional reciprocal coordinates, i1 slowest, each coordinate i/m mapped to
    (-1/2, 1/2].  No symmetry reduction; every point has the same weight."""
    m = np.asarray(mesh, dtype=np.int64).reshape(-1)
    if m.size != 3 or (m < 1).any():
        raise ValueError(f"mesh must be three positive integers, got {mesh!r}")
    axes = []
    for k in m:
        i = np.arange(k)
        axes.append(np.where(2 * i > k, i - k, i) / k)
    return np.stack(np.meshgrid(*axes, indexing="ij"), axis=-1).reshape(-1, 3)


def _cells(reps) -> np.ndarray:
    """(L, 3) cell indices l = (i1, i2, i3) in lexicographic order."""
    return np.stack(np.meshgrid(*[np.arange(r) for r in reps], indexing="ij"), axis=-1).reshape(-1, 3)


def supercell(lattice, cart, reps):
    """(supercell lattice (3,3), positions (N,3)) with atom j = l n + k at cart[k] + l . lattice, no wrapping."""
    reps = np.asarray(reps, dtype=np.int64)
    shift = _cells(reps) @ lattice
    return lattice * reps[:, None], (shift[:, None, :] + cart[None]).reshape(-1, 3)


def minimum_images(lattice, cart, reps):
    """(sv_ptr (n N + 1,) int64, sv (K, 3) float64): for each pair (k, j) (row k N + j) the minimum-image set of
    r_j - r_k in the supercell, each image as the unit-cell fractional coordinates of the lattice translation from cell
    0 to the image's cell (l + t * reps for the supercell translation t).  5^3 supercell images around the wrapped
    difference are searched; images within a relative ``IMAGE_RTOL`` of the shortest are all kept, in lexicographic
    order of t."""
    reps = np.asarray(reps, dtype=np.int64)
    S, pos = supercell(lattice, cart, reps)
    n, N = len(cart), len(pos)
    cells = np.repeat(_cells(reps), n, axis=0)              # (N, 3): cell of supercell atom j
    t = np.stack(np.meshgrid(*[np.arange(-2, 3)] * 3, indexing="ij"), axis=-1).reshape(-1, 3)
    tS = t @ S
    counts, vecs = [], []
    step = max(1, (1 << 21) // (N * len(t)))               # unit-cell atoms per pass: bounded temporaries
    for k0 in range(0, n, step):
        d0 = pos[None] - cart[k0:k0 + step, None]           # (k, N, 3)
        wrap = -np.floor(d0 @ np.linalg.inv(S) + 0.5)
        d = (d0 + wrap @ S)[:, :, None, :] + tS             # (k, N, 125, 3)
        r2 = np.einsum("knix,knix->kni", d, d)
        keep = r2 <= r2.min(axis=2, keepdims=True) * (1.0 + IMAGE_RTOL) ** 2
        counts.append(keep.sum(axis=2).reshape(-1))
        vecs.append((cells[None, :, None, :] + (wrap[:, :, None, :] + t) * reps)[keep])
    sv_ptr = np.concatenate([[0], np.cumsum(np.concatenate(counts))]).astype(np.int64)
    return sv_ptr, np.concatenate(vecs).astype(np.float64)


def _cum(counts, dtype):
    return np.concatenate([[0], np.cumsum(np.asarray(counts, dtype=np.int64))]).astype(dtype)


# the launches; the CPU tests substitute tests/phonon_oracle.py's restatements for these

def fc_launch(forces, st, h: float, symmetrize: int):
    """One m3g_phonon_force_constants call: st.fc, st.status and st.residual from forces (rows, 3), read as float32."""
    _lib.call("phonon_force_constants", forces.to(torch.float32).contiguous(), st.row_ptr, st.atom_ptr, st.reps,
              st.pair_ptr, st.B, st.max_n, h, symmetrize, st.fc, st.status, st.residual)


def frequencies_launch(st, q, q_ptr, f_ptr, out):
    """One m3g_phonon_frequencies call on q (Q, 3) float64: out.eig, out.freq, out.sweeps, out.q_status."""
    _lib.call("phonon_frequencies", st.fc, st.atom_ptr, st.reps, st.pair_ptr, st.sv_ptr, st.sv, st.mass, st.status,
              q, q_ptr, f_ptr, st.B, q.shape[0], st.max_n, THZ, out.eig, out.freq, out.sweeps, out.q_status)


def thermal_launch(st, freq, f_ptr, q_ptr, temps, cutoff: float, out):
    """One m3g_phonon_thermal call: out.values (B, T, 4), out.n_imag (B), out.fmin (B)."""
    _lib.call("phonon_thermal", freq, f_ptr, q_ptr, st.status, st.B, temps, temps.shape[0], KB, H_THZ, float(cutoff),
              out.values, out.n_imag, out.fmin)


def dynmat_launch(st, q, q_ptr, ld: int):
    """D(q) of every q-point (Q, ld, ld) complex128 (m3g_phonon_dynmat; zero outside each structure's 3n x 3n)."""
    out = torch.empty((q.shape[0], ld, ld, 2), dtype=torch.float64, device=q.device)
    _lib.call("phonon_dynmat", st.fc, st.atom_ptr, st.reps, st.pair_ptr, st.sv_ptr, st.sv, st.mass, q, q_ptr, st.B,
              q.shape[0], st.max_n, ld, out)
    return torch.view_as_complex(out)


class BatchPhonon:
    """Harmonic phonons of many structures at once (module docstring).

    ``structures``: unit cells as (lattice (3,3), cart (n,3), atomic_numbers (n,)) tuples or atoms objects, as
    ``BatchFire`` takes, at most ``MAX_ATOMS`` atoms each.  ``supercell``: one diagonal repetition (n1, n2, n3) or one
    per structure.  ``masses`` (amu): ``BatchMD``'s forms ({atomic number: mass} or one array per structure).
    ``displacement``: the step h in A.  ``symmetrize``: rounds of transpose averaging and acoustic sum rule (0 = the raw
    differences).  ``max_atoms`` bounds the atoms of each compute call (None = no bound)."""

    def __init__(self, calc, structures, supercell, masses, displacement: float = 0.01, symmetrize: int = 3,
                 max_atoms: Optional[int] = None):
        self.calc = calc
        self.structures = [as_arrays(s) for s in structures]
        B = len(self.structures)
        for i, s in enumerate(self.structures):
            if len(s[2]) > MAX_ATOMS:
                raise ValueError(f"structure {i} has {len(s[2])} atoms; unit cells of at most {MAX_ATOMS} atoms "
                                 "are supported")
        reps = np.asarray(supercell)
        if reps.size and not np.array_equal(reps, np.round(reps)):
            raise ValueError("supercell repetitions must be integers")
        reps = reps.astype(np.int64)
        if reps.shape == (3,):
            reps = np.tile(reps, (B, 1))
        if reps.shape != (B, 3):
            raise ValueError(f"supercell: expected (n1, n2, n3) or one per structure ({B}, 3), got shape {reps.shape}")
        if (reps < 1).any():
            raise ValueError("supercell repetitions must be at least 1")
        self.reps = reps
        h = float(displacement)
        if not (math.isfinite(h) and h > 0.0):
            raise ValueError("displacement must be finite and positive")
        self.h = h
        if int(symmetrize) != symmetrize or symmetrize < 0:
            raise ValueError("symmetrize must be a non-negative integer")
        self.symmetrize = int(symmetrize)
        if max_atoms is not None and int(max_atoms) < 1:
            raise ValueError("max_atoms must be positive or None")
        self.max_atoms = None if max_atoms is None else int(max_atoms)
        self.masses = _masses(masses, self.structures)
        dev = getattr(calc, "device", None)
        self.device = dev if dev is not None else torch.device("cuda", torch.cuda.current_device())
        self.n_compute_calls = 0
        self.minimum_image_seconds = 0.0
        self.last_sweeps: Optional[List[np.ndarray]] = None
        self._st = None

    @property
    def B(self) -> int:
        return len(self.structures)

    def _supercell(self, b: int, s: int):
        """(lattice, positions, numbers) of supercell s (0 = undisplaced, 1 + 2 (3 k + alpha) + {0: +h, 1: -h}) of
        structure b."""
        lat, cart, z = self.structures[b]
        S, pos = supercell(lat, cart, self.reps[b])
        if s > 0:
            k, rest = divmod(s - 1, 6)
            pos = pos.copy()
            pos[k, rest // 2] += self.h if rest % 2 == 0 else -self.h
        return S, pos, np.tile(z, int(np.prod(self.reps[b])))

    def run(self) -> List[dict]:
        """Force constants of every structure; one record per structure, in input order: ``status`` ("ok", or "failed"
        if any of its forces is not finite), ``force_constants`` (n, N, 3, 3) float64 eV/A^2 (NaN when failed),
        ``max_residual_force`` (largest |F| of the undisplaced supercell, eV/A; reported, not subtracted; NaN when
        failed), ``supercell_lattice`` (3, 3) and ``supercell`` (n1, n2, n3)."""
        if not self.B:
            return []
        dev = self.device
        n = [len(s[2]) for s in self.structures]
        L = [int(np.prod(r)) for r in self.reps]
        N = [a * c for a, c in zip(n, L)]
        t0 = time.perf_counter()
        tables = [minimum_images(s[0], s[1], r) for s, r in zip(self.structures, self.reps)]
        self.minimum_image_seconds = time.perf_counter() - t0
        # the evaluation list, structure-major
        jobs = [(b, s) for b in range(self.B) for s in range(6 * n[b] + 1)]
        sizes = [N[b] for b, _ in jobs]
        forces = None
        start = row = 0
        while start < len(jobs):
            end = admit(sizes, start, self.max_atoms, 0, 0)
            cells = [self._supercell(b, s) for b, s in jobs[start:end]]
            out = self.calc.compute(np.stack([c[0] for c in cells]), np.concatenate([c[1] for c in cells]),
                                    np.concatenate([c[2] for c in cells]), sizes[start:end])
            f = out[1].reshape(-1, 3)
            if forces is None:  # the calculator's precision (float32 for the model; the kernel reads float32)
                forces = torch.empty((sum(sizes), 3), dtype=f.dtype, device=dev)
            forces[row:row + f.shape[0]].copy_(f)
            row += f.shape[0]
            self.n_compute_calls += 1
            start = end
        pairs = [a * c for a, c in zip(n, N)]
        pair_ptr = _cum(pairs, np.int64)
        offs = _cum([len(t[1]) for t in tables], np.int64)
        sv_ptr = np.concatenate([t[0][:-1] + o for t, o in zip(tables, offs)] + [offs[-1:]])
        as_dev = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(dev)  # noqa: E731
        st = SimpleNamespace(
            B=self.B, max_n=max(n), n=n, N=N,
            row_ptr=as_dev(_cum([(6 * a + 1) * c for a, c in zip(n, N)], np.int64)),
            atom_ptr=as_dev(_cum(n, np.int32)), reps=as_dev(self.reps.astype(np.int32)), pair_ptr=as_dev(pair_ptr),
            sv_ptr=as_dev(sv_ptr), sv=as_dev(np.concatenate([t[1] for t in tables])),
            mass=as_dev(np.concatenate(self.masses)),
            fc=torch.empty((int(pair_ptr[-1]), 3, 3), dtype=torch.float64, device=dev),
            status=torch.empty(self.B, dtype=torch.int32, device=dev),
            residual=torch.empty(self.B, dtype=torch.float64, device=dev))
        fc_launch(forces, st, self.h, self.symmetrize)
        self._st = st
        fc = st.fc.cpu().numpy()
        status = st.status.cpu().numpy()
        residual = st.residual.cpu().numpy()
        return [dict(status=STATUS_NAMES[int(status[b])],
                     force_constants=fc[pair_ptr[b]:pair_ptr[b + 1]].reshape(n[b], N[b], 3, 3),
                     max_residual_force=float(residual[b]),
                     supercell_lattice=self.structures[b][0] * self.reps[b][:, None],
                     supercell=tuple(int(r) for r in self.reps[b])) for b in range(self.B)]

    def _qpoints(self, qpoints) -> List[np.ndarray]:
        try:
            arr = np.asarray(qpoints, dtype=np.float64)
        except ValueError:  # ragged: one array per structure
            arr = None
        if arr is not None and arr.ndim <= 2:
            arr = arr.reshape(-1, 3)
            qs = [arr] * self.B
        else:
            qs = [np.asarray(q, dtype=np.float64).reshape(-1, 3) for q in qpoints]
            if len(qs) != self.B:
                raise ValueError(f"qpoints: expected one (Q, 3) array for all or one per structure ({self.B}), "
                                 f"got {len(qs)}")
        for q in qs:
            if not np.isfinite(q).all():
                raise ValueError("qpoints must be finite")
        return qs

    def _frequencies(self, qs: List[np.ndarray]):
        """The device outputs of one m3g_phonon_frequencies call over the ragged q lists ``qs``."""
        if self._st is None:
            raise RuntimeError("BatchPhonon: call run() before asking for frequencies")
        st, dev = self._st, self.device
        dims = [3 * a for a in st.n]
        q_ptr = torch.as_tensor(_cum([len(q) for q in qs], np.int32)).to(dev)
        f_ptr = torch.as_tensor(_cum([len(q) * d for q, d in zip(qs, dims)], np.int64)).to(dev)
        q = torch.as_tensor(np.concatenate(qs)).to(dev)
        total = int(sum(len(x) * d for x, d in zip(qs, dims)))
        out = SimpleNamespace(eig=torch.empty(total, dtype=torch.float64, device=dev),
                              freq=torch.empty(total, dtype=torch.float64, device=dev),
                              sweeps=torch.empty(q.shape[0], dtype=torch.int32, device=dev),
                              q_status=torch.empty(q.shape[0], dtype=torch.int32, device=dev))
        frequencies_launch(st, q, q_ptr, f_ptr, out)
        return out, q_ptr, f_ptr

    def frequencies(self, qpoints) -> List[np.ndarray]:
        """Per structure the (Q_b, 3n) frequencies in THz, ascending per q-point; negative values are imaginary modes
        (sign(lambda) sqrt(|lambda|)).  ``qpoints``: fractional coordinates of the unit cell's reciprocal lattice, one
        (Q, 3) array for all structures or one array per structure.  A failed structure (or a q-point whose Jacobi
        iteration did not converge in 30 sweeps) gives NaN.  The Jacobi sweep counts are kept in ``last_sweeps``."""
        qs = self._qpoints(qpoints)
        out, _, _ = self._frequencies(qs)
        freq = out.freq.cpu().numpy()
        sweeps = out.sweeps.cpu().numpy()
        res, o, iq = [], 0, 0
        self.last_sweeps = []
        for q, a in zip(qs, self._st.n):
            res.append(freq[o:o + len(q) * 3 * a].reshape(len(q), 3 * a))
            self.last_sweeps.append(sweeps[iq:iq + len(q)])
            o, iq = o + len(q) * 3 * a, iq + len(q)
        return res

    def thermal_properties(self, mesh=(20, 20, 20), temperatures=np.arange(0, 1001, 10),
                           cutoff_frequency: float = 0.01) -> List[dict]:
        """Harmonic thermal properties per unit cell over the Gamma-centred ``mesh`` (``mesh_qpoints``), one record per
        structure: ``temperatures`` (K), ``free_energy`` (eV), ``entropy`` (eV/K), ``heat_capacity`` (eV/K, constant
        volume), ``energy`` (eV), each (T,); modes below ``cutoff_frequency`` (THz) are left out; ``n_imaginary`` (mesh
        modes below -cutoff_frequency) and ``min_frequency`` (THz).  A failed structure gives NaN and n_imaginary -1."""
        temps = np.asarray(temperatures, dtype=np.float64).reshape(-1)
        if not (np.isfinite(temps).all() and (temps >= 0).all()):
            raise ValueError("temperatures must be finite and non-negative")
        cutoff = float(cutoff_frequency)
        if not (math.isfinite(cutoff) and cutoff >= 0.0):
            raise ValueError("cutoff_frequency must be finite and non-negative")
        q = mesh_qpoints(mesh)
        out, q_ptr, f_ptr = self._frequencies([q] * self.B)
        dev = self.device
        th = SimpleNamespace(values=torch.empty((self.B, len(temps), 4), dtype=torch.float64, device=dev),
                             n_imag=torch.empty(self.B, dtype=torch.int32, device=dev),
                             fmin=torch.empty(self.B, dtype=torch.float64, device=dev))
        thermal_launch(self._st, out.freq, f_ptr, q_ptr, torch.as_tensor(temps).to(dev), cutoff, th)
        values = th.values.cpu().numpy()
        n_imag = th.n_imag.cpu().numpy()
        fmin = th.fmin.cpu().numpy()
        return [dict(temperatures=temps.copy(), free_energy=values[b, :, 0], entropy=values[b, :, 1],
                     heat_capacity=values[b, :, 2], energy=values[b, :, 3], n_imaginary=int(n_imag[b]),
                     min_frequency=float(fmin[b]), mesh=tuple(int(m) for m in np.asarray(mesh).reshape(-1)))
                for b in range(self.B)]
