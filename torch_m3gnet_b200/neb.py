"""Batched climbing-image NEB: the migration barriers of many bands (hops) at once, on one calculator.

A band is images 0 .. M+1 of one structure (same lattice, same atomic numbers in the same order); images 0 and M+1 are
fixed endpoints and the M interior images move.  Per band the method is ASE's ``NEB(method="improvedtangent")``
(Henkelman & Jonsson, J. Chem. Phys. 113, 9978 (2000)) with an optional climbing image (Henkelman, Uberuaga & Jonsson,
ibid. 9901), optimised by FIRE on the whole band as one vector, as ASE's FIRE does on an ``NEB`` object: power, norms
and the ``max_move`` clip over the band's M n interior rows, fmax = the largest row |G| among them.  DESIGN.md §8 gives
the equations, including the two choices ASE does not make: a flat triplet (E_{i-1} = E_i = E_{i+1}) takes the
tangent t+ + t-, and a band whose tangent is zero or not finite at some image fails.

``BatchNEB`` keeps a working set of bands in one ragged batch.  Each step makes one ``calc.compute(..., sizes=...)``
call on every interior image of the working set (one lattice and one size per image) and one launch of
``m3g_neb_step`` (csrc/neb.cu), which advances every running band; its one read-back is the statuses.  The kernel
reduces each band's rows in a fixed order that depends only on those rows, so given the same forces a band's path is
bit-identical whatever else is in the batch.  The endpoint energies are evaluated once, before the first step, and
never again.  Bands enter in input order while their interior atoms fit ``max_atoms`` and leave by relax.py's
fixed-cell regroup policy (``admit`` / ``should_regroup``).
"""
from __future__ import annotations

import time
from typing import List, Optional

import numpy as np
import torch

from torch_m3gnet_b200 import _lib
from torch_m3gnet_b200.relax import RUNNING, STATUS_NAMES, admit, as_arrays, should_regroup

MAX_IMAGES = 64  # interior images per band: M3G_NEB_MAX_IMAGES (include/m3gnet_b200.h)


def interpolate(initial, final, n_images: int, mic: bool = False):
    """``n_images + 2`` linearly interpolated images from ``initial`` to ``final``, as (lattice, cart, numbers) tuples.
    With ``mic`` each atom's displacement is first wrapped to the minimum image in fractional coordinates of the
    initial cell, and the last image is ``final`` translated by those lattice vectors (the same structure, with raw
    differences along the band that no longer cross the cell)."""
    lat, c0, z = as_arrays(initial)
    lat1, c1, z1 = as_arrays(final)
    _check_image(lat, z, lat1, z1, "final")
    if int(n_images) < 1:
        raise ValueError("n_images must be at least 1")
    d = c1 - c0
    if mic:
        f = d @ np.linalg.inv(lat)
        d = (f - np.round(f)) @ lat
    m = int(n_images) + 1
    return [(lat.copy(), c0 + (i / m) * d, z.copy()) for i in range(m + 1)]


def _check_image(lat0, z0, lat, z, what):
    if z.shape != z0.shape or not np.array_equal(z, z0):
        raise ValueError(f"the {what} image's atomic numbers differ from the first image's (count and order)")
    if np.abs(lat - lat0).max() > 1e-12:
        raise ValueError(f"the {what} image's lattice differs from the first image's (NEB runs on a fixed cell)")


def _band(spec, n_images):
    """[(lattice, cart, numbers)] * (M + 2) of one band: an explicit image list (>= 3) or an (initial, final) pair."""
    spec = list(spec)
    if len(spec) == 2:
        if n_images is None:
            raise ValueError("an (initial, final) band needs n_images")
        return interpolate(spec[0], spec[1], n_images)
    if len(spec) < 3:
        raise ValueError("a band is an (initial, final) pair or a list of at least 3 images")
    images = [as_arrays(s) for s in spec]
    for j, (lat, _, z) in enumerate(images[1:], 1):
        _check_image(images[0][0], images[0][2], lat, z, f"#{j}")
    return images


class _Bands:
    """Working-set state on the device: the arrays m3g_neb_step reads and writes, plus host bookkeeping.  Rows are the
    interior atoms (band-major, then image-major), images the interior images, ends the endpoints' atoms (2 n per
    band: the initial image's, then the final image's)."""

    ROW, IMAGE, END = ("pos", "v"), ("e_frame",), ("ends",)
    BAND = ("e_end", "k", "dt", "a", "fmax", "n_pos", "n_steps", "status", "i_climb")

    def __init__(self, device):
        self.device = device
        f64 = dict(dtype=torch.float64, device=device)
        i32 = dict(dtype=torch.int32, device=device)
        self.ids: List[int] = []
        self.M: List[int] = []
        self.n: List[int] = []
        for k in ("pos", "v", "ends"):
            setattr(self, k, torch.zeros((0, 3), **f64))
        self.e_end = torch.zeros((0, 2), **f64)
        for k in ("e_frame", "k", "dt", "a", "fmax"):
            setattr(self, k, torch.zeros(0, **f64))
        for k in ("n_pos", "n_steps", "status", "i_climb"):
            setattr(self, k, torch.zeros(0, **i32))
        self.reindex([], [])

    @property
    def B(self) -> int:
        return len(self.ids)

    @property
    def N(self) -> int:
        return int(sum(m * n for m, n in zip(self.M, self.n)))

    def _select(self, keep, counts, names):
        ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        idx = np.concatenate([np.arange(ptr[b], ptr[b + 1]) for b in keep]) if keep else np.zeros(0, np.int64)
        idx_d = torch.as_tensor(idx).to(self.device)
        for k in names:
            setattr(self, k, getattr(self, k).index_select(0, idx_d))

    def keep(self, keep: List[int]):
        """Only the bands at working-set positions ``keep`` (ascending) stay; their state is carried over."""
        self._select(keep, [m * n for m, n in zip(self.M, self.n)], self.ROW)
        self._select(keep, self.M, self.IMAGE)
        self._select(keep, [2 * n for n in self.n], self.END)
        self._select(keep, [1] * self.B, self.BAND)
        self.ids = [self.ids[b] for b in keep]
        self.M = [self.M[b] for b in keep]
        self.n = [self.n[b] for b in keep]
        self.reindex([self.z_h[b] for b in keep], [self.lat_h[b] for b in keep])

    def append(self, ids, bands, e_end, k, fire):
        """Fresh FIRE state (zero velocity) for the bands ``ids``."""
        dev = self.device
        f64 = dict(dtype=torch.float64, device=dev)
        i32 = dict(dtype=torch.int32, device=dev)
        m = len(ids)
        pos = torch.as_tensor(np.concatenate([np.concatenate([im[1] for im in bands[i][1:-1]]) for i in ids])).to(dev)
        ends = np.concatenate([np.concatenate([bands[i][0][1], bands[i][-1][1]]) for i in ids])
        new = dict(pos=pos, v=torch.zeros_like(pos), ends=torch.as_tensor(ends).to(dev),
                   e_frame=torch.zeros(sum(len(bands[i]) - 2 for i in ids), **f64),
                   e_end=torch.as_tensor(np.asarray([e_end[i] for i in ids], dtype=np.float64)).to(dev),
                   k=torch.as_tensor(np.asarray([k[i] for i in ids], dtype=np.float64)).to(dev),
                   dt=torch.full((m,), fire["dt"], **f64), a=torch.full((m,), fire["a_start"], **f64),
                   fmax=torch.zeros(m, **f64), n_pos=torch.zeros(m, **i32), n_steps=torch.zeros(m, **i32),
                   status=torch.zeros(m, **i32), i_climb=torch.zeros(m, **i32))
        for name in self.ROW + self.IMAGE + self.END + self.BAND:
            setattr(self, name, torch.cat([getattr(self, name), new[name]]))
        self.ids += list(ids)
        self.M += [len(bands[i]) - 2 for i in ids]
        self.n += [len(bands[i][0][2]) for i in ids]
        self.reindex(self.z_h + [bands[i][0][2] for i in ids], self.lat_h + [bands[i][0][0] for i in ids])

    def reindex(self, z_h, lat_h):
        self.z_h, self.lat_h = list(z_h), list(lat_h)
        cum = lambda c: torch.as_tensor(np.concatenate([[0], np.cumsum(c)]).astype(np.int32)).to(self.device)  # noqa
        self.row_ptr = cum([m * n for m, n in zip(self.M, self.n)])
        self.image_ptr = cum(self.M)
        self.end_ptr = cum([2 * n for n in self.n])
        # the compute call's layout: every interior image as a structure of its own
        self.sizes = [n for m, n in zip(self.M, self.n) for _ in range(m)]
        self.z_images = (np.concatenate([np.tile(z, m) for m, z in zip(self.M, self.z_h)]) if self.M
                         else np.zeros(0, np.int64))
        self.lat_images = (np.concatenate([np.repeat(lat[None], m, axis=0) for m, lat in zip(self.M, self.lat_h)])
                           if self.M else np.zeros((0, 3, 3)))


def neb_step(st: _Bands, forces, energy, climb: bool, fire, fmax: float, steps: int):
    """One m3g_neb_step call on the working set ``st`` (forces (rows,3), energy (images) float32)."""
    _lib.call("neb_step", forces, energy, st.row_ptr, st.image_ptr, st.end_ptr, st.B, max(st.M), st.ends, st.e_end,
              st.k, int(bool(climb)), fire["dt_max"], fire["max_move"], int(fire["n_min"]), fire["f_inc"],
              fire["f_dec"], fire["a_start"], fire["f_a"], float(fmax), int(steps), st.pos, st.v, st.dt, st.a,
              st.n_pos, st.n_steps, st.status, st.fmax, st.i_climb, st.e_frame)


class BatchNEB:
    """Climbing-image NEB of many bands at once (module docstring).

    ``bands``: per band an explicit image list (at least 3 structures, endpoints included) or an ``(initial, final)``
    pair, interpolated linearly with ``n_images`` interior images (``interpolate``; use it directly for ``mic``).
    Structures are (lattice (3,3), cart (n,3), atomic_numbers (n,)) tuples or atoms objects, as ``BatchFire`` takes.
    Every image of a band needs the band's lattice (to 1e-12 A) and atomic numbers; at most ``MAX_IMAGES`` interior
    images.  ``k``: spring constant in eV/A^2, one value or one per band.  ``climb``: the highest interior image climbs.
    ``max_atoms`` bounds the interior atoms of the working set and the atoms of each endpoint evaluation (None = no
    bound); a band larger than the budget runs alone.  The FIRE parameters have ``Fire``'s meaning, per band."""

    def __init__(self, calc, bands, n_images: Optional[int] = None, k=0.1, climb: bool = False,
                 max_atoms: Optional[int] = None, dt: float = 0.1, dt_max: float = 1.0, max_move: float = 0.2,
                 n_min: int = 5, f_inc: float = 1.1, f_dec: float = 0.5, a_start: float = 0.1, f_a: float = 0.99):
        self.calc = calc
        if n_images is not None and int(n_images) < 1:
            raise ValueError("n_images must be at least 1")
        self.bands = [_band(b, n_images) for b in bands]
        for i, band in enumerate(self.bands):
            if len(band) - 2 > MAX_IMAGES:
                raise ValueError(f"band {i} has {len(band) - 2} interior images; at most {MAX_IMAGES} are supported")
        kk = np.asarray(k, dtype=np.float64)
        kk = np.full(len(self.bands), float(kk)) if kk.ndim == 0 else kk.reshape(-1)
        if kk.size != len(self.bands):
            raise ValueError(f"k needs one value or one per band ({len(self.bands)}), got {kk.size}")
        if not (np.isfinite(kk).all() and (kk >= 0).all()):
            raise ValueError("k must be finite and non-negative")
        self.k = kk
        self.climb = bool(climb)
        if max_atoms is not None and int(max_atoms) < 1:
            raise ValueError("max_atoms must be positive or None")
        self.max_atoms = None if max_atoms is None else int(max_atoms)
        self.fire = dict(dt=float(dt), dt_max=float(dt_max), max_move=float(max_move), n_min=int(n_min),
                         f_inc=float(f_inc), f_dec=float(f_dec), a_start=float(a_start), f_a=float(f_a))
        dev = getattr(calc, "device", None)
        self.device = dev if dev is not None else torch.device("cuda", torch.cuda.current_device())
        self.n_iterations = self.n_regroups = self.n_endpoint_calls = 0
        self.regroup_seconds = 0.0

    def endpoint_energies(self) -> np.ndarray:
        """(bands, 2) float64 energies of every band's endpoints: compute calls over the endpoints in input order
        (initial, final, next band's initial, ...), in chunks of at most ``max_atoms`` atoms."""
        ends = [im for band in self.bands for im in (band[0], band[-1])]
        sizes = [len(s[2]) for s in ends]
        e = np.empty(len(ends))
        start = 0
        while start < len(ends):
            end = admit(sizes, start, self.max_atoms, 0, 0)
            chunk = ends[start:end]
            out = self.calc.compute(np.stack([s[0] for s in chunk]), np.concatenate([s[1] for s in chunk]),
                                    np.concatenate([s[2] for s in chunk]), sizes[start:end])
            e[start:end] = out[0].reshape(-1).double().cpu().numpy()
            self.n_endpoint_calls += 1
            start = end
        return e.reshape(-1, 2)

    def run(self, fmax: float = 0.05, steps: int = 200) -> List[dict]:
        """Optimise every band; one record per band, in input order, all of the frame at which the band stopped:
        ``status`` ("converged": fmax below ``fmax``; "not converged" within ``steps`` steps; "failed": a non-finite
        force or energy, or a degenerate tangent), ``n_steps``, ``fmax`` (eV/A, largest row |G| of the interior
        images), ``energies`` (M+2,) eV endpoints included, ``positions`` (M+2, n, 3) A, ``lattice`` (3,3),
        ``i_climb`` (the highest interior image, 1 .. M) and ``barrier_forward`` / ``barrier_backward`` (max energy
        minus the first / last image's).  A band with a non-finite endpoint energy fails with n_steps 0 before any
        step: its interior energies are NaN and i_climb is -1."""
        results: List[Optional[dict]] = [None] * len(self.bands)
        if not self.bands:
            return []
        e_end = self.endpoint_energies()
        queue = []
        for i, band in enumerate(self.bands):
            if np.isfinite(e_end[i]).all():
                queue.append(i)
                continue
            M = len(band) - 2
            energies = np.concatenate([[e_end[i][0]], np.full(M, np.nan), [e_end[i][1]]])
            results[i] = self._result(i, "failed", 0, np.inf, energies, np.stack([im[1] for im in band]), -1)
        sizes = [(len(self.bands[i]) - 2) * len(self.bands[i][0][2]) for i in queue]
        st = _Bands(self.device)
        pin = self.device.type == "cuda"
        nxt = admit(sizes, 0, self.max_atoms, 0, 0)
        if nxt:
            st.append(queue[:nxt], self.bands, e_end, self.k, self.fire)
        while st.B:
            out = self.calc.compute(st.lat_images, st.pos, st.z_images, st.sizes)
            energy = out[0].reshape(-1).to(torch.float32).contiguous()
            forces = out[1].reshape(-1, 3).to(torch.float32).contiguous()
            neb_step(st, forces, energy, self.climb, self.fire, fmax, steps)
            self.n_iterations += 1
            status_h = torch.empty(st.B, dtype=torch.int32, pin_memory=pin)  # the step's one read-back
            status_h.copy_(st.status, non_blocking=pin)
            if pin:
                torch.cuda.current_stream(self.device).synchronize()
            status = status_h.numpy()
            done = status != RUNNING
            band_atoms = np.asarray([m * n for m, n in zip(st.M, st.n)])
            if not should_regroup(int(band_atoms[done].sum()), st.N, bool(done.any()), bool(done.all()), False):
                continue
            t0 = time.perf_counter()
            self._record(st, np.flatnonzero(done), status, results)
            st.keep([int(b) for b in np.flatnonzero(~done)])
            end = admit(sizes, nxt, self.max_atoms, st.N, st.B)
            if end > nxt:
                st.append(queue[nxt:end], self.bands, e_end, self.k, self.fire)
                nxt = end
            self.n_regroups += 1
            self.regroup_seconds += time.perf_counter() - t0
        return results

    def _result(self, i, status, n_steps, fmax, energies, positions, i_climb):
        top = float(np.max(energies))
        return dict(status=status, n_steps=int(n_steps), fmax=float(fmax), energies=energies, positions=positions,
                    lattice=self.bands[i][0][0].copy(), i_climb=int(i_climb), barrier_forward=top - energies[0],
                    barrier_backward=top - energies[-1])

    def _record(self, st: _Bands, finished, status, results):
        if len(finished) == 0:
            return
        idx = torch.as_tensor(finished).to(self.device)
        host = {k: getattr(st, k).index_select(0, idx).cpu().numpy()
                for k in ("n_steps", "fmax", "i_climb", "e_end")}
        pos = st.pos.cpu().numpy()
        ends = st.ends.cpu().numpy()
        e_frame = st.e_frame.cpu().numpy()
        row = np.concatenate([[0], np.cumsum([m * n for m, n in zip(st.M, st.n)])])
        img = np.concatenate([[0], np.cumsum(st.M)])
        end = np.concatenate([[0], np.cumsum([2 * n for n in st.n])])
        for j, b in enumerate(finished):
            M, n = st.M[b], st.n[b]
            e = ends[end[b]:end[b + 1]]
            positions = np.concatenate([e[:n][None], pos[row[b]:row[b + 1]].reshape(M, n, 3), e[n:][None]])
            energies = np.concatenate([host["e_end"][j][:1], e_frame[img[b]:img[b + 1]], host["e_end"][j][1:]])
            results[st.ids[b]] = self._result(st.ids[b], STATUS_NAMES[int(status[b])], host["n_steps"][j],
                                              host["fmax"][j], energies, positions, host["i_climb"][j])

