"""Seeded synthetic periodic structures for the benchmarks (SURVEY.md §8(d) configurations C1–C5).
numpy float64; independent of the oracle so that the product arm of bench.py never imports ``oracle/``."""
from __future__ import annotations

import numpy as np

CU_Z = 29
A_CU = 3.615


def fcc_cu_supercell(reps: int, jitter: float, seed: int):
    """reps^3 conventional FCC Cu cells, positions + U(-jitter, jitter) from default_rng(seed).
    Returns (lattice (3,3), cart (n,3), atomic numbers (n))."""
    base = np.array([[0, 0, 0], [0, 0.5, 0.5], [0.5, 0, 0.5], [0.5, 0.5, 0]], dtype=np.float64)
    cells = np.stack(np.meshgrid(*[np.arange(reps)] * 3, indexing="ij"), axis=-1).reshape(-1, 3)
    cart = (cells[:, None, :] + base[None, :, :]).reshape(-1, 3) * A_CU
    if jitter > 0:
        cart = cart + np.random.default_rng(seed).uniform(-jitter, jitter, size=cart.shape)
    return np.eye(3) * (A_CU * reps), cart, np.full(len(cart), CU_Z, dtype=np.int64)


def config2_batch(n_structures: int = 256, first_seed: int = 0):
    """C2: n_structures copies of 3x3x3 cells (108 atoms), structure s perturbed U(-0.1, 0.1) with default_rng(s)."""
    lats, carts, zs, sizes = [], [], [], []
    for s in range(first_seed, first_seed + n_structures):
        lat, cart, z = fcc_cu_supercell(3, 0.1, s)
        lats.append(lat)
        carts.append(cart)
        zs.append(z)
        sizes.append(len(cart))
    return np.stack(lats), np.concatenate(carts), np.concatenate(zs), sizes


def mpf_like_structure(s: int):
    """C3: 20–200 atoms, 3–5 species from Z in [1,94], sheared cubic cell of density U(0.04,0.09) Å^-3, random
    sequential insertion with minimum distance 1.6 Å (jittered-lattice fallback if insertion stalls)."""
    rng = np.random.default_rng(1000 + s)
    n = int(rng.integers(20, 201))
    n_species = int(rng.integers(3, 6))
    species = rng.choice(np.arange(1, 95), size=n_species, replace=False)
    rho = rng.uniform(0.04, 0.09)
    a = (n / rho) ** (1.0 / 3.0)
    lattice = a * (np.eye(3) + rng.uniform(-0.1, 0.1, size=(3, 3)) * (1 - np.eye(3)))
    imgs = np.stack(np.meshgrid(*[np.arange(-1, 2)] * 3, indexing="ij"), axis=-1).reshape(-1, 3) @ lattice
    pts = []
    tries = 0
    while len(pts) < n and tries < 200 * n:
        tries += 1
        c = rng.uniform(0, 1, size=3) @ lattice
        if pts:
            d = np.asarray(pts)[:, None, :] + imgs[None, :, :] - c[None, None, :]
            if np.min(np.einsum("ijk,ijk->ij", d, d)) < 1.6**2:
                continue
        pts.append(c)
    if len(pts) < n:
        m = int(np.ceil(n ** (1 / 3)))
        grid = np.stack(np.meshgrid(*[np.arange(m)] * 3, indexing="ij"), axis=-1).reshape(-1, 3)[:n]
        pts = list(((grid + 0.5) / m + rng.uniform(-0.02, 0.02, size=(n, 3))) @ lattice)
    return lattice, np.asarray(pts), rng.choice(species, size=n).astype(np.int64)


def fcc_cu_vacancy_hop(reps: int):
    """(initial, final) of a vacancy hop in reps^3 conventional FCC Cu cells (4 reps^3 - 1 atoms): the vacancy at the
    origin, and the nearest neighbour at (0, a/2, a/2) moved into it.  Unrelaxed, same atom order in both."""
    lat, cart, z = fcc_cu_supercell(reps, 0.0, 0)
    cart, z = cart[1:], z[1:]
    j = int(np.argmin(np.linalg.norm(cart - np.array([0.0, 0.5, 0.5]) * A_CU, axis=1)))
    final = cart.copy()
    final[j] = 0.0
    return (lat, cart, z), (lat.copy(), final, z.copy())
