"""numpy float64 restatement of the batched Langevin step with the stochastic cell-rescaling barostat
(m3g_langevin_npt_step, csrc/md.cu, torch_m3gnet_b200/md.py), written from the ABI comment in include/m3gnet_b200.h.
It reuses tests/md_oracle.py's Philox and follows its arithmetic operation for operation, so with beta_T = 0 (mu = 1
exactly) it equals md_oracle.langevin_step bit for bit.  Structures of one size are stepped together (the statistical
tests run thousands of steps on hundreds of structures); numpy's sums over a structure's rows are the same whether the
rows come one structure or a stack of them at a time.

State: md_oracle's dict plus lattice (B,3,3) and P0, beta_T, tau_p (B) f64; updated in place."""
import numpy as np

from tests import md_oracle as MO

KB, RUNNING, FAILED = MO.KB, MO.RUNNING, MO.FAILED
STATE_KEYS = MO.STATE_KEYS + ("lattice", "P0", "beta_T", "tau_p")
ISOTROPIC, PER_AXIS = 0, 1
TAG_BAROSTAT = 2


def obs_width(coupling):
    return 6 if coupling == ISOTROPIC else 9


def normals(n, sids, ks, tag, seed):
    """(G, n, 3) normals of atoms 0..n-1 of G structures with stream ids ``sids`` at steps ``ks``: md_oracle.normals,
    one structure per row."""
    G = len(sids)
    ctr = np.zeros((G, n, 4), dtype=np.uint64)
    ctr[:, :, 0] = np.arange(n, dtype=np.uint64)[None]
    ctr[:, :, 1] = (np.asarray(sids, dtype=np.int64).astype(np.uint64))[:, None]
    ctr[:, :, 2] = np.asarray(ks, dtype=np.uint64)[:, None]
    ctr[:, :, 3] = np.uint64(tag)
    key = np.zeros((G, n, 2), dtype=np.uint64)
    key[..., 0] = np.uint64(MO.seed_word(seed))
    u = MO.uniform53(MO.philox4x64_10(ctr, key))
    r0, r2 = np.sqrt(-2.0 * np.log(u[..., 0])), np.sqrt(-2.0 * np.log(u[..., 2]))
    return np.stack([r0 * np.cos(2 * np.pi * u[..., 1]), r0 * np.sin(2 * np.pi * u[..., 1]),
                     r2 * np.cos(2 * np.pi * u[..., 3])], axis=-1)


def volume(L):
    """|det L| of (..., 3, 3) lattices by the kernel's cofactor expansion along the first row."""
    return np.abs(L[..., 0, 0] * (L[..., 1, 1] * L[..., 2, 2] - L[..., 1, 2] * L[..., 2, 1])
                  - L[..., 0, 1] * (L[..., 1, 0] * L[..., 2, 2] - L[..., 1, 2] * L[..., 2, 0])
                  + L[..., 0, 2] * (L[..., 1, 0] * L[..., 2, 1] - L[..., 1, 1] * L[..., 2, 0]))


def npt_step(st, forces, sigma, energy, atom_ptr, dt, max_step_move, seed, advance, slot, obs, coupling,
             max_step_strain):
    """One call for every running structure: close step k - 1, check frame k, form V and the pressures, draw the
    barostat noise and the scale factors mu, fail or record (obs (n_slots, B, 6 or 9) when slot >= 0), and unless
    ``advance`` is false advance to x_{k+1} by B A O A followed by the rescaling x, L by diag(mu), v by diag(mu)^-1."""
    forces = np.asarray(forces, dtype=np.float64)
    sigma = np.asarray(sigma, dtype=np.float64).reshape(-1, 3, 3)
    energy = np.asarray(energy, dtype=np.float64)
    atom_ptr = np.asarray(atom_ptr, dtype=np.int64)
    sizes = np.diff(atom_ptr)
    h = 0.5 * dt
    running = np.flatnonzero(st["status"] == RUNNING)
    for n in np.unique(sizes[running]):
        bs = running[sizes[running] == n]
        rows = atom_ptr[bs][:, None] + np.arange(n)[None]                   # (G, n)
        k = st["step"][bs].astype(np.int64)
        f, im = forces[rows], st["inv_mass"][rows]
        acc = f * im[..., None]
        v = np.where((k > 0)[:, None, None], st["v"][rows] + h * acc, st["v"][rows])
        with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
            w2 = (v * v).sum(axis=2)
            vmax = np.sqrt(w2.max(axis=1))
            ok = (np.isfinite(f).all(axis=(1, 2)) & np.isfinite(w2).all(axis=1) & np.isfinite(energy[bs])
                  & (vmax * dt <= max_step_move))
            ek = 0.5 * (w2 / im).sum(axis=1)
            kaa = 0.5 * ((v / im[..., None]) * v).sum(axis=1)                 # (G, 3)
            # the barostat
            L = st["lattice"][bs]
            sg = sigma[bs]
            V = volume(L)
            diag = np.stack([sg[:, 0, 0], sg[:, 1, 1], sg[:, 2, 2]], axis=1)
            p_int = 2.0 * ek / (3.0 * V) - (diag[:, 0] + diag[:, 1] + diag[:, 2]) / 3.0
            p_axis = 2.0 * kaa / V[:, None] - diag
            xi = normals(1, st["sid"][bs], k, TAG_BAROSTAT, seed)[:, 0]      # (G, 3)
            P0, bt, tau, kT = st["P0"][bs], st["beta_T"][bs], st["tau_p"][bs], st["kT"][bs]
            drift = bt * dt / tau
            diff = np.sqrt(2.0 * kT * bt * dt / (V * tau))
            if coupling == ISOTROPIC:
                le = np.repeat(((-drift * (P0 - p_int) + diff * xi[:, 0]) / 3.0)[:, None], 3, axis=1)
            else:
                le = -drift[:, None] * (P0[:, None] - p_axis) + diff[:, None] * xi
            ok &= np.isfinite(sg).all(axis=(1, 2)) & np.isfinite(V) & (np.abs(le) <= max_step_strain).all(axis=1)
            mu = np.exp(le)
        st["status"][bs[~ok]] = FAILED
        if slot >= 0:
            for j in np.flatnonzero(ok):
                b, nn = bs[j], float(n)
                row = [energy[b], ek[j], 2.0 * ek[j] / ((3.0 * nn - 3.0) * KB), st["bath"][b], V[j], p_int[j]]
                obs[slot, b] = row + (list(p_axis[j]) if coupling == PER_AXIS else [])
        g = np.flatnonzero(ok)
        if not len(g):
            continue
        bs, rows, k, v, acc, im, mu = bs[g], rows[g], k[g], v[g], acc[g], im[g], mu[g]
        if not advance:
            st["v"][rows] = v
            continue
        u = v + h * acc
        ke0 = 0.5 * ((u * u).sum(axis=2) / im).sum(axis=1)
        x = st["pos"][rows] + h * u
        xi = normals(n, st["sid"][bs], k, 0, seed)
        o = st["c1"][bs][:, None, None] * u + st["c2"][bs][:, None, None] * (np.sqrt(st["kT"][bs][:, None] * im)[..., None] * xi)
        m = 1.0 / im
        o = o - (o * m[..., None]).sum(axis=1)[:, None, :] / m.sum(axis=1)[:, None, None]
        st["pos"][rows] = (x + h * o) * mu[:, None, :]
        st["v"][rows] = o * (1.0 / mu)[:, None, :]
        st["lattice"][bs] = st["lattice"][bs] * mu[:, None, :]
        st["bath"][bs] += 0.5 * ((o * o).sum(axis=2) / im).sum(axis=1) - ke0
        st["step"][bs] = k + 1


def fresh_state(carts, lattices, masses, temperature, friction, dt, pressure, compressibility, barostat_time,
                ids=None):
    """md_oracle.fresh_state plus the cells and the barostat's per-structure parameters."""
    st, ptr = MO.fresh_state(carts, masses, temperature, friction, dt, ids)
    B = len(carts)
    st["lattice"] = np.stack([np.asarray(L, dtype=np.float64) for L in lattices])
    for key, val in (("P0", pressure), ("beta_T", compressibility), ("tau_p", barostat_time)):
        st[key] = np.asarray(val, dtype=np.float64) * np.ones(B)
    return st, ptr
