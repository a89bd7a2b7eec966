"""numpy float64 restatement of the batched Langevin step (m3g_langevin_step), the Maxwell-Boltzmann draw
(m3g_md_maxwell_boltzmann) and their Philox4x64-10 noise (csrc/md.cu, torch_m3gnet_b200/md.py), written from the ABI
comment in include/m3gnet_b200.h one structure at a time.  Shared by the CPU and GPU batched-MD tests.

State: a dict of numpy arrays with the names of md.py's working set (pos, v (N,3); inv_mass (N); c1, c2, kT, bath (B)
f64; sid (B) int64; step, status (B) int32); updated in place."""
import numpy as np

KB = 8.617333262e-5
RUNNING, FAILED = 0, 1
STATE_KEYS = ("pos", "v", "inv_mass", "c1", "c2", "kT", "bath", "sid", "step", "status")

_U = np.uint64
_M32 = _U(0xFFFFFFFF)
_PHILOX_M = (_U(0xD2E7470EE14C6C93), _U(0xCA5A826395121157))
_PHILOX_W = (_U(0x9E3779B97F4A7C15), _U(0xBB67AE8584CAA73B))


def _mulhilo(a, b):
    """(hi, lo) 64-bit words of the 128-bit products a * b (uint64 arrays), from 32-bit halves."""
    a0, a1 = a & _M32, a >> _U(32)
    b0, b1 = b & _M32, b >> _U(32)
    p00, p01, p10, p11 = a0 * b0, a0 * b1, a1 * b0, a1 * b1
    mid = (p00 >> _U(32)) + (p01 & _M32) + (p10 & _M32)
    hi = p11 + (p01 >> _U(32)) + (p10 >> _U(32)) + (mid >> _U(32))
    return hi, a * b


def philox4x64_10(ctr, key):
    """Philox4x64-10 words (..., 4) uint64 of counters (..., 4) and keys (..., 2) (Random123's philox4x64 with ten
    rounds: the key is bumped before every round but the first)."""
    with np.errstate(over="ignore"):
        c = [np.array(w, dtype=np.uint64) for w in np.moveaxis(np.asarray(ctr, dtype=np.uint64), -1, 0)]
        k = [np.array(w, dtype=np.uint64) for w in np.moveaxis(np.asarray(key, dtype=np.uint64), -1, 0)]
        for r in range(10):
            if r > 0:
                k = [k[0] + _PHILOX_W[0], k[1] + _PHILOX_W[1]]
            hi0, lo0 = _mulhilo(_PHILOX_M[0], c[0])
            hi1, lo1 = _mulhilo(_PHILOX_M[1], c[2])
            c = [hi1 ^ c[1] ^ k[0], lo1, hi0 ^ c[3] ^ k[1], lo0]
    return np.stack(c, axis=-1)


def uniform53(w):
    """((w >> 11) + 0.5) 2^-53 of uint64 words: in (0, 1), never 0."""
    return ((np.asarray(w, dtype=np.uint64) >> _U(11)).astype(np.float64) + 0.5) * 2.0 ** -53


def seed_word(seed) -> int:
    """The key word of a seed passed as int64 (reinterpreted as uint64)."""
    return int(seed) % (1 << 64)


def normals(n, sid, k, tag, seed):
    """(n, 3) standard normals of atoms 0..n-1 of the structure with stream id ``sid`` at step ``k``: one Philox call
    on the counter (i, sid, k, tag) under the key (seed, 0), Box-Muller."""
    ctr = np.zeros((n, 4), dtype=np.uint64)
    ctr[:, 0] = np.arange(n, dtype=np.uint64)
    ctr[:, 1], ctr[:, 2], ctr[:, 3] = _U(int(sid) % (1 << 64)), _U(int(k)), _U(int(tag))
    key = np.zeros((n, 2), dtype=np.uint64)
    key[:, 0] = _U(seed_word(seed))
    u = uniform53(philox4x64_10(ctr, key))
    r0, r2 = np.sqrt(-2.0 * np.log(u[:, 0])), np.sqrt(-2.0 * np.log(u[:, 2]))
    return np.stack([r0 * np.cos(2 * np.pi * u[:, 1]), r0 * np.sin(2 * np.pi * u[:, 1]),
                     r2 * np.cos(2 * np.pi * u[:, 3])], axis=1)


def _remove_com(v, im):
    m = 1.0 / im
    return v - (v * m[:, None]).sum(axis=0) / m.sum()


def maxwell_boltzmann(st, atom_ptr, seed):
    """v = sqrt(kT inv_mass) xi (step 0, tag 1), centre-of-mass velocity removed, per structure."""
    for b in range(len(atom_ptr) - 1):
        s, t = int(atom_ptr[b]), int(atom_ptr[b + 1])
        im = st["inv_mass"][s:t]
        v = np.sqrt(st["kT"][b] * im)[:, None] * normals(t - s, st["sid"][b], 0, 1, seed)
        st["v"][s:t] = _remove_com(v, im)


def langevin_step(st, forces, energy, atom_ptr, dt, max_step_move, seed, advance, slot, obs):
    """One call for every running structure: close step k - 1, check and record frame k (obs (n_slots, B, 4) when
    slot >= 0), and unless ``advance`` is false advance to x_{k+1} by B A O A."""
    forces = np.asarray(forces, dtype=np.float64)
    h = 0.5 * dt
    for b in range(len(atom_ptr) - 1):
        if st["status"][b] != RUNNING:
            continue
        s, t = int(atom_ptr[b]), int(atom_ptr[b + 1])
        n, k = t - s, int(st["step"][b])
        f, im = forces[s:t], st["inv_mass"][s:t]
        acc = f * im[:, None]
        v = st["v"][s:t] + h * acc if k > 0 else st["v"][s:t].copy()
        with np.errstate(invalid="ignore", over="ignore"):
            w2 = (v * v).sum(axis=1)
            vmax = float(np.sqrt(w2.max()))
        if not (np.isfinite(f).all() and np.isfinite(w2).all() and np.isfinite(energy[b])
                and vmax * dt <= max_step_move):
            st["status"][b] = FAILED
            continue
        ek = 0.5 * float((w2 / im).sum())
        if slot >= 0:
            obs[slot, b] = (energy[b], ek, 2.0 * ek / ((3.0 * n - 3.0) * KB), st["bath"][b])
        if not advance:
            st["v"][s:t] = v
            continue
        u = v + h * acc
        ke0 = 0.5 * float(((u * u).sum(axis=1) / im).sum())
        x = st["pos"][s:t] + h * u
        xi = normals(n, st["sid"][b], k, 0, seed)
        o = st["c1"][b] * u + st["c2"][b] * (np.sqrt(st["kT"][b] * im)[:, None] * xi)
        o = _remove_com(o, im)
        st["pos"][s:t] = x + h * o
        st["v"][s:t] = o
        st["bath"][b] += 0.5 * float(((o * o).sum(axis=1) / im).sum()) - ke0
        st["step"][b] = k + 1


def fresh_state(carts, masses, temperature, friction, dt, ids=None):
    """Starting state (zero velocities, no steps) of structures with positions ``carts`` [(n,3)], masses [(n,)] amu,
    temperature / friction per structure, and their atom_ptr; stream ids ``ids`` (default 0..B-1)."""
    from torch_m3gnet_b200.calculator import ACC_UNIT

    sizes = [len(c) for c in carts]
    B = len(sizes)
    pos = np.concatenate([np.asarray(c, dtype=np.float64) for c in carts])
    c1 = np.exp(-np.asarray(friction, dtype=np.float64) * dt) * np.ones(B)
    st = dict(pos=pos.copy(), v=np.zeros_like(pos), inv_mass=ACC_UNIT / np.concatenate(masses).astype(np.float64),
              c1=c1, c2=np.sqrt(1.0 - c1 * c1), kT=KB * np.asarray(temperature, dtype=np.float64) * np.ones(B),
              bath=np.zeros(B), sid=np.arange(B, dtype=np.int64) if ids is None else np.asarray(ids, np.int64),
              step=np.zeros(B, np.int32), status=np.zeros(B, np.int32))
    return st, np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
