"""numpy float64 restatement of one batched FIRE step (m3g_fire_step, torch_m3gnet_b200/relax.py::fire_step), written
from calculator.py::Fire.step / Fire.run / Fire.generalised_forces / Fire._set_generalised one structure at a time.
Shared by the CPU and GPU batched-FIRE tests.

State: a dict of numpy arrays with the names of relax.py::_State (pos, v, x (N,3); xc, vc, L0, lattice, sigma_frame
(B,3,3); dt, a, fmax, e_frame, cell_factor (B); n_pos, n_steps, status (B) int32); updated in place."""
import numpy as np

RUNNING, CONVERGED, NOT_CONVERGED, FAILED = 0, 1, 2, 3
STATE_KEYS = ("pos", "v", "x", "xc", "vc", "L0", "lattice", "sigma_frame", "dt", "a", "fmax", "e_frame", "cell_factor",
              "n_pos", "n_steps", "status")


def generalised_forces(forces, sigma, L0, lattice, cell_factor, pressure):
    """(n+3, 3) of one structure: F D and -V (sigma + p I) D^-T / cell_factor, D = solve(L0, L)^T."""
    D = np.linalg.solve(L0, lattice).T
    vol = abs(float(np.linalg.det(lattice)))
    virial = -vol * (np.asarray(sigma, dtype=np.float64) + pressure * np.eye(3))
    cell_f = np.linalg.solve(D, virial.T).T / cell_factor
    return np.concatenate([np.asarray(forces, dtype=np.float64) @ D, cell_f])


def fire_step(st, forces, sigma, energy, fire, fmax_target, steps, pressure, atom_ptr):
    """One step for every running structure; ``sigma`` (B,3,3) or None (fixed cells)."""
    cell = sigma is not None
    forces = np.asarray(forces, dtype=np.float64)
    for b in range(len(atom_ptr) - 1):
        if st["status"][b] != RUNNING:
            continue
        s, t = int(atom_ptr[b]), int(atom_ptr[b + 1])
        st["e_frame"][b] = energy[b]
        if cell:
            st["sigma_frame"][b] = sigma[b]
            g = generalised_forces(forces[s:t], sigma[b], st["L0"][b], st["lattice"][b], st["cell_factor"][b],
                                   pressure)
            v = np.concatenate([st["v"][s:t], st["vc"][b]])
        else:
            g = forces[s:t]
            v = st["v"][s:t].copy()
        if not np.isfinite(g).all():
            st["status"][b], st["fmax"][b] = FAILED, np.inf
            continue
        fm = float(np.sqrt((g * g).sum(axis=1)).max())
        st["fmax"][b] = fm
        if fm < fmax_target:
            st["status"][b] = CONVERGED
            continue
        if st["n_steps"][b] >= steps:
            st["status"][b] = NOT_CONVERGED
            continue
        a, dt, n_pos = float(st["a"][b]), float(st["dt"][b]), int(st["n_pos"][b])
        if float((g * v).sum()) > 0.0:
            fn = np.sqrt((g * g).sum())
            v = (1.0 - a) * v + a * np.sqrt((v * v).sum()) * g / max(fn, 1e-30)
            if n_pos > fire["n_min"]:
                dt = min(dt * fire["f_inc"], fire["dt_max"])
                a *= fire["f_a"]
            n_pos += 1
        else:
            v = np.zeros_like(v)
            a, dt, n_pos = fire["a_start"], dt * fire["f_dec"], 0
        v = v + dt * g
        dr = dt * v
        norm = float(np.sqrt((dr * dr).sum()))
        if norm > fire["max_move"]:
            dr = dr * (fire["max_move"] / norm)
        n = t - s
        st["v"][s:t] = v[:n]
        if cell:
            st["vc"][b] = v[n:]
            st["x"][s:t] = st["x"][s:t] + dr[:n]
            st["xc"][b] = st["xc"][b] + dr[n:]
            D = st["xc"][b] / st["cell_factor"][b]
            st["lattice"][b] = st["L0"][b] @ D.T
            st["pos"][s:t] = st["x"][s:t] @ D.T
        else:
            st["pos"][s:t] = st["pos"][s:t] + dr
        st["a"][b], st["dt"][b], st["n_pos"][b] = a, dt, n_pos
        st["n_steps"][b] += 1


def fresh_state(structures, fire, cell_factor=None):
    """Starting state of ``structures`` [(lattice, cart, numbers)] and their atom_ptr."""
    sizes = [len(s[2]) for s in structures]
    B = len(sizes)
    lats = np.stack([np.asarray(s[0], dtype=np.float64) for s in structures])
    pos = np.concatenate([np.asarray(s[1], dtype=np.float64) for s in structures])
    cf = np.asarray([float(n if cell_factor is None else cell_factor) for n in sizes])
    st = dict(pos=pos.copy(), v=np.zeros_like(pos), x=pos.copy(), xc=cf[:, None, None] * np.eye(3)[None],
              vc=np.zeros((B, 3, 3)), L0=lats.copy(), lattice=lats.copy(), sigma_frame=np.zeros((B, 3, 3)),
              dt=np.full(B, fire["dt"]), a=np.full(B, fire["a_start"]), fmax=np.zeros(B), e_frame=np.zeros(B),
              cell_factor=cf, n_pos=np.zeros(B, np.int32), n_steps=np.zeros(B, np.int32),
              status=np.zeros(B, np.int32))
    return st, np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


FIRE_DEFAULTS = dict(dt=0.1, dt_max=1.0, max_move=0.2, n_min=5, f_inc=1.1, f_dec=0.5, a_start=0.1, f_a=0.99)
