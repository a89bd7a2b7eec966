"""numpy float64 restatement of one batched climbing-image NEB step (m3g_neb_step, torch_m3gnet_b200/neb.py::neb_step),
written image by image from the improved-tangent equations (DESIGN.md §8; ASE's NEB(method="improvedtangent")) and
the FIRE step of tests/fire_oracle.py applied to the band's interior rows as one structure.  Shared by the CPU and GPU
NEB tests.

State: a dict of numpy arrays with the names of neb.py::_Bands (pos, v (rows,3); dt, a, fmax (B); n_pos, n_steps,
status, i_climb (B) int32; e_frame (images)); updated in place.  Band b: interior rows row_ptr[b] .. row_ptr[b+1]
(image-major), interior images image_ptr[b] .. image_ptr[b+1], endpoint rows end_ptr[b] .. end_ptr[b+1] of ``ends``
(the initial image's atoms, then the final image's)."""
import numpy as np

from tests import fire_oracle as FO
from tests.fire_oracle import CONVERGED, FAILED, NOT_CONVERGED, RUNNING  # noqa: F401
STATE_KEYS = ("pos", "v", "dt", "a", "fmax", "n_pos", "n_steps", "status", "i_climb", "e_frame")
MAX_IMAGES = 64


def tangent(E, R, i):
    """Improved tangent t (not normalised), t+ and t- of band image i; E (M+2,), R (M+2, n, 3)."""
    tp, tm = R[i + 1] - R[i], R[i] - R[i - 1]
    El, Ei, Er = E[i - 1], E[i], E[i + 1]
    if Er > Ei > El:
        return tp.copy(), tp, tm
    if Er < Ei < El:
        return tm.copy(), tp, tm
    dmax = max(abs(Er - Ei), abs(El - Ei))
    dmin = min(abs(Er - Ei), abs(El - Ei))
    if dmax == 0.0:
        return tp + tm, tp, tm                       # flat triplet: the limit of the mixed branch
    if Er > El:
        return dmax * tp + dmin * tm, tp, tm
    return dmin * tp + dmax * tm, tp, tm


def climbing_image(E):
    """Highest interior image (band numbering 1 .. M), ties to the lowest index."""
    ic = 1
    for i in range(2, len(E) - 1):
        if E[i] > E[ic]:
            ic = i
    return ic


def neb_forces(E, R, F, k, climb):
    """(G (M, n, 3), i_climb, ok) of one band: E (M+2,), R (M+2, n, 3), F (M, n, 3) forces of the interior images.
    ok is False for a degenerate tangent (|t| zero or not finite)."""
    M = len(E) - 2
    ic = climbing_image(E)
    G = np.empty_like(F)
    ok = True
    for i in range(1, M + 1):
        t, tp, tm = tangent(E, R, i)
        tn = np.sqrt((t * t).sum())
        if not (tn > 0.0 and np.isfinite(tn)):
            ok = False
            G[i - 1] = np.nan
            continue
        th = t / tn
        f = F[i - 1]
        ft = (f * th).sum()
        if climb and i == ic:
            G[i - 1] = f - 2.0 * ft * th
        else:
            G[i - 1] = f - ft * th + k * (np.sqrt((tp * tp).sum()) - np.sqrt((tm * tm).sum())) * th
    return G, ic, ok


def neb_step(st, forces, energy, ends, e_end, k, climb, fire, fmax_target, steps, row_ptr, image_ptr, end_ptr):
    """One step for every running band."""
    forces = np.asarray(forces, dtype=np.float64)
    energy = np.asarray(energy, dtype=np.float64)
    for b in range(len(row_ptr) - 1):
        if st["status"][b] != RUNNING:
            continue
        r0, r1 = int(row_ptr[b]), int(row_ptr[b + 1])
        i0, i1 = int(image_ptr[b]), int(image_ptr[b + 1])
        e0, e1 = int(end_ptr[b]), int(end_ptr[b + 1])
        M, n = i1 - i0, (e1 - e0) // 2
        if not 1 <= M <= MAX_IMAGES:
            st["status"][b], st["fmax"][b] = FAILED, np.inf
            continue
        E = np.concatenate([[e_end[b][0]], energy[i0:i1], [e_end[b][1]]])
        R = np.concatenate([ends[e0:e0 + n][None], st["pos"][r0:r1].reshape(M, n, 3), ends[e0 + n:e1][None]])
        st["e_frame"][i0:i1] = energy[i0:i1]
        st["i_climb"][b] = climbing_image(E)
        if not np.isfinite(E).all():
            st["status"][b], st["fmax"][b] = FAILED, np.inf
            continue
        G, _, ok = neb_forces(E, R, forces[r0:r1].reshape(M, n, 3), float(k[b]), climb)
        if not ok:
            st["status"][b], st["fmax"][b] = FAILED, np.inf
            continue
        fire_rows(st, b, r0, r1, G.reshape(-1, 3), fire, fmax_target, steps)


def fire_rows(st, b, r0, r1, g, fire, fmax_target, steps):
    """tests/fire_oracle.py::fire_step's fixed-cell step of band b (rows r0 .. r1) as one structure, forces g."""
    keys = ("dt", "a", "fmax", "n_pos", "n_steps", "status")
    one = dict(pos=st["pos"][r0:r1].copy(), v=st["v"][r0:r1].copy(), e_frame=np.zeros(1),
               **{k: st[k][b:b + 1].copy() for k in keys})
    FO.fire_step(one, g, None, np.zeros(1), fire, fmax_target, steps, 0.0, np.array([0, r1 - r0]))
    st["pos"][r0:r1], st["v"][r0:r1] = one["pos"], one["v"]
    for k in keys:
        st[k][b] = one[k][0]
