"""numpy float64 restatement of the batched phonon kernels (csrc/phonon.cu): finite-difference force constants and their
symmetrisation, the dynamical matrix D(q), the eigenvalues of its Hermitian part (numpy.linalg.eigvalsh in place of the
Jacobi method) and the harmonic thermal sums -- per structure, and as drop-in replacements for phonon.py's launches."""
import numpy as np
import torch

from torch_m3gnet_b200.phonon import FAILED, H_THZ, KB, OK, THZ

MAX_ATOMS = 32


def neg_cells(reps):
    """index of -l (wrapped) for every cell l, lexicographic."""
    r1, r2, r3 = (int(r) for r in reps)
    i = np.stack(np.meshgrid(np.arange(r1), np.arange(r2), np.arange(r3), indexing="ij"), -1).reshape(-1, 3)
    m = (-i) % np.array([r1, r2, r3])
    return (m[:, 0] * r2 + m[:, 1]) * r3 + m[:, 2]


def force_constants(forces, n, reps, h, symmetrize):
    """(fc (n, N, 3, 3), status, residual) of one structure from its ((6n+1) N, 3) forces (float32 values)."""
    F = np.asarray(forces, dtype=np.float64)
    L = int(np.prod(reps))
    N = n * L
    F = F.reshape(6 * n + 1, N, 3)
    if not np.isfinite(F).all():
        return np.full((n, N, 3, 3), np.nan), FAILED, np.nan
    residual = float(np.sqrt((F[0] ** 2).sum(axis=1)).max())
    X = F[1:].reshape(n, 3, 2, N, 3)                         # (k, alpha, +/-, j, beta)
    phi = (-(X[:, :, 0] - X[:, :, 1]) * (1.0 / (2.0 * h))).transpose(0, 2, 1, 3)
    phi = phi.reshape(n, L, n, 3, 3)                         # (k, l, k', alpha, beta)
    neg = neg_cells(reps)
    for _ in range(symmetrize):
        phi = 0.5 * (phi + phi.transpose(2, 1, 0, 4, 3)[:, neg])
        rows = phi.sum(axis=(1, 2))
        for k in range(n):
            phi[k, 0, k] -= rows[k]
    return phi.reshape(n, N, 3, 3), OK, residual


def dynmat(fc, sv_ptr, sv, mass, reps, q):
    """(3n, 3n) complex D(q) of one structure (fc (n, N, 3, 3), its minimum-image CSR table, masses (n,))."""
    n, N = fc.shape[:2]
    L = N // n
    ph = np.exp(2j * np.pi * (sv @ np.asarray(q, dtype=np.float64)))
    counts = np.diff(sv_ptr)
    mean = np.add.reduceat(ph, sv_ptr[:-1]) / counts       # every pair has at least one image
    D = np.einsum("klmab,klm->kamb", fc.reshape(n, L, n, 3, 3), mean.reshape(n, L, n))
    D = D / np.sqrt(np.outer(mass, mass))[:, None, :, None]
    return D.reshape(3 * n, 3 * n)


def eigenvalues(D):
    """Ascending eigenvalues of the Hermitian part of D."""
    return np.linalg.eigvalsh(0.5 * (D + D.conj().T))


def to_thz(lam):
    return np.sign(lam) * np.sqrt(np.abs(lam)) * THZ


def thermal(freq, temps, cutoff):
    """(values (T, 4): F, S, Cv, E per unit cell, n_imag, fmin) from all mesh frequencies (Q, 3n) of one structure."""
    f = np.asarray(freq, dtype=np.float64)
    nq = f.shape[0]
    f = f.reshape(-1)
    keep = ~(f < cutoff)
    e = H_THZ * f[keep]
    out = np.empty((len(temps), 4))
    for i, T in enumerate(temps):
        kT = KB * T
        if kT > 0:
            x = e / kT
            em = np.exp(-x)
            lg = np.log1p(-em)
            out[i] = [(0.5 * e + kT * lg).sum(), (KB * (x / np.expm1(x) - lg)).sum(),
                      (KB * x * x * em / np.expm1(-x) ** 2).sum(), (e * (0.5 + 1.0 / np.expm1(x))).sum()]
        else:
            out[i] = [0.5 * e.sum(), 0.0, 0.0, 0.5 * e.sum()]
    fmin = np.nan if np.isnan(f).any() else float(f.min())
    return out / nq, int((f < -cutoff).sum()), fmin


# ---------------------------------------------------------------------------------------------------------------------
# phonon.py's launches, restated (CPU tensors in, CPU tensors written)
# ---------------------------------------------------------------------------------------------------------------------

def _np(t):
    return t.detach().cpu().numpy()


def fc_launch(forces, st, h, symmetrize):
    F = _np(forces).astype(np.float64)
    row_ptr, pair_ptr, reps = _np(st.row_ptr), _np(st.pair_ptr), _np(st.reps)
    fc = _np(st.fc).copy()
    status = np.empty(st.B, np.int32)
    residual = np.empty(st.B)
    for b in range(st.B):
        phi, status[b], residual[b] = force_constants(F[row_ptr[b]:row_ptr[b + 1]], st.n[b], reps[b], h, symmetrize)
        fc[pair_ptr[b]:pair_ptr[b + 1]] = phi.reshape(-1, 3, 3)
    st.fc.copy_(torch.from_numpy(fc))
    st.status.copy_(torch.from_numpy(status))
    st.residual.copy_(torch.from_numpy(residual))


def structure_dynmat(st, b, q):
    pair_ptr, sv_ptr_all = _np(st.pair_ptr), _np(st.sv_ptr)
    atom_ptr = _np(st.atom_ptr)
    p0, p1 = pair_ptr[b], pair_ptr[b + 1]
    sv_ptr = sv_ptr_all[p0:p1 + 1]
    sv = _np(st.sv)[sv_ptr[0]:sv_ptr[-1]]
    fc = _np(st.fc)[p0:p1].reshape(st.n[b], st.N[b], 3, 3)
    return dynmat(fc, sv_ptr - sv_ptr[0], sv, _np(st.mass)[atom_ptr[b]:atom_ptr[b + 1]], _np(st.reps)[b], q)


def frequencies_launch(st, q, q_ptr, f_ptr, out):
    qs, q_ptr, f_ptr = _np(q), _np(q_ptr), _np(f_ptr)
    status = _np(st.status)
    eig = np.empty(out.eig.shape[0])
    for b in range(st.B):
        for i in range(q_ptr[b], q_ptr[b + 1]):
            o = f_ptr[b] + (i - q_ptr[b]) * 3 * st.n[b]
            eig[o:o + 3 * st.n[b]] = (np.nan if status[b] != OK else eigenvalues(structure_dynmat(st, b, qs[i])))
    fail = np.array([status[np.searchsorted(q_ptr, i, side="right") - 1] != OK for i in range(qs.shape[0])])
    out.eig.copy_(torch.from_numpy(eig))
    out.freq.copy_(torch.from_numpy(to_thz(eig)))
    out.sweeps.zero_()
    out.q_status.copy_(torch.from_numpy(fail.astype(np.int32)))


def thermal_launch(st, freq, f_ptr, q_ptr, temps, cutoff, out):
    f, f_ptr, q_ptr, T = _np(freq), _np(f_ptr), _np(q_ptr), _np(temps)
    status = _np(st.status)
    values = np.full((st.B, len(T), 4), np.nan)
    n_imag = np.full(st.B, -1, np.int32)
    fmin = np.full(st.B, np.nan)
    for b in range(st.B):
        if status[b] != OK:
            continue
        fb = f[f_ptr[b]:f_ptr[b + 1]].reshape(q_ptr[b + 1] - q_ptr[b], -1)
        values[b], n_imag[b], fmin[b] = thermal(fb, T, cutoff)
    out.values.copy_(torch.from_numpy(values))
    out.n_imag.copy_(torch.from_numpy(n_imag))
    out.fmin.copy_(torch.from_numpy(fmin))
