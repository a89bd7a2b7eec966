"""Batched phonons (BatchPhonon; kernels m3g_phonon_force_constants / _frequencies / _thermal / _dynmat).

Workloads (c1_default x3 weights):
  a  force phase: --structures conventional fcc Cu cells (4 atoms; lattice constants 3.615 A + 0.1 % spread) in 3x3x3
     supercells: 25 evaluations x 108 atoms each (64 cells: 172 800 atoms), max_atoms 30 000.  run() end to end, its
     atom-evaluations/s against the C2 batch (synthetic.config2_batch, bench.py's flagship) through the same calculator
     in this process; then an instrumented run for the shares (CUDA events around the calculator's compute and the
     model inside it, graph build = compute - model, the FC launch) and the host minimum-image table; and a sampled
     sequential loop of one supercell per compute call.
  b  mesh phase: the same structures on a 20^3 mesh (512 000 matrices of 12 x 12): m3g_phonon_frequencies, then
     m3g_phonon_thermal (101 temperatures), and as a comparison arm m3g_phonon_dynmat + torch.linalg.eigvalsh
     (cuSOLVER) on the same D matrices, alternating with the kernel.
  c  larger cells: --structures-c 16-atom cells (2x2x1 conventional Cu, 3n = 48) in 2x2x3 supercells on a 12^3 mesh.
Times are CUDA events (kernels) or host clocks around synchronised work (run()), medians of --repeats rounds.

  python tools/bench_phonon.py [--repeats 3] [--structures 64] [--structures-c 8] [--out profiles/phonon_bench.json]

Prints one JSON object (card name and power limit read in the same run) and writes it to --out when given.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch_m3gnet_b200 as m3g  # noqa: E402
from torch_m3gnet_b200 import _lib, phonon, synthetic  # noqa: E402
from tools.bench_relax import Timed, model  # noqa: E402
from tools.bench_stress import card  # noqa: E402

MASS = {29: 63.546}
TEMPS = np.arange(0, 1001, 10)
CUSOLVER_CHUNK = 4096


def cu_cells(count, reps=(1, 1, 1)):
    out = []
    for s in range(count):
        lat, cart, z = synthetic.fcc_cu_supercell(1, 0.0, 0)
        f = 1.0 + 0.001 * s / max(count - 1, 1)
        lat, cart = lat * f, cart * f
        if reps != (1, 1, 1):
            S, cart = phonon.supercell(lat, cart, reps)
            lat, z = S, np.tile(z, int(np.prod(reps)))
        out.append((lat, cart, z))
    return out


def events_ms(fn, n=1):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, out


def jacobi_flops(dim: int, sweeps: np.ndarray) -> float:
    """FP64 operations of the Jacobi phase from shapes and sweep counts: per sweep dim - 1 rounds of dim/2 rotations,
    each updating two rows and two columns (about 20 flops per updated entry pair: the phase multiply, 6, and two
    real-weighted combinations, 4 x 2 plus 6 for the other side) -> 20 dim (dim - 1) dim / 2 x 2; plus the
    off-diagonal norm (4 dim^2) per check, one more check than sweeps."""
    m = dim + (dim & 1)
    per_sweep = 20.0 * m * (m - 1) * dim
    return float(per_sweep * sweeps.sum() + 4.0 * dim * dim * (sweeps + 1).sum())


def dynmat_flops(pairs: int, images: int, Q: int) -> float:
    """FP64 operations of building D from shapes: each of the 9 components of every (k, j) pair goes over its images
    (phase argument 6, two accumulations 2; one sincospi each, counted separately) and is weighted into D (image
    weight 2, two FMAs 4): 9 (8 images + 6 pairs) per q-point."""
    return float(Q) * 9 * (8 * images + 6 * pairs)


def force_phase(mdl, dev, structs, reps, repeats):
    n_atoms = sum((6 * len(s[2]) + 1) * len(s[2]) * int(np.prod(reps)) for s in structs)
    walls = []
    for _ in range(repeats):
        calc = Timed(mdl, 5.0, 4.0, skin=0.5, device=dev)
        ph = m3g.BatchPhonon(calc, structs, reps, MASS, max_atoms=30000)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        recs = ph.run()
        torch.cuda.synchronize()
        walls.append(time.perf_counter() - t0)
    calc = Timed(mdl, 5.0, 4.0, skin=0.5, device=dev)
    calc.events = {"model": [], "compute": []}
    _lib.PROFILE = {}
    ph = m3g.BatchPhonon(calc, structs, reps, MASS, max_atoms=30000)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    recs = ph.run()
    torch.cuda.synchronize()
    inst_wall = time.perf_counter() - t0
    prof, _lib.PROFILE = _lib.PROFILE, None
    ms = lambda evs: sum(a.elapsed_time(b) for a, b in evs)  # noqa: E731
    compute_ms, model_ms = ms(calc.events["compute"]), ms(calc.events["model"])
    fc_ms = ms(prof["phonon_force_constants"])
    wall = statistics.median(walls)
    return ph, recs, dict(
        structures=len(structs), supercell=list(reps), evaluations=sum(6 * len(s[2]) + 1 for s in structs),
        atom_evaluations=n_atoms, compute_calls=ph.n_compute_calls, run_wall_s=[round(w, 4) for w in walls],
        run_wall_s_median=round(wall, 4), atom_evaluations_per_s=round(n_atoms / wall),
        instrumented_wall_s=round(inst_wall, 4),
        graph_build_pct=round(100 * 1e-3 * (compute_ms - model_ms) / inst_wall, 2),
        model_pct=round(100 * 1e-3 * model_ms / inst_wall, 2),
        fc_kernel_ms=round(fc_ms, 4), fc_kernel_pct=round(100 * 1e-3 * fc_ms / inst_wall, 3),
        minimum_image_table_s=round(ph.minimum_image_seconds, 4),
        minimum_image_table_pct=round(100 * ph.minimum_image_seconds / inst_wall, 2),
        max_residual_force_eV_per_A=max(r["max_residual_force"] for r in recs),
        statuses={s: sum(r["status"] == s for r in recs) for s in ("ok", "failed")})


def c2_rate(mdl, dev, repeats):
    lat, cart, z, sizes = synthetic.config2_batch()
    calc = m3g.M3GNetCalculator(mdl, 5.0, 4.0, skin=0.5, device=dev)
    calc.compute(lat, cart, z, sizes)
    ts = []
    for _ in range(max(repeats, 5)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        calc.compute(lat, cart + 1e-4 * len(ts), z, sizes)   # a new frame each call (no replay of an identical one)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    t = statistics.median(ts)
    return dict(atoms=int(sum(sizes)), compute_ms_median=round(1e3 * t, 3),
                atom_evaluations_per_s=round(sum(sizes) / t))


def sequential(mdl, dev, ph, samples):
    """One supercell per compute call on a fresh calculator, ``samples`` calls (after 3 warm-up calls)."""
    calc = m3g.M3GNetCalculator(mdl, 5.0, 4.0, skin=0.5, device=dev)
    per = 6 * len(ph.structures[0][2])
    cells = [ph._supercell(i % ph.B, 1 + i % per) for i in range(samples + 3)]
    ts = []
    for i, (S, pos, z) in enumerate(cells):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        calc.compute(S[None], pos, z, [len(z)])
        torch.cuda.synchronize()
        if i >= 3:
            ts.append(time.perf_counter() - t0)
    t = statistics.median(ts)
    total = sum(6 * len(s[2]) + 1 for s in ph.structures)
    return dict(samples=samples, call_ms_median=round(1e3 * t, 4), extrapolated_s=round(t * total, 3),
                atom_evaluations_per_s=round(len(cells[0][2]) / t))


def mesh_phase(ph, mesh, repeats, cusolver=True):
    q = phonon.mesh_qpoints(mesh)
    qs = [q] * ph.B
    ph._frequencies(qs)                                      # warm-up
    runs = []
    for _ in range(repeats):
        t, (out, q_ptr, f_ptr) = events_ms(lambda: ph._frequencies(qs))
        runs.append(t)
    sweeps = out.sweeps.cpu().numpy()
    st = ph._st
    n = st.n[0]
    dim = 3 * n
    Q = len(q) * ph.B
    pairs = int(st.pair_ptr[1].item())
    images = int(st.sv_ptr[pairs].item())
    th_ms = []
    temps = torch.as_tensor(TEMPS.astype(np.float64)).to(ph.device)
    th = types.SimpleNamespace(values=torch.empty((ph.B, len(TEMPS), 4), dtype=torch.float64, device=ph.device),
                               n_imag=torch.empty(ph.B, dtype=torch.int32, device=ph.device),
                               fmin=torch.empty(ph.B, dtype=torch.float64, device=ph.device))
    for _ in range(repeats):
        t, _ = events_ms(lambda: phonon.thermal_launch(st, out.freq, f_ptr, q_ptr, temps, 0.01, th))
        th_ms.append(t)
    k_ms = statistics.median(runs)
    fl_jac = jacobi_flops(dim, sweeps)
    fl_dyn = dynmat_flops(pairs, images, Q)
    res = dict(mesh=list(mesh), q_points=Q, dim=dim, frequencies_kernel_ms=[round(x, 3) for x in runs],
               frequencies_kernel_ms_median=round(k_ms, 3), q_points_per_s=round(Q / (1e-3 * k_ms)),
               sweeps_min=int(sweeps.min()), sweeps_median=float(np.median(sweeps)), sweeps_max=int(sweeps.max()),
               jacobi_fp64_ops=fl_jac, dynmat_fp64_ops=fl_dyn, sincospi_calls=float(Q) * 9 * images,
               fp64_tflops_achieved=round((fl_jac + fl_dyn) / (1e-3 * k_ms) / 1e12, 3),
               thermal_kernel_ms_median=round(statistics.median(th_ms), 4), temperatures=len(TEMPS),
               n_imaginary=th.n_imag.cpu().tolist()[:4], failed_q_points=int(out.q_status.sum().item()))
    if cusolver:
        try:
            res.update(cusolver_arm(ph, qs, q_ptr, dim, Q, repeats))
        except RuntimeError as e:                           # reported, not hidden: the arm is a comparison only
            res["cusolver_error"] = str(e)[:300]
    return res


def cusolver_arm(ph, qs, q_ptr, dim, Q, repeats):
    """The same matrices through m3g_phonon_dynmat, the Hermitian part (D + D^H) / 2 (what the kernel diagonalises;
    eigvalsh alone would read one triangle of D, which the float32 noise in the constants leaves slightly
    non-Hermitian) and torch.linalg.eigvalsh (cuSOLVER), alternating with the kernel.
    cuSOLVER's batched solver refused the whole 512 000-matrix batch (CUSOLVER_STATUS_INVALID_VALUE from its
    buffer-size query), so it runs in chunks of CUSOLVER_CHUNK matrices."""
    st = ph._st
    q_d = torch.as_tensor(np.concatenate(qs)).to(ph.device)

    def eigvalsh(D):
        return torch.cat([torch.linalg.eigvalsh(D[i:i + CUSOLVER_CHUNK]) for i in range(0, D.shape[0], CUSOLVER_CHUNK)])

    def hermitian_dynmat():
        D = phonon.dynmat_launch(st, q_d, q_ptr, dim)
        return 0.5 * (D + D.mH)

    eigvalsh(hermitian_dynmat())                            # warm-up (algorithm selection)
    dyn_ms, eig_ms, k2 = [], [], []
    for _ in range(repeats):
        t, D = events_ms(hermitian_dynmat)
        dyn_ms.append(t)
        t, lam = events_ms(lambda: eigvalsh(D))
        eig_ms.append(t)
        t, (out, _, _) = events_ms(lambda: ph._frequencies(qs))
        k2.append(t)
    ref = lam.cpu().numpy().reshape(Q, dim)
    got = out.eig.cpu().numpy().reshape(Q, dim)
    fro = torch.linalg.matrix_norm(D).cpu().numpy()
    pick = np.random.default_rng(0).choice(Q, size=min(Q, 256), replace=False)  # numpy.linalg.eigvalsh as the judge
    npy = np.linalg.eigvalsh(D[torch.as_tensor(pick).to(D.device)].cpu().numpy())
    dev_of = lambda x: float((np.abs(x[pick] - npy).max(axis=1) / fro[pick]).max())  # noqa: E731
    dyn, eig = statistics.median(dyn_ms), statistics.median(eig_ms)
    return dict(cusolver_chunk=CUSOLVER_CHUNK, cusolver_dynmat_and_hermitian_part_ms_median=round(dyn, 3),
                cusolver_eigvalsh_ms_median=round(eig, 3), cusolver_total_ms_median=round(dyn + eig, 3),
                kernel_ms_alternating_median=round(statistics.median(k2), 3),
                max_abs_dlambda_over_fro_kernel_vs_cusolver=float((np.abs(got - ref).max(axis=1) / fro).max()),
                sample_max_abs_dlambda_over_fro_kernel_vs_numpy=dev_of(got),
                sample_max_abs_dlambda_over_fro_cusolver_vs_numpy=dev_of(ref))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--structures", type=int, default=64)
    ap.add_argument("--structures-c", type=int, default=8)
    ap.add_argument("--sequential-samples", type=int, default=60)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    m3g.calculator.stabilise_allocator()
    mdl = model(dev)
    res = {"card": card(), "torch": torch.__version__}
    warm = m3g.BatchPhonon(m3g.M3GNetCalculator(mdl, 5.0, 4.0, skin=0.5, device=dev), cu_cells(2), (3, 3, 3), MASS)
    warm.run()
    warm.thermal_properties(mesh=(4, 4, 4))
    structs = cu_cells(args.structures)
    ph, recs, a = force_phase(mdl, dev, structs, (3, 3, 3), args.repeats)
    a["c2"] = c2_rate(mdl, dev, args.repeats)
    a["batched_over_c2_rate"] = round(a["atom_evaluations_per_s"] / a["c2"]["atom_evaluations_per_s"], 4)
    a["sequential_one_supercell_per_call"] = sequential(mdl, dev, ph, args.sequential_samples)
    a["speedup_over_sequential"] = round(a["sequential_one_supercell_per_call"]["extrapolated_s"]
                                         / a["run_wall_s_median"], 2)
    res["a_force_phase"] = a
    res["b_mesh_phase"] = mesh_phase(ph, (20, 20, 20), args.repeats)
    tp = ph.thermal_properties(mesh=(20, 20, 20), temperatures=[300.0])
    res["b_mesh_phase"]["first_structure_300K"] = {k: float(tp[0][k][0]) for k in
                                                   ("free_energy", "entropy", "heat_capacity", "energy")}
    res["b_mesh_phase"]["first_structure_min_frequency_THz"] = tp[0]["min_frequency"]
    big = cu_cells(args.structures_c, reps=(2, 2, 1))
    ph_c, _, c = force_phase(mdl, dev, big, (2, 2, 3), 1)
    c["mesh"] = mesh_phase(ph_c, (12, 12, 12), args.repeats)
    res["c_16_atom_cells"] = c
    res["card_after"] = card()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
