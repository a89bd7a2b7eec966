"""Batched climbing-image NEB (BatchNEB, kernel m3g_neb_step) against BatchFire on the same interior images.

Workloads (c1_default x3 weights; Cu vacancy hops, synthetic.fcc_cu_vacancy_hop with per-band jitter, endpoints
relaxed with BatchFire before timing, 5 interior images, climb on, k = 0.1 eV/A^2):
  a  --bands-a bands in 3x3x3 cells (107 atoms; 52 bands = 27 820 moving atoms, about C2's size)
  b  --bands-b bands in 2x2x2 cells (31 atoms)
Each runs --steps steps at fmax 0 (every band runs every step), --repeats times, alternating in this process with
BatchFire on the same interior images (the same ragged compute layout, one FIRE state per image), so the NEB overhead
is the difference.  Then once more instrumented: CUDA events around every m3g_neb_step call, around the calculator's
compute and around the model inside it (graph build = compute - model).  Timings cover run() end to end, including
the one endpoint evaluation.

  python tools/bench_neb.py [--steps 50] [--repeats 3] [--bands-a 52] [--bands-b 180] [--out profiles/neb_bench.json]

Prints one JSON object (card name and power limit read in the same run) and writes it to --out when given.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch_m3gnet_b200 as m3g  # noqa: E402
from torch_m3gnet_b200 import _lib, synthetic  # noqa: E402
from tools.bench_relax import HBM_BYTES_PER_S, Timed, model  # noqa: E402
from tools.bench_stress import card  # noqa: E402

M_IMAGES = 5


def neb_bytes(n_rows: int, n_images: int, n_bands: int, n_end_rows: int) -> int:
    """Algorithmic bytes of one advancing m3g_neb_step: per interior row forces read (12 B), positions read and written
    (48), velocities read and written (48); endpoint positions read (24 per endpoint row); per image its energy read
    and e_frame written (12); per band the FIRE scalars, status and step count (40), k and the endpoint energies (24),
    fmax and i_climb written (12) and the three offsets (12)."""
    return (12 + 48 + 48) * n_rows + 24 * n_end_rows + 12 * n_images + (40 + 24 + 12 + 12) * n_bands


def hop_bands(mdl, dev, reps, count):
    """``count`` (initial, final) pairs with relaxed endpoints (BatchFire, untimed)."""
    pairs = []
    for s in range(count):
        (lat, c0, z), (_, c1, _) = synthetic.fcc_cu_vacancy_hop(reps)
        jit = np.random.default_rng(s).uniform(-0.03, 0.03, c0.shape)
        pairs += [(lat, c0 + jit, z), (lat, c1 + jit, z)]
    calc = m3g.M3GNetCalculator(mdl, 5.0, 4.0, skin=0.5, device=dev)
    res = m3g.BatchFire(calc, pairs).run(fmax=0.05, steps=300)
    ends = [(r["lattice"], r["positions"], p[2]) for r, p in zip(res, pairs)]
    return [(ends[2 * i], ends[2 * i + 1]) for i in range(count)], [r["status"] for r in res]


def run(mdl, dev, kind, bands, images, steps, instrument=False):
    calc = Timed(mdl, 5.0, 4.0, skin=0.5, device=dev)
    if instrument:
        calc.events = {"model": [], "compute": []}
        _lib.PROFILE = {}
    if kind == "neb":
        opt = m3g.BatchNEB(calc, bands, n_images=M_IMAGES, climb=True)
    else:
        opt = m3g.BatchFire(calc, images)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = opt.run(fmax=0.0, steps=steps)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    out = dict(wall_s=wall, iterations=opt.n_iterations, rebuilds=calc.neighbor_list.n_rebuilds,
               statuses={s: sum(r["status"] == s for r in res) for s in ("converged", "not converged", "failed")})
    if kind == "neb":
        out["endpoint_calls"] = opt.n_endpoint_calls
        out["fmax_last_median"] = float(np.median([r["fmax"] for r in res]))
        out["barrier_forward_median_eV"] = float(np.median([r["barrier_forward"] for r in res]))
    if instrument:
        prof, _lib.PROFILE = _lib.PROFILE, None
        ms = lambda evs: [a.elapsed_time(b) for a, b in evs]  # noqa: E731
        out["kernel_us"] = [1e3 * x for x in ms(prof.get("neb_step" if kind == "neb" else "fire_step", []))]
        out["compute_ms"] = ms(calc.events["compute"])
        out["model_ms"] = ms(calc.events["model"])
    return out


def summary(runs, inst, moving_atoms, steps, kernel):
    wall = statistics.median(r["wall_s"] for r in runs)
    it = runs[0]["iterations"]
    step_s = wall / it
    k_us = statistics.median(inst["kernel_us"])
    graph = sum(inst["compute_ms"]) - sum(inst["model_ms"])
    return {"wall_s": [round(r["wall_s"], 4) for r in runs], "wall_s_median": round(wall, 4), "iterations": it,
            "statuses": runs[0]["statuses"], "step_ms_median": round(1e3 * step_s, 4),
            "moving_atom_steps_per_s_median": round(moving_atoms * steps / wall),
            f"{kernel}_call_us_median": round(k_us, 2), f"{kernel}_call_us_min": round(min(inst["kernel_us"]), 2),
            f"{kernel}_call_pct_of_step": round(100 * 1e-6 * k_us / step_s, 3),
            "instrumented_wall_s": round(inst["wall_s"], 4),
            "graph_build_pct": round(100 * 1e-3 * graph / inst["wall_s"], 2),
            "model_pct": round(100 * 1e-3 * sum(inst["model_ms"]) / inst["wall_s"], 2),
            "candidate_rebuilds": [r["rebuilds"] for r in runs],
            "candidate_rebuilds_per_step": round(statistics.median(r["rebuilds"] for r in runs) / it, 4)}


def workload(mdl, dev, reps, count, steps, repeats):
    from torch_m3gnet_b200.neb import interpolate

    pairs, relax_status = hop_bands(mdl, dev, reps, count)
    images = [im for a, b in pairs for im in interpolate(a, b, M_IMAGES)[1:-1]]
    n = len(pairs[0][0][2])
    moving = len(images) * n
    runs = {"neb": [], "fire": []}
    for _ in range(repeats):  # alternating
        for kind in ("neb", "fire"):
            runs[kind].append(run(mdl, dev, kind, pairs, images, steps))
    inst = {kind: run(mdl, dev, kind, pairs, images, steps, instrument=True) for kind in ("neb", "fire")}
    neb = summary(runs["neb"], inst["neb"], moving, steps, "neb_step")
    neb.update(endpoint_calls=runs["neb"][0]["endpoint_calls"],
               fmax_last_median=round(runs["neb"][0]["fmax_last_median"], 4),
               barrier_forward_median_eV_random_weights=round(runs["neb"][0]["barrier_forward_median_eV"], 4))
    fire = summary(runs["fire"], inst["fire"], moving, steps, "fire_step")
    b = neb_bytes(moving, len(images), count, 2 * n * count)
    return dict(bands=count, atoms_per_image=n, interior_images=M_IMAGES, moving_atoms=moving, steps=steps,
                repeats=repeats, endpoint_relax_statuses={s: relax_status.count(s) for s in set(relax_status)},
                neb=neb, batch_fire_same_images=fire,
                neb_over_fire_step_time=round(neb["step_ms_median"] / fire["step_ms_median"], 4),
                neb_step_bytes=b, neb_step_hbm_bound_us=round(1e6 * b / HBM_BYTES_PER_S, 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--bands-a", type=int, default=52)
    ap.add_argument("--bands-b", type=int, default=180)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    m3g.calculator.stabilise_allocator()
    mdl = model(dev)
    res = {"card": card(), "torch": torch.__version__}
    warm, _ = hop_bands(mdl, dev, 2, 4)  # warm-up: module loads, allocator
    run(mdl, dev, "neb", warm, None, 3)
    res["a_107_atom_cells"] = workload(mdl, dev, 3, args.bands_a, args.steps, args.repeats)
    res["b_31_atom_cells"] = workload(mdl, dev, 2, args.bands_b, args.steps, args.repeats)
    res["card_after"] = card()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
