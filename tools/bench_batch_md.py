"""Batched Langevin MD (BatchMD, kernel m3g_langevin_step) against sequential VelocityVerlet.

Workloads (c1_default x3 weights, Cu 63.546 amu, Maxwell-Boltzmann start):
  a  BASELINE.json configs[1] (C2: 256 x 108-atom Cu cells) at 600 K, dt 2 fs, friction 0.01 / fs, --steps steps
  b  --cells x 32-atom Cu cells, same conditions; baseline: VelocityVerlet on one 32-atom cell
Each is timed --repeats times end to end (median reported), then once more instrumented: CUDA events around every
m3g_langevin_step call, around the calculator's compute and around the model inside it (graph build = compute -
model), and the Verlet candidate rebuilds per step (one atom anywhere in the batch crossing skin / 2 rebuilds the
whole batch's candidates).

  python tools/bench_batch_md.py [--steps 100] [--repeats 3] [--cells 512] [--out profiles/batch_md_bench.json]

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

CU = {29: 63.546}
T, DT, GAMMA = 600.0, 2.0, 0.01


def langevin_bytes(n_atoms: int, n_structures: int) -> int:
    """Algorithmic bytes of one advancing m3g_langevin_step: forces read (12 B / atom), velocities read and written
    (48), positions read and written (48), inverse masses read (8); per structure c1, c2, kT, stream id, step, status
    and energy read (48), bath read and written (16), step written (4) and one observable row written (32)."""
    return (12 + 48 + 48 + 8) * n_atoms + (48 + 16 + 4 + 32) * n_structures


def batch_run(mdl, dev, structs, steps, instrument=False):
    calc = Timed(mdl, 5.0, 4.0, skin=0.5, device=dev)
    if instrument:
        calc.events = {"model": [], "compute": []}
        _lib.PROFILE = {}
    md = m3g.BatchMD(calc, structs, CU, T, friction=GAMMA, dt=DT, seed=1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = md.run(steps, record_every=10)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    out = dict(wall_s=wall, iterations=md.n_iterations, rebuilds=calc.neighbor_list.n_rebuilds,
               statuses={s: sum(r["status"] == s for r in res) for s in ("completed", "failed")},
               mean_temperature_last=float(np.mean([r["temperature"][-1] for r in res])))
    if instrument:
        prof, _lib.PROFILE = _lib.PROFILE, None
        ms = lambda evs: [a.elapsed_time(b) for a, b in evs]  # noqa: E731
        out["langevin_us"] = [1e3 * x for x in ms(prof.get("langevin_step", []))]
        out["compute_ms"] = ms(calc.events["compute"])
        out["model_ms"] = ms(calc.events["model"])
    return out


def workload(mdl, dev, structs, steps, repeats):
    runs = [batch_run(mdl, dev, structs, steps) for _ in range(repeats)]
    inst = batch_run(mdl, dev, structs, steps, instrument=True)
    wall = statistics.median(r["wall_s"] for r in runs)
    atoms = sum(len(s[2]) for s in structs)
    it = runs[0]["iterations"]
    step_s = wall / it
    lang = statistics.median(inst["langevin_us"])
    graph = sum(inst["compute_ms"]) - sum(inst["model_ms"])
    b = langevin_bytes(atoms, len(structs))
    return dict(
        structures=len(structs), atoms=atoms, steps=steps, temperature_K=T, dt_fs=DT, friction_per_fs=GAMMA,
        repeats=repeats, wall_s=[round(r["wall_s"], 4) for r in runs], wall_s_median=round(wall, 4),
        iterations=it, statuses=runs[0]["statuses"], step_ms_median=round(1e3 * step_s, 4),
        atom_steps_per_s_median=round(atoms * steps / wall), langevin_call_us_median=round(lang, 2),
        langevin_call_us_min=round(min(inst["langevin_us"]), 2),
        langevin_call_pct_of_step=round(100 * 1e-6 * lang / step_s, 3),
        langevin_bytes_per_step=b, langevin_hbm_bound_us=round(1e6 * b / HBM_BYTES_PER_S, 2),
        instrumented_wall_s=round(inst["wall_s"], 4),
        graph_build_pct=round(100 * 1e-3 * graph / inst["wall_s"], 2),
        model_pct=round(100 * 1e-3 * sum(inst["model_ms"]) / inst["wall_s"], 2),
        candidate_rebuilds=[r["rebuilds"] for r in runs],
        candidate_rebuilds_per_step=round(statistics.median(r["rebuilds"] for r in runs) / it, 4),
        mean_temperature_last_frame_K=round(runs[0]["mean_temperature_last"], 1))


def sequential_verlet(mdl, dev, steps, warmup=5):
    lat, cart, z = synthetic.fcc_cu_supercell(2, 0.05, 0)
    calc = m3g.M3GNetCalculator(mdl, 5.0, 4.0, skin=0.5, device=dev)
    sigma = np.sqrt(8.617333262e-5 * T * m3g.calculator.ACC_UNIT / CU[29])
    v0 = np.random.default_rng(0).normal(0.0, sigma, size=cart.shape)
    md = m3g.VelocityVerlet(calc, lat, cart, z, np.full(len(z), CU[29]), dt=DT, velocities=v0 - v0.mean(axis=0))
    md.step(warmup)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    md.step(steps)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return dict(atoms=len(z), steps=steps, wall_s=round(wall, 4), step_ms=round(1e3 * wall / steps, 4),
                atom_steps_per_s=round(len(z) * steps / wall))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--cells", type=int, default=512)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    m3g.calculator.stabilise_allocator()
    mdl = model(dev)
    res = {"card": card(), "torch": torch.__version__}
    lat, cart, z, sizes = synthetic.config2_batch(256)
    ptr = np.concatenate([[0], np.cumsum(sizes)])
    c2 = [(lat[b], cart[ptr[b]:ptr[b + 1]], z[ptr[b]:ptr[b + 1]]) for b in range(len(sizes))]
    small = [synthetic.fcc_cu_supercell(2, 0.05, s) for s in range(args.cells)]
    batch_run(mdl, dev, c2[:32], 3)  # warm-up: module loads, allocator
    res["a_c2_langevin"] = workload(mdl, dev, c2, args.steps, args.repeats)
    res["b_small_cells_langevin"] = workload(mdl, dev, small, args.steps, args.repeats)
    res["b_sequential_velocity_verlet_32_atoms"] = sequential_verlet(mdl, dev, args.steps)
    res["b_speedup_atom_steps"] = round(res["b_small_cells_langevin"]["atom_steps_per_s_median"]
                                        / res["b_sequential_velocity_verlet_32_atoms"]["atom_steps_per_s"], 1)
    res["card_after"] = card()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
