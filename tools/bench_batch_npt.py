"""Batched NPT MD (BatchMD(pressure=...), kernel m3g_langevin_npt_step) against the fixed-cell run (NVT) on the same
workloads, alternating in one process.

Workloads (c1_default x3 weights, Cu 63.546 amu, Maxwell-Boltzmann start, 600 K, dt 2 fs, friction 0.01 / fs, skin
0.5 A; NPT at P0 = 0, isotropic, default compressibility 1 / (100 GPa) and barostat time 1000 fs):
  a  BASELINE.json configs[1] (C2: 256 x 108-atom Cu cells)
  b  --cells x 32-atom Cu cells
Each arm is timed --rounds times end to end, NVT and NPT alternating (medians reported), then once more each
instrumented: CUDA events around every m3g_langevin_step / m3g_langevin_npt_step call, around the calculator's compute
and around the model inside it (graph build = compute - model), and the Verlet candidate rebuilds.  The per-step
lattice read-back (pinned copy of the (B,3,3) cells and one stream synchronisation) is also timed on its own.

  python tools/bench_batch_npt.py [--steps 100] [--rounds 3] [--cells 512] [--out profiles/batch_npt_bench.json]

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
from tools.bench_batch_md import CU, DT, GAMMA, T  # noqa: E402
from tools.bench_relax import Timed, model  # noqa: E402
from tools.bench_stress import card  # noqa: E402


def run(mdl, dev, structs, steps, npt, instrument=False):
    calc = Timed(mdl, 5.0, 4.0, skin=0.5, device=dev)
    if instrument:
        calc.events = {"model": [], "compute": []}
        _lib.PROFILE = {}
    md = m3g.BatchMD(calc, structs, CU, T, friction=GAMMA, dt=DT, seed=1, pressure=0.0 if npt else None)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = md.run(steps, record_every=10)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    out = dict(wall_s=wall, iterations=md.n_iterations, rebuilds=calc.neighbor_list.n_rebuilds,
               statuses={s: sum(r["status"] == s for r in res) for s in ("completed", "failed")})
    if npt:
        out["volume_change_pct"] = float(np.mean([100 * (r["volume"][-1] / r["volume"][0] - 1) for r in res]))
        out["mean_pressure_last_frame"] = float(np.mean([r["pressure"][-1] for r in res]))
    if instrument:
        prof, _lib.PROFILE = _lib.PROFILE, None
        ms = lambda evs: [a.elapsed_time(b) for a, b in evs]  # noqa: E731
        out["step_kernel_us"] = [1e3 * x for x in ms(prof.get("langevin_npt_step" if npt else "langevin_step", []))]
        out["compute_ms"] = ms(calc.events["compute"])
        out["model_ms"] = ms(calc.events["model"])
    return out


def readback_us(dev, B, reps=500):
    """Host time of the per-step lattice read-back alone: (B,3,3) f64 device -> pinned, then one synchronisation."""
    lat = torch.randn((B, 3, 3), dtype=torch.float64, device=dev)
    pin = torch.empty((B, 3, 3), dtype=torch.float64, pin_memory=True)
    stream = torch.cuda.current_stream(dev)
    for _ in range(20):
        pin.copy_(lat, non_blocking=True)
        stream.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        pin.copy_(lat, non_blocking=True)
        stream.synchronize()
    return 1e6 * (time.perf_counter() - t0) / reps


def summary(runs, inst, atoms, steps):
    wall = statistics.median(r["wall_s"] for r in runs)
    it = runs[0]["iterations"]
    step_s = wall / it
    kern = statistics.median(inst["step_kernel_us"])
    graph = sum(inst["compute_ms"]) - sum(inst["model_ms"])
    out = dict(wall_s=[round(r["wall_s"], 4) for r in runs], wall_s_median=round(wall, 4), iterations=it,
               statuses=runs[0]["statuses"], step_ms_median=round(1e3 * step_s, 4),
               atom_steps_per_s_median=round(atoms * steps / wall), step_kernel_us_median=round(kern, 2),
               step_kernel_us_min=round(min(inst["step_kernel_us"]), 2),
               step_kernel_pct_of_step=round(100 * 1e-6 * kern / step_s, 3),
               instrumented_wall_s=round(inst["wall_s"], 4),
               graph_build_pct=round(100 * 1e-3 * graph / inst["wall_s"], 2),
               graph_build_ms_per_step=round(graph / it, 4),
               model_pct=round(100 * 1e-3 * sum(inst["model_ms"]) / inst["wall_s"], 2),
               model_ms_per_step=round(sum(inst["model_ms"]) / it, 4),
               candidate_rebuilds=[r["rebuilds"] for r in runs])
    for k in ("volume_change_pct", "mean_pressure_last_frame"):
        if k in runs[0]:
            out[k] = round(runs[0][k], 5)
    return out


def workload(mdl, dev, structs, steps, rounds):
    atoms = sum(len(s[2]) for s in structs)
    runs = {False: [], True: []}
    for _ in range(rounds):
        for npt in (False, True):
            runs[npt].append(run(mdl, dev, structs, steps, npt))
    inst = {npt: run(mdl, dev, structs, steps, npt, instrument=True) for npt in (False, True)}
    nvt, npt = summary(runs[False], inst[False], atoms, steps), summary(runs[True], inst[True], atoms, steps)
    rb = readback_us(dev, len(structs))
    return dict(structures=len(structs), atoms=atoms, steps=steps, temperature_K=T, dt_fs=DT, friction_per_fs=GAMMA,
                pressure_eV_per_A3=0.0, rounds=rounds, nvt=nvt, npt=npt,
                npt_over_nvt_step=round(npt["step_ms_median"] / nvt["step_ms_median"], 4),
                lattice_readback_us_isolated=round(rb, 2),
                lattice_readback_pct_of_npt_step=round(100 * 1e-3 * rb / npt["step_ms_median"], 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=3)
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
    for npt in (False, True):
        run(mdl, dev, c2[:32], 3, npt)  # warm-up: module loads, allocator
    res["a_c2"] = workload(mdl, dev, c2, args.steps, args.rounds)
    res["b_small_cells"] = workload(mdl, dev, small, args.steps, args.rounds)
    res["card_after"] = card()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
