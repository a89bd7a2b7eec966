"""Batched FIRE relaxation (BatchFire, kernel m3g_fire_step) against sequential Fire runs.

Workloads (c1_default x3 weights):
  a  BASELINE.json configs[1] (C2: 256 x 108-atom Cu cells), fixed cell, --steps steps with fmax = 0 (nothing leaves)
  b  the same with relax_cell=True (every step changes the cells and rebuilds the neighbour candidates)
  c  --structures synthetic.mpf_like_structure cells relaxed to fmax 0.05 (at most 200 steps) under a
     --max-atoms working-set budget
Each is timed --repeats times end to end (median reported), then once more instrumented: CUDA events around every
m3g_fire_step call, around the calculator's compute and around the model inside it (graph build = compute - model),
and BatchFire's host clock around regroups.  The baseline is sequential Fire on a sample of the same structures.

  python tools/bench_relax.py [--steps 50] [--repeats 3] [--structures 1000] [--max-atoms 30000]
                              [--out profiles/relax_bench.json]

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
from torch_m3gnet_b200.relax import admit  # noqa: E402
from tools.bench_stress import card  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # B200 data sheet (one GPU of an HGX B200)


def fire_bytes(n_atoms: int, n_structures: int, relax_cell: bool) -> int:
    """Algorithmic bytes of one m3g_fire_step over running structures: forces read (12 B / atom), velocities read and
    written (48), coordinates read and written (48; with the cell filter x read and written + positions written, 72);
    per structure the FIRE scalars, status and step count (40), energy in / out (12) and, with the cell filter, stress
    in (36), stress out, L0, lattice in / out, cell rows of x and v in / out (6 x 72)."""
    per_atom = 12 + 48 + (72 if relax_cell else 48)
    per_struct = 52 + ((36 + 6 * 72) if relax_cell else 0)
    return per_atom * n_atoms + per_struct * n_structures


def model(dev):
    g = np.load(os.path.join(ROOT, "tests", "golden", "c1_default.npz"))
    sd = {k[3:]: torch.from_numpy(np.array(g[k])) for k in g.files if k.startswith("sd.")}
    mdl = m3g.build_model(5.0, 4.0, 3, 3, 95, 64, 3, device=dev)
    mdl.load_state_dict({k: (v * 3 if k.endswith("weight") else v) for k, v in sd.items()})
    return mdl


class Timed(m3g.M3GNetCalculator):
    """The calculator with CUDA events around compute and around the model inside it (instrumented runs only)."""

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.events = None

    def _eval(self, batch, stress):
        if self.events is None:
            return super()._eval(batch, stress)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = super()._eval(batch, stress)
        e1.record()
        self.events["model"].append((e0, e1))
        return out

    def compute(self, *a, **k):
        if self.events is None:
            return super().compute(*a, **k)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = super().compute(*a, **k)
        e1.record()
        self.events["compute"].append((e0, e1))
        return out


def relax(mdl, dev, structs, relax_cell, fmax, steps, max_atoms=None, instrument=False):
    calc = Timed(mdl, 5.0, 4.0, skin=0.5, device=dev)
    if instrument:
        calc.events = {"model": [], "compute": []}
        _lib.PROFILE = {}
    opt = m3g.BatchFire(calc, structs, relax_cell=relax_cell, max_atoms=max_atoms)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = opt.run(fmax=fmax, steps=steps)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    out = dict(wall_s=wall, iterations=opt.n_iterations, regroups=opt.n_regroups, regroup_s=opt.regroup_seconds,
               atom_steps=int(sum(r["n_steps"] * len(r["positions"]) for r in res)),
               statuses={s: sum(r["status"] == s for r in res) for s in ("converged", "not converged", "failed")})
    if instrument:
        prof, _lib.PROFILE = _lib.PROFILE, None
        ms = lambda evs: [a.elapsed_time(b) for a, b in evs]  # noqa: E731
        out["fire_us"] = [1e3 * x for x in ms(prof.get("fire_step", []))]
        out["compute_ms"] = ms(calc.events["compute"])
        out["model_ms"] = ms(calc.events["model"])
    return out, res


def sequential(mdl, dev, structs, relax_cell, fmax, steps):
    t, atom_steps = 0.0, 0
    for lat, cart, z in structs:
        calc = m3g.M3GNetCalculator(mdl, 5.0, 4.0, skin=0.5, device=dev)
        opt = m3g.Fire(calc, lat, cart, z, relax_cell=relax_cell)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        opt.run(fmax=fmax, steps=steps)
        torch.cuda.synchronize()
        t += time.perf_counter() - t0
        atom_steps += opt.n_steps * len(z)
    return dict(structures=len(structs), wall_s=round(t, 3), atom_steps=atom_steps,
                atom_steps_per_s=round(atom_steps / t), structures_per_s=round(len(structs) / t, 3))


def workload(mdl, dev, structs, relax_cell, fmax, steps, max_atoms, repeats, sample):
    runs = [relax(mdl, dev, structs, relax_cell, fmax, steps, max_atoms)[0] for _ in range(repeats)]
    inst, _ = relax(mdl, dev, structs, relax_cell, fmax, steps, max_atoms, instrument=True)
    wall = statistics.median(r["wall_s"] for r in runs)
    atoms = sum(len(s[2]) for s in structs)
    first = inst["iterations"]
    fire = statistics.median(inst["fire_us"])
    compute = sum(inst["compute_ms"])
    graph = compute - sum(inst["model_ms"])
    first_set = admit([len(s[2]) for s in structs], 0, max_atoms, 0, 0)
    b0 = fire_bytes(sum(len(s[2]) for s in structs[:first_set]), first_set, relax_cell)
    return dict(
        structures=len(structs), atoms=atoms, relax_cell=relax_cell, fmax=fmax, steps=steps, max_atoms=max_atoms,
        repeats=repeats, wall_s=[round(r["wall_s"], 4) for r in runs], wall_s_median=round(wall, 4),
        iterations=runs[0]["iterations"], regroups=runs[0]["regroups"], statuses=runs[0]["statuses"],
        atom_steps=runs[0]["atom_steps"], atom_steps_per_s_median=round(runs[0]["atom_steps"] / wall),
        structures_per_s_median=round(len(structs) / wall, 3),
        step_ms_median=round(1e3 * wall / runs[0]["iterations"], 4),
        fire_call_us_median=round(fire, 2), fire_call_us_min=round(min(inst["fire_us"]), 2),
        fire_call_pct_of_step=round(100 * 1e-6 * fire / (wall / runs[0]["iterations"]), 3),
        first_working_set=first_set, fire_bytes_first_working_set=b0, fire_hbm_bound_us=round(1e6 * b0 / HBM_BYTES_PER_S, 2),
        instrumented_wall_s=round(inst["wall_s"], 4), instrumented_iterations=first,
        graph_build_pct=round(100 * 1e-3 * graph / inst["wall_s"], 2),
        model_pct=round(100 * 1e-3 * sum(inst["model_ms"]) / inst["wall_s"], 2),
        regroup_pct=round(100 * inst["regroup_s"] / inst["wall_s"], 2),
        sequential_fire=sequential(mdl, dev, structs[:sample], relax_cell, fmax, steps))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--structures", type=int, default=1000)
    ap.add_argument("--max-atoms", type=int, default=30000)
    ap.add_argument("--sample", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    m3g.calculator.stabilise_allocator()
    mdl = model(dev)
    res = {"card": card(), "torch": torch.__version__}
    lat, cart, z, sizes = synthetic.config2_batch(256)
    ptr = np.concatenate([[0], np.cumsum(sizes)])
    c2 = [(lat[b], cart[ptr[b]:ptr[b + 1]], z[ptr[b]:ptr[b + 1]]) for b in range(len(sizes))]
    relax(mdl, dev, c2[:32], False, 0.0, 3)  # warm-up: module loads, allocator
    res["a_c2_fixed_cell"] = workload(mdl, dev, c2, False, 0.0, args.steps, None, args.repeats, args.sample)
    res["b_c2_relax_cell"] = workload(mdl, dev, c2, True, 0.0, args.steps, None, args.repeats, args.sample)
    mpf = [synthetic.mpf_like_structure(s) for s in range(args.structures)]
    res["c_mpf_to_convergence"] = workload(mdl, dev, mpf, False, 0.05, 200, args.max_atoms, args.repeats,
                                           2 * args.sample)
    res["card_after"] = card()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
