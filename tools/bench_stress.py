"""Cost of the cell stress (Gradient.compute_stress, kernel m3g_bond_virial): model steps with the stress off and on,
alternating in one process, on BASELINE.json configs[1] (C2: 256 x 108-atom Cu cells) and on the configs[3] cell (C4:
one 32 000-atom Cu cell, undecomposed), plus the stress call's own GPU time from CUDA events.

  python tools/bench_stress.py [--steps 20] [--rounds 5] [--warmup 3] [--out profiles/stress_bench.json]

Prints one JSON object (card name and power limit read in the same run) and writes it to --out when given.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch_m3gnet_b200 as m3g  # noqa: E402
from torch_m3gnet_b200 import _lib, synthetic  # noqa: E402
from torch_m3gnet_b200.data.material_graph import get_plan  # noqa: E402

BYTES_PER_BOND = 36  # vec4 16 B + g_vec4 16 B + g_dist 4 B read by the stage-1 kernel
HBM_BYTES_PER_S = 7.7e12  # B200 data sheet (one GPU of an HGX B200)


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else None
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def timed(fn, n):
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(n):
        fn()
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / n


def measure(model, batch, steps, rounds, warmup):
    plan = get_plan(batch)

    def step(stress):
        model.compute_stress = stress
        return model(batch)

    for _ in range(warmup):
        step(False)
        step(True)
    off, on = [], []
    for _ in range(rounds):  # alternate the two arms so that drifts of the shared host hit both
        off.append(timed(lambda: step(False), steps))
        on.append(timed(lambda: step(True), steps))
    # the stress call's own time: events around each m3g_bond_virial call (two kernels) inside full steps
    _lib.PROFILE = {}
    for _ in range(steps):
        step(True)
    torch.cuda.synchronize()
    evs = _lib.PROFILE.pop("bond_virial")
    _lib.PROFILE = None
    kern_ms = [a.elapsed_time(b) for a, b in evs]
    model.compute_stress = False
    kern = statistics.median(kern_ms)
    step_off, step_on = statistics.median(off), statistics.median(on)
    return dict(atoms=plan.N, bonds=plan.E, structures=plan.B, steps_per_round=steps, rounds=rounds,
                step_ms_off=[round(x, 4) for x in off], step_ms_on=[round(x, 4) for x in on],
                step_ms_off_median=round(step_off, 4), step_ms_on_median=round(step_on, 4),
                overhead_ms_median=round(step_on - step_off, 4),
                overhead_pct_median=round(100.0 * (step_on - step_off) / step_off, 3),
                stress_call_us_median=round(1e3 * kern, 2), stress_call_us_min=round(1e3 * min(kern_ms), 2),
                stress_call_pct_of_step=round(100.0 * kern / step_off, 3),
                bytes_read=plan.E * BYTES_PER_BOND,
                achieved_gb_per_s=round(plan.E * BYTES_PER_BOND / (kern * 1e-3) / 1e9, 1),
                hbm_bound_us=round(1e6 * plan.E * BYTES_PER_BOND / HBM_BYTES_PER_S, 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    model = m3g.build_model(5.0, 4.0, 3, 3, 95, 64, 3, device=dev)
    res = {"card": card(), "torch": torch.__version__}
    lat, cart, z, sizes = synthetic.config2_batch(256)
    c2 = m3g.Batch.from_arrays(lat, cart, z, sizes, 5.0, 4.0, device=dev)
    res["c2"] = measure(model, c2, args.steps, args.rounds, args.warmup)
    del c2
    lat, cart, z = synthetic.fcc_cu_supercell(20, 0.05, 4)
    c4 = m3g.Batch.from_arrays(lat[None], cart, z, [len(cart)], 5.0, 4.0, device=dev, want_triplet_index=False)
    res["c4"] = measure(model, c4, max(args.steps // 2, 1), args.rounds, args.warmup)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
