"""Fused conv-block adjoint (m3g_conv_tc_block_bwd) against the two m3g_conv_tc_bwd_saved launches it replaces, on
BASELINE.json configs[1] (C2: 256 x 108-atom Cu cells), in one process:

  (a) per block: CUDA-event time of one fused launch and of the two-launch sequence, alternating, on the saved
      activations of a real forward pass, for the three block kinds of a 3-block model (last: no residual base; middle;
      block 0: no g_z1), with the achieved rate on the algorithmic bytes of DESIGN.md §4;
  (b) whole step: model(batch) ms with M3G_CONV_BWD_FUSED on and off (module attribute), alternating rounds.

  python tools/bench_conv_bwd.py [--launches 30] [--steps 20] [--rounds 6] [--warmup 3] [--out profiles/conv_bwd_fused.json]

Prints one JSON object (card name and power limit read in the same run) and writes it to --out when given.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch_m3gnet_b200 as m3g  # noqa: E402
from bench_stress import card, timed  # noqa: E402
from torch_m3gnet_b200 import _lib, engine, synthetic  # noqa: E402
from torch_m3gnet_b200.data import MaterialGraphKey as K  # noqa: E402
from torch_m3gnet_b200.data.material_graph import get_plan  # noqa: E402
from torch_m3gnet_b200.nn import conv as conv_mod  # noqa: E402
from torch_m3gnet_b200.nn._functions import sm_count  # noqa: E402

# block kinds of the default 3-block model: (residual base g_e2 present, g_z1 stored)
KINDS = {"last": (False, True), "middle": (True, True), "block0": (True, False)}


def algorithmic_bytes(E, base, gz, fused):
    """Bytes per launch (sequence) the kernels are designed to move once, DESIGN.md §4 / conv_tc_bwd_saved:
    saved activations 2 x 1 KB, upstream g_x2[src] (+ ge2), residual bases, the ge2 round trip (two launches only),
    g_e, 2 x 512 B of g_z1 (blocks > 0), h / src / g_h."""
    per = 2048 + 256 + 256 * base + 256 + 1024 * gz
    per += 40 if fused else 56 + 256 + 256 + 256
    return per * E


def per_block(model, batch, launches):
    plan = get_plan(batch)
    eng = model.step_engine()
    desc, keep = eng.prepare(batch, plan)
    n = eng.n_blocks
    eng.run_phases(desc, 0, engine.phase_readout(n), batch[K.POS].device)  # forward: saves of every block, g_x
    torch.cuda.synchronize()
    scratch, off = keep["scratch"], keep["off"]
    E, N, R = plan.E, plan.N, 3
    dev = scratch.device

    def view(name, size):
        return scratch[off[name]:off[name] + size]

    n_save = int(_lib.LIB.load().m3g_conv_tc_save_floats(E))
    b = n - 1
    cw = eng.cvs[b]._packed.get()
    nd, ed = cw["node"], cw["edge"]
    save_n, save_e = view(f"save_n{b}", n_save), view(f"save_e{b}", n_save)
    h = keep["out"][K.EDGE_WEIGHTS]
    g_x2 = view("g_x0", 64 * N)
    g_e2 = torch.randn(E, 64, device=dev)
    ge2, g_e = torch.empty(E, 64, device=dev), torch.empty(E, 64, device=dev)
    gz_n, gz_e = torch.empty(E, 128, device=dev), torch.empty(E, 128, device=dev)
    gh = torch.empty(2, E, R, device=dev)
    passes, n_sm = 3, sm_count(dev)
    res = {}
    for kind, (base, gz) in KINDS.items():
        gb = g_e2 if base else None
        zn, ze = (gz_n, gz_e) if gz else (None, None)

        def two():
            _lib.call("conv_tc_bwd_saved", plan.src, h, nd["wimgT"], nd["WhT"], save_n, g_x2, gb, E, R, 1, passes,
                      n_sm, ge2, zn, gh[0], 1)
            _lib.call("conv_tc_bwd_saved", plan.src, h, ed["wimgT"], ed["WhT"], save_e, ge2, ge2, E, R, 0, passes,
                      n_sm, g_e, ze, gh[1], 1)

        def fused():
            _lib.call("conv_tc_block_bwd", plan.src, h, nd["wimgT"], nd["WhT"], save_n, ed["wimgT"], ed["WhT"], save_e,
                      g_x2, gb, E, R, passes, n_sm, g_e, zn, ze, gh[0], gh[1], 0)

        for _ in range(3):
            two()
            fused()
        t_two, t_fused = [], []
        for _ in range(launches):  # alternate the arms; one sample = one fused launch or one two-launch sequence
            t_two.append(timed(two, 1))
            t_fused.append(timed(fused, 1))
        m_two, m_fused = statistics.median(t_two), statistics.median(t_fused)
        b_two, b_fused = algorithmic_bytes(E, base, gz, False), algorithmic_bytes(E, base, gz, True)
        res[kind] = dict(residual_base=base, g_z1=gz, launches=launches,
                         two_launch_ms_median=round(m_two, 4), fused_ms_median=round(m_fused, 4),
                         two_launch_ms_min_max=[round(min(t_two), 4), round(max(t_two), 4)],
                         fused_ms_min_max=[round(min(t_fused), 4), round(max(t_fused), 4)],
                         fused_over_two=round(m_fused / m_two, 4),
                         two_launch_algorithmic_bytes=b_two, fused_algorithmic_bytes=b_fused,
                         two_launch_gb_per_s=round(b_two / (m_two * 1e-3) / 1e9, 1),
                         fused_gb_per_s=round(b_fused / (m_fused * 1e-3) / 1e9, 1))
    del keep
    return dict(atoms=N, bonds=E, **res)


def whole_step(model, batch, steps, rounds, warmup):
    old = conv_mod.CONV_BWD_FUSED

    def step(fused):
        conv_mod.CONV_BWD_FUSED = fused
        return model(batch)

    try:
        for _ in range(warmup):
            step(False)
            step(True)
        on, off = [], []
        for _ in range(rounds):
            off.append(timed(lambda: step(False), steps))
            on.append(timed(lambda: step(True), steps))
    finally:
        conv_mod.CONV_BWD_FUSED = old
    m_on, m_off = statistics.median(on), statistics.median(off)
    return dict(steps_per_round=steps, rounds=rounds, step_ms_fused=[round(x, 4) for x in on],
                step_ms_two_launch=[round(x, 4) for x in off], step_ms_fused_median=round(m_on, 4),
                step_ms_two_launch_median=round(m_off, 4), saved_ms_median=round(m_off - m_on, 4),
                saved_pct_median=round(100.0 * (m_off - m_on) / m_off, 2),
                spread_fused_ms=round(max(on) - min(on), 4), spread_two_launch_ms=round(max(off) - min(off), 4))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=30)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    model = m3g.build_model(5.0, 4.0, 3, 3, 95, 64, 3, device=dev)
    res = {"card": card(), "torch": torch.__version__}
    lat, cart, z, sizes = synthetic.config2_batch(256)
    c2 = m3g.Batch.from_arrays(lat, cart, z, sizes, 5.0, 4.0, device=dev)
    model(c2)  # plan, weight packing
    res["per_block"] = per_block(model, c2, args.launches)
    res["whole_step"] = whole_step(model, c2, args.steps, args.rounds, args.warmup)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
