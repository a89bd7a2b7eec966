"""GPU: the fused node + edge adjoint of a conv block (m3g_conv_tc_block_bwd) against the two m3g_conv_tc_bwd_saved
launches it replaces.  Same MMAs and the same fp32 adds per row, so every output must be bitwise equal."""
import numpy as np
import pytest
import torch

from oracle import m3gnet_oracle as O
from tests.util import golden, graph_dict, state_dict_of, to_batch

pytestmark = pytest.mark.gpu


def _images(device, seed):
    """[W2d^T, W2g^T, W1e_dense^T, W1e_gate^T] hi|lo image pairs of random 64x64 matrices."""
    from torch_m3gnet_b200 import _lib

    g = torch.Generator(device="cpu").manual_seed(seed)
    out = torch.empty(8 * 64 * 64, device=device)
    for i in range(4):
        W = (torch.randn(64, 64, generator=g) / 8).to(device)
        _lib.call("tc_pack_b", W, 64, 64, out[(2 * i) * 4096:(2 * i + 1) * 4096], out[(2 * i + 1) * 4096:(2 * i + 2) * 4096])
    return out


def _inputs(device, E, R, seed):
    from torch_m3gnet_b200 import _lib

    g = torch.Generator(device="cpu").manual_seed(seed)
    N = max(E // 12, 1)
    src = torch.sort(torch.randint(0, N, (E,), generator=g)).values.to(torch.int32)
    n_save = int(_lib.LIB.load().m3g_conv_tc_save_floats(E))

    def save():
        s = torch.randn(n_save, generator=g)
        # blocks 0, 1 of each tile hold SiLU'(z1) in [-0.1, 1.1]; blocks 2, 3 the layer-2 pre-activations
        return s.view(-1, 4, 128 * 64).mul_(torch.tensor([0.3, 0.3, 2.0, 2.0]).view(1, 4, 1)).view(-1)

    t = dict(src=src, h=torch.rand(E, R, generator=g), n_WhT=torch.randn(R, 64, generator=g),
             e_WhT=torch.randn(R, 64, generator=g), save_n=save(), save_e=save(), g_x2=torch.randn(N, 64, generator=g),
             g_e2=torch.randn(E, 64, generator=g))
    t = {k: v.to(device) for k, v in t.items()}
    t["n_wimgT"], t["e_wimgT"] = _images(device, seed + 1), _images(device, seed + 2)
    return t


def _nan(shape, device):
    return torch.full(shape, float("nan"), device=device)


def _two_launches(t, E, R, passes, n_sm, with_base, with_gz, gh_sum):
    from torch_m3gnet_b200 import _lib

    dev = t["h"].device
    g_e2 = t["g_e2"] if with_base else None
    ge2, g_e = _nan((E, 64), dev), _nan((E, 64), dev)
    gz_n = _nan((E, 128), dev) if with_gz else None
    gz_e = _nan((E, 128), dev) if with_gz else None
    gh_n, gh_e = _nan((E, R), dev), _nan((E, R), dev)
    _lib.call("conv_tc_bwd_saved", t["src"], t["h"], t["n_wimgT"], t["n_WhT"], t["save_n"], t["g_x2"], g_e2, E, R, 1,
              passes, n_sm, ge2, gz_n, gh_n, 1)
    if gh_sum:
        _lib.call("conv_tc_bwd_saved", t["src"], t["h"], t["e_wimgT"], t["e_WhT"], t["save_e"], ge2, ge2, E, R, 0,
                  passes, n_sm, g_e, gz_e, gh_n, 0)
        return g_e, gz_n, gz_e, gh_n
    _lib.call("conv_tc_bwd_saved", t["src"], t["h"], t["e_wimgT"], t["e_WhT"], t["save_e"], ge2, ge2, E, R, 0, passes,
              n_sm, g_e, gz_e, gh_e, 1)
    return g_e, gz_n, gz_e, gh_n, gh_e


def _fused(t, E, R, passes, n_sm, with_base, with_gz, gh_sum):
    from torch_m3gnet_b200 import _lib

    dev = t["h"].device
    g_e = _nan((E, 64), dev)
    gz_n = _nan((E, 128), dev) if with_gz else None
    gz_e = _nan((E, 128), dev) if with_gz else None
    gh_n = _nan((E, R), dev)
    gh_e = None if gh_sum else _nan((E, R), dev)
    _lib.call("conv_tc_block_bwd", t["src"], t["h"], t["n_wimgT"], t["n_WhT"], t["save_n"], t["e_wimgT"], t["e_WhT"],
              t["save_e"], t["g_x2"], t["g_e2"] if with_base else None, E, R, passes, n_sm, g_e, gz_n, gz_e, gh_n, gh_e,
              int(gh_sum))
    return (g_e, gz_n, gz_e, gh_n) if gh_sum else (g_e, gz_n, gz_e, gh_n, gh_e)


# E < 128, E not a multiple of 128, and enough tiles that every SM walks several of them
@pytest.mark.parametrize("E", [100, 1061, 3 * 148 * 128 + 77])
@pytest.mark.parametrize("R", [1, 2, 3])
@pytest.mark.parametrize("passes", [1, 3])
def test_block_bwd_equals_two_launches(device, E, R, passes):
    from torch_m3gnet_b200.nn._functions import sm_count

    t = _inputs(device, E, R, seed=E * 10 + R)
    n_sm = sm_count(device)
    for with_base in (False, True):
        for with_gz in (False, True):
            for gh_sum in (False, True):
                want = _two_launches(t, E, R, passes, n_sm, with_base, with_gz, gh_sum)
                got = _fused(t, E, R, passes, n_sm, with_base, with_gz, gh_sum)
                torch.cuda.synchronize()
                names = ("g_e", "gz_node", "gz_edge", "g_h") if gh_sum else ("g_e", "gz_node", "gz_edge", "g_h_node",
                                                                             "g_h_edge")
                for name, a, b in zip(names, got, want):
                    if b is None:
                        assert a is None
                        continue
                    assert torch.isfinite(b).all(), name
                    assert torch.equal(a, b), (f"{name} differs (base={with_base} gz={with_gz} gh_sum={gh_sum}): "
                                               f"max|diff|={(a - b).abs().max().item():.3e}")


# ---------------------------------------------------------------------------------------------------------------------
KEYS = ("total_energy", "forces", "stresses", "cell_stress")


def _outputs(model, make_batch, engine_on, fused):
    from torch_m3gnet_b200 import engine
    from torch_m3gnet_b200.data.material_graph import get_plan
    from torch_m3gnet_b200.nn import conv as conv_mod

    old = engine.ENABLED, conv_mod.CONV_BWD_FUSED
    engine.ENABLED, conv_mod.CONV_BWD_FUSED = engine_on, fused
    try:
        b = make_batch()
        assert model.step_engine().supports(b, get_plan(b)) == engine_on
        model.compute_stress = True
        out = model(b)
        torch.cuda.synchronize()
        return {k: out[k].detach().clone() for k in KEYS}
    finally:
        model.compute_stress = False
        engine.ENABLED, conv_mod.CONV_BWD_FUSED = old


def _model(device, sd, **kw):
    from torch_m3gnet_b200 import build_model

    model = build_model(5.0, 4.0, 3, 3, 95, 64, 3, device=device, **kw)
    model.load_state_dict(sd)
    return model


def _check_model(model, make_batch):
    for engine_on in (True, False):
        on = _outputs(model, make_batch, engine_on, True)
        off = _outputs(model, make_batch, engine_on, False)
        for k in KEYS:
            assert torch.isfinite(off[k]).all(), k
            assert torch.equal(on[k], off[k]), f"{k} (engine={engine_on}): max|diff|={(on[k] - off[k]).abs().max():.3e}"


@pytest.mark.parametrize("fixture", ["c1_default", "tio2_default"])
def test_model_bitwise_with_and_without_fusion(device, fixture):
    g, c1 = golden(fixture), golden("c1_default")
    sd = {k: (v * 3.0 if k.endswith("weight") else v) for k, v in state_dict_of(c1).items()}
    model = _model(device, sd)
    gd = graph_dict(g)
    _check_model(model, lambda: to_batch(gd, device))


def test_model_bitwise_ragged_batch(device):
    from torch_m3gnet_b200 import Batch

    hp = O.HyperParams(energy_scale=2.5, length_scale=1.3, elemental_energies=torch.linspace(-1.0, 1.0, 95))
    model = _model(device, O.init_params(hp, seed=3, gain=2.0), energy_scale=2.5, length_scale=1.3,
                   elemental_energies=hp.elemental_energies)
    structs = [O.mpf_like_structure(s) for s in (1, 2, 5)] + [O.fcc_supercell(2, jitter=0.1, seed=9)]
    lat = np.stack([s[0] for s in structs])
    cart = np.concatenate([s[1] for s in structs])
    z = np.concatenate([s[2] for s in structs])
    sizes = [len(s[1]) for s in structs]
    _check_model(model, lambda: Batch.from_arrays(lat, cart, z, sizes, 5.0, 4.0, device=device))


def test_model_bitwise_c2_and_launch_count(device):
    """Full C2 batch (256 x 108-atom Cu); the fused step makes one launch less per conv block."""
    import torch_m3gnet_b200 as m3g
    from torch_m3gnet_b200 import _lib, synthetic
    from torch_m3gnet_b200.nn import conv as conv_mod

    torch.manual_seed(0)
    model = m3g.build_model(5.0, 4.0, 3, 3, 95, 64, 3, device=device)
    lat, cart, z, sizes = synthetic.config2_batch(256)
    batch = m3g.Batch.from_arrays(lat, cart, z, sizes, 5.0, 4.0, device=device)
    _check_model(model, lambda: batch)
    eng = model.step_engine()
    old = conv_mod.CONV_BWD_FUSED
    try:
        counts = {}
        for fused in (True, False):
            conv_mod.CONV_BWD_FUSED = fused
            l0 = _lib.LAUNCHES
            model(batch)
            counts[fused] = _lib.LAUNCHES - l0
            assert counts[fused] == eng.launches(True)
    finally:
        conv_mod.CONV_BWD_FUSED = old
    assert counts[False] - counts[True] == 3
