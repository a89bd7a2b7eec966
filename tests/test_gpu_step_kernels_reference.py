"""GPU: the per-step kernels outside the tensor-core conv MLPs and the three-body op, through the C ABI, against the
float64 restatements in tests/step_kernels_oracle.py and tests/conv_oracle.py, at every branch of their dispatchers:
m3g_readout_fwd / _bwd / _fwd_bwd, m3g_structure_sum, m3g_linear_fwd / _bwd_input, m3g_conv_mlp_fwd / _bwd,
m3g_segment_sum_add, m3g_conv_gather_gz, m3g_radial_fwd / _bwd, m3g_edge_adjust_fwd / _bwd, m3g_geometry_fwd / _bwd,
m3g_angles_fwd / _bwd and m3g_forces_virial.

Accuracy.  Every output is checked per column (max over rows of |got - ref| over the column's largest scale) and per
row (the same over the row's largest scale), so that a wrong column block or a wrong tail row cannot hide behind the
largest entry.  The scale is condition-aware, the sum of |terms| of each dot product: forwards are the float64
restatement evaluated on the absolute values of every input and weight, adjoints are taken at the true operating point
with every local factor and the upstream gradient replaced by its absolute value (step_kernels_oracle.adjoint); sums
onto a prefill or a base add |prefill|.

Error model for tau.  A float32 dot product of length K accumulated in any order is within K * 2^-24 of its sum of
|terms|; each layer of a chain (a matvec followed by an activation) adds one such error.  tau(K, layers) =
2 * layers * (K + 8) * 2^-24: the 8 covers the bias, the activation (expf and a division, a few ulp) and the
products around the dot product, the 2 is margin.  Per kernel:
  readout forward        tau(F, 3)          readout adjoint         tau(F, 6)  (forward recomputed, three adjoints)
  linear                 tau(K)             structure_sum           tau(atoms of the structure)
  conv_mlp forward       tau(F + R, 3)      conv_mlp adjoint        tau(2F + R, 6)
  radial forward         tau(R, 2)          radial adjoint          tau(R, 4)  (sinf / cosf / division per term)
  edge_adjust forward    tau(R)             edge_adjust adjoint     tau(F + R, 2)
  geometry adjoint       tau(bonds of the atom)            angles adjoint  tau(triplets of the bond)
  virial                 tau(atoms of the structure)
The fwd4 / bwd64 edge-adjust forms evaluate the sigmoid with __expf / __fdividef, a relative error of a few 1e-7
(csrc/geometry.cu:190-192): they get TAU_Q = 2e-6 on top.  The worst error of each (kernel, branch, output) is printed
as a table at the end of the run; tau is never taken from it.

Bit for bit: m3g_geometry_fwd / m3g_angles_fwd against the float32 restatement of their rounding order,
m3g_segment_sum_add and both forms of m3g_conv_gather_gz against float32 sums in ascending edge order, forces = -g_pos.
Outputs do not depend on what their buffers held (NaN and a sentinel), guard rows after every output stay intact,
repeated calls are bitwise equal (except m3g_angles_bwd, which adds with float atomics), readout_fwd_bwd equals
readout_fwd + readout_bwd, and the shared-weight readout gives the same bits with 8 warps as with 16."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests import conv_oracle as C
from tests import step_kernels_oracle as S
from tests.test_gpu_conv_tc_reference import SENTINEL, guarded, same

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -24
TAU_Q = 2e-6
FS = (1, 4, 17, 31, 32, 33, 60, 64, 68, 96, 100, 128)
RS = tuple(range(1, 11))
SIZES = (1, 3, 4, 5, 15, 16, 17, 63, 64, 65)
MAX_F, MAX_R = 128, 10
SENT = str(SENTINEL)  # results of a run are keyed by str(fill): "nan" for NaN-filled outputs, SENT for the sentinel


def tau(K, layers=1):
    return 2.0 * layers * (K + 8) * U


RESULTS = {}  # (kernel, branch, output) -> [worst normalised error, tau]


@pytest.fixture(scope="module", autouse=True)
def _error_table(request):
    yield
    if not RESULTS:
        return
    lines = ["", "step kernels vs float64: worst normalised error (per column / per row)",
             f"{'kernel':<18}{'branch':<22}{'output':<28}{'worst':>11}{'tau':>10}"]
    for (k, b, o), (v, t) in sorted(RESULTS.items()):
        lines.append(f"{k:<18}{b:<22}{o:<28}{v:>11.2e}{t:>10.1e}")
    capman = request.config.pluginmanager.getplugin("capturemanager")
    if capman is None:
        print("\n".join(lines))
    else:
        with capman.global_and_fixture_disabled():
            print("\n".join(lines), flush=True)


def call(name, *args):
    from torch_m3gnet_b200 import _lib

    _lib.call(name, *args)


def n_sms(device):
    from torch_m3gnet_b200.nn._functions import sm_count

    return sm_count(device)


def nerr(got, ref, scale):
    """max over columns of max_i |got - ref| / max_i scale, and the same per row"""
    got = got.double().reshape(ref.shape[0], -1)
    ref = ref.double().reshape(ref.shape[0], -1)
    s = scale.double().reshape(ref.shape[0], -1)
    if ref.numel() == 0:
        return 0.0
    if not bool(torch.isfinite(got).all()):
        return math.inf
    err = (got - ref).abs()
    col = (err.amax(0) / s.amax(0).clamp_min(1e-300)).max().item()
    row = (err.amax(1) / s.amax(1).clamp_min(1e-300)).max().item()
    return max(col, row)


class Checks:
    def __init__(self):
        self.failed = []

    def acc(self, kern, branch, out, got, ref, scale, t, ctx=""):
        v = nerr(got, ref, scale)
        key = (kern, branch, out)
        old = RESULTS.get(key, [0.0, t])
        RESULTS[key] = [max(old[0], v), max(old[1], t)]
        if not v <= t:
            self.failed.append(f"{kern} [{branch}] {out} {ctx}: normalised error {v:.3e} > {t:.1e}")
        return v

    def true(self, cond, msg):
        if not cond:
            self.failed.append(msg)

    def done(self):
        assert not self.failed, "\n".join(self.failed[:40]) + (f"\n... {len(self.failed)} in all"
                                                               if len(self.failed) > 40 else "")


def out_buf(shape, device, fill=float("nan"), dtype=torch.float32):
    """(view, whole allocation with GUARD sentinel rows after it)"""
    return guarded(torch.full(shape, fill, dtype=dtype, device=device), SENTINEL)


def guard_ok(full, rows):
    return bool((full[rows:] == SENTINEL).all())


def rand(g, *shape, scale=1.0):
    return scale * torch.randn(*shape, generator=g)


# ---------------------------------------------------------------------------------------------------------------------
# mirrors of the dispatchers' conditions
def readout_branch(F, warps=16):
    """readout.cu launch_readout: the shared-weight (SW) form when F % 4 == 0, NJ <= 2 and the weights fit"""
    nj = (F + 31) // 32
    epw = 4 if warps == 16 else 8
    smem = (warps * epw * 5 * F + 8 * F * F) * 4
    if F % 4 == 0 and smem <= 227 * 1024 and nj <= 2:
        return f"sw{warps} nj{nj}"
    return f"nj{nj}"


def readout_persistent(F, N, n_sm, warps=16):
    """the SW grid is capped at one CTA per SM of warps x epw = 64 atoms: more atoms take the grid-stride loop"""
    return readout_branch(F, warps).startswith("sw") and N > n_sm * 64


def linear_branch(K, M):
    """conv.cu launch_linear_tiled / linear_kernel (K, M of the kernel: out (n,M) = in (n,K) Wt)"""
    if K % 32 == 0 and M % 64 == 0:
        return "tiled128" if M >= 256 else "tiled64"
    return "fallback" + (" K>128" if K > 128 else "") + (" M>128" if M > 128 else "")


def conv_mlp_branch(F, mode):
    return f"nj{(F + 31) // 32} mode{mode}"


def gather_branch(F, ldp, po):
    return "gz128" if F == 64 and ldp % 4 == 0 and po % 4 == 0 else "generic"


def adjust_fwd_branch(F, R):
    if F % 4 == 0 and R == 3:
        return "fwd4<3>"
    return "fwd4<4>" if F % 4 == 0 and R <= 4 else "generic"


def adjust_bwd_branch(F, R):
    if F == 64 and R == 3:
        return "bwd64<3>"
    return "bwd64<4>" if F == 64 and R <= 4 else "generic"


# ---------------------------------------------------------------------------------------------------------------------
# readout
def readout_weights(F, seed, device):
    g = torch.Generator().manual_seed(seed)
    w = {}
    for s in ("d", "g"):
        w[f"W0{s}"], w[f"b0{s}"] = rand(g, F, F, scale=F ** -0.5), rand(g, F, scale=0.5)
        w[f"W1{s}"], w[f"b1{s}"] = rand(g, F, F, scale=F ** -0.5), rand(g, F, scale=0.5)
        w[f"w2{s}"], w[f"b2{s}"] = rand(g, F, scale=F ** -0.5), rand(g, 1, scale=0.5)
    w = {k: v.to(device) for k, v in w.items()}
    for k in ("W0d", "W1d", "W0g", "W1g"):
        w[k + "T"] = w[k].t().contiguous()
    return w


RO_FWD = ("W0dT", "b0d", "W1dT", "b1d", "w2d", "b2d", "W0gT", "b0g", "W1gT", "b1g", "w2g", "b2g")
RO_BWD = ("W0d", "W1d", "W0g", "W1g")


class ReadoutCase:
    def __init__(self, F, N, device, seed=0):
        g = torch.Generator().manual_seed(seed + 1000 * F + N)
        self.F, self.N, self.device = F, N, device
        self.B = max(1, N // 7 + 2)
        self.w = readout_weights(F, seed + F, device)
        self.x = guarded(rand(g, N, F).to(device))[0]
        self.elemental = guarded(rand(g, N).to(device))[0]
        batch = torch.sort(torch.randint(0, self.B, (N,), generator=g)).values.to(torch.int32)
        self.batch = guarded(batch.to(device), 0)[0]
        self.ups = {"g_atomic": rand(g, N).to(device), "g_scaled_total": rand(g, self.B).to(device),
                    "g_total": rand(g, self.B).to(device)}
        self.scale = 1.7

    def fwd(self, out):
        call("readout_fwd", self.x, *[self.w[k] for k in RO_FWD], self.elemental, self.scale, self.N, self.F, out)

    def bwd(self, names, out):
        u = [self.ups[n] if n in names else None for n in ("g_atomic", "g_scaled_total", "g_total")]
        call("readout_bwd", self.x, *[self.w[k] for k in RO_FWD], *[self.w[k] for k in RO_BWD], *u, self.batch,
             self.scale, self.N, self.F, out)

    def fwd_bwd(self, atomic, g_x):
        call("readout_fwd_bwd", self.x, *[self.w[k] for k in RO_FWD], *[self.w[k] for k in RO_BWD], self.elemental,
             self.ups["g_total"], self.batch, self.scale, self.N, self.F, atomic, g_x)

    def refs(self, names):
        u = [self.ups[n] if n in names else None for n in ("g_atomic", "g_scaled_total", "g_total")]
        ref = S.readout_bwd(self.x, self.w, *u, self.batch, self.scale)
        ua = [None if t is None else t.abs() for t in u]
        scale = S.readout_bwd(self.x, self.w, *ua, self.batch, self.scale, S.ABS)
        return ref, scale


UPSTREAMS = (("g_atomic",), ("g_scaled_total",), ("g_total",), ("g_atomic", "g_scaled_total", "g_total"))


def readout_sizes(F, device):
    extra = (n_sms(device) * 64 + 5,) if readout_branch(F).startswith("sw") else ()
    return SIZES + extra


@pytest.mark.parametrize("F", FS)
def test_readout(device, F):
    """every branch of launch_readout x every upstream form, N across warp-group tails and past the SW grid"""
    ck = Checks()
    S_ = n_sms(device)
    for N in readout_sizes(F, device):
        c = ReadoutCase(F, N, device)
        br = readout_branch(F) + (" persist" if readout_persistent(F, N, S_) else "")
        ctx = f"F={F} N={N}"
        ref = S.readout_fwd(c.x, c.w, c.elemental, c.scale)
        sc = S.readout_fwd(c.x.abs(), S.absolute(c.w), c.elemental.abs(), c.scale)
        outs = {}
        for fill in (float("nan"), SENTINEL):
            a, af = out_buf((N,), device, fill)
            c.fwd(a)
            outs[str(fill)] = a
            ck.true(guard_ok(af, N), f"readout_fwd guard overwritten ({ctx})")
        ck.true(same(outs[SENT], outs["nan"]), f"readout_fwd depends on its buffer ({ctx})")
        ck.acc("readout_fwd", br, "atomic", outs[SENT], ref, sc, tau(F, 3), ctx)
        atomic = outs[SENT]
        for names in UPSTREAMS:
            r, s = c.refs(names)
            gx = {}
            for fill in (float("nan"), SENTINEL):
                g_x, gf = out_buf((N, F), device, fill)
                c.bwd(names, g_x)
                gx[str(fill)] = g_x
                ck.true(guard_ok(gf, N), f"readout_bwd guard overwritten ({ctx} {names})")
            ck.true(same(gx[SENT], gx["nan"]), f"readout_bwd depends on its buffer ({ctx} {names})")
            ck.acc("readout_bwd", br, "+".join(n[2:] for n in names), gx[SENT], r, s, tau(F, 6), ctx)
            if names == ("g_total",):
                a2, a2f = out_buf((N,), device)
                g2, g2f = out_buf((N, F), device)
                c.fwd_bwd(a2, g2)
                ck.true(same(a2, atomic) and same(g2, gx[SENT]),
                        f"readout_fwd_bwd differs from readout_fwd + readout_bwd ({ctx})")
                ck.true(guard_ok(a2f, N) and guard_ok(g2f, N), f"readout_fwd_bwd guard overwritten ({ctx})")
                a3, g3 = out_buf((N,), device)[0], out_buf((N, F), device)[0]
                c.fwd_bwd(a3, g3)
                ck.true(same(a3, a2) and same(g3, g2), f"readout_fwd_bwd repeat differs ({ctx})")
    ck.done()


_WARPS_SCRIPT = r"""
import json, sys, torch
sys.path.insert(0, sys.argv[1])
from tests.test_gpu_step_kernels_reference import ReadoutCase, readout_sizes
dev = torch.device("cuda:0")
out = {}
for F in json.loads(sys.argv[2]):
    for N in readout_sizes(F, dev):
        c = ReadoutCase(F, N, dev)
        a, g = torch.empty(N, device=dev), torch.empty(N, F, device=dev)
        c.fwd_bwd(a, g)
        a1, g1 = torch.empty(N, device=dev), torch.empty(N, F, device=dev)
        c.fwd(a1)
        c.bwd(("g_atomic", "g_scaled_total", "g_total"), g1)
        out[f"{F},{N}"] = [t.cpu() for t in (a, g, a1, g1)]
torch.save(out, sys.argv[3])
"""


def test_readout_sw_warps_bitwise(device, tmp_path):
    """readout.cu:13: the SW shapes (16 warps x 4 atoms, M3G_RO_WARPS=8: 8 warps x 8 atoms) accumulate in the same
    order, so they give the same bits.  The variable is read once per process, hence the subprocesses."""
    Fs = [F for F in FS if readout_branch(F).startswith("sw")]
    assert Fs == [4, 32, 60, 64] and all(readout_branch(F, 8).startswith("sw8") for F in Fs)
    res = {}
    for warps in ("16", "8"):
        env = {k: v for k, v in os.environ.items() if k != "M3G_RO_WARPS"}
        if warps == "8":
            env["M3G_RO_WARPS"] = "8"
        path = str(tmp_path / f"ro{warps}.pt")
        r = subprocess.run([sys.executable, "-c", _WARPS_SCRIPT, ROOT, json.dumps(Fs), path], env=env, cwd=ROOT,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        res[warps] = torch.load(path)
    assert res["16"].keys() == res["8"].keys()
    bad = [k for k in res["16"] if not all(same(a, b) for a, b in zip(res["16"][k], res["8"][k]))]
    assert not bad, f"M3G_RO_WARPS=8 differs from 16 warps at (F, N) = {bad}"


def _structures(sizes, device, seed):
    """atom_ptr (B+1) int32 on the device for the given structure sizes, and lattices (B,3,3), one with det < 0"""
    g = torch.Generator().manual_seed(seed)
    ptr = torch.tensor([0] + list(np.cumsum(sizes)), dtype=torch.int32)
    lat = 6.0 * torch.eye(3) + rand(g, len(sizes), 3, 3, scale=0.8)
    lat[0, 1] = -lat[0, 1]
    assert float(torch.linalg.det(lat[0])) < 0
    return guarded(ptr.to(device), 0)[0], guarded(lat.to(device))[0]


STRUCT_SIZES = (3, 0, 1, 33, 0, 100, 32, 5, 0)


def test_structure_sum_and_forces_virial(device):
    """zero-atom, one-atom and > 32-atom structures, a negative-determinant lattice; forces = -g_pos bit for bit"""
    ck = Checks()
    ptr, lat = _structures(STRUCT_SIZES, device, 1)
    B, N = len(STRUCT_SIZES), sum(STRUCT_SIZES)
    g = torch.Generator().manual_seed(2)
    atomic = guarded(rand(g, N).to(device))[0]
    pos = guarded(rand(g, N, 3, scale=4.0).to(device))[0]
    g_pos = guarded(rand(g, N, 3).to(device))[0]
    Kmax = max(STRUCT_SIZES)
    res = {}
    for fill in (float("nan"), SENTINEL):
        st, stf = out_buf((B,), device, fill)
        t, tf = out_buf((B,), device, fill)
        call("structure_sum", atomic, ptr, B, 2.5, st, t)
        f, ff = out_buf((N, 3), device, fill)
        sv, svf = out_buf((B, 6), device, fill)
        call("forces_virial", pos, g_pos, lat, ptr, N, B, f, sv)
        torch.cuda.synchronize()
        ck.true(all(guard_ok(a, r) for a, r in ((stf, B), (tf, B), (ff, N), (svf, B))), "guard overwritten")
        res[str(fill)] = (st, t, f, sv)
    ck.true(all(same(a, b) for a, b in zip(res[SENT], res["nan"])), "outputs depend on their buffers")
    st, t, f, sv = res[SENT]
    r_st, r_t = S.structure_sum(atomic, ptr, 2.5)
    a_st, a_t = S.structure_sum(atomic.abs(), ptr, 2.5)
    ck.acc("structure_sum", "-", "scaled", st, r_st, a_st, tau(Kmax))
    ck.acc("structure_sum", "-", "total", t, r_t, a_t, tau(Kmax))
    ck.true(same(f, -g_pos), "forces != -g_pos")
    r_f, r_sv = S.forces_virial(pos, g_pos, lat, ptr)
    ck.acc("forces_virial", "-", "stress", sv, r_sv, S.forces_virial(pos, g_pos, lat, ptr, True)[1], tau(Kmax))
    empty = torch.tensor([n == 0 for n in STRUCT_SIZES], device=device)
    ck.true(bool((st[empty] == 0).all() and (sv[empty] == 0).all()), "a zero-atom structure has a nonzero sum")
    out2 = [torch.empty_like(x) for x in (st, t, f, sv)]
    call("structure_sum", atomic, ptr, B, 2.5, out2[0], out2[1])
    call("forces_virial", pos, g_pos, lat, ptr, N, B, out2[2], out2[3])
    ck.true(all(same(a, b) for a, b in zip(out2, (st, t, f, sv))), "repeated calls differ")
    ck.done()


# ---------------------------------------------------------------------------------------------------------------------
# per-atom projections
LINEAR_CASES = [  # (K, M, in-kernel roles): linear_fwd (n,K)x(K,M); linear_bwd_input takes (n,M) g and W (M,K)
    (64, 512), (128, 1024), (64, 128), (32, 64), (17, 136), (136, 17), (1, 8), (96, 68), (200, 300), (128, 129),
]
LINEAR_N = SIZES + (129, 300)


@pytest.mark.parametrize("K,M", LINEAR_CASES)
def test_linear(device, K, M):
    """linear_fwd (bias null or not) and linear_bwd_input (base null or not) at both tiled shapes and the fallback with
    several K chunks and column passes"""
    ck = Checks()
    for n in LINEAR_N:
        g = torch.Generator().manual_seed(K * 7 + M + n)
        x = guarded(rand(g, n, K).to(device))[0]
        W = rand(g, M, K, scale=K ** -0.5).to(device)
        Wt = guarded(W.t().contiguous())[0]
        bias = rand(g, M).to(device)
        gup = guarded(rand(g, n, M).to(device))[0]
        Wb = guarded(W.clone())[0]
        baseK = guarded(rand(g, n, K).to(device))[0]
        ctx = f"K={K} M={M} n={n}"
        for b in (None, bias):
            res = {}
            for fill in (float("nan"), SENTINEL):
                y, yf = out_buf((n, M), device, fill)
                call("linear_fwd", x, Wt, b, n, K, M, y)
                ck.true(guard_ok(yf, n), f"linear_fwd guard overwritten ({ctx})")
                res[str(fill)] = y
            ck.true(same(res[SENT], res["nan"]), f"linear_fwd depends on its buffer ({ctx})")
            sc = S.linear(x.abs(), Wt.abs(), None if b is None else b.abs())
            ck.acc("linear_fwd", linear_branch(K, M), "out" + ("+bias" if b is not None else ""), res[SENT],
                   S.linear(x, Wt, b), sc, tau(K), ctx)
        for base in (None, baseK):
            res = {}
            for fill in (float("nan"), SENTINEL):
                y, yf = out_buf((n, K), device, fill)
                call("linear_bwd_input", gup, Wb, base, n, K, M, y)
                ck.true(guard_ok(yf, n), f"linear_bwd_input guard overwritten ({ctx})")
                res[str(fill)] = y
            ck.true(same(res[SENT], res["nan"]), f"linear_bwd_input depends on its buffer ({ctx})")
            y2 = torch.empty_like(res[SENT])
            call("linear_bwd_input", gup, Wb, base, n, K, M, y2)
            ck.true(same(y2, res[SENT]), f"linear_bwd_input repeat differs ({ctx})")
            sc = S.linear_bwd_input(gup.abs(), Wb.abs(), None if base is None else base.abs())
            ck.acc("linear_bwd_input", linear_branch(M, K), "out" + ("+base" if base is not None else ""),
                   res[SENT], S.linear_bwd_input(gup, Wb, base), sc, tau(M), ctx)
    ck.done()


# ---------------------------------------------------------------------------------------------------------------------
# generic conv MLPs, segment sums and the gradient gather
def _csr(src, dst, N):
    edge_ptr = C.edge_ptr_of(src, N)
    in_perm = torch.sort(dst, stable=True).indices
    in_ptr = C.edge_ptr_of(dst[in_perm], N)
    return edge_ptr, in_ptr, in_perm


class ConvCase:
    def __init__(self, kind, E, F, R, device, seed):
        src, dst, N = C.graph(kind, E, seed)
        g = torch.Generator().manual_seed(seed + 5)
        self.F, self.R, self.E, self.N, self.device = F, R, E, N, device
        self.src64, self.dst64 = src.to(device), dst.to(device)
        self.src = guarded(src.to(torch.int32).to(device), 0)[0]
        self.dst = guarded(dst.to(torch.int32).to(device), 0)[0]
        self.P = guarded(rand(g, N, 8 * F).to(device))[0]
        self.e = guarded(rand(g, E, F).to(device))[0]
        self.h = guarded(torch.rand(E, R, generator=g).to(device))[0]
        self.g_up = {0: guarded(rand(g, E, F).to(device))[0], 1: guarded(rand(g, N, F).to(device))[0]}
        self.base = guarded(rand(g, E, F).to(device))[0]
        self.gh_pre = rand(g, E, R).to(device)
        self.w = {k: v.to(device) for k, v in C.mlp_weights(R, seed + 9, F=F, scaled=False).items()}
        self.wT = {k: v.to(device) for k, v in C.transposed(self.w).items()}
        self.Wh = self.w["WhT"].t().contiguous()
        self.ptrs = [t.to(torch.int32).to(device) for t in _csr(src, dst, N)]

    def fwd(self, po, mode, y, w=None):
        w = self.w if w is None else w
        wT = self.wT if w is self.w else {k: v.to(self.device) for k, v in C.transposed(w).items()}
        call("conv_mlp_fwd", self.P, 8 * self.F, po, self.src, self.dst, self.e, self.h, wT["W1eT"], wT["W2dT"],
             w["b2d"], wT["W2gT"], w["b2g"], w["WhT"], self.E, self.F, self.R, mode, y)

    def bwd(self, po, mode, base, g_e, g_z1, g_h):
        w, wT = self.w, self.wT
        call("conv_mlp_bwd", self.P, 8 * self.F, po, self.src, self.dst, self.e, self.h, wT["W1eT"], wT["W2dT"],
             w["b2d"], wT["W2gT"], w["b2g"], w["WhT"], w["W1e"], w["W2d"], w["W2g"], self.Wh, self.g_up[mode], base,
             self.E, self.F, self.R, mode, g_e, g_z1, g_h)

    def ref_fwd(self, po, mode, w=None):
        w = self.w if w is None else w
        ref = C.forward(self.P, po, self.src64, self.dst64, self.e, self.h, w, mode)
        sc = C.forward(self.P.abs(), po, self.src64, self.dst64, self.e.abs(), self.h.abs(), S.absolute(w), 1)
        return ref, sc + (self.e.double().abs() if mode == 0 else 0.0)

    def ref_bwd(self, po, mode):
        ref = C.mlp_bwd(self.P, po, self.src64, self.dst64, self.e, self.h, self.w, self.g_up[mode], None, mode)
        sc = S.conv_mlp_bwd_scale(self.P, po, self.src64, self.dst64, self.e, self.h, self.w, self.g_up[mode], mode)
        return ref, sc


def conv_cases():
    """every (F, R) once, E and the graph kind cycling through the sizes and the degree-edge kinds"""
    kinds = ("deg31", "deg32", "deg33", "hubs", "one_atom", "self", "poisson", "single")
    out = []
    for i, F in enumerate(FS):
        for R in RS:
            j = i * len(RS) + R
            out.append((F, R, SIZES[j % len(SIZES)] + 64 * (j % 3), kinds[j % len(kinds)]))
    return out


@pytest.mark.parametrize("F", FS)
def test_conv_mlp(device, F):
    """m3g_conv_mlp_fwd / _bwd, NJ = 1..4, modes 0 and 1, R = 1..10, g_h onto a prefill, g_e_base null or not"""
    ck = Checks()
    for F_, R, E, kind in conv_cases():
        if F_ != F:
            continue
        c = ConvCase(kind, E, F, R, device, seed=F * 100 + R)
        ctx = f"F={F} R={R} E={E} {kind}"
        for mode, po in ((0, 0), (1, 4 * F)):
            br = conv_mlp_branch(F, mode)
            ref, sc = c.ref_fwd(po, mode)
            res = {}
            for fill in (float("nan"), SENTINEL):
                y, yf = out_buf((E, F), device, fill)
                c.fwd(po, mode, y)
                ck.true(guard_ok(yf, E), f"conv_mlp_fwd guard overwritten ({ctx})")
                res[str(fill)] = y
            ck.true(same(res[SENT], res["nan"]), f"conv_mlp_fwd depends on its buffer ({ctx})")
            ck.acc("conv_mlp_fwd", br, "y", res[SENT], ref, sc, tau(F + R, 3), ctx)
            (r_e, r_z, r_h), (s_e, s_z, s_h) = c.ref_bwd(po, mode)
            for base in (None, c.base):
                outs = []
                for fill in (float("nan"), SENTINEL):
                    g_e, gef = out_buf((E, F), device, fill)
                    g_z1, gzf = out_buf((E, 2 * F), device, fill)
                    g_h, ghf = guarded(c.gh_pre.clone(), SENTINEL)
                    c.bwd(po, mode, base, g_e, g_z1, g_h)
                    ck.true(guard_ok(gef, E) and guard_ok(gzf, E) and guard_ok(ghf, E),
                            f"conv_mlp_bwd guard overwritten ({ctx})")
                    outs.append((g_e, g_z1, g_h))
                ck.true(all(same(a, b) for a, b in zip(*outs)), f"conv_mlp_bwd depends on its buffers ({ctx})")
                g_e, g_z1, g_h = outs[1]
                b64 = 0.0 if base is None else base.double()
                ck.acc("conv_mlp_bwd", br, "g_e" + ("+base" if base is not None else ""), g_e, r_e + b64,
                       s_e + (0.0 if base is None else base.double().abs()), tau(2 * F + R, 6), ctx)
                ck.acc("conv_mlp_bwd", br, "g_z1", g_z1, r_z, s_z, tau(2 * F + R, 6), ctx)
                ck.acc("conv_mlp_bwd", br, "g_h+pre", g_h, r_h + c.gh_pre.double(), s_h + c.gh_pre.double().abs(),
                       tau(2 * F + R, 6), ctx)
    ck.done()


GATHER_CASES = [  # (F, ldp, po)
    (64, 512, 0), (64, 512, 256), (64, 513, 1), (64, 516, 2), (17, 136, 0), (17, 136, 68), (128, 1024, 512),
    (1, 8, 4), (33, 264, 0),
]


@pytest.mark.parametrize("kind", ("hubs", "deg31", "deg32", "deg33", "one_atom", "self", "poisson", "single"))
def test_segment_sum_and_gather(device, kind):
    """m3g_segment_sum_add and both forms of m3g_conv_gather_gz bit for bit against float32 sums in ascending edge
    order (and against float64), on graphs with bondless atoms and hubs of 129 and 200 bonds; g_P columns outside
    [po, po + 4F) are left alone"""
    ck = Checks()
    for i, (F, ldp, po) in enumerate(GATHER_CASES):
        E = SIZES[i % len(SIZES)] + 300 * (i % 2)
        src, dst, N = C.graph(kind, E, seed=i)
        g = torch.Generator().manual_seed(i)
        edge_ptr, in_ptr, in_perm = _csr(src, dst, N)
        dptr = [t.to(torch.int32).to(device) for t in (edge_ptr, in_ptr, in_perm)]
        ctx = f"{kind} F={F} ldp={ldp} po={po} E={E}"
        gz = guarded(rand(g, E, 2 * F).to(device))[0]
        want_out = S.segment_sum_f32(gz.cpu().numpy(), edge_ptr.numpy())
        want_in = S.segment_sum_f32(gz.cpu().numpy(), in_ptr.numpy(), in_perm.numpy())
        res = []
        for fill in (float("nan"), SENTINEL):
            gP, gPf = out_buf((N, ldp), device, fill)
            call("conv_gather_gz", gz, *dptr, N, F, ldp, po, gP)
            ck.true(guard_ok(gPf, N), f"conv_gather_gz guard overwritten ({ctx})")
            res.append(gP)
        ck.true(same(res[0][:, po:po + 4 * F], res[1][:, po:po + 4 * F]), f"gather depends on its buffer ({ctx})")
        gP = res[1].cpu()
        rest = torch.ones(ldp, dtype=torch.bool)
        rest[po:po + 4 * F] = False
        ck.true(bool((gP[:, rest] == SENTINEL).all()), f"gather wrote outside its columns ({ctx})")
        br = gather_branch(F, ldp, po)
        got = gP[:, po:po + 4 * F].numpy()
        ck.true(np.array_equal(got[:, :2 * F], want_out) and np.array_equal(got[:, 2 * F:], want_in),
                f"conv_gather_gz [{br}] is not the ascending float32 sum ({ctx})")
        r64 = torch.cat([C.segment_sum(torch.zeros(N, 2 * F), gz.cpu(), src, N),
                         C.segment_sum(torch.zeros(N, 2 * F), gz.cpu(), dst, N)], 1)
        s64 = torch.cat([C.segment_sum(torch.zeros(N, 2 * F), gz.cpu().abs(), src, N),
                         C.segment_sum(torch.zeros(N, 2 * F), gz.cpu().abs(), dst, N)], 1)
        deg = int(max((edge_ptr[1:] - edge_ptr[:-1]).max(), (in_ptr[1:] - in_ptr[:-1]).max()))
        ck.acc("conv_gather_gz", br, "g_P", gP[:, po:po + 4 * F], r64, s64, tau(deg), ctx)
        # segment_sum_add: x2 = x + messages summed per source atom
        msg = guarded(rand(g, E, F).to(device))[0]
        base = guarded(rand(g, N, F).to(device))[0]
        out, outf = out_buf((N, F), device)
        call("segment_sum_add", base, msg, dptr[0], N, F, out)
        ck.true(guard_ok(outf, N), f"segment_sum_add guard overwritten ({ctx})")
        want = base.cpu().numpy() + S.segment_sum_f32(msg.cpu().numpy(), edge_ptr.numpy())
        ck.true(np.array_equal(out.cpu().numpy(), want), f"segment_sum_add is not base + the ascending sum ({ctx})")
    ck.done()


# ---------------------------------------------------------------------------------------------------------------------
# radial basis and edge adjustor
@pytest.mark.parametrize("rc", [5.0, 4.2, 3.0, 6.5])
def test_radial(device, rc):
    """R = 1..10, r = 0 (the sinc's a == 0 branch: h from s(0) = 1, no gradient), r = r_c, r across (0, r_c]"""
    from torch_m3gnet_b200.nn.featurizer import radial_constants

    ck = Checks()
    for R in RS:
        E = SIZES[R % len(SIZES)] + 100
        g = torch.Generator().manual_seed(R)
        r = torch.rand(E, generator=g) * rc
        r[0], r[1], r[2] = 0.0, rc, rc * 1e-3
        r = guarded(r.to(device))[0]
        consts = radial_constants(R, rc)[0].to(device)
        g_h = guarded(rand(g, E, R).to(device))[0]
        ctx = f"R={R} rc={rc}"
        res = []
        for fill in (float("nan"), SENTINEL):
            h, hf = out_buf((E, R), device, fill)
            call("radial_fwd", r, consts, E, R, h)
            gd, gdf = out_buf((E,), device, fill)
            call("radial_bwd", r, consts, g_h, E, R, gd)
            ck.true(guard_ok(hf, E) and guard_ok(gdf, E), f"radial guard overwritten ({ctx})")
            res.append((h, gd))
        ck.true(same(res[0][0], res[1][0]) and same(res[0][1], res[1][1]), f"radial depends on its buffer ({ctx})")
        h, gd = res[1]
        ck.acc("radial_fwd", "-", "h", h, S.radial(r, consts, R), S.radial(r, consts, R, absolute_=True), tau(R, 2),
               ctx)
        ck.acc("radial_bwd", "-", "g_dist", gd, S.radial(r, consts, R, g_h),
               S.radial(r, consts, R, g_h, absolute_=True), tau(R, 4), ctx)
        ck.true(float(gd[0]) == 0.0, f"radial_bwd: nonzero gradient at r = 0 ({ctx})")
    ck.done()


@pytest.mark.parametrize("F", FS)
def test_edge_adjust(device, F):
    """fwd4<3>, fwd4<4> (R in 1, 2, 4), generic (F % 4 != 0 or R >= 5); bwd64<3>, bwd64<4>, generic up to R = 10"""
    ck = Checks()
    for R in RS:
        E = SIZES[(F + R) % len(SIZES)] + 64 * (R % 3)
        g = torch.Generator().manual_seed(F * 11 + R)
        h = guarded(torch.rand(E, R, generator=g).to(device))[0]
        Wt = guarded(rand(g, R, F, scale=R ** -0.5 * 2).to(device))[0]
        g_e0 = guarded(rand(g, E, F).to(device))[0]
        ctx = f"F={F} R={R} E={E}"
        res = []
        for fill in (float("nan"), SENTINEL):
            e0, ef = out_buf((E, F), device, fill)
            call("edge_adjust_fwd", h, Wt, E, R, F, e0)
            gh, ghf = out_buf((E, R), device, fill)
            call("edge_adjust_bwd", h, Wt, g_e0, E, R, F, gh)
            ck.true(guard_ok(ef, E) and guard_ok(ghf, E), f"edge_adjust guard overwritten ({ctx})")
            res.append((e0, gh))
        ck.true(same(res[0][0], res[1][0]) and same(res[0][1], res[1][1]),
                f"edge_adjust depends on its buffer ({ctx})")
        e0, gh = res[1]
        bf, bb = adjust_fwd_branch(F, R), adjust_bwd_branch(F, R)
        ck.acc("edge_adjust_fwd", bf, "e0", e0, S.edge_adjust_fwd(h, Wt), S.edge_adjust_fwd(h.abs(), Wt.abs()),
               tau(R) + (TAU_Q if bf != "generic" else 0.0), ctx)
        ck.acc("edge_adjust_bwd", bb, "g_h", gh, S.edge_adjust_bwd(h, Wt, g_e0),
               S.edge_adjust_bwd(h, Wt, g_e0, S.ABS), tau(F + R, 2) + (TAU_Q if bb != "generic" else 0.0),
               ctx)
    ck.done()


# ---------------------------------------------------------------------------------------------------------------------
# geometry and angles
class GeomCase:
    """Bonds of the "hubs" degree pattern (out-degrees 129, 3, 200, 0, 17, ...), a third of them pointing at one
    in-hub atom, the trailing atom without any bond; atoms spread over structures of STRUCT_SIZES-like sizes, one
    lattice with det < 0; triplets = every ordered pair of bonds of an atom (capped per atom)."""

    def __init__(self, E, device, seed=0, cap=40):
        src, dst, N = C.graph("hubs", E, seed)
        g = torch.Generator().manual_seed(seed + 3)
        N = max(N, 4)
        dst = dst % (N - 1)
        dst[::3] = min(3, N - 2)
        self.N, self.E, self.device = N, E, device
        sizes = [N // 3, 0, 1, N - N // 3 - 1, 0]
        self.ptr, self.lat = _structures(sizes, device, seed)
        batch = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes)).to(torch.int32)
        self.batch = guarded(batch.to(device), 0)[0]
        self.pos = guarded(rand(g, N, 3, scale=3.0).to(device))[0]
        shift = torch.randint(-2, 3, (E, 3), generator=g, dtype=torch.int32)
        shift[(src == dst) & (shift == 0).all(1), 0] = 1  # no zero-length bond
        self.shift = guarded(shift.to(device), 0)[0]
        self.src64, self.dst64 = src, dst
        self.src = guarded(src.to(torch.int32).to(device), 0)[0]
        self.dst = guarded(dst.to(torch.int32).to(device), 0)[0]
        self.ptrs = [t.to(torch.int32).to(device) for t in _csr(src, dst, N)]
        edge_ptr = self.ptrs[0].cpu()
        pairs = []
        for i in range(N):
            b = list(range(int(edge_ptr[i]), int(edge_ptr[i + 1])))[:cap]
            pairs += [(p, q) for p in b for q in b if p != q]
        self.tri = torch.tensor(pairs, dtype=torch.int64).t().contiguous().reshape(2, -1).to(device)
        self.T = self.tri.shape[1]
        deg_in = torch.bincount(dst, minlength=N)
        self.max_bonds = int((deg_in + torch.bincount(src, minlength=N)).max())

    def f32(self):
        v, r = S.geometry_f32(self.pos.cpu().numpy(), self.lat.cpu().numpy(), self.batch.cpu().numpy(),
                              self.src64.numpy(), self.dst64.numpy(), self.shift.cpu().numpy())
        return v, r


@pytest.mark.parametrize("E", [1, 5, 17, 65, 1000, 4099])
def test_geometry(device, E):
    """geometry_fwd and angles_fwd bit for bit; geometry_bwd with g_vec4 / g_dist each null or not and scale != 1, on
    hubs of > 32 in and out bonds, bondless atoms, zero- and one-atom structures and a det < 0 lattice; angles_bwd
    onto a prefill"""
    ck = Checks()
    c = GeomCase(E, device, seed=E)
    ctx = f"E={E}"
    res = []
    for fill in (float("nan"), SENTINEL):
        vec4, vf = out_buf((E, 4), device, fill)
        dist, df = out_buf((E,), device, fill)
        call("geometry_fwd", c.pos, c.lat, c.batch, c.src, c.dst, c.shift, E, vec4, dist)
        ck.true(guard_ok(vf, E) and guard_ok(df, E), f"geometry_fwd guard overwritten ({ctx})")
        res.append((vec4, dist))
    vec4, dist = res[1]
    ck.true(same(res[0][0], vec4) and same(res[0][1], dist), f"geometry_fwd depends on its buffer ({ctx})")
    v, r = c.f32()
    ck.true(np.array_equal(vec4[:, :3].cpu().numpy(), v) and np.array_equal(vec4[:, 3].cpu().numpy(), r) and
            np.array_equal(dist.cpu().numpy(), r), f"geometry_fwd is not the float32 restatement bit for bit ({ctx})")
    g = torch.Generator().manual_seed(E + 1)
    vec4 = guarded(vec4.clone())[0]
    if c.T:
        cos, cf = out_buf((c.T,), device)
        call("angles_fwd", vec4, c.tri, c.T, cos)
        ck.true(guard_ok(cf, c.T), f"angles_fwd guard overwritten ({ctx})")
        c_raw, c_cl = S.angles_f32(vec4.cpu().numpy(), c.tri.cpu().numpy())
        ck.true(np.array_equal(cos.cpu().numpy(), c_cl), f"angles_fwd is not the float32 restatement ({ctx})")
        g_cos = guarded(rand(g, c.T).to(device))[0]
        pre = rand(g, E, 4).to(device)
        gv, gvf = guarded(pre.clone(), SENTINEL)
        call("angles_bwd", vec4, c.tri, g_cos, c.T, gv)
        torch.cuda.synchronize()
        ck.true(guard_ok(gvf, E), f"angles_bwd guard overwritten ({ctx})")
        passes = torch.from_numpy((c_raw >= -1) & (c_raw <= 1)).to(device)
        per_bond = int(torch.bincount(c.tri.flatten(), minlength=E).max())
        ck.acc("angles_bwd", "-", "g_vec4+pre", gv, pre.double() + S.angles_bwd(vec4, c.tri, g_cos, passes),
               pre.double().abs() + S.angles_bwd(vec4, c.tri, g_cos, passes, True), tau(per_bond), ctx)
    g_vec4 = guarded(rand(g, E, 4).to(device))[0]
    g_dist = guarded(rand(g, E).to(device))[0]
    for gv4, gd in ((g_vec4, g_dist), (g_vec4, None), (None, g_dist)):
        for scale in (1.0, -0.37):
            sub = f"{ctx} g_vec4={gv4 is not None} g_dist={gd is not None} scale={scale}"
            outs = []
            for fill in (float("nan"), SENTINEL):
                gp, gpf = out_buf((c.N, 3), device, fill)
                call("geometry_bwd", vec4, gv4, gd, *c.ptrs, c.N, scale, gp)
                ck.true(guard_ok(gpf, c.N), f"geometry_bwd guard overwritten ({sub})")
                outs.append(gp)
            gp2 = torch.empty_like(outs[1])
            call("geometry_bwd", vec4, gv4, gd, *c.ptrs, c.N, scale, gp2)
            ck.true(same(outs[0], outs[1]) and same(gp2, outs[1]), f"geometry_bwd not bitwise repeatable ({sub})")
            ref = S.geometry_bwd(vec4, gv4, gd, c.src, c.dst, c.N, scale)
            sc = S.geometry_bwd(vec4, gv4, gd, c.src, c.dst, c.N, scale, absolute_=True)
            ck.acc("geometry_bwd", "+".join(n for n, t in (("g_vec4", gv4), ("g_dist", gd)) if t is not None),
                   "g_pos", outs[1], ref, sc, tau(c.max_bonds), sub)
            ck.true(bool((outs[1][c.N - 1] == 0).all()), f"geometry_bwd: the bondless atom has a gradient ({sub})")
    ck.done()


def _ulps(x, k):
    """x moved by k ulps (float32)"""
    return (torch.from_numpy(np.asarray(x, np.float32)).view(torch.int32) + torch.as_tensor(k, dtype=torch.int32)) \
        .view(torch.float32)


def test_collinear_triplets(device):
    """Bonds exactly parallel and exactly opposite (cos = +-1: every cubic cell has them) and a few ulps off: angles_fwd
    clamps as the float32 restatement does, and angles_bwd passes the gradient exactly where the forward's unclamped
    cos lies in [-1, 1] (torch.clamp's mask is taken from its input)."""
    g = torch.Generator().manual_seed(7)
    n = 4096
    a = rand(g, n, 3)
    a[: n // 4] = torch.tensor([1.0, 0.0, 0.0])  # axis bonds, as in a cubic cell
    a[n // 4: n // 2] = torch.tensor([1.0, 1.0, 0.0]) * 1.8075  # fcc nearest-neighbour direction
    sign = torch.where(torch.arange(n) % 2 == 0, 1.0, -1.0)[:, None]
    lam = torch.pow(2.0, torch.randint(-2, 3, (n, 1), generator=g).float())
    b = sign * lam * a  # exactly parallel / opposite
    k = torch.randint(-3, 4, (n,), generator=g)
    comp = b.abs().argmax(1)  # a nonzero component
    k[: n // 8] = 0
    b[torch.arange(n), comp] = _ulps(b[torch.arange(n), comp].numpy(), k)
    v = torch.cat([a, b]).numpy()
    r = np.sqrt((v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2])
    vec4 = torch.from_numpy(np.concatenate([v, r[:, None]], 1)).to(device)
    tri = torch.stack([torch.arange(n), torch.arange(n) + n]).to(device)
    c_raw, c_cl = S.angles_f32(vec4.cpu().numpy(), tri.cpu().numpy())
    assert (c_raw > 1).any() and (c_raw < -1).any() and (np.abs(c_raw) == 1).any() and (np.abs(c_raw) < 1).any()
    cos = torch.full((n,), float("nan"), device=device)
    call("angles_fwd", vec4, tri, n, cos)
    assert np.array_equal(cos.cpu().numpy(), c_cl), "angles_fwd does not clamp as the float32 restatement"
    g_cos = 1.0 + torch.rand(n, generator=g).to(device)
    gv = torch.zeros(2 * n, 4, device=device)
    call("angles_bwd", vec4, tri, g_cos, n, gv)
    passes = torch.from_numpy((c_raw >= -1) & (c_raw <= 1))
    got = (gv[:n].abs().sum(1) + gv[n:].abs().sum(1)).cpu() > 0
    wrong = torch.nonzero(got != passes).flatten()
    assert wrong.numel() == 0, (f"{wrong.numel()} of {n} collinear triplets: the gradient mask differs from the "
                                f"forward's clamp, e.g. unclamped cos {c_raw[wrong[:5].numpy()].tolist()}")
    ref = S.angles_bwd(vec4, tri, g_cos, passes.to(device))
    sc = S.angles_bwd(vec4, tri, g_cos, passes.to(device), True)
    ck = Checks()
    ck.acc("angles_bwd", "collinear", "g_vec4", gv, ref, sc, tau(1))
    ck.done()


# ---------------------------------------------------------------------------------------------------------------------
# branch coverage: the cases above reach every branch of every dispatcher
def test_branch_coverage(device):
    n_sm = n_sms(device)
    reached = set()
    for F in FS:
        for N in readout_sizes(F, device):
            reached.add(("readout", readout_branch(F) + (" persist" if readout_persistent(F, N, n_sm) else "")))
        reached |= {("readout", readout_branch(F, 8)) for F in FS if readout_branch(F).startswith("sw")}
    for K, M in LINEAR_CASES:
        reached |= {("linear", linear_branch(K, M)), ("linear", linear_branch(M, K))}
    for F, R, E, kind in conv_cases():
        reached |= {("conv_mlp", conv_mlp_branch(F, m) + f" R={R}") for m in (0, 1)}
    reached |= {("gather", gather_branch(F, ldp, po)) for F, ldp, po in GATHER_CASES}
    for F in FS:
        for R in RS:
            reached |= {("adjust_fwd", adjust_fwd_branch(F, R)), ("adjust_bwd", adjust_bwd_branch(F, R))}
    want = {("readout", b) for b in ("sw16 nj1", "sw16 nj2", "sw16 nj1 persist", "sw16 nj2 persist", "sw8 nj1",
                                     "sw8 nj2", "nj1", "nj2", "nj3", "nj4")}
    want |= {("linear", b) for b in ("tiled64", "tiled128", "fallback", "fallback K>128", "fallback M>128",
                                     "fallback K>128 M>128")}
    want |= {("conv_mlp", f"nj{nj} mode{m} R={R}") for nj in (1, 2, 3, 4) for m in (0, 1) for R in RS}
    want |= {("gather", "gz128"), ("gather", "generic")}
    want |= {("adjust_fwd", b) for b in ("fwd4<3>", "fwd4<4>", "generic")}
    want |= {("adjust_bwd", b) for b in ("bwd64<3>", "bwd64<4>", "generic")}
    assert not want - reached, f"dispatcher branches no case reaches: {sorted(want - reached)}"
    assert 128 in FS and MAX_F == 128 and MAX_R == 10 and RS[-1] == MAX_R
    assert any(N > n_sm * 64 for N in readout_sizes(64, device))


# ---------------------------------------------------------------------------------------------------------------------
# interface edges (host-side checks only: nothing is launched out of bounds)
def test_interface_edges(device):
    from torch_m3gnet_b200.nn.featurizer import radial_constants

    c = ReadoutCase(64, 5, device)
    w = c.w
    buf = torch.full((16384,), SENTINEL, device=device)
    ibuf = torch.zeros(64, dtype=torch.int32, device=device)
    consts = radial_constants(10, 5.0)[0].to(device)
    for F in (0, 129):
        with pytest.raises(RuntimeError, match=f"F={F}"):
            call("readout_fwd", buf, *[w[k] for k in RO_FWD], buf, 1.0, 5, F, buf)
        with pytest.raises(RuntimeError, match=f"F={F}"):
            call("readout_bwd", buf, *[w[k] for k in RO_FWD], *[w[k] for k in RO_BWD], None, None, buf, ibuf, 1.0, 5,
                 F, buf)
        with pytest.raises(RuntimeError, match=f"F={F}"):
            call("readout_fwd_bwd", buf, *[w[k] for k in RO_FWD], *[w[k] for k in RO_BWD], buf, buf, ibuf, 1.0, 5, F,
                 buf, buf)
        with pytest.raises(RuntimeError, match=f"F={F}"):
            call("conv_mlp_fwd", buf, 8, 0, ibuf, ibuf, buf, buf, buf, buf, buf, buf, buf, buf, 5, F, 3, 0, buf)
        with pytest.raises(RuntimeError, match=f"F={F}"):
            call("conv_mlp_bwd", buf, 8, 0, ibuf, ibuf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf,
                 buf, None, 5, F, 3, 0, buf, buf, buf)
        with pytest.raises(RuntimeError, match=f"F={F}"):
            call("edge_adjust_fwd", buf, buf, 5, 3, F, buf)
        with pytest.raises(RuntimeError, match=f"F={F}"):
            call("edge_adjust_bwd", buf, buf, buf, 5, 3, F, buf)
        with pytest.raises(RuntimeError, match=f"F={F}"):
            call("conv_gather_gz", buf, ibuf, ibuf, ibuf, 5, F, 8 * max(F, 1), 0, buf)
        with pytest.raises(RuntimeError, match=f"F={F}"):
            call("segment_sum_add", buf, buf, ibuf, 5, F, buf)
    for R in (0, 11):
        pat = f"(R|n_max)={R}"
        with pytest.raises(RuntimeError, match=pat):
            call("radial_fwd", buf, consts, 5, R, buf)
        with pytest.raises(RuntimeError, match=pat):
            call("radial_bwd", buf, consts, buf, 5, R, buf)
        with pytest.raises(RuntimeError, match=pat):
            call("edge_adjust_fwd", buf, buf, 5, R, 64, buf)
        with pytest.raises(RuntimeError, match=pat):
            call("edge_adjust_bwd", buf, buf, buf, 5, R, 64, buf)
        with pytest.raises(RuntimeError, match=pat):
            call("conv_mlp_fwd", buf, 512, 0, ibuf, ibuf, buf, buf, buf, buf, buf, buf, buf, buf, 5, 64, R, 0, buf)
        with pytest.raises(RuntimeError, match=pat):
            call("conv_mlp_bwd", buf, 512, 0, ibuf, ibuf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf,
                 buf, None, 5, 64, R, 0, buf, buf, buf)
    torch.cuda.synchronize()
    assert bool((buf == SENTINEL).all()), "a refused call wrote to a buffer"
    # N = 0 / E = 0: no-ops that leave every buffer untouched
    before = buf.clone()
    call("readout_fwd", buf, *[w[k] for k in RO_FWD], buf, 1.0, 0, 64, buf)
    call("readout_bwd", buf, *[w[k] for k in RO_FWD], *[w[k] for k in RO_BWD], None, None, buf, ibuf, 1.0, 0, 64, buf)
    call("readout_fwd_bwd", buf, *[w[k] for k in RO_FWD], *[w[k] for k in RO_BWD], buf, buf, ibuf, 1.0, 0, 64, buf,
         buf)
    call("structure_sum", buf, ibuf, 0, 1.0, buf, buf)
    call("linear_fwd", buf, buf, buf, 0, 64, 512, buf)
    call("linear_bwd_input", buf, buf, buf, 0, 64, 512, buf)
    call("conv_mlp_fwd", buf, 512, 0, ibuf, ibuf, buf, buf, buf, buf, buf, buf, buf, buf, 0, 64, 3, 0, buf)
    call("conv_mlp_bwd", buf, 512, 0, ibuf, ibuf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf,
         None, 0, 64, 3, 0, buf, buf, buf)
    call("segment_sum_add", buf, buf, ibuf, 0, 64, buf)
    call("conv_gather_gz", buf, ibuf, ibuf, ibuf, 0, 64, 512, 0, buf)
    call("radial_fwd", buf, consts, 0, 3, buf)
    call("radial_bwd", buf, consts, buf, 0, 3, buf)
    call("edge_adjust_fwd", buf, buf, 0, 3, 64, buf)
    call("edge_adjust_bwd", buf, buf, buf, 0, 3, 64, buf)
    call("geometry_fwd", buf, buf, ibuf, ibuf, ibuf, ibuf, 0, buf, buf)
    tri = torch.zeros(2, 0, dtype=torch.int64, device=device)
    call("angles_fwd", buf, tri, 0, buf)
    call("angles_bwd", buf, tri, buf, 0, buf)
    call("geometry_bwd", buf, buf, buf, ibuf, ibuf, ibuf, 0, 1.0, buf)
    call("forces_virial", buf, buf, buf, ibuf, 0, 0, buf, buf)
    torch.cuda.synchronize()
    assert same(buf, before), "a call with N = 0 or E = 0 wrote to a buffer"


# ---------------------------------------------------------------------------------------------------------------------
# negative controls: the check must reject the real kernel output against a plausibly wrong reference
def test_negative_controls(device):
    detected = {}
    # readout (F = 64, SW): the last k term of layer 0 dropped; one column of the dense and gate halves swapped
    c = ReadoutCase(64, 65, device, seed=5)
    a = torch.empty(65, device=device)
    c.fwd(a)
    sc = S.readout_fwd(c.x.abs(), S.absolute(c.w), c.elemental.abs(), c.scale)
    w_drop = dict(c.w, W0d=c.w["W0d"].clone(), W0g=c.w["W0g"].clone())
    w_drop["W0d"][:, -1] = 0.0
    w_drop["W0g"][:, -1] = 0.0
    w_swap = dict(c.w, W0d=c.w["W0d"].clone(), W0g=c.w["W0g"].clone())
    w_swap["W0d"][5], w_swap["W0g"][5] = c.w["W0g"][5], c.w["W0d"][5]
    clean = {"readout_fwd": nerr(a, S.readout_fwd(c.x, c.w, c.elemental, c.scale), sc) / tau(64, 3)}
    detected["readout_fwd: last k term dropped"] = nerr(a, S.readout_fwd(c.x, w_drop, c.elemental, c.scale), sc) / \
        tau(64, 3)
    detected["readout_fwd: dense/gate column swapped"] = nerr(a, S.readout_fwd(c.x, w_swap, c.elemental, c.scale),
                                                              sc) / tau(64, 3)
    # linear_bwd_input at F = 17 (fallback, K = 136 in two chunks): the last k term dropped; the last row missed
    n, K, M = 65, 17, 136
    g = torch.Generator().manual_seed(3)
    gup, W = rand(g, n, M).to(device), rand(g, M, K, scale=M ** -0.5).to(device)
    y = torch.empty(n, K, device=device)
    call("linear_bwd_input", gup, W, None, n, K, M, y)
    sc = S.linear_bwd_input(gup.abs(), W.abs())
    ref = S.linear_bwd_input(gup, W)
    clean["linear_bwd_input"] = nerr(y, ref, sc) / tau(M)
    detected["linear_bwd_input: last k term dropped"] = nerr(y, S.linear_bwd_input(gup[:, :-1], W[:-1]), sc) / tau(M)
    tail = ref.clone()
    tail[-1] = 0.0
    detected["linear_bwd_input: last row of the tail missed"] = nerr(y, tail, sc) / tau(M)
    # conv_mlp_fwd (F = 17, generic): one column of the dense and gate halves of layer 1 swapped
    cc = ConvCase("hubs", 261, 17, 3, device, seed=4)
    yv = torch.empty(261, 17, device=device)
    cc.fwd(0, 1, yv)
    ref, sc = cc.ref_fwd(0, 1)
    w_swap = dict(cc.w, W1e=cc.w["W1e"].clone())
    w_swap["W1e"][[3, 17 + 3]] = cc.w["W1e"][[17 + 3, 3]]
    clean["conv_mlp_fwd"] = nerr(yv, ref, sc) / tau(20, 3)
    detected["conv_mlp_fwd: dense/gate column swapped"] = nerr(yv, cc.ref_fwd(0, 1, w_swap)[0], sc) / tau(20, 3)
    # geometry_bwd: one hub atom's last bond dropped
    gc = GeomCase(1000, device, seed=9)
    vec4, dist = torch.empty(1000, 4, device=device), torch.empty(1000, device=device)
    call("geometry_fwd", gc.pos, gc.lat, gc.batch, gc.src, gc.dst, gc.shift, 1000, vec4, dist)
    gd = rand(g, 1000).to(device)
    gp = torch.empty(gc.N, 3, device=device)
    call("geometry_bwd", vec4, None, gd, *gc.ptrs, gc.N, 1.0, gp)
    sc = S.geometry_bwd(vec4, None, gd, gc.src, gc.dst, gc.N, absolute_=True)
    clean["geometry_bwd"] = nerr(gp, S.geometry_bwd(vec4, None, gd, gc.src, gc.dst, gc.N), sc) / tau(gc.max_bonds)
    last = int(gc.ptrs[0][1]) - 1  # the last bond of atom 0 (129 bonds)
    keep = torch.ones(1000, dtype=torch.bool, device=device)
    keep[last] = False
    drop = S.geometry_bwd(vec4[keep], None, gd[keep], gc.src[:1000][keep], gc.dst[:1000][keep], gc.N)
    detected["geometry_bwd: one atom's last bond dropped"] = nerr(gp, drop, sc) / tau(gc.max_bonds)
    lines = [f"{k:<52}{v:10.1f} x tau" for k, v in detected.items()] + \
        [f"clean {k:<46}{v:10.3f} x tau" for k, v in clean.items()]
    print("\n".join(lines))
    assert all(v <= 1.0 for v in clean.values()), "\n".join(lines)
    missed = [k for k, v in detected.items() if not v > 1.0]
    assert not missed, f"a wrong reference passed the check: {missed}\n" + "\n".join(lines)
