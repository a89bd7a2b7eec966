"""GPU: the tensor-core gated-MLP kernels (m3g_conv_tc_fwd, m3g_conv_tc_bwd_saved, m3g_conv_tc_bwd,
m3g_conv_tc_block_bwd) against the float64 restatement in tests/conv_oracle.py, across tile, schedule and graph shapes.

Accuracy: every output is checked per column (max over rows of |got - ref| <= tau * the column's scale) and per row
(the same with the row's scale), so a wrong column block or gate half cannot hide behind the largest entry of the
tensor.  For outputs that are sums (y in mode 0, g_e, ge2, g_h accumulated onto a prefill) the scale is the larger of
the two float64 terms.  The generic fp32 FMA kernels run on the same inputs as the yardstick of "fp32-faithful".

Error model for tau.  3xTF32 (passes = 3) splits each operand into a TF32 hi part (top 11 significant bits,
truncated) and the remainder read as TF32, and drops lo x lo: per product a relative error below 2^-20 (fp32: 2^-24),
so up to 16x the rounding error of fp32 FMAs.  On well-conditioned inputs fp32 reaches ~1e-6 of the column / row scale
after two GEMM layers and the adjoint, so 3xTF32 stays within 2e-5.  TF32 alone (passes = 1) truncates each operand by
up to 2^-10: ~5e-3 after two layers, 1e-2 at the worst of 10^5 rows.  A missing lo image leaves that TF32 error in one
GEMM, which the 3xTF32 tau must see (the negative controls below).

Weights with rows scaled by powers of two (variant "scaled": 1 row in 8 by 2^-6 .. 2^6) make the outputs
ill-conditioned on purpose: small columns computed from large terms.  There even the fp32 FMA kernels leave up to 4e-4
of the column scale, so the absolute tau does not apply; the tensor cores must instead stay within YARD_FACTOR of the
FMA kernels' error on the same inputs.

Bitwise properties: independence of n_sm and of repeated calls, saving changes nothing, outputs independent of what
the buffers held, guard rows after every input and output stay intact, row isolation and shift invariance, and the
edges of the interface."""
import math

import pytest
import torch

from tests import conv_oracle as C

pytestmark = pytest.mark.gpu

F = 64
# worst normalised error measured on an NVIDIA B200 (1000 W) over this file's well-conditioned cases:
# passes = 3: 1.35e-5 (block_bwd's chained edge phase 2.13e-5 against CHAIN * tau; FMA kernels 5.3e-6);
# passes = 1: 1.22e-2.  A zeroed lo image gives 8.6e-5 to 1.5e-3 (test_negative_controls).
TAU = {3: 2e-5, 1: 2e-2}
# passes = 3 against the FMA kernels on the same inputs: tc error <= YARD_FACTOR * fma error + YARD_FLOOR (the 2^-20
# vs 2^-24 per-product bound, with a factor 2 to spare); measured worst ratio 17.6 where the FMA error exceeds the
# floor (61.7 for bwd_saved0 g_h, whose FMA error is 7.8e-7)
YARD_FACTOR, YARD_FLOOR = 32.0, 1e-6
SCALE_FLOOR = 0.1
# outputs of m3g_conv_tc_block_bwd's edge phase: it consumes ge2, which carries the node phase's rounding error (up to
# tau of its scale), and adds its own, so these are held to CHAIN * tau
CHAINED = {("block_bwd", "g_e"), ("block_bwd", "gz_edge"), ("block_bwd", "gh_edge"), ("block_bwd", "gh_sum")}
CHAIN = 2.0
GUARD = 128  # guard rows after every input and output
SENTINEL = 3.0
SMALL_E = (1, 31, 32, 33, 127, 128, 129, 261)

# (kernel, output, passes) -> worst normalised error; ("fma", kernel, output) -> the FMA kernels' worst error
RESULTS = {}
RATIOS = {}  # (kernel, output) -> worst 3xTF32 / FMA error ratio


@pytest.fixture(scope="module", autouse=True)
def _error_table(request):
    yield
    if not RESULTS:
        return
    lines = ["", "conv tensor-core kernels vs float64: worst normalised error (per column / per row)",
             f"{'kernel':<16}{'output':<10}{'passes':>7}{'worst':>11}{'tau':>9}{'fma':>11}"]
    for (kern, out, passes), v in sorted(RESULTS.items(), key=lambda kv: tuple(map(str, kv[0]))):
        if kern == "fma":
            continue
        fma = RESULTS.get(("fma", kern, out))
        tau = TAU_BLOCK[kern.split()[1]] if kern.startswith("ConvFn") else tau_of(kern, out, passes)
        tau_s = "-" if kern.endswith("*") else f"{tau:.0e}"
        lines.append(f"{kern:<16}{out:<10}{passes:>7}{v:>11.2e}{tau_s:>9}" + (f"{fma:>11.2e}" if fma else ""))
    lines.append("* ill-conditioned inputs (rows scaled by 2^-6 .. 2^6): no tau, within YARD_FACTOR of the FMA kernels")
    lines += [f"3xTF32 / FMA error, worst ratio: {k} {o}: {r:.2f}" for (k, o), r in sorted(RATIOS.items())]
    # printed past pytest's output capture, so that the table shows in every run
    capman = request.config.pluginmanager.getplugin("capturemanager")
    if capman is None:
        print("\n".join(lines))
    else:
        with capman.global_and_fixture_disabled():
            print("\n".join(lines), flush=True)


def _lib():
    from torch_m3gnet_b200 import _lib

    return _lib


def call(name, *args):
    _lib().call(name, *args)


def n_sms(device):
    from torch_m3gnet_b200.nn._functions import sm_count

    return sm_count(device)


def resolve_E(E, device):
    """E given as an int or as "2S", "2S+1", "6S+77": multiples of S*128 bonds, S = number of SMs."""
    if isinstance(E, int):
        return E
    S = n_sms(device)
    k, _, extra = E.partition("S")
    return int(k) * S * 128 + (int(extra) if extra else 0)


def save_floats(E):
    return int(_lib().LIB.load().m3g_conv_tc_save_floats(E))


def same(a, b):
    """bitwise equality (NaN payloads included)"""
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


# ---------------------------------------------------------------------------------------------------------------------
# accuracy check
def nerr(got, ref, scale=None, rows=None, per_row=True):
    """Worst normalised error: max over columns of max_i |got - ref| / column scale, and the same per row.
    ``scale`` (default |ref|) is elementwise; ``rows`` (bool) restricts the check to those rows.  Row and column
    scales are floored at SCALE_FLOOR times the tensor's largest scale: an entry that is a sum of products can be near
    zero by cancellation (a row of g_h, any column when E is small), and its rounding error is set by the products, not
    by the result.  A column at a tenth of the tensor's scale is still held to tau of its own scale."""
    got = got.double().reshape(ref.shape[0], -1)
    ref = ref.reshape(ref.shape[0], -1)
    s = ref.abs() if scale is None else scale.reshape(ref.shape[0], -1)
    if rows is not None:
        got, ref, s = got[rows], ref[rows], s[rows]
    if ref.numel() == 0:
        return 0.0
    if not bool(torch.isfinite(got).all()):
        return math.inf
    err = (got - ref).abs()
    floor = max(SCALE_FLOOR * s.max().item(), 1e-30)
    col = (err.amax(0) / s.amax(0).clamp_min(floor)).max()
    if not per_row:
        return col.item()
    row = (err.amax(1) / s.amax(1).clamp_min(floor)).max()
    return max(col.item(), row.item())


def tau_of(kern, out, passes):
    return TAU[passes] * (CHAIN if (kern.rstrip("*"), out) in CHAINED else 1.0)


class Checks:
    """Collects every failed check of a test so that one run reports all of them."""

    def __init__(self):
        self.failed = []

    def acc(self, kern, out, passes, got, ref, scale=None, rows=None, ctx="", strict=True):
        """strict = False (ill-conditioned inputs): recorded under "<kern>*", finite values required, no tau"""
        v = nerr(got, ref, scale, rows)
        key = (kern if strict else kern + "*", out, passes)
        RESULTS[key] = max(RESULTS.get(key, 0.0), v)
        if not math.isfinite(v):
            self.failed.append(f"{kern} {out} passes={passes} {ctx}: non-finite result")
        elif strict and not v <= tau_of(kern, out, passes):
            self.failed.append(f"{kern} {out} passes={passes} {ctx}: normalised error {v:.3e} > "
                               f"{tau_of(kern, out, passes):.0e}")
        return v

    def fma(self, kern, out, got, ref, scale=None, strict=True):
        v = nerr(got, ref, scale)
        key = ("fma", kern if strict else kern + "*", out)
        RESULTS[key] = max(RESULTS.get(key, 0.0), v)
        return v

    def yard(self, kern, out, v_tc, v_fma, ctx=""):
        RATIOS[(kern, out)] = max(RATIOS.get((kern, out), 0.0), v_tc / max(v_fma, 1e-30))
        if not v_tc <= YARD_FACTOR * v_fma + YARD_FLOOR:
            self.failed.append(f"{kern} {out} {ctx}: 3xTF32 error {v_tc:.3e} vs FMA {v_fma:.3e}")

    def true(self, cond, msg):
        if not cond:
            self.failed.append(msg)

    def done(self):
        assert not self.failed, "\n".join(self.failed[:40]) + (f"\n... {len(self.failed)} in all"
                                                               if len(self.failed) > 40 else "")


def sum_scale(a, b):
    """elementwise scale of a sum a + b: the larger float64 term"""
    return torch.maximum(a.abs(), b.abs())


# ---------------------------------------------------------------------------------------------------------------------
# inputs
def guarded(t, fill=float("nan")):
    """``t`` copied into an allocation with GUARD rows of ``fill`` after it; returns (view of the rows of t, whole)."""
    rows = t.shape[0]
    full = torch.full((rows + GUARD,) + tuple(t.shape[1:]), fill, dtype=t.dtype, device=t.device)
    full[:rows] = t
    return full[:rows], full


def out_buf(shape, device, fill=float("nan")):
    return guarded(torch.full(shape, fill, device=device), SENTINEL)


class Mlp:
    """One gated MLP's weights on the device with the production images (nn/conv.py::_tc_images*)."""

    def __init__(self, w, device):
        from torch_m3gnet_b200.nn.conv import _tc_images, _tc_images_transposed

        self.cpu = w
        d = {k: v.to(device) for k, v in w.items()}
        self.ref = d
        t = C.transposed(w)
        self.W1e, self.W2d, self.W2g = d["W1e"], d["W2d"], d["W2g"]
        self.W1eT, self.W2dT, self.W2gT = (t[k].to(device) for k in ("W1eT", "W2dT", "W2gT"))
        self.b2d, self.b2g = d["b2d"], d["b2g"]
        R = w["WhT"].shape[0]
        self.WhT = guarded(d["WhT"])[0]  # NaN rows after the R rows of Wh^T
        self.Wh = d["WhT"].t().contiguous()
        self.img = _tc_images(self.W1e, self.W2d, self.W2g)
        self.imgT = _tc_images_transposed(self.W1eT, self.W2dT, self.W2gT)
        self.R = R


class Case:
    """Graph, per-atom projections P (N, 8F: edge MLP at column 0, node MLP at 4F), e, h and both MLPs.  Every input
    sits in front of GUARD NaN rows; src / dst guards name atom N, whose P row is NaN."""

    def __init__(self, kind, E, R, device, seed=0, variant="plain"):
        src, dst, N = C.graph(kind, E, seed)
        g = torch.Generator().manual_seed(seed + 101)
        scale = 6.0 if variant == "saturating" else 1.0  # saturating: |z| reaches 30-60
        P = scale * torch.randn(N, 8 * F, generator=g)
        e = scale * torch.randn(E, F, generator=g)
        h = torch.rand(E, R, generator=g)
        tf32 = variant == "tf32"
        if tf32:
            P, e, h = C.tf32_round(P), C.tf32_round(e), C.tf32_round(h)
        scaled = variant == "scaled"
        self.edge = Mlp(C.mlp_weights(R, seed + 1, scaled=scaled, tf32=tf32), device)
        self.node = Mlp(C.mlp_weights(R, seed + 2, scaled=scaled, tf32=tf32), device)
        self.kind, self.E, self.R, self.N, self.device = kind, E, R, N, device
        Pn = torch.cat([P, torch.full((1, 8 * F), float("nan"))])
        self.P = guarded(Pn.to(device))[0]
        self.src = guarded(src.to(torch.int32).to(device), N)[0]
        self.dst = guarded(dst.to(torch.int32).to(device), N)[0]
        self.src64 = src.to(device)
        self.dst64 = dst.to(device)
        self.e = guarded(e.to(device))[0]
        self.h = guarded(h.to(device))[0]
        self.g_up = guarded(torch.randn(E, F, generator=g).to(device))[0]
        gx = torch.cat([torch.randn(N, F, generator=g), torch.full((1, F), float("nan"))])
        self.g_x2 = guarded(gx.to(device))[0]
        self.base = guarded(torch.randn(E, F, generator=g).to(device))[0]
        self.gh_pre = torch.randn(E, R, generator=g).to(device)
        self.Pref = P.to(device)

    def mlp(self, which):
        return self.edge if which == "edge" else self.node

    # float64 references -------------------------------------------------------------------------------------------
    def out_ref(self, which, e_in):
        m = self.mlp(which)
        po = 0 if which == "edge" else 4 * F
        return C.mlp_out(C.z1_of(self.Pref, po, self.src64, self.dst64, e_in, m.ref), self.h[:, :self.R], m.ref)

    def bwd_ref(self, which, e_in, mode, g_up):
        """(g_e, g_z1, g_h, scale of g_h)"""
        po = 0 if which == "edge" else 4 * F
        args = (self.Pref, po, self.src64, self.dst64, e_in, self.h, self.mlp(which).ref,
                g_up[:self.N] if mode == 1 else g_up)
        return C.mlp_bwd(*args, None, mode) + (C.gh_scale(*args, mode),)

    # kernels ------------------------------------------------------------------------------------------------------
    def fwd(self, which, e_in, mode, passes, n_sm, y, save=None, R=None, img=None):
        m = self.mlp(which)
        po = 0 if which == "edge" else 4 * F
        call("conv_tc_fwd", self.P, 8 * F, po, self.src, self.dst, e_in, self.h, m.img if img is None else img,
             m.b2d, m.b2g, m.WhT, self.E, self.R if R is None else R, mode, passes, n_sm, y, save)

    def bwd_saved(self, which, save, mode, g_up, base, passes, n_sm, g_e, g_z1, g_h, gh_store, R=None, imgT=None):
        m = self.mlp(which)
        call("conv_tc_bwd_saved", self.src, self.h, m.imgT if imgT is None else imgT, m.WhT, save, g_up, base,
             self.E, self.R if R is None else R, mode, passes, n_sm, g_e, g_z1, g_h, gh_store)

    def bwd(self, which, e_in, mode, g_up, base, passes, n_sm, g_e, g_z1, g_h, R=None, img=None, imgT=None):
        m = self.mlp(which)
        po = 0 if which == "edge" else 4 * F
        call("conv_tc_bwd", self.P, 8 * F, po, self.src, self.dst, e_in, self.h, m.img if img is None else img,
             m.imgT if imgT is None else imgT, m.b2d, m.b2g, m.WhT, g_up, base, self.E, self.R if R is None else R,
             mode, passes, n_sm, g_e, g_z1, g_h)

    def block(self, save_n, save_e, g_e2, passes, n_sm, g_e, gz_n, gz_e, gh_n, gh_e, gh_mode, R=None, n_imgT=None,
              e_imgT=None):
        call("conv_tc_block_bwd", self.src, self.h, self.node.imgT if n_imgT is None else n_imgT, self.node.WhT,
             save_n, self.edge.imgT if e_imgT is None else e_imgT, self.edge.WhT, save_e, self.g_x2, g_e2, self.E,
             self.R if R is None else R, passes, n_sm, g_e, gz_n, gz_e, gh_n, gh_e, gh_mode)

    def fma_fwd(self, which, e_in, mode, y):
        m = self.mlp(which)
        po = 0 if which == "edge" else 4 * F
        call("conv_mlp_fwd", self.P, 8 * F, po, self.src, self.dst, e_in, self.h, m.W1eT, m.W2dT, m.b2d, m.W2gT,
             m.b2g, m.WhT, self.E, F, self.R, mode, y)

    def fma_bwd(self, which, e_in, mode, g_up, base, g_e, g_z1, g_h):
        m = self.mlp(which)
        po = 0 if which == "edge" else 4 * F
        call("conv_mlp_bwd", self.P, 8 * F, po, self.src, self.dst, e_in, self.h, m.W1eT, m.W2dT, m.b2d, m.W2gT,
             m.b2g, m.WhT, m.W1e, m.W2d, m.W2g, m.Wh, g_up, base, self.E, F, self.R, mode, g_e, g_z1, g_h)

    def new_save(self, fill=float("nan")):
        return guarded(torch.full((save_floats(self.E),), fill, device=self.device), SENTINEL)

    def forward_pair(self, passes, n_sm, node_mode=2):
        """edge forward (mode 0) and node forward on its output, both saving: (e2, y_node, save_e, save_n)"""
        e2, _ = out_buf((self.E, F), self.device)
        yn, _ = out_buf((self.E, F), self.device)
        save_e, _ = self.new_save()
        save_n, _ = self.new_save()
        self.fwd("edge", self.e, 0, passes, n_sm, e2, save_e)
        e2g = guarded(e2.clone())[0]
        self.fwd("node", e2g, node_mode, passes, n_sm, yn, save_n)
        return e2g, yn, save_e, save_n


def nan(shape, device):
    return out_buf(shape, device)[0]


# ---------------------------------------------------------------------------------------------------------------------
# forward accuracy
def _fwd_accuracy(device, kind, E, Rs, variant="plain"):
    ck = Checks()
    S = n_sms(device)
    strict = variant != "scaled"
    for R in Rs:
        c = Case(kind, E, R, device, seed=E + 7 * R, variant=variant)
        out = c.out_ref("edge", c.e)
        ref = {0: c.e.double() + out, 1: out}
        ref[2], mask = C.group_rows(out, c.src64)
        scale = {0: sum_scale(c.e.double(), out), 1: None, 2: None}
        fma_err = {}
        for mode in (0, 1):
            y = nan((E, F), device)
            c.fma_fwd("edge", c.e, mode, y)
            fma_err[mode] = ck.fma("fwd", f"y{mode}", y, ref[mode], scale[mode], strict)
        for passes in (1, 3):
            for mode in (0, 1, 2):
                y0 = nan((E, F), device)
                c.fwd("edge", c.e, mode, passes, S, y0)
                y1 = nan((E, F), device)
                save, _ = c.new_save()
                c.fwd("edge", c.e, mode, passes, S, y1, save)
                ctx = f"{kind} E={E} R={R} {variant}"
                ck.true(same(y0, y1), f"save changes y (mode {mode} passes {passes} {ctx})")
                rows = mask if mode == 2 else None
                v = ck.acc("fwd", f"y{mode}", passes, y1, ref[mode], scale[mode], rows, ctx, strict)
                if passes == 3 and mode in fma_err:
                    ck.yard("fwd", f"y{mode}", v, fma_err[mode], ctx)
                if mode == 2:
                    ck.true(bool(torch.isnan(y1[~mask]).all()), f"mode 2 wrote a non-partial row ({ctx})")
    ck.done()


@pytest.mark.parametrize("E", SMALL_E)
@pytest.mark.parametrize("kind", C.GRAPH_KINDS)
def test_fwd_accuracy_small(device, kind, E):
    _fwd_accuracy(device, kind, E, (1, 2, 3, 4))


@pytest.mark.parametrize("kind,E,variant", [
    ("poisson", 1380, "plain"), ("hubs", 1380, "plain"), ("deg32", 1380, "scaled"), ("poisson", 261, "scaled"),
    ("poisson", 1380, "saturating"), ("poisson", 261, "tf32"), ("poisson", 1380, "tf32"),
    ("poisson", "2S", "plain"), ("single", "2S+1", "plain"), ("hubs", "6S+77", "plain"),
    ("one_atom", "6S+77", "plain"), ("deg33", "2S+1", "saturating"), ("self", "6S+77", "scaled"),
])
def test_fwd_accuracy_large(device, kind, E, variant):
    _fwd_accuracy(device, kind, resolve_E(E, device), (1, 3, 4), variant)


# ---------------------------------------------------------------------------------------------------------------------
# backward accuracy, on the activations a real forward saved
def _bwd_accuracy(device, kind, E, Rs, variant="plain", full=True):
    ck = Checks()
    S = n_sms(device)
    strict = variant != "scaled"
    for R in Rs:
        c = Case(kind, E, R, device, seed=3 * E + R, variant=variant)
        base = c.base.double()
        pre = c.gh_pre.double()
        for passes in (1, 3):
            ctx = f"{kind} E={E} R={R} {variant}"
            e2, _, save_e, save_n = c.forward_pair(passes, S)
            refs = {"edge": c.bwd_ref("edge", c.e, 0, c.g_up), "node": c.bwd_ref("node", e2, 1, c.g_x2)}
            ups = {"edge": c.g_up, "node": c.g_x2}
            ins = {"edge": c.e, "node": e2}
            saves = {"edge": save_e, "node": save_n}
            for which, mode in (("edge", 0), ("node", 1)):
                r_ge, r_gz, r_gh, s_gh = refs[which]
                k = f"bwd_saved{mode}"
                fma_err = None
                if passes == 3:  # the FMA yardstick, on the same inputs (with a base and a g_h prefill)
                    g_e, g_z1, g_h = nan((E, F), device), nan((E, 2 * F), device), c.gh_pre.clone()
                    c.fma_bwd(which, ins[which], mode, ups[which], c.base, g_e, g_z1, g_h)
                    fma_err = (ck.fma(k, "g_e", g_e, r_ge + base, sum_scale(r_ge, base), strict),
                               ck.fma(k, "g_z1", g_z1, r_gz, None, strict),
                               ck.fma(k, "g_h", g_h, r_gh + pre, sum_scale(s_gh, pre), strict))
                combos = [(b, z, s) for b in (False, True) for z in (False, True) for s in (0, 1)] if full else \
                    [(True, True, 0), (False, False, 1)]
                for with_base, with_gz, gh_store in combos:
                    g_e, g_z1 = nan((E, F), device), nan((E, 2 * F), device) if with_gz else None
                    g_h = nan((E, R), device) if gh_store else guarded(c.gh_pre.clone(), SENTINEL)[0]
                    c.bwd_saved(which, saves[which], mode, ups[which], c.base if with_base else None, passes, S, g_e,
                                g_z1, g_h, gh_store)
                    sub = f"{ctx} base={with_base} gz={with_gz} gh_store={gh_store}"
                    v_e = ck.acc(k, "g_e", passes, g_e, r_ge + base if with_base else r_ge,
                                 sum_scale(r_ge, base) if with_base else None, ctx=sub, strict=strict)
                    v_z = ck.acc(k, "g_z1", passes, g_z1, r_gz, ctx=sub, strict=strict) if with_gz else 0.0
                    if gh_store:
                        v_h = ck.acc(k, "g_h", passes, g_h, r_gh, s_gh, ctx=sub, strict=strict)
                    else:
                        v_h = ck.acc(k, "g_h", passes, g_h, r_gh + pre, sum_scale(s_gh, pre), ctx=sub, strict=strict)
                    if fma_err is not None and with_base and with_gz and not gh_store:
                        for nm, v, vf in zip(("g_e", "g_z1", "g_h"), (v_e, v_z, v_h), fma_err):
                            ck.yard(k, nm, v, vf, sub)
                # forward recomputed inside the backward
                k = f"bwd{mode}"
                for with_base in ((False, True) if full else (True,)):
                    g_e, g_z1, g_h = nan((E, F), device), nan((E, 2 * F), device), guarded(c.gh_pre.clone())[0]
                    c.bwd(which, ins[which], mode, ups[which], c.base if with_base else None, passes, S, g_e, g_z1, g_h)
                    sub = f"{ctx} base={with_base}"
                    ck.acc(k, "g_e", passes, g_e, r_ge + base if with_base else r_ge,
                           sum_scale(r_ge, base) if with_base else None, ctx=sub, strict=strict)
                    ck.acc(k, "g_z1", passes, g_z1, r_gz, ctx=sub, strict=strict)
                    ck.acc(k, "g_h", passes, g_h, r_gh + pre, sum_scale(s_gh, pre), ctx=sub, strict=strict)
            # the fused block backward
            for with_e2 in ((False, True) if full else (True,)):
                g_e2 = c.base if with_e2 else None
                ge2, r_ge, r_gzn, r_gze, r_ghn, r_ghe = C.block_bwd(
                    c.Pref, c.src64, c.dst64, c.e, e2, c.h, c.edge.ref, c.node.ref, c.g_x2[:c.N], g_e2)
                s_ghn = refs["node"][3]
                s_ghe = C.gh_scale(c.Pref, 0, c.src64, c.dst64, c.e, c.h, c.edge.ref, ge2, 0)
                node_adj = ge2 - base if with_e2 else ge2
                # g_e = ge2 + edge adjoint, ge2 = g_e2 + node adjoint: scale by the largest of the three terms
                g_e_scale = torch.maximum(sum_scale(ge2, r_ge - ge2), node_adj.abs())
                if with_e2:
                    g_e_scale = torch.maximum(g_e_scale, base.abs())
                for with_gz in ((False, True) if full else (True,)):
                    for gh_mode in (0, 1):
                        g_e = nan((E, F), device)
                        gz_n = nan((E, 2 * F), device) if with_gz else None
                        gz_e = nan((E, 2 * F), device) if with_gz else None
                        gh_n = nan((E, R), device)
                        gh_e = nan((E, R), device) if gh_mode == 0 else None
                        c.block(save_n, save_e, g_e2, passes, S, g_e, gz_n, gz_e, gh_n, gh_e, gh_mode)
                        sub = f"{ctx} g_e2={with_e2} gz={with_gz} gh_mode={gh_mode}"
                        ck.acc("block_bwd", "g_e", passes, g_e, r_ge, g_e_scale, ctx=sub, strict=strict)
                        if with_gz:
                            ck.acc("block_bwd", "gz_node", passes, gz_n, r_gzn, ctx=sub, strict=strict)
                            ck.acc("block_bwd", "gz_edge", passes, gz_e, r_gze, ctx=sub, strict=strict)
                        if gh_mode == 0:
                            ck.acc("block_bwd", "gh_node", passes, gh_n, r_ghn, s_ghn, ctx=sub, strict=strict)
                            ck.acc("block_bwd", "gh_edge", passes, gh_e, r_ghe, s_ghe, ctx=sub, strict=strict)
                        else:
                            ck.acc("block_bwd", "gh_sum", passes, gh_n, r_ghn + r_ghe, sum_scale(s_ghn, s_ghe),
                                   ctx=sub, strict=strict)
    ck.done()


@pytest.mark.parametrize("E", SMALL_E)
@pytest.mark.parametrize("kind", C.GRAPH_KINDS)
def test_bwd_accuracy_small(device, kind, E):
    _bwd_accuracy(device, kind, E, (1, 2, 3))


@pytest.mark.parametrize("kind,E,variant", [
    ("poisson", 1380, "plain"), ("hubs", 1380, "plain"), ("poisson", 1380, "saturating"),
    ("poisson", 1380, "tf32"), ("deg32", 1380, "scaled"), ("poisson", "2S", "plain"), ("deg31", "2S+1", "plain"),
    ("one_atom", "6S+77", "plain"), ("self", "6S+77", "plain"), ("hubs", "6S+77", "scaled"),
])
def test_bwd_accuracy_large(device, kind, E, variant):
    _bwd_accuracy(device, kind, resolve_E(E, device), (1, 3), variant, full=False)


# ---------------------------------------------------------------------------------------------------------------------
# bitwise properties
def _run_all(c, n_sm, passes=3):
    """Every kernel once on one case; returns {name: output tensor} (all outputs cloned)."""
    dev, E, R = c.device, c.E, c.R
    out = {}
    for mode in (0, 1, 2):
        y = nan((E, F), dev)
        save, _ = c.new_save()
        c.fwd("edge", c.e, mode, passes, n_sm, y, save)
        out[f"fwd{mode}.y"], out[f"fwd{mode}.save"] = y.clone(), save.clone()
    e2, _, save_e, save_n = c.forward_pair(passes, n_sm)
    for which, mode, save, g_up, e_in in (("edge", 0, save_e, c.g_up, c.e), ("node", 1, save_n, c.g_x2, e2)):
        g_e, g_z1, g_h = nan((E, F), dev), nan((E, 2 * F), dev), guarded(c.gh_pre.clone())[0]
        c.bwd_saved(which, save, mode, g_up, c.base, passes, n_sm, g_e, g_z1, g_h, 0)
        out.update({f"bwds{mode}.g_e": g_e, f"bwds{mode}.g_z1": g_z1, f"bwds{mode}.g_h": g_h})
        g_e, g_z1, g_h = nan((E, F), dev), nan((E, 2 * F), dev), guarded(c.gh_pre.clone())[0]
        c.bwd(which, e_in, mode, g_up, c.base, passes, n_sm, g_e, g_z1, g_h)
        out.update({f"bwd{mode}.g_e": g_e, f"bwd{mode}.g_z1": g_z1, f"bwd{mode}.g_h": g_h})
    for gh_mode in (0, 1):
        g_e, gz_n, gz_e, gh_n = nan((E, F), dev), nan((E, 2 * F), dev), nan((E, 2 * F), dev), nan((E, R), dev)
        gh_e = nan((E, R), dev) if gh_mode == 0 else None
        c.block(save_n, save_e, c.base, passes, n_sm, g_e, gz_n, gz_e, gh_n, gh_e, gh_mode)
        out.update({f"block{gh_mode}.g_e": g_e, f"block{gh_mode}.gz_n": gz_n, f"block{gh_mode}.gz_e": gz_e,
                    f"block{gh_mode}.gh_n": gh_n})
        if gh_e is not None:
            out[f"block{gh_mode}.gh_e"] = gh_e
    return out


@pytest.mark.parametrize("kind,E", [("poisson", 261), ("hubs", "2S+1"), ("one_atom", "6S+77")])
@pytest.mark.parametrize("passes", [1, 3])
def test_schedule_independence(device, kind, E, passes):
    """n_sm = 1 makes one CTA walk every tile (many barrier parity flips); 2, 3 and S change which CTA and which warp
    group takes a tile.  Outputs are bitwise equal, and so are repeated calls."""
    E = resolve_E(E, device)
    S = n_sms(device)
    c = Case(kind, E, 3, device, seed=E)
    want = _run_all(c, S, passes)
    ck = Checks()
    for n_sm in (1, 2, 3, S):
        got = _run_all(c, n_sm, passes)
        for k in want:
            ck.true(same(got[k], want[k]), f"{k} differs with n_sm={n_sm} (E={E})")
    ck.done()


def _guard_ok(full, rows, fill):
    g = full[rows:]
    if math.isnan(fill):
        return bool(torch.isnan(g).all())
    return bool((g == fill).all())


@pytest.mark.parametrize("E", [1, 33, 129, 261, "2S+1"])
def test_buffers_and_guards(device, E):
    """Outputs do not depend on what their buffers held (except accumulated g_h); mode 2 leaves non-partial rows
    alone; guard rows after every input (NaN, or an atom with a NaN row for src / dst) and every output (sentinel)
    stay intact, and no NaN reaches a result."""
    E = resolve_E(E, device)
    S = n_sms(device)
    ck = Checks()
    c = Case("poisson", E, 3, device, seed=E + 5)
    mask = C.partial_rows(c.src64)

    def run(fill):
        res = {}
        bufs = {}

        def buf(name, shape):
            v, full = guarded(torch.full(shape, fill, device=device), SENTINEL)
            bufs[name] = (full, shape[0])
            return v

        for mode in (0, 1, 2):
            y = buf(f"y{mode}", (E, F))
            sv, svf = guarded(torch.full((save_floats(E),), fill, device=device), SENTINEL)
            bufs[f"save{mode}"] = (svf, save_floats(E))
            c.fwd("edge", c.e, mode, 3, S, y, sv)
            res[f"y{mode}"], res[f"save{mode}"] = y, sv
        e2 = guarded(res["y0"].clone())[0]
        save_e = guarded(res["save0"].clone())[0]
        save_n = guarded(torch.empty_like(res["save0"]))[0]
        c.fwd("node", e2, 2, 3, S, buf("y_node", (E, F)), save_n)
        for which, mode, save, g_up, e_in in (("edge", 0, save_e, c.g_up, c.e), ("node", 1, save_n, c.g_x2, e2)):
            for gh_store in (0, 1):
                g_e, g_z1 = buf(f"bs{mode}{gh_store}.g_e", (E, F)), buf(f"bs{mode}{gh_store}.g_z1", (E, 2 * F))
                if gh_store:
                    g_h = buf(f"bs{mode}1.g_h", (E, c.R))
                else:
                    g_h, ghf = guarded(c.gh_pre.clone(), SENTINEL)
                    bufs[f"bs{mode}0.g_h"] = (ghf, E)
                c.bwd_saved(which, save, mode, g_up, c.base, 3, S, g_e, g_z1, g_h, gh_store)
                res.update({f"bs{mode}{gh_store}.g_e": g_e, f"bs{mode}{gh_store}.g_z1": g_z1,
                            f"bs{mode}{gh_store}.g_h": g_h})
            g_e, g_z1 = buf(f"b{mode}.g_e", (E, F)), buf(f"b{mode}.g_z1", (E, 2 * F))
            g_h, ghf = guarded(c.gh_pre.clone(), SENTINEL)
            bufs[f"b{mode}.g_h"] = (ghf, E)
            c.bwd(which, e_in, mode, g_up, c.base, 3, S, g_e, g_z1, g_h)
            res.update({f"b{mode}.g_e": g_e, f"b{mode}.g_z1": g_z1, f"b{mode}.g_h": g_h})
        for gh_mode in (0, 1):
            p = f"blk{gh_mode}."
            outs = [buf(p + "g_e", (E, F)), buf(p + "gz_n", (E, 2 * F)), buf(p + "gz_e", (E, 2 * F)),
                    buf(p + "gh_n", (E, c.R)), buf(p + "gh_e", (E, c.R)) if gh_mode == 0 else None]
            c.block(save_n, save_e, None, 3, S, *outs, gh_mode)
            for nm, t in zip(("g_e", "gz_n", "gz_e", "gh_n", "gh_e"), outs):
                if t is not None:
                    res[p + nm] = t
        torch.cuda.synchronize()
        for name, (full, rows) in bufs.items():
            ck.true(_guard_ok(full, rows, SENTINEL), f"guard after {name} overwritten (E={E})")
        return res

    a = run(float("nan"))
    b = run(SENTINEL)
    for k in a:
        if k == "y2":
            ck.true(same(a[k][mask], b[k][mask]), "y2 partial rows depend on the buffer")
            ck.true(bool(torch.isnan(a[k][~mask]).all()) and bool((b[k][~mask] == SENTINEL).all()),
                    "mode 2 wrote a row that is not a partial row")
            ck.true(bool(torch.isfinite(a[k][mask]).all()), "NaN in the mode-2 partial rows")
            continue
        ck.true(same(a[k], b[k]), f"{k} depends on what its buffer held (E={E})")
        ck.true(bool(torch.isfinite(a[k]).all()), f"{k}: NaN or Inf in the result (E={E})")
    ck.done()


@pytest.mark.parametrize("kind,E", [("poisson", 261), ("deg33", 1380), ("hubs", "2S+1")])
def test_row_isolation_and_shift(device, kind, E):
    """A NaN in one bond's e or h, or in one atom's g_x2 row, changes only that bond's / atom's rows; shifting the bonds
    down by 1, 31, 32 or 128 rows leaves their rows bitwise unchanged (modes 0 and 1 and the backwards)."""
    E = resolve_E(E, device)
    S = n_sms(device)
    ck = Checks()
    c = Case(kind, E, 3, device, seed=E + 11)
    clean = _run_all(c, S)
    k = E // 2
    atom = int(c.src64[k])
    bond_rows = torch.zeros(E, dtype=torch.bool, device=device)
    bond_rows[k] = True
    atom_rows = c.src64 == atom
    part_rows = C.group_rows(torch.zeros(E, 1, device=device), c.src64)[1]
    run_of = torch.cumsum(part_rows.long(), 0) - 1
    k_run = run_of == run_of[k]
    for what in ("e", "h", "g_x2"):
        t = getattr(c, what)
        old = t.clone()
        if what == "g_x2":
            t[atom] = float("nan")
        else:
            t[k] = float("nan")
        got = _run_all(c, S)
        t.copy_(old)
        for name, v in got.items():
            if ".save" in name:
                continue
            if what == "g_x2":
                if name.startswith("fwd") or name.startswith(("bwds0", "bwd0")):
                    rows = torch.zeros_like(atom_rows)
                else:
                    rows = atom_rows
            elif name == "fwd2.y":
                rows = k_run
            else:
                rows = bond_rows
            keep = ~rows
            if name == "fwd2.y":
                keep = keep & part_rows
            ck.true(same(v[keep], clean[name][keep]), f"NaN in {what} changed rows of {name} outside its own")
    for s in (1, 31, 32, 128):
        sh = _shifted(c, s)
        got = _run_all(sh, S)
        for name, v in got.items():
            if ".save" in name or name == "fwd2.y":
                continue
            ck.true(same(v[s:], clean[name]), f"{name} changes when the bonds move down by {s} rows")
    ck.done()


def _shifted(c, s):
    """The same case with s extra bonds of a new atom 0 in front (all atoms renumbered +1)."""
    sh = object.__new__(Case)
    sh.__dict__.update(c.__dict__)
    dev = c.device
    g = torch.Generator().manual_seed(s)
    N = c.N + 1
    sh.N, sh.E = N, c.E + s
    P = torch.cat([torch.randn(1, 8 * F, generator=g).to(dev), c.Pref])
    sh.Pref = P
    sh.P = guarded(torch.cat([P, torch.full((1, 8 * F), float("nan"), device=dev)]))[0]
    src = torch.cat([torch.zeros(s, dtype=torch.long, device=dev), c.src64 + 1])
    dst = torch.cat([torch.zeros(s, dtype=torch.long, device=dev), c.dst64 + 1])
    sh.src64, sh.dst64 = src, dst
    sh.src = guarded(src.to(torch.int32), N)[0]
    sh.dst = guarded(dst.to(torch.int32), N)[0]

    def pre(t, rows):
        return guarded(torch.cat([torch.randn((rows,) + tuple(t.shape[1:]), generator=g).to(dev), t[:t.shape[0]]]))[0]

    sh.e, sh.h, sh.g_up, sh.base = pre(c.e, s), pre(c.h, s).abs(), pre(c.g_up, s), pre(c.base, s)
    sh.g_x2 = guarded(torch.cat([torch.randn(1, F, generator=g).to(dev), c.g_x2[:c.N + 1]]))[0]
    sh.gh_pre = torch.cat([torch.randn(s, c.R, generator=g).to(dev), c.gh_pre])
    return sh


def test_interface_edges(device):
    """E = 0 writes nothing; R = 5 (forward), R = 4 (backwards), passes = 2 and gh_mode = 2 are refused."""
    S = n_sms(device)
    c = Case("poisson", 261, 3, device, seed=1)
    c4 = Case("poisson", 261, 4, device, seed=1)
    dev, E = device, c.E
    bufs = [torch.full((E, 2 * F), SENTINEL, device=dev) for _ in range(6)]
    y, g_e, g_z1, gz_e, g_h, g_h2 = bufs
    save, _ = c.new_save()
    e2, _, save_e, save_n = c.forward_pair(3, S)
    before = [b.clone() for b in bufs]
    c.E = c4.E = 0
    try:
        c.fwd("edge", c.e, 0, 3, S, y, save)
        c.bwd_saved("edge", save_e, 0, c.g_up, c.base, 3, S, g_e, g_z1, g_h, 0)
        c.bwd("edge", c.e, 0, c.g_up, c.base, 3, S, g_e, g_z1, g_h)
        c.block(save_n, save_e, c.base, 3, S, g_e, g_z1, gz_e, g_h, g_h2, 0)
    finally:
        c.E = c4.E = E
    torch.cuda.synchronize()
    assert all(same(a, b) for a, b in zip(bufs, before)), "a call with E = 0 wrote to an output"
    R5 = guarded(torch.randn(5, F, device=dev))[0]
    h5 = guarded(torch.rand(E, 5, device=dev))[0]
    with pytest.raises(RuntimeError, match="R=5"):
        call("conv_tc_fwd", c.P, 8 * F, 0, c.src, c.dst, c.e, h5, c.edge.img, c.edge.b2d, c.edge.b2g, R5, E, 5, 0, 3,
             S, y, None)
    with pytest.raises(RuntimeError, match="R=4"):
        c4.bwd_saved("edge", save_e, 0, c4.g_up, None, 3, S, g_e, None, g_h, 1)
    with pytest.raises(RuntimeError, match="R=4"):
        c4.bwd("edge", c4.e, 0, c4.g_up, None, 3, S, g_e, g_z1, g_h)
    with pytest.raises(RuntimeError, match="R=4"):
        c4.block(save_n, save_e, None, 3, S, g_e, None, None, g_h, g_h2, 0)
    for fn in (lambda: c.fwd("edge", c.e, 0, 2, S, y, None),
               lambda: c.bwd_saved("edge", save_e, 0, c.g_up, None, 2, S, g_e, None, g_h, 1),
               lambda: c.bwd("edge", c.e, 0, c.g_up, None, 2, S, g_e, g_z1, g_h),
               lambda: c.block(save_n, save_e, None, 2, S, g_e, None, None, g_h, g_h2, 0)):
        with pytest.raises(RuntimeError, match="passes"):
            fn()
    with pytest.raises(RuntimeError, match="gh_mode"):
        c.block(save_n, save_e, None, 3, S, g_e, None, None, g_h, g_h2, 2)


# ---------------------------------------------------------------------------------------------------------------------
# negative controls: a missing lo image (plain TF32 in one GEMM) must fail the 3xTF32 accuracy check
FWD_LO = {"W1e": (8192, 16384), "W2d": (20480, 24576), "W2g": (28672, 32768)}
BWD_LO = {name: (i * 8192 + 4096, (i + 1) * 8192) for i, name in enumerate(("W2d^T", "W2g^T", "W1e_dense^T",
                                                                           "W1e_gate^T"))}


def _zero_lo(img, span):
    img = img.clone()
    img[span[0]:span[1]] = 0.0
    return img


def test_negative_controls(device):
    S = n_sms(device)
    c = Case("poisson", 1380, 3, device, seed=99)
    e2, _, save_e, save_n = c.forward_pair(3, S)
    detected = {}
    # forward (mode 1: no residual to dilute the scale)
    ref = c.out_ref("edge", c.e)
    y = nan((c.E, F), device)
    c.fwd("edge", c.e, 1, 3, S, y)
    clean = {"fwd": nerr(y, ref)}
    for name, span in FWD_LO.items():
        y = nan((c.E, F), device)
        c.fwd("edge", c.e, 1, 3, S, y, img=_zero_lo(c.edge.img, span))
        detected[f"fwd {name}"] = nerr(y, ref)
    # backwards
    r_ge, r_gz, r_gh, s_gh = c.bwd_ref("edge", c.e, 0, c.g_up)

    def worst(g_e, g_z1, g_h):
        return max(nerr(g_e, r_ge), nerr(g_z1, r_gz), nerr(g_h, r_gh, s_gh))

    g_e, g_z1, g_h = nan((c.E, F), device), nan((c.E, 2 * F), device), nan((c.E, 3), device)
    c.bwd_saved("edge", save_e, 0, c.g_up, None, 3, S, g_e, g_z1, g_h, 1)
    clean["bwd_saved"] = worst(g_e, g_z1, g_h)
    g_e, g_z1, g_h = nan((c.E, F), device), nan((c.E, 2 * F), device), torch.zeros((c.E, 3), device=device)
    c.bwd("edge", c.e, 0, c.g_up, None, 3, S, g_e, g_z1, g_h)
    clean["bwd"] = worst(g_e, g_z1, g_h)

    for name, span in BWD_LO.items():
        g_e, g_z1, g_h = nan((c.E, F), device), nan((c.E, 2 * F), device), nan((c.E, 3), device)
        c.bwd_saved("edge", save_e, 0, c.g_up, None, 3, S, g_e, g_z1, g_h, 1, imgT=_zero_lo(c.edge.imgT, span))
        detected[f"bwd_saved {name}"] = worst(g_e, g_z1, g_h)
        g_e, g_z1, g_h = nan((c.E, F), device), nan((c.E, 2 * F), device), torch.zeros((c.E, 3), device=device)
        c.bwd("edge", c.e, 0, c.g_up, None, 3, S, g_e, g_z1, g_h, imgT=_zero_lo(c.edge.imgT, span))
        detected[f"bwd {name}"] = worst(g_e, g_z1, g_h)
    for name, span in FWD_LO.items():
        g_e, g_z1, g_h = nan((c.E, F), device), nan((c.E, 2 * F), device), torch.zeros((c.E, 3), device=device)
        c.bwd("edge", c.e, 0, c.g_up, None, 3, S, g_e, g_z1, g_h, img=_zero_lo(c.edge.img, span))
        detected[f"bwd (recomputed forward) {name}"] = worst(g_e, g_z1, g_h)
    ge2, b_ge, b_gzn, b_gze, b_ghn, b_ghe = C.block_bwd(c.Pref, c.src64, c.dst64, c.e, e2, c.h, c.edge.ref, c.node.ref,
                                                        c.g_x2[:c.N], None)
    b_scales = (None, None, None, c.bwd_ref("node", e2, 1, c.g_x2)[3],
                C.gh_scale(c.Pref, 0, c.src64, c.dst64, c.e, c.h, c.edge.ref, ge2, 0))

    def worst_block(outs):
        """worst error in units of TAU[3]: each output normalised by its own tau (CHAIN * tau for the edge phase)"""
        names = ("g_e", "gz_node", "gz_edge", "gh_node", "gh_edge")
        return max(nerr(o, r, s) * TAU[3] / tau_of("block_bwd", n, 3)
                   for o, r, s, n in zip(outs, (b_ge, b_gzn, b_gze, b_ghn, b_ghe), b_scales, names))

    outs = [nan((c.E, F), device), nan((c.E, 2 * F), device), nan((c.E, 2 * F), device), nan((c.E, 3), device),
            nan((c.E, 3), device)]
    c.block(save_n, save_e, None, 3, S, *outs, 0)
    clean["block_bwd"] = worst_block(outs)
    for side in ("node", "edge"):
        for name, span in BWD_LO.items():
            outs = [nan((c.E, F), device), nan((c.E, 2 * F), device), nan((c.E, 2 * F), device),
                    nan((c.E, 3), device), nan((c.E, 3), device)]
            imgs = {"n_imgT": c.node.imgT, "e_imgT": c.edge.imgT}
            key = "n_imgT" if side == "node" else "e_imgT"
            imgs[key] = _zero_lo(imgs[key], span)
            c.block(save_n, save_e, None, 3, S, *outs, 0, **imgs)
            detected[f"block_bwd {side} {name}"] = worst_block(outs)
    lines = [f"{k:<40}{v:10.2e}" for k, v in detected.items()] + [f"clean {k:<34}{v:10.2e}" for k, v in clean.items()]
    print("\n".join(lines))
    # the unperturbed kernels pass on the same inputs, so the check itself separates the split from plain TF32
    assert all(v <= TAU[3] for v in clean.values()), "\n".join(lines)
    missed = [k for k, v in detected.items() if not v > TAU[3]]
    assert not missed, f"a zeroed lo image passed the 3xTF32 check: {missed}\n" + "\n".join(lines)


# ---------------------------------------------------------------------------------------------------------------------
# the whole block through ConvFn against oracle.conv in float64
# Per-column check only (x2 sums up to E messages per atom and g_h both MLPs' terms, so single rows can cancel); the
# FMA path and tc3 at the 3xTF32 tau, tc3 also within YARD_FACTOR of the FMA path.  Worst measured on an NVIDIA B200
# (1000 W): fma 4.3e-6, tc3 1.05e-5, tc1 8.0e-3
TAU_BLOCK = {"tc3": 2e-5, "fma": 2e-5, "tc1": 2e-2}
CONFIGS = [  # (CONV_PATH, TC_BWD_VARIANT, MSG_REDUCE, CONV_BWD_FUSED)
    ("fma", 4, True, True),
    ("tc3", 4, True, True), ("tc3", 4, True, False), ("tc3", 4, False, True), ("tc3", 4, False, False),
    ("tc3", 2, True, True), ("tc3", 2, False, True),
    ("tc1", 4, True, True), ("tc1", 4, False, False), ("tc1", 2, True, True),
]


def _batch(src, dst, N, device):
    from torch_m3gnet_b200.data.material_graph import Batch

    E = src.numel()
    b = Batch(pos=torch.rand(N, 3, device=device), atom_types=torch.zeros(N, dtype=torch.long, device=device),
              num_triplet_i=torch.zeros(N, dtype=torch.long, device=device),
              edge_index=torch.stack([src, dst]).to(device),
              edge_cell_shift=torch.zeros(E, 3, device=device),
              num_triplet_ij=torch.zeros(E, dtype=torch.long, device=device),
              triplet_edge_index=torch.zeros(2, 0, dtype=torch.long, device=device),
              lattice=(10.0 * torch.eye(3, device=device))[None])
    b["batch"] = torch.zeros(N, dtype=torch.long, device=device)
    return b


@pytest.mark.parametrize("kind,E", [("poisson", 1380), ("hubs", 1380), ("one_atom", 261), ("deg33", 700),
                                    ("self", 1380), ("single", 300), ("poisson", "2S+1")])
def test_conv_block_against_oracle(device, kind, E):
    from oracle import m3gnet_oracle as O
    from torch_m3gnet_b200.data.material_graph import get_plan
    from torch_m3gnet_b200.nn import conv as conv_mod
    from torch_m3gnet_b200.nn.conv import M3GNetConv

    E = resolve_E(E, device)
    big = E > 10000
    src, dst, N = C.graph(kind, E, seed=E)
    ck = Checks()
    old = (conv_mod.CONV_PATH, conv_mod.TC_BWD_VARIANT, conv_mod.MSG_REDUCE, conv_mod.CONV_BWD_FUSED)
    try:
        for R in ((3,) if big else (1, 2, 3, 4)):
            torch.manual_seed(E + R)
            cv = M3GNetConv(R, F, F, device=device)
            with torch.no_grad():
                for name, prm in cv.named_parameters():  # nonzero biases, activations of order one
                    prm.copy_(torch.randn_like(prm) * (0.5 if name.endswith("bias") else 1.0 / math.sqrt(prm.shape[-1])))
            p = {"c." + k: v.detach().double() for k, v in cv.state_dict().items()}
            g = torch.Generator().manual_seed(R)
            x = torch.randn(N, F, generator=g).to(device)
            e = torch.randn(E, F, generator=g).to(device)
            h = torch.rand(E, R, generator=g).to(device)
            gx2 = torch.randn(N, F, generator=g).to(device)
            ge2 = torch.randn(E, F, generator=g).to(device)
            ei = torch.stack([src, dst]).to(device)
            x64, e64, h64 = (t.double().requires_grad_(True) for t in (x, e, h))
            rx, re = O.conv(p, "c", x64, e64, h64, ei)
            refs = {}
            for loss in ("x2", "e2", "both"):
                outs = [o for o, k in ((rx, "x2"), (re, "e2")) if loss in (k, "both")]
                gos = [go.double() for go, k in ((gx2, "x2"), (ge2, "e2")) if loss in (k, "both")]
                refs[loss] = torch.autograd.grad(outs, (x64, e64, h64), gos, retain_graph=True)
            b = _batch(src, dst, N, device)
            get_plan(b)
            fma = {}
            for path, bwd, reduce, fused in (CONFIGS[:2] if big else CONFIGS):
                conv_mod.CONV_PATH, conv_mod.TC_BWD_VARIANT = path, bwd
                conv_mod.MSG_REDUCE, conv_mod.CONV_BWD_FUSED = reduce, fused
                tau = TAU_BLOCK[path]
                for loss in ("x2", "e2", "both"):
                    b["x"], b["edge_attr"], b["edge_weights"] = (t.clone().requires_grad_(True) for t in (x, e, h))
                    ins = (b["x"], b["edge_attr"], b["edge_weights"])
                    out = cv(b)
                    outs = [o for o, k in ((out["x"], "x2"), (out["edge_attr"], "e2")) if loss in (k, "both")]
                    gos = [go for go, k in ((gx2, "x2"), (ge2, "e2")) if loss in (k, "both")]
                    grads = torch.autograd.grad(outs, ins, gos)
                    ctx = f"{path} bwd={bwd} reduce={reduce} fused={fused} {kind} E={E} R={R} loss={loss}"
                    checks = list(zip(("gx", "ge", "gh"), grads, refs[loss]))
                    if loss == "both":
                        checks += [("x2", out["x"], rx.detach()), ("e2", out["edge_attr"], re.detach())]
                    for nm, got, want in checks:
                        v = nerr(got, want, per_row=False)
                        key = ("ConvFn " + path, nm, 3 if path != "tc1" else 1)
                        RESULTS[key] = max(RESULTS.get(key, 0.0), v)
                        ck.true(v <= tau, f"{nm} {ctx}: normalised error {v:.3e} > {tau:.0e}")
                        if path == "fma":
                            fma[(loss, nm)] = v
                        elif path == "tc3":
                            ck.yard("ConvFn tc3", nm, v, fma[(loss, nm)], ctx)
    finally:
        conv_mod.CONV_PATH, conv_mod.TC_BWD_VARIANT, conv_mod.MSG_REDUCE, conv_mod.CONV_BWD_FUSED = old
    ck.done()
