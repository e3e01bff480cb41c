"""The tensor-core convolution (conv_tc.cu) alone, through ev_test_conv_epilogue, against a float64 convolution with the same fused
epilogue: bias, mask_pre select, alpha, residual and MRF partial sum, 1/div, LeakyReLU / ReLU / SnakeBeta, mask_act, fp32 and bf16
outputs, polyphase transposed convolutions, fused GroupNorm statistics, ragged tile lists and the split fp32 paths.

The reference applies the kernel's roundings and nothing else: bf16 x and w on the bf16 path, exact bias and residuals, the
multiplication by fp32(1/div), bf16 rounding of the activated output.  Every output buffer belongs to the test: it sits between guard
rows, its rows may carry padding columns and its items padding rows, all filled with a sentinel (all bits set; -0.0 for the fp64
GroupNorm sums, which adding +0.0 would turn into +0.0), and each of them must still hold it afterwards.  One check function takes
every result: fp32 outputs bound rel-L2, the worst row and the worst channel (a bug confined to one 32-column block or one tile-edge
row hides under a global norm at N = 1024), bf16 outputs are bounded per element, masked rows must be exactly 0.  The CPU tests at
the top show that the check accepts an fp32 emulation of the kernel and rejects planted bugs; they need no GPU."""
import ctypes
import dataclasses
import itertools
import math
from collections import defaultdict

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ACT = {"none": 0, "relu": 1, "lrelu": 2, "snake": 4}
SCHED_NAMES = ("lean", "mb", "ctas_per_sm", "epi_warps", "resident", "bk32", "halo", "share")
REPORT_NAMES = ("bn", "mb", "ctas_per_sm", "epi_warps", "issuers", "resident", "a_slots", "b_slots", "bk", "halo", "a_boxes", "act_only",
                "vec_ok", "split", "flush_groups", "tf32_share", "ragged", "grid", "total_tiles")
TOL_F32 = (1e-5, 2e-5, 2e-5)      # fp32 outputs (rel-L2, worst row, worst channel): one conv, fp32 accumulation of exact products
ACT_FLOOR = 3e-5                  # bf16 outputs: 1 bf16 ulp of the reference + this times rms(reference)
SNAKE_FLOOR = 3e-4                # ... SnakeBeta: __sinf is inexact outside [-pi, pi]
GN_TOL = 1e-6                     # GroupNorm sums: |err| <= GN_TOL * sum |v| (sum of squares: * sum v^2)
GUARD = 3                         # guard rows before and after every output
PREC = {"bf16": 1, "tf32x3": 2, "f16x3": 3}
SENTINEL = {torch.float32: (torch.int32, -1), torch.bfloat16: (torch.int16, -1), torch.float64: (torch.int64, -(2 ** 63))}


def bf(t):
    return t.to(torch.bfloat16).to(t.dtype)


def f32(v):
    return float(np.float32(v))


@dataclasses.dataclass(frozen=True)
class Case:
    B: int = 2
    C_in: int = 64
    T: int = 129
    C_out: int = 64
    K: int = 1
    stride: int = 1
    pad: int = 0
    dil: int = 1
    transposed: bool = False
    prec: str = "bf16"
    bias: bool = True
    f32: bool = False                 # fp32 output
    act_out: bool = False             # bf16 output
    act: str = "none"
    slope: float = 0.0
    f32_is_act: bool = False
    res: str = ""                     # "" none, "sep" its own buffer, "out" the fp32 output itself (the Euler update)
    res2: str = ""                    # ditto ("out": the MRF partial sum)
    alpha: float = 1.0
    div: float = 1.0
    lengths: tuple = ()               # valid frames per item; () = no mask
    len_shift: int = 0
    mask_pre: bool = False
    mask_act: bool = False
    gn: bool = False
    f32_pad: int = 0                  # padding columns of an fp32 output row
    act_pad: int = 0                  # ... of a bf16 output row
    pad_rows: int = 0                 # padding rows after every item of every output
    x_col0: int = 0                   # bf16 x rows: x_col0 other columns, C_in channels, x_pad more (x_ld = their sum)
    x_pad: int = 0
    ragged: tuple = ()                # (frame lengths, rows_per_frame, margin) of a compact tile list

    @property
    def T_out(self):
        if self.transposed:
            return (self.T - 1) * self.stride - 2 * self.pad + self.K
        return (self.T + 2 * self.pad - self.dil * (self.K - 1) - 1) // self.stride + 1

    @property
    def N(self):
        return self.stride * self.C_out if self.transposed else self.C_out

    @property
    def x_ld(self):
        return self.x_col0 + self.C_in + self.x_pad


def pick_bn(N):
    return 128 if N % 128 == 0 else 32 if N <= 32 else 64 if N <= 64 else 128


def vec_ok(cs):
    lds = [cs.C_out + cs.f32_pad, cs.C_out + cs.act_pad]
    return cs.C_out % 4 == 0 and cs.N % 4 == 0 and all(ld % 4 == 0 for ld in lds)


def lean_ok(cs):
    ld = cs.C_out + cs.act_pad
    return (cs.prec == "bf16" and vec_ok(cs) and cs.act_out and not (cs.f32 or cs.res or cs.res2 or cs.mask_pre or cs.transposed) and
            cs.alpha == 1.0 and cs.div == 1.0 and cs.N % 32 == 0 and ld % 8 == 0 and (cs.T_out + cs.pad_rows) * ld % 8 == 0)


# ------------------------------------------------------------------------------------------------ caller-owned outputs
class Out:
    """B items of `rows` x C elements at interior offset `off` of a flat sentinel-filled buffer: item b, row t, column c lives at
    off + b*bs + t*ld + c with ld = C + pad_cols and bs = (rows + pad_rows) * ld; `guard` rows of ld elements come before and after."""

    def __init__(self, B, rows, C, dtype, device, pad_cols=0, pad_rows=0, guard=GUARD):
        self.B, self.rows, self.C, self.dtype = B, rows, C, dtype
        self.ld, self.off = C + pad_cols, guard * (C + pad_cols)
        self.bs = (rows + pad_rows) * self.ld
        ity, s = SENTINEL[dtype]
        self.full = torch.full((2 * self.off + B * self.bs,), s, dtype=ity, device=device).view(dtype)
        b, t, c = torch.arange(B).view(-1, 1, 1), torch.arange(rows).view(1, -1, 1), torch.arange(C).view(1, 1, -1)
        self.index = self.off + b * self.bs + t * self.ld + c
        self.inside = torch.zeros(self.full.numel(), dtype=torch.bool)
        self.inside[self.index.flatten()] = True

    def ptr(self):
        return self.full.data_ptr() + self.off * self.full.element_size()

    def values(self):
        return self.full.cpu()[self.index]

    def set(self, v):
        self.full[self.index.to(self.full.device)] = v.to(self.dtype).to(self.full.device)

    def untouched(self):
        """True where an element outside the interior region still holds the sentinel, bit for bit."""
        ity, s = SENTINEL[self.dtype]
        out = self.full.cpu()
        return out.view(ity)[~self.inside] == s


# ------------------------------------------------------------------------------------------------ inputs and the reference
def make_inputs(cs, seed):
    g = torch.Generator().manual_seed(seed)
    B, T_out, C = cs.B, cs.T_out, cs.C_out
    w_shape = (cs.C_in, cs.C_out, cs.K) if cs.transposed else (cs.C_out, cs.C_in, cs.K)
    fan = cs.C_in * cs.K / (cs.stride if cs.transposed else 1)
    return dict(
        x=torch.randn(B, cs.T, cs.C_in, generator=g),
        w=torch.randn(*w_shape, generator=g) / math.sqrt(fan),
        bias=torch.randn(C, generator=g) * 0.3 if cs.bias else None,
        res=torch.randn(B, T_out, C, generator=g) if cs.res else None,
        res2=torch.randn(B, T_out, C, generator=g) if cs.res2 else None,
        snake_a=torch.exp(torch.randn(C, generator=g) * 0.3),
        snake_invb=1.0 / (torch.exp(torch.randn(C, generator=g) * 0.3) + 1e-9),
    )


def row_mask(cs, lengths=None, shift=None):
    """(B, T_out) bool: output row t of item b is valid while (t << len_shift) < lengths[b]."""
    lengths = cs.lengths if lengths is None else lengths
    shift = cs.len_shift if shift is None else shift
    if not lengths:
        return torch.ones(cs.B, cs.T_out, dtype=torch.bool)
    t = torch.arange(cs.T_out).view(1, -1)
    return (t << shift) < torch.tensor(lengths).view(-1, 1)


def reference(cs, inp, *, dtype=torch.float64, plant=()):
    """-> dict f32 / act: (B, T_out, C_out) in `dtype` (act rounded to bf16), or None when the case has no such output; zero_f32 /
    zero_act: (B, T_out) rows that masking makes exactly 0.  dtype=float32 is an emulation of the kernel.  `plant` lists the planted
    bugs of the CPU tests: bias_block, mask_off_by_one, ignore_shift, drop_res2, alpha_after_res, swap_phases, snake_column, div."""
    rnd = bf if cs.prec == "bf16" else (lambda t: t)
    x = rnd(inp["x"]).to(dtype).transpose(1, 2)
    w = rnd(inp["w"]).to(dtype)
    if cs.transposed:
        acc = F.conv_transpose1d(x, w, stride=cs.stride, padding=cs.pad)
    else:
        acc = F.conv1d(x, w, stride=cs.stride, padding=cs.pad, dilation=cs.dil)
    v = acc.transpose(1, 2)
    if "swap_phases" in plant:                   # output rows of phases 0 and 1 exchanged (t + pad = s*r + phase)
        t0 = torch.arange(-cs.pad, cs.T_out, cs.stride)
        t0 = t0[(t0 >= 0) & (t0 + 1 < cs.T_out)]
        v = v.clone()
        v[:, t0], v[:, t0 + 1] = v[:, t0 + 1].clone(), v[:, t0].clone()
    if inp["bias"] is not None:
        b = inp["bias"].to(dtype).clone()
        if "bias_block" in plant:
            b[32:64] = 0
        v = v + b
    lengths = tuple(n + 1 for n in cs.lengths) if "mask_off_by_one" in plant else cs.lengths
    m = row_mask(cs, lengths, 0 if "ignore_shift" in plant else cs.len_shift).unsqueeze(-1)
    if cs.mask_pre:
        v = torch.where(m, v, torch.zeros_like(v))
    alpha = torch.tensor(f32(cs.alpha), dtype=dtype)
    res = sum(inp[k].to(dtype) for k in ("res", "res2") if inp[k] is not None and not (k == "res2" and "drop_res2" in plant))
    v = (v + res) * alpha if "alpha_after_res" in plant else v * alpha + res
    if cs.div != 1.0:
        v = v / torch.tensor(f32(cs.div), dtype=dtype) if "div" in plant else v * torch.tensor(f32(1.0 / np.float32(cs.div)), dtype=dtype)
    if cs.act == "relu":
        a = torch.clamp_min(v, 0)
    elif cs.act == "lrelu":
        a = torch.where(v > 0, v, v * f32(cs.slope))
    elif cs.act == "snake":
        sa, sb = inp["snake_a"].to(dtype), inp["snake_invb"].to(dtype)
        if "snake_column" in plant:
            sa, sb = sa.roll(1), sb.roll(1)
        a = v + sb * torch.sin(v * sa) ** 2
    else:
        a = v
    if cs.mask_act:
        a = torch.where(m, a, torch.zeros_like(a))
    masked = ~row_mask(cs)
    no_res = not (cs.res or cs.res2)
    return dict(f32=(a if cs.f32_is_act else v) if cs.f32 else None, act=bf(a) if cs.act_out else None,
                zero_act=masked & cs.mask_act,
                zero_f32=masked & ((cs.mask_act and cs.f32_is_act) or (cs.mask_pre and no_res and not cs.f32_is_act)))


def gn_reference(cs, got_f32, rows=None):
    """Per (item, 32-channel group) sum and sum of squares of the kernel's own fp32 output over rows t < T_out (or `rows`)."""
    v = got_f32.double()[:, : cs.T_out if rows is None else rows]
    v = v.reshape(cs.B, v.shape[1], cs.C_out // 32, 32)
    return torch.stack([v.sum((1, 3)), (v * v).sum((1, 3))], -1), torch.stack([v.abs().sum((1, 3)), (v * v).sum((1, 3))], -1)


# ------------------------------------------------------------------------------------------------ the one check
WORST = defaultdict(float)            # measured worst errors per group (printed by the coverage test)


def group(cs, what):
    if cs.prec != "bf16":
        return "split paths, fp32 out"
    if what == "act":
        return "bf16, snake" if cs.act == "snake" else "bf16, bf16 out"
    return "bf16, fp32 out"


def bf16_ulp(r):
    _, e = torch.frexp(r.double())
    return torch.where(r == 0, torch.zeros_like(r.double()), torch.ldexp(torch.ones_like(r.double()), e - 8))


def check(cs, outs, ref, what="", record=False):
    """Every result passes here.  outs: name -> Out ("f32", "act", "gn"); ref: reference(cs, ...).  record: a kernel result whose
    errors go into WORST."""
    worst = WORST if record else defaultdict(float)
    for name, o in outs.items():
        ok = o.untouched()
        assert ok.all(), f"{what}: {name}: {int((~ok).sum())} elements outside the output (guard rows, padding) lost their sentinel"
    if cs.f32:
        got, r = outs["f32"].values().double(), ref["f32"].double()
        assert torch.isfinite(got).all(), f"{what}: fp32 output has non-finite values"
        assert (got[ref["zero_f32"]] == 0).all(), f"{what}: masked rows of the fp32 output are not 0"
        err = got - r
        rms = r.pow(2).mean().sqrt().clamp_min(1e-30)
        rel = float(err.norm() / r.norm().clamp_min(1e-30))
        row = float(err.pow(2).mean(-1).sqrt().max() / rms)
        chan = float(err.pow(2).mean((0, 1)).sqrt().max() / rms)
        g = group(cs, "f32")
        for k, val in (("rel-L2", rel), ("worst row", row), ("worst channel", chan)):
            worst[(g, k)] = max(worst[(g, k)], val)
        assert rel <= TOL_F32[0] and row <= TOL_F32[1] and chan <= TOL_F32[2], \
            f"{what}: fp32 output rel-L2 {rel:.3g}, worst row {row:.3g}, worst channel {chan:.3g} (bounds {TOL_F32})"
    if cs.act_out:
        got, r = outs["act"].values().double(), ref["act"].double()
        assert torch.isfinite(got).all(), f"{what}: bf16 output has non-finite values"
        assert (got[ref["zero_act"]] == 0).all(), f"{what}: masked rows of the bf16 output are not 0"
        floor = (SNAKE_FLOOR if cs.act == "snake" else ACT_FLOOR) * float(r.pow(2).mean().sqrt())
        err = (got - r).abs()
        ulp = bf16_ulp(r)
        bad = err > ulp + floor
        g = group(cs, "act")
        worst[(g, "ulps")] = max(worst[(g, "ulps")], float((err / (ulp + floor)).max()))
        assert not bad.any(), (f"{what}: {int(bad.sum())} bf16 outputs beyond 1 ulp + {floor:.2g}, first (b, t, c) = {bad.nonzero()[0].tolist()}, "
                               f"got {float(got[bad][0])}, reference {float(r[bad][0])}")
    if cs.gn:
        got = outs["gn"].values().double()
        ref_gn, scale = gn_reference(cs, outs["f32"].values())
        err = float(((got - ref_gn).abs() / scale.clamp_min(1e-30)).max())
        worst[("GroupNorm sums", "relative to sum |v|")] = max(worst[("GroupNorm sums", "relative to sum |v|")], err)
        assert err <= GN_TOL, f"{what}: GroupNorm sums off by {err:.3g} of their magnitude (bound {GN_TOL})"


def alloc_outputs(cs, device):
    outs = {}
    if cs.f32:
        outs["f32"] = Out(cs.B, cs.T_out, cs.C_out, torch.float32, device, cs.f32_pad, cs.pad_rows)
    if cs.act_out:
        outs["act"] = Out(cs.B, cs.T_out, cs.C_out, torch.bfloat16, device, cs.act_pad, cs.pad_rows)
    if cs.gn:
        outs["gn"] = Out(cs.B, cs.C_out // 32, 2, torch.float64, device, guard=4)
        outs["gn"].set(torch.zeros(cs.B, cs.C_out // 32, 2, dtype=torch.float64))
    return outs


def emulated(cs, inp, plant=(), gn_rows=None):
    """What a kernel with `plant` would leave in the caller's buffers, on the CPU (fp32 arithmetic)."""
    r = reference(cs, inp, dtype=torch.float32, plant=plant)
    outs = alloc_outputs(cs, "cpu")
    if cs.f32:
        outs["f32"].set(r["f32"])
    if cs.act_out:
        outs["act"].set(r["act"])
    if cs.gn:
        v = r["f32"][:, : cs.T_out if gn_rows is None else gn_rows].reshape(cs.B, -1, cs.C_out // 32, 32)
        outs["gn"].set(torch.stack([v.sum((1, 3)), (v * v).sum((1, 3))], -1).double())
    return outs


# ------------------------------------------------------------------------------------------------ the check, without a GPU
EMUL_CASES = {
    "lean lrelu": Case(C_in=80, C_out=128, K=7, pad=3, act_out=True, act="lrelu", slope=0.1),
    "fp32 + bias": Case(C_in=64, C_out=128, K=3, pad=1, f32=True),
    "masked operand": Case(C_in=64, T=130, C_out=64, K=3, pad=1, act_out=True, lengths=(130, 71), mask_act=True),
    "half-rate mask": Case(C_in=64, T=130, C_out=64, K=3, stride=2, pad=1, act_out=True, lengths=(130, 71), len_shift=1, mask_act=True),
    "MRF mean": Case(C_in=32, C_out=32, K=7, pad=3, f32=True, act_out=True, act="lrelu", slope=0.1, res="sep", res2="out", div=3.0),
    "Euler": Case(C_in=64, C_out=80, f32=True, act_out=True, res="out", alpha=0.1, lengths=(129, 50), mask_pre=True, mask_act=True, act_pad=80),
    "polyphase": Case(C_in=64, T=65, C_out=32, K=4, stride=2, pad=1, transposed=True, f32=True),
    "snake": Case(C_in=64, C_out=256, act_out=True, act="snake"),
    "groupnorm": Case(C_in=64, T=257, C_out=96, K=3, pad=1, f32=True, gn=True),
    "padded rows": Case(C_in=64, C_out=64, act_out=True, act="relu", act_pad=8, pad_rows=2),
}
PLANTED = [  # (case, planted bug): each must fail the check
    ("fp32 + bias", "bias_block"), ("lean lrelu", "bias_block"), ("masked operand", "mask_off_by_one"), ("half-rate mask", "ignore_shift"),
    ("MRF mean", "drop_res2"), ("Euler", "alpha_after_res"), ("polyphase", "swap_phases"), ("snake", "snake_column"),
    ("groupnorm", "gn_last_row"), ("padded rows", "padding_write"),
]


@pytest.mark.parametrize("name", sorted(EMUL_CASES))
def test_check_accepts_fp32_emulation(name):
    cs = EMUL_CASES[name]
    inp = make_inputs(cs, seed=len(name))
    ref = reference(cs, inp)
    check(cs, emulated(cs, inp), ref, what=f"emulation {name}")
    if cs.div != 1.0:    # x / div in place of x * (1/div): one rounding apart, accepted
        check(cs, emulated(cs, inp, plant=("div",)), ref, what=f"emulation {name}, x / div")


@pytest.mark.parametrize("name,bug", PLANTED)
def test_check_rejects_planted_bug(name, bug):
    cs = EMUL_CASES[name]
    inp = make_inputs(cs, seed=len(name))
    ref = reference(cs, inp)
    if bug == "gn_last_row":
        outs = emulated(cs, inp, gn_rows=cs.T_out - 1)
    elif bug == "padding_write":
        outs = emulated(cs, inp)
        o = outs["act"]
        o.full[o.off + o.bs + 5 * o.ld + cs.C_out + 3] = 0.0          # one store into a padding column of item 1
    else:
        outs = emulated(cs, inp, plant=(bug,))
    with pytest.raises(AssertionError):
        check(cs, outs, ref, what=f"{name} with {bug}")


def test_check_catches_a_stray_groupnorm_add_past_the_last_item():
    """+0.0 added one group past the end changes the -0.0 guard's bits (the overrun of a block past C_out)."""
    cs = EMUL_CASES["groupnorm"]
    inp = make_inputs(cs, seed=3)
    outs = emulated(cs, inp)
    o = outs["gn"]
    o.full[o.off + cs.B * o.bs] += 0.0
    with pytest.raises(AssertionError):
        check(cs, outs, reference(cs, inp), what="stray GroupNorm add")


# ------------------------------------------------------------------------------------------------ the kernel on the GPU
@pytest.fixture(scope="module")
def ctx():
    from emojivoice_b200 import _lib

    return _lib.Context()


SEEN = defaultdict(set)               # launch variants run by this file (checked by test_every_launch_variant_was_run)


def run(ctx, cs, inp, schedule=None, expect_rc=0):
    """One ev_test_conv_epilogue call -> (outs on the device, report dict)."""
    from emojivoice_b200 import _lib

    dev = "cuda"
    outs = alloc_outputs(cs, dev)
    keep = []

    def d(t):
        if t is None:
            return None
        t = t.contiguous().to(dev)
        keep.append(t)
        return t.data_ptr()

    if cs.prec == "bf16":
        xb = torch.zeros(cs.B, cs.T, cs.x_ld, dtype=torch.bfloat16)
        xb[..., cs.x_col0: cs.x_col0 + cs.C_in] = inp["x"].bfloat16()
        x_ptr = d(xb) + 2 * cs.x_col0
        x_ld = cs.x_ld
    else:
        x_ptr, x_ld = d(inp["x"]), cs.C_in
    a = _lib.EvConvEpilogueTest()
    a.B, a.C_in, a.T, a.C_out, a.K, a.stride, a.pad, a.dilation = cs.B, cs.C_in, cs.T, cs.C_out, cs.K, cs.stride, cs.pad, cs.dil
    a.transposed, a.precision = int(cs.transposed), PREC[cs.prec]
    a.w, a.bias, a.x, a.x_ld, a.x_bs = d(inp["w"]), d(inp["bias"]), x_ptr, x_ld, cs.T * x_ld
    for name, ptr_f, ld_f, bs_f in (("res", "res", "res_ld", "res_bs"), ("res2", "res2", "res2_ld", "res2_bs")):
        mode = getattr(cs, name)
        if mode == "sep":
            setattr(a, ptr_f, d(inp[name]))
            setattr(a, ld_f, cs.C_out)
            setattr(a, bs_f, cs.T_out * cs.C_out)
        elif mode == "out":
            o = outs["f32"]
            o.set(inp[name])
            setattr(a, ptr_f, o.ptr())
            setattr(a, ld_f, o.ld)
            setattr(a, bs_f, o.bs)
    if cs.f32:
        o = outs["f32"]
        a.out_f32, a.f32_ld, a.f32_bs = o.ptr(), o.ld, o.bs
    if cs.act_out:
        o = outs["act"]
        a.out_act, a.act_ld, a.act_bs = o.ptr(), o.ld, o.bs
    if cs.gn:
        a.gn_sum, a.gn_groups = outs["gn"].ptr(), cs.C_out // 32
    if cs.lengths:
        a.lengths = d(torch.tensor(cs.lengths, dtype=torch.int64))
    a.len_shift, a.mask_pre, a.mask_act = cs.len_shift, int(cs.mask_pre), int(cs.mask_act)
    a.act, a.slope, a.f32_is_act = ACT[cs.act], cs.slope, int(cs.f32_is_act)
    a.snake_a, a.snake_invb = d(inp["snake_a"]), d(inp["snake_invb"])
    a.alpha, a.div = cs.alpha, cs.div
    if cs.ragged:
        frames, a.rows_per_frame, a.ragged_margin = cs.ragged
        a.ragged_lengths = d(torch.tensor(frames, dtype=torch.int64))
    sched = (ctypes.c_int32 * 8)(*[(schedule or {}).get(n, -1) for n in SCHED_NAMES])
    rep = (ctypes.c_int32 * 19)()
    a.schedule_host = ctypes.cast(sched, ctypes.c_void_p)
    a.report_host = ctypes.cast(rep, ctypes.c_void_p)
    rc = _lib.lib().ev_test_conv_epilogue(ctx.handle, ctypes.byref(a), _lib.stream_ptr())
    if expect_rc is None:             # the caller takes refusals
        if rc != 0:
            assert rc == -1, f"{cs} {schedule}: rc {rc}: {_lib.lib().ev_last_error(ctx.handle).decode()}"
            return None, None
    elif expect_rc:
        assert rc == expect_rc, f"{schedule}: expected {expect_rc}, got {rc}: {_lib.lib().ev_last_error(ctx.handle).decode()}"
        return None, None
    else:
        ctx.check(rc, f"ev_test_conv_epilogue {cs} schedule={schedule}")
    r = dict(zip(REPORT_NAMES, list(rep)))
    for k in ("bn", "mb", "ctas_per_sm", "epi_warps", "issuers", "resident", "bk", "halo", "a_boxes", "act_only", "vec_ok", "split",
              "tf32_share", "ragged"):
        SEEN[k].add(r[k])
    SEEN["flush"].add(r["flush_groups"] > 1)
    return outs, r


def check_report(cs, rep):
    """The report agrees with the layer: tile width, K-chunk, split mode, epilogue kind, tiles, grid."""
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    M = cs.T + 1 if cs.transposed else cs.T_out
    assert rep["bn"] == pick_bn(cs.N), rep
    assert rep["split"] == PREC[cs.prec] - 1, rep
    assert rep["vec_ok"] == vec_ok(cs), rep
    assert rep["act_only"] <= lean_ok(cs), rep
    assert rep["total_tiles"] == cs.B * math.ceil(M / (128 * rep["mb"])) * math.ceil(cs.N / rep["bn"]), rep
    assert rep["grid"] == min(rep["total_tiles"], rep["ctas_per_sm"] * sms), rep
    assert rep["epi_warps"] == (8 if rep["issuers"] == 1 else 16), rep
    if cs.prec == "tf32x3":
        assert rep["bk"] == 32, rep
    elif cs.prec == "f16x3" or cs.C_in > 32:
        assert rep["bk"] == 64, rep


def schedules(cs):
    """Every forced schedule the launcher may accept for the case (refused ones are skipped by the caller)."""
    if cs.prec != "bf16":
        return [dict(share=0), dict(share=1), dict(share=0, resident=1)]
    n_tiles = math.ceil(cs.N / pick_bn(cs.N))
    axes = [("lean", (0, 1) if lean_ok(cs) else (-1,)), ("mb", (1, 2)), ("occ", ((2, 8), (1, 8), (1, 16))),
            ("resident", (0, 1) if n_tiles == 1 else (-1,)), ("bk32", (0, 1) if cs.C_in <= 32 else (-1,)),
            ("halo", (0, 1) if cs.K > 1 and cs.stride == 1 else (-1,))]
    out = []
    for vals in itertools.product(*[v for _, v in axes]):
        sc = {}
        for (name, _), v in zip(axes, vals):
            if name == "occ":
                sc["ctas_per_sm"], sc["epi_warps"] = v
            elif v != -1:
                sc[name] = v
        out.append(sc)
    return out


def same_bits(outs_a, outs_b):
    return all(torch.equal(outs_a[k].full.view(SENTINEL[outs_a[k].dtype][0]), outs_b[k].full.view(SENTINEL[outs_b[k].dtype][0])) for k in outs_a)


def verify(ctx, cs, seed, walk=True):
    """The default launch against the reference; then every accepted forced schedule: bit-identical to it on the bf16 path (every
    walk issues each accumulator's MMAs K-chunk-major, tap-minor and the lean and generic epilogues round alike), within the bound
    on the split paths (operand sharing reorders the three products).  -> the default report."""
    inp = make_inputs(cs, seed)
    ref = reference(cs, inp)
    base, rep = run(ctx, cs, inp)
    check_report(cs, rep)
    check(cs, base, ref, what=f"{cs} default", record=True)
    if not walk:
        return rep
    accepted = 0
    for sc in schedules(cs):
        outs, r = run(ctx, cs, inp, schedule=sc, expect_rc=None)
        if outs is None:
            continue
        accepted += 1
        check_report(cs, r)
        if cs.prec == "bf16":
            assert same_bits(outs, base), f"{cs}: schedule {sc} ({r}) differs from the default ({rep})"
        else:
            check(cs, outs, ref, what=f"{cs} schedule {sc}", record=True)
    assert accepted >= 2, f"{cs}: the launcher accepted {accepted} forced schedules"
    return rep


# ---- every epilogue the models build, at the widths they use
LRELU = dict(act="lrelu", slope=0.1)
MODEL_CASES = {
    # vocoder (HiFi-GAN v1): conv_pre, ResBlock conv1 (lean), conv2 with residual, the MRF branch that closes a stage, upsamplers
    "voc conv_pre": Case(C_in=80, T=200, C_out=512, K=7, pad=3, act_out=True, **LRELU),
    "voc rb conv1 C32": Case(C_in=32, T=300, C_out=32, K=11, pad=25, dil=5, act_out=True, **LRELU),
    "voc rb conv1 C128": Case(C_in=128, T=257, C_out=128, K=3, pad=3, dil=3, act_out=True, **LRELU),
    "voc rb conv2": Case(C_in=64, T=300, C_out=64, K=7, pad=3, res="sep", f32=True, act_out=True, **LRELU),
    "voc mrf close": Case(C_in=128, T=255, C_out=128, K=11, pad=5, res="sep", res2="out", div=3.0, f32=True, act_out=True, **LRELU),
    "voc mrf close, no fp32": Case(C_in=64, T=129, C_out=64, K=3, pad=1, res="sep", res2="sep", div=3.0, act_out=True, **LRELU),
    "voc up s8 p4": Case(C_in=512, T=33, C_out=256, K=16, stride=8, pad=4, transposed=True, f32=True, act_out=True, **LRELU),
    "voc up s8 p0": Case(C_in=128, T=40, C_out=64, K=16, stride=8, pad=0, transposed=True, f32=True, act_out=True, **LRELU),
    "voc up s8 p7": Case(C_in=128, T=40, C_out=64, K=16, stride=8, pad=7, transposed=True, f32=True, act_out=True, **LRELU),
    "voc up s2 p1": Case(C_in=64, T=150, C_out=32, K=4, stride=2, pad=1, transposed=True, f32=True, act_out=True, **LRELU),
    "voc up s2 p0": Case(C_in=64, T=150, C_out=32, K=4, stride=2, pad=0, transposed=True, f32=True, act_out=True, **LRELU),
    # decoder (U-Net of the flow-matching estimator, D = 256): down / up convs into the skip buffers, FF1 (SnakeBeta), FF2,
    # ResNet convs with fused GroupNorm statistics, QKV, the up-sampling transposed conv, the Euler update
    "dec down0 stride2": Case(C_in=256, T=258, C_out=256, K=3, stride=2, pad=1, act_out=True, lengths=(258, 161), len_shift=1, mask_act=True,
                              x_col0=256),
    "dec up1_conv": Case(C_in=256, T=257, C_out=256, K=3, pad=1, act_out=True, lengths=(257, 100), mask_act=True),
    "dec ff1 snake": Case(C_in=256, T=200, C_out=1024, act_out=True, act="snake"),
    "dec ff2": Case(C_in=1024, T=200, C_out=256, res="sep", act_out=True, lengths=(200, 77), mask_act=True, act_pad=256),
    "dec resnet conv gn 256": Case(C_in=512, T=130, C_out=256, K=3, pad=1, f32=True, gn=True),
    "dec resnet conv gn 128": Case(C_in=128, T=257, C_out=128, K=3, pad=1, f32=True, gn=True),
    "dec qkv": Case(C_in=256, T=129, C_out=384, act_out=True),
    "dec up0 transposed": Case(C_in=256, T=65, C_out=256, K=4, stride=2, pad=1, transposed=True, act_out=True, lengths=(130, 61),
                               mask_act=True, act_pad=256),
    "dec euler": Case(C_in=256, T=257, C_out=80, f32=True, act_out=True, res="out", alpha=0.1, lengths=(257, 140), mask_pre=True,
                      mask_act=True, act_pad=80),
    "dec estimator out": Case(C_in=256, T=128, C_out=80, f32=True, alpha=0.25, lengths=(128, 3), mask_pre=True),
    # text encoder, split fp32 paths: ffn1 (ReLU, masked, into the fp32 "activation"), ffn2 (residual, masked first)
    "enc ffn1 3xTF32": Case(prec="tf32x3", C_in=192, T=181, C_out=768, K=3, pad=1, f32=True, f32_is_act=True, act="relu", lengths=(181, 90),
                            mask_act=True),
    "enc ffn1 3xFP16": Case(prec="f16x3", C_in=192, T=181, C_out=768, K=3, pad=1, f32=True, f32_is_act=True, act="relu", lengths=(181, 90),
                            mask_act=True),
    "enc ffn2 3xTF32": Case(prec="tf32x3", C_in=768, T=130, C_out=192, K=3, pad=1, f32=True, res="sep", lengths=(130, 64), mask_pre=True),
    "enc ffn2 3xFP16": Case(prec="f16x3", C_in=768, T=130, C_out=192, K=3, pad=1, f32=True, res="sep", lengths=(130, 64), mask_pre=True),
    "enc proj_m 3xFP16": Case(prec="f16x3", C_in=192, T=77, C_out=80, f32=True, lengths=(77, 20), mask_pre=True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MODEL_CASES))
def test_model_epilogues(ctx, name):
    verify(ctx, MODEL_CASES[name], seed=sum(map(ord, name)))


# ---- geometry: tile edges, BN edges, K-chunk widths, padded layouts
@pytest.mark.gpu
@pytest.mark.parametrize("T", [127, 128, 129, 255, 256, 257])
@pytest.mark.parametrize("lean", [True, False])
def test_output_rows_on_tile_edges(ctx, T, lean):
    if lean:
        cs = Case(C_in=64, T=T, C_out=64, K=3, pad=1, act_out=True, lengths=(T, T // 2 + 1), mask_act=True, **LRELU)
    else:
        cs = Case(C_in=64, T=T, C_out=64, K=3, pad=1, res="sep", f32=True, act_out=True, lengths=(T, T - 3), mask_act=True, **LRELU)
    verify(ctx, cs, seed=T + 1000 * lean)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [32, 64, 96, 128, 160, 192, 224, 384])
@pytest.mark.parametrize("mode", ["lean", "lean, dense rows", "generic", "groupnorm", "groupnorm, dense rows"])
def test_output_channels_on_tile_edges(ctx, N, mode):
    """N = 96 / 160 / 192 / 224 leave 32-column blocks past C_out in the last 128-wide tile: the lean epilogue must neither read the bias
    past C_out nor store into columns >= C_out, and the GroupNorm statistics must not add into a group past the last.  With padding
    columns a stray store lands on a sentinel; with the production layout (ld == C_out) it lands in the next row, which the reference
    comparison catches."""
    dense = "dense" in mode
    pad = 0 if dense else 32
    if mode.startswith("lean"):
        cs = Case(B=3, C_in=64, T=150, C_out=N, K=3, pad=1, act_out=True, act_pad=pad, **LRELU)
    elif mode == "generic":
        cs = Case(B=3, C_in=64, T=150, C_out=N, K=3, pad=1, res="sep", f32=True, act_out=True, f32_pad=pad, act_pad=pad, **LRELU)
    else:
        cs = Case(B=3, C_in=64, T=150, C_out=N, K=3, pad=1, f32=True, gn=True, f32_pad=pad)
    rep = verify(ctx, cs, seed=N + len(mode))
    if mode.startswith("lean"):
        assert rep["act_only"] == 1, rep


@pytest.mark.gpu
@pytest.mark.parametrize("C_in,K", [(16, 3), (32, 7), (80, 7), (224, 3)])
def test_reduction_widths(ctx, C_in, K):
    """C_in <= 32 (BK 32, the 64-byte swizzle) and C_in not a multiple of 64 (a zero-filled tail of the last K-chunk)."""
    verify(ctx, Case(C_in=C_in, T=200, C_out=64, K=K, pad=K // 2, res="sep", f32=True, act_out=True, **LRELU), seed=C_in * K)
    verify(ctx, Case(C_in=C_in, T=200, C_out=128, K=K, pad=K // 2, act_out=True, x_pad=8, **LRELU), seed=C_in * K + 1)


@pytest.mark.gpu
def test_padded_item_stride_and_single_row(ctx):
    verify(ctx, Case(C_in=64, T=131, C_out=128, K=3, pad=1, act_out=True, act_pad=8, pad_rows=5, **LRELU), seed=1)
    verify(ctx, Case(C_in=64, T=131, C_out=128, K=3, pad=1, f32=True, act_out=True, res="sep", f32_pad=4, act_pad=8, pad_rows=3, **LRELU), seed=2)
    verify(ctx, Case(B=3, C_in=64, T=1, C_out=64, K=3, pad=1, f32=True, act_out=True, res="sep", **LRELU), seed=3)
    verify(ctx, Case(B=3, C_in=64, T=1, C_out=64, K=1, act_out=True, **LRELU), seed=4)


@pytest.mark.gpu
@pytest.mark.parametrize("lean", [True, False])
def test_more_tiles_than_ctas(ctx, lean):
    """Hundreds of tiles per launch: each CTA hands its two accumulator sets back and forth many times (the parity turns over)."""
    if lean:
        cs = Case(B=8, C_in=32, T=8200, C_out=256, K=3, pad=1, act_out=True, lengths=(8200, 3000, 1, 8200, 2048, 17, 5000, 129), mask_act=True,
                  **LRELU)
    else:
        cs = Case(B=8, C_in=32, T=8200, C_out=256, K=3, pad=1, f32=True, res="sep", act_out=True, **LRELU)
    rep = verify(ctx, cs, seed=5 + lean, walk=False)
    assert rep["total_tiles"] > 2 * rep["grid"], rep
    for sc in (dict(ctas_per_sm=2, mb=1), dict(ctas_per_sm=1, epi_warps=16, mb=2)):
        inp = make_inputs(cs, 5 + lean)
        outs, r = run(ctx, cs, inp, schedule=sc)
        assert r["total_tiles"] > 2 * r["grid"], r
        check(cs, outs, reference(cs, inp), what=f"{cs} {sc}", record=True)


# ---- the scalar epilogue (N % 4 != 0, or a row stride that is not a multiple of 4)
SCALAR_FEATURES = {
    "bias + fp32": dict(f32=True),
    "lrelu bf16": dict(act_out=True, **LRELU),
    "snake bf16": dict(act_out=True, act="snake"),
    "mask_pre + alpha + res (Euler)": dict(f32=True, act_out=True, res="out", alpha=0.1, lengths=(140, 51), mask_pre=True, mask_act=True),
    "res + res2 + div": dict(f32=True, act_out=True, res="sep", res2="out", div=3.0, **LRELU),
    "f32_is_act relu + mask_act": dict(f32=True, f32_is_act=True, act="relu", lengths=(140, 9), len_shift=1, mask_act=True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("feature", sorted(SCALAR_FEATURES))
@pytest.mark.parametrize("N,pad", [(1, 0), (3, 0), (30, 0), (32, 1)])
def test_scalar_epilogue(ctx, N, pad, feature):
    cs = Case(C_in=64, T=140, C_out=N, K=3, pad=1, f32_pad=pad, act_pad=pad, **SCALAR_FEATURES[feature])
    rep = verify(ctx, cs, seed=N * 7 + pad + len(feature))
    assert rep["vec_ok"] == 0, rep


@pytest.mark.gpu
def test_polyphase_with_scalar_epilogue(ctx):
    verify(ctx, Case(C_in=64, T=50, C_out=6, K=4, stride=2, pad=1, transposed=True, f32=True, act_out=True, **LRELU), seed=9)


# ---- ragged tile lists
@pytest.mark.gpu
@pytest.mark.parametrize("lean", [True, False])
def test_ragged_tile_list(ctx, lean):
    """Compact tile lists: rows below (frames + margin) * rows_per_frame equal the dense launch bit for bit; every other row either
    equals it too (its tile was computed) or still holds the sentinel (skipped)."""
    frames, rpf, margin = (0, 3, 40, 17), 8, 2
    if lean:
        base = Case(B=4, C_in=64, T=320, C_out=128, K=7, pad=3, act_out=True, **LRELU)
    else:
        base = Case(B=4, C_in=64, T=320, C_out=64, K=16, stride=8, pad=4, transposed=True, f32=True, act_out=True, **LRELU)
    inp = make_inputs(base, seed=11)
    rag_cs = dataclasses.replace(base, ragged=(frames, rpf, margin))
    M = base.T + 1 if base.transposed else base.T_out
    skipped = 0
    for sc in (dict(mb=1), dict(mb=2)):
        dense, _ = run(ctx, base, inp, schedule=sc)
        rag, rep = run(ctx, rag_cs, inp, schedule=sc)
        assert rep["ragged"] == 1, rep
        for k, o in rag.items():
            d, r = dense[k].values(), o.values()
            ity, s = SENTINEL[o.dtype]
            for b, n in enumerate(frames):
                need_rows = min(M, (n + margin) * rpf)
                valid = min(base.T_out, need_rows * (base.stride if base.transposed else 1) - (base.pad if base.transposed else 0))
                valid = max(valid, 0)
                assert torch.equal(r[b, :valid].view(ity), d[b, :valid].view(ity)), f"{k}: item {b}, schedule {sc}"
                rest_equal = (r[b, valid:].view(ity) == d[b, valid:].view(ity)).all(-1)
                rest_sent = (r[b, valid:].view(ity) == s).all(-1)
                assert (rest_equal | rest_sent).all(), f"{k}: item {b}, schedule {sc}: rows past the needed ones hold other values"
                skipped += int(rest_sent.sum())
            assert o.untouched().all()
    assert skipped > 0, "no tile was skipped"


# ---- refusals and coverage
@pytest.mark.gpu
def test_forced_schedule_that_cannot_run_is_refused(ctx):
    """A forced choice is launched as asked or refused with EV_ERR_INVALID, never swapped for another variant."""
    lean = Case(C_in=64, T=300, C_out=128, K=3, pad=1, act_out=True, **LRELU)
    wide = Case(C_in=64, T=300, C_out=384, K=3, pad=1, act_out=True, **LRELU)
    big_w = Case(C_in=1024, T=300, C_out=128, K=3, pad=1, act_out=True, **LRELU)
    generic = Case(C_in=64, T=300, C_out=128, K=1, f32=True)
    split = Case(prec="tf32x3", C_in=192, T=100, C_out=256, K=3, pad=1, f32=True)
    cases = [
        (wide, dict(resident=1)),                        # three n-tiles: resident weights are loaded at n0 = 0
        (big_w, dict(resident=1)),                       # 48 weight tiles of 16 KB do not fit in shared memory
        (lean, dict(ctas_per_sm=2, mb=2)),               # 2 * mb * BN = 512 TMEM columns: one CTA per SM
        (lean, dict(ctas_per_sm=2, epi_warps=16)),       # two CTAs per SM run 8 epilogue warps each
        (generic, dict(lean=1)),                         # the lean epilogue writes only a bf16 output
        (lean, dict(bk32=1)),                            # BK 32 serves C_in <= 32
        (generic, dict(halo=1)),                         # a 1x1 conv has one tap
        (lean, dict(share=1)),                           # operand sharing is a split-path walk
        (split, dict(mb=2)),                             # the split paths run one m-block per tile
        (split, dict(epi_warps=8)),                      # ... and their two-level flush needs 16 epilogue warps
        (split, dict(bk32=0)),                           # ... and a fixed K-chunk width
        (split, dict(ctas_per_sm=2)),
        (lean, dict(mb=3)),                              # not a choice
    ]
    for cs, sc in cases:
        inp = make_inputs(cs, seed=1)
        run(ctx, cs, inp, schedule=sc, expect_rc=-1)
    inp = make_inputs(lean, seed=2)
    outs, _ = run(ctx, lean, inp, schedule=dict(ctas_per_sm=1, epi_warps=16, mb=1, resident=1))     # the context is still usable
    check(lean, outs, reference(lean, inp), what="after refusals")


@pytest.mark.gpu
def test_every_launch_variant_was_run(ctx):
    """The union of the launch reports of this file covers every variant of the launcher (run the whole file)."""
    expect = dict(bn={32, 64, 128}, mb={1, 2}, ctas_per_sm={1, 2}, epi_warps={8, 16}, issuers={1, 2}, resident={0, 1}, bk={32, 64},
                  halo={0, 1}, a_boxes={1, 2}, act_only={0, 1}, vec_ok={0, 1}, split={0, 1, 2}, flush={False, True}, tf32_share={0, 1},
                  ragged={0, 1})
    missing = {k: v - SEEN[k] for k, v in expect.items() if v - SEEN[k]}
    print("\nworst errors measured by this file:")
    for (g, k), v in sorted(WORST.items()):
        print(f"  {g:24s} {k:22s} {v:.3g}")
    assert not missing, f"launch variants never run: {missing} (seen {dict(SEEN)})"
