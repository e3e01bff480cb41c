"""The fused HiFi-GAN ResBlock kernel (resblock_tc.cu) and the layer-by-layer ResBlock path, each alone through
ev_test_resblock, against a float64 ResBlock1 (hifigan/models.py:90-97) and the multi-receptive-field mean (:186-192).

The reference applies the kernel's roundings and nothing else: bf16 lrelu(x), bf16 weights, bf16 lrelu(conv1 + b1), exact
biases and residual stream, act = bf16(lrelu((sum + y) * inv_n, slope)).  A global rel-L2 bound alone misses the errors this
kernel is prone to -- a halo exchange that does not land touches a few rows next to one window boundary -- so every
comparison also bounds the worst row, sqrt(mean_c err^2) / rms(ref).  The CPU tests at the top show that the bounds accept
an fp32 emulation of the kernel and reject a set of planted bugs; they need no GPU."""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as F

DIL = (1, 3, 5)
SLOPE = 0.1                       # LRELU_SLOPE, hifigan/models.py:11
TOL_BF16 = (1.5e-3, 1e-2)         # (rel-L2, worst row): bf16 operands, fp32 accumulation
TOL_BIAS = (1e-4, 5e-4)           # bias-dominated input: the bf16 hi + lo bias split keeps the bias to ~2^-17
TOL_FP32 = (2e-6, 2e-5)           # fp32 layer-by-layer path


def bf(t):
    return t.to(torch.bfloat16).to(t.dtype)


def lrelu(t, slope=SLOPE):
    return torch.where(t > 0, t, t * slope)


def block_weights(C, k, seed, bias_dominated=False):
    """Unit-gain weights and small biases, or (bias_dominated) weak weights and biases of 5 +- 3."""
    g = torch.Generator().manual_seed(seed)
    w = {}
    for l in range(3):
        for name in ("convs1", "convs2"):
            scale = (C * k) ** -0.5 * (0.1 if bias_dominated else 1.0)
            w[f"{name}.{l}.weight"] = torch.randn(C, C, k, generator=g) * scale
            w[f"{name}.{l}.bias"] = torch.randn(C, generator=g) * 3 + 5 if bias_dominated else torch.randn(C, generator=g) * 0.1
    return w


def block_input(B, C, L, seed, scale=0.5):
    return torch.randn(B, C, L, generator=torch.Generator().manual_seed(seed)) * scale


def reference(x, w, k, *, sum_in=None, mode=0, inv_n=1.0, slope_out=SLOPE, dtype=torch.float64, bf16_ops=True, bias_round=None,
              drop_bias=None, halo_cut=None):
    """ResBlock1 + the MRF step in `dtype`.  x (B, C, L) -> (sum, act) as (B, L, C); act is None unless mode == 2.
    bf16_ops: round operands and act like the tensor-core path.  bias_round, drop_bias, halo_cut plant bugs (see the CPU tests)."""
    rnd = bf if bf16_ops else (lambda t: t)
    xs = x.to(dtype)
    for l in range(3):
        d = DIL[l]
        w1, w2 = (rnd(w[f"convs{i}.{l}.weight"].to(dtype)) for i in (1, 2))
        b1, b2 = (w[f"convs{i}.{l}.bias"].to(dtype) for i in (1, 2))
        if bias_round is not None:
            b1, b2 = bias_round(b1), bias_round(b2)
        if drop_bias == l:
            b2 = torch.zeros_like(b2)
        a = rnd(lrelu(F.conv1d(rnd(lrelu(xs)), w1, b1, padding=(k * d - d) // 2, dilation=d)))
        y = F.conv1d(a, w2, b2, padding=(k - 1) // 2)
        if halo_cut is not None and l == 2:
            # the 32 edge rows the right neighbour pushes before the last conv never arrive: the left CTA's rows see zeros there
            a_bad = a.clone()
            a_bad[..., halo_cut:halo_cut + 32] = 0
            y[..., :halo_cut] = F.conv1d(a_bad, w2, b2, padding=(k - 1) // 2)[..., :halo_cut]
        xs = xs + y
    s = xs.transpose(1, 2)
    if mode >= 1:
        s = sum_in.to(dtype) + s
    if mode == 2:
        s = s * inv_n
        return s, rnd(lrelu(s, slope_out))
    return s, None


def block_errors(got, ref):
    """(rel-L2, worst row) of got against ref, both (B, L, C); a row is one (b, t)."""
    err = got.double() - ref.double()
    rms = ref.double().pow(2).mean().sqrt().clamp_min(1e-30)
    rel = err.norm() / ref.double().norm().clamp_min(1e-30)
    row = err.pow(2).mean(-1).sqrt().max() / rms
    return float(rel), float(row)


def check_block(sum_out, act_out, ref_sum, ref_act, *, mode, write_f32=1, sum_in=None, tol=TOL_BF16, what=""):
    """The one check every ResBlock result passes.  sum_out / act_out: what the call returned, (B, L, C) fp32 (act_out may be
    None when it was not returned).  Rows t < L must be finite and within tol; outputs the call must not write must still hold
    the NaN fill (act_out in modes 0 and 1 and when not requested); sum with write_f32 = 0 in mode 2 must equal sum_in bit for bit."""
    rel_tol, row_tol = tol

    def compare(got, ref, name):
        bad = (~torch.isfinite(got)).any(-1)
        assert not bad.any(), f"{what}: {name} has {int(bad.sum())} non-finite rows, first (b, t) = {bad.nonzero()[0].tolist()}"
        rel, row = block_errors(got, ref)
        assert rel <= rel_tol and row <= row_tol, f"{what}: {name} rel-L2 {rel:.3g} (<= {rel_tol}), worst row {row:.3g} (<= {row_tol})"

    if mode == 2 and not write_f32:
        assert torch.equal(sum_out.view(torch.int32), sum_in.float().view(torch.int32)), f"{what}: sum written although write_f32 = 0"
    else:
        compare(sum_out, ref_sum, "sum")
    if act_out is not None:
        if ref_act is None:
            assert torch.isnan(act_out).all(), f"{what}: act written in mode {mode} or without being requested"
        else:
            compare(act_out, ref_act, "act")


# ------------------------------------------------------------------------------------------------ the bounds, without a GPU
EMUL_SHAPES = [(32, 11, 4096), (64, 7, 2048), (128, 11, 1024)]


def _emulation(C, k, L, seed):
    """fp32 with the kernel's roundings (the error a correct kernel has) and the float64 reference, dense mode 0."""
    w = block_weights(C, k, seed)
    x = block_input(1, C, L, seed + 1)
    ref, _ = reference(x, w, k)
    emu, _ = reference(x, w, k, dtype=torch.float32)
    return w, x, ref, emu


@pytest.mark.parametrize("C,k,L", EMUL_SHAPES)
def test_check_accepts_fp32_emulation_and_rejects_planted_bugs(C, k, L):
    w, x, ref, emu = _emulation(C, k, L, seed=C + k)
    check_block(emu, None, ref, None, mode=0, what="fp32 emulation")
    cut = L // 2
    halo, _ = reference(x, w, k, halo_cut=cut)                           # 1. one missing halo exchange
    shifted = ref.clone()                                                # 3. the stored rows of one window one row off
    shifted[:, cut:cut + 200] = ref[:, cut + 1:cut + 201]
    dropped, _ = reference(x, w, k, drop_bias=1)                         # 4. one conv2 bias left out
    unwritten = ref.clone()                                              # 5. one row never written (NaN fill)
    unwritten[0, cut] = float("nan")
    for name, bad in [("halo", halo), ("shifted window", shifted), ("conv2 bias dropped", dropped), ("row unwritten", unwritten)]:
        with pytest.raises(AssertionError):
            check_block(bad, None, ref, None, mode=0, what=name)


@pytest.mark.parametrize("C", [32, 128])
def test_check_rejects_a_bias_without_its_low_half(C):
    """2. The bias of a conv as bf16 hi only: invisible at unit gain, 1e-3 on a bias-dominated block."""
    k, L = 7, 1024
    w = block_weights(C, k, seed=5, bias_dominated=True)
    x = block_input(1, C, L, seed=6, scale=0.05)
    ref, _ = reference(x, w, k)
    hilo = lambda b: bf(b) + bf(b - bf(b))
    check_block(reference(x, w, k, dtype=torch.float32, bias_round=hilo)[0], None, ref, None, mode=0, tol=TOL_BIAS, what="hi + lo bias")
    with pytest.raises(AssertionError):
        check_block(reference(x, w, k, dtype=torch.float32, bias_round=bf)[0], None, ref, None, mode=0, tol=TOL_BIAS, what="hi-only bias")


def test_check_covers_mode_two_outputs():
    C, k, L = 32, 3, 600
    w = block_weights(C, k, seed=9)
    x = block_input(2, C, L, seed=10)
    sum_in = torch.randn(2, L, C, generator=torch.Generator().manual_seed(11))
    ref, act = reference(x, w, k, sum_in=sum_in, mode=2, inv_n=1 / 3)
    emu, emu_act = reference(x, w, k, sum_in=sum_in, mode=2, inv_n=1 / 3, dtype=torch.float32)
    check_block(emu, emu_act, ref, act, mode=2, what="mode 2")
    check_block(sum_in.clone(), emu_act, ref, act, mode=2, write_f32=0, sum_in=sum_in, what="mode 2, no fp32 write")
    with pytest.raises(AssertionError):
        check_block(emu, emu_act, ref, act, mode=2, write_f32=0, sum_in=sum_in, what="sum written")
    with pytest.raises(AssertionError):
        check_block(emu, torch.zeros_like(emu), ref, None, mode=1, what="act written in mode 1")


# ------------------------------------------------------------------------------------------------ the kernel on the GPU
def _W(C):
    return 256 if C == 128 else 512          # rows per CTA window (m-blocks x 128)


def _H(k):
    return 6 * (k - 1)                       # halo rows per window side: sum_l (k-1)/2 * (d_l + 1)


def _Wv(C, k, cl):
    return cl * _W(C) - 2 * _H(k)            # output rows per (cluster) window


SCHED_NAMES = ("cluster", "occ2", "wave", "resident")


def schedules(C):
    """Every forced alternative the launcher offers at C: single and paired windows; at C = 32 also one CTA per SM with resident
    weights (16 or, at k = 11, 8 epilogue warps), the wavefront schedule, and weights streamed through the ring."""
    out = [dict(cluster=1), dict(cluster=3)]
    if C == 32:
        out += [dict(cluster=1, occ2=0), dict(cluster=3, occ2=0), dict(occ2=0, wave=1),
                dict(cluster=1, occ2=0, resident=0), dict(cluster=3, occ2=0, resident=0)]
    return out


def expected_variants(C, k):
    """(CTAs per cluster, CTAs per SM, wavefront, resident weights, epilogue warps) of every kernel variant the launcher can pick."""
    if C != 32:
        return {(1, 1, 0, 0, 16), (2, 1, 0, 0, 16)}
    n_res = 8 if k == 11 else 16             # 6k resident 2 KB weight tiles beside 16 epilogue warps' buffers exceed 224 KB at k = 11
    return {(1, 2, 0, 0, 8), (2, 2, 0, 0, 8), (1, 1, 0, 1, n_res), (2, 1, 0, 1, n_res), (1, 1, 1, 1, n_res), (1, 1, 0, 0, 16), (2, 1, 0, 0, 16)}


@pytest.fixture(scope="module")
def ctx():
    from emojivoice_b200 import _lib

    return _lib.Context()


def run_block(ctx, w, x, k, *, sum_in=None, mode=0, inv_n=1.0, slope_out=SLOPE, write_f32=1, want_act=False, lengths=None, rpf=1, margin=0,
              impl=1, prec="bf16", schedule=None, expect_rc=0):
    """-> (sum, act, report) on the CPU; report = dict of what the fused kernel launched."""
    from emojivoice_b200 import _lib

    B, C, L = x.shape
    arr, keep = _lib.tensor_list(w, ctx.device)
    xd = x.contiguous().cuda()
    sd = None if sum_in is None else sum_in.float().contiguous().cuda()
    ld = None if lengths is None else torch.as_tensor(lengths, dtype=torch.int64).cuda()
    out, act = torch.empty(B, L, C, device="cuda"), torch.empty(B, L, C, device="cuda")
    sched = None
    if schedule is not None:
        sched = (ctypes.c_int32 * 4)(*[schedule.get(n, -1) for n in SCHED_NAMES])
    rep = (ctypes.c_int32 * 9)()
    rc = _lib.lib().ev_test_resblock(ctx.handle, arr, len(keep), C, k, _lib.ptr(xd), _lib.ptr(sd), B, L, mode, inv_n, slope_out, write_f32,
                                     int(want_act), _lib.ptr(ld), rpf, margin, impl, _lib.PREC[prec],
                                     None if sched is None else ctypes.cast(sched, ctypes.c_void_p), _lib.ptr(out), _lib.ptr(act),
                                     ctypes.cast(rep, ctypes.c_void_p), _lib.stream_ptr())
    if expect_rc:
        assert rc == expect_rc, f"expected {expect_rc}, got {rc}: {_lib.lib().ev_last_error(ctx.handle).decode()}"
        return None
    ctx.check(rc, f"ev_test_resblock C={C} k={k} L={L} schedule={schedule}")
    names = ("cl", "occ", "wave", "resident", "w_slots", "n_epi", "grid", "Wv", "total_tiles")
    return out.cpu(), act.cpu(), dict(zip(names, list(rep)))


def variant(rep):
    return rep["cl"], rep["occ"], rep["wave"], rep["resident"], rep["n_epi"]


def check_report(rep, C, k, B, L):
    """The launch report agrees with the kernel's geometry."""
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    cl, occ = rep["cl"], rep["occ"]
    assert rep["Wv"] == _Wv(C, k, cl), rep
    assert rep["total_tiles"] == B * math.ceil(L / rep["Wv"]), rep
    assert rep["grid"] == cl * min(rep["total_tiles"], occ * sms // cl), rep
    assert (rep["w_slots"] == 1) if rep["resident"] else (rep["w_slots"] >= 3), rep


def same_bits(a, b):
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


def lengths_for(C, k):
    """L = n Wv + r for both window widths, n Wv >= 1024 (the vocoder runs the fused kernel from L = 1024 on): r = 0 (windows end on
    L), 1 (a last window of one row), H (a last window that is all halo), W - H (the rank-1 CTA of the last cluster wholly past L),
    W, W + 1 (the interior / non-interior switch of the last CTA) and Wv - 1."""
    W, H, out = _W(C), _H(k), set()
    for cl in (1, 2):
        Wv = _Wv(C, k, cl)
        n = max(1, -(-1024 // Wv))
        for r in (0, 1, H, W - H, W, W + 1, Wv - 1):
            out.add(n * Wv + r)
    return sorted(out)


CK = [(C, k) for C in (32, 64, 128) for k in (3, 7, 11)]


@pytest.mark.gpu
@pytest.mark.parametrize("C,k", CK)
def test_fused_resblock_lengths_and_every_schedule(ctx, C, k):
    """Every length edge under the default policy and every forced schedule: the default result is checked against the
    reference, every schedule must reproduce it bit for bit (paired == single == wavefront == one / two CTAs per SM == resident /
    streamed weights: every row sums the same products in the same order), and together the calls hit every kernel variant
    the launcher can pick at this (C, k)."""
    w = block_weights(C, k, seed=100 * C + k)
    seen = set()
    for i, L in enumerate(lengths_for(C, k)):
        x = block_input(1, C, L, seed=1000 * C + 10 * k + i)
        ref, _ = reference(x, w, k)
        base, act, rep = run_block(ctx, w, x, k)
        check_report(rep, C, k, 1, L)
        seen.add(variant(rep))
        check_block(base, act, ref, None, mode=0, what=f"C={C} k={k} L={L} default {variant(rep)}")
        for sc in schedules(C):
            out, act, rep = run_block(ctx, w, x, k, schedule=sc)
            check_report(rep, C, k, 1, L)
            seen.add(variant(rep))
            assert same_bits(out, base), f"C={C} k={k} L={L}: schedule {sc} ({variant(rep)}) differs from the default"
            assert torch.isnan(act).all()
    assert seen == expected_variants(C, k), f"variants hit {sorted(seen)}, launcher variants {sorted(expected_variants(C, k))}"


@pytest.mark.gpu
@pytest.mark.parametrize("C", [32, 64, 128])
def test_fused_resblock_short_sequences(ctx, C):
    """Lengths below one window: a single row, a sequence shorter than one halo, one window exactly."""
    k = 11
    H, W = _H(k), _W(C)
    w = block_weights(C, k, seed=7 * C)
    for i, L in enumerate(sorted({1, 2, H - 1, H, H + 1, W - H, _Wv(C, k, 1) - 1, _Wv(C, k, 1), W, 2 * W - 2 * H - 1})):
        x = block_input(2, C, L, seed=31 * C + i)
        ref, _ = reference(x, w, k)
        base = None
        for sc in [None] + schedules(C):
            out, _, rep = run_block(ctx, w, x, k, schedule=sc)
            check_report(rep, C, k, 2, L)
            if base is None:
                check_block(out, None, ref, None, mode=0, what=f"C={C} L={L}")
                base = out
            else:
                assert same_bits(out, base), f"C={C} L={L}: schedule {sc} differs from the default"


@pytest.mark.gpu
@pytest.mark.parametrize("C,k,B,L,schedule", [
    (32, 3, 3, 201 * 488 - 7, None),                     # two CTAs per SM: 603 windows on 296 CTAs
    (32, 3, 3, 201 * 488 - 7, dict(occ2=0)),             # resident weights: 603 windows on 148 CTAs
    (64, 7, 2, 151 * 952 - 3, dict(cluster=3)),          # paired windows: 302 cluster windows on 74 clusters
])
def test_fused_resblock_more_windows_than_ctas(ctx, C, k, B, L, schedule):
    w = block_weights(C, k, seed=C + k + B)
    x = block_input(B, C, L, seed=L)
    out, _, rep = run_block(ctx, w, x, k, schedule=schedule)
    check_report(rep, C, k, B, L)
    assert rep["total_tiles"] > 2 * rep["grid"] // rep["cl"] and rep["total_tiles"] % (rep["grid"] // rep["cl"]), rep
    ref, _ = reference(x, w, k)
    check_block(out, None, ref, None, mode=0, what=f"C={C} k={k} B={B} L={L}")


def _mrf_stage(ctx, C, L, last, impl, prec, seed):
    """The three branches k = 3, 7, 11 of one generator stage: modes 0 -> 1 -> 2, inv_n = 1/3; a stage in the middle writes only
    the bf16 operand of the next stage (write_f32 = 0), the last one only the fp32 mean.  Each branch is compared with the
    reference given the same sum_in (the previous branch's result)."""
    tol = TOL_FP32 if prec == "fp32" else TOL_BF16
    x = block_input(2, C, L, seed=seed)
    sum_in = None
    for j, k in enumerate((3, 7, 11)):
        w = block_weights(C, k, seed=seed + k)
        mode = j
        write_f32 = 1 if (mode < 2 or last) else 0
        want_act = mode == 2 and not last
        out, act, _ = run_block(ctx, w, x, k, sum_in=sum_in, mode=mode, inv_n=1 / 3, write_f32=write_f32, want_act=want_act, impl=impl,
                                prec=prec)
        ref, ref_act = reference(x, w, k, sum_in=sum_in, mode=mode, inv_n=1 / 3, bf16_ops=prec == "bf16")
        check_block(out, act, ref, ref_act if want_act else None, mode=mode, write_f32=write_f32, sum_in=sum_in, tol=tol,
                    what=f"{prec} impl={impl} C={C} k={k} mode={mode}")
        sum_in = out


@pytest.mark.gpu
@pytest.mark.parametrize("last", [False, True])
@pytest.mark.parametrize("C", [32, 64, 128])
def test_fused_mrf_stage(ctx, C, last):
    _mrf_stage(ctx, C, 1500, last, impl=1, prec="bf16", seed=C + 17 * last)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["bf16", "fp32"])
@pytest.mark.parametrize("C", [32, 64, 128, 256])
def test_layer_by_layer_resblock_path(ctx, C, prec):
    """The six conv launches with their fused epilogues (residual, MRF accumulator, division by n, the next stage's lrelu) --
    the path every C = 256 block and the fp32 vocoder take."""
    for last in (False, True):
        _mrf_stage(ctx, C, 700 if C == 256 else 1100, last, impl=0, prec=prec, seed=3 * C + last)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [32, 64, 128])
def test_fused_resblock_bias_dominated(ctx, C):
    """Biases of 5 +- 3 under weak weights and a small input: the bias reaches the result at its own precision."""
    k, L = 7, 1500
    w = block_weights(C, k, seed=C, bias_dominated=True)
    x = block_input(1, C, L, seed=C + 1, scale=0.05)
    ref, _ = reference(x, w, k)
    for sc in (dict(cluster=1), dict(cluster=3)):
        out, _, rep = run_block(ctx, w, x, k, schedule=sc)
        check_block(out, None, ref, None, mode=0, tol=TOL_BIAS, what=f"C={C} {variant(rep)}")


@pytest.mark.gpu
@pytest.mark.parametrize("C,k", [(32, 11), (64, 3), (128, 7)])
def test_fused_resblock_ragged_batch(ctx, C, k):
    """Compact window lists: rows below len * rows_per_frame equal the dense call bit for bit; every other row is either equal
    too (its window was computed) or still holds the NaN fill (skipped)."""
    rpf, margin = 64, 2
    L = 40 * rpf
    frames = [0, 1, 40, 17]
    w = block_weights(C, k, seed=C * k)
    x = block_input(len(frames), C, L, seed=C * k + 1)
    for sc in (dict(cluster=1), dict(cluster=3)):
        dense, _, _ = run_block(ctx, w, x, k, schedule=sc)
        rag, _, _ = run_block(ctx, w, x, k, schedule=sc, lengths=frames, rpf=rpf, margin=margin)
        for b, n in enumerate(frames):
            valid = n * rpf
            assert same_bits(rag[b, :valid], dense[b, :valid]), f"item {b} ({n} frames), schedule {sc}"
            rest_equal = (rag[b, valid:].view(torch.int32) == dense[b, valid:].view(torch.int32)).all(-1)
            rest_nan = torch.isnan(rag[b, valid:]).all(-1)
            assert (rest_equal | rest_nan).all(), f"item {b} ({n} frames), schedule {sc}: rows past the needed ones hold other values"
        assert torch.isnan(rag[0]).any(), "no window was skipped"


@pytest.mark.gpu
def test_forced_schedule_that_cannot_run_is_refused(ctx):
    """A forced schedule is launched as asked or refused (EV_ERR_INVALID); so are shapes the fused kernel does not take."""
    L = 1100
    cases = [(32, 3, dict(wave=1)),                          # two CTAs per SM stream their weights: no wavefront
             (32, 11, dict(resident=1)),                     # ... and do not keep them resident
             (32, 3, dict(occ2=0, wave=1, cluster=3)),       # the wavefront schedule keeps single windows
             (64, 7, dict(wave=1)), (64, 7, dict(occ2=1)), (128, 3, dict(resident=1))]
    for C, k, sc in cases:
        run_block(ctx, block_weights(C, k, seed=1), block_input(1, C, L, seed=2), k, schedule=sc, expect_rc=-1)
    run_block(ctx, block_weights(256, 3, seed=1), block_input(1, 256, L, seed=2), 3, expect_rc=-1)       # C = 256: layer by layer only
    run_block(ctx, block_weights(64, 5, seed=1), block_input(1, 64, L, seed=2), 5, expect_rc=-1)         # k = 5
    run_block(ctx, block_weights(64, 3, seed=1), block_input(1, 64, L, seed=2), 3, prec="fp32", expect_rc=-1)   # fp32 is not fused
    # the context is still usable
    w, x = block_weights(32, 3, seed=3), block_input(1, 32, L, seed=4)
    out, _, _ = run_block(ctx, w, x, 3, schedule=dict(occ2=0, wave=1))
    check_block(out, None, reference(x, w, 3)[0], None, mode=0, what="after refusals")
