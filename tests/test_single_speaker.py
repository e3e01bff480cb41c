"""Single-speaker Matcha-TTS (n_spks = 1, the LJSpeech layout synthesis.ipynb loads): no speaker channels, so the text encoder
is 192 wide with two 96-wide heads and the decoder input is 160 channels (x | mu).

CPU: the oracle's single-speaker branches against the unmodified reference (skipped where the reference tree is absent).
GPU: the 96-wide encoder attention kernels alone against float64, the whole model against the oracle (synthesise, vocoder,
graph replay, training forward, estimator, corpus lanes), which kernels ran, and the refusal of a head width no kernel has."""
import dataclasses
import math

import pytest
import torch

from emojivoice_b200 import synthetic
from emojivoice_b200.config import HIFIGAN_V1, VCTK
from oracle import hifigan_oracle as ho
from oracle import matcha_oracle as mo
from oracle import reference_shim as shim
from tests.conftest import rel_l2

LJ = dataclasses.replace(VCTK, n_spks=1)
TOL = {"fp32": 1e-4, "bf16": 1e-2}
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def lj_sd():
    return synthetic.matcha_state_dict(LJ, seed=1234)


def test_layout():
    assert (LJ.enc_hidden, LJ.enc_hidden // LJ.enc_heads, LJ.dec_in) == (192, 96, 160)


# ------------------------------------------------------------------------------------------------ CPU: oracle vs reference
needs_reference = pytest.mark.skipif(not shim.available(), reason="/root/reference not present")


@needs_reference
def test_oracle_bit_equal_to_reference_synthesise_single_speaker(lj_sd):
    ref = shim.build_matcha(LJ, lj_sd)
    x, xl, _ = synthetic.phoneme_batch(3, 4, 14, seed=11)
    for ls in (0.8, 1.0, 1.2):
        probe = mo.synthesise(lj_sd, LJ, x, xl, 1, 0.667, None, ls)
        z = synthetic.prior_noise(3, 80, probe["t_pad"], seed=12)
        out = mo.synthesise(lj_sd, LJ, x, xl, 3, 0.667, None, ls, z=z)
        with shim.injected_noise(z):
            r = ref.synthesise(x, xl, n_timesteps=3, temperature=0.667, spks=None, length_scale=ls)
        assert torch.equal(out["mel_lengths"], r["mel_lengths"])
        for k in ("encoder_outputs", "decoder_outputs", "attn", "mel"):
            assert torch.equal(out[k], r[k]), (ls, k)


@needs_reference
def test_oracle_bit_equal_to_reference_training_forward_single_speaker(lj_sd):
    import random

    ref = shim.build_matcha(LJ, lj_sd).eval()
    for seed, out_size in ((31, None), (33, 16)):
        x, xl, _, y, yl = synthetic.training_batch(3, 4, 14, seed, LJ.n_feats)
        torch.manual_seed(seed)
        random.seed(seed)
        with torch.no_grad():
            dur, prior, diff, attn = ref(x, xl, y, yl, spks=None, out_size=out_size)
        torch.manual_seed(seed)
        random.seed(seed)
        off = None
        if out_size is not None:           # the reference's draw, matcha_tts.py:213-216
            mx = (yl - out_size).clamp(0).tolist()
            off = torch.tensor([random.choice(range(0, e)) if e > 0 else 0 for e in mx])
        t = torch.rand([x.shape[0], 1, 1])
        z = torch.randn(x.shape[0], LJ.n_feats, out_size or y.shape[-1])
        o = mo.forward_losses(lj_sd, LJ, x, xl, y, yl, None, out_size=out_size, t=t, z=z, out_offset=off)
        assert torch.equal(o["attn"], attn)
        assert torch.equal(o["dur_loss"], dur) and torch.equal(o["prior_loss"], prior) and torch.equal(o["diff_loss"], diff)


# ------------------------------------------------------------------------------------------------ GPU fixtures
@pytest.fixture(scope="module")
def ctx():
    from emojivoice_b200 import _lib

    return _lib.Context()


@pytest.fixture(scope="module")
def model(lj_sd):
    import emojivoice_b200 as ev

    m = ev.MatchaTTS(**LJ.constructor_kwargs())
    m.load_state_dict(lj_sd)
    return m


@pytest.fixture(scope="module")
def vocoder():
    import emojivoice_b200 as ev

    sd = synthetic.hifigan_state_dict(HIFIGAN_V1, seed=4321, gain=1.0)
    g = ev.Generator(HIFIGAN_V1)
    g.load_state_dict(sd)
    g.remove_weight_norm()
    return g, sd


# ------------------------------------------------------------------------------------------------ GPU: the kernel alone
@gpu
@pytest.mark.parametrize("impl", [0, 1])
@pytest.mark.parametrize("case", [(3, 177, 2), (2, 64, 2), (1, 1, 2), (2, 129, 1), (2, 300, 2), (1, 384, 2), (2, 65, 2), (2, 700, 2)])
def test_encoder_attention_head_width_96_matches_float64(ctx, case, impl):
    """text_encoder.py:223-246 in float64 at head width 96: RoPE on the first 48 features (pairs d, d + 24), scores / sqrt(96),
    -1e4 where the query OR the key is padded.  impl 0 = fp32 CUDA cores, 1 = tcgen05 with 3xFP16 split operands."""
    from emojivoice_b200 import _lib

    B, T, H = case
    hd = 96
    g = torch.Generator().manual_seed(7 * B + T + 96)
    qkv = torch.randn(B, T, 3 * H * hd, generator=g) * 1.7
    lens = torch.randint(1, T + 1, (B,), generator=g)
    lens[0] = T
    if B > 2:
        lens[1] = 1
    q, k, v = (z.reshape(B, T, H, hd).transpose(1, 2).double() for z in qkv.chunk(3, dim=2))
    q, k = mo._rope(q, hd // 2).double(), mo._rope(k, hd // 2).double()
    m = (torch.arange(T)[None, :] < lens[:, None]).double()
    scores = (q @ k.transpose(-2, -1)) / math.sqrt(hd)
    scores = scores.masked_fill((m[:, None, :, None] * m[:, None, None, :]) == 0, -1e4)
    ref = (torch.softmax(scores, dim=-1) @ v).transpose(1, 2).reshape(B, T, H * hd)
    out = torch.full((B, T, H * hd), float("nan"), device="cuda")
    qd, ld = qkv.cuda(), lens.cuda()
    ctx.check(_lib.lib().ev_test_encoder_attention_hd(ctx.handle, _lib.ptr(qd), _lib.ptr(ld), B, T, H, hd, impl, _lib.ptr(out), 0,
                                                      None, _lib.stream_ptr()), "ev_test_encoder_attention_hd")
    assert torch.isfinite(out).all()
    valid = m.bool()[:, :, None].expand_as(ref)
    assert rel_l2(out.cpu()[valid], ref[valid]) < 2e-6
    assert rel_l2(out.cpu(), ref) < 2e-6                  # padded queries: a uniform softmax, the mean of v


@gpu
def test_encoder_attention_hook_refuses_widths_without_a_kernel(ctx):
    from emojivoice_b200 import _lib

    qkv = torch.zeros(1, 8, 3 * 2 * 64, device="cuda")
    out = torch.zeros(1, 8, 2 * 64, device="cuda")
    for hd, impl in ((64, 1), (48, 0), (48, 1)):
        rc = _lib.lib().ev_test_encoder_attention_hd(ctx.handle, _lib.ptr(qkv), None, 1, 8, 2, hd, impl, _lib.ptr(out), 0, None,
                                                     _lib.stream_ptr())
        assert rc != 0, (hd, impl)
    ctx.check(_lib.lib().ev_test_encoder_attention_hd(ctx.handle, _lib.ptr(qkv), None, 1, 8, 2, 64, 0, _lib.ptr(out), 0, None,
                                                      _lib.stream_ptr()), "ev_test_encoder_attention_hd")


# ------------------------------------------------------------------------------------------------ GPU: end to end vs the oracle
def _pick(sd, make, ls):
    """The first of five seeded batches whose oracle durations hold no near-tie token (|w - round(w)| < 1e-4, where a last-ulp
    difference of exp() may legitimately flip a ceil) -> x, x_lengths, t_pad"""
    for seed in range(int(ls * 100), int(ls * 100) + 5000, 1000):
        x, xl = make(seed)
        ref = mo.synthesise(sd, LJ, x, xl, 1, 0.667, None, ls)
        w = torch.exp(ref["logw"]) * ref["x_mask"]
        if not bool((((w - torch.round(w)).abs() < 1e-4) & (ref["x_mask"] > 0)).any()):
            return x, xl, ref["t_pad"]
    raise AssertionError("no near-tie-free batch among 5 seeds")


def _check(out, ref, prec):
    assert torch.equal(out["w_ceil"].cpu(), ref["w_ceil"])
    assert out["mel_lengths"].cpu().tolist() == ref["mel_lengths"].tolist()
    assert torch.equal(out["attn"].cpu(), ref["attn"])
    assert rel_l2(out["mel"].cpu(), ref["mel"]) < TOL[prec]
    assert rel_l2(out["decoder_outputs_full"].cpu(), ref["decoder_outputs_full"]) < TOL[prec]


def _tx151(seed):
    x, xl, _ = synthetic.phoneme_batch(1, 75, 75, seed=seed)     # Tx = 2 * 75 + 1
    return x, xl


def _ragged(seed):
    x, xl, _ = synthetic.phoneme_batch(3, 20, 40, seed=seed)
    x[1] = 0
    xl[1] = 1                                            # a one-token item (a lone blank)
    return x, xl


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", ["b1_tx151", "ragged_b3"])
@pytest.mark.parametrize("n", [2, 10])
def test_synthesise_matches_oracle(model, lj_sd, shape, n, prec):
    x, xl, t_pad = _pick(lj_sd, _tx151 if shape == "b1_tx151" else _ragged, 1.0)
    assert x.shape[1] == (151 if shape == "b1_tx151" else int(xl.max())) and int(xl.min()) == (151 if shape == "b1_tx151" else 1)
    z = synthetic.prior_noise(x.shape[0], 80, t_pad, seed=152)
    ref = mo.synthesise(lj_sd, LJ, x, xl, n, 0.667, None, 1.0, z=z)
    out = model.synthesise(x, xl, n, 0.667, None, 1.0, z=z, dtype=prec)
    _check(out, ref, prec)
    assert rel_l2(out["mu_x"].cpu(), ref["mu_x"]) < 2e-5


@gpu
@pytest.mark.parametrize("ls", [0.8, 1.0, 1.2])
def test_length_scales_match_oracle(model, lj_sd, ls):
    x, xl, t_pad = _pick(lj_sd, lambda seed: synthetic.phoneme_batch(4, 10, 60, seed=seed)[:2], ls)
    z = synthetic.prior_noise(4, 80, t_pad, seed=153)
    ref = mo.synthesise(lj_sd, LJ, x, xl, 2, 0.667, None, ls, z=z)
    for prec in ("fp32", "bf16"):
        _check(model.synthesise(x, xl, 2, 0.667, None, ls, z=z, dtype=prec), ref, prec)


@gpu
def test_waveform_through_v1_vocoder_and_graph_replay(model, lj_sd, vocoder):
    gen, hsd = vocoder
    x, xl, t_pad = _pick(lj_sd, _ragged, 1.0)
    z = synthetic.prior_noise(3, 80, t_pad, seed=154)
    ref = mo.synthesise(lj_sd, LJ, x, xl, 4, 0.667, None, 1.0, z=z)
    ref_wav = ho.generator(hsd, HIFIGAN_V1, ref["mel"])
    for prec in ("fp32", "bf16"):
        runs = [model.synthesise(x, xl, 4, 0.667, None, 1.0, z=z, dtype=prec) for _ in range(3)]   # eager, capture, replay
        _check(runs[0], ref, prec)
        for k in ("mel", "decoder_outputs_full", "attn", "mu_x"):
            assert torch.equal(runs[0][k], runs[2][k]), (prec, k)
        lens = runs[0]["mel_lengths"]
        wav = gen(runs[0]["mel"], dtype=prec, lengths=lens)
        for b, nf in enumerate(lens.cpu().tolist()):
            assert rel_l2(wav[b, :, : nf * 256].cpu(), ref_wav[b, :, : nf * 256]) < TOL[prec], (prec, b)
            assert float(wav[b, :, nf * 256:].abs().sum()) == 0.0


@gpu
def test_intended_kernels_ran(model):
    """bf16 synthesise: the encoder attention ran on tcgen05 (no fp32 fallback), and the first ResNet block (C_in = 160) through
    the fused resnet_tc kernel like the other five."""
    x, xl, _ = synthetic.phoneme_batch(2, 30, 75, seed=155)
    model.cuda_graphs = False
    try:
        model._ctx.profile_begin()
        model.synthesise(x, xl, 2, 0.667, None, 1.0, dtype="bf16")
        torch.cuda.synchronize()
        stats = {s["name"]: s["launches"] for s in model._ctx.profile_end()}
    finally:
        model.cuda_graphs = True
    names = " ".join(stats)
    assert "attention_enc_tc" in names and "attention_enc_f32" not in names, stats
    rn = sum(v for k, v in stats.items() if k.startswith("resnet_tc"))
    assert rn == 6 * 2, stats                            # six ResNet blocks per step, every one fused
    assert not any(k.startswith("gn_stats") or k.startswith("gn_apply") for k in stats), stats


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_training_forward_and_estimator_match_oracle(model, lj_sd, prec):
    import random

    x, xl, _, y, yl = synthetic.training_batch(4, 10, 40, 71, LJ.n_feats)
    t, z = synthetic.training_draws(4, LJ.n_feats, y.shape[-1], 72)
    o = mo.forward_losses(lj_sd, LJ, x, xl, y, yl, None, t=t, z=z)
    dur, prior, diff, attn = model.forward(x, xl, y, yl, spks=None, t=t, z=z, dtype=prec)
    assert torch.equal(attn.cpu(), o["attn"])
    rel = lambda a, b: abs(float(a) - float(b)) / max(abs(float(b)), 1e-30)
    assert rel(dur, o["dur_loss"]) < 1e-4 and rel(prior, o["prior_loss"]) < 1e-4 and rel(diff, o["diff_loss"]) < TOL[prec]
    v = model.decoder.estimator(o["y_t"], o["y_mask"], o["mu_y"], t, None, dtype=prec)
    assert torch.isfinite(v).all()
    if prec == "fp32":
        assert rel_l2(v.cpu(), o["v"]) < 1e-4
    # a random crop (out_size) as the reference's training step draws it
    random.seed(5)
    out_size = 16
    off = torch.tensor([random.choice(range(0, e)) if e > 0 else 0 for e in (yl - out_size).clamp(0).tolist()])
    t2, z2 = synthetic.training_draws(4, LJ.n_feats, out_size, 73)
    o2 = mo.forward_losses(lj_sd, LJ, x, xl, y, yl, None, out_size=out_size, t=t2, z=z2, out_offset=off)
    dur2, prior2, diff2, attn2 = model.forward(x, xl, y, yl, out_size=out_size, t=t2, z=z2, out_offset=off, dtype=prec)
    assert torch.equal(attn2.cpu(), o2["attn"])
    assert rel(prior2, o2["prior_loss"]) < 1e-4 and rel(diff2, o2["diff_loss"]) < TOL[prec]


@gpu
def test_corpus_lanes_do_not_change_results(model, vocoder):
    import emojivoice_b200 as ev

    gen, _ = vocoder
    x, xl, _ = synthetic.phoneme_batch(8, 5, 30, seed=156)
    utts = [(x[i, : int(xl[i])].tolist(), 0) for i in range(8)]
    zs = {}

    def z_fn(mb, m, x_, xl_, spks_):
        probe = m.synthesise(x_, xl_, 1, 0.667, None, 1.0)
        return zs.setdefault(tuple(mb.items), synthetic.prior_noise(len(mb.items), 80, probe["t_pad"], seed=157))

    r1, s1 = ev.synthesise_corpus(model, gen, utts, batch_size=2, n_timesteps=2, z_fn=z_fn)
    r2, s2 = ev.synthesise_corpus(model, gen, utts, batch_size=2, n_timesteps=2, z_fn=z_fn, in_flight=2)
    assert sorted(r1) == sorted(r2) == list(range(8)) and s1.utterances == s2.utterances == 8
    for i in r1:
        assert r1[i]["mel_length"] == r2[i]["mel_length"]
        assert torch.equal(r1[i]["waveform"], r2[i]["waveform"])


@gpu
def test_head_width_without_a_kernel_is_refused_at_load(model):
    import emojivoice_b200 as ev

    cfg = dataclasses.replace(LJ, enc_heads=4)           # 192 channels / 4 heads = 48-wide heads
    m = ev.MatchaTTS(**cfg.constructor_kwargs())
    with pytest.raises(RuntimeError, match="head width"):
        m.load_state_dict(synthetic.matcha_state_dict(cfg, seed=5))
    x, xl, _ = synthetic.phoneme_batch(1, 3, 3, seed=158)
    out = model.synthesise(x, xl, 2, 0.667, None, 1.0)    # the device is still usable
    torch.cuda.synchronize()
    assert torch.isfinite(out["mel"]).all()


@gpu
def test_load_from_checkpoint_single_speaker(model, lj_sd, tmp_path):
    """A Lightning-style checkpoint of a single-speaker model (hyper_parameters + state_dict) loads and synthesises like the model
    built from the constructor kwargs, bit for bit."""
    import emojivoice_b200 as ev

    path = tmp_path / "lj.ckpt"
    torch.save({"hyper_parameters": LJ.constructor_kwargs(), "state_dict": lj_sd}, path)
    m = ev.MatchaTTS.load_from_checkpoint(str(path), map_location="cuda:0")
    assert m.n_spks == 1
    x, xl, _ = synthetic.phoneme_batch(2, 5, 20, seed=159)
    probe = model.synthesise(x, xl, 1, 0.667, None, 1.0)
    z = synthetic.prior_noise(2, 80, probe["t_pad"], seed=160)
    a = model.synthesise(x, xl, 3, 0.667, None, 1.0, z=z)
    b = m.synthesise(x, xl, 3, 0.667, None, 1.0, z=z)
    assert torch.equal(a["mel"], b["mel"]) and torch.equal(a["attn"], b["attn"])
