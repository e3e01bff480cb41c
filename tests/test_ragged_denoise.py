"""Ragged vocoder + denoiser (ev_to_waveform_ragged, ev_denoise_ragged, Generator.vocode_denoised, Denoiser(lengths=)): on a
padded batch, each utterance's denoised samples [: len_b*256] must equal the dense path -- vocoder(mel).clamp(-1, 1), then the
denoiser over the whole padded waveform -- bit for bit, with zeros beyond, while only the frames those samples reach are computed.

CPU: the reach of the denoised samples into the audio, on the oracle (torch.stft / torch.istft, hifigan/denoiser.py).
GPU: bit-identity against the dense path, graph replay, the corpus driver, the work skipped, refusals."""
import ctypes as C

import pytest
import torch

from emojivoice_b200.hifigan import check_lengths
from oracle import hifigan_oracle as ho

HOP = 256


# ------------------------------------------------------------------------------------------------ CPU: reach on the oracle
@pytest.mark.parametrize("strength", [0.1, 1.0])
def test_denoised_samples_read_no_audio_at_or_past_len_plus_3_frames(strength):
    """Output sample t < len*256 is an overlap-add of STFT frames f <= len + 1, whose windows end below (len + 3)*256: audio
    there and beyond does not reach [: len*256], while a large change at (len + 3)*256 - 1 does.  Lengths T-4 .. T are where
    the row end clips the margin.  (Pairing adds one frame in the kernel; the GPU tests cover that.)"""
    T = 24
    g = torch.Generator().manual_seed(11)
    audio = (torch.rand(2, T * HOP, generator=g) - 0.5)
    bias = torch.rand(1, 513, 1, generator=g) * 1.5 + 0.5
    base = ho.denoise(audio, bias, strength)
    for n in [1, 2, 7, 8, T - 4, T - 3, T - 2, T - 1, T]:
        cut = (n + 3) * HOP
        if cut < T * HOP:
            far = audio.clone()
            far[:, cut:] += torch.randn(2, T * HOP - cut, generator=g) * 10.0
            assert torch.equal(ho.denoise(far, bias, strength)[:, : n * HOP], base[:, : n * HOP]), n
        if cut - 1 < T * HOP:
            edge = audio.clone()
            edge[:, cut - 1] += 1000.0
            assert not torch.equal(ho.denoise(edge, bias, strength)[:, : n * HOP], base[:, : n * HOP]), n


def test_host_lengths_outside_one_to_T_are_refused():
    check_lengths([1, 5, 10], 10)
    check_lengths(torch.tensor([10]), 10)
    for bad in ([0, 5], [1, 11], torch.tensor([-1])):
        with pytest.raises(ValueError):
            check_lengths(bad, 10)
    with pytest.raises(ValueError):
        check_lengths(None, 10)


# ------------------------------------------------------------------------------------------------ GPU
STRENGTHS = (0.00025, 0.0005, 0.1)


@pytest.fixture(scope="module")
def gen_den():
    import emojivoice_b200 as ev
    from emojivoice_b200 import synthetic
    from emojivoice_b200.config import HIFIGAN_V1

    g = ev.Generator(HIFIGAN_V1)
    g.load_state_dict(synthetic.hifigan_state_dict(HIFIGAN_V1, seed=4321, gain=1.0))
    g.remove_weight_norm()
    return g, ev.Denoiser(g)


def _mel(B, T, seed):
    from emojivoice_b200 import synthetic

    return synthetic.synthetic_mel(B, T, seed=seed)


def _check(fused, dense, lens):
    assert fused.shape == (dense.shape[0], 1, dense.shape[1])
    for b, n in enumerate(lens):
        n = max(0, min(int(n), dense.shape[1] // HOP)) * HOP
        assert torch.equal(fused[b, 0, :n], dense[b, :n]), (lens, b)
        if n < dense.shape[1]:
            assert float(fused[b, 0, n:].abs().max()) == 0.0, (lens, b)


LEN_CASES = {
    # odd and even lengths, lengths within 4 frames of T, 1- and 2-frame utterances next to long ones
    "mixed": (300, [137, 138, 299, 296, 1, 2]),
    "near_end": (300, [300, 297, 298, 299, 296, 295]),
    "b1_full": (50, [50]),
    "b1_short": (50, [37]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("case", list(LEN_CASES))
def test_vocode_denoised_equals_dense_path(gen_den, prec, case):
    gen, den = gen_den
    T, lens = LEN_CASES[case]
    mel = _mel(len(lens), T, seed=90 + T)
    wav = gen(mel, dtype=prec).clamp(-1, 1).squeeze(1)
    for strength in STRENGTHS:
        dense = den(wav, strength=strength)
        _check(gen.vocode_denoised(mel, torch.tensor(lens), strength, dtype=prec), dense, lens)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_vocode_denoised_config2_shape(gen_den, prec):
    """32 utterances of 368-548 frames padded to 668 (BASELINE config 2)."""
    gen, den = gen_den
    g = torch.Generator().manual_seed(5)
    lens = torch.randint(368, 549, (32,), generator=g).tolist()
    lens[0], lens[1] = 548, 369
    mel = _mel(32, 668, seed=91)
    dense = den(gen(mel, dtype=prec).clamp(-1, 1).squeeze(1), strength=0.00025)
    _check(gen.vocode_denoised(mel, lens, 0.00025, dtype=prec), dense, lens)


@pytest.mark.gpu
def test_vocode_denoised_graph_replay(gen_den):
    """Eager, capture, replay; and replays of one graph with other lengths follow those lengths."""
    gen, den = gen_den
    T = 120
    mel = _mel(4, T, seed=92)
    dense = den(gen(mel).clamp(-1, 1).squeeze(1), strength=0.00025)
    before = len(gen._graphs.entries)
    for lens in ([120, 3, 61, 118], [120, 3, 61, 118], [120, 3, 61, 118], [1, 2, 119, 60], [117, 120, 4, 5]):
        _check(gen.vocode_denoised(mel, torch.tensor(lens).cuda(), 0.00025), dense, lens)
    assert len(gen._graphs.entries) == before + 1


@pytest.mark.gpu
def test_device_lengths_are_clamped_to_zero_and_T(gen_den):
    gen, den = gen_den
    T = 40
    mel = _mel(3, T, seed=93)
    dense = den(gen(mel).clamp(-1, 1).squeeze(1), strength=0.0005)
    got = gen.vocode_denoised(mel, torch.tensor([T + 9, 0, -3]).cuda(), 0.0005)
    _check(got, dense, [T, 0, 0])


@pytest.mark.gpu
def test_denoiser_with_lengths_equals_dense_call(gen_den):
    gen, den = gen_den
    T = 200
    lens = [200, 1, 2, 77, 198, 150]
    wav = gen(_mel(6, T, seed=94)).clamp(-1, 1).squeeze(1)
    for strength in STRENGTHS:
        _check(den(wav, strength=strength, lengths=lens).unsqueeze(1), den(wav, strength=strength), lens)
        _check(den(wav, strength=strength, lengths=torch.tensor(lens).cuda()).unsqueeze(1), den(wav, strength=strength), lens)
    # audio that is not a whole number of hops: the output has (n // 256) * 256 samples, lengths up to n // 256
    cut = wav[:, : T * HOP - 100]
    lens2 = [199, 5, 100, 198, 1, 2]
    _check(den(cut, strength=0.00025, lengths=lens2).unsqueeze(1), den(cut, strength=0.00025), lens2)
    with pytest.raises(ValueError):
        den(cut, strength=0.00025, lengths=[200] * 6)
    with pytest.raises(ValueError):
        den(wav, strength=0.00025, lengths=[0] * 6)


@pytest.mark.gpu
def test_work_skipped(gen_den):
    """The ragged denoiser computes sum_b (floor((len_b + 1) / 2) + 1) frame pairs (the launch report's algorithmic FLOPs count
    the device-built list), and the vocoder inside the call does exactly the work of ev_vocode_ragged on min(len_b + 4, T)."""
    gen, den = gen_den
    T = 300
    lens = [137, 138, 299, 296, 1, 2, 300, 40]
    mel = _mel(len(lens), T, seed=95)
    ctx = gen._ctx
    gen.cuda_graphs = False
    try:
        ctx.profile_begin()
        gen.vocode_denoised(mel, lens, 0.00025)
        fused = {r["name"]: r for r in ctx.profile_end()}
        ctx.profile_begin()
        gen(mel, lengths=[min(n + 4, T) for n in lens])
        voc = {r["name"]: r for r in ctx.profile_end()}
    finally:
        gen.cuda_graphs = True
    pairs = fused["denoise_fft_ragged"]["flops"] / (2.0 * 5.0 * 1024 * 10.0)
    want = sum(min((n + 1) // 2 + 1, (T + 2) // 2) for n in lens)
    assert pairs == want and want < len(lens) * ((T + 2) // 2)
    assert "denoise_fft" not in fused
    for name, r in voc.items():
        assert fused[name]["launches"] == r["launches"], name
        assert fused[name]["flops"] == pytest.approx(r["flops"], rel=1e-12), name


@pytest.mark.gpu
def test_corpus_with_denoiser_ragged_equals_dense(matcha_sd, gen_den):
    """synthesise_corpus(denoiser=...) returns the same cropped waveforms with ragged=True (one ragged vocoder + denoiser call)
    and ragged=False (dense vocoder, dense denoiser), one and three micro-batches in flight."""
    import emojivoice_b200 as ev
    from emojivoice_b200 import synthetic
    from emojivoice_b200.config import VCTK

    gen, den = gen_den
    matcha = ev.MatchaTTS(**VCTK.constructor_kwargs())
    matcha.load_state_dict(matcha_sd)
    x, xl, spks = synthetic.phoneme_batch(10, 5, 40, seed=23)
    utts = [(x[i, : int(xl[i])].tolist(), int(spks[i])) for i in range(10)]
    zs = {}

    def z_fn(mb, model, x_, xl_, spks_):
        probe = model.synthesise(x_, xl_, 1, 0.667, spks_, 1.0)
        return zs.setdefault(tuple(mb.items), synthetic.prior_noise(len(mb.items), 80, probe["t_pad"], seed=6))

    ref, _ = ev.synthesise_corpus(matcha, gen, utts, batch_size=4, n_timesteps=2, z_fn=z_fn, denoiser=den, ragged=False)
    ctx = gen._ctx
    ctx.profile_begin()
    r1, _ = ev.synthesise_corpus(matcha, gen, utts, batch_size=4, n_timesteps=2, z_fn=z_fn, denoiser=den, ragged=True)
    names = {r["name"] for r in ctx.profile_end()}
    assert "denoise_fft_ragged" in names and "denoise_fft" not in names
    r3, _ = ev.synthesise_corpus(matcha, gen, utts, batch_size=4, n_timesteps=2, z_fn=z_fn, denoiser=den, ragged=True, in_flight=3)
    r3d, _ = ev.synthesise_corpus(matcha, gen, utts, batch_size=4, n_timesteps=2, z_fn=z_fn, denoiser=den, ragged=False, in_flight=3)
    assert sorted(ref) == sorted(r1) == sorted(r3) == sorted(r3d) == list(range(10))
    for i in ref:
        for r in (r1, r3, r3d):
            assert r[i]["mel_length"] == ref[i]["mel_length"]
            assert torch.equal(r[i]["waveform"], ref[i]["waveform"]), i


@pytest.mark.gpu
def test_refusals(gen_den):
    """Before ev_denoiser_init: EV_ERR_STATE; null lengths, T < 3, unknown precision: EV_ERR_INVALID; a short workspace:
    EV_ERR_STATE; host lengths outside [1, T]: ValueError.  ev_last_error says why."""
    import emojivoice_b200 as ev
    from emojivoice_b200 import _lib, synthetic
    from emojivoice_b200.config import HIFIGAN_V1

    L = _lib.lib()
    fresh = ev.Generator(HIFIGAN_V1)
    fresh.load_state_dict(synthetic.hifigan_state_dict(HIFIGAN_V1, seed=4321, gain=1.0))
    fresh.remove_weight_norm()
    mel = _mel(2, 20, seed=96).cuda()
    lens = torch.tensor([20, 7]).cuda()
    wav = torch.empty(2, 1, 20 * HOP, device="cuda")

    def call(g, mel_, lens_, T, prec=1, ws_bytes=None):
        ctx = g._ctx
        nb = L.ev_to_waveform_ragged_workspace_bytes(ctx.handle, 2, T)
        ws = ctx.workspace(nb)
        rc = L.ev_to_waveform_ragged(ctx.handle, _lib.ptr(mel_), _lib.ptr(lens_), 2, T, prec, C.c_float(0.00025), _lib.ptr(wav),
                                     _lib.ptr(ws), ws.numel() if ws_bytes is None else ws_bytes, _lib.stream_ptr())
        return rc, L.ev_last_error(ctx.handle).decode()

    rc, msg = call(fresh, mel, lens, 20)
    assert rc == -4 and "ev_denoiser_init" in msg
    with pytest.raises(RuntimeError, match="ev_denoiser_init"):
        fresh.vocode_denoised(mel, [20, 7])
    gen, _ = gen_den
    rc, msg = call(gen, mel, None, 20)
    assert rc == -1 and "null" in msg
    rc, msg = call(gen, mel[:, :, :2].contiguous(), lens, 2)
    assert rc == -1 and "reflect padding" in msg
    rc, msg = call(gen, mel, lens, 20, prec=7)
    assert rc == -1 and "precision" in msg
    rc, msg = call(gen, mel, lens, 20, ws_bytes=1024)
    assert rc == -4 and "workspace" in msg
    for bad in ([21, 7], [0, 7]):
        with pytest.raises(ValueError, match=r"\[1, 20\]"):
            gen.vocode_denoised(mel, bad)
