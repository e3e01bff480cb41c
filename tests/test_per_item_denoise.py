"""A denoiser strength per utterance, or none (ev_to_waveform_items, ev_denoise_items, Generator.vocode_denoised and Denoiser with
per-item strengths, synthesise_corpus's "denoiser_strength" key): in one padded batch, each utterance gets bit for bit what the
scalar call with its own strength gives it, or the vocoder's (Denoiser: its input's) samples when it is not denoised.

CPU: argument parsing, the corpus settings and their refusals, the micro-batch plan.
GPU: per-item calls against scalar calls and the oracle, launch counts, graph replay, device lengths, the work skipped, the
corpus driver, the C ABI's refusals."""
import pytest
import torch

from tests.conftest import rel_l2
from emojivoice_b200 import batch, sharding
from emojivoice_b200.hifigan import per_item_strength
from oracle import hifigan_oracle as ho

HOP = 256


# ------------------------------------------------------------------------------------------------ CPU
def test_per_item_strength_arguments():
    assert per_item_strength(0.00025, 3) == 0.00025
    assert per_item_strength(torch.tensor(0.5), 3) == 0.5
    assert per_item_strength(None, 3) is None
    assert per_item_strength([None, None], 2) is None                                   # nothing denoised
    assert per_item_strength([0.1, 0.1, 0.1], 3) == 0.1                                 # equal values are the scalar call
    assert per_item_strength(torch.tensor([0.0005, 0.0005]), 2) == pytest.approx(0.0005)
    assert per_item_strength([0.1, None, 0], 3) == (0.1, None, 0.0)
    assert per_item_strength([0.1, 0.1, None], 3) == (0.1, 0.1, None)                  # equal strengths with an "off" stay per item
    assert per_item_strength(torch.tensor([0.5, 0.25]), 2) == (0.5, 0.25)
    assert per_item_strength((0, 1), 2) == (0.0, 1.0)
    for bad in ([0.1, 0.2], [0.1] * 4, [float("nan"), 0.1, 0.1], [0.1, float("inf"), None], torch.tensor([0.1, float("-inf"), 0.0]),
                ["0.1", 0.1, 0.1]):
        with pytest.raises(ValueError):
            per_item_strength(bad, 3)


def test_corpus_denoiser_strength_settings():
    d = dict(length_scale=1.0, temperature=0.667, n_timesteps=10, denoiser_strength=0.0005)
    utts = [([1, 2], 3), ([4], 5, {"denoiser_strength": None}), ([4], 5, {"denoiser_strength": 0.1, "temperature": 0.5}),
            ([6], 7, {"denoiser_strength": 0.0})]
    s, own = batch.utterance_settings(utts[:2] + utts[3:], d)
    assert not own                                                # a strength alone is not a synthesis setting
    assert [x["denoiser_strength"] for x in s] == [0.0005, None, 0.0]
    s, own = batch.utterance_settings(utts, d)
    assert own and s[2] == dict(d, denoiser_strength=0.1, temperature=0.5)
    assert batch.denoiser_strengths(s, denoiser=object()) == [0.0005, None, 0.1, 0.0]
    with pytest.raises(ValueError, match="unknown"):
        batch.utterance_settings([([1], 3, {"strength": 0.1})], d)
    with pytest.raises(ValueError):
        batch.denoiser_strengths([dict(d, denoiser_strength=float("nan"))], denoiser=object())
    # without a denoiser the default is "off", and a strength asked for is refused before any work
    for u in ([([1], 3, {"denoiser_strength": 0.1})], [([1], 3), ([2], 4, {"denoiser_strength": 0.0})]):
        with pytest.raises(ValueError, match="needs a denoiser"):
            batch.synthesise_corpus(None, None, u, denoiser=None)
    no_den = dict(d, denoiser_strength=None)
    s, _ = batch.utterance_settings([([1], 3), ([2], 4, {"denoiser_strength": None})], no_den)
    assert batch.denoiser_strengths(s, denoiser=None) == [None, None]


class _PlanSeen(Exception):
    pass


def test_plan_does_not_depend_on_per_utterance_strengths(monkeypatch):
    """synthesise_corpus hands sharding.shard the same arguments with and without per-utterance strengths (stopped there)."""
    seen, real = [], sharding.shard

    def shard(*a, **kw):
        seen.append((a, kw, real(*a, **kw)))
        raise _PlanSeen

    monkeypatch.setattr(sharding, "shard", shard)
    g = torch.Generator().manual_seed(3)
    lens = torch.randint(5, 80, (70,), generator=g).tolist()
    plain = [(list(range(n)), 1) for n in lens]
    strengths = [None, 0.0, 0.00025, 0.1]
    mixed = [(ids, spk, {"denoiser_strength": strengths[i % 4]}) if i % 5 else (ids, spk) for i, (ids, spk) in enumerate(plain)]
    for utts in (plain, mixed):
        with pytest.raises(_PlanSeen):
            batch.synthesise_corpus(None, None, utts, batch_size=16, denoiser=object(), world_size=2, rank=1)
    (a0, kw0, p0), (a1, kw1, p1) = seen
    assert a0 == a1 and kw0 == kw1
    assert [(m.items, m.cost) for m in p0] == [(m.items, m.cost) for m in p1]


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def gen_den():
    import emojivoice_b200 as ev
    from emojivoice_b200 import synthetic
    from emojivoice_b200.config import HIFIGAN_V1

    sd = synthetic.hifigan_state_dict(HIFIGAN_V1, seed=4321, gain=1.0)
    g = ev.Generator(HIFIGAN_V1)
    g.load_state_dict(sd)
    g.remove_weight_norm()
    return g, ev.Denoiser(g), sd


def _mel(B, T, seed):
    from emojivoice_b200 import synthetic

    return synthetic.synthetic_mel(B, T, seed=seed)


def _scalar_refs(gen, mel, lens, strengths, prec=None):
    """Each distinct setting's scalar call on the whole batch: vocode_denoised(strength), or the ragged vocoder for None."""
    refs = {}
    for s in set(strengths):
        refs[s] = gen(mel, lengths=lens, dtype=prec) if s is None else gen.vocode_denoised(mel, lens, s, dtype=prec)
    return refs


def _check_items(got, refs, strengths, lens, T):
    assert got.shape == (len(strengths), 1, T * HOP)
    for b, (s, n) in enumerate(zip(strengths, lens)):
        n = max(0, min(int(n), T)) * HOP
        assert torch.equal(got[b], refs[s][b]), (b, s)
        assert float(got[b, 0, n:].abs().sum()) == 0.0, (b, s)


RAGGED_LENS = [300, 300, 300, 300, 300, 300, 137, 138, 1, 2, 299, 296]      # six full items, short ones, lengths near T
MIXED = (None, 0.0, 0.00025, 0.0005, 0.1)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_mixed_strengths_equal_scalar_calls(gen_den, prec):
    gen, _, _ = gen_den
    T = 300
    strengths = [MIXED[(b * 3) % 5] for b in range(len(RAGGED_LENS))]
    mel = _mel(len(RAGGED_LENS), T, seed=70)
    refs = _scalar_refs(gen, mel, RAGGED_LENS, strengths, prec)
    for _ in range(3):                                       # eager, capture, replay
        _check_items(gen.vocode_denoised(mel, RAGGED_LENS, strengths, dtype=prec), refs, strengths, RAGGED_LENS, T)
    # strength 0 is not "off": the STFT / ISTFT round trip changes low bits
    b = strengths.index(0.0)
    n = RAGGED_LENS[b] * HOP
    assert not torch.equal(refs[0.0][b, 0, :n], refs[None][b, 0, :n])
    assert rel_l2(refs[0.0][b, 0, :n], refs[None][b, 0, :n]) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_all_off_and_all_equal_are_the_scalar_calls(gen_den, prec):
    gen, _, _ = gen_den
    T, lens = 120, [120, 7, 64, 119]
    mel = _mel(4, T, seed=71)
    gen.cuda_graphs = False
    try:
        for strengths, scalar in (([None] * 4, lambda: gen(mel, lengths=lens, dtype=prec)),
                                  ([0.0005] * 4, lambda: gen.vocode_denoised(mel, lens, 0.0005, dtype=prec)),
                                  (torch.full((4,), 0.1), lambda: gen.vocode_denoised(mel, lens, 0.1, dtype=prec))):
            gen.launch_count(reset=True)
            want = scalar()
            n_scalar = gen.launch_count(reset=True)
            got = gen.vocode_denoised(mel, lens, strengths, dtype=prec)
            assert gen.launch_count(reset=True) == n_scalar
            assert torch.equal(got, want)
    finally:
        gen.cuda_graphs = True


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_config2_shape(gen_den, prec):
    """32 utterances of 368-548 frames padded to 668 (BASELINE config 2), strengths {off, 0.00025, 0.0005, 0.001} dealt in turn."""
    gen, _, _ = gen_den
    g = torch.Generator().manual_seed(5)
    lens = torch.randint(368, 549, (32,), generator=g).tolist()
    lens[0], lens[1] = 548, 369
    strengths = [(None, 0.00025, 0.0005, 0.001)[b % 4] for b in range(32)]
    mel = _mel(32, 668, seed=72)
    refs = _scalar_refs(gen, mel, lens, strengths, prec)
    _check_items(gen.vocode_denoised(mel, torch.tensor(lens), strengths, dtype=prec), refs, strengths, lens, 668)


@pytest.mark.gpu
def test_graph_replay_reads_new_strengths(gen_den):
    """One graph for every mixed call of a shape; replays follow new strengths, items flipping between on and off, and new lengths."""
    gen, _, _ = gen_den
    T = 120
    mel = _mel(4, T, seed=73)
    items_keys = lambda: [k for k in gen._graphs.entries if k[-1] == "items"]
    before = len(items_keys())
    cases = [([120, 3, 61, 118], [None, 0.00025, 0.1, 0.0005])] * 3 + [
        ([120, 3, 61, 118], [0.1, None, 0.00025, None]),
        ([120, 3, 61, 118], [0.0005, 0.0005, None, 0.0]),
        ([1, 2, 119, 60], [None, 0.1, 0.1, 0.00025]),
    ]
    for lens, strengths in cases:
        dev_lens = torch.tensor(lens).cuda()
        refs = _scalar_refs(gen, mel, dev_lens, strengths)
        _check_items(gen.vocode_denoised(mel, dev_lens, strengths), refs, strengths, lens, T)
    assert len(items_keys()) == before + 1


@pytest.mark.gpu
def test_device_lengths_are_clamped_to_zero_and_T(gen_den):
    gen, _, _ = gen_den
    T = 40
    mel = _mel(5, T, seed=74)
    strengths = [0.0005, None, 0.1, None, None]
    got = gen.vocode_denoised(mel, torch.tensor([T + 9, 0, -3, T + 1, 17]).cuda(), strengths)
    clamped = torch.tensor([T, 0, 0, T, 17]).cuda()
    _check_items(got, _scalar_refs(gen, mel, clamped, strengths), strengths, [T, 0, 0, T, 17], T)


@pytest.mark.gpu
def test_denoiser_per_item_strengths(gen_den):
    gen, den, _ = gen_den
    T = 200
    lens = [200, 1, 2, 77, 198, 150]
    strengths = [None, 0.0, 0.00025, 0.1, None, 0.0005]
    wav = gen(_mel(6, T, seed=75)).clamp(-1, 1).squeeze(1)
    for audio, lens_ in ((wav, lens), (wav[:, : T * HOP - 100], [199, 5, 100, 198, 1, 2])):   # and a length not a multiple of 256
        n_out = (audio.shape[1] // HOP) * HOP
        for lengths in (None, lens_, torch.tensor(lens_).cuda()):
            got = den(audio, strengths, lengths=lengths)
            assert got.shape == (6, n_out)
            for b, s in enumerate(strengths):
                if s is not None:
                    assert torch.equal(got[b], den(audio, strength=s, lengths=lengths)[b]), (b, s)
                    continue
                want = audio[b, :n_out].clone()
                if lengths is not None:
                    want[lens_[b] * HOP:] = 0.0
                assert torch.equal(got[b], want), b
    assert torch.equal(den(wav, [None] * 6), wav)                       # nothing denoised: the input
    assert torch.equal(den(wav, [0.1] * 6), den(wav, 0.1))
    with pytest.raises(ValueError):
        den(wav, [0.1, None])


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_items_match_oracle(gen_den, prec):
    """Each item against oracle.hifigan_oracle.to_waveform with its own strength (or no denoiser), on the padded mel and cropped
    to its length, at the vocoder's parity tolerances; the bias spectrum is the one the GPU computed (tested on its own elsewhere)."""
    from emojivoice_b200.config import HIFIGAN_V1

    gen, den, sd = gen_den
    T = 48
    lens = [48, 30, 47, 12, 40]
    strengths = [None, 0.00025, 0.1, 0.0, 0.0005]
    mel = _mel(5, T, seed=76)
    got = gen.vocode_denoised(mel, lens, strengths, dtype=prec).cpu()
    bias = den.bias_spec.cpu()
    for b, (n, s) in enumerate(zip(lens, strengths)):
        ref = ho.to_waveform(sd, HIFIGAN_V1, mel[b: b + 1], None if s is None else bias, 0.0 if s is None else s)
        assert rel_l2(got[b, 0, : n * HOP], ref[: n * HOP]) < {"fp32": 1e-4, "bf16": 1e-2}[prec], (b, s)


@pytest.mark.gpu
def test_work_skipped(gen_den):
    """Items not denoised add no STFT pairs, and the vocoder runs them on their own length instead of length + 4."""
    gen, _, _ = gen_den
    T = 300
    lens = [137, 138, 299, 296, 1, 2, 300, 40]
    strengths = [None, 0.00025, None, 0.1, 0.0005, None, 0.0, None]
    mel = _mel(len(lens), T, seed=77)
    ctx = gen._ctx
    gen.cuda_graphs = False
    try:
        ctx.profile_begin()
        gen.vocode_denoised(mel, lens, strengths)
        fused = {r["name"]: r for r in ctx.profile_end()}
        ctx.profile_begin()
        gen(mel, lengths=[n if s is None else min(n + 4, T) for n, s in zip(lens, strengths)])
        voc = {r["name"]: r for r in ctx.profile_end()}
    finally:
        gen.cuda_graphs = True
    pairs = fused["denoise_fft_ragged"]["flops"] / (2.0 * 5.0 * 1024 * 10.0)
    assert pairs == sum(min((n + 1) // 2 + 1, (T + 2) // 2) for n, s in zip(lens, strengths) if s is not None)
    for name, r in voc.items():
        assert fused[name]["launches"] == r["launches"], name
        assert fused[name]["flops"] == pytest.approx(r["flops"], rel=1e-12), name


@pytest.mark.gpu
@pytest.mark.parametrize("in_flight", [1, 2])
def test_corpus_per_utterance_strengths(matcha_sd, gen_den, in_flight):
    """Each waveform equals the corpus run with its utterance's setting applied to all (no denoiser for "off"), ragged or not,
    and every mel equals the run without a denoiser."""
    import emojivoice_b200 as ev
    from emojivoice_b200 import synthetic
    from emojivoice_b200.config import VCTK

    gen, den, _ = gen_den
    matcha = ev.MatchaTTS(**VCTK.constructor_kwargs())
    matcha.load_state_dict(matcha_sd)
    x, xl, spks = synthetic.phoneme_batch(11, 5, 40, seed=24)
    own = [None, 0.00025, "default", 0.1, None, 0.0, "default", 0.00025, 0.1, None, 0.0]
    utts = [(x[i, : int(xl[i])].tolist(), int(spks[i])) + (() if own[i] == "default" else ({"denoiser_strength": own[i]},))
            for i in range(11)]
    plain = [u[:2] for u in utts]
    setting = [0.0005 if s == "default" else s for s in own]
    zs = {}

    def z_fn(mb, model, x_, xl_, spks_):
        probe = model.synthesise(x_, xl_, 1, 0.667, spks_, 1.0)
        return zs.setdefault(tuple(mb.items), synthetic.prior_noise(len(mb.items), 80, probe["t_pad"], seed=7))

    kw = dict(batch_size=4, n_timesteps=2, z_fn=z_fn, keep_mel=True, in_flight=in_flight)
    refs = {None: ev.synthesise_corpus(matcha, gen, plain, **kw)[0]}
    for s in set(setting) - {None}:
        refs[s] = ev.synthesise_corpus(matcha, gen, plain, denoiser=den, denoiser_strength=s, **kw)[0]
    for ragged in (True, False):
        got, _ = ev.synthesise_corpus(matcha, gen, utts, denoiser=den, denoiser_strength=0.0005, ragged=ragged, **kw)
        assert sorted(got) == list(range(11))
        for i, s in enumerate(setting):
            assert got[i]["mel_length"] == refs[None][i]["mel_length"]
            assert torch.equal(got[i]["mel"], refs[None][i]["mel"]), i
            assert torch.equal(got[i]["waveform"], refs[s][i]["waveform"]), (i, s, ragged)


@pytest.mark.gpu
def test_refusals(gen_den):
    """Before ev_denoiser_init: EV_ERR_STATE; null strengths or lengths: EV_ERR_INVALID; a short workspace: EV_ERR_STATE."""
    import emojivoice_b200 as ev
    from emojivoice_b200 import _lib, synthetic
    from emojivoice_b200.config import HIFIGAN_V1

    L = _lib.lib()
    fresh = ev.Generator(HIFIGAN_V1)
    fresh.load_state_dict(synthetic.hifigan_state_dict(HIFIGAN_V1, seed=4321, gain=1.0))
    fresh.remove_weight_norm()
    mel = _mel(2, 20, seed=78).cuda()
    lens = torch.tensor([20, 7]).cuda()
    st = torch.tensor([0.1, 0.0]).cuda()
    on = torch.tensor([1, 0], dtype=torch.uint8).cuda()
    wav = torch.empty(2, 1, 20 * HOP, device="cuda")

    def call(g, lens_, st_, ws_bytes=None):
        ctx = g._ctx
        ws = ctx.workspace(L.ev_to_waveform_items_workspace_bytes(ctx.handle, 2, 20))
        rc = L.ev_to_waveform_items(ctx.handle, _lib.ptr(mel), _lib.ptr(lens_), 2, 20, 1, _lib.ptr(st_), _lib.ptr(on), _lib.ptr(wav),
                                    _lib.ptr(ws), ws.numel() if ws_bytes is None else ws_bytes, _lib.stream_ptr())
        return rc, L.ev_last_error(ctx.handle).decode()

    def call_dn(g, st_):
        ctx = g._ctx
        ws = ctx.workspace(L.ev_denoise_items_workspace_bytes(ctx.handle, 2, 20 * HOP))
        rc = L.ev_denoise_items(ctx.handle, _lib.ptr(wav), None, 2, 20 * HOP, _lib.ptr(st_), None, _lib.ptr(wav), _lib.ptr(ws), ws.numel(),
                                _lib.stream_ptr())
        return rc, L.ev_last_error(ctx.handle).decode()

    assert call(fresh, lens, st)[0] == -4 and "ev_denoiser_init" in call(fresh, lens, st)[1]
    assert call_dn(fresh, st)[0] == -4
    gen, _, _ = gen_den
    rc, msg = call(gen, None, st)
    assert rc == -1 and "null" in msg
    rc, msg = call(gen, lens, None)
    assert rc == -1 and "strengths" in msg
    rc, msg = call_dn(gen, None)
    assert rc == -1 and "strengths" in msg
    rc, msg = call(gen, lens, st, ws_bytes=1024)
    assert rc == -4 and "workspace" in msg
    torch.cuda.synchronize()
