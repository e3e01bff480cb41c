"""CPU-side checks: the C ABI exports what the header declares, host-only helpers, emoji front-end, synthetic data."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

import emojivoice_b200 as ev
from emojivoice_b200 import _lib, synthetic
from emojivoice_b200.config import VCTK

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "emojivoice_b200.h")).read()
    declared = set(re.findall(r"EV_API\s+[\w\s\*]+?\b(ev_\w+)\s*\(", header))
    assert declared, "no declarations parsed"
    lib = _lib.lib()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert lib.ev_version() >= 100


def test_no_gpu_means_loud_failure(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)      # what a machine without a GPU reports
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.Context()
    m = ev.MatchaTTS(**VCTK.constructor_kwargs())
    with pytest.raises(RuntimeError):
        m.load_state_dict({})


@pytest.mark.parametrize("n", [1, 2, 4, 10, 50])
def test_euler_schedule_matches_torch_float32(n):
    t = (C.c_float * n)()
    d = (C.c_float * n)()
    assert _lib.lib().ev_test_euler_schedule(n, t, d) == 0
    # flow_matching.py:52,68-83
    span = torch.linspace(0, 1, n + 1)
    tt, dt = span[0], span[1] - span[0]
    for step in range(1, n + 1):
        assert float(tt) == t[step - 1] and float(dt) == d[step - 1], (step, float(tt), t[step - 1], float(dt), d[step - 1])
        tt = tt + dt
        if step < n:
            dt = span[step + 1] - tt


def test_emoji_front_end():
    # feel_me.py:298-312: first emoji of the text that is in the map wins; emoji and brackets are stripped
    assert ev.emoji_to_spk("wow \U0001F62E (so cool) \U0001F60D") == ("wow  so cool ", 54)
    assert ev.emoji_to_spk("no emoji here") == ("no emoji here", 0)
    assert ev.emoji_to_spk("unknown \U0001F984 then \U0001F923", default=0) == ("unknown  then ", 15)
    # demo_story_script.py:177-182: mapping order, default 12
    txt = "\U0001F923 first in text, \U0001F60D first in map"
    assert ev.emoji_to_spk(txt, order="mapping", default=12)[1] == 107
    assert ev.emoji_to_spk("plain", order="mapping", default=12)[1] == 12
    assert ev.emoji_to_spk("x \U0001F60E", mapping=ev.EMOJI_MAPPING_MALE)[1] == 6


def test_emoji_recognition_follows_the_unicode_emoji_property():
    """`emoji.is_emoji` / `emoji.replace_emoji` semantics (feel_me.py:298-312): plain arrows, maths and technical symbols, digits
    and stand-alone joiners are NOT emoji and stay in the text; whole sequences (ZWJ families, flags, keycaps, skin tones,
    text-presentation emoji with VS16) are removed as one unit."""
    from emojivoice_b200.emoji_frontend import is_emoji, replace_emoji

    for ch in "\u2192\u2191\u2193\u2200\u2211\u2318\u23000123456789#*\u200d\ufe0f\u20e3\U0001F1E8a ":
        assert not is_emoji(ch), hex(ord(ch))
    for ch in "\u2194\u21a9\u00a9\u00ae\u2122\u231a\u2600\u2764\u2b50\u3030\U0001F600\U0001F984\U0001F3FD\U0001FAE0":
        assert is_emoji(ch), hex(ord(ch))
    assert all(is_emoji(k) for k in list(ev.EMOJI_MAPPING_FEMALE) + list(ev.EMOJI_MAPPING_MALE))
    assert not is_emoji("\U0001F600\U0001F600")                      # the apps pass single characters
    txt = "a \u2192 b \U0001F468\u200d\U0001F469\u200d\U0001F467 c 5\ufe0f\u20e3 d \u20e3 e \U0001F1E8\U0001F1E6 f \U0001F44D\U0001F3FD g\ufe0f \u2639\ufe0f 7"
    assert replace_emoji(txt) == "a \u2192 b  c  d \u20e3 e  f  g\ufe0f  7"
    assert replace_emoji("x\U0001F600y", "_") == "x_y"
    assert ev.emoji_to_spk("go \u2192 there \U0001F60D")[0] == "go \u2192 there "
    assert ev.intersperse([5, 6, 7]) == [0, 5, 0, 6, 0, 7, 0]


def test_synthetic_inputs_are_blank_interspersed_and_in_range():
    x, xl, spk = synthetic.phoneme_batch(6, 3, 20, seed=3)
    assert x.shape[1] == int(xl.max()) and (xl % 2 == 1).all()
    for b in range(6):
        row = x[b, : xl[b]]
        assert (row[0::2] == 0).all() and (row[1::2] > 0).all() and (row < 178).all()
        assert (x[b, xl[b]:] == 0).all()
    assert set(spk.tolist()) <= set(ev.EMOJI_MAPPING_FEMALE.values())
    a = synthetic.matcha_state_dict(VCTK, seed=5)
    b = synthetic.matcha_state_dict(VCTK, seed=5)
    assert synthetic.checksum(a) == synthetic.checksum(b)
    assert sum(v.numel() for k, v in a.items() if k not in ("mel_mean", "mel_std")) == 20_857_569


def test_aten_sum_order_restatement_matches_torch():
    """numpy restatement of SURVEY.md Appendix B (the order the CUDA length stage reproduces) vs torch.sum on CPU."""
    from tests.aten_sum_ref import sum_f32

    rng = np.random.default_rng(0)
    for n in (1, 3, 7, 8, 9, 15, 16, 17, 33, 64, 151, 333, 511, 512, 513, 1100, 2100):
        for ls in (0.8, 0.9, 1.1, 1.2):
            w = (np.ceil(np.exp(rng.normal(0.9, 0.6, size=n))).astype(np.float32) * np.float32(ls)).astype(np.float32)
            w[rng.integers(0, n + 1):] = 0.0
            want = float(torch.sum(torch.from_numpy(w).view(1, 1, n), [1, 2])[0])
            assert sum_f32(w) == want, (n, ls)


def test_ragged_vocoder_margins_cover_the_generators_look_ahead():
    """ev_vocode_ragged computes item b only up to (len_b + margin) frames per layer.  The margins come from the configuration
    (hifigan.cu: vocoder_margins); here they are pinned against the ORACLE generator's real receptive field: perturbing the
    mel from frame f on must not change any sample before (f - look_ahead) * 256, and the look-ahead measured that way must
    not exceed what the first layers keep (margin - 1 spare frame)."""
    from emojivoice_b200.config import HIFIGAN_V1
    from oracle import hifigan_oracle as ho

    h = HIFIGAN_V1
    cfg = _lib.EvHifiganCfg()
    cfg.num_mels, cfg.upsample_initial_channel = 80, int(h["upsample_initial_channel"])
    cfg.n_ups, cfg.n_kernels = len(h["upsample_rates"]), len(h["resblock_kernel_sizes"])
    for i, (u, k) in enumerate(zip(h["upsample_rates"], h["upsample_kernel_sizes"])):
        cfg.upsample_rates[i], cfg.upsample_kernel_sizes[i] = int(u), int(k)
    for j, (k, dil) in enumerate(zip(h["resblock_kernel_sizes"], h["resblock_dilation_sizes"])):
        cfg.resblock_kernel_sizes[j] = int(k)
        for l in range(3):
            cfg.resblock_dilation_sizes[j][l] = int(dil[l])
    stage, up, pre = (C.c_int32 * 8)(), (C.c_int32 * 8)(), C.c_int32(0)
    assert _lib.lib().ev_test_vocoder_margins(C.byref(cfg), stage, up, C.byref(pre)) == 0
    n = cfg.n_ups
    assert list(stage)[:n] == [11, 3, 2, 2] and list(up)[:n] == [13, 3, 2, 2] and pre.value == 13      # HiFi-GAN v1
    # measured look-ahead of the oracle: first output sample that reacts to a change of the frames >= f
    sd = synthetic.hifigan_state_dict(h, seed=4321, gain=1.0)
    T, f = 48, 32
    mel = synthetic.synthetic_mel(1, T, seed=3)
    mel2 = mel.clone()
    mel2[:, :, f:] += torch.randn(1, 80, T - f, generator=torch.Generator().manual_seed(1))
    a, b = ho.generator(sd, h, mel)[0, 0], ho.generator(sd, h, mel2)[0, 0]
    first = int((a != b).nonzero()[0])
    look_ahead_frames = (f * 256 - first + 255) // 256        # measured on the mel INPUT: 13 frames for v1
    # conv_pre (k = 7) itself reaches 3 frames ahead and reads the dense mel, so its OUTPUT rows must be right up to
    # look_ahead - 3 frames past the end; the margin keeps one spare frame on top of its own (conservative) bound
    assert 5 < look_ahead_frames - 3 <= pre.value - 1, look_ahead_frames
    # stage by stage the margins shrink with the remaining depth of the generator and never drop below one spare frame
    assert all(stage[i] >= stage[i + 1] >= 2 for i in range(n - 1)) and all(up[i] >= stage[i] for i in range(n))


def test_lanes_host_logic():
    """ev.Lanes / lanes_for without a GPU: argument check, lane 0 is the caller's own pair, the cache is keyed by the vocoder OBJECT."""
    import emojivoice_b200 as ev

    class Fake:
        pass

    m, v1, v2 = Fake(), Fake(), Fake()
    with pytest.raises(ValueError):
        ev.Lanes(m, v1, 0)
    one = ev.lanes_for(m, v1, 1)
    assert len(one) == 1 and one.models[0] is m and one.vocoders[0] is v1 and one.streams == [None]
    assert ev.lanes_for(m, v1, 1) is one
    assert ev.lanes_for(m, v2, 1) is not one and ev.lanes_for(m, v2, 1).vocoders[0] is v2
    d = object()
    assert one.denoiser(0, d) is d and one.denoiser(0, None) is None
