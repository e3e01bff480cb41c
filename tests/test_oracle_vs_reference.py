"""Build-container-only: re-derive the pins through the stub-imported reference (skipped on the GPU box)."""
import dataclasses

import pytest
import torch

from emojivoice_b200 import synthetic
from emojivoice_b200.config import HIFIGAN_V1, VCTK
from oracle import hifigan_oracle as ho
from oracle import matcha_oracle as mo
from oracle import reference_shim as shim

pytestmark = pytest.mark.skipif(not shim.available(), reason="/root/reference not present")


def test_parameter_counts_pin_the_restated_diffusers_attention():
    lj = dataclasses.replace(VCTK, n_spks=1)
    ref = shim.build_matcha(lj, synthetic.matcha_state_dict(lj, seed=1))
    assert sum(p.numel() for p in ref.parameters()) == 18_204_193      # synthesis.ipynb:127


def test_oracle_bit_equal_to_reference_synthesise(matcha_sd):
    ref = shim.build_matcha(VCTK, matcha_sd)
    x, xl, spk = synthetic.phoneme_batch(3, 4, 14, seed=11)
    for ls in (0.8, 1.0, 1.2):
        probe = mo.synthesise(matcha_sd, VCTK, x, xl, 1, 0.667, spk, ls)
        z = synthetic.prior_noise(3, 80, probe["t_pad"], seed=12)
        out = mo.synthesise(matcha_sd, VCTK, x, xl, 3, 0.667, spk, ls, z=z)
        with shim.injected_noise(z):
            r = ref.synthesise(x, xl, n_timesteps=3, temperature=0.667, spks=spk, length_scale=ls)
        assert torch.equal(out["mel_lengths"], r["mel_lengths"])
        for k in ("encoder_outputs", "decoder_outputs", "attn", "mel"):
            assert torch.equal(out[k], r[k]), k


def test_oracle_bit_equal_to_reference_vocoder_and_denoiser():
    hs = synthetic.hifigan_state_dict(HIFIGAN_V1, seed=9, gain=0.7)
    gen = shim.build_hifigan(HIFIGAN_V1, hs)
    mel = synthetic.synthetic_mel(2, 21, seed=10)
    with torch.inference_mode():
        w_ref = gen(mel)
    w = ho.generator(hs, HIFIGAN_V1, mel)
    assert torch.equal(w, w_ref)
    den = shim.build_denoiser(gen)
    bias = ho.denoiser_bias(hs, HIFIGAN_V1)
    assert torch.equal(bias, den.bias_spec)
    assert torch.equal(ho.denoise(w.clamp(-1, 1).squeeze(1), bias, 0.00025), den(w_ref.clamp(-1, 1).squeeze(), strength=0.00025))


def _training_batch(seed, b=3):
    return synthetic.training_batch(b, 4, 14, seed, VCTK.n_feats)


def test_oracle_bit_equal_to_reference_training_forward(matcha_sd):
    """MatchaTTS.forward (matcha_tts.py:154-245) of the unmodified reference -- its own monotonic_align wrapper on its own Cython
    kernel when oracle/_ref holds the build -- against the restatement, under the same random draws."""
    import random

    ref = shim.build_matcha(VCTK, matcha_sd).eval()
    for seed, out_size in ((31, None), (32, None), (33, 16)):
        x, xl, spk, y, yl = _training_batch(seed)
        torch.manual_seed(seed)
        random.seed(seed)
        with torch.no_grad():
            dur, prior, diff, attn = ref(x, xl, y, yl, spks=spk, out_size=out_size)
        torch.manual_seed(seed)
        random.seed(seed)
        off = None
        if out_size is not None:           # the reference's draw, matcha_tts.py:213-216
            mx = (yl - out_size).clamp(0).tolist()
            off = torch.tensor([random.choice(range(0, e)) if e > 0 else 0 for e in mx])
        t = torch.rand([x.shape[0], 1, 1])
        z = torch.randn(x.shape[0], VCTK.n_feats, out_size or y.shape[-1])
        o = mo.forward_losses(matcha_sd, VCTK, x, xl, y, yl, spk, out_size=out_size, t=t, z=z, out_offset=off)
        assert torch.equal(o["attn"], attn)
        assert torch.equal(o["dur_loss"], dur) and torch.equal(o["prior_loss"], prior) and torch.equal(o["diff_loss"], diff), (seed, o["diff_loss"], diff)
