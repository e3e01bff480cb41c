"""The CPU oracle against the fixtures the reference itself produced (scripts/make_golden.py)."""
import pytest
import torch

from emojivoice_b200 import synthetic
from emojivoice_b200.config import HIFIGAN_V1, VCTK
from oracle import hifigan_oracle as ho
from oracle import matcha_oracle as mo
from tests import golden_io
from tests.conftest import rel_l2

TOL = 2e-5  # fp32 CPU kernels may differ in summation order between hosts; on the generating host it is 0


@pytest.mark.parametrize("name", golden_io.MATCHA)
def test_matcha_oracle_matches_reference_fixture(name, matcha_sd):
    g = golden_io.load(name)
    assert abs(synthetic.checksum(matcha_sd) - float(g["weights_checksum"])) < 1e-6 * abs(float(g["weights_checksum"]))
    out = mo.synthesise(matcha_sd, VCTK, **golden_io.matcha_inputs(g))
    assert out["mel_lengths"].tolist() == g["mel_lengths"].tolist()          # bit-exact
    assert torch.equal(out["attn"][:, 0], g["attn"])                          # bit-exact
    for k in ("encoder_outputs", "decoder_outputs", "mel"):
        assert rel_l2(out[k], torch.from_numpy(g[k])) < TOL, k


@pytest.mark.parametrize("name", list(golden_io.HIFIGAN))
def test_hifigan_oracle_matches_reference_fixture(name):
    g = golden_io.load(name)
    sd = synthetic.hifigan_state_dict(HIFIGAN_V1, **golden_io.HIFIGAN[name])
    assert abs(synthetic.checksum(sd) - float(g["weights_checksum"])) < 1e-6 * abs(float(g["weights_checksum"]))
    b, frames, seed = (int(v) for v in g["meta"])
    mel = synthetic.synthetic_mel(b, frames, seed=seed)
    wav = ho.generator(sd, HIFIGAN_V1, mel)
    assert wav.shape == (b, 1, frames * 256)
    assert rel_l2(wav, torch.from_numpy(g["wav"])) < TOL
    bias = ho.denoiser_bias(sd, HIFIGAN_V1)
    assert rel_l2(bias, torch.from_numpy(g["bias_spec"])) < 1e-4
    den = ho.denoise(wav.clamp(-1, 1).squeeze(1), bias, 0.00025)
    assert rel_l2(den, torch.from_numpy(g["denoised"])) < 1e-4


def test_parameter_counts_match_the_reference():
    """The state dicts the oracle and the CUDA loaders consume hold exactly the reference's parameters: 18,204,193 for the
    single-speaker Matcha-TTS (the count its synthesis.ipynb:127 prints; mel_mean / mel_std are buffers) and 13,926,017 for
    HiFi-GAN v1."""
    import dataclasses

    lj = synthetic.matcha_state_dict(dataclasses.replace(VCTK, n_spks=1), seed=1)
    assert sum(v.numel() for k, v in lj.items() if k not in ("mel_mean", "mel_std")) == 18_204_193
    assert sum(v.numel() for v in synthetic.hifigan_state_dict(HIFIGAN_V1).values()) == 13_926_017


def test_weight_norm_checkpoint_form_folds_to_plain_weights():
    plain = synthetic.hifigan_state_dict(HIFIGAN_V1, seed=7)
    wn = synthetic.hifigan_state_dict(HIFIGAN_V1, seed=7, weight_norm=True)
    folded = ho.fold_weight_norm(wn)
    assert set(folded) == set(plain)
    w, v, gk = folded["ups.0.weight"], wn["ups.0.weight_v"], wn["ups.0.weight_g"]
    assert torch.allclose(w.flatten(1).norm(dim=1), gk.flatten(), rtol=1e-5)
    assert torch.allclose(w / w.flatten(1).norm(dim=1).view(-1, 1, 1), v / v.flatten(1).norm(dim=1).view(-1, 1, 1), atol=1e-6)
