#!/usr/bin/env python
"""Vocoder + bias denoiser on a padded batch, dense against ragged, on one GPU.

    python scripts/ragged_denoise_bench.py [--reps 30] [--corpus-passes 2] [--out FILE.json]

Synthetic weights (VCTK Matcha-TTS seed 1234, HiFi-GAN v1 seed 4321, bf16).  Prints the GPU name and power limit, then
  * the BASELINE config-2 batch (32 utterances of 60-90 phonemes, n = 10, temperature 0.667, length_scale 0.8) synthesised
    once; on its mel, CUDA events around steady-state calls (graph replay, calls alternated between the arms) of
      dense:  Denoiser(vocoder(mel).clamp(-1, 1)) -- the whole padded batch vocoded and denoised;
      ragged: vocoder.vocode_denoised(mel, mel_lengths) -- ev_to_waveform_ragged;
      and, for scale, the ragged vocoder alone and the dense denoiser alone;
    the cropped waveforms of the two arms are compared bit for bit;
  * synthesise_corpus(denoiser=...) over the BASELINE config-3 corpus (1024 mixed-length utterances, micro-batches of 32,
    three in flight), ragged=False against ragged=True, host wall clock per pass after a warm-up pass of each.
Writes nothing unless --out is given."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import emojivoice_b200 as ev  # noqa: E402
from emojivoice_b200 import synthetic  # noqa: E402
from emojivoice_b200.config import HIFIGAN_V1, VCTK  # noqa: E402

STRENGTH = 0.00025          # feel_me.py:185


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 else None}


def device_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=5, help="alternations of the arms; each times --reps calls")
    ap.add_argument("--corpus-passes", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (B200)")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "strength": STRENGTH}

    model = ev.MatchaTTS(**VCTK.constructor_kwargs()).eval()
    model.load_state_dict(synthetic.matcha_state_dict(VCTK, seed=1234))
    voc = ev.Generator(HIFIGAN_V1)
    voc.load_state_dict(synthetic.hifigan_state_dict(HIFIGAN_V1, seed=4321))
    voc.remove_weight_norm()
    den = ev.Denoiser(voc)

    # ---- config-2 batch
    x, xl, spks = synthetic.phoneme_batch(32, 60, 90, seed=2000)
    out = model.synthesise(x, xl, 10, 0.667, spks, 0.8)
    mel, lens = out["mel"], out["mel_lengths"]
    ml = lens.cpu().tolist()
    T = mel.shape[-1]
    arms = {
        "dense_vocoder_denoiser": lambda: den(voc(mel).clamp(-1, 1).squeeze(1), strength=STRENGTH),
        "ragged_vocoder_denoiser": lambda: voc.vocode_denoised(mel, lens, STRENGTH),
        "ragged_vocoder_alone": lambda: voc(mel, lengths=lens),
    }
    wav_dense = voc(mel).clamp(-1, 1).squeeze(1)
    arms["dense_denoiser_alone"] = lambda: den(wav_dense, strength=STRENGTH)
    for fn in arms.values():          # warm up: first sight, capture, replays
        for _ in range(4):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, fn in arms.items():
            times[k].append(device_ms(fn, args.reps))
    dense, ragged = arms["dense_vocoder_denoiser"](), arms["ragged_vocoder_denoiser"]()
    identical = all(torch.equal(ragged[b, 0, : n * 256], dense[b, : n * 256]) and float(ragged[b, 0, n * 256:].abs().sum()) == 0.0
                    for b, n in enumerate(ml))
    frames = sum(ml)
    res["config2"] = {
        "batch": 32, "T_pad": T, "valid_frames": frames, "padded_frames": 32 * T, "audio_seconds": frames * 256 / 22050,
        "ms_per_call_median": {k: sorted(v)[len(v) // 2] for k, v in times.items()},
        "ms_per_call_all_rounds": times,
        "cropped_waveforms_bit_identical": identical,
        "timing": "CUDA events around --reps back-to-back calls (CUDA-graph replay), --rounds rounds alternating the arms",
    }

    # ---- config-3 corpus through synthesise_corpus
    utts = synthetic.mixed_length_corpus(1024)
    lanes = ev.lanes_for(model, voc, 3)
    passes = {"ragged_false": [], "ragged_true": []}
    results = {}
    for rep in range(args.corpus_passes + 1):
        for name, rag in (("ragged_false", False), ("ragged_true", True)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r, st = ev.synthesise_corpus(model, voc, utts, batch_size=32, n_timesteps=10, temperature=0.667, length_scale=0.8,
                                         denoiser=den, denoiser_strength=STRENGTH, ragged=rag, lanes=lanes)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            if rep > 0:       # pass 0 warms both arms (new shapes, workspace growth)
                passes[name].append({"wall_s": round(wall, 3), "audio_s_per_s_wall": round(st.audio_seconds / wall, 1)})
            results[name] = r
    same_mel = all(results["ragged_true"][i]["mel_length"] == results["ragged_false"][i]["mel_length"] for i in results["ragged_false"])
    res["config3_denoised"] = {
        "utterances": len(utts), "in_flight": 3, "passes": passes, "mel_lengths_equal": same_mel,
        "timing": "host wall clock around synthesise_corpus incl. D2H + crop, after one warm-up pass of each arm; the prior noise is "
                  "drawn per call, so waveforms are not compared here (tests/test_ragged_denoise.py compares them with shared noise)",
    }
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
