#!/usr/bin/env python
"""Vocoder + bias denoiser with a strength per utterance, or none, on one GPU.

    python scripts/per_item_denoise_bench.py [--reps 30] [--rounds 7] [--out FILE.json]

Synthetic weights (VCTK Matcha-TTS seed 1234, HiFi-GAN v1 seed 4321, bf16).  Prints the GPU name and power limit, then, on the
mel of the BASELINE config-2 batch (32 utterances of 60-90 phonemes, n = 10, temperature 0.667, length_scale 0.8), CUDA events
around steady-state calls (graph replay, the arms alternated, the median of --rounds rounds of --reps calls) of
  mixed:          one vocode_denoised call, strengths {off, 0.00025, 0.0005, 0.001} dealt round-robin (ev_to_waveform_items);
  split:          the same utterances as one call per setting on its sub-batch (vocode_denoised, or the ragged vocoder for off);
  all_denoised:   the mixed call with the off utterances denoised at 0.00025 instead (what "off" saves);
  scalar:         vocode_denoised at 0.00025 for the whole batch (ev_to_waveform_ragged);
  equal_items:    the per-item kernels with 0.00025 in every entry (callers that pass equal values get the scalar call instead).
The waveforms of mixed and split are compared bit for bit per utterance, as are scalar and equal_items.
Writes nothing unless --out is given."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import emojivoice_b200 as ev  # noqa: E402
from emojivoice_b200 import synthetic  # noqa: E402
from emojivoice_b200.config import HIFIGAN_V1, VCTK  # noqa: E402

SETTINGS = (None, 0.00025, 0.0005, 0.001)


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
    ap.add_argument("--rounds", type=int, default=7, help="alternations of the arms; each times --reps calls")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (B200)")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "settings_round_robin": list(SETTINGS)}

    model = ev.MatchaTTS(**VCTK.constructor_kwargs()).eval()
    model.load_state_dict(synthetic.matcha_state_dict(VCTK, seed=1234))
    voc = ev.Generator(HIFIGAN_V1)
    voc.load_state_dict(synthetic.hifigan_state_dict(HIFIGAN_V1, seed=4321))
    voc.remove_weight_norm()
    ev.Denoiser(voc)

    x, xl, spks = synthetic.phoneme_batch(32, 60, 90, seed=2000)
    out = model.synthesise(x, xl, 10, 0.667, spks, 0.8)
    mel, lens = out["mel"].contiguous(), out["mel_lengths"]
    ml = lens.cpu().tolist()
    B, T = mel.shape[0], mel.shape[-1]
    mixed = [SETTINGS[b % len(SETTINGS)] for b in range(B)]
    all_on = [0.00025 if s is None else s for s in mixed]
    groups = {s: [b for b in range(B) if mixed[b] == s] for s in SETTINGS}
    subs = {s: (mel[idx].contiguous(), lens[idx].contiguous()) for s, idx in ((s, torch.tensor(g, device=mel.device)) for s, g in groups.items())}

    def split():
        return {s: (voc(m, lengths=l) if s is None else voc.vocode_denoised(m, l, s)) for s, (m, l) in subs.items()}

    arms = {
        "mixed": lambda: voc.vocode_denoised(mel, lens, mixed),
        "split": split,
        "all_denoised": lambda: voc.vocode_denoised(mel, lens, all_on),
        "scalar": lambda: voc.vocode_denoised(mel, lens, 0.00025),
        "equal_items": torch.inference_mode()(lambda: voc._run(mel, None, lens, (0.00025,) * B)),
    }
    for fn in arms.values():          # warm up: first sight, capture, replays
        for _ in range(4):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, fn in arms.items():
            times[k].append(device_ms(fn, args.reps))
    got, parts = arms["mixed"](), arms["split"]()
    mixed_equals_split = all(torch.equal(got[b], parts[s][j]) for s, idx in groups.items() for j, b in enumerate(idx))
    equal_items_equals_scalar = torch.equal(arms["equal_items"](), arms["scalar"]())
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    frames = sum(ml)
    res["config2"] = {
        "batch": B, "T_pad": T, "valid_frames": frames, "audio_seconds": frames * 256 / 22050,
        "utterances_per_setting": {str(s): len(g) for s, g in groups.items()},
        "ms_per_call_median": med,
        "ms_per_call_all_rounds": times,
        "mixed_over_split": med["mixed"] / med["split"],
        "mixed_over_all_denoised": med["mixed"] / med["all_denoised"],
        "equal_items_over_scalar": med["equal_items"] / med["scalar"],
        "mixed_bit_identical_to_split": mixed_equals_split,
        "equal_items_bit_identical_to_scalar": equal_items_equals_scalar,
        "timing": "CUDA events around --reps back-to-back calls (CUDA-graph replay), --rounds rounds alternating the arms, median",
    }
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
