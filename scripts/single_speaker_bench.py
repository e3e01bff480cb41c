#!/usr/bin/env python
"""Single-speaker Matcha-TTS (n_spks = 1, the LJSpeech layout: 96-wide text-encoder heads, 160-channel decoder input) on one GPU.

    python scripts/single_speaker_bench.py [--reps 20] [--out FILE.json]

Synthetic weights (synthetic.matcha_state_dict, seed 1234) and HiFi-GAN v1 (seed 4321): durations follow the synthetic
duration predictor, not a trained one.  Prints the GPU name and power limit, then
  * B = 1, Tx = 151, n = 10, temperature 0.667, length_scale 1.0 (synthesis.ipynb's settings): synthesise and synthesise +
    vocoder timed with CUDA events (steady state, graph replay), as RTF and audio seconds per second, and the reference-style
    RTF (host clock around the call, no synchronisation: matcha_tts.py:142-143), plus the mel's rel-L2 against the CPU oracle;
  * the BASELINE config-2 shape (B = 32, 60-90 phonemes, length_scale 0.8, n = 10), one batch at a time;
  * the text-encoder attention alone at head width 96, tcgen05 (impl 1) vs fp32 CUDA cores (impl 0), microseconds per launch
    and rel-L2 against float64, at (B 32, Tx 177, H 2) and (B 32, Tx 384, H 2).
Writes nothing unless --out is given."""
import argparse
import ctypes as C
import dataclasses
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import emojivoice_b200 as ev  # noqa: E402
from emojivoice_b200 import _lib, synthetic  # noqa: E402
from emojivoice_b200.config import HIFIGAN_V1, VCTK  # noqa: E402
from oracle import matcha_oracle as mo  # noqa: E402

LJ = dataclasses.replace(VCTK, n_spks=1)


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


def workload(model, gen, x, xl, ls, reps, ragged):
    res = {}

    def synth():
        res["out"] = model.synthesise(x, xl, 10, 0.667, None, ls)

    def synth_voc():
        synth()
        o = res["out"]
        res["wav"] = gen(o["mel"], lengths=o["mel_lengths"] if ragged else None)

    for _ in range(3):                                      # eager, capture, replay: every timed call below replays
        synth_voc()
    torch.cuda.synchronize()
    audio_s = float(res["out"]["mel_lengths"].sum()) * 256 / 22050
    ms_s, ms_sv = device_ms(synth, reps), device_ms(synth_voc, reps)
    host_rtf = []
    for _ in range(reps):
        host_rtf.append(model.synthesise(x, xl, 10, 0.667, None, ls)["rtf"])
        torch.cuda.synchronize()
    return {"B": int(x.shape[0]), "Tx_max": int(x.shape[1]), "frames": res["out"]["mel_lengths"].cpu().tolist() if x.shape[0] == 1
            else int(res["out"]["mel_lengths"].sum()), "audio_s": round(audio_s, 4),
            "synthesise_ms": round(ms_s, 3), "synthesise_rtf": round(ms_s / 1e3 / audio_s, 6), "synthesise_audio_s_per_s": round(audio_s / (ms_s / 1e3), 1),
            "synth_vocoder_ms": round(ms_sv, 3), "synth_vocoder_rtf": round(ms_sv / 1e3 / audio_s, 6),
            "synth_vocoder_audio_s_per_s": round(audio_s / (ms_sv / 1e3), 1),
            "reference_style_host_rtf_mean": round(sum(host_rtf) / len(host_rtf), 6)}


def attention(ctx, B, T, H, hd, reps):
    g = torch.Generator().manual_seed(1)
    qkv = torch.randn(B, T, 3 * H * hd, generator=g) * 1.7
    lens = torch.randint(T // 2, T + 1, (B,), generator=g)
    q, k, v = (z.reshape(B, T, H, hd).transpose(1, 2).double() for z in qkv.chunk(3, dim=2))
    q, k = mo._rope(q, hd // 2).double(), mo._rope(k, hd // 2).double()
    m = (torch.arange(T)[None, :] < lens[:, None]).double()
    sc = ((q @ k.transpose(-2, -1)) / math.sqrt(hd)).masked_fill((m[:, None, :, None] * m[:, None, None, :]) == 0, -1e4)
    ref = (torch.softmax(sc, dim=-1) @ v).transpose(1, 2).reshape(B, T, H * hd)
    qd, ld = qkv.cuda(), lens.cuda()
    row = {"B": B, "Tx": T, "H": H, "head_width": hd}
    for impl, name in ((1, "attention_enc_tc"), (0, "attention_enc_f32")):
        out = torch.empty(B, T, H * hd, device="cuda")
        us = C.c_float(0.0)
        ctx.check(_lib.lib().ev_test_encoder_attention_hd(ctx.handle, _lib.ptr(qd), _lib.ptr(ld), B, T, H, hd, impl, _lib.ptr(out), 10,
                                                          None, _lib.stream_ptr()), "warm-up")
        ctx.check(_lib.lib().ev_test_encoder_attention_hd(ctx.handle, _lib.ptr(qd), _lib.ptr(ld), B, T, H, hd, impl, _lib.ptr(out), reps,
                                                          C.byref(us), _lib.stream_ptr()), name)
        row[name] = {"us_per_launch": round(us.value, 2), "rel_l2_vs_float64": float((out.cpu().double() - ref).norm() / ref.norm())}
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "weights": "synthetic (matcha seed 1234, hifigan v1 seed 4321)"}
    print(json.dumps(res["gpu"]))
    sd = synthetic.matcha_state_dict(LJ, seed=1234)
    model = ev.MatchaTTS(**LJ.constructor_kwargs())
    model.load_state_dict(sd)
    gen = ev.Generator(HIFIGAN_V1)
    gen.load_state_dict(synthetic.hifigan_state_dict(HIFIGAN_V1, seed=4321, gain=1.0))
    gen.remove_weight_norm()

    x, xl, _ = synthetic.phoneme_batch(1, 75, 75, seed=151)              # Tx = 151
    res["notebook_b1_tx151"] = workload(model, gen, x, xl, 1.0, args.reps, ragged=False)
    print("B=1 Tx=151 n=10:", json.dumps(res["notebook_b1_tx151"]))
    probe = mo.synthesise(sd, LJ, x, xl, 1, 0.667, None, 1.0)
    z = synthetic.prior_noise(1, 80, probe["t_pad"], seed=152)
    ref = mo.synthesise(sd, LJ, x, xl, 10, 0.667, None, 1.0, z=z)
    acc = {}
    for prec in ("fp32", "bf16"):
        o = model.synthesise(x, xl, 10, 0.667, None, 1.0, z=z, dtype=prec)
        acc[prec] = {"mel_rel_l2_vs_oracle": float((o["mel"].cpu().double() - ref["mel"].double()).norm() / ref["mel"].double().norm()),
                     "attn_equal": bool(torch.equal(o["attn"].cpu(), ref["attn"]))}
    res["notebook_b1_tx151"]["accuracy"] = acc
    print("B=1 Tx=151 n=10 vs oracle:", json.dumps(acc))

    x, xl, _ = synthetic.phoneme_batch(32, 60, 90, seed=2000)             # BASELINE config-2 shape
    res["config2_b32"] = workload(model, gen, x, xl, 0.8, args.reps, ragged=True)
    print("B=32 config-2 shape:", json.dumps(res["config2_b32"]))

    ctx = _lib.Context("cuda:0")
    res["encoder_attention"] = [attention(ctx, 32, T, 2, hd, 200) for T in (177, 384) for hd in (96, 128)]
    for r in res["encoder_attention"]:
        print("encoder attention:", json.dumps(r))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
