#!/usr/bin/env python
"""Seeded prior noise on one GPU: what ev_prior_noise costs, alone and inside MatchaTTS.synthesise.

    python scripts/seeded_noise_bench.py [--launches 1000] [--reps 30] [--rounds 5] [--out profiles/seeded_noise_bench_v1.json]

  1. kernel   ev_prior_noise at the config-2 shape (32 x 80 x 668): CUDA events around --launches back-to-back launches,
              --rounds times; the 6.8 MB output stays in L2 between launches, so this is the kernel's compute-bound time.
  2. synthesise  the BASELINE config-2 batch (32 utterances of 60-90 phonemes, seed 2000; synthetic VCTK weights seed 1234,
              bf16, n = 10, CUDA-graph replay), text to mel only: seed= (an int64 device tensor, and a Python list) against
              z=None (torch.randn).  CUDA events around --reps back-to-back calls, --rounds rounds alternating the arms.
Prints the GPU name and power limit read in the same run, and one JSON line of the headline numbers."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import emojivoice_b200 as ev  # noqa: E402
from emojivoice_b200 import _lib, synthetic  # noqa: E402
from emojivoice_b200.config import VCTK  # noqa: E402
from emojivoice_b200.matcha import per_item_seed  # noqa: E402


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


def compare(arms, reps, rounds, warm=4):
    for fn in arms.values():          # first sight, capture, replays
        for _ in range(warm):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(device_ms(fn, reps))
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    return {"ms_per_call_median": {k: round(v, 4) for k, v in med.items()},
            "ms_per_call_spread": {k: round(max(v) - min(v), 4) for k, v in times.items()}, "ms_per_call_all_rounds": times}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=5, help="alternations of the arms; each times --reps calls")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "seeded_noise_bench_v1.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (B200)")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "launches": args.launches, "reps": args.reps, "rounds": args.rounds}

    # 1. the kernel alone
    B, F, T = 32, 80, 668
    ctx, L = _lib.Context(), _lib.lib()
    seeds = per_item_seed(list(range(B)), B).cuda()
    z = torch.empty(B, F, T, device="cuda")

    def launch():
        ctx.check(L.ev_prior_noise(ctx.handle, _lib.ptr(seeds), B, F, T, _lib.ptr(z), _lib.stream_ptr()), "ev_prior_noise")

    for _ in range(10):
        launch()
    torch.cuda.synchronize()
    us = [device_ms(launch, args.launches) * 1e3 for _ in range(args.rounds)]
    med = sorted(us)[len(us) // 2]
    nbytes = B * F * T * 4
    res["kernel"] = {"shape": [B, F, T], "us_per_launch_median": round(med, 3), "us_per_launch_all_rounds": [round(v, 3) for v in us],
                     "output_bytes": nbytes, "achieved_GB_per_s": round(nbytes / (med * 1e-6) / 1e9, 1),
                     "normal_draws_per_s": round(B * F * T / (med * 1e-6), 1)}

    # 2. synthesise with and without a seed
    model = ev.MatchaTTS(**VCTK.constructor_kwargs()).eval()
    model.load_state_dict(synthetic.matcha_state_dict(VCTK, seed=1234))
    x, xl, spks = synthetic.phoneme_batch(32, 60, 90, seed=2000)
    dev_seeds = per_item_seed(list(range(1000, 1032)), 32).cuda()
    host_seeds = list(range(1000, 1032))
    res["synthesise"] = compare({
        "randn": lambda: model.synthesise(x, xl, 10, 0.667, spks, 1.0),
        "seed_device_tensor": lambda: model.synthesise(x, xl, 10, 0.667, spks, 1.0, seed=dev_seeds),
        "seed_list": lambda: model.synthesise(x, xl, 10, 0.667, spks, 1.0, seed=host_seeds),
    }, args.reps, args.rounds)
    res["synthesise"]["t_pad"] = model.synthesise(x, xl, 10, 0.667, spks, 1.0, seed=dev_seeds)["t_pad"]
    res["synthesise"]["workload"] = "BASELINE config-2 batch (32 x 60-90 phonemes, seed 2000), synthesise only, bf16, n = 10, graph replay"

    print(json.dumps(res, indent=1))
    m = res["synthesise"]["ms_per_call_median"]
    print(json.dumps({"gpu": res["gpu"]["nvidia_smi"], "prior_noise_us": res["kernel"]["us_per_launch_median"],
                      "synthesise_ms_randn": m["randn"], "synthesise_ms_seed": m["seed_device_tensor"],
                      "synthesise_ms_seed_list": m["seed_list"]}))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
