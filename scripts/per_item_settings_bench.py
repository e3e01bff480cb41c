#!/usr/bin/env python
"""Per-utterance synthesis settings on one GPU: what a batch with mixed (length_scale, temperature, n_timesteps) costs.

    python scripts/per_item_settings_bench.py [--reps 10] [--rounds 5] [--out profiles/per_item_settings_bench_v1.json]

Synthetic weights (VCTK Matcha-TTS seed 1234, bf16, CUDA-graph replay), the BASELINE config-2 batch (32 utterances of 60-90
phonemes, seed 2000), MatchaTTS.synthesise only (text to mel; the vocoder is not part of any arm).  Every arm is timed with CUDA
events around --reps back-to-back steady-state calls, --rounds rounds alternating the arms of a comparison:
  1. scalar   synthesise(x, n=10, temperature=0.667, length_scale=0.8)  against the same call with per-item arrays that are
     all equal;
  2. mixed    one batch mixing length scales {0.8, 0.9, 1.0}, temperatures {0.5, 0.667} and n in {4, 10} (12 setting triples)
     against the same utterances split into one sub-batch per triple, run one after another; both with one batch in flight
     and with three (model replicas on their own streams, as synthesise_corpus(in_flight=3)): there, three copies of the
     workload are dealt to the lanes and the time is divided by three;
  3. held     the mixed batch against the same batch at a uniform n = 10 (the steps past an item's own n are computed and
     discarded).
Prints the GPU name and power limit read in the same run."""
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
    return {"ms_per_call_median": {k: round(v, 3) for k, v in med.items()}, "ms_per_call_all_rounds": times}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5, help="alternations of the arms; each times --reps calls")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "per_item_settings_bench_v1.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (B200)")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "workload": "BASELINE config-2 batch (32 x 60-90 phonemes, seed 2000), synthesise only, bf16, graph replay",
           "timing": "CUDA events around --reps back-to-back calls, --rounds rounds alternating the arms, median round reported",
           "reps": args.reps, "rounds": args.rounds}

    model = ev.MatchaTTS(**VCTK.constructor_kwargs()).eval()
    model.load_state_dict(synthetic.matcha_state_dict(VCTK, seed=1234))
    voc = ev.Generator(HIFIGAN_V1)
    voc.load_state_dict(synthetic.hifigan_state_dict(HIFIGAN_V1, seed=4321))
    voc.remove_weight_norm()
    x, xl, spks = synthetic.phoneme_batch(32, 60, 90, seed=2000)
    B = x.shape[0]

    # 1. scalar call against equal per-item arrays
    res["scalar_vs_equal_arrays"] = compare({
        "scalar": lambda: model.synthesise(x, xl, 10, 0.667, spks, 0.8),
        "equal_per_item_arrays": lambda: model.synthesise(x, xl, [10] * B, [0.667] * B, spks, [0.8] * B),
    }, args.reps, args.rounds)

    # 2. one mixed batch against one sub-batch per setting triple
    ls = [(0.8, 0.9, 1.0)[i % 3] for i in range(B)]
    temps = [(0.5, 0.667)[(i // 3) % 2] for i in range(B)]
    ns = [(4, 10)[(i // 6) % 2] for i in range(B)]
    groups = {}
    for i in range(B):
        groups.setdefault((ls[i], temps[i], ns[i]), []).append(i)
    subs = []
    for (l, t, n), items in sorted(groups.items()):
        idx = torch.tensor(items)
        tx = int(xl[idx].max())
        subs.append((x[idx, :tx].contiguous(), xl[idx].contiguous(), spks[idx].contiguous(), n, t, l))

    def mixed(m):
        return m.synthesise(x, xl, ns, temps, spks, ls)

    def split(m):
        for xs, xls, ss, n, t, l in subs:
            m.synthesise(xs, xls, n, t, ss, l)

    lanes = ev.lanes_for(model, voc, 3)

    def in_flight(work):
        caller = torch.cuda.current_stream()
        for st in lanes.streams:
            st.wait_stream(caller)
        for k, w in enumerate(work):
            lane = k % len(lanes)
            with torch.cuda.stream(lanes.streams[lane]):
                w(lanes.models[lane])
        for st in lanes.streams:
            caller.wait_stream(st)

    three_mixed = [mixed] * 3
    three_split = [lambda m, s=s: m.synthesise(s[0], s[1], s[3], s[4], s[2], s[5]) for s in subs] * 3
    res["setting_triples"] = len(subs)
    res["sub_batch_sizes"] = [len(v) for _, v in sorted(groups.items())]
    one = compare({"mixed_batch": lambda: mixed(model), "split_sub_batches": lambda: split(model)}, args.reps, args.rounds)
    three = compare({"mixed_batch": lambda: in_flight(three_mixed), "split_sub_batches": lambda: in_flight(three_split)},
                    args.reps, args.rounds)
    three["ms_per_batch_of_32_median"] = {k: round(v / 3, 3) for k, v in three["ms_per_call_median"].items()}
    res["mixed_vs_split"] = {"in_flight_1": one, "in_flight_3": three}

    # 3. cost of held items: the mixed batch against the same batch at a uniform n = 10
    res["held_items"] = compare({
        "mixed_n_4_and_10": lambda: mixed(model),
        "uniform_n_10": lambda: model.synthesise(x, xl, 10, temps, spks, ls),
    }, args.reps, args.rounds)
    res["held_items"]["steps_computed_and_discarded"] = sum(max(ns) - n for n in ns)
    res["held_items"]["steps_total"] = B * max(ns)

    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
