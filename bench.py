#!/usr/bin/env python
"""Headline benchmark: audio-seconds synthesised per second (22.05 kHz, mel + vocoder) on N x B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: MatchaTTS.synthesise(x, x_lengths, n_timesteps=10,
temperature=0.667, spks=emoji ids, length_scale=0.8) followed by vocoder(mel).clamp(-1, 1), on BASELINE.json
configs[1] (batch 32 emoji-tagged utterances of ~5 s, bf16, random-init VCTK Matcha-TTS + HiFi-GAN v1).
For N > 1 the driver launches one rank per GPU with torch.distributed.run; utterances shard by batch, every
rank synthesises the same 32-utterance batch (weak scaling: identical work per GPU), no collective on the data path.

Throughput is measured with `--in-flight` (default 3) batches in flight per GPU: step i runs on lane i % 3, a lane being
its own model / vocoder instance and CUDA stream (emojivoice_b200.Lanes, what synthesise_corpus does with a corpus) --
a step is a chain of ~70 dependent launches, many latency-bound, and the other lanes' kernels fill its gaps.  K steps are
still timed as one bracket (barrier + synchronize, CUDA events, max over ranks); `one_step_at_a_time` is the same loop
without the overlap (the figure every earlier bench line of this repo reports).

One JSON line is printed by rank 0 (see the task contract): `value` is measured with the inputs resident in HBM,
`e2e` through the same public API with pinned HOST inputs and the waveform read back, `roofline` for the dominant
kernel class (plus `rooflines` per stage) from a CUDA-event-instrumented step, `cpu_baseline` = the reference's own CPU
PyTorch path (the unmodified files staged under baseline/_ref, else the oracle port) timed on this box's host cores on a
bounded sample.  Further blocks: `padded_vocoder` (the reference's literal work list, with its own e2e), `denoiser`,
`config3` (BASELINE configs[2]: 1024 mixed-length utterances sharded over the N ranks through synthesise_corpus, strong
scaling, wall clock incl. D2H + crop, cold = never-seen shapes and warm) and `config5` (vocoder only, 60-s segments).

`--dump-outputs DIR` writes what the last timed step returned to its caller (the synthesise dict of the reference and the
waveform) as DIR/<name>.npy.  The prior noise is drawn from a generator seeded before the timed region, so with the same
arguments two runs, or two builds, compute the same step and can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SR, HOP = 22050, 256
N_TIMESTEPS, TEMPERATURE, LENGTH_SCALE = 10, 0.667, 0.8      # feel_me.py:71-77 (the operating point of every app)
BATCH, P_LO, P_HI = 32, 60, 90                                # SURVEY.md 8d config 2: Tx = 2P+1 in [121, 181]
CPU_SAMPLE = 8                                                # utterances the `cpu_baseline` leg / reference warm-up synthesise (~4.5 s per pass)
DUMP_BYTES = 64 * 10**6                                       # cap on what --dump-outputs writes in all
DUMPED = ("encoder_outputs", "decoder_outputs", "attn", "mel", "mel_lengths")      # the dict the reference's synthesise returns


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=float(p["hbm_gbs"]), tflops=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                    source="MEASURED_PEAKS.json (sustained bf16, copy bandwidth)")
    return dict(hbm_gbs=6650.0, tflops=1400.0, source="fallback of B200_PROFILING.md")


class ClockSampler:
    """SM clock + throttle reasons sampled every 100 ms while the timed region runs, through NVML in-process
    (spawning `nvidia-smi -lms` was measurably perturbing the launch path on the GPU box)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index: int):
        self.gpu, self.sm, self.bits, self.stop_flag, self.thread, self.h, self.mx = gpu_index, [], 0, False, None, None, None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception:
                pass
            time.sleep(0.1)

    def start(self):
        if self.h is not None:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.thread.join(timeout=1.0)
        reasons = sorted(n for b, n in self.REASONS.items() if self.bits & b)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.mx, "reasons": reasons,
                "samples": len(self.sm)}


TRAFFIC_FILE = ["r02_launch_summary.json"]


def measured_traffic(kernel_class: str):
    """DRAM bytes per launch of a kernel function from the committed ncu launch list of this same command
    (profiles/r02_launch_summary.json -- r01 when this round's capture is not there yet -- written by
    scripts/ncu_launch_summary.py); None when no capture is committed."""
    import re

    path = os.path.join(ROOT, "profiles", TRAFFIC_FILE[0])
    if not os.path.exists(path):
        TRAFFIC_FILE[0] = "r01_launch_summary.json"
        path = os.path.join(ROOT, "profiles", TRAFFIC_FILE[0])
    if not os.path.exists(path):
        return None, None
    k = json.load(open(path))["kernels"]
    m = re.match(r"conv_tc_(bn|tf32x)(\d+)", kernel_class)
    fn = "conv_tc_kernel<%s>" % (m.group(2) if m.group(1) == "bn" else "128") if m else None
    if kernel_class.startswith("resblock_tc"):
        hits = [v for n, v in k.items() if n.startswith("resblock_tc_kernel")]
        if hits:
            n = sum(h["launches"] for h in hits)
            return sum(h["dram_bytes_per_launch"] * h["launches"] for h in hits) / n, "resblock_tc_kernel<*>"
    if fn in k:
        return k[fn]["dram_bytes_per_launch"], fn
    return None, None


def audio_seconds(mel_lengths) -> float:
    return float(mel_lengths.sum()) * HOP / SR


def dump_outputs(out_dir, tensors, cap=DUMP_BYTES):
    """Write each tensor as out_dir/<name>.npy: floating point as float32, integers as float64 (exact).  Should the whole
    exceed `cap` bytes, every array above 1 MiB keeps the same fraction of its elements, flattened, at ascending positions
    drawn with a fixed seed (identical positions from run to run as long as the shapes agree); its original shape is then
    written beside it as <name>.shape.npy."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrs = {k: (t.detach().float() if t.is_floating_point() else t.detach().double()).cpu().numpy() for k, t in tensors.items()}
    big = [k for k, a in arrs.items() if a.nbytes > 2**20]
    need = sum(arrs[k].nbytes for k in big)
    room = cap - 8192 * len(arrs) - sum(a.nbytes for k, a in arrs.items() if k not in big)      # (8192: .npy headers, shapes)
    for name, a in arrs.items():
        if name in big and need > room:
            np.save(os.path.join(out_dir, name + ".shape.npy"), np.array(a.shape, dtype=np.float64))
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, a.size * room // need, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


class CpuArm:
    """The reference's CPU PyTorch implementation of the path on this box's host cores, all host threads:
    kind "reference" = the reference's UNMODIFIED files (staged under baseline/_ref by scripts/install_reference.py, or
    /root/reference in the build container) driven through oracle/reference_shim.py -- MatchaTTS.synthesise(...) then
    Generator(mel).clamp(-1, 1) exactly as feel_me.py:193-200,183 calls them; kind "port" = the oracle's restatement, only
    when no copy of the reference travelled."""

    def __init__(self):
        from emojivoice_b200 import synthetic
        from emojivoice_b200.config import HIFIGAN_V1, VCTK
        from oracle import reference_shim as shim

        torch.set_num_threads(os.cpu_count() or 1)
        self.cores = torch.get_num_threads()
        sd = synthetic.matcha_state_dict(VCTK, seed=1234)
        hsd = synthetic.hifigan_state_dict(HIFIGAN_V1, seed=4321)
        if shim.available():
            self.kind, self.src = "reference", shim.REFERENCE_ROOT
            self.model, self.voc = shim.build_matcha(VCTK, sd), shim.build_hifigan(HIFIGAN_V1, hsd)
        else:
            from oracle import hifigan_oracle as ho
            from oracle import matcha_oracle as mo

            self.kind, self.src = "port", "oracle/"
            self.model = lambda x, xl, n, t, s, ls: mo.synthesise(sd, VCTK, x, xl, n, t, s, ls)
            self.voc = lambda mel: ho.generator(hsd, HIFIGAN_V1, mel)

    @torch.inference_mode()
    def once(self, x, xl, spks, n_utts=None):
        """One pass over the first n_utts utterances (all when None) -> (audio seconds, wall seconds)."""
        n = x.shape[0] if n_utts is None else min(n_utts, x.shape[0])
        xs, ls, ss = x[:n, : int(xl[:n].max())].contiguous(), xl[:n], spks[:n]
        t0 = time.perf_counter()
        if self.kind == "reference":
            out = self.model.synthesise(xs, ls, n_timesteps=N_TIMESTEPS, temperature=TEMPERATURE, spks=ss, length_scale=LENGTH_SCALE)
        else:
            out = self.model(xs, ls, N_TIMESTEPS, TEMPERATURE, ss, LENGTH_SCALE)
        wav = self.voc(out["mel"]).clamp(-1, 1)
        dt = time.perf_counter() - t0
        assert wav.shape[-1] == out["mel"].shape[-1] * HOP
        return audio_seconds(out["mel_lengths"]), dt


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path, all host threads, on the SAME workload as our arm:
    every timed step synthesises the whole 32-utterance batch (about 19 s of CPU work); the W warm-up steps run the first
    CPU_SAMPLE utterances only, so the default K = 20 finishes in about 6.5 minutes."""
    if rank != 0:
        return
    from emojivoice_b200 import synthetic

    x, xl, spks = synthetic.phoneme_batch(BATCH, P_LO, P_HI, seed=2000)
    arm = CpuArm()
    for _ in range(args.warmup):
        arm.once(x, xl, spks, CPU_SAMPLE)
    t0 = time.perf_counter()
    secs = 0.0
    for _ in range(args.steps):
        a, _ = arm.once(x, xl, spks)
        secs += a
    dt = time.perf_counter() - t0
    val = secs / dt
    sample = (f"all {BATCH} utterances of the batch per timed step ({secs / args.steps:.1f} audio-s), fp32 torch CPU, "
              f"{arm.kind} ({arm.src}); warm-up steps: first {CPU_SAMPLE} utterances")
    print(json.dumps({
        "impl": "reference", "metric": "audio_seconds_per_second", "value": val, "unit": "audio-s/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(),
        "cpu_baseline": {"value": val, "unit": "audio-s/s", "cores": arm.cores, "kind": arm.kind, "sample": sample},
        "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "rtf": 1.0 / val}))


def workload_config():
    return {"workload": "BASELINE.json configs[1]: batch 32 emoji-tagged utterances (~5 s each), n_timesteps=10, "
                        "Matcha-TTS VCTK arch + HiFi-GAN v1, random init, synthetic blank-interspersed phoneme ids",
            "batch_per_gpu": BATCH, "n_timesteps": N_TIMESTEPS, "temperature": TEMPERATURE, "length_scale": LENGTH_SCALE,
            "tokens_per_utt": f"2P+1, P~U[{P_LO},{P_HI}]", "speakers": "11 emoji voices (feel_me.py:84-96)"}


def roofline_of(a, peaks, ksum):
    """Roofline entry of one kernel class of the instrumented step (algorithmic FLOPs / bytes of the valid, un-padded work)."""
    sec = a["total_ms"] / 1e3
    ridge = peaks["tflops"] * 1e12 / (peaks["hbm_gbs"] * 1e9)
    ai = a["flops"] / max(a["bytes"], 1.0)
    if a["flops"] > 0 and ai >= ridge:
        ach, peak, unit, bound = a["flops"] / sec / 1e12, peaks["tflops"], "TFLOP/s", "tensor"
    else:
        ach, peak, unit, bound = a["bytes"] / sec / 1e9, peaks["hbm_gbs"], "GB/s", "hbm"
    n = max(a["launches"], 1)
    return {"kernel": a["name"], "bound": bound, "achieved": round(ach, 2), "peak": peak, "unit": unit, "frac": round(ach / peak, 4),
            "traffic": None, "launches": a["launches"], "algorithmic_bytes_per_launch": round(a["bytes"] / n),
            "algorithmic_flops_per_launch": round(a["flops"] / n), "avg_launch_us": round(a["total_ms"] * 1e3 / n, 2),
            "share_of_step": round(a["total_ms"] / ksum, 4), "arith_intensity": round(ai, 1),
            "tflops": round(a["flops"] / sec / 1e12, 2) if sec else 0.0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the config3 / config5 / denoiser blocks (headline numbers only)")
    ap.add_argument("--in-flight", type=int, default=3,
                    help="batches in flight on one GPU (lanes = model/vocoder instances on their own streams, ev.Lanes); 1 = one step at a time")
    ap.add_argument("--dense-vocoder", action="store_true",
                    help="vocode the padded frames of every utterance too (the default skips the time tiles past each utterance's "
                         "own length: identical waveform on [: length*256], zero beyond -- what cli.py:307-311 crops away)")
    ap.add_argument("--profile-one-step", action="store_true",
                    help="after warm-up, bracket ONE step with cudaProfilerStart/Stop and exit (for `ncu --profile-from-start off`)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (%s, waveform) as DIR/<name>.npy, float32 "
                         "(float64 for the lengths), at most 64 MB in all" % ", ".join(DUMPED))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.profile_one_step):
        ap.error("--dump-outputs writes the outputs of the timed CUDA path: not with --impl reference or --profile-one-step")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    n_warm_min = max(args.warmup, 3)                             # the contract's floor; the JSON line echoes the requested value

    import torch.distributed as dist

    import emojivoice_b200 as ev
    from emojivoice_b200 import _lib as _lib_mod
    from emojivoice_b200 import synthetic
    from emojivoice_b200.config import HIFIGAN_V1, VCTK

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the CUDA path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(vals, op):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=op)
        return t.tolist()

    MAX, SUM = (dist.ReduceOp.MAX, dist.ReduceOp.SUM)

    model = ev.MatchaTTS(**VCTK.constructor_kwargs(), device=dev, precision=args.precision).eval()
    model.load_state_dict(synthetic.matcha_state_dict(VCTK, seed=1234))
    voc = ev.Generator(HIFIGAN_V1, device=dev, precision=args.precision)
    voc.load_state_dict(synthetic.hifigan_state_dict(HIFIGAN_V1, seed=4321))
    voc.eval()
    voc.remove_weight_norm()

    # weak scaling: every rank synthesises the SAME 32-utterance batch (identical work per GPU, so the per-N values are
    # comparable; round 1 drew a different batch per rank and rank 0's happened to be the heaviest)
    x, xl, spks = synthetic.phoneme_batch(BATCH, P_LO, P_HI, seed=2000)
    x_pin, xl_pin, spk_pin = x.pin_memory(), xl.pin_memory(), spks.pin_memory()
    x_dev, xl_dev, spk_dev = x.to(dev), xl.to(dev), spks.to(dev)

    ragged = [not args.dense_vocoder]
    # batches in flight: step i runs on lane i % n (its own model / vocoder instance and stream, emojivoice_b200/batch.py Lanes);
    # `serial[0]` pins every step to lane 0, i.e. one step at a time
    lanes = ev.lanes_for(model, voc, max(1, args.in_flight))
    n_lanes = len(lanes)
    caller = torch.cuda.current_stream(dev)
    serial = [False]
    counter = [0]

    def next_lane():
        i = counter[0]
        counter[0] += 1
        lane = 0 if serial[0] else i % n_lanes
        return lane, lanes.models[lane], lanes.vocoders[lane], lanes.streams[lane] or caller

    def vocode(v, out):
        # to_waveform (feel_me.py:183).  Ragged: item b is vocoded up to mel_lengths[b] (+ receptive field) only
        return v(out["mel"], lengths=out["mel_lengths"] if ragged[0] else None).clamp(-1, 1)

    lane_done = [None] * n_lanes
    last_step = [False, None]                                    # [recording, (out, wav) of the last step recorded]

    def step_resident():
        lane, m, v, st = next_lane()
        if lane_done[lane] is not None and n_lanes > 1 and not serial[0]:
            lane_done[lane].synchronize()                        # one step per lane in flight: the host does not run further ahead
        with torch.cuda.stream(st):
            out = m.synthesise(x_dev, xl_dev, N_TIMESTEPS, TEMPERATURE, spk_dev, LENGTH_SCALE)
            wav = vocode(v, out)
            lane_done[lane] = torch.cuda.Event()
            lane_done[lane].record()
        if last_step[0]:
            last_step[1] = (out, wav)
        return out, wav

    host = [dict(wav=None, len=torch.empty(BATCH, dtype=torch.int64).pin_memory(), done=None) for _ in range(n_lanes)]

    def step_e2e():
        lane, m, v, st = next_lane()
        h = host[lane]
        if h["done"] is not None:
            h["done"].synchronize()                              # the host has this lane's previous result before the slot is reused
        with torch.cuda.stream(st):
            xd = x_pin.to(dev, non_blocking=True)
            ld = xl_pin.to(dev, non_blocking=True)
            sd_ = spk_pin.to(dev, non_blocking=True)
            out = m.synthesise(xd, ld, N_TIMESTEPS, TEMPERATURE, sd_, LENGTH_SCALE)
            wav = vocode(v, out)
            if h["wav"] is None or h["wav"].shape != wav.shape:
                h["wav"] = torch.empty(wav.shape, dtype=wav.dtype).pin_memory()
            h["wav"].copy_(wav, non_blocking=True)               # .cpu() of to_waveform (feel_me.py:187)
            h["len"].copy_(out["mel_lengths"], non_blocking=True)
            h["done"] = torch.cuda.Event()
            h["done"].record()
        if n_lanes == 1 or serial[0]:
            h["done"].synchronize()                              # one step at a time: the result is on the host before the next step starts
        return out, wav

    def settle(fn, floor, window, cap_s=15.0, cap_n=60):
        """Run fn until the last `window` per-step wall times agree within 15 % (a freshly booted box stalls the host for
        100s of ms now and then), at least `floor` times."""
        t0, recent = time.perf_counter(), []
        while True:
            t_s = time.perf_counter()
            res = fn()
            torch.cuda.synchronize()
            recent.append(time.perf_counter() - t_s)
            last = recent[-window:]
            if len(recent) >= floor and ((len(last) >= window and max(last) < 1.15 * min(last)) or
                                         time.perf_counter() - t0 > cap_s or len(recent) >= cap_n):
                return res, len(recent)

    def timed(fn, steps):
        """K steps bracketed by barrier + synchronize, CUDA events on the launching stream -> ms (this rank).  The lanes'
        streams fork from the start event and join before the end event, so the events span every step's last kernel."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for st in lanes.streams:
            if st is not None:
                st.wait_event(e0)
        for _ in range(steps):
            fn()
        for st in lanes.streams:
            if st is not None:
                caller.wait_stream(st)
        e1.record()
        barrier()
        return e0.elapsed_time(e1)

    # warm-up: W steps at least (graphs are captured on the second sight of a shape), then until the step time has settled
    (out, wav), n_warm = settle(step_resident, max(n_warm_min, 2 * n_lanes + 2), 6)     # every lane captures its graphs on its second step
    secs_per_step = audio_seconds(out["mel_lengths"].cpu())
    frames = int(out["mel_lengths"].sum())
    t_pad = int(out["t_pad"])
    ws_bytes = (_lib_mod.lib().ev_vocode_workspace_bytes(voc._ctx.handle, BATCH, int(out["mel"].shape[2])) +
                _lib_mod.lib().ev_decode_workspace_bytes(model._ctx.handle, BATCH, t_pad, N_TIMESTEPS))

    if args.profile_one_step:
        serial[0] = True
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step_resident()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        print(json.dumps({"profiled_step": True, "t_pad": t_pad, "frames": frames}))
        return

    # ---------------- timed region: K steps, inputs resident in HBM
    # every step draws its prior noise from the device's generator; the warm-up above runs until the step time settles, so
    # the generator is seeded here, a fixed number of steps before the last timed one
    torch.cuda.manual_seed(0)
    sampler = ClockSampler(local_rank)
    sampler.start()
    def count_launches(reset=False):
        return sum(m.launch_count(reset) + v.launch_count(reset) for m, v in zip(lanes.models, lanes.vocoders))

    if n_lanes > 1:
        timed(step_resident, 2 * n_lanes)                        # untimed: brings the lanes into their steady overlap
    count_launches(reset=True)
    last_step[0] = bool(args.dump_outputs) and rank == 0
    ms = timed(step_resident, args.steps)
    launches = count_launches()
    clocks = sampler.stop()
    if last_step[0]:
        out_last, wav_last = last_step[1]
        dump_outputs(args.dump_outputs, {**{k: out_last[k] for k in DUMPED}, "waveform": wav_last})
        last_step[:] = [False, None]
        del out_last, wav_last
    # one step at a time (every step on lane 0): the loop rounds 1 and 2 reported until in-flight lanes existed
    ms_serial = None
    if n_lanes > 1:
        serial[0] = True
        timed(step_resident, 3)
        ms_serial = timed(step_resident, args.steps)
        serial[0] = False

    # ---------------- e2e: same steps through the public API with pinned host inputs and the waveform read back
    settle(step_e2e, 2 * n_lanes + 2, 4, cap_n=40)
    ms_e2e = timed(step_e2e, args.steps)
    ms_e2e_serial = None
    if n_lanes > 1:
        serial[0] = True
        timed(step_e2e, 3)
        ms_e2e_serial = timed(step_e2e, args.steps)
        serial[0] = False

    # ---------------- the same with the padded frames vocoded too: the reference's literal work list (vocoder(mel), no kwarg)
    ms_dense = ms_e2e_dense = None
    if ragged[0]:
        ragged[0] = False
        settle(step_resident, 2 * n_lanes + 1, 3, cap_n=20)
        ms_dense = timed(step_resident, args.steps)
        settle(step_e2e, 2 * n_lanes + 1, 3, cap_n=20)
        ms_e2e_dense = timed(step_e2e, args.steps)
        ragged[0] = True

    red = reduce([ms, ms_e2e, ms_dense or 0.0, ms_e2e_dense or 0.0, ms_serial or 0.0, ms_e2e_serial or 0.0], MAX)        # the slowest rank bounds the job
    ms, ms_e2e = red[0], red[1]
    ms_dense, ms_e2e_dense = (red[2], red[3]) if ms_dense is not None else (None, None)
    ms_serial, ms_e2e_serial = (red[4], red[5]) if ms_serial is not None else (None, None)
    total_secs, launches = reduce([secs_per_step, float(launches)], SUM)
    launches = int(launches)
    per_s = lambda t_ms: total_secs * args.steps / (t_ms / 1e3)
    value, value_e2e = per_s(ms), per_s(ms_e2e)
    h2d = x.numel() * 8 + xl.numel() * 8 + spks.numel() * 8
    d2h = int(wav.numel()) * 4 + BATCH * 8
    peaks = load_peaks()

    # ---------------- denoiser (hifigan/denoiser.py:59-64; every app calls it after the vocoder, feel_me.py:183-185)
    denoiser_block = None
    if not args.no_extras:
        den = ev.Denoiser(voc, mode="zeros")
        wav_d = voc(out["mel"]).clamp(-1, 1).squeeze(1)          # the denoiser needs the dense waveform (STFT windows reach into the padding)
        for _ in range(3):
            den(wav_d, strength=0.00025)
        ms_den = reduce([timed(lambda: den(wav_d, strength=0.00025), args.steps)], MAX)[0] / args.steps
        den_bytes = 8.0 * wav_d.numel()                          # algorithmic: read the waveform once, write it once
        denoiser_block = {"ms_per_step": round(ms_den, 3), "samples": int(wav_d.numel()), "algorithmic_bytes": int(den_bytes),
                          "gbs": round(den_bytes / (ms_den / 1e3) / 1e9, 1), "frac_of_hbm_peak": round(den_bytes / (ms_den / 1e3) / 1e9 / peaks["hbm_gbs"], 4),
                          "share_of_step": round(ms_den / (ms_dense / args.steps + ms_den), 4) if ms_dense else None,
                          "what": "Denoiser(vocoder)(audio, 0.00025) on the batch's dense waveform: STFT (1024/256 hann) -> magnitude - bias*strength -> ISTFT"}
        del wav_d

    # ---------------- roofline: one more step with CUDA events around every launch
    model.cuda_graphs = voc.cuda_graphs = False                  # per-launch events need eager launches, not a graph replay
    serial[0] = True                                             # lane 0 = `model` / `voc`, alone on the GPU
    model._ctx.profile_begin(); voc._ctx.profile_begin()
    step_resident()
    torch.cuda.synchronize()
    stats = model._ctx.profile_end() + voc._ctx.profile_end()
    model.cuda_graphs = voc.cuda_graphs = True
    serial[0] = False
    agg = {}
    for s in stats:
        a = agg.setdefault(s["name"], dict(name=s["name"], launches=0, total_ms=0.0, flops=0.0, bytes=0.0))
        for k in ("launches", "total_ms", "flops", "bytes"):
            a[k] += s[k]
    klist = sorted(agg.values(), key=lambda a: -a["total_ms"])
    ksum = sum(a["total_ms"] for a in klist) or 1.0
    table = []
    for a in klist[:12]:
        sec = a["total_ms"] / 1e3
        table.append({"name": a["name"], "launches": a["launches"], "ms": round(a["total_ms"], 3),
                      "share": round(a["total_ms"] / ksum, 4), "tflops": round(a["flops"] / sec / 1e12, 2) if sec else 0,
                      "gbs": round(a["bytes"] / sec / 1e9, 1) if sec else 0})
    # one roofline per kernel CLASS = (__global__ function, stage): the decoder's and the vocoder's launches of the same conv
    # function are different populations (small latency-bound tiles vs long MMA-bound ones) and are reported separately;
    # `roofline` is the class with the largest share of the step
    rooflines = [roofline_of(a, peaks, ksum) for a in klist if a["total_ms"] / ksum >= 0.02]
    how = ("CUDA events around every launch on the launching stream, one instrumented (eager) step right after the timed region; "
           "algorithmic FLOPs/bytes (valid un-padded work)")
    for r in rooflines:
        tr, tr_fn = measured_traffic(r["kernel"])
        if tr is not None:
            r["traffic"] = round(tr)
            r["traffic_source"] = ("dram__bytes_read.sum + dram__bytes_write.sum per launch of %s, averaged over its launches in one bench step "
                                   "(profiles/%s, ncu --clock-control none)" % (tr_fn, TRAFFIC_FILE[0]))
    roofline = dict(rooflines[0], peak_source=peaks["source"], how=how)
    # whole-path algorithmic FLOPs (SURVEY.md 8d) as a fraction of the tensor roofline
    tx = xl.double()
    flops_step = float((tx * (19309056 + 6144 * tx)).sum()) + 0.0
    ml = out["mel_lengths"].double().cpu()
    flops_step += float((N_TIMESTEPS * ml * (11116544 + 1536 * ml)).sum()) + float((ml * 614105088).sum())
    path_tflops = flops_step * args.steps / (ms / 1e3) / 1e12 * world

    # ---------------- BASELINE configs[2]: 1024 mixed-length utterances, sharded over the ranks (strong scaling)
    config3 = config5 = None
    if not args.no_extras:
        utts = synthetic.mixed_length_corpus(1024)
        passes = []
        for rep in range(4):
            barrier()
            t0 = time.perf_counter()
            res, st = ev.synthesise_corpus(model, voc, utts, batch_size=32, n_timesteps=N_TIMESTEPS, temperature=TEMPERATURE,
                                           length_scale=LENGTH_SCALE, rank=rank, world_size=world, lanes=lanes)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            wall_max, dev_max = reduce([wall, st.seconds], MAX)
            secs3, n3 = reduce([st.audio_seconds, float(len(res))], SUM)
            passes.append({"pass": rep, "wall_s": round(wall_max, 3), "audio_s_per_s_wall": round(secs3 / wall_max, 1),
                           "audio_s_per_s_device": round(secs3 / dev_max, 1)})
            del res
        config3 = {"workload": "BASELINE.json configs[2]: 1024 mixed-length utterances (P~U[20,150]), 11 emoji voices, micro-batches of 32 "
                               "sorted by length, dealt to the ranks by estimated FLOPs (sharding.shard), synthesise_corpus: "
                               "collate -> synthesise -> ragged vocoder -> pinned D2H on a copy stream -> per-utterance crop, "
                               "%d micro-batches in flight per GPU" % n_lanes,
                   "scaling": "strong", "utterances": int(n3), "audio_seconds": round(secs3, 1), "n_gpus": world,
                   "timing": "host wall clock around the whole call incl. D2H + crop, max over ranks (pass 0 = shapes never seen before)",
                   "passes": passes, "value_first_pass": passes[0]["audio_s_per_s_wall"], "value_warm": passes[-1]["audio_s_per_s_wall"]}
        # ---------------- BASELINE configs[4]: vocoder only, 60-second segments (T = 5168 frames), 4 segments per GPU
        T5 = int(round(60 * SR / HOP))
        mel5 = synthetic.synthetic_mel(4, T5, seed=5).to(dev)
        for _ in range(3):
            voc(mel5)
        ms5 = reduce([timed(lambda: voc(mel5), 10)], MAX)[0] / 10
        secs5 = 4 * T5 * HOP / SR
        config5 = {"workload": "BASELINE.json configs[4]: HiFi-GAN only, synthetic 80-bin mel, 4 x 60-s segments per GPU (T = 5168)",
                   "scaling": "weak", "n_gpus": world, "ms_per_step": round(ms5, 3), "value": round(world * secs5 / (ms5 / 1e3), 1),
                   "unit": "audio-s/s", "tflops_per_gpu": round(4 * T5 * 614105088 / (ms5 / 1e3) / 1e12, 1)}
        del mel5

    result = {
        "metric": "audio_seconds_per_second", "value": round(value, 2), "unit": "audio-s/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": args.precision if args.precision != "fp32" else "f32",
        "data": "synthetic",
        "config": workload_config(),
        "details": dict(audio_seconds_per_step_per_gpu=round(secs_per_step, 2), mel_frames_per_step_per_gpu=frames, t_pad=t_pad,
                        warmup_steps_run=n_warm, per_rank_batch="identical on every rank (seed 2000)",
                        steps_in_flight=("%d batches in flight per GPU (step i on lane i %% %d: own model / vocoder instance + stream, ev.Lanes; a lane "
                                         "takes its next step when its previous one is done); `one_step_at_a_time` is the same loop with a step "
                                         "starting only when the previous one has finished" % (n_lanes, n_lanes)) if n_lanes > 1 else "one step at a time",
                        l2="no flush: each step streams a %.1f GB activation workspace (>> 126 MB L2); weights "
                        "(35 MB bf16) stay L2-resident as they would in service" % (ws_bytes / 1e9),
                        launch="encoder, alignment + decoder and vocoder replayed as CUDA graphs (captured during warm-up, per lane)",
                        vocoder=("ragged: time tiles past each utterance's own length (+ the receptive field behind each layer: 13 frames at conv_pre ... 2 at the last stage) are "
                                 "not computed; waveform bit-identical to the dense generator on [: mel_length*256] and zero beyond "
                                 "-- the part the reference's batched caller crops away (cli.py:307-311); `padded_vocoder` is the "
                                 "same run with the padded frames vocoded too") if not args.dense_vocoder else "dense (padded frames vocoded too)"),
        "rtf": round(1.0 / value, 8), "x_realtime": round(value, 1),
        "clocks": clocks,
        "e2e": {"value": round(value_e2e, 2), "unit": "audio-s/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": round(ms_e2e / args.steps, 3)},
        "gpu_launches": int(launches),
        "in_flight": n_lanes,
        "one_step_at_a_time": ({"value": round(per_s(ms_serial), 2), "unit": "audio-s/s", "ms_per_step": round(ms_serial / args.steps, 3),
                                "e2e": {"value": round(per_s(ms_e2e_serial), 2), "unit": "audio-s/s", "ms_per_step": round(ms_e2e_serial / args.steps, 3)},
                                "what": "the same K steps issued one after another on one stream (a step starts when the previous one has "
                                        "finished; e2e: host sync per step) -- the loop every earlier bench line of this repo reports"}
                               if ms_serial else None),
        "padded_vocoder": ({"value": round(per_s(ms_dense), 2), "unit": "audio-s/s", "ms_per_step": round(ms_dense / args.steps, 3),
                            "e2e": {"value": round(per_s(ms_e2e_dense), 2), "unit": "audio-s/s", "h2d_bytes_per_step": h2d,
                                    "d2h_bytes_per_step": d2h, "ms_per_step": round(ms_e2e_dense / args.steps, 3)},
                            "what": "vocoder(mel) without the `lengths` kwarg: the reference's literal work list (padded frames vocoded, cropped afterwards)"}
                           if ms_dense else None),
        "roofline": roofline, "rooflines": rooflines,
        "path_tflops": round(path_tflops, 2), "path_frac_of_tensor_peak": round(path_tflops / (peaks["tflops"] * world), 4),
        "kernels": table, "denoiser": denoiser_block, "config3": config3, "config5": config5,
    }
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        arm = CpuArm()
        arm.once(x, xl, spks, CPU_SAMPLE)
        best = None
        for _ in range(3):
            a, dt = arm.once(x, xl, spks, CPU_SAMPLE)
            best = (a, dt) if best is None or dt < best[1] else best
        result["cpu_baseline"] = {"value": round(best[0] / best[1], 3), "unit": "audio-s/s", "cores": arm.cores, "kind": arm.kind,
                                  "sample": f"first {CPU_SAMPLE} utterances of the batch ({best[0]:.1f} audio-s), fp32 torch CPU, "
                                  f"{arm.kind} ({arm.src}), warm-up 1, best of 3, {os.cpu_count()} host cpus"}
    elif rank == 0:
        result["cpu_baseline"] = None
    if rank == 0:
        print(json.dumps(result))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
