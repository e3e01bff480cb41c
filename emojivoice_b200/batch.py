"""Batched corpus synthesis: the caller side of the hot path as `matcha/cli.py:264-317` (batched_synthesis) does it --
collate (pad) -> MatchaTTS.synthesise -> to_waveform -> per-utterance crop `[: length * 256]` -- over the micro-batch
plan of `sharding.py`, so the same call runs one GPU's shard or the whole list."""
from __future__ import annotations

import torch

from . import sharding


SETTINGS = ("length_scale", "temperature", "n_timesteps")
VOCODER_SETTINGS = ("denoiser_strength",)      # per utterance too, but read after synthesis: the plan does not depend on them
NOISE_SETTINGS = ("seed",)                     # the prior noise's seed: the plan does not depend on it either


def collate(utterances, items):
    """cli.py:109-120 batched_collate_fn: right-pad the id sequences with 0.  utterances[i] = (ids, speaker_id[, settings])."""
    seqs = [torch.as_tensor(utterances[i][0], dtype=torch.long).reshape(-1) for i in items]
    x = torch.nn.utils.rnn.pad_sequence(seqs, batch_first=True)
    x_lengths = torch.tensor([s.numel() for s in seqs], dtype=torch.long)
    spks = torch.tensor([int(utterances[i][1]) for i in items], dtype=torch.long)
    return x, x_lengths, spks


class Lanes:
    """`n` (model, vocoder) instances on one device, one CUDA stream each: `synthesise_corpus` deals micro-batch k to lane k % n,
    so n batches are in flight at once.  A batch is a chain of ~70 dependent launches, many of them latency-bound or on
    partial waves (the decoder runs one tile per CTA on 75-148 SMs); the other lanes' kernels fill those gaps: 7.5 k ->
    8.2 k (n = 2) -> 8.6 k (n = 3) audio-s/s on the config-2 batch (profiles/r02_batches_in_flight.txt).  Every lane owns its
    context (packed weights, workspace, graph cache), the arithmetic is the same kernels on the same inputs, so results do
    not depend on n.  Lane 0 is the caller's own pair."""

    def __init__(self, model, vocoder, n: int):
        if n < 1:
            raise ValueError("in_flight must be >= 1")
        self.models = [model] + [model.replica() for _ in range(n - 1)]
        self.vocoders = [vocoder] + [vocoder.replica() for _ in range(n - 1)]
        self.streams = [torch.cuda.Stream(device=model.device) for _ in range(n)] if n > 1 else [None]
        self.denoisers = {}

    def __len__(self):
        return len(self.models)

    def denoiser(self, lane: int, denoiser):
        """The caller's denoiser belongs to lane 0's vocoder context; the other lanes get their own (same bias spectrum)."""
        if denoiser is None or lane == 0:
            return denoiser
        if lane not in self.denoisers:
            self.denoisers[lane] = type(denoiser)(self.vocoders[lane])
        return self.denoisers[lane]


def lanes_for(model, vocoder, n: int) -> Lanes:
    """The (cached) lanes of a model / vocoder pair: replicas are built once per (vocoder, n) and kept on the model."""
    cache = model.__dict__.setdefault("_lanes", [])
    for lanes in cache:
        if lanes.vocoders[0] is vocoder and len(lanes) == int(n):
            return lanes
    cache.append(Lanes(model, vocoder, int(n)))
    return cache[-1]


def utterance_settings(utterances, defaults):
    """Each utterance's settings (SETTINGS, VOCODER_SETTINGS and NOISE_SETTINGS): an utterance is (ids, speaker_id) or (ids,
    speaker_id, settings) with a dict holding any of those keys; a missing key takes its value from `defaults`.
    -> (per-utterance dicts, True when some utterance has its own synthesis settings (SETTINGS))"""
    out, own = [], False
    for u in utterances:
        s = dict(defaults)
        if len(u) > 2 and u[2]:
            known = SETTINGS + VOCODER_SETTINGS + NOISE_SETTINGS
            extra = set(u[2]) - set(known)
            if extra:
                raise ValueError(f"unknown per-utterance settings {sorted(extra)}; expected keys among {known}")
            s.update(u[2])
            own = own or any(k in SETTINGS for k in u[2])
        out.append(s)
    return out, own


def denoiser_strengths(settings, denoiser):
    """Each utterance's denoiser strength from its settings, None = not denoised; refuses a strength without a denoiser."""
    from .hifigan import per_item_strength

    dn = [s["denoiser_strength"] for s in settings]
    if denoiser is None and any(v is not None for v in dn):
        raise ValueError("a per-utterance denoiser_strength needs a denoiser: pass denoiser=Denoiser(vocoder)")
    per_item_strength(dn, len(dn))          # the host-side checks, before any work is done
    return dn


def splitmix64(seed, n):
    """The first n outputs of splitmix64 seeded with `seed` mod 2^64 (Steele, Lea and Flood 2014).  Utterance i of a corpus
    seeded with S draws its noise from output i: consecutive seeds S + i would give corpora S and S + 1 all but one noise in
    common, while these streams share none."""
    m = (1 << 64) - 1
    x, out = seed & m, []
    for _ in range(n):
        x = (x + 0x9E3779B97F4A7C15) & m
        v = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & m
        v = ((v ^ (v >> 27)) * 0x94D049BB133111EB) & m
        out.append(v ^ (v >> 31))
    return out


def utterance_seeds(settings, seed, z_fn=None):
    """Each utterance's noise seed (a uint64), or None when the corpus is not seeded.  Utterance i takes its settings' "seed",
    else output i of splitmix64(seed) when `seed` is given.  Refuses, before any work is done, a corpus in which some utterances
    are seeded and others are not, and seeds together with z_fn (which supplies the noise itself)."""
    from .matcha import seed_value

    derived = splitmix64(seed_value(seed), len(settings)) if seed is not None else None
    seeds = []
    for i, s in enumerate(settings):
        v = s.get("seed", derived[i] if derived is not None else None)
        seeds.append(None if v is None else seed_value(v, f"utterance {i}"))
    if all(v is None for v in seeds):
        return None
    if any(v is None for v in seeds):
        raise ValueError("some utterances have a noise seed and others do not: pass seed= or give every utterance a \"seed\"")
    if z_fn is not None:
        raise ValueError("z_fn supplies the prior noise itself: it cannot be combined with noise seeds")
    return seeds


@torch.inference_mode()
def synthesise_corpus(model, vocoder, utterances, batch_size=32, n_timesteps=10, temperature=0.667, length_scale=1.0,
                      rank=0, world_size=1, denoiser=None, denoiser_strength=0.00025, sort=True, keep_mel=False, z_fn=None,
                      ragged=True, cuda_graphs=False, in_flight=1, lanes=None, seed=None):
    """Synthesise this rank's share of `utterances`: a list of (phoneme ids, speaker id) or (phoneme ids, speaker id, settings),
    where settings is a dict with any of "length_scale", "temperature", "n_timesteps" for that utterance (a missing key takes
    the keyword's value).  Utterances with different settings share micro-batches (MatchaTTS.synthesise with per-utterance
    values); the micro-batch plan does not depend on them, only its cost estimate uses each utterance's own step count.
    settings may also hold "denoiser_strength": a number, or None for an utterance that is not denoised; a missing key takes
    `denoiser_strength`, or None when `denoiser` is None (a strength without a denoiser is a ValueError).  The vocoder stage of
    a micro-batch then denoises each utterance with its own strength (Generator.vocode_denoised, Denoiser with per-item
    strengths), so an utterance's mel and waveform do not depend on what the other utterances asked of the denoiser.

    -> (results, stats): results maps utterance index -> dict(waveform (L,) cpu float32, mel_length, [mel]), stats is a
    sharding.ShardStats with this rank's device time.  `z_fn(mb, model, x, x_lengths, spks)` may supply the prior noise per
    micro-batch (parity runs share it with the oracle).  ragged: the vocoder skips the time tiles past each utterance's own length
    (identical cropped waveforms, see Generator.__call__); with a denoiser, vocoder and denoiser run as one ragged call that
    vocodes 4 frames past each end, which the denoiser's STFT windows reach, and transforms only each utterance's own frames
    (identical cropped waveforms, see Generator.vocode_denoised; a denoiser built on another generator than `vocoder` runs
    the dense path).  ragged=False vocodes and denoises the whole padded batch.  cuda_graphs: a corpus hardly ever repeats a (B, Tx, T_pad) shape, so by default the
    stages are launched eagerly -- measured within 2 % of a graph replay (the host enqueues a step in 5 ms of the GPU's 29),
    whereas capturing costs ~250 ms per new shape (profiles/r02_host_cost.txt); True restores capture-on-second-sight.
    in_flight / lanes: micro-batches in flight at once (see `Lanes`; `lanes` passes a prebuilt set, else `lanes_for` builds and
    caches one); the waveforms do not depend on it.  stats.seconds is the sum of the micro-batches' device times for one
    lane and the device span from the first launch to the last kernel's end for several.

    seed: utterance i (its index in `utterances`) draws its prior noise on the GPU from output i of splitmix64(seed)
    (MatchaTTS.synthesise(seed=...)); a "seed" in its settings overrides that value and does not change the plan.  The noise,
    and so every waveform, is then the same for any rank / world_size split, in_flight, cuda_graphs and RNG history; without a
    seed the noise comes from torch.randn as before.  The mel depends on the micro-batch (the decoder is not padding-invariant),
    which the plan fixes independently of world_size.  Some utterances seeded and others not, or seeds with z_fn, are a
    ValueError."""
    lens = [len(u[0]) for u in utterances]
    settings, own = utterance_settings(utterances, dict(length_scale=length_scale, temperature=temperature, n_timesteps=n_timesteps,
                                                        denoiser_strength=denoiser_strength if denoiser is not None else None))
    strengths = denoiser_strengths(settings, denoiser)
    seeds = utterance_seeds(settings, seed, z_fn)
    steps = [int(s["n_timesteps"]) for s in settings] if own else n_timesteps
    plan = sharding.shard(lens, batch_size, rank, world_size, n_timesteps=steps, sort=sort)
    results, stats = {}, sharding.ShardStats()
    if lanes is None:
        lanes = lanes_for(model, vocoder, in_flight)
    n_lanes = len(lanes)
    dev = model.device
    copy_stream = torch.cuda.Stream(device=dev)
    pinned = {}                      # n_lanes + 1 pinned staging buffers (grown on demand), used in turn
    pending = []                     # the micro-batches in flight: their read-back and crops overlap the later ones' GPU work
    span = []                        # (first start event, end events) for the several-lane device time

    def finish(p):
        p["done"].synchronize()
        mel_len = p["len_host"].tolist()
        stats.add(mel_len, p["xl"], [steps[i] for i in p["items"]] if own else n_timesteps,
                  p["e0"].elapsed_time(p["e1"]) / 1e3 if n_lanes == 1 else 0.0)
        for j, i in enumerate(p["items"]):
            n = int(mel_len[j])
            rec = {"waveform": p["wav_host"][j, 0, : n * 256].clone(), "mel_length": n}     # cli.py:308-309 crop
            if keep_mel:
                rec["mel"] = p["mel"][j, :, :n].cpu()
            results[i] = rec

    saved_graphs = [(m.cuda_graphs, v.cuda_graphs) for m, v in zip(lanes.models, lanes.vocoders)]

    def restore_graphs():
        for (mg, vg), m, v in zip(saved_graphs, lanes.models, lanes.vocoders):
            m.cuda_graphs, v.cuda_graphs = mg, vg

    if not cuda_graphs:
        for m, v in zip(lanes.models, lanes.vocoders):
            m.cuda_graphs = v.cuda_graphs = False
    try:
        caller = torch.cuda.current_stream(dev)
        for st in lanes.streams:
            if st is not None:
                st.wait_stream(caller)
        # largest micro-batch first: the workspace and the caching allocator's blocks are sized once, every later batch fits
        plan = sorted(plan, key=lambda m: -m.cost)
        for k, mb in enumerate(plan):
            lane = k % n_lanes
            m, v, st = lanes.models[lane], lanes.vocoders[lane], lanes.streams[lane] or caller
            x, xl, spks = collate(utterances, mb.items)
            with torch.cuda.stream(st):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                kw = {}
                if z_fn is not None:
                    kw["z"] = z_fn(mb, m, x, xl, spks)
                if seeds is not None:
                    kw["seed"] = [seeds[i] for i in mb.items]
                if own:      # one value per utterance of the micro-batch
                    n_b, temp_b, ls_b = ([settings[i][k] for i in mb.items] for k in ("n_timesteps", "temperature", "length_scale"))
                else:
                    n_b, temp_b, ls_b = n_timesteps, temperature, length_scale
                out = m.synthesise(x, xl, n_b, temp_b, spks if m.n_spks > 1 else None, ls_b, **kw)
                d = lanes.denoiser(lane, denoiser)
                dn = [strengths[i] for i in mb.items]        # equal values are the scalar call (per_item_strength)
                if ragged and d is not None and d.vocoder is v:
                    wav = v.vocode_denoised(out["mel"], out["mel_lengths"], dn)
                else:
                    wav = v(out["mel"], lengths=out["mel_lengths"] if ragged and d is None else None).clamp(-1, 1)   # to_waveform, cli.py:121-126
                    if d is not None:
                        wav = d(wav.squeeze(1), strength=dn).unsqueeze(1)
                e1.record()
                # read-back on a copy stream into pinned memory (the `.cpu()` of to_waveform): the host crops an EARLIER micro-batch
                # while this one's copy -- and the next ones' kernels -- are in flight
                slot = pinned.setdefault(k % (n_lanes + 1), {})
                if "wav" not in slot or slot["wav"].numel() < wav.numel():
                    slot["wav"] = torch.empty(wav.numel(), dtype=wav.dtype).pin_memory()
                if "len" not in slot or slot["len"].numel() < len(mb.items):
                    slot["len"] = torch.empty(len(mb.items), dtype=torch.int64).pin_memory()
                wav_host = slot["wav"][: wav.numel()].view(wav.shape)
                len_host = slot["len"][: len(mb.items)]
                copy_stream.wait_stream(st)
                with torch.cuda.stream(copy_stream):
                    wav_host.copy_(wav, non_blocking=True)
                    len_host.copy_(out["mel_lengths"], non_blocking=True)
                    done = torch.cuda.Event()
                    done.record()
                wav.record_stream(copy_stream)                        # both sources are read by the copy stream after this iteration
                out["mel_lengths"].record_stream(copy_stream)         # rebinds `out`: the allocator must not recycle them early
            if not span:
                span.append(e0)
            span.append(e1)
            pending.append(dict(done=done, e0=e0, e1=e1, wav_host=wav_host, len_host=len_host, xl=xl.tolist(), items=mb.items,
                                mel=out["mel"] if keep_mel else None))
            if len(pending) > n_lanes:
                finish(pending.pop(0))
        while pending:
            finish(pending.pop(0))
        for st in lanes.streams:
            if st is not None:
                caller.wait_stream(st)
        if n_lanes > 1 and len(span) > 1:
            for e in span[1:]:
                e.synchronize()
            stats.seconds += max(span[0].elapsed_time(e) for e in span[1:]) / 1e3
        stats.extra["in_flight"] = n_lanes
    finally:
        restore_graphs()
    return results, stats


def synthesise_file(model, vocoder, script, out_dir, *, phonemizer=None, cleaner="english_cleaners2", spk=None, emoji_mapping=None,
                    default_spk: int = 12, batch_size: int = 32, n_timesteps: int = 10, temperature: float = 0.667,
                    length_scale: float = 1.0, denoiser=None, denoiser_strength: float = 0.00025, rank: int = 0,
                    world_size: int = 1, in_flight: int = 1, seed=None):
    """One call from a script file to audio on disk: the reference's batched file path composed end to end
    (`matcha/cli.py:226-250` get_texts / `:277-317` batched_synthesis / `:129-135` save_to_folder).

    script : path of a text file or an iterable of lines.  Three line formats, decided per line:
               `text|speaker_id`   (cli.py:326-330)            -> that speaker
               text with an emoji  (feel_me.py:298-312)         -> the emoji's voice from `emoji_mapping`, emoji stripped
               plain text                                       -> `spk` if given, else `default_spk`
    phonemizer : callable text -> phoneme string standing for espeak-ng (absent offline); the rule-based half of the cleaner
                 (`text_cleaners`) runs in front of it.  None: the line must already be a phoneme string of the symbol table.
    Writes `<out_dir>/utterance_{i:03d}_speaker_{spk:03d}.wav` (PCM_24, 22.05 kHz) + `.npy` (mel), i = line index, for the
    lines this rank owns (`sharding.shard`); `in_flight` micro-batches at once (see `Lanes`).  seed: as synthesise_corpus, with
    i the utterance's index among the script's non-empty lines, so every rank split writes the same files.
    -> (list of (index, wav_path, mel_length), ShardStats)"""
    from . import audio_io, text_cleaners, text_frontend
    from .emoji_frontend import emoji_to_spk
    from .config import EMOJI_MAPPING_FEMALE

    if isinstance(script, (str, bytes)) or hasattr(script, "__fspath__"):
        with open(script, "r", encoding="utf-8") as f:
            lines = f.read().splitlines()
    else:
        lines = list(script)
    mapping = EMOJI_MAPPING_FEMALE if emoji_mapping is None else emoji_mapping
    utterances, speakers = [], []
    for ln in (l.strip() for l in lines):
        if not ln:
            continue
        head, bar, tail = ln.rpartition("|")
        if bar and head and tail.strip().lstrip("-").isdigit():
            text, speaker = head.strip(), int(tail)
        else:
            text, speaker = emoji_to_spk(ln, mapping, default_spk if spk is None else int(spk))
        g2p = (lambda t, _c=cleaner: text_cleaners.clean_text(t, [_c], phonemizer)) if phonemizer is not None else None
        rec = text_frontend.process_text(text, g2p)
        utterances.append((rec["x"][0].tolist(), speaker))
        speakers.append(speaker)
    results, stats = synthesise_corpus(model, vocoder, utterances, batch_size=batch_size, n_timesteps=n_timesteps, temperature=temperature,
                                       length_scale=length_scale, rank=rank, world_size=world_size, denoiser=denoiser,
                                       denoiser_strength=denoiser_strength, keep_mel=True, in_flight=in_flight, seed=seed)
    written = []
    for i in sorted(results):
        name = f"utterance_{i:03d}_speaker_{speakers[i]:03d}"
        path = audio_io.save_to_folder(name, {"mel": results[i]["mel"], "waveform": results[i]["waveform"]}, out_dir)
        written.append((i, path, results[i]["mel_length"]))
    return written, stats
