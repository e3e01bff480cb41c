"""Drop-in for the reference vocoder objects: `Generator(h)` (hifigan/models.py:148-206) and `Denoiser`
(hifigan/denoiser.py), plus `to_waveform` (feel_me.py:181-187 / cli.py:121-126)."""
from __future__ import annotations

import ctypes as C
import numbers

import torch

from . import _lib
from .config import HIFIGAN_V1


class Generator:
    def __init__(self, h=None, device=None, precision="bf16", cuda_graphs=True):
        self.h = dict(h) if h is not None else dict(HIFIGAN_V1)
        if str(self.h.get("resblock", "1")) != "1":
            raise ValueError("only ResBlock1 (config v1) is implemented")
        self.num_kernels = len(self.h["resblock_kernel_sizes"])
        self.num_upsamples = len(self.h["upsample_rates"])
        self.precision = precision
        self._device = torch.device(device) if device is not None else None
        self._sd = None
        self._ctx = None
        self.cuda_graphs = cuda_graphs            # replay the generator as a CUDA graph once a (B, T) shape repeats
        self._graphs = _lib.GraphCache()
        self._replayed_launches = 0
        self.hop = 1
        for u in self.h["upsample_rates"]:
            self.hop *= int(u)

    def to(self, device):
        self._device = torch.device(device)
        return self

    def cuda(self, device=None):
        return self.to(torch.device("cuda", torch.cuda.current_device() if device is None else device))

    def eval(self):
        return self

    def parameters(self):
        return iter((self._sd or {}).values())

    @property
    def device(self):
        return self._ctx.device if self._ctx is not None else self._device

    def load_state_dict(self, state_dict, strict=True):
        """Accepts plain `weight` keys or the checkpoint's weight-norm form (`weight_g`/`weight_v`,
        feel_me.py:161-167); the library folds the latter as `remove_weight_norm()` would."""
        self._sd = {k: v for k, v in state_dict.items()}
        return self

    def remove_weight_norm(self):
        self._materialise()

    def replica(self):
        """Another generator on the same device with its own context (weights, workspace, graph cache): see MatchaTTS.replica."""
        if self._sd is None:
            raise RuntimeError("load_state_dict() first")
        g = Generator(self.h, device=self.device, precision=self.precision, cuda_graphs=self.cuda_graphs)
        g.load_state_dict(self._sd)
        g._materialise()
        return g

    def _materialise(self):
        if self._ctx is not None:
            return
        if self._sd is None:
            raise RuntimeError("load_state_dict() first")
        self._ctx = _lib.Context(self._device)
        h = self.h
        cfg = _lib.EvHifiganCfg()
        cfg.num_mels = int(h.get("num_mels", 80))
        cfg.upsample_initial_channel = int(h["upsample_initial_channel"])
        cfg.n_ups, cfg.n_kernels = self.num_upsamples, self.num_kernels
        for i, (u, k) in enumerate(zip(h["upsample_rates"], h["upsample_kernel_sizes"])):
            cfg.upsample_rates[i], cfg.upsample_kernel_sizes[i] = int(u), int(k)
        for j, (k, dil) in enumerate(zip(h["resblock_kernel_sizes"], h["resblock_dilation_sizes"])):
            cfg.resblock_kernel_sizes[j] = int(k)
            if len(dil) != 3:
                raise ValueError("ResBlock1 needs three dilations per kernel size")
            for l in range(3):
                cfg.resblock_dilation_sizes[j][l] = int(dil[l])
        arr, keep = _lib.tensor_list(self._sd, self._ctx.device)
        with torch.cuda.device(self._ctx.device):
            rc = _lib.lib().ev_load_hifigan(self._ctx.handle, arr, len(keep), C.byref(cfg), _lib.stream_ptr())
        self._ctx.check(rc, "ev_load_hifigan")

    @torch.inference_mode()
    def __call__(self, mel, dtype=None, lengths=None):
        """mel (B, num_mels, T) -> wav (B, 1, T*hop); tanh output already clamped to [-1, 1].

        lengths (B,) int, optional: valid mel frames per item (the `mel_lengths` of synthesise) of a padded batch.  The
        waveform of item b is then bit-identical on [: lengths[b]*hop] -- all the reference's batched caller keeps
        (cli.py:307-311) -- and zero beyond; time tiles further than the generator's receptive field past an utterance's
        end are never computed (ev_vocode_ragged)."""
        return self._run(mel, dtype, lengths, None)

    forward = __call__

    @torch.inference_mode()
    def vocode_denoised(self, mel, lengths, strength=0.00025, dtype=None):
        """The batched reply path in one call: `Denoiser(self)(self(mel).clamp(-1, 1).squeeze(1), strength)` followed by the
        per-utterance crop `[: lengths[b]*hop]` (feel_me.py:181-187, cli.py:300,307-311) -> wav (B, 1, T*hop).

        wav[b] is bit-identical to that dense path on [: lengths[b]*hop] and zero beyond: the generator runs ragged on
        lengths[b] + 4 frames (all the denoised samples read) and the denoiser transforms only the STFT frames of each
        utterance's own samples (ev_to_waveform_ragged).  A Denoiser built on this generator must exist (it holds the bias
        spectrum).  lengths (B,) valid mel frames per item; lengths given on the host must lie in [1, T] (device tensors are
        clamped to [0, T] on the device, as checking them would synchronise).

        strength: a number for the whole batch, or a (B,) sequence / tensor with one per utterance, in which None means "not
        denoised" (see `per_item_strength`).  Utterance b then gets, bit for bit, this call with its own strength, or
        `self(mel, lengths=lengths)[b]` when it is not denoised (ev_to_waveform_items); strength 0 is not the same as None."""
        s = per_item_strength(strength, mel.shape[0] if mel.dim() == 3 else 1)
        if s is None:                     # no utterance is denoised: the ragged generator alone
            check_lengths(lengths, mel.shape[-1])
        return self._run(mel, dtype, lengths, s if s is None or isinstance(s, tuple) else float(s))

    def _run(self, mel, dtype, lengths, strength):
        """ev_vocode_ragged (strength None), ev_to_waveform_ragged (a number) or ev_to_waveform_items (a tuple with None for the
        items not denoised), replayed as a CUDA graph once a call shape repeats."""
        self._materialise()
        ctx, L = self._ctx, _lib.lib()
        dev = ctx.device
        denoise = strength is not None
        items = isinstance(strength, tuple)
        if mel.dim() == 2:
            mel = mel.unsqueeze(0)
        with torch.cuda.device(dev):
            mel = mel.to(device=dev, dtype=torch.float32).contiguous()
            B, _, T = mel.shape
            prec = _lib.PREC[dtype if dtype is not None else self.precision]
            nb = (L.ev_to_waveform_items_workspace_bytes if items else L.ev_to_waveform_ragged_workspace_bytes if denoise
                  else L.ev_vocode_workspace_bytes)(ctx.handle, B, T)
            if denoise:
                check_lengths(lengths, T)
            if lengths is not None:
                lengths = torch.as_tensor(lengths).reshape(-1).to(device=dev, dtype=torch.int64).contiguous()
                if lengths.numel() != B:
                    raise ValueError(f"lengths has {lengths.numel()} entries for a batch of {B}")
            st = strength_tensors(strength, dev) if items else (None, None)

            def call(mel_, wav_, ws_, len_=None, st_=(None, None)):
                if items:
                    ctx.check(L.ev_to_waveform_items(ctx.handle, _lib.ptr(mel_), _lib.ptr(len_), B, T, prec, _lib.ptr(st_[0]), _lib.ptr(st_[1]),
                                                     _lib.ptr(wav_), _lib.ptr(ws_), ws_.numel(), _lib.stream_ptr()), "ev_to_waveform_items")
                    return
                if denoise:
                    ctx.check(L.ev_to_waveform_ragged(ctx.handle, _lib.ptr(mel_), _lib.ptr(len_), B, T, prec, strength, _lib.ptr(wav_),
                                                      _lib.ptr(ws_), ws_.numel(), _lib.stream_ptr()), "ev_to_waveform_ragged")
                    return
                ctx.check(L.ev_vocode_ragged(ctx.handle, _lib.ptr(mel_), _lib.ptr(len_) if len_ is not None else None, B, T, prec,
                                             _lib.ptr(wav_), _lib.ptr(ws_), ws_.numel(), _lib.stream_ptr()), "ev_vocode")

            # per-item strengths and flags are static inputs of the graph: a replay reads the values of its own call
            key = (B, T, prec, lengths is not None) + (("items",) if items else (strength,) if denoise else ())
            ws_shared = ctx.workspace(nb)                   # (may grow the workspace: do it before looking graphs up)
            ent = self._graphs.get(key, ctx.ws_version) if self.cuda_graphs else None
            if ent is None and self.cuda_graphs and self._graphs.should_capture(key):
                ent = dict(mel=mel.clone(), wav=torch.empty(B, 1, T * self.hop, device=dev), ws=ws_shared, ws_version=ctx.ws_version,
                           len=lengths.clone() if lengths is not None else None, st=tuple(t.clone() if t is not None else None for t in st))
                ent["graph"], ent["launches"] = _lib.capture(ctx, lambda: call(ent["mel"], ent["wav"], ent["ws"], ent["len"], ent["st"]))
                self._graphs.put(key, ent)
            if ent is None:
                wav = torch.empty(B, 1, T * self.hop, device=dev)
                call(mel, wav, ws_shared, lengths, st)
            else:
                ent["mel"].copy_(mel)
                if lengths is not None:
                    ent["len"].copy_(lengths)
                if items:
                    for dst, src in zip(ent["st"], st):
                        dst.copy_(src)
                ent["graph"].replay()
                self._replayed_launches += ent["launches"]
                wav = ent["wav"].clone()
        return wav

    def launch_count(self, reset=False):
        """Kernels launched by this generator's context, graph replays included."""
        n = self._ctx.launch_count(reset) + self._replayed_launches
        if reset:
            self._replayed_launches = 0
        return n


def check_lengths(lengths, max_len):
    """Lengths the caller holds on the host must lie in [1, max_len]; a CUDA tensor is not read back (that would synchronise)."""
    if lengths is None:
        raise ValueError("lengths are required")
    if isinstance(lengths, torch.Tensor) and lengths.is_cuda:
        return
    t = torch.as_tensor(lengths).reshape(-1)
    if t.numel() and (int(t.min()) < 1 or int(t.max()) > max_len):
        raise ValueError(f"lengths must lie in [1, {max_len}] frames, got [{int(t.min())}, {int(t.max())}]")


def per_item_strength(value, B):
    """The denoiser setting of a batch of B utterances: a number for the whole batch, None for "not denoised", or a (B,)
    sequence / tensor with one of those per utterance.  -> the number, None when no utterance is denoised, or a tuple of B
    floats and Nones; values that are all equal are the number, as MatchaTTS.synthesise does with its settings
    (matcha.per_item_setting, whose rules the per-utterance strengths follow: finite numbers, since the library reads them on
    the device)."""
    from .matcha import per_item_setting

    if value is None or isinstance(value, numbers.Number) or (torch.is_tensor(value) and value.dim() == 0):
        return value.item() if torch.is_tensor(value) else value
    vals = value.detach().reshape(-1).tolist() if torch.is_tensor(value) else list(value)
    if len(vals) != B:
        raise ValueError(f"strength: expected a number or {B} values (one per utterance), got {len(vals)}")
    on = [v for v in vals if v is not None]
    if not on:
        return None
    per_item_setting(on, len(on), "strength")
    vals = [None if v is None else float(v) for v in vals]
    return vals[0] if all(v == vals[0] for v in vals) else tuple(vals)


def strength_tensors(strengths, device):
    """A tuple of per_item_strength -> (strengths (B,) fp32, flags (B,) uint8: 0 = not denoised) on the device."""
    s = torch.tensor([0.0 if v is None else v for v in strengths], dtype=torch.float32)
    on = torch.tensor([v is not None for v in strengths], dtype=torch.uint8)
    return s.to(device), on.to(device)


class Denoiser:
    """hifigan/denoiser.py:7-64 (mode="zeros").  bias_spec is computed on the GPU with the given generator."""

    def __init__(self, vocoder: Generator, filter_length=1024, n_overlap=4, win_length=1024, mode="zeros"):
        if mode != "zeros":
            raise Exception(f"Mode {mode} if not supported")
        if (filter_length, n_overlap, win_length) != (1024, 4, 1024):
            raise ValueError("the denoiser kernel is built for filter_length=1024, n_overlap=4, win_length=1024")
        vocoder._materialise()
        self.vocoder = vocoder
        self.device = vocoder.device
        ctx, L = vocoder._ctx, _lib.lib()
        self.bias_spec = torch.empty(1, 513, 1, device=self.device)
        with torch.cuda.device(self.device):
            ws = ctx.workspace(L.ev_denoise_workspace_bytes(ctx.handle, 1, 88 * vocoder.hop) +
                               L.ev_vocode_workspace_bytes(ctx.handle, 1, 88) + (1 << 20))
            ctx.check(L.ev_denoiser_init(ctx.handle, _lib.ptr(self.bias_spec), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()),
                      "ev_denoiser_init")

    @torch.inference_mode()
    def __call__(self, audio, strength=0.0005, lengths=None):
        """lengths (B,) optional: valid mel frames per item of a padded batch, as `mel_lengths`.  Item b is then bit-identical
        to the call without lengths on [: lengths[b]*256] and zero beyond, and only the STFT frames those samples reach are
        transformed (ev_denoise_ragged).  Lengths given on the host must lie in [1, n // 256].

        strength: a number, or a (B,) sequence / tensor with one per item in which None means "not denoised" (see
        `per_item_strength`).  Item b then gets, bit for bit, this call with its own strength, or its input truncated to
        (n // 256) * 256 samples (and zero past lengths[b]*256) when it is not denoised (ev_denoise_items)."""
        ctx, L = self.vocoder._ctx, _lib.lib()
        squeeze = audio.dim() == 1
        a = audio.reshape(-1, audio.shape[-1]).to(device=self.device, dtype=torch.float32).contiguous()
        B, n = a.shape
        s = per_item_strength(strength, B)
        out = torch.empty(B, (n // 256) * 256, device=self.device)
        with torch.cuda.device(self.device):
            if lengths is not None:
                check_lengths(lengths, n // 256)
                lengths = torch.as_tensor(lengths).reshape(-1).to(device=self.device, dtype=torch.int64).contiguous()
                if lengths.numel() != B:
                    raise ValueError(f"lengths has {lengths.numel()} entries for a batch of {B}")
            if s is not None and not isinstance(s, tuple):
                ws = ctx.workspace(L.ev_denoise_workspace_bytes(ctx.handle, B, n))
                ctx.check(L.ev_denoise_ragged(ctx.handle, _lib.ptr(a), _lib.ptr(lengths), B, n, float(s), _lib.ptr(out), _lib.ptr(ws),
                                              ws.numel(), _lib.stream_ptr()), "ev_denoise")
            else:
                st, on = strength_tensors(s if s is not None else (None,) * B, self.device)
                ws = ctx.workspace(L.ev_denoise_items_workspace_bytes(ctx.handle, B, n))
                ctx.check(L.ev_denoise_items(ctx.handle, _lib.ptr(a), _lib.ptr(lengths), B, n, _lib.ptr(st), _lib.ptr(on), _lib.ptr(out),
                                             _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "ev_denoise_items")
        return out[0] if squeeze else out

    forward = __call__


@torch.inference_mode()
def to_waveform(mel, vocoder, denoiser=None, strength=0.00025, lengths=None):
    """feel_me.py:181-187: vocoder(mel).clamp(-1, 1) -> optional denoiser -> .cpu().squeeze().

    lengths: optional valid frames per item of a padded batch (see Generator.__call__).  With a denoiser, the denoiser still
    transforms the whole padded waveform here (the ragged vocoder leaves zeros past each utterance's end, so the last samples
    differ from the dense path); `vocoder.vocode_denoised` is the padded batch's exact form."""
    audio = (vocoder(mel, lengths=lengths) if lengths is not None else vocoder(mel)).clamp(-1, 1)
    if denoiser is not None:
        audio = denoiser(audio.squeeze(1), strength=strength)
    return audio.cpu().squeeze()
