"""Drop-in for the reference's `MatchaTTS` inference surface (Matcha-TTS/matcha/models/matcha_tts.py:26-152).

Same constructor kwargs, `load_state_dict` with the reference key names, `eval()`, `synthesise(x, x_lengths,
n_timesteps, temperature, spks, length_scale)` with the same return dict.  All arithmetic runs in
libemojivoice_b200.so; this file only allocates tensors and sequences four C-ABI calls.
"""
from __future__ import annotations

import ctypes as C
import datetime as dt
import math
import numbers

import torch

from . import _lib
from .config import MatchaConfig


class MatchaTTS:
    def __init__(self, n_vocab, n_spks, spk_emb_dim, n_feats, encoder, decoder, cfm, data_statistics, out_size=None,
                 optimizer=None, scheduler=None, prior_loss=True, use_precomputed_durations=False, device=None,
                 precision="bf16", cuda_graphs=True):
        self.cfg = MatchaConfig.from_constructor_kwargs(n_vocab, n_spks, spk_emb_dim, n_feats, encoder, decoder, cfm,
                                                        data_statistics)
        self.n_vocab, self.n_spks, self.spk_emb_dim, self.n_feats = n_vocab, n_spks, spk_emb_dim, n_feats
        self.out_size, self.prior_loss, self.use_precomputed_durations = out_size, prior_loss, use_precomputed_durations
        self.hparams = dict(n_vocab=n_vocab, n_spks=n_spks, spk_emb_dim=spk_emb_dim, n_feats=n_feats, encoder=encoder,
                            decoder=decoder, cfm=cfm, data_statistics=data_statistics, out_size=out_size)
        self.mel_mean = torch.tensor(self.cfg.mel_mean)
        self.mel_std = torch.tensor(self.cfg.mel_std)
        self.precision = precision
        self._device = torch.device(device) if device is not None else None
        self._ctx = None
        self._loaded = False
        self.cuda_graphs = cuda_graphs            # replay the decoder as a CUDA graph once a (B, T_pad, n, ...) key repeats
        self._graphs = _lib.GraphCache()

    # -- nn.Module-ish surface the callers touch (feel_me.py:156-159, cli.py:110-118)
    def eval(self):
        return self

    def to(self, device):
        if self._loaded and torch.device(device) != self.device:
            raise RuntimeError("weights already live on " + str(self.device))
        self._device = torch.device(device)
        return self

    def cuda(self, device=None):
        return self.to(torch.device("cuda", torch.cuda.current_device() if device is None else device))

    @property
    def device(self):
        return self._ctx.device if self._ctx is not None else self._device

    @classmethod
    def load_from_checkpoint(cls, checkpoint_path, map_location=None, **kw):
        """Lightning checkpoint shim: needs `hyper_parameters` + `state_dict` (feel_me.py:156-159)."""
        ckpt = torch.load(checkpoint_path, map_location="cpu", weights_only=False)
        hp = dict(ckpt["hyper_parameters"])
        model = cls(**{k: hp.get(k) for k in ("n_vocab", "n_spks", "spk_emb_dim", "n_feats", "encoder", "decoder", "cfm",
                                               "data_statistics", "out_size")}, device=map_location, **kw)
        model.load_state_dict(ckpt["state_dict"])
        return model

    def load_state_dict(self, state_dict, strict=True):
        if self._loaded:
            raise RuntimeError("weights are packed once per model instance; create a new MatchaTTS to reload")
        self._ctx = _lib.Context(self._device)
        c = self.cfg
        if len(c.dec_channels) != 2 or c.dec_channels[0] != c.dec_channels[1] or c.dec_n_blocks != 1:
            raise ValueError("only the reference decoder layout channels=(c,c), n_blocks=1 is implemented")
        if c.dec_act != "snakebeta":
            raise ValueError("only act_fn='snakebeta' is implemented (configs/model/decoder/default.yaml:7)")
        cfg = _lib.EvMatchaCfg(c.n_vocab, c.n_spks, c.spk_emb_dim, c.n_feats, c.enc_channels, c.enc_filter_channels,
                               c.enc_filter_channels_dp, c.enc_heads, c.enc_layers, c.enc_kernel, int(c.enc_prenet),
                               c.dec_channels[0], c.dec_heads, c.dec_head_dim, c.dec_mid_blocks,
                               float(state_dict.get("mel_mean", c.mel_mean)), float(state_dict.get("mel_std", c.mel_std)))
        self.mel_mean = torch.tensor(cfg.mel_mean, device=self._ctx.device)
        self.mel_std = torch.tensor(cfg.mel_std, device=self._ctx.device)
        arr, keep = _lib.tensor_list(state_dict, self._ctx.device)
        with torch.cuda.device(self._ctx.device):
            rc = _lib.lib().ev_load_matcha(self._ctx.handle, arr, len(keep), C.byref(cfg), _lib.stream_ptr())
        self._ctx.check(rc, "ev_load_matcha")
        del keep
        self._loaded = True
        self._sd = state_dict                     # kept by reference for replica()
        return self

    def replica(self):
        """Another instance of this model on the same device with its own context -- packed weights (35 MB), workspace and
        graph cache -- so that a second batch can be in flight on another stream (`batch.Lanes`)."""
        if not self._loaded:
            raise RuntimeError("load_state_dict() / load_from_checkpoint() first")
        m = MatchaTTS(**self.hparams, device=self.device, precision=self.precision, cuda_graphs=self.cuda_graphs)
        return m.load_state_dict(self._sd)

    @staticmethod
    def fix_len_compatibility(length: int, num_downsamplings_in_unet: int = 2) -> int:
        """utils/model.py:14-20"""
        f = 2 ** num_downsamplings_in_unet
        return -(-int(length) // f) * f

    @torch.inference_mode()
    def synthesise(self, x, x_lengths, n_timesteps, temperature=1.0, spks=None, length_scale=1.0, z=None, dtype=None, seed=None):
        """Same contract as matcha_tts.py:77-152.  Extras: `z` injects the prior noise (B, n_feats, T_pad) *before*
        temperature scaling (the reference draws it at flow_matching.py:51); `dtype` picks "fp32" | "bf16".

        `n_timesteps`, `temperature` and `length_scale` each take a number (the whole batch) or a (B,) sequence / tensor (one
        value per utterance).  Utterance b of a batch with per-utterance values gets the durations, alignment and lengths of
        the batch called with length_scale[b], and the mel of the batch called with (n_timesteps[b], temperature[b]) at the
        same padded length T_pad (ev_encode_items / ev_decode_items in include/emojivoice_b200.h); per-utterance values that
        are all equal are the call with that number.

        `seed` draws the prior noise on the GPU from a seed per utterance instead of torch.randn: a Python int (every
        utterance; ints in [-2^63, 2^64) are taken mod 2^64), a (B,) sequence of ints or an int64 tensor (two's complement of
        the uint64 seeds; never read back).  Utterance b's noise is then a function of (seed[b], feature, frame) only
        (ev_prior_noise): it does not depend on B, T_pad, its row or the process's RNG state, and is returned in out["z"].
        The mel still depends on the batch: the decoder is not padding-invariant (GroupNorm statistics and attention keys
        cover T_pad), so a seeded utterance gets the same mel only in the same micro-batch.  None (the default) draws with
        torch.randn as before; `z` and `seed` together are a ValueError."""
        if not self._loaded:
            raise RuntimeError("load_state_dict() / load_from_checkpoint() first")
        t0 = dt.datetime.now()
        ctx, L = self._ctx, _lib.lib()
        dev = ctx.device
        prec = _lib.PREC[dtype if dtype is not None else self.precision]
        with torch.cuda.device(dev):
            x = x.to(device=dev, dtype=torch.int64).contiguous()
            x_lengths = x_lengths.to(device=dev, dtype=torch.int64).contiguous()
            B, Tx = x.shape
            n_timesteps = per_item_setting(n_timesteps, B, "n_timesteps")
            temperature = per_item_setting(temperature, B, "temperature")
            length_scale = per_item_setting(length_scale, B, "length_scale")
            ls_items = isinstance(length_scale, tuple)
            seeds = per_item_seed(seed, B)
            if seeds is not None and z is not None:
                raise ValueError("pass either `z` (the prior noise itself) or `seed` (to draw it), not both")
            if self.n_spks > 1:
                if spks is None:
                    raise ValueError("multi-speaker model: `spks` (speaker / emoji ids) is required")
                spks = spks.to(device=dev).long().contiguous()          # matcha_tts.py:118 spks.long()
                if spks.numel() != B:
                    raise ValueError("spks must hold one id per utterance")
            else:
                spks = None
            F = self.n_feats
            S = self.spk_emb_dim if self.n_spks > 1 else 0

            def encode(i, o, ws):
                if ls_items:
                    ctx.check(L.ev_encode_items(ctx.handle, _lib.ptr(i["x"]), _lib.ptr(i["x_lengths"]), _lib.ptr(i["spks"]), B, Tx,
                                                _lib.ptr(i["length_scales"]), _lib.ptr(o.get("spk_emb")), _lib.ptr(o["mu_x"]),
                                                _lib.ptr(o["logw"]), _lib.ptr(o["w_ceil"]), _lib.ptr(o["y_lengths"]), _lib.ptr(o["summary"]),
                                                _lib.ptr(ws), ws.numel(), _lib.stream_ptr()),
                              "ev_encode_items")
                    return
                ctx.check(L.ev_encode(ctx.handle, _lib.ptr(i["x"]), _lib.ptr(i["x_lengths"]), _lib.ptr(i["spks"]), B, Tx,
                                      float(length_scale), _lib.ptr(o.get("spk_emb")), _lib.ptr(o["mu_x"]), _lib.ptr(o["logw"]),
                                      _lib.ptr(o["w_ceil"]), _lib.ptr(o["y_lengths"]), _lib.ptr(o["summary"]), _lib.ptr(ws), ws.numel(),
                                      _lib.stream_ptr()),
                          "ev_encode")

            f32, i64 = torch.float32, torch.int64
            enc_out = {"mu_x": ((B, F, Tx), f32), "logw": ((B, 1, Tx), f32), "w_ceil": ((B, 1, Tx), f32), "y_lengths": ((B,), i64),
                       "summary": ((2,), i64)}
            if S:
                enc_out["spk_emb"] = ((B, S), f32)
            enc_in = {"x": x, "x_lengths": x_lengths, "spks": spks}
            if ls_items:    # a static input of the captured graph: a replay reads the values of its own call
                enc_in["length_scales"] = torch.tensor(length_scale, dtype=torch.float32).to(dev)
            e = self._run("encode", (B, Tx, "items" if ls_items else float(length_scale)), L.ev_encode_workspace_bytes(ctx.handle, B, Tx),
                          enc_in, enc_out, encode)
            mu_x, logw, w_ceil, y_lengths, spk_emb = e["mu_x"], e["logw"], e["w_ceil"], e["y_lengths"], e.get("spk_emb")
            # the reference's one host sync (y_lengths.max(), utils/model.py:18): the library reduced it on the device, together
            # with the id-range flags (nn.Embedding raises IndexError where the kernels clamp)
            y_max_length, bad_ids = (int(v) for v in e["summary"].tolist())
            if bad_ids:
                raise IndexError("index out of range in self: " + " and ".join(
                    n for bit, n in ((1, f"token id outside [0, {self.n_vocab})"), (2, f"speaker id outside [0, {self.n_spks})")) if bad_ids & bit))
            T_pad = self.fix_len_compatibility(y_max_length)
            seeded = seeds is not None                                   # ev_prior_noise writes z inside the decode stage
            if z is None and not seeded:
                z = torch.randn(B, F, T_pad, device=dev)                 # flow_matching.py:51
            elif z is not None:
                z = z.to(device=dev, dtype=torch.float32).contiguous()
                if tuple(z.shape) != (B, F, T_pad):
                    raise ValueError(f"z must have shape {(B, F, T_pad)}, got {tuple(z.shape)}")
            dec_items = isinstance(n_timesteps, tuple) or isinstance(temperature, tuple)
            dec_in = {"w_ceil": w_ceil, "x_lengths": x_lengths, "y_lengths": y_lengths, "mu_x": mu_x, "z": z, "spk_emb": spk_emb}
            if dec_items:
                # the step counts are read on the host while the launches are enqueued (part of the graph key); the temperatures
                # are a static device input of the graph
                n_list = n_timesteps if isinstance(n_timesteps, tuple) else (int(n_timesteps),) * B
                n_host = (C.c_int32 * B)(*n_list)
                temps = temperature if isinstance(temperature, tuple) else (float(temperature),) * B
                dec_in["temperatures"] = torch.tensor(temps, dtype=torch.float32).to(dev)
                dec_key = (B, Tx, T_pad, ("n",) + n_list, "items", prec)
                dec_bytes = L.ev_decode_items_workspace_bytes(ctx.handle, B, T_pad, max(n_list))
            else:
                n_steps, temp = int(n_timesteps), float(temperature)
                dec_key = (B, Tx, T_pad, n_steps, temp, prec)
                dec_bytes = L.ev_decode_workspace_bytes(ctx.handle, B, T_pad, n_steps)
            dec_out = {"attn": ((B, Tx, T_pad), f32), "mu_y": ((B, F, T_pad), f32), "y_mask": ((B, 1, T_pad), f32),
                       "dec": ((B, F, T_pad), f32), "mel": ((B, F, T_pad), f32)}
            if seeded:      # the seeds are a static device input of the graph, z one of its outputs
                dec_in["seeds"] = seeds.to(dev)
                dec_out["z"] = ((B, F, T_pad), f32)
                dec_key += ("seeded",)

            def align_decode(i, o, ws):
                if seeded:
                    ctx.check(L.ev_prior_noise(ctx.handle, _lib.ptr(i["seeds"]), B, F, T_pad, _lib.ptr(o["z"]), _lib.stream_ptr()),
                              "ev_prior_noise")
                zp = _lib.ptr(o["z"] if seeded else i["z"])
                ctx.check(L.ev_align(ctx.handle, _lib.ptr(i["w_ceil"]), _lib.ptr(i["x_lengths"]), _lib.ptr(i["y_lengths"]),
                                     _lib.ptr(i["mu_x"]), B, Tx, T_pad, _lib.ptr(o["attn"]), _lib.ptr(o["mu_y"]), _lib.ptr(o["y_mask"]),
                                     _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "ev_align")
                if dec_items:
                    ctx.check(L.ev_decode_items(ctx.handle, _lib.ptr(o["mu_y"]), _lib.ptr(i["y_lengths"]), zp,
                                                _lib.ptr(i["spk_emb"]), B, T_pad, n_host, _lib.ptr(i["temperatures"]), prec,
                                                _lib.ptr(o["dec"]), _lib.ptr(o["mel"]), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()),
                              "ev_decode_items")
                    return
                ctx.check(L.ev_decode(ctx.handle, _lib.ptr(o["mu_y"]), _lib.ptr(i["y_lengths"]), zp, _lib.ptr(i["spk_emb"]),
                                      B, T_pad, n_steps, temp, prec, _lib.ptr(o["dec"]), _lib.ptr(o["mel"]), _lib.ptr(ws), ws.numel(),
                                      _lib.stream_ptr()), "ev_decode")

            nb = max(L.ev_align_workspace_bytes(ctx.handle, B, Tx, T_pad), dec_bytes)
            d = self._run("decode", dec_key, nb, dec_in, dec_out, align_decode)
            attn, mu_y, y_mask, dec, mel = d["attn"], d["mu_y"], d["y_mask"], d["dec"], d["mel"]
            if seeded:
                z = d["z"]
        t = (dt.datetime.now() - t0).total_seconds()
        rtf = t * 22050 / (max(y_max_length, 1) * 256)                    # matcha_tts.py:142-143 (host clock, no sync)
        return {
            "encoder_outputs": mu_y[:, :, :y_max_length],
            "decoder_outputs": dec[:, :, :y_max_length],
            # NB the reference slices the 4-D (B,1,Tx,T_pad) tensor with [:, :, :y_max_length], i.e. along the TOKEN
            # axis (matcha_tts.py:148) -- a no-op whenever y_max_length >= Tx.  Kept verbatim for drop-in parity.
            "attn": attn.unsqueeze(1)[:, :, :y_max_length],
            "mel": mel[:, :, :y_max_length],
            "mel_lengths": y_lengths,
            "rtf": rtf,
            # extras (not in the reference dict): intermediates the parity tests compare
            "logw": logw, "w_ceil": w_ceil, "mu_x": mu_x, "y_mask": y_mask, "t_pad": T_pad, "z": z,
            "decoder_outputs_full": dec, "mel_full": mel,
        }

    # ---- training-side forward pass (SURVEY 8 f4): loss VALUES through the same kernels, no autograd -----------------
    @torch.no_grad()
    def forward(self, x, x_lengths, y, y_lengths, spks=None, out_size=None, cond=None, durations=None, *, t=None, z=None,
                out_offset=None, dtype="fp32"):
        """matcha_tts.py:154-245 -> (dur_loss, prior_loss, diff_loss, attn), same argument meaning.  The reference's random
        draws can be injected: `t` (B,) ~ U[0,1) and `z` like the (cut) target (flow_matching.py:106-108), `out_offset` (B,) the
        segment starts it draws with random.choice (matcha_tts.py:213-216); when omitted they are drawn here the same way.
        Values only: this build has no backward pass (training itself is outside SURVEY 8)."""
        if not self._loaded:
            raise RuntimeError("load_state_dict() / load_from_checkpoint() first")
        if cond is not None:
            raise NotImplementedError("`cond` is unused by the reference estimator (decoder.py:363) and not accepted here")
        ctx, L = self._ctx, _lib.lib()
        dev = ctx.device
        with torch.cuda.device(dev):
            x = x.to(device=dev, dtype=torch.int64).contiguous()
            x_lengths = x_lengths.to(device=dev, dtype=torch.int64).contiguous()
            y = y.to(device=dev, dtype=torch.float32).contiguous()
            y_lengths = y_lengths.to(device=dev, dtype=torch.int64).contiguous()
            B, Tx = x.shape
            F, Ty = self.n_feats, y.shape[-1]
            if self.n_spks > 1:
                if spks is None:
                    raise ValueError("multi-speaker model: `spks` is required")
                spks = spks.to(device=dev).long().contiguous()
            else:
                spks = None
            enc = self._encode_eager(x, x_lengths, spks, 1.0)
            Tc = Ty if out_size is None else int(out_size)
            if out_size is not None and out_offset is None:     # matcha_tts.py:211-216
                import random
                mx = (y_lengths - Tc).clamp(0).tolist()
                out_offset = torch.tensor([random.choice(range(0, e)) if e > 0 else 0 for e in mx], dtype=torch.int64)
            if out_offset is not None:
                out_offset = out_offset.to(device=dev, dtype=torch.int64).contiguous()
            t = torch.rand(B, device=dev) if t is None else t.to(device=dev, dtype=torch.float32).reshape(B).contiguous()
            z = torch.randn(B, F, Tc, device=dev) if z is None else z.to(device=dev, dtype=torch.float32).contiguous()
            if tuple(z.shape) != (B, F, Tc):
                raise ValueError(f"z must have shape {(B, F, Tc)}")
            if self.use_precomputed_durations:
                if durations is None:
                    raise ValueError("use_precomputed_durations=True needs `durations`")
                durations = durations.to(device=dev, dtype=torch.float32).reshape(B, Tx).contiguous()
            else:
                durations = None
            losses = torch.empty(3, dtype=torch.float32, device=dev)
            attn = torch.empty(B, Tx, Tc, dtype=torch.float32, device=dev)
            ws = ctx.workspace(L.ev_train_forward_workspace_bytes(ctx.handle, B, Tx, Ty, 0 if out_size is None else Tc))
            ctx.check(L.ev_train_forward(ctx.handle, _lib.ptr(enc["mu_x"]), _lib.ptr(enc["logw"]), _lib.ptr(x_lengths), _lib.ptr(y),
                                         _lib.ptr(y_lengths), _lib.ptr(enc.get("spk_emb")), _lib.ptr(t), _lib.ptr(z), _lib.ptr(durations),
                                         0 if out_size is None else Tc, _lib.ptr(out_offset), B, Tx, Ty, float(self.cfg.sigma_min),
                                         int(bool(self.prior_loss)), _lib.PREC[dtype], _lib.ptr(losses), _lib.ptr(attn), _lib.ptr(ws),
                                         ws.numel(), _lib.stream_ptr()), "ev_train_forward")
        prior = losses[1] if self.prior_loss else 0
        return losses[0], prior, losses[2], attn

    __call__ = forward

    def _encode_eager(self, x, x_lengths, spks, length_scale):
        """ev_encode without the CUDA-graph cache -> dict(mu_x, logw, w_ceil, y_lengths[, spk_emb])."""
        ctx, L = self._ctx, _lib.lib()
        dev = ctx.device
        B, Tx = x.shape
        F, S = self.n_feats, (self.spk_emb_dim if self.n_spks > 1 else 0)
        f32 = torch.float32
        o = {"mu_x": torch.empty(B, F, Tx, dtype=f32, device=dev), "logw": torch.empty(B, 1, Tx, dtype=f32, device=dev),
             "w_ceil": torch.empty(B, 1, Tx, dtype=f32, device=dev), "y_lengths": torch.empty(B, dtype=torch.int64, device=dev),
             "summary": torch.empty(2, dtype=torch.int64, device=dev)}
        if S:
            o["spk_emb"] = torch.empty(B, S, dtype=f32, device=dev)
        ws = ctx.workspace(L.ev_encode_workspace_bytes(ctx.handle, B, Tx))
        ctx.check(L.ev_encode(ctx.handle, _lib.ptr(x), _lib.ptr(x_lengths), _lib.ptr(spks), B, Tx, float(length_scale), _lib.ptr(o.get("spk_emb")),
                              _lib.ptr(o["mu_x"]), _lib.ptr(o["logw"]), _lib.ptr(o["w_ceil"]), _lib.ptr(o["y_lengths"]), _lib.ptr(o["summary"]),
                              _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "ev_encode")
        return o

    @property
    def decoder(self):
        """`model.decoder.compute_loss(...)` / `model.decoder.estimator(...)` as on the reference's CFM (flow_matching.py:87-118)."""
        return _CFMFacade(self)

    def _run(self, name, key, nbytes, inputs, out_specs, call):
        """One stage (`call(inputs, outputs, workspace)` enqueues library calls only), eagerly or -- once the same shape key has
        been seen before -- as a CUDA-graph replay over static buffers: inputs are copied in, outputs cloned out, so callers
        own fresh tensors as with the reference.  The text encoder (~230 launches), alignment + the decoder's n-step loop (~750)
        and the vocoder (~50) are replayed this way, which takes the host out of the critical path."""
        ctx, dev = self._ctx, self._ctx.device
        ws = ctx.workspace(nbytes)                              # (may grow the workspace: do it before looking graphs up)
        gkey = (name,) + tuple(key)
        ent = self._graphs.get(gkey, ctx.ws_version) if self.cuda_graphs else None
        if ent is None and self.cuda_graphs and self._graphs.should_capture(gkey):
            st_in = {k: (None if v is None else torch.empty_like(v)) for k, v in inputs.items()}
            for k, v in inputs.items():
                if v is not None:
                    st_in[k].copy_(v)
            st_out = {k: torch.empty(shape, dtype=dtp, device=dev) for k, (shape, dtp) in out_specs.items()}
            graph, launches = _lib.capture(ctx, lambda: call(st_in, st_out, ws))
            ent = dict(inp=st_in, out=st_out, graph=graph, launches=launches, ws_version=ctx.ws_version)
            self._graphs.put(gkey, ent)
        if ent is None:
            out = {k: torch.empty(shape, dtype=dtp, device=dev) for k, (shape, dtp) in out_specs.items()}
            call(inputs, out, ws)
            return out
        for k, v in inputs.items():
            if v is not None:
                ent["inp"][k].copy_(v)
        ent["graph"].replay()
        self._replayed_launches += ent["launches"]
        return {k: v.clone() for k, v in ent["out"].items()}

    _replayed_launches = 0

    def launch_count(self, reset=False):
        """Kernels launched by this model's context, graph replays included (a replay launches every captured kernel)."""
        n = self._ctx.launch_count(reset) + self._replayed_launches
        if reset:
            self._replayed_launches = 0
        return n


def per_item_setting(value, B, name):
    """One synthesis setting of a batch of B utterances: a number for the whole batch, or a (B,) sequence / tensor with one
    value per utterance.  -> the number, or a tuple of B values when they differ (values that are all equal are the number).
    Per-utterance values are checked here, since the library reads the length scales and temperatures on the device:
    n_timesteps must be integers >= 1, length_scale finite and positive, temperature finite."""
    if isinstance(value, numbers.Number) or (torch.is_tensor(value) and value.dim() == 0):
        return value.item() if torch.is_tensor(value) else value
    vals = value.detach().reshape(-1).tolist() if torch.is_tensor(value) else list(value)
    if len(vals) != B:
        raise ValueError(f"{name}: expected a number or {B} values (one per utterance), got {len(vals)}")
    for v in vals:
        if not isinstance(v, numbers.Real) or not math.isfinite(v):
            raise ValueError(f"{name}: per-utterance values must be finite numbers, got {v!r}")
    if name == "n_timesteps":
        if any(v != int(v) or v < 1 for v in vals):
            raise ValueError(f"n_timesteps: per-utterance step counts must be integers >= 1, got {vals}")
        vals = [int(v) for v in vals]
    elif name == "length_scale":
        if any(v <= 0 for v in vals):
            raise ValueError(f"length_scale: per-utterance values must be positive, got {vals}")
        vals = [float(v) for v in vals]
    else:
        vals = [float(v) for v in vals]
    return vals[0] if all(v == vals[0] for v in vals) else tuple(vals)


_U64 = 1 << 64


def seed_value(v, what="seed"):
    """One noise seed as the uint64 it stands for: a Python (or numpy) int in [-2^63, 2^64), taken mod 2^64.  Bools and
    non-integers are a ValueError."""
    if isinstance(v, bool) or not isinstance(v, numbers.Integral):
        raise ValueError(f"{what}: seeds must be integers, got {v!r}")
    v = int(v)
    if not -(1 << 63) <= v < _U64:
        raise ValueError(f"{what}: seeds must lie in [-2^63, 2^64), got {v}")
    return v % _U64


def per_item_seed(seed, B):
    """The noise seeds of a batch of B utterances: None, a number (every utterance), a (B,) sequence of ints or an integer
    tensor with one seed per utterance.  -> None, or a (B,) int64 tensor holding the uint64 seeds in two's complement (on the
    device of a tensor argument, else on the CPU).  An int64 tensor is taken as it is: every value is a valid seed, so it is
    not read back."""
    if seed is None:
        return None
    if torch.is_tensor(seed):
        if seed.dtype == torch.int64:
            if seed.dim() == 0:
                return seed.reshape(1).expand(B).contiguous()
            if seed.numel() != B:
                raise ValueError(f"seed: expected a number or {B} seeds (one per utterance), got {seed.numel()}")
            return seed.detach().reshape(B).contiguous()
        if seed.dtype == torch.bool or seed.is_floating_point() or seed.is_complex():
            raise ValueError(f"seed: seeds must be integers, got a {seed.dtype} tensor")
        seed = seed.item() if seed.dim() == 0 else seed.detach().reshape(-1).tolist()
    if isinstance(seed, numbers.Number):
        vals = [seed_value(seed)] * B
    else:
        if isinstance(seed, (str, bytes)) or not hasattr(seed, "__iter__"):
            raise ValueError(f"seed: seeds must be integers, got {seed!r}")
        vals = [seed_value(v) for v in seed]
        if len(vals) != B:
            raise ValueError(f"seed: expected a number or {B} seeds (one per utterance), got {len(vals)}")
    return torch.tensor([v - _U64 if v >= (1 << 63) else v for v in vals], dtype=torch.int64)


class _CFMFacade:
    """The two calls of the reference's `CFM` object that the training forward uses, on an already loaded MatchaTTS."""

    def __init__(self, model):
        self._m = model
        self.sigma_min = model.cfg.sigma_min
        self.n_feats = model.n_feats

    @torch.no_grad()
    def estimator(self, x, mask, mu, t, spks=None, cond=None, dtype="fp32"):
        """decoder.py:363-443: x, mu (B,n_feats,T), mask (B,1,T) a prefix mask, t (B,) or scalar, spks (B,spk_emb_dim) EMBEDDINGS."""
        m, L = self._m, _lib.lib()
        ctx = m._ctx
        dev = ctx.device
        with torch.cuda.device(dev):
            x = x.to(device=dev, dtype=torch.float32).contiguous()
            mu = mu.to(device=dev, dtype=torch.float32).contiguous()
            B, F, T = x.shape
            y_lengths = mask.to(dev).reshape(B, T).sum(-1).to(torch.int64).contiguous()      # sequence_mask prefix length
            t = torch.as_tensor(t, dtype=torch.float32, device=dev).reshape(-1)
            t = (t.expand(B) if t.numel() == 1 else t).contiguous()
            spk = None if spks is None else spks.to(device=dev, dtype=torch.float32).contiguous()
            v = torch.empty(B, F, T, dtype=torch.float32, device=dev)
            ws = ctx.workspace(L.ev_estimator_workspace_bytes(ctx.handle, B, T))
            ctx.check(L.ev_estimator(ctx.handle, _lib.ptr(x), _lib.ptr(y_lengths), _lib.ptr(mu), _lib.ptr(t), _lib.ptr(spk), B, T,
                                     _lib.PREC[dtype], _lib.ptr(v), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "ev_estimator")
        return v

    @torch.no_grad()
    def compute_loss(self, x1, mask, mu, spks=None, cond=None, *, t=None, z=None, dtype="fp32"):
        """flow_matching.py:87-118 -> (loss, y): the conditional-flow-matching loss value and the sampled point y."""
        dev = self._m._ctx.device
        x1 = x1.to(device=dev, dtype=torch.float32)
        b = x1.shape[0]
        t = torch.rand([b, 1, 1], device=dev) if t is None else t.to(dev, torch.float32).reshape(b, 1, 1)
        z = torch.randn_like(x1) if z is None else z.to(dev, torch.float32)
        y = (1 - (1 - self.sigma_min) * t) * z + t * x1
        u = x1 - (1 - self.sigma_min) * z
        v = self.estimator(y, mask, mu.to(dev), t.reshape(b), spks, dtype=dtype)
        loss = ((v - u).double() ** 2).sum() / (mask.to(dev).double().sum() * u.shape[1])
        return loss.float(), y
