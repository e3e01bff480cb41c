"""ctypes binding of libemojivoice_b200.so (include/emojivoice_b200.h).  PyTorch only supplies device memory and the
current CUDA stream; every kernel lives in the shared library.  There is NO fallback: if the library is missing or
the device is not sm_100, the calls raise."""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EV_LIB_PATH") or os.path.join(_HERE, "lib", "libemojivoice_b200.so")   # EV_LIB_PATH: A/B-test another build

PREC = {"fp32": 0, "float32": 0, torch.float32: 0, "bf16": 1, "bfloat16": 1, torch.bfloat16: 1,
        "tf32x3": 2}    # unit-test hook only: fp32-accurate tensor-core path (3xTF32 split) the text encoder uses


class EvTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("ndim", C.c_int32), ("shape", C.c_int64 * 4)]


class EvMatchaCfg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_vocab", "n_spks", "spk_emb_dim", "n_feats", "enc_channels", "enc_filter_channels",
        "enc_filter_channels_dp", "enc_heads", "enc_layers", "enc_kernel", "enc_prenet", "dec_channels", "dec_heads",
        "dec_head_dim", "dec_mid_blocks")] + [("mel_mean", C.c_float), ("mel_std", C.c_float)]


class EvHifiganCfg(C.Structure):
    _fields_ = [("num_mels", C.c_int32), ("upsample_initial_channel", C.c_int32), ("n_ups", C.c_int32),
                ("n_kernels", C.c_int32), ("upsample_rates", C.c_int32 * 8), ("upsample_kernel_sizes", C.c_int32 * 8),
                ("resblock_kernel_sizes", C.c_int32 * 4), ("resblock_dilation_sizes", (C.c_int32 * 3) * 4)]


class EvConvEpilogueTest(C.Structure):
    _fields_ = ([(n, C.c_int32) for n in ("B", "C_in", "T", "C_out", "K", "stride", "pad", "dilation", "transposed", "precision")] +
                [("w", C.c_void_p), ("bias", C.c_void_p), ("x", C.c_void_p), ("x_ld", C.c_int64), ("x_bs", C.c_int64),
                 ("res", C.c_void_p), ("res_ld", C.c_int64), ("res_bs", C.c_int64),
                 ("res2", C.c_void_p), ("res2_ld", C.c_int64), ("res2_bs", C.c_int64),
                 ("out_f32", C.c_void_p), ("f32_ld", C.c_int64), ("f32_bs", C.c_int64),
                 ("out_act", C.c_void_p), ("act_ld", C.c_int64), ("act_bs", C.c_int64),
                 ("gn_sum", C.c_void_p), ("lengths", C.c_void_p), ("snake_a", C.c_void_p), ("snake_invb", C.c_void_p)] +
                [(n, C.c_int32) for n in ("gn_groups", "len_shift", "mask_pre", "mask_act", "act", "f32_is_act")] +
                [("slope", C.c_float), ("alpha", C.c_float), ("div", C.c_float), ("ragged_margin", C.c_int32), ("rows_per_frame", C.c_int32),
                 ("ragged_lengths", C.c_void_p), ("schedule_host", C.c_void_p), ("report_host", C.c_void_p)])


class EvKernelStat(C.Structure):
    _fields_ = [("name", C.c_char * 48), ("launches", C.c_int64), ("total_ms", C.c_double), ("flops", C.c_double),
                ("bytes", C.c_double)]


_P, _I, _F, _SZ, _I64 = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.c_int64
# name -> (restype, argtypes); must list every symbol include/emojivoice_b200.h declares (tests check it)
SIGNATURES = {
    "ev_create": (_I, [C.POINTER(_P), _I]),
    "ev_destroy": (_I, [_P]),
    "ev_last_error": (C.c_char_p, [_P]),
    "ev_version": (_I, []),
    "ev_load_matcha": (_I, [_P, C.POINTER(EvTensor), _I, C.POINTER(EvMatchaCfg), _P]),
    "ev_load_hifigan": (_I, [_P, C.POINTER(EvTensor), _I, C.POINTER(EvHifiganCfg), _P]),
    "ev_encode_workspace_bytes": (_SZ, [_P, _I, _I]),
    "ev_encode": (_I, [_P, _P, _P, _P, _I, _I, _F, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "ev_encode_items": (_I, [_P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "ev_align_workspace_bytes": (_SZ, [_P, _I, _I, _I]),
    "ev_align": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _SZ, _P]),
    "ev_decode_workspace_bytes": (_SZ, [_P, _I, _I, _I]),
    "ev_decode": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _F, _I, _P, _P, _P, _SZ, _P]),
    "ev_decode_items_workspace_bytes": (_SZ, [_P, _I, _I, _I]),
    "ev_decode_items": (_I, [_P, _P, _P, _P, _P, _I, _I, _P, _P, _I, _P, _P, _P, _SZ, _P]),
    "ev_prior_noise": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "ev_vocode_workspace_bytes": (_SZ, [_P, _I, _I]),
    "ev_vocode": (_I, [_P, _P, _I, _I, _I, _P, _P, _SZ, _P]),
    "ev_vocode_ragged": (_I, [_P, _P, _P, _I, _I, _I, _P, _P, _SZ, _P]),
    "ev_denoise_workspace_bytes": (_SZ, [_P, _I, _I]),
    "ev_denoiser_init": (_I, [_P, _P, _P, _SZ, _P]),
    "ev_denoise": (_I, [_P, _P, _I, _I, _F, _P, _P, _SZ, _P]),
    "ev_denoise_ragged": (_I, [_P, _P, _P, _I, _I, _F, _P, _P, _SZ, _P]),
    "ev_to_waveform_ragged_workspace_bytes": (_SZ, [_P, _I, _I]),
    "ev_to_waveform_ragged": (_I, [_P, _P, _P, _I, _I, _I, _F, _P, _P, _SZ, _P]),
    "ev_denoise_items_workspace_bytes": (_SZ, [_P, _I, _I]),
    "ev_denoise_items": (_I, [_P, _P, _P, _I, _I, _P, _P, _P, _P, _SZ, _P]),
    "ev_to_waveform_items_workspace_bytes": (_SZ, [_P, _I, _I]),
    "ev_to_waveform_items": (_I, [_P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _SZ, _P]),
    "ev_maximum_path_workspace_bytes": (_SZ, [_P, _I, _I, _I]),
    "ev_maximum_path": (_I, [_P, _P, _P, _P, _I, _I, _I, _F, _P, _P, _SZ, _P]),
    "ev_estimator_workspace_bytes": (_SZ, [_P, _I, _I]),
    "ev_estimator": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P, _SZ, _P]),
    "ev_train_forward_workspace_bytes": (_SZ, [_P, _I, _I, _I, _I]),
    "ev_train_forward": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P, _I, _I, _I, _F, _I, _I, _P, _P, _P, _SZ, _P]),
    "ev_launch_count": (_I64, [_P, _I]),
    "ev_profile_begin": (_I, [_P]),
    "ev_profile_end": (_I, [_P, C.POINTER(EvKernelStat), _I, C.POINTER(_I)]),
    "ev_test_conv1d": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P]),
    "ev_test_attention": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P]),
    "ev_test_encoder_attention": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, _I, C.POINTER(_F), _P]),
    "ev_test_encoder_attention_hd": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _I, C.POINTER(_F), _P]),
    "ev_test_ff_block": (_I, [_P] * 11 + [_I, _I, _I, _I, _P, _I, C.POINTER(_F), _P]),
    "ev_test_tf_tail": (_I, [_P] * 14 + [_I, _I, _I, _I, _P, _I, C.POINTER(_F), _P]),
    "ev_test_resnet_block": (_I, [_P, C.POINTER(EvTensor), _I, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _I, C.POINTER(_F), _P]),
    "ev_test_resblock": (_I, [_P, C.POINTER(EvTensor), _I, _I, _I, _P, _P, _I, _I, _I, _F, _F, _I, _I, _P, _I, _I, _I, _I,
                              _P, _P, _P, _P, _P]),
    "ev_test_conv_epilogue": (_I, [_P, C.POINTER(EvConvEpilogueTest), _P]),
    "ev_test_resnet_trace": (_I, [_P, _P, _I]),
    "ev_test_vocoder_margins": (_I, [C.POINTER(EvHifiganCfg), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "ev_test_euler_schedule": (_I, [_I, C.POINTER(_F), C.POINTER(_F)]),
    "ev_test_euler_tables": (_I, [C.POINTER(C.c_int32), _I, C.POINTER(_F), C.POINTER(_F)]),
    "ev_test_row_sum": (_I, [_P, _P, _I, _I, _P, _P]),
    "ev_test_conv_trace": (_I, [_P, _P, _I]),
    "ev_test_ff_trace": (_I, [_P, _P, _I]),
}

_lib = None


def lib() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built -- there is no python/CPU substitute."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build the CUDA library first (python -m emojivoice_b200.build). "
                "emojivoice_b200 has no CPU or eager-PyTorch fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Context:
    """One ev_ctx per (process, device).  Owns the packed weights; hands out a growing scratch workspace."""

    def __init__(self, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("emojivoice_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError(f"emojivoice_b200 runs on CUDA devices only, got {self.device}")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        torch.cuda.init()
        with torch.cuda.device(self.device):
            torch.zeros(1, device=self.device)  # make sure the primary context exists
            h = C.c_void_p()
            rc = lib().ev_create(C.byref(h), self.device.index)
        if rc != 0:
            raise RuntimeError(f"ev_create failed ({rc}): {lib().ev_last_error(None).decode()}")
        self.handle = h
        self._ws = None
        self.ws_version = 0          # bumped whenever the workspace is reallocated (captured graphs hold its address)

    def check(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"{what} failed ({rc}): {lib().ev_last_error(self.handle).decode()}")

    def workspace(self, nbytes: int) -> torch.Tensor:
        """The context's one scratch buffer (calls run one after another on the stream, so eager calls and every captured
        graph share it).  Growing it invalidates the graphs captured so far: `ws_version` tells the caches."""
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = None
            self._ws = torch.empty(int(nbytes * 1.25) + 4096, dtype=torch.uint8, device=self.device)
            self.ws_version += 1
        return self._ws

    def launch_count(self, reset=False) -> int:
        return int(lib().ev_launch_count(self.handle, 1 if reset else 0))

    def profile_begin(self):
        self.check(lib().ev_profile_begin(self.handle), "ev_profile_begin")

    def profile_end(self):
        """-> list of dicts {name, launches, total_ms, flops, bytes}, one per kernel class launched since begin."""
        arr = (EvKernelStat * 256)()
        n = C.c_int(0)
        self.check(lib().ev_profile_end(self.handle, arr, 256, C.byref(n)), "ev_profile_end")
        return [dict(name=arr[i].name.decode(), launches=int(arr[i].launches), total_ms=float(arr[i].total_ms),
                     flops=float(arr[i].flops), bytes=float(arr[i].bytes)) for i in range(n.value)]

    def close(self):
        if getattr(self, "handle", None):
            lib().ev_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GraphCache:
    """CUDA graphs of one library call per shape key (the decoder's n-step loop is ~750 launches, the vocoder ~50:
    replaying them as a graph takes the host out of the critical path).  A key is captured the second time it is seen
    (a one-off shape is not worth a capture); entries own their small static I/O buffers and share the context's
    workspace (so a corpus of many micro-batch shapes stays cheap); least recently used entries are dropped beyond
    `capacity`, and every entry is dropped when the workspace has been reallocated since its capture."""

    def __init__(self, capacity=64):
        self.capacity, self.entries, self.seen = capacity, {}, {}

    def get(self, key, ws_version=None):
        e = self.entries.get(key)
        if e is not None and ws_version is not None and e.get("ws_version") != ws_version:
            self.entries.pop(key)                                # captured against a workspace that no longer exists
            return None
        if e is not None:
            self.entries[key] = self.entries.pop(key)            # move to the back (most recent)
        return e

    def should_capture(self, key):
        self.seen[key] = self.seen.get(key, 0) + 1
        if len(self.seen) > 4096:
            self.seen.clear()
        return self.seen[key] >= 2

    def put(self, key, entry):
        self.entries[key] = entry
        while len(self.entries) > self.capacity:
            self.entries.pop(next(iter(self.entries)))

    def clear(self):
        self.entries.clear()


def capture(ctx, fn):
    """Run fn() once eagerly on a side stream (one-time kernel attribute setup must not happen inside a capture) and
    count the kernels it launches, then capture it into a torch.cuda.CUDAGraph.  -> (graph, kernels per replay)"""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    before = ctx.launch_count()
    with torch.cuda.stream(side):
        fn()
    launches = ctx.launch_count() - before
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g, launches


def tensor_list(sd: dict, device):
    """state_dict -> (ctypes array of EvTensor, keep-alive list).  Tensors are moved to `device` as contiguous fp32."""
    keep, arr = [], (EvTensor * len(sd))()
    for i, (k, v) in enumerate(sd.items()):
        t = v.detach().to(device=device, dtype=torch.float32).contiguous()
        name = k.encode()
        keep.append((t, name))
        arr[i].name = name
        arr[i].data = t.data_ptr()
        arr[i].ndim = min(t.dim(), 4)
        for d in range(min(t.dim(), 4)):
            arr[i].shape[d] = t.shape[d]
        if t.dim() == 0:
            arr[i].ndim, arr[i].shape[0] = 1, 1
    return arr, keep
