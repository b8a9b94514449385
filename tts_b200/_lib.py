"""ctypes binding of libtts_b200.so (the C ABI in include/tts_b200.h).

There is deliberately NO fallback: if the CUDA library is missing or a call fails, the product
path raises.  (The CPU oracle under oracle/ is test infrastructure and is never imported here.)
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtts_b200.so")
_lib = None


class HifiganConfigC(ctypes.Structure):
    _fields_ = [
        ("in_channels", ctypes.c_int),
        ("out_channels", ctypes.c_int),
        ("upsample_initial_channel", ctypes.c_int),
        ("cond_channels", ctypes.c_int),
        ("resblock_type", ctypes.c_int),
        ("num_upsamples", ctypes.c_int),
        ("upsample_factors", ctypes.c_int * 8),
        ("upsample_kernel_sizes", ctypes.c_int * 8),
        ("num_kernels", ctypes.c_int),
        ("resblock_kernel_sizes", ctypes.c_int * 8),
        ("num_dilations", ctypes.c_int),
        ("resblock_dilations", (ctypes.c_int * 8) * 8),
    ]


class FlowConfigC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in ("channels", "hidden_channels", "kernel_size", "dilation_rate",
                                            "num_layers", "num_flows", "cond_channels")]


class TextEncoderConfigC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in ("n_vocab", "out_channels", "hidden_channels", "hidden_channels_ffn",
                                            "num_heads", "num_layers", "kernel_size", "rel_attn_window_size",
                                            "language_emb_dim")]


class SdpConfigC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in ("in_channels", "hidden_channels", "kernel_size", "num_flows",
                                            "cond_channels", "language_emb_dim", "num_bins")] + \
               [("tail_bound", ctypes.c_float)]


class PosteriorConfigC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in ("in_channels", "out_channels", "hidden_channels", "kernel_size",
                                            "dilation_rate", "num_layers", "cond_channels")]


class DurationPredictorConfigC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in ("in_channels", "hidden_channels", "kernel_size", "cond_channels",
                                            "language_emb_dim")]


class Conv1dConfigC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in ("in_channels", "out_channels", "kernel_size", "dilation", "padding",
                                            "transposed", "stride")]


class AudioNormC(ctypes.Structure):
    _fields_ = [("signal_norm", ctypes.c_int), ("symmetric_norm", ctypes.c_int), ("clip_norm", ctypes.c_int),
                ("max_norm", ctypes.c_float), ("min_level_db", ctypes.c_float), ("ref_level_db", ctypes.c_float),
                ("scaler_mean", ctypes.c_void_p), ("scaler_scale", ctypes.c_void_p)]


DISPATCH_NAMES = {0: "fma", 1: "tc1", 2: "tc2", 3: "tc3", 4: "tc3_staged", 5: "tc3_grouped", 6: "row1", 7: "resblock",
                  8: "tc3_tf32", 9: "tc3_grouped_tf32"}

# B200TTS_PRECISION_* of include/tts_b200.h: numerics of the tensor-core conv layers
PRECISIONS = {"fp32": 0, "tf32": 1}


def precision_id(precision):
    """``"fp32"`` (3xTF32, the default) or ``"tf32"`` (single-pass TF32) -> the C ABI constant; anything else raises.
    Pure Python: validating a setting needs no CUDA library."""
    if not isinstance(precision, str) or precision not in PRECISIONS:
        raise ValueError(f"tts_b200: precision must be one of {sorted(PRECISIONS)}, got {precision!r}")
    return PRECISIONS[precision]


def _declare(lib):
    vp, sz, ci = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
    lib.b200tts_last_error.restype = ctypes.c_char_p
    lib.b200tts_launch_count.restype = ctypes.c_ulonglong
    lib.b200tts_version.restype = ci
    lib.b200tts_debug_tc_error.restype = ci
    lib.b200tts_debug_dispatch_begin.restype = None
    lib.b200tts_debug_dispatch_end.restype = ci
    lib.b200tts_debug_dispatch_end.argtypes = [vp, ci]
    lib.b200tts_conv1d_create.restype = ci
    lib.b200tts_conv1d_create.argtypes = [ctypes.POINTER(Conv1dConfigC), vp, vp, ci, ctypes.POINTER(vp)]
    lib.b200tts_conv1d_create_ex.restype = ci
    lib.b200tts_conv1d_create_ex.argtypes = [ctypes.POINTER(Conv1dConfigC), vp, vp, ci, ci, ctypes.POINTER(vp)]
    lib.b200tts_conv1d_destroy.restype = None
    lib.b200tts_conv1d_destroy.argtypes = [vp]
    lib.b200tts_conv1d_out_len.restype = ci
    lib.b200tts_conv1d_out_len.argtypes = [vp, ci]
    lib.b200tts_conv1d_forward.restype = ci
    lib.b200tts_conv1d_forward.argtypes = [vp, vp, ci, ci, ctypes.c_float, vp, ctypes.c_float, ci, ctypes.c_float, vp, vp]
    lib.b200tts_hifigan_forward_ex.restype = ci
    lib.b200tts_hifigan_forward_ex.argtypes = [vp, vp, vp, ci, ci, vp, vp, vp, vp, sz, vp]
    lib.b200tts_hifigan_margin_frames.restype = ci
    lib.b200tts_hifigan_margin_frames.argtypes = [vp]
    lib.b200tts_flow_reverse_ragged.restype = ci
    lib.b200tts_flow_reverse_ragged.argtypes = [vp, vp, vp, vp, vp, ci, ci, vp, sz, vp]
    lib.b200tts_vocoder_input_len.restype = ci
    lib.b200tts_vocoder_input_len.argtypes = [ci, ctypes.c_float, ci]
    lib.b200tts_vocoder_input.restype = ci
    lib.b200tts_vocoder_input.argtypes = [vp, ctypes.c_longlong, ci, ci, ci, ci, ci, ctypes.POINTER(AudioNormC),
                                          ctypes.POINTER(AudioNormC), ctypes.c_float, ci, vp, ci, vp]
    lib.b200tts_absmax.restype = ci
    lib.b200tts_absmax.argtypes = [vp, ctypes.c_longlong, vp, vp]
    lib.b200tts_to_int16.restype = ci
    lib.b200tts_to_int16.argtypes = [vp, ctypes.c_longlong, vp, vp, vp]
    lib.b200tts_mas_workspace_bytes.restype = sz
    lib.b200tts_mas_workspace_bytes.argtypes = [ci, ci, ci]
    lib.b200tts_mas.restype = ci
    lib.b200tts_mas.argtypes = [vp, vp, vp, vp, ci, ci, ci, vp, ci, vp, sz, vp]
    lib.b200tts_mas_from_stats_workspace_bytes.restype = sz
    lib.b200tts_mas_from_stats_workspace_bytes.argtypes = [ci, ci, ci]
    lib.b200tts_mas_from_stats.restype = ci
    lib.b200tts_mas_from_stats.argtypes = [vp, vp, vp, vp, vp, ci, ci, ci, ci, vp, ci, vp, vp, sz, vp]
    lib.b200tts_hifigan_create.restype = ci
    lib.b200tts_hifigan_create.argtypes = [ctypes.POINTER(HifiganConfigC), ctypes.POINTER(vp), ci,
                                           ctypes.POINTER(vp)]
    lib.b200tts_hifigan_create_ex.restype = ci
    lib.b200tts_hifigan_create_ex.argtypes = [ctypes.POINTER(HifiganConfigC), ctypes.POINTER(vp), ci, ci,
                                              ctypes.POINTER(vp)]
    lib.b200tts_hifigan_precision.restype = ci
    lib.b200tts_hifigan_precision.argtypes = [vp]
    lib.b200tts_hifigan_destroy.restype = None
    lib.b200tts_hifigan_destroy.argtypes = [vp]
    lib.b200tts_hifigan_workspace_bytes.restype = sz
    lib.b200tts_hifigan_workspace_bytes.argtypes = [vp, ci, ci]
    lib.b200tts_hifigan_out_len.restype = ci
    lib.b200tts_hifigan_out_len.argtypes = [vp, ci]
    lib.b200tts_hifigan_forward.restype = ci
    lib.b200tts_hifigan_forward.argtypes = [vp, vp, vp, ci, ci, vp, vp, sz, vp]
    cf = ctypes.c_float
    for name, cfgt in (("flow", FlowConfigC), ("text_encoder", TextEncoderConfigC), ("sdp", SdpConfigC),
                       ("posterior", PosteriorConfigC), ("duration_predictor", DurationPredictorConfigC)):
        f = getattr(lib, f"b200tts_{name}_create")
        f.restype = ci
        f.argtypes = [ctypes.POINTER(cfgt), ctypes.POINTER(vp), ci, ctypes.POINTER(vp)]
        f = getattr(lib, f"b200tts_{name}_destroy")
        f.restype = None
        f.argtypes = [vp]
        f = getattr(lib, f"b200tts_{name}_workspace_bytes")
        f.restype = sz
        f.argtypes = [vp, ci, ci]
    lib.b200tts_stft_create.restype = ci
    lib.b200tts_stft_create.argtypes = [ci, ci, vp, vp, ci, ctypes.POINTER(vp)]
    lib.b200tts_stft_destroy.restype = None
    lib.b200tts_stft_destroy.argtypes = [vp]
    lib.b200tts_stft_magnitude.restype = ci
    lib.b200tts_stft_magnitude.argtypes = [vp, vp, ci, ci, ci, ci, ci, cf, vp, ci, vp]
    lib.b200tts_stft_mel_project.restype = ci
    lib.b200tts_stft_mel_project.argtypes = [vp, vp, ci, ci, cf, vp, vp]
    lib.b200tts_flow_create_forward.restype = ci
    lib.b200tts_flow_create_forward.argtypes = [ctypes.POINTER(FlowConfigC), ctypes.POINTER(vp), ci, ctypes.POINTER(vp)]
    lib.b200tts_posterior_forward.restype = ci
    lib.b200tts_posterior_forward.argtypes = [vp, vp, vp, vp, vp, ci, ci, vp, vp, vp, sz, vp]
    lib.b200tts_duration_predictor_forward.restype = ci
    lib.b200tts_duration_predictor_forward.argtypes = [vp, vp, vp, vp, vp, ci, ci, vp, vp, sz, vp]
    lib.b200tts_upsample_linear.restype = ci
    lib.b200tts_upsample_linear.argtypes = [vp, ci, ci, cf, vp, ci, vp]
    lib.b200tts_flow_reverse.restype = ci
    lib.b200tts_flow_reverse.argtypes = [vp, vp, vp, vp, ci, ci, vp, sz, vp]
    lib.b200tts_text_encoder_forward.restype = ci
    lib.b200tts_text_encoder_forward.argtypes = [vp, vp, vp, vp, ci, ci, vp, vp, vp, vp, sz, vp]
    lib.b200tts_sdp_reverse.restype = ci
    lib.b200tts_sdp_reverse.argtypes = [vp, vp, vp, vp, vp, vp, cf, ci, ci, vp, vp, vp, sz, vp]
    lib.b200tts_durations.restype = ci
    lib.b200tts_durations.argtypes = [vp, vp, cf, ci, ci, vp, vp, vp, vp, vp, vp]
    lib.b200tts_expand_prior.restype = ci
    lib.b200tts_expand_prior.argtypes = [vp, vp, vp, vp, vp, cf, ci, ci, ci, ci, vp, vp, vp, vp, vp, vp]


def lib():
    """The loaded CUDA library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"tts_b200: {LIB_PATH} is missing -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(tts_b200/csrc/build.sh).  There is no CPU fallback.")
        _lib = ctypes.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().b200tts_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"tts_b200.{what} failed (status {rc}): {msg}")


def ptr(t):
    """Raw device (or host) pointer of a tensor; None -> NULL."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t, name):
    if not t.is_cuda:
        raise RuntimeError(f"tts_b200: `{name}` must be a CUDA tensor -- this package has no CPU path")
    return t


class dispatch_log:
    """``with dispatch_log() as log: ...`` -> ``log.names``: the kernel family of every conv launch inside the block."""

    def __enter__(self):
        lib().b200tts_debug_dispatch_begin()
        self.names = []
        return self

    def __exit__(self, *exc):
        buf = (ctypes.c_int32 * 4096)()
        n = lib().b200tts_debug_dispatch_end(buf, 4096)
        self.names = [DISPATCH_NAMES.get(int(buf[i]), str(int(buf[i]))) for i in range(min(n, 4096))]
        return False


def launch_count():
    return int(lib().b200tts_launch_count())


_workspaces = {}


def workspace(device, nbytes, tag="default"):
    """A cached per-(device, stream, tag) scratch buffer that only ever grows."""
    key = (device, torch.cuda.current_stream(device).cuda_stream, tag)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    return buf
