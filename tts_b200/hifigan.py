"""Drop-in for TTS.vocoder.models.hifigan_generator.HifiganGenerator
(/root/reference/TTS/vocoder/models/hifigan_generator.py:162-301).

Same constructor signature, same ``state_dict`` keys (the torch modules below are only parameter
containers -- weight-norm parametrizations included -- so reference checkpoints load unchanged),
same ``forward(x, g=None)`` / ``inference(c)`` / ``remove_weight_norm()`` / ``load_checkpoint``.
The arithmetic runs in libtts_b200.so (b200tts_hifigan_forward); there is no PyTorch fallback.

``precision`` selects the numerics of the tensor-core convolutions (conv_pre, upsamplers, ResBlocks): ``"fp32"``
(default, 3xTF32: waveform within 1e-4 RMS of an fp32 computation) or ``"tf32"`` (single-pass TF32 with operands
rounded to nearest -- what the reference gets from cuDNN with torch's default ``allow_tf32`` -- and faster).  It is a
plain attribute, not part of ``state_dict``; torch's global TF32 flags are deliberately not consulted.
"""
import ctypes

import torch
from torch import nn
from torch.nn.utils.parametrizations import weight_norm
from torch.nn.utils.parametrize import is_parametrized, remove_parametrizations

from . import _lib

LRELU_SLOPE = 0.1


def get_padding(k, d):
    return int((k * d - d) / 2)


class _ParamResBlock1(nn.Module):
    """Parameter container with the key layout of ResBlock1 (hifigan_generator.py:33-82)."""

    def __init__(self, channels, kernel_size=3, dilation=(1, 3, 5)):
        super().__init__()
        self.convs1 = nn.ModuleList([
            weight_norm(nn.Conv1d(channels, channels, kernel_size, 1, dilation=d, padding=get_padding(kernel_size, d)))
            for d in dilation])
        self.convs2 = nn.ModuleList([
            weight_norm(nn.Conv1d(channels, channels, kernel_size, 1, dilation=1, padding=get_padding(kernel_size, 1)))
            for _ in dilation])

    def remove_weight_norm(self):
        for l in list(self.convs1) + list(self.convs2):
            if is_parametrized(l, "weight"):
                remove_parametrizations(l, "weight")

    def ordered_convs(self):
        out = []
        for c1, c2 in zip(self.convs1, self.convs2):
            out += [c1, c2]
        return out


class _ParamResBlock2(nn.Module):
    """Parameter container with the key layout of ResBlock2 (hifigan_generator.py:123-148)."""

    def __init__(self, channels, kernel_size=3, dilation=(1, 3)):
        super().__init__()
        self.convs = nn.ModuleList([
            weight_norm(nn.Conv1d(channels, channels, kernel_size, 1, dilation=d, padding=get_padding(kernel_size, d)))
            for d in dilation])

    def remove_weight_norm(self):
        for l in self.convs:
            if is_parametrized(l, "weight"):
                remove_parametrizations(l, "weight")

    def ordered_convs(self):
        return list(self.convs)


class HifiganGenerator(nn.Module):
    def __init__(self, in_channels, out_channels, resblock_type, resblock_dilation_sizes, resblock_kernel_sizes,
                 upsample_kernel_sizes, upsample_initial_channel, upsample_factors, inference_padding=5,
                 cond_channels=0, conv_pre_weight_norm=True, conv_post_weight_norm=True, conv_post_bias=True):
        super().__init__()
        self.inference_padding = inference_padding
        self.num_kernels = len(resblock_kernel_sizes)
        self.num_upsamples = len(upsample_factors)
        self._cfg = dict(in_channels=in_channels, out_channels=out_channels, resblock_type=str(resblock_type),
                         resblock_dilation_sizes=[list(d) for d in resblock_dilation_sizes],
                         resblock_kernel_sizes=list(resblock_kernel_sizes),
                         upsample_kernel_sizes=list(upsample_kernel_sizes),
                         upsample_initial_channel=upsample_initial_channel,
                         upsample_factors=list(upsample_factors), cond_channels=cond_channels)
        self.conv_pre = weight_norm(nn.Conv1d(in_channels, upsample_initial_channel, 7, 1, padding=3))
        resblock = _ParamResBlock1 if str(resblock_type) == "1" else _ParamResBlock2
        self.ups = nn.ModuleList()
        for i, (u, k) in enumerate(zip(upsample_factors, upsample_kernel_sizes)):
            self.ups.append(weight_norm(nn.ConvTranspose1d(upsample_initial_channel // (2 ** i),
                                                           upsample_initial_channel // (2 ** (i + 1)), k, u,
                                                           padding=(k - u) // 2)))
        self.resblocks = nn.ModuleList()
        ch = upsample_initial_channel
        for i in range(len(self.ups)):
            ch = upsample_initial_channel // (2 ** (i + 1))
            for k, d in zip(resblock_kernel_sizes, resblock_dilation_sizes):
                self.resblocks.append(resblock(ch, k, d))
        self.conv_post = weight_norm(nn.Conv1d(ch, out_channels, 7, 1, padding=3, bias=conv_post_bias))
        if cond_channels > 0:
            self.cond_layer = nn.Conv1d(cond_channels, upsample_initial_channel, 1)
        if not conv_pre_weight_norm:
            remove_parametrizations(self.conv_pre, "weight")
        if not conv_post_weight_norm:
            remove_parametrizations(self.conv_post, "weight")
        self._handle = None
        self._handle_device = None
        self._precision = "fp32"
        # a parent's load_state_dict never calls a child's load_state_dict() override (it recurses through
        # _load_from_state_dict), so the packed handle is dropped from a pre-hook: Vits.load_checkpoint twice in a row
        # must not keep the first checkpoint's decoder weights
        self._register_load_state_dict_pre_hook(lambda *a, **k: self._drop_handle())

    # ------------------------------------------------------------------ numerics
    @property
    def precision(self):
        """``"fp32"`` (3xTF32, default) or ``"tf32"`` (single-pass TF32) for the tensor-core layers."""
        return self._precision

    @precision.setter
    def precision(self, value):
        _lib.precision_id(value)              # validates (ValueError) without loading the CUDA library
        self._drop_handle()                   # the packed handle holds the weights in the old mode's format
        self._precision = value

    # ------------------------------------------------------------------ engine handle
    def _drop_handle(self):
        if getattr(self, "_handle", None) is not None:
            _lib.lib().b200tts_hifigan_destroy(self._handle)
        self._handle = None

    def __del__(self):
        try:
            self._drop_handle()
        except Exception:  # pragma: no cover - interpreter shutdown
            pass

    def _apply(self, fn, *a, **kw):
        self._drop_handle()
        return super()._apply(fn, *a, **kw)

    def repack(self):
        """Re-read the parameters (call after modifying weights in place)."""
        self._drop_handle()

    def _ordered_weights(self):
        """Host fp32 tensors in the order include/tts_b200.h documents (weight norm folded by torch)."""
        def wb(m):
            w = m.weight.detach().to(torch.float32).cpu().contiguous()
            b = None if m.bias is None else m.bias.detach().to(torch.float32).cpu().contiguous()
            return [w, b]

        out = wb(self.conv_pre)
        if hasattr(self, "cond_layer"):
            out += wb(self.cond_layer)
        for i in range(self.num_upsamples):
            out += wb(self.ups[i])
            for j in range(self.num_kernels):
                for conv in self.resblocks[i * self.num_kernels + j].ordered_convs():
                    out += wb(conv)
        out += wb(self.conv_post)
        return out

    def _ensure_handle(self, device):
        if self._handle is not None and self._handle_device == device:
            return self._handle
        self._drop_handle()
        c = self._cfg
        cfg = _lib.HifiganConfigC()
        cfg.in_channels, cfg.out_channels = c["in_channels"], c["out_channels"]
        cfg.upsample_initial_channel, cfg.cond_channels = c["upsample_initial_channel"], c["cond_channels"]
        cfg.resblock_type = 1 if c["resblock_type"] == "1" else 2
        cfg.num_upsamples = len(c["upsample_factors"])
        for i, (u, k) in enumerate(zip(c["upsample_factors"], c["upsample_kernel_sizes"])):
            cfg.upsample_factors[i], cfg.upsample_kernel_sizes[i] = u, k
        cfg.num_kernels = len(c["resblock_kernel_sizes"])
        nd = len(c["resblock_dilation_sizes"][0])
        cfg.num_dilations = nd
        for j, (k, ds) in enumerate(zip(c["resblock_kernel_sizes"], c["resblock_dilation_sizes"])):
            if len(ds) != nd:
                raise ValueError("tts_b200: all resblocks must use the same number of dilations")
            cfg.resblock_kernel_sizes[j] = k
            for n, d in enumerate(ds):
                cfg.resblock_dilations[j][n] = d
        tensors = self._ordered_weights()
        arr = (ctypes.c_void_p * len(tensors))(*[None if t is None else t.data_ptr() for t in tensors])
        handle = ctypes.c_void_p()
        with torch.cuda.device(device):
            rc = _lib.lib().b200tts_hifigan_create_ex(ctypes.byref(cfg), arr, len(tensors),
                                                      _lib.precision_id(self._precision), ctypes.byref(handle))
        _lib.check(rc, "hifigan_create")
        self._handle, self._handle_device = handle, device
        return handle

    # ------------------------------------------------------------------ reference API
    @torch.no_grad()
    def forward(self, x, g=None, peak=None, lengths=None):
        """x [B, C, T] (CUDA), g [B, cond, 1] -> waveform [B, out_channels, T*prod(upsample_factors)]
        (hifigan_generator.py:236-265).  ``peak`` (optional int32[1] device word, zeroed by the caller): conv_post folds
        max|wav| into it while storing -- the first half of save_wav's peak normalisation (tts_b200.vocoder.wav_to_int16).
        ``lengths`` (optional [B] valid frames per row of a padded batch): padded frames are neither computed nor read;
        samples below ``lengths[b] * prod(upsample_factors)`` are bit-identical to the dense call, the rest of the row is
        zero (the dense call -- like the reference -- fills it with the network's response to zero input)."""
        _lib.require_cuda(x, "x")
        if hasattr(self, "cond_layer") and g is None:
            raise ValueError("tts_b200.HifiganGenerator: model has a cond_layer but g is None")
        x = x.to(torch.float32).contiguous()
        b, cin, t = x.shape
        if cin != self._cfg["in_channels"]:
            raise ValueError(f"expected {self._cfg['in_channels']} input channels, got {cin}")
        h = self._ensure_handle(x.device)
        L = _lib.lib()
        gl = None
        if hasattr(self, "cond_layer"):
            gl = g.to(device=x.device, dtype=torch.float32).contiguous()
        with torch.cuda.device(x.device):
            tout = L.b200tts_hifigan_out_len(h, t)
            wav = torch.empty((b, self._cfg["out_channels"], tout), dtype=torch.float32, device=x.device)
            nbytes = L.b200tts_hifigan_workspace_bytes(h, b, t)
            ws = _lib.workspace(x.device, nbytes, "hifigan")
            if peak is None and lengths is None:
                rc = L.b200tts_hifigan_forward(h, _lib.ptr(x), _lib.ptr(gl), b, t, _lib.ptr(wav), _lib.ptr(ws),
                                               ctypes.c_size_t(ws.numel()), _lib.stream_ptr(x.device))
            else:
                lens = None if lengths is None else lengths.to(device=x.device, dtype=torch.int32).contiguous()
                rc = L.b200tts_hifigan_forward_ex(h, _lib.ptr(x), _lib.ptr(gl), b, t, _lib.ptr(wav), _lib.ptr(lens),
                                                  _lib.ptr(peak), _lib.ptr(ws), ctypes.c_size_t(ws.numel()),
                                                  _lib.stream_ptr(x.device))
        _lib.check(rc, "hifigan_forward")
        return wav

    @torch.no_grad()
    def inference(self, c):
        """Replicate-pad ``inference_padding`` frames each side, then forward (hifigan_generator.py:267-282)."""
        from .vocoder import AudioNorm, vocoder_input
        c = c.to(self.conv_pre.bias.device)
        # the replicate padding comes from the hand-off kernel (one pass together with any re-normalisation /
        # interpolation a caller folds in through tts_b200.vocoder.vocoder_input), not from a torch op
        c = vocoder_input(c, AudioNorm.identity(), AudioNorm.identity(), padding=self.inference_padding)
        return self.forward(c)

    def remove_weight_norm(self):
        self._drop_handle()
        for l in self.ups:
            if is_parametrized(l, "weight"):
                remove_parametrizations(l, "weight")
        for l in self.resblocks:
            l.remove_weight_norm()
        for l in (self.conv_pre, self.conv_post):
            if is_parametrized(l, "weight"):
                remove_parametrizations(l, "weight")

    def load_checkpoint(self, config, checkpoint_path, eval=False, cache=False):  # pylint: disable=redefined-builtin
        """hifigan_generator.py:293-301."""
        state = torch.load(checkpoint_path, map_location=torch.device("cpu"), weights_only=False)
        self.load_state_dict(state["model"])
        if eval:
            self.eval()
            assert not self.training
            self.remove_weight_norm()
