"""One conv layer of the path with its fused prologue / epilogue (``b200tts_conv1d_*``): the building block the
HiFiGAN / flow / posterior engines run on, exposed so a layer can be checked or reused on its own.

Replaces one ``F.conv1d`` / ``F.conv_transpose1d`` call plus the element-wise ops around it, e.g. the ResBlock1 step
``xt = F.leaky_relu(x, 0.1); xt = c(xt); x = xt + x`` (/root/reference/TTS/vocoder/models/hifigan_generator.py:93-99):

    y = ((conv(leaky_relu(x, in_slope)) + bias) + residual) * scale [+ y if accumulate] / post_div
"""
import ctypes

import torch

from . import _lib


class FusedConv1d:
    """weight [Cout,Cin,K] (or [Cin,Cout,K] with ``transposed=True``), bias [Cout] or None -- host or device tensors;
    the packed device copy is created on first use per device.

    ``precision`` chooses the numerics of the tensor-core kernels: ``"fp32"`` (default, 3xTF32, within ~1e-5 relative
    of fp32) or ``"tf32"`` (single-pass TF32 with round-to-nearest operands, cuDNN's default numerics; faster).  A layer
    the tensor cores do not take (fewer than 32 output rows, ``tensor_cores=False``, ...) is exact FP32 either way."""

    def __init__(self, weight, bias=None, dilation=1, padding=0, transposed=False, stride=1, tensor_cores=True,
                 precision="fp32"):
        self.weight = weight.detach().to(torch.float32).cpu().contiguous()
        self.bias = None if bias is None else bias.detach().to(torch.float32).cpu().contiguous()
        self.dilation, self.padding, self.transposed, self.stride = int(dilation), int(padding), bool(transposed), int(stride)
        self.tensor_cores = bool(tensor_cores)
        _lib.precision_id(precision)
        self.precision = precision
        if transposed:
            self.cin, self.cout, self.k = self.weight.shape
        else:
            self.cout, self.cin, self.k = self.weight.shape
        self._handles = {}

    def __del__(self):
        try:
            for h in self._handles.values():
                _lib.lib().b200tts_conv1d_destroy(h)
        except Exception:  # pragma: no cover - interpreter shutdown
            pass

    def _handle(self, device):
        h = self._handles.get(device)
        if h is None:
            cfg = _lib.Conv1dConfigC(self.cin, self.cout, self.k, self.dilation, self.padding, int(self.transposed), self.stride)
            out = ctypes.c_void_p()
            with torch.cuda.device(device):
                rc = _lib.lib().b200tts_conv1d_create_ex(ctypes.byref(cfg), _lib.ptr(self.weight), _lib.ptr(self.bias),
                                                         int(self.tensor_cores), _lib.precision_id(self.precision),
                                                         ctypes.byref(out))
            _lib.check(rc, "conv1d_create")
            self._handles[device] = h = out
        return h

    @torch.no_grad()
    def __call__(self, x, in_slope=1.0, residual=None, scale=1.0, accumulate_into=None, post_div=1.0):
        _lib.require_cuda(x, "x")
        x = x.to(torch.float32).contiguous()
        b, cin, t = x.shape
        if cin != self.cin:
            raise ValueError(f"tts_b200.FusedConv1d: expected {self.cin} input channels, got {cin}")
        h = self._handle(x.device)
        L = _lib.lib()
        tout = L.b200tts_conv1d_out_len(h, t)
        if accumulate_into is not None:
            y = accumulate_into
            if tuple(y.shape) != (b, self.cout, tout) or not y.is_contiguous():
                raise ValueError("tts_b200.FusedConv1d: accumulate_into has the wrong shape")
        else:
            y = torch.empty((b, self.cout, tout), dtype=torch.float32, device=x.device)
        if residual is not None:
            residual = residual.to(torch.float32).contiguous()
            if tuple(residual.shape) != (b, self.cout, tout):
                raise ValueError("tts_b200.FusedConv1d: residual has the wrong shape")
        with torch.cuda.device(x.device):
            rc = L.b200tts_conv1d_forward(h, _lib.ptr(x), b, t, ctypes.c_float(in_slope), _lib.ptr(residual),
                                          ctypes.c_float(scale), 0 if accumulate_into is None else 1,
                                          ctypes.c_float(post_div), _lib.ptr(y), _lib.stream_ptr(x.device))
        _lib.check(rc, "conv1d_forward")
        return y
