"""The single-pass TF32 mode of the tensor-core convolutions (``precision="tf32"``) on the GPU.

What it promises (include/tts_b200.h): operands rounded to TF32 to nearest (ties away from zero), one MMA per tap,
fp32 accumulation -- the numerics cuDNN gives the reference with torch's default ``allow_tf32`` -- with the same
determinism as the default 3xTF32 mode.  The default mode is unchanged.
"""
import pytest
import torch
import torch.nn.functional as F

import vits_oracle as O

pytestmark = pytest.mark.gpu

# layer shapes of the benchmark's decoder, 10..45 tiles per CTA: (C, K, dil, B, T)
LAYER_CASES = [
    (128, 11, 5, 32, 9600),
    (128, 3, 1, 32, 9600),
    (128, 7, 3, 32, 9600),
    (256, 7, 1, 32, 2400),
    (256, 11, 5, 16, 4800),
    (64, 11, 1, 32, 19200),
    (64, 3, 3, 32, 19200),
    (64, 7, 5, 32, 19200),
    (32, 7, 5, 32, 38400),
    (32, 3, 1, 32, 38400),
    (32, 11, 3, 32, 38400),
]
UPSAMPLER_CASES = [(256, 128, 16, 8, 32, 1200), (512, 256, 16, 8, 32, 152), (128, 64, 4, 2, 32, 9600),
                   (64, 32, 4, 2, 32, 19200)]


def _tc_clean():
    from tts_b200 import _lib
    torch.cuda.synchronize()
    assert _lib.lib().b200tts_debug_tc_error() == 0


def _rel_rms(got, want):
    err = got.double() - want.double()
    return float(err.pow(2).mean().sqrt() / want.double().pow(2).mean().sqrt().clamp_min(1e-30))


def _bits(t, fn):
    u = t.float().contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    u = fn(u) & 0xFFFFFFFF
    return torch.where(u >= 2 ** 31, u - 2 ** 32, u).to(torch.int32).view(torch.float32)


def _rna(t):
    return _bits(t, lambda u: (u + 0x1000) & 0xFFFFE000)


def _trunc(t):
    return _bits(t, lambda u: u & 0xFFFFE000)


# ----------------------------------------------------------------------------- 1. rounding known answer
def _known_answer_operands():
    # 1 + 3*2^-12 (0.75 ulp of TF32 above 1), 1 + 2^-11 (an exact tie), 1 + 2^-12 (0.25 ulp), both signs; scaled by
    # powers of two per channel, so every column's sum is exact in fp32 under every rounding and the roundings of a
    # column all point the same way
    v = torch.tensor([1 + 3 * 2 ** -12, -(1 + 3 * 2 ** -12), 1 + 2 ** -11, -(1 + 2 ** -11), 1 + 2 ** -12, -(1 + 2 ** -12)])
    scale = torch.tensor([2.0 ** (ci % 3 - 1) for ci in range(8)])
    inexact = v[torch.arange(256) % 6][None, :] * scale[:, None]                    # [8, 256]
    exact = torch.tensor([1.0, -0.5, 2.0, 0.25])[torch.arange(8) % 4][:, None].expand(8, 256).contiguous()
    return inexact, exact


@pytest.mark.parametrize("rounded", ["activation", "weight"])
def test_rna_rounding_known_answer(rounded):
    """RNA, truncation and fp32 give different, exactly representable sums: torch.equal tells them apart."""
    from tts_b200 import _lib
    from tts_b200.conv import FusedConv1d
    inexact, exact = _known_answer_operands()
    if rounded == "activation":
        w = torch.ones(128, 8, 1)
        x = inexact[None]                                                          # [1, 8, 256]
        xs = {"rna": _rna(x), "trunc": _trunc(x), "fp32": x}
        ws = {k: w for k in xs}
    else:
        w = (inexact[:, :128].t() * (1 + torch.arange(128) % 2)[:, None]).unsqueeze(-1).contiguous()   # [128, 8, 1]
        x = exact[None]
        ws = {"rna": _rna(w), "trunc": _trunc(w), "fp32": w}
        xs = {k: x for k in ws}
    want = {k: torch.einsum("oc,bct->bot", ws[k][:, :, 0].double(), xs[k].double()).float() for k in ws}
    for k in want:   # the sums are exact in fp32
        assert torch.equal(want[k].double(), torch.einsum("oc,bct->bot", ws[k][:, :, 0].double(), xs[k].double()))
    assert not torch.equal(want["rna"], want["fp32"]) and not torch.equal(want["rna"], want["trunc"])
    tf32 = FusedConv1d(w, None, precision="tf32")
    default = FusedConv1d(w, None)
    with _lib.dispatch_log() as log:
        got_tf32 = tf32(x.cuda(), in_slope=1.0).cpu()
        got_fp32 = default(x.cuda(), in_slope=1.0).cpu()
    _tc_clean()
    assert log.names == ["tc3_tf32", "tc3"], log.names
    assert torch.equal(got_tf32, want["rna"]), (got_tf32 - want["rna"]).abs().max()
    assert torch.equal(got_fp32, want["fp32"]), (got_fp32 - want["fp32"]).abs().max()


# ----------------------------------------------------------------------------- 2. single layers at bench scale
def _bound(A, n_acc, post_div, extras):
    """Largest |y - y64| the single-pass mode may give.
    - operands: each rounded to TF32 (relative error <= 2^-11), so a product is off by <= (2^-10 + 2^-22) |w x|;
    - accumulation: n_acc fp32 additions that may truncate, each <= 2^-23 of a partial sum <= sum|w~ x~|;
      1.01 covers the second-order terms (2^-10 * n_acc * 2^-23 and the 2^-22);
    - the accumulator passes through post_div;
    - epilogue: at most three fp32 additions (bias, residual, old y) and one division, each rounded to nearest
      (<= 2^-24 of its result), every intermediate <= 1.01 A + |bias| + |res| + |y_old|: <= 4 * 2^-24 <= 2^-22 of it."""
    return 1.01 * (2.0 ** -10 + n_acc * 2.0 ** -23) * A / post_div + 2.0 ** -22 * (1.01 * A + extras)


def _check_layer(got, y64, A, n_acc, post_div, extras):
    err = (got.double() - y64).abs()
    bound = _bound(A, n_acc, post_div, extras)
    worst = float((err / bound).max())
    rel = _rel_rms(got, y64)
    assert worst <= 1.0, f"error exceeds the derived bound by {worst:.3f}x"
    assert rel <= 1e-3, rel
    return rel, worst


@pytest.mark.parametrize("c,k,dil,b,t", LAYER_CASES)
def test_tf32_conv_layer_bench_scale(c, k, dil, b, t):
    """ResBlock1's second-conv form y_old + ((conv(lrelu(x)) + bias) + residual), MRF mean on top; then the plain form.
    The whole batch runs on the GPU; the float64 reference covers the first and the last row (other rows are the same
    arithmetic on other CTAs' tiles)."""
    from tts_b200 import _lib
    from tts_b200.conv import FusedConv1d
    torch.manual_seed(c * 1000 + k * 10 + dil)
    w = torch.randn(c, c, k) / (c * k) ** 0.5
    bias = torch.randn(c) * 0.1
    x = torch.randn(b, c, t)
    res = torch.randn(b, c, t)
    yold = torch.randn(b, c, t)
    pad = (k * dil - dil) // 2
    default = FusedConv1d(w, bias, dilation=dil, padding=pad)
    conv = FusedConv1d(w, bias, dilation=dil, padding=pad, precision="tf32")
    with _lib.dispatch_log() as log:
        default(x[:, :, :512].cuda(), in_slope=0.1)
    family = log.names
    y = yold.cuda().clone()
    with _lib.dispatch_log() as log:
        got = conv(x.cuda(), in_slope=0.1, residual=res.cuda(), accumulate_into=y, post_div=3.0).cpu()
    _tc_clean()
    assert len(family) == 1 and log.names == [family[0].replace("_staged", "") + "_tf32"], (family, log.names)
    rows = [0, b - 1]
    xl = F.leaky_relu(x[rows], 0.1).double()
    conv64 = F.conv1d(xl, w.double(), None, dilation=dil, padding=pad)
    A = F.conv1d(xl.abs(), w.double().abs(), None, dilation=dil, padding=pad)
    bb = bias.double()[None, :, None]
    y64 = (yold[rows].double() + ((conv64 + bb) + res[rows].double())) / 3.0
    rel, worst = _check_layer(got[rows], y64, A, c * k, 3.0, bb.abs() + res[rows].double().abs() + yold[rows].double().abs())
    # plain form through the lean epilogue, another tile count (a multiple of 4 columns: 16-byte aligned rows keep the
    # layer on the tensor cores)
    t2 = t - 76
    with _lib.dispatch_log() as log2:
        got2 = conv(x[:, :, :t2].cuda(), in_slope=0.1).cpu()
    _tc_clean()
    assert log2.names == log.names, log2.names
    A2 = F.conv1d(xl[:, :, :t2].abs(), w.double().abs(), None, dilation=dil, padding=pad)
    y2 = F.conv1d(xl[:, :, :t2], w.double(), None, dilation=dil, padding=pad) + bb
    rel2, worst2 = _check_layer(got2[rows], y2, A2, c * k, 1.0, bb.abs())
    print(f"C={c} K={k} dil={dil}: rel rms {rel:.2e} / {rel2:.2e}, worst error / bound {worst:.3f} / {worst2:.3f}")


@pytest.mark.parametrize("cin,cout,k,s,b,t", UPSAMPLER_CASES)
def test_tf32_upsampler_bench_scale(cin, cout, k, s, b, t):
    """o = ups(leaky_relu(o, 0.1)) as a polyphase conv: each output sums cin * taps-per-phase products."""
    from tts_b200 import _lib
    from tts_b200.conv import FusedConv1d
    torch.manual_seed(cin + k)
    w = torch.randn(cin, cout, k) / (cin * k / s) ** 0.5
    bias = torch.randn(cout) * 0.1
    x = torch.randn(b, cin, t)
    p = (k - s) // 2
    conv = FusedConv1d(w, bias, padding=p, transposed=True, stride=s, precision="tf32")
    with _lib.dispatch_log() as log:
        got = conv(x.cuda(), in_slope=0.1).cpu()
    _tc_clean()
    assert log.names == ["tc3_tf32"], log.names
    rows = [0, b - 1]
    xl = F.leaky_relu(x[rows], 0.1).double()
    y64 = F.conv_transpose1d(xl, w.double(), bias.double(), stride=s, padding=p)
    A = F.conv_transpose1d(xl.abs(), w.double().abs(), None, stride=s, padding=p)
    taps = (k - 1 - p) // s + (s - 1 + p) // s + 1          # polyphase taps per output phase (conv1d.cu)
    rel, worst = _check_layer(got[rows], y64, A, cin * taps, 1.0, bias.double().abs()[None, :, None])
    print(f"ups {cin}->{cout} k={k} s={s}: rel rms {rel:.2e}, worst error / bound {worst:.3f}")


# ----------------------------------------------------------------------------- decoders
def _decoder_args(cin=192):
    return dict(in_channels=cin, out_channels=1, resblock_type="1", resblock_dilation_sizes=[[1, 3, 5]] * 3,
                resblock_kernel_sizes=[3, 7, 11], upsample_kernel_sizes=[16, 16, 4, 4], upsample_initial_channel=512,
                upsample_factors=[8, 8, 2, 2], inference_padding=0, cond_channels=0, conv_pre_weight_norm=False,
                conv_post_weight_norm=False, conv_post_bias=False)


@pytest.mark.parametrize("precision", ["tf32", "fp32"])
def test_decoder_is_bit_stable(precision):
    """Identical calls give identical bits; a ragged batch equals the dense one on valid samples and is zero beyond."""
    from tts_b200.hifigan import HifiganGenerator
    torch.manual_seed(7)
    m = HifiganGenerator(**_decoder_args()).eval().cuda()
    m.precision = precision
    lens = torch.tensor([256, 200, 77, 131])
    x = (torch.randn(4, 192, 256) * (torch.arange(256)[None, None, :] < lens[:, None, None])).cuda()
    a, b = m(x), m(x)
    assert torch.equal(a, b)
    ragged = m(x, lengths=lens.cuda())
    _tc_clean()
    for i, n in enumerate(lens.tolist()):
        assert torch.equal(ragged[i, :, : n * 256], a[i, :, : n * 256]), i
        assert float(ragged[i, :, n * 256:].abs().sum()) == 0.0, i


@pytest.fixture
def cudnn_tf32():
    """The reference's default numerics on a GPU: cuDNN convolutions with TF32 allowed (torch's default)."""
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = True
    yield
    torch.backends.cudnn.allow_tf32 = old


def _wav_rel(got, want):
    return float((got.double() - want.double()).pow(2).mean().sqrt() / want.double().pow(2).mean().sqrt())


@pytest.mark.parametrize("case", ["cfg1_4x80x256", "decoder192_4x1024"])
def test_tf32_waveform_quality(case, cudnn_tf32):
    from tts_b200.hifigan import HifiganGenerator
    if case == "cfg1_4x80x256":
        torch.manual_seed(1234)
        m = HifiganGenerator(80, 1, "1", [[1, 3, 5]] * 3, [3, 7, 11], [16, 16, 4, 4], 512, [8, 8, 2, 2]).eval()
        x = torch.randn(4, 80, 256)
    else:
        torch.manual_seed(41)
        m = HifiganGenerator(**_decoder_args()).eval()
        x = torch.randn(4, 192, 1024)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    want = O.hifigan_forward(sd, x)                                   # fp32 on the CPU
    cudnn = O.hifigan_forward({k: v.cuda() for k, v in sd.items()}, x.cuda()).cpu()
    m.precision = "tf32"
    got = m.cuda()(x.cuda()).cpu()
    _tc_clean()
    ours, theirs = _wav_rel(got, want), _wav_rel(cudnn, want)
    print(f"{case}: relative waveform RMS vs fp32 -- tf32 mode {ours:.3e}, cuDNN with allow_tf32 {theirs:.3e}")
    assert ours <= 5e-3, ours
    if theirs >= 1e-4:                                                # cuDNN really used TF32
        assert ours <= 2 * theirs, (ours, theirs)


def test_default_mode_is_unchanged():
    from tts_b200 import _lib
    from tts_b200.hifigan import HifiganGenerator
    torch.manual_seed(5)
    a = HifiganGenerator(**_decoder_args()).eval()
    b = HifiganGenerator(**_decoder_args()).eval()
    b.load_state_dict(a.state_dict())
    b.precision = "fp32"
    a, b = a.cuda(), b.cuda()
    x = torch.randn(2, 192, 64).cuda()
    with _lib.dispatch_log() as log:
        ya = a(x)
    yb = b(x)
    _tc_clean()
    assert a.precision == "fp32"
    assert torch.equal(ya, yb)
    assert not any(n.endswith("_tf32") for n in log.names), log.names


def test_tf32_decoder_dispatch_is_pinned():
    """Same walk as the default mode's pin: every tensor-core layer on its single-pass kernel, conv_post exact."""
    from tts_b200 import _lib
    from tts_b200.vits import Vits, VitsConfig
    torch.manual_seed(0)
    m = Vits(VitsConfig()).eval().cuda()
    m.waveform_decoder.precision = "tf32"
    with _lib.dispatch_log() as log:
        m.waveform_decoder(torch.randn(2, 192, 256).cuda())
    _tc_clean()
    names = log.names
    assert names[0] == "tc3_tf32" and names[-1] == "row1", names
    body = names[1:-1]
    assert len(body) == 4 * 19, len(body)
    for s in range(4):
        stage = body[s * 19:(s + 1) * 19]
        assert stage[0] == "tc3_tf32", (s, stage)
        assert set(stage[1:]) == ({"tc3_tf32"} if s < 2 else {"tc3_grouped_tf32"}), (s, stage)
    assert "tc3_staged" not in names
    with _lib.dispatch_log() as log:                  # the flow is not affected by the decoder's setting
        m.flow(torch.randn(2, 192, 192).cuda(), torch.ones(2, 1, 192).cuda(), reverse=True)
    assert not any(n.endswith("_tf32") for n in log.names), log.names


# ----------------------------------------------------------------------------- 7. end to end
def _perturb(m, seed):
    gen = torch.Generator().manual_seed(seed)
    for _, p in m.named_parameters():
        if float(p.detach().abs().sum()) == 0.0:
            p.data.copy_(torch.randn(p.shape, generator=gen) * 0.05)


def test_tf32_vits_cfg2_end_to_end(tmp_path):
    """cfg2 (32 utterances x 64 tokens) with the decoder in TF32 mode: everything before the decoder is untouched."""
    from dataclasses import asdict

    from tts_b200 import _lib
    from tts_b200.vits import Vits, VitsConfig
    cfg, seed = VitsConfig(), 1234
    tok = torch.randint(0, 100, (32, 64), generator=torch.Generator().manual_seed(4321))
    lens = torch.full((32,), 64)
    torch.manual_seed(seed)
    m = Vits(cfg).eval()
    _perturb(m, seed)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    sdp_noise = torch.randn(32, 2, 64, generator=torch.Generator().manual_seed(seed + 1))
    store = {}

    def prior_noise(shape):
        store["n"] = torch.randn(shape, generator=torch.Generator().manual_seed(seed + 2))
        return store["n"].cuda()

    m.waveform_decoder.precision = "tf32"
    m.cuda()
    aux = {"x_lengths": lens.cuda(), "speaker_ids": None}
    got = m.inference(tok.cuda(), aux, sdp_noise=sdp_noise, prior_noise=prior_noise)
    _tc_clean()
    want = O.vits_inference(sd, tok, lens, sdp_noise, lambda s: store["n"], args=asdict(cfg.model_args))
    assert torch.equal(got["durations"].cpu(), want["durations"])
    assert torch.equal(got["y_lengths"].cpu(), want["y_lengths"])
    assert torch.equal(got["alignments"].cpu(), want["alignments"])
    assert torch.equal(got["y_mask"].cpu(), want["y_mask"])
    n = want["model_outputs"].shape[-1]
    valid = (torch.arange(n)[None, None, :] < (want["y_lengths"] * 256)[:, None, None]).double()
    g, w_ = got["model_outputs"].cpu().double() * valid, want["model_outputs"].double() * valid
    rel = float((g - w_).pow(2).sum().sqrt() / w_.pow(2).sum().sqrt())
    print(f"cfg2 tf32 decoder: relative waveform RMS on valid samples {rel:.3e}")
    assert rel <= 5e-3, rel
    # the setting survives a checkpoint reload and a device move, and the rebuilt handle is single-pass again
    p = tmp_path / "vits.pth"
    torch.save({"model": sd}, p)
    m.load_checkpoint(cfg, str(p), eval=True)
    m.cuda()
    assert m.waveform_decoder.precision == "tf32"
    with _lib.dispatch_log() as log:
        again = m.inference(tok.cuda(), aux, sdp_noise=sdp_noise, prior_noise=prior_noise)
    _tc_clean()
    assert "tc3_tf32" in log.names
    assert torch.equal(again["model_outputs"], got["model_outputs"])
