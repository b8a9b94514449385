"""Same-run A/B of the two numerics of the HiFiGAN decoder's tensor-core convolutions: "fp32" (3xTF32, the default and
what bench.py measures) against "tf32" (single-pass TF32, opt-in).

Modes alternate inside one process (fp32, tf32, fp32, tf32, ...), REPS rounds; every number is reported as the median
of the rounds with its min / max, so a difference can be read against the spread of the same measurement.  L2 (126 MB)
is overwritten before every timed window.  Reported:
  - the 11 conv and 4 upsampler layer shapes of tests/test_precision_gpu.py (ResBlock interior form: residual, lean
    epilogue; upsamplers: leaky ReLU -> polyphase transposed conv), ms per call;
  - the decoder alone at the benchmark's shape (32 rows, the frame count and per-row lengths of a cfg2 inference, ragged
    as bench.py runs it);
  - the full cfg2 Vits.inference step as bench.py configures it (random-init VitsConfig, 32 x 64 tokens,
    trim_padding=True), ms per step and valid samples per second;
  - the card name and its power limit, read in the same run.
Usage: python scripts/dev_bench_precision.py OUT.json
"""
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from tts_b200 import _lib  # noqa: E402
from tts_b200.conv import FusedConv1d  # noqa: E402

REPS = int(os.environ.get("REPS", "7"))
MODES = ("fp32", "tf32")
LAYER_CASES = [(128, 11, 5, 32, 9600), (128, 3, 1, 32, 9600), (128, 7, 3, 32, 9600), (256, 7, 1, 32, 2400),
               (256, 11, 5, 16, 4800), (64, 11, 1, 32, 19200), (64, 3, 3, 32, 19200), (64, 7, 5, 32, 19200),
               (32, 7, 5, 32, 38400), (32, 3, 1, 32, 38400), (32, 11, 3, 32, 38400)]
UPSAMPLER_CASES = [(256, 128, 16, 8, 32, 1200), (512, 256, 16, 8, 32, 152), (128, 64, 4, 2, 32, 9600),
                   (64, 32, 4, 2, 32, 19200)]


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=False).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def timed(fn, iters, flush):
    """ms per call of fn over `iters` back-to-back calls, L2 overwritten first."""
    flush.fill_(1)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def ab(fns, iters, flush):
    """Alternate the modes REPS times; median / min / max per mode and the median ratio fp32 / tf32."""
    for f in fns.values():          # warm-up: module loads, handle packing, allocator
        f()
        f()
    torch.cuda.synchronize()
    runs = {m: [] for m in fns}
    for _ in range(REPS):
        for m, f in fns.items():
            runs[m].append(timed(f, iters, flush))
    out = {m: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)} for m, v in runs.items()}
    out["speedup_median"] = out["fp32"]["median_ms"] / out["tf32"]["median_ms"]
    # the spread: how far apart two rounds of the SAME mode were, relative to its median
    out["spread_fp32"] = (out["fp32"]["max_ms"] - out["fp32"]["min_ms"]) / out["fp32"]["median_ms"]
    out["spread_tf32"] = (out["tf32"]["max_ms"] - out["tf32"]["min_ms"]) / out["tf32"]["median_ms"]
    return out


def main():
    assert torch.cuda.is_available(), "dev_bench_precision.py needs a CUDA device"
    out_path = sys.argv[1] if len(sys.argv) > 1 else "precision_ab.json"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = {"card": card(), "reps": REPS, "layers": [], "upsamplers": []}

    for c, k, dil, b, t in LAYER_CASES:
        torch.manual_seed(c + k + dil)
        w, bias = torch.randn(c, c, k) / (c * k) ** 0.5, torch.randn(c) * 0.1
        x, res = torch.randn(b, c, t, device=dev), torch.randn(b, c, t, device=dev)
        pad = (k * dil - dil) // 2
        convs = {m: FusedConv1d(w, bias, dilation=dil, padding=pad, precision=m) for m in MODES}
        fams = {}
        for m in MODES:
            with _lib.dispatch_log() as log:
                convs[m](x, in_slope=0.1, residual=res)
            fams[m] = log.names
        r = ab({m: (lambda m=m: convs[m](x, in_slope=0.1, residual=res)) for m in MODES}, 20, flush)
        r.update(shape=dict(C=c, K=k, dil=dil, B=b, T=t), kernels=fams)
        result["layers"].append(r)
        print(json.dumps(r), flush=True)

    for cin, cout, k, s, b, t in UPSAMPLER_CASES:
        torch.manual_seed(cin + k)
        w, bias = torch.randn(cin, cout, k) / (cin * k / s) ** 0.5, torch.randn(cout) * 0.1
        x = torch.randn(b, cin, t, device=dev)
        convs = {m: FusedConv1d(w, bias, padding=(k - s) // 2, transposed=True, stride=s, precision=m) for m in MODES}
        r = ab({m: (lambda m=m: convs[m](x, in_slope=0.1)) for m in MODES}, 20, flush)
        r.update(shape=dict(Cin=cin, Cout=cout, K=k, stride=s, B=b, T=t))
        result["upsamplers"].append(r)
        print(json.dumps(r), flush=True)

    # ---- cfg2 as bench.py runs it: one model per mode (same weights), so switching never repacks
    from tts_b200.vits import Vits, VitsConfig
    models = {}
    for m in MODES:
        torch.manual_seed(1234)
        models[m] = Vits(VitsConfig()).eval().to(dev)
        models[m].trim_padding = True
        models[m].waveform_decoder.precision = m
    gen = torch.Generator().manual_seed(4321)
    tokens = torch.randint(0, 100, (32, 64), generator=gen).to(dev)
    lengths = torch.full((32,), 64, dtype=torch.int64).to(dev)
    sdp_noise = torch.randn(32, 2, 64, generator=gen).to(dev)
    ngen = torch.Generator(device=dev).manual_seed(99)

    def prior_noise(shape):
        return torch.randn(shape, generator=ngen, device=dev, dtype=torch.float32)

    def step(m):
        return models[m].inference(tokens, {"x_lengths": lengths}, sdp_noise=sdp_noise, prior_noise=prior_noise,
                                   return_alignments=True)

    ref = step("fp32")
    frames = int(ref["y_mask"].shape[-1])
    ylen = ref["y_lengths"].to(torch.int32)
    samples = int(ref["wav_lengths"].sum())
    torch.manual_seed(5)
    z = torch.randn(32, 192, frames, device=dev) * ref["y_mask"]
    wav = {m: models[m].waveform_decoder(z, lengths=ylen) for m in MODES}
    d = ab({m: (lambda m=m: models[m].waveform_decoder(z, lengths=ylen)) for m in MODES}, 10, flush)
    valid = (torch.arange(wav["fp32"].shape[-1], device=dev)[None, None, :] < (ylen * 256)[:, None, None]).double()
    e = (wav["tf32"].double() - wav["fp32"].double()) * valid
    d.update(shape=dict(B=32, frames=frames, ragged=True),
             tf32_vs_fp32_rel_rms=float(e.pow(2).sum().sqrt() / (wav["fp32"].double() * valid).pow(2).sum().sqrt()))
    result["decoder"] = d
    print(json.dumps(d), flush=True)

    s = ab({m: (lambda m=m: step(m)) for m in MODES}, 10, flush)
    for m in MODES:
        s[m]["Msamples_per_s"] = samples / s[m]["median_ms"] / 1e3
    s.update(valid_samples_per_step=samples, frames=frames)
    result["vits_cfg2_step"] = s
    print(json.dumps(s), flush=True)
    result["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
    worst = max(result["layers"] + result["upsamplers"], key=lambda r: -r["speedup_median"])
    print(f"decoder {d['fp32']['median_ms']:.3f} -> {d['tf32']['median_ms']:.3f} ms ({d['speedup_median']:.2f}x), "
          f"step {s['fp32']['median_ms']:.3f} -> {s['tf32']['median_ms']:.3f} ms, slowest layer ratio "
          f"{worst['speedup_median']:.2f}x at {worst['shape']}")


if __name__ == "__main__":
    main()
