#!/usr/bin/env python
"""bench.py -- audio-samples/sec of batched VITS end-to-end inference (BASELINE.json configs[1]).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU)
  python bench.py --impl reference ...                      # the reference's CPU algorithm (oracle port) on host cores
  python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs as DIR/<name>.npy

A "step" is one pass of the hot path over one batch: Vits.inference on a [32, 64] token batch per GPU
(random-init VitsConfig, LJSpeech-shaped synthetic tokens), i.e. text encoder -> stochastic duration predictor
-> path expansion -> flow (reverse) -> HiFiGAN.  `value` times it with inputs resident in HBM; `e2e` times the
same call from pinned HOST buffers (tokens + SDP noise in, waveform out) per step.  Weak scaling: every rank
synthesises its own batch and rank 0 gathers the waveforms over NCCL inside the timed region.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_GPU = 32
T_TEXT = 64
SR = 22050
HIFIGAN_FLOP_PER_SAMPLE = 2.402e6      # SURVEY.md section 8d (Cin=192)
FLOW_FLOP_PER_FRAME = 14.16e6          # SURVEY.md section 8d


def load_measured(name, default=None):
    """Numbers that only a GPU box can produce are committed under profiles/ by the run that measured them
    (profiles/measured.json: FP32-FMA and dense-TF32 peaks from tools/microbench_*.cu, DRAM bytes of a decoder pass
    per shape from an ncu capture); nothing here is a hand-typed constant.  Missing key -> `default` (None)."""
    try:
        with open(os.path.join(ROOT, "profiles", "measured.json")) as f:
            return json.load(f).get(name, default)
    except Exception:
        return default


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line).

    NVML through pynvml when importable (one nvmlInit before the warm-up, then cheap per-sample queries from a
    thread); otherwise one looping `nvidia-smi -lms` process.  Either way nothing is spawned inside the timed region:
    attaching a new NVML client stalls the GPU for tens of milliseconds."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nvml, self._stop = index, [], None, None, False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
            threading.Thread(target=self._poll_nvml, daemon=True).start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        bits = [(getattr(n, "nvmlClocksEventReasonHwSlowdown", getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8))),
                (getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40))),
                (getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20))),
                (getattr(n, "nvmlClocksEventReasonSwPowerCap", getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)))]
        try:
            mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        except Exception:
            mx = None
        while not self._stop:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
                mask = int(get(self.handle))
                self.rows.append([str(sm), str(mx)] + ["Active" if mask & b else "Not Active" for b in bits])
            except Exception:
                pass
            time.sleep(0.05)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        """Index of the next sample: call at the start of the timed region."""
        return len(self.rows)

    def stop(self, first=0):
        self._stop = True
        if self.proc is not None:
            self.proc.terminate()
        rows = self.rows[first:] or self.rows[-1:]
        self.rows = rows
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = [n for i, n in enumerate(self.NAMES) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": "nvml" if self.nvml else "nvidia-smi"}


DUMP_BYTES = 64_000_000


def dump_outputs(out, directory):
    """Writes every tensor of one Vits.inference result as <directory>/<name>.npy, floating-point ones as float32 and
    integer ones as float64 (exact), so two builds can be compared output for output.  Should they exceed DUMP_BYTES in
    all, each array is cut to the same fixed, seeded sample of its flattened values in every run."""
    import numpy as np
    import torch
    arrays = {k: v.detach().cpu().numpy().astype(np.float32 if v.is_floating_point() else np.float64)
              for k, v in out.items() if torch.is_tensor(v)}
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_BYTES - 1024 * len(arrays)           # room for the .npy headers
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        if total > budget:
            n = max(1, a.size * budget // total)
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, n, replace=False))]
        np.save(os.path.join(directory, k + ".npy"), a)


def build_model(seed=1234):
    import torch
    from tts_b200.vits import Vits, VitsConfig
    torch.manual_seed(seed)
    return Vits(VitsConfig()).eval()


def make_batch(rank, device=None):
    import torch
    gen = torch.Generator().manual_seed(4321 + rank)
    tokens = torch.randint(0, 100, (B_PER_GPU, T_TEXT), generator=gen)
    lengths = torch.full((B_PER_GPU,), T_TEXT, dtype=torch.int64)
    sdp_noise = torch.randn(B_PER_GPU, 2, T_TEXT, generator=gen)
    return tokens, lengths, sdp_noise


def host_threads():
    """Threads the CPU arm can really use: the affinity mask capped by the container's CPU quota.  (On this pool the
    GPU boxes report 128 logical CPUs but run under a 16-CPU cgroup quota; 128 torch threads then run ~100x slower
    than 16 -- measured with tools/probe_host_threads.py -- which would flatter the GPU/CPU ratio.)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, -(-int(quota) // int(period))))
    except Exception:
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = min(n, max(1, -(-quota // period)))
        except Exception:
            pass
    return max(1, n)


def _oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vits_oracle as O
    return O


def cpu_reference_samples_per_s(nbatch, steps=1, warmup=0, threads=None, first_noise=None):
    """The reference's CPU algorithm (oracle port, bit-identical to the reference modules) on host cores.
    ``first_noise``: prior-noise tensor for the FIRST (warm-up) pass -- the parity gate feeds the GPU step's own
    draw here and compares that pass's output; returns (samples/s, s/step, samples, threads, first_output)."""
    import torch
    O = _oracle()
    from dataclasses import asdict
    # every host thread the container may use (torchrun exports OMP_NUM_THREADS=1; override it at run time)
    torch.set_num_threads(threads or host_threads())
    model = build_model()
    sd = model.state_dict()
    args = asdict(model.args)
    tokens, lengths, sdp_noise = make_batch(0)
    tokens, lengths, sdp_noise = tokens[:nbatch], lengths[:nbatch], sdp_noise[:nbatch]
    gen = torch.Generator().manual_seed(7)
    times, samples, first = [], 0, None
    with torch.no_grad():
        for i in range(warmup + steps):
            def noise_fn(shape, i=i):
                if i == 0 and first_noise is not None and tuple(shape) == tuple(first_noise[:nbatch].shape):
                    return first_noise[:nbatch]
                return torch.randn(shape, generator=gen)
            t0 = time.perf_counter()
            out = O.vits_inference(sd, tokens, lengths, sdp_noise, noise_fn, args=args)
            dt = time.perf_counter() - t0
            if i == 0:
                first = out
            if i >= warmup:
                times.append(dt)
                samples = int(out["y_lengths"].sum()) * 256
    return samples / (sum(times) / len(times)), sum(times) / len(times), samples, torch.get_num_threads(), first


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    nb = B_PER_GPU if host_threads() >= 8 else 4          # the whole batch per step when the host can afford it
    v, sec, samples, cores, _ = cpu_reference_samples_per_s(nb, steps=args.steps, warmup=args.warmup)
    line = {"impl": "reference", "metric": "audio_samples_per_sec", "value": v, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "vits_e2e_inference_b32_t64 (BASELINE configs[1])", "tokens": T_TEXT,
                       "batch_per_gpu": B_PER_GPU, "sample": f"first {nb} of {B_PER_GPU} utterances of the batch per step"},
            "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": "port",
                             "sample": f"{nb} of {B_PER_GPU} utterances, {samples} samples per step",
                             "logical_cpus": os.cpu_count()},
            "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def parity_report(got, want, nb):
    """The parity gate of the measured workload: the GPU step's outputs against the oracle's on the same tokens and
    the same random draws (north_star: MAS/duration indices bit-exact, waveform within 1e-4 RMS)."""
    import torch
    g = {k: (v[:nb].detach().float().cpu() if torch.is_tensor(v) else v) for k, v in got.items()}
    w = want
    rep = {"utterances": nb,
           "durations_equal": bool(torch.equal(g["durations"], w["durations"])),
           "y_lengths_equal": bool(torch.equal(got["y_lengths"][:nb].cpu(), w["y_lengths"]))}
    tw = w["alignments"].shape[-1]
    rep["path_equal"] = bool(g["alignments"].shape[-1] >= tw and torch.equal(g["alignments"][..., :tw], w["alignments"])
                             and float(g["alignments"][..., tw:].abs().sum()) == 0.0)
    n = w["model_outputs"].shape[-1]
    if g["model_outputs"].shape[-1] >= n:
        err = g["model_outputs"][..., :n] - w["model_outputs"]
        # compare the samples every caller keeps (valid lengths); the padded tail is reported separately
        valid = (torch.arange(n)[None, None, :] < (w["y_lengths"] * 256)[:, None, None]).float()
        nv = float(valid.sum())
        rms = float(((err * valid) ** 2).sum() / nv) ** 0.5
        ref_rms = float(((w["model_outputs"] * valid) ** 2).sum() / nv) ** 0.5
        rep.update({"wav_rms": rms, "wav_rel_rms": rms / max(ref_rms, 1e-30), "wav_ref_rms": ref_rms,
                    "wav_max_abs": float((err * valid).abs().max()),
                    "wav_rms_padded_tail": float((((err * (1 - valid)) ** 2).sum() / max(float((1 - valid).sum()), 1.0)) ** 0.5)})
        z_err = float((g["z"][..., :tw] - w["z"]).abs().max()) if g["z"].shape[-1] >= tw else None
        rep["z_max_abs"] = z_err
        rep["ok"] = bool(rep["durations_equal"] and rep["path_equal"] and rep["y_lengths_equal"] and rms <= 1e-4
                         and rep["wav_rel_rms"] <= 1e-4)
    else:
        rep["ok"] = False
    return rep


def gpu_eager_baseline(dev, steps=3):
    """The bar SURVEY 2a names: the same algorithm as PyTorch eager library kernels (cuDNN / cuBLAS) on the GPU, TF32
    off (fp32 like the reference), same batch and noise.  It is the oracle port moved to the device -- measured
    outside the product arm's timed region, reported beside it, never on the product path."""
    import torch
    O = _oracle()
    from dataclasses import asdict
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        model = build_model()
        sd = {k: v.to(dev) for k, v in model.state_dict().items()}
        args = asdict(model.args)
        tokens, lengths, sdp_noise = (t.to(dev) for t in make_batch(0))
        gen = torch.Generator(device=dev).manual_seed(7)
        fn = lambda shape: torch.randn(shape, generator=gen, device=dev)
        ev = []
        samples = 0
        with torch.no_grad():
            for i in range(1 + steps):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                out = O.vits_inference(sd, tokens, lengths, sdp_noise, fn, args=args)
                e.record()
                if i > 0:
                    ev.append((s, e))
                    samples += int(out["y_lengths"].sum()) * 256
        torch.cuda.synchronize()
        sec = sum(s.elapsed_time(e) for s, e in ev) / 1e3
        return {"value": samples / sec, "unit": "samples/s", "ms_per_step": sec / steps * 1e3,
                "kind": "oracle port on cuda (torch eager: cuDNN conv / cuBLAS matmul), allow_tf32=False",
                "steps": steps, "warmup": 1}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def secondary_results(dev, peaks):
    """Sub-results on the other BASELINE configs that fit one GPU (not the headline; same JSON line, key `secondary`):
    cfg3 per-GPU shard (flow reverse + HiFiGAN, B=32, 1024 frames), cfg4 MAS (512 x 200 x 1000), cfg5 multi-speaker
    B=128 mixed lengths.  CUDA events, 1 warm-up + 3 timed passes each, L2 flushed between passes."""
    import torch
    from tts_b200.helpers import maximum_path
    from tts_b200.vits import Vits, VitsArgs, VitsConfig
    res = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timed(fn, n=3):
        fn()
        ts = []
        for _ in range(n):
            flush.fill_(1)
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e))
        return sum(ts) / len(ts)

    try:   # cfg3 shard
        model = build_model().to(dev)
        g = torch.Generator(device=dev).manual_seed(3)
        z_p = torch.randn(32, 192, 1024, generator=g, device=dev)
        mask = torch.ones(32, 1, 1024, device=dev)
        ms_flow = timed(lambda: model.flow(z_p, mask, reverse=True))
        z = model.flow(z_p, mask, reverse=True)
        ms_dec = timed(lambda: model.waveform_decoder(z))
        n = 32 * 1024 * 256
        res["cfg3_shard_flow_hifigan_b32_t1024"] = {
            "flow_ms": ms_flow, "hifigan_ms": ms_dec, "samples_per_s": n / ((ms_flow + ms_dec) / 1e3),
            "hifigan_tflops": n * HIFIGAN_FLOP_PER_SAMPLE / (ms_dec / 1e3) / 1e12,
            "flow_tflops": 32 * 1024 * FLOW_FLOP_PER_FRAME / (ms_flow / 1e3) / 1e12}
        del z_p, z, mask
    except Exception as ex:  # noqa: BLE001 - a sub-result must not take the headline down
        res["cfg3_shard_flow_hifigan_b32_t1024"] = {"error": repr(ex)[:200]}
    try:   # cfg4 MAS
        g = torch.Generator(device=dev).manual_seed(4)
        v = torch.randn(512, 200, 1000, generator=g, device=dev)
        m = torch.ones(512, 200, 1000, device=dev)
        from tts_b200.helpers import maximum_path_lengths
        tx = torch.full((512,), 200, dtype=torch.int32, device=dev)
        ty = torch.full((512,), 1000, dtype=torch.int32, device=dev)
        ms = timed(lambda: maximum_path_lengths(v, tx, ty))
        gbs = 512 * 200 * 1000 * 8 / (ms / 1e3) / 1e9
        res["cfg4_mas_b512_200x1000"] = {"ms": ms, "gbs": gbs, "frac_hbm": gbs / peaks["hbm_gbs"],
                                         "bytes": "8 B per cell (f32 value in, i32 path out)"}
        del v, m
    except Exception as ex:  # noqa: BLE001
        res["cfg4_mas_b512_200x1000"] = {"error": repr(ex)[:200]}
    try:   # cfg5
        torch.manual_seed(1234)
        cfg = VitsConfig(model_args=VitsArgs(use_speaker_embedding=True, num_speakers=109))
        m5 = Vits(cfg).eval().to(dev)
        gen = torch.Generator().manual_seed(55)
        lens = torch.randint(20, 129, (128,), generator=gen)
        tok = torch.randint(0, 100, (128, 128), generator=gen)
        tok = tok * (torch.arange(128)[None, :] < lens[:, None])
        sid = torch.randint(0, 109, (128,), generator=gen)
        noise = torch.randn(128, 2, 128, generator=gen).to(dev)
        tok_d, lens_d, sid_d = tok.to(dev), lens.to(dev), sid.to(dev)
        out = {}

        def step():
            out["o"] = m5.inference(tok_d, {"x_lengths": lens_d, "speaker_ids": sid_d}, sdp_noise=noise)
        ms = timed(step)
        n = int(out["o"]["wav_lengths"].sum())
        res["cfg5_multispeaker_b128_mixed"] = {"ms": ms, "samples_per_s": n / (ms / 1e3), "valid_samples": n,
                                               "frames_padded": int(out["o"]["y_mask"].shape[-1]) * 128}
    except Exception as ex:  # noqa: BLE001
        res["cfg5_multispeaker_b128_mixed"] = {"error": repr(ex)[:200]}
    return res


def run_cuda(args):
    import torch
    import torch.distributed as dist
    from tts_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    _lib.lib()
    model = build_model().to(dev)
    # ragged batches: skip the padded frames of the batch in the flow and the decoder (every valid sample stays
    # bit-identical, tests/test_ragged_gpu.py; the padded tail of model_outputs, which no caller keeps and the metric
    # never counted, becomes zero instead of the decoder's response to zero input).  BENCH_DENSE=1 measures the
    # reference's dense batch semantics instead.
    model.trim_padding = not os.environ.get("BENCH_DENSE")
    tokens_h, lengths_h, sdp_noise_h = make_batch(rank)
    tokens_pin, lengths_pin, noise_pin = tokens_h.pin_memory(), lengths_h.pin_memory(), sdp_noise_h.pin_memory()
    tokens_d, lengths_d, noise_d = tokens_h.to(dev), lengths_h.to(dev), sdp_noise_h.to(dev)
    gen = torch.Generator(device=dev).manual_seed(99 + rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    gatherer = None
    if world > 1:
        from tts_b200.parallel import WaveformGather
        gatherer = WaveformGather(dev, dst=0)
    gather_ev = []

    def prior_noise(shape):
        return torch.randn(shape, generator=gen, device=dev, dtype=torch.float32)

    def gather(out, timed=False):
        if world == 1:
            return
        # the one collective on the data path: rank 0 receives every rank's padded waveforms + valid lengths over
        # NVLink.  Shapes are exchanged as host integers on a side stream, the payload follows the decoder there;
        # the step's end event waits for it (current stream <- side stream), so the timed region contains it.
        if timed:
            a = torch.cuda.Event(enable_timing=True)
            a.record()
        gatherer.gather(out["model_outputs"], out["wav_lengths"]).wait()
        if timed:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            gather_ev.append((a, b))

    def step_resident(stage_events=None):
        model._stage_events = stage_events
        out = model.inference(tokens_d, {"x_lengths": lengths_d}, sdp_noise=noise_d, prior_noise=prior_noise,
                              return_alignments=True)
        model._stage_events = None
        gather(out, timed=stage_events is not None)
        return out

    host_wav = {}

    def step_e2e():
        tok = tokens_pin.to(dev, non_blocking=True)
        ln = lengths_pin.to(dev, non_blocking=True)
        nz = noise_pin.to(dev, non_blocking=True)
        out = model.inference(tok, {"x_lengths": ln}, sdp_noise=nz, prior_noise=prior_noise, return_alignments=True)
        gather(out)
        wav = out["model_outputs"]
        key = tuple(wav.shape)
        if key not in host_wav:
            host_wav[key] = torch.empty(wav.shape, dtype=wav.dtype).pin_memory()
        host_wav[key].copy_(wav, non_blocking=True)
        yl = out["wav_lengths"].cpu()  # device->host read of the step's result (also synchronises)
        return out, wav.numel() * 4 + yl.numel() * 8, int(yl.sum())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the sampler process attaches to the GPU when it starts (a tens-of-ms stall): start it before the warm-up and
    # only keep the samples taken inside the timed region
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        step_resident()
    barrier()

    # ---------------- timed region 1: device-resident inputs
    first_sample = sampler.mark()
    launches0 = _lib.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    stage_ev = []
    lens_out = []
    padded_samples = 0
    frames_padded = 0
    barrier()
    for s, e in ev:
        flush.fill_(1)       # evict L2 between timed iterations (outside the events)
        torch.cuda.synchronize()
        s.record()
        out = step_resident(stage_ev)
        e.record()
        lens_out.append(out["wav_lengths"])          # read after the loop: no extra host sync inside a step
        padded_samples += out["model_outputs"].numel()
        frames_padded += out["y_mask"].shape[0] * out["y_mask"].shape[-1]
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    samples_rank = int(sum(int(l.sum().item()) for l in lens_out))
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop(first_sample)
    t_resident = sum(s.elapsed_time(e) for s, e in ev) / 1e3
    dec_ms = sum(a.elapsed_time(b) for n, a, b in stage_ev if n == "waveform_decoder")
    stage_ms = {}
    for n, a, b in stage_ev:
        stage_ms[n] = stage_ms.get(n, 0.0) + a.elapsed_time(b)
    gather_ms = sum(a.elapsed_time(b) for a, b in gather_ev)
    if os.environ.get("BENCH_DEBUG") and rank == 0:
        print("per-step ms:", [round(s.elapsed_time(e), 2) for s, e in ev], file=sys.stderr)
        print("per-stage:", [(n, round(a.elapsed_time(b), 2)) for n, a, b in stage_ev], file=sys.stderr)
    if _lib.lib().b200tts_debug_tc_error():
        raise RuntimeError("bench: a tcgen05 conv launch hit a pipeline timeout -- results are invalid")

    # ---------------- timed region 2: end to end from pinned host buffers
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    e2e_samples, d2h = 0, 0
    for _ in range(args.steps):
        out, nbytes, nvalid = step_e2e()
        e2e_samples += nvalid
        d2h = nbytes
    barrier()
    t_e2e = time.perf_counter() - t0

    def allred(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    allmax = lambda x: allred(x, dist.ReduceOp.MAX)
    allsum = lambda x: allred(x, dist.ReduceOp.SUM)
    t_resident_max, t_e2e_max = allmax(t_resident), allmax(t_e2e)
    total_samples, total_e2e_samples = allsum(samples_rank), allsum(e2e_samples)
    frames_max, frames_sum = allmax(frames_padded / args.steps), allsum(frames_padded / args.steps)
    compute_ms_max = allmax((t_resident * 1e3 - gather_ms) / args.steps)
    compute_ms_sum = allsum((t_resident * 1e3 - gather_ms) / args.steps)
    gather_ms_max = allmax(gather_ms / args.steps)

    # ---------------- parity gate of the measured workload (rank 0, N = 1): same tokens, same draws, vs the oracle
    parity, cpu = None, None
    if rank == 0 and world == 1 and not os.environ.get("BENCH_SKIP_CPU"):
        store = {}

        def fixed_noise(shape):
            store["n"] = torch.randn(shape, generator=torch.Generator().manual_seed(777))
            return store["n"].to(dev)

        got = model.inference(tokens_d, {"x_lengths": lengths_d}, sdp_noise=noise_d, prior_noise=fixed_noise)
        torch.cuda.synchronize()
        cpu_nb = B_PER_GPU if host_threads() >= 8 else 2
        cpu_v, cpu_sec, cpu_samples, cores, first = cpu_reference_samples_per_s(cpu_nb, steps=2, warmup=1,
                                                                                 first_noise=store["n"])
        cpu = (cpu_nb, cpu_v, cpu_sec, cpu_samples, cores)
        parity = parity_report(got, first, cpu_nb)
        del got

    if rank == 0:
        peaks = load_peaks()
        value = total_samples / t_resident_max
        e2e_value = total_e2e_samples / t_e2e_max
        # algorithmic work of the decoder pass: the frames it really computes (valid frames + the exactness margin per
        # utterance in ragged mode, every padded frame in dense mode)
        if model.trim_padding:
            margin = _lib.lib().b200tts_hifigan_margin_frames(model.waveform_decoder._handle)
            computed_samples = total_samples / max(world, 1) + args.steps * B_PER_GPU * margin * 256
            computed_samples = min(computed_samples, padded_samples)
        else:
            computed_samples = padded_samples
        dec_tflops = computed_samples * HIFIGAN_FLOP_PER_SAMPLE / (dec_ms / 1e3) / 1e12 if dec_ms > 0 else None
        h2d = tokens_pin.numel() * 8 + lengths_pin.numel() * 8 + noise_pin.numel() * 4
        if cpu is None:   # developer A/B runs (BENCH_SKIP_CPU) and N > 1: the contract's cpu_baseline is an N = 1 item
            cpu_nb, cpu_v, cpu_sec, cpu_samples, cores = 0, None, 0.0, 0, 0
        else:
            cpu_nb, cpu_v, cpu_sec, cpu_samples, cores = cpu
        tf32_peak = load_measured("tf32_dense_tflops")          # tools/microbench_mma.cu on this pool (None: not measured)
        fma_peak = load_measured("fp32_fma_tflops")
        traffic = (load_measured("decoder_dram_bytes_per_pass") or {}).get(str(frames_padded // args.steps))
        eager = None
        secondary = None
        if world == 1 and not os.environ.get("BENCH_SKIP_EXTRA"):
            try:
                eager = gpu_eager_baseline(dev)
            except Exception as ex:  # noqa: BLE001
                eager = {"error": repr(ex)[:200]}
            secondary = secondary_results(dev, peaks)
        line = {
            "metric": "audio_samples_per_sec", "value": value, "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": t_resident_max / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "vits_e2e_inference_b32_t64 (BASELINE configs[1])", "batch_per_gpu": B_PER_GPU,
                       "tokens": T_TEXT, "frames_padded_per_step": frames_padded // args.steps,
                       "frames_valid_per_step": int(total_samples / args.steps / 256),
                       "padding": ("ragged: padded frames of the batch are skipped in flow + decoder, valid samples bit-identical "
                                   "to the dense call, padded tail zero (Vits.trim_padding)") if model.trim_padding else
                                  "dense: the reference's batch semantics, padded tail computed",
                       "parallelism": f"dp{world}", "l2": "256 MiB buffer written between timed steps (outside the events)",
                       "rtf": (t_resident_max / args.steps) / (total_samples / args.steps / SR),
                       "stage_ms_per_step": {k: v / args.steps for k, v in stage_ms.items()},
                       "multi_gpu": None if world == 1 else {
                           "compute_ms_per_step_max": compute_ms_max, "compute_ms_per_step_mean": compute_ms_sum / world,
                           "gather_wait_ms_per_step_max": gather_ms_max,
                           "padded_frames_per_rank_max": frames_max, "padded_frames_per_rank_mean": frames_sum / world,
                           "note": "ranks synthesise different random batches; max/mean padded frames is the work skew "
                                   "the max-over-ranks time contains"}},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "parity": parity,
            "roofline": {"bound": "tensor", "kernel": "HiFiGAN decoder pass (tcgen05 3xTF32 conv kernels + conv_post)",
                         "achieved": dec_tflops, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                         "frac": (dec_tflops / peaks["bf16_tflops_sustained"]) if dec_tflops else None,
                         "traffic": traffic,
                         "traffic_unit": "bytes per decoder pass, ncu dram__bytes_read+write (profiles/measured.json, keyed by padded frames); algorithmic layer-granular = 21.2 KB/sample",
                         "peak_source": peaks["source"],
                         "note": "algorithmic fp32 FLOPs; the convs run on tcgen05 kind::tf32 as 3xTF32 (3 MMAs per "
                                 "algorithmic MAC) => ceiling = dense TF32 peak / 3; conv_post is a streaming FP32 kernel",
                         "tf32_dense_peak_measured": tf32_peak,
                         "frac_of_3xtf32_ceiling": (dec_tflops / (tf32_peak / 3.0)) if (dec_tflops and tf32_peak) else None,
                         "frac_fp32_fma": (dec_tflops / fma_peak) if (dec_tflops and fma_peak) else None},
            "cpu_baseline": {"value": cpu_v, "unit": "samples/s", "cores": cores, "kind": "port",
                             "sample": f"{cpu_nb} of {B_PER_GPU} utterances, 1 warm-up (= the parity pass) + 2 timed steps ({cpu_samples} samples, {cpu_sec:.2f} s per step)",
                             "logical_cpus": os.cpu_count()},
            "gpu_eager_baseline": eager,
            "secondary": secondary,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_RESULT_FD = None


def emit(line):
    """The one JSON line of the contract, on the real stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    # stdout carries exactly one JSON line: libraries that print to fd 1 (NCCL's "NCCL version ..." banner under
    # torchrun, NCCL_DEBUG output) are sent to stderr instead, the result is written to the saved descriptor
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (float32 / float64 .npy files, at most 64 MB in all)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
