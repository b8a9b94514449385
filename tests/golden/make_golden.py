"""Generates the committed golden fixtures from the UNMODIFIED reference modules.

Run in the build container only (needs /root/reference):  python tests/golden/make_golden.py
Each fixture stores the reference module's state_dict, the inputs and the reference outputs for a
SMALL configuration of the same classes the hot path uses (full-size weights would be >50 MB);
the kernels are config-driven, so the small shapes exercise the same code.  Zero-initialised
layers of the reference (flow `post`, ConvFlow `proj`) are perturbed so the tests are not vacuous.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import fixtures  # noqa: E402
import ref_import  # noqa: E402

R = ref_import.load()


def perturb_zero_params(m, std=0.05):
    for _, p in m.named_parameters():
        if float(p.abs().sum()) == 0.0:
            p.data.normal_(0, std)


def seq_mask(lengths, t):
    return (torch.arange(t)[None, :] < lengths[:, None]).unsqueeze(1).float()


def save(name, obj):
    path = os.path.join(HERE, name + ".pt")
    if os.path.exists(path) and "--force" not in sys.argv:   # fixtures are append-only: keep committed bytes stable
        print("kept ", name)
        return
    torch.save(obj, path)
    print("wrote", name)


@torch.no_grad()
def main():
    torch.set_num_threads(fixtures.THREADS)
    torch.manual_seed(1234)
    H = R["hifigan"].HifiganGenerator
    # 1. HiFiGAN v1 topology, narrow channels, standalone vocoder flavour
    args = dict(in_channels=80, out_channels=1, resblock_type="1", resblock_dilation_sizes=[[1, 3, 5]] * 3,
                resblock_kernel_sizes=[3, 7, 11], upsample_kernel_sizes=[16, 16, 4, 4],
                upsample_initial_channel=32, upsample_factors=[8, 8, 2, 2])
    m = H(**args).eval()
    x = torch.randn(2, 80, 13)
    save("hifigan_v1_small", {"args": args, "state": m.state_dict(), "x": x, "y": m(x), "y_inference": m.inference(x)})
    # 2. VITS flavour: cond, no weight norm on pre/post, no post bias, ResBlock2, odd sizes
    args = dict(in_channels=24, out_channels=1, resblock_type="2", resblock_dilation_sizes=[[1, 3], [1, 3]],
                resblock_kernel_sizes=[3, 5], upsample_kernel_sizes=[8, 4], upsample_initial_channel=48,
                upsample_factors=[4, 2], inference_padding=0, cond_channels=12, conv_pre_weight_norm=False,
                conv_post_weight_norm=False, conv_post_bias=False)
    m = H(**args).eval()
    x, g = torch.randn(3, 24, 19), torch.randn(3, 12, 1)
    save("hifigan_cond_rb2_small", {"args": args, "state": m.state_dict(), "x": x, "g": g, "y": m(x, g)})
    # 3. flow (reverse and forward), with speaker conditioning and ragged lengths
    args = dict(channels=16, hidden_channels=24, kernel_size=5, dilation_rate=1, num_layers=3, num_flows=4,
                cond_channels=10)
    m = R["networks"].ResidualCouplingBlocks(**args).eval()
    perturb_zero_params(m)
    z, g = torch.randn(3, 16, 37), torch.randn(3, 10, 1)
    mask = seq_mask(torch.tensor([37, 20, 5]), 37)
    save("flow_small", {"args": args, "state": m.state_dict(), "z": z, "g": g, "mask": mask,
                        "rev": m(z, mask, g=g, reverse=True), "fwd": m(z, mask, g=g, reverse=False)})
    # 4. text encoder
    args = dict(n_vocab=30, out_channels=16, hidden_channels=16, hidden_channels_ffn=40, num_heads=2, num_layers=3,
                kernel_size=3, dropout_p=0.1)
    m = R["networks"].TextEncoder(**args).eval()
    tok = torch.randint(0, 30, (4, 23))
    lens = torch.tensor([23, 17, 9, 2])
    x, mp, logs, xm = m(tok, lens)
    save("text_encoder_small", {"args": args, "state": m.state_dict(), "tokens": tok, "lengths": lens, "x": x,
                                "m_p": mp, "logs_p": logs, "x_mask": xm})
    # 5. stochastic duration predictor, reverse
    args = dict(in_channels=16, hidden_channels=16, kernel_size=3, dropout_p=0.5, num_flows=4, cond_channels=10)
    m = R["sdp"].StochasticDurationPredictor(**args).eval()
    perturb_zero_params(m)
    g4 = torch.randn(4, 10, 1)
    torch.manual_seed(77)
    noise = torch.randn(4, 2, 23)
    torch.manual_seed(77)  # the reference draws the same tensor inside forward (sdp.py:287)
    logw = m(x, xm, g=g4, reverse=True, noise_scale=0.8)
    save("sdp_small", {"args": args, "state": m.state_dict(), "x": x, "x_mask": xm, "g": g4, "noise": noise,
                       "noise_scale": 0.8, "logw": logw})
    # 6. monotonic alignment search through the reference's own Cython kernel
    assert R["helpers"].CYTHON, "oracle/_ref was not built (make -C oracle)"
    cases = []
    rng = np.random.RandomState(5)
    for (b, tx, ty) in [(3, 7, 19), (4, 33, 70), (2, 1, 5), (2, 40, 40)]:
        v = torch.from_numpy(rng.randn(b, tx, ty).astype(np.float32)) * 3
        t_x = torch.from_numpy(rng.randint(1, tx + 1, size=b))
        t_y = torch.tensor([int(rng.randint(int(a), ty + 1)) for a in t_x])
        t_x[0], t_y[0] = tx, ty
        mask = ((torch.arange(tx)[None, :, None] < t_x[:, None, None]) &
                (torch.arange(ty)[None, None, :] < t_y[:, None, None])).float()
        cases.append({"value": v, "mask": mask, "path": R["helpers"].maximum_path(v, mask)})
    save("mas_cases", {"cases": cases})
    # 7. generate_path: the reference's own known-answer structure (tests/tts_tests/test_helpers.py:71-88)
    dur = torch.randint(1, 4, (10, 21)).float()
    dur_mask = torch.ones(10, 21, int(dur.sum(1).max()))
    save("generate_path", {"duration": dur, "mask": dur_mask, "path": R["helpers"].generate_path(dur, dur_mask)})
    # 8. posterior encoder (voice conversion); the reference draws randn_like(mean) inside forward (networks.py:287)
    args = dict(in_channels=33, out_channels=16, hidden_channels=24, kernel_size=5, dilation_rate=1, num_layers=3,
                cond_channels=10)
    m = R["networks"].PosteriorEncoder(**args).eval()
    y, g3 = torch.randn(3, 33, 29).abs(), torch.randn(3, 10, 1)
    ylen = torch.tensor([29, 14, 3])
    torch.manual_seed(99)
    noise = torch.randn(3, 16, 29)
    torch.manual_seed(99)
    z, mean, log_scale, ymask = m(y, ylen, g=g3)
    save("posterior_small", {"args": args, "state": m.state_dict(), "y": y, "y_lengths": ylen, "g": g3,
                             "noise": noise, "z": z, "mean": mean, "log_scale": log_scale, "y_mask": ymask})
    # 9. deterministic duration predictor (use_sdp=False), speaker + language conditioned
    args = dict(in_channels=16, hidden_channels=32, kernel_size=3, dropout_p=0.5, cond_channels=10, language_emb_dim=4)
    m = R["duration_predictor"].DurationPredictor(**args).eval()
    for p_ in m.parameters():           # default init leaves gamma=0.1/beta=0: make every parameter informative
        p_.data.add_(torch.randn_like(p_) * 0.05)
    xd, gd, ld = torch.randn(4, 20, 23), torch.randn(4, 10, 1), torch.randn(4, 4, 1)
    xmd = seq_mask(torch.tensor([23, 17, 9, 2]), 23)
    save("duration_predictor_small", {"args": args, "state": m.state_dict(), "x": xd, "x_mask": xmd, "g": gd,
                                      "lang_emb": ld, "logw": m(xd, xmd, g=gd, lang_emb=ld)})
    # 10. voice-conversion chain built from the reference modules (vits.py:1226-1232): posterior encoder -> flow
    #     forward (source speaker) -> flow reverse (target speaker) -> HiFiGAN
    hid = 16
    pe = R["networks"].PosteriorEncoder(33, hid, hid, 5, 1, 3, cond_channels=10).eval()
    fl = R["networks"].ResidualCouplingBlocks(hid, hid, 5, 1, 2, cond_channels=10).eval()
    perturb_zero_params(fl)
    dec = H(hid, 1, "1", [[1, 3, 5]] * 3, [3, 7, 11], [8, 4], 32, [4, 2], inference_padding=0, cond_channels=10,
            conv_pre_weight_norm=False, conv_post_weight_norm=False, conv_post_bias=False).eval()
    yv, lv = torch.randn(2, 33, 21).abs(), torch.tensor([21, 9])
    g_src, g_tgt = torch.randn(2, 10, 1), torch.randn(2, 10, 1)
    torch.manual_seed(123)
    nv = torch.randn(2, hid, 21)
    torch.manual_seed(123)
    z, _, _, ym = pe(yv, lv, g=g_src)
    z_p = fl(z, ym, g=g_src)
    z_hat = fl(z_p, ym, g=g_tgt, reverse=True)
    o_hat = dec(z_hat * ym, g=g_tgt)
    state = {}
    for prefix, mod in (("posterior_encoder", pe), ("flow", fl), ("waveform_decoder", dec)):
        state.update({f"{prefix}.{k}": v for k, v in mod.state_dict().items()})
    save("vc_small", {"state": state, "y": yv, "y_lengths": lv, "g_src": g_src, "g_tgt": g_tgt, "noise": nv,
                      "z": z, "z_p": z_p, "z_hat": z_hat, "o_hat": o_hat, "y_mask": ym,
                      "args": {"hidden_channels": hid, "kernel_size_posterior_encoder": 5,
                               "dilation_rate_posterior_encoder": 1, "num_layers_posterior_encoder": 3,
                               "kernel_size_flow": 5, "dilation_rate_flow": 1, "num_layers_flow": 2,
                               "upsample_rates_decoder": [4, 2], "upsample_kernel_sizes_decoder": [8, 4],
                               "resblock_kernel_sizes_decoder": [3, 7, 11],
                               "resblock_dilation_sizes_decoder": [[1, 3, 5]] * 3, "resblock_type_decoder": "1"}})
    main_r02()


@torch.no_grad()
def main_r02():
    """Round-2 fixtures: produced by the REAL reference classes that became importable once third-party packages got
    placeholders (oracle/ref_import.load_full): Vits.inference itself, AudioProcessor, TTSTokenizer,
    interpolate_vocoder_input, HifiganGenerator.inference, save_wav's arithmetic."""
    F = ref_import.load_full()
    # 11. the real Vits.inference on a narrow multi-speaker model: the fixture the GPU box checks the product against
    args = F["vits_model"].VitsArgs(hidden_channels=64, upsample_initial_channel_decoder=32, num_layers_text_encoder=2,
                                    hidden_channels_ffn_text_encoder=128, use_speaker_embedding=True, num_speakers=7,
                                    speaker_embedding_channels=32, init_discriminator=False,
                                    num_layers_posterior_encoder=2, out_channels=33, num_layers_flow=2)
    cfg = F["vits_config"].VitsConfig()
    cfg.model_args = args
    cfg.__post_init__()
    torch.manual_seed(77)
    m = F["vits_model"].Vits(cfg).eval()
    perturb_zero_params(m)
    tok = torch.randint(0, 100, (3, 15))
    lens = torch.tensor([15, 8, 2])
    sid = torch.tensor([6, 0, 3])
    torch.manual_seed(78)
    sdp_noise = torch.randn(3, 2, 15)
    torch.manual_seed(78)
    out = m.inference(tok, aux_input={"x_lengths": lens, "speaker_ids": sid, "d_vectors": None, "language_ids": None,
                                      "durations": None})
    # recover the prior noise the reference drew (randn_like on a transposed view; see test_oracle_vs_reference_model)
    torch.manual_seed(78)
    torch.randn(3, 2, 15)
    prior = torch.randn_like(torch.empty(3, out["m_p"].shape[2], 64).transpose(1, 2)).contiguous()
    import dataclasses
    # inference never reads the posterior encoder or the SDP's training-only post_* stack: left out to keep the fixture small
    state = {k: v for k, v in m.state_dict().items()
             if not k.startswith(("posterior_encoder.", "duration_predictor.post_", "disc."))}
    save("vits_real_model_small", {"args": dataclasses.asdict(args), "state": state, "tokens": tok, "x_lengths": lens,
                                   "speaker_ids": sid, "sdp_noise": sdp_noise, "prior_noise": prior,
                                   "out": {k: v.contiguous() for k, v in out.items()}})
    # 12. AudioProcessor.normalize / denormalize, every branch; interpolate_vocoder_input; the Synthesizer hand-off
    AP = F["processor"].AudioProcessor
    rng = np.random.RandomState(5)
    S = (rng.randn(80, 37) * 35 - 45).astype(np.float32)
    cases = []
    base = dict(sample_rate=22050, num_mels=80, fft_size=1024, hop_length=256, win_length=1024, mel_fmin=0, mel_fmax=8000,
                verbose=False)
    for kw in (dict(signal_norm=True, symmetric_norm=True, max_norm=4.0, clip_norm=True, min_level_db=-100, ref_level_db=20),
               dict(signal_norm=True, symmetric_norm=True, max_norm=4.0, clip_norm=False, min_level_db=-100, ref_level_db=20),
               dict(signal_norm=True, symmetric_norm=False, max_norm=1.0, clip_norm=True, min_level_db=-100, ref_level_db=0),
               dict(signal_norm=True, symmetric_norm=False, max_norm=2.0, clip_norm=False, min_level_db=-80, ref_level_db=10),
               dict(signal_norm=False, symmetric_norm=True, max_norm=4.0, clip_norm=True, min_level_db=-100, ref_level_db=20)):
        ap = AP(**base, **kw)
        n = ap.normalize(S)
        cases.append({"kw": kw, "S": torch.from_numpy(S), "normalized": torch.from_numpy(np.asarray(n, dtype=np.float32)),
                      "denormalized": torch.from_numpy(np.asarray(ap.denormalize(n * 1.1), dtype=np.float32)),
                      "denorm_input": torch.from_numpy(np.asarray(n * 1.1, dtype=np.float32))})
    # mean-var scaler branch (stats_path): StandardScaler set by hand with float32 statistics
    ap = AP(**base, signal_norm=True, symmetric_norm=True, max_norm=4.0, clip_norm=True, min_level_db=-100, ref_level_db=20)
    mean, std = rng.randn(80).astype(np.float32) * 5 - 40, (rng.rand(80).astype(np.float32) + 0.5) * 20
    ap.setup_scaler(mean, std, np.zeros(513, np.float32), np.ones(513, np.float32))
    n = ap.normalize(S)
    cases.append({"kw": dict(signal_norm=True, mel_mean=torch.from_numpy(mean), mel_std=torch.from_numpy(std)),
                  "S": torch.from_numpy(S), "normalized": torch.from_numpy(np.asarray(n, dtype=np.float32)),
                  "denormalized": torch.from_numpy(np.asarray(ap.denormalize(n), dtype=np.float32)),
                  "denorm_input": torch.from_numpy(np.asarray(n, dtype=np.float32))})
    interp = []
    for r in (1.5, 22050 / 16000, 0.5, 24000 / 22050):
        spec = rng.randn(80, 29).astype(np.float32)
        interp.append({"scale": r, "spec": torch.from_numpy(spec),
                       "out": F["vocoder_generic_utils"].interpolate_vocoder_input([1, r], spec)})
    # the chain of synthesizer.py:412-429 with two different AudioProcessors, then HifiganGenerator.inference's pad
    tts_ap = AP(**base, signal_norm=True, symmetric_norm=True, max_norm=4.0, clip_norm=True, min_level_db=-100, ref_level_db=20)
    voc_kw = dict(signal_norm=True, symmetric_norm=False, max_norm=1.0, clip_norm=True, min_level_db=-100, ref_level_db=0)
    voc_ap = AP(**{**base, "sample_rate": 24000}, **voc_kw)
    mel_tc = tts_ap.normalize(S).T                                   # what a spectrogram TTS model returns: [T, C]
    mel = tts_ap.denormalize(mel_tc.T).T
    vin = voc_ap.normalize(mel.T)
    vin = F["vocoder_generic_utils"].interpolate_vocoder_input([1, 24000 / 22050], vin)
    padded = torch.nn.functional.pad(vin, (5, 5), "replicate")
    wav = (rng.randn(4000) * 0.2).astype(np.float32)
    wav_norm = wav * (32767 / max(0.01, np.max(np.abs(wav))))        # numpy_transforms.save_wav:439-441
    save("vocoder_handoff", {"normalize_cases": cases, "interpolate_cases": interp,
                             "chain": {"mel_tc": torch.from_numpy(np.ascontiguousarray(mel_tc)),
                                       "tts_kw": dict(signal_norm=True, symmetric_norm=True, max_norm=4.0, clip_norm=True,
                                                      min_level_db=-100, ref_level_db=20),
                                       "voc_kw": voc_kw, "sr_tts": 22050, "sr_voc": 24000, "out": padded},
                             "wav": torch.from_numpy(wav), "wav_int16": torch.from_numpy(wav_norm.astype(np.int16))})
    # 13. tokenizer: the reference's TTSTokenizer over its default grapheme set and over a plain vocabulary
    ch = F["characters"]
    T = F["tokenizer"].TTSTokenizer
    texts = ["Hello,  World!", "a b", "Zürich is   nice; isn't it?", "", "ALL CAPS and 123 digits"]
    g = ch.Graphemes()
    tok_cases = []
    for add_blank in (False, True):
        for bos in (False, True):
            t = T(False, F["cleaners"].basic_cleaners, g, None, add_blank=add_blank, use_eos_bos=bos)
            tok_cases.append({"add_blank": add_blank, "use_eos_bos": bos, "ids": [t.text_to_ids(x) for x in texts]})
    save("tokenizer_cases", {"texts": texts, "graphemes": {"characters": g.characters, "punctuations": g.punctuations,
                                                           "pad": g.pad, "eos": g.eos, "bos": g.bos, "blank": g.blank},
                             "vocab": list(g.vocab), "cases": tok_cases})
    main_full_width()
    main_real_model()
    main_reference_objects()


def _regenerate(m, seed):
    """Replaces the module's weights by the compact fixture's regenerated ones; returns what the fixture stores."""
    # the discriminator of the Vits model is training-only: it keeps its own initialisation and stays out of the fixture
    stats = fixtures.state_stats({k: v for k, v in m.state_dict().items() if not k.startswith("disc.")})
    m.load_state_dict(fixtures.state_from_stats(stats, seed), strict=False)
    return {"stats": stats, "seed": seed}


@torch.no_grad()
def main_full_width():
    """The reference layer modules at full VITS width (tests/test_oracle_vs_reference.py): weights regenerated from
    per-entry statistics of the reference's own initialisation, inputs re-drawn from fixed seeds by the test."""
    cases = {}
    torch.manual_seed(0)
    m = R["hifigan"].HifiganGenerator(192, 1, "1", [[1, 3, 5]] * 3, [3, 7, 11], [16, 16, 4, 4], 512, [8, 8, 2, 2],
                                      inference_padding=0, cond_channels=256, conv_pre_weight_norm=False,
                                      conv_post_weight_norm=False, conv_post_bias=False).eval()
    c = _regenerate(m, 1000)
    torch.manual_seed(10)
    x, g = torch.randn(1, 192, 6), torch.randn(1, 256, 1)
    c["y"] = fixtures.record(m(x, g))
    cases["hifigan"] = c

    torch.manual_seed(1)
    te = R["networks"].TextEncoder(100, 192, 192, 768, 2, 6, 3, 0.1).eval()
    c = {"text_encoder": _regenerate(te, 2000)}
    torch.manual_seed(11)
    tok, lens = torch.randint(0, 100, (3, 21)), torch.tensor([21, 13, 5])
    ref = te(tok, lens)
    c["text_encoder_out"] = [fixtures.record(t) for t in ref]
    sdp = R["sdp"].StochasticDurationPredictor(192, 192, 3, 0.5, 4, cond_channels=256).eval()
    perturb_zero_params(sdp)
    c["sdp"] = _regenerate(sdp, 3000)
    torch.manual_seed(12)
    g = torch.randn(3, 256, 1)
    torch.manual_seed(9)           # the reference draws the SDP noise inside forward (sdp.py:287)
    c["logw"] = fixtures.record(sdp(ref[0], ref[3], g=g, reverse=True, noise_scale=1.0))
    fl = R["networks"].ResidualCouplingBlocks(192, 192, 5, 1, 4, cond_channels=256).eval()
    perturb_zero_params(fl)
    c["flow"] = _regenerate(fl, 4000)
    torch.manual_seed(13)
    z = torch.randn(3, 192, 40)
    mask = seq_mask(torch.tensor([40, 22, 3]), 40)
    c["flow_out"] = fixtures.record(fl(z, mask, g=g, reverse=True))
    cases["vits_stack"] = c

    rng = np.random.RandomState(0)
    v = torch.from_numpy(rng.randn(8, 200, 1000).astype(np.float32))
    t_x = torch.from_numpy(rng.randint(100, 201, size=8))
    t_y = torch.tensor([int(rng.randint(5 * int(a) if 5 * int(a) <= 1000 else 1000, 1001)) for a in t_x])
    mask = ((torch.arange(200)[None, :, None] < t_x[:, None, None]) &
            (torch.arange(1000)[None, None, :] < t_y[:, None, None])).float()
    assert R["helpers"].CYTHON, "oracle/_ref was not built (make -C oracle)"
    cases["mas_cfg4"] = {"path": fixtures.record(R["helpers"].maximum_path(v, mask))}

    torch.manual_seed(4)
    pe = R["networks"].PosteriorEncoder(513, 192, 192, 5, 1, 16, cond_channels=256).eval()
    c = {"posterior": _regenerate(pe, 5000)}
    torch.manual_seed(14)
    y, g = torch.randn(2, 513, 33).abs(), torch.randn(2, 256, 1)
    lens = torch.tensor([33, 12])
    torch.manual_seed(5)           # PosteriorEncoder draws randn_like(mean) inside forward (networks.py:287)
    ref = pe(y, lens, g=g)
    c["posterior_out"] = [fixtures.record(t) for t in ref]
    fl = R["networks"].ResidualCouplingBlocks(192, 192, 5, 1, 4, cond_channels=256).eval()
    perturb_zero_params(fl)
    c["flow"] = _regenerate(fl, 6000)
    c["flow_out"] = fixtures.record(fl(ref[0], ref[3], g=g))
    dp = R["duration_predictor"].DurationPredictor(192, 256, 3, 0.5, cond_channels=256).eval()
    c["dp"] = _regenerate(dp, 7000)
    torch.manual_seed(15)
    x = torch.randn(2, 192, 17)
    xm = seq_mask(torch.tensor([17, 6]), 17)
    c["dp_out"] = fixtures.record(dp(x, xm, g=g))
    cases["voice_conversion_stack"] = c

    def keys(m):
        return {k: tuple(v.shape) for k, v in m.state_dict().items()}

    cases["state_dict_keys"] = {
        "TextEncoder": keys(R["networks"].TextEncoder(50, 192, 192, 768, 2, 6, 3, 0.1, language_emb_dim=4)),
        "ResidualCouplingBlocks": keys(R["networks"].ResidualCouplingBlocks(192, 192, 5, 1, 4, cond_channels=256)),
        "PosteriorEncoder": keys(R["networks"].PosteriorEncoder(513, 192, 192, 5, 1, 16, cond_channels=256)),
        "StochasticDurationPredictor": keys(R["sdp"].StochasticDurationPredictor(192, 192, 3, 0.5, 4, cond_channels=256,
                                                                                 language_emb_dim=4)),
        "DurationPredictor": keys(R["duration_predictor"].DurationPredictor(192, 256, 3, 0.5, cond_channels=256,
                                                                            language_emb_dim=4)),
        "HifiganGenerator": keys(R["hifigan"].HifiganGenerator(
            in_channels=192, out_channels=1, resblock_type="1", resblock_dilation_sizes=[[1, 3, 5]] * 3,
            resblock_kernel_sizes=[3, 7, 11], upsample_kernel_sizes=[16, 16, 4, 4], upsample_initial_channel=512,
            upsample_factors=[8, 8, 2, 2], inference_padding=0, cond_channels=256, conv_pre_weight_norm=False,
            conv_post_weight_norm=False, conv_post_bias=False)),
    }
    save("oracle_vs_reference_full_width", cases)


def _perturb_seeded(m, seed=0):
    gen = torch.Generator().manual_seed(seed)
    for _, p in m.named_parameters():
        if float(p.abs().sum()) == 0.0:
            p.data.copy_(torch.randn(p.shape, generator=gen) * 0.05)


@torch.no_grad()
def main_real_model():
    """The real Vits.inference / voice_conversion / forward_mas with a narrow decoder
    (tests/test_oracle_vs_reference_model.py); the test replays the same random draws for the oracle."""
    import dataclasses
    import types
    F = ref_import.load_full()
    base = dict(upsample_initial_channel_decoder=64, num_layers_text_encoder=2, hidden_channels_ffn_text_encoder=256)
    cases = {}

    def run(name, b, t, lens, seed, model_args=None, aux_extra=None, audio_sample_rate=None, attrs=None,
            language_manager=None):
        args = F["vits_model"].VitsArgs(**{**base, **(model_args or {})})
        cfg = F["vits_config"].VitsConfig()
        cfg.model_args = args
        cfg.__post_init__()
        if audio_sample_rate:
            cfg.audio.sample_rate = audio_sample_rate
        torch.manual_seed(seed)
        m = F["vits_model"].Vits(cfg, language_manager=language_manager).eval()
        _perturb_seeded(m, seed)
        for k, v in (attrs or {}).items():
            setattr(m, k, v)
        c = _regenerate(m, 100000 * seed)
        torch.manual_seed(seed + 100)
        tok = torch.randint(0, args.num_chars, (b, t))
        aux = {"x_lengths": lens, "d_vectors": None, "speaker_ids": None, "language_ids": None, "durations": None}
        aux.update(aux_extra or {})
        torch.manual_seed(seed + 1)
        want = m.inference(tok, aux_input=dict(aux))
        a = dataclasses.asdict(args)
        a["length_scale"] = m.length_scale
        a["max_inference_len"] = m.max_inference_len
        a["sample_rate"] = cfg.audio.sample_rate
        c.update({"args": a, "b": b, "t": t, "x_lengths": lens, "aux": aux_extra or {},
                  "out": {k: fixtures.record(v) for k, v in want.items()}})
        cases[name] = c

    run("single_speaker", 3, 17, torch.tensor([17, 9, 4]), 3)
    run("speaker_embedding_and_length_scale", 3, 12, torch.tensor([12, 7, 3]), 4,
        dict(use_speaker_embedding=True, num_speakers=11), {"speaker_ids": torch.tensor([10, 0, 4])},
        attrs={"length_scale": 1.6})
    torch.manual_seed(50)
    run("d_vectors", 2, 10, torch.tensor([10, 6]), 5, dict(use_d_vector_file=True, d_vector_dim=32),
        {"d_vectors": torch.randn(2, 32)})
    run("language_embedding", 2, 9, torch.tensor([9, 5]), 6,
        dict(use_language_embedding=True, num_languages=3, embedded_language_dim=4), {"language_ids": torch.tensor([2, 0])},
        language_manager=types.SimpleNamespace(num_languages=3))   # sizes emb_l like the LanguageManager (vits.py:795-799)
    run("deterministic_dp_and_max_inference_len", 2, 11, torch.tensor([11, 6]), 7,
        dict(use_sdp=False, use_speaker_embedding=True, num_speakers=4), {"speaker_ids": torch.tensor([1, 3])},
        attrs={"max_inference_len": 9})
    run("encoder_sample_rate", 2, 8, torch.tensor([8, 3]), 8,
        dict(encoder_sample_rate=11025, upsample_rates_decoder=[8, 8, 4, 2], upsample_kernel_sizes_decoder=[16, 16, 8, 4]),
        audio_sample_rate=22050)

    args = F["vits_model"].VitsArgs(**base, use_speaker_embedding=True, num_speakers=5)
    cfg = F["vits_config"].VitsConfig()
    cfg.model_args = args
    cfg.__post_init__()
    torch.manual_seed(9)
    m = F["vits_model"].Vits(cfg).eval()
    _perturb_seeded(m, 9)
    c = _regenerate(m, 900000)
    torch.manual_seed(19)
    y = torch.rand(1, 513, 14)
    torch.manual_seed(10)          # PosteriorEncoder: torch.randn_like(mean), networks.py:287
    o_hat, y_mask, (z, z_p, z_hat) = m.voice_conversion(y, torch.tensor([14]), 1, 4)
    c.update({"args": dataclasses.asdict(args), "out": [fixtures.record(t) for t in (o_hat, y_mask, z, z_p, z_hat)]})
    cases["voice_conversion"] = c

    args = F["vits_model"].VitsArgs(**base)
    cfg = F["vits_config"].VitsConfig()
    cfg.model_args = args
    cfg.__post_init__()
    torch.manual_seed(12)
    m = F["vits_model"].Vits(cfg).train()
    b, ch, tx, ty = 3, 192, 11, 47
    x_mask = seq_mask(torch.tensor([11, 7, 4]), tx)
    y_mask = seq_mask(torch.tensor([47, 30, 21]), ty)
    torch.manual_seed(13)
    z_p, m_p, logs_p = torch.randn(b, ch, ty), torch.randn(b, ch, tx), torch.randn(b, ch, tx) * 0.3
    x = torch.randn(b, ch, tx)
    _, attn = m.forward_mas({}, z_p, m_p, logs_p, x, x_mask, y_mask, g=None, lang_emb=None)
    cases["forward_mas"] = {"attn": fixtures.record(attn)}
    save("oracle_vs_reference_model", cases)


@torch.no_grad()
def main_reference_objects():
    """Answers of the reference's tokenizer / vocabulary, fairseq re-keying and vocoder config objects
    (tests/test_handoff_cpu.py)."""
    F = ref_import.load_full()
    vocab = list("_ abcdefghijklmnopqrstuvwxyz'!?") + ["<x>"]
    ref_v = F["characters"].BaseVocabulary(vocab, pad="_", blank=None, bos=None, eos=None)
    out = {"vocab": vocab, "ids": {n: getattr(ref_v, n) for n in ("pad_id", "blank_id", "bos_id", "eos_id", "num_chars")}}
    texts = ("What's  up?", "", "UPPER lower", "x")
    tok = {}
    for add_blank in (False, True):
        t = F["tokenizer"].TTSTokenizer(False, F["cleaners"].basic_cleaners, ref_v, None, add_blank=add_blank)
        tok[add_blank] = {"text_to_ids": [t.text_to_ids(x) for x in texts],
                          "intersperse_blank": t.intersperse_blank_char([1, 2, 3], True),
                          "intersperse_no_blank": t.intersperse_blank_char([1, 2], False),
                          "pad_with_bos_eos": t.pad_with_bos_eos([4, 5])}
    out.update({"texts": list(texts), "tokenizer": [tok[False], tok[True]]})

    import tempfile
    sys.path.insert(0, os.path.dirname(HERE))
    from test_handoff_cpu import _fake_fairseq_state
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "G_100000.pth")
        torch.save({"model": _fake_fairseq_state()}, p)
        out["fairseq"] = F["fairseq"].rehash_fairseq_vits_checkpoint(p)

    rc = F["hifigan_config"].HifiganConfig()
    ref_g = F["vocoder_models"].setup_generator(rc)
    ra = rc.audio
    out["hifigan_config"] = {
        "generator_model": rc.generator_model, "generator_model_params": rc.generator_model_params,
        "generator_state": [(k, tuple(v.shape)) for k, v in ref_g.state_dict().items()],
        "audio": {f: getattr(ra, f) for f in ("fft_size", "win_length", "hop_length", "sample_rate", "num_mels",
                                              "ref_level_db", "min_level_db", "signal_norm", "symmetric_norm",
                                              "max_norm", "clip_norm")}}
    save("reference_objects", out)


if __name__ == "__main__":
    main()
