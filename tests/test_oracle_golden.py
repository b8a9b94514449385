"""Pins oracle/vits_oracle.py (+ the C MAS port) against fixtures produced by the unmodified reference
(tests/golden/make_golden.py).  Bit-exact on CPU: the oracle issues the same torch ops."""
import numpy as np
import pytest
import torch

import fixtures
import vits_oracle as O


@pytest.fixture(autouse=True)
def _recorded_threads():
    yield from fixtures.recorded_threads()


def test_hifigan_v1_small(golden):
    g = golden("hifigan_v1_small")
    a = g["args"]
    kw = dict(upsample_factors=a["upsample_factors"], upsample_kernel_sizes=a["upsample_kernel_sizes"],
              resblock_kernel_sizes=a["resblock_kernel_sizes"], resblock_dilation_sizes=a["resblock_dilation_sizes"],
              resblock_type=a["resblock_type"])
    assert torch.equal(O.hifigan_forward(g["state"], g["x"], **kw), g["y"])
    assert torch.equal(O.hifigan_inference(g["state"], g["x"], **kw), g["y_inference"])
    assert g["y"].shape == (2, 1, 13 * 256)  # length contract (tests/tts_tests2/test_delightful_tts_layers.py:89)


def test_hifigan_cond_resblock2(golden):
    g = golden("hifigan_cond_rb2_small")
    a = g["args"]
    y = O.hifigan_forward(g["state"], g["x"], g["g"], upsample_factors=a["upsample_factors"],
                          upsample_kernel_sizes=a["upsample_kernel_sizes"],
                          resblock_kernel_sizes=a["resblock_kernel_sizes"],
                          resblock_dilation_sizes=a["resblock_dilation_sizes"], resblock_type="2")
    assert torch.equal(y, g["y"])


def test_flow(golden):
    g = golden("flow_small")
    a = g["args"]
    kw = dict(num_flows=a["num_flows"], hidden=a["hidden_channels"], kernel_size=a["kernel_size"],
              dilation_rate=a["dilation_rate"], num_layers=a["num_layers"])
    assert torch.equal(O.flow_forward(g["state"], g["z"], g["mask"], g["g"], reverse=True, **kw), g["rev"])
    assert torch.equal(O.flow_forward(g["state"], g["z"], g["mask"], g["g"], reverse=False, **kw), g["fwd"])


def test_text_encoder(golden):
    g = golden("text_encoder_small")
    a = g["args"]
    x, m, logs, mask = O.text_encoder(g["state"], g["tokens"], g["lengths"], hidden=a["hidden_channels"],
                                      out_channels=a["out_channels"], num_heads=a["num_heads"],
                                      num_layers=a["num_layers"], kernel_size=a["kernel_size"])
    for got, key in ((x, "x"), (m, "m_p"), (logs, "logs_p"), (mask, "x_mask")):
        assert torch.allclose(got, g[key], atol=1e-6, rtol=0), key


def test_sdp_reverse(golden):
    g = golden("sdp_small")
    a = g["args"]
    logw = O.sdp_reverse(g["state"], g["x"], g["x_mask"], g["noise"], g=g["g"], noise_scale=g["noise_scale"],
                         hidden=a["hidden_channels"], kernel_size=a["kernel_size"], num_flows=a["num_flows"])
    assert torch.allclose(logw, g["logw"], atol=1e-6, rtol=0)


def test_posterior_encoder(golden):
    g = golden("posterior_small")
    a = g["args"]
    z, mean, logs, mask = O.posterior_encoder(g["state"], g["y"], g["y_lengths"], g=g["g"], noise=g["noise"],
                                              out_channels=a["out_channels"], hidden=a["hidden_channels"],
                                              kernel_size=a["kernel_size"], dilation_rate=a["dilation_rate"],
                                              num_layers=a["num_layers"])
    for got, key in ((z, "z"), (mean, "mean"), (logs, "log_scale"), (mask, "y_mask")):
        assert torch.equal(got, g[key]), key


def test_deterministic_duration_predictor(golden):
    g = golden("duration_predictor_small")
    logw = O.duration_predictor(g["state"], g["x"], g["x_mask"], g=g["g"], lang_emb=g["lang_emb"])
    assert torch.allclose(logw, g["logw"], atol=1e-6, rtol=0)
    assert logw.shape == (4, 1, 23)


def test_voice_conversion_chain(golden):
    """The restated Vits.voice_conversion glue (vits.py:1226-1232) against the same chain run on reference modules."""
    g = golden("vc_small")
    o, mask, (z, z_p, z_hat) = O.voice_conversion(g["state"], g["y"], g["y_lengths"], g["g_src"], g["g_tgt"], g["noise"],
                                                   args=g["args"])
    assert torch.equal(mask, g["y_mask"])
    for got, key in ((z, "z"), (z_p, "z_p"), (z_hat, "z_hat"), (o, "o_hat")):
        assert torch.equal(got, g[key]), key


def test_mas_ports_match_reference_kernel(golden):
    for case in golden("mas_cases")["cases"]:
        for impl in ("c", "py"):
            got = O.maximum_path(case["value"], case["mask"], impl=impl)
            assert torch.equal(got, case["path"]), impl
        # structural invariants the reference pins (tests/tts_tests/test_vits.py:164-165)
        assert case["path"].max() == 1 and case["path"].min() == 0


def test_generate_path(golden):
    g = golden("generate_path")
    assert torch.equal(O.generate_path(g["duration"], g["mask"]), g["path"])
    # tests/tts_tests/test_helpers.py:71-88: each token owns exactly `duration` consecutive frames
    dur, path = g["duration"], g["path"]
    for b in range(dur.shape[0]):
        cur = 0
        for t in range(dur.shape[1]):
            d = int(dur[b, t])
            assert path[b, t, cur:cur + d].sum() == d and path[b, t].sum() == d
            cur += d


def test_mel_basis_matches_torchaudio_slaney():
    import torchaudio

    mb = O.slaney_mel_basis(22050, 1024, 80, 0, None)
    tb = torchaudio.functional.melscale_fbanks(513, 0.0, 11025.0, 80, 22050, norm="slaney", mel_scale="slaney").T
    assert mb.shape == (80, 513)
    assert np.abs(mb - tb.numpy()).max() < 1e-6


def test_wav_to_mel_is_spec_to_mel_of_wav_to_spec():
    # the one relation the reference pins for the front end (tests/tts_tests/test_vits.py:56)
    torch.manual_seed(0)
    wav = torch.rand(2, 1, 8192) * 2 - 1
    spec = O.wav_to_spec(wav, 1024, 256, 1024)
    assert spec.shape == (2, 513, 32)
    mel = O.wav_to_mel(wav, 1024, 80, 22050, 256, 1024, 0, None)
    assert torch.equal(mel, O.spec_to_mel(spec, 1024, 80, 22050, 0, None))
