"""Pins the oracle port against the UNMODIFIED reference modules at FULL model sizes, through the compact fixture
tests/golden/oracle_vs_reference_full_width.pt (tests/golden/make_golden.py ran the reference on the same regenerated
weights and the same seeded inputs; oracle/fixtures.py says what is stored)."""
import numpy as np
import pytest
import torch

import fixtures
import vits_oracle as O
from fixtures import check, state_from_stats


@pytest.fixture(autouse=True)
def _recorded_threads():
    yield from fixtures.recorded_threads()


@pytest.fixture(scope="module")
def F(golden):
    return golden("oracle_vs_reference_full_width")


def _state(c):
    return state_from_stats(c["stats"], c["seed"])


def _mask(lengths, t):
    return O.sequence_mask(torch.tensor(lengths), t).unsqueeze(1).float()


@torch.no_grad()
def test_hifigan_full_width(F):
    c = F["hifigan"]
    torch.manual_seed(10)
    x, g = torch.randn(1, 192, 6), torch.randn(1, 256, 1)
    check(O.hifigan_forward(_state(c), x, g), c["y"], "waveform")


@torch.no_grad()
def test_vits_stack_full_width(F):
    c = F["vits_stack"]
    torch.manual_seed(11)
    tok, lens = torch.randint(0, 100, (3, 21)), torch.tensor([21, 13, 5])
    got = O.text_encoder(_state(c["text_encoder"]), tok, lens)
    for i, (a, b) in enumerate(zip(got, c["text_encoder_out"])):
        check(a, b, f"text_encoder[{i}]")
    torch.manual_seed(12)
    g = torch.randn(3, 256, 1)
    torch.manual_seed(9)
    noise = torch.randn(3, 2, 21)
    check(O.sdp_reverse(_state(c["sdp"]), got[0], got[3], noise, g=g), c["logw"], "logw")
    torch.manual_seed(13)
    z = torch.randn(3, 192, 40)
    check(O.flow_forward(_state(c["flow"]), z, _mask([40, 22, 3], 40), g, reverse=True), c["flow_out"], "flow")


def test_mas_cfg4_shape_against_compiled_reference(F):
    rng = np.random.RandomState(0)
    v = torch.from_numpy(rng.randn(8, 200, 1000).astype(np.float32))
    t_x = torch.from_numpy(rng.randint(100, 201, size=8))
    t_y = torch.tensor([int(rng.randint(5 * int(a) if 5 * int(a) <= 1000 else 1000, 1001)) for a in t_x])
    mask = ((torch.arange(200)[None, :, None] < t_x[:, None, None]) &
            (torch.arange(1000)[None, None, :] < t_y[:, None, None])).float()
    check(O.maximum_path(v, mask, impl="c"), F["mas_cfg4"]["path"], "c port")
    check(O.maximum_path(v, mask, impl="py"), F["mas_cfg4"]["path"], "python port")


@torch.no_grad()
def test_voice_conversion_stack_full_width(F):
    """Posterior encoder, flow forward and the deterministic duration predictor at VITS width vs the reference."""
    c = F["voice_conversion_stack"]
    torch.manual_seed(14)
    y, g = torch.randn(2, 513, 33).abs(), torch.randn(2, 256, 1)
    lens = torch.tensor([33, 12])
    torch.manual_seed(5)
    noise = torch.randn(2, 192, 33)
    got = O.posterior_encoder(_state(c["posterior"]), y, lens, g=g, noise=noise)
    for i, (a, b) in enumerate(zip(got, c["posterior_out"])):
        check(a, b, f"posterior_encoder[{i}]")
    check(O.flow_forward(_state(c["flow"]), got[0], got[3], g, reverse=False), c["flow_out"], "flow")
    torch.manual_seed(15)
    x = torch.randn(2, 192, 17)
    logw = O.duration_predictor(_state(c["dp"]), x, _mask([17, 6], 17), g=g)
    assert torch.allclose(logw, c["dp_out"], atol=1e-6, rtol=0)


def test_drop_in_state_dict_keys_match_reference(F):
    """The Python mirror must load reference checkpoints unchanged: same state_dict keys and shapes."""
    from tts_b200 import layers as L
    from tts_b200.hifigan import HifiganGenerator

    def keys(m):
        return {k: tuple(v.shape) for k, v in m.state_dict().items()}

    ours = {
        "TextEncoder": L.TextEncoder(50, 192, 192, 768, 2, 6, 3, 0.1, language_emb_dim=4),
        "ResidualCouplingBlocks": L.ResidualCouplingBlocks(192, 192, 5, 1, 4, cond_channels=256),
        "PosteriorEncoder": L.PosteriorEncoder(513, 192, 192, 5, 1, 16, cond_channels=256),
        "StochasticDurationPredictor": L.StochasticDurationPredictor(192, 192, 3, 0.5, 4, cond_channels=256,
                                                                     language_emb_dim=4),
        "DurationPredictor": L.DurationPredictor(192, 256, 3, 0.5, cond_channels=256, language_emb_dim=4),
        "HifiganGenerator": HifiganGenerator(
            in_channels=192, out_channels=1, resblock_type="1", resblock_dilation_sizes=[[1, 3, 5]] * 3,
            resblock_kernel_sizes=[3, 7, 11], upsample_kernel_sizes=[16, 16, 4, 4], upsample_initial_channel=512,
            upsample_factors=[8, 8, 2, 2], inference_padding=0, cond_channels=256, conv_pre_weight_norm=False,
            conv_post_weight_norm=False, conv_post_bias=False),
    }
    assert set(ours) == set(F["state_dict_keys"])
    for name, m in ours.items():
        assert keys(m) == F["state_dict_keys"][name], name
