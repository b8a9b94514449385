"""Pins the oracle's restated ``Vits.inference`` glue (oracle/vits_oracle.py: vits_inference, voice_conversion) against
the REAL, unmodified reference model class ``TTS.tts.models.vits.Vits``: same weights, same random draws,
``torch.equal`` on every output of the reference's 8-key dict.  The reference's answers come from the compact fixture
tests/golden/oracle_vs_reference_model.pt (tests/golden/make_golden.py; oracle/fixtures.py says what is stored)."""
import pytest
import torch

import fixtures
import vits_oracle as O
from fixtures import check, state_from_stats


@pytest.fixture(autouse=True)
def _recorded_threads():
    yield from fixtures.recorded_threads()


KEYS = ("model_outputs", "alignments", "durations", "z", "z_p", "m_p", "logs_p", "y_mask")


def _run(golden, name, seed):
    c = golden("oracle_vs_reference_model")[name]
    a, b, t = c["args"], c["b"], c["t"]
    torch.manual_seed(seed + 100)
    tok = torch.randint(0, a["num_chars"], (b, t))
    # the reference draws the SDP noise first (stochastic_duration_predictor.py:287, CPU generator), then
    # randn_like(m_p) (vits.py:1155): replay the same stream for the oracle
    torch.manual_seed(seed + 1)
    sdp_noise = torch.randn(b, 2, t) if a["use_sdp"] else None
    # m_p is a transposed view there ([B,T,C] storage seen as [B,C,T]); randn_like keeps the strides and a non-contiguous
    # CPU normal_() takes the serial sampler, not the vectorised fill: replay with the same call on the same layout
    got = O.vits_inference(state_from_stats(c["stats"], c["seed"]), tok, c["x_lengths"], sdp_noise,
                           lambda s: torch.randn_like(torch.empty(s[0], s[2], s[1]).transpose(1, 2)), args=a,
                           speaker_ids=c["aux"].get("speaker_ids"), d_vectors=c["aux"].get("d_vectors"),
                           language_ids=c["aux"].get("language_ids"))
    assert set(c["out"]) == set(KEYS)
    for k in KEYS:
        check(got[k], c["out"][k], k)
    return got


@torch.no_grad()
def test_single_speaker_glue_bit_exact(golden):
    out = _run(golden, "single_speaker", 3)
    assert out["model_outputs"].shape[-1] == out["y_mask"].shape[-1] * 256


@torch.no_grad()
def test_speaker_embedding_and_length_scale(golden):
    _run(golden, "speaker_embedding_and_length_scale", 4)


@torch.no_grad()
def test_d_vectors(golden):
    _run(golden, "d_vectors", 5)


@torch.no_grad()
def test_language_embedding(golden):
    _run(golden, "language_embedding", 6)


@torch.no_grad()
def test_deterministic_duration_predictor_and_max_inference_len(golden):
    _run(golden, "deterministic_dp_and_max_inference_len", 7)


@torch.no_grad()
def test_encoder_sample_rate_upsampling(golden):
    _run(golden, "encoder_sample_rate", 8)


@torch.no_grad()
def test_voice_conversion_glue_bit_exact(golden):
    c = golden("oracle_vs_reference_model")["voice_conversion"]
    torch.manual_seed(19)
    y = torch.rand(1, 513, 14)
    torch.manual_seed(10)
    noise = torch.randn(1, 192, 14)       # PosteriorEncoder: torch.randn_like(mean), networks.py:287
    sd = state_from_stats(c["stats"], c["seed"])
    # the reference embeds `speaker_cond` as emb_g(tensor(id).unsqueeze(0)) (vits.py:1216-1217): one utterance, scalar ids
    g = lambda i: torch.nn.functional.embedding(torch.tensor([i]), sd["emb_g.weight"]).unsqueeze(-1)
    go, gm, (gz, gzp, gzh) = O.voice_conversion(sd, y, torch.tensor([14]), g(1), g(4), noise, args=c["args"])
    for i, a in enumerate((go, gm, gz, gzp, gzh)):
        check(a, c["out"][i], ("o_hat", "y_mask", "z", "z_p", "z_hat")[i])


@torch.no_grad()
def test_forward_mas_alignment_vs_real_model(golden):
    """Vits.forward_mas (vits.py:909-919) on the real model class: the oracle's logp / attn restatement is bit-exact
    (the real maximum_path ran the reference's compiled Cython kernel)."""
    want = golden("oracle_vs_reference_model")["forward_mas"]["attn"]
    b, c, tx, ty = 3, 192, 11, 47
    x_mask = O.sequence_mask(torch.tensor([11, 7, 4]), tx).unsqueeze(1).float()
    y_mask = O.sequence_mask(torch.tensor([47, 30, 21]), ty).unsqueeze(1).float()
    torch.manual_seed(13)
    z_p, m_p, logs_p = torch.randn(b, c, ty), torch.randn(b, c, tx), torch.randn(b, c, tx) * 0.3
    for impl in ("c", "py"):
        got, _ = O.forward_mas_attn(z_p, m_p, logs_p, x_mask, y_mask, impl=impl)
        check(got, want, impl)
