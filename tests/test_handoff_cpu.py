"""Host-side widening of the path (SURVEY 8 f3 / f4), CPU only: tokenizer hand-off, fairseq checkpoint re-keying,
HifiganConfig / setup_generator / GAN surface, and the oracle's restated vocoder hand-off -- each against the committed
golden vectors (produced by the real reference, tests/golden/make_golden.py), including the recorded answers of the
reference objects themselves (tests/golden/reference_objects.pt)."""
import numpy as np
import pytest
import torch

import fixtures
import vits_oracle as O


@pytest.fixture(autouse=True)
def _recorded_threads():
    yield from fixtures.recorded_threads()


# ----------------------------------------------------------------------------- tokenizer
def _tokenizer(g, add_blank, bos):
    from tts_b200.text import BaseCharacters, TTSTokenizer, basic_cleaners
    chars = BaseCharacters(g["characters"], g["punctuations"], pad=g["pad"], eos=g["eos"], bos=g["bos"], blank=g["blank"])
    return TTSTokenizer(False, basic_cleaners, chars, None, add_blank=add_blank, use_eos_bos=bos), chars


def test_tokenizer_matches_reference_golden(golden, capsys):
    gd = golden("tokenizer_cases")
    for case in gd["cases"]:
        tok, chars = _tokenizer(gd["graphemes"], case["add_blank"], case["use_eos_bos"])
        assert list(chars.vocab) == gd["vocab"]
        one_by_one = [tok.text_to_ids(t) for t in gd["texts"]]
        assert one_by_one == case["ids"]
        block, lens = tok.batch_text_to_ids(gd["texts"], pin_memory=False)
        assert lens.tolist() == [len(i) for i in case["ids"]]
        for r, ids in enumerate(case["ids"]):
            assert block[r, : len(ids)].tolist() == ids
            assert (block[r, len(ids):] == chars.pad_id).all()
    capsys.readouterr()
    tok, _ = _tokenizer(gd["graphemes"], True, False)
    assert tok.decode(tok.encode("abc")) == "abc"
    assert "ü" in tok.not_found_characters or tok.text_to_ids("ü") == [tok.characters.blank_id]   # unknown chars are dropped


def test_tokenizer_and_vocabulary_vs_reference_objects(golden, capsys):
    from tts_b200.text import BaseVocabulary, TTSTokenizer, basic_cleaners
    ref = golden("reference_objects")
    my_v = BaseVocabulary(ref["vocab"], pad="_")
    for name, want in ref["ids"].items():
        assert getattr(my_v, name) == want, name
    for add_blank, want in zip((False, True), ref["tokenizer"]):
        my_t = TTSTokenizer(False, basic_cleaners, my_v, None, add_blank=add_blank)
        assert [my_t.text_to_ids(text) for text in ref["texts"]] == want["text_to_ids"]
        assert my_t.intersperse_blank_char([1, 2, 3], True) == want["intersperse_blank"]
        assert my_t.intersperse_blank_char([1, 2], False) == want["intersperse_no_blank"]
        assert my_t.pad_with_bos_eos([4, 5]) == want["pad_with_bos_eos"]
    capsys.readouterr()


# ----------------------------------------------------------------------------- fairseq checkpoints
def _fake_fairseq_state():
    keys = ["enc_p.emb.weight", "enc_p.encoder.attn_layers.0.conv_q.weight", "dec.conv_pre.weight", "dec.ups.0.weight_g",
            "enc_q.pre.weight", "enc_q.enc.in_layers.3.weight_v", "flow.flows.0.pre.weight", "flow.flows.2.enc.in_layers.1.bias",
            "flow.flows.4.post.bias", "flow.flows.6.pre.bias", "dp.flows.0.m", "dp.flows.0.logs", "dp.flows.1.pre.weight",
            "dp.flows.3.convs.convs_sep.0.weight", "dp.flows.5.proj.bias", "dp.flows.7.pre.bias", "dp.post_flows.0.m",
            "dp.post_flows.0.logs", "dp.post_flows.1.proj.weight", "dp.post_flows.3.pre.bias", "dp.post_flows.5.pre.bias",
            "dp.post_flows.7.pre.bias", "dp.pre.weight", "dp.convs.norms_1.0.gamma", "dp.post_pre.bias", "emb_g.weight"]
    return {k: torch.full((1,), float(i)) for i, k in enumerate(keys)}


def test_fairseq_rekeying(tmp_path, golden):
    from tts_b200.text import rehash_fairseq_vits_checkpoint
    sd = _fake_fairseq_state()
    p = tmp_path / "G_100000.pth"
    torch.save({"model": sd}, p)
    got = rehash_fairseq_vits_checkpoint(str(p))
    want_names = {
        "enc_p.emb.weight": "text_encoder.emb.weight", "dec.ups.0.weight_g": "waveform_decoder.ups.0.weight_g",
        "enc_q.enc.in_layers.3.weight_v": "posterior_encoder.enc.in_layers.3.weight_v",
        "flow.flows.0.pre.weight": "flow.flows.0.pre.weight", "flow.flows.2.enc.in_layers.1.bias": "flow.flows.1.enc.in_layers.1.bias",
        "flow.flows.4.post.bias": "flow.flows.2.post.bias", "flow.flows.6.pre.bias": "flow.flows.3.pre.bias",
        "dp.flows.0.m": "duration_predictor.flows.0.translation", "dp.flows.0.logs": "duration_predictor.flows.0.log_scale",
        "dp.flows.1.pre.weight": "duration_predictor.flows.1.pre.weight", "dp.flows.3.convs.convs_sep.0.weight": "duration_predictor.flows.2.convs.convs_sep.0.weight",
        "dp.flows.5.proj.bias": "duration_predictor.flows.3.proj.bias", "dp.flows.7.pre.bias": "duration_predictor.flows.4.pre.bias",
        "dp.post_flows.0.m": "duration_predictor.post_flows.0.translation", "dp.post_flows.7.pre.bias": "duration_predictor.post_flows.4.pre.bias",
        "dp.pre.weight": "duration_predictor.pre.weight", "dp.post_pre.bias": "duration_predictor.post_pre.bias", "emb_g.weight": "emb_g.weight"}
    for old, new in want_names.items():
        assert new in got and torch.equal(got[new], sd[old]), (old, new)
    assert len(got) == len(sd)
    ref = golden("reference_objects")["fairseq"]
    assert set(ref.keys()) == set(got.keys())
    for k in ref:
        assert torch.equal(ref[k], got[k])


def test_fairseq_vocab_and_tokenizer(tmp_path):
    from tts_b200.text import FairseqVocab, TTSTokenizer, basic_cleaners
    p = tmp_path / "vocab.txt"
    p.write_text("_\na\nb\n \nc\n", encoding="utf-8")
    v = FairseqVocab(str(p))
    assert v.blank == "_" and v.pad == " " and v.num_chars == 5 and v.blank_id == 0 and v.pad_id == 3
    t = TTSTokenizer(False, basic_cleaners, v, None, add_blank=True, use_eos_bos=False)
    assert t.text_to_ids("AB c") == [0, 1, 0, 2, 0, 3, 0, 4, 0]


# ----------------------------------------------------------------------------- vocoder config surface
def test_hifigan_config_and_setup_generator_surface(golden):
    from tts_b200.vocoder import GAN, BaseAudioConfig, HifiganConfig, setup_generator, to_camel
    c = HifiganConfig()
    assert c.generator_model == "hifigan_generator" and c["generator_model_params"]["upsample_factors"] == [8, 8, 2, 2]
    assert to_camel("hifigan_generator") == "HifiganGenerator"
    g = setup_generator(c)
    assert type(g).__name__ == "HifiganGenerator" and g._cfg["in_channels"] == c.audio.num_mels == 80
    assert g.inference_padding == 5
    gan = GAN(c)
    assert set(k.split(".")[0] for k in gan.state_dict()) == {"model_g"}
    with pytest.raises(NotImplementedError):
        setup_generator(HifiganConfig(generator_model="melgan_generator"))
    rc = golden("reference_objects")["hifigan_config"]
    assert rc["generator_model_params"] == c.generator_model_params and rc["generator_model"] == c.generator_model
    assert rc["generator_state"] == [(k, tuple(v.shape)) for k, v in g.state_dict().items()]
    for f, want in rc["audio"].items():
        assert getattr(BaseAudioConfig(), f) == want, f


# ----------------------------------------------------------------------------- oracle hand-off vs golden / reference
def test_oracle_normalize_denormalize_vs_reference_golden(golden):
    gd = golden("vocoder_handoff")
    for case in gd["normalize_cases"]:
        kw = {k: (v.numpy() if torch.is_tensor(v) else v) for k, v in case["kw"].items()}
        n = O.audio_normalize(case["S"].numpy(), **kw)
        assert np.array_equal(n, case["normalized"].numpy()), case["kw"]
        d = O.audio_denormalize(case["denorm_input"].numpy(), **kw)
        assert np.array_equal(d, case["denormalized"].numpy()), case["kw"]
    for case in gd["interpolate_cases"]:
        assert torch.equal(O.interpolate_vocoder_input([1, case["scale"]], case["spec"].numpy()), case["out"])
    ch = gd["chain"]
    out = O.vocoder_handoff(ch["mel_tc"].numpy(), ch["tts_kw"], ch["voc_kw"], ch["sr_tts"], ch["sr_voc"], 5)
    assert torch.equal(out, ch["out"])
    assert np.array_equal(O.wav_to_int16(gd["wav"].numpy()), gd["wav_int16"].numpy())


def test_real_model_fixture_matches_oracle(golden):
    """The fixture produced by the REAL Vits.inference (multi-speaker, narrow) replays bit-exactly through the oracle --
    on the GPU box this is what ties the product to the reference model class itself."""
    g = golden("vits_real_model_small")
    got = O.vits_inference(g["state"], g["tokens"], g["x_lengths"], g["sdp_noise"], lambda s: g["prior_noise"],
                           args=g["args"], speaker_ids=g["speaker_ids"])
    for k, v in g["out"].items():
        assert torch.equal(got[k], v), k
