"""The `precision` setting of the HiFiGAN generator and of FusedConv1d, on the host side: default, validation, state_dict
and persistence.  Nothing here needs a GPU or the CUDA library."""
import pytest
import torch

from tts_b200 import _lib
from tts_b200.conv import FusedConv1d
from tts_b200.hifigan import HifiganGenerator


def _small_generator():
    return HifiganGenerator(32, 1, "1", [[1, 3, 5]] * 3, [3, 7, 11], [16, 16, 4, 4], 64, [8, 8, 2, 2],
                            inference_padding=0)


@pytest.fixture
def no_cuda_library(monkeypatch):
    """Any attempt to load libtts_b200.so fails the test."""
    def refuse():
        raise AssertionError("the CUDA library was loaded")
    monkeypatch.setattr(_lib, "lib", refuse)


def test_default_is_fp32_and_only_known_values_are_accepted(no_cuda_library):
    m = _small_generator()
    assert m.precision == "fp32"
    m.precision = "tf32"
    assert m.precision == "tf32"
    for bad in ("TF32", "bf16", "fp16", "", None, 1):
        with pytest.raises(ValueError):
            m.precision = bad
    assert m.precision == "tf32"
    m.precision = "fp32"
    assert m.precision == "fp32"


def test_fused_conv_precision_is_validated(no_cuda_library):
    w = torch.randn(128, 8, 1)
    assert FusedConv1d(w).precision == "fp32"
    assert FusedConv1d(w, precision="tf32").precision == "tf32"
    with pytest.raises(ValueError):
        FusedConv1d(w, precision="half")


def test_state_dict_keys_do_not_depend_on_the_mode(no_cuda_library):
    a, b = _small_generator(), _small_generator()
    b.precision = "tf32"
    assert list(a.state_dict().keys()) == list(b.state_dict().keys())
    assert "precision" not in dict(b.named_parameters()) and "precision" not in dict(b.named_buffers())
    b.load_state_dict(a.state_dict())                     # a checkpoint from either mode loads into the other
    assert b.precision == "tf32"


def test_mode_survives_apply_checkpoints_and_weight_norm_removal(tmp_path, no_cuda_library):
    m = _small_generator()
    m.precision = "tf32"
    m.float()
    m.to("cpu")
    assert m.precision == "tf32"
    p = tmp_path / "g.pth"
    torch.save({"model": _small_generator().state_dict()}, p)
    m.load_checkpoint({}, str(p))
    assert m.precision == "tf32"
    m.load_checkpoint({}, str(p), eval=True)              # eval=True also removes the weight norm
    assert m.precision == "tf32" and not m.training
    m.repack()
    assert m.precision == "tf32"


def test_mode_reaches_every_wrapper(no_cuda_library):
    from tts_b200.vits import Vits, VitsConfig
    from tts_b200.vocoder import GAN

    v = Vits(VitsConfig())
    assert v.waveform_decoder.precision == "fp32"
    v.waveform_decoder.precision = "tf32"
    v.repack()
    assert v.waveform_decoder.precision == "tf32"
    cfg = {"generator_model": "hifigan_generator", "audio": {"num_mels": 80},
           "generator_model_params": dict(resblock_type="1", resblock_dilation_sizes=[[1, 3, 5]] * 3,
                                          resblock_kernel_sizes=[3, 7, 11], upsample_kernel_sizes=[16, 16, 4, 4],
                                          upsample_initial_channel=64, upsample_factors=[8, 8, 2, 2])}
    gan = GAN(cfg)
    gan.model_g.precision = "tf32"
    assert gan.model_g.precision == "tf32"
