"""TEST INFRASTRUCTURE ONLY -- compact golden fixtures for the full-width comparisons with the reference.

Full-width weights and outputs are far too large to commit, so a fixture stores instead:
  * for every state_dict entry its shape and the mean / std of the reference module's own initialisation;
    ``state_from_stats`` regenerates the weights from a seed (the fixture was produced by loading exactly these
    regenerated weights into the reference module, so reference and oracle see the same numbers);
  * every small output tensor in full, every large one as its SHA-256 (bit-exact check) plus a fixed, seeded sample
    of its values (so a mismatch reports how far off it is).
"""
import hashlib
import json
import zlib

import torch

FULL_LIMIT = 512       # outputs up to this many elements are stored in full
SAMPLE = 128
# Every fixture under tests/golden was recorded with this many intra-op threads.  The summation order of torch's CPU
# convolutions depends on the thread count, so comparing bit for bit with a fixture needs the same count on any host.
THREADS = 8


def recorded_threads():
    """Body of a pytest fixture: runs the test with THREADS intra-op threads, then restores the previous count."""
    old = torch.get_num_threads()
    torch.set_num_threads(THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(old)


def state_stats(sd):
    """Shape, mean and std (4 significant digits) of every entry, as zlib-compressed JSON in a uint8 tensor."""
    assert all(v.is_floating_point() for v in sd.values())
    stats = [[k, list(v.shape), float(f"{float(v.double().mean()):.4g}"),
              float(f"{float(v.double().std()):.4g}") if v.numel() > 1 else 0.0] for k, v in sd.items()]
    return torch.frombuffer(bytearray(zlib.compress(json.dumps(stats).encode(), 9)), dtype=torch.uint8)


def state_from_stats(blob, seed):
    """Deterministic float32 weights with the recorded per-entry mean / std (entry i draws from seed + i)."""
    sd = {}
    for i, (k, shape, mean, std) in enumerate(json.loads(zlib.decompress(blob.numpy().tobytes()))):
        gen = torch.Generator().manual_seed(seed + i)
        sd[k] = (torch.randn(shape, generator=gen, dtype=torch.float64) * std + mean).float()
    return sd


def _digest(t):
    t = t.detach().contiguous().cpu()
    return hashlib.sha256(t.numpy().tobytes()).hexdigest()


def _sample_index(numel):
    gen = torch.Generator().manual_seed(numel)
    return torch.randperm(numel, generator=gen)[:SAMPLE].sort().values


def record(t):
    """What a fixture keeps of one output tensor."""
    t = t.detach().contiguous().cpu()
    if t.numel() <= FULL_LIMIT:
        return t.clone()
    idx = _sample_index(t.numel())
    return {"shape": tuple(t.shape), "dtype": str(t.dtype), "sha256": _digest(t), "sample": t.reshape(-1)[idx].clone()}


def check(got, rec, name=""):
    """Asserts ``got`` is bit-identical to the recorded tensor."""
    got = got.detach().contiguous().cpu()
    if torch.is_tensor(rec):
        assert got.shape == rec.shape and got.dtype == rec.dtype, (name, got.shape, got.dtype, rec.shape, rec.dtype)
        assert torch.equal(got, rec), (name, float((got.double() - rec.double()).abs().max()))
        return
    assert tuple(got.shape) == rec["shape"] and str(got.dtype) == rec["dtype"], (name, got.shape, got.dtype, rec["shape"])
    sample = got.reshape(-1)[_sample_index(got.numel())]
    assert torch.equal(sample, rec["sample"]), (name, float((sample.double() - rec["sample"].double()).abs().max()))
    assert _digest(got) == rec["sha256"], (name, "sampled values agree, full tensor differs")
