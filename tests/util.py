import os

import torch


def rel_fro(a: torch.Tensor, b: torch.Tensor) -> float:
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def max_rel(a: torch.Tensor, b: torch.Tensor) -> float:
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def mismatch_fraction(a: torch.Tensor, b: torch.Tensor) -> float:
    return float((a.detach().cpu() != b.detach().cpu()).float().mean())


def seeded(seed: int) -> torch.Generator:
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    return g


def randn_bf16(shape, gen, scale=1.0):
    return (torch.randn(shape, generator=gen) * scale).to(torch.bfloat16)


# ---- outputs of the reference's own code, recorded once and stored in tests/golden/ref_recorded.pt ----
RECORDED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_recorded.pt")
_recorded = None


def recording() -> bool:
    """LV_RECORD_GOLDEN=1: run the reference (oracle/ref_loader.py, where its sources are mounted) and store what it
    returns, instead of reading the stored values."""
    return os.environ.get("LV_RECORD_GOLDEN") == "1"


def recorded(key: str, compute, store: bool = True):
    """The stored output of the reference's own code under `key`.  When recording, `compute()` runs the reference and
    its result replaces the stored value (written at once unless `store` is False, e.g. on all but one rank)."""
    global _recorded
    if _recorded is None:
        _recorded = torch.load(RECORDED) if os.path.exists(RECORDED) else {}
    if recording():
        from oracle import ref_loader

        assert ref_loader.available(), "LV_RECORD_GOLDEN=1 needs the reference sources (oracle/ref_loader.py)"
        value = compute()
        if store:
            _recorded = torch.load(RECORDED) if os.path.exists(RECORDED) else {}
            _recorded[key] = value
            torch.save(_recorded, RECORDED)
        return value
    assert key in _recorded, f"{key} is not in {RECORDED}: record it with LV_RECORD_GOLDEN=1"
    return _recorded[key]


def digest(t) -> tuple:
    """(shape, dtype, sha256 of the bytes) - for a bit-exact comparison with an output too large to store.
    -0.0 is folded into +0.0, as torch.equal / numpy.array_equal do."""
    import hashlib

    import numpy as np

    if torch.is_tensor(t):
        t = t.detach().cpu().contiguous()
        if t.is_floating_point():
            t = t + 0.0
        b = t.view(torch.uint8).numpy().tobytes() if t.numel() else b""
        return tuple(t.shape), str(t.dtype), hashlib.sha256(b).hexdigest()
    a = np.ascontiguousarray(t)
    if a.dtype.kind == "f":
        a = a + a.dtype.type(0)
    return tuple(a.shape), str(a.dtype), hashlib.sha256(a.tobytes()).hexdigest()
