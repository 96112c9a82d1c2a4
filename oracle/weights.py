"""ORACLE (test infrastructure): deterministic, name-keyed random initialisation.

No pretrained checkpoints are available offline (SURVEY.md section 8c), so parity work uses seeded random weights.
Every parameter is filled from a generator seeded by crc32(parameter name) so that the reference classes, the oracle
and the CUDA modules -- which may construct their sub-modules in different orders -- receive identical values for
identical state-dict keys.  Zero-initialised convolutions (``zero_module``) are overwritten too, otherwise a random
ControlNet outputs exactly 0 and nothing downstream is exercised.
"""
from __future__ import annotations

import zlib

import torch


def _std_for(name: str, p: torch.Tensor) -> float:
    if p.dim() >= 2:
        fan_in = p[0].numel()
        return 1.0 / (fan_in ** 0.5)
    return 0.1


@torch.no_grad()
def seeded_init_(module: torch.nn.Module, seed: int = 0) -> torch.nn.Module:
    for name, p in sorted(module.named_parameters(), key=lambda kv: kv[0]):
        # CPU parameters use the CPU generator (the stream the committed golden vectors were produced with);
        # parameters that already live on a GPU are filled there (GPU-only parity tests: much faster for 10^9 weights,
        # both sides of those tests share the values through a state_dict copy)
        g = torch.Generator(device=p.device if p.is_cuda else "cpu")
        g.manual_seed((zlib.crc32(name.encode()) + 7919 * seed) & 0x7FFFFFFF)
        v = torch.randn(p.shape, generator=g, dtype=torch.float32, device=p.device if p.is_cuda else "cpu")
        leaf = name.rsplit(".", 1)[-1]
        is_norm_weight = leaf == "weight" and p.dim() == 1
        if name.endswith("mix_factor"):
            v = v * 0.5
        elif is_norm_weight:
            v = 1.0 + 0.1 * v
        else:
            v = v * _std_for(name, p)
        p.copy_(v.to(p.dtype))
    return module


def seeded_tensor(name: str, shape, seed: int = 0, scale: float = 1.0, dtype=torch.float32) -> torch.Tensor:
    g = torch.Generator(device="cpu")
    g.manual_seed((zlib.crc32(name.encode()) + 104729 * seed) & 0x7FFFFFFF)
    return (torch.randn(tuple(shape), generator=g, dtype=torch.float32) * scale).to(dtype)


def sample_indices(numel: int, k: int = 512, seed: int = 1234) -> torch.Tensor:
    g = torch.Generator(device="cpu")
    g.manual_seed(seed + numel)
    if numel <= k:
        return torch.arange(numel)
    return torch.randint(0, numel, (k,), generator=g)


def fingerprint(t: torch.Tensor, k: int = 512) -> dict:
    """Compact, order-sensitive summary of a tensor used as a golden vector."""
    f = t.detach().double().reshape(-1).cpu()
    idx = sample_indices(f.numel(), k)
    return {
        "shape": list(t.shape),
        "mean": float(f.double().mean()),
        "std": float(f.double().std()) if f.numel() > 1 else 0.0,
        "absmax": float(f.abs().max()),
        "samples": [float(x) for x in f[idx]],
    }
