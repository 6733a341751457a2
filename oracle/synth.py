"""Platform-stable synthetic parameters and frames (TEST INFRASTRUCTURE, see oracle/__init__.py).

The golden vectors under tests/golden/ were produced by the *reference* model holding
``synth_state_dict(...)`` weights and fed ``synth_images(...)`` frames.  Because both are a
pure function of (name, shape, seed) through numpy's Philox bit generator -- whose stream
numpy guarantees stable -- the GPU box can rebuild the identical tensors without the
fixtures having to carry ~20 MB of weights.  Nothing here depends on module construction
order or on torch's RNG.
"""
from __future__ import annotations

import zlib
from typing import Dict, Iterable, Tuple

import numpy as np


def _gen(seed: int, name: str) -> np.random.Generator:
    return np.random.Generator(np.random.Philox(key=[int(seed) & 0xFFFFFFFF, zlib.crc32(name.encode())]))


def synth_tensor(name: str, shape: Tuple[int, ...], seed: int = 0) -> np.ndarray:
    """Deterministic value for one state_dict entry, chosen by its name and rank.

    conv weights  : N(0, g/fan_in), g = 2 for the encoders (kaiming), 1/3 for the update block
                    (the variance of torch default conv init, keeps flows at a few px / iteration)
    norm weights  : 1 + 0.1 N(0,1)      (rank-1 ``*.weight``)
    biases        : 0.05 N(0,1)
    running_mean  : 0.05 N(0,1);  running_var: 1 + 0.2 |N(0,1)|;  num_batches_tracked: 0
    """
    g = _gen(seed, name)
    shape = tuple(int(s) for s in shape)
    if name.endswith("num_batches_tracked"):
        return np.zeros(shape, dtype=np.int64)
    if name.endswith("rel_ind"):  # GMA RelPosEmb index buffer: deltas + max_pos - 1 (gma_utils.py:12-16), not random
        n = shape[0]
        return (np.arange(n)[None, :] - np.arange(n)[:, None] + n - 1).astype(np.int64)
    n = g.standard_normal(shape, dtype=np.float64)
    if name.endswith("running_var"):
        return (1.0 + 0.2 * np.abs(n)).astype(np.float32)
    if name.endswith("running_mean"):
        return (0.05 * n).astype(np.float32)
    if len(shape) == 4:
        fan_in = shape[1] * shape[2] * shape[3]
        gain = 2.0 if name.startswith(("fnet.", "cnet.")) else 1.0 / 3.0  # encoders: kaiming; update block: torch default-init variance
        return (n * np.sqrt(gain / fan_in)).astype(np.float32)
    if len(shape) == 1 and name.endswith("weight"):
        return (1.0 + 0.1 * n).astype(np.float32)
    if name.endswith("gamma"):  # GMA Aggregate.gamma (scalar, zero-init in the reference)
        return (0.5 + 0.1 * n).astype(np.float32)
    return (0.05 * n).astype(np.float32)


def synth_state_dict(shapes: Dict[str, Tuple[int, ...]], seed: int = 0):
    """name -> torch tensor for every entry of ``shapes`` (an ordered name->shape map)."""
    import torch

    return {k: torch.from_numpy(synth_tensor(k, tuple(v), seed)) for k, v in shapes.items()}


def shapes_of(state_dict) -> Dict[str, Tuple[int, ...]]:
    return {k: tuple(v.shape) for k, v in state_dict.items()}


def synth_images(batch: int, height: int, width: int, seed: int = 0, kind: str = "noise") -> np.ndarray:
    """Frame pairs [B, 2, 3, H, W] float32 in [0, 1), BGR like the reference expects.

    kind="noise"  : i.i.d. uniform (what model_benchmark.py feeds, model_benchmark.py:445-453).
    kind="smooth" : box-blurred coarse noise; frame 2 is frame 1 moved by (+4, -3) px, so the
                    lookups stay mostly in bounds (SURVEY.md section 8(d) "smooth" input).
    """
    g = _gen(seed, f"images/{kind}/{batch}x{height}x{width}")
    if kind == "noise":
        return g.random((batch, 2, 3, height, width), dtype=np.float32)
    if kind != "smooth":
        raise ValueError(kind)
    ch, cw = height // 8 + 2, width // 8 + 2
    coarse = g.random((batch, 3, ch, cw), dtype=np.float32)
    img = np.repeat(np.repeat(coarse, 8, axis=2), 8, axis=3)
    # separable 9-tap box blur, twice, keeps it cheap and numpy-only
    k = 9
    for _ in range(2):
        c = np.cumsum(np.pad(img, ((0, 0), (0, 0), (k, 0), (0, 0))), axis=2, dtype=np.float64)
        img = ((c[:, :, k:] - c[:, :, :-k]) / k).astype(np.float32)
        c = np.cumsum(np.pad(img, ((0, 0), (0, 0), (0, 0), (k, 0))), axis=3, dtype=np.float64)
        img = ((c[:, :, :, k:] - c[:, :, :, :-k]) / k).astype(np.float32)
    f1 = img[:, :, 8 : 8 + height, 8 : 8 + width]
    f2 = img[:, :, 8 + 3 : 8 + 3 + height, 8 - 4 : 8 - 4 + width]  # content moves +4 in x, -3 in y
    out = np.stack([f1, f2], axis=1)
    lo, hi = out.min(), out.max()
    return ((out - lo) / max(hi - lo, 1e-6) * 0.999).astype(np.float32)


def synth_normal(name: str, shape: Iterable[int], seed: int = 0, scale: float = 1.0) -> np.ndarray:
    """Generic N(0, scale^2) float32 tensor for operator-level fixtures (features, coords noise)."""
    return (scale * _gen(seed, name).standard_normal(tuple(shape), dtype=np.float64)).astype(np.float32)


def sample_index(n: int, k: int) -> np.ndarray:
    """Up to k distinct flat positions spread over [0, n), ascending (all of them when n <= k).  A fixed multiplicative
    stride rather than an RNG: a fixture that stores a sample of a large output and the test that reads it always agree
    on the positions."""
    if n <= k:
        return np.arange(n)
    return np.unique((np.arange(k, dtype=np.int64) * 2654435761) % n)
