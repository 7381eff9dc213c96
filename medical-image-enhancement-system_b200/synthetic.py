"""Seeded synthetic inputs of the shapes BASELINE.json names (SURVEY.md §8(d)).

  U  uniform noise over the full dtype range (best case for histogram atomics)
  P  CT-like phantom: >= 40 % of the pixels are exactly 0 ("air") outside a body
     ellipse; inside, piecewise-constant ellipses in [800, 3000] plus N(0, 25)
     noise, 12-bit occupancy of the 16-bit container (headline distribution)
  K  constant image (worst-case contention, CLAHE edge case)

numpy only (host side); used by bench.py, tests/ and the batching loader demo.
"""
from __future__ import annotations

import numpy as np

__all__ = ["uniform", "phantom", "constant", "phantom_volume", "vessel_volume", "make"]


def uniform(shape, dtype=np.uint16, seed: int = 0) -> np.ndarray:
    rng = np.random.default_rng(seed)
    info = np.iinfo(dtype)
    return rng.integers(info.min, info.max + 1, size=shape, dtype=dtype)


def constant(shape, dtype=np.uint16, value: int = 1000) -> np.ndarray:
    info = np.iinfo(dtype)
    return np.full(shape, min(max(value, info.min), info.max), dtype=dtype)


def _phantom_slice(rng, h, w, z=0.0):
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    cy, cx = h / 2.0 + rng.uniform(-0.02, 0.02) * h, w / 2.0 + rng.uniform(-0.02, 0.02) * w
    ry, rx = 0.40 * h * (1.0 - 0.3 * z * z), 0.34 * w * (1.0 - 0.3 * z * z)
    body = ((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1.0
    img = np.zeros((h, w), np.float32)
    img[body] = 1000.0
    for _ in range(int(rng.integers(5, 11))):
        ey, ex = cy + rng.uniform(-0.6, 0.6) * ry, cx + rng.uniform(-0.6, 0.6) * rx
        sy, sx = rng.uniform(0.05, 0.3) * ry, rng.uniform(0.05, 0.3) * rx
        inside = (((yy - ey) / sy) ** 2 + ((xx - ex) / sx) ** 2 <= 1.0) & body
        img[inside] = rng.uniform(800.0, 3000.0)
    noise = rng.normal(0.0, 25.0, size=(h, w)).astype(np.float32)
    img = np.where(body, np.clip(img + noise, 1.0, 4095.0), 0.0)
    return np.rint(img)


def phantom(shape, dtype=np.uint16, seed: int = 0, unique: int = 16) -> np.ndarray:
    """(..., H, W) phantom slices; `unique` distinct slices are generated and cycled
    (with a per-slice flip) so that large batches stay cheap to synthesise."""
    h, w = shape[-2:]
    n = int(np.prod(shape[:-2], dtype=np.int64)) if len(shape) > 2 else 1
    rng = np.random.default_rng(seed)
    base = [_phantom_slice(rng, h, w) for _ in range(min(unique, n))]
    out = np.empty((n, h, w), np.float32)
    for i in range(n):
        s = base[i % len(base)]
        k = (i // len(base)) % 4
        out[i] = s if k == 0 else (s[:, ::-1] if k == 1 else (s[::-1] if k == 2 else s[::-1, ::-1]))
    if np.dtype(dtype) == np.int16:
        out = out - 1024.0  # HU-like: air = -1024
    return out.astype(dtype).reshape(shape)


def phantom_volume(shape, dtype=np.int16, seed: int = 0) -> np.ndarray:
    """(D, H, W) volume whose body ellipse shrinks towards the ends (HU-like for int16)."""
    d, h, w = shape
    rng = np.random.default_rng(seed)
    key = [_phantom_slice(rng, h, w, z=0.0) for _ in range(min(d, 8))]
    out = np.empty((d, h, w), np.float32)
    for z in range(d):
        out[z] = key[(z * len(key)) // d]
    nz = rng.normal(0.0, 10.0, size=(d, 1, 1)).astype(np.float32)
    out = np.where(out > 0, np.clip(out + nz, 1.0, 4095.0), 0.0)
    if np.dtype(dtype) == np.int16:
        out = out - 1024.0
    return np.rint(out).astype(dtype)


def vessel_volume(shape, dtype=np.int16, seed: int = 0, tubes: int = 12) -> np.ndarray:
    """(D, H, W) angiography-like volume: `tubes` bright straight vessels of radius 1 to 6 voxels in random orientations
    (contrast-enhanced blood, 250 to 450 HU, with a soft edge) on soft tissue (40 HU) with N(0, 20) noise.  int16 is
    in HU; uint16 is HU + 1024; uint8 is (HU + 1024) / 8 clipped to 255; float32 is (HU + 1024) / 4096."""
    d, h, w = shape
    rng = np.random.default_rng(seed)
    centre = rng.uniform(0.2, 0.8, size=(tubes, 3)) * np.array([d, h, w])
    axis = rng.normal(size=(tubes, 3))
    axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    radius = rng.uniform(1.0, 6.0, size=tubes)
    level = rng.uniform(250.0, 450.0, size=tubes)
    out = np.empty((d, h, w), np.float32)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    for z in range(d):
        sl = np.full((h, w), 40.0, np.float32)
        for c, u, r, v in zip(centre, axis, radius, level):
            pz, py, px = np.float32(z - c[0]), yy - np.float32(c[1]), xx - np.float32(c[2])
            along = pz * np.float32(u[0]) + py * np.float32(u[1]) + px * np.float32(u[2])
            dist2 = pz * pz + py * py + px * px - along * along
            inside = np.clip(np.float32(r) + 0.5 - np.sqrt(np.maximum(dist2, 0.0)), 0.0, 1.0)
            sl = np.maximum(sl, 40.0 + (v - 40.0) * inside)
        out[z] = sl
    out += rng.normal(0.0, 20.0, size=(d, h, w)).astype(np.float32)
    dt = np.dtype(dtype)
    if dt == np.int16:
        return np.rint(out).astype(np.int16)
    if dt == np.uint16:
        return np.rint(out + 1024.0).clip(0, 65535).astype(np.uint16)
    if dt == np.uint8:
        return np.rint((out + 1024.0) / 8.0).clip(0, 255).astype(np.uint8)
    return ((out + 1024.0) / 4096.0).astype(np.float32)


def make(kind: str, shape, dtype=np.uint16, seed: int = 0) -> np.ndarray:
    if kind == "U":
        return uniform(shape, dtype, seed)
    if kind == "P":
        return phantom(shape, dtype, seed)
    if kind == "K":
        return constant(shape, dtype)
    raise ValueError(f"unknown synthetic kind {kind!r} (U, P, K)")
