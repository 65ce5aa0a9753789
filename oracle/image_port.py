"""numpy restatement of the LayoutLMv3 image processor on 8-bit L / RGB pages (the reference pins transformers 4.26,
which resizes with Pillow): `Image.resize((S, S), BILINEAR)` as Pillow's Resample.c computes it, then rescale and
normalise to (r / 255 - 0.5) / 0.5 in fp32.  The engine's image kernels (csrc/image.cuh) must equal this bit for bit.

Pillow's 8-bit resample, per axis:
  scale = in / out, fs = max(scale, 1), support = fs (bilinear support 1), ksize = 2 * ceil(support) + 1
  for each output index xx: center = (xx + 0.5) * scale, xmin = max(int(center - support + 0.5), 0),
  n = min(int(center + support + 0.5), in) - xmin, w[x] = tri((x + xmin - center + 0.5) * (1 / fs)) for x < n,
  divided by their sequential sum when it is non-zero, then k = int(w * 2^22 + 0.5) (PRECISION_BITS = 22).
A pass computes clip((2^21 + sum byte * k) >> 22, 0, 255) into uint8.  The horizontal pass runs first and the
vertical one over its output, except for a page more than 100 times taller than wide that is shrunk in height: there
`Image.resize` (Pillow 12.2) runs the vertical pass first, as a resize of its own.  Python floats and numpy float64
arrays are IEEE doubles without fused multiply-adds.
"""
from __future__ import annotations

import numpy as np

PRECISION_BITS = 22


def coeffs(in_size: int, out_size: int):
    """-> (xmin int64 [out], n int64 [out], k int64 [out, ksize]) of one axis; k is zero past n."""
    scale = float(in_size) / out_size
    fs = max(scale, 1.0)
    support = fs * 1.0
    ksize = int(np.ceil(support)) * 2 + 1
    center = (np.arange(out_size, dtype=np.float64) + 0.5) * scale
    ss = 1.0 / fs
    xmin = np.maximum((center - support + 0.5).astype(np.int64), 0)
    n = np.minimum((center + support + 0.5).astype(np.int64), in_size) - xmin
    w = np.zeros((out_size, ksize), dtype=np.float64)
    ww = np.zeros(out_size, dtype=np.float64)
    for x in range(ksize):                       # column by column: the sum is sequential in x, as in Pillow
        t = np.abs(((x + xmin).astype(np.float64) - center + 0.5) * ss)
        wx = np.where((x < n) & (t < 1.0), 1.0 - t, 0.0)
        w[:, x] = wx
        ww = ww + wx
    w = np.where(ww[:, None] != 0.0, w / np.where(ww == 0.0, 1.0, ww)[:, None], w)
    scaled = w * float(1 << PRECISION_BITS)
    k = np.where(w < 0, (scaled - 0.5).astype(np.int64), (scaled + 0.5).astype(np.int64))
    return xmin, n, k


def _pass(a: np.ndarray, out_size: int, axis: int) -> np.ndarray:
    """Resample uint8 `a` [rows, cols, C] along `axis` (1: horizontal, 0: vertical) to out_size."""
    xmin, n, k = coeffs(a.shape[axis], out_size)
    ksize = k.shape[1]
    idx = np.minimum(xmin[:, None] + np.arange(ksize)[None, :], a.shape[axis] - 1)   # k = 0 where clipped
    src = np.moveaxis(a, axis, 0).astype(np.int64)                                    # [in, other, C]
    acc = np.full((out_size,) + src.shape[1:], 1 << (PRECISION_BITS - 1), dtype=np.int64)
    for x in range(ksize):
        acc += src[idx[:, x]] * k[:, x][:, None, None]
    out = np.clip(acc >> PRECISION_BITS, 0, 255).astype(np.uint8)
    return np.moveaxis(out, 0, axis)


def vertical_first(h: int, w: int, size: int) -> bool:
    """Pillow's `Image.resize` shrinks a page more than 100 times taller than wide vertically first."""
    return h > 100 * w and size < h


def resize(a: np.ndarray, size: int) -> np.ndarray:
    """Pillow `Image.fromarray(a).resize((size, size), BILINEAR)` of a uint8 (h, w) or (h, w, C) array, as uint8
    (size, size) or (size, size, C).  A pass whose input already has `size` entries is the identity and is skipped."""
    a = np.asarray(a)
    if a.dtype != np.uint8 or a.ndim not in (2, 3):
        raise ValueError("expected a uint8 (h, w) or (h, w, C) array")
    x = a[:, :, None] if a.ndim == 2 else a
    axes = (0, 1) if vertical_first(x.shape[0], x.shape[1], size) else (1, 0)
    for axis in axes:
        if x.shape[axis] != size:
            x = _pass(x, size, axis)
    return x[:, :, 0] if a.ndim == 2 else x


def normalise(r: np.ndarray) -> np.ndarray:
    """Rescale and normalise uint8 bytes: (r / 255 - 0.5) / 0.5 in fp32, correctly rounded division."""
    f = np.float32
    return (np.asarray(r).astype(f) / f(255.0) - f(0.5)) / f(0.5)


def preprocess(a: np.ndarray, size: int = 224) -> np.ndarray:
    """fp32 [3, size, size] pixel values of one L (h, w) or RGB (h, w, 3) page: what the reference's processor gives
    for `Image.fromarray(a).convert("RGB")`."""
    r = resize(a, size)
    if r.ndim == 2:
        r = np.repeat(r[:, :, None], 3, axis=2)
    return np.ascontiguousarray(normalise(r).transpose(2, 0, 1))
