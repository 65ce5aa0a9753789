"""uint8 document images for the engine's device preprocess (`mmee_preprocess_images`, `mmee_forward_images`).

`pack_images` lays a batch of decoded pages out the way the C ABI reads it (`mmee_images` in include/mmee.h): all
bytes back to back, row-major HWC, with per-image offsets and (height, width).  The engine then resizes, rescales and
normalises them on the device, bit for bit as the reference's LayoutLMv3 image processor does on the host
(oracle/image_port.py).  Decoding (TIFF / PNG / JPEG) stays with the caller.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Sequence

import numpy as np
import torch

from . import _lib

MAX_SIDE = 16384     # image.cuh IMG_MAX_SIDE


@dataclass
class PackedImages:
    data: torch.Tensor       # uint8 [total_bytes]: all images back to back, row-major HWC (host, pinned if asked, or CUDA)
    offsets: np.ndarray      # int64 [B] byte offset of each image in data
    sizes: np.ndarray        # int32 [B, 2] (height, width)
    channels: int            # 1 (grayscale) or 3 (RGB), the whole batch

    def __len__(self) -> int:
        return int(self.offsets.shape[0])

    def c_struct(self, data: torch.Tensor = None) -> _lib.Images:
        """The `mmee_images` view of this batch, with `data` (same bytes, e.g. a device copy) in place of self.data.
        The struct borrows the arrays: keep this object alive while it is used."""
        d = self.data if data is None else data
        s = _lib.Images()
        s.data = d.data_ptr()
        s.offsets = self.offsets.ctypes.data
        s.sizes = self.sizes.ctypes.data
        s.channels = self.channels
        s.total_bytes = d.numel()
        return s


def _as_array(img) -> np.ndarray:
    if isinstance(img, np.ndarray):
        a = img
    elif torch.is_tensor(img):
        if img.dtype != torch.uint8:
            raise ValueError(f"image tensors must be uint8, got {img.dtype}")
        a = img.detach().cpu().numpy()
    elif hasattr(img, "mode") and hasattr(img, "size"):          # PIL.Image.Image
        if img.mode not in ("L", "RGB"):
            raise ValueError(f"PIL images must be mode L or RGB, got {img.mode!r}")
        a = np.asarray(img)
    else:
        raise ValueError(f"unsupported image type {type(img).__name__}: expected a uint8 numpy array, torch tensor or "
                         "PIL image")
    if a.dtype != np.uint8:
        raise ValueError(f"images must be uint8, got {a.dtype}")
    if not (a.ndim == 2 or (a.ndim == 3 and a.shape[2] == 3)):
        raise ValueError(f"images must be shaped (h, w) or (h, w, 3), got {a.shape}")
    h, w = a.shape[:2]
    if not (1 <= h <= MAX_SIDE and 1 <= w <= MAX_SIDE):
        raise ValueError(f"image size ({h}, {w}) outside [1, {MAX_SIDE}]")
    return a


def pack_images(images: Sequence, pin: bool = True) -> PackedImages:
    """Pack decoded pages: uint8 numpy arrays or torch tensors shaped (h, w) (grayscale) or (h, w, 3) (RGB), or PIL
    images in mode L or RGB.  Every page of a batch must have the same number of channels.  `pin=True` puts the bytes
    in pinned host memory, so the upload to the GPU is asynchronous."""
    if isinstance(images, (np.ndarray, torch.Tensor)) or not isinstance(images, Sequence) or len(images) == 0:
        raise ValueError("expected a non-empty list of images")
    arrays = [_as_array(im) for im in images]
    chans = {1 if a.ndim == 2 else 3 for a in arrays}
    if len(chans) != 1:
        raise ValueError("all images of a batch must have the same number of channels (1 or 3)")
    sizes = np.array([a.shape[:2] for a in arrays], dtype=np.int32)
    nbytes = np.array([a.size for a in arrays], dtype=np.int64)
    offsets = np.concatenate([[0], np.cumsum(nbytes)[:-1]]).astype(np.int64)
    data = torch.empty(int(nbytes.sum()), dtype=torch.uint8, pin_memory=pin)
    flat = data.numpy()
    for a, o, n in zip(arrays, offsets, nbytes):
        flat[o:o + n] = a.reshape(-1)
    return PackedImages(data=data, offsets=offsets, sizes=sizes, channels=chans.pop())


def as_packed(images, pin: bool = True) -> PackedImages:
    """`images` as given if already packed, else `pack_images(images, pin)`."""
    return images if isinstance(images, PackedImages) else pack_images(images, pin=pin)
