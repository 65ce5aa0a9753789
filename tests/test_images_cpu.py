"""CPU tests of the uint8 image path: the numpy restatement of Pillow's bilinear resize (oracle/image_port.py, what the
device kernels of csrc/image.cuh are checked against) equals Pillow and the LayoutLMv3 image processor, and
`mmee.images.pack_images` rejects malformed input."""
import numpy as np
import pytest
import torch
from PIL import Image

from mmee.images import pack_images
from oracle import image_port

S = 224


def size_set():
    """>= 200 seeded (h, w): edge cases, then random sizes across up- and downscaling and extreme aspect ratios."""
    sizes = [(1, 1), (224, 224), (223, 223), (225, 225), (223, 225), (225, 223), (1000, 754), (1000, 762),
             (100, 80), (300, 224), (224, 500), (2200, 1700), (7, 999), (16384, 1), (16384, 3), (1, 16384),
             (5, 16384), (16384, 224), (224, 16384), (16384, 163), (16384, 164), (101, 1), (100, 1),
             (2, 16384), (13, 17), (8191, 7), (127, 131), (2, 3), (449, 448)]
    primes = [2, 3, 5, 7, 11, 97, 211, 223, 227, 229, 509, 1009, 2003, 4099]
    rng = np.random.default_rng(20261022)
    for _ in range(12):
        sizes.append((int(rng.choice(primes)), int(rng.choice(primes))))
    while len(sizes) < 210:
        kind = rng.integers(0, 4)
        if kind == 0:
            h, w = rng.integers(1, 3000, 2)
        elif kind == 1:
            h, w = rng.integers(500, 1400), rng.integers(400, 1100)
        elif kind == 2:
            h, w = rng.integers(1000, 16385), rng.integers(1, 80)
        else:
            h, w = rng.integers(1, 80), rng.integers(1000, 16385)
        sizes.append((int(h), int(w)))
    return sizes


SIZES = size_set()


def page(h, w, channels, seed, kind="random"):
    """A seeded uint8 page: random bytes, constant 0 / 255 or a checkerboard."""
    shape = (h, w) if channels == 1 else (h, w, 3)
    if kind == "zeros":
        return np.zeros(shape, np.uint8)
    if kind == "ones":
        return np.full(shape, 255, np.uint8)
    if kind == "checker":
        c = ((np.arange(h)[:, None] + np.arange(w)[None, :]) % 2 * 255).astype(np.uint8)
        return c if channels == 1 else np.repeat(c[:, :, None], 3, axis=2)
    return np.random.default_rng(seed).integers(0, 256, shape, dtype=np.uint8)


KINDS = ["random", "zeros", "ones", "checker"]


def test_size_set_covers_the_cases():
    assert len(SIZES) >= 200
    assert max(max(s) for s in SIZES) == 16384
    assert any(image_port.vertical_first(h, w, S) for h, w in SIZES)


@pytest.mark.parametrize("i", range(len(SIZES)))
def test_resize_equals_pillow(i):
    h, w = SIZES[i]
    channels = 1 if i % 3 else 3
    a = page(h, w, channels, seed=i, kind=KINDS[i % 4] if i % 5 == 0 else "random")
    want = np.asarray(Image.fromarray(a).resize((S, S), Image.BILINEAR))
    got = image_port.resize(a, S)
    assert got.dtype == np.uint8 and got.shape == want.shape
    bad = np.argwhere(got != want)
    assert bad.size == 0, f"({h}, {w}) x{channels}: first mismatch at {bad[0].tolist()}"


@pytest.mark.parametrize("n", [1, 7, 224, 1000])
def test_pass_over_an_axis_of_output_length_is_identity(n):
    """The device kernels run both passes even when an axis already has S entries: the coefficients are {2^22, 0}."""
    xmin, cnt, k = image_port.coeffs(n, n)
    assert np.array_equal(xmin, np.arange(n))
    assert np.all(k[:, 0] == 1 << image_port.PRECISION_BITS) and np.all(k[:, 1:] == 0)


def test_grayscale_resizes_as_its_rgb_conversion():
    a = page(1000, 754, 1, seed=5)
    rgb = np.asarray(Image.fromarray(a).convert("RGB").resize((S, S), Image.BILINEAR))
    got = image_port.resize(a, S)
    for c in range(3):
        assert np.array_equal(rgb[:, :, c], got)


def test_normalise_is_correctly_rounded_division():
    r = np.arange(256, dtype=np.uint8)
    want = np.array([(np.float32(v) / np.float32(255.0) - np.float32(0.5)) / np.float32(0.5) for v in range(256)],
                    dtype=np.float32)
    assert np.array_equal(image_port.normalise(r), want)
    # transformers 4.26 order: fp64 r * (1 / 255) rounded to fp32, then the fp32 normalisation
    old = ((r.astype(np.float64) * (1 / 255)).astype(np.float32) - np.float32(0.5)) / np.float32(0.5)
    assert np.array_equal(image_port.normalise(r), old)


def _processor():
    try:
        from transformers import LayoutLMv3ImageProcessorPil as P
    except ImportError:
        try:        # transformers 4.x: the Pillow-backed processor under its own name
            from transformers import LayoutLMv3ImageProcessor as P
        except ImportError:
            return None
    return P(apply_ocr=False)


@pytest.mark.parametrize("channels", [1, 3])
@pytest.mark.parametrize("hw", [(1000, 754), (224, 224), (100, 80), (2200, 1700), (7, 999), (16384, 3)])
def test_preprocess_equals_layoutlmv3_image_processor(hw, channels):
    proc = _processor()
    if proc is None:
        pytest.skip("transformers has no Pillow-backed LayoutLMv3 image processor in this environment")
    a = page(*hw, channels, seed=hw[0] + channels)
    want = np.asarray(proc(Image.fromarray(a).convert("RGB"), return_tensors="np")["pixel_values"][0])
    got = image_port.preprocess(a, S)
    assert got.dtype == np.float32 and want.shape == got.shape == (3, S, S)
    assert np.array_equal(got, want)


# ---------------------------------------------------------------------------------------------------- pack_images
def test_pack_images_layout():
    a = page(30, 20, 1, seed=1)
    b = torch.from_numpy(page(5, 7, 1, seed=2))
    c = Image.fromarray(page(3, 4, 1, seed=3))
    p = pack_images([a, b, c], pin=False)
    assert p.channels == 1 and len(p) == 3
    assert p.sizes.tolist() == [[30, 20], [5, 7], [3, 4]]
    assert p.offsets.tolist() == [0, 600, 635]
    flat = p.data.numpy()
    assert flat.size == 647
    assert np.array_equal(flat[600:635].reshape(5, 7), b.numpy())
    rgb = pack_images([page(4, 5, 3, seed=4), Image.fromarray(page(2, 2, 3, seed=5))], pin=False)
    assert rgb.channels == 3 and rgb.offsets.tolist() == [0, 60] and rgb.data.numel() == 72


@pytest.mark.parametrize("bad", [
    "empty", "not_a_list", "float", "int16_tensor", "two_channels", "four_channels", "rank4", "zero_height",
    "too_wide", "too_tall", "mixed_channels", "pil_rgba", "pil_palette", "string",
])
def test_pack_images_rejects(bad):
    ok = page(8, 8, 1, seed=0)
    cases = {
        "empty": [],
        "not_a_list": ok,
        "float": [ok.astype(np.float32)],
        "int16_tensor": [torch.zeros((8, 8), dtype=torch.int16)],
        "two_channels": [np.zeros((8, 8, 2), np.uint8)],
        "four_channels": [np.zeros((8, 8, 4), np.uint8)],
        "rank4": [np.zeros((1, 8, 8, 3), np.uint8)],
        "zero_height": [np.zeros((0, 8), np.uint8)],
        "too_wide": [np.zeros((1, 16385), np.uint8)],
        "too_tall": [np.zeros((16385, 1), np.uint8)],
        "mixed_channels": [ok, page(8, 8, 3, seed=1)],
        "pil_rgba": [Image.new("RGBA", (8, 8))],
        "pil_palette": [Image.new("P", (8, 8))],
        "string": ["page.png"],
    }
    with pytest.raises(ValueError):
        pack_images(cases[bad], pin=False)
