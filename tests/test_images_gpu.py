"""GPU tests (B200) of the uint8 image path (csrc/image.cuh, `mmee_preprocess_images`, `mmee_forward_images`): the
device preprocess equals the numpy restatement of the LayoutLMv3 image processor (oracle/image_port.py, itself checked
against Pillow by test_images_cpu.py) bit for bit, and every forward over `images=` equals the same forward over the
oracle's pixel values, bit for bit."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from helpers import load_case
from mmee import _lib, synth
from mmee.config import ExitConfig, ModelDims
from mmee.images import pack_images
from oracle import image_port
from test_images_cpu import KINDS, SIZES, page

pytestmark = pytest.mark.gpu

_models = {}


def _engine(name, dtype="bf16", max_batch=8):
    from mmee.model import B200EEForSequenceClassification

    key = (name, dtype, max_batch)
    if key not in _models:
        g, dims, ee, sd, docs = load_case(name)
        mb = max(max_batch, docs["pixel_values"].shape[0])
        _models[key] = (B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=mb, dtype=dtype), dims, docs)
    return _models[key]


@functools.lru_cache(maxsize=None)
def _size_set_case(channels):
    """(pages, oracle pixels f32 [B, 3, 224, 224]) for SIZES: mostly random bytes, every fifth page constant 0 / 255
    or a checkerboard."""
    pages = [page(h, w, channels, seed=100 * channels + i, kind=KINDS[i % 4] if i % 5 == 0 else "random")
             for i, (h, w) in enumerate(SIZES)]
    return pages, np.stack([image_port.preprocess(a, 224) for a in pages])


def _assert_pixels(got, pages, want, tag):
    got = got.cpu().numpy()
    for b, a in enumerate(pages):
        bad = np.argwhere(got[b] != want[b])
        if bad.size:
            c, y, x = bad[0].tolist()
            raise AssertionError(f"{tag}: image {b} {a.shape}: {len(bad)} mismatches, first at channel {c}, row {y}, "
                                 f"column {x}: got {got[b, c, y, x]!r}, want {want[b, c, y, x]!r}")


@pytest.mark.parametrize("channels", [1, 3])
def test_preprocess_ragged_batch_equals_oracle(channels):
    model, dims, _ = _engine("tiny_ramp_conf", max_batch=len(SIZES))
    pages, want = _size_set_case(channels)
    got = model.preprocess_images(pages)
    torch.cuda.synchronize()
    assert got.shape == (len(pages), 3, dims.image, dims.image) and got.dtype == torch.float32
    _assert_pixels(got, pages, want, f"ragged batch x{channels}")
    # neither the neighbours nor the order matter
    rev = model.preprocess_images(pages[::-1])
    torch.cuda.synchronize()
    assert torch.equal(rev.flip(0), got)


@pytest.mark.parametrize("channels", [1, 3])
def test_preprocess_one_image_per_batch_equals_oracle(channels):
    model, dims, _ = _engine("tiny_ramp_conf", max_batch=len(SIZES))
    pages, want = _size_set_case(channels)
    outs = [model.preprocess_images([a]) for a in pages]
    torch.cuda.synchronize()
    _assert_pixels(torch.cat(outs), pages, want, f"one per batch x{channels}")


def _doc_pages(n, seed, channels=1):
    """n document pages of assorted sizes (RVL-CDIP-like heights, a small page, a tall strip)."""
    rng = np.random.default_rng(seed)
    hw = [(1000, int(rng.integers(600, 1001))) for _ in range(n)]
    hw[0] = (224, 224)
    if n > 2:
        hw[1], hw[2] = (97, 61), (12000, 100)
    return [page(h, w, channels, seed=seed + i) for i, (h, w) in enumerate(hw)]


def _oracle_px(pages, S):
    return torch.from_numpy(np.stack([image_port.preprocess(a, S) for a in pages]))


def _same(a, b):
    if torch.is_tensor(a):
        return torch.equal(a.cpu(), b.cpu()) or (a.dtype.is_floating_point and
                                                  np.array_equal(a.cpu().numpy(), b.cpu().numpy(), equal_nan=True))
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


PATHS = ["forward", "infer_host", "infer_device", "plan_device", "plan_host"]


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("early_exit", [True, False])
@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
@pytest.mark.parametrize("name", ["tiny_ramp_conf", "base_gate_ent", "tiny_image_only"])
def test_forward_images_equals_pixel_values(name, dtype, early_exit, path):
    if path == "forward" and early_exit:
        pytest.skip("forward is the dense reference-shaped call: one mode")
    model, dims, docs = _engine(name, dtype)
    n = docs["pixel_values"].shape[0]
    pages = _doc_pages(n, seed=len(name))
    px = _oracle_px(pages, dims.image)
    text = {k: v for k, v in docs.items() if k != "pixel_values"}
    if dims.n_text == 0:
        text = {}
    dev = {k: v.cuda() for k, v in text.items()}
    kw = dict(exit_threshold=0.6 if model._default_criterion() == "max_confidence" else 0.5, early_exit=early_exit)
    pages_dev = pack_images(pages)          # device paths get device bytes: the image-only engine has no text inputs
    pages_dev.data = pages_dev.data.cuda()
    if path == "forward":
        got = model.forward(**text, images=pages)
        want = model.forward(**text, pixel_values=px)
        for f in ("logits", "exit_logits", "exit_index"):
            assert _same(getattr(got, f), getattr(want, f)), f
        for (gh, gc), (wh, wc) in zip(got.exit_states, want.exit_states):
            assert _same(gh, wh) and _same(gc, wc)
        return
    if path in ("infer_host", "infer_device"):
        src = text if path == "infer_host" else dev
        got = model.infer(**src, images=pages, return_all=True, **kw) if path == "infer_host" else \
            model.infer_device(**src, images=pages_dev, **kw)
        want = model.infer(**src, pixel_values=px if path == "infer_host" else px.cuda(), return_all=True, **kw) \
            if path == "infer_host" else model.infer_device(**src, pixel_values=px.cuda(), **kw)
        torch.cuda.synchronize()
    else:
        plan = model.plan(n, early_exit=early_exit, return_all=True)
        src = dev if path == "plan_device" else text
        got = plan.infer(**src, images=pages_dev if path == "plan_device" else pages, exit_threshold=kw["exit_threshold"])
        want = plan.infer(**src, pixel_values=px.cuda() if path == "plan_device" else px,
                          exit_threshold=kw["exit_threshold"])
        plan.close()
        assert got.logits.device == want.logits.device
    if isinstance(got, dict):
        for k in got:
            assert _same(got[k], want[k]), k
        return
    for f in ("exits_store", "logits", "criteria", "exit_hist", "predictions", "all_exit_logits", "all_criteria"):
        assert _same(getattr(got, f), getattr(want, f)), f


def test_image_forwards_are_ordered_with_plan_runs():
    """Host image forwards (their preprocess runs on the engine's copy stream) interleaved with plan runs and device
    preprocesses on other streams give the results each gives alone."""
    model, dims, docs = _engine("base_gate_ent")
    n = docs["pixel_values"].shape[0]
    text = {k: v for k, v in docs.items() if k != "pixel_values"}
    dev = {k: v.cuda() for k, v in text.items()}
    pages, other = _doc_pages(n, seed=1), _doc_pages(n, seed=2)
    kw = dict(exit_threshold=0.6)
    ref = model.infer(**text, images=pages, **kw)
    ref_other = model.infer(**text, images=other, **kw)
    plan = model.plan(n)
    s1 = torch.cuda.Stream()
    torch.cuda.synchronize()
    for _ in range(3):
        with torch.cuda.stream(s1):
            r1 = plan.infer_device(**dev, images=other, **kw)
        r2 = model.infer(**text, images=pages, **kw)                     # host path, no dependency on s1
        with torch.cuda.stream(s1):
            r3 = plan.infer_device(**dev, images=pages, **kw)
        torch.cuda.synchronize()
        assert torch.equal(r1["logits"].cpu(), ref_other.logits.cpu())
        assert torch.equal(r2.logits, ref.logits) and np.array_equal(r2.exits_store, ref.exits_store)
        assert torch.equal(r3["logits"].cpu(), ref.logits.cpu())
    model.sync()
    plan.close()


def _c_preprocess(model, B, data, offsets, sizes, channels, total=None, out=None):
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    sizes = np.ascontiguousarray(sizes, dtype=np.int32)
    img = _lib.Images()
    img.data, img.offsets, img.sizes = data.data_ptr(), offsets.ctypes.data, sizes.ctypes.data
    img.channels = channels
    img.total_bytes = data.numel() if total is None else total
    S = model.dims.image
    if out is None:
        out = torch.empty((max(B, 1), 3, S, S), dtype=torch.float32, device="cuda")
    rc = model._lib.mmee_preprocess_images(model._h, B, C.byref(img), C.c_void_p(out.data_ptr()), None)
    return rc, out


def test_c_abi_errors_leave_the_engine_usable():
    model, dims, docs = _engine("tiny_ramp_conf")
    lib = model._lib
    a = page(30, 20, 1, seed=3)
    data = torch.from_numpy(a.reshape(-1).copy()).cuda()
    want = image_port.preprocess(a, dims.image)
    bad = {
        "channels 2": dict(channels=2),
        "channels 0": dict(channels=0),
        "height 0": dict(sizes=[[0, 20]]),
        "width 16385": dict(sizes=[[1, 16385]]),
        "height -1": dict(sizes=[[-1, 20]]),
        "past total_bytes": dict(offsets=[1]),
        "negative offset": dict(offsets=[-1]),
        "total_bytes too small": dict(total=599),
        "B = 0": dict(B=0),
        "B > max_batch": dict(B=model.max_batch + 1),
    }
    for tag, kw in bad.items():
        args = dict(B=1, offsets=[0], sizes=[[30, 20]], channels=1)
        args.update(kw)
        B = args.pop("B")
        rc, _ = _c_preprocess(model, B, data, **args)
        msg = lib.mmee_last_error().decode()
        assert rc != 0 and msg, tag
        rc, out = _c_preprocess(model, 1, data, [0], [[30, 20]], 1)
        assert rc == 0, lib.mmee_last_error().decode()
        assert np.array_equal(out[0].cpu().numpy(), want), tag
    # the host forward checks the same before anything is enqueued
    text = {k: v[:1].contiguous() for k, v in docs.items() if k != "pixel_values"}
    img = _lib.Images()
    host = a.reshape(-1).copy()
    offs, szs = np.zeros(1, np.int64), np.array([[30, 20]], np.int32)
    img.data, img.offsets, img.sizes, img.channels, img.total_bytes = host.ctypes.data, offs.ctypes.data, \
        szs.ctypes.data, 2, host.size
    thr = np.full(max(model.n_exits, 1), 0.5, np.float32)
    pol = _lib.Policy()
    pol.criterion, pol.mode, pol.thresholds = 0, 1, thr.ctypes.data_as(C.POINTER(C.c_float))
    logits = torch.empty((1, dims.n_labels)); ex = torch.empty(1, dtype=torch.int32)
    out = _lib.Outputs()
    out.logits, out.exit_index = logits.data_ptr(), ex.data_ptr()
    rc = lib.mmee_forward_images(model._h, 1, C.c_void_p(text["input_ids"].data_ptr()),
                                 C.c_void_p(text["bbox"].data_ptr()), C.c_void_p(text["attention_mask"].data_ptr()),
                                 C.byref(img), C.byref(pol), C.byref(out))
    assert rc != 0 and "channels" in lib.mmee_last_error().decode()
    r = model.infer(**text, images=[a], exit_threshold=0.5)
    w = model.infer(**text, pixel_values=torch.from_numpy(want[None]), exit_threshold=0.5)
    assert torch.equal(r.logits, w.logits)


def test_engine_without_rgb_channels_rejects_images():
    from mmee.model import B200EEForSequenceClassification

    dims = ModelDims.tiny(channels=1)
    ee = ExitConfig.from_dict(dict(exits=[1, 2, 3], encoder_layer_strategy="ramp", inference_strategy="max_confidence"))
    model = B200EEForSequenceClassification(dims, ee, synth.make_state_dict(dims, ee, seed=0), device=0, max_batch=2)
    with pytest.raises(RuntimeError, match="channels"):
        model.preprocess_images([page(40, 30, 1, seed=0)])
    model.close()


def test_entry_points_without_images_refuse_them():
    model, dims, docs = _engine("tiny_ramp_conf")
    with pytest.raises(ValueError, match="images"):
        model.infer_submit(**docs, images=[page(10, 10, 1, seed=0)] * docs["pixel_values"].shape[0])
    with pytest.raises(ValueError, match="not both"):
        model.infer(**docs, images=[page(10, 10, 1, seed=0)] * docs["pixel_values"].shape[0])
    text = {k: v for k, v in docs.items() if k != "pixel_values"}
    with pytest.raises(ValueError, match="images for"):
        model.infer(**text, images=[page(10, 10, 1, seed=0)])
    assert pack_images([page(4, 4, 1, seed=0)]).data.is_pinned()
