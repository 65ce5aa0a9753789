"""Python mirror of the reference's model API for the early-exit inference path, backed by libmmee.

`B200EEForSequenceClassification.forward(**batch)` takes the same keyword arguments as the reference's
`LayoutLMv3EEForSequenceClassification.forward` (EE/models/LayoutLMv3.py:696-711; call site
EE/utils.py:179) and returns an object with the fields its consumers read (EE/utils.py:182-193,
EE/IC_only.py:93): `logits`, `exit_states` (tuple of (head_logits, criterion)), `exit_criteria`,
`gated_logits` (gate mode).  That is the DENSE mode: every exit for every document, exactly what the
reference computes.

`infer(**batch, exit_threshold=..., temperatures=...)` is the path the reference only emulates post-hoc
(EE/policy.py:12-53): documents leave at the first exit whose calibrated criterion passes its threshold
and deeper layers run on the survivors only.  It returns what `Policy` returns — `(exits_store,
predictions, exit_distribution)` — plus per-document criteria and the exit histogram.

Everything numeric happens in the CUDA engine; torch is used for tensor storage and streams only.
"""
from __future__ import annotations

import ctypes as C
import weakref
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib
from .config import ExitConfig, ModelDims
from .images import PackedImages, as_packed


@dataclass
class EESequenceClassifierOutput:
    """Field-compatible with the reference dataclass (EE/models/EE_modules.py:231-273)."""
    logits: torch.Tensor = None
    loss: Optional[torch.Tensor] = None
    hidden_states: Optional[Tuple[torch.Tensor]] = None
    attentions: Optional[Tuple[torch.Tensor]] = None
    exit_losses: Optional[Tuple[torch.Tensor]] = None
    exit_criteria: Optional[List[torch.Tensor]] = None
    exit_states: Optional[Tuple[Tuple[torch.Tensor, torch.Tensor], ...]] = None
    gated_logits: Optional[Tuple[torch.Tensor, ...]] = None
    lte_output: Optional[Tuple[torch.Tensor]] = None
    # engine extras
    exit_logits: Optional[torch.Tensor] = None      # [E+1, B, K] as stored by EE/utils.py:160-193
    exit_index: Optional[torch.Tensor] = None       # [B] first exit passing the configured threshold

    def __getitem__(self, i):
        return (self.logits,)[i] if self.loss is None else (self.loss, self.logits)[i]


@dataclass
class EarlyExitResult:
    exits_store: np.ndarray            # int32 [N]   (Policy return 0)
    predictions: torch.Tensor          # float64 [N, K] on CPU (Policy return 1)
    exit_distribution: Dict[int, float]  # (Policy return 2)
    criteria: np.ndarray               # float32 [N] criterion at the exit taken
    exit_hist: np.ndarray              # int64 [E+1]
    logits: torch.Tensor               # float32 [N, K] (device or host, as the inputs were)

    def __iter__(self):                # unpack like the reference Policy methods
        return iter((self.exits_store, self.predictions, self.exit_distribution))


def bucket_lut(num_buckets: int, max_distance: int, n: int = 1024) -> np.ndarray:
    """|rel| -> bucket offset with the exact torch ops of HF relative_position_bucket
    (modeling_layoutlmv3.py:393-414), so device lookups are bit-identical to the reference."""
    import math

    nb = num_buckets // 2
    rel = torch.arange(n, dtype=torch.long)
    max_exact = nb // 2
    is_small = rel < max_exact
    large = max_exact + (
        torch.log(rel.float() / max_exact) / math.log(max_distance / max_exact) * (nb - max_exact)
    ).to(torch.long)
    large = torch.min(large, torch.full_like(large, nb - 1))
    return torch.where(is_small, rel, large).to(torch.uint8).numpy()


EMBEDDING_EXIT_CODES = {"vision_avg": -2, "text_avg": -1, "text_visual_concat": 0}   # include/mmee.h MMEE_EXIT_*
CRITERION_CODES = {"max_confidence": 0, "entropy": 1, "lte": 2}                        # include/mmee.h MMEE_CRIT_*


class B200EEForSequenceClassification:
    def __init__(self, dims: ModelDims, ee: Union[ExitConfig, dict], state_dict: Dict[str, torch.Tensor],
                 device: int = 0, max_batch: int = 256, dtype: str = "bf16"):
        """dtype: arithmetic of the dense contractions — "bf16" (default: bf16 tensor-core operands, logits within
        1e-2 of the reference) or "fp32" (fp32-parity mode: split-bf16 operands, three tensor-core products per
        contraction, logits within 1e-4; the reference itself computes in fp32, EE/utils.py:160-164)."""
        if isinstance(ee, dict):
            ee = ExitConfig.from_dict(ee)
        if dtype not in _lib.COMPUTE_DTYPES:
            raise ValueError(f"dtype must be one of {sorted(_lib.COMPUTE_DTYPES)}")
        self.dtype = dtype
        dims.check()
        for x in ee.exits:
            if isinstance(x, str) and x not in EMBEDDING_EXIT_CODES:
                raise NotImplementedError(f"unknown embedding-level exit {x!r}")
        self.dims, self.ee = dims, ee
        self.device_index = device
        self.max_batch = max_batch
        # reference order: vision_avg, text_avg, text_visual_concat, then the encoder layers (EE/models/LayoutLMv3.py:465-606)
        self.exit_layers = sorted(EMBEDDING_EXIT_CODES[x] for x in ee.exits if isinstance(x, str)) \
            + sorted(ee.encoder_exit_layers)
        self.n_exits = len(self.exit_layers)
        self._plans = weakref.WeakSet()     # live ForwardPlans: closed before the engine they run on
        self._lib = _lib.load()
        d = _lib.ModelDesc()
        d.hidden, d.layers, d.heads, d.inter = dims.hidden, dims.layers, dims.heads, dims.inter
        d.n_text, d.image, d.patch, d.channels = dims.n_text, dims.image, dims.patch, dims.channels
        d.n_labels, d.coord, d.shape = dims.n_labels, dims.coord, dims.shape
        d.vocab, d.max_pos, d.max_2d = dims.vocab, dims.max_pos, dims.max_2d
        d.rel_bins, d.max_rel, d.rel2d_bins, d.max_rel2d = dims.rel_bins, dims.max_rel, dims.rel2d_bins, dims.max_rel2d
        d.pad_id, d.ln_eps, d.vis_ln_eps = dims.pad_id, dims.ln_eps, dims.vis_ln_eps
        d.n_exits = self.n_exits
        for i, l in enumerate(self.exit_layers):
            d.exit_after_layer[i] = l
        d.head_kind = 0 if ee.encoder_layer_strategy == "ramp" else 1
        d.head_layers = ee.exit_head_num_layers
        d.compute_dtype = _lib.COMPUTE_DTYPES[dtype]
        self._h = C.c_void_p()
        _lib.check(self._lib.mmee_create(C.byref(d), device, max_batch, C.byref(self._h)))
        self._load_weights(state_dict)

    # ------------------------------------------------------------------ construction helpers
    @staticmethod
    def spec_from_reference(model):
        """(ModelDims, ExitConfig, fp32 CPU state dict) of a constructed reference
        `LayoutLMv3EEForSequenceClassification` (or anything with the same `.config` / `.state_dict()`)."""
        c = model.config
        dims = ModelDims(hidden=c.hidden_size, layers=c.num_hidden_layers, heads=c.num_attention_heads,
                         inter=c.intermediate_size, image=c.input_size, patch=c.patch_size,
                         channels=c.num_channels, n_labels=c.num_labels, coord=c.coordinate_size,
                         shape=c.shape_size, vocab=c.vocab_size, max_pos=c.max_position_embeddings,
                         max_2d=c.max_2d_position_embeddings, rel_bins=c.rel_pos_bins, max_rel=c.max_rel_pos,
                         rel2d_bins=c.rel_2d_pos_bins, max_rel2d=c.max_rel_2d_pos, pad_id=c.pad_token_id,
                         ln_eps=c.layer_norm_eps)
        ee = ExitConfig.from_dict({k: (v if isinstance(v, (list, tuple, int, float)) else str(v))
                                   for k, v in dict(c.EE_config).items()})
        sd = {k: v.detach().float().cpu() for k, v in model.state_dict().items()}
        return dims, ee, sd

    @classmethod
    def from_reference(cls, model, device: int = 0, max_batch: int = 256, dtype: str = "bf16"):
        """Build the engine from a constructed reference model (reads HF dims, `config.EE_config`, weights)."""
        dims, ee, sd = cls.spec_from_reference(model)
        return cls(dims, ee, sd, device=device, max_batch=max_batch, dtype=dtype)

    def _load_weights(self, sd: Dict[str, torch.Tensor]) -> None:
        keep = []
        for name, t in sd.items():
            if not torch.is_tensor(t) or not t.dtype.is_floating_point:
                continue
            t = t.detach().to(torch.float32).contiguous().cpu()
            keep.append(t)
            shape = (C.c_int64 * max(t.dim(), 1))(*t.shape)
            _lib.check(self._lib.mmee_set_weight(self._h, name.encode(), C.c_void_p(t.data_ptr()), shape, t.dim()))
        l1 = bucket_lut(self.dims.rel_bins, self.dims.max_rel)
        l2 = bucket_lut(self.dims.rel2d_bins, self.dims.max_rel2d)
        _lib.check(self._lib.mmee_set_bucket_lut(self._h, 0, l1.ctypes.data_as(C.c_void_p), len(l1)))
        _lib.check(self._lib.mmee_set_bucket_lut(self._h, 1, l2.ctypes.data_as(C.c_void_p), len(l2)))
        _lib.check(self._lib.mmee_finalize_weights(self._h))

    def close(self) -> None:
        for p in list(getattr(self, "_plans", ())):
            p.close()
        if getattr(self, "_h", None) and self._h.value:
            self._lib.mmee_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def eval(self):
        return self

    def _default_criterion(self) -> str:
        """Early-exit decision rule of `infer*`: the learned-to-exit scorer when EE_config["use_lte"] is set
        (EE/models/LayoutLMv3.py:140, 231-268: sigmoid(lte_classifier(CLS)) < global_threshold, encoder exits
        after layer l < number of encoder exits only), else the configured confidence criterion."""
        return "lte" if self.ee.use_lte else self.ee.inference_strategy

    def __call__(self, *a, **k):
        return self.forward(*a, **k)

    # ------------------------------------------------------------------ engine call
    def _run(self, input_ids, attention_mask, bbox, pixel_values, criterion: str, mode: int,
             thresholds: Sequence[float], temperatures: Optional[Sequence[float]], want_all: bool,
             blocking: bool = True, plan: Optional["ForwardPlan"] = None, images=None):
        """One forward through the engine; `plan` given: a run of that captured forward plan instead (same inputs,
        same outputs).  `images` (uint8 pages, see `mmee.images`) in place of `pixel_values`: with host inputs and no
        plan the forward is `mmee_forward_images`; otherwise the pages are preprocessed on the device first
        (`preprocess_images`) and the forward runs on the device (results read back for host inputs)."""
        if images is not None:
            if pixel_values is not None:
                raise ValueError("pass either pixel_values or images, not both")
            images = as_packed(images)
            n_docs, px_device = len(images), images.data.device
        elif pixel_values is None:
            raise ValueError("pixel_values (or images) are required (multimodal and image-only paths)")
        else:
            n_docs, px_device = pixel_values.shape[0], pixel_values.device
        if input_ids is None:
            if self.dims.n_text != 0:
                raise ValueError("this engine was built for the multimodal path: input_ids and bbox are required "
                                 "(build it with ModelDims(n_text=0) for the image-only path)")
            input_ids = torch.zeros((n_docs, 0), dtype=torch.int64, device=px_device)
        B, T = input_ids.shape
        if T != self.dims.n_text:
            raise ValueError(f"expected {self.dims.n_text} text tokens (padding='max_length'), got {T}")
        if images is not None and len(images) != B:
            raise ValueError(f"{len(images)} images for {B} documents")
        if attention_mask is None:
            attention_mask = torch.ones_like(input_ids)
        if bbox is None:
            bbox = torch.zeros((B, T, 4), dtype=torch.long, device=input_ids.device)
        on_dev = input_ids.is_cuda
        to_host = False
        if images is not None and (on_dev or plan is not None):
            pixel_values = self.preprocess_images(images)
            images = None
            if not on_dev:          # a plan over host inputs: run its device path and read the results back
                input_ids, to_host, on_dev = input_ids.to(pixel_values.device), True, True
        dev = input_ids.device
        ids = input_ids.to(torch.int64).contiguous()
        msk = attention_mask.to(device=dev, dtype=torch.int64).contiguous()
        bb = bbox.to(device=dev, dtype=torch.int64).contiguous()
        px = None if images is not None else pixel_values.to(device=dev, dtype=torch.float32).contiguous()
        E1, K = self.n_exits + 1, self.dims.n_labels
        kw = dict(device=dev)
        logits = torch.empty((B, K), dtype=torch.float32, **kw)
        exit_index = torch.empty((B,), dtype=torch.int32, **kw)
        crit = torch.empty((B,), dtype=torch.float32, **kw)
        hist = torch.zeros((E1,), dtype=torch.int64, **kw)
        out = _lib.Outputs()
        out.logits, out.exit_index, out.criterion = logits.data_ptr(), exit_index.data_ptr(), crit.data_ptr()
        out.exit_hist = hist.data_ptr()
        all_l = all_h = all_c = None
        if want_all:
            all_l = torch.empty((E1, B, K), dtype=torch.float32, **kw)
            all_h = torch.empty((E1, B, K), dtype=torch.float32, **kw)
            all_c = torch.empty((E1, B), dtype=torch.float32, **kw)
            out.all_exit_logits, out.all_head_logits, out.all_criteria = all_l.data_ptr(), all_h.data_ptr(), all_c.data_ptr()
        thr = np.broadcast_to(np.asarray(thresholds, dtype=np.float32), (max(self.n_exits, 1),)).copy()
        pol = _lib.Policy()
        pol.criterion = CRITERION_CODES[criterion]
        pol.mode = mode
        pol.thresholds = thr.ctypes.data_as(C.POINTER(C.c_float))
        tmp = None
        if temperatures is not None:
            tmp = np.asarray(temperatures, dtype=np.float32).reshape(-1).copy()
            if tmp.shape[0] != E1:
                raise ValueError(f"temperatures must have {E1} entries (one per exit + final)")
            pol.temperatures = tmp.ctypes.data_as(C.POINTER(C.c_float))
        if images is not None:      # host forward over uint8 pages
            if images.data.is_cuda:
                images = PackedImages(images.data.cpu(), images.offsets, images.sizes, images.channels)
            img = images.c_struct()
            _lib.check(self._lib.mmee_forward_images(self._h, B, C.c_void_p(ids.data_ptr()), C.c_void_p(bb.data_ptr()),
                                                     C.c_void_p(msk.data_ptr()), C.byref(img), C.byref(pol),
                                                     C.byref(out)))
            return dict(logits=logits, exit_index=exit_index, criterion=crit, hist=hist, all_logits=all_l,
                        all_head=all_h, all_crit=all_c, _keep=(ids, msk, bb, images, thr, tmp))
        args = (C.c_void_p(ids.data_ptr()), C.c_void_p(bb.data_ptr()), C.c_void_p(msk.data_ptr()),
                C.c_void_p(px.data_ptr()), C.byref(pol), C.byref(out))
        if plan is None:
            args = (self._h, B) + args
            fwd_device, fwd_host = self._lib.mmee_forward_device, self._lib.mmee_forward
        else:
            if B != plan.batch_size:
                raise ValueError(f"this plan was captured for {plan.batch_size} documents, got {B}")
            args = (plan._handle(),) + args
            fwd_device, fwd_host = self._lib.mmee_plan_forward_device, self._lib.mmee_plan_forward
        if on_dev:
            if dev.index is not None and dev.index != self.device_index:
                raise ValueError("inputs live on a different GPU than the engine")
            # torch's legacy default stream has handle 0, which the C ABI reads as "the engine's own stream,
            # synchronous": pass cudaStreamLegacy (1) instead, so the forward is ordered after the torch work that
            # produced the inputs and stays asynchronous; blocking callers wait explicitly below
            stream = torch.cuda.current_stream(dev).cuda_stream or 1
            _lib.check(fwd_device(*args, C.c_void_p(stream)))
            if blocking:
                _lib.check(self._lib.mmee_sync(self._h, C.c_void_p(stream)))
        else:
            _lib.check(fwd_host(*args))
        r = dict(logits=logits, exit_index=exit_index, criterion=crit, hist=hist, all_logits=all_l,
                 all_head=all_h, all_crit=all_c, _keep=(ids, msk, bb, px, thr, tmp))
        if to_host:
            r.update({k: v.cpu() for k, v in r.items() if torch.is_tensor(v)})
        return r

    # ------------------------------------------------------------------ reference-shaped forward (dense)
    def forward(self, input_ids=None, attention_mask=None, bbox=None, pixel_values=None, labels=None,
                temperatures: Optional[Sequence[float]] = None, images=None, **unused) -> EESequenceClassifierOutput:
        """`images`: uint8 pages (a `mmee.images.PackedImages` or what `pack_images` takes) instead of `pixel_values`;
        the engine resizes and normalises them as the reference's image processor does.  Same for `infer*`."""
        crit_name = self.ee.inference_strategy
        r = self._run(input_ids, attention_mask, bbox, pixel_values, crit_name, 0,
                      [float(self.ee.global_threshold)], temperatures, True, images=images)
        E, K = self.n_exits, self.dims.n_labels
        gate = self.ee.encoder_layer_strategy == "gate"
        n_head = 2 if gate else K
        fn = _entropy if crit_name == "entropy" else _max_confidence
        exit_states = []
        exit_criteria = []
        for j in range(E):
            head = r["all_head"][j, :, :n_head]
            c = fn(head)                     # reference: criterion of the raw head output (EE/models/LayoutLMv3.py:240)
            exit_states.append((head, c))
            exit_criteria.append(c)
        final = r["all_logits"][E]
        exit_criteria.append(fn(final))      # EE/models/LayoutLMv3.py:871-872
        gated = tuple(r["all_logits"][j] for j in range(E)) if gate else ()
        loss = None
        if labels is not None:
            loss = torch.nn.functional.cross_entropy(final, labels.to(final.device).view(-1))
        return EESequenceClassifierOutput(
            logits=final, loss=loss, exit_losses=[], exit_criteria=exit_criteria, exit_states=tuple(exit_states),
            gated_logits=gated, exit_logits=r["all_logits"], exit_index=r["exit_index"])

    # ------------------------------------------------------------------ real early exit
    def infer(self, input_ids=None, attention_mask=None, bbox=None, pixel_values=None, labels=None,
              exit_threshold: Union[float, Sequence[float], None] = None,
              temperatures: Optional[Sequence[float]] = None, criterion: Optional[str] = None,
              early_exit: bool = True, return_all: bool = False, images=None, **unused) -> EarlyExitResult:
        thr = self.ee.global_threshold if exit_threshold is None else exit_threshold
        crit_name = criterion or self._default_criterion()
        r = self._run(input_ids, attention_mask, bbox, pixel_values, crit_name, 1 if early_exit else 0,
                      np.atleast_1d(np.asarray(thr, dtype=np.float32)), temperatures, return_all, images=images)
        return self._early_exit_result(r, return_all)

    def _early_exit_result(self, r, return_all: bool) -> EarlyExitResult:
        ex = r["exit_index"].cpu().numpy().astype(np.int32)
        hist = r["hist"].cpu().numpy()
        n = ex.shape[0]
        dist = {e: float(hist[e]) / n for e in range(self.n_exits + 1)}
        res = EarlyExitResult(exits_store=ex, predictions=r["logits"].detach().cpu().to(torch.float64),
                              exit_distribution=dist, criteria=r["criterion"].cpu().numpy(), exit_hist=hist,
                              logits=r["logits"])
        if return_all:
            res.all_exit_logits = r["all_logits"]
            res.all_criteria = r["all_crit"]
        return res

    def infer_device(self, input_ids=None, attention_mask=None, bbox=None, pixel_values=None, labels=None,
                     exit_threshold: Union[float, Sequence[float], None] = None,
                     temperatures: Optional[Sequence[float]] = None, criterion: Optional[str] = None,
                     early_exit: bool = True, images=None, **unused) -> Dict[str, torch.Tensor]:
        """`infer` without the device->host read-back: results stay on the GPU (logits f32 [B,K], exit_index i32 [B],
        criterion f32 [B], hist i64 [E+1]) and the call is asynchronous on the current stream — what the
        data-parallel gather (`mmee.dist`) and pipelined callers want.  Inputs must be CUDA tensors."""
        thr = self.ee.global_threshold if exit_threshold is None else exit_threshold
        crit_name = criterion or self._default_criterion()
        r = self._run(input_ids, attention_mask, bbox, pixel_values, crit_name, 1 if early_exit else 0,
                      np.atleast_1d(np.asarray(thr, dtype=np.float32)), temperatures, False, blocking=False,
                      images=images)
        return self._device_result(r)

    @staticmethod
    def _device_result(r) -> Dict[str, torch.Tensor]:
        return {"logits": r["logits"], "exit_index": r["exit_index"], "criterion": r["criterion"], "hist": r["hist"]}

    # ------------------------------------------------------------------ uint8 images
    def preprocess_images(self, images) -> torch.Tensor:
        """Pixel values f32 [B, 3, S, S] (S = dims.image) on this engine's GPU from uint8 pages (a `PackedImages` or
        what `mmee.images.pack_images` takes), computed on the device and asynchronous on the current stream:
        Pillow's bilinear resize to S x S, then (r / 255 - 0.5) / 0.5, bit for bit as the reference's LayoutLMv3 image
        processor (`mmee_preprocess_images`)."""
        p = as_packed(images)
        dev = torch.device("cuda", self.device_index)
        data = p.data.to(dev, non_blocking=True)
        S = self.dims.image
        out = torch.empty((len(p), 3, S, S), dtype=torch.float32, device=dev)
        img = p.c_struct(data)
        stream = torch.cuda.current_stream(dev).cuda_stream or 1     # see _run: 0 would mean "engine stream, sync"
        _lib.check(self._lib.mmee_preprocess_images(self._h, len(p), C.byref(img), C.c_void_p(out.data_ptr()),
                                                    C.c_void_p(stream)))
        return out

    # ------------------------------------------------------------------ captured forwards
    def plan(self, batch_size: int, criterion: Optional[str] = None, early_exit: bool = True,
             return_all: bool = False) -> "ForwardPlan":
        """Capture the forward for exactly `batch_size` documents into a CUDA graph (`mmee_plan_create`) and return
        a `ForwardPlan` whose `infer` / `infer_device` run it: one graph launch per call instead of ~100 kernel
        launches, and in early-exit mode no launches at all for the layers after the last document has left.
        Thresholds and temperatures stay arguments of every call; the criterion, the mode and `return_all` are fixed
        here.  Results are bit-identical to `infer` / `infer_device` on the same documents."""
        p = ForwardPlan(self, batch_size, criterion or self._default_criterion(), early_exit, return_all)
        self._plans.add(p)
        return p

    # ------------------------------------------------------------------ pipelined host path
    def infer_submit(self, input_ids=None, attention_mask=None, bbox=None, pixel_values=None, labels=None,
                     exit_threshold: Union[float, Sequence[float], None] = None,
                     temperatures: Optional[Sequence[float]] = None, criterion: Optional[str] = None,
                     early_exit: bool = True, **unused):
        """Enqueue one early-exit forward over HOST tensors (pinned memory recommended) and return a ticket without
        waiting; at most two tickets may be outstanding.  The upload of this batch overlaps the forward of the
        previous one (`mmee_forward_submit`).  Pass the ticket to `infer_collect`."""
        if "images" in unused:
            raise ValueError("infer_submit takes pixel_values only (use infer / infer_device for uint8 images)")
        if pixel_values is None or pixel_values.is_cuda:
            raise ValueError("infer_submit takes host tensors (use infer / infer_device for CUDA tensors)")
        if input_ids is None:
            input_ids = torch.zeros((pixel_values.shape[0], 0), dtype=torch.int64)
        B, T = input_ids.shape
        if T != self.dims.n_text:
            raise ValueError(f"expected {self.dims.n_text} text tokens (padding='max_length'), got {T}")
        if attention_mask is None:
            attention_mask = torch.ones_like(input_ids)
        if bbox is None:
            bbox = torch.zeros((B, T, 4), dtype=torch.long)
        ids = input_ids.to(torch.int64).contiguous()
        msk = attention_mask.to(torch.int64).contiguous()
        bb = bbox.to(torch.int64).contiguous()
        px = pixel_values.to(torch.float32).contiguous()
        thr = self.ee.global_threshold if exit_threshold is None else exit_threshold
        thr = np.broadcast_to(np.asarray(thr, dtype=np.float32), (max(self.n_exits, 1),)).copy()
        pol = _lib.Policy()
        pol.criterion = CRITERION_CODES[criterion or self._default_criterion()]
        pol.mode = 1 if early_exit else 0
        pol.thresholds = thr.ctypes.data_as(C.POINTER(C.c_float))
        tmp = None
        if temperatures is not None:
            tmp = np.asarray(temperatures, dtype=np.float32).reshape(-1).copy()
            if tmp.shape[0] != self.n_exits + 1:
                raise ValueError(f"temperatures must have {self.n_exits + 1} entries (one per exit + final)")
            pol.temperatures = tmp.ctypes.data_as(C.POINTER(C.c_float))
        t = self._lib.mmee_forward_submit(self._h, B, C.c_void_p(ids.data_ptr()), C.c_void_p(bb.data_ptr()),
                                          C.c_void_p(msk.data_ptr()), C.c_void_p(px.data_ptr()), C.byref(pol))
        if t < 0:
            _lib.check(t)
        return {"ticket": t, "B": B, "_keep": (ids, msk, bb, px, thr, tmp)}

    def infer_collect(self, ticket) -> EarlyExitResult:
        """Wait for a submitted forward and read its results back (same result object as `infer`)."""
        B, K, E1 = ticket["B"], self.dims.n_labels, self.n_exits + 1
        logits = torch.empty((B, K), dtype=torch.float32)
        exit_index = torch.empty((B,), dtype=torch.int32)
        crit = torch.empty((B,), dtype=torch.float32)
        hist = torch.zeros((E1,), dtype=torch.int64)
        out = _lib.Outputs()
        out.logits, out.exit_index, out.criterion = logits.data_ptr(), exit_index.data_ptr(), crit.data_ptr()
        out.exit_hist = hist.data_ptr()
        _lib.check(self._lib.mmee_forward_collect(self._h, ticket["ticket"], C.byref(out)))
        ticket["_keep"] = None
        ex = exit_index.numpy().astype(np.int32)
        h = hist.numpy()
        dist = {e: float(h[e]) / B for e in range(E1)}
        return EarlyExitResult(exits_store=ex, predictions=logits.to(torch.float64), exit_distribution=dist,
                               criteria=crit.numpy(), exit_hist=h, logits=logits)

    def sync(self) -> None:
        """Wait for the forwards enqueued on torch's current stream (`infer_device` is asynchronous) and raise if a
        device-side check tripped (input ids / boxes out of range, attention guard): `mmee_sync`."""
        stream = torch.cuda.current_stream(torch.device("cuda", self.device_index)).cuda_stream or 1
        _lib.check(self._lib.mmee_sync(self._h, C.c_void_p(stream)))

    # ------------------------------------------------------------------ introspection
    def last_launch_count(self) -> int:
        return int(self._lib.mmee_last_launch_count(self._h))

    def set_profiling(self, on: bool) -> None:
        self._lib.mmee_set_profiling(self._h, 1 if on else 0)

    def debug_read(self, name: str, dtype, count: int) -> np.ndarray:
        """Test hook: first `count` elements of an internal activation buffer."""
        buf = np.zeros(count, dtype=dtype)
        n = self._lib.mmee_debug_read(self._h, name.encode(), buf.ctypes.data_as(C.c_void_p), buf.nbytes)
        if n < 0:
            _lib.check(-1)
        return buf

    def last_stage_ms(self) -> Dict[str, float]:
        """Per-stage device time in ms, AVERAGED over the forwards run since `set_profiling(True)` (or the previous
        call); "forwards" = how many that were."""
        _lib.check(self._lib.mmee_collect_profile(self._h))
        n = float(self._lib.mmee_last_stage_ms(self._h, b"forwards")) or 1.0
        out = {k: float(self._lib.mmee_last_stage_ms(self._h, k.encode())) / n
               for k in ("total", "embed", "gemm", "attention", "norm", "exit", "end")}
        out["forwards"] = n
        return out

    def bucket_lut_in_use(self, which: int) -> np.ndarray:
        buf = np.zeros(4096, dtype=np.uint8)
        n = self._lib.mmee_get_bucket_lut(self._h, which, buf.ctypes.data_as(C.c_void_p), buf.size)
        return buf[:n]


class ForwardPlan:
    """A forward captured for a fixed batch size, criterion, mode and `return_all` (`B200EEForSequenceClassification.plan`).

    `infer` / `infer_device` take the same inputs as the model's methods of that name (host or CUDA tensors, same
    rules) for exactly `batch_size` documents and return the same results, bit for bit.  The plan holds a reference to
    its model; `close()` (or garbage collection) frees the graph."""

    def __init__(self, model: B200EEForSequenceClassification, batch_size: int, criterion: str, early_exit: bool,
                 return_all: bool):
        if criterion not in CRITERION_CODES:
            raise ValueError(f"criterion must be one of {sorted(CRITERION_CODES)}")
        self.model = model
        self.batch_size = int(batch_size)
        self.criterion, self.early_exit, self.return_all = criterion, bool(early_exit), bool(return_all)
        self._h = C.c_void_p()
        shape = _lib.Policy()
        shape.criterion = CRITERION_CODES[criterion]
        shape.mode = 1 if early_exit else 0
        _lib.check(model._lib.mmee_plan_create(model._h, self.batch_size, C.byref(shape), 1 if return_all else 0,
                                               C.byref(self._h)))

    def _handle(self) -> C.c_void_p:
        if not self._h.value:
            raise RuntimeError("this forward plan has been closed")
        return self._h

    def _call(self, batch, exit_threshold, temperatures, criterion, early_exit, want_all, blocking):
        m = self.model
        thr = m.ee.global_threshold if exit_threshold is None else exit_threshold
        # criterion / early_exit default to the plan's; others are passed on and rejected by mmee_plan_forward
        crit_name = criterion or self.criterion
        mode = 1 if (self.early_exit if early_exit is None else early_exit) else 0
        return m._run(batch.get("input_ids"), batch.get("attention_mask"), batch.get("bbox"),
                      batch.get("pixel_values"), crit_name, mode, np.atleast_1d(np.asarray(thr, dtype=np.float32)),
                      temperatures, want_all, blocking=blocking, plan=self, images=batch.get("images"))

    def infer(self, exit_threshold: Union[float, Sequence[float], None] = None,
              temperatures: Optional[Sequence[float]] = None, criterion: Optional[str] = None,
              early_exit: Optional[bool] = None, **batch) -> EarlyExitResult:
        """Same as `B200EEForSequenceClassification.infer` (with this plan's `return_all`)."""
        r = self._call(batch, exit_threshold, temperatures, criterion, early_exit, self.return_all, True)
        return self.model._early_exit_result(r, self.return_all)

    def infer_device(self, exit_threshold: Union[float, Sequence[float], None] = None,
                     temperatures: Optional[Sequence[float]] = None, criterion: Optional[str] = None,
                     early_exit: Optional[bool] = None, **batch) -> Dict[str, torch.Tensor]:
        """Same as `B200EEForSequenceClassification.infer_device`: asynchronous on the current stream."""
        r = self._call(batch, exit_threshold, temperatures, criterion, early_exit, False, False)
        return self.model._device_result(r)

    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            self.model._lib.mmee_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _entropy(x: torch.Tensor) -> torch.Tensor:
    """EE/models/EE_modules.py:149-154 (output packaging only; the exit decision is made on the device)."""
    ex = torch.exp(x)
    a = ex.sum(dim=1)
    return torch.log(a) - (x * ex).sum(dim=1) / a


def _max_confidence(x: torch.Tensor) -> torch.Tensor:
    """EE/models/EE_modules.py:157-160."""
    return torch.softmax(x, dim=1).max(dim=1)[0]
