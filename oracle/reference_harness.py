"""TEST INFRASTRUCTURE — runs the UNMODIFIED reference model on CPU (dev container only).

Imports `/root/reference/EE/models/LayoutLMv3.py` verbatim and applies the five
API shims of SURVEY.md Appendix B that bridge the reference's pinned
transformers ^4.26 to the installed 5.x (signature drift only; arithmetic is
untouched).  `/root/reference` does not exist on the GPU box, so nothing here
may be imported by `-m gpu` tests, `smoke()` or `bench.py`; it is used by
`tests/golden/make_golden.py` to generate the committed golden vectors and by
CPU tests that validate `oracle/port.py` when the reference is present.
"""
from __future__ import annotations

import os
import sys
import types

REFERENCE_ROOT = os.environ.get("MMEE_REFERENCE_ROOT", "/root/reference")
_loaded = None


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "EE", "models", "LayoutLMv3.py"))


def _install_stubs() -> None:
    # fvcore is imported at EE/models/EE_modules.py:10 but only used by training/accounting code.
    if "fvcore" not in sys.modules:
        fv = types.ModuleType("fvcore")
        fvnn = types.ModuleType("fvcore.nn")
        fvnn.FlopCountAnalysis = object
        fvnn.parameter_count = lambda *a, **k: {}
        fv.nn = fvnn
        sys.modules["fvcore"] = fv
        sys.modules["fvcore.nn"] = fvnn


def load():
    """Return the reference module `models.LayoutLMv3` with shims applied (idempotent)."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not available():
        raise RuntimeError(f"reference not present at {REFERENCE_ROOT}")
    _install_stubs()
    ee_dir = os.path.join(REFERENCE_ROOT, "EE")
    if ee_dir not in sys.path:
        sys.path.insert(0, ee_dir)
    import models.LayoutLMv3 as L  # noqa: E402  (the reference, verbatim)
    from transformers.models.layoutlmv3 import modeling_layoutlmv3 as HF

    # (1) v5 dropped the `device` positional of get_extended_attention_mask (ref :622)
    _ext = HF.LayoutLMv3Model.get_extended_attention_mask
    L.LayoutLMv3ModelEE.get_extended_attention_mask = (
        lambda s, am, shape, device=None, dtype=None: _ext(s, am, shape, dtype=dtype))
    # (2) get_head_mask removed in v5 (ref :631)
    L.LayoutLMv3ModelEE.get_head_mask = lambda s, hm, n, *a, **k: [None] * n
    # (3) v5 dropped the `hidden_states` arg of the bias builders (ref :171, :176)
    _o1, _o2 = HF.LayoutLMv3Encoder._cal_1d_pos_emb, HF.LayoutLMv3Encoder._cal_2d_pos_emb
    L.LayoutLMv3EncoderEE._cal_1d_pos_emb = lambda s, hs, pid: _o1(s, pid)
    L.LayoutLMv3EncoderEE._cal_2d_pos_emb = lambda s, hs, bb: _o2(s, bb)
    # (4) v5 layer.forward: no head_mask positional, returns a Tensor instead of a tuple (ref :209-218)
    if not getattr(HF.LayoutLMv3Layer.forward, "_mmee_shim", False):
        _lf = HF.LayoutLMv3Layer.forward

        def _layer_forward(s, hs, am=None, hm=None, oa=False, rel_pos=None, rel_2d_pos=None, **k):
            return (_lf(s, hs, am, rel_pos=rel_pos, rel_2d_pos=rel_2d_pos),)

        _layer_forward._mmee_shim = True
        HF.LayoutLMv3Layer.forward = _layer_forward
    # (5) offline: the processor is never used on the forward path (ref :674)
    L.AutoProcessor.from_pretrained = staticmethod(lambda *a, **k: None)
    _loaded = L
    return L


def reference_config(dims, ee):
    """The HF LayoutLMv3Config with the `EE_config` dict the reference model is constructed from."""
    cfg = dims.to_hf_config()
    cfg.EE_config = {
        "training_strategy": "one_stage_subgraphs_weighted",
        "exits": list(ee.exits),
        "encoder_layer_strategy": ee.encoder_layer_strategy,
        "inference_strategy": ee.inference_strategy,
        "exit_head_num_layers": ee.exit_head_num_layers,
        "global_threshold": ee.global_threshold,
        "model_weights": "microsoft/layoutlmv3-base",
    }
    if getattr(ee, "use_lte", False):
        cfg.EE_config["use_lte"] = True
    return cfg


def build_reference_model(dims, ee, state_dict=None):
    """Construct the reference `LayoutLMv3EEForSequenceClassification` for (dims, ee) in eval mode.

    `ee.exits` must contain an embedding-level exit for encoder exits to be reported
    (reference quirk, EE/models/LayoutLMv3.py:402,648-649)."""
    import torch

    L = load()
    cfg = reference_config(dims, ee)
    torch.manual_seed(0)
    model = L.LayoutLMv3EEForSequenceClassification(cfg).eval()
    if state_dict is not None:
        missing, unexpected = model.load_state_dict(state_dict, strict=False)
        # non-persistent buffers never appear; anything else is a naming bug in mmee.synth
        assert not unexpected, unexpected
        assert not missing, missing
    return model


def reference_forward(model, docs):
    """One reference forward (EE/utils.py:179 call shape).  Returns dict of CPU tensors:
    exit_logits [E+1,B,K] (what get_logits stores: exit_states[j][0] for ramps, gated_logits[j]
    for gates, then final logits — EE/utils.py:182-193), head_logits (raw head outputs),
    criteria [E+1,B], last_hidden [B,S,H]."""
    import torch

    with torch.no_grad():
        out = model(**docs)
        inner = model.layoutlmv3(
            docs["input_ids"], attention_mask=docs["attention_mask"], bbox=docs["bbox"],
            pixel_values=docs["pixel_values"], return_dict=True)
    heads = [s[0] for s in out.exit_states]
    gate = model.apply_gating
    per_exit = list(out.gated_logits) if gate else heads
    return {
        "exit_logits": torch.stack(per_exit + [out.logits]).float(),
        "head_logits": torch.stack(heads).float(),
        "criteria": torch.stack(list(out.exit_criteria)).float(),
        "last_hidden": inner.last_hidden_state.float(),
    }


def reference_forward_image_only(model, pixel_values):
    """BASELINE config 5 (image-only, patch tokens only, ramps).  The reference EE model cannot run this through
    `forward` (UnboundLocalError, EE/models/LayoutLMv3.py:549-565; author's note EE/configs.py:52), so the verified
    recipe of SURVEY.md Appendix B drives its sub-modules directly with stock-HF image-only semantics (HF:730-768):
    forward_image -> model LayerNorm -> [concat exit on the mean] -> LayoutLMv3EncoderEE over the 197 visual tokens
    (visual boxes / positions) -> classifier on the visual CLS token."""
    import torch

    m = model.layoutlmv3
    B = pixel_values.shape[0]
    with torch.no_grad():
        x = m.dropout(m.LayerNorm(m.forward_image(pixel_values)))
        n_vis = x.shape[1]
        heads = []
        rows = []
        if hasattr(m, "concat_exit_embeddings"):
            z = x.mean(1)
            rows.append(z)
            heads.append(m.concat_exit_embeddings(z))
        ext = m.get_extended_attention_mask(torch.ones(B, n_vis), None, x.device, dtype=x.dtype)
        side = int(pixel_values.shape[2] / m.config.patch_size)
        enc = m.encoder(x, bbox=m.calculate_visual_bbox(x.device, dtype=torch.long, batch_size=B),
                        position_ids=torch.arange(n_vis)[None].repeat(B, 1), attention_mask=ext,
                        head_mask=[None] * m.config.num_hidden_layers, return_dict=True,
                        patch_height=side, patch_width=side)
        for st in enc.exit_states:
            heads.append(st[0] if isinstance(st, tuple) else st)
        rows += list(enc.gate_inputs) if model.apply_gating else []
        last = enc[0]
        final = model.classifier(last[:, 0, :])
        gate = model.apply_gating
        per_exit = [model.classifier(z) for z in rows] if gate else heads
        crit = [model.layoutlmv3.exit_criterion(h) for h in heads] + [model.layoutlmv3.exit_criterion(final)]
    return {
        "exit_logits": torch.stack(per_exit + [final]).float(),
        "head_logits": torch.stack(heads).float(),
        "criteria": torch.stack(crit).float(),
        "last_hidden": last.float(),
    }


def reference_forward_lte(model, docs):
    """The reference's learned-to-exit inference (EE_config["use_lte"], EE/models/LayoutLMv3.py:231-268, 728-748).
    Its exit test compares a squeezed tensor with a float, which is only defined for ONE document, so the model is
    run document by document; no labels are passed (they would only add losses).  Returns logits [B,K] (the
    `outputs.logits` of each call: the exit ramp's logits / classifier(CLS_j) in gate mode when the encoder raised
    EarlyExitException, else the final classifier) and exit_layer [B] (encoder layer of the exit taken, 0 = ran to
    the end), read from the exception the inner model raises."""
    import torch

    L = load()
    B = docs["pixel_values"].shape[0]
    logits, layers = [], []
    with torch.no_grad():
        for i in range(B):
            d1 = {k: v[i:i + 1] for k, v in docs.items() if k != "labels"}
            out = model(**d1)
            logits.append(out.logits.reshape(-1).float())
            try:
                model.layoutlmv3(d1["input_ids"], attention_mask=d1["attention_mask"], bbox=d1["bbox"],
                                 pixel_values=d1["pixel_values"], return_dict=True)
                layers.append(0)
            except L.EarlyExitException as ex:
                # identifier = "encoder_exit_<layer>_<head type>" (EE/models/LayoutLMv3.py:82, 115-118)
                layers.append(int(str(ex.exit_layer).split("_")[2]))
    return {"logits": torch.stack(logits), "exit_layer": torch.tensor(layers, dtype=torch.int64)}
