"""GPU tests (B200) of forward plans (`B200EEForSequenceClassification.plan`, `mmee_plan_*`): a forward captured into
a CUDA graph, with the launches after the last exit skipped by IF nodes in early-exit mode.  The plan runs the same
kernels in the same order as the eager forward, so every result must be bit-identical to `infer` on the same inputs.
"""
import numpy as np
import pytest
import torch

from helpers import load_case
from mmee import synth
from mmee.calibration import spread_temperatures, thresholds_for
from mmee.config import ExitConfig, ModelDims

pytestmark = pytest.mark.gpu

_models = {}


def _engine(name, dtype="bf16", max_batch=8):
    from mmee.model import B200EEForSequenceClassification

    key = (name, dtype)
    if key not in _models:
        g, dims, ee, sd, docs = load_case(name)
        mb = max(max_batch, docs["pixel_values"].shape[0])
        _models[key] = (B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=mb, dtype=dtype), dims, docs)
    return _models[key]


def _cuda(docs):
    return {k: v.cuda() for k, v in docs.items()}


def _policy(model, dims, dev, criterion, conf=0.7):
    """(threshold, temperatures) at which some documents leave early and some do not."""
    if criterion == "lte":
        return 0.5, None
    dense = model.infer(**dev, exit_threshold=2.0 if criterion == "max_confidence" else -1.0, criterion=criterion,
                        early_exit=False, return_all=True)
    temps = spread_temperatures(dense.all_exit_logits.cpu().numpy(), criterion)
    return thresholds_for(criterion, conf, dims.n_labels), temps


def _assert_same(got, want, all_outputs=True):
    assert np.array_equal(got.exits_store, want.exits_store)
    assert torch.equal(got.logits.cpu(), want.logits.cpu())
    assert np.array_equal(got.criteria, want.criteria, equal_nan=True)
    assert np.array_equal(got.exit_hist, want.exit_hist)
    assert torch.equal(got.predictions, want.predictions)
    if all_outputs:
        for f in ("all_exit_logits", "all_criteria"):
            a, b = getattr(got, f).cpu().numpy(), getattr(want, f).cpu().numpy()
            assert np.array_equal(a, b, equal_nan=True), f


PARITY_CASES = ["tiny_ramp_conf", "tiny_gate_ent", "tiny_ramp_1layer_head", "tiny_modality_ramp", "tiny_modality_gate",
                "tiny_image_only", "base_gate_ent", "config0_base_ramp16"]


@pytest.mark.parametrize("early_exit", [True, False])
@pytest.mark.parametrize("criterion", ["max_confidence", "entropy"])
@pytest.mark.parametrize("name", PARITY_CASES)
def test_plan_equals_eager(name, criterion, early_exit):
    model, dims, docs = _engine(name)
    dev = _cuda(docs)
    thr, temps = _policy(model, dims, dev, criterion)
    plan = model.plan(docs["pixel_values"].shape[0], criterion=criterion, early_exit=early_exit, return_all=True)
    got = plan.infer(**dev, exit_threshold=thr, temperatures=temps)
    want = model.infer(**dev, exit_threshold=thr, temperatures=temps, criterion=criterion, early_exit=early_exit,
                       return_all=True)
    _assert_same(got, want)
    if early_exit:
        print(f"{name} [{criterion}]: exit histogram {want.exit_hist.tolist()}")
    plan.close()


@pytest.mark.parametrize("early_exit", [True, False])
@pytest.mark.parametrize("name", ["tiny_lte_ramp", "tiny_lte_gate"])
def test_plan_equals_eager_lte(name, early_exit):
    model, dims, docs = _engine(name)
    dev = _cuda(docs)
    plan = model.plan(docs["pixel_values"].shape[0], criterion="lte", early_exit=early_exit, return_all=True)
    for thr in (0.3, 0.5, 0.7):
        got = plan.infer(**dev, exit_threshold=thr)
        want = model.infer(**dev, exit_threshold=thr, criterion="lte", early_exit=early_exit, return_all=True)
        _assert_same(got, want)
    plan.close()


@pytest.mark.parametrize("name", ["tiny_ramp_conf", "base_gate_ent"])
def test_plan_equals_eager_fp32(name):
    model, dims, docs = _engine(name, dtype="fp32")
    dev = _cuda(docs)
    criterion = model._default_criterion()
    thr, temps = _policy(model, dims, dev, criterion)
    for early_exit in (True, False):
        plan = model.plan(docs["pixel_values"].shape[0], criterion=criterion, early_exit=early_exit, return_all=True)
        got = plan.infer(**dev, exit_threshold=thr, temperatures=temps)
        want = model.infer(**dev, exit_threshold=thr, temperatures=temps, criterion=criterion, early_exit=early_exit,
                           return_all=True)
        _assert_same(got, want)
        plan.close()


def test_one_plan_many_policies():
    """Thresholds and temperatures are inputs of every run, not part of the captured graph."""
    model, dims, docs = _engine("tiny_gate_ent")
    dev = _cuda(docs)
    _, temps = _policy(model, dims, dev, "max_confidence")
    plan = model.plan(docs["pixel_values"].shape[0], criterion="max_confidence", return_all=True)
    hists = set()
    for tv in (temps, np.ones_like(temps)):
        for thr in (0.1, 0.5, 0.7, 0.9):
            got = plan.infer(**dev, exit_threshold=thr, temperatures=tv)
            want = model.infer(**dev, exit_threshold=thr, temperatures=tv, criterion="max_confidence", return_all=True)
            _assert_same(got, want)
            hists.add(tuple(want.exit_hist.tolist()))
    assert len(hists) > 1          # the policies do lead to different exits


def test_plan_skips_the_tail():
    """Once every document has left, the exit kernels of the deeper stages do not run in a plan (their stage count
    keeps the -1 the run starts from), while the eager forward launches them and they publish 0 survivors."""
    model, dims, docs = _engine("tiny_ramp_conf")
    dev = _cuda(docs)
    n = docs["pixel_values"].shape[0]
    E = model.n_exits
    plan = model.plan(n, criterion="max_confidence", return_all=True)
    # max-softmax > 0 always: every document leaves at exit 0
    got = plan.infer(**dev, exit_threshold=0.0)
    nd_plan = model.debug_read("NDEV", np.int32, E + 3)
    want = model.infer(**dev, exit_threshold=0.0, criterion="max_confidence", return_all=True)
    nd_eager = model.debug_read("NDEV", np.int32, E + 3)
    _assert_same(got, want)
    assert (got.exits_store == 0).all()
    assert nd_plan[0] == n and nd_plan[1] == 0 and (nd_plan[2:] == -1).all(), nd_plan
    assert nd_eager[0] == n and (nd_eager[1:E + 2] == 0).all(), nd_eager
    # strict > 1.0 never holds: nobody leaves before the final classifier, every stage runs
    got = plan.infer(**dev, exit_threshold=1.0)
    nd_plan = model.debug_read("NDEV", np.int32, E + 3)
    want = model.infer(**dev, exit_threshold=1.0, criterion="max_confidence", return_all=True)
    _assert_same(got, want)
    assert (got.exits_store == E).all()
    assert (nd_plan[:E + 1] == n).all() and nd_plan[E + 1] == 0, nd_plan
    plan.close()


def test_new_inputs_every_run():
    """Two plans (B = 1 and B = 4, below max_batch) on one engine, alternated, host and device inputs: each run equals
    the eager forward on the same documents."""
    model, dims, docs = _engine("tiny_ramp_conf")
    pool = synth.make_docs(dims, 8, seed=77, pad=True)
    dev_pool = _cuda(pool)
    p1 = model.plan(1, criterion="max_confidence", return_all=True)
    p4 = model.plan(4, criterion="max_confidence", return_all=True)
    thr, temps = _policy(model, dims, dev_pool, "max_confidence", conf=0.6)
    for i in range(6):
        for plan, b in ((p1, 1), (p4, 4)):
            lo = (i * b) % 8
            src = dev_pool if i % 2 == 0 else pool
            batch = {k: v[lo:lo + b].contiguous() for k, v in src.items()}
            got = plan.infer(**batch, exit_threshold=thr, temperatures=temps)
            want = model.infer(**batch, exit_threshold=thr, temperatures=temps, return_all=True)
            assert got.logits.is_cuda == (i % 2 == 0)
            _assert_same(got, want)
    p1.close()
    p4.close()


def test_plan_runs_are_ordered_with_eager_forwards():
    """Plan runs and eager forwards on different streams share one set of scratch buffers and stay ordered."""
    model, dims, docs = _engine("base_gate_ent")
    dev = _cuda(docs)
    n = docs["pixel_values"].shape[0]
    thr, temps = _policy(model, dims, dev, "max_confidence", conf=0.5)
    kw = dict(exit_threshold=thr, temperatures=temps)
    flipped = {k: v.flip(0).contiguous() for k, v in dev.items()}
    ref = model.infer(**dev, criterion="max_confidence", **kw)
    ref_flip = model.infer(**flipped, criterion="max_confidence", **kw)
    plan = model.plan(n, criterion="max_confidence")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    for _ in range(3):
        with torch.cuda.stream(s1):
            r1 = plan.infer_device(**dev, **kw)
        with torch.cuda.stream(s2):                                     # no explicit dependency on s1
            r2 = model.infer_device(**flipped, criterion="max_confidence", **kw)
        with torch.cuda.stream(s1):
            r3 = plan.infer_device(**flipped, **kw)
        r4 = plan.infer(**docs, **kw)                                   # host path
        torch.cuda.synchronize()
        assert torch.equal(r1["logits"], ref.logits) and torch.equal(r2["logits"], ref_flip.logits)
        assert torch.equal(r3["logits"], ref_flip.logits)
        assert torch.equal(r1["exit_index"].cpu(), torch.from_numpy(ref.exits_store))
        assert torch.equal(r4.logits, ref.logits.cpu())
    model.sync()
    plan.close()


def test_plan_errors_leave_the_engine_usable():
    model, dims, docs = _engine("tiny_ramp_conf")
    dev = _cuda(docs)
    n = docs["pixel_values"].shape[0]
    plan = model.plan(n, criterion="max_confidence")
    with pytest.raises(ValueError, match="captured for"):
        plan.infer(**{k: v[:n - 1] for k, v in dev.items()}, exit_threshold=0.5)
    with pytest.raises(RuntimeError, match="criterion / mode"):
        plan.infer(**dev, exit_threshold=0.5, criterion="entropy")
    with pytest.raises(RuntimeError, match="criterion / mode"):
        plan.infer(**dev, exit_threshold=0.5, early_exit=False)
    with pytest.raises(RuntimeError, match="batch out of range"):
        model.plan(model.max_batch + 1)
    with pytest.raises(RuntimeError, match="LTE"):
        model.plan(n, criterion="lte")
    bad = {k: v.clone() for k, v in docs.items()}
    bad["input_ids"][0, 5] = dims.vocab + 10
    with pytest.raises(RuntimeError, match="input out of range"):
        plan.infer(**bad, exit_threshold=0.5)
    # the engine and the plan still work, and still agree
    got = plan.infer(**dev, exit_threshold=0.5)
    want = model.infer(**dev, exit_threshold=0.5, criterion="max_confidence")
    _assert_same(got, want, all_outputs=False)
    plan.close()
    with pytest.raises(RuntimeError, match="closed"):
        plan.infer(**dev, exit_threshold=0.5)


def test_plan_equals_eager_at_bench_size():
    """The headline configuration (base, gates after every layer, entropy, calibrated temperatures, the entropy
    equivalent of 0.7 confidence) at 256 documents."""
    from mmee.model import B200EEForSequenceClassification

    dims = ModelDims.base()
    ee = ExitConfig.from_dict(dict(exits=["text_visual_concat"] + list(range(1, dims.layers + 1)),
                                   encoder_layer_strategy="gate", inference_strategy="entropy"))
    sd = synth.make_state_dict(dims, ee, seed=0)
    model = B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=256)
    cal = _cuda(synth.make_docs(dims, 64, seed=12345, pad=False))
    thr, temps = _policy(model, dims, cal, "entropy")
    docs = _cuda(synth.make_docs(dims, 256, seed=1, pad=False))
    plan = model.plan(256, return_all=True)
    got = plan.infer(**docs, exit_threshold=thr, temperatures=temps)
    want = model.infer(**docs, exit_threshold=thr, temperatures=temps, return_all=True)
    _assert_same(got, want)
    print(f"headline B=256: exit histogram {want.exit_hist.tolist()}")
    plan.close()
    model.close()
