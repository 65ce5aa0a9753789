"""GPU parity tests (B200): the CUDA engine, called through the C ABI, against the golden vectors
(outputs of the unmodified reference) and the oracle port / policy port on the same seeded inputs.

Tolerances (north_star): logits within 1e-2 absolute in the bf16 engine mode and 1e-4 in the fp32 mode; predicted
classes identical wherever the reference's top-2 logit gap exceeds 2x that tolerance; exit indices bit-exact for
every document that is decisive in the sense of `helpers.exit_agreement` (the criterion margin to the threshold
exceeds 1.5x the engine's own criterion error at every exit), with the agreement over ALL documents and the decisive
fraction printed and — in the fp32 mode, where the error is small enough for the notion to be non-vacuous at the
calibration temperatures of random-init heads — floored.
"""
import numpy as np
import pytest
import torch

from helpers import ALL_CASES, exit_agreement, load_case, port_forward_chunked
from mmee import synth
from mmee.calibration import spread_temperatures, thresholds_for
from mmee.config import ExitConfig, ModelDims

pytestmark = pytest.mark.gpu

LOGIT_TOL = 1e-2          # bf16 engine mode, absolute (north_star)
LOGIT_TOL_FP32 = 1e-4     # fp32 engine mode, absolute (north_star)
TOL = {"bf16": LOGIT_TOL, "fp32": LOGIT_TOL_FP32}

_models = {}


def _engine(name, max_batch=8, dtype="bf16"):
    from mmee.model import B200EEForSequenceClassification

    key = (name, dtype)
    if key not in _models:
        g, dims, ee, sd, docs = load_case(name)
        mb = max(max_batch, docs["pixel_values"].shape[0])
        _models[key] = (B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=mb, dtype=dtype), g, dims, ee, sd, docs)
    return _models[key]


def _cuda(docs):
    return {k: v.cuda() for k, v in docs.items()}


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
@pytest.mark.parametrize("name", ALL_CASES)
def test_dense_logits_match_reference_golden(name, dtype):
    model, g, dims, ee, sd, docs = _engine(name, dtype=dtype)
    tol = TOL[dtype]
    out = model.forward(**_cuda(docs))
    got = out.exit_logits.cpu().numpy()
    ref = g["exit_logits"]
    assert got.shape == ref.shape
    err = np.abs(got - ref).max()
    print(f"{name} [{dtype}]: max|logits - reference| = {err:.3e} (tolerance {tol:g})")
    assert err <= tol
    # predicted classes identical wherever the reference's decision is not a numerical tie
    srt = np.sort(ref, axis=-1)
    decisive = (srt[..., -1] - srt[..., -2]) > 2 * tol
    assert (got.argmax(-1) == ref.argmax(-1))[decisive].all()
    # raw head outputs (exit_states[j][0]) and the reference-shaped output object
    n_head = g["head_logits"].shape[-1]
    heads = torch.stack([s[0] for s in out.exit_states]).cpu().numpy()
    assert heads.shape == g["head_logits"].shape
    assert np.abs(heads - g["head_logits"]).max() <= tol
    assert len(out.exit_criteria) == ref.shape[0]
    assert np.abs(torch.stack(out.exit_criteria).cpu().numpy() - g["criteria"]).max() <= 2 * tol
    assert np.abs(out.logits.cpu().numpy() - ref[-1]).max() <= tol
    if ee.encoder_layer_strategy == "gate":
        assert n_head == 2 and len(out.gated_logits) == ref.shape[0] - 1
        assert np.abs(torch.stack(out.gated_logits).cpu().numpy() - ref[:-1]).max() <= tol


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
@pytest.mark.parametrize("name", ALL_CASES)
def test_early_exit_matches_reference_policy(name, dtype):
    """Exit indices of the real early-exit forward vs the reference Policy results stored in the golden (calibrated
    logits, four thresholds).  Bit-exact on the decisive documents; agreement over ALL documents and the decisive
    fraction are printed, and floored in the fp32 mode."""
    model, g, dims, ee, sd, docs = _engine(name, dtype=dtype)
    tol = TOL[dtype]
    temps = g["temps"]
    dense = model.infer(**_cuda(docs), exit_threshold=2.0, criterion="max_confidence", early_exit=False, return_all=True)
    eng_logits = dense.all_exit_logits.cpu().numpy()
    total = agree = n_dec = 0
    for thr in (0.1, 0.5, 0.7, 0.9):
        res = model.infer(**_cuda(docs), exit_threshold=thr, temperatures=temps, criterion="max_confidence")
        st = exit_agreement(res.exits_store, eng_logits, g["exit_logits"], temps, thr, "max_confidence")
        want = g[f"policy_cal_{thr}_exits"]
        assert np.array_equal(st["want"], want)                     # the policy port reproduces the reference's Policy
        dm = st["decisive_mask"]
        assert (res.exits_store[dm] == want[dm]).all(), (thr, res.exits_store, want)
        total += want.size
        agree += int(st["agree"].sum())
        n_dec += int(dm.sum())
        # returned logits are those of the exit taken
        same = st["agree"]
        if same.any():
            assert np.abs(res.predictions.numpy()[same] - g[f"policy_cal_{thr}_pred"][same] * temps[want[same]][:, None]
                          ).max() <= tol
        assert res.exit_hist.sum() == want.size
        assert abs(sum(res.exit_distribution.values()) - 1.0) < 1e-9
    print(f"{name} [{dtype}]: exit-layer agreement with the reference policy: all documents {agree}/{total}, "
          f"decisive {n_dec}/{total} (all agree)")
    if dtype == "fp32":
        assert n_dec >= 0.9 * total and agree >= 0.9 * total


@pytest.mark.parametrize("name", ["tiny_ramp_conf", "tiny_gate_ent", "base_gate_ent", "tiny_modality_ramp",
                                  "tiny_modality_gate"])
@pytest.mark.parametrize("criterion", ["max_confidence", "entropy"])
def test_early_exit_equals_dense_posthoc(name, criterion):
    """Real compaction == post-hoc policy on the engine's own dense logits, bit-exact (per-document
    arithmetic does not depend on which slot a document occupies)."""
    from oracle import policy_port

    model, g, dims, ee, sd, docs = _engine(name)
    dense = model.infer(**_cuda(docs), exit_threshold=2.0 if criterion == "max_confidence" else -1.0,
                        criterion=criterion, early_exit=False, return_all=True)
    all_logits = dense.all_exit_logits.cpu().numpy()
    temps = spread_temperatures(all_logits, criterion)
    for conf_thr in (0.3, 0.6, 0.8, 0.95):
        thr = thresholds_for(criterion, conf_thr, dims.n_labels)
        ee_res = model.infer(**_cuda(docs), exit_threshold=thr, temperatures=temps, criterion=criterion,
                             return_all=True)
        dn_res = model.infer(**_cuda(docs), exit_threshold=thr, temperatures=temps, criterion=criterion,
                             early_exit=False, return_all=True)
        assert np.array_equal(ee_res.exits_store, dn_res.exits_store)
        assert torch.equal(ee_res.logits, dn_res.logits)
        assert np.array_equal(ee_res.criteria, dn_res.criteria)
        assert np.array_equal(ee_res.exit_hist, dn_res.exit_hist)
        # exits a document reached carry identical logits; the ones it skipped are NaN
        a, b = ee_res.all_exit_logits.cpu().numpy(), dn_res.all_exit_logits.cpu().numpy()
        reached = np.arange(a.shape[0])[:, None] <= ee_res.exits_store[None, :]
        assert np.array_equal(a[reached], b[reached])
        assert np.isnan(a[~reached]).all()
        # and both agree with the fp64 policy oracle applied to the engine's dense logits (outside the margin)
        cal = policy_port.temperature_scale(all_logits, temps)
        want, _, crit = policy_port.exit_policy_vectorised(cal, thr, criterion)
        margin = np.abs(crit[:-1] - thr).min(axis=0)
        decisive = margin > 1e-4
        assert (ee_res.exits_store[decisive] == want[decisive]).all() and decisive.mean() >= 0.5


def test_host_path_equals_device_path():
    model, g, dims, ee, sd, docs = _engine("tiny_ramp_conf")
    temps = g["temps"]
    a = model.infer(**_cuda(docs), exit_threshold=0.5, temperatures=temps, return_all=True)
    b = model.infer(**docs, exit_threshold=0.5, temperatures=temps, return_all=True)     # CPU tensors -> mmee_forward
    assert not b.logits.is_cuda
    assert np.array_equal(a.exits_store, b.exits_store)
    assert torch.equal(a.logits.cpu(), b.logits)
    assert np.array_equal(a.exit_hist, b.exit_hist)
    o1 = model.forward(**_cuda(docs))
    o2 = model.forward(**docs)
    assert torch.equal(o1.exit_logits.cpu(), o2.exit_logits)


def test_batch_composition_invariance():
    """A document's result does not depend on its neighbours or its position in the batch."""
    model, g, dims, ee, sd, docs = _engine("tiny_ramp_conf")
    full = model.forward(**_cuda(docs)).exit_logits.cpu()
    perm = torch.tensor([3, 0, 5, 1])
    sub = {k: v[perm].cuda() for k, v in docs.items()}
    part = model.forward(**sub).exit_logits.cpu()
    assert torch.equal(part, full[:, perm])
    one = {k: v[2:3].cuda() for k, v in docs.items()}
    assert torch.equal(model.forward(**one).exit_logits.cpu(), full[:, 2:3])


def test_edge_cases_thresholds():
    model, g, dims, ee, sd, docs = _engine("tiny_ramp_conf")
    n = docs["input_ids"].shape[0]
    E1 = g["exit_logits"].shape[0]
    # threshold that can never be exceeded (strict >): everything leaves at the final classifier
    r = model.infer(**_cuda(docs), exit_threshold=1.0)
    assert (r.exits_store == E1 - 1).all() and r.exit_hist[-1] == n
    # threshold 0: max-softmax > 0 always -> everything leaves at exit 0 (no encoder layer runs)
    r = model.infer(**_cuda(docs), exit_threshold=0.0)
    assert (r.exits_store == 0).all() and r.exit_hist[0] == n
    assert np.abs(r.predictions.numpy() - g["exit_logits"][0]).max() <= LOGIT_TOL
    # per-exit thresholds: only exit 2 can fire
    thr = [1.0] * (E1 - 1)
    thr[2] = 0.0
    r = model.infer(**_cuda(docs), exit_threshold=thr)
    assert (r.exits_store == 2).all()
    # batch of one document, fully padded text except <s> </s>
    d1 = synth.make_docs(dims, 1, seed=9)
    d1["input_ids"][0, 2:] = dims.pad_id
    d1["input_ids"][0, 1] = 2
    d1["attention_mask"][0, 2:] = 0
    d1["bbox"][0] = 0
    from oracle import port

    want = port.forward(sd, dims, ee, d1)["exit_logits"].numpy()
    got = model.forward(**_cuda(d1)).exit_logits.cpu().numpy()
    assert np.abs(got - want).max() <= LOGIT_TOL


def test_bucket_lut_c_default_equals_torch():
    """The C default |rel|->bucket table equals the table computed with the reference's torch ops."""
    from mmee.model import B200EEForSequenceClassification, bucket_lut
    from mmee import _lib
    import ctypes as C

    model, g, dims, *_ = _engine("tiny_ramp_conf")
    assert np.array_equal(model.bucket_lut_in_use(0), bucket_lut(dims.rel_bins, dims.max_rel))
    assert np.array_equal(model.bucket_lut_in_use(1), bucket_lut(dims.rel2d_bins, dims.max_rel2d))


def test_full_size_batch_properties():
    """BASELINE config-2 shape (base, B=256 per GPU is covered by bench; here B=32 full-length documents):
    size-independent properties — early-exit == dense, histogram sums to B, duplicated documents give
    bit-identical rows, exit depth is monotone in the threshold."""
    dims = ModelDims.base()
    ee = ExitConfig.from_dict(dict(exits=["text_visual_concat"] + list(range(1, 13)), encoder_layer_strategy="ramp",
                                   inference_strategy="max_confidence"))
    from mmee.model import B200EEForSequenceClassification

    sd = synth.make_state_dict(dims, ee, seed=0)
    model = B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=32)
    docs = synth.make_docs(dims, 16, seed=21, pad=False)
    docs = {k: torch.cat([v, v]) for k, v in docs.items()}          # every document twice
    dev = _cuda(docs)
    dense = model.infer(**dev, exit_threshold=2.0, early_exit=False, return_all=True)
    al = dense.all_exit_logits.cpu().numpy()
    assert np.array_equal(al[:, :16], al[:, 16:])
    assert np.isfinite(al).all()
    temps = spread_temperatures(al, "max_confidence")
    prev_mean = -1.0
    for thr in (0.5, 0.7, 0.9, 0.99):
        a = model.infer(**dev, exit_threshold=thr, temperatures=temps)
        b = model.infer(**dev, exit_threshold=thr, temperatures=temps, early_exit=False)
        assert np.array_equal(a.exits_store, b.exits_store) and torch.equal(a.logits, b.logits)
        assert a.exit_hist.sum() == 32
        assert np.array_equal(a.exits_store[:16], a.exits_store[16:])
        assert a.exits_store.mean() >= prev_mean
        prev_mean = a.exits_store.mean()
    model.close()


def test_get_logits_store_matches_reference_layout(tmp_path):
    """SURVEY.md §8f row 1: the batched logits-store loop writes what EE/utils.py:125-271 writes (names, keys, dtypes,
    which logits per exit) and the post-hoc Policy on that store equals the engine's on-device early exit."""
    import json
    import os

    from mmee.pipeline import get_logits
    from mmee.policy import Policy

    for name in ("tiny_ramp_conf", "tiny_gate_ent"):
        model, g, dims, ee, sd, docs = _engine(name)
        n = docs["input_ids"].shape[0]
        docs = dict(docs)
        docs["labels"] = torch.arange(n) % dims.n_labels
        loader = [{k: v[i:i + 4] for k, v in docs.items()} for i in range(0, n, 4)]       # batches of 4 (last: 2)
        cfg = {"checkpoint": f"org/{name}", "test_dataset": "synthetic/rvl", "downsampling": 0, "labelset": "test",
               "results_root": str(tmp_path), "exit_threshold": 0.5, "device": "cpu"}
        logits, refs, _ = get_logits(model, cfg, loader)
        assert logits.dtype == np.float64 and logits.shape == g["exit_logits"].shape
        assert np.abs(logits - g["exit_logits"]).max() <= LOGIT_TOL                   # the reference's stored logits
        assert np.array_equal(refs, docs["labels"].numpy())
        out = os.path.join(str(tmp_path), "results", f"{name}-rvl")
        assert sorted(os.listdir(out)) == ["config.json", "exit_logits-test.npz", "references-test.npz"]
        assert np.array_equal(np.load(os.path.join(out, "exit_logits-test.npz"))["arr_0"], logits)
        saved = json.load(open(os.path.join(out, "config.json")))
        assert "exit_threshold" not in saved and saved["checkpoint"] == f"org/{name}"
        again, refs2, _ = get_logits(model, cfg, loader)                              # cache short-cut
        assert np.array_equal(again, logits) and np.array_equal(refs2, refs)
        # post-hoc policy on the store == real early exit on the device (raw logits, max-confidence)
        ex, pred, _ = Policy(logits=logits, config=cfg).max_confidence_global_thresholding_policy()
        res = model.infer(**_cuda({k: v for k, v in docs.items()}), exit_threshold=0.5, criterion="max_confidence")
        crit = policy_port_criterion(logits)
        decisive = np.abs(crit[:-1] - 0.5).min(axis=0) > 1e-4
        assert np.array_equal(res.exits_store[decisive], ex[decisive])


def policy_port_criterion(logits):
    from oracle import policy_port

    return policy_port.criterion(logits, "max_confidence")


@pytest.mark.parametrize("pad,dtype", [(True, "bf16"), (False, "bf16"), (True, "fp32")])
def test_batch256_parity_and_exit_agreement_vs_port(pad, dtype):
    """The benchmarked shape: 256 base documents (16 exit groups, two CTA waves of attention, compaction across warps),
    gates + entropy policy (BASELINE configs[1]), 2 encoder layers + the concat exit so that the oracle port finishes
    in seconds per chunk.  Dense logits vs the port (itself pinned to the reference goldens, max|d| = 0); real early
    exit == the post-hoc policy on the engine's dense logits, bit for bit; agreement with the REFERENCE policy
    (port logits + policy port) over all 256 documents, bit-exact on the decisive ones."""
    from mmee.model import B200EEForSequenceClassification
    from oracle import policy_port

    dims = ModelDims.base(layers=2)
    ee = ExitConfig.from_dict(dict(exits=["text_visual_concat", 1, 2], encoder_layer_strategy="gate",
                                   inference_strategy="entropy"))
    sd = synth.make_state_dict(dims, ee, seed=3)
    docs = synth.make_docs(dims, 256, seed=31, pad=pad)
    model = B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=256, dtype=dtype)
    dev = _cuda(docs)
    dense = model.infer(**dev, exit_threshold=-1.0, early_exit=False, return_all=True)
    got = dense.all_exit_logits.cpu().numpy()
    want = port_forward_chunked(sd, dims, ee, docs).numpy()
    err = np.abs(got - want)
    print(f"256 base docs (pad={pad}) [{dtype}]: max|logits - port| = {err.max():.3e}, mean = {err.mean():.3e}")
    assert err.max() <= TOL[dtype]
    srt = np.sort(want, axis=-1)
    dec = (srt[..., -1] - srt[..., -2]) > 2 * TOL[dtype]
    assert (got.argmax(-1) == want.argmax(-1))[dec].all()
    temps = spread_temperatures(want, "entropy")
    fracs = []
    for conf_thr in (0.5, 0.7, 0.9):
        thr = thresholds_for("entropy", conf_thr, dims.n_labels)
        early = model.infer(**dev, exit_threshold=thr, temperatures=temps, return_all=True)
        posthoc = model.infer(**dev, exit_threshold=thr, temperatures=temps, early_exit=False)
        assert np.array_equal(early.exits_store, posthoc.exits_store) and torch.equal(early.logits, posthoc.logits)
        assert early.exit_hist.sum() == 256
        mine, _, _ = policy_port.exit_policy_vectorised(policy_port.temperature_scale(got, temps), thr, "entropy")
        st = exit_agreement(early.exits_store, got, want, temps, thr, "entropy")
        dm = st["decisive_mask"]
        assert (early.exits_store[dm] == st["want"][dm]).all()
        # against the engine's OWN dense logits the only slack is fp32-vs-fp64 criterion arithmetic
        own_crit = policy_port.criterion(policy_port.temperature_scale(got, temps), "entropy")
        own_dec = np.abs(own_crit[:-1] - thr).min(axis=0) > 1e-4
        assert (early.exits_store == mine)[own_dec].all() and own_dec.mean() > 0.99
        fracs.append((conf_thr, st["all"], st["decisive_frac"], early.exit_hist.tolist()))
        print(f"  threshold@{conf_thr}: agreement with the reference policy {st['all']:.3f} over all 256 documents, "
              f"decisive fraction {st['decisive_frac']:.3f}, exits {early.exit_hist.tolist()}")
    if dtype == "fp32":
        assert min(f[1] for f in fracs) >= 0.98 and min(f[2] for f in fracs) >= 0.95
    else:
        assert min(f[1] for f in fracs) >= 0.80                     # bf16: 3e-3 logit error / T ~ 0.01 (see helpers.exit_agreement)
    model.close()


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_many_ragged_documents_multi_chunk_compaction(dtype):
    """600 documents (the compaction / row-plan block walks the slots in three chunks of 256) with text lengths from 2
    to 512, all three embedding-level exits and encoder exits: real early exit == post-hoc policy on the dense run, bit
    for bit, at thresholds that spread the documents over every exit; dense logits vs the oracle port; the row plan
    keeps every document's rows together (a wrong prefix sum shows up as garbage logits)."""
    from mmee.model import B200EEForSequenceClassification

    dims = ModelDims.tiny(layers=3)
    ee = ExitConfig.from_dict(dict(exits=["vision_avg", "text_avg", "text_visual_concat", 1, 2, 3],
                                   encoder_layer_strategy="ramp", inference_strategy="max_confidence"))
    sd = synth.make_state_dict(dims, ee, seed=13, std=0.05)
    n = 600
    docs = synth.make_docs(dims, n, seed=61, pad=True)
    g = torch.Generator().manual_seed(3)
    short = torch.randint(2, 40, (n,), generator=g)
    for d in range(0, n, 7):                                      # every 7th document is very short
        L = int(short[d])
        docs["input_ids"][d, L:] = dims.pad_id
        docs["input_ids"][d, L - 1] = 2
        docs["attention_mask"][d, L:] = 0
        docs["bbox"][d, L - 1:] = 0
    model = B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=n, dtype=dtype)
    dev = _cuda(docs)
    dense = model.infer(**dev, exit_threshold=2.0, early_exit=False, return_all=True)
    al = dense.all_exit_logits.cpu().numpy()
    assert np.isfinite(al).all()
    want = port_forward_chunked(sd, dims, ee, docs, chunk=64).numpy()
    err = np.abs(al - want).max()
    print(f"600 ragged tiny documents [{dtype}]: max|logits - port| = {err:.3e}")
    assert err <= TOL[dtype]
    temps = spread_temperatures(al, "max_confidence")
    seen = np.zeros(al.shape[0], dtype=np.int64)
    for thr in (0.46, 0.55, 0.7, 0.85, 0.97):
        a = model.infer(**dev, exit_threshold=thr, temperatures=temps, return_all=True)
        b = model.infer(**dev, exit_threshold=thr, temperatures=temps, early_exit=False)
        assert np.array_equal(a.exits_store, b.exits_store) and torch.equal(a.logits, b.logits)
        assert np.array_equal(a.exit_hist, b.exit_hist) and a.exit_hist.sum() == n
        x, y = a.all_exit_logits.cpu().numpy(), al
        reached = np.arange(x.shape[0])[:, None] <= a.exits_store[None, :]
        assert np.array_equal(x[reached], y[reached]) and np.isnan(x[~reached]).all()
        seen += a.exit_hist
    print("  documents per exit over the five thresholds:", seen.tolist())
    assert (seen > 0).sum() >= 5                                   # the thresholds really spread the exits
    model.close()


def test_out_of_range_inputs_raise_like_the_reference():
    """ADVICE r1: the reference raises IndexError for an input_id >= vocab or a bbox coordinate outside [0, max_2d);
    the engine must not read out of bounds: it clamps on the device and the synchronous call reports an error."""
    model, g, dims, ee, sd, docs = _engine("tiny_ramp_conf")
    good = model.forward(**_cuda(docs)).exit_logits.cpu()
    for field, value in (("input_ids", dims.vocab), ("input_ids", -1), ("bbox", dims.max_2d), ("bbox", -5)):
        bad = {k: v.clone() for k, v in docs.items()}
        if field == "input_ids":
            bad["input_ids"][1, 7] = value
        else:
            bad["bbox"][2, 9, 2] = value
        with pytest.raises(RuntimeError, match="out of range"):
            model.forward(**_cuda(bad))
        with pytest.raises(RuntimeError, match="out of range"):
            model.infer(**bad, exit_threshold=0.5)                      # host path
    # the engine is still usable and the flag does not stick
    assert torch.equal(model.forward(**_cuda(docs)).exit_logits.cpu(), good)


def test_forwards_on_different_streams_are_ordered():
    """ADVICE r1: one set of scratch buffers per engine — a forward on another stream (or the host path, which uses the
    engine's own stream) must not start before the previous forward has finished with them."""
    model, g, dims, ee, sd, docs = _engine("base_gate_ent")
    temps = g["temps"]
    dev = _cuda(docs)
    ref = model.infer(**dev, exit_threshold=0.5, temperatures=temps, criterion="max_confidence")
    ref_flip = model.infer(**{k: v.flip(0) for k, v in dev.items()}, exit_threshold=0.5, temperatures=temps,
                           criterion="max_confidence")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    flipped = {k: v.flip(0).contiguous() for k, v in dev.items()}
    torch.cuda.synchronize()
    for _ in range(3):
        with torch.cuda.stream(s1):
            r1 = model.infer_device(**dev, exit_threshold=0.5, temperatures=temps, criterion="max_confidence")
        with torch.cuda.stream(s2):                                     # no explicit dependency on s1
            r2 = model.infer_device(**flipped, exit_threshold=0.5, temperatures=temps, criterion="max_confidence")
        r3 = model.infer(**docs, exit_threshold=0.5, temperatures=temps, criterion="max_confidence")   # host path
        torch.cuda.synchronize()
        assert torch.equal(r1["logits"], ref.logits) and torch.equal(r2["logits"], ref_flip.logits)
        assert torch.equal(r3.logits, ref.logits.cpu())


# hidden size -> (coord, shape): 4 coord + 2 shape = hidden, both multiples of 4 so the vectorised text embedding runs
HIDDEN_SPATIAL = {256: (40, 48), 384: (64, 64), 512: (88, 80), 640: (108, 104), 896: (152, 144)}


@pytest.mark.parametrize("n_text,layers,hidden,dtype", [
    pytest.param(77, 2, None, "bf16", id="77-2"), pytest.param(200, 1, None, "bf16", id="200-1"),
    pytest.param(448, 1, None, "bf16", id="448-1")] + [
    pytest.param(77, 1, h, dt, id=f"h{h}-{dt}") for h in sorted(HIDDEN_SPATIAL) for dt in ("bf16", "fp32")])
def test_odd_sequence_lengths_vs_port(n_text, layers, hidden, dtype):
    """Sequence lengths that are not 709: partial key / query tiles, other pitches.  Engine vs the oracle port.
    `hidden`: every hidden size mmee_create accepts that the tiny / base / large models do not use (hidden / 128 = 2..7,
    heads = hidden / 64), with the embedding-level exits, in both engine modes."""
    from mmee.model import B200EEForSequenceClassification
    from oracle import port

    if hidden is None:
        dims = ModelDims.tiny(n_text=n_text, layers=layers)
        exits = ["text_visual_concat"] + list(range(1, layers + 1))
    else:
        coord, shape = HIDDEN_SPATIAL[hidden]
        dims = ModelDims.tiny(n_text=n_text, layers=layers, hidden=hidden, heads=hidden // 64, inter=2 * hidden,
                              coord=coord, shape=shape)
        exits = ["vision_avg", "text_avg", "text_visual_concat", 1]
    ee = ExitConfig.from_dict(dict(exits=exits, encoder_layer_strategy="ramp", inference_strategy="max_confidence"))
    sd = synth.make_state_dict(dims, ee, seed=5)
    docs = synth.make_docs(dims, 5 if hidden is None else 4, seed=41, pad=True)
    model = B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=8, dtype=dtype)
    got = model.forward(**_cuda(docs)).exit_logits.cpu().numpy()
    want = port.forward(sd, dims, ee, docs)["exit_logits"].numpy()
    assert np.isfinite(got).all()
    err = np.abs(got - want).max()
    if hidden is not None:
        print(f"hidden {hidden} [{dtype}]: max|logits - port| = {err:.3e}")
    assert err <= TOL[dtype]
    dense = model.infer(**_cuda(docs), exit_threshold=0.2, early_exit=False)
    early = model.infer(**_cuda(docs), exit_threshold=0.2)
    assert np.array_equal(dense.exits_store, early.exits_store) and torch.equal(dense.logits, early.logits)
    model.close()


def test_pipelined_submit_collect_equals_blocking():
    """mmee_forward_submit / mmee_forward_collect (two forwards in flight) return what the blocking call returns."""
    model, g, dims, ee, sd, docs = _engine("tiny_ramp_conf")
    temps = g["temps"]
    a = {k: v.clone().pin_memory() for k, v in docs.items()}
    b = {k: v.flip(0).clone().pin_memory() for k, v in docs.items()}
    ra = model.infer(**a, exit_threshold=0.5, temperatures=temps)
    rb = model.infer(**b, exit_threshold=0.5, temperatures=temps)
    t1 = model.infer_submit(**a, exit_threshold=0.5, temperatures=temps)
    t2 = model.infer_submit(**b, exit_threshold=0.5, temperatures=temps)
    with pytest.raises(RuntimeError, match="in flight"):
        model.infer_submit(**a, exit_threshold=0.5, temperatures=temps)
    pa = model.infer_collect(t1)
    t3 = model.infer_submit(**a, exit_threshold=0.9, temperatures=temps)
    pb = model.infer_collect(t2)
    pc = model.infer_collect(t3)
    for p, r in ((pa, ra), (pb, rb)):
        assert np.array_equal(p.exits_store, r.exits_store) and torch.equal(p.logits, r.logits.cpu())
        assert np.array_equal(p.exit_hist, r.exit_hist) and np.array_equal(p.criteria, r.criteria)
    rc = model.infer(**a, exit_threshold=0.9, temperatures=temps)
    assert np.array_equal(pc.exits_store, rc.exits_store) and torch.equal(pc.logits, rc.logits.cpu())
    with pytest.raises(RuntimeError, match="ticket"):
        model.infer_collect(t1)


@pytest.mark.parametrize("gain", [8.0, 25.0, 60.0])
def test_large_scores_exercise_lazy_rescale(gain):
    """Trained-model-like score ranges: scale W_q / W_k and the relative-position tables so that attention scores
    span tens of log2 units within a row and the row maximum moves from key tile to key tile.  This drives the lazy
    O-rescale path of the attention kernel (reference raised by more than 2^8 after the first tile), which the
    random-init fixtures never reach.  Engine vs the fp32 oracle port; probabilities are peaky here, so the bar is the
    bf16 one on the logits plus finiteness."""
    from mmee.model import B200EEForSequenceClassification
    from oracle import port

    dims = ModelDims.tiny(layers=2)
    ee = ExitConfig.from_dict(dict(exits=["text_visual_concat", 1, 2], encoder_layer_strategy="ramp",
                                   inference_strategy="max_confidence"))
    sd = synth.make_state_dict(dims, ee, seed=9)
    for k in list(sd):
        if k.endswith("attention.self.query.weight") or k.endswith("attention.self.key.weight"):
            sd[k] = sd[k] * gain
        if "rel_pos" in k:
            sd[k] = sd[k] * (gain * 10.0)
    docs = synth.make_docs(dims, 4, seed=51, pad=True)
    model = B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=4)
    got = model.forward(**_cuda(docs)).exit_logits.cpu().numpy()
    want = port.forward(sd, dims, ee, docs)["exit_logits"].numpy()
    assert np.isfinite(got).all()
    err = np.abs(got - want).max()
    print(f"gain {gain}: max|logits - port| = {err:.3e}")
    assert err <= LOGIT_TOL
    model.close()


DELTA_LTE = 2.5e-3        # decisive margin on the learned-to-exit score sigmoid(w . CLS + b); measured engine-vs-port
                          # score error: 5e-4 (base, std 0.02 weights), 1.8e-3 (tiny cases, std 0.08 weights)


@pytest.mark.parametrize("name", ["tiny_lte_ramp", "tiny_lte_gate", "base4_lte_ramp"])
def test_lte_early_exit_matches_reference_golden(name):
    """EE_config["use_lte"] (EE/models/LayoutLMv3.py:142-149, 231-268): documents leave at the first eligible
    encoder exit whose learned score is below the global threshold.  Exit layers equal the reference's (run one
    document at a time, golden) for every document whose visited scores keep DELTA_LTE from the threshold;
    returned logits within 1e-2; early-exit mode == dense mode bit for bit."""
    from helpers import LTE_CASES  # noqa: F401
    from oracle import port
    model, g, dims, ee, sd, docs = _engine(name, max_batch=16)
    thr = float(ee.global_threshold)
    res = model.infer(**_cuda(docs), return_all=True)               # criterion defaults to "lte"
    layer_of = [max(l, 0) for l in model.exit_layers] + [0]          # exit index -> encoder layer (0 = none / final)
    got_layer = np.array([layer_of[e] for e in res.exits_store])
    ref_layer = g["exit_layer"]
    scores = port.lte_scores(sd, port.forward(sd, dims, ee, docs)).numpy()
    E = model.n_exits
    decisive = np.ones(len(ref_layer), bool)
    for d_i, l in enumerate(ref_layer):
        stop = model.exit_layers.index(int(l)) if l > 0 else E - 1
        decisive[d_i] = np.abs(scores[:stop + 1, d_i] - thr).min() > DELTA_LTE
    agree = (got_layer == ref_layer)
    print(f"{name}: exit layers {got_layer.tolist()} reference {ref_layer.tolist()} decisive {int(decisive.sum())}/{len(decisive)}")
    assert decisive.sum() >= 3
    assert agree[decisive].all()
    err = np.abs(res.logits.cpu().numpy() - g["logits"])[agree].max()
    print(f"{name}: max|logits - reference| = {err:.3e}")
    assert err <= LOGIT_TOL
    # the engine's scores at the exits each document reached equal the port's
    got_scores = res.all_criteria.cpu().numpy()
    reached = ~np.isnan(got_scores)
    print(f"{name}: max|score - port| = {np.abs(got_scores - scores)[reached].max():.3e}")
    assert np.abs(got_scores - scores)[reached].max() < DELTA_LTE
    # dense mode takes the same decisions and returns the same bits
    dense = model.infer(**_cuda(docs), early_exit=False)
    assert np.array_equal(dense.exits_store, res.exits_store)
    assert torch.equal(dense.logits, res.logits)
    # max-confidence policy on the same engine still works (the scorer is only read by criterion "lte")
    conf = model.infer(**_cuda(docs), criterion="max_confidence", exit_threshold=0.5)
    assert conf.exits_store.shape == res.exits_store.shape


def test_lte_needs_its_weights():
    model, g, dims, ee, sd, docs = _engine("tiny_ramp_conf")
    with pytest.raises(RuntimeError, match="lte_classifier"):
        model.infer(**_cuda(docs), criterion="lte")


def test_ragged_attention_masks_vs_port():
    """Masks the tokenizer never emits but the interface allows: holes in the middle, a document with every text token
    masked (all eight text key tiles are skipped), a single live token, an all-ones mask.  Engine vs the oracle port."""
    from mmee.model import B200EEForSequenceClassification
    from oracle import port

    dims = ModelDims.tiny(layers=2)
    ee = ExitConfig.from_dict(dict(exits=["text_visual_concat", 1, 2], encoder_layer_strategy="ramp",
                                   inference_strategy="max_confidence"))
    sd = synth.make_state_dict(dims, ee, seed=9)
    docs = synth.make_docs(dims, 6, seed=51, pad=False)
    g = torch.Generator().manual_seed(7)
    m = docs["attention_mask"].clone()
    m[0] = (torch.rand(dims.n_text, generator=g) < 0.5).long()       # random holes
    m[1] = 0                                                          # no text token visible
    m[2] = 0; m[2, 0] = 1                                             # only <s>
    m[3, 64:192] = 0                                                  # two whole key tiles masked in the middle
    m[4, :448] = 0                                                    # only the last text tile is live
    docs["attention_mask"] = m
    model = B200EEForSequenceClassification(dims, ee, sd, device=0, max_batch=8)
    got = model.forward(**_cuda(docs)).exit_logits.cpu().numpy()
    want = port.forward(sd, dims, ee, docs)["exit_logits"].numpy()
    assert np.isfinite(got).all()
    err = np.abs(got - want).max()
    print(f"ragged masks: max|logits - port| = {err:.3e}")
    assert err <= LOGIT_TOL
    early = model.infer(**_cuda(docs), exit_threshold=0.0701)
    dense = model.infer(**_cuda(docs), exit_threshold=0.0701, early_exit=False)
    assert np.array_equal(dense.exits_store, early.exits_store) and torch.equal(dense.logits, early.logits)
    model.close()


def test_infer_device_is_stream_ordered_and_async():
    """infer_device enqueues on torch's current stream (the legacy default stream included) without waiting: inputs
    produced by torch kernels just before the call are seen, results feed torch ops just after it, and two calls may be
    in flight back to back; mmee_sync (through `infer`) is the blocking form."""
    model, g, dims, ee, sd, docs = _engine("tiny_ramp_conf")
    dev_docs = _cuda(docs)
    ref = model.infer(**dev_docs, exit_threshold=0.0701)
    for stream in (torch.cuda.current_stream(), torch.cuda.Stream()):
        with torch.cuda.stream(stream):
            # inputs made by torch kernels on this stream immediately before the call
            shifted = {k: (v.clone() if v.dtype != torch.float32 else v * 1.0) for k, v in dev_docs.items()}
            r1 = model.infer_device(**shifted, exit_threshold=0.0701)
            s1 = r1["logits"].sum()                      # consumer on the same stream, no host sync in between
            l1, e1 = r1["logits"].clone(), r1["exit_index"].clone()
            r2 = model.infer_device(**shifted, exit_threshold=0.0701)
            l2 = r2["logits"].clone()
        stream.synchronize()
        assert torch.equal(l1, ref.logits) and torch.equal(l2, ref.logits)
        assert np.array_equal(e1.cpu().numpy(), ref.exits_store)
        assert torch.isfinite(s1).item()
