"""CPU tests (no GPU): C-ABI surface, host-side logic, data-parallel plumbing (gloo, world_size 2)."""
import ctypes as C
import os
import re
import socket

import numpy as np
import pytest
import torch

from mmee import _lib, synth
from mmee.calibration import TemperatureScaler, spread_temperatures, thresholds_for
from mmee.config import ExitConfig, ModelDims
from oracle import policy_port, port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "mmee.h")).read()
    declared = sorted(set(re.findall(r"\b(mmee_[a-z_0-9]+)\s*\(", hdr)))
    assert declared, "no declarations parsed"
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/mmee.h but not exported by libmmee.so"
    assert set(_lib.EXPORTED_SYMBOLS) <= set(declared)
    assert b"sm_100a" in lib.mmee_version()


def test_struct_layout_matches_header():
    # field order/count of the ctypes mirrors must follow include/mmee.h
    hdr = open(os.path.join(ROOT, "include", "mmee.h")).read()
    desc = hdr[hdr.index("typedef struct {", hdr.index("Model description")):hdr.index("} mmee_model_desc;")]
    names = [f[0] for f in _lib.ModelDesc._fields_]
    for tok in ["hidden", "layers", "heads", "inter", "n_text", "image", "patch", "channels", "n_labels", "coord",
                "shape", "vocab", "max_pos", "max_2d", "rel_bins", "max_rel", "rel2d_bins", "max_rel2d", "pad_id",
                "ln_eps", "vis_ln_eps", "n_exits", "exit_after_layer", "head_kind", "head_layers", "compute_dtype"]:
        assert tok in names and tok in desc
    pos = [desc.index(t) for t in names]
    assert pos == sorted(pos), "ctypes ModelDesc field order differs from the header"
    assert C.sizeof(_lib.ModelDesc) == 4 * (21 + 1 + 64 + 3)
    assert _lib.COMPUTE_DTYPES == {"bf16": int(re.search(r"#define MMEE_DTYPE_BF16 (\d+)", hdr).group(1)),
                                   "fp32": int(re.search(r"#define MMEE_DTYPE_FP32 (\d+)", hdr).group(1))}
    assert [f[0] for f in _lib.Outputs._fields_] == ["logits", "exit_index", "criterion", "all_exit_logits",
                                                     "all_head_logits", "all_criteria", "exit_hist"]


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a box WITHOUT a GPU")
def test_engine_fails_loudly_without_gpu():
    """No CPU fallback: creating an engine without a CUDA device is an error, not a silent slow path."""
    from mmee.model import B200EEForSequenceClassification

    dims = ModelDims.tiny(layers=1)
    ee = ExitConfig.from_dict(dict(exits=["text_visual_concat", 1]))
    with pytest.raises(RuntimeError, match="no CUDA device|libmmee"):
        B200EEForSequenceClassification(dims, ee, {}, device=0, max_batch=2)
    lib = _lib.load()
    h = C.c_void_p()
    d = _lib.ModelDesc()
    assert lib.mmee_create(C.byref(d), 0, 1, C.byref(h)) != 0
    assert lib.mmee_last_error()


def test_exit_config_mirrors_reference_fields():
    ee = ExitConfig.from_dict({"training_strategy": "one_stage_subgraphs_weighted", "exits": "text_visual_concat,1,4,8",
                               "encoder_layer_strategy": "gate", "inference_strategy": "entropy",
                               "global_threshold": 0.3, "model_weights": "microsoft/layoutlmv3-base", "unknown": 1})
    assert ee.exits == ["text_visual_concat", 1, 4, 8] and ee.encoder_exit_layers == [1, 4, 8] and ee.has_concat_exit
    assert ee.encoder_layer_strategy == "gate" and ee.inference_strategy == "entropy" and ee.exit_head_num_layers == 2
    with pytest.raises(NotImplementedError):
        ExitConfig.from_dict({"inference_strategy": "patience"})
    with pytest.raises(NotImplementedError):
        ExitConfig.from_dict({"encoder_layer_strategy": "embexit"})


def test_synthetic_inputs_are_deterministic_and_well_formed():
    dims = ModelDims.base()
    a, b = synth.make_docs(dims, 5, seed=3), synth.make_docs(dims, 5, seed=3)
    for k in a:
        assert torch.equal(a[k], b[k])
    assert a["input_ids"].shape == (5, 512) and a["bbox"].shape == (5, 512, 4) and a["pixel_values"].shape == (5, 3, 224, 224)
    assert (a["input_ids"][:, 0] == 0).all()
    assert int(a["bbox"].max()) <= 1000 and int(a["bbox"].min()) >= 0
    pad = a["attention_mask"] == 0
    assert (a["input_ids"][pad] == dims.pad_id).all() and (a["bbox"][pad] == 0).all()
    assert a["attention_mask"][0].all()                      # one unpadded document
    assert float(a["pixel_values"].abs().max()) <= 1.0
    ee = ExitConfig.from_dict(dict(exits=["text_visual_concat", 1, 2, 3]))
    sd1, sd2 = synth.make_state_dict(ModelDims.tiny(), ee, 0), synth.make_state_dict(ModelDims.tiny(), ee, 0)
    assert all(torch.equal(sd1[k], sd2[k]) for k in sd1)
    assert "layoutlmv3.encoder.early_exits.2.out_proj.weight" in sd1 and "classifier.dense.weight" in sd1


def test_bucket_lut_matches_hf_function():
    from mmee.model import bucket_lut

    for bins, maxd in ((32, 128), (64, 256)):
        lut = bucket_lut(bins, maxd)
        rel = torch.arange(-1023, 1024)
        want = port.relative_position_bucket(rel, bins, maxd)
        got = (rel > 0).long() * (bins // 2) + torch.from_numpy(lut.astype(np.int64))[rel.abs()]
        assert torch.equal(got, want)


def test_temperature_scaler_fails_loudly_without_gpu_and_spread():
    rng = np.random.default_rng(0)
    logits = rng.normal(size=(512, 16)) * 4.0
    labels = logits.argmax(-1)
    ts = TemperatureScaler()
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CUDA device"):       # device fit, no CPU fallback
            ts.fit(labels, logits)
    assert np.allclose(ts.temperature_scale(logits), logits)            # T = 1 until fitted
    assert np.allclose(TemperatureScaler(2.0).temperature_scale(logits), logits / 2.0)
    # the host-side ECE equals the oracle's restatement of the same definition
    from mmee.calibration import ece_equal_mass
    from oracle import calibration_port
    from scipy.special import softmax
    assert ece_equal_mass(labels, logits) == pytest.approx(calibration_port.ece_equal_mass(labels, softmax(logits, -1)))
    assert 0.0 <= ece_equal_mass(labels, logits) <= 1.0
    stack = rng.normal(size=(5, 200, 16)) * 0.1
    for kind in ("max_confidence", "entropy"):
        temps = spread_temperatures(stack, kind)
        crit = policy_port.criterion(policy_port.temperature_scale(stack, temps), kind)
        med = np.median(crit, axis=1)
        assert (np.diff(med) > 0).all() if kind == "max_confidence" else (np.diff(med) < 0).all()
    assert thresholds_for("max_confidence", 0.7, 16) == 0.7
    assert 0 < thresholds_for("entropy", 0.9, 16) < thresholds_for("entropy", 0.5, 16) < np.log(16)


def test_shard_range_partitions_exactly():
    from mmee.dist import shard_range

    for n in (1, 7, 8, 8192, 8191):
        for w in (1, 2, 3, 8):
            spans = [shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gather_worker(rank, world, port_no, n_total, out_dir):
    import torch.distributed as dist

    from mmee.dist import gather_results, gather_results_fixed, shard_range

    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port_no}", rank=rank, world_size=world)
    g = torch.Generator().manual_seed(5)
    logits = torch.randn(n_total, 16, generator=g)
    exits = torch.randint(0, 14, (n_total,), generator=g, dtype=torch.int32)
    crit = torch.rand(n_total, generator=g)
    a, b = shard_range(n_total, rank, world)
    hist = torch.bincount(exits[a:b].long(), minlength=14)
    res = gather_results(logits[a:b], exits[a:b], crit[a:b], hist)
    ok = (torch.equal(res["logits"], logits) and torch.equal(res["exit_index"], exits) and torch.equal(res["criterion"], crit)
          and torch.equal(res["exit_hist"], torch.bincount(exits.long(), minlength=14)))
    # equal-shard hot-loop variant
    n_eq = (n_total // world) * world
    per = n_eq // world
    packed = torch.cat([logits[rank * per:(rank + 1) * per], exits[rank * per:(rank + 1) * per, None].float(),
                        crit[rank * per:(rank + 1) * per, None]], dim=1)
    out = torch.empty(n_eq, 18)
    h2 = torch.bincount(exits[rank * per:(rank + 1) * per].long(), minlength=14)
    gather_results_fixed(packed, h2, out)
    ok = ok and torch.equal(out[:, :16], logits[:n_eq]) and torch.equal(out[:, 16].int(), exits[:n_eq])
    ok = ok and torch.equal(h2, torch.bincount(exits[:n_eq].long(), minlength=14))
    # per-step asynchronous gather into a ring, one read-back at the end (what bench.py does at N > 1)
    from mmee.dist import JobGatherer, pack_results
    jg = JobGatherer(per, 18, 14, capacity=3, device="cpu")
    want_hist = torch.zeros(14, dtype=torch.int64)
    for step in range(5):                                         # more steps than ring slots: the last 3 survive
        lg = logits[:n_eq] + step
        mine = slice(rank * per, (rank + 1) * per)
        slot = jg.push(pack_results(lg[mine], exits[mine], crit[mine]), torch.bincount(exits[mine].long(), minlength=14))
        ok = ok and slot == step % 3
        want_hist += torch.bincount(exits[:n_eq].long(), minlength=14)
    fin = jg.finish()
    ok = ok and fin["steps"] == 5 and torch.equal(fin["exit_hist"], want_hist)
    for step in (2, 3, 4):
        rows = fin["results"][step % 3]
        ok = ok and torch.equal(rows[:, :16], logits[:n_eq] + step) and torch.equal(rows[:, 16].int(), exits[:n_eq])
        ok = ok and torch.equal(rows[:, 17], crit[:n_eq])
    ok = ok and jg.steps == 0 and int(jg.hist.sum()) == 0
    open(os.path.join(out_dir, f"ok{rank}"), "w").write("1" if ok else "0")
    dist.destroy_process_group()


def test_two_rank_gather_equals_single_process(tmp_path):
    """N>1 path on CPU: block-sharded results gathered over gloo == the unsharded arrays (uneven shards included)."""
    import torch.multiprocessing as mp

    world = 2
    mp.spawn(_gather_worker, args=(world, _free_port(), 37, str(tmp_path)), nprocs=world, join=True)
    assert all(open(os.path.join(tmp_path, f"ok{r}")).read() == "1" for r in range(world))


class _ReferenceLike:
    """What spec_from_reference reads off a reference model: its config (HF LayoutLMv3Config + EE_config, as the
    reference is constructed) and the state dict it loaded strictly."""

    def __init__(self, config, state_dict):
        self.config = config
        self._sd = state_dict

    def state_dict(self):
        return dict(self._sd)


def test_spec_from_reference_model():
    """from_reference() reads dims, exit config and weights off a constructed reference model (the reference itself
    when its source tree is present, else an object with the same `.config` / `.state_dict()`)."""
    from mmee.model import B200EEForSequenceClassification
    from oracle import reference_harness as RH

    dims = ModelDims.tiny(layers=2)
    ee = ExitConfig.from_dict(dict(exits=["text_visual_concat", 1, 2], encoder_layer_strategy="gate",
                                   inference_strategy="entropy", global_threshold=0.4))
    sd = synth.make_state_dict(dims, ee, seed=1)
    if RH.available():
        ref = RH.build_reference_model(dims, ee, sd)
    else:
        # checks the config half in full; the weight half only checks that names and values pass through, not that
        # mmee.synth names parameters as the reference does (its strict load in build_reference_model checks that)
        ref = _ReferenceLike(RH.reference_config(dims, ee), sd)
    d2, e2, sd2 = B200EEForSequenceClassification.spec_from_reference(ref)
    assert d2 == dims
    assert list(e2.exits) == list(ee.exits) and e2.encoder_layer_strategy == "gate" and e2.inference_strategy == "entropy"
    assert e2.global_threshold == 0.4
    for k, v in sd.items():
        assert torch.equal(sd2[k], v), k
    assert set(sd2) - set(sd) <= {"layoutlmv3.visual_bbox", "layoutlmv3.embeddings.position_ids"}


def test_policy_host_logic_and_loud_failure():
    """Host side of mmee.policy: per-exit thresholds of accuracy_calibration_heuristic (EE/policy.py:68-79) and
    argument checks; the scan itself has no CPU fallback."""
    from mmee.policy import Policy, heuristic_thresholds, policy_scan

    cm = {"accuracy": [0.5, 0.7, 0.9], "ece": [0.2, 0.1, 0.05]}
    thr = heuristic_thresholds(cm, 0.1, 3)
    metrics = np.array([1 - 0.5 / 0.2, 1 - 0.7 / 0.1, 1 - 0.9 / 0.05])
    want = (metrics - (metrics.min() - 0.1)) / ((metrics.max() + 0.1) - (metrics.min() - 0.1))
    assert np.allclose(thr, want) and (thr > 0).all() and (thr < 1).all()
    # threshold shapes are explicit, never guessed from a length (ADVICE r1): 1-D = T global thresholds, always
    from mmee.policy import _threshold_rows, generate_thresholds
    assert _threshold_rows(0.5, 4, False).shape == (1, 4)
    rows = _threshold_rows(np.array([0.1, 0.2, 0.3, 0.4]), 4, False)            # T == E1: still 4 sweep points
    assert rows.shape == (4, 4) and (rows == rows[:, :1]).all()
    assert np.array_equal(_threshold_rows(np.array([0.1, 0.2, 0.3, 0.4]), 4, True), [[0.1, 0.2, 0.3, 0.4]])
    assert _threshold_rows(np.zeros((7, 4)), 4, True).shape == (7, 4)
    with pytest.raises(ValueError):
        _threshold_rows(np.zeros(3), 4, True)
    with pytest.raises(ValueError):
        _threshold_rows(np.zeros((2, 5)), 4, False)
    # mixtures: same numpy stream as the reference's generate_thresholds (restated in the oracle)
    from oracle import policy_port
    csf = np.random.default_rng(0).random((5, 300))
    assert np.array_equal(generate_thresholds(csf, 10, 257), policy_port.generate_thresholds(csf, 10, 257))
    with pytest.raises(ValueError):
        policy_scan(np.zeros((3, 4)), 0.5)
    with pytest.raises(ValueError):
        policy_scan(np.zeros((3, 4, 5)), np.zeros((2, 4)))
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CUDA device|libmmee"):
            Policy(np.zeros((3, 4, 5)), {"exit_threshold": 0.5}).max_confidence_global_thresholding_policy()


def test_image_only_documents_and_port():
    """BASELINE config 5 shape: n_text = 0 -> 197 visual tokens; the oracle port runs it (CPU, tiny dims)."""
    dims = ModelDims.tiny(n_text=0, layers=1)
    assert dims.seq == dims.n_vis == 197
    docs = synth.make_docs(dims, 2, seed=4)
    assert docs["input_ids"].shape == (2, 0) and docs["bbox"].shape == (2, 0, 4)
    ee = ExitConfig.from_dict(dict(exits=["text_visual_concat", 1]))
    sd = synth.make_state_dict(dims, ee, seed=1)
    out = port.forward(sd, dims, ee, docs)
    assert out["exit_logits"].shape == (3, 2, dims.n_labels) and out["last_hidden"].shape == (2, 197, dims.hidden)
    assert torch.isfinite(out["exit_logits"]).all()
