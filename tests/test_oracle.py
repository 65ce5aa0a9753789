"""CPU tests: the oracle port and policy port against the golden vectors (outputs of the
unmodified reference, tests/golden/make_golden.py) and, when the original project's source tree is present
(MMEE_REFERENCE_ROOT), against the reference's own classes live."""
import os

import numpy as np
import pytest
import torch

from helpers import ALL_CASES, load_case
from oracle import policy_port, port, reference_harness


@pytest.mark.parametrize("name", ALL_CASES)
def test_port_matches_reference_golden(name):
    g, dims, ee, sd, docs = load_case(name)
    out = port.forward(sd, dims, ee, docs)
    # same torch build => bit-exact in practice; 2e-6 leaves room for a different BLAS thread split
    assert np.abs(out["exit_logits"].numpy() - g["exit_logits"]).max() <= 2e-6
    assert np.abs(out["head_logits"].numpy() - g["head_logits"]).max() <= 2e-6
    assert np.abs(out["last_hidden"][:, 0].numpy() - g["last_hidden_cls"]).max() <= 2e-5
    assert np.abs(out["last_hidden"].numpy()[:, ::37, ::5] - g["last_hidden_sample"]).max() <= 2e-5
    assert (out["exit_logits"].argmax(-1).numpy() == g["exit_logits"].argmax(-1)).all()


@pytest.mark.parametrize("name", ALL_CASES)
def test_policy_port_matches_reference_policy_golden(name):
    g, *_ = load_case(name)
    lg = g["exit_logits"].astype(np.float64)
    for tag, l in (("raw", lg), ("cal", policy_port.temperature_scale(lg, g["temps"]))):
        for thr in (0.1, 0.5, 0.7, 0.9):
            ex, pred, dist = policy_port.exit_policy(l, thr, "max_confidence")
            assert np.array_equal(ex, g[f"policy_{tag}_{thr}_exits"])
            assert np.array_equal(pred, g[f"policy_{tag}_{thr}_pred"])
            ex2, pred2, _ = policy_port.exit_policy_vectorised(l, thr, "max_confidence")
            assert np.array_equal(ex2, ex) and np.array_equal(pred2, pred)   # thresh.py:308-318 property
            assert abs(sum(dist.values()) - 1.0) < 1e-12


@pytest.mark.parametrize("name", ["tiny_gate_ent", "base_gate_ent"])
def test_criteria_match_reference_functions(name):
    g, *_ = load_case(name)
    cal = policy_port.temperature_scale(g["exit_logits"].astype(np.float64), g["temps"])
    assert np.abs(policy_port.criterion(cal, "entropy") - g["ref_entropy_cal"]).max() < 2e-5
    assert np.abs(policy_port.criterion(cal, "max_confidence") - g["ref_maxconf_cal"]).max() < 2e-6
    cal32 = torch.from_numpy(cal).float()
    for e in range(cal.shape[0]):
        assert torch.allclose(port.entropy(cal32[e]), torch.from_numpy(g["ref_entropy_cal"][e]), atol=1e-6)
        assert torch.allclose(port.max_confidence(cal32[e]), torch.from_numpy(g["ref_maxconf_cal"][e]), atol=1e-7)


def test_policy_edge_cases():
    rng = np.random.default_rng(0)
    lg = rng.normal(size=(5, 64, 16)) * 3
    # threshold 1.0 can never be exceeded (strict >): everything leaves at the last exit
    ex, pred, dist = policy_port.exit_policy(lg, 1.0)
    assert (ex == 4).all() and dist[4] == 1.0 and np.array_equal(pred, lg[4])
    # threshold 0 always fires at exit 0
    ex, pred, _ = policy_port.exit_policy(lg, 0.0)
    assert (ex == 0).all() and np.array_equal(pred, lg[0])
    # per-exit thresholds, entropy criterion; loop == vectorised
    thr = np.array([0.5, 1.0, 1.5, 2.0, 0.0])
    a = policy_port.exit_policy(lg, thr, "entropy")
    b = policy_port.exit_policy_vectorised(lg, thr, "entropy")
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    # single exit (E+1 == 1)
    ex, pred, _ = policy_port.exit_policy(lg[:1], 0.99)
    assert (ex == 0).all()


@pytest.mark.skipif(not reference_harness.available(),
                    reason="needs the original project's source tree (MMEE_REFERENCE_ROOT), which the repository does not contain")
def test_port_matches_live_reference_tiny():
    from mmee import synth
    from mmee.config import ExitConfig, ModelDims

    dims = ModelDims.tiny(layers=2)
    ee = ExitConfig.from_dict(dict(exits=["text_visual_concat", 1, 2], encoder_layer_strategy="gate",
                                   inference_strategy="entropy"))
    sd = synth.make_state_dict(dims, ee, seed=11)
    docs = synth.make_docs(dims, 3, seed=12)
    model = reference_harness.build_reference_model(dims, ee, sd)
    ref = reference_harness.reference_forward(model, docs)
    out = port.forward(sd, dims, ee, docs)
    assert torch.allclose(out["exit_logits"], ref["exit_logits"], atol=2e-6)
    assert torch.allclose(out["head_logits"], ref["head_logits"], atol=2e-6)
    assert torch.allclose(out["last_hidden"], ref["last_hidden"], atol=2e-5)


@pytest.mark.parametrize("name", ["cal_a", "cal_b", "cal_c"])
def test_calibration_port_matches_reference_temperatures(name):
    """oracle/calibration_port.py against the temperatures the reference's own TemperatureScaler produced
    (tests/golden/make_calibration_golden.py; one scaler reused across exits as EE/eval.py:298-313 does)."""
    from oracle import calibration_port
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "calibration.npz"))
    seed, E1, N, K = (int(v) for v in g[f"{name}_shape"])
    logits, labels = calibration_port.synthetic_exit_logits(seed, E1, N, K)
    scaler = calibration_port.TemperatureScalerPort()
    for e in range(E1):
        t = float(scaler.fit(labels, logits[e])[0])
        assert abs(t - g[f"{name}_t_ref"][e]) <= 1e-3 * g[f"{name}_t_ref"][e]
        assert abs(calibration_port.nll(labels, logits[e], t) - g[f"{name}_nll_ref"][e]) < 1e-8
        # both sit at the minimiser up to L-BFGS-B's tolerance
        assert abs(t - g[f"{name}_t_opt"][e]) <= 1e-3 * g[f"{name}_t_opt"][e]


@pytest.mark.parametrize("name", ["tiny_lte_ramp", "tiny_lte_gate", "base4_lte_ramp"])
def test_lte_port_matches_reference_golden(name):
    """Learned-to-exit inference (EE_config["use_lte"]): the port's per-document decision and returned logits
    against what the unmodified reference produced document by document (tests/golden/make_golden.py)."""
    g, dims, ee, sd, docs = load_case(name)
    assert ee.use_lte and "layoutlmv3.encoder.lte_classifier.weight" in sd
    out = port.forward(sd, dims, ee, docs)
    r = port.lte_exit(sd, ee, out, float(ee.global_threshold))
    assert r["exit_layer"].tolist() == g["exit_layer"].tolist()
    assert len(set(g["exit_layer"].tolist())) >= 2                   # the case exercises several exits
    assert np.abs(r["logits"].numpy() - g["logits"]).max() < 1e-4


@pytest.mark.parametrize("tag", ["mix_a_msp", "mix_a_entropy", "mix_a_margin", "mix_b_msp", "mix_b_entropy"])
def test_mixture_port_matches_reference_golden(tag):
    """oracle check_2d_threshold / opt0_2d / generate_thresholds / evaluate_exit_logits against what the reference's
    own functions produced (tests/golden/make_mixture_golden.py runs them unmodified)."""
    import sys
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "mixtures.npz"))
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    from make_mixture_golden import synthetic_store
    seed, E1, N, K, npe, M = (int(v) for v in g[tag + "_shape"])
    lg, labels = synthetic_store(seed, E1, N, K)
    csf = policy_port.csf(lg, tag.split("_")[-1])
    assert np.allclose(csf.sum(1), g[tag + "_csf_sum"], rtol=1e-13)
    thr2d = policy_port.generate_thresholds(csf, npe, M)
    assert np.array_equal(thr2d, g[tag + "_thr2d"])
    exits = policy_port.opt0_2d(csf, thr2d)
    assert np.array_equal(exits, g[tag + "_exits"])
    for t in (0, 1, M // 2, M - 1):
        acc, avg, dist = policy_port.evaluate_exit_logits(lg, labels, exits[t])
        assert acc == g[tag + "_acc"][t] and avg == g[tag + "_avg_exit"][t]
        assert abs(sum(dist.values()) - 1.0) < 1e-12


def test_policy_port_properties_randomised():
    """Randomised properties of the policy restatement (hypothesis): the per-sample double loop of EE/policy.py:28-45
    equals the vectorised form for any logits / per-exit thresholds, exits are monotone in a global threshold, the last
    exit always fires, and check_2d_threshold is the argmax-of->= rule with its all-False -> 0 corner."""
    from hypothesis import given, settings, strategies as st
    from hypothesis.extra import numpy as hnp

    @settings(max_examples=60, deadline=None)
    @given(hnp.arrays(np.float64, st.tuples(st.integers(1, 5), st.integers(1, 12), st.integers(2, 6)),
                      elements=st.floats(-6, 6, allow_nan=False, width=32)),
           st.floats(0.05, 0.999), st.floats(0.05, 0.999), st.sampled_from(["max_confidence", "entropy"]))
    def check(lg, t1, t2, kind):
        E1, N, K = lg.shape
        lo, hi = sorted((t1, t2))
        scale = 1.0 if kind == "max_confidence" else np.log(K)
        a = policy_port.exit_policy(lg, lo * scale, kind)
        b = policy_port.exit_policy_vectorised(lg, lo * scale, kind)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
        c = policy_port.exit_policy_vectorised(lg, hi * scale, kind)
        # a higher confidence threshold exits later; a higher entropy threshold exits earlier
        assert (c[0] >= b[0]).all() if kind == "max_confidence" else (c[0] <= b[0]).all()
        assert (a[0] <= E1 - 1).all() and abs(sum(a[2].values()) - 1.0) < 1e-12
        thr = np.linspace(lo, hi, E1)
        d = policy_port.exit_policy(lg, thr * scale, kind)
        e = policy_port.exit_policy_vectorised(lg, thr * scale, kind)
        assert np.array_equal(d[0], e[0])
        csf = policy_port.csf(lg, "msp")
        ex = policy_port.check_2d_threshold(csf, thr)
        fire = csf >= thr[:, None]
        assert np.array_equal(ex, np.where(fire.any(0), fire.argmax(0), 0))

    check()
