"""The oracle (CPU restatement) and the bonito_b200 module tree replayed against golden vectors produced by the
reference's own modules (tests/golden/forward_fast.npz, written by oracle/make_golden.py).  The fixtures hold the
reference's outputs at a seeded sample of their last axis; full outputs are compared at those indices."""
import json
import os

import numpy as np
import pytest
import torch
from _helpers import at_sample

from oracle import build_ref, crf_oracle as O
from oracle import synth


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "forward_fast.npz"))


@pytest.fixture(scope="module")
def oracle_scores(gold):
    """Full [T, N, C + blanks] scores of the oracle on the fixture's weights and input, which the decode tests take as
    input; checked against the reference's scores first."""
    spec = synth.model_spec("fast", n_lstm=2)
    w, _ = _fused_weights(gold, spec)
    with torch.no_grad():
        s = O.lstm_crf_forward(w, spec, torch.from_numpy(gold["x"]), expand_blanks=True).numpy()
    np.testing.assert_allclose(at_sample(s, gold, "scores"), gold["scores"], atol=2e-5)
    return s


def _fused_weights(gold, spec):
    """Oracle-named fp32 weights with the reference's fused (BN-folded) convolutions."""
    pre = {k[4:]: torch.from_numpy(np.asarray(gold[k], dtype=np.float32)) for k in gold.files if k.startswith("pre.")}
    w = {}
    for i in range(3):
        w[f"conv{i}.weight"] = torch.from_numpy(gold[f"fused.encoder.{i}.conv.weight"])
        w[f"conv{i}.bias"] = torch.from_numpy(gold[f"fused.encoder.{i}.conv.bias"])
    for i in range(spec["n_lstm"]):
        p = f"encoder.{4 + i}.rnn."
        w[f"lstm{i}.w_ih"], w[f"lstm{i}.w_hh"] = pre[p + "weight_ih_l0"], pre[p + "weight_hh_l0"]
        w[f"lstm{i}.b_ih"], w[f"lstm{i}.b_hh"] = pre[p + "bias_ih_l0"], pre[p + "bias_hh_l0"]
    w["crf.weight"] = pre[f"encoder.{4 + spec['n_lstm']}.linear.weight"]
    return w, pre


def test_oracle_forward_matches_reference(gold):
    spec = synth.model_spec("fast", n_lstm=2)
    w, _ = _fused_weights(gold, spec)
    x = torch.from_numpy(gold["x"])
    with torch.no_grad():
        scores, feats = O.lstm_crf_forward(w, spec, x, expand_blanks=True, return_features=True)
    np.testing.assert_allclose(at_sample(feats["conv1"], gold, "feat_1"), gold["feat_1"], atol=2e-6)
    np.testing.assert_allclose(at_sample(feats["conv2"], gold, "feat_2"), gold["feat_2"], atol=2e-6)
    np.testing.assert_allclose(at_sample(feats["lstm0"], gold, "feat_4"), gold["feat_4"], atol=5e-6)
    np.testing.assert_allclose(at_sample(feats["lstm1"], gold, "feat_5"), gold["feat_5"], atol=5e-6)
    np.testing.assert_allclose(at_sample(scores, gold, "scores"), gold["scores"], atol=2e-5)
    assert scores.shape == (250, 3, 320)


def test_module_tree_forward_matches_reference(gold):
    """bonito_b200.nn builds the same torch modules from the same config and folds BN the same way."""
    from bonito_b200.crf.model import Model
    from bonito_b200.nn import fuse_bn_
    cfg = json.loads(str(gold["config"]))
    model = Model(cfg)
    sd = model.state_dict()
    for k in sd:
        if "pre." + k in gold.files:
            sd[k] = torch.from_numpy(np.asarray(gold["pre." + k], dtype=np.float32))
    model.load_state_dict(sd)
    model.eval()
    model.apply(fuse_bn_)
    for i in range(3):
        np.testing.assert_allclose(model.state_dict()[f"encoder.{i}.conv.weight"].numpy(),
                                   gold[f"fused.encoder.{i}.conv.weight"], atol=1e-7)
    with torch.inference_mode():
        scores = model(torch.from_numpy(gold["x"]))
    assert scores.shape == (250, 3, 320)
    np.testing.assert_allclose(at_sample(scores, gold, "scores"), gold["scores"], atol=2e-5)
    assert model.stride == int(gold["stride"])


def test_oracle_decode_batch_matches_reference_glue(gold, oracle_scores):
    strings, path = O.decode_batch(oracle_scores, state_len=3)
    assert strings == json.loads(str(gold["strings"]))
    assert all(len(s) > 50 for s in strings) and len(set(strings)) == len(strings)


def test_native_layout_decode_equals_decode_batch(gold, oracle_scores):
    """decode_native (kernel conventions, no blank column) == decode_batch on the blank-expanded scores."""
    s = oracle_scores.reshape(250, 3, 64, 5)
    assert np.all(s[..., 0] == 2.0)
    ntc = np.ascontiguousarray(s[..., 1:].reshape(250, 3, 256).transpose(1, 0, 2))
    moves, seq, qual, mass = O.decode_native(ntc, 3, blank_score=2.0)
    got = [r[r != 0].tobytes().decode() for r in seq]
    assert got == json.loads(str(gold["strings"]))
    assert np.array_equal(moves, (seq != 0).astype(np.uint8)) and np.array_equal(seq != 0, qual != 0)
    assert np.all(mass >= 0) and np.all(mass.sum(-1) <= 1 + 1e-9)


def test_c_decode_matches_numpy_oracle(gold, oracle_scores):
    """oracle/csrc/crf_decode_ref.c (the CPU-baseline decode) == crf_oracle.decode_native, incl. qualities, on the golden
    model's scores and on seeded random scores of every state length."""
    s = oracle_scores.reshape(250, 3, 64, 5)
    scores = np.ascontiguousarray(s[..., 1:].reshape(250, 3, 256).transpose(1, 0, 2))
    a = build_ref.decode(scores, 3, 2.0, 1.05, 0.2)
    b = O.decode_native(scores, 3, 2.0, 1.05, 0.2)[:3]
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert [r[r != 0].tobytes().decode() for r in a[1]] == json.loads(str(gold["strings"]))
    g = np.random.default_rng(3)
    for k, n, t in [(3, 3, 200), (4, 2, 150), (5, 1, 40)]:
        sc = np.clip(g.normal(size=(n, t, 4 ** (k + 1))) * 1.7, -5, 5).astype(np.float16).astype(np.float32)
        a = build_ref.decode(sc, k)
        b = O.decode_native(sc, k)[:3]
        for x, y in zip(a, b):
            assert np.array_equal(x, y)


def _hac_fixture(golden_dir):
    from oracle.make_golden import weights_digest
    gold = np.load(os.path.join(golden_dir, "forward_hac.npz"))
    spec = synth.model_spec("hac")
    weights = synth.make_weights(spec, seed=int(gold["seed"]))
    if weights_digest(weights) != str(gold["digest"]):
        pytest.skip("seeded hac weights round differently on this CPU (QR in the orthogonal init): fixture not comparable")
    return gold, spec, weights


def test_oracle_matches_reference_on_the_headline_shape(golden_dir):
    """hac shape (H = 384, 5 LSTM layers, 1024 scores): oracle forward == the reference module tree's scores
    (tests/golden/forward_hac.npz), oracle decode == the reference's decode_batch strings."""
    gold, spec, weights = _hac_fixture(golden_dir)
    x = torch.from_numpy(gold["x"].astype(np.float32))
    with torch.no_grad():
        s = O.lstm_crf_forward(weights, spec, x).permute(1, 0, 2).numpy()      # [N, T, C]
    np.testing.assert_allclose(at_sample(s, gold, "scores_ntc"), gold["scores_ntc"], atol=5e-5)
    seq = build_ref.decode(s, spec["state_len"], 2.0)[1]
    assert [r[r != 0].tobytes().decode() for r in seq] == json.loads(str(gold["strings"]))


def test_cpu_reference_model_matches_the_reference_fixtures(gold, golden_dir):
    """`oracle/cpu_reference.py::CpuReferenceModel` -- what bench.py times as `cpu_baseline` and under `--impl reference` --
    reproduces the scores the reference's own module tree produced (fast fixture with folded BN; hac headline shape) and
    the reference's decode_batch strings."""
    from oracle.cpu_reference import CpuReferenceModel
    spec = dict(synth.model_spec("fast", n_lstm=2), clamp=None)          # the fast fixture's config has no Clamp layer
    w, _ = _fused_weights(gold, spec)
    cfg = json.loads(str(gold["config"]))
    if any(layer.get("type") == "clamp" for layer in cfg["encoder"]["sublayers"]):
        spec["clamp"] = (-5.0, 5.0)
    ref = CpuReferenceModel(spec, w)
    s = ref(torch.from_numpy(gold["x"]))                                   # [T, N, C] without the blank column
    idx = gold["scores_idx"]                                               # blank-expanded column 5 * state + j, blank at j = 0
    real = idx % 5 != 0
    np.testing.assert_allclose(s.numpy()[..., 4 * (idx[real] // 5) + idx[real] % 5 - 1], gold["scores"][..., real], atol=2e-5)

    hac, hspec, hweights = _hac_fixture(golden_dir)
    href = CpuReferenceModel(hspec, hweights)
    x = torch.from_numpy(hac["x"].astype(np.float32))
    np.testing.assert_allclose(at_sample(href(x).permute(1, 0, 2), hac, "scores_ntc"), hac["scores_ntc"], atol=5e-5)
    seq = href.basecall_batch(x)[1]
    assert [r[r != 0].tobytes().decode() for r in seq] == json.loads(str(hac["strings"]))
