"""Transformer (sup) oracle and host module replayed against tests/golden/forward_sup.npz, which was produced by the
reference's own bonito.transformer classes (oracle/make_golden.py, oracle/reference_shim.load_transformer)."""
import json
import os

import numpy as np
import pytest
import torch
from _helpers import at_sample

from oracle import synth
from oracle import transformer_oracle as TO


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "forward_sup.npz"))


def _spec_weights(gold):
    spec = json.loads(str(gold["spec"]))
    spec["convs"] = [tuple(c) for c in spec["convs"]]
    spec["window"] = tuple(spec["window"])
    w = {k[2:]: torch.from_numpy(gold[k].astype(np.float32)) for k in gold.files if k.startswith("w.")}
    return spec, w


def _strip_blanks(scores_tnc):
    t, n, c = scores_tnc.shape
    s = scores_tnc.reshape(t, n, c // 5, 5)
    assert np.all(s[..., 0] == 2.0)
    return np.ascontiguousarray(s[..., 1:].reshape(t, n, -1).transpose(1, 0, 2))


def test_oracle_matches_reference_transformer(gold):
    spec, w = _spec_weights(gold)
    with torch.no_grad():
        s, feats = TO.transformer_forward(w, spec, torch.from_numpy(gold["x"]), return_features=True)
    np.testing.assert_allclose(feats["conv4"].permute(0, 2, 1).numpy(), gold["conv"], atol=2e-5)
    np.testing.assert_allclose(feats["layer0"].numpy(), gold["layer0"], atol=2e-5)
    np.testing.assert_allclose(s.numpy(), _strip_blanks(gold["scores"]), atol=1e-4)


def test_host_module_matches_reference_transformer(gold):
    from bonito_b200.transformer import Model
    from bonito_b200.transformer.model import deepnorm_params, sliding_window_mask
    spec, w = _spec_weights(gold)
    model = Model(synth.sup_config(spec))
    model.load_state_dict(synth.sup_state_dict(spec, w))
    model.eval()
    with torch.inference_mode():
        scores = model(torch.from_numpy(gold["x"]))
    np.testing.assert_allclose(scores.numpy(), gold["scores"], atol=1e-4)
    assert model.stride == int(gold["stride"]) == 6
    assert deepnorm_params(18) == (2.4494897, 0.2886751)            # dna_r10.4.1@v5.0.toml:98-99
    m = sliding_window_mask(6, (1, 2), "cpu")
    assert m[3].tolist() == [False, False, True, True, True, True] and m[0].tolist() == [True, True, True, False, False, False]


def test_use_koi_rewrites_the_encoder_like_the_reference():
    from bonito_b200.nn import LinearCRFEncoder, MakeContiguous, Permute, Serial
    from bonito_b200.transformer import Model
    spec = synth.sup_spec(depth=1, d_model=64, nhead=2, dim_feedforward=128, state_len=3)
    spec["convs"] = [(1, 8, 5, 1, 2, "swish"), (8, 8, 5, 1, 2, "swish"), (8, 16, 9, 3, 4, "swish"),
                     (16, 16, 9, 2, 4, "swish"), (16, 64, 5, 2, 2, "swish")]
    model = Model(synth.sup_config(spec))
    model.use_koi(batchsize=4, chunksize=1200, quantize=False)
    assert isinstance(model.encoder, Serial) and isinstance(model.encoder[1], Permute) and isinstance(model.encoder[2], MakeContiguous)
    crf = [m for m in model.encoder.modules() if isinstance(m, LinearCRFEncoder)][0]
    assert crf.expand_blanks is False
    with pytest.raises(Exception):      # armed native path without a CUDA device: loud failure
        model(torch.zeros(1, 1, 1200))


def _wide(golden_dir):
    from oracle.make_golden import weights_digest
    gold = np.load(os.path.join(golden_dir, "forward_sup_wide.npz"))
    spec = synth.sup_spec(depth=int(gold["depth"]))
    weights = synth.make_sup_weights(spec, seed=int(gold["seed"]))
    if weights_digest(weights) != str(gold["digest"]):
        pytest.skip("seeded sup weights differ on this machine: fixture not comparable")
    return gold, spec, weights


def test_oracle_matches_reference_transformer_at_sup_width(golden_dir):
    """d_model 512, 8 heads, ff 2048, 6 layers, k = 5: the oracle against the reference's own classes (fp32)."""
    gold, spec, w = _wide(golden_dir)
    with torch.no_grad():
        s, feats = TO.transformer_forward(w, spec, torch.from_numpy(gold["x"].astype(np.float32)), return_features=True)
    np.testing.assert_allclose(at_sample(feats["conv4"].permute(0, 2, 1), gold, "conv"), gold["conv"], atol=5e-5)
    np.testing.assert_allclose(at_sample(feats["layer0"], gold, "layer0"), gold["layer0"], atol=5e-5)
    np.testing.assert_allclose(at_sample(feats["layer5"], gold, "layer5"), gold["layer5"], atol=1e-4)
    np.testing.assert_allclose(at_sample(s, gold, "scores_ntc"), gold["scores_ntc"], atol=5e-4)   # |x| ~ 11 (x5 scale)
    # the same-rounding (fp16 storage) oracle the GPU tests compare with stays within half-precision distance of it
    with torch.no_grad():
        s16 = TO.transformer_forward(w, spec, torch.from_numpy(gold["x"].astype(np.float32)), fp16=True)
    err = np.abs(at_sample(s16, gold, "scores_ntc") - gold["scores_ntc"])
    assert err.max().item() <= 8e-2 and err.mean().item() <= 6e-3, (err.max().item(), err.mean().item())
