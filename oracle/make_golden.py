"""
ORACLE -- TEST INFRASTRUCTURE ONLY.  Generate tests/golden/*.npz by running the REFERENCE's own code
(imported from /root/reference through oracle/reference_shim.py) in the authoring container.

    python -m oracle.make_golden

The fixtures are committed; the GPU box (no /root/reference) only replays them.
Contents
  host_logic.npz   chunk / stitch / batchify results of bonito.util on arange signals, CTC_CRF.idx tables,
                   get_stride, conv length table
  forward_sup.npz  narrow transformer through the reference's bonito.transformer classes (Triton / CUDA-only pieces
                   replaced by flash-attn's torch reference functions, see oracle/reference_shim.load_transformer)
  forward_hac.npz  the headline shape (H = 384, 5 LSTM, k = 4) through the reference module tree, fp32 CPU: input, scores
                   without the blank column [N,T,1024] (sampled), decode_batch strings, digest of the seeded weights
  revcomp.npz      CTC_CRF.reverse_complement of the reference on small random scores, k = 3, 4, 5
  forward_sup_wide.npz  the sup v5 width (d_model 512, 8 heads, ff 2048, k = 5), 6 layers, through the reference's
                   bonito.transformer classes: input, conv output, layers 0 and 5, scores [N,2T',4096] (all sampled);
                   weights by digest
  forward_fast.npz reference module tree (bonito.nn via from_dict, BatchNorm folded by fuse_bn_) forward in
                   fp32 on CPU: input, every parameter, per-layer features and scores [T,N,C+blanks] (sampled);
                   + decode_batch strings (reference glue over the oracle's posteriors stand-in)

"Sampled" outputs keep a seeded subset of the indices of their last axis (channels or score columns; every chunk and
every time step stays), listed beside them as `<name>_idx`: each fixture file stays under 1 MB.  Inputs, parameters and
decoded strings are always stored whole.
"""

import json
import os

import numpy as np
import torch

from oracle import reference_shim, synth

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def sample_last_axis(out, names, fraction, seed=0):
    """Replace each named output by a seeded subset of its last axis (sorted indices stored as `<name>_idx`)."""
    rng = np.random.default_rng(seed)
    for name in names:
        n = out[name].shape[-1]
        idx = np.sort(rng.choice(n, max(1, round(n * fraction)), replace=False)).astype(np.int32)
        out[name] = np.ascontiguousarray(out[name][..., idx])
        out[name + "_idx"] = idx


class _Read:
    def __init__(self, rid, n):
        self.read_id = rid
        self.signal = np.arange(n, dtype=np.float32)


def host_logic(ref):
    out = {}
    cases = [(25000, 3996, 492, 6), (100000, 9996, 492, 6), (60000, 12000, 600, 6), (3000, 3996, 492, 6),
             (25000, 4000, 500, 6), (9996, 9996, 492, 6), (20000, 4000, 0, 5)]
    meta = []
    for i, (L, cs, ov, stride) in enumerate(cases):
        sig = torch.arange(L, dtype=torch.float32)
        chunks = ref.util.chunk(sig, cs, ov)
        # frames = every stride-th sample of each chunk, then the reference's stitch_results logic
        frames = chunks[:, 0, ::stride]
        if L < cs:
            stitched = frames[0, :int(np.floor(L / stride))]
        else:
            stitched = ref.util.stitch(frames, cs, ov, L, stride)
            stitched_rev = ref.util.stitch(frames, cs, ov, L, stride, reverse=True)
            out[f"stitch_rev_{i}"] = stitched_rev.numpy()
        out[f"chunk_first_{i}"] = chunks[:, 0, 0].numpy()   # first sample of every chunk identifies the window
        out[f"chunk_shape_{i}"] = np.array(chunks.shape)
        out[f"stitch_{i}"] = stitched.numpy()
        meta.append([L, cs, ov, stride])
    out["cases"] = np.array(meta)

    # batchify / unbatchify keys (SURVEY.md Appendix A)
    items = [(f"r{j}", torch.arange(n * 3, dtype=torch.float32).reshape(n, 3) + 100 * j) for j, n in enumerate([3, 5, 1, 7])]
    batches = list(ref.util.batchify(items, 4))
    out["batchify_keys"] = np.array(json.dumps([[[k, list(se)] for k, se in keys] for keys, _ in batches]))
    out["batchify_sizes"] = np.array([v.shape[0] for _, v in batches])
    rebuilt = list(ref.util.unbatchify(batches))
    out["unbatchify_keys"] = np.array(json.dumps([k for k, _ in rebuilt]))
    out["unbatchify_cat"] = torch.cat([v for _, v in rebuilt]).numpy()

    for k in (3, 4, 5):
        out[f"idx_k{k}"] = ref.crf_model.CTC_CRF(k, ["N", "A", "C", "G", "T"]).idx.numpy()
    np.savez_compressed(os.path.join(OUT, "host_logic.npz"), **out)
    print("host_logic.npz", len(out), "arrays")


def forward_fast(ref):
    torch.manual_seed(25)
    spec = synth.model_spec("fast", n_lstm=2)
    cfg = synth.model_config(spec, batchnorm=True)
    model = ref.crf_model.Model(cfg)
    weights = synth.make_weights(spec, seed=7)
    sd = synth.state_dict_from_weights(spec, weights)
    # non-trivial BatchNorm statistics so that fuse_bn_ matters
    gen = torch.Generator().manual_seed(11)
    full = model.state_dict()
    for k in full:
        if k in sd:
            full[k] = sd[k]
        elif k.endswith("bn.weight"):
            full[k] = 1.0 + 0.2 * torch.randn(full[k].shape, generator=gen)
        elif k.endswith("bn.bias"):
            full[k] = 0.1 * torch.randn(full[k].shape, generator=gen)
        elif k.endswith("running_mean"):
            full[k] = 0.2 * torch.randn(full[k].shape, generator=gen)
        elif k.endswith("running_var"):
            full[k] = 0.5 + torch.rand(full[k].shape, generator=gen)
    model.load_state_dict(full)
    model.eval()
    pre_fusion = {k: v.clone() for k, v in model.state_dict().items()}
    model.apply(ref.nn.fuse_bn_)           # bonito/cli/basecaller.py:61
    assert get_stride_ok(ref, model)
    x = synth.squiggle(3, 1500, seed=5)
    with torch.inference_mode():
        scores, feats = model.encoder(x, return_features=True)
        strings = model.decode_batch(scores)
    out = {"x": x.numpy(), "scores": scores.numpy(), "strings": np.array(json.dumps(strings)),
           "config": np.array(json.dumps(cfg)), "stride": np.array(model.stride)}
    for i, f in enumerate(feats):
        if i in (1, 2, 4, 5):  # conv1 (stem output), conv2, lstm0, lstm1; the head is `scores`
            out[f"feat_{i}"] = f.numpy()
    def compact(a):  # exactly fp16-representable tensors are stored as fp16
        h = a.astype(np.float16)
        return h if np.array_equal(h.astype(a.dtype), a) else a
    for k, v in pre_fusion.items():
        if "num_batches_tracked" not in k:
            out["pre." + k] = compact(v.numpy())
    for k, v in model.state_dict().items():
        if ".conv." in k:  # only the convolutions change under fuse_bn_
            out["fused." + k] = v.numpy()
    sample_last_axis(out, ["scores", "feat_1", "feat_2", "feat_4", "feat_5"], 1 / 6)   # the parameters take half the budget
    np.savez_compressed(os.path.join(OUT, "forward_fast.npz"), **out)
    print("forward_fast.npz scores", tuple(scores.shape), "strings", [len(s) for s in strings])


def forward_sup(ref):
    """Narrow transformer (d_model 64, 2 heads, 2 layers) through the reference's own transformer package."""
    tm = reference_shim.load_transformer()
    spec = synth.sup_spec(depth=2, d_model=64, nhead=2, dim_feedforward=128, state_len=3)
    spec["convs"] = [(1, 8, 5, 1, 2, "swish"), (8, 8, 5, 1, 2, "swish"), (8, 16, 9, 3, 4, "swish"),
                     (16, 16, 9, 2, 4, "swish"), (16, 64, 5, 2, 2, "swish")]
    cfg = synth.sup_config(spec)
    torch.manual_seed(25)
    model = tm.Model(cfg)
    weights = synth.make_sup_weights(spec, seed=9)
    missing, unexpected = model.load_state_dict(synth.sup_state_dict(spec, weights), strict=False)
    assert not unexpected and all("rotary" in k or "inv_freq" in k for k in missing), (missing, unexpected)
    model.eval()
    x = synth.squiggle(2, 1200, seed=6)
    with torch.inference_mode():
        scores = model(x)                                   # [2T', N, C + blanks]
        conv = model.encoder.conv(x)                        # [N, T', d]
        layer0 = model.encoder.transformer_encoder[0](conv)
    out = {"x": x.numpy(), "scores": scores.numpy(), "conv": conv.numpy(), "layer0": layer0.numpy(),
           "spec": np.array(json.dumps({k: v for k, v in spec.items()})), "stride": np.array(model.stride)}
    for k, v in weights.items():
        out["w." + k] = v.numpy().astype(np.float16)
    np.savez_compressed(os.path.join(OUT, "forward_sup.npz"), **out)
    print("forward_sup.npz scores", tuple(scores.shape))


def weights_digest(weights):
    """sha256 over the fp16 bytes of every tensor (sorted by name): the fixture stores it instead of 12 MB of weights."""
    import hashlib
    h = hashlib.sha256()
    for k in sorted(weights):
        h.update(k.encode())
        h.update(weights[k].numpy().astype(np.float16).tobytes())
    return h.hexdigest()


def forward_hac(ref):
    """The headline shape (H = 384, 5 LSTM layers, 1024 scores) through the reference's module tree, fp32 on CPU.
    Weights are `synth.make_weights(spec, seed=31)`: regenerated by the tests and compared by digest (the QR inside the
    orthogonal init may round differently on another CPU; the tests then skip rather than compare apples with pears)."""
    spec = synth.model_spec("hac")
    cfg = synth.model_config(spec, batchnorm=False)
    model = ref.crf_model.Model(cfg)
    weights = synth.make_weights(spec, seed=31)
    model.load_state_dict(synth.state_dict_from_weights(spec, weights))
    model.eval()
    x = synth.squiggle(2, 1200, seed=12).half().float()     # fp16-representable input: identical for every implementation
    with torch.inference_mode():
        scores = model.encoder(x)                            # [T, N, C + blanks]
        strings = model.decode_batch(scores)
    t, n, _ = scores.shape
    s4 = scores.reshape(t, n, -1, 5)
    assert torch.all(s4[..., 0] == 2.0)
    ntc = s4[..., 1:].reshape(t, n, -1).permute(1, 0, 2).contiguous()
    out = {"x": x.numpy().astype(np.float16), "scores_ntc": ntc.numpy(), "strings": np.array(json.dumps(strings)),
           "digest": np.array(weights_digest(weights)), "seed": np.array(31), "stride": np.array(model.stride)}
    sample_last_axis(out, ["scores_ntc"], 1 / 2)
    np.savez_compressed(os.path.join(OUT, "forward_hac.npz"), **out)
    print("forward_hac.npz scores", tuple(ntc.shape), "strings", [len(s) for s in strings], "max|s|", float(ntc.abs().max()))


def revcomp(ref):
    """CTC_CRF.reverse_complement (bonito/crf/model.py:84-96) of the reference on small random blank-expanded scores."""
    out = {}
    gen = torch.Generator().manual_seed(3)
    for k, (T, N) in ((3, (7, 2)), (4, (5, 3)), (5, (3, 1))):
        sd = ref.crf_model.CTC_CRF(k, ["N", "A", "C", "G", "T"])
        scores = torch.randn(T, N, sd.n_score(), generator=gen)
        out[f"in_k{k}"] = scores.numpy()
        out[f"out_k{k}"] = sd.reverse_complement(scores).numpy()
    np.savez_compressed(os.path.join(OUT, "revcomp.npz"), **out)
    print("revcomp.npz", {k: v.shape for k, v in out.items()})


def forward_sup_wide(ref):
    """The sup v5 width (d_model 512, 8 heads of 64, feed-forward 2048, the full 5-convolution stack, k = 5: 4096 scores per
    frame), 6 layers, through the reference's own transformer classes in fp32 on the CPU.  The 24 M seeded weights are
    regenerated by the tests (`synth.make_sup_weights(spec, seed=11)`, plain torch.randn draws) and checked by digest."""
    tm = reference_shim.load_transformer()
    spec = synth.sup_spec(depth=6)
    cfg = synth.sup_config(spec)
    torch.manual_seed(25)
    model = tm.Model(cfg)
    weights = synth.make_sup_weights(spec, seed=11)
    missing, unexpected = model.load_state_dict(synth.sup_state_dict(spec, weights), strict=False)
    assert not unexpected and all("rotary" in k or "inv_freq" in k for k in missing), (missing, unexpected)
    model.eval()
    x = synth.squiggle(2, 600, seed=16).half().float()      # fp16-representable input
    with torch.inference_mode():
        scores = model(x)                                   # [2T', N, C + blanks]
        conv = model.encoder.conv(x)                        # [N, T', d]
        h, layers = conv, []
        for layer in model.encoder.transformer_encoder:
            h = layer(h)
            layers.append(h)
    t, n, _ = scores.shape
    s5 = scores.reshape(t, n, -1, 5)
    assert torch.all(s5[..., 0] == 2.0)
    ntc = s5[..., 1:].reshape(t, n, -1).permute(1, 0, 2).contiguous()
    out = {"x": x.numpy().astype(np.float16), "scores_ntc": ntc.numpy(), "conv": conv.numpy(),
           "layer0": layers[0].numpy(), "layer5": layers[5].numpy(), "digest": np.array(weights_digest(weights)),
           "seed": np.array(11), "depth": np.array(6), "stride": np.array(model.stride)}
    sample_last_axis(out, ["scores_ntc", "conv", "layer0", "layer5"], 1 / 5)
    np.savez_compressed(os.path.join(OUT, "forward_sup_wide.npz"), **out)
    print("forward_sup_wide.npz scores", tuple(ntc.shape), "std %.2f max %.1f" % (float(ntc.std()), float(ntc.abs().max())))


def get_stride_ok(ref, model):
    return ref.crf_model.get_stride(model.encoder) == 6 and model.stride == 6


def main(names=None):
    """`python -m oracle.make_golden [name ...]`: all fixtures, or only the named ones."""
    os.makedirs(OUT, exist_ok=True)
    ref = reference_shim.load()
    makers = dict(host_logic=host_logic, forward_fast=forward_fast, forward_sup=forward_sup, forward_hac=forward_hac,
                  revcomp=revcomp, forward_sup_wide=forward_sup_wide)
    for name in (names or list(makers)):
        makers[name](ref)


if __name__ == "__main__":
    import sys
    main(sys.argv[1:])
