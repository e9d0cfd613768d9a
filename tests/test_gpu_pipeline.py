"""GPU parity tests of the whole chunked forward + decode path against the CPU oracle."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import crf_oracle as O
from oracle import synth

pytestmark = pytest.mark.gpu


def _model(name, n_lstm=5, seed=25, batchnorm=False):
    from bonito_b200.crf.model import Model
    spec = synth.model_spec(name, n_lstm=n_lstm)
    weights = synth.make_weights(spec, seed=seed)
    model = Model(synth.model_config(spec, batchnorm=batchnorm))
    model.load_state_dict(synth.state_dict_from_weights(spec, weights), strict=not batchnorm)
    model.use_koi(batchsize=32, chunksize=1998, quantize=False)
    return model.half().eval().to("cuda"), spec, weights


# Tolerances.  BASELINE.json asks for "1e-3 fp16 tolerance": fp16 carries 11 significant bits, so one ulp of a score
# of magnitude 4..8 is 3.9e-3 and 1e-3 is a RELATIVE bound (~1 ulp).  Against the oracle run with the same fp16
# storage rounding points the engine must stay within a few ulp (accumulation order differs); against the pure
# fp32 oracle the bound is what half-precision storage of 7 stacked layers costs any implementation.
TOL_FP16_MAX, TOL_FP16_MEAN = 8.0e-3, 6.0e-4       # measured 3.9e-3 / 3.5e-4 (one fp16 ulp at |x| in [4, 8))
TOL_FP32_MAX, TOL_FP32_MEAN = 6.0e-2, 3.0e-3


@pytest.mark.parametrize("name,n,L", [("fast", 5, 1998), ("fast", 33, 600), ("hac", 6, 1998), ("hac", 35, 996)])
def test_forward_scores_match_oracle(name, n, L):
    model, spec, weights = _model(name)
    x = synth.squiggle(n, L, seed=n).half()
    with torch.inference_mode():
        scores, feats = model.native_plan("cuda").forward(x.cuda(), return_features=True)
    torch.cuda.synchronize()
    for fp16, tol_max, tol_mean in ((True, TOL_FP16_MAX, TOL_FP16_MEAN), (False, TOL_FP32_MAX, TOL_FP32_MEAN)):
        with torch.no_grad():
            ref, rfeats = O.lstm_crf_forward(weights, spec, x.float(), return_features=True, fp16=fp16)
        errs = {"stem": (feats["stem"].float().cpu().permute(0, 2, 1) - rfeats["conv1"]).abs().max().item(),
                "conv": (feats["conv"].float().cpu() - rfeats["conv2"].permute(2, 0, 1)).abs().max().item()}
        for i in range(spec["n_lstm"]):
            errs[f"lstm{i}"] = (feats[f"lstm{i}"].float().cpu() - rfeats[f"lstm{i}"]).abs().max().item()
        err = (scores.float().cpu() - ref.permute(1, 0, 2)).abs()
        errs["scores_max"] = err.max().item()
        errs["scores_mean"] = err.mean().item()
        errs["scores_rel_1e-3"] = (err <= 1e-3 * ref.permute(1, 0, 2).abs().clamp(min=1.0) + 1e-3).float().mean().item()
        print(name, n, L, "oracle-fp16" if fp16 else "oracle-fp32", {k: f"{v:.2e}" for k, v in errs.items()})
        assert scores.shape == (n, ref.shape[0], 4 ** (spec["state_len"] + 1))
        assert errs["scores_max"] <= tol_max, errs
        assert errs["scores_mean"] <= tol_mean, errs


@pytest.mark.parametrize("n", [33, 70, 128])
def test_tile_pipelined_forward_is_bit_identical(n, monkeypatch):
    """Per-tile streams (the default for batches above one tile) vs the single-stream layer-by-layer schedule, and the
    second-generation recurrent kernel (48-chunk tiles, default) vs the first (32-chunk tiles, B200_LSTM_TILE=0)."""
    model, spec, _ = _model("hac", n_lstm=3)
    x = synth.squiggle(n, 1200, seed=n).half().cuda()
    plan = model.native_plan("cuda")
    with torch.inference_mode():
        a = plan.forward(x, tiled=False).clone()
        b = plan.forward(x, tiled=True).clone()
        c = plan.forward(x).clone()
        monkeypatch.setenv("B200_COARSE_FWD", "0")       # the same launches one ctypes call at a time
        f = plan.forward(x, tiled=False).clone()
        monkeypatch.setenv("B200_LSTM_TILE", "0")
        d = plan.forward(x, tiled=False).clone()
        e = plan.forward(x, tiled=True).clone()
    torch.cuda.synchronize()
    assert torch.equal(a, b) and torch.equal(a, c)       # a, c: the whole encoder from one C call (b200_lstm_crf_fwd)
    assert torch.equal(a, f)
    assert torch.equal(d, e) and torch.equal(a, d)


def test_gemm_paths_agree_end_to_end():
    from bonito_b200 import native
    model, spec, _ = _model("hac", n_lstm=2)
    x = synth.squiggle(4, 1200, seed=3).half().cuda()
    plan = model.native_plan("cuda")
    with torch.inference_mode():
        a = plan.forward(x, gemm_impl=native.GEMM_TCGEN05).clone()
        b = plan.forward(x, gemm_impl=native.GEMM_MMA_SYNC).clone()
    assert (a.float() - b.float()).abs().max().item() <= 2e-2


def test_identical_sequences_and_basecall_pipeline():
    """basecall() over synthetic reads == oracle forward + oracle decode + reference-style stitching."""
    from _helpers import identity
    from bonito_b200.crf.basecall import basecall, stitch_results
    from bonito_b200.util import chunk

    model, spec, weights = _model("fast", n_lstm=3, seed=4)
    model.config["qscore"] = {"scale": 1.05, "bias": 0.2}

    class Read:
        def __init__(self, rid, sig):
            self.read_id, self.signal = rid, sig

    lengths = [5000, 1200, 3996, 9000]  # multi-chunk, short (tiled), exactly one chunk, stubbed
    reads = [Read(f"r{i}", synth.squiggle(1, n, seed=10 + i)[0, 0].numpy()) for i, n in enumerate(lengths)]
    cs, ov = 1998, 120
    got = {r.read_id: res for r, res in basecall(model, reads, chunksize=cs, overlap=ov, batchsize=4,
                                                 qscore_calibration=True)}
    plain = {r.read_id: res for r, res in basecall(model, reads, chunksize=cs, overlap=ov, batchsize=4)}
    for read in reads:
        chunks = chunk(torch.from_numpy(read.signal), cs, ov).half()
        with torch.no_grad():
            s = O.lstm_crf_forward(weights, spec, chunks.float())
        ntc = s.permute(1, 0, 2).half().float().numpy()
        moves, seq, qual, _ = O.decode_native(ntc, spec["state_len"], 2.0, 1.05, 0.2)
        attrs = {"moves": torch.from_numpy(moves), "sequence": torch.from_numpy(seq), "qstring": torch.from_numpy(qual)}
        st = stitch_results(attrs, len(read.signal), cs, ov, 6)
        want = st["sequence"].numpy()
        want = want[want != 0].tobytes().decode()
        res = got[read.read_id]
        assert res["stride"] == 6 and len(res["moves"]) == len(st["moves"])
        # fp16-vs-fp32 forward differences may flip an occasional near-tie: demand >= 99% identity, report it
        same = identity(res["sequence"], want)
        print(read.read_id, len(want), len(res["sequence"]), f"identity (edit distance) {same:.4f}")
        assert len(res["qstring"]) == len(res["sequence"]) == int(res["moves"].sum())
        assert same >= 0.99, (read.read_id, same)
        # default = the reference's behaviour: scale 1.0 / offset 0.0, same bases, different quality string
        assert plain[read.read_id]["sequence"] == res["sequence"]
        moves1, seq1, qual1, _ = O.decode_native(ntc, spec["state_len"], 2.0, 1.0, 0.0)
        st1 = stitch_results({"qstring": torch.from_numpy(qual1)}, len(read.signal), cs, ov, 6)["qstring"].numpy()
        want_q = st1[st1 != 0].tobytes().decode()
        if res["sequence"] == want:
            dq = [abs(ord(a) - ord(b)) for a, b in zip(plain[read.read_id]["qstring"], want_q)]
            assert max(dq) <= 1 and sum(d != 0 for d in dq) <= 0.02 * len(dq)


def test_decode_of_own_scores_is_exact():
    """Same fp16 scores into the oracle decoder and the kernel -> identical base sequences."""
    from bonito_b200.decode import beam_search
    model, spec, _ = _model("hac", n_lstm=5)
    x = synth.squiggle(6, 3996, seed=8).half().cuda()
    with torch.inference_mode():
        scores = model(x)
        seq, qstring, moves = beam_search(scores, scale=1.05, offset=0.2)
    o_moves, o_seq, o_q, _ = O.decode_native(scores.float().cpu().numpy(), 4, 2.0, 1.05, 0.2)
    got = [r[r != 0].tobytes() for r in seq.numpy()]
    want = [r[r != 0].tobytes() for r in o_seq]
    assert got == want                                   # identical base sequences
    # Where a base is emitted may legitimately differ by one frame when "move now, stay next" and "stay now,
    # move next" have log-posterior sums equal to fp32 rounding (the kernel uses ex2/lg2 intrinsics, the oracle
    # float64 libm): allow isolated one-frame shifts, nothing else.
    diff = np.argwhere(moves.numpy() != o_moves)
    print("frames with a shifted move:", len(diff), "of", o_moves.size)
    assert len(diff) <= 0.005 * o_moves.size and len(diff) % 2 == 0
    for (n0, t0), (n1, t1) in zip(diff[0::2], diff[1::2]):
        assert n0 == n1 and t1 == t0 + 1
    lens = [len(w) for w in want]
    assert min(lens) > 100 and len(set(want)) == 6


def test_headline_shape_scores_and_sequences_match_oracle():
    """
    BASELINE config 2 at full size: hac, batch 512 x 9996 samples (T = 1666), 64 distinct chunks repeated 8 times.
    16 chunks spread over the batch (different tiles, different copies) are compared with the CPU oracle run with the
    same fp16 storage rounding: scores within fp16 tolerance (north star: 1e-3 relative; one fp16 ulp at |x| in [4, 8)
    is 3.9e-3, the budget is two), and the base sequences of CUDA forward + CUDA decode against oracle forward + oracle
    decode by edit distance.
    """
    from _helpers import edit_distance
    from bonito_b200.decode import beam_search, to_str
    from oracle import build_ref
    model, spec, weights = _model("hac")
    x64 = synth.squiggle(64, 9996, seed=7).half()
    x = x64.repeat(8, 1, 1)
    with torch.inference_mode():
        scores = model(x.cuda())
        seq, qstring, moves = beam_search(scores, scale=1.05, offset=0.2)
    assert scores.shape == (512, 1666, 1024)
    picks = [0, 37, 63, 64 + 5, 128 + 31, 128 + 32, 192 + 47, 256 + 48, 300, 333, 383, 400, 449, 480, 500, 511]
    with torch.no_grad():
        ref = O.lstm_crf_forward(weights, spec, x[picks].float(), fp16=True).permute(1, 0, 2).contiguous()
    got = scores[picks].float().cpu()
    err = (got - ref).abs()
    within = (err <= 1e-3 * ref.abs().clamp(min=1.0) + 1e-3).float().mean().item()
    print(f"headline shape vs fp16-rounding oracle: max {err.max().item():.2e} mean {err.mean().item():.2e} "
          f"within 1e-3 rel: {within:.5f}")
    assert err.max().item() <= 8e-3, err.max().item()
    assert err.mean().item() <= 6e-4, err.mean().item()
    assert within >= 0.999, within
    # (1) the decoder at full length on real scores: the oracle decoder fed the CUDA scores gives the CUDA sequences exactly
    c_moves, c_seq, c_q = build_ref.decode(got.numpy(), spec["state_len"], 2.0, 1.05, 0.2)
    for k, i in enumerate(picks):
        assert to_str(seq[i]) == c_seq[k][c_seq[k] != 0].tobytes().decode(), i
    # (2) end to end: oracle forward + oracle decode against CUDA forward + CUDA decode.  The two forwards differ by at most
    # one fp16 ulp in 0.003 % of the scores; where the posterior is flat (synthetic random weights have such stretches) that
    # is enough to move a few calls, so identity is asserted by edit distance and the exact-match count is reported.
    o_moves, o_seq, o_q = build_ref.decode(ref.numpy(), spec["state_len"], 2.0, 1.05, 0.2)
    total = dist = exact = 0
    for k, i in enumerate(picks):
        a, b = to_str(seq[i]), o_seq[k][o_seq[k] != 0].tobytes().decode()
        d = edit_distance(a, b)
        dist, total, exact = dist + d, total + len(b), exact + (d == 0)
        assert len(b) > 500 and d <= 0.03 * len(b), (i, d, len(b))
    print(f"sequences: {exact}/{len(picks)} chunks identical, edit distance {dist} over {total} bases "
          f"(identity {1 - dist / total:.5f})")
    assert dist <= 1e-2 * total and exact >= len(picks) // 2, (dist, total, exact)
    # the copies of a chunk decode identically wherever they sit in the batch
    assert torch.equal(seq[:64], seq[448:]) and torch.equal(moves[:64], moves[64:128])


def test_full_size_properties():
    """BASELINE config 2 (hac, batch 512, 9996 samples): determinism and chunk independence."""
    from bonito_b200.decode import beam_search
    model, spec, _ = _model("hac")
    x = synth.squiggle(64, 9996, seed=1).half()
    x = x.repeat(8, 1, 1).cuda()            # 512 chunks, 8 copies of 64 distinct ones
    with torch.inference_mode():
        s1 = model(x).clone()
        s2 = model(x).clone()
        assert torch.equal(s1, s2)          # run-to-run bitwise determinism
        assert s1.shape == (512, 1666, 1024)
        for r in range(1, 8):               # a chunk's scores do not depend on where it sits in the batch
            assert torch.equal(s1[:64], s1[64 * r:64 * (r + 1)])
        small = model(x[:40]).clone()       # ... nor on the batch size
        assert torch.equal(small, s1[:40])
        seq, q, moves = beam_search(s1)
    assert torch.equal(seq[:64], seq[448:]) and int(moves.sum()) > 512 * 300
    assert float((s1.float().abs() >= 5).float().mean()) < 0.05


def test_cli_basecaller_end_to_end(tmp_path):
    """`python -m bonito_b200 basecaller <model dir> <reads dir>` on synthetic .npy reads -> FASTQ on stdout."""
    import os, subprocess, sys
    from bonito_b200.crf.basecall import basecall
    from bonito_b200.nn import fuse_bn_
    from bonito_b200.reader import Reader
    from bonito_b200.util import load_model
    spec = synth.model_spec("fast", n_lstm=3)
    weights = synth.make_weights(spec, seed=4)
    mdir = synth.write_model_dir(str(tmp_path / "model"), spec, weights, batchsize=8, chunksize=2000, overlap=120)
    rdir = tmp_path / "reads"
    rdir.mkdir()
    for i, n in enumerate([5000, 1500, 7777]):
        np.save(rdir / f"read{i}.npy", 93.7 + 23.5 * synth.squiggle(1, n, seed=20 + i)[0, 0].numpy())   # picoamperes
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "bonito_b200", "basecaller", mdir, str(rdir), "--no-trim"], cwd=root,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "> samples per second" in out.stderr and "> completed reads: 3" in out.stderr, out.stderr[-1500:]
    lines = out.stdout.strip().split("\n")
    records = {lines[i][1:]: (lines[i + 1], lines[i + 3]) for i in range(0, len(lines), 4)}
    assert sorted(records) == ["read0", "read1", "read2"]
    model = load_model(mdir, "cuda", use_koi=True).apply(fuse_bn_)
    reads = Reader(str(rdir)).get_reads(str(rdir), do_trim=False, scaling_strategy=model.config["scaling"],
                                        norm_params=model.config["standardisation"])
    p = model.config["basecaller"]
    for read, res in basecall(model, reads, batchsize=p["batchsize"], chunksize=p["chunksize"], overlap=p["overlap"]):
        assert records[read.read_id] == (res["sequence"], res["qstring"]) and len(res["sequence"]) > 50


def test_score_batches_equals_compute_scores():
    """The pipelined generator basecall() runs == one synchronous compute_scores per batch: same bytes, same order, ragged
    last batch, chunk length that is not a multiple of the stride, empty input."""
    from bonito_b200.crf.basecall import compute_scores, score_batches
    model, spec, weights = _model("fast", n_lstm=3, seed=4)
    sizes = [(5, 1998), (5, 1998), (5, 1998), (3, 1998), (2, 4000), (5, 1998)]
    batches = [(f"k{i}", synth.squiggle(n, L, seed=20 + i)) for i, (n, L) in enumerate(sizes)]
    got = list(score_batches(model, iter(batches), scale=1.05, offset=0.2))
    assert [k for k, _ in got] == [k for k, _ in batches]
    for (key, batch), (_, res) in zip(batches, got):
        want = compute_scores(model, batch, scale=1.05, offset=0.2)
        for name in ("moves", "sequence", "qstring"):
            assert res[name].shape == want[name].shape and res[name].dtype == torch.uint8
            assert torch.equal(res[name], want[name]), (key, name)
        assert int(res["moves"].sum()) > 10
    assert list(score_batches(model, iter([]))) == []


def test_headline_shape_against_the_reference_fixture(golden_dir):
    """hac shape through the native engine vs scores produced by the reference's own module tree (fp32 CPU,
    tests/golden/forward_hac.npz, a sample of its score columns): fp16 tolerance on the scores, same base sequences."""
    from _helpers import at_sample, identity
    from oracle.make_golden import weights_digest
    from bonito_b200.crf.model import Model
    from bonito_b200.decode import beam_search, to_str
    gold = np.load(os.path.join(golden_dir, "forward_hac.npz"))
    spec = synth.model_spec("hac")
    weights = synth.make_weights(spec, seed=int(gold["seed"]))
    if weights_digest(weights) != str(gold["digest"]):
        pytest.skip("seeded hac weights round differently on this CPU: fixture not comparable")
    model = Model(synth.model_config(spec, batchsize=8, chunksize=1200, overlap=0))
    model.load_state_dict(synth.state_dict_from_weights(spec, weights))
    model.use_koi(batchsize=8, chunksize=1200, quantize=False)
    model = model.half().eval().cuda()
    x = torch.from_numpy(gold["x"].astype(np.float16)).cuda()
    with torch.inference_mode():
        scores = model(x)
        seq, _, _ = beam_search(scores)
    assert scores.shape == (2, 200, 1024)
    ref = torch.from_numpy(gold["scores_ntc"])
    err = (torch.from_numpy(at_sample(scores.float().cpu(), gold, "scores_ntc")) - ref).abs()
    print("vs reference fixture: max", err.max().item(), "mean", err.mean().item())
    assert err.max().item() <= 2e-2 and err.mean().item() <= 2e-3
    want = json.loads(str(gold["strings"]))
    for got, w in zip([to_str(r) for r in seq], want):
        same = identity(got, w)
        assert same >= 0.99, (len(got), len(w), same)


def test_reverse_complement_on_the_native_layout():
    """--revcomp (bonito/crf/basecall.py:35, bonito/crf/model.py:84-96): the native-layout helper equals the reference
    definition on the blank-expanded [T, N, C] layout (pinned on the CPU against tests/golden/revcomp.npz), and basecalling
    the reverse-complemented scores yields the reverse complement of the sequence."""
    from _helpers import identity
    from bonito_b200.crf.basecall import _revcomp_native, compute_scores
    from bonito_b200.decode import to_str
    model, spec, _ = _model("hac", n_lstm=2)
    g = torch.Generator().manual_seed(12)
    scores = (torch.randn(3, 50, 1024, generator=g) * 1.7).clamp(-5, 5).half()
    got = _revcomp_native(model, scores.cuda(), 2.0).cpu()
    full = torch.nn.functional.pad(scores.permute(1, 0, 2).reshape(50, 3, 256, 4), (1, 0), value=2.0).reshape(50, 3, -1)
    want = model.seqdist.reverse_complement(full).reshape(50, 3, 256, 5)[..., 1:].reshape(50, 3, 1024).permute(1, 0, 2)
    assert torch.equal(got, want)
    assert torch.equal(_revcomp_native(model, got.cuda(), 2.0).cpu(), scores)

    x = synth.squiggle(5, 3996, seed=31)
    fwd = compute_scores(model, x)
    rev = compute_scores(model, x, reverse=True)
    comp = str.maketrans("ACGT", "TGCA")
    exact = 0
    for a, b in zip(fwd["sequence"], rev["sequence"]):
        sa, sb = to_str(a), to_str(b)
        assert len(sa) > 200
        same = identity(sa[::-1].translate(comp), sb)
        exact += same == 1.0
        # not exactly 1: scores saturated at the +-5 clamp produce exact ties between paths, and the tie-break (lowest
        # in-edge, lowest state) is not symmetric under reverse complement
        assert same >= 0.97, same
    print("reverse-complement basecalls identical to the reverse complement of the forward basecall:", exact, "of 5")


def test_quantized_input_projection_stays_close_to_fp16():
    """--quantize: int8 input projections (per-row weight scale, activations x127).  Its own parity budget: the scores of the
    quantised model against the fp16 model of the same weights, and the base sequences of both by edit distance."""
    from _helpers import identity
    from bonito_b200.crf.model import Model
    from bonito_b200.decode import beam_search, to_str
    spec = synth.model_spec("hac")
    weights = synth.make_weights(spec, seed=25)
    x = synth.squiggle(50, 3996, seed=11).half().cuda()
    out = {}
    for q in (False, True):
        model = Model(synth.model_config(spec))
        model.load_state_dict(synth.state_dict_from_weights(spec, weights))
        model.use_koi(batchsize=50, chunksize=3996, quantize=q)
        model = model.half().eval().cuda()
        with torch.inference_mode():
            scores = model(x)
            seq, _, _ = beam_search(scores)
        out[q] = (scores.float().cpu(), [to_str(r) for r in seq])
    err = (out[True][0] - out[False][0]).abs()
    ids = [identity(a, b) for a, b in zip(out[True][1], out[False][1])]
    print(f"int8 input projection vs fp16: scores max {err.max().item():.3f} mean {err.mean().item():.4f}; "
          f"sequence identity mean {sum(ids) / len(ids):.4f} min {min(ids):.4f}")
    assert err.mean().item() <= 0.08 and err.max().item() <= 3.0, (err.mean().item(), err.max().item())
    assert sum(ids) / len(ids) >= 0.95 and min(ids) >= 0.85


@pytest.mark.parametrize("name,n,L", [("hac", 6, 1998), ("fast", 5, 1998)])
def test_old_style_crf_head_tanh_and_scale(name, n, L):
    """LinearCRFEncoder(activation="tanh", scale=5.0) without a Clamp layer (the dna_r9.4.1-era configs, bonito/nn.py:283-298):
    the tanh -> fp16 -> x scale -> fp16 epilogue of the CRF GEMM against the oracle with the same rounding points, and the
    decode of those scores."""
    from bonito_b200.crf.model import Model
    from bonito_b200.decode import beam_search
    spec = dict(synth.model_spec(name), clamp=None, crf_activation="tanh", crf_scale=5.0)
    weights = synth.make_weights(spec, seed=31)
    model = Model(synth.model_config(spec))
    model.load_state_dict(synth.state_dict_from_weights(spec, weights))
    model.use_koi(batchsize=32, chunksize=L, quantize=False)
    model = model.half().eval().to("cuda")
    x = synth.squiggle(n, L, seed=n + 1).half()
    with torch.inference_mode():
        scores = model(x.cuda())
        seqs, _, moves = beam_search(scores)
    with torch.no_grad():
        ref = O.lstm_crf_forward(weights, spec, x.float(), fp16=True).permute(1, 0, 2)
    got = scores.float().cpu()
    err = (got - ref).abs()
    print(f"tanh + scale head ({name}): max |err| {err.max().item():.2e} mean {err.mean().item():.2e}, |scores| max {ref.abs().max().item():.2f}")
    assert got.abs().max().item() <= 5.0 + 1e-6
    # one fp16 ulp of the pre-activation (2e-3 at |x| in [2, 4)) times the slope of tanh times 5, plus the output rounding
    assert err.max().item() <= 2.5e-2 and err.mean().item() <= 1.5e-3, (err.max().item(), err.mean().item())
    _, o_seq, _, _ = O.decode_native(got.numpy(), spec["state_len"], spec["blank_score"])
    assert [r[r != 0].tobytes() for r in seqs.cpu().numpy()] == [r[r != 0].tobytes() for r in o_seq]     # identical base sequences
