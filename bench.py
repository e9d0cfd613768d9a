#!/usr/bin/env python
"""
bench.py -- raw-signal samples/sec basecalled (forward + decode) on synthetic chunks.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload all|hac|sup] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload (BASELINE.json configs[1], the one the metric is quoted on): hac-shaped LSTM-CRF (H=384, 5-mer scores,
seeded random weights -- the real checkpoint needs the network), batch 512 chunks per GPU, 10 000-sample chunks trimmed
to a stride multiple (9996) exactly as `_load_model(use_koi=True)` does (bonito/util.py:288-291).  A step = one batch
through conv stem -> strided conv GEMM -> 5 x (input GEMM + persistent LSTM) -> CRF linear + clamp -> CRF decode.

  value  whole-job samples/s with the batch already resident in HBM (CUDA events, max over ranks)
  e2e    the same through the reference-facing generator `score_batches(model, host float32 batches)` (the loop
         `basecall()` runs): fp16 staging in pinned memory, H2D, forward, decode, D2H of moves/sequence/qstring inside
         the timed region
  roofline / stages: per-kernel CUDA-event durations recorded inside the timed region

`configs` (workload "all", the default) adds the other BASELINE.json configurations to the same JSON line:
  config3_sup        sup-shaped transformer (18 layers, d_model 512, k = 5), batch 256/GPU, 9996-sample chunks
  config5_sup_sweep  the same at chunk lengths 3996 / 7992 / 12000 (multiples of 12, SURVEY.md H6), batch 256/GPU
  config1_fast_cpu   fast-shaped LSTM-CRF, batch 8 x 4000 samples, the reference's PyTorch-CPU path on the host cores
(config 4 is this script under torchrun: the driver runs N = 1, 2, 4, 8.)

Multi-GPU: chunks shard by batch (one process per GPU, weights broadcast once over NCCL, no steady-state collective)
=> weak scaling.
--impl reference: the reference's PyTorch-CPU execution of the headline path (oracle/cpu_reference.py) on all host cores,
a bounded sample of the workload per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# The engine drives one CUDA stream per tile (11 + 11 at batch 512).  With the default of 8 hardware work queues, streams
# that share a queue serialise behind each other's not-yet-dispatched cluster launches; set before the CUDA context exists.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark leaves the tree it runs from as it found it (it may be read-only)

METRIC = "raw-signal samples/sec basecalled (forward+decode), 10k-sample chunks, hac-shaped LSTM-CRF"
CHUNK = 10000
BATCH = 512
SUP_BATCH = 256
SUP_SWEEP = (3996, 7992, 12000)


def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return dict(hbm=p["hbm_gbs"], tflops=p["bf16_tflops_sustained"], tflops_burst=p["bf16_tflops"], source="measured")
    except Exception:
        return dict(hbm=6650.0, tflops=1400.0, tflops_burst=1590.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.t_begin = self.t_end = None

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for stamp, r in self.rows:
            if self.t_begin is not None and not (self.t_begin <= stamp <= (self.t_end or stamp) + 0.06):
                continue   # only samples taken while the timed region ran
            try:
                pw.append(float(r[2]))
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, flag in zip(names, r[3:7]):
                    if flag.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "sm_mhz_min": sm[0] if sm else None, "power_w_max": max(pw) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------
# models
# ---------------------------------------------------------------------------------------------------------------
def build_hac(device, rank, world, name="hac", batch=BATCH, chunk=CHUNK, quantize=False):
    from bonito_b200.crf.model import Model
    from bonito_b200 import synth
    spec = synth.model_spec(name)
    weights = synth.make_weights(spec, seed=25)
    cfg = synth.model_config(spec, batchsize=batch, chunksize=chunk, overlap=500)
    model = Model(cfg)
    if rank == 0:
        model.load_state_dict(synth.state_dict_from_weights(spec, weights))
    chunksize = chunk - chunk % model.stride
    model.use_koi(batchsize=batch, chunksize=chunksize, quantize=quantize)
    model = model.half().eval().to(device)
    if world > 1:  # the one collective of the path: weights from rank 0 (NCCL over NVLink)
        from bonito_b200.distributed import broadcast_parameters
        broadcast_parameters(model, src=0)
    return model, spec, weights, chunksize


def build_sup(device, rank, world, batch=SUP_BATCH):
    from bonito_b200 import synth
    from bonito_b200.transformer import Model
    spec = synth.sup_spec(depth=18)
    model = Model(synth.sup_config(spec, batchsize=batch))
    if rank == 0:
        model.load_state_dict(synth.sup_state_dict(spec, synth.make_sup_weights(spec, seed=25)))
    model.use_koi(batchsize=batch, chunksize=9996, quantize=False)
    model = model.half().eval().to(device)
    if world > 1:
        from bonito_b200.distributed import broadcast_parameters
        broadcast_parameters(model, src=0)
    return model, spec


# ---------------------------------------------------------------------------------------------------------------
# timing helpers
# ---------------------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, args, rank, local_rank, world, device):
        self.args, self.rank, self.local_rank, self.world, self.device = args, rank, local_rank, world, device

    def barrier(self):
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, values):
        if self.world == 1:
            return list(values)
        import torch.distributed as dist
        t = torch.tensor(list(values), device=self.device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()


N_SLOTS = int(os.environ.get("B200_BENCH_SLOTS", "2"))     # batches in flight in the resident loop (as in score_batches)


def time_resident(ctx, step, steps, warmup, sampler=None, slots=1):
    """
    W untimed + exactly K timed steps, CUDA events on the launch stream, barrier + synchronize on both sides.
    slots > 1: step i is enqueued on stream i % slots with buffer set i % slots (what score_batches does): consecutive
    batches overlap on the device; the timed region still contains exactly K complete steps.
    Returns (elapsed ms, events, host enqueue ms per step, what the last timed step returned).
    """
    main = torch.cuda.current_stream()
    from bonito_b200 import native
    # streams of their own (torch.cuda.Stream() hands out 32 pooled streams round-robin: two of them may be the same stream)
    streams = [native.new_stream(ctx.device) for _ in range(slots)] if slots > 1 else [main]

    def run(i, events):
        if slots == 1:
            return step(events, 0)
        with torch.cuda.stream(streams[i % slots]):
            return step(events, i % slots)

    for i in range(warmup):
        run(i, None)
    ctx.barrier()
    if sampler is not None:
        sampler.mark_begin()
    events = []
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(main)
    for st in streams:
        st.wait_event(t0)
    h0 = time.perf_counter()
    for i in range(steps - 1):
        run(i, events)
    last = run(steps - 1, events)     # only the last step's outputs are kept (the others are released as they are made)
    enqueue_ms = (time.perf_counter() - h0) * 1e3 / steps
    for st in streams:
        main.wait_stream(st)
    t1.record(main)
    ctx.barrier()
    if sampler is not None:
        sampler.mark_end()
    return t0.elapsed_time(t1), events, enqueue_ms, last


def time_e2e(ctx, model, host_batch, steps, qs):
    """The generator basecall() runs, host float32 batches in, host byte arrays out; wall clock around K batches."""
    from bonito_b200.crf.basecall import score_batches
    feed = lambda n: ((i, host_batch) for i in range(n))
    for _ in score_batches(model, feed(2), scale=qs["scale"], offset=qs["bias"]):
        pass
    ctx.barrier()
    t0 = time.perf_counter()
    n_out = 0
    for _, out in score_batches(model, feed(steps), scale=qs["scale"], offset=qs["bias"]):
        n_out += int(out["moves"].shape[0])
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    assert n_out == host_batch.shape[0] * steps
    ctx.barrier()
    return ms


DUMP_BYTES = 64_000_000


def dump_outputs(directory, scores, decoded):
    """
    `--dump-outputs DIR`: what the timed step computed in its last step, as float32 .npy files, so that two builds can be
    compared output for output (the inputs and weights are seeded, so the same arguments give the same inputs):
      moves.npy, sequence.npy, qstring.npy  [N, T] the decoder's outputs (what score_batches hands to basecall())
      scores.npy                            [S, T, C] the scores of S chunks, a fixed seeded sample of the N chunks, as many
                                            as fit in DUMP_BYTES with the rest
      scores_chunks.npy                     [S] which chunks those are
    """
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    arrays = {name: t.cpu().numpy().astype(np.float32) for name, t in zip(("moves", "sequence", "qstring"), decoded)}
    n, t, c = scores.shape
    room = DUMP_BYTES - sum(a.nbytes for a in arrays.values()) - 4 * n - 5 * 4096     # chunk list, .npy headers
    if room < t * c * 4:
        raise SystemExit(f"--dump-outputs: batch {n} leaves no room for the scores of one chunk in {DUMP_BYTES} bytes")
    rows = np.sort(np.random.default_rng(0).choice(n, min(n, room // (t * c * 4)), replace=False))
    arrays["scores"] = scores[torch.from_numpy(rows).to(scores.device)].float().cpu().numpy()
    arrays["scores_chunks"] = rows.astype(np.float32)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)
    log(f"outputs of the last timed step -> {directory}: " + ", ".join(f"{k} {list(a.shape)}" for k, a in arrays.items()))


def stage_table(events, steps):
    per = {}
    for name, a, b in events:
        per.setdefault(name, []).append(a.elapsed_time(b))
    return ({k: sum(v) / steps for k, v in per.items()}, {k: len(v) // steps for k, v in per.items()},
            sum(len(v) for v in per.values()))


# ---------------------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------------------
def bench_hac(ctx, peaks, sampler):
    from bonito_b200 import synth
    from bonito_b200.crf.basecall import compute_scores
    from bonito_b200.decode import _decoder
    args, rank, world, device = ctx.args, ctx.rank, ctx.world, ctx.device
    model, spec, weights, L = build_hac(device, rank, world, batch=args.batch)
    N = args.batch
    host_batch = synth.squiggle(64, L, seed=100 + rank).repeat(N // 64 + 1, 1, 1)[:N].contiguous()  # float32 host
    x_dev = host_batch.to(device, torch.float16)
    log("hac model built")
    plan = model.native_plan(device)
    T = plan.frames(L)
    qs = model.config["qscore"]

    def step(events, slot):
        scores = plan.forward(x_dev, events=events, slot=slot)
        return scores, _decoder(scores, spec["state_len"], blank_score=plan.blank_score, qscale=qs["scale"],
                                qbias=qs["bias"], events=events, slot=slot)

    slots = N_SLOTS if plan.supports_slots else 1
    elapsed_ms, events, enqueue_ms, last = time_resident(ctx, step, args.steps, max(args.warmup, 3), sampler, slots=slots)
    log(f"hac resident: {elapsed_ms / args.steps:.2f} ms/step ({slots} batches in flight)")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    del last
    e2e_ms = time_e2e(ctx, model, host_batch, args.steps, qs)
    for _ in range(2):
        compute_scores(model, host_batch, scale=qs["scale"], offset=qs["bias"])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        compute_scores(model, host_batch, scale=qs["scale"], offset=qs["bias"])
    torch.cuda.synchronize()
    single_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    ctx.barrier()
    log(f"hac e2e: {e2e_ms / args.steps:.2f} ms/step pipelined, {single_ms:.2f} ms/step one synchronous call per batch")
    elapsed_ms, e2e_ms = ctx.max_over_ranks([elapsed_ms, e2e_ms])
    if rank != 0:
        return None, None

    per_step, launches, n_launches = stage_table(events, args.steps)
    step_ms = elapsed_ms / args.steps
    H = spec["hidden"]
    tile_mode = bool(plan.tile) and os.environ.get("B200_LSTM_TILE", "1") != "0"
    tile_chunks = plan.tile if tile_mode else plan.TILE
    cluster = plan.tile_cs if tile_mode else 8
    n_tiles = -(-N // tile_chunks)
    flops_step = {  # algorithmic FLOPs per step, all launches of the kernel (DESIGN.md section 4)
        "lstm_rec": spec["n_lstm"] * 2.0 * N * T * 4 * H * H,
        "lstm_in_gemm": spec["n_lstm"] * 2.0 * N * T * 4 * H * H,
        "conv_gemm": 2.0 * N * T * H * plan.k3 * plan.c2,
        "crf_gemm": 2.0 * N * T * plan.n_scores * H,
    }
    sms = torch.cuda.get_device_properties(device).multi_processor_count
    dominant = "lstm_rec"
    dur = per_step[dominant] / launches[dominant] * 1e-3
    ach = flops_step[dominant] / launches[dominant] / dur / 1e12
    # one launch = one cluster (6 or 8 SMs) working on one tile-layer, or all tiles of a layer: compare with that share of the chip
    launch_sms = cluster if launches[dominant] > spec["n_lstm"] else min(cluster * n_tiles, sms)
    peak_share = peaks["tflops"] * launch_sms / sms
    chip_ach = flops_step[dominant] / (step_ms * 1e-3) / 1e12
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            rec = json.load(fh)["lstm_rec_tile" if tile_mode else "lstm_rec"]
            traffic = rec["bytes"] if N == BATCH and launches[dominant] == rec.get("launches_per_step", launches[dominant]) else None
    except Exception:
        pass
    chunks_per_launch = N * spec["n_lstm"] / launches[dominant]
    roof = {"kernel": ("lstm_rec_tc6_kernel (persistent tcgen05 LSTM layer, one 6-CTA cluster per 48-chunk tile)" if tile_mode else
                       "lstm_rec_tc_kernel (persistent tcgen05 LSTM layer, one 8-CTA cluster per 32-chunk tile)"),
            "bound": "tensor", "achieved": ach, "peak": peak_share, "unit": "TFLOP/s", "frac": ach / peak_share,
            "traffic": traffic, "traffic_algorithmic": 2.0 * T * chunks_per_launch * 5 * H,
            "peak_source": f"{peaks['source']} sustained bf16 GEMM {peaks['tflops']} TFLOP/s x {launch_sms}/{sms} SMs "
                           "(the share of the chip one launch occupies)",
            "launch_ms": dur * 1e3, "launches_per_step": launches[dominant],
            "flops_per_launch": flops_step[dominant] / launches[dominant],
            "chip_level": {"achieved": chip_ach, "peak": peaks["tflops"], "frac": chip_ach / peaks["tflops"],
                           "note": "all lstm_rec FLOPs of a step / whole step time (other kernels overlap)"}}
    total_flops = sum(flops_step.values())
    line = {
        "metric": METRIC, "value": world * N * L * args.steps / (elapsed_ms * 1e-3), "unit": "samples/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": step_ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": f"hac-shaped LSTM-CRF (H={H}, {spec['n_lstm']} LSTM, {plan.n_scores} scores/frame), "
                               f"batch {N}/GPU, {CHUNK}->{L}-sample chunks ({T} frames), forward+decode",
                   "weights": "seeded synthetic (bonito_b200/synth.py)", "l2": "per-step tensors (0.16-2.6 GB) exceed the 126 MB L2",
                   "parallelism": f"chunk-sharded replicas x{world}",
                   "batches_in_flight": slots},
        "e2e": {"value": world * N * L * args.steps / (e2e_ms * 1e-3), "unit": "samples/s",
                "h2d_bytes_per_step": N * L * 2, "d2h_bytes_per_step": 3 * N * T, "ms_per_step": e2e_ms / args.steps,
                "api": "bonito_b200.crf.basecall.score_batches(model, float32 host batches): the loop basecall() runs",
                "single_call_ms_per_step": single_ms},
        "gpu_launches": n_launches,
        "roofline": roof,
        "stage_launch_ms_summed_per_step": {k: round(v, 4) for k, v in per_step.items()},
        "launches_per_step": launches,
        "host_enqueue_ms_per_step": round(enqueue_ms, 3),
        "model_tflops_per_s": total_flops / (step_ms * 1e-3) / 1e12,
    }
    del model, plan
    return line, (spec, weights, L)


def bench_hac_quantized(ctx):
    """The `--quantize` option of the basecaller (int8 LSTM input projections): the headline shape once more, resident only.
    A separate configuration: its scores differ from the fp16 path (tests/test_gpu_pipeline.py states the budget)."""
    from bonito_b200 import synth
    from bonito_b200.decode import _decoder
    args, device = ctx.args, ctx.device
    model, spec, _, L = build_hac(device, ctx.rank, ctx.world, batch=args.batch, quantize=True)
    N = args.batch
    x_dev = synth.squiggle(64, L, seed=100 + ctx.rank).repeat(N // 64 + 1, 1, 1)[:N].contiguous().to(device, torch.float16)
    plan = model.native_plan(device)
    qs = model.config["qscore"]

    def step(events, slot):
        scores = plan.forward(x_dev, events=None, slot=slot)
        return _decoder(scores, spec["state_len"], blank_score=plan.blank_score, qscale=qs["scale"], qbias=qs["bias"], slot=slot)

    steps = min(args.steps, 10)
    elapsed_ms, _, _, _ = time_resident(ctx, step, steps, 3, None, slots=N_SLOTS if plan.supports_slots else 1)
    (elapsed_ms,) = ctx.max_over_ranks([elapsed_ms])
    del model, plan
    torch.cuda.empty_cache()
    return {"workload": f"hac-shaped LSTM-CRF, batch {N} x {L} samples, int8 input projections (basecaller --quantize)",
            "value": ctx.world * N * L * steps / (elapsed_ms * 1e-3), "unit": "samples/s", "n_gpus": ctx.world, "steps": steps,
            "warmup": 3, "ms_per_step": elapsed_ms / steps, "dtype": "i8 input projections, f16 elsewhere"}


def sup_flops(spec, plan, N, L):
    """Algorithmic FLOPs of one sup step by stage (SURVEY.md section 8d)."""
    geo = plan._geometry(L)
    d, ff, depth = spec["d_model"], spec["dim_feedforward"], spec["depth"]
    Tq = geo[-1]["lout"]
    M = N * Tq
    wl, wr = spec["window"]
    keys = sum(min(Tq - 1, i + wr) - max(0, i - wl) + 1 for i in range(Tq)) / Tq     # visible keys per query, averaged
    conv = sum(2.0 * N * g["lout"] * c["cout"] * c["k"] * c["cin"] for g, c in zip(geo, plan.convs))
    return {"conv_gemm": conv, "qkv_gemm": depth * 2.0 * M * 3 * d * d, "attention": depth * 4.0 * M * d * keys,
            "proj_gemm": depth * 2.0 * M * d * d, "fc1_swiglu_gemm": depth * 2.0 * M * 2 * ff * d,
            "fc2_gemm": depth * 2.0 * M * d * ff, "upsample_gemm": 2.0 * M * 2 * d * d,
            "crf_gemm": 2.0 * 2 * M * plan.n_scores * d}, Tq


def bench_sup(ctx, peaks, model, spec, L, steps, warmup, with_e2e=True, dump=None):
    """One sup configuration: batch 256 x L samples per GPU; returns the block that goes under `configs`.
    `dump`: directory for the outputs of the last timed step (see dump_outputs)."""
    from bonito_b200 import synth
    from bonito_b200.decode import _decoder
    rank, world, device = ctx.rank, ctx.world, ctx.device
    N = SUP_BATCH
    host_batch = synth.squiggle(32, L, seed=200 + rank).repeat(N // 32 + 1, 1, 1)[:N].contiguous()
    x_dev = host_batch.to(device, torch.float16)
    plan = model.native_plan(device)
    qs = model.config["qscore"]

    def step(events, slot):
        scores = plan.forward(x_dev, events=events, slot=slot)
        return scores, _decoder(scores, spec["state_len"], blank_score=plan.blank_score, qscale=qs["scale"],
                                qbias=qs["bias"], events=events, slot=slot)

    # one batch at a time: the sup step is one long chain of chip-filling GEMMs, a second batch in flight buys nothing
    # (54.5 vs 56.2 ms measured) and would blur the per-kernel event times
    elapsed_ms, events, enqueue_ms, last = time_resident(ctx, step, steps, warmup, slots=1)
    if dump and rank == 0:
        dump_outputs(dump, *last)
    del last
    e2e_ms = time_e2e(ctx, model, host_batch, steps, qs) if with_e2e else 0.0
    elapsed_ms, e2e_ms = ctx.max_over_ranks([elapsed_ms, e2e_ms])
    log(f"sup L={L}: resident {elapsed_ms / steps:.2f} ms/step" + (f", e2e {e2e_ms / steps:.2f}" if with_e2e else ""))
    if rank != 0:
        return None
    per_step, launches, n_launches = stage_table(events, steps)
    flops, Tq = sup_flops(spec, plan, N, L)
    step_ms = elapsed_ms / steps
    # dominant kernel = the tensor-core stage with the largest share of the step (the launches run on one stream: no overlap)
    dominant = max((k for k in per_step if k in flops), key=lambda k: per_step[k])
    ach = flops[dominant] / (per_step[dominant] * 1e-3) / 1e12
    block = {
        "workload": f"sup-shaped transformer ({spec['depth']} layers, d_model {spec['d_model']}, {spec['nhead']} heads, window "
                    f"{spec['window'][0]}/{spec['window'][1]}, {4 ** (spec['state_len'] + 1)} scores/frame), batch {N}/GPU, "
                    f"{L}-sample chunks ({Tq} tokens, {2 * Tq} frames), forward+decode",
        "value": world * N * L * steps / (elapsed_ms * 1e-3), "unit": "samples/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": step_ms, "dtype": "f16",
        "roofline": {"kernel": dominant, "bound": "tensor", "achieved": ach, "peak": peaks["tflops"], "unit": "TFLOP/s",
                     "frac": ach / peaks["tflops"], "traffic": None,
                     "peak_source": f"{peaks['source']} sustained bf16 GEMM", "ms_per_step": per_step[dominant],
                     "launches_per_step": launches[dominant]},
        "stage_ms_per_step": {k: round(v, 3) for k, v in per_step.items()},
        "stage_tflops": {k: round(flops[k] / (per_step[k] * 1e-3) / 1e12, 1) for k in flops if k in per_step},
        "model_tflops_per_s": sum(flops.values()) / (step_ms * 1e-3) / 1e12,
        "gpu_launches": n_launches, "host_enqueue_ms_per_step": round(enqueue_ms, 3),
    }
    if with_e2e:
        block["e2e"] = {"value": world * N * L * steps / (e2e_ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": N * L * 2,
                        "d2h_bytes_per_step": 3 * N * 2 * Tq, "ms_per_step": e2e_ms / steps}
    return block


# ---------------------------------------------------------------------------------------------------------------
# CPU legs (oracle port of the reference's PyTorch-CPU path; rank 0, N = 1 only)
# ---------------------------------------------------------------------------------------------------------------
def _cpu_run(ref, x, threads):
    torch.set_num_threads(threads)
    os.environ["OMP_NUM_THREADS"] = str(threads)
    ref.forward(x[:2])  # warm-up
    _, _, _, tf, td = ref.basecall_batch(x)
    return tf, td


def _cpu_thread_sweep(ref, chunksize, label):
    """
    Thread counts 32 -> 64 -> all on a 32-chunk sample; the sweep stops as soon as more threads are slower (measured on the
    128-core GPU host: 64 threads are 1.8x SLOWER than 32 for this recurrent workload, and 128 threads did not finish a
    128-chunk sample in 7 minutes), then a larger sample is tried at the best thread count.  Returns
    (value, threads, n_chunks, t_forward, t_decode, tried, x).
    """
    from oracle import synth
    cores = os.cpu_count() or 1
    best, tried = None, []
    x32 = synth.squiggle(32, chunksize, seed=25)
    for threads in sorted({min(cores, 32), min(cores, 64), cores}):
        tf, td = _cpu_run(ref, x32, threads)
        v = 32 * chunksize / (tf + td)
        tried.append({"threads": threads, "chunks": 32, "samples_per_s": round(v, 1)})
        log(f"{label}: 32 chunks on {threads} threads: forward {tf:.2f}s decode {td:.2f}s -> {v:.3g} samples/s")
        if best is not None and v < best[0]:
            break
        best = (v, threads, 32, tf, td, x32)
    if best[3] + best[4] < 4.0:
        x64 = synth.squiggle(64, chunksize, seed=25)
        tf, td = _cpu_run(ref, x64, best[1])
        v = 64 * chunksize / (tf + td)
        tried.append({"threads": best[1], "chunks": 64, "samples_per_s": round(v, 1)})
        log(f"{label}: 64 chunks on {best[1]} threads: forward {tf:.2f}s decode {td:.2f}s -> {v:.3g} samples/s")
        if v > best[0]:
            best = (v, best[1], 64, tf, td, x64)
    return (*best[:5], tried, best[5])


def cpu_baseline(spec, weights, chunksize):
    """hac on the host cores (oracle port of the reference's PyTorch-CPU path), best of a bounded thread / sample sweep."""
    from oracle.cpu_reference import CpuReferenceModel
    ref = CpuReferenceModel(spec, weights)
    v, threads, n_chunks, tf, td, tried, _ = _cpu_thread_sweep(ref, chunksize, "cpu baseline")
    return {"value": v, "unit": "samples/s", "cores": threads, "host_cores": os.cpu_count(), "kind": "port",
            "forward_only": n_chunks * chunksize / tf, "tried": tried,
            "sample": f"{n_chunks} chunks x {chunksize} samples, torch {torch.__version__} fp32 modules as bonito.nn builds them + "
                      f"OpenMP C posterior-Viterbi decode (forward {tf:.2f}s, decode {td:.2f}s); thread count from a sweep that "
                      "stops when more threads are slower"}


def cpu_config1():
    """BASELINE config 1: fast-shaped LSTM-CRF, batch 8 x 4000 samples, PyTorch-CPU, best of a few thread counts."""
    from oracle import synth
    from oracle.cpu_reference import CpuReferenceModel
    spec = synth.model_spec("fast")
    ref = CpuReferenceModel(spec, synth.make_weights(spec, seed=25))
    x = synth.squiggle(8, 4000, seed=25)
    cores = os.cpu_count() or 1
    best, tried = None, []
    for threads in sorted({1, min(cores, 8), min(cores, 32)}):     # (8 x 4000 samples cannot use more)
        torch.set_num_threads(threads)
        os.environ["OMP_NUM_THREADS"] = str(threads)
        for _ in range(2):
            ref.basecall_batch(x)
        times = []
        for _ in range(5):
            _, _, _, tf, td = ref.basecall_batch(x)
            times.append((tf + td, tf, td))
        t, tf, td = sorted(times)[len(times) // 2]
        v = 8 * 4000 / t
        tried.append({"threads": threads, "samples_per_s": round(v, 1), "forward_s": round(tf, 4), "decode_s": round(td, 4)})
        if best is None or v > best[0]:
            best = (v, threads, tf, td)
    v, threads, tf, td = best
    log(f"config 1 (fast, 8 x 4000, CPU): {v:.3g} samples/s on {threads} threads")
    return {"workload": "fast-shaped LSTM-CRF (H=96, 5 LSTM, 256 scores/frame), batch 8, 4000-sample chunks, forward+decode, "
                        "PyTorch-CPU fp32 (reference path) + OpenMP C decode", "value": v, "unit": "samples/s",
            "cores": threads, "host_cores": cores, "kind": "port", "forward_only": 8 * 4000 / tf, "tried": tried,
            "protocol": "2 warm-up + 5 timed iterations, median"}


def run_reference(args, rank, world):
    """Reference arm: PyTorch-CPU path of the headline workload on all host cores; rank 0 only."""
    if rank != 0:
        return
    from oracle import synth
    from oracle.cpu_reference import CpuReferenceModel
    spec = synth.model_spec("hac")
    weights = synth.make_weights(spec, seed=25)
    chunksize = CHUNK - CHUNK % 6
    cores = os.cpu_count() or 1
    ref = CpuReferenceModel(spec, weights)
    _, threads, n_chunks, _, _, tried, x = _cpu_thread_sweep(ref, chunksize, "reference arm probe")
    torch.set_num_threads(threads)
    os.environ["OMP_NUM_THREADS"] = str(threads)
    for _ in range(max(args.warmup, 1)):
        ref.forward(x[:2])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ref.basecall_batch(x)
    dt = time.perf_counter() - t0
    value = n_chunks * chunksize * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"hac-shaped LSTM-CRF, {chunksize}-sample chunks, forward+decode",
                   "sample_chunks_per_step": n_chunks},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": threads, "host_cores": cores, "kind": "port",
                         "tried": tried,
                         "sample": f"{n_chunks} chunks x {chunksize} samples per step (torch fp32 modules as bonito.nn builds "
                                   f"them + OpenMP C decode), thread count from a sweep that stops when more threads are slower"},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--workload", default="all", choices=["all", "hac", "sup"],
                    help="all: hac headline line + the other BASELINE configurations under `configs`; hac: headline only; "
                         "sup: config 3 as the headline of the line")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (float32, at most "
                         "64 MB: decoder outputs of every chunk, scores of a seeded sample of chunks; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")

    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
        if os.environ.get("B200_PIN", "1") != "0":   # one slice of the host cores per rank (8 Python processes per node)
            from bonito_b200.distributed import pin_to_local_cores
            pin_to_local_cores(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    ctx = Ctx(args, rank, local_rank, world, device)
    peaks = load_peaks()

    with torch.inference_mode():
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()          # nvidia-smi needs a moment before its first sample: start it before the warm-up
        line = hac_state = None
        if args.workload in ("all", "hac"):
            line, hac_state = bench_hac(ctx, peaks, sampler)
        clocks = sampler.stop() if rank == 0 else None
        torch.cuda.empty_cache()

        configs = {}
        if args.workload in ("all", "hac"):
            cq = bench_hac_quantized(ctx)
            if rank == 0:
                configs["hac_quantize_int8"] = cq
                log(f"hac --quantize: {cq['ms_per_step']:.2f} ms/step")
        if args.workload in ("all", "sup"):
            model, spec = build_sup(device, rank, world)
            log("sup model built")
            sup_steps, sup_warm = min(args.steps, 10), 3
            if args.workload == "sup":
                sampler = ClockSampler(local_rank)
                if rank == 0:
                    sampler.start()
                    time.sleep(0.3)
                    sampler.mark_begin()
            headline = args.workload == "sup"
            c3 = bench_sup(ctx, peaks, model, spec, 9996, args.steps if headline else sup_steps, sup_warm,
                           dump=args.dump_outputs if headline else None)
            if args.workload == "sup" and rank == 0:
                sampler.mark_end()
                clocks = sampler.stop()
            sweep = [bench_sup(ctx, peaks, model, spec, L, max(3, sup_steps // 2), 3, with_e2e=False) for L in SUP_SWEEP]
            if rank == 0:
                configs["config3_sup"] = c3
                configs["config5_sup_sweep"] = [{k: b[k] for k in ("workload", "value", "unit", "n_gpus", "ms_per_step",
                                                                     "model_tflops_per_s", "stage_ms_per_step")} for b in sweep]
            del model
            torch.cuda.empty_cache()

    if rank == 0:
        if args.workload == "sup":
            c3 = configs.pop("config3_sup")
            line = {"metric": "raw-signal samples/sec basecalled (forward+decode), 10k-sample chunks, sup-shaped transformer",
                    "value": c3["value"], "unit": "samples/s", "n_gpus": world, "steps": c3["steps"], "warmup": c3["warmup"],
                    "ms_per_step": c3["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                    "dtype": "f16", "data": "synthetic",
                    "config": {"workload": c3["workload"], "weights": "seeded synthetic (bonito_b200/synth.py)",
                               "l2": "per-step tensors (0.2-3.5 GB) exceed the 126 MB L2",
                               "parallelism": f"chunk-sharded replicas x{world}"},
                    "e2e": c3["e2e"], "gpu_launches": c3["gpu_launches"], "roofline": c3["roofline"],
                    "stage_ms_per_step": c3["stage_ms_per_step"], "stage_tflops": c3["stage_tflops"],
                    "model_tflops_per_s": c3["model_tflops_per_s"]}
        line["clocks"] = clocks
        if world == 1 and not args.no_cpu_baseline:
            if hac_state is not None:
                line["cpu_baseline"] = cpu_baseline(*hac_state)
            if args.workload == "all":
                configs["config1_fast_cpu"] = cpu_config1()
        if configs:
            line["configs"] = configs
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
