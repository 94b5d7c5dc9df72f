#!/usr/bin/env python
"""bench.py -- audio-sec/sec (RTF^-1) and p50 chunk latency of the WhisperLive per-chunk hot path
(PCM -> log-mel -> encoder -> beam-search decoder) on N B200s of one node.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the CPU arm (oracle port; CT2/faster-whisper are absent)

Workload (BASELINE.json metric): Whisper large-v3, 32 concurrent streams in total, beam 4, chunk
durations U[5,30] s (VAD-gated chunk emulation, seed 1234+stream), synthetic speech-like 16 kHz PCM,
random-init weights of the large-v3 architecture (no checkpoints offline).  Streams are sharded
round-robin over the ranks (weights replicated, no data-path collective; one all_gather of the
emitted token ids per batch so every rank holds the whole batch's result).  With random weights the
decode length is pinned: EOT is suppressed and each stream decodes ceil(3.2 * seconds) + 8 tokens
(a typical Whisper token rate incl. timestamps), so both arms execute the same number of steps.

One "step" = one pass of the hot path over the batch of chunks:
  value : inputs resident in HBM (PCM uploaded by the warm-up), device time (CUDA events on the
          library stream, max over ranks)
  e2e   : the public API call B200WhisperModel.transcribe_batch(host numpy PCM) -> Segment lists on the
          host; H2D of the PCM/features and D2H of features/token ids inside the timed region
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "audio-sec/sec (RTF^-1) Whisper large-v3, 32 streams, beam 4"


def metric_name(args) -> str:
    """BASELINE's metric at the default flags; the same quantity named after the flags otherwise (parity-config runs)."""
    if (args.model, args.streams, args.beam) == ("large-v3", 32, 4):
        return METRIC
    return f"audio-sec/sec (RTF^-1) Whisper {args.model}, {args.streams} streams, beam {args.beam}"
UNIT = "audio-sec/sec"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="large-v3")
    ap.add_argument("--streams", type=int, default=32, help="total concurrent streams (sharded over the ranks)")
    ap.add_argument("--beam", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=8.0, help="chunk length of the bounded CPU sample")
    ap.add_argument("--cpu-steps", type=int, default=3, help="timed steps of the in-run CPU baseline")
    ap.add_argument("--word-timestamps", action="store_true", help="BASELINE config 4: K14 word alignment on every chunk (e2e only)")
    ap.add_argument("--no-streaming", action="store_true", help="skip the staggered-arrival latency phase (RoundScheduler, step-level admission)")
    ap.add_argument("--stream-load", type=float, default=0.6, help="offered load of the streaming phase as a fraction of the batch throughput")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step of each timed path "
                    "returned as DIR/<name>.npy (float64; rank 0's streams for the resident path)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def tokens_for(seconds: float) -> int:
    return int(math.ceil(3.2 * seconds)) + 8


def make_streams(n_total: int):
    from whisperlive_b200 import synth
    durs = synth.chunk_durations(n_total, 5.0, 30.0, seed=1234)
    return durs, [synth.speech_like(d, seed=1234 + i) for i, d in enumerate(durs)]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        top = sorted(sm)[len(sm) // 2:] if sm else []   # upper half = samples under load
        return {"sm_mhz": statistics.median(top) if top else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def physical_cores():
    try:
        import psutil
        return psutil.cpu_count(logical=False)
    except Exception:
        return None


def cpu_oracle_sample(model: str, beam: int, seconds: float, threads: int):
    """The CPU arm: oracle port (torch fp32 + restated CT2 search) on one bounded chunk."""
    import torch
    from oracle.engine import OracleWhisper
    from oracle import mel as omel
    from whisperlive_b200 import synth
    from whisperlive_b200.config import dims_for
    from whisperlive_b200.weights import random_init
    torch.set_num_threads(threads)
    dims = dims_for(model)
    eng = OracleWhisper(random_init(dims, seed=0), dims)
    sp = eng.spec
    prompt = [sp.sot] if not dims.multilingual else [sp.sot, sp.sot + 1, sp.sot + 1 + dims.num_languages + 1]
    n_new = tokens_for(seconds)
    wav = synth.speech_like(seconds, seed=1234)

    def step():
        t0 = time.perf_counter()
        feats = omel.pad_or_trim(omel.log_mel(wav, dims.n_mels)[:, :-1])
        enc = eng.encode(feats[None])
        eng.generate(enc, [prompt], beam_size=beam, suppress_tokens=[sp.eot], max_length=2 * n_new, suppress_blank=False)
        return time.perf_counter() - t0
    return step, seconds, n_new


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    threads = min(os.cpu_count() or 1, 32)   # torch intra-op threads; more only adds synchronisation overhead
    step, seconds, n_new = cpu_oracle_sample(args.model, args.beam, args.cpu_seconds, threads)
    for _ in range(min(args.warmup, 1)):
        step()
    times = [step() for _ in range(args.steps)]
    total = sum(times)
    value = seconds * len(times) / total
    sample = (f"1 stream x {seconds:.0f} s chunk per step, {n_new} decoded tokens, beam {args.beam}, torch fp32 oracle port "
              f"(stand-in: faster-whisper / CTranslate2 are not installed, not the reference binary)")
    line = {
        "metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000 * total / len(times), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "impl": "reference",
        "config": {"workload": f"Whisper {args.model} random-init, CPU sample of the bench workload", "beam": args.beam,
                   "sample": sample},
        "p50_chunk_latency_ms": 1000 * statistics.median(times),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "physical_cores": physical_cores(),
                         "logical_cpus": os.cpu_count(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from whisperlive_b200.config import dims_for
    from whisperlive_b200.engine import B200Whisper
    from whisperlive_b200.feature_extractor import FeatureExtractor
    from whisperlive_b200.tokenizer import build_synthetic_tokenizer
    from whisperlive_b200.transcriber import B200WhisperModel
    from whisperlive_b200.weights import random_init

    dims = dims_for(args.model)
    durs, waves = make_streams(args.streams)
    mine = [i for i in range(args.streams) if i % world == rank]
    my_waves = [waves[i] for i in mine]
    my_durs = [durs[i] for i in mine]
    n_local = len(mine)
    heads = [(dims.dec_layers - 1 - (i // 4), (3 * i) % dims.n_heads) for i in range(10)]
    eng = B200Whisper(dims, random_init(dims, seed=0), device_index=local, max_streams=max(1, n_local), max_beam=max(args.beam, 1),
                      enc_slots=2 * max(1, n_local) + 2, alignment_heads=heads)
    model = B200WhisperModel(args.model, engine=eng, hf_tokenizer=build_synthetic_tokenizer(dims.vocab),
                             feature_extractor=FeatureExtractor(eng, dims.n_mels))
    tok_eot = eng.eot
    n_sot = 3 if dims.multilingual else 1   # CT2 decodes min(max_length/2, max_length - prompt) tokens: 2N gives N
    all_kws = [dict(beam_size=args.beam, temperature=[0.0], log_prob_threshold=None, compression_ratio_threshold=None,
                    no_speech_threshold=None, suppress_tokens=[-1, tok_eot], suppress_blank=False,
                    max_new_tokens=2 * tokens_for(d) - n_sot, language="en" if dims.multilingual else None,
                    condition_on_previous_text=False, word_timestamps=bool(args.word_timestamps), _single_window=True)
               for d in durs]
    audio_sec_total = float(sum(durs))
    # the product's multi-GPU front end: streams placed i mod W, one all-gather of ids + times per batch
    from whisperlive_b200.parallel import DistributedTranscriber
    dist_tr = DistributedTranscriber(model)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}   # what the latest step of each timed path returned (--dump-outputs)

    def e2e_step():
        t0 = time.perf_counter()
        out = dist_tr.transcribe_batch(waves, all_kws)      # whole batch in, whole batch out on every rank
        n_ids = sum(len(s.tokens) for segs, _ in out for s in (segs or []))
        last["e2e"] = out
        return time.perf_counter() - t0, n_ids

    # ---- resident-input step: PCM / features already in HBM, device-timed
    feats_cache = {}

    def resident_step():
        ms = 0.0
        eng.lib.wl_mel_resident(eng.ctx)
        ms += eng.last_device_ms(0)
        slots = feats_cache["slots"]
        import ctypes as C
        from whisperlive_b200 import _lib
        rc = eng.lib.wl_encode_resident(eng.ctx, len(slots), _lib.ptr(slots, C.c_int32))
        _lib.check(eng.lib, eng.ctx, rc, "wl_encode_resident")
        ms += eng.last_device_ms(1)
        last["resident"] = eng.generate(feats_cache["enc"], feats_cache["prompts"], **feats_cache["gen_kw"])
        ms += eng.last_device_ms(2)
        return ms / 1000.0

    def prime_resident():
        feats = model.feature_extractor.batch(my_waves)
        from whisperlive_b200.transcriber import pad_or_trim
        f3 = np.stack([pad_or_trim(f[:, :-1], 3000) for f in feats])
        enc = eng.encode(f3)
        sot_seq = [eng.sot] if not dims.multilingual else [eng.sot, eng.sot + 1, eng.sot + 1 + dims.num_languages + 1]
        feats_cache["enc"] = enc
        feats_cache["slots"] = np.asarray(enc.slots, dtype=np.int32)
        feats_cache["prompts"] = [sot_seq] * n_local
        n_max = max(tokens_for(d) for d in my_durs)
        sup = sorted(set(model_suppress + [tok_eot]))
        feats_cache["gen_kw"] = dict(beam_size=args.beam, suppress_tokens=sup, suppress_blank=False, max_length=2 * n_max,
                                     max_length_per_stream=[2 * tokens_for(d) for d in my_durs])

    from whisperlive_b200.tokenizer import Tokenizer
    from whisperlive_b200.transcriber import get_suppressed_tokens
    _tk = Tokenizer(model.hf_tokenizer, dims.multilingual, task="transcribe" if dims.multilingual else None,
                    language="en" if dims.multilingual else None)
    model_suppress = list(get_suppressed_tokens(_tk, [-1]))

    # ---- warm-up
    for _ in range(max(3, args.warmup)):
        e2e_step()
    prime_resident()
    resident_step()
    barrier()

    # ---- timed: value (resident, device-timed)
    launches0 = eng.kernel_launches()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    t_res = [resident_step() for _ in range(args.steps)]
    barrier()
    launches_res = eng.kernel_launches() - launches0
    # ---- timed: e2e (host buffers through the public API)
    barrier()
    t0 = time.perf_counter()
    lat, n_ids = [], 0
    for _ in range(args.steps):
        dt, n_ids = e2e_step()
        lat.append(dt)
        if os.environ.get("WLB200_TRACE") and rank == 0:
            print("e2e step %.1f ms; host split (ms): %s" % (1000 * dt, {k: round(1000 * v, 1) for k, v in model.last_timing.items()}),
                  file=sys.stderr)
    barrier()
    t_e2e = time.perf_counter() - t0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, feats_cache["enc"], last["resident"], last["e2e"])

    loop_ms, loop_steps = eng.last_device_ms(2), getattr(eng, "last_steps", None)   # the last e2e step's decode loop
    # ---- streaming phase: staggered arrivals through the product scheduler (N=1 rank-local; reported, not the headline)
    streaming = None
    if not args.no_streaming and not args.word_timestamps:
        try:
            streaming = streaming_latency(model, my_waves, [all_kws[i] for i in mine], my_durs, sum(lat) / len(lat), args.stream_load)
        except Exception as ex:   # the phase is additional evidence: report why it is missing instead of losing the line
            streaming = {"error": repr(ex)}
    barrier()

    res_total = sum(t_res)
    stats = torch.tensor([res_total, t_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    res_total, t_e2e = float(stats[0]), float(stats[1])
    value = audio_sec_total * args.steps / res_total
    e2e_value = audio_sec_total * args.steps / t_e2e
    # bytes the e2e step moves per rank, counted from the buffers libwlb200 copies: PCM up (wl_mel_device; the log-mel and
    # the encoder input never leave HBM), prompts + per-stream metadata up, and per generate call the finished-hypothesis
    # tables down (wl_generate: hyp_tok [B][16][448] + lengths / scores / counters)
    h2d = sum(w.nbytes for w in my_waves) + n_local * (448 + 16) * 4
    d2h = n_local * (16 * 448 * 4 + 16 * 8 + 16)
    if args.word_timestamps:   # K14: text-token probabilities + DTW path (<= 448 + 1500 pairs) per stream
        d2h += n_local * ((448 + 1500 + 2) * 8 + 448 * 4)

    # ---- roofline of the dominant kernel (cross-attention K/V streaming), measured live
    roof = dominant_kernel_roofline(eng, dims, n_local, args.beam, feats_cache, loop_ms, loop_steps)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = min(os.cpu_count() or 1, 32)
        step, seconds, n_new = cpu_oracle_sample(args.model, args.beam, args.cpu_seconds, threads)
        step()                                               # warm-up (thread pool, allocator)
        cts = [step() for _ in range(max(1, args.cpu_steps))]
        cpu = {"value": seconds * len(cts) / sum(cts), "unit": UNIT, "cores": threads, "physical_cores": physical_cores(),
               "logical_cpus": os.cpu_count(), "kind": "port", "steps": len(cts), "step_s": [round(x, 2) for x in cts],
               "sample": f"{len(cts)} timed steps after 1 warm-up, each 1 stream x {seconds:.0f} s chunk, {n_new} decoded tokens, beam "
                         f"{args.beam}, torch fp32 oracle port on {threads} threads (stand-in, not the reference binary: "
                         f"faster-whisper/CTranslate2 absent)"}
    if rank == 0:
        line = {
            "metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": 1000 * res_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic",
            "config": {"workload": f"Whisper {args.model} (random-init), {args.streams} streams total sharded round-robin over "
                                   f"{world} GPU(s), beam {args.beam}, chunks U[5,30] s (sum {audio_sec_total:.0f} s audio/step), "
                                   "decode length pinned to ceil(3.2*s)+8 tokens (EOT suppressed)",
                       "streams": args.streams, "streams_per_gpu": n_local, "beam": args.beam, "parallelism": f"dp{world}",
                       "l2": "working set (3.1 GB weights + 246 MB/stream cross-KV) >> 126 MB L2, no flush needed"},
            "p50_chunk_latency_ms": 1000 * statistics.median(lat),
            "streaming": streaming,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": 1000 * t_e2e / args.steps,
                    "api": "whisperlive_b200.parallel.DistributedTranscriber(B200WhisperModel).transcribe_batch(host PCM)",
                    "gather_bytes_per_step": int(dist_tr.last_gather_bytes), "word_timestamps": bool(args.word_timestamps)},
            "gpu_launches": int(launches_res),
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir: str, eng, enc, resident, e2e):
    """The last timed step's results as float64 arrays, padded with -1 where lengths differ.

    resident_*: what ``generate`` returned for this rank's streams (best hypothesis), and the encoder output it decoded
    from -- 64 frames per stream drawn with a fixed seed, all channels.  e2e_*: what ``transcribe_batch`` returned for
    every stream: segment tokens, and one row per segment (stream, start, end, avg_logprob, no_speech_prob,
    compression_ratio)."""
    os.makedirs(out_dir, exist_ok=True)

    def padded(rows):
        a = np.full((len(rows), max([len(r) for r in rows] + [1])), -1.0)
        for i, r in enumerate(rows):
            a[i, :len(r)] = r
        return a
    frames = np.sort(np.random.default_rng(0).choice(1500, 64, replace=False))
    arrays = {
        "resident_tokens": padded([r.sequences_ids[0] for r in resident]),
        "resident_scores": np.array([r.scores[0] for r in resident], dtype=np.float64),
        "resident_no_speech_prob": np.array([r.no_speech_prob for r in resident], dtype=np.float64),
        "resident_encoder_output_sample": np.stack([eng._encoder_output(s)[frames] for s in enc.slots]).astype(np.float64),
        "e2e_tokens": padded([[t for s in (segs or []) for t in s.tokens] for segs, _ in e2e]),
        "e2e_segments": np.array([[i, s.start, s.end, s.avg_logprob, s.no_speech_prob, s.compression_ratio]
                                  for i, (segs, _) in enumerate(e2e) for s in (segs or [])], dtype=np.float64).reshape(-1, 6),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def streaming_latency(model, waves, kws, durs, batch_step_s: float, load: float, cycles: int = 3, step_tokens: int = 16):
    """p50 chunk latency the way a live server sees it (reference definition: wall time of ``transcribe_audio`` per
    chunk, whisper_live/backend/base.py:123-130): every stream's chunk ARRIVES at its own time -- uniformly spread so
    that the offered load is ``load`` x the batch throughput -- and is submitted to the product's scheduler
    (``RoundScheduler``: step-level admission into the running decode loop, N2).  Latency = submit -> segments."""
    import random
    from whisperlive_b200.scheduler import BatchRequest, RoundScheduler

    class Req(BatchRequest):
        def kwargs(self_):
            return self_.kw

    n = len(waves)
    period = batch_step_s / max(load, 1e-3)
    rng = random.Random(4321)
    sch = RoundScheduler(model, max_batch_size=model.model.max_streams, step_tokens=step_tokens)
    sch.start()
    lat, reqs = [], []
    try:
        # warm-up cycle (captures the session's graph), then `cycles` measured ones
        for cyc in range(cycles + 1):
            t_start = time.monotonic()
            offs = sorted((rng.uniform(0.0, period), i) for i in range(n))
            batch = []
            for off, i in offs:
                dt = t_start + off - time.monotonic()
                if dt > 0:
                    time.sleep(dt)
                r = Req(audio=waves[i])
                r.kw = kws[i]
                sch.submit(r)
                batch.append(r)
            for r in batch:
                if not r.future.wait(120):
                    raise RuntimeError("streaming phase: a chunk was not answered within 120 s")
                if r.error is not None:
                    raise r.error
            left = t_start + period - time.monotonic()
            if left > 0:
                time.sleep(left)
            if cyc > 0:
                lat += [1000.0 * (r.finished_at - r.submitted_at) for r in batch]
                reqs += batch
    finally:
        sch.stop()
    lat.sort()
    q = lambda f: lat[min(len(lat) - 1, int(f * len(lat)))]
    return {"p50_chunk_latency_ms": q(0.5), "p90_chunk_latency_ms": q(0.9), "max_chunk_latency_ms": lat[-1], "chunks": len(lat),
            "offered_load": load, "arrival_period_ms": 1000.0 * period, "scheduler": f"RoundScheduler(step_tokens={step_tokens})",
            "rounds": sch.rounds_run, "admitted_mid_flight": sch.admitted_mid_flight,
            "what": "each stream's chunk arrives at its own uniformly drawn time inside the period; latency = submit -> segments "
                    "through the product scheduler (streams join the running device-side decode loop)"}


def dominant_kernel_roofline(eng, dims, n_streams, beam, feats_cache, loop_ms, loop_steps):
    """Roofline of the dominant kernel, decoder cross-attention (K11, cross_attn_kernel): one launch streams the
    encoder K and V of every live stream for one layer, 2 * 1500 * d_model fp16 values per stream (DESIGN.md
    section 4) -- HBM-bound.  Its launch duration is measured live: a short graph-less generate pass over the
    bench's own resident encoder outputs with CUDA events around every launch on the library stream
    (wl_profile_cross_attn).  `step` keeps the whole decode loop (weights + cross-KV + self-KV per token) for context."""
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    which = "measured burst copy bandwidth (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    d, L, V = dims.d_model, dims.dec_layers, dims.vocab
    # whole decode loop of the last timed generate call
    steps, ms = loop_steps, loop_ms
    step_info = None
    if steps and ms > 0:
        w_step = (14 * d * d * L + V * d) * 2
        kv_cross = n_streams * L * 2 * 1500 * d * 2
        kv_self = n_streams * beam * L * 2 * (0.5 * steps) * d * 2   # cache grows linearly: mean length over the loop
        bytes_step = w_step + kv_cross + kv_self
        ach = bytes_step * steps / (ms / 1000.0) / 1e9
        step_info = {"what": "decode loop: weights + cross-KV + self-KV per token (K9-K12)", "achieved": ach, "frac": ach / peak,
                     "algorithmic_bytes_per_step": int(bytes_step), "steps": int(steps), "ms_per_token_step": ms / steps}
    # the kernel itself
    graph0 = eng.use_cuda_graph
    kw = dict(feats_cache["gen_kw"])
    kw["max_length"] = 2 * 12
    kw["max_length_per_stream"] = [2 * 12] * n_streams          # 12 decode steps: every stream stays live
    try:
        eng.use_cuda_graph = False
        eng.profile_cross_attn(True)
        eng.generate(feats_cache["enc"], feats_cache["prompts"], **kw)
        avg_ms, n_launch = eng.last_device_ms(3), int(eng.last_device_ms(4))
    finally:
        eng.profile_cross_attn(False)
        eng.use_cuda_graph = graph0
    alg = n_streams * 2 * 1500 * d * 2          # bytes one launch has to read: K and V of every stream, fp16
    traffic = None
    try:   # DRAM bytes per launch from the committed ncu --set full capture of this kernel at this configuration
        for fn in ("traffic_r2.json", "traffic_r1.json"):      # newest committed ncu --set full capture of this kernel
            path = os.path.join(ROOT, "profiles", fn)
            if not os.path.exists(path):
                continue
            t = json.load(open(path)).get("cross_attn_kernel", {})
            if int(t.get("streams", -1)) == n_streams and t.get("model") == dims.name:
                traffic = float(t["dram_bytes_per_launch"])
                break
    except Exception:
        pass
    if avg_ms <= 0:
        return {"bound": "hbm", "kernel": "cross_attn_kernel (K11)", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None,
                "traffic": traffic, "peak_source": which, "step": step_info}
    achieved = alg / (avg_ms / 1000.0) / 1e9
    return {"bound": "hbm", "kernel": "cross_attn_kernel (K11 decoder cross-attention, one launch per decoder layer per token)",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "algorithmic_bytes_per_launch": int(alg), "avg_launch_us": 1000.0 * avg_ms, "launches_timed": n_launch,
            "timing": "CUDA events around each launch on the library stream (includes the launch gap), graph-less pass",
            "peak_source": which, "step": step_info}


if __name__ == "__main__":
    main()
