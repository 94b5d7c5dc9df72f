"""CPU tests of the drop-in boundary: C-ABI export list, plugin surface (ServeClientB200 on the
reference's own ServeClientBase), scheduler batching, and the multi-rank stream sharding (gloo)."""
import json
import os
import re
import subprocess
import sys
import threading

import numpy as np
import pytest
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_c_abi_exports_every_declared_symbol():
    """The library loads without a GPU and exports exactly what include/wlb200.h declares."""
    from whisperlive_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "wlb200.h")).read()
    declared = set(re.findall(r"\b(wl_[a-z_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), name
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (wl_[a-z_]+)", out))
    assert declared <= exported


def test_wl_init_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from whisperlive_b200.config import dims_for
    from whisperlive_b200.engine import B200Whisper
    from whisperlive_b200 import _lib
    with pytest.raises(_lib.WlError, match="no CUDA device|no CPU fallback"):
        B200Whisper(dims_for("micro.en"), {}, max_streams=1, max_beam=1)


def test_product_never_imports_oracle():
    """No module under whisperlive_b200/ may import the oracle (it is test infrastructure)."""
    pkg = os.path.join(ROOT, "whisperlive_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), fn


def test_no_silent_random_weights_or_synthetic_tokenizer(tmp_path):
    """ADVICE r1 (high): a size name without a checkpoint must raise (the reference resolves it through the hub,
    faster_whisper_backend.py:133-178); random weights / the fabricated vocabulary are explicit opt-ins only."""
    from whisperlive_b200.engine import B200Whisper
    from whisperlive_b200.transcriber import B200WhisperModel
    with pytest.raises(FileNotFoundError, match="no checkpoint"):
        B200Whisper.from_model("small.en", local_files_only=True, download_root=str(tmp_path))
    with pytest.raises(ValueError):
        B200Whisper.from_model("small.en", weights="zeros")
    with pytest.raises(FileNotFoundError, match="no checkpoint"):
        B200WhisperModel("small.en", local_files_only=True, download_root=str(tmp_path))
    m = _oracle_model()
    with pytest.raises(FileNotFoundError, match="tokenizer.json"):
        B200WhisperModel("micro.en", engine=m.model, feature_extractor=m.feature_extractor)
    ok = B200WhisperModel("micro.en", engine=m.model, feature_extractor=m.feature_extractor, hf_tokenizer="synthetic")
    assert ok.hf_tokenizer.get_vocab_size() >= m.model.vocab_size - 1


def _oracle_model(name="micro.en", seed=0):
    from oracle.engine import OracleWhisper
    from oracle.mel import OracleFeatureExtractor
    from whisperlive_b200.config import dims_for
    from whisperlive_b200.tokenizer import build_synthetic_tokenizer
    from whisperlive_b200.transcriber import B200WhisperModel
    from whisperlive_b200.weights import random_init
    dims = dims_for(name)
    return B200WhisperModel(name, engine=OracleWhisper(random_init(dims, seed=seed), dims),
                            hf_tokenizer=build_synthetic_tokenizer(dims.vocab),
                            feature_extractor=OracleFeatureExtractor(dims.n_mels))


def test_scheduler_survives_errors_and_isolates_them():
    """The owner thread keeps serving after a failing call; with a plain ``transcribe_batch`` transcriber (no sessions)
    every round is one call over whatever is in the inbox."""
    from whisperlive_b200.scheduler import BatchRequest, RoundScheduler

    class Fake:
        def __init__(self):
            self.calls = []

        def transcribe_batch(self, audios, kws):
            self.calls.append(len(audios))
            if any(len(a) == 13 for a in audios):
                raise RuntimeError("boom")
            return [([f"seg{len(a)}"], "info") for a in audios]
    fake = Fake()
    sch = RoundScheduler(fake, max_batch_size=4, linger_ms=200)
    sch.start()
    reqs = [BatchRequest(audio=np.zeros(n, np.float32), use_vad=False) for n in (5, 6, 7)]
    for r in reqs:
        sch.submit(r)
    assert all(r.future.wait(5) for r in reqs)
    assert [r.result for r in reqs] == [["seg5"], ["seg6"], ["seg7"]] and fake.calls == [3]
    bad = BatchRequest(audio=np.zeros(13, np.float32))
    sch.submit(bad)
    assert bad.future.wait(5) and isinstance(bad.error, RuntimeError)
    ok = BatchRequest(audio=np.zeros(2, np.float32))
    sch.submit(ok)
    assert ok.future.wait(5) and ok.result == ["seg2"]   # the owner thread is still alive
    sch.stop()


def test_round_scheduler_admits_mid_flight_and_answers_early():
    """N2: a chunk submitted while others are already decoding joins THEIR rounds (it is not queued behind the batch),
    and a short chunk is answered before a long multi-window one it shared rounds with; results equal the one-shot
    ``transcribe_batch`` of the same audio."""
    from whisperlive_b200 import synth
    from whisperlive_b200.scheduler import BatchRequest, RoundScheduler
    torch.set_num_threads(4)
    model = _oracle_model()
    long_wave, short_wave = synth.speech_like(65.0, seed=50), synth.speech_like(3.0, seed=51)

    class Req(BatchRequest):      # no sampling rungs: the comparison below is token for token
        def kwargs(self):
            return dict(super().kwargs(), temperature=[0.0], log_prob_threshold=None)
    BatchRequest = Req
    ref = model.transcribe_batch([long_wave, short_wave], [Req(audio=long_wave, use_vad=False, language="en").kwargs()] * 2)

    entered = threading.Event()
    orig_round = type(model.open_session()).round

    sch = RoundScheduler(model, max_batch_size=4, step_tokens=None)     # window-level rounds (step-level: next test)

    def patched_round(self_):
        entered.set()
        return orig_round(self_)
    sess_cls = type(model.open_session())
    sess_cls.round = patched_round
    try:
        sch.start()
        r_long = BatchRequest(audio=long_wave, use_vad=False, language="en")
        sch.submit(r_long)
        assert entered.wait(30)                      # the long stream is being decoded (3 windows ahead of it)
        r_short = BatchRequest(audio=short_wave, use_vad=False, language="en")
        sch.submit(r_short)
        assert r_short.future.wait(120) and r_long.future.wait(240)
    finally:
        sess_cls.round = orig_round
        sch.stop()
    assert r_short.error is None and r_long.error is None
    assert sch.admitted_mid_flight >= 1 and sch.max_in_flight == 2
    assert r_short.finished_at < r_long.finished_at      # answered without waiting for the stream it shared rounds with
    for r, (segs, _info) in zip((r_long, r_short), ref):
        assert [s.tokens for s in r.result] == [s.tokens for s in segs]
        assert [(s.start, s.end) for s in r.result] == [(s.start, s.end) for s in segs]


def test_step_scheduler_joins_the_running_decode_loop():
    """N2, token-step level: a chunk submitted while another stream is in the MIDDLE of its decode loop is admitted into
    that loop (``TranscribeSession.step_round`` over the engine's decode session) after a few token steps -- it does not
    wait for the running ``generate`` to end -- and is answered first; results equal the one-shot ``transcribe_batch``.
    (The oracle engine models the session's timing; ``tests/test_gpu_parity.py`` runs the real one.)"""
    from whisperlive_b200 import synth
    from whisperlive_b200.scheduler import BatchRequest, RoundScheduler
    torch.set_num_threads(4)
    model = _oracle_model()
    long_wave, short_wave = synth.speech_like(65.0, seed=50), synth.speech_like(3.0, seed=51)

    class Req(BatchRequest):      # no sampling rungs: the comparison below is token for token
        def kwargs(self):
            return dict(super().kwargs(), temperature=[0.0], log_prob_threshold=None)
    ref = model.transcribe_batch([long_wave, short_wave], [Req(audio=long_wave, use_vad=False, language="en").kwargs()] * 2)

    first_steps_done, short_submitted = threading.Event(), threading.Event()
    sess_cls = type(model.open_session())
    orig = sess_cls.step_round
    seen = {}

    def gated(self_, max_steps=16):
        seen["session"] = self_
        out = orig(self_, max_steps)
        if not first_steps_done.is_set():
            first_steps_done.set()                   # the long stream has run its first token steps ...
            short_submitted.wait(30)                 # ... and the short one arrives before the next ones
        return out
    sess_cls.step_round = gated
    sch = RoundScheduler(model, max_batch_size=4, step_tokens=2)
    try:
        sch.start()
        r_long = Req(audio=long_wave, use_vad=False, language="en")
        sch.submit(r_long)
        assert first_steps_done.wait(120)
        r_short = Req(audio=short_wave, use_vad=False, language="en")
        sch.submit(r_short)
        short_submitted.set()
        assert r_short.future.wait(240) and r_long.future.wait(480)
    finally:
        sess_cls.step_round = orig
        sch.stop()
    assert r_short.error is None and r_long.error is None
    sess = seen["session"]
    assert sess.admitted_steps[0] == 0 and any(a > 0 for a in sess.admitted_steps[1:])   # joined a loop that was already running
    assert sch.admitted_mid_flight >= 1 and sch.max_in_flight == 2
    assert r_short.finished_at < r_long.finished_at
    for r, (segs, _info) in zip((r_long, r_short), ref):
        assert [s.tokens for s in r.result] == [s.tokens for s in segs]
        assert [(s.start, s.end) for s in r.result] == [(s.start, s.end) for s in segs]


def test_backend_plugin_streams_segments_through_reference_base():
    """ServeClientB200 subclasses the reference's ServeClientBase; frames go in through the base's loop and segment JSON
    comes out of the base's send path.  tests/golden/record_plugin_base.py ran the plugin on the reference's own base and
    recorded every call across that boundary; here a stand-in base replays the record: its loop hands the plugin the
    same audio chunk and duration, and every call the plugin makes into the base (update_segments, prepare_segments,
    send_transcription_to_client) must come in the recorded order with the recorded arguments, and gets the reference
    base's answer back.  The plugin's own websocket messages and its transcription result must match too."""
    import importlib

    from tests.golden import record_plugin_base as R
    import whisperlive_b200.backend as backend
    from whisperlive_b200.scheduler import BatchRequest
    torch.set_num_threads(8)
    rec = json.load(open(os.path.join(ROOT, "tests", "golden", "plugin_base_calls.json")))
    stand_in = R.replay_module(rec)
    names = ("whisper_live", "whisper_live.backend", "whisper_live.backend.base")
    saved = {n: sys.modules.get(n) for n in names}
    sys.modules.update(zip(names, (type(sys)("whisper_live"), type(sys)("whisper_live.backend"), stand_in)))
    orig_kwargs = BatchRequest.kwargs
    BatchRequest.kwargs = lambda self: dict(orig_kwargs(self), **R.CHEAP)
    try:
        ServeClientB200 = importlib.reload(backend).ServeClientB200
        assert issubclass(ServeClientB200, stand_in.ServeClientBase)
        model = _oracle_model()
        ServeClientB200.MODEL_FACTORY = lambda name: model
        ws = R.WS()
        client = ServeClientB200(ws, **R.CLIENT)
        assert client.language == "en"
        assert stand_in.ServeClientBase.done.wait(120)
        client.trans_thread.join(timeout=30)
        assert not stand_in.ServeClientBase.mismatches, stand_in.ServeClientBase.mismatches
        # what the plugin sent itself; the segments message is the base's (checked above as send_transcription_to_client)
        assert ws.sent == [m for m in rec["sent"] if "segments" not in m] and ws.sent[0]["message"] == "SERVER_READY"
        segs = [m for m in rec["sent"] if "segments" in m]
        assert segs and set(segs[0]["segments"][0]) >= {"start", "end", "text", "completed"} and segs[0]["uid"] == "u1"
    finally:
        BatchRequest.kwargs = orig_kwargs
        backend.ServeClientB200.shutdown()
        backend.ServeClientB200.MODEL_FACTORY = None
        for n, m in saved.items():
            if m is None:
                sys.modules.pop(n, None)
            else:
                sys.modules[n] = m
        importlib.reload(backend)


GLOO_WORKER = r"""
import os, sys, json
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from tests.test_boundary_cpu import _oracle_model
from whisperlive_b200 import synth
from whisperlive_b200.parallel import DistributedTranscriber
torch.set_num_threads(2)
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + sys.argv[2], rank=int(sys.argv[3]), world_size=2)
n_streams = 3
waves = [synth.speech_like(2.0 + i, seed=40 + i) for i in range(n_streams)]
kw = dict(temperature=[0.0], beam_size=2, log_prob_threshold=None, max_new_tokens=16)
dt = DistributedTranscriber(_oracle_model())          # the product API: shards by rank, gathers ids + times
out = dt.transcribe_batch(waves, [kw] * n_streams)      # every rank passes (and gets back) the whole batch
res = [[[s.tokens, round(s.start, 3), round(s.end, 3)] for s in segs] for segs, _ in out]
owned = dt.owned(n_streams)
print("RESULT%d " % dist.get_rank() + json.dumps({"res": res, "owned": owned, "bytes": dt.last_gather_bytes}))
dist.destroy_process_group()
"""


def test_two_rank_stream_sharding_matches_single_process(tmp_path):
    """world_size=2 (gloo) through whisperlive_b200.parallel.DistributedTranscriber: streams sharded i mod W, one
    all-gather of ids + times per batch; BOTH ranks end up with the single-process result for every stream."""
    from whisperlive_b200 import synth
    torch.set_num_threads(4)
    model = _oracle_model()
    kw = dict(temperature=[0.0], beam_size=2, log_prob_threshold=None, max_new_tokens=16)
    waves = [synth.speech_like(2.0 + i, seed=40 + i) for i in range(3)]
    single = [[[s.tokens, round(s.start, 3), round(s.end, 3)] for s in segs] for segs, _ in model.transcribe_batch(waves, [kw] * 3)]
    script = tmp_path / "w.py"
    script.write_text(GLOO_WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                              text=True) for r in range(2)]
    outs = [p.communicate(timeout=300) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    for r in range(2):
        line = next(l for l in outs[r][0].splitlines() if l.startswith(f"RESULT{r} "))
        got = json.loads(line[len(f"RESULT{r} "):])
        assert got["owned"] == [i for i in range(3) if i % 2 == r] and got["bytes"] > 0
        assert got["res"] == single, (r, got["res"], single)


def test_multi_device_model_fans_out_and_keeps_order():
    """One process, several engine contexts (MultiDeviceWhisperModel): sticky i mod G placement, results in input order,
    explicit placement honoured, a failing device propagates its error."""
    from whisperlive_b200.parallel import MultiDeviceWhisperModel, owner_of

    class Fake:
        def __init__(self, g):
            self.g, self.calls = g, []
            self.model = self
            self.hf_tokenizer = None

        def transcribe_batch(self, audios, kws):
            self.calls.append([len(a) for a in audios])
            if any(len(a) == 13 for a in audios):
                raise RuntimeError("boom")
            return [((self.g, len(a)), k.get("tag")) for a, k in zip(audios, kws)]
    fakes = [Fake(0), Fake(1), Fake(2)]
    m = MultiDeviceWhisperModel(models=fakes, device_index=[0, 1, 2])
    audios = [np.zeros(n, np.float32) for n in (5, 6, 7, 8, 9)]
    out = m.transcribe_batch(audios, [dict(tag=i) for i in range(5)])
    assert out == [((owner_of(i, 3), 5 + i), i) for i in range(5)]
    assert fakes[0].calls == [[5, 8]] and fakes[1].calls == [[6, 9]] and fakes[2].calls == [[7]]
    out = m.transcribe_batch(audios[:2], None, placement=[2, 2])
    assert [o[0][0] for o in out] == [2, 2]
    with pytest.raises(RuntimeError):
        m.transcribe_batch([np.zeros(13, np.float32)], None)
    m.close()


def test_multi_device_session_places_and_steps_every_device():
    """The scheduler-facing session of a multi-GPU model: streams go to the least-loaded device and stay there, the
    rounds of all devices run, every stream comes back under its own handle with the single-device result."""
    from whisperlive_b200 import synth
    from whisperlive_b200.parallel import MultiDeviceWhisperModel
    from whisperlive_b200.scheduler import BatchRequest, RoundScheduler
    torch.set_num_threads(2)
    models = [_oracle_model(), _oracle_model()]
    md = MultiDeviceWhisperModel("micro.en", device_index=[0, 1], models=models)
    waves = [synth.speech_like(3.0 + i, seed=80 + i) for i in range(3)]
    kw = dict(temperature=[0.0], log_prob_threshold=None, language="en", vad_filter=False)
    ref = models[0].transcribe_batch(waves, [kw] * 3)
    sess = md.open_session()
    h01 = sess.add_streams(waves[:2], [kw] * 2)
    sess.step_round(4)
    h2 = sess.add_streams(waves[2:], [kw])               # joins while the first two are decoding
    assert sess.placed[:2] == [0, 1] and sess.placed[2] in (0, 1)
    got, guard = {}, 0
    while sess.pending():
        sess.step_round(4)
        for e in sess.pop_finished():
            got[e.handle] = sess.result_of(e)
        guard += 1
        assert guard < 500
    for e in sess.pop_finished():
        got[e.handle] = sess.result_of(e)
    sess.close()
    for h, (segs, _info) in zip(h01 + h2, ref):
        assert [s.tokens for s in got[h][0]] == [s.tokens for s in segs]

    class Req(BatchRequest):
        def kwargs(self):
            return dict(kw)
    sch = RoundScheduler(md, max_batch_size=4, step_tokens=4)
    sch.start()
    try:
        reqs = [Req(audio=w) for w in waves]
        for r in reqs:
            sch.submit(r)
        assert all(r.future.wait(240) for r in reqs)
    finally:
        sch.stop()
        md.close()
    for r, (segs, _info) in zip(reqs, ref):
        assert r.error is None and [s.tokens for s in r.result] == [s.tokens for s in segs]


def test_bench_reference_arm_prints_the_contract_line():
    """bench.py --impl reference (the CPU arm the driver runs beside ours) works without a GPU and prints one JSON line
    with the contract's keys; a tiny architecture keeps it to seconds."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--model", "micro.en", "--steps", "1",
                          "--warmup", "0", "--cpu-seconds", "2", "--beam", "2"], capture_output=True, text=True, timeout=240)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "audio-sec/sec" and line["value"] > 0
    assert line["higher_is_better"] is True and line["steps"] == 1
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and "stand-in" in line["cpu_baseline"]["sample"]


def test_reference_batcher_runs_unmodified_on_the_b200_transcriber():
    """SURVEY.md section 8(b): the reference's own BatchInferenceWorker (batch_inference.py:193-438) over the reference's
    WhisperModel, recorded by tests/golden/run_reference_batcher.py for the batched path and the batch-of-one path: every
    attribute it read and every call the transcriber answered (encode, get_prompt, _split_segments_by_timestamps,
    transcribe) is replayed on B200WhisperModel over the same CPU oracle engine and must get the same answer -- so the
    batcher driving B200WhisperModel agrees with the reference segment for segment (tokens, times, avg_logprob,
    no_speech_prob, temperature, language)."""
    from oracle import mel as omel
    from oracle.engine import OracleWhisper
    from oracle.mel import OracleFeatureExtractor
    from tests.golden import run_reference_batcher as R
    from whisperlive_b200.config import dims_for
    from whisperlive_b200.tokenizer import Tokenizer, build_synthetic_tokenizer
    from whisperlive_b200.transcriber import B200WhisperModel
    from whisperlive_b200.weights import random_init
    torch.set_num_threads(8)
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_batcher_calls.json")))
    assert set(gold) == set(R.MODELS)
    for name, log in gold.items():
        dims = dims_for(name)
        mine = B200WhisperModel(name, engine=OracleWhisper(random_init(dims, seed=0), dims),
                                hf_tokenizer=build_synthetic_tokenizer(dims.vocab), feature_extractor=OracleFeatureExtractor(dims.n_mels))
        waves = R.audios()

        def tok(key):
            return Tokenizer(mine.hf_tokenizer, key[0], task=key[1], language=key[2])
        calls = [e.get("call") for e in log]
        assert {"encode", "get_prompt", "_split_segments_by_timestamps", "transcribe"} <= set(calls), calls
        for e in log:
            if "attr" in e:
                assert getattr(mine, e["attr"]) == e["value"], (name, e)
            elif e["call"] == "encode":
                feats = np.stack([omel.pad_or_trim(mine.feature_extractor(waves[i])) for i in e["audios"]])
                np.testing.assert_allclose(R.encoder_sample(mine.encode(feats)), e["sample"], atol=1e-4, rtol=0)
            elif e["call"] == "get_prompt":
                assert list(mine.get_prompt(tok(e["tokenizer"]), **e["kwargs"])) == e["result"], (name, e)
            elif e["call"] == "_split_segments_by_timestamps":
                got = R.split_result(mine._split_segments_by_timestamps(tokenizer=tok(e["tokenizer"]), **e["kwargs"]))
                assert got == e["result"], (name, got, e)
            else:
                segs, info = mine.transcribe(waves[e["audio"]], **e["kwargs"])
                got, ref = R.result_row(None if segs is None else list(segs), info), e["result"]
                assert ref["segments"] and got["segment_type"] == ref["segment_type"] == "Segment"
                assert [s["tokens"] for s in got["segments"]] == [s["tokens"] for s in ref["segments"]], name
                assert got["segments"] == pytest.approx(ref["segments"], abs=2e-6) and got["language"] == ref["language"]
                assert got["duration"] == pytest.approx(ref["duration"])


def test_bench_reference_arm_under_torchrun_two_ranks():
    """The driver launches the reference arm like ours for N > 1: rank 0 alone measures and prints the line, the other
    ranks exit 0 without work."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29577", os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--model", "micro.en",
           "--steps", "1", "--warmup", "0", "--cpu-seconds", "2", "--beam", "2"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=400, cwd=root)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["n_gpus"] == 2 and line["value"] > 0
