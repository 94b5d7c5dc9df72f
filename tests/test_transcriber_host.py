"""Host logic of whisperlive_b200.transcriber (SURVEY.md §8a rows H4-H8, K14 host part)
against tests/golden/transcribe_reference.json, which was produced by running the
reference's own WhisperModel orchestration over the same CPU oracle engine
(tests/golden/make_golden_transcribe.py).  The engine here is the oracle -- injected for
the test only; the product constructs the CUDA engine."""
import json
import os

import numpy as np
import pytest
import torch

from oracle.engine import OracleWhisper
from oracle.mel import OracleFeatureExtractor
from tests.golden.make_golden_transcribe import SCENARIOS, make_audio
from whisperlive_b200.config import dims_for
from whisperlive_b200.tokenizer import build_synthetic_tokenizer
from whisperlive_b200.transcriber import B200WhisperModel
from whisperlive_b200.weights import random_init

GOLD = os.path.join(os.path.dirname(__file__), "golden", "transcribe_reference.json")


def _model(sc):
    dims = dims_for(sc["model"])
    eng = OracleWhisper(random_init(dims, seed=sc["seed"]), dims)
    from tests import stub_vad
    return B200WhisperModel(sc["model"], engine=eng, hf_tokenizer=build_synthetic_tokenizer(dims.vocab),
                            feature_extractor=OracleFeatureExtractor(dims.n_mels), vad=stub_vad)


def _check(segs, gold):
    assert len(segs) == len(gold)
    for s, g in zip(segs, gold):
        assert s.id == g["id"] and s.seek == g["seek"] and s.tokens == g["tokens"] and s.text == g["text"]
        assert s.temperature == g["temperature"]
        for k in ("start", "end", "avg_logprob", "compression_ratio", "no_speech_prob"):
            assert getattr(s, k) == pytest.approx(g[k], abs=1e-6), k
        if g["words"] is None:
            assert s.words is None
        else:
            assert [(w.word, w.start, w.end) for w in s.words] == [(w["word"], w["start"], w["end"]) for w in g["words"]]
            for w, gw in zip(s.words, g["words"]):
                assert w.probability == pytest.approx(gw["probability"], abs=1e-6)


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_transcribe_matches_reference_orchestration(name):
    torch.set_num_threads(8)
    gold = json.load(open(GOLD))[name]
    sc = SCENARIOS[name]
    segs, info = _model(sc).transcribe(make_audio(sc["audio"]), **sc["kw"])
    if gold["segments"] is None:      # nothing left after VAD: (None, None) like reference :860-861
        assert segs is None and info is None
        return
    _check(segs, gold["segments"])
    if sc["kw"].get("vad_filter"):
        assert info.duration_after_vad == pytest.approx(gold["duration_after_vad"]) and info.duration_after_vad < info.duration
    assert info.language == gold["language"]
    assert float(info.language_probability) == pytest.approx(gold["language_probability"], abs=1e-6)
    assert info.duration == pytest.approx(gold["duration"])


def test_batched_equals_single():
    """transcribe_batch advances streams in lockstep; results equal per-stream transcribe."""
    torch.set_num_threads(8)
    gold = json.load(open(GOLD))
    names = ["en_two_windows_prompt_hotwords", "en_silence", "en_short_ladder"]
    m = _model(SCENARIOS[names[0]])
    res = m.transcribe_batch([make_audio(SCENARIOS[n]["audio"]) for n in names], [SCENARIOS[n]["kw"] for n in names])
    for n, (segs, info) in zip(names, res):
        _check(segs, gold[n]["segments"])


def test_empty_audio_returns_none():
    m = _model(SCENARIOS["en_silence"])
    assert m.transcribe(np.zeros(0, np.float32)) == (None, None)


# ------------------------------------------------------------------ N1: on-disk formats either side of create_model
def test_ct2_model_bin_round_trip(tmp_path):
    """model.bin writer -> reader gives back the canonical HF-named weights (fp16 rounding only); the tied output
    projection travels as an alias; k_proj biases (absent in Whisper) do not appear.  Format restated from memory of
    ctranslate2's ModelSpec._serialize -- this pins self-consistency, not agreement with a real converter."""
    import torch
    from whisperlive_b200 import ct2_format
    from whisperlive_b200.config import dims_for
    from whisperlive_b200.weights import infer_dims, load_model_dir, random_init

    dims = dims_for("micro")
    w = random_init(dims, seed=3)
    d = tmp_path / "ct2"
    d.mkdir()
    ct2_format.save_ct2_model_bin(w, str(d / "model.bin"))
    (d / "config.json").write_text('{"alignment_heads": [[1, 0], [1, 1]], "lang_ids": [5, 6], "suppress_ids": [1, 2]}')
    variables, aliases, header = ct2_format.read_variables(str(d / "model.bin"))
    assert header == {"spec": "WhisperSpec", "revision": 3, "version": 6}
    assert aliases == {"decoder/projection/weight": "decoder/embeddings/weight"}
    assert variables["encoder/layer_0/self_attention/linear_0/weight"].shape == (3 * dims.d_model, dims.d_model)
    assert variables["decoder/layer_0/attention/linear_1/weight"].shape == (2 * dims.d_model, dims.d_model)
    back = load_model_dir(str(d))
    assert set(back) == {k for k in w if not k.endswith("k_proj.bias")}
    for k, t in back.items():
        assert t.dtype == torch.float32
        torch.testing.assert_close(t, w[k].half().float(), rtol=0, atol=0)
    got = infer_dims(back, "micro-from-ct2")
    assert (got.d_model, got.enc_layers, got.dec_layers, got.n_mels, got.vocab) == \
        (dims.d_model, dims.enc_layers, dims.dec_layers, dims.n_mels, dims.vocab)
    assert ct2_format.read_ct2_config(str(d))["alignment_heads"] == [(1, 0), (1, 1)]


def test_ct2_model_bin_rejects_what_it_does_not_understand(tmp_path):
    import struct

    import numpy as np
    import pytest
    from whisperlive_b200 import ct2_format

    p = tmp_path / "model.bin"
    p.write_bytes(struct.pack("<I", 5))
    with pytest.raises(ValueError, match="binary version 5"):
        ct2_format.read_variables(str(p))
    ct2_format.write_variables(str(p), {"encoder/conv1/weight": np.zeros((2, 2, 3), np.int8)}, spec="WhisperSpec")
    with pytest.raises((ValueError, KeyError)):
        ct2_format.load_ct2_model_bin(str(p))
    ct2_format.write_variables(str(p), {"x": np.zeros((2,), np.float32)}, spec="TransformerSpec")
    with pytest.raises(ValueError, match="not a WhisperSpec"):
        ct2_format.load_ct2_model_bin(str(p))
    with open(p, "ab") as f:
        f.write(b"junk")
    with pytest.raises(ValueError, match="trailing bytes"):
        ct2_format.read_variables(str(p))


def test_window_batch_buffer_equals_pad_and_stack():
    """_stack_windows (reused per-thread buffer) gives exactly np.stack(pad_or_trim(view)) -- including after a larger
    batch left stale data in the buffer, and independently per thread."""
    import threading

    import numpy as np
    from whisperlive_b200.transcriber import pad_or_trim

    m = _model(next(iter(SCENARIOS.values())))
    n_mels = m.feature_extractor.mel_filters.shape[0] if hasattr(m.feature_extractor, "mel_filters") else 80
    rng = np.random.default_rng(0)

    def views(lengths):
        return [rng.standard_normal((n_mels, t)).astype(np.float32) for t in lengths]

    big = views([3000, 17, 1234, 2999])
    got = m._stack_windows(big).copy()
    assert got.shape == (4, n_mels, 3000) and got.flags.c_contiguous
    np.testing.assert_array_equal(got, np.stack([pad_or_trim(v, 3000) for v in big]))
    small = views([5, 300])                                  # shorter windows over the stale rows of the previous batch
    got2 = m._stack_windows(small)
    assert got2.flags.c_contiguous
    np.testing.assert_array_equal(got2, np.stack([pad_or_trim(v, 3000) for v in small]))
    other = {}
    t = threading.Thread(target=lambda: other.setdefault("buf", m._stack_windows(views([10]))))
    t.start(); t.join()
    assert not np.shares_memory(other["buf"], got2)          # a second thread never sees this thread's buffer


def test_host_helpers_match_reference_code_live():
    """Differential run against what the reference's own functions (imported with ctranslate2 / faster_whisper stubbed)
    returned on ~1400 randomised inputs, stored by tests/golden/diff_reference_host.py: timestamp splitting, prompt
    assembly, suppress list, language detection, punctuation merge, compression ratio."""
    from tests.golden import diff_reference_host as D
    from whisperlive_b200 import transcriber as ours

    torch.set_num_threads(8)
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "host_helpers_reference.json")))["cases"]
    got = D.run_cases(ours, lambda name, engine, dims: B200WhisperModel(
        name, engine=engine, hf_tokenizer=build_synthetic_tokenizer(dims.vocab), feature_extractor=OracleFeatureExtractor(dims.n_mels)))
    assert len(gold) > 1000 and [n for n, _ in got] == [n for n, _ in gold]
    bad = []
    for i, ((name, out), (_, ref)) in enumerate(zip(got, gold)):
        if name == "detect_language":
            same = out[0] == ref[0] and abs(out[1] - ref[1]) < D.APPROX[name] and [x[0] for x in out[2]] == [x[0] for x in ref[2]] \
                and all(abs(x[1] - y[1]) < D.APPROX[name] for x, y in zip(out[2], ref[2]))
        elif name == "get_compression_ratio":
            same = abs(out - ref) <= D.APPROX[name]
        else:
            same = D.digest(out) == ref
        if not same:
            bad.append((i, name, str(out)[:300]))
    assert not bad, (len(bad), bad[:10])


def test_ct2_model_bin_reads_bfloat16_payloads(tmp_path):
    """dtype id 5 (bfloat16) is widened to float32 on read; a hand-assembled record exercises that branch and aliases."""
    import struct

    import numpy as np
    from whisperlive_b200 import ct2_format

    vals = np.array([[1.0, -2.5, 0.15625], [3.0e4, -1.0e-3, 0.0]], dtype=np.float32)
    bf16 = (vals.view(np.uint32) >> 16).astype(np.uint16)          # truncation: exact for these values' top 16 bits

    def wstr(s):
        b = s.encode()
        return struct.pack("<H", len(b) + 1) + b + b"\0"

    blob = struct.pack("<I", 6) + wstr("WhisperSpec") + struct.pack("<II", 3, 1)
    blob += wstr("decoder/embeddings/weight") + struct.pack("<B", 2) + struct.pack("<II", 2, 3) + struct.pack("<BI", 5, bf16.nbytes)
    blob += bf16.tobytes() + struct.pack("<I", 1) + wstr("decoder/projection/weight") + wstr("decoder/embeddings/weight")
    p = tmp_path / "model.bin"
    p.write_bytes(blob)
    variables, aliases, header = ct2_format.read_variables(str(p))
    got = variables["decoder/embeddings/weight"]
    assert got.dtype == np.float32 and got.shape == (2, 3)
    expect = (bf16.astype(np.uint32) << 16).view(np.float32).reshape(2, 3)
    np.testing.assert_array_equal(got, expect)
    assert abs(got[0, 1] + 2.5) < 1e-6 and aliases == {"decoder/projection/weight": "decoder/embeddings/weight"}


def test_decode_audio_wav_flac_and_paths(tmp_path):
    """``transcribe`` takes a path / file object like the reference (``decode_audio``, transcriber_faster_whisper.py:820-821):
    RIFF/WAVE PCM and FLAC are decoded natively (the FLAC decoder checks the STREAMINFO MD5), resampled to 16 kHz mono;
    other containers raise with the magic named."""
    import wave

    from whisperlive_b200.audio import decode_audio, decode_flac, resample
    rng = np.random.default_rng(5)
    # stereo 8 kHz 16-bit WAV -> mono 16 kHz
    t = np.arange(8000) / 8000.0
    left, right = 0.4 * np.sin(2 * np.pi * 220 * t), 0.2 * np.sin(2 * np.pi * 330 * t)
    inter = np.stack([left, right], axis=1)
    p = tmp_path / "a.wav"
    with wave.open(str(p), "wb") as w:
        w.setnchannels(2); w.setsampwidth(2); w.setframerate(8000)
        w.writeframes(np.round(inter * 32767).astype("<i2").tobytes())
    y = decode_audio(str(p))
    assert y.dtype == np.float32 and y.shape == (16000,)
    ref = resample((np.round(inter * 32767) / 32768.0).mean(axis=1), 8000, 16000)
    assert np.abs(y - ref).max() < 1e-6
    with open(p, "rb") as f:
        assert np.array_equal(decode_audio(f), y)            # file object
    assert np.array_equal(decode_audio(p.read_bytes()), y)    # bytes
    assert resample(left, 16000, 16000).shape == left.shape
    with pytest.raises(ValueError, match="unsupported container"):
        decode_audio(b"OggS" + bytes(64))
    # the head of the reference's asset: decoded FLAC == the committed fixture (to the fixture's int16 rounding, away from
    # the cut where the resampling filter runs off the end); a flipped byte is caught
    src = os.path.join(os.path.dirname(__file__), "golden", "jfk_head.flac")
    fx = np.load(os.path.join(os.path.dirname(__file__), "golden", "jfk_16k_i16.npy")).astype(np.float32) / 32768.0
    y = decode_audio(src)
    n = len(y) - 64
    assert len(y) == -(-46080 * 160 // 441) and np.abs(y[:n] - fx[:n]).max() <= 0.5 / 32768 + 1e-7
    data = bytearray(open(src, "rb").read())
    data[len(data) // 2] ^= 0x10
    with pytest.raises(Exception):
        decode_flac(bytes(data))
    # through the transcriber: a path gives what the samples give
    from tests.test_boundary_cpu import _oracle_model
    from whisperlive_b200 import synth
    model = _oracle_model()
    wav16 = synth.speech_like(3.0, seed=3)
    q = tmp_path / "b.wav"
    with wave.open(str(q), "wb") as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(16000)
        w.writeframes(np.round(wav16 * 32768).clip(-32768, 32767).astype("<i2").tobytes())
    kw = dict(temperature=[0.0], beam_size=2, log_prob_threshold=None, max_new_tokens=12, language="en")
    a_segs, a_info = model.transcribe(str(q), **kw)
    b_segs, _ = model.transcribe(decode_audio(str(q)), **kw)
    assert a_info.duration == pytest.approx(3.0) and [s.tokens for s in a_segs] == [s.tokens for s in b_segs]
