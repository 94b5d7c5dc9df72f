"""Record what the original project's OWN cross-stream batcher (whisper_live/batch_inference.py
BatchInferenceWorker._process_multi / _process_single, :193-438) asks of the transcriber it drives, and what the original
project's WhisperModel answers, into tests/golden/reference_batcher_calls.json.

The drop-in claim of SURVEY.md section 8(b) is that everything the batcher reads from the transcriber
(feature_extractor, encode, model.generate / detect_language / is_multilingual, hf_tokenizer, get_prompt, max_length,
frames_per_second, _split_segments_by_timestamps, transcribe) exists on whisperlive_b200.transcriber.B200WhisperModel
with the original's meaning.  The batcher runs once, over the original WhisperModel wrapped in a recorder; the engine
underneath is the CPU oracle and ctranslate2 / faster_whisper are stubbed exactly as in make_golden_transcribe.py.  The
recorder logs the plain attributes read and every call answered by the transcriber's own code (the engine is shared by
both sides, so model.generate / detect_language are not transcriber code): tests/test_boundary_cpu.py replays each call
on B200WhisperModel over the same engine and requires the same answers, and with them the batcher's results would be the
same segment for segment.

    python tests/golden/run_reference_batcher.py <original project checkout>
"""
import functools
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, "..", ".."))
sys.path.insert(0, ROOT)

from tests.golden import make_golden_transcribe as G  # noqa: E402
from oracle import mel as omel  # noqa: E402
from oracle.engine import OracleWhisper  # noqa: E402
from whisperlive_b200 import synth  # noqa: E402
from whisperlive_b200.config import dims_for  # noqa: E402
from whisperlive_b200.weights import random_init  # noqa: E402

GOLD = os.path.join(HERE, "reference_batcher_calls.json")
MODELS = ("micro.en", "micro")


def audios():
    return [synth.speech_like(6.0, seed=1), synth.speech_like(3.0, seed=2), synth.speech_like(9.5, seed=3)]


def encoder_sample(enc) -> list:
    """A fixed sub-grid of the encoder output: [stream][frame::100][channel::16]."""
    return np.asarray(enc, dtype=np.float32)[:, ::100, ::16].tolist()


def tokenizer_key(tok) -> list:
    """What the batcher builds its Tokenizer from: (multilingual, task, language)."""
    if tok.task is None:
        return [False, None, None]
    return [True, tok.tokenizer.id_to_token(tok.task).strip("<|>"), tok.language_code]


def split_result(r) -> list:
    return [[{k: (float(v) if isinstance(v, (float, np.floating)) else v) for k, v in s.items()} for s in r[0]], int(r[1]),
            bool(r[2])]


def result_row(segs, info) -> dict:
    """Segments and info the way the batcher hands them on, rounded to 6 decimals."""
    return dict(segments=None if segs is None else [dict(
        tokens=list(s.tokens), start=round(float(s.start), 6), end=round(float(s.end), 6), text=s.text,
        avg_logprob=round(float(s.avg_logprob), 6), no_speech_prob=round(float(s.no_speech_prob), 6), temperature=s.temperature,
        compression_ratio=round(float(s.compression_ratio), 6)) for s in segs],
        segment_type=None if not segs else type(segs[0]).__name__,
        language=getattr(info, "language", None), duration=round(float(getattr(info, "duration", -1.0)), 6))


class Recorder:
    """Forwards everything to the wrapped transcriber and logs what the batcher asked and got."""

    def __init__(self, inner, waves):
        self.__dict__.update(_inner=inner, log=[],
                             _padded=[omel.pad_or_trim(inner.feature_extractor(w)) for w in waves], _waves=waves)

    def __getattr__(self, name):
        v = getattr(self._inner, name)
        if name in ("encode", "get_prompt", "_split_segments_by_timestamps", "transcribe"):
            return functools.partial(getattr(self, "_rec" + name.lstrip("_")), v)
        if isinstance(v, (bool, int, float, str)):
            self.log.append(dict(attr=name, value=v))
        return v

    def _recencode(self, fn, features):
        idx = [next(i for i, p in enumerate(self._padded) if np.array_equal(p, f)) for f in features]
        out = fn(features)
        self.log.append(dict(call="encode", audios=idx, sample=encoder_sample(out)))
        return out

    def _recget_prompt(self, fn, tokenizer, **kw):
        out = fn(tokenizer, **kw)
        self.log.append(dict(call="get_prompt", tokenizer=tokenizer_key(tokenizer), kwargs=kw, result=list(out)))
        return out

    def _recsplit_segments_by_timestamps(self, fn, tokenizer, **kw):
        out = fn(tokenizer=tokenizer, **kw)
        self.log.append(dict(call="_split_segments_by_timestamps", tokenizer=tokenizer_key(tokenizer),
                             kwargs=dict(kw, tokens=list(kw["tokens"])), result=split_result(out)))
        return out

    def _rectranscribe(self, fn, audio, **kw):
        segs, info = fn(audio, **kw)
        segs = None if segs is None else list(segs)
        idx = next(i for i, w in enumerate(self._waves) if w is audio)
        self.log.append(dict(call="transcribe", audio=idx, kwargs=kw, result=result_row(segs, info)))
        return segs, info


def main():
    G.install_stubs()
    sys.path.insert(0, os.path.abspath(sys.argv[1]))
    from whisper_live import batch_inference as ref_bi
    from whisper_live.transcriber import transcriber_faster_whisper as ref_tr

    out = {}
    for model_name in MODELS:
        dims = dims_for(model_name)
        engine = OracleWhisper(random_init(dims, seed=0), dims)
        rec = Recorder(G.reference_model(ref_tr, engine, dims), audios())
        worker = ref_bi.BatchInferenceWorker(rec, max_batch_size=4, batch_window_ms=1)
        lang = None if dims.multilingual else "en"
        reqs = [ref_bi.BatchRequest(audio=a, language=lang, use_vad=False, initial_prompt="hello" if i == 1 else None)
                for i, a in enumerate(rec._waves)]
        worker._process_multi(reqs)          # the batched path, called synchronously (no thread needed)
        single = ref_bi.BatchRequest(audio=rec._waves[0], language=lang, use_vad=False)
        worker._process_single(single)       # batch of one: delegates to transcriber.transcribe()
        for r in reqs + [single]:
            assert r.error is None and r.future.is_set() and r.result, (model_name, r.error)
        out[model_name] = rec.log
    with open(GOLD, "w") as f:
        json.dump(out, f, indent=0)
        f.write("\n")
    print("wrote", GOLD, {k: len(v) for k, v in out.items()})


if __name__ == "__main__":
    main()
