"""Record how ServeClientB200 and the original project's ServeClientBase (whisper_live/backend/base.py) talk to each other
into tests/golden/plugin_base_calls.json, and replay that record without the original package.

The plugin subclasses ServeClientBase: the base's ``speech_to_text`` loop hands audio chunks to the plugin's
``transcribe_audio`` and the result to ``handle_transcription_output``, which calls back into the base
(``update_segments``, ``prepare_segments``, ``send_transcription_to_client``).  Run as a script with the original
checkout, the plugin runs on the real base over the CPU oracle engine (one 3 s chunk, until the first segments are
sent) and every crossing of that boundary is logged with its arguments and answers.  ``replay_module`` builds a
stand-in ``whisper_live.backend.base`` from the log: its loop makes the same calls into the plugin, its methods check
the plugin's calls against the log and answer with what the real base answered.  tests/test_boundary_cpu.py runs the
plugin on it.

    python tests/golden/record_plugin_base.py <original project checkout>
"""
import functools
import json
import os
import sys
import threading
import time
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, "..", ".."))
sys.path.insert(0, ROOT)

GOLD = os.path.join(HERE, "plugin_base_calls.json")
CLIENT = dict(client_uid="u1", model="micro.en", use_vad=False, no_speech_thresh=1.1)
# keep the CPU oracle cheap: the plugin's requests carry the reference defaults (beam 5, six-rung temperature ladder,
# up to 224 new tokens), which is tens of seconds per chunk on the oracle and trips the plugin's 30 s request timeout
CHEAP = dict(temperature=[0.0], beam_size=2, log_prob_threshold=None, max_new_tokens=24)


def wave():
    from whisperlive_b200 import synth
    return synth.speech_like(3.0, seed=1)


def oracle_model():
    from oracle.engine import OracleWhisper
    from oracle.mel import OracleFeatureExtractor
    from whisperlive_b200.config import dims_for
    from whisperlive_b200.tokenizer import build_synthetic_tokenizer
    from whisperlive_b200.transcriber import B200WhisperModel
    from whisperlive_b200.weights import random_init
    dims = dims_for("micro.en")
    return B200WhisperModel("micro.en", engine=OracleWhisper(random_init(dims, seed=0), dims),
                            hf_tokenizer=build_synthetic_tokenizer(dims.vocab), feature_extractor=OracleFeatureExtractor(dims.n_mels))


class WS:
    def __init__(self):
        self.sent, self.closed = [], False

    def send(self, msg):
        self.sent.append(json.loads(msg))

    def close(self):
        self.closed = True


def rows(result):
    """The transcriber's segments as the base reads them."""
    return None if result is None else [dict(start=float(s.start), end=float(s.end), text=s.text, tokens=list(s.tokens),
                                             no_speech_prob=float(s.no_speech_prob)) for s in result]


def plain(x):
    return json.loads(json.dumps(x))


def init_args(args) -> list:
    """super().__init__ arguments after (client_uid, websocket): send_last_n_segments, no_speech_thresh, clip_audio,
    same_output_threshold, translation_queue, diarization, word_timestamps (queue / diarizer: whether given)."""
    a = list(args[2:])
    return a[:4] + [a[4] is not None, a[5] is not None] + a[6:]


def same(got, ref, tol=1e-5) -> bool:
    if isinstance(ref, dict):
        return isinstance(got, dict) and set(got) == set(ref) and all(same(got[k], ref[k], tol) for k in ref)
    if isinstance(ref, list):
        return isinstance(got, list) and len(got) == len(ref) and all(same(g, r, tol) for g, r in zip(got, ref))
    if isinstance(ref, float) and not isinstance(got, bool):
        return isinstance(got, (int, float)) and abs(got - ref) <= tol
    return got == ref


def replay_module(rec):
    """A ``whisper_live.backend.base`` module whose ServeClientBase replays ``rec``; the class collects mismatches in
    ``ServeClientBase.mismatches`` and sets ``ServeClientBase.done`` when the record is used up."""
    mod = types.ModuleType("whisper_live.backend.base")
    audio = wave()

    class ServeClientBase:
        mismatches = []
        done = threading.Event()

        def __init__(self, client_uid, websocket, *args):
            self.client_uid, self.websocket = client_uid, websocket
            self.word_timestamps = args[-1]
            self.exit = False
            if [client_uid] + init_args((None, None) + args) != rec["init"]:
                self.mismatches.append(("__init__", [client_uid] + init_args((None, None) + args)))
            self._expect = [e for e in rec["events"] if "to_base" in e]

        def _check(self, name, **got):
            e = self._expect.pop(0) if self._expect else {"to_base": None}
            if e["to_base"] != name or not all(same(plain(v), e[k]) for k, v in got.items()):
                self.mismatches.append((name, str(got)[:500], str(e)[:500]))
            return e.get("returns")

        def speech_to_text(self):
            try:
                for e in rec["events"]:
                    if self.exit:
                        return
                    if e.get("to_plugin") == "transcribe_audio":
                        result = self.transcribe_audio(audio[e["offset"]:e["offset"] + e["length"]].copy())
                        if not same(rows(result), e["result"]):
                            self.mismatches.append(("transcribe_audio", str(rows(result))[:500], str(e["result"])[:500]))
                    elif e.get("to_plugin") == "handle_transcription_output":
                        self.handle_transcription_output(result, e["duration"])
                if self._expect:
                    self.mismatches.append(("calls into the base never made", self._expect))
            except Exception as ex:
                self.mismatches.append(("exception", repr(ex)))
            finally:
                self.done.set()

        def update_segments(self, segments, duration):
            return self._check("update_segments", segments=rows(segments), duration=duration)

        def prepare_segments(self, last_segment=None):
            return self._check("prepare_segments", last_segment=last_segment)

        def send_transcription_to_client(self, segments):
            self._check("send_transcription_to_client", segments=segments)

    for k, v in rec["class_attrs"].items():
        setattr(ServeClientBase, k, v)
    mod.ServeClientBase = ServeClientBase
    return mod


def main():
    sys.path.insert(0, os.path.abspath(sys.argv[1]))
    import torch
    from whisper_live.backend import base
    from whisperlive_b200.backend import ServeClientB200
    from whisperlive_b200.scheduler import BatchRequest
    torch.set_num_threads(8)
    B = base.ServeClientBase
    audio = wave()
    rec = {"init": None, "events": [], "class_attrs": {"SERVER_READY": B.SERVER_READY, "RATE": B.RATE}}

    def on_base(name, fn):
        @functools.wraps(fn)
        def w(self, *a, **k):
            out = fn(self, *a, **k)
            if name == "update_segments":
                e = dict(segments=rows(a[0]), duration=a[1])
            elif name == "prepare_segments":
                e = dict(last_segment=a[0] if a else k.get("last_segment"))
            else:
                e = dict(segments=a[0])
                self.exit = True                     # the first segments sent end the recording
            rec["events"].append(dict(to_base=name, **plain(e), returns=plain(out)))
            return out
        return w

    def on_plugin(name, fn):
        @functools.wraps(fn)
        def w(self, *a):
            if name == "transcribe_audio":
                x = a[0]
                off = next(i for i in range(len(audio) - len(x) + 1) if np.array_equal(audio[i:i + len(x)], x))
                out = fn(self, *a)
                rec["events"].append(dict(to_plugin=name, offset=off, length=len(x), result=rows(out)))
                return out
            rec["events"].append(dict(to_plugin=name, duration=a[1]))
            return fn(self, *a)
        return w

    real_init = B.__init__

    def init(self, *a, **k):
        rec["init"] = [a[0]] + init_args(a)
        real_init(self, *a, **k)
    B.__init__ = init
    for n in ("update_segments", "prepare_segments", "send_transcription_to_client"):
        setattr(B, n, on_base(n, getattr(B, n)))
    for n in ("transcribe_audio", "handle_transcription_output"):
        setattr(ServeClientB200, n, on_plugin(n, getattr(ServeClientB200, n)))
    orig_kwargs = BatchRequest.kwargs
    BatchRequest.kwargs = lambda self: dict(orig_kwargs(self), **CHEAP)
    model = oracle_model()
    ServeClientB200.MODEL_FACTORY = lambda name: model
    ws = WS()
    try:
        client = ServeClientB200(ws, **CLIENT)
        client.add_frames(audio)
        deadline = time.time() + 120
        while time.time() < deadline and not any("segments" in m for m in ws.sent):
            time.sleep(0.1)
        client.exit = True
        client.trans_thread.join(timeout=30)
    finally:
        ServeClientB200.shutdown()
    assert any("segments" in m for m in ws.sent), ws.sent
    rec["sent"] = ws.sent
    with open(GOLD, "w") as f:
        json.dump(rec, f, indent=1)
        f.write("\n")
    print("wrote", GOLD, [e.get("to_base") or e.get("to_plugin") for e in rec["events"]])


if __name__ == "__main__":
    main()
