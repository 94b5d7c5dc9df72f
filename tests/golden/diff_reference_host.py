"""Differential check of the host-side helpers against the original project's own Python, on randomised inputs.

``run_cases`` calls, on ~1400 inputs drawn from a fixed seed, either the original project's
whisper_live/transcriber/transcriber_faster_whisper.py or whisperlive_b200.transcriber:
    _split_segments_by_timestamps (:970-1047)   get_prompt (:1480-1513)
    get_suppressed_tokens (:1831-1853)          merge_punctuations (:1856-1887)      get_compression_ratio (:1826-1828)
    detect_language (:1716-1789, multilingual model: first-segment threshold and majority vote)
Run as a script with the original project's checkout, it imports that module with the same sys.modules stubs as
make_golden_transcribe.py (in its own process: the stubs must not leak into pytest) and writes what it returned to
tests/golden/host_helpers_reference.json: the first 16 hex digits of the SHA-1 of each output that
tests/test_transcriber_host.py compares exactly, the value itself for the two helpers compared with a tolerance.

    python tests/golden/diff_reference_host.py <original project checkout>
"""
import copy
import hashlib
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, "..", ".."))
sys.path.insert(0, ROOT)

from oracle.engine import OracleWhisper  # noqa: E402
from whisperlive_b200 import tokenizer as wtok  # noqa: E402
from whisperlive_b200.config import dims_for  # noqa: E402
from whisperlive_b200.weights import random_init  # noqa: E402

GOLD = os.path.join(HERE, "host_helpers_reference.json")
APPROX = {"detect_language": 1e-6, "get_compression_ratio": 1e-12}    # compared with this tolerance, the rest exactly


def _plain(x):
    if hasattr(x, "item"):
        return x.item()
    if isinstance(x, (tuple, set)):
        return list(x)
    raise TypeError(type(x))


def digest(x) -> str:
    return hashlib.sha1(json.dumps(x, sort_keys=True, default=_plain).encode()).hexdigest()[:16]


def run_cases(mod, make_model):
    """[(helper name, output)] of ``mod``'s helpers on the fixed inputs; ``make_model(name, engine, dims)`` builds the
    transcriber whose methods are called."""
    rnd = random.Random(20260922)
    out = []
    for model_name in ("micro.en", "micro"):
        dims = dims_for(model_name)
        engine = OracleWhisper(random_init(dims, seed=0), dims)
        m = make_model(model_name, engine, dims)
        tok = wtok.Tokenizer(wtok.build_synthetic_tokenizer(dims.vocab), dims.multilingual,
                             task="transcribe" if dims.multilingual else None, language="en" if dims.multilingual else None)
        tb = tok.timestamp_begin
        # ---- _split_segments_by_timestamps: random mixes of text and timestamp tokens, all edge shapes
        for _ in range(400):
            L = rnd.choice([0, 1, 2, 3, 5, 9, 17, 40])
            toks, ts = [], tb + rnd.randrange(0, 50)
            for _i in range(L):
                r = rnd.random()
                if r < 0.35:
                    ts += rnd.randrange(0, 40)
                    toks.append(min(ts, tb + 1500))
                else:
                    toks.append(rnd.randrange(0, min(tb, 50000)))
            if L and rnd.random() < 0.3:
                toks.append(toks[-1] if toks[-1] >= tb else tb + rnd.randrange(0, 1500))
            args = (rnd.choice([0.0, 30.0, 12.34]), rnd.choice([3000, 1234, 17]), rnd.choice([30.0, 12.34, 0.17]),
                    rnd.choice([0, 3000, 777]))
            if not toks:
                continue
            a = m._split_segments_by_timestamps(tok, list(toks), *args)
            out.append(("split", [list(a[0]), a[1], bool(a[2])]))
        # ---- get_prompt
        for _ in range(200):
            prev = [rnd.randrange(0, 50000) for _i in range(rnd.choice([0, 0, 3, 50, 223, 224, 300]))]
            kw = dict(without_timestamps=rnd.random() < 0.5, prefix=rnd.choice([None, None, "hello there", " world"]),
                      hotwords=rnd.choice([None, None, "foo bar", "x" * 400]))
            out.append(("get_prompt", list(m.get_prompt(tok, list(prev), **kw))))
        # ---- get_suppressed_tokens
        for sup in ([-1], [], [-1, 5, 7], [11, 12], [-1, tok.eot]):
            a = mod.get_suppressed_tokens(tok, sup)
            out.append(("get_suppressed_tokens", None if a is None else list(a)))
        # ---- detect_language wrapper (:1716-1789): threshold hit on the first segment, and the majority-vote path
        if dims.multilingual:
            from whisperlive_b200 import synth
            for sec, nseg, thr in ((7.0, 1, 0.5), (41.0, 2, 0.999), (65.0, 3, 0.0)):
                audio = synth.speech_like(sec, seed=int(sec))
                a = m.detect_language(audio=audio, language_detection_segments=nseg, language_detection_threshold=thr)
                out.append(("detect_language", [a[0], float(a[1]), [[x[0], float(x[1])] for x in a[2]]]))
    # ---- merge_punctuations / get_compression_ratio (tokenizer independent)
    words = ["hello", " world", " \"", "quoted", ",", " and", " (", "paren", ")", ".", " ¿", "que", "?", " -", "dash", "!"]
    for _ in range(300):
        al = []
        for _i in range(rnd.randrange(0, 12)):
            w = rnd.choice(words)
            al.append(dict(word=w, tokens=[rnd.randrange(0, 1000) for _j in range(rnd.randrange(1, 3))],
                           start=rnd.random(), end=rnd.random(), probability=rnd.random()))
        a = copy.deepcopy(al)
        mod.merge_punctuations(a, "\"'“¿([{-", "\"'.。,，!！?？:：”)]}、")
        out.append(("merge_punctuations", a))
    for s in ("a", "aaaaaaaaaaaaaaaaaaaaaaaa", "the quick brown fox", "ab" * 200, "héllo wörld " * 7):
        out.append(("get_compression_ratio", float(mod.get_compression_ratio(s))))
    return out


def main():
    from tests.golden import make_golden_transcribe as G
    G.install_stubs()
    sys.path.insert(0, os.path.abspath(sys.argv[1]))
    from whisper_live.transcriber import transcriber_faster_whisper as ref

    cases = run_cases(ref, lambda name, engine, dims: G.reference_model(ref, engine, dims))
    rows = [[name, out] if name in APPROX else [name, digest(out)] for name, out in cases]
    with open(GOLD, "w") as f:
        f.write('{"cases": [\n' + ",\n".join(json.dumps(r) for r in rows) + "\n]}\n")
    print("wrote", GOLD, len(rows), "cases")


if __name__ == "__main__":
    main()
