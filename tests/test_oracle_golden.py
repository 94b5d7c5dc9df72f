"""The oracle against the committed golden vectors (CPU).

mel_reference.npz   <- reference's in-repo mel code (tests/golden/make_golden_mel.py)
model_hf.npz        <- HF transformers Whisper (tests/golden/make_golden_model.py)
"""
import os

import numpy as np
import pytest
import torch

from oracle import mel as omel
from oracle import model as om
from whisperlive_b200 import synth
from whisperlive_b200.config import dims_for
from whisperlive_b200.weights import random_init

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_mel_oracle_matches_reference_formula():
    g = np.load(os.path.join(GOLD, "mel_reference.npz"))
    keys = [k for k in g.files if not k.startswith("wav__")]
    assert len(keys) == 10
    for k in keys:
        name, n_mels = k.split("__")
        out = omel.log_mel(g["wav__" + name], int(n_mels))
        assert out.shape == g[k].shape and out.dtype == np.float32
        # fp32 FFT implementations differ in the last bits; log-mel units
        np.testing.assert_allclose(out, g[k], atol=5e-5, rtol=0)


def test_mel_filterbank_matches_hf():
    from transformers.audio_utils import mel_filter_bank
    for n in (80, 128):
        hf = mel_filter_bank(num_frequency_bins=201, num_mel_filters=n, min_frequency=0.0, max_frequency=8000.0,
                             sampling_rate=16000, norm="slaney", mel_scale="slaney").T
        np.testing.assert_allclose(omel.slaney_mel_filters(n), hf.astype(np.float32), atol=1e-7)


def test_mel_shapes_and_padding():
    for n in (1600, 16000, 17001, 480000):
        f = omel.log_mel(np.zeros(n, np.float32), 80)
        assert f.shape == (80, n // 160 + 1)
    f = omel.pad_or_trim(np.ones((80, 10), np.float32))
    assert f.shape == (80, 3000) and f[:, 10:].sum() == 0  # zero padding in feature space
    assert omel.pad_or_trim(np.ones((80, 3100), np.float32)).shape == (80, 3000)


@pytest.mark.parametrize("name", ["micro.en", "tiny"])
def test_network_oracle_matches_hf(name):
    g = np.load(os.path.join(GOLD, "model_hf.npz"))
    dims = dims_for(name)
    w = random_init(dims, seed=int(g[name + "__init_seed"][0]))
    wav = synth.speech_like(7.3, seed=int(g[name + "__wav_seed"][0]))
    feats = omel.pad_or_trim(omel.log_mel(wav, dims.n_mels)[:, :-1])
    with torch.no_grad():
        enc = om.encoder_forward(w, torch.from_numpy(feats)[None], dims.n_heads, dims.enc_layers)
        xkv = om.cross_kv(w, enc, dims.n_heads, dims.dec_layers)
        toks = torch.from_numpy(g[name + "__tokens"])
        logits = om.decoder_forward(w, toks, xkv, om.DecoderState(dims.dec_layers), dims.n_heads, dims.dec_layers)
        st = om.DecoderState(dims.dec_layers)
        inc = torch.cat([om.decoder_forward(w, toks[:, i:i + 1], xkv, st, dims.n_heads, dims.dec_layers)
                         for i in range(toks.shape[1])], 1)
    np.testing.assert_allclose(enc[0, ::25].numpy(), g[name + "__enc_sub"], atol=2e-4)
    np.testing.assert_allclose(logits[0, :, :512].numpy(), g[name + "__logits_head"], atol=5e-4)
    np.testing.assert_allclose(logits[0, :, -1700:].numpy(), g[name + "__logits_tail"], atol=5e-4)
    np.testing.assert_allclose(torch.logsumexp(logits[0], -1).numpy(), g[name + "__logits_lse"], atol=5e-4)
    # KV-cached incremental decoding == full teacher-forced pass
    np.testing.assert_allclose(inc.numpy(), logits.numpy(), atol=2e-4)


def test_timestamp_rules_match_transformers_port():
    """oracle/search.py::apply_processors (suppress list, suppress-blank, timestamp rules a-e, log-softmax) against
    transformers' WhisperTimeStampLogitsProcessor + SuppressTokens(AtBegin)LogitsProcessor -- an independent port of
    OpenAI whisper's ApplyTimestampRules, the same rule set CTranslate2's models/whisper.cc ports.  CTranslate2 itself is
    not available offline, so this is the closest executable anchor for the logits rules (the beam search proper stays
    unpinned).  600 random histories (valid and invalid ones: both sides are pure functions of the history)."""
    from types import SimpleNamespace

    from transformers.generation.logits_process import (SuppressTokensAtBeginLogitsProcessor, SuppressTokensLogitsProcessor,
                                                        WhisperTimeStampLogitsProcessor)

    from oracle.search import GenOptions, VocabSpec, apply_processors

    rng = np.random.default_rng(7)
    for vocab in (51864, 51866):
        spec = VocabSpec.from_vocab_size(vocab)
        tb = spec.timestamp_begin
        begin = 3
        cfg = SimpleNamespace(no_timestamps_token_id=spec.no_timestamps, eos_token_id=spec.eot, bos_token_id=spec.eot,
                              max_initial_timestamp_index=50, _detect_timestamp_from_logprob=True)
        ts_proc = WhisperTimeStampLogitsProcessor(cfg, begin_index=begin)
        for case in range(300):
            n = int(rng.choice([0, 0, 1, 2, 3, 6, 15]))
            gen = [int(tb + rng.integers(0, 1200)) if rng.random() < 0.4 else int(rng.integers(0, spec.eot)) for _ in range(n)]
            if n >= 2 and rng.random() < 0.3:
                gen[-1] = gen[-2] if gen[-2] >= tb else int(tb + rng.integers(0, 1200))     # closed timestamp pair
            logits = torch.from_numpy((3.0 * rng.standard_normal(vocab)).astype(np.float32))
            if rng.random() < 0.3:
                logits[tb:] += 4.0                                                          # make rule e fire sometimes
            suppress = sorted(set(int(t) for t in rng.integers(0, vocab, int(rng.choice([0, 0, 5, 90])))))
            blank = bool(rng.random() < 0.5)
            opts = GenOptions(beam_size=1, suppress_blank=blank, suppress_tokens=suppress, max_initial_timestamp_index=50)
            mine = apply_processors(logits, gen, spec, opts, True)
            ids = torch.tensor([[spec.sot, spec.sot + 1, spec.sot + 2][:begin] + gen])
            x = logits[None].clone()
            if suppress:
                x = SuppressTokensLogitsProcessor(suppress, device="cpu")(ids, x)
            if blank:
                x = SuppressTokensAtBeginLogitsProcessor([spec.blank, spec.eot], begin, device="cpu")(ids, x)
            ref = torch.log_softmax(ts_proc(ids, x)[0], dim=-1)
            m_inf, r_inf = torch.isinf(mine), torch.isinf(ref)
            assert torch.equal(m_inf, r_inf), (vocab, case, gen, int((m_inf != r_inf).sum()))
            assert torch.allclose(mine[~m_inf], ref[~r_inf], atol=1e-5), (vocab, case)


def test_alignment_helpers_match_transformers_port():
    """oracle/align.py median filter and DTW against transformers' `_median_filter` / `_dynamic_time_warping` (ports of
    OpenAI whisper/timing.py, which CTranslate2's align also follows): identical outputs, ties included."""
    from transformers.models.whisper.generation_whisper import _dynamic_time_warping, _median_filter

    from oracle.align import dtw_path, median_filter_time

    rng = np.random.default_rng(11)
    for _ in range(40):
        n, m = int(rng.integers(1, 24)), int(rng.integers(1, 70))
        cost = rng.standard_normal((n, m)).astype(np.float32)
        if rng.random() < 0.4:
            cost = np.round(cost, 0)                  # plenty of exact ties: the tie-breaking order must agree too
        a_t, a_f = dtw_path(cost)
        b_t, b_f = _dynamic_time_warping(cost.astype(np.float64))
        assert a_t.tolist() == b_t.tolist() and a_f.tolist() == b_f.tolist(), (n, m)
    for width in (3, 7):
        for t in (1, 2, 3, 4, 9, 150):
            x = rng.standard_normal((2, 5, t)).astype(np.float32)
            ref = _median_filter(torch.from_numpy(x), width).numpy()
            np.testing.assert_array_equal(median_filter_time(x, width), ref)


def test_alignment_pipeline_matches_transformers_order():
    """oracle/align.py::alignment_from_attention (slice the softmaxed weights to num_frames // 2, standardise over the token
    axis, median filter, mean over heads, DTW on the negated matrix without the start sequence and <eot>) step for step
    against the same pipeline assembled from transformers' helpers in the order of
    WhisperGenerationMixin._extract_token_timestamps."""
    from transformers.models.whisper.generation_whisper import _dynamic_time_warping, _median_filter

    from oracle.align import alignment_from_attention

    rng = np.random.default_rng(13)
    for _ in range(12):
        heads, n_tok, n_start = int(rng.integers(1, 7)), int(rng.integers(6, 30)), int(rng.integers(1, 5))
        num_frames = int(rng.integers(40, 3000))
        logits = rng.standard_normal((heads, n_tok, 1500)).astype(np.float32) * 2.0
        attn = torch.softmax(torch.from_numpy(logits), dim=-1).numpy()
        got = alignment_from_attention(attn, n_start, num_frames, 7)
        w = torch.from_numpy(attn)[None][..., : num_frames // 2]            # [batch, heads, tokens, frames]
        std = torch.std(w, dim=-2, keepdim=True, unbiased=False)
        mean = torch.mean(w, dim=-2, keepdim=True)
        w = _median_filter((w - mean) / std, 7).mean(dim=1)[0]
        ti, fi = _dynamic_time_warping(-w[n_start:-1].double().numpy())
        assert got == list(zip(ti.tolist(), fi.tolist()))


def test_jfk_fixture_is_the_reference_asset():
    """tests/golden/jfk_16k_i16.npy = the original project's assets/jfk.flac (input of its WER test, tests/test_server.py:
    92-118; BASELINE config 1) decoded by the self-checking FLAC decoder of make_golden_jfk.py (STREAMINFO MD5 verified) and
    resampled to 16 kHz mono: 176 000 samples = 11.0 s.  The oracle's K1 on it has the reference feature geometry.  The
    first 10 frames of that FLAC file (tests/golden/jfk_head.flac, make_jfk_head.py) go through the same recipe and must
    give the fixture's first samples exactly (the last few are left out: the resampling filter sees the cut there)."""
    pcm = np.load(os.path.join(GOLD, "jfk_16k_i16.npy"))
    assert pcm.dtype == np.int16 and pcm.shape == (176000,)
    assert 20000 < int(np.abs(pcm).max()) < 32768
    mel = omel.log_mel(pcm.astype(np.float32) / 32768.0, 80)
    assert mel.shape == (80, 1101) and np.isfinite(mel).all()
    assert float(mel.max() - mel.min()) <= 2.0 + 1e-6          # (clamp to max - 8, + 4) / 4 -> a dynamic range of at most 2
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden_jfk", os.path.join(GOLD, "make_golden_jfk.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    raw, info = mod.decode_flac(open(os.path.join(GOLD, "jfk_head.flac"), "rb").read())
    assert raw.shape == (2, 46080) and info["rate"] == 44100 and info["bps"] == 24
    from scipy.signal import resample_poly
    mono = raw.astype(np.float64).mean(axis=0) / float(1 << 23)
    y = np.clip(np.round(resample_poly(mono, 160, 441) * 32768.0), -32768, 32767).astype(np.int16)
    n = len(y) - 64
    assert n > 16000
    np.testing.assert_array_equal(y[:n], pcm[:n])
