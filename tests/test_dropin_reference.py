"""Drop-in test through the reference's OWN orchestration code (SURVEY.md section 7 step 2, section 8b).

`do_whisper` and `do_translate` of the reference's main.py (main.py:91-94, 514-547, 554-770) were run with
  ctranslate2            := willow_inference_server_b200              (the two-line integration diff of INTEGRATION.md)
  log_mel_spectrogram .. := the log-mel oracle + willow_inference_server_b200.audio
and a recording engine; tests/golden/dropin_trace.json holds every engine call they made (method, feature windows,
prompt tokens, keyword arguments) and what they returned (scripts/gen_golden_dropin.py).  These tests replay those calls
exactly as recorded and assemble the transcript the way do_whisper does (one window: the window's tokens; chunked: the
LCS merge of the windows' tokens with their strides), so no reference source is needed to run them.

  * CPU test: a recording engine with the signature of models.Whisper.generate / detect_language behind the real
    StorageView: every recorded call binds to the shim's API, and the replayed transcript equals the recorded one.
  * GPU test: the real engine; the tokens of the replayed calls equal a direct wisb_generate on the same features.
"""
import inspect
import json
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRACE = json.load(open(os.path.join(ROOT, "tests", "golden", "dropin_trace.json")))
CANNED_LANGUAGE = TRACE["canned"]["detect_language"][0][0]

PROMPT = [50258, 50259, 50359, 50363]


class FakeTokenizer:
    """Stands in for the HF tokenizer WIS loads (main.py:331-333): the four prompt tokens and the special-id list."""

    def __init__(self, dims):
        from willow_inference_server_b200.languages import LANGUAGE_CODES

        self.table = {"<|startoftranscript|>": dims["sot"], "<|transcribe|>": dims["transcribe"], "<|translate|>": dims["translate"],
                      "<|notimestamps|>": dims["no_timestamps"]}
        for i, c in enumerate(LANGUAGE_CODES):
            self.table[f"<|{c}|>"] = dims["lang_first"] + i
        self.all_special_ids = list(range(dims["eot"], dims["n_vocab"]))

    def convert_tokens_to_ids(self, toks):
        return [self.table[t] for t in toks]


class FakeProcessor:
    def __init__(self, dims):
        self.tokenizer = FakeTokenizer(dims)

    def decode(self, tokens):
        return " ".join(str(int(t)) for t in tokens)


def _synth(n, seed):
    from oracle import logmel as om

    return om.synth_utterance(n, seed)


def _windows(entry, pcm, pad_or_trim, log_mel):
    """The feature windows do_whisper built for `pcm` (main.py:598-617): one zero-padded window, or the chunk_iter windows."""
    from willow_inference_server_b200 import audio

    if entry["features"] == "whole":
        return [log_mel(pad_or_trim(pcm))], None
    chunks = list(audio.chunk_iter(pcm))
    assert [list(s) for _, s in chunks] == entry["strides"]
    return [log_mel(pad_or_trim(c)) for c, _ in chunks], entry["strides"]


def _replay(calls, engine, processor, windows):
    """Make the recorded engine calls -> (language detect_language returned or None, the generate results in order).
    A prompt's language token taken from the canned detection stands for whatever detect_language answers."""
    from willow_inference_server_b200 import models

    detected, results = None, []
    for call in calls:
        feats = models.StorageView.from_array(np.stack([windows[i] for i in call["windows"]]))
        if call["method"] == "detect_language":
            assert call["positional"] == 1
            detected = engine.detect_language(feats, **call["kwargs"])[0][0][0]
            continue
        assert call["method"] == "generate" and call["positional"] == 2
        prompts = [processor.tokenizer.convert_tokens_to_ids([detected if detected and t == CANNED_LANGUAGE else t for t in p])
                   for p in call["prompts"]]
        results.extend(engine.generate(feats, prompts, **call["kwargs"]))
    return detected, results


def _transcript(results, strides, processor):
    """do_whisper's result assembly (main.py:712-721): LCS merge of the windows when chunked, then decode and strip."""
    from willow_inference_server_b200 import audio

    if strides:
        tokens = audio.find_longest_common_sequence([(r.sequences_ids[0], s) for r, s in zip(results, strides)], processor.tokenizer)
    else:
        tokens = results[0].sequences_ids[0]
    return processor.decode(tokens).strip()


# ------------------------------------------------------------------------------------------------------------------ CPU
class RecordingWhisper:
    """Binds every call to the signature of the real shim methods and returns canned results."""

    def __init__(self):
        self.calls = []

    def generate(self, *a, **kw):
        from willow_inference_server_b200 import models

        bound = inspect.signature(models.Whisper.generate).bind(self, *a, **kw)
        feats, prompts = bound.arguments["features"], bound.arguments["prompts"]
        assert isinstance(feats, models.StorageView) and feats.shape[1:] == [80, 3000]
        assert len(prompts) == feats.shape[0] and all(len(p) == 4 for p in prompts)
        self.calls.append(("generate", feats.shape[0], list(prompts[0]), bound.arguments.get("beam_size", 5)))
        return [models.WhisperGenerationResult([[100 + i, 200 + i, 50257]]) for i in range(feats.shape[0])]

    def detect_language(self, *a, **kw):
        from willow_inference_server_b200 import models

        bound = inspect.signature(models.Whisper.detect_language).bind(self, *a, **kw)
        assert bound.arguments["features"].shape == [1, 80, 3000]
        self.calls.append(("detect_language",))
        return [[("<|de|>", 0.9), ("<|en|>", 0.1)]]


def test_reference_do_whisper_drives_the_shim_api_on_cpu():
    from oracle import logmel as om
    from willow_inference_server_b200 import weights as W

    d = W.WhisperDims()
    dims = {"sot": d.sot, "eot": d.eot, "transcribe": d.transcribe, "translate": d.translate, "no_timestamps": d.no_timestamps,
            "lang_first": d.lang_first, "n_vocab": d.n_vocab}
    proc = FakeProcessor(dims)
    short, long_, translate_flag = TRACE["do_whisper"]
    eng = RecordingWhisper()
    # one 3.84 s utterance, language forced
    assert short["args"] == ["x.flac", "large", 5, "transcribe", False, "en"]
    wins, strides = _windows(short, _synth(short["n_samples"], 1), om.pad_or_trim, om.log_mel_spectrogram)
    _, res = _replay(short["calls"], eng, proc, wins)
    ret = short["returned"]
    assert (ret["language"], ret["text"], ret["translation"], ret["duration_ms"]) == ("en", "100 200 50257", None, 3840)
    assert _transcript(res, strides, proc) == ret["text"]
    assert eng.calls == [("generate", 1, PROMPT, 5)]
    # language detection + the long-audio path: 75 s -> 6 windows, two per engine call, beam 3 (long mode), LCS merge
    eng.calls.clear()
    assert long_["args"] == ["x.flac", "medium", 5, "transcribe", True, None] and long_["n_samples"] == 75 * 16000
    wins, strides = _windows(long_, _synth(long_["n_samples"], 2), om.pad_or_trim, om.log_mel_spectrogram)
    detected, res = _replay(long_["calls"], eng, proc, wins)
    assert long_["returned"]["language"] == "de" == re.findall("[A-Za-z0-9]+", detected)[0]
    assert eng.calls[0] == ("detect_language",)
    assert [c[1] for c in eng.calls[1:]] == [2, 2, 2] and all(c[3] == 3 for c in eng.calls[1:])
    assert eng.calls[1][2] == [d.sot, d.lang_first + 2, d.transcribe, d.no_timestamps]  # <|de|>
    assert _transcript(res, strides, proc) == long_["returned"]["text"]
    # do_translate: positional generate(features, prompts, beam_size=...) with the <|translate|> prompt (main.py:535-537)
    eng.calls.clear()
    tr = TRACE["do_translate"][0]
    assert tr["args"] == ["<|de|>", 4]
    _, res = _replay(tr["calls"], eng, proc, [np.zeros((80, 3000), np.float32)])
    out = proc.decode(res[0].sequences_ids[0])
    assert eng.calls == [("generate", 1, [d.sot, d.lang_first + 2, d.translate, d.no_timestamps], 4)] and out == tr["returned"] == "100 200 50257"
    # the latent reference bug is still the reference's: translate=True trips over len(int) (main.py:729, SURVEY section 2)
    # inside the reference's own code, after an engine call that the shim serves
    eng.calls.clear()
    assert translate_flag["args"][-1] is True and translate_flag["raised"] == {"type": "TypeError", "in_reference_code": True}
    wins, _ = _windows(translate_flag, _synth(translate_flag["n_samples"], 1), om.pad_or_trim, om.log_mel_spectrogram)
    _replay(translate_flag["calls"], eng, proc, wins)
    assert eng.calls == [("generate", 1, PROMPT, 5)]


# ------------------------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_reference_do_whisper_over_the_real_engine():
    from tests.gpu_common import model_pair
    from willow_inference_server_b200 import audio, models

    dims, oracle, h = model_pair()
    model = models.Whisper(None, device="cuda", _handles=[h])
    d = model.dims
    proc = FakeProcessor(d)
    short, long_, _ = TRACE["do_whisper"]
    log_mel = lambda x: audio.log_mel_spectrogram(x).numpy()  # noqa: E731  (what do_whisper calls, main.py:605,614)
    # ---- one short utterance: the tokens do_whisper decodes are the tokens of a direct engine call on the same features
    pcm = _synth(61440, 7)
    wins, strides = _windows(short, pcm, audio.pad_or_trim, log_mel)
    _, res = _replay(short["calls"], model, proc, wins)
    text = _transcript(res, strides, proc)
    mel = audio.log_mel_spectrogram(audio.pad_or_trim(pcm)).numpy()[None]
    want, _ = h.generate(mel, [PROMPT], beam_size=5)
    assert text == " ".join(str(t) for t in want[0]) and short["returned"]["duration_ms"] == 3840
    # ---- 75 s: chunked, long-mode beam 3, two windows per call, stitched by the LCS merge; detect_language first
    pcm = _synth(75 * 16000, 8)
    wins, strides = _windows(long_, pcm, audio.pad_or_trim, log_mel)
    lang, res = _replay(long_["calls"], model, proc, wins)
    text = _transcript(res, strides, proc)
    mels, strides = audio.log_mel_chunks(pcm)
    top = model.detect_language(models.StorageView.from_array(mels[:1]))[0][0][0]
    assert lang == top
    prompt = proc.tokenizer.convert_tokens_to_ids(["<|startoftranscript|>", top, "<|transcribe|>", "<|notimestamps|>"])
    seqs, _ = h.generate(mels, [prompt] * mels.shape[0], beam_size=3)
    merged = audio.find_longest_common_sequence(list(zip(seqs, strides)), proc.tokenizer)
    assert text == " ".join(str(int(t)) for t in merged)
    # ---- do_translate on the short utterance's features
    tr = TRACE["do_translate"][1]
    assert tr["args"] == ["<|en|>", 5]
    _, res = _replay(tr["calls"], model, proc, list(mel))
    out = proc.decode(res[0].sequences_ids[0])
    want, _ = h.generate(mel, [[PROMPT[0], PROMPT[1], d["translate"], PROMPT[3]]], beam_size=5)
    assert out == " ".join(str(t) for t in want[0])
