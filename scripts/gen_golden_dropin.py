#!/usr/bin/env python
"""Generate tests/golden/dropin_trace.json by RUNNING THE REFERENCE's own orchestration code.

    python scripts/gen_golden_dropin.py <reference checkout>/main.py

`chunkit`, `do_translate` and `do_whisper` are cut out of the reference's main.py with `ast` (main.py itself cannot be
imported: aiortc, av, librosa, ctranslate2 ... are not installed) and executed with
  ctranslate2            := willow_inference_server_b200
  log_mel_spectrogram .. := the log-mel oracle (oracle.logmel) + this package's chunk_iter / LCS merge
and a recording engine with canned results.  Every engine call they make is written down: method, the feature windows
it was given, the prompt as token strings, the keyword arguments; and what do_whisper / do_translate return.  Nothing
from main.py is stored.  tests/test_dropin_reference.py replays the trace against the shim's API (CPU) and the real
engine (GPU).
"""
import ast
import datetime
import json
import logging
import math
import os
import re
import sys
import traceback
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import willow_inference_server_b200 as pkg  # noqa: E402
from oracle import logmel as om  # noqa: E402
from willow_inference_server_b200 import audio, weights as W  # noqa: E402

DETECTED = [("<|de|>", 0.9), ("<|en|>", 0.1)]  # canned detect_language answer
CONCURRENT_GPU_CHUNKS = 2


def canned(i):
    return [100 + i, 200 + i, 50257]


class Tokenizer:
    """The HF tokenizer WIS loads (main.py:331-333), reduced to the prompt tokens and the special-id list."""

    def __init__(self, d):
        from willow_inference_server_b200.languages import LANGUAGE_CODES

        self.table = {"<|startoftranscript|>": d.sot, "<|transcribe|>": d.transcribe, "<|translate|>": d.translate,
                      "<|notimestamps|>": d.no_timestamps}
        for i, c in enumerate(LANGUAGE_CODES):
            self.table[f"<|{c}|>"] = d.lang_first + i
        self.names = {v: k for k, v in self.table.items()}
        self.all_special_ids = list(range(d.eot, d.n_vocab))

    def convert_tokens_to_ids(self, toks):
        return [self.table[t] for t in toks]


class Processor:
    def __init__(self, d):
        self.tokenizer = Tokenizer(d)

    def decode(self, tokens):
        return " ".join(str(int(t)) for t in tokens)


class Recorder:
    def __init__(self, windows, tokenizer):
        self.windows, self.tok, self.calls = windows, tokenizer, []

    def _window_ids(self, feats):
        return [next(i for i, w in enumerate(self.windows) if np.array_equal(w, row)) for row in feats.array]

    def generate(self, *a, **kw):
        feats, prompts = a[0], (a[1] if len(a) > 1 else kw["prompts"])
        self.calls.append({"method": "generate", "positional": len(a), "windows": self._window_ids(feats),
                           "prompts": [[self.tok.names[t] for t in p] for p in prompts],
                           "kwargs": {k: v for k, v in kw.items() if k != "prompts"}})
        return [pkg.models.WhisperGenerationResult([canned(i)]) for i in range(len(prompts))]

    def detect_language(self, *a, **kw):
        self.calls.append({"method": "detect_language", "positional": len(a), "windows": self._window_ids(a[0]), "kwargs": kw})
        return [DETECTED]


def extract(main_py):
    tree = ast.parse(open(main_py).read())
    picked = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in {"chunkit", "do_translate", "do_whisper"}]
    assert len(picked) == 3
    return compile(ast.Module(body=picked, type_ignores=[]), main_py, "exec")


def windows_of(pcm):
    """The feature windows of one recording: one zero-padded window up to 30 s, chunk_iter windows beyond."""
    if pcm.shape[0] <= om.N_SAMPLES:
        return "whole", [om.log_mel_spectrogram(om.pad_or_trim(pcm))], None
    chunks = list(audio.chunk_iter(pcm))
    return "chunks", [om.log_mel_spectrogram(om.pad_or_trim(c)) for c, _ in chunks], [list(s) for _, s in chunks]


def namespace(code, rec, d, pcm):
    librosa = types.SimpleNamespace(load=lambda f, sr=16000, mono=True: (pcm, sr), get_duration=lambda y, sr: len(y) / float(sr))
    ns = {
        "datetime": datetime, "math": math, "re": re, "np": np, "librosa": librosa, "ctranslate2": pkg,
        "logger": logging.getLogger("dropin"), "settings": types.SimpleNamespace(language="en"),
        "models": types.SimpleNamespace(whisper_model_large=rec, whisper_model_medium=rec, whisper_model_small=rec,
                                        whisper_model_base=rec, whisper_model_tiny=rec, whisper_processor=Processor(d)),
        "chunk_iter": audio.chunk_iter, "pad_or_trim": om.pad_or_trim,
        "log_mel_spectrogram": lambda x: types.SimpleNamespace(numpy=lambda: om.log_mel_spectrogram(x)),
        "find_longest_common_sequence": audio.find_longest_common_sequence,
        "beam_size": 1, "long_beam_size": 3, "long_beam_size_threshold": 12000, "support_chunking": True,
        "concurrent_gpu_chunks": CONCURRENT_GPU_CHUNKS,
    }
    exec(code, ns)
    return ns


def main():
    main_py = sys.argv[1]
    code = extract(main_py)
    d = W.WhisperDims()
    out = {"canned": {"generate_row_i": "[100 + i, 200 + i, 50257]", "detect_language": DETECTED},
           "settings": {"language": "en", "beam_size": 1, "long_beam_size": 3, "long_beam_size_threshold_ms": 12000,
                        "support_chunking": True, "concurrent_gpu_chunks": CONCURRENT_GPU_CHUNKS},
           "do_whisper": [], "do_translate": []}
    cases = [(61440, ("x.flac", "large", 5, "transcribe", False, "en")),
             (75 * 16000, ("x.flac", "medium", 5, "transcribe", True, None)),
             (61440, ("x.flac", "large", 5, "transcribe", False, "en", True))]
    for n, args in cases:
        pcm = om.synth_utterance(n, 1)
        layout, wins, strides = windows_of(pcm)
        rec = Recorder(wins, Processor(d).tokenizer)
        ns = namespace(code, rec, d, pcm)
        entry = {"n_samples": n, "args": list(args), "features": layout, "strides": strides}
        try:
            lang, text, _ms, translation, _speedup, dur = ns["do_whisper"](*args)
            entry["returned"] = {"language": lang, "text": text, "translation": translation, "duration_ms": dur}
        except Exception as e:  # noqa: BLE001 -- the reference's own latent bugs are part of the record
            frame = traceback.extract_tb(e.__traceback__)[-1]
            entry["raised"] = {"type": type(e).__name__, "in_reference_code": os.path.abspath(frame.filename) == os.path.abspath(main_py)}
        entry["calls"] = rec.calls
        out["do_whisper"].append(entry)
    for language, beam in (("<|de|>", 4), ("<|en|>", 5)):
        pcm = om.synth_utterance(61440, 1)
        _, wins, _ = windows_of(pcm)
        rec = Recorder(wins, Processor(d).tokenizer)
        ns = namespace(code, rec, d, pcm)
        text = ns["do_translate"](rec, pkg.StorageView.from_array(np.stack(wins)), 1, language, beam)
        out["do_translate"].append({"args": [language, beam], "windows": 1, "returned": text, "calls": rec.calls})
    dst = os.path.join(ROOT, "tests", "golden", "dropin_trace.json")
    with open(dst, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print(open(dst).read())


if __name__ == "__main__":
    main()
