"""Timestamp decoding on the host side (no GPU): how models.Whisper.generate picks the mode and passes it to the engine,
the refusal in audio.transcribe_long, and the batcher keeping the two modes apart.  A fake handle stands in for the C ABI."""
import threading

import numpy as np
import pytest

from willow_inference_server_b200 import _lib, audio, models, weights as W
from willow_inference_server_b200.batcher import TranscribeBatcher

D = W.WhisperDims()
PLAIN = [D.sot, D.lang_first, D.transcribe, D.no_timestamps]
TS = [D.sot, D.lang_first, D.transcribe]
TB = D.no_timestamps + 1


class FakeHandle:
    """Answers like the engine would: a timestamp call returns ids that start with a timestamp token."""

    def __init__(self):
        self.calls = []
        self.lock = threading.Lock()

    def dims(self):
        d = {k: getattr(D, k) for k in _lib.DIM_NAMES if k != "n_vocab_pad"}
        d["n_vocab_pad"] = D.n_vocab_pad
        return d

    def set_option(self, key, value):
        pass

    def generate(self, mel, prompts, beam_size, patience, length_penalty, max_length, extra, **kw):
        with self.lock:
            self.calls.append((mel.shape[0], [list(p) for p in prompts], dict(kw)))
        ts = kw.get("timestamps", False)
        ids = [([TB + int(w[0, 0])] if ts else []) + [int(w[0, 0]), 100] for w in mel]
        return ids, [0.0] * mel.shape[0]


def _mel(tags):
    a = np.zeros((len(tags), 80, 3000), np.float32)
    a[:, 0, 0] = tags
    return a


def test_prompt_without_notimestamps_selects_timestamp_decoding():
    h = FakeHandle()
    m = models.Whisper(None, device="cuda", _handles=[h])
    out = m.generate(models.StorageView.from_array(_mel([1, 2])), [TS, TS], beam_size=5, max_initial_timestamp_index=7)
    assert h.calls[-1][2] == {"timestamps": True, "max_initial_timestamp_index": 7}
    assert [r.sequences_ids[0] for r in out] == [[TB + 1, 1, 100], [TB + 2, 2, 100]]
    m.generate(models.StorageView.from_array(_mel([3])), [TS])
    assert h.calls[-1][2] == {"timestamps": True, "max_initial_timestamp_index": 50}  # CTranslate2's default
    m.generate(models.StorageView.from_array(_mel([3])), [PLAIN], max_initial_timestamp_index=7)
    assert h.calls[-1][2] == {}  # <|notimestamps|>: the plain call, unchanged


def test_mixed_modes_and_bad_initial_index_are_refused():
    h = FakeHandle()
    m = models.Whisper(None, device="cuda", _handles=[h])
    mel = models.StorageView.from_array(_mel([1, 2]))
    with pytest.raises(ValueError, match="notimestamps"):
        m.generate(mel, [TS + [D.blank], PLAIN])  # same length, different modes
    n_ts = D.n_vocab - TB
    for bad in (-1, n_ts, 10 ** 6):
        with pytest.raises(ValueError, match="max_initial_timestamp_index"):
            m.generate(mel, [TS, TS], max_initial_timestamp_index=bad)
    m.generate(mel, [TS, TS], max_initial_timestamp_index=n_ts - 1)  # the last timestamp is a valid bound
    m.generate(mel, [PLAIN, PLAIN], max_initial_timestamp_index=-1)  # ignored without timestamps, as before
    assert len(h.calls) == 2


def test_transcribe_long_refuses_timestamp_prompts(monkeypatch):
    h = FakeHandle()
    m = models.Whisper(None, device="cuda", _handles=[h])

    class Tok:
        all_special_ids = [D.eot, D.sot]

    monkeypatch.setattr(audio, "log_mel_window", lambda a, handle=None: _mel([5]))
    with pytest.raises(ValueError, match="timestamps"):
        audio.transcribe_long(m, np.zeros(16000, np.float32), TS, Tok())
    with TranscribeBatcher(m, max_batch=4, max_wait_ms=1) as b:
        with pytest.raises(ValueError, match="timestamps"):
            audio.transcribe_long(None, np.zeros(16000, np.float32), TS, Tok(), batcher=b)
    assert not h.calls
    assert audio.transcribe_long(m, np.zeros(16000, np.float32), PLAIN, Tok()).tolist() == [5, 100]


def test_batcher_keeps_timestamp_and_plain_requests_apart():
    h = FakeHandle()
    m = models.Whisper(None, device="cuda", _handles=[h])
    reqs = [(1, TS), (2, PLAIN), (3, TS), (4, PLAIN), (5, TS)]
    alone = {tag: m.generate(models.StorageView.from_array(_mel([tag])), [p])[0].sequences_ids[0] for tag, p in reqs}
    h.calls.clear()
    with TranscribeBatcher(m, max_batch=8, max_wait_ms=50) as b:
        futs = {tag: b.submit(_mel([tag]), p) for tag, p in reqs}
        got = {tag: f.result(timeout=5)[0].sequences_ids[0] for tag, f in futs.items()}
    assert got == alone
    assert got[1][0] == TB + 1 and got[2] == [2, 100]
    for n, prompts, kw in h.calls:  # every engine call is in one mode
        assert all((D.no_timestamps not in p) == kw.get("timestamps", False) for p in prompts)
    assert len(h.calls) == 2  # and the requests of each mode were coalesced
