"""Timestamp decoding on top of the fp32 CPU oracle (``oracle.whisper_ref.WhisperOracle``): the reference for the CUDA
search's timestamp rules.  TEST INFRASTRUCTURE ONLY.

CTranslate2 applies Whisper's timestamp rules when the prompt lacks <|notimestamps|> (the reference's prompts keep that
token, main.py:529, :661).  ``timestamp_rules`` restates them after HF transformers'
``WhisperTimeStampLogitsProcessor`` (a port of openai-whisper's ``ApplyTimestampRules``) and is PINNED against that
processor in ``tests/test_oracle_timestamps.py`` (golden ``tests/golden/timestamps_hf.npz``, written by
scripts/gen_golden_timestamps_hf.py: the processor's bans on seeded rows, and a greedy timestamp decode).  CTranslate2
4.1.0 restates the same rules, but agreement with it is **PARITY UNPINNED**: no CTranslate2 binary, source or golden
transcript is available; one known grey zone is what its ``max_initial_timestamp_index=0`` means.

``TimestampOracle`` decodes with the oracle's own greedy / beam search, unchanged: the rules are applied after its
logits processors, and each row's generated tokens travel with the row's K/V cache, so the beam search's reordering
(``cache[i][parents]``) reorders them too.
"""
from __future__ import annotations

import torch

from oracle.whisper_ref import NEG_INF, WhisperOracle


def timestamp_rules(logits: torch.Tensor, hist, ts_begin: int, eot: int, max_initial_timestamp_index: int):
    """Whisper's timestamp rules on one row of (already suppressed) logits [V], after HF
    ``WhisperTimeStampLogitsProcessor.__call__``; ``hist`` are the row's generated tokens (prompt excluded).
    Returns (processed copy, whether rule 5's test held)."""
    lg = logits.clone()
    lg[ts_begin - 1] = NEG_INF  # 1. <|notimestamps|>
    seq = [int(t) for t in hist]
    last_ts = len(seq) >= 1 and seq[-1] >= ts_begin
    pen_ts = len(seq) < 2 or seq[-2] >= ts_begin
    if last_ts:  # 2. timestamps come in pairs, except directly before <|endoftext|>
        if pen_ts:
            lg[ts_begin:] = NEG_INF
        else:
            lg[:eot] = NEG_INF
    stamps = [t for t in seq if t >= ts_begin]
    if stamps:  # 3. timestamps never decrease; a segment may open at the time the previous one closed
        lg[ts_begin : stamps[-1] + (0 if last_ts and not pen_ts else 1)] = NEG_INF
    if not seq:  # 4. the first token is a timestamp, no later than ts_begin + max_initial_timestamp_index
        lg[:ts_begin] = NEG_INF
        lg[ts_begin + max_initial_timestamp_index + 1 :] = NEG_INF
    # 5. timestamps' total probability above every text token -> a timestamp (the log-softmax shift cancels)
    fired = bool(torch.logsumexp(lg[ts_begin:], 0) > lg[:ts_begin].max())
    if fired:
        lg[:ts_begin] = NEG_INF
    return lg, fired


class TimestampOracle(WhisperOracle):
    """``WhisperOracle`` plus ``generate(..., timestamps=True, max_initial_timestamp_index=50)``; without
    ``timestamps`` every call is the base class's."""

    _ts = None      # (ts_begin, max_initial_timestamp_index) while a timestamp decode runs
    _start = 0      # position of the last prompt token (decoding starts there)
    _hist = None    # [rows, generated] tokens of the rows of the current step

    def generate(self, features, prompts, *args, timestamps: bool = False, max_initial_timestamp_index: int = 50,
                 **kw):
        """As ``WhisperOracle.generate``; ``timestamps=True`` applies the timestamp rules (the prompts must not contain
        <|notimestamps|>) and the results keep the timestamp tokens."""
        if not timestamps:
            return super().generate(features, prompts, *args, **kw)
        if any(self.dims.no_timestamps in p for p in prompts):
            raise ValueError("timestamp decoding: the prompt must not contain <|notimestamps|>")
        self._ts = (self.dims.no_timestamps + 1, int(max_initial_timestamp_index))
        try:
            return super().generate(features, prompts, *args, **kw)
        finally:
            self._ts = self._hist = None

    def _prefill(self, prompt, ckv):
        cache = super()._prefill(prompt, ckv)
        if self._ts is None:
            return cache
        self._start = len(prompt) - 1
        # one more cache "layer" holds the generated tokens: [rows, n] (empty at the first generated step)
        empty = torch.zeros((1, 0), dtype=torch.long)
        return (cache or []) + [(empty, empty)]

    def decode_rows(self, tokens, pos: int, cache, ckv):
        if self._ts is None or not cache or cache[-1][0].dtype != torch.long:  # no history entry: prompt prefill
            return super().decode_rows(tokens, pos, cache, ckv)
        hist = cache[-1][0]
        logits, new_cache = super().decode_rows(tokens, pos, cache[:-1] or None, ckv)
        if pos > self._start:  # the token fed here is the row's previous output
            hist = torch.cat([hist, torch.as_tensor(tokens, dtype=torch.long)[:, None]], 1)
        self._hist = hist
        return logits, new_cache + [(hist, hist)]

    def _process(self, logits, gen_step: int, extra_suppress=None):
        logits = super()._process(logits, gen_step, extra_suppress)
        if self._ts is not None:
            for i in range(logits.shape[0]):
                logits[i] = timestamp_rules(logits[i], self._hist[i].tolist(), self._ts[0], self.dims.eot, self._ts[1])[0]
        return logits
