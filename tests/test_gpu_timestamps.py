"""GPU parity of timestamp decoding (wisb_generate_ts): the CUDA search with Whisper's timestamp rules vs the fp32 oracle
on a timestamp-scripted synthetic model, through every decoder path, plus isolation from the plain mode on one handle.

Token parity is exact on the cases whose oracle transcript is a robust decision (tests/gpu_common.robust_cases); every
output, robust or not, must obey the timestamp rules when replayed through tests.timestamp_oracle.timestamp_rules."""
import functools

import numpy as np
import pytest
import torch

from tests.gpu_common import LOGIT_TOL, PROMPT, RAMP, SCRIPT, mel_inputs, robust_cases
from tests.timestamp_oracle import TimestampOracle, timestamp_rules
from willow_inference_server_b200 import _lib, models, weights as W

pytestmark = pytest.mark.gpu

TS_PROMPT = PROMPT[:3]  # <|startoftranscript|><|en|><|transcribe|>, no <|notimestamps|>
# decoder position -> first timestamp index of its scripted alternatives (prompt of 3: generated token g comes from
# position 2 + g): an opening timestamp, text, then closing / opening pairs before the <|endoftext|> ramp
TS_SCRIPT = ((2, 0), (6, 12), (7, 16), (10, 30), (11, 34), (14, 50), (15, 54))
SEED = 11


@functools.lru_cache(maxsize=1)
def ts_pair():
    dims = W.WhisperDims(d_model=128, n_heads=2, n_enc_layers=2, n_dec_layers=2)
    tensors = W.synth_engine_tensors(dims, seed=SEED, eot_ramp=RAMP, script=SCRIPT, ts_script=TS_SCRIPT)
    buf = np.zeros(W.blob_nbytes(tensors), np.uint8)
    W.write_blob_into(buf, dims, tensors)
    return dims, TimestampOracle.from_blob(buf), _lib.Handle.from_host(buf, 0)


@pytest.fixture(scope="module")
def pair():
    return ts_pair()


@functools.lru_cache(maxsize=4)
def oracle_cases(beam, n=6):
    dims, oracle, _ = ts_pair()
    mel = mel_inputs(n)
    res, robust = robust_cases(oracle, mel, [TS_PROMPT] * n, beam, n_probe=4, timestamps=True)
    if beam > 1:
        # two finished hypotheses that differ in one early token and agree afterwards can tie far below the logit
        # tolerance while the noise probe happens to leave them in order: such a tie is not a robust decision either
        # (the gap between the two best hypotheses, length-normalised, is taken back to log-probability units)
        trace = []
        oracle.generate(mel, [TS_PROMPT] * n, beam_size=beam, timestamps=True, trace=trace)
        gap = [dict(x for x in t if isinstance(x, tuple))["final"] * (len(r.sequences_ids[0]) + 1) for t, r in zip(trace, res)]
        robust = [i for i in robust if gap[i] > LOGIT_TOL]
    return res, robust


def assert_rules(dims, seq, mi=50):
    """Replay `seq` through the oracle's rule function (rules 1-4 do not depend on the logits; a row whose text
    tokens all beat the timestamps keeps rule 5 out of the way) and check the structure directly."""
    tb = dims.no_timestamps + 1
    row = torch.zeros(dims.n_vocab)
    row[tb:] = -1e4
    for i, t in enumerate(seq):
        lg, _ = timestamp_rules(row, seq[:i], tb, dims.eot, mi)
        assert lg[t] != float("-inf"), (i, seq)
    assert dims.no_timestamps not in seq and dims.eot not in seq
    assert seq and tb <= seq[0] <= tb + mi
    stamps = [t for t in seq if t >= tb]
    assert stamps == sorted(stamps)
    runs, k = [], 0  # timestamps come in pairs, except a single one at the end (directly before <|endoftext|>)
    while k < len(seq):
        if seq[k] >= tb:
            j = k
            while j < len(seq) and seq[j] >= tb:
                j += 1
            runs.append((k, j - k))
            k = j
        else:
            k += 1
    for start, n in runs:
        assert n <= 2, seq
        if n == 2:
            assert start > 0  # a pair closes one segment and opens the next
        elif start > 0 and start + n < len(seq):
            raise AssertionError(f"unpaired timestamp inside the transcript: {seq}")


def has_structure(dims, seq):
    tb = dims.no_timestamps + 1
    pairs = any(a >= tb and b >= tb for a, b in zip(seq[1:], seq[2:]))
    return seq[0] >= tb and seq[1] < tb and pairs


@pytest.mark.parametrize("beam", [1, 2, 5])
def test_generate_matches_oracle(pair, beam):
    dims, oracle, h = pair
    mel = mel_inputs(6)
    res, robust = oracle_cases(beam)
    assert len(robust) >= 4, f"only {len(robust)} of 6 oracle transcripts are robust decisions"
    m = models.Whisper(None, device="cuda", _handles=[h])
    out = m.generate(models.StorageView.from_array(mel), [TS_PROMPT] * 6, beam_size=beam, return_scores=True)
    for i in robust:  # exact token parity, no tolerated mismatch
        assert out[i].sequences_ids[0] == res[i].sequences_ids[0], (beam, i)
        if beam > 1:
            assert abs(out[i].scores[0] - res[i].scores[0]) < 5e-2, (beam, i)
        assert has_structure(dims, res[i].sequences_ids[0]), res[i].sequences_ids[0]
    assert len({tuple(res[i].sequences_ids[0]) for i in robust}) >= 3
    for o in out:
        assert_rules(dims, o.sequences_ids[0])


@pytest.mark.parametrize("n_utt,beam", [(2, 3), (4, 2), (8, 1)])
def test_persistent_pass_several_utterances(pair, n_utt, beam):
    dims, oracle, h = pair
    mel = mel_inputs(8)[:n_utt]
    for mma in (1, 0):  # the warp-MMA pass and the SIMT pass
        h.set_option("mega_mma", mma)
        try:
            ids, _ = h.generate(mel, [TS_PROMPT] * n_utt, beam_size=beam, timestamps=True)
            solo = [h.generate(mel[i : i + 1], [TS_PROMPT], beam_size=beam, timestamps=True)[0][0] for i in range(n_utt)]
        finally:
            h.set_option("mega_mma", 1)
        assert ids == solo, (mma, n_utt, beam)
        for s in ids:
            assert_rules(dims, s)


def test_batched_pass(pair):
    dims, oracle, h = pair
    mel = mel_inputs(16)
    ids, scores = h.generate(mel, [TS_PROMPT] * 16, beam_size=5, timestamps=True)  # 80 rows: the batched pass
    solo = [h.generate(mel[i : i + 1], [TS_PROMPT], beam_size=5, timestamps=True) for i in range(16)]
    assert ids == [s[0][0] for s in solo]
    assert np.allclose(scores, [s[1][0] for s in solo], atol=2e-2)
    res, robust = oracle_cases(5)
    for i in robust:
        assert ids[i] == res[i].sequences_ids[0], i
    for s in ids:
        assert_rules(dims, s)


def test_per_op_chain_graphs_on_and_off(pair):
    dims, oracle, h = pair
    mel = mel_inputs(4)[:2]
    want, _ = h.generate(mel, [TS_PROMPT] * 2, beam_size=3, timestamps=True)
    h.set_option("decoder_mega", 0)
    try:
        chain, _ = h.generate(mel, [TS_PROMPT] * 2, beam_size=3, timestamps=True)
        h.set_option("use_graphs", 0)
        eager, _ = h.generate(mel, [TS_PROMPT] * 2, beam_size=3, timestamps=True)
    finally:
        h.set_option("use_graphs", 1)
        h.set_option("decoder_mega", 1)
    assert chain == eager == want


@pytest.mark.parametrize("mega,B", [(1, 1), (0, 1), (1, 3)])  # persistent pass; per-op chain (graphs); batched pass
def test_no_cross_contamination_between_modes(pair, mega, B):
    dims, oracle, h = pair
    mel = mel_inputs(4)[:B]
    h.set_option("decoder_mega", mega)
    try:
        a = h.generate(mel, [PROMPT] * B, beam_size=5)
        t = h.generate(mel, [TS_PROMPT] * B, beam_size=5, timestamps=True)
        b = h.generate(mel, [PROMPT] * B, beam_size=5)
        t2 = h.generate(mel, [TS_PROMPT] * B, beam_size=5, timestamps=True)
    finally:
        h.set_option("decoder_mega", 1)
    assert a == b and t == t2
    tb = dims.no_timestamps + 1
    for s in t[0]:
        assert_rules(dims, s)
    # without the rules the scripted timestamps are ordinary tokens: the plain transcripts break rule 4 or the pairing
    assert a[0] != t[0]


def test_max_initial_timestamp_index(pair):
    dims, oracle, h = pair
    tb = dims.no_timestamps + 1
    mel = mel_inputs(6)
    for mi in (5, 1):
        res, robust = robust_cases(oracle, mel, [TS_PROMPT] * 6, 1, timestamps=True, max_initial_timestamp_index=mi)
        assert robust
        ids, _ = h.generate(mel, [TS_PROMPT] * 6, beam_size=1, timestamps=True, max_initial_timestamp_index=mi)
        for i, s in enumerate(ids):
            assert tb <= s[0] <= tb + mi
            assert_rules(dims, s, mi)
        for i in robust:
            assert ids[i] == res[i].sequences_ids[0], (mi, i)


def test_argument_errors(pair):
    dims, oracle, h = pair
    mel = mel_inputs(4)[:1]
    with pytest.raises(ValueError, match="notimestamps"):  # wisb_generate_ts returns 1
        h.generate(mel, np.array([PROMPT], np.int32), beam_size=1, timestamps=True)
    n_ts = dims.n_vocab - dims.no_timestamps - 1
    for bad in (-1, n_ts):
        with pytest.raises(ValueError):
            h.generate(mel, np.array([TS_PROMPT], np.int32), beam_size=1, timestamps=True, max_initial_timestamp_index=bad)
    # the plain entry point keeps its behaviour for a prompt without <|notimestamps|>: no timestamp rules
    ids, _ = h.generate(mel, np.array([TS_PROMPT], np.int32), beam_size=1)
    res, robust = robust_cases(oracle, mel, [TS_PROMPT], 1)
    if robust:
        assert ids[0] == res[0].sequences_ids[0]
