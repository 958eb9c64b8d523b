"""Pin the oracle's timestamp rules (tests/timestamp_oracle.py) against HF transformers'
WhisperTimeStampLogitsProcessor (tests/golden/timestamps_hf.npz, written by scripts/gen_golden_timestamps_hf.py), and
check that the timestamp-scripted synthetic weights leave the default weights untouched."""
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import logmel as om
from tests.timestamp_oracle import TimestampOracle, timestamp_rules
from willow_inference_server_b200 import weights as W

TINY = dict(d_model=128, n_heads=2, n_enc_layers=2, n_dec_layers=2)


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "timestamps_hf.npz"))


def _row(dims, seed, boost, first, std):
    # same construction as scripts/gen_golden_timestamps_hf.py row_logits
    lg = np.random.default_rng(int(seed)).standard_normal(dims.n_vocab, dtype=np.float32) * np.float32(std)
    lg[dims.no_timestamps + 1 :] += np.float32(boost)
    lg[sorted(set(dims.suppress_ids))] = -np.inf
    if first:
        lg[dims.suppress_ids_begin] = -np.inf
    return torch.from_numpy(lg)


def _intervals(banned):
    d = np.diff(np.concatenate([[0], banned.astype(np.int8), [0]]))
    return np.stack([np.flatnonzero(d == 1), np.flatnonzero(d == -1)], 1)


def test_rule_function_matches_hf_processor(golden):
    dims = W.WhisperDims()
    tb = dims.no_timestamps + 1
    n = len(golden["seeds"])
    assert n >= 20 and 0 < golden["fired"].sum() < n  # rule 5 both fires and does not
    seen = set()
    for i in range(n):
        hist = golden["hist_flat"][golden["hist_off"][i] : golden["hist_off"][i + 1]].tolist()
        row = _row(dims, golden["seeds"][i], golden["boost"][i], not hist, golden["row_std"])
        out, fired = timestamp_rules(row, hist, tb, dims.eot, int(golden["max_init"][i]))
        want = golden["ban"][golden["ban_off"][i] : golden["ban_off"][i + 1]]
        got = _intervals(torch.isneginf(out).numpy())
        assert np.array_equal(got, want), (i, hist)
        assert fired == bool(golden["fired"][i]), (i, hist)
        if not hist:
            seen.add("empty")
        elif len(hist) == 1:
            seen.add("len1")
        elif hist[-1] >= tb and hist[-2] < tb:
            seen.add("closed")
        elif hist[-1] >= tb:
            seen.add("pair")
        if dims.n_vocab - 1 in hist:
            seen.add("last51864")
    assert seen >= {"empty", "len1", "closed", "pair", "last51864"}
    assert len(set(golden["max_init"].tolist())) >= 3


def _ts_model(golden):
    dims = W.WhisperDims(**dict(zip(TINY, (int(v) for v in golden["cfg"]))))
    r = golden["eot_ramp"]
    s = golden["script"]
    tensors = W.synth_engine_tensors(dims, seed=int(golden["seed"]), eot_ramp=(int(r[0]), float(r[1])),
                                     script=(int(s[0]), float(s[1]), float(s[2])),
                                     ts_script=tuple(tuple(int(v) for v in p) for p in golden["ts_script"]))
    return dims, TimestampOracle(dims, tensors)


def test_greedy_timestamp_decode_matches_hf(golden):
    dims, o = _ts_model(golden)
    mel = om.log_mel_batch([om.synth_utterance(int(n), int(s)) for n, s in golden["utts"]])
    prompt = golden["prompt"].tolist()
    assert dims.no_timestamps not in prompt
    res = o.generate(mel, [prompt] * mel.shape[0], beam_size=1, timestamps=True,
                     max_initial_timestamp_index=int(golden["max_init_decode"]))
    tb = dims.no_timestamps + 1
    for b in range(mel.shape[0]):
        got = res[b].sequences_ids[0]
        assert got == golden[f"greedy{b}"].tolist(), b
        assert got[0] >= tb and sum(t >= tb for t in got) >= 3  # not vacuous: the decode really speaks in timestamps
    with pytest.raises(ValueError):
        o.generate(mel[:1], [prompt + [dims.no_timestamps]], beam_size=1, timestamps=True)


def _digest(sd):
    m = hashlib.sha256()
    for k in sorted(sd):
        m.update(k.encode())
        m.update(np.ascontiguousarray(sd[k]).tobytes())
    return m.hexdigest()


def test_ts_script_none_leaves_weights_unchanged():
    dims = W.WhisperDims(**TINY)
    base = W.synth_state_dict(dims, seed=11, eot_ramp=(8, 12.0), script=(4, 3.3, 1.67))
    # digest of the same call before ts_script existed
    assert _digest(base) == "0df91748052d72742784dd7e80321a34be997adc3af901c293ce41a282b0e3c4"
    assert _digest(W.synth_state_dict(dims, seed=11, eot_ramp=(8, 12.0), script=(4, 3.3, 1.67), ts_script=None)) == _digest(base)
    ts = ((2, 0), (7, 20))
    alt = W.synth_state_dict(dims, seed=11, eot_ramp=(8, 12.0), script=(4, 3.3, 1.67), ts_script=ts)
    pos = "model.decoder.embed_positions.weight"
    for k in base:  # only the positional rows of the scripted positions change
        if k != pos:
            assert np.array_equal(base[k], alt[k]), k
    changed = np.flatnonzero(np.any(base[pos] != alt[pos], axis=1)).tolist()
    assert changed == [2, 7]
    with pytest.raises(ValueError):
        W.synth_state_dict(dims, seed=11, script=(4, 3.3, 1.67), ts_script=((2, 10), (7, 8)))  # overlapping ranges
    with pytest.raises(ValueError):
        W.synth_state_dict(dims, seed=11, ts_script=ts)  # needs script
