#!/usr/bin/env python
"""Generate tests/golden/timestamps_hf.npz with HF transformers' ``WhisperTimeStampLogitsProcessor`` (a port of
openai-whisper's ``ApplyTimestampRules``; CTranslate2 restates the same rules).

    python scripts/gen_golden_timestamps_hf.py

(a) Processor level: seeded random rows (the suppress masks already applied, as the engine does) with hand-picked and
    random histories; we record which tokens the processor bans, as [lo, hi) intervals, and whether rule 5's test ("the
    timestamps' total probability beats every text token") held.
(b) A greedy timestamp decode of the timestamp-scripted tiny model (weights.synth_state_dict(ts_script=...)) with
    ``WhisperForConditionalGeneration``, full re-forward per step.
Tests rebuild the rows / weights / inputs from the seeds stored here and compare the oracle with these; they never
import transformers.
"""
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from transformers import WhisperConfig, WhisperForConditionalGeneration  # noqa: E402
from transformers.generation.logits_process import WhisperTimeStampLogitsProcessor  # noqa: E402

from oracle import logmel as om  # noqa: E402
from willow_inference_server_b200 import weights as W  # noqa: E402

# (b): the timestamp-scripted tiny model of tests/test_gpu_timestamps.py
CFG = dict(d_model=128, n_heads=2, n_enc_layers=2, n_dec_layers=2)
SEED = 11
EOT_RAMP = (8, 12.0)
SCRIPT = (4, 3.3, 1.67)
TS_SCRIPT = ((2, 0), (6, 12), (7, 16), (10, 30), (11, 34), (14, 50), (15, 54))
PROMPT = [50258, 50259, 50359]  # no <|notimestamps|>: timestamp decoding
MAX_INIT = 50
UTTS = [(61440, 1234), (160000, 5)]
ROW_STD = 3.0


def row_logits(dims, seed, boost, first):
    """(a) input row: seeded N(0, ROW_STD), timestamps shifted by `boost`, the engine's suppress masks applied."""
    lg = np.random.default_rng(seed).standard_normal(dims.n_vocab, dtype=np.float32) * np.float32(ROW_STD)
    lg[dims.no_timestamps + 1 :] += np.float32(boost)
    lg[sorted(set(dims.suppress_ids))] = -np.inf
    if first:
        lg[dims.suppress_ids_begin] = -np.inf
    return lg


def intervals(banned):
    """bool mask -> [[lo, hi), ...] of its True runs"""
    d = np.diff(np.concatenate([[0], banned.astype(np.int8), [0]]))
    return np.stack([np.flatnonzero(d == 1), np.flatnonzero(d == -1)], 1)


def processor_cases(dims):
    tb = dims.no_timestamps + 1
    last = dims.n_vocab - 1
    cases = [  # (history, max_initial_timestamp_index, timestamp boost)
        ([], 50, 0.0), ([], 0, 0.0), ([], 1, 4.0), ([], 5, -6.0), ([], dims.n_vocab - tb - 1, 0.0),
        ([tb + 3], 50, 0.0),                        # len == 1, a timestamp: text next
        ([500], 50, 0.0),                           # len == 1, text
        ([tb + 2, 500, 600, tb + 10], 50, 0.0),     # a segment just closed
        ([tb, 500, tb + 10, tb + 12], 50, 0.0),     # a pair just completed
        ([tb, 500, tb + 10, tb + 12, 700], 50, 0.0),
        ([tb, 500, tb + 10, tb + 10, 700], 50, 4.0),
        ([tb, 500, last], 50, 0.0),                 # last timestamp 51864 closes a segment
        ([tb, 500, last, last, 600], 50, 6.0),      # ... and after it every timestamp is banned
        ([tb + 1, 400, 500], 50, 6.0),              # rule 5 fires
        ([tb + 1, 400, 500], 50, -6.0),             # rule 5 does not fire
        ([tb + 30, 400, tb + 20, 500], 50, 3.0),    # "last" timestamp is not the largest
    ]
    rng = np.random.default_rng(77)
    for _ in range(12):  # random histories (not necessarily ones the rules would produce)
        n = int(rng.integers(1, 12))
        h = [int(tb + rng.integers(0, 1501)) if rng.random() < 0.4 else int(rng.integers(300, 50000)) for _ in range(n)]
        cases.append((h, int(rng.choice([0, 3, 50, 200])), float(rng.uniform(-4.0, 7.0))))
    return cases


def hf_processor(dims, prompt_len, mi, detect):
    cfg = SimpleNamespace(no_timestamps_token_id=dims.no_timestamps, eos_token_id=dims.eot, bos_token_id=dims.eot,
                          max_initial_timestamp_index=mi)
    return WhisperTimeStampLogitsProcessor(cfg, begin_index=prompt_len, _detect_timestamp_from_logprob=detect)


def main():
    dims = W.WhisperDims(**CFG)
    prompt = torch.tensor([PROMPT])
    # ---- (a)
    seeds, mis, boosts, fired, hist_flat, hist_off, ban_flat, ban_off = [], [], [], [], [], [0], [], [0]
    for i, (hist, mi, boost) in enumerate(processor_cases(dims)):
        seed = 1000 + i
        lg = torch.from_numpy(row_logits(dims, seed, boost, not hist))[None]
        ids = torch.cat([prompt, torch.tensor([hist], dtype=torch.long).reshape(1, -1)], 1)
        out = hf_processor(dims, len(PROMPT), mi, True)(ids, lg)[0]
        without5 = hf_processor(dims, len(PROMPT), mi, False)(ids, lg)[0]
        iv = intervals(torch.isneginf(out).numpy())
        seeds.append(seed)
        mis.append(mi)
        boosts.append(boost)
        lp = torch.log_softmax(without5.float(), -1)  # rule 5's test, as the processor evaluates it
        fired.append(bool(lp[dims.no_timestamps + 1 :].logsumexp(-1) > lp[: dims.no_timestamps + 1].max()))
        assert fired[-1] or torch.equal(out, without5)
        hist_flat += hist
        hist_off.append(len(hist_flat))
        ban_flat.append(iv)
        ban_off.append(ban_off[-1] + len(iv))
    print("rule 5 fired in", sum(fired), "of", len(fired), "rows")
    # ---- (b)
    sd = W.synth_state_dict(dims, seed=SEED, eot_ramp=EOT_RAMP, script=SCRIPT, ts_script=TS_SCRIPT)
    cfg = WhisperConfig(
        vocab_size=dims.n_vocab, num_mel_bins=80, d_model=dims.d_model,
        encoder_layers=dims.n_enc_layers, encoder_attention_heads=dims.n_heads, encoder_ffn_dim=4 * dims.d_model,
        decoder_layers=dims.n_dec_layers, decoder_attention_heads=dims.n_heads, decoder_ffn_dim=4 * dims.d_model,
        max_source_positions=1500, max_target_positions=448, activation_function="gelu",
        pad_token_id=50257, bos_token_id=50257, eos_token_id=50257, decoder_start_token_id=50258,
    )
    model = WhisperForConditionalGeneration(cfg).eval()
    tsd = {k: torch.from_numpy(v) for k, v in sd.items()}
    tsd["proj_out.weight"] = tsd["model.decoder.embed_tokens.weight"]
    print(model.load_state_dict(tsd, strict=False))
    mel = om.log_mel_batch([om.synth_utterance(n, s) for n, s in UTTS])
    feats = torch.from_numpy(mel)
    proc = hf_processor(dims, len(PROMPT), MAX_INIT, True)
    sup = sorted(set(dims.suppress_ids))
    greedy = []
    with torch.no_grad():
        for b in range(len(UTTS)):
            toks = list(PROMPT)
            for s in range(W.WhisperDims().n_text_ctx // 2):
                lg = model(input_features=feats[b : b + 1], decoder_input_ids=torch.tensor([toks])).logits[0, -1].clone()
                lg[sup] = -float("inf")
                if s == 0:
                    lg[dims.suppress_ids_begin] = -float("inf")
                lg = proc(torch.tensor([toks]), lg[None])[0]
                t = int(torch.argmax(lg))
                if t == dims.eot:
                    break
                toks.append(t)
            greedy.append(toks[len(PROMPT) :])
    tb = dims.no_timestamps + 1
    for g in greedy:
        print("greedy", ["T%d" % (t - tb) if t >= tb else t for t in g])
    np.savez_compressed(
        os.path.join(ROOT, "tests", "golden", "timestamps_hf.npz"),
        row_std=np.float32(ROW_STD), seeds=np.array(seeds), max_init=np.array(mis), boost=np.array(boosts),
        fired=np.array(fired), hist_flat=np.array(hist_flat, np.int64), hist_off=np.array(hist_off),
        ban=np.concatenate(ban_flat).astype(np.int64), ban_off=np.array(ban_off),
        cfg=np.array([CFG["d_model"], CFG["n_heads"], CFG["n_enc_layers"], CFG["n_dec_layers"]]), seed=np.int64(SEED),
        eot_ramp=np.array(EOT_RAMP, np.float64), script=np.array(SCRIPT, np.float64), ts_script=np.array(TS_SCRIPT),
        prompt=np.array(PROMPT), max_init_decode=np.int64(MAX_INIT), utts=np.array(UTTS),
        greedy0=np.array(greedy[0]), greedy1=np.array(greedy[1]),
    )


if __name__ == "__main__":
    main()
