#!/usr/bin/env python
"""Per-step cost of timestamp decoding: large-v2-sized synthetic weights, beam 5, at B = 1 (the persistent decoder pass)
and B = 64 (the batched pass), <|notimestamps|> prompts and timestamp prompts alternated in one process.

    python scripts/bench_timestamps.py [--reps 5] [--out profiles/bench_timestamps.json]

For each (B, mode) it prints the decode time per step (engine timing decode_ms / decode_steps, CUDA events, profiler
off) and, from a separate torch.profiler run, the device time per step of the two search kernels (topk_partial_kernel,
search_tail_kernel).  <|endoftext|> is suppressed so both modes decode the same number of steps (15, as bench.py).
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (SYNTH_KW, synth_utterance, make_blob_host: the same synthetic model as the headline)

SEARCH_KERNELS = ("topk_partial_kernel", "search_tail_kernel")
MAX_LENGTH = 30  # 15 new tokens for both prompts (min(30 // 2, 30 - prompt length))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    from willow_inference_server_b200 import _lib, weights as W

    dims = W.WhisperDims.for_size(bench.MODEL)
    host, _ = bench.make_blob_host(dims)
    h = _lib.Handle.from_host(host.numpy(), 0)
    modes = {"notimestamps": (bench.PROMPT, False), "timestamps": (bench.PROMPT[:3], True)}
    extra = [dims.eot]
    result = {"card": card(), "model": bench.MODEL, "beam": bench.BEAM, "configs": []}
    for B in (1, 64):
        pcm = [bench.synth_utterance(bench.AUDIO_SAMPLES, 1234 + i) for i in range(B)]
        mel = h.logmel(np.concatenate(pcm), np.arange(B, dtype=np.int64) * bench.AUDIO_SAMPLES,
                       np.full(B, bench.AUDIO_SAMPLES, np.int32))

        def run(mode):
            prompt, ts = modes[mode]
            ids, _ = h.generate(mel, np.asarray([prompt] * B, np.int32), bench.BEAM, 1.0, 1.0, MAX_LENGTH, extra,
                                timestamps=ts)
            return ids, h.timing()

        per_step = {m: [] for m in modes}
        for m in modes:  # warm-up: allocations, graph capture
            run(m)
        for _ in range(args.reps):
            for m in modes:
                ids, t = run(m)
                per_step[m].append(t["decode_ms"] / t["decode_steps"])
                steps = t["decode_steps"]
        search_us = {}
        for m in modes:  # profiler in its own runs
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                _, t = run(m)
                torch.cuda.synchronize()
            tot = sum(e.device_time_total for e in prof.key_averages() if any(k in e.key for k in SEARCH_KERNELS))
            search_us[m] = tot / t["decode_steps"]
        cfg = {"B": B, "rows": B * bench.BEAM, "decode_steps": steps,
               "pass": "persistent" if B * bench.BEAM <= 8 else "batched"}
        for m in modes:
            v = np.asarray(per_step[m])
            cfg[m] = {"decode_ms_per_step_median": round(float(np.median(v)), 4),
                      "decode_ms_per_step_min": round(float(v.min()), 4),
                      "decode_ms_per_step_max": round(float(v.max()), 4),
                      "search_kernels_us_per_step": round(float(search_us[m]), 2)}
        cfg["delta_ms_per_step_median"] = round(cfg["timestamps"]["decode_ms_per_step_median"]
                                                - cfg["notimestamps"]["decode_ms_per_step_median"], 4)
        cfg["delta_search_us_per_step"] = round(cfg["timestamps"]["search_kernels_us_per_step"]
                                                - cfg["notimestamps"]["search_kernels_us_per_step"], 2)
        print(json.dumps(cfg), flush=True)
        result["configs"].append(cfg)
    print(json.dumps(result))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
