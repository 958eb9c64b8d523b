#!/usr/bin/env python
"""bench.py -- Whisper large-v2 realtime multiple on B200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps K --warmup W                  # our arm (CUDA engine through the C ABI)
    python bench.py ... --dump-outputs DIR                         # + the last timed step's outputs as DIR/<name>.npy
    python bench.py --impl reference --gpus 1 --steps K --warmup W # reference arm: CTranslate2 on the host cores when it
                                                                   # is installed on the box, else the oracle port
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Headline workload (configs[1] of BASELINE.json): whisper-large-v2, beam 5, one 3.84 s synthetic 16 kHz utterance per step,
padded to a 30 s window exactly as WIS does (main.py:613).  Weights are seeded synthetic (no checkpoints in the image),
peaked like a trained model's output (weights.synth_state_dict(script=...)), so the decode length is pinned as SURVEY.md
section 8(d) prescribes: ceil(3.5 tok/s * 3.84 s) + 1 = 15 generated tokens (max_length = 30, <|endoftext|> suppressed
through CT2's own `suppress_tokens` option), after the 4-token prompt.
One "step" = log-mel + encoder + cross-K/V + 1 prompt-prefix pass + 15 beam-search passes for one utterance per GPU.

  value : whole-job audio-seconds / second with the PCM already resident in HBM (wisb_logmel on a device pointer,
          wisb_generate on the device-resident features), timed with the library's CUDA events on its launching stream
  e2e   : the same metric through the reference-facing surface with HOST buffers:
          audio.log_mel_spectrogram(pcm).numpy() -> StorageView.from_array -> Whisper.generate (wall clock, synchronised)
N > 1   : one process per GPU, utterances are independent (weak scaling, no data-path collective); the weight blob is
          generated on rank 0 and broadcast over NCCL at load time only.
Extra keys on the same JSON line (N = 1, rank 0): the other BASELINE.json configs --
  configs0 : whisper-base greedy on client/3sec.flac through audio.load_audio (FLAC decode included)
  configs2 : large-v2 beam 5, batch 64 mixed 3.84 / 10 / 30 s utterances in ONE engine call (shared decoder passes)
  configs4 : whisper-medium beam 1, one 30 s window, p50 latency
  configs3 : (N = 8 under torchrun) 512 x 10 s utterances, 64 per GPU, + the reference's own one-process mode
             models.Whisper(device_index=[0..7]) behind the cross-request batcher
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = "large-v2"
AUDIO_SAMPLES = 61440  # 3.84 s
AUDIO_SECONDS = AUDIO_SAMPLES / 16000.0
BEAM = 5
N_OUT = int(math.ceil(3.5 * AUDIO_SECONDS)) + 1  # 15
MAX_LENGTH = 2 * N_OUT  # -> max_new = min(15, 30 - 4) = 15
PROMPT = [50258, 50259, 50359, 50363]
SEED = 0
SYNTH_KW = dict(seed=SEED, script=(4, 3.3, 1.67))  # peaked synthetic model: beam decisions are not near-ties


def n_out_for(n_samples: int) -> int:
    """SURVEY.md section 8(d): decode length pinned to ceil(3.5 tokens/s x duration) + 1."""
    return int(math.ceil(3.5 * n_samples / 16000.0)) + 1


def synth_utterance(n_samples: int, seed: int = 1234) -> np.ndarray:
    """SURVEY.md section 8(d) input recipe: 0.3 sin(2 pi (200 + 300 t) t) + 0.05 N(0,1), 16 kHz mono float32."""
    rng = np.random.default_rng(seed)
    t = np.arange(n_samples, dtype=np.float64) / 16000.0
    return (0.3 * np.sin(2.0 * np.pi * (200.0 + 300.0 * t) * t) + 0.05 * rng.standard_normal(n_samples)).astype(np.float32)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def ncu_dram_traffic_per_launch(*names):
    """dram__bytes_read + dram__bytes_write per launch from a committed ncu --set full capture under profiles/
    (the first of `names` that exists), averaged over the captured launches; None if no summary is there."""
    import csv

    for summary in names:
        p = os.path.join(ROOT, "profiles", summary)
        if not os.path.exists(p):
            continue
        rows = list(csv.reader(open(p)))
        hdr, units = rows[0], rows[1]
        try:
            ir, iw = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
        except ValueError:
            continue
        scale = {"Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0, "Gbyte": 1e9}
        tot = [float(r[ir]) * scale.get(units[ir], 1e6) + float(r[iw]) * scale.get(units[iw], 1e6) for r in rows[2:]]
        if tot:
            return int(sum(tot) / len(tot)), summary
    return None, None


def encoder_gemm_flops(dims, windows=1):
    """Algorithmic FLOPs of the tcgen05 GEMM launches per window (SURVEY.md section 8d): conv2 + 4 GEMMs per encoder
    layer + the cross-K/V projection, 1500 valid rows each."""
    d, L = dims.d_model, dims.n_enc_layers
    conv2 = 2 * 1500 * (3 * d) * d
    layers = L * 2 * 1500 * d * (3 * d + d + 4 * d + 4 * d)
    ckv = 2 * 1500 * d * (dims.n_dec_layers * 2 * d)
    return windows * (conv2 + layers + ckv), 1 + 4 * L + 1


def decoder_pass_bytes(dims, n_utt=1):
    """Bytes one decoder pass streams (fp16): per layer the QKV (3 d^2), out (d^2), cross-q (d^2), cross-out (d^2), fc1 and
    fc2 (8 d^2) matrices = 14 L d^2, the tied vocabulary projection V d, and 2 x 1500 x d of cross K/V per layer and
    utterance (read once for all beams).  SURVEY.md section 8(d) writes 16 L d^2: that also counts the cross-K/V
    projection weights (2 L d^2), which the encoder-side GEMM consumes once per window, not once per pass."""
    d, L = dims.d_model, dims.n_dec_layers
    return 2 * (14 * L * d * d + dims.n_vocab * d) + n_utt * 4 * L * 1500 * d


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_blob_host(dims, pinned=True, **kw):
    import torch

    from willow_inference_server_b200 import weights as W

    tensors = W.synth_engine_tensors(dims, **(kw or SYNTH_KW))
    n = W.blob_nbytes(tensors)
    host = torch.empty(n, dtype=torch.uint8)
    if pinned:
        host = host.pin_memory()
    W.write_blob_into(host.numpy(), dims, tensors)
    return host, tensors


# --------------------------------------------------------------------------------------------------------------- extra configs
def bench_configs2(handle, dims, device, reps=3):
    """BASELINE.json configs[2]: large-v2, beam 5, batch 64 = 22 x 3.84 s + 21 x 10 s + 21 x 30 s (shuffled, seed 1234) in ONE
    engine call: every decoder pass is shared by all utterances still decoding (per-utterance length limits)."""
    from willow_inference_server_b200 import _lib, audio, models

    durs = [61440] * 22 + [160000] * 21 + [480000] * 21
    np.random.default_rng(1234).shuffle(durs)
    B = len(durs)
    pcm = [synth_utterance(n, 1234 + i) for i, n in enumerate(durs)]
    n_out = [n_out_for(n) for n in durs]
    max_len = np.asarray([2 * k for k in n_out], np.int32)
    audio_s = sum(durs) / 16000.0
    flat = np.concatenate(pcm)
    off = np.cumsum([0] + [len(p) for p in pcm[:-1]]).astype(np.int64)
    ns = np.asarray(durs, np.int32)
    prompts = np.asarray([PROMPT] * B, np.int32)
    import torch

    flat_dev = torch.from_numpy(flat).to(device)
    model = models.Whisper(None, device="cuda", _handles=[handle], reuse_encoder=False)

    def step_device():
        handle.logmel(flat_dev.data_ptr(), off, ns, to_host=False, keep=True, pcm_on_device=True, pcm_dtype=_lib.PCM_F32, B=B)
        tl = handle.timing()["logmel_ms"]
        ids, _ = handle.generate(None, prompts, BEAM, 1.0, 1.0, max_len, [dims.eot], B=B)
        t = handle.timing()
        return ids, tl, t

    def step_e2e():
        mel = audio.log_mel_batch(pcm, handle)
        res = model.generate(models.StorageView.from_array(mel), [PROMPT] * B, beam_size=BEAM, max_length=max_len,
                             suppress_tokens=[-1, dims.eot])
        return [r.sequences_ids[0] for r in res]

    ids, _, _ = step_device()  # warm-up: allocations, graph capture
    assert [len(x) for x in ids] == n_out, "decode lengths are not the pinned ones"
    ids_e2e = step_e2e()
    assert ids_e2e == ids, "host-buffer path and device-resident path disagree (configs2)"
    dev_ms, stages = [], {}
    for _ in range(reps):
        _, tl, t = step_device()
        dev_ms.append(tl + t["generate_ms"])
        for k in ("encoder_ms", "cross_kv_ms", "decode_ms"):
            stages[k] = stages.get(k, 0.0) + t[k] / reps
        stages["logmel_ms"] = stages.get("logmel_ms", 0.0) + tl / reps
    t0 = time.perf_counter()
    for _ in range(reps):
        step_e2e()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / reps
    ms = float(np.mean(dev_ms))
    passes = int(t["decode_steps"])
    utt_steps = sum(n_out)
    return {"workload": "whisper-large-v2 beam=5, batch=64 mixed 3.84/10/30 s utterances (22/21/21, seed 1234), one engine call "
                        "(BASELINE.json configs[2]); WIS would switch to beam 3 for >= 12 s audio (main.py:582-586), the config pins 5",
            "value": round(audio_s / (ms * 1e-3), 1), "unit": "x realtime", "ms_per_batch": round(ms, 2),
            "audio_seconds": round(audio_s, 1), "decoder_passes": passes,
            "decode_length_policy": "per utterance ceil(3.5 tok/s x duration) + 1 = 15 / 36 / 106 tokens (per-utterance max_length, "
                                    "<|endoftext|> suppressed); finished utterances leave the shared pass",
            "stages_ms": {k: round(v, 2) for k, v in stages.items()},
            "e2e": {"value": round(audio_s / wall, 1), "unit": "x realtime", "ms_per_batch": round(wall * 1e3, 2),
                    "h2d_bytes_per_step": int(flat.nbytes + B * 80 * 3000 * 4 + B * 4 * 4),
                    "d2h_bytes_per_step": int(B * 80 * 3000 * 4 + 4 * utt_steps + 8 * B)},
            "serial_estimate_x_realtime": 135.0,
            "note": "the serial estimate is VERDICT r01's figure for one-utterance-at-a-time decoding of the same batch"}


def bench_small_model(size, beam, n_samples, device_index, reps, flac=None):
    """configs[0] / configs[4]: a small model on one utterance, latency oriented.  Returns p50 / mean latency (device
    timed and end to end with host buffers) and the realtime multiple."""
    from willow_inference_server_b200 import _lib, audio, models, weights as W

    dims = W.WhisperDims.for_size(size)
    host, _ = make_blob_host(dims, pinned=False)
    h = _lib.Handle.from_host(host.numpy(), device_index)
    del host
    model = models.Whisper(None, device="cuda", _handles=[h], reuse_encoder=False)
    if flac is not None:
        raw = open(flac, "rb").read()
        pcm = audio.load_audio(raw)
        n_samples = int(pcm.shape[0])
    else:
        raw = None
        pcm = synth_utterance(n_samples, 4321)
    n_out = n_out_for(n_samples)
    ml = 2 * n_out

    def step():
        x = audio.load_audio(raw) if raw is not None else pcm  # configs0: FLAC decode is part of the request
        mel = audio.log_mel_spectrogram(audio.pad_or_trim(x)).numpy()[None]
        res = model.generate(models.StorageView.from_array(mel), [PROMPT], beam_size=beam, max_length=ml,
                             suppress_tokens=[-1, dims.eot])
        return res[0].sequences_ids[0]

    ids = step()
    step()
    assert len(ids) == n_out
    lat, dev = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        step()
        lat.append((time.perf_counter() - t0) * 1e3)
        dev.append(model.timing()["generate_ms"])
    audio_s = n_samples / 16000.0
    out = {"model": size, "beam": beam, "audio_seconds": round(audio_s, 3), "generated_tokens": n_out,
           "p50_latency_ms": round(float(np.median(lat)), 3), "mean_latency_ms": round(float(np.mean(lat)), 3),
           "generate_ms_device": round(float(np.median(dev)), 3),
           "value": round(audio_s / (float(np.median(lat)) * 1e-3), 1), "unit": "x realtime (e2e, host buffers, p50)",
           "decode_length_policy": "ceil(3.5 tok/s x duration) + 1 tokens, <|endoftext|> suppressed", "tokens": ids[:8]}
    h.close()
    return out, dims, pcm


def cpu_port_small(size, beam, pcm, n_threads):
    """The oracle port of the same small-model request on the host cores (+ the log-mel front end timed on its own)."""
    import torch

    from oracle import logmel as om
    from oracle.whisper_ref import WhisperOracle
    from willow_inference_server_b200 import weights as W

    dims = W.WhisperDims.for_size(size)
    tensors = W.synth_engine_tensors(dims, **SYNTH_KW)
    torch.set_num_threads(n_threads)
    oracle = WhisperOracle(dims, tensors)
    n_out = n_out_for(len(pcm))
    t0 = time.perf_counter()
    mel = om.log_mel_spectrogram(om.pad_or_trim(pcm))[None]
    t_mel = time.perf_counter() - t0
    res = oracle.generate(mel, [PROMPT], beam_size=beam, max_length=2 * n_out, suppress_tokens=(-1, dims.eot))
    dt = time.perf_counter() - t0
    return {"kind": "port", "cores": n_threads, "seconds": round(dt, 3), "logmel_seconds": round(t_mel, 4),
            "value": round(len(pcm) / 16000.0 / dt, 3), "unit": "x realtime", "tokens": res[0].sequences_ids[0][:8],
            "sample": "1 request, fp32 torch oracle port incl. the numpy restatement of wis.audio.log_mel_spectrogram "
                      "(/root/reference is not on the GPU box; published anchor: base / beam 1 / 3.84 s = 245 ms on 16 cores, README.md:100)"}


def run_ours(args):
    import torch
    import torch.distributed as dist

    from willow_inference_server_b200 import _lib, audio, models, weights as W

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dims = W.WhisperDims.for_size(MODEL)
    # ---- load: rank 0 builds the blob, everyone receives it over NCCL (the only collective in the system)
    from willow_inference_server_b200 import parallel

    t0 = time.time()
    if rank == 0:
        host, tensors = make_blob_host(dims)
    else:
        host, tensors = torch.empty(0, dtype=torch.uint8), None
    torch.cuda.synchronize()
    tb = time.time()
    blob_dev = parallel.broadcast_blob(host, torch.device("cuda", local))
    torch.cuda.synchronize()
    t_bcast = (time.time() - tb) if world > 1 else None
    handle = _lib.Handle.from_device(blob_dev.data_ptr(), blob_dev.numel(), local, keepalive=blob_dev)
    load_s = time.time() - t0
    os.environ["WISB_DEVICE"] = str(local)
    for kv in args.opt:
        k, v = kv.split("=")
        handle.set_option(k, int(v))

    pcm = synth_utterance(AUDIO_SAMPLES, seed=1234 + rank)
    pcm_dev = torch.from_numpy(pcm).cuda()
    prompts = np.array([PROMPT], np.int32)
    off, ns = np.zeros(1, np.int64), np.array([AUDIO_SAMPLES], np.int32)
    extra = [dims.eot]

    def step_device():
        handle.logmel(pcm_dev.data_ptr(), off, ns, to_host=False, keep=True, pcm_on_device=True, pcm_dtype=_lib.PCM_F32, B=1)
        t_l = handle.timing()["logmel_ms"]
        ids, scores = handle.generate(None, prompts, BEAM, 1.0, 1.0, MAX_LENGTH, extra, B=1)
        t = handle.timing()
        return ids, scores, t_l + t["generate_ms"], t

    # reuse_encoder=False: the same utterance is replayed every step, nothing may be skipped behind the benchmark's back
    model = models.Whisper(None, device="cuda", _handles=[handle], reuse_encoder=False)
    pcm_pin = torch.from_numpy(pcm).pin_memory().numpy()

    def step_e2e():
        mel = audio.log_mel_spectrogram(pcm_pin).numpy()[None]  # H2D pcm, D2H mel (what WIS does, main.py:613-616)
        res = model.generate(models.StorageView.from_array(mel), [PROMPT], beam_size=BEAM, max_length=MAX_LENGTH,
                             suppress_tokens=[-1, dims.eot])  # H2D mel, D2H ids
        return res[0].sequences_ids[0], mel

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (graph capture, allocations)
    for _ in range(max(args.warmup, 3)):
        ids, _, _, _ = step_device()
    assert len(ids[0]) == N_OUT, f"decode length {len(ids[0])} != pinned {N_OUT}"
    for _ in range(2):
        e_ids, _ = step_e2e()
    assert e_ids == ids[0], "host-buffer path and device-resident path disagree"
    gpu_tokens = [int(t) for t in ids[0]]

    # ---- timed region 1: device-resident inputs
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    w0 = time.perf_counter()
    dev_ms, launches, stage = 0.0, 0, {}
    for _ in range(args.steps):
        ids, scores, ms, t = step_device()
        dev_ms += ms
        launches += int(t["launches"]) + 3
        for k in ("encoder_ms", "cross_kv_ms", "decode_ms", "logmel_ms", "h2d_ms"):
            stage[k] = stage.get(k, 0.0) + t[k]
    barrier()
    wall_dev = time.perf_counter() - w0
    # ---- timed region 2: end to end through the reference-facing surface
    barrier()
    w0 = time.perf_counter()
    for _ in range(args.steps):
        e_ids, e_mel = step_e2e()
    barrier()
    wall_e2e = time.perf_counter() - w0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"tokens": np.asarray(ids, np.float64), "scores": np.asarray(scores, np.float64),
                                         "e2e_tokens": np.asarray([e_ids], np.float64), "e2e_log_mel": e_mel})

    # ---- kernel-level profile pass (not timed): per-family CUDA-event sums
    handle.set_option("profile", 1)
    prof = {}
    for _ in range(3):
        _, _, _, t = step_device()
        for k in ("gemm_ms", "attn_ms", "ln_ms", "conv1_ms", "gemm_launches", "encoder_ms", "cross_kv_ms"):
            prof[k] = prof.get(k, 0.0) + t[k] / 3
    handle.set_option("profile", 0)

    # ---- configs[3] (8 ranks): 512 x 10 s utterances, 64 per GPU, one shared-pass engine call per rank
    configs3 = None
    if world == 8 and not args.no_extra:
        configs3 = bench_configs3_rank(handle, dims, torch.device("cuda", local), dist, rank, world)

    if world > 1:
        tt = torch.tensor([dev_ms, wall_dev, wall_e2e], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dev_ms, wall_dev, wall_e2e = tt.tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk, pk_src = peaks()
    flops, n_gemm = encoder_gemm_flops(dims)
    gemm_tf = flops / (prof["gemm_ms"] * 1e-3) / 1e12 if prof.get("gemm_ms") else None
    peak_tf = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
    ms_per_step = dev_ms / args.steps
    value = world * AUDIO_SECONDS / (ms_per_step * 1e-3)
    e2e_value = world * AUDIO_SECONDS * args.steps / wall_e2e
    dec_bytes = decoder_pass_bytes(dims, 1)
    steps_per = int(t["decode_steps"])  # decoder passes per utterance (prompt prefix in one pass + N_OUT search steps)
    dec_traffic, dec_traffic_src = ncu_dram_traffic_per_launch("r02_dec_pass_mma_kernel_full.csv", "r02_dec_pass_kernel_full.csv", "r01_dec_pass_kernel_full.csv")
    gemm_traffic, gemm_traffic_src = ncu_dram_traffic_per_launch("r02_gemm_tc_full.csv", "r01_gemm_tc_full.csv")
    out = {
        "metric": "Whisper large-v2 realtime multiple (audio s / s), beam 5, 3.84 s utterance",
        "value": round(value, 2), "unit": "x realtime", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": round(ms_per_step, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": "whisper-large-v2 beam=5, 3.84 s synthetic 16 kHz utterance, 1 utterance per GPU per step "
                               "(BASELINE.json configs[1])",
                   "model": MODEL, "beam": BEAM, "prompt_len": 4, "generated_tokens": N_OUT, "decoder_passes": steps_per,
                   "weights": f"seeded synthetic (seed {SEED}, peaked output distribution), fp16 weights / fp32 accumulate",
                   "l2": "no explicit flush: each step streams 3.1 GB of weights (>> 126 MB L2)",
                   "timer": "CUDA events on the library's launching stream (wisb_get_timing), max over ranks",
                   "parallelism": f"dp{world} (independent utterances, weights broadcast once over NCCL)"},
        "p50_latency_ms": round(ms_per_step, 3),
        "wall_ms_per_step": round(1e3 * wall_dev / args.steps, 3),
        "stages_ms": {k: round(v / args.steps, 3) for k, v in stage.items()},
        "e2e": {"value": round(e2e_value, 2), "unit": "x realtime",
                "h2d_bytes_per_step": int(AUDIO_SAMPLES * 4 + 80 * 3000 * 4 + 4 * 4),
                "d2h_bytes_per_step": int(80 * 3000 * 4 + N_OUT * 4 + 8), "ms_per_step": round(1e3 * wall_e2e / args.steps, 3)},
        "gpu_launches": launches,
        "clocks": clocks,
        # dominant kernel of the step: the persistent decoder pass; HBM-bound weight streaming (bytes per pass: decoder_pass_bytes)
        "roofline": {"bound": "hbm", "kernel": "dec_pass_mma_kernel<5> (persistent decoder pass on the warp-level tensor path, one launch per generated token)",
                     "achieved": round(dec_bytes * steps_per / (stage["decode_ms"] / args.steps * 1e-3) / 1e9, 1),
                     "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": None,
                     "traffic": dec_traffic,
                     "traffic_note": f"dram bytes per launch from the ncu --set full capture in profiles/{dec_traffic_src}",
                     "peak_source": pk_src + " hbm_gbs",
                     "algorithmic_bytes_per_launch": dec_bytes,
                     "algorithmic_bytes_formula": "2 (14 L d^2 + V d) + 4 L 1500 d  (fp16 weights + one utterance's cross K/V)",
                     "launches_per_step": steps_per,
                     "avg_launch_ms": round(stage["decode_ms"] / args.steps / steps_per, 4),
                     "timing_note": "CUDA events around the decode stage on the launching stream / passes; the stage also holds "
                                    "the small search kernels of every pass (about 2 % of it)"},
        "encoder_roofline": {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05, encoder + cross-K/V GEMMs)",
                             "achieved": round(gemm_tf, 1) if gemm_tf else None, "peak": peak_tf, "unit": "TFLOP/s",
                             "frac": round(gemm_tf / peak_tf, 4) if gemm_tf else None,
                             "traffic": gemm_traffic,
                             "traffic_note": f"bytes per launch, mean of the ncu --set full capture in profiles/{gemm_traffic_src}",
                             "peak_source": pk_src + " bf16_tflops_sustained (kernel timed inside a long step)",
                             "algorithmic_flops_per_step": flops, "launches_per_step": n_gemm,
                             "avg_launch_ms": round(prof["gemm_ms"] / n_gemm, 4) if prof.get("gemm_ms") else None,
                             "encoder_share": {k: round(prof[k], 3) for k in ("gemm_ms", "attn_ms", "ln_ms", "conv1_ms")}},
        "load": {"seconds": round(load_s, 1), "nccl_broadcast_s": round(t_bcast, 3) if t_bcast else None,
                 "blob_gb": round(blob_dev.numel() / 1e9, 2)},
    }
    out["roofline"]["frac"] = round(out["roofline"]["achieved"] / pk["hbm_gbs"], 4)
    if configs3 is not None:
        out["configs3"] = configs3
    if world == 1 and not args.no_extra:
        try:
            out["configs2"] = bench_configs2(handle, dims, torch.device("cuda", local))
        except Exception as e:  # an extra config must never take the headline down
            out["configs2"] = {"error": repr(e)[:300]}
    if not args.no_cpu_baseline and world == 1:
        del tensors, host  # free the host copies before the CPU leg builds its own fp32 model
        out["cpu_baseline"] = cpu_baseline_subprocess()
        toks = out["cpu_baseline"].get("tokens")
        # full-size parity: the fp32 CPU oracle decodes the same utterance with the same weights
        out["tokens_identical_to_cpu_oracle"] = (toks == gpu_tokens) if toks is not None else None
        out["gpu_tokens"] = gpu_tokens
    if world == 1 and not args.no_extra:
        handle.close()
        del blob_dev
        torch.cuda.empty_cache()
        threads = cpu_threads()
        try:
            c4, _, _ = bench_small_model("medium", 1, 480000, local, reps=7)
            c4["workload"] = ("whisper-medium beam=1, one 30 s window, request latency (BASELINE.json configs[4]: the WebRTC path runs "
                              "do_whisper on the whole recording at `stop`, main.py:935-971)")
            out["configs4"] = c4
        except Exception as e:
            out["configs4"] = {"error": repr(e)[:300]}
        try:
            flac = os.path.join(ROOT, "tests", "golden", "client_3sec.flac")
            c0, _, pcm0 = bench_small_model("base", 1, 0, local, reps=7, flac=flac)
            c0["workload"] = "whisper-base greedy (beam=1) on client/3sec.flac, FLAC decode + log-mel + generate (BASELINE.json configs[0])"
            if not args.no_cpu_baseline:
                c0["cpu_baseline"] = cpu_port_small("base", 1, pcm0, threads)
                c0["tokens_identical_to_cpu_oracle"] = c0["cpu_baseline"]["tokens"] == c0["tokens"]
            out["configs0"] = c0
        except Exception as e:
            out["configs0"] = {"error": repr(e)[:300]}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, arrays):
    """What the timed path handed its caller in its last step, one float32 / float64 .npy per array (token ids are exact
    in float64).  The inputs are seeded, so two builds run with the same arguments can be compared array for array."""
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20, "dumped outputs exceed 64 MB"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def bench_configs3_rank(handle, dims, device, dist, rank, world, reps=2):
    """BASELINE.json configs[3]: large-v2 beam 5, 512 x 10 s utterances over 8 GPUs = 64 per GPU, each rank one engine call;
    then (rank 0 only, the other ranks idle) the reference's own mode: ONE process, models.Whisper(device_index=[0..7]) behind
    the cross-request batcher."""
    import torch

    from willow_inference_server_b200 import _lib, models

    B, n = 64, 160000
    pcm = [synth_utterance(n, 5000 + rank * B + i) for i in range(B)]
    flat = torch.from_numpy(np.concatenate(pcm)).to(device)
    off = (np.arange(B) * n).astype(np.int64)
    ns = np.full(B, n, np.int32)
    prompts = np.asarray([PROMPT] * B, np.int32)
    ml = 2 * n_out_for(n)

    def step():
        handle.logmel(flat.data_ptr(), off, ns, to_host=False, keep=True, pcm_on_device=True, pcm_dtype=_lib.PCM_F32, B=B)
        tl = handle.timing()["logmel_ms"]
        handle.generate(None, prompts, BEAM, 1.0, 1.0, ml, [dims.eot], B=B)
        return tl + handle.timing()["generate_ms"]

    step()
    dist.barrier()
    ms = [step() for _ in range(reps)]
    tt = torch.tensor([float(np.mean(ms))], dtype=torch.float64, device=device)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    audio_s = world * B * n / 16000.0
    res = {"workload": "whisper-large-v2 beam=5, 512 x 10 s utterances, 64 per GPU (BASELINE.json configs[3])",
           "torchrun": {"value": round(audio_s / (tt.item() * 1e-3), 1), "unit": "x realtime", "ms_per_batch_max_over_ranks": round(tt.item(), 2)},
           "generated_tokens": n_out_for(n)}
    # one process driving all 8 GPUs (what WIS does: ctranslate2 device_index=[0..N-1], main.py:295,346)
    dist.barrier()
    if rank == 0:
        try:
            from willow_inference_server_b200 import audio
            from willow_inference_server_b200.batcher import TranscribeBatcher

            # replicas 1..7 need their own copy of the weights in this process (the other ranks' copies live in other processes)
            host, _ = make_blob_host(dims, pinned=True)
            hs = [handle] + [_lib.Handle.from_host(host.numpy(), d) for d in range(1, world)]
            del host
            m = models.Whisper(None, device="cuda", device_index=list(range(world)), _handles=hs, reuse_encoder=False)
            all_pcm = [synth_utterance(n, 5000 + i) for i in range(world * B)]
            mel = audio.log_mel_batch(all_pcm, handle)
            feats = models.StorageView.from_array(mel)
            kw = dict(beam_size=BEAM, max_length=ml, suppress_tokens=[-1, dims.eot])
            m.generate(feats, [PROMPT] * (world * B), **kw)
            t0 = time.perf_counter()
            m.generate(feats, [PROMPT] * (world * B), **kw)
            dt = time.perf_counter() - t0
            res["in_process_device_index_list"] = {"value": round(audio_s / dt, 1), "unit": "x realtime (generate on host features, wall clock)",
                                                   "seconds": round(dt, 3)}
            with TranscribeBatcher(m, max_batch=world * B, max_wait_ms=20) as b:
                t0 = time.perf_counter()
                futs = [b.submit(mel[i : i + 1], PROMPT, **kw) for i in range(world * B)]
                [f.result(timeout=600) for f in futs]
                dt = time.perf_counter() - t0
            res["in_process_batcher_512_requests"] = {"value": round(audio_s / dt, 1), "unit": "x realtime (512 single-window requests, wall clock)",
                                                      "seconds": round(dt, 3), "engine_calls": b.stats["engine_calls"]}
            for h_ in hs[1:]:
                h_.close()
        except Exception as e:
            res["in_process_device_index_list"] = {"error": repr(e)[:300]}
    dist.barrier()
    return res


CPU_THREADS_MAX = 32  # more OpenMP threads than this slow the small decoder GEMVs down on many-core hosts


def cpu_threads() -> int:
    return max(1, min(os.cpu_count() or 1, CPU_THREADS_MAX))


def cpu_baseline_subprocess(timeout_s: int = 420) -> dict:
    """Run the CPU leg in its own process so that a slow host cannot take the GPU result down with it."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-baseline-only"], capture_output=True, text=True,
                           timeout=timeout_s)
        line = [l for l in r.stdout.splitlines() if l.startswith("{")]
        if r.returncode == 0 and line:
            return json.loads(line[-1])
        return {"value": None, "unit": "x realtime", "cores": cpu_threads(), "kind": "port", "sample": "failed: " + r.stderr[-300:]}
    except subprocess.TimeoutExpired:
        return {"value": None, "unit": "x realtime", "cores": cpu_threads(), "kind": "port",
                "sample": f"oracle port did not finish one utterance within {timeout_s} s on this host"}


def cpu_baseline(dims, tensors, steps=1):
    """The oracle port of the reference path (fp32 torch on the host cores) on the same utterance/config."""
    import torch

    from oracle import logmel as om
    from oracle.whisper_ref import WhisperOracle

    cores = cpu_threads()
    torch.set_num_threads(cores)
    oracle = WhisperOracle(dims, tensors)
    pcm = synth_utterance(AUDIO_SAMPLES, seed=1234)
    t0 = time.perf_counter()
    for _ in range(steps):
        mel = om.log_mel_spectrogram(om.pad_or_trim(pcm))[None]
        res = oracle.generate(mel, [PROMPT], beam_size=BEAM, max_length=MAX_LENGTH, suppress_tokens=(-1, dims.eot))
    dt = (time.perf_counter() - t0) / steps
    assert len(res[0].sequences_ids[0]) == N_OUT
    return {"value": round(AUDIO_SECONDS / dt, 4), "unit": "x realtime", "cores": cores, "kind": "port",
            "sample": f"{steps} utterance(s) of the same workload (log-mel + large-v2 encoder + {N_OUT}-token beam-5 decode), "
                      f"fp32 torch oracle, {cores} threads; ctranslate2 is not installable here (no wheel, no network)",
            "seconds_per_utterance": round(dt, 2), "tokens": res[0].sequences_ids[0]}


# --------------------------------------------------------------------------------------------------------------- reference arm
def probe_ctranslate2():
    """BASELINE.md section 3 steps 1-2: is the reference's own engine on this box?  Looks for an importable ctranslate2
    (site-packages or baseline/_ref) and a converted large-v2 model directory.  Returns (module, model_dir) or (None, why)."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(ref) and ref not in sys.path:
        sys.path.insert(0, ref)
    try:
        import ctranslate2  # noqa: F401
    except Exception as e:  # ModuleNotFoundError in this image
        return None, f"import ctranslate2 failed ({type(e).__name__})"
    import ctranslate2

    cands = []
    for base in (os.path.join(ROOT, "models"), os.path.join(ref, "models"), "/models", os.path.join(ROOT, "baseline", "models")):
        for name in ("tovera-wis-whisper-large-v2", "tovera-wis-whisper-large", "whisper-large-v2-ct2", "large-v2"):
            cands.append(os.path.join(base, name))
    for c in cands:
        if os.path.isfile(os.path.join(c, "model.bin")):
            return ctranslate2, c
    return None, "ctranslate2 imports but no converted large-v2 model directory (model.bin) was found"


def run_reference_ct2(args, ct2, model_dir):
    """The reference path verbatim (main.py:297-301, 349-355): CTranslate2 on the host cores, int8, inter = intra = cores // 2,
    fed by the log-mel restatement (the reference's wis/audio.py is not on the GPU box)."""
    from oracle import logmel as om

    cores = os.cpu_count() or 2
    half = max(1, cores // 2)
    model = ct2.models.Whisper(model_dir, device="cpu", compute_type="int8", inter_threads=half, intra_threads=half)
    pcm = synth_utterance(AUDIO_SAMPLES, seed=1234)

    def step():
        mel = om.log_mel_spectrogram(om.pad_or_trim(pcm))[None].astype(np.float32)
        return model.generate(ct2.StorageView.from_array(np.ascontiguousarray(mel)), [PROMPT], beam_size=BEAM,
                              max_length=MAX_LENGTH, suppress_tokens=[-1, 50257], return_scores=False)

    for _ in range(max(1, args.warmup)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    return dt, {"kind": "ct2", "cores": cores,
                "sample": f"CTranslate2 {getattr(ct2, '__version__', '?')} int8 on the host cores, inter_threads = intra_threads = {half} "
                          f"(main.py:297-301, 349-355), real weights from {model_dir}, each step = 1 utterance"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ct2, where = probe_ctranslate2()
    if ct2 is not None:
        dt, base = run_reference_ct2(args, ct2, where)
        probe_note = f"ctranslate2 found, model {where}"
    else:
        probe_note = where
        from willow_inference_server_b200 import weights as W

        dims = W.WhisperDims.for_size(MODEL)
        tensors = W.synth_engine_tensors(dims, **SYNTH_KW)
        import torch

        from oracle import logmel as om
        from oracle.whisper_ref import WhisperOracle

        cores = cpu_threads()
        torch.set_num_threads(cores)
        oracle = WhisperOracle(dims, tensors)
        pcm = synth_utterance(AUDIO_SAMPLES, seed=1234)

        def step():
            mel = om.log_mel_spectrogram(om.pad_or_trim(pcm))[None]
            return oracle.generate(mel, [PROMPT], beam_size=BEAM, max_length=MAX_LENGTH, suppress_tokens=(-1, dims.eot))

        # warm-up is bounded too (a step is ~10-20 s of host work): at least one step, then stop after ~30 s
        t_w = time.perf_counter()
        warmed = 0
        while warmed < args.warmup and (warmed == 0 or time.perf_counter() - t_w < 30.0):
            step()
            warmed += 1
        args.warmup = warmed
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        dt = (time.perf_counter() - t0) / args.steps
        base = {"kind": "port", "cores": cores,
                "sample": f"each step = 1 utterance of the same workload on the host cores (fp32 torch oracle port, {cores} threads); "
                          "the reference's own engine, ctranslate2==4.1.0, is an un-vendored pip dependency that is absent from "
                          "this image and cannot be installed offline"}
    v = round(AUDIO_SECONDS / dt, 4)
    print(json.dumps({
        "impl": "reference", "metric": "Whisper large-v2 realtime multiple (audio s / s), beam 5, 3.84 s utterance",
        "value": v, "unit": "x realtime", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt * 1e3, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int8" if base["kind"] == "ct2" else "f32", "data": "synthetic",
        "config": {"workload": "whisper-large-v2 beam=5, 3.84 s synthetic 16 kHz utterance (BASELINE.json configs[1])",
                   "model": MODEL, "beam": BEAM, "generated_tokens": N_OUT},
        "reference_probe": probe_note,
        "cpu_baseline": dict(base, value=v, unit="x realtime"),
        "e2e": {"value": v, "unit": "x realtime", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="headline config only (skip configs0 / 2 / 3 / 4)")
    ap.add_argument("--opt", action="append", default=[], help="engine option key=value (diagnostics), e.g. --opt mega_barrier=1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step returned "
                    "(token ids, beam scores, the end-to-end path's log-mel features) to DIR/<name>.npy")
    ap.add_argument("--cpu-baseline-only", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.cpu_baseline_only:
        from willow_inference_server_b200 import weights as W

        dims = W.WhisperDims.for_size(MODEL)
        print(json.dumps(cpu_baseline(dims, W.synth_engine_tensors(dims, **SYNTH_KW), steps=1)))
        return
    if args.impl == "reference":
        args.warmup = min(args.warmup, 1)
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
