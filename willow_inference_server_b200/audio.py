"""Drop-in for ``wis/audio.py`` (the names ``main.py:52-57`` imports), running on the B200.

    from willow_inference_server_b200.audio import (
        log_mel_spectrogram, pad_or_trim, chunk_iter, find_longest_common_sequence)

* ``log_mel_spectrogram`` replaces /root/reference/wis/audio.py:72-103: same argument (float32 numpy PCM), returns an
  object with ``.numpy()`` -> float32 [80, n_frames] exactly as the call sites use it (main.py:608,614).  The STFT /
  mel / log pipeline runs in the CUDA kernel csrc/logmel.cu; there is no CPU path.
* ``pad_or_trim`` (wis/audio.py:28-51) is kept for API compatibility; the kernel fuses padding/trimming, so calling
  it first is allowed but not required (``log_mel_spectrogram`` accepts the unpadded utterance too).
* ``chunk_iter`` / ``find_longest_common_sequence`` (wis/audio.py:106-159) are host logic on token lists and are
  restated here with the same behaviour (goldens: tests/golden/host_logic.json).
"""
from __future__ import annotations

import os
import threading

import numpy as np

from . import _lib

SAMPLE_RATE = 16000
N_FFT = 400
N_MELS = 80
HOP_LENGTH = 160
CHUNK_LENGTH = 30
N_SAMPLES = CHUNK_LENGTH * SAMPLE_RATE
N_FRAMES = N_SAMPLES // HOP_LENGTH

chunk_length_s = 22
stride_length_s = [4, 4]
chunk_len = chunk_length_s * SAMPLE_RATE
stride_left = stride_length_s[0] * SAMPLE_RATE
stride_right = stride_length_s[1] * SAMPLE_RATE

_frontend = None
_frontend_lock = threading.Lock()


def _get_frontend() -> "_lib.Handle":
    global _frontend
    with _frontend_lock:
        if _frontend is None:
            _frontend = _lib.Handle.frontend(int(os.environ.get("WISB_DEVICE", "0")))
        return _frontend


class MelFeatures:
    """What the reference gets back from torch: something with ``.numpy()`` and a shape."""

    def __init__(self, arr: np.ndarray):
        self._a = arr

    def numpy(self) -> np.ndarray:
        return self._a

    @property
    def shape(self):
        return self._a.shape

    def __array__(self, dtype=None, copy=None):
        return self._a if dtype is None else self._a.astype(dtype)


def pad_or_trim(array, length: int = N_SAMPLES, *, axis: int = -1):
    array = np.asarray(array)
    n = array.shape[axis]
    if n > length:
        array = np.take(array, np.arange(length), axis=axis)
    elif n < length:
        widths = [(0, 0)] * array.ndim
        widths[axis] = (0, length - n)
        array = np.pad(array, widths)
    return array


def log_mel_spectrogram(audio, n_mels: int = N_MELS) -> MelFeatures:
    if n_mels != N_MELS:
        raise AssertionError(f"Unsupported n_mels: {n_mels}")
    if isinstance(audio, str):
        raise TypeError("log_mel_spectrogram takes PCM samples (numpy), not a path")
    pcm = np.asarray(audio)
    if pcm.dtype not in (np.float32, np.int16):
        pcm = pcm.astype(np.float32)
    if pcm.ndim != 1:
        raise ValueError("audio must be a 1-D array of 16 kHz samples")
    mel = _get_frontend().logmel(pcm, [0], [pcm.shape[0]])
    return MelFeatures(mel[0])


def log_mel_batch(pcm_list, handle=None) -> np.ndarray:
    """Batched form used by the engine-side tests/bench: list of 1-D arrays -> float32 [B, 80, 3000]."""
    h = handle or _get_frontend()
    dt = np.int16 if all(np.asarray(p).dtype == np.int16 for p in pcm_list) else np.float32
    arrs = [np.ascontiguousarray(p, dt) for p in pcm_list]
    n = np.array([a.shape[0] for a in arrs], np.int32)
    off = np.zeros(len(arrs), np.int64)
    off[1:] = np.cumsum(n[:-1])
    flat = np.concatenate(arrs) if arrs else np.zeros(0, dt)
    return h.logmel(flat, off, n)


def chunk_iter(inputs):
    """30-s windows (22 s payload + 4 s context each side, 14 s step) -- wis/audio.py:106-134."""
    if not isinstance(inputs, np.ndarray):
        raise AssertionError("chunk_iter only takes numpy array")
    total = inputs.shape[0]
    step = chunk_len - stride_left - stride_right
    for start in range(0, total, step):
        piece = inputs[start : start + chunk_len]
        left = 0 if start == 0 else stride_left
        last = start + step + stride_left >= total
        right = 0 if last else stride_right
        if piece.shape[0] > left:
            yield piece, (piece.shape[0], left, right)


def chunk_table(total: int):
    """The windows ``chunk_iter`` yields for a ``total``-sample input, as index arithmetic only:
    (offsets int64 [N], lengths int32 [N], strides [(length, left, right)] * N)."""
    step = chunk_len - stride_left - stride_right
    offs, lens, strides = [], [], []
    for start in range(0, total, step):
        n = min(chunk_len, total - start)
        left = 0 if start == 0 else stride_left
        right = 0 if start + step + stride_left >= total else stride_right
        if n > left:
            offs.append(start)
            lens.append(n)
            strides.append((n, left, right))
    return np.asarray(offs, np.int64), np.asarray(lens, np.int32), strides


def log_mel_chunks(audio, handle=None):
    """Long-audio front end (main.py:603-611 does ``[log_mel_spectrogram(pad_or_trim(c)) for c in chunk_iter(audio)]``):
    every 22-s window is framed by the log-mel kernel straight out of the one PCM buffer (offset + length per window,
    zero padding to 30 s fused), so neither the padded copies nor a [N, 480000] batch is ever materialised.
    Returns (float32 [N, 80, 3000], strides) with the strides ``chunk_iter`` would have produced."""
    pcm = np.asarray(audio)
    if pcm.dtype not in (np.float32, np.int16):
        pcm = pcm.astype(np.float32)
    if pcm.ndim != 1:
        raise ValueError("audio must be a 1-D array of 16 kHz samples")
    offs, lens, strides = chunk_table(pcm.shape[0])
    if not strides:
        return np.zeros((0, N_MELS, N_FRAMES), np.float32), strides
    return (handle or _get_frontend()).logmel(np.ascontiguousarray(pcm), offs, lens), strides


def log_mel_window(audio, handle=None):
    """One utterance of at most 30 s -> float32 [1, 80, 3000] (zero padding to the window fused in the kernel): what
    ``log_mel_spectrogram(pad_or_trim(audio)).numpy()[None]`` yields in main.py:612-617."""
    pcm = np.asarray(audio)
    if pcm.dtype not in (np.float32, np.int16):
        pcm = pcm.astype(np.float32)
    n = min(int(pcm.shape[0]), N_SAMPLES)
    return (handle or _get_frontend()).logmel(np.ascontiguousarray(pcm[:n]), [0], [n])


def transcribe_long(model, audio, prompt, tokenizer, *, beam_size: int = 5, batcher=None, max_windows_per_call: int = 64,
                    **generate_options):
    """The long-audio path of ``do_whisper`` (main.py:582-617, 676-714) on top of the pieces above: window the
    utterance, decode all windows as batch rows (the reference goes two at a time, ``concurrent_gpu_chunks``), stitch
    the token lists with ``find_longest_common_sequence``.  ``model`` is a ``models.Whisper`` (or anything with its
    ``generate``); with ``batcher`` (a ``TranscribeBatcher``) the windows join other requests' batches.
    Returns the merged token ids (numpy int array), ready for ``whisper_processor.decode``."""
    from .models import StorageView

    # Timestamps are relative to their window: stitching them with the token-level LCS merge would give wrong times, so
    # a prompt that asks for timestamps is refused (checked with the engine's ids, when it has them)
    dims = getattr(model if model is not None else getattr(batcher, "_model", None), "dims", None)
    if isinstance(dims, dict) and "no_timestamps" in dims and dims["no_timestamps"] not in list(prompt):
        raise ValueError("transcribe_long does not decode timestamps: the prompt must contain <|notimestamps|>")
    pcm = np.asarray(audio)
    if pcm.ndim == 1 and pcm.shape[0] <= N_SAMPLES:
        # <= 30 s: the reference does not window at all (main.py:587-617), it decodes one zero-padded 30-s window
        mel = log_mel_window(pcm)
        strides = [(pcm.shape[0], 0, 0)]
    else:
        mel, strides = log_mel_chunks(audio)
    if not strides:
        return np.zeros(0, np.int64)
    seqs = []
    for s in range(0, mel.shape[0], max_windows_per_call):
        part = mel[s : s + max_windows_per_call]
        if batcher is not None:
            res = batcher.submit(part, prompt, beam_size=beam_size, **generate_options).result()
        else:
            res = model.generate(StorageView.from_array(part), [list(prompt)] * part.shape[0], beam_size=beam_size,
                                 **generate_options)
        seqs += [r.sequences_ids[0] for r in res]
    if len(seqs) == 1:
        special = set(tokenizer.all_special_ids)
        return np.array([t for t in seqs[0] if t not in special])
    return find_longest_common_sequence([(ids, st) for ids, st in zip(seqs, strides)], tokenizer)


def find_longest_common_sequence(sequences, tokenizer):
    """Token-level stitch of overlapping windows -- wis/audio.py:139-159 (same scoring: fraction of matches + i/10000,
    at least two matches).  Unlike the reference this does not raise when a later window is longer than the text
    accumulated so far (numpy broadcasting error there, SURVEY.md section 5): the comparison is limited to the overlap."""
    special = set(tokenizer.all_special_ids)
    merged = [t for t in sequences[0][0] if t not in special]
    for item in sequences[1:]:
        new = [t for t in item[0] if t not in special]
        best_i, best = 0, 0.0
        for i in range(1, len(new) + 1):
            tail, head = merged[-i:], new[:i]
            # (the reference compares numpy arrays here and raises once i exceeds len(merged))
            matches = sum(1 for a, b in zip(tail, head) if a == b) if len(tail) == len(head) else 0
            score = matches / i + i / 10000.0
            if matches > 1 and score > best:
                best_i, best = i, score
        merged.extend(new[best_i:])
    return np.array(merged)


def decode_flac(src, verify: bool = True, return_bps: bool = False):
    """FLAC file path / bytes -> (pcm, sample_rate[, bits_per_sample]).  pcm: int16 (<= 16 bits per sample) or int32, shape [n] for mono,
    [n, channels] otherwise.  The decode half of ``librosa.load`` (/root/reference/main.py:579) for the FLAC inputs WIS
    is tested with; with ``verify`` the decoded PCM is checked against the MD5 the encoder stored in STREAMINFO (an
    all-zero signature means "not set" and is skipped).  Host code in libwisb200 (csrc/flac.cu); no GPU involved."""
    import hashlib

    data = src if isinstance(src, (bytes, bytearray, memoryview)) else open(src, "rb").read()
    pcm, sr, bps, md5 = _lib.flac_decode(bytes(data))
    if verify and any(md5):
        nbytes = (bps + 7) // 8
        raw = pcm.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :nbytes].tobytes()  # little-endian, sign-extended
        if hashlib.md5(raw).digest() != md5:
            raise ValueError("FLAC: decoded audio does not match the MD5 signature in STREAMINFO")
    out = pcm.astype(np.int16) if bps <= 16 else pcm
    out = out[:, 0] if out.shape[1] == 1 else out
    return (out, sr, bps) if return_bps else (out, sr)


def load_audio(src, sr: int = SAMPLE_RATE) -> np.ndarray:
    """FLAC -> float32 mono in [-1, 1) at 16 kHz, as ``librosa.load(file, sr=16000)`` returns it for inputs that are
    already sampled at 16 kHz (the reference's fixtures are).  Other rates raise: resampling stays with the caller."""
    pcm, rate, bps = decode_flac(src, return_bps=True)
    if rate != sr:
        raise ValueError(f"{rate} Hz input: resampling to {sr} Hz is not implemented here")
    # the decoder returns right-justified samples: full scale is 2^(bps-1) whatever the container width
    # (soundfile / librosa normalise the same way; 8-, 12-, 20- and 24-bit streams included)
    x = pcm.astype(np.float32) / np.float32(1 << (bps - 1))
    return x if x.ndim == 1 else x.mean(axis=1, dtype=np.float32)
