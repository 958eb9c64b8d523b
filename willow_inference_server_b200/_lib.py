"""ctypes binding of libwisb200.so (include/wisb200.h).  No CPU fallback: a missing library or a missing CUDA
device is an error, never a silent downgrade."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libwisb200.so")

N_DIMS = 20
DIM_NAMES = [
    "d_model", "n_heads", "n_enc_layers", "n_dec_layers", "n_vocab", "n_vocab_pad", "n_text_ctx", "n_mels",
    "n_audio_ctx", "sot", "eot", "transcribe", "translate", "no_timestamps", "sot_prev", "sot_lm", "no_speech",
    "blank", "lang_first", "n_langs",
]
PCM_F32, PCM_S16 = 0, 1

_lib = None

_SIGS = {
    "wisb_abi_version": (C.c_int, []),
    "wisb_last_error": (C.c_char_p, []),
    "wisb_create": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]),
    "wisb_create_from_host": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]),
    "wisb_create_from_device": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]),
    "wisb_create_frontend": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "wisb_destroy": (C.c_int, [C.c_void_p]),
    "wisb_get_dims": (C.c_int, [C.c_void_p, C.c_void_p]),
    "wisb_logmel": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "wisb_generate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float,
                                C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "wisb_generate_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float,
                                   C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "wisb_generate_ts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float,
                                   C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                   C.c_void_p]),
    "wisb_detect_language": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "wisb_get_timing": (C.c_int, [C.c_void_p, C.c_void_p]),
    "wisb_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "wisb_debug_gemm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "wisb_debug_gemv_tc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_void_p]),
    "wisb_debug_read_trace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "wisb_debug_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "wisb_debug_forced_logits": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "wisb_flac_last_error": (C.c_char_p, []),
    "wisb_flac_info": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wisb_flac_decode": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int64, C.c_void_p]),
}
EXPORTS = sorted(_SIGS)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `python willow_inference_server_b200/build.py`). There is no CPU / PyTorch fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)  # AttributeError here = the .so does not match include/wisb200.h
            fn.restype = res
            fn.argtypes = args
        if l.wisb_abi_version() != 1:
            raise ImportError("libwisb200.so ABI version mismatch")
        _lib = l
    return _lib


def check(rc: int):
    if rc == 0:
        return
    msg = lib().wisb_last_error().decode("utf-8", "replace")
    if rc == 1:
        raise ValueError(msg)
    raise RuntimeError(msg)


def ptr(a):
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


class Handle:
    """Owns one wisb_handle (one model replica or one front end on one GPU)."""

    def __init__(self, raw, keepalive=None):
        self._h = raw
        self._keep = keepalive

    @classmethod
    def from_path(cls, path: str, device: int = 0):
        h = C.c_void_p()
        check(lib().wisb_create(path.encode(), device, C.byref(h)))
        return cls(h)

    @classmethod
    def from_host(cls, blob: np.ndarray, device: int = 0):
        blob = np.ascontiguousarray(blob, np.uint8)
        h = C.c_void_p()
        check(lib().wisb_create_from_host(ptr(blob), blob.size, device, C.byref(h)))
        return cls(h)

    @classmethod
    def from_device(cls, dev_ptr: int, nbytes: int, device: int = 0, keepalive=None):
        h = C.c_void_p()
        check(lib().wisb_create_from_device(C.c_void_p(dev_ptr), nbytes, device, C.byref(h)))
        return cls(h, keepalive)

    @classmethod
    def frontend(cls, device: int = 0):
        h = C.c_void_p()
        check(lib().wisb_create_frontend(device, C.byref(h)))
        return cls(h)

    def close(self):
        if self._h:
            lib().wisb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ calls
    def dims(self) -> dict:
        out = np.zeros(N_DIMS, np.int32)
        check(lib().wisb_get_dims(self._h, ptr(out)))
        return dict(zip(DIM_NAMES, (int(v) for v in out)))

    def set_option(self, key: str, value: int):
        check(lib().wisb_set_option(self._h, key.encode(), int(value)))

    def timing(self) -> dict:
        out = np.zeros(16, np.float32)
        check(lib().wisb_get_timing(self._h, ptr(out)))
        keys = ["logmel_ms", "h2d_ms", "encoder_ms", "cross_kv_ms", "decode_ms", "generate_ms", "decode_steps", "launches",
                "gemm_ms", "attn_ms", "ln_ms", "conv1_ms", "gemm_launches"]
        return dict(zip(keys, (float(v) for v in out)))

    def logmel(self, pcm, offsets, n_samples, *, to_host=True, keep=False, pcm_on_device=False, pcm_dtype=None, B=None):
        offsets = np.ascontiguousarray(offsets, np.int64)
        n_samples = np.ascontiguousarray(n_samples, np.int32)
        B = int(offsets.shape[0]) if B is None else B
        if pcm_on_device:
            p, dt = C.c_void_p(int(pcm)), pcm_dtype
        else:
            if pcm.dtype == np.int16:
                dt = PCM_S16
            elif pcm.dtype == np.float32:
                dt = PCM_F32
            else:
                raise ValueError("pcm must be float32 or int16")
            pcm = np.ascontiguousarray(pcm)
            p = ptr(pcm)
        out = np.empty((B, 80, 3000), np.float32) if to_host else None
        check(lib().wisb_logmel(self._h, p, dt, 1 if pcm_on_device else 0, ptr(offsets), ptr(n_samples), B, ptr(out),
                                1 if keep else 0))
        return out

    def generate(self, mel, prompts, beam_size=5, patience=1.0, length_penalty=1.0, max_length=448, extra_suppress=(),
                 B=None, timestamps=False, max_initial_timestamp_index=50):
        """-> (token ids per window, scores).  ``timestamps=True`` applies Whisper's timestamp rules (wisb_generate_ts):
        the prompts must not contain <|notimestamps|>, and the ids keep the timestamp tokens."""
        prompts = np.ascontiguousarray(prompts, np.int32)
        if prompts.ndim != 2:
            raise ValueError("prompts must be [B, prompt_len]")
        if mel is not None:
            if mel.dtype != np.float32 or mel.ndim != 3 or mel.shape[1:] != (80, 3000) or not mel.flags["C_CONTIGUOUS"]:
                raise ValueError("features must be a C-contiguous float32 array of shape [n, 80, 3000]")
            B = mel.shape[0]
        if B is None or prompts.shape[0] != B:
            raise ValueError("one prompt per feature window is required")
        per_utt = None
        if not np.isscalar(max_length):  # one limit per utterance (requests coalesced by the batcher)
            per_utt = np.ascontiguousarray(max_length, np.int32)
            if per_utt.shape != (B,):
                raise ValueError("max_length must be an int or one int per utterance")
            max_length = int(per_utt.max())
        stride = max(1, int(max_length) // 2)
        ids = np.zeros((B, stride), np.int32)
        lens = np.zeros(B, np.int32)
        scores = np.zeros(B, np.float32)
        extra = np.ascontiguousarray(list(extra_suppress), np.int32)
        if timestamps:
            check(lib().wisb_generate_ts(self._h, ptr(mel), B, ptr(prompts), prompts.shape[1], int(beam_size),
                                         float(patience), float(length_penalty), int(max_length), ptr(per_utt),
                                         ptr(extra) if extra.size else None, extra.size, int(max_initial_timestamp_index),
                                         ptr(ids), stride, ptr(lens), ptr(scores)))
        else:
            check(lib().wisb_generate_ex(self._h, ptr(mel), B, ptr(prompts), prompts.shape[1], int(beam_size),
                                         float(patience), float(length_penalty), int(max_length), ptr(per_utt),
                                         ptr(extra) if extra.size else None, extra.size, ptr(ids), stride, ptr(lens),
                                         ptr(scores)))
        return [ids[b, : lens[b]].tolist() for b in range(B)], scores.tolist()

    def detect_language(self, mel, B=None):
        if mel is not None:
            B = mel.shape[0]
        nl = self.dims()["n_langs"]
        ids = np.zeros((B, nl), np.int32)
        probs = np.zeros((B, nl), np.float32)
        check(lib().wisb_detect_language(self._h, ptr(mel), B, ptr(ids), ptr(probs)))
        return ids, probs

    # ------------------------------------------------------------------ diagnostics (tests)
    def debug_gemm(self, a16: np.ndarray, w16: np.ndarray, impl: int = 0, bn: int = 0) -> np.ndarray:
        a16 = np.ascontiguousarray(a16, np.float16)
        w16 = np.ascontiguousarray(w16, np.float16)
        M, K = a16.shape
        N = w16.shape[0]
        c = np.zeros((M, N), np.float32)
        check(lib().wisb_debug_gemm(self._h, ptr(a16), ptr(w16), ptr(c), M, N, K, impl, bn))
        return c

    def debug_gemv_tc(self, x: np.ndarray, w16: np.ndarray, bias=None, iters: int = 0):
        """tcgen05 skinny GEMV on caller data -> (out float32 [R, N], average kernel time in us over `iters` launches)."""
        x = np.ascontiguousarray(x, np.float32)
        w16 = np.ascontiguousarray(w16, np.float16)
        R, K = x.shape
        N = w16.shape[0]
        out = np.zeros((R, N), np.float32)
        us = C.c_float(0.0)
        b = None if bias is None else np.ascontiguousarray(bias, np.float32)
        check(lib().wisb_debug_gemv_tc(self._h, ptr(x), ptr(w16), ptr(b), ptr(out), R, N, K, int(iters), C.byref(us)))
        return out, float(us.value)

    def debug_read_trace(self, n: int = 600) -> np.ndarray:
        out = np.zeros(n, np.uint64)
        check(lib().wisb_debug_read_trace(self._h, ptr(out), n))
        return out

    def debug_encode(self, mel: np.ndarray, n_layers: int = -1) -> np.ndarray:
        mel = np.ascontiguousarray(mel, np.float32)
        out = np.zeros((mel.shape[0], 1500, self.dims()["d_model"]), np.float32)
        check(lib().wisb_debug_encode(self._h, ptr(mel), mel.shape[0], ptr(out), n_layers))
        return out

    def debug_forced_logits(self, mel: np.ndarray, tokens) -> np.ndarray:
        mel = np.ascontiguousarray(mel, np.float32)
        tokens = np.ascontiguousarray(tokens, np.int32)
        out = np.zeros((tokens.shape[0], self.dims()["n_vocab"]), np.float32)
        check(lib().wisb_debug_forced_logits(self._h, ptr(mel), ptr(tokens), tokens.shape[0], ptr(out)))
        return out


def flac_decode(data: bytes):
    """FLAC stream -> (int32 ndarray [n_frames, channels], sample_rate, bits_per_sample, md5 bytes).  Host code only."""
    l = lib()
    buf = np.frombuffer(data, np.uint8)
    sr, ch, bps, n = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
    md5 = (C.c_uint8 * 16)()
    if l.wisb_flac_info(buf.ctypes.data, buf.size, C.byref(sr), C.byref(ch), C.byref(bps), C.byref(n), md5):
        raise ValueError("FLAC: " + l.wisb_flac_last_error().decode())
    # STREAMINFO is untrusted input: a frame is >= 9 bytes and carries <= 65535 samples per channel, so the stream
    # cannot hold more inter-channel samples than that, whatever the header claims (and 2^30 samples is the hard cap)
    bound = (buf.size // 9 + 1) * 65535
    if n.value < 0 or n.value > bound or n.value * max(ch.value, 1) > (1 << 30):
        raise ValueError(f"FLAC: STREAMINFO announces {n.value} samples, impossible for a {buf.size}-byte stream")
    out = np.zeros((n.value, ch.value), np.int32)
    got = C.c_int64()
    if l.wisb_flac_decode(buf.ctypes.data, buf.size, out.ctypes.data, n.value, C.byref(got)):
        raise ValueError("FLAC: " + l.wisb_flac_last_error().decode())
    return out[: got.value], sr.value, bps.value, bytes(md5)
