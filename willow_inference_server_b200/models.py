"""Drop-in for the part of ``ctranslate2`` that WIS calls (main.py:39, 341-355, 454, 535-537, 638-640, 685-692).

    import willow_inference_server_b200 as ctranslate2
    model = ctranslate2.models.Whisper(path, device="cuda", compute_type=..., inter_threads=..., device_index=[0..N-1])
    feats = ctranslate2.StorageView.from_array(mel)            # float32 [n, 80, 3000]
    results = model.generate(feats, [prompt] * n, beam_size=5, return_scores=False)
    results[i].sequences_ids[0]                                # list[int]
    model.detect_language(feats)[0][0]                         # ("<|en|>", prob)

Same names, argument meaning and error behaviour (ValueError for bad shapes/arguments, RuntimeError for device
failures).  What differs by design: ``device`` must be "cuda" (no CPU fallback), ``compute_type`` is accepted and
ignored (one fp16-weights / fp32-accumulate path, no multi-backend dispatch), ``model_path`` points at a WISB200 weight
blob (file, or directory containing ``model.wisb``).  ``device_index=[...]`` builds one replica per GPU; a batch is
split across the replicas (weights are read once and copied to every GPU at load; bench.py does the same step with an
NCCL broadcast when launched under torchrun).
"""
from __future__ import annotations

import os
import threading
import zlib
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from .languages import LANGUAGE_CODES


class StorageView:
    """ctranslate2.StorageView stand-in: a borrowed view of a host float32 array (main.py:638,685)."""

    def __init__(self, array: np.ndarray):
        self.array = array

    @classmethod
    def from_array(cls, array):
        a = np.asarray(array)
        if a.dtype != np.float32:
            raise ValueError(f"StorageView.from_array: unsupported dtype {a.dtype} (float32 expected)")
        if not a.flags["C_CONTIGUOUS"]:
            raise ValueError("StorageView.from_array: the array must be C-contiguous")
        return cls(a)

    @property
    def shape(self):
        return list(self.array.shape)


@dataclass
class WhisperGenerationResult:
    sequences_ids: list
    scores: list = field(default_factory=list)
    no_speech_prob: float = 0.0

    @property
    def sequences(self):  # CT2 returns token strings here; WIS never reads them (main.py:707,713 use ids)
        return [[str(t) for t in seq] for seq in self.sequences_ids]


def get_supported_compute_types(device: str, device_index: int = 0):
    """main.py:454 only logs this.  One compute path exists: fp16 weights/activations, fp32 accumulation."""
    if device != "cuda":
        raise ValueError("willow_inference_server_b200 supports device='cuda' only")
    return {"float16"}


def _features_array(features) -> np.ndarray:
    a = features.array if isinstance(features, StorageView) else np.asarray(features)
    if a.dtype != np.float32 or a.ndim != 3 or tuple(a.shape[1:]) != (80, 3000):
        raise ValueError(f"features must be float32 [n, 80, 3000], got {a.dtype} {tuple(a.shape)}")
    return np.ascontiguousarray(a)


class Whisper:
    def __init__(self, model_path, device: str = "cuda", *, device_index=0, compute_type: str = "default",
                 inter_threads: int = 1, intra_threads: int = 0, max_queued_batches: int = 0, files=None,
                 reuse_encoder=None, _handles=None, **_ignored):
        if device != "cuda":
            raise ValueError("willow_inference_server_b200.models.Whisper runs on device='cuda' only (no CPU fallback)")
        idx = [device_index] if isinstance(device_index, int) else list(device_index)
        if not idx:
            raise ValueError("device_index must name at least one GPU")
        self.device = device
        self.device_index = idx
        self.compute_type = "float16"
        if _handles is not None:
            self._handles = list(_handles)
        else:
            path = str(model_path)
            if os.path.isdir(path) and os.path.isfile(os.path.join(path, "model.wisb")):
                path = os.path.join(path, "model.wisb")
            if os.path.isfile(path):
                blob = np.fromfile(path, np.uint8)  # read once, copied to every replica
            elif os.path.isdir(path) and any(os.path.exists(os.path.join(path, f)) for f in
                                             ("model.bin", "model.safetensors", "model.safetensors.index.json",
                                              "pytorch_model.bin")):
                # a CTranslate2 directory as main.py:342 passes it, or an HF checkpoint: converted in memory
                from . import loaders, weights as _W

                dims, tensors = loaders.load_any(path)
                blob = np.zeros(_W.blob_nbytes(tensors), np.uint8)
                _W.write_blob_into(blob, dims, tensors)
            else:
                raise RuntimeError(f"Unable to open model '{path}' (expected model.wisb, a CTranslate2 model.bin "
                                   "or a Hugging Face Whisper checkpoint)")
            self._handles = [_lib.Handle.from_host(blob, d) for d in idx]
        # detect_language -> generate -> (translate) on the same window encode once (SURVEY 8f row 4); opt-in because a
        # caller that replays identical features on purpose (a benchmark) must not have work skipped behind its back
        if reuse_encoder is None:
            reuse_encoder = os.environ.get("WISB_ENCODER_CACHE", "0") not in ("", "0")
        self.reuse_encoder = bool(reuse_encoder)
        for h in self._handles:
            h.set_option("encoder_cache", 1 if self.reuse_encoder else 0)
        self._dims = self._handles[0].dims()
        self._pool = ThreadPoolExecutor(max_workers=len(self._handles)) if len(self._handles) > 1 else None
        self._rr = 0
        self._lock = threading.Lock()

    # ----------------------------------------------------------------------------------------------------------
    @property
    def is_multilingual(self) -> bool:
        return self._dims["n_vocab"] >= 51865

    @property
    def num_languages(self) -> int:
        return self._dims["n_langs"]

    @property
    def dims(self) -> dict:
        return dict(self._dims)

    def _split(self, n: int, mel=None):
        k = len(self._handles)
        if k > 1 and self.reuse_encoder and n <= 2 and mel is not None:
            # same features -> same replica, so the cached encoder output is found again
            return [(zlib.crc32(np.ascontiguousarray(mel[0, :, :64]).tobytes()) % k, 0, n)]
        if k == 1 or n == 1:
            with self._lock:
                i = self._rr % k
                self._rr += 1
            return [(i, 0, n)]
        per = -(-n // k)
        return [(i, s, min(n, s + per)) for i, s in enumerate(range(0, n, per))]

    def _run(self, jobs):
        if self._pool is None or len(jobs) == 1:
            return [fn() for fn in jobs]
        return [f.result() for f in [self._pool.submit(fn) for fn in jobs]]

    def generate(self, features, prompts, *, asynchronous: bool = False, beam_size: int = 5, patience: float = 1,
                 num_hypotheses: int = 1, length_penalty: float = 1, repetition_penalty: float = 1,
                 no_repeat_ngram_size: int = 0, max_length: int = 448, return_scores: bool = False,
                 return_no_speech_prob: bool = False, max_initial_timestamp_index: int = 50,
                 suppress_blank: bool = True, suppress_tokens=(-1,), sampling_topk: int = 1,
                 sampling_temperature: float = 1):
        """ctranslate2.models.Whisper.generate for the options WIS relies on (SURVEY.md section 8b defaults).  As in
        CTranslate2, prompts without <|notimestamps|> decode with Whisper's timestamp rules (``max_initial_timestamp_index``
        bounds the first timestamp) and ``sequences_ids`` then contain the timestamp tokens."""
        mel = _features_array(features)
        n = mel.shape[0]
        if len(prompts) != n:
            raise ValueError(f"expected {n} prompts (one per feature window), got {len(prompts)}")
        lens = {len(p) for p in prompts}
        if len(lens) != 1 or 0 in lens:
            raise ValueError("all prompts must be non-empty and of the same length")
        if isinstance(prompts[0][0], str):
            raise ValueError("prompts must be token ids (WIS builds them with convert_tokens_to_ids, main.py:656-663)")
        if num_hypotheses != 1 or repetition_penalty != 1 or no_repeat_ngram_size != 0 or sampling_topk != 1:
            raise ValueError("only num_hypotheses=1, repetition_penalty=1, no_repeat_ngram_size=0, sampling_topk=1 "
                             "(the CTranslate2 defaults WIS uses) are implemented")
        if not suppress_blank or -1 not in suppress_tokens or asynchronous:
            raise ValueError("suppress_blank=True, suppress_tokens containing -1 and asynchronous=False are required")
        # CTranslate2's switch: a prompt without <|notimestamps|> turns the timestamp rules on (main.py:529, :661)
        no_ts = self._dims["no_timestamps"]
        modes = {no_ts not in p for p in prompts}
        if len(modes) != 1:
            raise ValueError("all prompts of one call must agree on <|notimestamps|> (timestamp decoding or not)")
        timestamps = modes.pop()
        n_ts = self._dims["n_vocab"] - no_ts - 1  # timestamp tokens [no_timestamps + 1, n_vocab)
        if timestamps and not 0 <= int(max_initial_timestamp_index) < n_ts:
            raise ValueError(f"max_initial_timestamp_index must be in [0, {n_ts - 1}], got {max_initial_timestamp_index}")
        extra = [int(t) for t in suppress_tokens if t >= 0]
        p = np.asarray(prompts, np.int32)
        parts = self._split(n, mel)
        # extension over CTranslate2: `max_length` may be one int per window (requests with different limits coalesced
        # into one call by batcher.TranscribeBatcher); a plain int is the CTranslate2 meaning
        ml = None if np.isscalar(max_length) else np.asarray(max_length, np.int32)
        if ml is not None and ml.shape != (n,):
            raise ValueError("max_length must be an int or one int per feature window")

        ts_kw = {"timestamps": True, "max_initial_timestamp_index": int(max_initial_timestamp_index)} if timestamps else {}

        def job(i, s, e):
            return lambda: self._handles[i].generate(mel[s:e], p[s:e], beam_size, patience, length_penalty,
                                                     max_length if ml is None else ml[s:e], extra, **ts_kw)

        outs = self._run([job(*pt) for pt in parts])
        results = []
        for ids, scores in outs:
            for seq, sc in zip(ids, scores):
                results.append(WhisperGenerationResult([seq], [sc] if return_scores else []))
        return results

    def detect_language(self, features):
        mel = _features_array(features)
        parts = self._split(mel.shape[0], mel)

        def job(i, s, e):
            return lambda: self._handles[i].detect_language(mel[s:e])

        out = []
        first = self._dims["lang_first"]
        for ids, probs in self._run([job(*pt) for pt in parts]):
            for row_ids, row_p in zip(ids, probs):
                out.append([(f"<|{LANGUAGE_CODES[int(t) - first]}|>" if int(t) - first < len(LANGUAGE_CODES) else f"<|{int(t)}|>",
                             float(pr)) for t, pr in zip(row_ids, row_p)])
        return out

    def timing(self, replica: int = 0) -> dict:
        return self._handles[replica].timing()

    def unload_model(self, to_cpu: bool = False):
        for h in self._handles:
            h.close()
