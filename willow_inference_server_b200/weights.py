"""Flat weight blob shared by the CUDA engine (csrc/weights.cu) and the CPU oracle.

The reference loads CTranslate2 model directories ``models/tovera-wis-whisper-<size>/``
(/root/reference/main.py:342,364,386,408,430) -- none exist in this image and
ctranslate2 is absent, so the engine defines its own container: one file, one
``cudaMemcpy`` (or one NCCL broadcast) to place it in HBM.

Layout (little endian):
    [0,256)            header  : magic "WISB200\\0", u32 version, 21 x i32 dims/special ids
    [256, 256+96*n)    table   : n entries {char name[48]; u32 dtype; u32 ndim; i64 shape[4]; u64 offset}
    data                       : every tensor 256-byte aligned (TMA needs >= 16 B)

dtypes: 0 = float16, 1 = float32, 2 = int32.  GEMM weights are float16 [N, K]
row-major (K contiguous = "K-major" for tcgen05 / TMA); biases, LayerNorm
parameters and positional tables are float32.

Canonical (HF-named) state dict -> engine tensors is done by ``pack_state_dict``;
names follow [HF] transformers/models/whisper/modeling_whisper.py so that real
``openai/whisper-*`` / ``tovera/wis-whisper-*`` safetensors drop in unchanged.
"""
from __future__ import annotations

import struct
from dataclasses import dataclass, field, asdict

import numpy as np

MAGIC = b"WISB200\x00"
VERSION = 1
HEADER_BYTES = 256
ENTRY_BYTES = 96
ALIGN = 256
T_ENC = 1500  # encoder positions per 30-s window
N_MELS = 80
N_FRAMES = 3000

# [HF] configuration_whisper.py NON_SPEECH_TOKENS_MULTI, plus the task/sot tokens CTranslate2
# converts into config.json:suppress_ids (SURVEY.md section 8a row A11).
NON_SPEECH_TOKENS_MULTI = [
    1, 2, 7, 8, 9, 10, 14, 25, 26, 27, 28, 29, 31, 58, 59, 60, 61, 62, 63, 90, 91, 92, 93, 359, 503, 522, 542, 873,
    893, 902, 918, 922, 931, 1350, 1853, 1982, 2460, 2627, 3246, 3253, 3268, 3536, 3846, 3961, 4183, 4667, 6585,
    6647, 7273, 9061, 9383, 10428, 10929, 11938, 12033, 12331, 12562, 13793, 14157, 14635, 15265, 15618, 16553,
    16604, 18362, 18956, 20075, 21675, 22520, 26130, 26161, 26435, 28279, 29464, 31650, 32302, 32470, 36865,
    42863, 47425, 49870, 50254, 50258, 50358, 50359, 50360, 50361, 50362,
]

SIZES = {  # name -> (d_model, layers, heads)   SURVEY.md section 8
    "tiny": (384, 4, 6),
    "base": (512, 6, 8),
    "small": (768, 12, 12),
    "medium": (1024, 24, 16),
    "large-v2": (1280, 32, 20),
    "large": (1280, 32, 20),
}


@dataclass
class WhisperDims:
    d_model: int = 1280
    n_heads: int = 20
    n_enc_layers: int = 32
    n_dec_layers: int = 32
    n_vocab: int = 51865
    n_text_ctx: int = 448
    n_mels: int = N_MELS
    n_audio_ctx: int = T_ENC
    sot: int = 50258
    eot: int = 50257
    transcribe: int = 50359
    translate: int = 50358
    no_timestamps: int = 50363
    sot_prev: int = 50361
    sot_lm: int = 50360
    no_speech: int = 50362
    blank: int = 220
    lang_first: int = 50259  # <|en|>
    n_langs: int = 99
    suppress_ids: list = field(default_factory=lambda: list(NON_SPEECH_TOKENS_MULTI))
    suppress_ids_begin: list = field(default_factory=lambda: [220, 50257])

    @property
    def n_vocab_pad(self) -> int:
        return (self.n_vocab + 127) // 128 * 128

    @property
    def lang_ids(self) -> list:
        return list(range(self.lang_first, self.lang_first + self.n_langs))

    @staticmethod
    def for_size(name: str, **kw) -> "WhisperDims":
        d, layers, heads = SIZES[name]
        return WhisperDims(d_model=d, n_heads=heads, n_enc_layers=layers, n_dec_layers=layers, **kw)

    def validate(self):
        if self.d_model % 64 or self.d_model != 64 * self.n_heads:
            raise ValueError("engine requires head_dim == 64 (true for every Whisper size)")
        if self.n_mels != N_MELS or self.n_audio_ctx != T_ENC:
            raise ValueError("engine is built for 80 mels x 1500 encoder positions")
        if not (0 <= self.eot < self.n_vocab and 0 <= self.sot < self.n_vocab):
            raise ValueError("special ids outside the vocabulary")


_HDR_FIELDS = [
    "d_model", "n_heads", "n_enc_layers", "n_dec_layers", "n_vocab", "n_vocab_pad", "n_text_ctx", "n_mels",
    "n_audio_ctx", "sot", "eot", "transcribe", "translate", "no_timestamps", "sot_prev", "sot_lm", "no_speech",
    "blank", "lang_first", "n_langs",
]
_DT = {np.dtype(np.float16): 0, np.dtype(np.float32): 1, np.dtype(np.int32): 2}
_DT_INV = {0: np.float16, 1: np.float32, 2: np.int32}


# ---------------------------------------------------------------------------
# canonical (HF-named, float32 values that are exactly float16-representable for
# every GEMM weight) -> engine tensors
# ---------------------------------------------------------------------------
def sinusoids(length: int, channels: int, max_timescale: float = 10000.0) -> np.ndarray:
    """[HF] modeling_whisper.py:55 ``sinusoids`` -- encoder positional table."""
    inc = np.log(max_timescale) / (channels // 2 - 1)
    inv = np.exp(-inc * np.arange(channels // 2, dtype=np.float64))
    t = np.arange(length, dtype=np.float64)[:, None] * inv[None, :]
    return np.concatenate([np.sin(t), np.cos(t)], axis=1).astype(np.float32)


def pack_state_dict(sd: dict, dims: WhisperDims) -> dict:
    """HF ``WhisperForConditionalGeneration.state_dict()`` (numpy values) -> engine tensors."""
    dims.validate()
    d = dims.d_model
    f16 = lambda a: np.ascontiguousarray(np.asarray(a, np.float32).astype(np.float16))  # noqa: E731
    f32 = lambda a: np.ascontiguousarray(np.asarray(a, np.float32))  # noqa: E731
    z = np.zeros(d, np.float32)
    out = {}
    e = "model.encoder."
    # conv weights [co, ci, k] -> [co, k*ci] so that one A row = 3 consecutive time rows
    out["enc.conv1.w"] = f16(np.transpose(sd[e + "conv1.weight"], (0, 2, 1)).reshape(d, 3 * dims.n_mels))
    out["enc.conv1.b"] = f32(sd[e + "conv1.bias"])
    out["enc.conv2.w"] = f16(np.transpose(sd[e + "conv2.weight"], (0, 2, 1)).reshape(d, 3 * d))
    out["enc.conv2.b"] = f32(sd[e + "conv2.bias"])
    out["enc.pos"] = f32(sd[e + "embed_positions.weight"])
    for i in range(dims.n_enc_layers):
        p = f"{e}layers.{i}."
        q = f"enc.{i}."
        out[q + "ln1.g"] = f32(sd[p + "self_attn_layer_norm.weight"])
        out[q + "ln1.b"] = f32(sd[p + "self_attn_layer_norm.bias"])
        out[q + "qkv.w"] = f16(np.concatenate([sd[p + "self_attn.q_proj.weight"], sd[p + "self_attn.k_proj.weight"],
                                               sd[p + "self_attn.v_proj.weight"]], 0))
        out[q + "qkv.b"] = f32(np.concatenate([sd[p + "self_attn.q_proj.bias"], z, sd[p + "self_attn.v_proj.bias"]]))
        out[q + "o.w"] = f16(sd[p + "self_attn.out_proj.weight"])
        out[q + "o.b"] = f32(sd[p + "self_attn.out_proj.bias"])
        out[q + "ln2.g"] = f32(sd[p + "final_layer_norm.weight"])
        out[q + "ln2.b"] = f32(sd[p + "final_layer_norm.bias"])
        out[q + "fc1.w"] = f16(sd[p + "fc1.weight"])
        out[q + "fc1.b"] = f32(sd[p + "fc1.bias"])
        out[q + "fc2.w"] = f16(sd[p + "fc2.weight"])
        out[q + "fc2.b"] = f32(sd[p + "fc2.bias"])
    out["enc.ln_post.g"] = f32(sd[e + "layer_norm.weight"])
    out["enc.ln_post.b"] = f32(sd[e + "layer_norm.bias"])

    dd = "model.decoder."
    emb = np.zeros((dims.n_vocab_pad, d), np.float16)
    emb[: dims.n_vocab] = np.asarray(sd[dd + "embed_tokens.weight"], np.float32).astype(np.float16)
    out["dec.tok_emb"] = emb
    out["dec.pos"] = f32(sd[dd + "embed_positions.weight"])
    ckv_w, ckv_b = [], []
    for i in range(dims.n_dec_layers):
        p = f"{dd}layers.{i}."
        q = f"dec.{i}."
        out[q + "ln1.g"] = f32(sd[p + "self_attn_layer_norm.weight"])
        out[q + "ln1.b"] = f32(sd[p + "self_attn_layer_norm.bias"])
        out[q + "qkv.w"] = f16(np.concatenate([sd[p + "self_attn.q_proj.weight"], sd[p + "self_attn.k_proj.weight"],
                                               sd[p + "self_attn.v_proj.weight"]], 0))
        out[q + "qkv.b"] = f32(np.concatenate([sd[p + "self_attn.q_proj.bias"], z, sd[p + "self_attn.v_proj.bias"]]))
        out[q + "o.w"] = f16(sd[p + "self_attn.out_proj.weight"])
        out[q + "o.b"] = f32(sd[p + "self_attn.out_proj.bias"])
        out[q + "ln2.g"] = f32(sd[p + "encoder_attn_layer_norm.weight"])
        out[q + "ln2.b"] = f32(sd[p + "encoder_attn_layer_norm.bias"])
        out[q + "cq.w"] = f16(sd[p + "encoder_attn.q_proj.weight"])
        out[q + "cq.b"] = f32(sd[p + "encoder_attn.q_proj.bias"])
        out[q + "co.w"] = f16(sd[p + "encoder_attn.out_proj.weight"])
        out[q + "co.b"] = f32(sd[p + "encoder_attn.out_proj.bias"])
        out[q + "ln3.g"] = f32(sd[p + "final_layer_norm.weight"])
        out[q + "ln3.b"] = f32(sd[p + "final_layer_norm.bias"])
        out[q + "fc1.w"] = f16(sd[p + "fc1.weight"])
        out[q + "fc1.b"] = f32(sd[p + "fc1.bias"])
        out[q + "fc2.w"] = f16(sd[p + "fc2.weight"])
        out[q + "fc2.b"] = f32(sd[p + "fc2.bias"])
        ckv_w += [sd[p + "encoder_attn.k_proj.weight"], sd[p + "encoder_attn.v_proj.weight"]]
        ckv_b += [z, sd[p + "encoder_attn.v_proj.bias"]]
    out["dec.crosskv.w"] = f16(np.concatenate(ckv_w, 0))
    out["dec.crosskv.b"] = f32(np.concatenate(ckv_b))
    out["dec.ln.g"] = f32(sd[dd + "layer_norm.weight"])
    out["dec.ln.b"] = f32(sd[dd + "layer_norm.bias"])
    out["meta.suppress_ids"] = np.asarray(sorted(set(dims.suppress_ids)), np.int32)
    out["meta.suppress_ids_begin"] = np.asarray(dims.suppress_ids_begin, np.int32)
    out["meta.lang_ids"] = np.asarray(dims.lang_ids, np.int32)
    return out


# ---------------------------------------------------------------------------
# seeded synthetic weights (there are no real checkpoints in this image)
# ---------------------------------------------------------------------------
def synth_state_dict(dims: WhisperDims, seed: int = 0, logit_std: float = 4.0, qk_gain: float = 2.5,
                     resid_std: float = 8.0, eot_ramp: tuple | None = None, script: tuple | None = None,
                     ts_script: tuple | None = None) -> dict:
    """Deterministic random Whisper weights under HF names.

    Every GEMM weight is rounded to float16 so oracle (fp32 math) and engine
    (fp16 tensor-core inputs) hold IDENTICAL parameters.  ``eot_ramp=(p0, slope)``
    adds ``slope * max(0, p - p0)`` along the <|endoftext|> embedding direction to
    the decoder positional table so that hypotheses terminate at data-dependent
    steps (exercises the beam-search finish rules); ``None`` means EOT is
    essentially never the arg-max and decoding runs to ``max_length``.

    ``script=(n_alt, rho, off)`` makes the output distribution PEAKED the way a trained model's is
    (SURVEY.md section 7: "peaked-logit scaling so argmax margins >> rounding noise"): every text
    position gets ``n_alt`` seeded "plausible next tokens" whose logits are lifted through the decoder
    positional table to ``(off + k) * rho`` times the standard deviation of the Gaussian (audio / history
    dependent) part of the logits, k = n_alt-1 .. 0 -- far above the bulk of the vocabulary (the maximum of
    51865 Gaussian draws is ~4.3 of those deviations).  Which alternative wins still depends on the audio, but
    candidates are separated by O(rho) deviations instead of the ~0.01-wide near-ties of a flat random model,
    so greedy / beam transcripts are robust to fp16-vs-fp32 rounding.  The share of the residual stream the
    script takes is solved from ``rho`` and d_model, so the same setting works at every model size.

    ``ts_script=((pos, first), ...)`` (needs ``script``) makes a model that speaks in timestamps: at each listed decoder
    position the ``n_alt`` plausible next tokens are the timestamps ``no_timestamps + 1 + first + [0, n_alt)`` instead of
    text tokens.  The ranges must be disjoint and increase with the position (timestamps never decrease), and the first
    one should lie within the ``max_initial_timestamp_index`` the model is decoded with.  ``None`` leaves the weights
    byte-identical to a call without it.
    """
    dims.validate()
    if ts_script is not None and script is None:
        raise ValueError("ts_script needs script=(n_alt, rho, off)")
    d = dims.d_model
    # logits = LN(x) . E[v] ~ N(0, d * emb_std^2): pick emb_std for the requested logit spread, and
    # make the sub-layer outputs large enough (residual stream std ~ resid_std) that the direct
    # "copy the previous token" path E[prev].E[prev] / std(x) stays far below the top of the vocabulary.
    emb_std = logit_std / np.sqrt(d)
    dec_gain = resid_std / (0.6 * np.sqrt(3.0 * dims.n_dec_layers))
    ss = np.random.SeedSequence(seed)
    counter = [0]
    deferred = []  # (name-slot, thunk): tensors are drawn in parallel, each from its own counter-derived stream

    def stream():
        counter[0] += 1
        key = counter[0]
        return lambda: np.random.default_rng(np.random.SeedSequence(entropy=ss.entropy, spawn_key=(key,)))

    def h(a):  # round to fp16 grid
        return a.astype(np.float16).astype(np.float32)

    class Lazy:
        def __init__(self, fn):
            self.fn = fn

    def normal(shape, scale, half=True, mean=0.0):
        mk = stream()

        def fn():
            a = mk().standard_normal(shape, dtype=np.float32) * np.float32(scale)
            if mean:
                a = a + np.float32(mean)
            return h(a) if half else a.astype(np.float32)

        return Lazy(fn)

    def lin(n_out, n_in, gain=1.0):
        return normal((n_out, n_in), gain / np.sqrt(n_in))

    def vec(n, std=0.02, mean=0.0):
        return normal(n, std, half=False, mean=mean)

    sd = {}
    e = "model.encoder."
    sd[e + "conv1.weight"] = normal((d, dims.n_mels, 3), 1.0 / np.sqrt(3 * dims.n_mels))
    sd[e + "conv1.bias"] = vec(d)
    sd[e + "conv2.weight"] = normal((d, d, 3), 1.5 / np.sqrt(3 * d))
    sd[e + "conv2.bias"] = vec(d)
    sd[e + "embed_positions.weight"] = sinusoids(dims.n_audio_ctx, d)

    def attn(prefix, gain=1.0):
        sd[prefix + "q_proj.weight"] = lin(d, d, qk_gain)
        sd[prefix + "q_proj.bias"] = vec(d)
        sd[prefix + "k_proj.weight"] = lin(d, d, qk_gain)
        sd[prefix + "v_proj.weight"] = lin(d, d, 2.0)
        sd[prefix + "v_proj.bias"] = vec(d)
        sd[prefix + "out_proj.weight"] = lin(d, d, gain)
        sd[prefix + "out_proj.bias"] = vec(d)

    def ln(prefix):
        sd[prefix + ".weight"] = vec(d, 0.05, 1.0)
        sd[prefix + ".bias"] = vec(d, 0.02)

    def mlp(prefix, gain=1.0):
        sd[prefix + "fc1.weight"] = lin(4 * d, d)
        sd[prefix + "fc1.bias"] = vec(4 * d)
        sd[prefix + "fc2.weight"] = lin(d, 4 * d, gain)
        sd[prefix + "fc2.bias"] = vec(d)

    for i in range(dims.n_enc_layers):
        p = f"{e}layers.{i}."
        ln(p + "self_attn_layer_norm")
        attn(p + "self_attn.")
        ln(p + "final_layer_norm")
        mlp(p)
    ln(e + "layer_norm")

    dd = "model.decoder."
    sd[dd + "embed_tokens.weight"] = normal((dims.n_vocab, d), emb_std)
    sd[dd + "embed_positions.weight"] = normal((dims.n_text_ctx, d), emb_std, half=False)
    for i in range(dims.n_dec_layers):
        p = f"{dd}layers.{i}."
        ln(p + "self_attn_layer_norm")
        attn(p + "self_attn.", dec_gain)
        ln(p + "encoder_attn_layer_norm")
        attn(p + "encoder_attn.", dec_gain)
        ln(p + "final_layer_norm")
        mlp(p, dec_gain)
    ln(dd + "layer_norm")
    # materialise (numpy's Generator releases the GIL: one thread per tensor)
    from concurrent.futures import ThreadPoolExecutor
    import os as _os

    names = [k for k, v in sd.items() if isinstance(v, Lazy)]
    with ThreadPoolExecutor(max_workers=max(1, min(32, (_os.cpu_count() or 1)))) as ex:
        for k, a in zip(names, ex.map(lambda k: sd[k].fn(), names)):
            sd[k] = a
    if script is not None:
        n_alt, rho, off = script
        emb = sd[dd + "embed_tokens.weight"]
        mult = np.asarray([off + (int(n_alt) - 1 - j) for j in range(int(n_alt))], np.float64)
        # xn = LN(x) has |xn|^2 = d; a share `frac` of it goes to the scripted directions, the rest (the "noise") keeps
        # the audio / history dependence:  boost_j = c_j * logit_std with c_j = c0 * mult_j, noise = sqrt(1 - frac) *
        # logit_std, c0 = rho * sqrt(1 - frac), sum_j c_j^2 = d * frac
        kk = float((mult ** 2).sum()) * rho * rho
        frac = kk / (d + kk)
        c = rho * np.sqrt(1.0 - frac) * mult
        s_eff = resid_std / np.sqrt(1.0 - frac)  # residual-stream std once the scripted components are in it
        banned = set(dims.suppress_ids) | set(dims.suppress_ids_begin)
        rng = np.random.default_rng(np.random.SeedSequence(entropy=ss.entropy, spawn_key=(10 ** 6,)))
        ts_alts = {}
        if ts_script is not None:
            ts_rng = np.random.default_rng(np.random.SeedSequence(entropy=ss.entropy, spawn_key=(10 ** 6 + 1,)))
            ts_begin = dims.no_timestamps + 1
            prev_end = 0
            for p, first in sorted((int(p), int(f)) for p, f in ts_script):
                if p in ts_alts or first < prev_end or ts_begin + first + int(n_alt) > dims.n_vocab:
                    raise ValueError("ts_script: timestamp ranges must be disjoint, increasing and inside the vocabulary")
                prev_end = first + int(n_alt)
                ts_alts[p] = [ts_begin + first + int(j) for j in ts_rng.permutation(int(n_alt))]
        pos = sd[dd + "embed_positions.weight"].astype(np.float64)
        for p in range(dims.n_text_ctx):
            alts = []
            while len(alts) < int(n_alt):
                t = int(rng.integers(300, dims.eot))  # ordinary text tokens only
                if t not in banned and t not in alts:
                    alts.append(t)
            alts = ts_alts.get(p, alts)  # (the text draw above still happens: later positions keep their tokens)
            for j, t in enumerate(alts):
                nrm = np.linalg.norm(emb[t])
                pos[p] += (c[j] * s_eff * logit_std / (nrm * nrm)) * emb[t].astype(np.float64)
        sd[dd + "embed_positions.weight"] = pos.astype(np.float32)
    if eot_ramp is not None:
        p0, slope = eot_ramp
        emb = sd[dd + "embed_tokens.weight"]
        u = emb[dims.eot] / np.linalg.norm(emb[dims.eot])
        ramp = np.maximum(0.0, np.arange(dims.n_text_ctx, dtype=np.float32) - p0) * np.float32(slope)
        sd[dd + "embed_positions.weight"] = (sd[dd + "embed_positions.weight"] + ramp[:, None] * u[None, :]).astype(np.float32)
    return sd


def synth_engine_tensors(dims: WhisperDims, seed: int = 0, **kw) -> dict:
    return pack_state_dict(synth_state_dict(dims, seed, **kw), dims)


# ---------------------------------------------------------------------------
# blob (de)serialisation
# ---------------------------------------------------------------------------
def _layout(tensors: dict):
    names = list(tensors.keys())
    off = HEADER_BYTES + ENTRY_BYTES * len(names)
    off = (off + ALIGN - 1) // ALIGN * ALIGN
    offsets = {}
    for n in names:
        offsets[n] = off
        off += (tensors[n].nbytes + ALIGN - 1) // ALIGN * ALIGN
    return names, offsets, off


def blob_nbytes(tensors: dict) -> int:
    return _layout(tensors)[2]


def write_blob_into(buf: np.ndarray, dims: WhisperDims, tensors: dict) -> int:
    """Serialise into a pre-allocated uint8 buffer (e.g. pinned host memory). Returns bytes used."""
    names, offsets, total = _layout(tensors)
    assert buf.dtype == np.uint8 and buf.size >= total
    hdr = bytearray(HEADER_BYTES)
    hdr[:8] = MAGIC
    vals = [getattr(dims, f) for f in _HDR_FIELDS]
    struct.pack_into("<II%di" % len(vals), hdr, 8, VERSION, len(names), *vals)
    buf[:HEADER_BYTES] = np.frombuffer(bytes(hdr), np.uint8)
    for i, n in enumerate(names):
        a = tensors[n]
        assert a.flags["C_CONTIGUOUS"] and a.ndim <= 4 and len(n) < 48, n
        shape = list(a.shape) + [1] * (4 - a.ndim)
        ent = struct.pack("<48sII4qQ", n.encode(), _DT[a.dtype], a.ndim, *shape, offsets[n])
        ent = ent.ljust(ENTRY_BYTES, b"\0")
        o = HEADER_BYTES + i * ENTRY_BYTES
        buf[o : o + ENTRY_BYTES] = np.frombuffer(ent, np.uint8)
        buf[offsets[n] : offsets[n] + a.nbytes] = a.reshape(-1).view(np.uint8)
    return total


def write_blob(path: str, dims: WhisperDims, tensors: dict) -> int:
    total = blob_nbytes(tensors)
    buf = np.zeros(total, np.uint8)
    write_blob_into(buf, dims, tensors)
    buf.tofile(path)
    return total


def read_blob(src) -> tuple:
    """path or uint8 array -> (WhisperDims, {name: ndarray view})."""
    buf = np.fromfile(src, np.uint8) if isinstance(src, str) else np.asarray(src, np.uint8)
    if bytes(buf[:8]) != MAGIC:
        raise ValueError("not a WISB200 weight blob")
    n_fields = len(_HDR_FIELDS)
    vals = struct.unpack_from("<II%di" % n_fields, buf[:HEADER_BYTES].tobytes(), 8)
    if vals[0] != VERSION:
        raise ValueError(f"unsupported blob version {vals[0]}")
    n = vals[1]
    hv = dict(zip(_HDR_FIELDS, vals[2:]))
    hv.pop("n_vocab_pad")
    tensors = {}
    for i in range(n):
        o = HEADER_BYTES + i * ENTRY_BYTES
        name, dt, nd, s0, s1, s2, s3, off = struct.unpack_from("<48sII4qQ", buf[o : o + ENTRY_BYTES].tobytes(), 0)
        name = name.rstrip(b"\0").decode()
        shape = (s0, s1, s2, s3)[:nd]
        dtype = np.dtype(_DT_INV[dt])
        cnt = int(np.prod(shape)) if nd else 1
        tensors[name] = buf[off : off + cnt * dtype.itemsize].view(dtype).reshape(shape)
    dims = WhisperDims(**hv)
    dims.suppress_ids = [int(v) for v in tensors["meta.suppress_ids"]]
    dims.suppress_ids_begin = [int(v) for v in tensors["meta.suppress_ids_begin"]]
    return dims, tensors


def dims_dict(dims: WhisperDims) -> dict:
    return asdict(dims)
