"""FLAC ingest (SURVEY 8f row 3a): csrc/flac.cu through the C ABI and audio.decode_flac -- host code, runs without a GPU.

Goldens: the PCM MD5s of the reference's libFLAC-made fixtures (SURVEY.md section 4, parsed from their STREAMINFO):
client/3sec.flac as it is, and the first 10 frames of client/{10sec,30sec}.flac (tests/golden/client_*_head.flac, cut by
scripts/gen_golden_flac.py; the MD5 of the full 10 s / 30 s recordings is c5b99673... / 3a541ad6...), plus streams made
by tests/flac_writer.py for every decoder path the libFLAC-made mono fixtures do not reach."""
import hashlib
import os

import numpy as np
import pytest

from tests import flac_writer as fw
from willow_inference_server_b200 import _lib, audio

FIXTURES = [("3sec.flac", 61440, "ad790df21d4d9d223d3f34227b5cfedd"),
            ("10sec_head.flac", 40960, "b8310575537022d81af8341b0aa377ec"),
            ("30sec_head.flac", 40960, "97c9c8e0886212e3deadeaf1e58e88a7")]


@pytest.mark.parametrize("name,n,md5", FIXTURES)
def test_reference_fixtures_decode_to_their_md5(name, n, md5, golden_dir):
    path = os.path.join(golden_dir, "client_" + name)
    pcm, sr = audio.decode_flac(path)                              # verify=True already checks STREAMINFO's MD5
    assert sr == 16000 and pcm.dtype == np.int16 and pcm.shape == (n,)
    assert hashlib.md5(pcm.astype("<i2").tobytes()).hexdigest() == md5
    x = audio.load_audio(path)
    assert x.dtype == np.float32 and x.shape == (n,) and np.abs(x).max() <= 1.0
    assert np.array_equal(x, pcm.astype(np.float32) / 32768.0)


def _signal(n, ch, bps, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    amp = (1 << (bps - 1)) * 0.4
    x = np.stack([amp * np.sin(2 * np.pi * (0.01 + 0.003 * c) * t + c) + rng.normal(0, amp * 0.02, n) for c in range(ch)], 1)
    return np.clip(np.round(x), -(1 << (bps - 1)), (1 << (bps - 1)) - 1).astype(np.int64)


def _roundtrip(pcm, **kw):
    data = fw.encode(pcm, **kw)
    got, sr = audio.decode_flac(data)
    want = np.asarray(pcm)
    want = want[:, 0] if want.ndim == 2 and want.shape[1] == 1 else want
    assert got.shape == want.shape and np.array_equal(got.astype(np.int64), want), kw
    return data


def test_every_subframe_type_and_residual_coding():
    n = 4096 + 1000 + 192 + 37
    x = _signal(n, 1, 16, 1)[:, 0]
    x[4096 : 4096 + 1000] = -1234                       # constant block
    blocks = [4096, 1000, 192, 37]
    for method in (0, 1):
        specs = [[{"kind": "lpc", "order": 3, "coefs": [1400, -900, 200], "shift": 9, "prec": 12, "method": method, "po": 3,
                   "escape": (2,)}],
                 [{"kind": "constant"}],
                 [{"kind": "fixed", "order": 4, "method": method, "po": 2, "escape": (0,)}],
                 [{"kind": "verbatim"}]]
        _roundtrip(x, blocks=blocks, specs=specs)
    for order in range(5):
        _roundtrip(x[:2048], blocks=[2048], specs=[[{"kind": "fixed", "order": order, "po": 4}]])
    # 32nd-order LPC with a long warm-up and the largest legal coefficient precision
    coefs = [((-1) ** j) * (3000 >> (j // 4)) for j in range(32)]
    _roundtrip(x[:1024], blocks=[1024], specs=[[{"kind": "lpc", "order": 32, "coefs": coefs, "shift": 14, "prec": 15, "po": 0}]])


@pytest.mark.parametrize("bps", [8, 16, 24])
def test_stereo_decorrelation_wasted_bits_and_sample_widths(bps):
    n = 3 * 1152 + 500
    x = _signal(n, 2, bps, 7)
    x[1152:2304] = (x[1152:2304] >> 3) << 3             # three wasted bits in the second block
    blocks = [1152, 1152, 1152, 500]
    modes = ["ls", "sr", "ms", "indep"]
    specs = [[{"kind": "fixed", "order": 2, "po": 1}, {"kind": "fixed", "order": 1, "po": 0}],
             [{"kind": "fixed", "order": 2, "po": 0, "wasted": 3}, {"kind": "fixed", "order": 0, "po": 2, "wasted": 3}],
             [{"kind": "lpc", "order": 2, "coefs": [500, -200], "shift": 8, "prec": 11, "po": 2}, {"kind": "fixed", "order": 3, "po": 0}],
             [{"kind": "verbatim"}, {"kind": "fixed", "order": 1, "po": 2}]]
    data = _roundtrip(x, bps=bps, blocks=blocks, stereo_modes=modes, specs=specs)
    pcm, sr, got_bps, md5 = _lib.flac_decode(data)
    assert (sr, got_bps, pcm.shape) == (16000, bps, (n, 2)) and any(md5)
    if bps <= 16:
        assert audio.load_audio(data).shape == (n,)     # stereo is averaged to mono, as librosa.load(mono=True) does


def test_many_frames_unknown_md5_and_8_channels():
    x = _signal(300 * 256 + 13, 1, 16, 3)[:, 0]
    _roundtrip(x, blocks=[256] * 300 + [13], md5=False)  # frame numbers >= 128 need the multi-byte number coding
    y = _signal(1024, 8, 16, 4)
    _roundtrip(y, blocks=[1024])


def test_corruption_is_detected():
    x = _signal(4096, 1, 16, 5)[:, 0]
    good = fw.encode(x, blocks=[4096])
    for where in (len(good) // 2, len(good) - 1):        # payload byte, CRC-16 byte
        bad = bytearray(good)
        bad[where] ^= 0x10
        with pytest.raises(ValueError, match="FLAC"):
            audio.decode_flac(bytes(bad))
    with pytest.raises(ValueError, match="fLaC"):
        audio.decode_flac(b"RIFF" + good[4:])
    with pytest.raises(ValueError, match="FLAC"):
        audio.decode_flac(good[: len(good) // 2])        # truncated
    lying = bytearray(good)
    lying[26 + 8] ^= 0xFF                                 # MD5 field of STREAMINFO (4 + 4 + 18 = offset 26)
    with pytest.raises(ValueError, match="MD5"):
        audio.decode_flac(bytes(lying))
    assert audio.decode_flac(bytes(lying), verify=False)[0].shape == (4096,)
    with pytest.raises(ValueError, match="resampling"):
        audio.load_audio(fw.encode(x, blocks=[4096], sample_rate=44100))


@pytest.mark.parametrize("seed", range(12))
def test_random_streams_roundtrip(seed):
    # seeded fuzz over the writer's degrees of freedom: block sizes, widths, channel layouts, predictors, partitions
    rng = np.random.default_rng(seed)
    bps = int(rng.choice([8, 12, 16, 20, 24]))
    ch = int(rng.choice([1, 2, 2, 3]))
    blocks = [int(rng.choice([192, 256, 576, 1000, 1152, 4096, 17, 255, 257])) for _ in range(int(rng.integers(1, 6)))]
    n = sum(blocks)
    x = _signal(n, ch, bps, seed + 100)
    modes, specs = [], []
    for bs in blocks:
        modes.append(str(rng.choice(["indep", "ls", "sr", "ms"])) if ch == 2 else "indep")
        row = []
        for _ in range(ch):
            kind = str(rng.choice(["verbatim", "fixed", "fixed", "lpc"]))
            po = int(rng.integers(0, 4))
            while po > 0 and (bs % (1 << po) or (bs >> po) <= 8):
                po -= 1
            if kind == "fixed":
                row.append({"kind": "fixed", "order": int(rng.integers(0, 5)), "po": po, "method": int(rng.integers(0, 2)),
                            "escape": tuple(int(p) for p in range(1 << po) if rng.random() < 0.2)})
            elif kind == "lpc":
                order = int(rng.integers(1, 9))
                prec = int(rng.integers(5, 13))
                coefs = [int(c) for c in rng.integers(-(1 << (prec - 1)), 1 << (prec - 1), order) // order]
                row.append({"kind": "lpc", "order": order, "coefs": coefs, "shift": prec - 1, "prec": prec, "po": po,
                            "method": int(rng.integers(0, 2))})
            else:
                row.append({"kind": "verbatim"})
        specs.append(row)
    _roundtrip(x, bps=bps, blocks=blocks, stereo_modes=modes, specs=specs, md5=bool(seed % 2))


@pytest.mark.parametrize("bps", [8, 12, 16, 20, 24])
def test_load_audio_amplitude_for_every_sample_width(bps):
    # full scale is 2^(bps-1) whatever the width (what soundfile / librosa.load hand do_whisper, main.py:579): the log-mel
    # front end is not gain invariant, so a 24-bit stream decoded 48 dB too quiet would silently change every feature
    n = 3000
    x = _signal(n, 1, bps, 11)[:, 0]
    data = fw.encode(x, bps=bps, blocks=[n])
    got = audio.load_audio(data)
    want = (x.astype(np.float64) / float(1 << (bps - 1))).astype(np.float32)
    assert got.dtype == np.float32 and got.shape == (n,)
    assert np.array_equal(got, want)
    assert 0.35 < np.abs(got).max() < 0.5


def test_streaminfo_sample_count_is_not_trusted():
    # a 42-byte "file" whose STREAMINFO claims 2^36 - 1 samples must be rejected before anything is allocated
    x = _signal(64, 1, 16, 3)[:, 0]
    data = bytearray(fw.encode(x, blocks=[64]))
    # STREAMINFO body starts at byte 8; total samples = low 36 bits of bytes 13..17 of the body
    data[8 + 13] |= 0x0F
    data[8 + 14 : 8 + 18] = b"\xff\xff\xff\xff"
    with pytest.raises(ValueError):
        _lib.flac_decode(bytes(data[:42]))
