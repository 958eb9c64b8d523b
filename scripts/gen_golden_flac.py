#!/usr/bin/env python
"""Cut the reference's client/*.flac fixtures down to tests/golden/client_<name>_head.flac.

    python scripts/gen_golden_flac.py <reference checkout>/client

The full 10 s and 30 s recordings are larger than a test vector should be.  The head of each stream keeps the encoder's
own frames byte for byte: STREAMINFO, then the first N_FRAMES frames (frame numbers 0.., so the cut stream is a valid
FLAC file), with STREAMINFO's total-sample count and PCM MD5 rewritten for the shorter stream.  The MD5 is taken from
the full file's decode, which csrc/flac.cu first checks against the encoder's MD5 of the whole recording.  Other
metadata blocks (a VORBIS_COMMENT with the encoder's vendor string) are dropped.
"""
import hashlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from willow_inference_server_b200 import audio  # noqa: E402

N_FRAMES = {"10sec": 10, "30sec": 10}


def crc8(data):
    c = 0
    for b in data:
        c ^= b
        for _ in range(8):
            c = ((c << 1) ^ 0x07) & 0xFF if c & 0x80 else (c << 1) & 0xFF
    return c


def frame_offsets(b, start):
    """Byte offsets of frames 0, 1, ... of a fixed-block-size stream whose frame numbers fit one byte (< 128): a sync
    code, the expected frame number and a matching header CRC-8 (8-bit sample rate / block size codes are not used)."""
    offs, k, p = [], 0, start
    while True:
        p = b.find(b"\xff\xf8", p)
        if p < 0 or k >= 128:
            return offs
        bs, sr = b[p + 2] >> 4, b[p + 2] & 15
        hdr_len = 5 + (1 if bs in (6, 7) else 0) + (2 if bs == 7 else 0) + (1 if sr == 12 else 2 if sr in (13, 14) else 0)
        if b[p + 4] == k and crc8(b[p : p + hdr_len]) == b[p + hdr_len]:
            offs.append(p)
            k += 1
        p += 2


def main():
    src = sys.argv[1]
    for name, n_frames in N_FRAMES.items():
        b = open(os.path.join(src, f"{name}.flac"), "rb").read()
        pcm, _ = audio.decode_flac(b)  # verify=True: the full decode matches the encoder's MD5
        assert b[4] & 0x7F == 0 and int.from_bytes(b[5:8], "big") == 34  # STREAMINFO first
        info = bytearray(b[8:42])
        bs = int.from_bytes(info[0:2], "big")
        assert bs == int.from_bytes(info[2:4], "big")  # fixed block size
        p = 4
        while not b[p] & 0x80:
            p += 4 + int.from_bytes(b[p + 1 : p + 4], "big")
        first = p + 4 + int.from_bytes(b[p + 1 : p + 4], "big")
        offs = frame_offsets(b, first)
        n = n_frames * bs
        head = pcm[:n]
        x = int.from_bytes(info[10:18], "big")
        info[10:18] = ((x & ~((1 << 36) - 1)) | n).to_bytes(8, "big")
        info[18:34] = hashlib.md5(head.astype("<i2").tobytes()).digest()
        out = b"fLaC" + bytes([0x80, 0, 0, 34]) + bytes(info) + b[offs[0] : offs[n_frames]]
        got, _ = audio.decode_flac(out)
        assert got.shape == (n,) and (got == head).all()
        dst = os.path.join(ROOT, "tests", "golden", f"client_{name}_head.flac")
        open(dst, "wb").write(out)
        print(dst, len(out), n, hashlib.md5(head.astype("<i2").tobytes()).hexdigest(),
              [offs[i + 1] - offs[i] for i in range(min(len(offs) - 1, 60))])


if __name__ == "__main__":
    main()
