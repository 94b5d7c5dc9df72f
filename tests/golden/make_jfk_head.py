"""Cut the first frames of the original project's jfk.flac into tests/golden/jfk_head.flac, a valid FLAC stream small
enough to commit (the whole asset is 1.15 MB).

FLAC frames decode independently, so the head is STREAMINFO (sample count and MD5 rewritten for the kept samples, every
other metadata block dropped) followed by the first N frames byte for byte: the tests decode real encoder output
(LPC / fixed subframes, stereo decorrelation, 24-bit samples) and the decoder's MD5 check still covers every sample.

    python tests/golden/make_jfk_head.py <original project>/assets/jfk.flac [--frames 10]
"""
import argparse
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "jfk_head.flac")
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from whisperlive_b200.audio import decode_flac  # noqa: E402


def crc8(b: bytes) -> int:
    c = 0
    for x in b:
        c ^= x
        for _ in range(8):
            c = ((c << 1) ^ 0x07) & 0xFF if c & 0x80 else (c << 1) & 0xFF
    return c


def frame_start(data: bytes, start: int, number: int) -> int:
    """Byte offset of the fixed-blocksize frame ``number`` (< 128): sync code, that frame number, valid header CRC-8."""
    pos = data.find(b"\xff\xf8", start)
    while pos >= 0:
        bs, sr = data[pos + 2] >> 4, data[pos + 2] & 15
        n = 5 + (1 if bs == 6 else 2 if bs == 7 else 0) + (1 if sr == 12 else 2 if sr in (13, 14) else 0)
        if data[pos + 4] == number and crc8(data[pos:pos + n]) == data[pos + n]:
            return pos
        pos = data.find(b"\xff\xf8", pos + 1)
    raise ValueError(f"frame {number} not found")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("src")
    ap.add_argument("--frames", type=int, default=10)
    args = ap.parse_args()
    data = open(args.src, "rb").read()
    pcm, info = decode_flac(data)                          # raises unless the whole stream matches its MD5
    pos = 4
    while True:                                            # metadata blocks: keep STREAMINFO, find the first frame
        last, btype, size = data[pos] >> 7, data[pos] & 127, int.from_bytes(data[pos + 1:pos + 4], "big")
        if btype == 0:
            si = bytearray(data[pos + 4:pos + 4 + size])
        pos += 4 + size
        if last:
            break
    min_bs, max_bs = int.from_bytes(si[0:2], "big"), int.from_bytes(si[2:4], "big")
    assert min_bs == max_bs, "variable block size"
    end = frame_start(data, pos, args.frames)
    total = args.frames * max_bs
    head = pcm[:, :total]
    raw = b"".join(int(v).to_bytes((info["bps"] + 7) // 8, "little", signed=True) for v in head.T.reshape(-1))
    packed = int.from_bytes(si[10:18], "big")
    packed = (packed & ~((1 << 36) - 1)) | total           # low 36 bits: total samples per channel
    si[10:18] = packed.to_bytes(8, "big")
    si[18:34] = hashlib.md5(raw).digest()
    out = b"fLaC" + bytes([0x80]) + len(si).to_bytes(3, "big") + bytes(si) + data[pos:end]
    got, ginfo = decode_flac(out)
    assert ginfo["total"] == total and np.array_equal(got, head)
    with open(OUT, "wb") as f:
        f.write(out)
    print("wrote", OUT, len(out), "bytes,", total, "samples at", info["rate"], "Hz")


if __name__ == "__main__":
    main()
