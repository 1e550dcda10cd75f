"""Saved stream state (nvx_engine_save_streams / nvx_engine_load_streams / nvx_stream_state_info) is part of the published ABI,
and nvx_stream_state_info validates a state on the host.  No GPU needed: the states here are built byte by byte after the layout
in engine.cu (96-byte header, device records, message part) and the checksum of nvx::hash_bytes."""
import os
import re
import struct

import pytest

from navtex_b200 import engine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("nvx_engine_save_streams", "nvx_engine_load_streams", "nvx_stream_state_info")
HEADER = struct.Struct("<IIQQq3qQq6i")
MAGIC, VERSION = 0x5358564E, 1
M64, P64, SEED = (1 << 64) - 1, 0x100000001B3, 1469598103934665603


def _hash(data, h=SEED):
    n8 = len(data) // 8 * 8
    for (w,) in struct.iter_unpack("<Q", data[:n8]):
        h = ((h ^ w) * P64) & M64
        h ^= h >> 29
    for b in data[n8:]:
        h = ((h ^ b) * P64) & M64
        h ^= h >> 29
    return h


def _state(count=1, magic=MAGIC, version=VERSION, C=2, fmt=1, position=280 * 9000):
    words = (1960, 0, 0)                                   # the fused path's int16 tail: 1960 words per stream
    rec_words = 1960 + C * 1336                            # + per channel: y3 / corr histories, clock, fsm, epoch
    msg = b""
    for _ in range(count * C):
        line, text, bbbb = b"NAVAREA", b"ZCZC EA12\n", b"EA12"
        msg += struct.pack("<5i", 518, 1, len(line), len(text), len(bbbb)) + line + text + bbbb
    body = bytes(count * rec_words * 4) + msg
    size = HEADER.size + len(body)
    raw = HEADER.pack(magic, version, size, 0, position, *words, 0, rec_words, count, C, fmt, 0, 0, 0) + body
    cs = _hash(raw[24:], _hash(raw[:16]))
    return raw[:16] + struct.pack("<Q", cs) + raw[24:]


def test_state_entry_points_are_declared_and_exported():
    with open(os.path.join(ROOT, "include", "navtex_b200.h")) as f:
        header = f.read()
    for name in NAMES:
        assert name in engine.EXPORTS, name
        assert re.search(r"\bint " + name + r"\(", header), name


def test_state_info_reads_a_valid_state():
    info = engine.stream_state_info(_state(count=2, C=2, fmt=1, position=280 * 9000))
    assert info == {"count": 2, "position": 280 * 9000, "n_channels": 2, "sample_format": "s16"}


@pytest.mark.parametrize("case", ["empty", "short", "magic", "version", "flipped", "truncated", "extended"])
def test_state_info_rejects_a_bad_state(case):
    good = _state()
    bad = {
        "empty": b"",
        "short": good[:40],
        "magic": _state(magic=MAGIC ^ 1),
        "version": _state(version=VERSION + 1),
        "flipped": good[:5000] + bytes([good[5000] ^ 0x10]) + good[5001:],
        "truncated": good[:-1],
        "extended": good + b"\0",
    }[case]
    with pytest.raises(engine.NvxError):
        engine.stream_state_info(bad)
    # every single flipped byte of the header and the message part is caught, not only one
    if case == "flipped":
        for k in list(range(HEADER.size)) + list(range(len(good) - 60, len(good))):
            with pytest.raises(engine.NvxError):
                engine.stream_state_info(good[:k] + bytes([good[k] ^ 0x01]) + good[k + 1:])
