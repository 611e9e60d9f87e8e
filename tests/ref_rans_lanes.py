"""Reference of the library's laned rANS format (DESIGN.md section 7), for tests of the GPU coder.

Built only on `oracle.ref_rans`' restatement of compressai's coder, with no arithmetic of its own:
- `encode_lanes`    lane l = encode_with_indexes of symbols[l::W] / indexes[l::W], behind the header {W, lane byte lengths}
- `split_lanes`     header parsing: the W lane streams, ValueError for a malformed header
- `decode_lanes`    decode_with_indexes of every lane, interleaved back into symbol order
"""
from __future__ import annotations

import struct
from typing import List

import numpy as np

from oracle.ref_rans import decode_with_indexes, encode_with_indexes


def encode_lanes(symbols, indexes, W: int, cdfs, cdf_lengths, offsets) -> bytes:
    """The laned stream of W lanes: little-endian uint32 words {W, byte length of every lane}, then the lanes in order."""
    if not 1 <= W <= 32:
        raise ValueError("W must be in 1..32")
    sym, idx = np.asarray(symbols).ravel(), np.asarray(indexes).ravel()
    lanes = [encode_with_indexes(sym[l::W], idx[l::W], cdfs, cdf_lengths, offsets) for l in range(W)]
    return struct.pack(f"<{1 + W}I", W, *[len(b) for b in lanes]) + b"".join(lanes)


def split_lanes(data: bytes, W: int) -> List[bytes]:
    """The W lane streams of a laned stream.  Raises ValueError for a malformed header: another lane count, a length that is not
    a multiple of 4 or below 8, or lengths that do not add up to the stream."""
    if len(data) % 4 or len(data) < 4 * (1 + W):
        raise ValueError("laned stream shorter than its header or not a multiple of 4")
    head = struct.unpack(f"<{1 + W}I", data[: 4 * (1 + W)])
    if head[0] != W:
        raise ValueError(f"header gives {head[0]} lanes, expected {W}")
    lens = head[1:]
    if any(n % 4 or n < 8 for n in lens) or 4 * (1 + W) + sum(lens) != len(data):
        raise ValueError("lane lengths are not multiples of 4 of at least 8 bytes adding up to the stream")
    out, pos = [], 4 * (1 + W)
    for n in lens:
        out.append(data[pos: pos + n])
        pos += n
    return out


def decode_lanes(data: bytes, indexes, W: int, cdfs, cdf_lengths, offsets) -> List[int]:
    """decode_with_indexes of every lane of a laned stream, interleaved back into symbol order.  Raises ValueError for a
    malformed header or a lane shorter than its decode needs."""
    idx = np.asarray(indexes).ravel()
    out = [0] * len(idx)
    for l, lane in enumerate(split_lanes(data, W)):
        out[l::W] = decode_with_indexes(lane, idx[l::W], cdfs, cdf_lengths, offsets)
    return out
