"""ORACLE (test infrastructure only): plain-Python twin of the BGZF reader of include/v2p_vcf.h (v2p_vcf_load_bgzf),
with zlib as the independent inflater.

  inflate(data) -> the text, or BgzfError(block, offset, cls) for the first bad block in file order

Classes, in order of precedence within one block: HEADER (the walk stops there, but a bad block before it still comes
first), DEFLATE (zlib refuses the data, or it does not reach the end of its final block), SIZE (!= ISIZE), CRC.
"""
from __future__ import annotations

import struct
import zlib
from typing import List, Optional, Tuple

HEADER, DEFLATE, SIZE, CRC = 1, 2, 3, 4
MAX_ISIZE = 65536


class BgzfError(ValueError):
    def __init__(self, block: int, offset: int, cls: int):
        super().__init__("BGZF block %d at byte %d: class %d" % (block, offset, cls))
        self.block, self.offset, self.cls = block, offset, cls


def walk(data: bytes) -> Tuple[List[Tuple[int, bytes, int, int]], Optional[int]]:
    """-> [(offset, cdata, crc, isize)] of the blocks before the first bad header, and that header's offset (or None)."""
    out, o, n = [], 0, len(data)
    while o < n:
        h = data[o:o + 18]
        if len(h) < 18 or h[:4] != b"\x1f\x8b\x08\x04":
            return out, o
        xlen = struct.unpack_from("<H", h, 10)[0]
        if xlen < 6 or 12 + xlen > n - o:
            return out, o
        extra, x, bsize = data[o + 12:o + 12 + xlen], 0, None
        while x + 4 <= xlen:
            slen = struct.unpack_from("<H", extra, x + 2)[0]
            if x + 4 + slen > xlen:
                break
            if extra[x:x + 2] == b"BC" and slen == 2:
                bsize = struct.unpack_from("<H", extra, x + 4)[0]
            x += 4 + slen
        if bsize is None or bsize + 1 < 12 + xlen + 8 or bsize + 1 > n - o:
            return out, o
        crc, isize = struct.unpack_from("<II", data, o + bsize + 1 - 8)
        if isize > MAX_ISIZE:
            return out, o
        out.append((o, data[o + 12 + xlen:o + bsize + 1 - 8], crc, isize))
        o += bsize + 1
    return out, None


def block_class(cdata: bytes, crc: int, isize: int) -> Tuple[int, bytes]:
    d = zlib.decompressobj(-15)
    try:
        text = d.decompress(cdata)
    except zlib.error:
        return DEFLATE, b""
    if not d.eof:
        return DEFLATE, b""
    if len(text) != isize:
        return SIZE, b""
    if zlib.crc32(text) & 0xFFFFFFFF != crc:
        return CRC, b""
    return 0, text


def inflate(data: bytes) -> bytes:
    blocks, bad_header = walk(data)
    out = []
    for k, (off, cdata, crc, isize) in enumerate(blocks):
        cls, text = block_class(cdata, crc, isize)
        if cls:
            raise BgzfError(k, off, cls)
        out.append(text)
    if bad_header is not None:
        raise BgzfError(len(blocks), bad_header, HEADER)
    return b"".join(out)
