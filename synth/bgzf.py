"""BGZF writer (SAM spec section 4.1), laid out as bgzip lays it out: the text cut into 0xff00-byte inputs, each one raw
DEFLATE member with XLEN 6 holding the BC subfield, then the 28-byte EOF block.  Test and measurement input only.

  members(text, level, strategy, block_size, flush_at, threads) -> [member bytes]  (one BGZF block each, no EOF block)
  write(text, ..., eof=True)                                     -> the file

flush_at: offsets inside each input where the compressor does a Z_FULL_FLUSH (the member then holds several DEFLATE
blocks and an empty stored block at each point).  A member whose data does not fit BSIZE (incompressible input at
block_size 65536) is split in two, as bgzip shrinks its input.  Blocks compress on a thread pool: zlib releases the GIL.
"""
from __future__ import annotations

import os
import struct
import zlib
from concurrent.futures import ThreadPoolExecutor
from typing import List, Sequence

EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
BLOCK_INPUT = 0xFF00
MAX_BLOCK = 65536
STRATEGIES = {"default": zlib.Z_DEFAULT_STRATEGY, "filtered": zlib.Z_FILTERED, "huffman_only": zlib.Z_HUFFMAN_ONLY,
              "rle": zlib.Z_RLE, "fixed": zlib.Z_FIXED}


def member(cdata: bytes, raw: bytes) -> bytes:
    """One BGZF block: gzip header with FEXTRA (XLEN 6, BC = BSIZE), raw DEFLATE data, CRC32, ISIZE."""
    bsize = 18 + len(cdata) + 8 - 1
    hdr = struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 0xFF, 6, ord("B"), ord("C"), 2, bsize)
    return hdr + cdata + struct.pack("<II", zlib.crc32(raw) & 0xFFFFFFFF, len(raw))


def deflate(raw: bytes, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, flush_at: Sequence[int] = ()) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    out, at = [], 0
    for f in sorted(p for p in set(flush_at) if 0 < p < len(raw)):
        out += [c.compress(raw[at:f]), c.flush(zlib.Z_FULL_FLUSH)]
        at = f
    out += [c.compress(raw[at:]), c.flush()]
    return b"".join(out)


def _members_of(raw: bytes, level, strategy, flush_at) -> List[bytes]:
    cdata = deflate(raw, level, strategy, flush_at)
    if 26 + len(cdata) <= MAX_BLOCK:
        return [member(cdata, raw)]
    h = len(raw) // 2
    return _members_of(raw[:h], level, strategy, flush_at) + _members_of(raw[h:], level, strategy, [f - h for f in flush_at])


def members(text: bytes, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, block_size: int = BLOCK_INPUT,
            flush_at: Sequence[int] = (), threads: int = 0) -> List[bytes]:
    assert 1 <= block_size <= MAX_BLOCK
    chunks = [text[i:i + block_size] for i in range(0, len(text), block_size)]
    work = lambda raw: _members_of(raw, level, strategy, flush_at)
    if len(chunks) < 64:
        parts = [work(c) for c in chunks]
    else:
        with ThreadPoolExecutor(threads or os.cpu_count() or 1) as ex:
            parts = list(ex.map(work, chunks, chunksize=max(1, len(chunks) // 256)))
    return [m for p in parts for m in p]


def write(text: bytes, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, block_size: int = BLOCK_INPUT,
          flush_at: Sequence[int] = (), eof: bool = True, threads: int = 0) -> bytes:
    return b"".join(members(text, level, strategy, block_size, flush_at, threads)) + (EOF_BLOCK if eof else b"")
