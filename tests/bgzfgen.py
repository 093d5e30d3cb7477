"""BGZF inputs whose result is known by construction, for tests/test_bgzf_twin.py (checked against the twin,
oracle/bgzf.py) and tests/test_gpu_vcf_bgzf.py (the device against the twin): small VCF texts cut into blocks, the
deflategen streams wrapped as blocks, corruptions with the (block, offset, class) they must report, seeded flips."""
from __future__ import annotations

import re
import struct
import zlib
from typing import Dict, List, Sequence, Tuple

import numpy as np

from synth import bgzf as W
from tests import deflategen as D

HEADER, DEFLATE, SIZE, CRC = 1, 2, 3, 4
WHAT = {"bad BGZF block header": HEADER, "invalid DEFLATE data": DEFLATE,
        "inflated size differs from the trailer's ISIZE": SIZE, "CRC-32 differs from the trailer's": CRC}


def error_triple(msg: str) -> Tuple[int, int, int]:
    """(block, offset, class) of a V2P_ERR_BGZF message."""
    m = re.match(r"BGZF block (\d+) at byte (\d+): ([^(]*?)(?: \(.*)?$", msg)
    assert m and m.group(3) in WHAT, msg
    return int(m.group(1)), int(m.group(2)), WHAT[m.group(3)]


def small_vcf(n_records: int = 40, n_samples: int = 5, seed: int = 1) -> bytes:
    rng = np.random.default_rng(seed)
    hdr = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT" + b"".join(b"\tS%d" % i for i in range(n_samples))
    lines = [b"##fileformat=VCFv4.2", hdr]
    for r in range(n_records):
        cells = [b"0|1:%d" % int(rng.integers(0, 1 << 20)) if rng.random() < 0.5 else b"%d,%d" % tuple(rng.integers(0, 9, 2))
                 for _ in range(n_samples)]
        lines.append(b"1\t%d\t.\tC\tT\t.\t.\tBCSQ=missense|G%d|T1|protein_coding|+|1A>1C|x\tGT:BCSQ\t%s" % (r + 1, r % 7, b"\t".join(cells)))
    return b"\r\n".join(lines[:3]) + b"\r\n" + b"\n".join(lines[3:]) + b"\n"


def split(text: bytes, cuts: Sequence[int], level: int = 6) -> bytes:
    """One block per piece between the cuts, then the EOF block."""
    at = [0] + sorted(cuts) + [len(text)]
    return b"".join(W.member(W.deflate(text[a:b], level), text[a:b]) for a, b in zip(at, at[1:])) + W.EOF_BLOCK


def offsets(members: Sequence[bytes]) -> List[int]:
    return list(np.cumsum([0] + [len(m) for m in members])[:-1])


def put(data: bytes, at: int, fmt: str, *v) -> bytes:
    b = bytearray(data)
    struct.pack_into(fmt, b, at, *v)
    return bytes(b)


def corruptions(text: bytes) -> Dict[str, Tuple[bytes, Tuple[int, int, int]]]:
    """name -> (file, (block, offset, class) it must report).  The text is cut into 9 blocks of level 6 data."""
    ms = W.members(text, 6, block_size=max(1, len(text) // 8))
    assert len(ms) >= 9
    off = offsets(ms)
    good = b"".join(ms)
    eof_at = len(good)

    def with_block(k, m):
        return b"".join(ms[:k] + [m] + ms[k + 1:]) + W.EOF_BLOCK

    c = {}
    k = 3
    m = ms[k]
    bsize = len(m) - 1
    c["header_magic"] = (with_block(k, b"\x1f\x8c" + m[2:]), (k, off[k], HEADER))
    c["header_flg"] = (with_block(k, m[:3] + b"\x05" + m[4:]), (k, off[k], HEADER))
    c["header_xlen_5"] = (with_block(k, put(m, 10, "<H", 5)), (k, off[k], HEADER))
    c["header_no_bc"] = (with_block(k, m[:12] + b"XC" + m[14:]), (k, off[k], HEADER))
    c["header_bc_slen_4"] = (with_block(k, put(m, 14, "<H", 4)), (k, off[k], HEADER))
    c["header_bsize_past_end"] = (b"".join(ms[:k]) + put(m, 16, "<H", bsize + 100), (k, off[k], HEADER))
    c["header_bsize_too_small"] = (with_block(k, put(m, 16, "<H", 18 + 8 - 2)), (k, off[k], HEADER))
    c["header_isize_65537"] = (with_block(k, put(m, len(m) - 4, "<I", 65537)), (k, off[k], HEADER))
    c["header_truncated"] = (good + W.EOF_BLOCK[:17], (len(ms), eof_at, HEADER))
    c["plain_text"] = (text, (0, 0, HEADER))
    c["plain_gzip"] = (_gzip(text), (0, 0, HEADER))
    c["deflate_btype_3"] = (with_block(k, m[:18] + bytes([m[18] | 0b110]) + m[19:]), (k, off[k], DEFLATE))
    c["size_isize_plus_1"] = (with_block(k, put(m, len(m) - 4, "<I", struct.unpack_from("<I", m, len(m) - 4)[0] + 1)),
                              (k, off[k], SIZE))
    c["crc_flipped"] = (with_block(k, put(m, len(m) - 8, "<I", struct.unpack_from("<I", m, len(m) - 8)[0] ^ 1)), (k, off[k], CRC))
    # several bad blocks: the lowest wins, a header error behind an earlier DEFLATE error included
    bad = list(ms)
    bad[2] = bad[2][:18] + bytes([bad[2][18] | 0b110]) + bad[2][19:]
    bad[6] = b"\x00" + bad[6][1:]
    bad[7] = put(bad[7], len(bad[7]) - 8, "<I", 0)
    c["deflate_before_header"] = (b"".join(bad) + W.EOF_BLOCK, (2, off[2], DEFLATE))
    bad[2] = ms[2]
    c["header_after_good_blocks"] = (b"".join(bad) + W.EOF_BLOCK, (6, off[6], HEADER))
    bad = list(ms)
    bad[1] = put(bad[1], len(bad[1]) - 8, "<I", 0)
    bad[5] = bad[5][:18] + bytes([bad[5][18] | 0b110]) + bad[5][19:]
    c["crc_before_deflate"] = (b"".join(bad) + W.EOF_BLOCK, (1, off[1], CRC))
    return c


def _gzip(text: bytes) -> bytes:
    c = zlib.compressobj(6, zlib.DEFLATED, 31)
    return c.compress(text) + c.flush()


def flips(data: bytes, seed: int, n: int = 300):
    """n seeded corruptions of `data`: single bit flips and byte overwrites anywhere (headers, data, trailers)."""
    rng = np.random.default_rng(seed)
    for i in range(n):
        b = bytearray(data)
        for _ in range(int(rng.integers(1, 3))):
            p = int(rng.integers(0, len(b)))
            if rng.random() < 0.7:
                b[p] ^= 1 << int(rng.integers(0, 8))
            else:
                b[p] = int(rng.integers(0, 256))
        yield i, bytes(b)


def edge_blocks() -> Dict[str, Tuple[bytes, bytes]]:
    """Each deflategen stream as one BGZF block (CRC and ISIZE of its intended text; 0 / 0 when it is malformed), with
    a good block in front, so that the bad one is block 1, and a #CHROM line after it, so that the text indexes.
    name -> (file, intended text or None)."""
    lead, tail = b"##lead block\n", b"\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS0\n"
    out = {}
    for name, (stream, want) in D.CASES.items():
        body = want if want is not None else b""
        blk = struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 0xFF, 6, 66, 67, 2, 18 + len(stream) + 8 - 1) + stream + \
            struct.pack("<II", zlib.crc32(body) & 0xFFFFFFFF, len(body))
        out[name] = (W.member(W.deflate(lead), lead) + blk + W.member(W.deflate(tail), tail) + W.EOF_BLOCK,
                     None if want is None else lead + want + tail)
    return out
