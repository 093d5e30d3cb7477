"""A small hand DEFLATE (RFC 1951) encoder for the streams zlib never writes: stored, fixed and dynamic blocks from a
token list (a byte value is a literal, (length, distance) a match) with code lengths given by the caller, and every
malformed construct include/v2p_vcf.h lists.

  CASES -> {name: (raw DEFLATE stream, the text it inflates to, or None when zlib must refuse it)}
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
CL_LENS = [4, 5, 5, 5, 4, 4, 4, 4, 4, 4, 4, 4, 4, 5, 5, 5, 4, 4, 4]  # a complete code-length code: 13 x 4 + 6 x 5 bits
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 32


class BitWriter:
    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def bits(self, v: int, n: int):
        self.acc |= (v & ((1 << n) - 1)) << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def code(self, c: int, n: int):  # Huffman codes go most-significant bit first
        self.bits(int(format(c, "0%db" % n)[::-1], 2) if n else 0, n)

    def align(self):
        if self.n:
            self.bits(0, 8 - self.n)

    def bytes(self) -> bytes:
        return bytes(self.out) + (bytes([self.acc & 255]) if self.n else b"")


def canonical(lens: Sequence[int]) -> List[int]:
    """Canonical codes (RFC 1951 3.2.2) of a length set; codes of an over-subscribed set are still assigned."""
    bl = [0] * 16
    for l in lens:
        bl[l] += 1
    bl[0], code, nxt = 0, 0, [0] * 16
    for b in range(1, 16):
        code = (code + bl[b - 1]) << 1
        nxt[b] = code
    out = []
    for l in lens:
        out.append(nxt[l] if l else 0)
        if l:
            nxt[l] += 1
    return out


def len_sym(length: int) -> Tuple[int, int, int]:
    s = max(i for i in range(29) if LEN_BASE[i] <= length) if length != 258 else 28
    return 257 + s, length - LEN_BASE[s], LEN_EXTRA[s]


def dist_sym(d: int) -> Tuple[int, int, int]:
    s = max(i for i in range(30) if DIST_BASE[i] <= d)
    return s, d - DIST_BASE[s], DIST_EXTRA[s]


def expand(tokens) -> bytes:
    out = bytearray()
    for t in tokens:
        if isinstance(t, int):
            out.append(t)
        else:
            ln, d = t
            for _ in range(ln):
                out.append(out[-d])
    return bytes(out)


def symbols(w: BitWriter, tokens, lit: Sequence[int], dist: Sequence[int], end: bool = True):
    lc, dc = canonical(lit), canonical(dist)
    for t in tokens:
        if isinstance(t, int):
            w.code(lc[t], lit[t])
        elif t[0] == "sym":  # a raw lit/len or distance symbol: ("sym", lit_sym, dist_sym or None)
            w.code(lc[t[1]], lit[t[1]])
            if t[2] is not None:
                w.code(dc[t[2]], dist[t[2]])
        else:
            s, e, n = len_sym(t[0])
            w.code(lc[s], lit[s])
            w.bits(e, n)
            s, e, n = dist_sym(t[1])
            w.code(dc[s], dist[s])
            w.bits(e, n)
    if end:
        w.code(lc[256], lit[256])


def stored(w: BitWriter, data: bytes, final: bool, nlen: Optional[int] = None):
    w.bits(int(final), 1), w.bits(0, 2)
    w.align()
    w.bits(len(data), 16), w.bits((~len(data) & 0xFFFF) if nlen is None else nlen, 16)
    for b in data:
        w.bits(b, 8)


def fixed(w: BitWriter, tokens, final: bool):
    w.bits(int(final), 1), w.bits(1, 2)
    symbols(w, tokens, FIXED_LIT, FIXED_DIST)


def rle(lens: Sequence[int]) -> List[Tuple[int, int]]:
    """Plain code-length symbols, one per length: [(symbol, extra value)]."""
    return [(l, 0) for l in lens]


def dynamic(w: BitWriter, tokens, lit: Sequence[int], dist: Sequence[int], final: bool, cl_lens: Sequence[int] = CL_LENS,
            cl_seq: Optional[List[Tuple[int, int]]] = None, hlit: Optional[int] = None, hdist: Optional[int] = None,
            hclen: int = 19):
    """cl_seq: the code-length symbols to send (default: one per length of lit + dist); hlit/hdist: the header fields
    (default: len(lit), len(dist))."""
    hlit = len(lit) if hlit is None else hlit
    hdist = len(dist) if hdist is None else hdist
    w.bits(int(final), 1), w.bits(2, 2)
    w.bits(hlit - 257, 5), w.bits(hdist - 1, 5), w.bits(hclen - 4, 4)
    for i in range(hclen):
        w.bits(cl_lens[CL_ORDER[i]], 3)
    cc = canonical(cl_lens)
    for s, e in (rle(list(lit) + list(dist)) if cl_seq is None else cl_seq):
        w.code(cc[s], cl_lens[s])
        if s >= 16:
            w.bits(e, {16: 2, 17: 3, 18: 7}[s])
    symbols(w, tokens, list(lit) + [0] * (288 - len(lit)), list(dist) + [0] * (32 - len(dist)))


def stream(*blocks) -> bytes:
    w = BitWriter()
    for fn, args in blocks:
        fn(w, *args)
    return w.bytes()


def _lit(pairs: Dict[int, int], n: int = 286) -> List[int]:
    lens = [0] * n
    for s, l in pairs.items():
        lens[s] = l
    return lens


def ok_lit() -> List[int]:
    """A complete lit/len code over 0..257: 254 codes of 8 bits, four of 9."""
    return _lit({s: 8 for s in range(254)} | {254: 9, 255: 9, 256: 9, 257: 9})


def _cases():
    c = {}
    # 15-bit codes: lengths 1..14 and two of 15 (complete); a single distance code of length 1 (incomplete, allowed)
    deep = {97 + i: i + 1 for i in range(12)}
    deep.update({257: 13, 109: 14, 256: 15, 110: 15})
    toks = [97, 110, 109, 98, 110, (3, 1), 108, 110]
    c["codes_of_15_bits"] = (stream((dynamic, (toks, _lit(deep), [1], True))), expand(toks))
    # HDIST = 1 with a zero length: no distance codes at all, literals only
    toks = list(b"no distances here")
    c["no_distance_codes"] = (stream((dynamic, (toks, ok_lit(), [0], True))), expand(toks))
    # repeat codes at their extreme counts (16: 3 and 6, 17: 3 and 10, 18: 11 and 138); 15 literals + EOB of 4 bits
    lit = [0] * 97 + [4] * 15 + [0] * 144 + [4] + [0] * 29
    seq = [(17, 10 - 3), (17, 3 - 3), (18, 81 - 11), (0, 0), (0, 0), (0, 0),     # 0..96: 10 + 3 + 81 + 3 zeros
           (4, 0), (16, 6 - 3), (16, 3 - 3), (4, 0), (4, 0), (4, 0), (4, 0), (4, 0),  # 97..111: 1 + 6 + 3 + 5 fours
           (18, 138 - 11), (17, 6 - 3),                                          # 112..255: 138 + 6 zeros
           (4, 0),                                                               # 256
           (18, 11 - 11), (18, 19 - 11)]                                         # 257..285 and the one distance: 30 zeros
    assert sum(1 if s < 16 else 3 + e if s in (16, 17) else 11 + e for s, e in seq) == 287
    toks = [97 + i for i in range(15)] * 3
    c["repeat_codes_at_extreme_counts"] = (stream((dynamic, (toks, lit, [0], True, CL_LENS, seq))), expand(toks))
    # distance 32768 with length 258, from a fixed block back into the stored block before it
    data = bytes((i * 7 + (i >> 8)) & 255 for i in range(32768))
    toks = [(258, 32768), 65, (258, 1)]
    c["distance_32768_length_258"] = (stream((stored, (data, False)), (fixed, (toks, True))), expand(list(data) + toks))
    # several blocks, an empty stored block between them (as Z_FULL_FLUSH writes), bytes after the end of the stream
    toks = list(b"abcabcabc") + [(12, 3)]
    c["empty_stored_and_trailing_bytes"] = (stream((fixed, (toks, False)), (stored, (b"", False)), (stored, (b"xyz", True))) +
                                            b"\x00junk", expand(toks) + b"xyz")
    # --- malformed: zlib refuses every one
    c["bad_over_subscribed_lit"] = (stream((dynamic, ([65], _lit({65: 1, 66: 1, 256: 1}), [1], True))), None)
    c["bad_incomplete_lit"] = (stream((dynamic, ([65], _lit({65: 2, 256: 2, 66: 2}), [1], True))), None)
    c["bad_incomplete_cl_code"] = (stream((dynamic, ([65], ok_lit(), [1], True, [5] * 19))), None)
    c["bad_over_subscribed_dist"] = (stream((dynamic, ([65], ok_lit(), [1, 1, 1], True))), None)
    c["bad_missing_end_of_block"] = (stream((dynamic, ([65], _lit({s: 8 for s in range(256)}), [1], True))), None)
    c["bad_lit_symbol_286"] = (stream((fixed, ([65, ("sym", 286, None)], True))), None)
    c["bad_dist_symbol_30"] = (stream((fixed, ([65, 66, 67, ("sym", 257, 30)], True))), None)
    c["bad_hlit_287"] = (stream((dynamic, ([65], ok_lit() + [0], [1], True))), None)
    c["bad_hdist_31"] = (stream((dynamic, ([65], ok_lit(), [1] + [0] * 30, True))), None)
    c["bad_repeat_with_no_previous"] = (stream((dynamic, ([65], ok_lit(), [1], True, CL_LENS, [(16, 0)] + rle(ok_lit() + [1])))),
                                        None)
    c["bad_repeat_past_hlit_hdist"] = (stream((dynamic, ([65], ok_lit(), [1], True, CL_LENS, rle(ok_lit()) + [(18, 0)]))), None)
    c["bad_stored_nlen"] = (stream((stored, (b"abc", True, 0x1234))), None)
    c["bad_btype_3"] = (bytes([0b111]) + b"\x00" * 8, None)
    c["bad_distance_too_far"] = (stream((fixed, ([65, 66, (3, 3)], True))), None)
    c["bad_distance_too_far_after_stored"] = (stream((stored, (b"ab", False)), (fixed, ([(3, 4)], True))), None)
    c["bad_unfinished_stream"] = (stream((fixed, ([65, 66], False))), None)
    c["bad_truncated_stream"] = (stream((stored, (b"abcdef", True)))[:-2], None)
    c["bad_empty_data"] = (b"", None)
    return c


CASES = _cases()
