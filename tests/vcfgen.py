"""Inputs for the device VCF reader at scale, with their ground truth known by construction.

The plain-Python twin (oracle/vcftext.py) walks every byte and is too slow for texts of tens of MB, so the large tests
get their truth from how the text was made instead:
  - line_tables(text)        numpy restatement of v2p_vcf_load's line table (newlines, '\r' strip, '#' / empty lines,
                             the first #CHROM line, the 9th tab of each data line)
  - decodable_masks(...)     a mask matrix whose bits name only csqs the record has (maskdecode can decode it);
                             synth/vcftext.py writes it as text, decorate() adds meta / comment / empty / CRLF lines
  - filler_line(...)         records whose cells carry long ':'-fields in front of the mask (only the last field counts)
  - cell_starts(...)         byte offset of every sample cell of a data line; word_starts(...) of its mask words
  - a1_error_cases(...)      malformed spots in a short_records_text and the error each one must give
  - fuzz_text(rng)           seeded grammar-based texts with random byte edits (small: checked against the twin directly)
  - site_lists(...)          vectorized restatement of maskdecode.site_lists
tests/test_vcf_edges_twin.py checks each of these against the twin or maskdecode on small instances.
"""
from __future__ import annotations

import re
from typing import Dict, List, Sequence

import numpy as np

from oracle import vcftext as O
from synth import vcftext as S

HDR = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT"

# v2p_vcf_parse_masks: "VCF line L, sample column C: <what>", one phrase per error class
WHAT = {
    "a mask word with a character other than a decimal digit": O.BAD_CHAR,
    "an empty mask word": O.EMPTY,
    "a mask word above 2^32-1": O.OVERFLOW,
    "a number of sample cells other than the #CHROM line's": O.COUNT,
}
_MSG = re.compile(r"VCF line (\d+), sample column (\d+): ([^(]+?)(?: \(status \d+ \w+\))?$")


def error_triple(msg: str):
    """message of a V2P_ERR_VCF_PARSE (bare, or as EngineError prints it) -> (1-based file line, 1-based sample column,
    class)"""
    m = _MSG.search(msg)
    assert m and m.group(3) in WHAT, msg
    return int(m.group(1)), int(m.group(2)), WHAT[m.group(3)]


def header(n_samples: int, name: bytes = b"S%d") -> bytes:
    return HDR + b"".join(b"\t" + name % i for i in range(n_samples))


def record(pos: int, cells: Sequence[bytes], id_pad: int = 0) -> bytes:
    """A data line; id_pad extra bytes in the ID column move the 9th tab without touching the cells."""
    return b"1\t%d\t%s\tC\tT\t.\t.\tAC=1\tGT:BCSQ\t" % (pos, b"." + b"i" * id_pad) + b"\t".join(cells)


# ------------------------------------------------------------------------------------------------------ line tables
def line_tables(text) -> Dict:
    """The twin's index(text) with numpy: same keys, same values."""
    t = np.frombuffer(text, np.uint8) if isinstance(text, (bytes, bytearray)) else np.asarray(text, np.uint8)
    n = len(t)
    if n == 0:
        raise O.VcfParseError(0, 0, O.COUNT)
    starts = np.concatenate([[0], np.flatnonzero(t[:n - 1] == 10) + 1]).astype(np.int64)
    ends = np.empty_like(starts)
    ends[:-1] = starts[1:] - 1
    ends[-1] = n - 1 if t[n - 1] == 10 else n
    ends -= (ends > starts) & (t[np.maximum(ends - 1, 0)] == 13)
    nonempty = ends > starts
    hashed = nonempty & (t[starts] == 35)
    data = nonempty & ~hashed
    cand = np.flatnonzero(hashed & (ends - starts >= 6))
    probe = t[np.minimum(starts[cand][:, None] + np.arange(6), n - 1)]
    chrom = cand[(probe == np.frombuffer(b"#CHROM", np.uint8)).all(axis=1)]
    if not len(chrom):
        raise O.VcfParseError(0, 0, O.COUNT)
    hb, he = int(starts[chrom[0]]), int(ends[chrom[0]])
    tabs = np.flatnonzero(t == 9)
    n_tabs = int(np.searchsorted(tabs, he) - np.searchsorted(tabs, hb))
    b, e = starts[data], ends[data]
    k = np.searchsorted(tabs, b) + 8
    tab9 = tabs[np.minimum(k, len(tabs) - 1)] if len(tabs) else np.zeros_like(k)
    has = (k < len(tabs)) & (tab9 < e)
    u = lambda x: np.asarray(x, np.uint64)
    return dict(n_samples=max(n_tabs - 8, 0), n_lines=int(data.sum()), header_begin=hb, header_end=he, line_begin=u(b),
                cells_begin=u(np.where(has, tab9 + 1, e)), line_end=u(e), has_cells=has, line_no=np.flatnonzero(data) + 1)


def cell_starts(text: np.ndarray, ix: Dict, line: int) -> np.ndarray:
    """Offsets of the first byte of every sample cell of data line `line` (which must have cells)."""
    cb, e = int(ix["cells_begin"][line]), int(ix["line_end"][line])
    return np.concatenate([[cb], np.flatnonzero(text[cb:e] == 9) + cb + 1])


def word_starts(text, start):
    """Offsets of the words of the last ':'-field of the cell starting at `start`."""
    end = start
    while text[end] not in (9, 10, 13):
        end += 1
    f = start + text[start:end].tobytes().rfind(b":") + 1
    return [f] + [f + i + 1 for i, c in enumerate(text[f:end]) if c == 44], end


# ----------------------------------------------------------------------------------------------- masks and texts
def decodable_masks(rng, n_csq: np.ndarray, n_samples: int, p_zero: float = 0.5) -> np.ndarray:
    """masks[n_rec, n_samples, W] (W = words_for of the largest n_csq) with bits only for csqs the record has: word w
    bit pair i is csq 15*w + i (MaskDecoder.rs:122-153), so pair 15 of word w and pair 0 of word w+1 name the same csq.
    Words past a record's own word count are 0.  A mix of wide and small values gives words of 1-10 digits."""
    n_csq = np.asarray(n_csq, np.int64)
    W = S.words_for(int(n_csq.max()))
    k = 15 * np.arange(W)[:, None] + np.arange(16)[None, :]  # [W, 16] csq of each bit pair
    pair = np.uint64(3) << (2 * np.arange(16, dtype=np.uint64))
    allowed = ((k[None] < n_csq[:, None, None]) * pair).sum(axis=2).astype(np.uint32)  # [n_rec, W]
    own = np.arange(W)[None, :] < np.array([S.words_for(int(c)) for c in n_csq])[:, None]
    allowed &= np.where(own, 0xFFFFFFFF, 0).astype(np.uint32)
    v = rng.integers(0, 1 << 32, size=(len(n_csq), n_samples, W), dtype=np.uint64).astype(np.uint32)
    small = rng.random((len(n_csq), n_samples, W)) < 0.3
    v = np.where(small, v & np.uint32(0x3ff), v) & allowed[:, None, :]
    v[rng.random((len(n_csq), n_samples)) < p_zero] = 0
    return v


JUNK = (b"", b"##meta=%d", b"#comment %d", b"\r", b"#", b"#CHROM\tPOS\tID\tlater #CHROM lines are comments %d")


def decorate(text: bytes, rng, p_junk: float = 0.05, p_crlf: float = 0.2) -> bytes:
    """Insert meta, comment, empty and '\r'-only lines between the records of a synth/vcftext.py text and end some
    records with CRLF, so that a file line number is not a data ordinal.  Data lines keep their order."""
    lines = text.split(b"\n")
    assert lines[-1] == b"" and lines[1].startswith(b"#CHROM")
    recs = lines[2:-1]
    junk = rng.random(len(recs)) < p_junk
    kind = rng.integers(0, len(JUNK), len(recs))
    crlf = rng.random(len(recs)) < p_crlf
    out = lines[:2]
    for i, r in enumerate(recs):
        if junk[i]:
            j = JUNK[kind[i]]
            out.append(j % i if b"%d" in j else j)
        out.append(r + b"\r" if crlf[i] else r)
    return b"\n".join(out) + b"\n"


def short_records_text(rng, n_lines: int, n_samples: int, max_csq: int = 45, p_junk: float = 0.05):
    """(text, masks, n_csq): n_lines records of W = 1..words_for(max_csq), decorated."""
    n_csq = rng.integers(1, max_csq + 1, n_lines)
    n_csq[: min(n_lines, 3)] = [1, 16, max_csq][: min(n_lines, 3)]  # the widths at both ends, csq 15 aliasing
    masks = decodable_masks(rng, n_csq, n_samples)
    if masks.shape[2] >= 2:  # bits 30/31 of word 0: csq 15, which word 1 bits 0/1 also name
        hit = (n_csq >= 16)[:, None] & (rng.random((n_lines, n_samples)) < 0.2)
        top = rng.integers(1, 4, hit.shape).astype(np.uint32) << np.uint32(30)
        masks[:, :, 0] |= np.where(hit, top, np.uint32(0))
    text = S.vcf_text(["S%d" % i for i in range(n_samples)], [[""] * int(c) for c in n_csq], masks, block=2048)
    return decorate(text, rng, p_junk=p_junk), masks, n_csq


def want_rows(masks: np.ndarray, n_csq: np.ndarray, rows: Sequence[int]) -> np.ndarray:
    """The matrix parse_masks(rows) must give for a text written from masks: W = the widest selected record."""
    rows = np.asarray(rows, np.int64)
    W = max([1] + [S.words_for(int(c)) for c in np.unique(n_csq[rows])]) if len(rows) else 1
    return masks[rows][:, :, :W]


# --------------------------------------------------------------------------------- long cells: ':'-fields in front
FILL = np.frombuffer(b"0123456789,|/.x", np.uint8)


def filler(rng, n: int) -> bytes:
    """n bytes with no ':', tab or line end: digits, commas and a few non-digits (a field the mask does not use)."""
    return FILL[rng.integers(0, len(FILL), n)].tobytes()


def words_cell(words: Sequence[int]) -> bytes:
    return b",".join(b"%d" % w for w in words)


def filler_line(rng, pos: int, rows_words: List[Sequence[int]], fill_len: Sequence[int]) -> bytes:
    """A record whose cell s is `<fill_len[s] filler bytes>:<words>` (no ':' when fill_len[s] < 0)."""
    cells = [(filler(rng, f) + b":" if f >= 0 else b"") + words_cell(w) for w, f in zip(rows_words, fill_len)]
    return record(pos, cells)


def matrix_of(cells_words: List[List[Sequence[int]]], n_samples: int) -> np.ndarray:
    W = max([1] + [len(w) for row in cells_words for w in row])
    out = np.zeros((len(cells_words), n_samples, W), np.uint32)
    for r, row in enumerate(cells_words):
        for s, w in enumerate(row):
            out[r, s, :len(w)] = w
    return out


def a1_error_cases(t: np.ndarray, ix: Dict, masks: np.ndarray):
    """Malformed spots in a short_records_text (at least 4 records, 24 samples): [(name, [(offset, byte)], bad data
    lines, (file line, sample column, class) of the first error)].  Early, middle and late records; a count error
    alone and with a cell error further left; all three first ones at once."""
    n, ns = ix["n_lines"], ix["n_samples"]
    L_ = lambda r: int(ix["line_no"][r])
    cell = lambda r, s: int(cell_starts(t, ix, r)[s])
    big = [r for r in range(n - 1, 0, -1) if (masks[r, :, 0] >= 10 ** 9).any()][0]
    big_s = int(np.flatnonzero(masks[big, :, 0] >= 10 ** 9)[0])
    spots = {  # name -> ([(offset, byte)], record, want)
        "early_bad_char": ([(word_starts(t, cell(2, 5))[0][0], ord("x"))], 2, (L_(2), 6, O.BAD_CHAR)),
        "middle_empty": ([(word_starts(t, cell(n // 2, 0))[0][0], ord(","))], n // 2, (L_(n // 2), 1, O.EMPTY)),
        "late_overflow": ([(word_starts(t, cell(big, big_s))[0][0], ord("9"))], big, (L_(big), big_s + 1, O.OVERFLOW)),
        "count": ([(cell(n // 3, ns - 1) - 1, ord(","))], n // 3, (L_(n // 3), ns, O.COUNT)),
        "count_and_a_cell_error_left_of_it": ([(cell(n // 3, ns - 1) - 1, ord(",")), (word_starts(t, cell(n // 3, 2))[0][0], ord("x"))],
                                              n // 3, (L_(n // 3), 3, O.BAD_CHAR)),
    }
    assert t[cell(n // 3, ns - 1) - 1] == 9
    cases = [(k, v[0], [v[1]], v[2]) for k, v in spots.items()]
    cases.append(("early_middle_late_at_once", sum((spots[k][0] for k in ("late_overflow", "middle_empty", "early_bad_char")), []),
                  [2, n // 2, big], spots["early_bad_char"][2]))
    return cases


FUZZ_BYTES = np.frombuffer(b"\t\t\n\n\r::,,0123456789#x.", np.uint8)


def fuzz_text(rng):
    """Grammar: meta lines, a #CHROM line of 0-8 samples, records with GT-like fields and 1-4 word masks, empty and
    comment lines, CRLF; then 1-3 random byte inserts / deletes / replaces, half of them digits."""
    ns = int(rng.integers(1, 9)) if rng.random() < 0.95 else 0
    target = int(rng.integers(1 << 10, 1 << 16))
    lines = [b"##fileformat=VCFv4.2"] * int(rng.integers(0, 3)) + [header(ns)]
    size = 0
    flawed = rng.random() < 0.5  # malformed words and cell counts; the byte edits below may break any text

    def word():
        if flawed and rng.random() < 0.001:
            return [b"", b".", b"4294967296", b"1x"][int(rng.integers(0, 4))]
        w = b"%d" % int(rng.integers(0, 1 << 32) >> int(rng.integers(0, 32)))
        return b"0" * int(rng.integers(0, 4)) + w if rng.random() < 0.1 else w

    def cell():
        pre = b"".join(rng.choice([b"0|1", b"1/0", b".", b"12,3"]) + b":" for _ in range(int(rng.integers(0, 3))))
        return pre + b",".join(word() for _ in range(int(rng.integers(1, 5))))

    while size < target:
        if rng.random() < 0.05:
            line = [b"", b"#c", b"##x=1", b"\r"][int(rng.integers(0, 4))]
        else:
            k = ns + (int(rng.integers(-1, 2)) if flawed and rng.random() < 0.01 else 0)
            line = record(len(lines), [cell() for _ in range(max(k, 0))], id_pad=int(rng.integers(0, 16)))
        lines.append(line + (b"\r" if rng.random() < 0.1 else b""))
        size += len(line) + 1
    text = bytearray(b"\n".join(lines) + (b"\n" if rng.random() < 0.8 else b""))
    for _ in range(int(rng.integers(1, 4))):
        p = int(rng.integers(0, len(text)))
        u = rng.random()
        b = 48 + int(rng.integers(0, 10)) if u < 0.5 else int(FUZZ_BYTES[rng.integers(0, len(FUZZ_BYTES))]) if u < 0.9 else int(rng.integers(0, 256))
        op = int(rng.integers(0, 3))
        if op == 0:
            text.insert(p, b)
        elif op == 1:
            del text[p]
        else:
            text[p] = b
    return bytes(text)


# -------------------------------------------------------------------------------------------------- site lists
def site_lists(masks: np.ndarray, csq_begin: np.ndarray, csq_site: np.ndarray):
    """maskdecode.site_lists without the Python loops: every set bit -> (haplotype, site), sorted and deduplicated."""
    n_rec, n_samp, W = masks.shape
    r, s, w = np.nonzero(masks)
    v = masks[r, s, w].astype(np.uint64)
    bit = np.arange(32, dtype=np.uint64)
    on = ((v[:, None] >> bit[None, :]) & np.uint64(1)).astype(bool)
    i, b = np.nonzero(on)
    r, s, w = r[i], s[i], w[i]
    k = 15 * w.astype(np.int64) + b // 2
    n_csq = (csq_begin[1:].astype(np.int64) - csq_begin[:-1].astype(np.int64))[r]
    if (k >= n_csq).any():
        raise IndexError("a mask selects a csq the record does not have")
    site = np.asarray(csq_site, np.int64)[csq_begin[r].astype(np.int64) + k]
    hap = 2 * s.astype(np.int64) + (b & 1)
    keep = site >= 0
    span = int(site.max(initial=0)) + 1
    key = np.unique(hap[keep] * span + site[keep])
    hk, sk = key // span, key % span
    site_begin = np.zeros(2 * n_samp + 1, np.uint64)
    np.cumsum(np.bincount(hk, minlength=2 * n_samp), out=site_begin[1:])
    return site_begin, sk.astype(np.uint32)
