"""ORACLE (test infrastructure only): plain-Python twin of the VCF dialect of include/v2p_vcf.h, and the host's
per-record step that sits between v2p_vcf_load and v2p_vcf_parse_masks.

  index(text)                   -> the line table v2p_vcf_load returns (plus each data line's end and file line number)
  parse_masks(text, ix, rows)   -> masks[n_records, n_samples, W] (uint32), or VcfParseError for the first error in
                                   file order (lowest line, then lowest sample column)
  bcsq(text, ix, line)          -> the record's INFO/BCSQ consequence strings (columns 1-9 only)
  supported(csqs)               -> the record is kept when one of its classes is in taskgen.SUP_TYPE (Constants.rs:3-8)
"""
from __future__ import annotations

from typing import Dict, List, Sequence

import numpy as np

from oracle import taskgen

BAD_CHAR, EMPTY, OVERFLOW, COUNT = 1, 2, 3, 4  # tie order at one (line, sample column), as in csrc/v2p_vcf.cu


class VcfParseError(ValueError):
    def __init__(self, line: int, sample: int, kind: int):
        """line: 1-based line of the file; sample: 1-based sample column (0 = the file has no #CHROM line)."""
        super().__init__("VCF line %d, sample column %d: error %d" % (line, sample, kind))
        self.line, self.sample, self.kind = line, sample, kind


def index(text: bytes) -> Dict:
    n = len(text)
    starts = [0] + [i + 1 for i in range(n - 1) if text[i] == 10] if n else []
    begin, end, cells, has_cells, line_no = [], [], [], [], []
    chrom = None
    for i, b in enumerate(starts):
        e = starts[i + 1] - 1 if i + 1 < len(starts) else (n - 1 if text[n - 1] == 10 else n)
        if e > b and text[e - 1] == 13:
            e -= 1
        if e == b:
            continue
        if text[b] == 35:  # '#'
            if chrom is None and text[b:b + 6] == b"#CHROM":
                chrom = (b, e)
            continue
        tabs = [p for p in range(b, e) if text[p] == 9]
        begin.append(b), end.append(e), line_no.append(i + 1)
        cells.append(tabs[8] + 1 if len(tabs) >= 9 else e), has_cells.append(len(tabs) >= 9)
    if chrom is None:
        raise VcfParseError(0, 0, COUNT)
    n_tabs = text[chrom[0]:chrom[1]].count(b"\t")
    u = lambda x: np.asarray(x, np.uint64)
    return dict(n_samples=max(n_tabs - 8, 0), n_lines=len(begin), header_begin=chrom[0], header_end=chrom[1], line_begin=u(begin),
                cells_begin=u(cells), line_end=u(end), has_cells=has_cells, line_no=line_no)


def _cell(cell: bytes):
    """-> (words, class of the first malformed word or 0)"""
    words, err = [], 0
    for w in cell.split(b":")[-1].split(b","):
        kind = EMPTY if not w else BAD_CHAR if any(not (48 <= c <= 57) for c in w) else OVERFLOW if int(w) > 0xFFFFFFFF else 0
        err = err or kind
        words.append(int(w) if kind == 0 else 0)
    return words, err


def parse_masks(text: bytes, ix: Dict, rec_line: Sequence[int]) -> np.ndarray:
    ns = ix["n_samples"]
    rows, errs = [], []
    for l in rec_line:
        b, e = int(ix["cells_begin"][l]), int(ix["line_end"][l])
        cells = text[b:e].split(b"\t") if ix["has_cells"][l] else []
        row = []
        for k, c in enumerate(cells):
            words, err = _cell(c)
            if err:
                errs.append((ix["line_no"][l], k + 1, err))
            row.append(words)
        if len(cells) != ns:
            errs.append((ix["line_no"][l], min(len(cells), ns) + 1, COUNT))
        rows.append(row)
    if errs:
        raise VcfParseError(*min(errs))
    w = max([1] + [len(x) for row in rows for x in row])
    out = np.zeros((len(rows), ns, w), np.uint32)
    for r, row in enumerate(rows):
        for k, words in enumerate(row):
            out[r, k, :len(words)] = words
    return out


def bcsq(text: bytes, ix: Dict, line: int) -> List[str]:
    """INFO's BCSQ= list of a data line (column 8), [] when it has none."""
    cols = text[int(ix["line_begin"][line]):int(ix["cells_begin"][line])].rstrip(b"\t").split(b"\t")
    if len(cols) < 8:
        return []
    for kv in cols[7].split(b";"):
        if kv.startswith(b"BCSQ="):
            return kv[5:].decode().split(",")
    return []


def supported(csqs: Sequence[str]) -> bool:
    return any(c.split("|")[0] in taskgen.SUP_TYPE for c in csqs)
