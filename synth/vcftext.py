"""Synthetic VCF text at bench sizes: FORMAT/BCSQ mask matrix + per-record csq strings -> the text
oracle.refbin.vcf_text writes (the minimal dialect of include/v2p_vcf.h), built with numpy a block of records at a
time instead of one Python string per cell.  Byte-identical to refbin.vcf_text on the same records
(tests/test_vcftext.py)."""
from __future__ import annotations

from typing import Sequence

import numpy as np

HEADER = b"##fileformat=VCFv4.2\n"
COLUMNS = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT"


def words_for(n_csq: int) -> int:
    """Words of a record's cells: one 15-csq word each (MaskDecoder.rs:122-153), at least one."""
    return max(1, (n_csq + 14) // 15)


def _digits(v: np.ndarray):
    """uint32 values -> (digits[n, D] most significant first, left-aligned; lengths[n]); D = the longest"""
    v = v.astype(np.uint64)
    n_dig = np.ones(len(v), np.int64)
    for p in range(1, 10):
        big = v >= 10 ** p
        if not big.any():
            break
        n_dig += big
    width = int(n_dig.max()) if len(v) else 1
    out = np.zeros((len(v), width), np.uint8)
    if width == 1:
        out[:, 0] = v + 48
        return out, n_dig
    for d in range(width):
        pw = np.power(10, np.maximum(n_dig - 1 - d, 0)).astype(np.uint64)
        out[:, d] = np.where(d < n_dig, (v // pw) % 10 + 48, 0)
    return out, n_dig


def vcf_text(samples: Sequence[str], csqs: Sequence[Sequence[str]], masks: np.ndarray, block: int = 512) -> bytes:
    """masks[n_records, n_samples, W] (W >= every record's words_for(len(csqs[r])); words past a record's own count are
    ignored).  Record r is written at POS 100 + r with INFO `AC=1;BCSQ=<csqs joined by ','>`, FORMAT GT:BCSQ and the
    cell `<h1>|<h2>:<words joined by ','>`, h1 / h2 = whether any even / odd bit is set."""
    n_rec, n_samp = masks.shape[0], len(samples)
    assert masks.shape[1] == n_samp and len(csqs) == n_rec
    parts = [HEADER, COLUMNS + b"".join(b"\t" + s.encode() for s in samples) + b"\n"]
    for r0 in range(0, n_rec, block):
        r1 = min(n_rec, r0 + block)
        m = masks[r0:r1].astype(np.uint32)
        nw = np.array([words_for(len(csqs[r])) for r in range(r0, r1)], np.int64)
        prefix = [b"1\t%d\t.\tC\tT\t.\t.\tAC=1;BCSQ=%s\tGT:BCSQ\t" % (100 + r, ",".join(csqs[r]).encode()) for r in range(r0, r1)]
        if n_samp == 0:
            parts.append(b"".join(p + b"\n" for p in prefix))
            continue
        used = np.arange(m.shape[2])[None, None, :] < nw[:, None, None]  # [rec, 1, W]
        mw = np.where(used, m, 0)
        h1 = (mw & np.uint32(0x55555555)).any(axis=2)
        h2 = (mw & np.uint32(0xAAAAAAAA)).any(axis=2)
        dig, nd = _digits(m.reshape(-1))
        nd = nd.reshape(m.shape)
        # bytes per cell: "a|b:" + words + commas, then '\t' or '\n'
        cell_len = 4 + np.where(used, nd + 1, 0).sum(axis=2) - 1 + 1
        plen = np.array([len(p) for p in prefix], np.int64)
        rec_len = plen + cell_len.sum(axis=1)
        rec_off = np.zeros(len(prefix) + 1, np.int64)
        np.cumsum(rec_len, out=rec_off[1:])
        out = np.zeros(int(rec_off[-1]), np.uint8)
        for i, p in enumerate(prefix):
            out[rec_off[i]:rec_off[i] + plen[i]] = np.frombuffer(p, np.uint8)
        cell_off = np.zeros_like(cell_len)
        cell_off[:, 1:] = np.cumsum(cell_len, axis=1)[:, :-1]
        cell_off += (rec_off[:-1] + plen)[:, None]
        out[cell_off] = 48 + h1
        out[cell_off + 1] = ord("|")
        out[cell_off + 2] = 48 + h2
        out[cell_off + 3] = ord(":")
        pos = cell_off + 4
        dig = dig.reshape(m.shape + (dig.shape[1],))
        for w in range(m.shape[2]):
            sel = np.broadcast_to(used[:, :, w], m.shape[:2])
            if not sel.any():
                break
            p, dd, ln = pos[sel], dig[:, :, w][sel], nd[:, :, w][sel]
            for d in range(dd.shape[1]):
                k = ln > d
                out[p[k] + d] = dd[k, d]
            comma = sel & (w + 1 < nw)[:, None]
            out[pos[comma] + nd[:, :, w][comma]] = ord(",")
            pos = np.where(sel, pos + nd[:, :, w] + 1, pos)
        sep = np.full(m.shape[:2], ord("\t"), np.uint8)
        sep[:, -1] = ord("\n")
        out[cell_off + cell_len - 1] = sep
        parts.append(out.tobytes())
    return b"".join(parts)


def masks_of(records, n_samples: int) -> np.ndarray:
    """refbin-style records [(csqs, per_sample[(h1 indices, h2 indices)])] -> masks[n_records, n_samples, W]."""
    w = max([1] + [words_for(len(c)) for c, _ in records])
    out = np.zeros((len(records), n_samples, w), np.uint32)
    for r, (_, cells) in enumerate(records):
        for s, (h1, h2) in enumerate(cells):
            for hap, idx in ((0, h1), (1, h2)):
                for k in idx:
                    out[r, s, k // 15] |= np.uint32(1 << (2 * (k % 15) + hap))
    return out
