"""CPU suite: the plain-Python twin of the VCF dialect (oracle/vcftext.py), the bench-size text writer
(synth/vcftext.py), and the ctypes binding of include/v2p_vcf.h."""
import os
import re

import numpy as np
import pytest

from oracle import maskdecode, refbin
from oracle import vcftext as O
from synth import vcftext as S
from tests.helpers import cohort_haplotype_csqs, load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT"


def rec(pos, cells, fmt=b"GT:BCSQ", info=b"BCSQ=missense|G|T1|protein_coding|+|1A>1C|x"):
    return b"1\t%d\t.\tC\tT\t.\t.\t%s\t%s\t%s" % (pos, info, fmt, b"\t".join(cells))


@pytest.mark.parametrize("name", ["cohort_a.json", "cohort_b.json", "cohort_c.json"])
def test_twin_decodes_the_golden_texts_back_to_the_selections(name):
    """refbin.vcf_text wrote the texts the reference binary ran on: twin parse + maskdecode gives every haplotype's csqs."""
    co = load_golden(name)
    text = refbin.vcf_text(co["samples"], co["records"]).encode()
    ix = O.index(text)
    assert ix["n_samples"] == len(co["samples"]) and ix["n_lines"] == len(co["records"])
    hdr = text[ix["header_begin"]:ix["header_end"]].split(b"\t")[9:]
    assert [h.decode() for h in hdr] == co["samples"]
    kept = [l for l in range(ix["n_lines"]) if O.supported(O.bcsq(text, ix, l))]
    masks = O.parse_masks(text, ix, kept)
    csqs = [O.bcsq(text, ix, l) for l in kept]
    pool = sorted({c for cs in csqs for c in cs})
    site_of = {c: i for i, c in enumerate(pool)}
    cb = np.cumsum([0] + [len(c) for c in csqs]).astype(np.uint64)
    cs = np.array([site_of[c] for cc in csqs for c in cc], np.int32)
    sb, sites = maskdecode.site_lists(masks, cb, cs)
    want = cohort_haplotype_csqs(co)
    for s, smp in enumerate(co["samples"]):
        for hap in (1, 2):
            h = 2 * s + hap - 1
            got = [pool[i] for i in sites[int(sb[h]):int(sb[h + 1])]]
            assert got == sorted(set(want.get((smp, hap), []))), (smp, hap)


@pytest.mark.parametrize("name", ["cohort_a.json", "cohort_b.json", "cohort_c.json"])
def test_synth_writer_is_byte_identical_to_refbin(name):
    co = load_golden(name)
    want = refbin.vcf_text(co["samples"], co["records"]).encode()
    got = S.vcf_text(co["samples"], [c for c, _ in co["records"]], S.masks_of(co["records"], len(co["samples"])), block=37)
    assert got == want


def test_synth_writer_multi_word_cells_of_mixed_widths():
    rng = np.random.default_rng(3)
    records = []
    for r in range(30):
        n = int(rng.choice([1, 2, 15, 16, 31, 44]))
        csqs = ["missense|G|T%d|protein_coding|+|%dA>%dC|x" % (r, k, k) for k in range(n)]
        cells = [(sorted(rng.choice(n, int(rng.integers(0, min(n, 5) + 1)), replace=False).tolist()),
                  sorted(rng.choice(n, int(rng.integers(0, min(n, 3) + 1)), replace=False).tolist())) for _ in range(9)]
        records.append((csqs, cells))
    samples = ["S%d" % i for i in range(9)]
    want = refbin.vcf_text(samples, records).encode()
    assert S.vcf_text(samples, [c for c, _ in records], S.masks_of(records, 9), block=4) == want
    ix = O.index(want)
    m = O.parse_masks(want, ix, range(ix["n_lines"]))
    assert m.shape[2] == 3 and np.array_equal(m, S.masks_of(records, 9))


def test_dialect_line_ends_meta_lines_and_fields():
    text = (b"##fileformat=VCFv4.2\r\n##x=1\n\n" + HDR + b"\tA\tB\r\n" + rec(1, [b"0|1:5", b"7"]) + b"\r\n\r\n#comment\n" +
            rec(2, [b"1/1:3:12,4", b"0"], fmt=b"GT:AD:BCSQ") + b"\n" + rec(3, [b"1", b"2"]))  # last line without newline
    ix = O.index(text)
    assert ix["n_samples"] == 2 and ix["n_lines"] == 3 and ix["line_no"] == [5, 8, 9]
    assert text[ix["header_begin"]:ix["header_end"]] == HDR + b"\tA\tB"
    m = O.parse_masks(text, ix, [2, 0, 1])
    assert m.shape == (3, 2, 2)
    assert m[:, :, 0].tolist() == [[1, 2], [5, 7], [12, 0]] and m[2, 0, 1] == 4 and m[:2, :, 1].sum() == 0
    assert O.parse_masks(text, ix, []).shape == (0, 2, 1)
    assert text[int(ix["line_begin"][1]):int(ix["cells_begin"][1])].endswith(b"GT:AD:BCSQ\t")


@pytest.mark.parametrize("cell,kind", [(b"0|1:", O.EMPTY), (b"1,,2", O.EMPTY), (b"0|1:.", O.BAD_CHAR), (b"-1", O.BAD_CHAR),
                                       (b"+1", O.BAD_CHAR), (b" 1", O.BAD_CHAR), (b"4294967296", O.OVERFLOW),
                                       (b"1,99999999999", O.OVERFLOW)])
def test_dialect_errors_name_line_and_sample(cell, kind):
    text = HDR + b"\tA\tB\tC\n" + rec(1, [b"1", b"2", b"3"]) + b"\n" + rec(2, [b"1", b"2", cell]) + b"\n"
    ix = O.index(text)
    with pytest.raises(O.VcfParseError) as e:
        O.parse_masks(text, ix, [0, 1])
    assert (e.value.line, e.value.sample, e.value.kind) == (3, 3, kind)
    assert O.parse_masks(text, ix, [0]).shape == (1, 3, 1)  # a malformed line that is not selected is never read
    assert O.parse_masks(HDR + b"\tA\n" + rec(1, [b"4294967295"]), O.index(HDR + b"\tA\n" + rec(1, [b"4294967295"])), [0])[0, 0, 0] == 0xFFFFFFFF


def test_dialect_cell_counts_and_the_first_error_in_file_order():
    text = HDR + b"\tA\tB\n" + rec(1, [b"1"]) + b"\n" + rec(2, [b"x", b"1", b"2"]) + b"\n" + rec(3, [b"1", b"."]) + b"\n"
    ix = O.index(text)
    for rows, want in (([0], (2, 2, O.COUNT)), ([1], (3, 1, O.BAD_CHAR)), ([2, 1], (3, 1, O.BAD_CHAR)), ([2], (4, 2, O.BAD_CHAR))):
        with pytest.raises(O.VcfParseError) as e:
            O.parse_masks(text, ix, rows)
        assert (e.value.line, e.value.sample, e.value.kind) == want, rows
    with pytest.raises(O.VcfParseError):  # no #CHROM line
        O.index(b"##fileformat=VCFv4.2\n" + rec(1, [b"1"]))


def test_binding_covers_the_vcf_header():
    from vcf2prot_b200 import _lib

    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "v2p_vcf.h")).read(), flags=re.S)
    names = set(re.findall(r"\b(v2p_[a-z0-9_]+)\s*\(", src))
    assert len(names) == 5 and all(n in _lib.SYMBOLS for n in names)
    assert _lib.ERR_VCF_PARSE == 11 and _lib.STATUS_NAMES[11] == "VCF_PARSE"
    if os.path.isfile(_lib.LIB_PATH):
        lib = _lib.load()
        assert all(hasattr(lib, n) for n in names)
