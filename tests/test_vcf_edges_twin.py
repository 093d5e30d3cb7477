"""CPU suite: the ground truth of tests/test_gpu_vcf_edges.py.  The large GPU tests trust tests/vcfgen.py instead of
the twin (oracle/vcftext.py), so here every generator is checked against the twin, and the vectorized site-list
restatement against oracle/maskdecode.py, on instances small enough for the twin."""
import os
import re

import numpy as np
import pytest

from oracle import maskdecode
from oracle import vcftext as O
from tests import vcfgen as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def twin_error(text, ix, rows):
    with pytest.raises(O.VcfParseError) as e:
        O.parse_masks(text, ix, rows)
    return e.value.line, e.value.sample, e.value.kind


def same_index(a, b):
    assert sorted(a) == sorted(b)
    for k in a:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k


def test_error_table_matches_the_library_messages():
    """The four phrases of v2p_vcf_parse_masks and the class numbers of csrc/v2p_vcf.cu, as the tests parse them."""
    src = open(os.path.join(ROOT, "vcf2prot_b200", "csrc", "v2p_vcf.cu")).read()
    what = re.findall(r'"([^"]*)"', re.search(r"static const char\* what\[\] = \{(.*?)\};", src, re.S).group(1))
    assert what[0] == "" and len(what) == 5
    enum = dict(re.findall(r"E_([A-Z_]+) = (\d)", re.search(r"enum \{ (E_BAD_CHAR[^}]*)\}", src).group(1)))
    assert {k: int(v) for k, v in enum.items()} == dict(BAD_CHAR=O.BAD_CHAR, EMPTY=O.EMPTY, OVERFLOW=O.OVERFLOW, COUNT=O.COUNT)
    assert {w: k for k, w in enumerate(what) if k} == G.WHAT
    assert '"VCF line %llu, sample column %llu: %s"' in src
    for k, w in enumerate(what[1:], 1):
        assert G.error_triple("VCF line 12, sample column 345: %s" % w) == (12, 345, k)
        assert G.error_triple("VCF line 3, sample column 1: %s (status 11 VCF_PARSE)" % w) == (3, 1, k)
    with pytest.raises(AssertionError):
        G.error_triple("VCF line 3, sample column 1: something else")


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_short_records_text_by_construction(seed):
    """Decorated synth texts: numpy line tables = the twin's index; the matrix of any selection = masks by construction;
    the masks decode (no bit names a csq the record lacks) and have csq 15 in word 0 bits 30/31."""
    rng = np.random.default_rng(seed)
    text, masks, n_csq = G.short_records_text(rng, 400, int(rng.integers(8, 33)), p_junk=0.2)
    ix = O.index(text)
    same_index(G.line_tables(text), ix)
    assert ix["n_lines"] == 400 and ix["line_no"][-1] > 400 + 40
    assert b"\r\n" in text and b"\n\n" in text and b"\n#CHROM\tPOS\tID\tlater" in text
    for rows in (range(400), rng.permutation(400)[:123], [7] * 9, [0], [1]):
        assert np.array_equal(O.parse_masks(text, ix, rows), G.want_rows(masks, n_csq, list(rows)))
    assert ((masks[:, :, 0] >> np.uint32(30)) != 0).any() and masks.shape[2] == 3
    cb = np.concatenate([[0], np.cumsum(n_csq)]).astype(np.uint64)
    cs = rng.integers(-1, 50, int(cb[-1])).astype(np.int32)
    want = maskdecode.site_lists(masks, cb, cs)
    got = G.site_lists(masks, cb, cs)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def test_cell_and_word_offsets():
    rng = np.random.default_rng(4)
    text, masks, n_csq = G.short_records_text(rng, 50, 9)
    t = np.frombuffer(text, np.uint8)
    ix = G.line_tables(t)
    for l in range(50):
        st = G.cell_starts(t, ix, l)
        cells = text[int(ix["cells_begin"][l]):int(ix["line_end"][l])].split(b"\t")
        assert [text[s:s + len(c)] for s, c in zip(st, cells)] == cells
        for s, c in zip(st, cells):
            ws, end = G.word_starts(t, int(s))
            assert text[int(s):end] == c and [text[w:w + 1] for w in ws] == [w[:1] for w in c.split(b":")[-1].split(b",")]


def test_filler_lines_by_construction():
    """Long ':'-fields in front of the mask (digits, commas, '|', '/', '.', 'x'): only the last field counts."""
    rng = np.random.default_rng(5)
    ns = 6
    words = [[rng.integers(0, 1 << 32, int(rng.integers(1, 5)), dtype=np.uint64).tolist() for _ in range(ns)] for _ in range(12)]
    fills = [rng.integers(-1, 3000, ns) for _ in range(12)]
    text = G.header(ns) + b"\n" + b"\n".join(G.filler_line(rng, i, words[i], fills[i]) for i in range(12)) + b"\n"
    ix = O.index(text)
    same_index(G.line_tables(text), ix)
    assert np.array_equal(O.parse_masks(text, ix, range(12)), G.matrix_of(words, ns))
    assert b"x" in text and b"." in text


def test_a1_error_cases_by_construction():
    """The malformed spots of the GPU error-at-scale test, made the same way in a small text: the twin reports the
    (line, sample column, class) the construction says, and the rows left out are clean."""
    rng = np.random.default_rng(6)
    text, masks, n_csq = G.short_records_text(rng, 300, 24)
    t = np.frombuffer(text, np.uint8)
    ix = G.line_tables(t)
    cases = G.a1_error_cases(t, ix, masks)
    assert len(cases) == 6 and {c[3][2] for c in cases} == {O.BAD_CHAR, O.EMPTY, O.OVERFLOW, O.COUNT}
    for name, edits, bad, want in cases:
        u = t.copy()
        for o, b in edits:
            u[o] = b
        bad_text = u.tobytes()
        bix = O.index(bad_text)
        same_index(G.line_tables(u), bix)
        assert twin_error(bad_text, bix, range(300)) == want, name
        clean = np.setdiff1d(np.arange(300), bad)
        assert np.array_equal(O.parse_masks(bad_text, bix, clean), G.want_rows(masks, n_csq, clean)), name


def test_big_header_tables():
    text = b"\r\n".join([b"##x", G.header(5000, b"S%07d"), G.record(1, [b"1"] * 5000), b"", G.record(2, [b"2"] * 5000)])
    ix = O.index(text)
    same_index(G.line_tables(text), ix)
    assert ix["n_samples"] == 5000 and ix["header_end"] - ix["header_begin"] == len(G.header(5000, b"S%07d"))


def test_line_tables_equal_the_twin_on_fuzz_texts():
    rng = np.random.default_rng(7)
    extra = [b"", b"\n", b"\r", b"#CHROM", b"#CHRO\n", b"x\n#CHROM\t1\n", b"\n\r\n#CHROM\r", b"#CHROM\t" + b"\t" * 9 + b"\n\t"]
    n_ok = 0
    for i in range(60 + len(extra)):
        text = G.fuzz_text(rng)[: int(rng.integers(1, 4000))] if i < 60 else extra[i - 60]
        try:
            ix = O.index(text)
        except O.VcfParseError:
            with pytest.raises(O.VcfParseError):
                G.line_tables(text)
            continue
        same_index(G.line_tables(text), ix)
        n_ok += 1
    assert n_ok >= 50


@pytest.mark.parametrize("W", [1, 2, 3])
def test_vectorized_site_lists_equal_maskdecode(W):
    rng = np.random.default_rng(10 + W)
    for _ in range(20):
        n_rec, ns = int(rng.integers(0, 12)), int(rng.integers(1, 7))
        n_csq = rng.integers(15 * (W - 1) + 1, 15 * W + 1, n_rec)
        masks = G.decodable_masks(rng, n_csq, ns, p_zero=0.3) if n_rec else np.zeros((0, ns, W), np.uint32)
        if n_rec and W > 1:  # csq 15 by word 0 bit 30
            masks[:, :, 0] |= np.where(rng.random((n_rec, ns)) < 0.3, np.uint32(1 << 30), np.uint32(0))
        cb = np.concatenate([[0], np.cumsum(n_csq)]).astype(np.uint64)
        cs = rng.integers(-1, 30, int(cb[-1])).astype(np.int32)
        want = maskdecode.site_lists(masks, cb, cs)
        got = G.site_lists(masks, cb, cs)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    masks = np.zeros((2, 1, 1), np.uint32)
    masks[1, 0, 0] = 1 << 6  # csq 3 of a record with 3
    cb, cs = np.array([0, 4, 7], np.uint64), np.arange(7, dtype=np.int32)
    for f in (maskdecode.site_lists, G.site_lists):
        with pytest.raises(IndexError):
            f(masks, cb, cs)
