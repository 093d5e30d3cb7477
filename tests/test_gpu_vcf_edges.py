"""GPU suite: the device VCF reader (csrc/v2p_vcf.cu) where a text parser goes wrong.

  A  the kernels' scheduling loops at sizes where they loop: k_find_cells past its grid, k_parse with several segments
     per warp and records changing inside a warp's run, k_header_tabs over several passes, errors at scale;
     ground truth by construction (tests/vcfgen.py), because the twin is too slow for tens of MB
  B  every byte boundary of the cell parse: the 9th tab and cells at every offset of a 16-byte chunk and around 512-byte
     segments, values and leading zeros at every alignment, every byte value, field syntax, error order, seeded fuzz;
     ground truth: the plain-Python twin (oracle/vcftext.py)
  C  state left between calls on one object: stale text after n_bytes, reused matrix buffers, n_samples = 0
  D  the A-size matrix, still on the device, into v2p_sites_from_masks
Every error is compared whole: (file line, sample column, class)."""
import numpy as np
import pytest

from oracle import vcftext as O
from synth import vcftext as S
from tests import vcfgen as G
from tests.vcfgen import header, record
from vcf2prot_b200 import _lib as L
from vcf2prot_b200.engine import EngineError
from vcf2prot_b200.vcf import DeviceVcf

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vcf():
    v = DeviceVcf(0)
    yield v
    v.close()


@pytest.fixture(scope="module")
def sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def to_device(text):
    import torch

    return torch.from_numpy(np.frombuffer(text, np.uint8).copy()).cuda()


def outcome(vcf, rows):
    """The matrix of parse_masks(rows), or the (line, sample column, class) of its V2P_ERR_VCF_PARSE."""
    try:
        m = vcf.parse_masks(rows)
    except EngineError as e:
        assert e.status == L.ERR_VCF_PARSE, str(e)
        return G.error_triple(str(e))
    return m.read()


def twin_outcome(text, ix, rows):
    try:
        return O.parse_masks(text, ix, rows)
    except O.VcfParseError as e:
        return e.line, e.sample, e.kind


def same(got, want, what=""):
    if isinstance(want, tuple):
        assert isinstance(got, tuple) and got == want, (got if isinstance(got, tuple) else "a matrix", want, what)
    else:
        assert isinstance(got, np.ndarray), (got, what)
        assert got.shape == want.shape and np.array_equal(got, want), what


def same_tables(got, ix):
    assert (got.n_samples, got.header_begin, got.header_end, got.n_lines) == (
        ix["n_samples"], ix["header_begin"], ix["header_end"], ix["n_lines"])
    assert np.array_equal(got.line_begin, ix["line_begin"]) and np.array_equal(got.cells_begin, ix["cells_begin"])


def against_twin(vcf, text, row_sets=(), single_rows=True, device=False):
    """Load `text`, compare the line table and the outcome of every row alone, of all rows and of `row_sets` with the
    twin.  -> the twin's index."""
    ix = O.index(text)
    keep = to_device(text) if device else None
    got = vcf.load((keep.data_ptr(), len(text)) if device else text)
    same_tables(got, ix)
    n = ix["n_lines"]
    sets = [list(range(n))] + [list(r) for r in row_sets] + ([[l] for l in range(n)] if single_rows else [])
    for rows in sets:
        same(outcome(vcf, rows), twin_outcome(text, ix, rows), rows[:8])
    del keep
    return ix


def segments(ix, rows=None):
    """Parse segments of the selected lines: 512 bytes each from cells_begin's 16-byte block, at least one."""
    a0 = ix["cells_begin"].astype(np.int64) & ~15
    n = np.maximum((ix["line_end"].astype(np.int64) - a0 + 511) // 512, 1)
    return n if rows is None else n[np.asarray(rows)]


# ====================================================================================================== A: scale
@pytest.fixture(scope="module")
def a1(sms):
    """Many short records (24 samples, W = 1-3) among meta / comment / empty / CRLF lines."""
    n = 3 * sms * 32 * 8 + 1237
    text, masks, n_csq = G.short_records_text(np.random.default_rng(101), n, 24)
    t = np.frombuffer(text, np.uint8)
    return dict(text=text, t=t, masks=masks, n_csq=n_csq, ix=G.line_tables(t))


def test_a1_many_short_records(vcf, sms, a1):
    ix, masks, n_csq = a1["ix"], a1["masks"], a1["n_csq"]
    n = ix["n_lines"]
    assert n == len(masks) >= 3 * sms * 32 * 8  # k_find_cells: 8 warps a block, at most sms*32 blocks -> 3 strides
    assert n >= 3 * 64 * sms  # k_parse: >= 1 segment a record, at most 64 warps an SM -> >= 3 segments a warp
    assert ix["line_no"][-1] > n + 1000 and ix["n_samples"] == 24
    same_tables(vcf.load(a1["text"]), ix)
    rng = np.random.default_rng(11)
    for rows in (np.arange(n), rng.permutation(n)[: 2 * n // 3], np.full(3000, n // 2 + 7)):
        m = vcf.parse_masks(rows)
        want = G.want_rows(masks, n_csq, rows)
        assert m.shape == want.shape and np.array_equal(m.read(), want)


def test_a1_device_text(vcf, a1):
    t = to_device(a1["text"])
    got = vcf.load((t.data_ptr(), len(a1["text"])))
    same_tables(got, a1["ix"])
    rows = np.arange(a1["ix"]["n_lines"])[::-1]
    assert np.array_equal(vcf.parse_masks(rows).read(), G.want_rows(a1["masks"], a1["n_csq"], rows))


def test_a2_long_lines(vcf, sms):
    """At most 40 lines, >= 3 segments a warp: every warp's run lies inside one or two long records."""
    need, n_rec = 3 * 64 * sms, 40
    rng = np.random.default_rng(102)
    n_samples = need * 512 // n_rec // 9
    n_csq = rng.integers(1, 46, n_rec)
    masks = G.decodable_masks(rng, n_csq, n_samples)
    text = G.decorate(S.vcf_text(["P%d" % i for i in range(n_samples)], [[""] * int(c) for c in n_csq], masks), rng, 0.3, 0.5)
    ix = G.line_tables(text)
    assert ix["n_lines"] == n_rec and segments(ix).sum() >= need and len(text) < 40e6
    same_tables(vcf.load(text), ix)
    for rows in (np.arange(n_rec), [39, 0, 17, 17, 5]):
        assert np.array_equal(vcf.parse_masks(rows).read(), G.want_rows(masks, n_csq, rows))


@pytest.fixture(scope="module")
def a3(sms):
    """16 samples: short synth records, then 30 long records whose cells carry 0-30 KB ':'-fields in front of the mask."""
    rng = np.random.default_rng(103)
    n_short, n_long, ns = 3 * 64 * sms, 30, 16
    text, masks, n_csq = G.short_records_text(rng, n_short, ns, max_csq=30)
    long_words = [[rng.integers(0, 1 << 32, int(rng.integers(1, 4)), dtype=np.uint64).tolist() for _ in range(ns)]
                  for _ in range(n_long)]
    fills = [np.where(rng.random(ns) < 0.5, rng.integers(0, 30000, ns), rng.integers(900, 1500, ns)) for _ in range(n_long)]
    longs = [G.filler_line(rng, 10 ** 6 + i, long_words[i], fills[i]) for i in range(n_long)]
    text += b"\n".join(longs) + b"\n"
    want = np.zeros((n_short + n_long, ns, 3), np.uint32)
    want[:n_short, :, :masks.shape[2]] = masks
    want[n_short:] = G.matrix_of(long_words, ns)
    t = np.frombuffer(text, np.uint8)
    return dict(text=text, t=t, want=want, ix=G.line_tables(t), n_short=n_short, n_long=n_long)


def test_a3_long_and_short_records_share_warp_runs(vcf, sms, a3):
    ix, want, n_short = a3["ix"], a3["want"], a3["n_short"]
    same_tables(vcf.load(a3["text"]), ix)
    longs = np.arange(n_short, n_short + a3["n_long"])
    groups = np.array_split(np.arange(n_short), a3["n_long"])
    rows = np.concatenate([np.concatenate([[lg], g]) for lg, g in zip(longs, groups)])
    rng = np.random.default_rng(13)
    for sel in (rows, rng.permutation(rows), np.concatenate([longs[:3], np.arange(40), longs[3:6], np.arange(40)])):
        if sel is rows:
            assert segments(ix, sel).sum() >= 3 * 64 * sms
        m = vcf.parse_masks(sel)
        assert m.shape[2] == 3 and np.array_equal(m.read(), want[sel])


def test_a4_the_widest_cell_anywhere_in_a_warps_run(vcf, sms):
    """One line whose only wide cell has 40 words, among >= 3*64*sms one-segment lines (so every warp gets a run of at
    least two segments): at selection positions p and p+1, one of which is inside a run, W must be 40."""
    rng = np.random.default_rng(104)
    n, ns = 3 * 64 * sms + 17, 8
    n_csq = rng.integers(1, 16, n)
    masks = G.decodable_masks(rng, n_csq, ns)
    wide = [int(x) for x in rng.integers(0, 10, 40)]
    line_a = np.zeros((ns, 40), np.uint32)
    line_a[:, 0] = rng.integers(0, 10, ns)
    line_a[5] = wide
    cells = [G.words_cell(w) if s == 5 else b"%d" % w[0] for s, w in enumerate(line_a)]
    text = S.vcf_text(["P%d" % i for i in range(ns)], [[""] * int(c) for c in n_csq], masks) + record(7, cells) + b"\n"
    ix = G.line_tables(text)
    assert ix["n_lines"] == n + 1 and (segments(ix) == 1).all() and n + 1 >= 3 * 64 * sms
    same_tables(vcf.load(text), ix)
    for p in (n // 2 + 3, n // 2 + 4):
        rows = np.insert(np.arange(n), p, n)
        m = vcf.parse_masks(rows)
        assert m.shape == (n + 1, ns, 40), p
        got = m.read()
        assert np.array_equal(got[p], line_a), p
        assert np.array_equal(np.delete(got, p, axis=0)[:, :, :1], masks) and not np.delete(got, p, axis=0)[:, :, 1:].any(), p


def test_a5_errors_at_scale(vcf, a1, a3):
    """Each malformed spot known by construction; every case 3 times (the first error must not depend on timing), then a
    clean selection of the same text."""
    t, ix, masks, n_csq = a1["t"], a1["ix"], a1["masks"], a1["n_csq"]
    n = ix["n_lines"]
    cases = G.a1_error_cases(t, ix, masks)
    dev = to_device(a1["text"])
    rng = np.random.default_rng(15)
    for name, edits, bad, want in cases:
        for o, b in edits:
            dev[o] = b
        vcf.load((dev.data_ptr(), len(t)))
        for _ in range(3):
            same(outcome(vcf, np.arange(n)), want, name)
        clean = np.setdiff1d(rng.permutation(n)[: n // 2], bad)
        assert np.array_equal(vcf.parse_masks(clean).read(), G.want_rows(masks, n_csq, clean)), name
        same(outcome(vcf, np.arange(n)), want, name)  # the clean parse left nothing behind
        for o, _ in edits:
            dev[o] = int(t[o])
    # one malformed cell that starts in one segment and ends two segments later (a long ':'-field in front)
    t, ix = a3["t"], a3["ix"]
    found = None
    for r in range(a3["n_short"], a3["n_short"] + a3["n_long"]):
        a0 = int(ix["cells_begin"][r]) & ~15
        st = G.cell_starts(t, ix, r)
        for s in range(len(st)):
            end = G.word_starts(t, int(st[s]))[1]
            if (end - 1 - a0) // 512 - (int(st[s]) - a0) // 512 == 2:
                found = r, s, end - 1
                break
        if found:
            break
    assert found
    r, s, o = found
    dev = to_device(a3["text"])
    dev[o] = ord(".")
    vcf.load((dev.data_ptr(), len(t)))
    rows = np.concatenate([np.arange(0, a3["n_short"], 7), [r], np.arange(a3["n_short"], len(a3["want"]))])
    for _ in range(3):
        same(outcome(vcf, rows), (int(ix["line_no"][r]), s + 1, O.BAD_CHAR))
    clean = rows[rows != r]
    assert np.array_equal(vcf.parse_masks(clean).read(), a3["want"][clean])


@pytest.mark.parametrize("n_rec", [0, 2])
def test_a6_big_header(vcf, sms, n_rec):
    """A #CHROM line longer than three passes of k_header_tabs (sms blocks of 256 threads, 16 bytes a thread)."""
    n_samples = 3 * sms * 256 * 16 // 9 + 1001
    rng = np.random.default_rng(106)
    vals = rng.integers(0, 10, (n_rec, n_samples))
    lines = [b"##fileformat=VCFv4.2", header(n_samples, b"S%07d")] + [record(i, [b"%d" % v for v in vals[i]]) for i in range(n_rec)]
    text = b"\r\n".join(lines)
    ix = G.line_tables(text)
    assert ix["header_end"] - ix["header_begin"] >= 3 * sms * 256 * 16 and ix["n_samples"] == n_samples
    got = vcf.load(text)
    same_tables(got, ix)
    m = vcf.parse_masks(np.arange(n_rec))
    assert m.shape == (n_rec, n_samples, 1) and np.array_equal(m.read()[:, :, 0], vals)


# ================================================================================================ B: byte boundaries
def zcell(n, v):
    """A one-word cell of exactly n bytes with value v (leading zeros)."""
    return b"%0*d" % (n, v)


def test_b1_ninth_tab_and_cells_at_every_alignment(vcf):
    """The ID column padded by 0-15 bytes moves the 9th tab over every offset of a 16-byte chunk; cell lengths put tabs on
    the last and the first byte of a 512-byte segment (counted from cells_begin & ~15), line ends on a segment boundary,
    and cells over 2 and 3 segments."""
    seen = dict(tab9=set(), tab_last=0, tab_first=0, end_on_seg=0, span3=0)
    for pad in range(16):
        buf = header(3) + b"\n"
        lines = []
        for shape in ("short", "tab_last", "tab_first", "end_1seg", "end_2seg", "span2", "span3", "second_spans3", "crlf"):
            start = len(buf)
            pre = record(pad, [], id_pad=pad)
            cb = start + len(pre)
            a0 = cb & ~15
            lens = {"short": [1, 2, 3], "tab_last": [a0 + 511 - cb, 3, 4], "tab_first": [a0 + 512 - cb, 3, 4],
                    "end_1seg": [5, 6, a0 + 512 - cb - 13], "end_2seg": [300, 400, a0 + 1024 - cb - 702],
                    "span2": [700, 2, 3], "span3": [1100, 1, 1], "second_spans3": [40, 1100, 9], "crlf": [a0 + 512 - cb - 1, 1, 2]}[shape]
            line = pre + b"\t".join(zcell(k, (i + pad) % 9 + 1) for i, k in enumerate(lens))
            end = start + len(line)
            tabs = [cb + sum(lens[:i + 1]) + i for i in range(2)]
            seen["tab9"].add((cb - 1) % 16)
            seen["tab_last"] += any((x - a0) % 512 == 511 for x in tabs)
            seen["tab_first"] += any((x - a0) % 512 == 0 for x in tabs)
            seen["end_on_seg"] += (end - a0) % 512 == 0
            seen["span3"] += any((cb + sum(lens[:i]) + i + k - 1 - a0) // 512 - (cb + sum(lens[:i]) + i - a0) // 512 == 2
                                 for i, k in enumerate(lens))
            nl = b"\r\n" if shape == "crlf" else b"\n"
            lines.append(line)
            buf += line + nl
        against_twin(vcf, buf, row_sets=[[8, 0, 3], [1, 1]], device=pad % 2 == 1)
        # the 9th tab on the line's last byte: one sample, an empty cell (cells_begin == line_end)
        one = b"\n".join([header(1), record(0, [], id_pad=pad), record(1, [b"5"], id_pad=pad), record(2, [], id_pad=pad) + b"\r"])
        ix = against_twin(vcf, one)
        assert ix["cells_begin"][0] == ix["line_end"][0] and twin_outcome(one, ix, [0]) == (2, 1, O.EMPTY)
    assert seen["tab9"] == set(range(16)) and all(seen[k] for k in ("tab_last", "tab_first", "end_on_seg", "span3"))


VALID = ([b"9" * k for k in range(1, 10)] + [b"1" + b"0" * (k - 1) for k in range(1, 11)] +
         [b"4294967295", b"0000000000004294967295", b"0", b"00", b"3735928559", b"2147483648"] +
         [b"0" * (k - 1) + b"5" for k in range(11, 26)] + [b"0" * (k - 10) + b"4294967295" for k in range(11, 26)])
OVER = ([b"4294967296", b"9999999999", b"10000000000", b"42949672950", b"18446744073709551616", b"18446744073709551621",
         b"18446744073709551615", b"36893488147419103232", b"9" * 30, b"4294967296" + b"0" * 15] +
        [b"0" * (k - 10) + b"4294967296" for k in range(11, 26)] + [b"0" * (k - 11) + b"42949672950" for k in range(11, 26)])


def test_b2_values_at_every_alignment(vcf):
    for pad in range(16):
        lines = [header(3)]
        for i, w in enumerate(VALID + OVER):
            lines += [record(i, [b"1", w, b"2"], id_pad=pad), record(i, [b"0|1:" + w, b"1," + w + b",2", w], id_pad=pad)]
        text = b"\n".join(lines) + b"\n"
        ix = against_twin(vcf, text, row_sets=[range(0, 2 * len(VALID))])
        if pad == 0:
            m = O.parse_masks(text, ix, range(2 * len(VALID)))
            assert m[::2, 1, 0].tolist() == [int(w) for w in VALID]
            for l in range(2 * len(VALID), ix["n_lines"]):
                assert twin_outcome(text, ix, [l])[2] == O.OVERFLOW


def test_b3_every_byte_value_in_a_word(vcf):
    """Each byte 0-255 but '\\n' at the start, middle and end of a word, in a middle and in the last column."""
    for pad in (0, 9):
        lines = [header(3)]
        for b in range(256):
            if b == 10:
                continue
            c = bytes([b])
            for cell in (c + b"12", b"1" + c + b"2", b"12" + c):
                lines += [record(b, [b"1", cell, b"2"], id_pad=pad), record(b, [b"1", b"2", cell], id_pad=pad)]
        lines += [record(1, [b"1", b"2", b"3\r\r"], id_pad=pad), record(2, [b"1", b"2\r", b"3\r"], id_pad=pad)]
        text = b"\n".join(lines) + b"\n"
        ix = against_twin(vcf, text)
        k = 6 * (0xB0 - 1)  # data lines of byte 0xB0 ('0' | 0x80), which is not a digit
        assert all(twin_outcome(text, ix, [l])[2] == O.BAD_CHAR for l in range(k, k + 6))
        assert twin_outcome(text, ix, [ix["n_lines"] - 2]) == (len(lines) - 1, 3, O.BAD_CHAR)  # "\r\r": one '\r' ends it


def test_b4_field_syntax(vcf):
    cells = [b":5", b"5:", b"::5", b"x:5", b"5,", b",5", b",", b":", b"0|1:x:7,8", b"1/0:.:9", b"1,2:3,4,5", b"a:b:c:"]
    lines = [header(3)]
    for i, c in enumerate(cells):
        lines += [record(i, [c, b"1", b"2"]), record(i, [b"1", b"2", c])]
    lines += [record(90, [b"1,2:3,4,5", b"1,2,3,4,5,6", b"7"]), record(91, [b"9,9,9,9,9,9,9:1", b"1", b"2"])]
    for k in range(1, 65):  # cells of 1-64 words
        lines.append(record(100 + k, [b",".join(b"%d" % (j * 7 + k) for j in range(k)), b"3", b",".join([b"1"] * (65 - k))]))
    text = b"\n".join(lines) + b"\n"
    ok = list(range(2 * len(cells), len(lines) - 1))
    ix = against_twin(vcf, text, row_sets=[ok])
    m = O.parse_masks(text, ix, ok)
    assert m.shape[2] == 64 and m[0, 0, :4].tolist() == [3, 4, 5, 0] and m[1, 0, :2].tolist() == [1, 0]
    kinds = {c: twin_outcome(text, ix, [2 * i]) for i, c in enumerate(cells)}
    assert not isinstance(kinds[b"x:5"], tuple) and kinds[b"5:"][2] == O.EMPTY and kinds[b",5"][2] == O.EMPTY


def test_b5_error_order_inside_a_cell_and_across_cells(vcf):
    lines = [header(3)]
    for c in (b"x,,1", b",x", b"99999999999,x", b"x,99999999999", b",99999999999", b"1,x,", b"0|1:,:x"):
        lines += [record(1, [b"1", c, b"2"])]
    lines += [record(2, [b"1", b"2", b"3", b"x"]), record(3, [b"1", b"2", b"3", b""]), record(4, [b"1", b"2", b"3", b"4"]),
              record(5, [b"x", b"2"]), record(6, [b"1", b"2", b"3", b"4", b"y"]), record(7, [b"1", b""])]
    text = b"\n".join(lines) + b"\n"
    ix = against_twin(vcf, text, row_sets=[[8, 7], [9, 8], [12, 11, 10]])
    got = [twin_outcome(text, ix, [l]) for l in range(ix["n_lines"])]
    assert [g[2] for g in got[:3]] == [O.BAD_CHAR, O.EMPTY, O.OVERFLOW]
    assert got[7] == (9, 4, O.BAD_CHAR) and got[8] == (10, 4, O.EMPTY) and got[9] == (11, 4, O.COUNT)  # the tie at ns + 1



def test_b6_seeded_fuzz(vcf):
    rng = np.random.default_rng(106)
    kinds = {"ok": 0, "error": 0, "no_chrom": 0}
    for i in range(300):
        text = G.fuzz_text(rng)
        try:
            ix = O.index(text)
        except O.VcfParseError:
            with pytest.raises(EngineError) as e:
                vcf.load(text)
            assert e.value.status == L.ERR_VCF_PARSE and "#CHROM" in str(e.value), i
            kinds["no_chrom"] += 1
            continue
        keep = to_device(text) if i % 3 == 0 else None
        same_tables(vcf.load((keep.data_ptr(), len(text)) if keep is not None else text), ix)
        n = ix["n_lines"]
        for rows in (list(range(n)), rng.integers(0, max(n, 1), int(rng.integers(0, n + 2))).tolist() if n else []):
            want = twin_outcome(text, ix, rows)
            same(outcome(vcf, rows), want, (i, rows[:8]))
            if len(rows) == n:
                kinds["error" if isinstance(want, tuple) else "ok"] += 1
    assert kinds["ok"] >= 30 and kinds["error"] >= 100, kinds


# ============================================================================================= C: state between calls
def test_c_stale_upload_buffer_after_n_bytes(vcf):
    """A large upload leaves digits and tabs in the buffer after a small text's last byte."""
    big = header(2) + b"\n" + b"123456789\t" * 200_000 + b"\n"
    for pad in range(10):
        vcf.load(big)
        for tail in (b"", b"\t", b"\r", b"0", b",", b"\t12"):
            small = header(2) + b"\n" + record(1, [b"1", b"2"], id_pad=pad) + b"\n" + record(2, [b"3", b"45"], id_pad=pad) + tail
            against_twin(vcf, small)


def test_c_borrowed_device_text_inside_a_larger_buffer(vcf):
    import torch

    texts = [header(2) + b"\n" + record(1, [b"1", b"2,3"]) + b"\n" + record(2, [b"4", b"5"]),
             header(3) + b"\r\n" + record(1, [b"7", b"8", b"9\r"]) + b"\r\n" + record(2, [b"1", b"2", b""]),
             header(1) + b"\n" + record(1, [b"0|1:6"]) + b"\n" + record(2, [], id_pad=5)]
    junk = np.frombuffer((b"98\t7\n65\t" * 1024), np.uint8)
    for text in texts:
        ix = O.index(text)
        for off in (0, 16, 48, 4096 + 16):
            buf = torch.from_numpy(np.concatenate([junk[:off], np.frombuffer(text, np.uint8), junk])).cuda()
            got = vcf.load((buf.data_ptr() + off, len(text)))
            same_tables(got, ix)
            for rows in (list(range(ix["n_lines"])), [ix["n_lines"] - 1], [0]):
                same(outcome(vcf, rows), twin_outcome(text, ix, rows), (off, rows))
            del buf


def test_c_wide_narrow_wide_on_one_object(vcf):
    """The second wide matrix reuses the first one's buffer: its zero padding has to be written by the kernel."""
    text = b"\n".join([header(3), record(1, [b"11,12,13,14,15", b"21,22,23,24,25", b"31,32,33,34,35"]), record(2, [b"7", b"8", b"9"]),
                       record(3, [b"1,2,3,4,5", b"6", b"0|1:4,5"]), record(4, [b"1,1,1,1,1", b"2,2", b"3,3,3,3"])]) + b"\n"
    ix = O.index(text)
    vcf.load(text)
    first = vcf.parse_masks([0, 0, 0])
    ptr = first.ptr
    same(first.read(), O.parse_masks(text, ix, [0, 0, 0]))
    same(outcome(vcf, [1]), O.parse_masks(text, ix, [1]))
    last = vcf.parse_masks([2, 3, 2])
    assert last.ptr == ptr and last.shape == (3, 3, 5)
    same(last.read(), O.parse_masks(text, ix, [2, 3, 2]))


def test_c_no_samples_and_empty_selections(vcf):
    text = b"\n".join([header(0), b"1\t2\t.\tC\tT\t.\t.\tX", b"1\t2\t.\tC\tT\t.\t.\tX\tGT", b"1\t2\t.\tC\tT\t.\t.\tX\tGT\t", b"1\t3\t.\tC\tT\t.\t.\tX\tGT\t5"]) + b"\n"
    ix = against_twin(vcf, text, row_sets=[[0, 1, 1, 0], []])
    assert ix["n_samples"] == 0 and vcf.parse_masks([0, 1]).shape == (2, 0, 1) and vcf.parse_masks([]).shape == (0, 0, 1)
    assert twin_outcome(text, ix, [3]) == (5, 1, O.COUNT) and twin_outcome(text, ix, [2]) == (4, 1, O.EMPTY)
    vcf.load(header(4) + b"\n" + record(1, [b"1"] * 4) + b"\n")
    assert vcf.parse_masks([]).shape == (0, 4, 1)


# ====================================================================================== D: chained into the decode
def test_d_sites_from_the_device_matrix_at_scale(vcf, sms, a1):
    from synth import cohort as C
    from vcf2prot_b200.taskgen import DeviceCatalogue

    masks, n_csq = a1["masks"], a1["n_csq"]
    n = len(masks)
    assert masks.size >= 3 * sms * 16 * 1024 and masks.shape[2] >= 2  # k_md_count / k_md_emit loop: sms*16 blocks of 1024
    top = (masks[:, :, 0] >> np.uint32(30)) != 0
    assert top.any() and (masks[:, :, 1][top] & 3).any()  # csq 15 named by word 0, and in some cells by word 1 as well
    vcf.load(a1["text"])
    m = vcf.parse_masks(np.arange(n))
    assert m.shape == masks.shape
    prot = C.make_proteome(seed=41, n_tx=300, mu=5.3, sigma=0.7, lo=30, hi=3000)
    cat = C.make_catalogue(prot, 6000, seed=42, mix=(0.55, 0.10, 0.10, 0.08, 0.07, 0.05, 0.05), fs_mean=30, fs_max=600, sl_max=120)
    rng = np.random.default_rng(107)
    cb = np.concatenate([[0], np.cumsum(n_csq)]).astype(np.uint64)
    cs = rng.integers(0, cat.n, int(cb[-1])).astype(np.int32)
    cs[rng.random(len(cs)) < 0.1] = -1
    want_sb, want_sites = G.site_lists(masks, cb, cs)
    dc = DeviceCatalogue(prot, cat, 0)
    try:
        lst = dc.sites_from_masks(m.ptr, cb, cs, shape=m.shape)
        sb = dc.read(lst.site_begin, lst.n_hap + 1, np.uint64)
        sites = dc.read(lst.sites, lst.n_sites, np.uint32)
    finally:
        dc.close()
    assert np.array_equal(sb, want_sb) and np.array_equal(sites, want_sites)
