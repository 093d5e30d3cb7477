"""CPU suite: the ground truth of tests/test_gpu_vcf_bgzf.py.  The BGZF writer (synth/bgzf.py) against Python's gzip
module and SAM spec section 4.1, the hand DEFLATE streams (tests/deflategen.py) against zlib, the corruption generators
(tests/bgzfgen.py) against the twin (oracle/bgzf.py), and the error phrases against csrc/v2p_vcf.cu."""
import gzip
import os
import re
import struct
import zlib

import pytest

from oracle import bgzf as O
from synth import bgzf as W
from tests import bgzfgen as G
from tests import deflategen as D

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TEXT = G.small_vcf(300, 7)


def check_blocks(data: bytes, eof: bool = True):
    o, n_blocks = 0, 0
    while o < len(data):
        id1, id2, cm, flg, _, _, _, xlen, si1, si2, slen, bsize = struct.unpack_from("<BBBBIBBHBBHH", data, o)
        assert (id1, id2, cm, flg, xlen, si1, si2, slen) == (31, 139, 8, 4, 6, 66, 67, 2)
        assert o + bsize + 1 <= len(data)
        crc, isize = struct.unpack_from("<II", data, o + bsize + 1 - 8)
        d = zlib.decompressobj(-15)
        raw = d.decompress(data[o + 18:o + bsize + 1 - 8])
        assert d.eof and len(raw) == isize <= 65536 and zlib.crc32(raw) & 0xFFFFFFFF == crc
        o += bsize + 1
        n_blocks += 1
    assert o == len(data)
    assert data.endswith(W.EOF_BLOCK) == eof
    return n_blocks


@pytest.mark.parametrize("level,strategy", [(0, "default"), (1, "default"), (6, "default"), (9, "default"), (6, "filtered"),
                                            (6, "huffman_only"), (6, "rle"), (6, "fixed")])
@pytest.mark.parametrize("block_size", [1, 17, 4096, 0xFF00, 65536])
def test_writer_reads_back_through_gzip_and_obeys_the_spec(level, strategy, block_size):
    text = TEXT * (1 if block_size < 4096 else 40)
    data = W.write(text, level, W.STRATEGIES[strategy], block_size, flush_at=(5, 300) if level else ())
    assert gzip.decompress(data) == text and O.inflate(data) == text
    n = check_blocks(data)
    assert n >= -(-len(text) // block_size) + 1


def test_eof_block_bytes_and_optional_eof():
    assert W.EOF_BLOCK.hex() == "1f8b08040000000000ff0600424302001b0003000000000000000000"
    data = W.write(TEXT, eof=False)
    check_blocks(data, eof=False)
    assert O.inflate(data) == TEXT and O.inflate(b"") == b""


def test_flush_points_make_several_deflate_blocks():
    raw = TEXT[:4000]
    plain = W.deflate(raw, 6)
    flushed = W.deflate(raw, 6, flush_at=(1000, 2000, 3000))
    assert b"\x00\x00\xff\xff" in flushed and b"\x00\x00\xff\xff" not in plain  # the empty stored blocks
    assert zlib.decompress(flushed, -15) == raw


@pytest.mark.parametrize("name", sorted(D.CASES))
def test_deflategen_streams_inflate_under_zlib_as_intended(name):
    stream, want = D.CASES[name]
    d = zlib.decompressobj(-15)
    try:
        got = d.decompress(stream)
        ok = d.eof
    except zlib.error:
        ok = False
    if want is None:
        assert not ok
    else:
        assert ok and got == want


def test_deflategen_codes_are_what_their_names_say():
    lit = [0] * 288
    for s, l in {97 + i: i + 1 for i in range(12)}.items():
        lit[s] = l
    assert max(D.canonical(lit)) < 1 << 12
    stream, want = D.CASES["distance_32768_length_258"]
    assert len(want) == 32768 + 258 + 1 + 258 and want[32768:32768 + 258] == want[:258]


@pytest.mark.parametrize("name", sorted(G.corruptions(TEXT)))
def test_twin_reports_each_corruption_as_intended(name):
    data, want = G.corruptions(TEXT)[name]
    with pytest.raises(O.BgzfError) as e:
        O.inflate(data)
    assert (e.value.block, e.value.offset, e.value.cls) == want


def test_edge_blocks_by_construction():
    for name, (data, want) in G.edge_blocks().items():
        if want is None:
            with pytest.raises(O.BgzfError) as e:
                O.inflate(data)
            assert (e.value.block, e.value.cls) == (1, O.DEFLATE), name
        else:
            assert O.inflate(data) == want, name


def test_block_boundaries_at_every_offset_read_back():
    text = G.small_vcf(3, 2)
    for k in range(1, len(text)):
        assert O.inflate(G.split(text, [k])) == text


def test_flips_are_deterministic():
    data = W.write(TEXT, 6, block_size=4096)
    a = [x for _, x in G.flips(data, 7, 20)]
    assert a == [x for _, x in G.flips(data, 7, 20)] and all(x != data for x in a)


def test_error_phrases_match_the_library():
    src = open(os.path.join(ROOT, "vcf2prot_b200", "csrc", "v2p_vcf.cu")).read()
    what = re.findall(r'"([^"]*)"', re.search(r"const char\* const kBgzfWhat\[\] = \{(.*?)\};", src, re.S).group(1))
    assert what[0] == "" and {w: k for k, w in enumerate(what) if k} == G.WHAT
    inf = open(os.path.join(ROOT, "vcf2prot_b200", "csrc", "v2p_inflate.cuh")).read()
    enum = dict(re.findall(r"BGZF_([A-Z]+) = (\d)", inf))
    assert {k: int(v) for k, v in enum.items()} == dict(HEADER=O.HEADER, DEFLATE=O.DEFLATE, SIZE=O.SIZE, CRC=O.CRC)
    assert (G.HEADER, G.DEFLATE, G.SIZE, G.CRC) == (O.HEADER, O.DEFLATE, O.SIZE, O.CRC)
    assert '"BGZF block %llu at byte %llu: %s (%s)"' in src and '"BGZF block %llu at byte %llu: %s"' in src
    assert "not BGZF: recompress with bgzip" in src
    for k, w in enumerate(what[1:], 1):
        assert G.error_triple("BGZF block 12 at byte 345: %s" % w) == (12, 345, k)
        assert G.error_triple("BGZF block 0 at byte 0: %s (why) (status 12 BGZF)" % w) == (0, 0, k)
    with pytest.raises(AssertionError):
        G.error_triple("BGZF block 1 at byte 2: something else")


def test_product_does_not_import_the_test_generators():
    pkg = os.path.join(ROOT, "vcf2prot_b200")
    for dp, _, fns in os.walk(pkg):
        for fn in fns:
            if fn.endswith(".py"):
                assert not re.search(r"^\s*(from|import)\s+(synth|tests)\b", open(os.path.join(dp, fn)).read(), re.M), fn


def test_bgzf_struct_binding_matches_the_header():
    import ctypes as C

    from vcf2prot_b200 import _lib as L

    assert C.sizeof(L.VcfBgzf) == 6 * 8 + 2 * 4 and L.ERR_BGZF == 12 and L.STATUS_NAMES[12] == "BGZF"
    assert [f for f, _ in L.VcfBgzf._fields_] == ["n_blocks", "text_bytes", "text", "head", "fixed", "fixed_begin",
                                                  "inflate_ms", "fixed_ms"]
    hdr = open(os.path.join(ROOT, "include", "v2p_vcf_bgzf.h")).read()
    assert re.search(r"int v2p_vcf_load_bgzf\(v2p_vcf\* v, const uint8_t\* data, uint64_t n_bytes, uint32_t flags, v2p_vcf_lines\* out,"
                     r"\s+v2p_vcf_bgzf\* bz\);", hdr)
    assert "V2P_ERR_BGZF = 12" in open(os.path.join(ROOT, "include", "v2p_engine.h")).read()
