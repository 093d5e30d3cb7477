"""GPU suite: bgzip'd VCF in, inflated and indexed on the device (v2p_vcf_load_bgzf, include/v2p_vcf.h), against the
plain-text load of the same object, the BGZF twin (oracle/bgzf.py, zlib inside) and the VCF twin (oracle/vcftext.py).
Every error is compared as a whole (block, offset, class) triple read from the library's message."""
import ctypes as C
import gzip

import numpy as np
import pytest

from oracle import bgzf as OB
from oracle import refbin
from oracle import vcftext as O
from synth import bgzf as W
from tests import bgzfgen as G
from tests import deflategen as D
from tests.helpers import assert_sample_matches_reference, load_golden
from tests.test_gpu_vcf import golden_world, random_text
from vcf2prot_b200 import _lib as L
from vcf2prot_b200.engine import EngineError
from vcf2prot_b200.vcf import DeviceVcf

pytestmark = pytest.mark.gpu

TEXT = random_text(11, 33, 700)  # ~4 blocks of 0xff00


@pytest.fixture(scope="module")
def vcf():
    v = DeviceVcf(0)
    yield v
    v.close()


def same_lines(a, b):
    assert (a.n_samples, a.header_begin, a.header_end, a.n_lines) == (b.n_samples, b.header_begin, b.header_end, b.n_lines)
    assert np.array_equal(a.line_begin, b.line_begin) and np.array_equal(a.cells_begin, b.cells_begin)


def check(vcf, text, data, twin=True):
    """load_bgzf(data) == text: the text, the index (== plain load, == twin), head, fixed, the matrix (== plain)."""
    got = vcf.load_bgzf(data)
    assert got.text_bytes == len(text) and got.read_text() == text
    assert got.h2d_bytes == len(data) and got.n_blocks >= 1 and got.inflate_ms > 0
    assert got.head == text[:got.header_end]
    fixed = b"".join(text[int(b):int(c)] for b, c in zip(got.line_begin, got.cells_begin))
    assert got.fixed_text.tobytes() == fixed and int(got.fixed_begin[-1]) == len(fixed)
    assert np.array_equal(np.diff(got.fixed_begin.astype(np.int64)), (got.cells_begin - got.line_begin).astype(np.int64))
    if got.n_lines:
        assert got.fixed(got.n_lines - 1) == text[int(got.line_begin[-1]):int(got.cells_begin[-1])]
    if twin:
        ix = O.index(text)
        assert (got.n_samples, got.header_begin, got.header_end, got.n_lines) == (ix["n_samples"], ix["header_begin"], ix["header_end"], ix["n_lines"])
        assert np.array_equal(got.line_begin, ix["line_begin"]) and np.array_equal(got.cells_begin, ix["cells_begin"])
    rows = np.arange(got.n_lines)
    m = vcf.parse_masks(rows).read()
    plain = vcf.load(text)
    same_lines(got, plain)
    assert np.array_equal(vcf.parse_masks(rows).read(), m)
    return got


def bgzf_error(vcf, data):
    with pytest.raises(EngineError) as e:
        vcf.load_bgzf(data)
    assert e.value.status == L.ERR_BGZF, str(e.value)
    return G.error_triple(str(e.value))


def twin_result(data):
    try:
        return OB.inflate(data), None
    except OB.BgzfError as e:
        return None, (e.block, e.offset, e.cls)


ROUND_TRIP = {"L%d_%s" % (lv, st): dict(level=lv, strategy=W.STRATEGIES[st])
              for lv, st in [(0, "default"), (1, "default"), (6, "default"), (9, "default"), (6, "filtered"),
                             (6, "huffman_only"), (6, "rle"), (6, "fixed"), (1, "huffman_only"), (9, "rle")]}
ROUND_TRIP.update({"block_%d" % b: dict(block_size=b) for b in (1, 17, 4096, 0xFF00, 65536)})
ROUND_TRIP.update({"L0_block_65536": dict(level=0, block_size=65536), "flush": dict(flush_at=(1, 777, 30000)),
                   "flush_no_eof": dict(flush_at=(100, 20000), eof=False), "no_eof": dict(eof=False),
                   "L1_flush_4096": dict(level=1, block_size=4096, flush_at=(3, 2000))})


@pytest.mark.parametrize("case", sorted(ROUND_TRIP))
def test_round_trip(vcf, case):
    kw = ROUND_TRIP[case]
    text = TEXT if kw.get("block_size", 4096) >= 4096 else random_text(12, 5, 60, crlf=True)
    data = W.write(text, **kw)
    assert OB.inflate(data) == text
    check(vcf, text, data)


def test_block_boundary_at_every_byte_offset(vcf):
    """A '\\r' | '\\n' split, a split #CHROM line, a cell cut inside a word: every cut of a small file."""
    text = G.small_vcf(3, 2)
    assert b"\r\n#CHROM" in text
    plain = vcf.load(text)
    m = vcf.parse_masks(np.arange(plain.n_lines)).read()
    for k in range(1, len(text)):
        got = vcf.load_bgzf(G.split(text, [k]))
        assert got.n_blocks == 3 and got.read_text() == text, k
        same_lines(got, plain)
        assert got.head == text[:got.header_end]
        assert got.fixed_text.tobytes() == b"".join(text[int(b):int(c)] for b, c in zip(plain.line_begin, plain.cells_begin))
        assert np.array_equal(vcf.parse_masks(np.arange(plain.n_lines)).read(), m), k


@pytest.mark.parametrize("name", sorted(D.CASES))
def test_deflategen_streams(vcf, name):
    data, want = G.edge_blocks()[name]
    if want is None:
        assert bgzf_error(vcf, data) == twin_result(data)[1] and twin_result(data)[1][0] == 1
    else:
        assert vcf.load_bgzf(data).read_text() == want == OB.inflate(data)
        if b"junk" not in D.CASES[name][0]:  # Python's gzip reads the trailer right after the DEFLATE end
            assert gzip.decompress(data) == want


def test_scale_strides_over_the_resident_warps(vcf):
    """At least 3x the most warps the B200 can hold (64 per SM) in blocks, so that k_inflate loops on every warp."""
    import torch

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    need = 3 * 64 * sms
    text = G.small_vcf(int(need * 64 / 500) + 50, 61, seed=3)
    ms = W.members(text, 6, block_size=64)
    data, n_blocks = b"".join(ms) + W.EOF_BLOCK, len(ms) + 1
    assert n_blocks >= need, (n_blocks, need)
    got = check(vcf, text, data, twin=False)
    assert got.n_blocks == n_blocks


@pytest.mark.parametrize("name", sorted(G.corruptions(G.small_vcf(300, 7))))
def test_each_error_class_against_the_twin(vcf, name):
    text = G.small_vcf(300, 7)
    data, want = G.corruptions(text)[name]
    assert twin_result(data)[1] == want
    assert bgzf_error(vcf, data) == want
    if name.startswith("plain"):
        with pytest.raises(EngineError) as e:
            vcf.load_bgzf(data)
        assert "not BGZF: recompress with bgzip" in str(e.value)
    # the object stays usable
    check(vcf, text, W.write(text, 6, block_size=4096), twin=False)
    assert vcf.load(text).n_lines == 300


def test_seeded_flips_equal_the_twin(vcf):
    text = G.small_vcf(120, 9, seed=5)
    data = W.write(text, 6, block_size=2048, flush_at=(700,))
    n_err = 0
    for i, bad in G.flips(data, 2024, 300):
        want_text, want_err = twin_result(bad)
        if want_err is not None:
            assert bgzf_error(vcf, bad) == want_err, i
            n_err += 1
        else:
            assert vcf.load_bgzf(bad).read_text() == want_text, i
    assert n_err > 200
    check(vcf, text, data)


def test_state_flags_and_symbols(vcf):
    lib = L.load()
    assert "v2p_vcf_load_bgzf" in L.SYMBOLS and hasattr(lib, "v2p_vcf_load_bgzf") and L.ERR_BGZF == 12
    data = np.frombuffer(W.write(TEXT), np.uint8)
    for flags in (L.FLAG_DEVICE_PTRS, 1, 8):
        res, bz = L.VcfLines(), L.VcfBgzf()
        assert lib.v2p_vcf_load_bgzf(vcf._h, data.ctypes.data_as(C.c_void_p), data.nbytes, flags, C.byref(res), C.byref(bz)) == L.ERR_INVALID_ARG
        with pytest.raises(EngineError) as e:  # nothing loaded after the refused call
            vcf.parse_masks([0])
        assert e.value.status == L.ERR_INVALID_ARG
    with pytest.raises(EngineError) as e:  # inflates, but the text has no #CHROM line
        vcf.load_bgzf(W.write(b"##x\n1\t2\n"))
    assert e.value.status == L.ERR_VCF_PARSE
    empty = vcf.load_bgzf(W.write(b"#CHROM\n", eof=True))
    assert empty.n_lines == 0 and empty.head == b"#CHROM" and empty.fixed_begin.tolist() == [0]
    check(vcf, TEXT, W.write(TEXT))


@pytest.mark.parametrize("name", ["cohort_a.json", "cohort_b.json", "cohort_c.json"])
def test_golden_cohorts_from_vcf_gz_to_the_reference_binarys_records(gpu_engine, vcf, name):
    """load_bgzf -> the host's BCSQ step on `fixed` (no host text) -> parse_masks -> pipeline -> the reference's records."""
    from vcf2prot_b200.pipeline import DevicePipeline
    from vcf2prot_b200.taskgen import DeviceCatalogue

    co = load_golden(name)
    text = refbin.vcf_text(co["samples"], co["records"]).encode()
    ix = vcf.load_bgzf(W.write(text, 6, block_size=997))
    assert ix.sample_names() == co["samples"]

    class FixedView:  # the index golden_world reads, over the fixed columns instead of the text
        n_lines = ix.n_lines
        line_begin, cells_begin = ix.fixed_begin[:-1], ix.fixed_begin[1:]

    w, kept, cb, cs = golden_world(ix.fixed_text.tobytes(), FixedView, co["refs"])
    m = vcf.parse_masks(kept)
    name_off = np.cumsum([0] + [len(n) for n in w.names]).astype(np.uint64)
    cats = []
    for _ in range(2):
        dc = DeviceCatalogue.from_instructions(*w.cat_args)
        dc.set_names(name_off, np.frombuffer("".join(w.names).encode(), np.uint8))
        cats.append(dc)
    gpu_engine.set_reference(w.tape)
    pipe = DevicePipeline(gpu_engine, cats=cats)
    files = {}

    def sink(first, n, data, begins):
        for i in range(n):
            files[first + i] = bytes(data[int(begins[i]):int(begins[i + 1])])
        return 0

    _, res = pipe.run_masks(m.ptr, cb, cs, shape=m.shape, chunk_samples=16, sink=sink)
    pipe.close()
    assert sorted(files) == list(range(len(co["samples"])))
    for s, smp in enumerate(co["samples"]):
        assert_sample_matches_reference(co, smp, refbin.parse_fasta_records(files[s].decode()))
    assert res.n_records > 0
