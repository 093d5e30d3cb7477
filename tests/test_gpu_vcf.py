"""GPU suite: VCF text -> FORMAT/BCSQ mask matrix on the device (include/v2p_vcf.h) against the plain-Python twin of
the dialect (oracle/vcftext.py), and chained into the pipeline / cohort runner up to the reference binary's records."""
import numpy as np
import pytest

from oracle import refbin
from oracle import taskgen as T
from oracle import vcftext as O
from synth import vcftext as S
from tests.helpers import assert_sample_matches_reference, load_golden
from vcf2prot_b200 import _lib as L
from vcf2prot_b200.engine import EngineError
from vcf2prot_b200.vcf import DeviceVcf

pytestmark = pytest.mark.gpu

HDR = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT"


@pytest.fixture(scope="module")
def vcf():
    v = DeviceVcf(0)
    yield v
    v.close()


def rec(pos, cells, fmt=b"GT:BCSQ", info=b"BCSQ=missense|G|T1|protein_coding|+|1A>1C|x"):
    return b"1\t%d\t.\tC\tT\t.\t.\t%s\t%s\t%s" % (pos, info, fmt, b"\t".join(cells))


def header(n):
    return HDR + b"".join(b"\tS%d" % i for i in range(n))


def random_cell(rng):
    words = [str(int(x)) for x in rng.choice([0, 1, 2, 3, 1 << 20, 0xFFFFFFFF], size=int(rng.choice([1, 1, 1, 2, 3])))]
    body = ",".join(words).encode()
    return rng.choice([b"", b"0|1:", b"1/0:7,3:", b"0|0:"]) + body


def random_text(seed, n_samples, n_records, crlf=False):
    rng = np.random.default_rng(seed)
    nl = b"\r\n" if crlf else b"\n"
    lines = [b"##fileformat=VCFv4.2", header(n_samples)]
    for r in range(n_records):
        lines.append(rec(r, [random_cell(rng) for _ in range(n_samples)], fmt=rng.choice([b"GT:BCSQ", b"BCSQ", b"GT:AD:BCSQ"])))
    return nl.join(lines) + nl


def load(vcf, text, device):
    if not device:
        return vcf.load(text), None
    import torch

    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    return vcf.load((t.data_ptr(), len(text))), t


def check(vcf, text, rows=None, device=False):
    ix = O.index(text)
    got, keep = load(vcf, text, device)
    assert (got.n_samples, got.header_begin, got.header_end, got.n_lines) == (ix["n_samples"], ix["header_begin"], ix["header_end"], ix["n_lines"])
    assert np.array_equal(got.line_begin, ix["line_begin"]) and np.array_equal(got.cells_begin, ix["cells_begin"])
    assert got.h2d_bytes == (0 if device else len(text))
    rows = list(range(ix["n_lines"])) if rows is None else rows
    m = vcf.parse_masks(rows)
    want = O.parse_masks(text, ix, rows)
    assert m.shape == want.shape
    assert np.array_equal(m.read(), want)
    del keep
    return got, m


CASES = {
    "crlf_and_last_line_without_newline": lambda: random_text(1, 5, 40, crlf=True)[:-2],
    "meta_and_empty_lines": lambda: b"##a=1\n\n##b=2\r\n" + header(3) + b"\n\n" + rec(1, [b"1", b"2", b"3"]) + b"\n\r\n#x\n" +
                                    rec(2, [b"0|1:4", b"5", b"0:6"]) + b"\n\n",
    "extra_format_fields_and_no_colon": lambda: header(2) + b"\n" + rec(1, [b"0|1:3,4:9", b"8"], fmt=b"GT:AD:BCSQ") + b"\n",
    "multi_word_mixed_widths": lambda: header(4) + b"\n" + rec(1, [b"1", b"2,3", b"0|1:4,5,6,7", b"0"]) + b"\n" + rec(2, [b"1"] * 4),
    "one_sample": lambda: random_text(2, 1, 100),
    "zero_records": lambda: b"##fileformat=VCFv4.2\n" + header(7) + b"\n",
    "header_only_no_newline": lambda: header(3),
    "many_lines": lambda: random_text(3, 61, 700),
    "long_lines": lambda: random_text(4, 110_000, 3),  # > 600 KB a line: cells straddle every segment boundary
}


@pytest.mark.parametrize("device", [False, True])
@pytest.mark.parametrize("case", sorted(CASES))
def test_tables_and_matrices_equal_the_twin(vcf, case, device):
    text = CASES[case]()
    got, m = check(vcf, text, device=device)
    if case == "long_lines":
        assert min(np.diff(got.line_begin)) > 600_000
    if case == "zero_records":
        assert m.shape == (0, 7, 1)
    if case == "multi_word_mixed_widths":
        assert m.shape == (2, 4, 4)


@pytest.mark.parametrize("device", [False, True])
def test_subset_and_permuted_rows(vcf, device):
    text = random_text(5, 33, 200)
    rng = np.random.default_rng(5)
    for rows in (rng.permutation(200)[:57].tolist(), [199, 0, 199, 3], [17]):
        check(vcf, text, rows, device=device)


def test_sample_names(vcf):
    ix = vcf.load(header(3) + b"\r\n" + rec(1, [b"1", b"2", b"3"]))
    assert ix.sample_names() == ["S0", "S1", "S2"]


def test_every_error_class_names_line_and_sample(vcf):
    base = [b"##fileformat=VCFv4.2", header(3), rec(1, [b"1", b"2", b"3"])]
    for cell, what in ((b"0|1:", "empty"), (b"1,,2", "empty"), (b".", "character"), (b"0|1:-1", "character"), (b"+1", "character"),
                       (b" 1", "character"), (b"4294967296", "above"), (b"1,99999999999", "above")):
        text = b"\n".join(base + [rec(2, [b"1", cell, b"3"])]) + b"\n"
        vcf.load(text)
        with pytest.raises(EngineError) as e:
            vcf.parse_masks([0, 1])
        assert e.value.status == L.ERR_VCF_PARSE and "line 4, sample column 2" in str(e.value) and what in str(e.value), cell
        assert vcf.parse_masks([0]).read().tolist() == [[[1], [2], [3]]]  # usable afterwards; unselected line never read
    for cells, col in (([b"1", b"2"], 3), ([b"1", b"2", b"3", b"4"], 4), ([], 1)):
        text = b"\n".join(base + [rec(2, cells) if cells else b"1\t2\t.\tC\tT\t.\t.\tX"]) + b"\n"
        vcf.load(text)
        with pytest.raises(EngineError) as e:
            vcf.parse_masks([1])
        assert e.value.status == L.ERR_VCF_PARSE and "line 4, sample column %d" % col in str(e.value) and "number" in str(e.value)
    with pytest.raises(EngineError) as e:
        vcf.load(b"##fileformat=VCFv4.2\n" + rec(1, [b"1"]) + b"\n")
    assert e.value.status == L.ERR_VCF_PARSE and "#CHROM" in str(e.value)
    with pytest.raises(EngineError) as e:  # nothing loaded after the failed load
        vcf.parse_masks([0])
    assert e.value.status == L.ERR_INVALID_ARG
    vcf.load(b"\n".join(base) + b"\n")
    with pytest.raises(EngineError) as e:
        vcf.parse_masks([1])
    assert e.value.status == L.ERR_INVALID_ARG


def test_first_error_in_file_order_wins(vcf):
    """Errors in lines far apart and in one long line: the lowest (line, sample column) is reported every time."""
    n = 20_000
    good = [b"1"] * n
    late = list(good)
    late[n - 5] = b"x"
    early = list(good)
    early[n - 700] = b"7,"
    early[n - 1] = b"."
    lines = [header(n)] + [rec(i, good) for i in range(30)] + [rec(30, late), rec(31, early), rec(32, good[:-1])]
    text = b"\n".join(lines) + b"\n"
    vcf.load(text)
    for rows, want in (([32, 31, 30], "line 32, sample column %d" % (n - 4)), ([31, 32], "line 33, sample column %d" % (n - 699)),
                       ([32, 0], "line 34, sample column %d" % n)):
        for _ in range(3):
            with pytest.raises(EngineError) as e:
                vcf.parse_masks(rows)
            assert want in str(e.value), (rows, str(e.value))
            with pytest.raises(O.VcfParseError):
                O.parse_masks(text, O.index(text), rows)


def golden_world(text, ix, refs):
    """The host's per-record step: BCSQ lists of the supported records -> general catalogue (csq -> site or -1)."""
    from tests.test_gpu_taskgen_general import World
    from tests.test_taskgen_rules import static_instruction

    tix = dict(line_begin=ix.line_begin, cells_begin=ix.cells_begin)
    kept = [l for l in range(ix.n_lines) if O.supported(O.bcsq(text, tix, l))]
    csqs = [O.bcsq(text, tix, l) for l in kept]
    good = set()
    for c in {c for cs in csqs for c in cs}:
        try:
            if T.Mutation.from_csq(c).transcript_name in refs:
                static_instruction(T.Mutation.from_csq(c))
                good.add(c)
        except T.TaskGenError:  # dropped by AltTranscript::new (vcf_ds.rs:366-373)
            pass
    w = World(refs, [sorted(good)])
    csq_begin = np.cumsum([0] + [len(c) for c in csqs]).astype(np.uint64)
    csq_site = np.array([w.site_of.get(c, -1) for cs in csqs for c in cs], np.int32)
    return w, kept, csq_begin, csq_site


@pytest.mark.parametrize("name", ["cohort_a.json", "cohort_b.json", "cohort_c.json"])
def test_golden_cohorts_from_vcf_text_to_the_reference_binarys_records(gpu_engine, vcf, name):
    from vcf2prot_b200.pipeline import DevicePipeline
    from vcf2prot_b200.taskgen import DeviceCatalogue

    co = load_golden(name)
    text = refbin.vcf_text(co["samples"], co["records"]).encode()
    ix = vcf.load(text)
    assert ix.sample_names() == co["samples"]
    w, kept, cb, cs = golden_world(text, ix, co["refs"])
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


@pytest.mark.parametrize("n_workers", [2, 3])
def test_cohort_runner_takes_the_device_matrix(vcf, n_workers):
    from synth import cohort as C
    from tests.test_gpu_cohort_run import devices, runner
    from tests.test_gpu_pipeline import RICH_MIX, cohort_sites

    prot = C.make_proteome(seed=81, n_tx=300, mu=5.3, sigma=0.7, lo=30, hi=3000)
    cat = C.make_catalogue(prot, 6000, seed=82, mix=RICH_MIX, fs_mean=30, fs_max=600, sl_max=120)
    cat.af[:] = np.random.default_rng(9).choice([0.01, 0.05, 0.2, 0.5], size=cat.n)
    n_samples = 31
    rec_ = C.make_records(cat, 6, 3, 0.2, 4)
    assert rec_.words > 1
    hap, site = cohort_sites(cat, n_samples, 90 + n_workers)
    masks = C.encode_masks(rec_, n_samples, hap, site)
    csqs = [["c%d" % k for k in range(int(rec_.csq_begin[r + 1] - rec_.csq_begin[r]))] for r in range(rec_.n_rec)]
    text = S.vcf_text(["P%d" % i for i in range(n_samples)], csqs, masks)
    ix = vcf.load(text)
    m = vcf.parse_masks(np.arange(ix.n_lines))
    assert np.array_equal(m.read(), masks)
    out, h2d = {}, {}
    for key in ("host", "device"):
        got = out.setdefault(key, {})

        def sink(first, n, data, begins):
            for i in range(n):
                got[first + i] = bytes(data[int(begins[i]):int(begins[i + 1])])
            return 0

        r = runner(prot, cat, devices(n_workers))
        try:
            if key == "host":
                res = r.run_masks(masks, rec_.csq_begin, rec_.csq_site, chunk_samples=4, sink=sink)
            else:
                res = r.run_masks(m.ptr, rec_.csq_begin, rec_.csq_site, chunk_samples=4, sink=sink, shape=m.shape)
        finally:
            r.close()
        assert int(res.total.n_sites) == len(site)
        h2d[key] = int(res.total.h2d_bytes)
    assert sorted(out["device"]) == list(range(n_samples)) and out["device"] == out["host"]
    assert h2d["device"] == h2d["host"] - masks.nbytes  # the matrix is not uploaded
