"""CPU suite: the C-ABI library loads and exports every symbol include/v2p_engine.h declares (no compute)."""
import ctypes as C
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADERS = [os.path.join(ROOT, "include", h) for h in ("v2p_engine.h", "v2p_taskgen.h", "v2p_gzip.h", "v2p_pipeline.h", "v2p_cohort.h")]


@pytest.fixture(scope="module")
def lib():
    from vcf2prot_b200 import _lib

    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__ as g

        g.build()
    return _lib.load()


def header_functions():
    names = set()
    for h in HEADERS:
        src = re.sub(r"/\*.*?\*/", "", open(h).read(), flags=re.S)
        names |= set(re.findall(r"\b(v2p_[a-z0-9_]+)\s*\(", src))
    return sorted(names)


def test_every_declared_symbol_is_exported(lib):
    from vcf2prot_b200 import _lib

    names = header_functions()
    assert len(names) >= 19
    for n in names:
        assert hasattr(lib, n), "libv2p_engine.so does not export %s" % n
        assert n in _lib.SYMBOLS, "ctypes binding lacks %s" % n
    assert lib.v2p_abi_version() == 1


def test_struct_layouts_match_header():
    from vcf2prot_b200 import _lib

    assert C.sizeof(_lib.Task16) == 16
    assert C.sizeof(_lib.Batch) == 13 * 8
    assert C.sizeof(_lib.Result) == 32
    assert C.sizeof(_lib.Generated) == 13 * 8 + 8 + 4 * 8 + 8 + 8 + 8 + 8


def test_engine_from_str_contract(lib):
    """engines.rs:20-29: exactly st|ST|mt|MT|gpu|GPU."""
    from vcf2prot_b200 import Engine, EngineError

    assert Engine.from_str("st") is Engine.ST and Engine.from_str("ST") is Engine.ST
    assert Engine.from_str("mt") is Engine.MT and Engine.from_str("MT") is Engine.MT
    assert Engine.from_str("gpu") is Engine.GPU and Engine.from_str("GPU") is Engine.GPU
    for bad in ("Gpu", "cuda", "", "st ", "mT"):
        with pytest.raises(EngineError):
            Engine.from_str(bad)


def test_library_is_sm100a_and_uses_tma_bulk_store():
    from vcf2prot_b200 import _lib

    out = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    txt = out.stdout.decode()
    assert "sm_100a" in txt
    assert "UBLKCP" in txt  # cp.async.bulk shared->global (TMA bulk copy)


def test_no_cpu_fallback_without_device(lib):
    """Without a CUDA device the product path must fail loudly, never compute on the host."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from vcf2prot_b200 import EngineError, GpuEngine

    with pytest.raises(EngineError):
        GpuEngine(0)


def test_product_never_imports_oracle():
    """The product path may not import, link, dlopen or execute anything under oracle/."""
    pkg = os.path.join(ROOT, "vcf2prot_b200")
    pat = re.compile(r"^\s*(from|import)\s+oracle\b|libv2p_oracle|oracle[/\\](_ref|ref_engine|taskgen|cengine|refbin)", re.M)
    for dp, _, fns in os.walk(pkg):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp", "Makefile")):
                txt = open(os.path.join(dp, fn)).read()
                assert not pat.search(txt), "%s reaches into the oracle" % fn


def _without_bodies(src, names):
    """src with the definitions of the named functions cut out (from the name to the brace that closes the body)."""
    for name in names:
        m = re.search(r"\b%s\([^)]*\)\s*\{" % name, src)
        assert m, "no definition of %s" % name
        depth, i = 1, m.end()
        while depth:
            depth += {"{": 1, "}": -1}.get(src[i], 0)
            i += 1
        src = src[:m.start()] + src[i:]
    return src


def test_host_objects_share_one_buffer_and_error_implementation():
    """Device and pinned memory is allocated and freed only by the owning buffer types of csrc/v2p_hostres.cuh and
    csrc/v2p_mapped.cuh (whose destructors free it, so no destroy function keeps a list of buffers to forget one from)
    and by the public v2p_host_alloc / v2p_host_free.  Error messages are formatted only in csrc/v2p_hostres.cuh."""
    csrc = os.path.join(ROOT, "vcf2prot_b200", "csrc")
    alloc = re.compile(r"\b(cudaMalloc\w*|cudaHostAlloc|cudaFree\w*)\s*\(")
    fmt = re.compile(r"\bvsnprintf\s*\(")
    names = sorted(fn for fn in os.listdir(csrc) if fn.endswith((".cu", ".cuh")))
    assert "v2p_hostres.cuh" in names and "v2p_engine.cu" in names
    for fn in names:
        src = open(os.path.join(csrc, fn)).read()
        if fn == "v2p_engine.cu":
            src = _without_bodies(src, ("v2p_host_alloc", "v2p_host_free"))
        if fn not in ("v2p_hostres.cuh", "v2p_mapped.cuh"):
            m = alloc.search(src)
            assert not m, "%s calls %s: use DevBuf / PinnedBuf (v2p_hostres.cuh) or MappedBuf" % (fn, m.group(1))
        if fn != "v2p_hostres.cuh":
            assert not fmt.search(src), "%s formats its own messages: use v2p::fail / v2p::vformat" % fn


def test_dir_writer_sink_writes_one_file_per_proband(lib, tmp_path):
    """The ready-made sink of include/v2p_pipeline.h is host code (parts/io.rs:35-57 naming): no GPU needed."""
    import numpy as np

    from vcf2prot_b200.pipeline import DirWriter

    names = ["HG%05d" % i for i in range(7)]
    w = DirWriter(str(tmp_path), names, compressed=False, threads=3)
    data = np.frombuffer(b">T_1\nMEDL\n>T_2\nMEDK\n" + b"" + b">U_1\n\n", np.uint8).copy()
    fb = np.array([0, 10, 20, 20, 26], np.uint64)  # third file is empty
    rc = lib.v2p_dir_writer_sink(w._h, 2, 4, data.ctypes.data_as(C.c_void_p), fb.ctypes.data_as(C.POINTER(C.c_uint64)))
    assert rc == 0 and w.files_written == 4 and w.bytes_written == 26
    assert (tmp_path / "HG00002.fasta").read_bytes() == b">T_1\nMEDL\n"
    assert (tmp_path / "HG00003.fasta").read_bytes() == b">T_2\nMEDK\n"
    assert (tmp_path / "HG00004.fasta").read_bytes() == b""
    assert (tmp_path / "HG00005.fasta").read_bytes() == b">U_1\n\n"
    assert not (tmp_path / "HG00000.fasta").exists()
    # a chunk beyond the proband list, and an unwritable directory, stop the run (non-zero)
    assert lib.v2p_dir_writer_sink(w._h, 5, 4, data.ctypes.data_as(C.c_void_p), fb.ctypes.data_as(C.POINTER(C.c_uint64))) != 0
    w.close()
    w2 = DirWriter(str(tmp_path / "missing_dir"), names, compressed=True)
    assert lib.v2p_dir_writer_sink(w2._h, 0, 4, data.ctypes.data_as(C.c_void_p), fb.ctypes.data_as(C.POINTER(C.c_uint64))) != 0
    assert "missing_dir" in w2.last_error() and ".fasta.gz" in w2.last_error()
    w2.close()


def test_copy_kernel_is_built_on_tma_and_has_no_tensor_core_code(lib):
    """The sm_100a build keeps what DESIGN.md section 4 says it has: TMA bulk loads and stores with mbarrier completion
    and cp.async staging in k_copy_tiles, and not one tensor-core instruction anywhere (the path has no flops)."""
    import shutil

    from vcf2prot_b200 import _lib

    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump not on PATH")
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], stdout=subprocess.PIPE, text=True, check=True).stdout
    assert "sm_100a" in subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], stdout=subprocess.PIPE, text=True).stdout
    copy = "".join(b for b in sass.split("Function : ")[1:] if b.startswith("_ZN3v2p12k_copy_tilesILi8192ELi2ELi3ELi3"))
    assert copy, "default copy-kernel instantiation missing"
    for op in ("UBLKCP.G.S", "UBLKCP.S.G", "SYNCS.ARRIVE.TRANS64", "SYNCS.PHASECHK.TRANS64.TRYWAIT", "LDGSTS.E.128", "FENCE.VIEW.ASYNC"):
        assert op in copy, "%s not in k_copy_tiles" % op
    assert not re.search(r"\b(HMMA|IMMA|QMMA|UTCHMMA|UTCQMMA|UTCIMMA)\b", sass)
