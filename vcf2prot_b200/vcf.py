"""ctypes harness for the device VCF reader (include/v2p_vcf.h, csrc/v2p_vcf.cu): VCF text in, the FORMAT/BCSQ mask
matrix out, on the device -- the per-cell text parse and transpose the reference does on the host (readers.rs,
text_parser.rs:163-194, vcf_ds.rs:126-213).  The host keeps columns 1-9 (INFO/BCSQ) and chooses the records."""
from __future__ import annotations

import ctypes as C
from typing import List, Sequence, Tuple, Union

import numpy as np

from . import _lib as L
from .engine import EngineError


class VcfIndex:
    """What v2p_vcf_load found: n_samples, the #CHROM line's byte range, and per data line (file order) the offsets of
    its first byte (line_begin) and of its first sample cell (cells_begin; the line end if it has fewer columns)."""

    def __init__(self, res: L.VcfLines, header: bytes):
        n = int(res.n_lines)
        as_np = lambda p: np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint64)), shape=(n,)).copy() if n else np.zeros(0, np.uint64)
        self.n_samples, self.n_lines = int(res.n_samples), n
        self.header_begin, self.header_end = int(res.header_begin), int(res.header_end)
        self.line_begin, self.cells_begin = as_np(res.line_begin), as_np(res.cells_begin)
        self.h2d_bytes, self.h2d_ms, self.index_ms = int(res.h2d_bytes), float(res.h2d_ms), float(res.index_ms)
        self._header = header

    def sample_names(self) -> List[str]:
        """Columns after FORMAT on the #CHROM line."""
        return [c.decode() for c in self._header.split(b"\t")[9:]] if self.n_samples else []


class BgzfVcfIndex(VcfIndex):
    """What v2p_vcf_load_bgzf found: the VcfIndex of the inflated text (offsets are into that text), plus what the host
    needs without a text of its own: `head` (every line up to and including #CHROM) and columns 1-9 of every data line
    (`fixed_text`, sliced by `fixed_begin`).  The text itself stays on the device at `text_ptr` until the next load."""

    def __init__(self, res: L.VcfLines, bz: L.VcfBgzf, owner: "DeviceVcf"):
        self.head = C.string_at(bz.head, int(res.header_end)) if res.header_end else b""
        super().__init__(res, self.head[int(res.header_begin):])
        n = int(res.n_lines)
        self.fixed_begin = np.ctypeslib.as_array(C.cast(bz.fixed_begin, C.POINTER(C.c_uint64)), shape=(n + 1,)).copy()
        n_fixed = int(self.fixed_begin[-1])
        self.fixed_text = np.frombuffer(C.string_at(bz.fixed, n_fixed), np.uint8).copy() if n_fixed else np.zeros(0, np.uint8)
        self.text_ptr, self.text_bytes, self.n_blocks = int(bz.text or 0), int(bz.text_bytes), int(bz.n_blocks)
        self.inflate_ms, self.fixed_ms = float(bz.inflate_ms), float(bz.fixed_ms)
        self._owner = owner

    def fixed(self, l: int) -> bytes:
        """Columns 1-9 of data line l, with the tab after FORMAT when the line has sample cells."""
        return self.fixed_text[int(self.fixed_begin[l]):int(self.fixed_begin[l + 1])].tobytes()

    def read_text(self) -> bytes:
        """Device -> host copy of the inflated text (tests, debugging); valid until the owner's next load."""
        out = np.zeros(self.text_bytes, np.uint8)
        if out.size and self._owner._lib.v2p_device_read(out.ctypes.data_as(C.c_void_p), C.c_void_p(self.text_ptr), out.nbytes):
            raise EngineError(L.ERR_CUDA, "v2p_device_read failed")
        return out.tobytes()


class DeviceMasks:
    """masks[n_records][n_samples][words_per_cell] (uint32) on the device, owned by the DeviceVcf until its next call.
    `ptr` / `shape` go straight to DevicePipeline.run_masks(ptr, ..., shape=shape) and CohortRunner.run_masks."""

    def __init__(self, res: L.VcfMasks, owner: "DeviceVcf"):
        self.ptr = int(res.masks or 0)
        self.shape = (int(res.n_records), int(res.n_samples), int(res.words_per_cell))
        self.parse_ms = float(res.parse_ms)
        self._owner = owner

    def read(self) -> np.ndarray:
        """Device -> host copy of the matrix (tests, debugging)."""
        out = np.zeros(self.shape, np.uint32)
        if out.size:
            st = self._owner._lib.v2p_device_read(out.ctypes.data_as(C.c_void_p), C.c_void_p(self.ptr), out.nbytes)
            if st:
                raise EngineError(st, "v2p_device_read failed")
        return out


class DeviceVcf:
    def __init__(self, device: int = 0):
        self._lib = L.load()
        h = C.c_void_p()
        st = self._lib.v2p_vcf_create(device, C.byref(h))
        if st:
            raise EngineError(st, "v2p_vcf_create(%d) failed (no such device? there is no CPU fallback)" % device)
        self._h = h
        self._text = None

    def close(self):
        if getattr(self, "_h", None):
            self._lib.v2p_vcf_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _err(self) -> str:
        return (self._lib.v2p_vcf_last_error(self._h) or b"").decode()

    def load(self, text: Union[bytes, np.ndarray, Tuple[int, int]]) -> VcfIndex:
        """bytes or a uint8 array (host; pinned memory uploads at the full PCIe rate), or (device_ptr, n_bytes): device
        memory on this object's device, 16-byte aligned, kept alive by the caller until the next load / close."""
        res = L.VcfLines()
        if isinstance(text, tuple):
            ptr, n = int(text[0]), int(text[1])
            st = self._lib.v2p_vcf_load(self._h, C.c_void_p(ptr), n, L.FLAG_DEVICE_PTRS, C.byref(res))
            self._text = None
        else:
            buf = np.frombuffer(text, np.uint8) if isinstance(text, (bytes, bytearray, memoryview)) else np.ascontiguousarray(text, np.uint8)
            st = self._lib.v2p_vcf_load(self._h, buf.ctypes.data_as(C.c_void_p), buf.nbytes, 0, C.byref(res))
            self._text = buf
        if st:
            raise EngineError(st, self._err())
        hb, he = int(res.header_begin), int(res.header_end)
        if self._text is not None:
            header = self._text[hb:he].tobytes()
        else:
            hdr = np.zeros(he - hb, np.uint8)
            if he > hb and self._lib.v2p_device_read(hdr.ctypes.data_as(C.c_void_p), C.c_void_p(int(text[0]) + hb), he - hb):
                raise EngineError(L.ERR_CUDA, "reading the #CHROM line back failed")
            header = hdr.tobytes()
        return VcfIndex(res, header)

    def load_bgzf(self, data: Union[bytes, np.ndarray]) -> BgzfVcfIndex:
        """A bgzip'd VCF (bytes or a uint8 array in host memory; pinned memory uploads at the full PCIe rate), inflated
        and indexed on the device.  parse_masks then works as after load()."""
        buf = np.frombuffer(data, np.uint8) if isinstance(data, (bytes, bytearray, memoryview)) else np.ascontiguousarray(data, np.uint8)
        res, bz = L.VcfLines(), L.VcfBgzf()
        st = self._lib.v2p_vcf_load_bgzf(self._h, buf.ctypes.data_as(C.c_void_p), buf.nbytes, 0, C.byref(res), C.byref(bz))
        self._text = None
        if st:
            raise EngineError(st, self._err())
        return BgzfVcfIndex(res, bz, self)

    def parse_masks(self, rec_line: Sequence[int]) -> DeviceMasks:
        """Row r of the matrix = data line rec_line[r] of the last load (any order)."""
        rl = np.ascontiguousarray(rec_line, np.uint64)
        res = L.VcfMasks()
        st = self._lib.v2p_vcf_parse_masks(self._h, len(rl), rl.ctypes.data_as(C.c_void_p), 0, C.byref(res))
        if st:
            raise EngineError(st, self._err())
        return DeviceMasks(res, self)
