"""ctypes harness for the single-process multi-GPU cohort runner (include/v2p_cohort.h, csrc/v2p_cohort.cu): one host
thread + engine + pipeline per device, contiguous sample ranges, no launcher -- parts/exec.rs:34-40 on GPUs."""
from __future__ import annotations

import ctypes as C
from typing import Callable, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from .engine import EngineError
from .pipeline import DevicePipeline


class CohortRunner:
    def __init__(self, devices: Sequence[int], proteome: np.ndarray, tx_offsets: np.ndarray, names: Tuple[np.ndarray, np.ndarray],
                 site_tx, site_pos, site_cls, site_rlen, site_doff, site_dlen, pool, lanes: int = 2):
        """Seven-class catalogue arrays as for v2p_catalogue_create (DeviceCatalogue takes the same ones)."""
        self._lib = L.load()
        a = lambda x, dt: np.ascontiguousarray(x, dt)
        self._keep = dict(prot=a(proteome, np.uint8), off=a(tx_offsets, np.uint64), noff=a(names[0], np.uint64), npool=a(names[1], np.uint8),
                          tx=a(site_tx, np.uint32), pos=a(site_pos, np.uint32), cls=a(site_cls, np.uint8), rlen=a(site_rlen, np.uint32),
                          doff=a(site_doff, np.uint64), dlen=a(site_dlen, np.uint32), pool=a(pool, np.uint8))
        k = self._keep
        p = lambda x: x.ctypes.data_as(C.c_void_p)
        inp = L.CohortInputs()
        inp.proteome, inp.n_proteome, inp.n_tx, inp.tx_offsets = p(k["prot"]), len(k["prot"]), len(k["off"]) - 1, p(k["off"])
        inp.name_off, inp.names, inp.general, inp.n_sites = p(k["noff"]), p(k["npool"]), 0, len(k["tx"])
        inp.site_tx, inp.site_pos, inp.site_cls, inp.site_rlen = p(k["tx"]), p(k["pos"]), p(k["cls"]), p(k["rlen"])
        inp.site_doff, inp.site_dlen, inp.pool, inp.n_pool = p(k["doff"]), p(k["dlen"]), p(k["pool"]), len(k["pool"])
        self._inputs = inp
        devs = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        st = self._lib.v2p_cohort_create(devs, len(devices), C.byref(inp), lanes, C.byref(h))
        if st:
            raise EngineError(st, "v2p_cohort_create failed (a device is missing? there is no CPU fallback)")
        self._h = h
        self.n_devices = len(devices)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.v2p_cohort_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def launch_count(self) -> int:
        return int(self._lib.v2p_cohort_launch_count(self._h))

    def enable_all_records(self) -> None:
        """The reference's `-a` (write_all) on every device; afterwards run_lists(..., all_records=True)."""
        st = self._lib.v2p_cohort_enable_all_records(self._h, C.byref(self._inputs))
        if st:
            raise EngineError(st, (self._lib.v2p_cohort_last_error(self._h) or b"").decode())

    def run_lists(self, site_begin: np.ndarray, sites: np.ndarray, n_samples: int, chunk_samples: int = 128, gzip: bool = False,
                  sink: Optional[Callable] = None, concurrent_sink: bool = False, all_records: bool = False) -> L.CohortResult:
        """sink(first_sample, n, data, file_begin) per chunk (cohort-wide sample numbers), or a DirWriter."""
        sb, st_ = np.ascontiguousarray(site_begin, np.uint64), np.ascontiguousarray(sites, np.uint32)
        cb, user, keep = DevicePipeline._sink(sink)
        res = L.CohortResult()
        flags = (L.PIPE_GZIP if gzip else 0) | (L.COHORT_CONCURRENT_SINK if concurrent_sink else 0) | (L.PIPE_ALL_RECORDS if all_records else 0)
        st = self._lib.v2p_cohort_run_lists(self._h, n_samples, sb.ctypes.data_as(C.c_void_p), st_.ctypes.data_as(C.c_void_p),
                                            chunk_samples, flags, cb, user, C.byref(res))
        del keep
        if st:
            raise EngineError(st, (self._lib.v2p_cohort_last_error(self._h) or b"").decode())
        return res

    def run_masks(self, masks, csq_begin: np.ndarray, csq_site: np.ndarray, chunk_samples: int = 128, gzip: bool = False,
                  sink: Optional[Callable] = None, concurrent_sink: bool = False, all_records: bool = False, shape=None) -> L.CohortResult:
        """masks[n_records, n_samples, W] (FORMAT/BCSQ integers): decoded once on the first device, then as run_lists.
        numpy array, or a device pointer (int) on the first worker's device with shape=(n_records, n_samples, W)."""
        flags = (L.PIPE_GZIP if gzip else 0) | (L.COHORT_CONCURRENT_SINK if concurrent_sink else 0) | (L.PIPE_ALL_RECORDS if all_records else 0)
        if isinstance(masks, np.ndarray):
            masks = np.ascontiguousarray(masks, np.uint32)
            n_rec, n_samp, w = masks.shape
            mp = masks.ctypes.data_as(C.c_void_p)
        else:
            n_rec, n_samp, w = shape
            mp, flags = C.c_void_p(int(masks)), flags | L.COHORT_DEVICE_MASKS
        cbeg, csite = np.ascontiguousarray(csq_begin, np.uint64), np.ascontiguousarray(csq_site, np.int32)
        cb, user, keep = DevicePipeline._sink(sink)
        res = L.CohortResult()
        st = self._lib.v2p_cohort_run_masks(self._h, n_rec, n_samp, w, mp, cbeg.ctypes.data_as(C.c_void_p),
                                            csite.ctypes.data_as(C.c_void_p), chunk_samples, flags, cb, user, C.byref(res))
        del keep
        if st:
            raise EngineError(st, (self._lib.v2p_cohort_last_error(self._h) or b"").decode())
        return res
