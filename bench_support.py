"""bench_support.py -- pieces of bench.py that are not the timed loop: the synthetic workload, the clock sampler, the CPU
legs (oracle port = `cpu_baseline` / `--impl reference`; the reference's prebuilt binary timed beside it) and the
measurements of the rows either side of the hot path (gzip, the whole-cohort pipeline).

This module is test/bench infrastructure like bench.py itself: it is the one place besides tests/ and smoke() that may
use oracle/ -- as the checker and as the CPU baseline, never as the thing measured on the GPU arm."""
from __future__ import annotations

import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


# ------------------------------------------------------------------------------------------------ workload
def make_workload(kind: str, n_samples: int, rank: int, layout: str = "packed", fasta: bool = False):
    from synth import cohort as C

    prot = C.make_proteome(seed=0x5EED0001, giant=(20 if kind == "c4" else 0))
    if kind == "c2":
        cat = C.make_catalogue(prot, 280000, seed=0x5EED0002)
    else:
        cat = C.make_catalogue(prot, 120000, seed=0x5EED0004, mix=C.MIX_C4, fs_mean=60, fs_max=4000, sl_max=500,
                               long_ins_mean=50, long_ins_max=5000, lognormal_tails=True)
    n_hap = 2 * n_samples
    parts = []
    step = 256
    for i, h0 in enumerate(range(0, n_hap, step)):
        parts.append(C.synth_batch(prot, cat, min(step, n_hap - h0), seed=(0x5EED0002 + 7919 * rank) * 1000 + i,
                                   layout=layout))
    if fasta:  # record framing as copy segments (SURVEY 8f.1): the result tape is the .fasta file image
        parts = [C.fasta_image(prot, b) for b in parts]
    return prot, cat, C.concat_batches(parts)


def alg_bytes(batch) -> int:
    """SURVEY.md 8(d): sum(len) read + sum(len) written + '.' gap bytes + 16 B per packed task."""
    covered = int(batch.tasks[:, 1].astype(np.int64).sum())
    n_out = batch.n_residues
    return covered + n_out + 16 * len(batch.tasks)  # n_out = covered + gap bytes


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons, pw = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                clk, mxc, p = float(f[1]), float(f[2]), float(f[3])
            except ValueError:
                continue
            mx = mxc
            if t0 - 0.05 <= ts <= t1 + 0.1:
                sm.append(clk)
                pw.append(p)
                for n, v in zip(names, f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------------------------------------ CPU side
def oracle_check_range(batch, prot, h0: int, h1: int, gpu_bytes: np.ndarray) -> bool:
    """Oracle (1-byte port) on haplotypes [h0,h1) of the cohort vs the GPU's bytes for the same range."""
    from oracle import cengine

    t0, t1 = int(batch.task_begin[h0]), int(batch.task_begin[h1])
    a0, a1 = int(batch.alt_base[h0]), int(batch.alt_base[h1])
    o0, o1 = int(batch.out_base[h0]), int(batch.out_base[h1])
    out = np.zeros(o1 - o0, np.uint8)
    rebase = lambda a, x: (a[h0:h1 + 1] - np.uint64(x)).astype(np.uint64)
    st, _, _ = cengine.batch_execute(rebase(batch.task_begin, t0), batch.tasks[t0:t1], prot.residues, batch.alt[a0:a1],
                                     rebase(batch.alt_base, a0), out, rebase(batch.out_base, o0), threads=os.cpu_count() or 1)
    return st == 0 and bool(np.array_equal(out, gpu_bytes))


def cpu_engine_rate(batch, prot, n_haps: int, seconds: float, threads: int, width: int, check_against=None):
    """Reference-equivalent CPU engine (oracle port) on the first n_haps haplotypes; returns residues/s."""
    from oracle import cengine

    n_haps = min(n_haps, batch.n_hap)
    t1 = int(batch.task_begin[n_haps])
    a1, o1 = int(batch.alt_base[n_haps]), int(batch.out_base[n_haps])
    dt = np.uint32 if width == 4 else np.uint8
    ref = prot.residues.astype(dt)
    alt = batch.alt[:a1].astype(dt)
    out = np.zeros(o1, dt)
    args = (batch.task_begin[:n_haps + 1], batch.tasks[:t1], ref, alt, batch.alt_base[:n_haps + 1], out,
            batch.out_base[:n_haps + 1])
    st, _, _ = cengine.batch_execute(*args, threads=threads)  # warm-up + page-in
    assert st == 0
    reps, t0 = 0, time.perf_counter()
    while True:
        st, _, _ = cengine.batch_execute(*args, threads=threads)
        reps += 1
        el = time.perf_counter() - t0
        if el >= seconds or reps >= 1000:
            break
    ok = None
    if check_against is not None:
        ok = bool(np.array_equal(out.astype(np.uint8), check_against[:o1]))
    return o1 * reps / el, el, reps, n_haps, o1, ok


def reference_binary_rate(prot, cat, batch, n_samples: int):
    """Whole-tool timing of the reference's own prebuilt binary on the first n_samples of the cohort."""
    from oracle import refbin
    from synth import cohort as C

    if not refbin.available() or n_samples <= 0:
        return None
    n_samples = min(n_samples, batch.n_hap // 2)
    sel = batch.kept_hap < 2 * n_samples if batch.kept_hap is not None else None
    return None if sel is None else _ref_binary_run(prot, cat, batch, n_samples, sel, refbin, C)


def _ref_binary_run(prot, cat, batch, n_samples, sel, refbin, C):
    hap, site = batch.kept_hap[sel], batch.kept_site[sel]
    used, inv = np.unique(site, return_inverse=True)
    mask = np.zeros((len(used), n_samples), np.uint8)
    np.bitwise_or.at(mask, (inv, hap // 2), (1 << (hap % 2)).astype(np.uint8))  # both haplotypes may carry a site
    refs = {prot.name(t): prot.seq(t) for t in range(prot.n_tx)}
    samples = ["S%05d" % i for i in range(n_samples)]
    lines = [refbin.VCF_HEADER, "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(samples) + "\n"]
    cell = ["0|0:0", "1|0:1", "0|1:2", "1|1:3"]
    for r, i in enumerate(used):
        lines.append("1\t%d\t.\tC\tT\t.\t.\tAC=1;BCSQ=%s\tGT:BCSQ\t%s\n" %
                     (100 + r, C.site_csq(prot, cat, int(i)), "\t".join(cell[m] for m in mask[r])))
    t0 = time.perf_counter()
    recs, stdout, rc = refbin.run_reference("".join(lines), refs, "mt", verbose=True, timeout=1200)
    wall = time.perf_counter() - t0
    st = refbin.stage_seconds(stdout)
    n_res = sum(len(s) for v in recs.values() for _, s in v)
    if rc != 0 or not st:
        return {"error": "reference binary rc=%d" % rc}
    return {"samples": n_samples, "residues": n_res, "wall_s": round(wall, 2), "parse_s": round(st["parse"], 2),
            "exec_stage_s": round(st["exec"], 3), "write_s": round(st["write"], 2),
            "exec_stage_residues_per_s": n_res / max(st["exec"], 1e-9), "whole_tool_residues_per_s": n_res / st["total"],
            "engine": "mt", "version": "0.1.2 (bins/Linux/vcf2prot)"}


def gzip_measure(args, prot, cat, eng, dev, local_rank, torch):
    """FASTA image of `--gzip-samples` samples produced on the device, then v2p_gzip_files device -> device; only the
    compressed bytes cross PCIe.  Beside it: zlib level 9 (what flate2 Compression::best amounts to) on one host core."""
    import zlib

    from synth import cohort as C
    from vcf2prot_b200.gzipdev import DeviceGzip

    ns = args.gzip_samples
    parts = [C.fasta_image(prot, C.synth_batch(prot, cat, min(256, 2 * ns - h0), seed=0x5EED0011 * 1000 + i, layout="packed"))
             for i, h0 in enumerate(range(0, 2 * ns, 256))]
    img = C.concat_batches(parts)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)
    d = [up(img.task_begin), up(img.tasks), up(img.alt), up(img.alt_base), up(img.out_base)]
    d_img = torch.empty(img.n_residues + 64, dtype=torch.uint8, device=dev)
    eng.execute_batch_device(img.n_hap, d[0], d[1], None, d[2], d[3], d_img, d[4], len(img.tasks), len(img.alt), img.n_residues)
    torch.cuda.synchronize()
    gz = DeviceGzip(local_rank)
    file_begin = np.ascontiguousarray(img.out_base[::2])
    cap = gz.bound(img.n_residues, ns)
    d_gz = torch.empty(cap, dtype=torch.uint8, device=dev)
    gz.compress_device(d_img.data_ptr(), file_begin, d_gz.data_ptr(), cap)  # warm-up (allocations)
    runs = [gz.compress_device(d_img.data_ptr(), file_begin, d_gz.data_ptr(), cap) for _ in range(5)]
    ob, res = runs[-1]
    ms = sorted(r.ms for _, r in runs)
    h_gz = torch.empty(int(ob[-1]), dtype=torch.uint8).pin_memory()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    h_gz.copy_(d_gz[: int(ob[-1])], non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    d2h_ms = e0.elapsed_time(e1)
    # the judge: zlib inflates the first and the last sample's member back to the image the device produced
    image = d_img[: img.n_residues].cpu().numpy()
    ok = True
    for s_ in (0, ns - 1):
        dec = zlib.decompressobj(wbits=31)
        got = dec.decompress(h_gz.numpy()[int(ob[s_]):int(ob[s_ + 1])].tobytes())
        ok = ok and dec.eof and got == image[int(file_begin[s_]):int(file_begin[s_ + 1])].tobytes()
    one = image[int(file_begin[0]):int(file_begin[1])].tobytes()
    t0 = time.perf_counter()
    z9 = len(zlib.compress(one, 9))
    t_z9 = time.perf_counter() - t0
    gz.close()
    return {"samples": ns, "image_bytes": int(res.in_bytes), "gz_bytes": int(res.out_bytes), "ratio": res.in_bytes / max(1, res.out_bytes),
            "chunks": int(res.n_chunks), "stored_chunks": int(res.n_stored_chunks), "ms_median": ms[len(ms) // 2], "ms_best": ms[0],
            "image_gbs": res.in_bytes / (ms[len(ms) // 2] * 1e-3) / 1e9, "d2h_ms_of_gz_bytes": d2h_ms,
            "d2h_ms_if_uncompressed": d2h_ms * res.in_bytes / max(1, res.out_bytes), "inflates_to_the_image": bool(ok),
            "cpu_zlib9_one_core": {"mbs": len(one) / t_z9 / 1e6, "ratio": len(one) / z9, "sample_bytes": len(one)},
            "what": "v2p_gzip_files, device -> device: one gzip member per sample file, 16 KiB dynamic-Huffman chunks"}


def oracle_file_text(batch, prot, s: int) -> bytes:
    """Sample s's .fasta text from the ORACLE's tapes (hap-1 records, then hap-2 records, tape order)."""
    from oracle import cengine
    from synth import cohort as C

    h0, h1 = 2 * s, 2 * s + 2
    t0, t1 = int(batch.task_begin[h0]), int(batch.task_begin[h1])
    a0, a1 = int(batch.alt_base[h0]), int(batch.alt_base[h1])
    o0, o1 = int(batch.out_base[h0]), int(batch.out_base[h1])
    tape = np.zeros(o1 - o0, np.uint8)
    rebase = lambda a, x: (a[h0:h1 + 1] - np.uint64(x)).astype(np.uint64)
    st, _, _ = cengine.batch_execute(rebase(batch.task_begin, t0), batch.tasks[t0:t1], prot.residues, batch.alt[a0:a1],
                                     rebase(batch.alt_base, a0), tape, rebase(batch.out_base, o0))
    assert st == 0
    txt = []
    for k in (0, 1):
        base = int(batch.out_base[h0 + k]) - o0
        lo, hi = np.searchsorted(batch.ann_hap, [h0 + k, h0 + k + 1])
        for r in range(lo, hi):
            seq = tape[base + int(batch.ann_start[r]): base + int(batch.ann_end[r])].tobytes()
            txt.append(b">" + prot.name(int(batch.ann_tx[r])).encode() + b"_%d\n" % (k + 1) + seq + b"\n")
    return b"".join(txt)


def pipeline_measure(args, prot, cat, batch, eng, local_rank, barrier, shard, dev):
    """v2p_pipeline_run_lists on the timed cohort: the per-haplotype site lists go up (4 B/site), every sample's .fasta
    (then .fasta.gz) image lands in the pipeline's pinned ring and is handed to a sink; tasks, tapes and images never
    exist on the host.  First and last file are compared with the oracle's text."""
    import zlib

    from synth import cohort as C
    from vcf2prot_b200.pipeline import DevicePipeline, csr_lists

    ns = batch.n_hap // 2 if args.pipeline_samples < 0 else min(args.pipeline_samples, batch.n_hap // 2)
    sel = batch.kept_hap < 2 * ns
    sb, sites = csr_lists(batch.kept_hap[sel], batch.kept_site[sel], 2 * ns)
    n_res = int((batch.ann_end - batch.ann_start)[batch.ann_hap < 2 * ns].sum())
    want_first, want_last = oracle_file_text(batch, prot, 0), oracle_file_text(batch, prot, ns - 1)
    pipe = DevicePipeline(eng, prot, cat, C.default_names(prot), lanes=2, device=local_rank)
    out = {"samples": ns, "chunk_samples": args.pipeline_chunk, "lanes": 2, "residues": n_res,
           "api": "v2p_pipeline_run_lists (host site lists in, file images to a sink through the pipeline's pinned ring)"}
    warm = min(ns, 2 * args.pipeline_chunk)
    for gz in (False, True):
        got = {}

        def sink(first, n, data, begins):
            if first == 0:
                got["first"] = bytes(data[: int(begins[1])])
            if first + n == ns:
                got["last"] = bytes(data[int(begins[n - 1]): int(begins[n])])
            return 0

        pipe.run_lists(sb[: 2 * warm + 1], sites[: int(sb[2 * warm])], warm, args.pipeline_chunk, gz, sink=lambda *a: 0)  # allocations
        barrier()
        _, r = pipe.run_lists(sb, sites, ns, args.pipeline_chunk, gz, sink=sink)
        un = (lambda b: zlib.decompress(b, wbits=31)) if gz else (lambda b: b)
        wall = shard.max_over_ranks(r.wall_s, dev)  # all ranks run their own sample range at once (weak scaling)
        out["fasta_gz" if gz else "fasta"] = {
            "residues_per_s": shard.sum_over_ranks(n_res, dev) / wall, "wall_s": wall, "h2d_bytes": int(r.h2d_bytes), "d2h_bytes": int(r.out_bytes),
            "image_bytes": int(r.image_bytes), "records": int(r.n_records), "tasks": int(r.n_tasks), "chunks": int(r.n_chunks),
            "gen_ms": r.gen_ms, "exec_ms": r.exec_ms, "gzip_ms": r.gzip_ms,
            "first_and_last_file_equal_oracle_text": bool(un(got["first"]) == want_first and un(got["last"]) == want_last)}
    # ---- and onto the file system: {tmpdir}/{proband}.fasta[.gz] through the native directory writer (rank 0 only)
    nw = min(args.written_samples, ns)
    if nw > 0 and int(os.environ.get("RANK", "0")) == 0:
        import shutil
        import tempfile

        from vcf2prot_b200.pipeline import DirWriter

        n_res_w = int((batch.ann_end - batch.ann_start)[batch.ann_hap < 2 * nw].sum())
        names = ["S%06d" % i for i in range(nw)]
        out["written"] = {"samples": nw, "residues": n_res_w, "writer_threads": 8,
                          "what": "v2p_pipeline_run_lists -> v2p_dir_writer_sink: write(2) of the file images, one file per proband"}
        for gz in (False, True):
            tmpdir = tempfile.mkdtemp(prefix="v2p_written_")
            try:
                w = DirWriter(tmpdir, names, compressed=gz, threads=8)
                _, r = pipe.run_lists(sb[: 2 * nw + 1], sites[: int(sb[2 * nw])], nw, args.pipeline_chunk, gz, sink=w)
                one = open(os.path.join(tmpdir, names[0] + (".fasta.gz" if gz else ".fasta")), "rb").read()
                ok = (zlib.decompress(one, wbits=31) if gz else one) == want_first and w.files_written == nw
                out["written"]["fasta_gz" if gz else "fasta"] = {
                    "residues_per_s": n_res_w / r.wall_s, "wall_s": r.wall_s, "bytes": w.bytes_written, "files": w.files_written,
                    "file_gbs": w.bytes_written / r.wall_s / 1e9, "first_file_equals_oracle_text": bool(ok)}
                w.close()
            finally:
                shutil.rmtree(tmpdir, ignore_errors=True)
    pipe.close()
    return out


# ------------------------------------------------------------------------------------------------ output dump
DUMP_BYTES = 8 << 20  # result-tape bytes written by dump_outputs: 32 MiB as float32
DUMP_WINDOW = 4096
DUMP_SEED = 0x5EED00D0


def dump_outputs(out_dir: str, tape, n_out: int) -> None:
    """Write the result tape the timed path handed its caller (torch uint8 tape[:n_out]) under out_dir, so that two builds
    can be compared output for output: result_tape.npy (float32 residue bytes) and result_tape_window_starts.npy (float64
    tape offsets).  A tape of more than DUMP_BYTES is sampled in non-overlapping DUMP_WINDOW-byte windows whose starts
    come from a fixed seed, so the same bench arguments always dump the same positions."""
    import torch

    if n_out <= DUMP_BYTES:
        starts = np.zeros(1, np.int64)
        sample = tape[:n_out]
    else:
        n_win = DUMP_BYTES // DUMP_WINDOW
        rng = np.random.default_rng(DUMP_SEED)
        starts = np.sort(rng.choice(n_out // DUMP_WINDOW, n_win, replace=False)).astype(np.int64) * DUMP_WINDOW
        idx = torch.from_numpy((starts[:, None] + np.arange(DUMP_WINDOW)).reshape(-1)).to(tape.device)
        sample = tape[idx]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "result_tape.npy"), sample.cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "result_tape_window_starts.npy"), starts.astype(np.float64))


# ------------------------------------------------------------------------------------------------ whole-cohort parity
class _DevPtr:
    """A raw device pointer as a __cuda_array_interface__ object (so torch can view library-owned HBM)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def dev_view(torch, ptr: int, nbytes: int, dev):
    return torch.as_tensor(_DevPtr(ptr, nbytes), device=dev) if nbytes else torch.empty(0, dtype=torch.uint8, device=dev)


class StreamChecker:
    """GPU result tapes against the oracle, whole batches at a time and at copy speed: the tape comes back in
    ~256-haplotype pieces through two pinned buffers while the previous piece is checked by oracle.batch_check on
    `threads` host threads (each haplotype is executed into a cache-resident scratch tape and compared)."""

    def __init__(self, torch, dev, ref: np.ndarray, threads: int, piece_bytes: int = 1 << 30):
        self.torch, self.dev, self.ref, self.threads = torch, dev, np.ascontiguousarray(ref, np.uint8), max(1, threads)
        self.bufs = [torch.empty(piece_bytes, dtype=torch.uint8).pin_memory() for _ in range(2)]
        self.stream = torch.cuda.Stream(device=dev)
        self.checked_haps = self.checked_bytes = self.bad_haps = 0
        self.first_bad = None
        self.seconds = 0.0

    def check(self, d_out, task_begin, tasks, alt, alt_base, out_base, hap_offset: int = 0):
        """d_out: torch uint8 tensor on the device holding the tapes of out_base[0]..out_base[-1]; the other arrays
        are host numpy arrays of the same batch (v2p_batch layout)."""
        from oracle import cengine

        torch = self.torch
        t_start = time.perf_counter()
        n_hap = len(out_base) - 1
        ob = out_base.astype(np.int64) - int(out_base[0])
        cap = self.bufs[0].numel()
        pieces, h0 = [], 0
        while h0 < n_hap:  # as many haplotypes as fit one pinned buffer (at least one)
            h1 = int(np.searchsorted(ob, ob[h0] + cap, side="right")) - 1
            h1 = min(max(h1, h0 + 1), n_hap)
            if ob[h1] - ob[h0] > cap:
                raise ValueError("one haplotype is larger than the pinned piece buffer")
            pieces.append((h0, h1))
            h0 = h1
        result = {}

        def work(i, a, b, host):
            t0, t1 = int(task_begin[a]), int(task_begin[b])
            a0, a1 = int(alt_base[a]), int(alt_base[b])
            result[i] = cengine.batch_check(task_begin[a:b + 1], tasks[t0 - int(task_begin[0]):t1 - int(task_begin[0])], self.ref,
                                            alt[a0 - int(alt_base[0]):a1 - int(alt_base[0])], alt_base[a:b + 1], host,
                                            out_base[a:b + 1], threads=self.threads)

        th = None
        for i, (a, b) in enumerate(pieces):
            buf = self.bufs[i % 2]
            n = int(ob[b] - ob[a])
            with torch.cuda.stream(self.stream):
                buf[:n].copy_(d_out[int(ob[a]):int(ob[b])], non_blocking=True)
            self.stream.synchronize()
            if th is not None:
                th.join()  # piece i-1 checked (its buffer is the other one; buffer i%2 was checked before this copy began)
            th = threading.Thread(target=work, args=(i, a, b, buf[:n].numpy()))
            th.start()
            # the NEXT copy goes into the other buffer, whose check (piece i-1) has just been joined
        if th is not None:
            th.join()
        for i, (a, b) in enumerate(pieces):
            nb, fb = result[i]
            if nb and self.first_bad is None:
                self.first_bad = hap_offset + a + fb
            self.bad_haps += nb
        self.checked_haps += n_hap
        self.checked_bytes += int(ob[-1])
        self.seconds += time.perf_counter() - t_start
        return self.bad_haps == 0


# ------------------------------------------------------------------------------------------------ C3: the 50k-sample cohort
def c3_measure(args, eng, prot, rank, world, local_rank, dev, shard, barrier, peak_gbs, dram_bytes_per_residue):
    """BASELINE.json configs[2] / north_star: ONE seeded 50,000-sample cohort, contiguous sample ranges over the ranks
    (parts/exec.rs:34-40: the reference's parallel unit is the proband), every rank streaming its range through HBM
    in chunks: [synthetic site lists, made on the device] -> v2p_generate_tasks_from_lists -> v2p_execute_batch
    (DEVICE_PTRS).  At N = 1 all ~320 GB of result tape go through the one GPU.  STRONG scaling: total work is fixed.
    Timed pass: device time (CUDA events) of every chunk's launch group, summed, max over ranks.  Check pass: every
    chunk's tapes and Task arrays come back and the oracle re-executes ALL of them (every rank its own range)."""
    import torch

    from synth import cohort as C
    from synth import devgen
    from vcf2prot_b200 import _lib as L
    from vcf2prot_b200.taskgen import DeviceCatalogue, execute_generated

    n_samples, chunk = args.c3_samples, args.c3_chunk_samples
    seed = 0x5EED0003
    cat = C.make_catalogue(prot, 280000, seed=seed)
    gen = devgen.DeviceCohort(cat, seed, local_rank)
    dc = DeviceCatalogue(prot, cat, local_rank)

    def generate(s0, ns):
        begin, sites, n = gen.lists(2 * s0, 2 * ns)
        lists = L.SiteLists()
        lists.n_hap, lists.n_sites, lists.site_begin, lists.sites = 2 * ns, n, begin.data_ptr(), sites.data_ptr()
        return dc.generate_from_lists(lists, aligned=False), n

    # ---- pass 0 (planning, untimed): result-tape bytes of every sample -> contiguous ranges balanced by bytes
    t0 = time.perf_counter()
    weights = np.zeros(n_samples, np.int64)
    for s0 in range(0, n_samples, chunk):
        ns = min(chunk, n_samples - s0)
        g, _ = generate(s0, ns)
        ob = dc.read(g.batch.out_base, 2 * ns + 1, np.uint64).astype(np.int64)
        weights[s0:s0 + ns] = ob[2::2] - ob[:-2:2]
    ranges = shard.balanced_ranges(weights.tolist(), world)
    lo, hi = ranges[rank]
    per_rank = [int(weights[a:b].sum()) for a, b in ranges]
    plan_s = time.perf_counter() - t0

    # ---- timed pass
    chunks = [(s0, min(chunk, hi - s0)) for s0 in range(lo, hi, chunk)]
    for s0, ns in chunks[:1]:  # warm-up: allocations of the largest buffers
        g, _ = generate(s0, ns)
        for _ in range(3):
            execute_generated(eng, g)
    launches0 = eng.launch_count()
    barrier()
    w0 = time.perf_counter()
    exec_ms = copy_ms = gen_ms = 0.0
    n_res = n_tasks = n_sites = 0
    for s0, ns in chunks:
        g, n = generate(s0, ns)
        gm, cm = execute_generated(eng, g)
        exec_ms, copy_ms, gen_ms = exec_ms + gm, copy_ms + cm, gen_ms + g.gen_ms
        n_res, n_tasks, n_sites = n_res + int(g.batch.n_out), n_tasks + int(g.batch.n_tasks), n_sites + n
    torch.cuda.synchronize()
    wall_s = time.perf_counter() - w0
    launches = eng.launch_count() - launches0
    alg = 2 * n_res + 16 * n_tasks  # SURVEY 8d: read + written + 16 B/task (these classes leave no '.' gaps)
    t_exec = shard.max_over_ranks(exec_ms, dev)
    t_copy = shard.max_over_ranks(copy_ms, dev)
    t_gen_exec = shard.max_over_ranks(exec_ms + gen_ms, dev)
    t_wall = shard.max_over_ranks(wall_s, dev)
    tot_res, tot_tasks, tot_alg = shard.sum_over_ranks(n_res, dev), shard.sum_over_ranks(n_tasks, dev), shard.sum_over_ranks(alg, dev)

    # ---- check pass: every haplotype of this rank's range against the oracle
    parity = None
    if not args.no_c3_parity:
        threads = max(1, (os.cpu_count() or 1) // world)
        ck = StreamChecker(torch, dev, prot.residues, threads)
        for s0, ns in chunks:
            g, _ = generate(s0, ns)
            execute_generated(eng, g)
            b = g.batch
            nh = 2 * ns
            ck.check(dev_view(torch, b.out, b.n_out, dev), dc.read(b.task_begin, nh + 1, np.uint64),
                     dc.read(b.tasks, 4 * b.n_tasks, np.uint32).reshape(-1, 4), dc.read(b.alt, b.n_alt, np.uint8),
                     dc.read(b.alt_base, nh + 1, np.uint64), dc.read(b.out_base, nh + 1, np.uint64), hap_offset=2 * s0)
        bad_all = shard.sum_over_ranks(ck.bad_haps, dev)
        haps_all = shard.sum_over_ranks(ck.checked_haps, dev)
        bytes_all = shard.sum_over_ranks(ck.checked_bytes, dev)
        parity = {"checked_haplotypes": haps_all, "haplotypes": 2 * n_samples, "checked_residues": bytes_all,
                  "mismatching_haplotypes": bad_all, "gpu_equals_oracle": bad_all == 0 and haps_all == 2 * n_samples,
                  "all_ranks": True, "oracle_threads_per_rank": threads, "seconds": round(shard.max_over_ranks(ck.seconds, dev), 1),
                  "what": "every chunk's result tape + Task arrays D2H, oracle.batch_check re-executes every haplotype (u8 tapes)"}
    gen.close()
    dc.close()
    kernel_gbs = tot_alg / (t_copy * 1e-3) / 1e9
    return {"workload": "c3: ONE %d-sample phased cohort (seed 0x5EED0003, %d haplotypes) x 20k-transcript proteome, missense-dominated "
                        "mix, contiguous sample ranges balanced by result-tape bytes over %d rank(s), streamed in %d-sample chunks"
                        % (n_samples, 2 * n_samples, world, chunk),
            "scaling": "strong", "n_gpus": world, "samples": n_samples, "residues": tot_res, "tasks": tot_tasks,
            "value": tot_res / (t_exec * 1e-3), "unit": "residues/s", "exec_ms_max_rank": t_exec, "copy_kernel_ms_max_rank": t_copy,
            "value_with_task_generation": tot_res / (t_gen_exec * 1e-3), "gen_plus_exec_ms_max_rank": t_gen_exec,
            "wall_s_max_rank": t_wall, "haplotypes_per_s": 2 * n_samples / (t_exec * 1e-3),
            "chunks_this_rank": len(chunks), "chunk_samples": chunk, "sample_range_rank0": [int(ranges[0][0]), int(ranges[0][1])],
            "range_bytes_max_over_mean": max(per_rank) / (sum(per_rank) / world), "plan_pass_s": round(plan_s, 2),
            "gpu_launches": int(launches), "sites": shard.sum_over_ranks(n_sites, dev),
            "roofline": {"bound": "hbm", "alg_bytes": tot_alg, "alg_gbs_kernel": kernel_gbs, "peak_gbs_aggregate": peak_gbs * world,
                         "frac": kernel_gbs / (peak_gbs * world),
                         "dram_gbs_kernel": None if dram_bytes_per_residue is None else dram_bytes_per_residue * tot_res / (t_copy * 1e-3) / 1e9,
                         "dram_frac": None if dram_bytes_per_residue is None else dram_bytes_per_residue * tot_res / (t_copy * 1e-3) / 1e9 / (peak_gbs * world),
                         "note": "kernel = k_copy_tiles time summed over this rank's chunks, max over ranks; alg = SURVEY 8d bytes; dram = "
                                 "ncu DRAM bytes per residue of the C2 capture x residues"},
            "parity": parity}


# ------------------------------------------------------------------------------------------------ the literal drop-in
def dropin_measure(args, eng, prot, cat, n_haps: int = 32, seconds: float = 4.0):
    """Throughput of the call INTEGRATION.md section 3 pastes into gir.rs:236-239 -- v2p_gir_execute, one haplotype per
    call, the reference's own GIR hand-off (four usize arrays + UTF-32 `char` tapes, per-haplotype ref tape) -- driven
    the way the reference drives it: many host threads at once (rayon workers, parts/exec.rs:36-39).  Beside it the
    CPU port on the SAME inputs and thread count.  Both sides are bounded by moving 4-byte residues through host
    memory; the GPU side also crosses PCIe, so this entry is parity, not speed -- the batch ABI is the fast path."""
    import ctypes as C_
    import threading

    from oracle import cengine
    from synth import cohort as C
    from vcf2prot_b200 import _lib as L

    threads = max(1, min(16, os.cpu_count() or 1))
    b = C.synth_batch(prot, cat, n_haps, seed=0x5EED0D01, ref_mode="per_hap")
    lib = L.load()
    calls, total_res = [], 0
    for h in range(n_haps):
        t0, t1 = int(b.task_begin[h]), int(b.task_begin[h + 1])
        tk = b.tasks[t0:t1].astype(np.uint64)
        cols = [np.ascontiguousarray(tk[:, i]) for i in (3, 0, 1, 2)]  # exec_code, start_pos, length, start_pos_res
        ref = b.ref[int(b.ref_base[h]):int(b.ref_base[h + 1])].astype(np.uint32)
        alt = b.alt[int(b.alt_base[h]):int(b.alt_base[h + 1])].astype(np.uint32)
        n_res = int(b.out_base[h + 1] - b.out_base[h])
        res = np.zeros(n_res, np.uint32)
        calls.append((cols, ref, alt, res, n_res))
        total_res += n_res
    p = lambda a: a.ctypes.data_as(C_.c_void_p)

    def one(c):
        cols, ref, alt, res, n_res = c
        bad = C_.c_uint64(0)
        st = lib.v2p_gir_execute(eng._h, L.ENGINE_GPU, len(cols[0]), p(cols[0]), p(cols[1]), p(cols[2]), p(cols[3]), p(ref), len(ref),
                                 p(alt), len(alt), p(res), n_res, L.FLAG_FILL_DOT, C_.byref(bad))
        if st:
            raise RuntimeError("v2p_gir_execute failed: %d" % st)

    for c in calls[:threads]:
        one(c)  # warm-up: slot allocations
    # parity of the warm-up results against the oracle (UTF-32 tapes)
    ok = True
    for cols, ref, alt, res, n_res in calls[:min(4, threads)]:
        out = np.zeros(n_res, np.uint32)
        lib2 = cengine.load()
        bad = C_.c_uint64(0)
        st = lib2.ref_gir_execute_u32(len(cols[0]), p(cols[0]), p(cols[1]), p(cols[2]), p(cols[3]), p(ref), len(ref), p(alt), len(alt),
                                      p(out), n_res, 1, 0, C_.byref(bad))
        ok = ok and st == 0 and bool(np.array_equal(out, res))
    done = [0] * threads
    stop = time.perf_counter() + seconds

    def worker(w):
        i = w
        while time.perf_counter() < stop:
            one(calls[i % n_haps])
            done[w] += calls[i % n_haps][4]
            i += threads

    t0 = time.perf_counter()
    th = [threading.Thread(target=worker, args=(w,)) for w in range(threads)]
    [t.start() for t in th]
    [t.join() for t in th]
    el = time.perf_counter() - t0
    gpu_rate = sum(done) / el
    # the CPU port on the same inputs: UTF-32 tapes, per-haplotype ref tapes, haplotypes over the same number of threads
    ref32, alt32 = b.ref.astype(np.uint32), b.alt.astype(np.uint32)
    out32 = np.zeros(int(b.out_base[-1]), np.uint32)
    a = (b.task_begin, b.tasks, ref32, alt32, b.alt_base, out32, b.out_base)
    cengine.batch_execute(*a, ref_base=b.ref_base, threads=threads)
    reps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < min(seconds, 3.0):
        cengine.batch_execute(*a, ref_base=b.ref_base, threads=threads)
        reps += 1
    cpu_rate = total_res * reps / (time.perf_counter() - t0)
    return {"api": "v2p_gir_execute (gir.rs:283-299 hand-off: 4 x usize arrays + UTF-32 tapes, one haplotype per call)",
            "host_threads": threads, "haplotypes": n_haps, "mean_residues_per_haplotype": total_res // n_haps,
            "haplotypes_per_s": gpu_rate / (total_res / n_haps), "residues_per_s": gpu_rate,
            "cpu_port_same_inputs_residues_per_s": cpu_rate, "ratio_vs_cpu_port": gpu_rate / cpu_rate,
            "gpu_equals_oracle": bool(ok), "seconds": round(el, 2),
            "note": "both sides move 4-byte residues through host memory (the CPU engine IS a memcpy of that size); the GPU side "
                    "narrows / widens them on the host and crosses PCIe as well: this entry exists for parity with the reference's "
                    "call site, the batched ABI (e2e) is the fast path"}
