"""VCF text -> mask matrix on the device (include/v2p_vcf.h) at the C2 size: 2,504 samples x the taskgen.maskdecode
records of bench.py (one csq per record), written by synth/vcftext.py.

Reports the text size, the H2D time from pinned and from pageable memory, index / parse device time (CUDA events,
warm-up, repeats, spread), each phase's text bytes/s and its algorithmic bytes over the measured HBM copy rate, and
pinned text -> .fasta.gz images through v2p_pipeline_run_masks(DEVICE_PTRS) next to the same cohort's host matrix through
run_masks.  The device matrix is checked against the synthetic masks before any number is printed.  Needs a GPU.

    python profiles/dev/vcf_probe.py --out profiles/r3/vcf_probe_c2.json
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def spread(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1], "n": len(xs)}


def card():
    import torch

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def hbm_copy_gbs(torch, n=4 << 30, reps=10):
    x = torch.empty(n, dtype=torch.uint8, device="cuda")
    y = torch.empty_like(x)
    y.copy_(x)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(reps):
        a.record()
        y.copy_(x)
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    del x, y
    return 2 * n / (spread(ms)["median"] * 1e-3) / 1e9  # read + write


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch

    from synth import cohort as C
    from synth import vcftext as S
    from vcf2prot_b200 import GpuEngine
    from vcf2prot_b200.pipeline import DevicePipeline
    from vcf2prot_b200.vcf import DeviceVcf

    if not torch.cuda.is_available():
        raise SystemExit("vcf_probe needs a GPU")
    res = {"card": card()}
    t0 = time.time()
    prot = C.make_proteome(seed=0x5EED0001)
    cat = C.make_catalogue(prot, 280000, seed=0x5EED0002)
    rec = C.make_records(cat, 0x5EED0009, 1)  # bench.py's taskgen.maskdecode records
    ns = args.samples
    hap, site = C.select_sites(cat, 2 * ns, np.random.default_rng(0x5EED0010))
    masks = C.encode_masks(rec, ns, hap, site)
    csqs = [["missense|GENE|ENST%011d|protein_coding|+|%dA>%dC|%dC>T" % (r, 1 + r % 900, 1 + r % 900, 1000 + r)]
            for r in range(rec.n_rec)]
    text = S.vcf_text(["NA%05d" % i for i in range(ns)], csqs, masks)
    n = len(text)
    res["workload"] = {"samples": ns, "records": rec.n_rec, "words_per_cell": int(masks.shape[2]), "text_bytes": n,
                       "carrier_bits": int(len(site)), "host_setup_s": round(time.time() - t0, 1)}
    pinned = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = np.frombuffer(text, np.uint8)
    pageable = np.frombuffer(text, np.uint8)
    d_text = pinned.cuda()
    del text
    vcf = DeviceVcf(0)

    ix = vcf.load(pinned.numpy())  # warm-up (allocations, module load)
    rows = np.arange(ix.n_lines)
    m = vcf.parse_masks(rows)
    assert ix.n_samples == ns and ix.n_lines == rec.n_rec
    ok = bool(np.array_equal(m.read(), masks))  # at the timed size, before any number
    assert ok, "device matrix differs from the synthetic masks"
    cell_bytes = int((np.append(ix.line_begin[1:], n) - ix.cells_begin).sum())  # sample cells (+ line ends)
    h2d_p, idx_p, h2d_g, idx_d, parse = [], [], [], [], []
    for _ in range(args.repeats):
        ix = vcf.load(pinned.numpy())
        h2d_p.append(ix.h2d_ms), idx_p.append(ix.index_ms)
    for _ in range(3):
        h2d_g.append(vcf.load(pageable).h2d_ms)
    for _ in range(args.repeats):
        idx_d.append(vcf.load((d_text.data_ptr(), n)).index_ms)
    for _ in range(args.repeats):
        parse.append(vcf.parse_masks(rows).parse_ms)
    hbm = hbm_copy_gbs(torch)
    i_ms, p_ms = spread(idx_d)["median"], spread(parse)["median"]
    alg_index = 2 * n + 24 * ix.n_lines  # the text twice + line tables
    alg_parse = 2 * cell_bytes + masks.nbytes
    res["h2d"] = {"pinned_ms": spread(h2d_p), "pageable_ms": spread(h2d_g),
                  "pinned_gbs": n / (spread(h2d_p)["median"] * 1e-3) / 1e9, "pageable_gbs": n / (spread(h2d_g)["median"] * 1e-3) / 1e9}
    res["index"] = {"ms_device_text": spread(idx_d), "ms_after_pinned_upload": spread(idx_p), "text_gbs": n / (i_ms * 1e-3) / 1e9,
                    "alg_bytes": alg_index, "alg_bytes_over_hbm_copy_rate_ms": alg_index / (hbm * 1e9) * 1e3}
    res["parse"] = {"ms": spread(parse), "cell_bytes": cell_bytes, "text_gbs": cell_bytes / (p_ms * 1e-3) / 1e9,
                    "matrix_bytes": int(masks.nbytes), "alg_bytes": alg_parse,
                    "alg_bytes_over_hbm_copy_rate_ms": alg_parse / (hbm * 1e9) * 1e3}
    res["hbm_copy_gbs_measured"] = hbm
    res["index_plus_parse_over_pinned_upload"] = (i_ms + p_ms) / spread(h2d_p)["median"]
    res["matrix_equals_synth_masks"] = ok

    # ---- text -> .fasta.gz images, next to the host matrix through run_masks
    eng = GpuEngine(0)
    eng.set_reference(prot.residues)
    pipe = DevicePipeline(eng, prot, cat, C.default_names(prot), lanes=2)
    digests = {}

    def run(kind):
        h = hashlib.sha256()

        def sink(first, k, data, begins):
            h.update(bytes(data))
            return 0

        torch.cuda.synchronize()
        t = time.perf_counter()
        if kind == "device_text":
            vcf.load(pinned.numpy())
            mm = vcf.parse_masks(rows)
            _, r = pipe.run_masks(mm.ptr, rec.csq_begin, rec.csq_site, shape=mm.shape, chunk_samples=128, gzip=True, sink=sink)
        else:
            _, r = pipe.run_masks(masks, rec.csq_begin, rec.csq_site, chunk_samples=128, gzip=True, sink=sink)
        wall = time.perf_counter() - t
        digests[kind] = h.hexdigest()
        return wall, r

    out = {}
    for kind in ("device_text", "host_matrix"):
        run(kind)  # warm-up
        walls = []
        for _ in range(2):
            w, r = run(kind)
            walls.append(w)
        out[kind] = {"wall_s": spread(walls), "decode_ms": float(r.decode_ms), "out_bytes": int(r.out_bytes), "h2d_bytes": int(r.h2d_bytes)}
    out["same_files"] = digests["device_text"] == digests["host_matrix"]
    out["what"] = ("device_text: pinned text -> v2p_vcf_load -> v2p_vcf_parse_masks -> v2p_pipeline_run_masks(DEVICE_PTRS), "
                   "gzip, 2 lanes, 128-sample chunks, sink hashing every byte; host_matrix: the same cohort's mask matrix from "
                   "host memory through run_masks")
    res["to_fasta_gz"] = out
    pipe.close()
    eng.close()
    vcf.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
