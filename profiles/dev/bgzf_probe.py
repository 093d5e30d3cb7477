"""bgzip'd VCF -> inflated text -> index on the device (v2p_vcf_load_bgzf, include/v2p_vcf.h) at the C2 size: the text
of profiles/dev/vcf_probe.py (2,504 samples x bench.py's taskgen.maskdecode records, one csq per record), written as
BGZF by synth/bgzf.py at level 6 (bgzip's default), level 1, Z_HUFFMAN_ONLY (all literals: the decoder's worst case)
and level 0 (stored).

Per variant: compressed bytes, the pinned compressed upload, inflate (device time and GB/s of text), index, the
columns 1-9 gather + copy-back, parse; in the same run the plain text's pinned upload + index.  Before any number is
printed: the inflated text equals the original, the matrix equals the synthetic masks, and the .fasta.gz images from the
level-6 .vcf.gz equal those from the plain text.  Needs a GPU.

    python profiles/dev/bgzf_probe.py --out profiles/r4/bgzf_probe_c2.json
"""
import argparse
import ctypes as Ct
import hashlib
import json
import os
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402

from vcf_probe import card, spread  # noqa: E402

VARIANTS = {"level6": (6, zlib.Z_DEFAULT_STRATEGY), "level1": (1, zlib.Z_DEFAULT_STRATEGY),
            "huffman_only": (6, zlib.Z_HUFFMAN_ONLY), "level0_stored": (0, zlib.Z_DEFAULT_STRATEGY)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--variants", default=",".join(VARIANTS))
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch

    from synth import bgzf as W
    from synth import cohort as C
    from synth import vcftext as S
    from vcf2prot_b200 import GpuEngine
    from vcf2prot_b200 import _lib as L
    from vcf2prot_b200.pipeline import DevicePipeline
    from vcf2prot_b200.vcf import DeviceVcf

    if not torch.cuda.is_available():
        raise SystemExit("bgzf_probe needs a GPU")
    res = {"card": card()}
    t0 = time.time()
    prot = C.make_proteome(seed=0x5EED0001)
    cat = C.make_catalogue(prot, 280000, seed=0x5EED0002)
    rec = C.make_records(cat, 0x5EED0009, 1)
    ns = args.samples
    hap, site = C.select_sites(cat, 2 * ns, np.random.default_rng(0x5EED0010))
    masks = C.encode_masks(rec, ns, hap, site)
    csqs = [["missense|GENE|ENST%011d|protein_coding|+|%dA>%dC|%dC>T" % (r, 1 + r % 900, 1 + r % 900, 1000 + r)]
            for r in range(rec.n_rec)]
    text = S.vcf_text(["NA%05d" % i for i in range(ns)], csqs, masks)
    n = len(text)
    res["workload"] = {"samples": ns, "records": rec.n_rec, "text_bytes": n, "host_setup_s": round(time.time() - t0, 1),
                       "host_cpus": os.cpu_count()}
    pinned = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = np.frombuffer(text, np.uint8)
    back = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    vcf = DeviceVcf(0)
    lib = L.load()

    # plain text: pinned upload + index, the yardstick
    ix = vcf.load(pinned.numpy())
    rows = np.arange(ix.n_lines)
    h2d, idx = [], []
    for _ in range(args.repeats):
        ix = vcf.load(pinned.numpy())
        h2d.append(ix.h2d_ms), idx.append(ix.index_ms)
    plain_ms = spread(h2d)["median"] + spread(idx)["median"]
    res["plain"] = {"h2d_ms": spread(h2d), "index_ms": spread(idx), "upload_plus_index_ms": plain_ms}

    gz6 = None
    for name in args.variants.split(","):
        level, strategy = VARIANTS[name]
        t = time.time()
        data = W.write(text, level, strategy)
        comp_s = time.time() - t
        cz = torch.empty(len(data), dtype=torch.uint8, pin_memory=True)
        cz.numpy()[:] = np.frombuffer(data, np.uint8)
        if name == "level6":
            gz6 = cz
        del data
        bx = vcf.load_bgzf(cz.numpy())  # warm-up, then the checks at the timed size
        assert bx.text_bytes == n and lib.v2p_device_read(Ct.c_void_p(back.data_ptr()), Ct.c_void_p(bx.text_ptr), n) == 0
        text_ok = bool(torch.equal(back, pinned))
        assert text_ok, "%s: inflated text differs from the original" % name
        m = vcf.parse_masks(rows)
        mat_ok = bool(np.array_equal(m.read(), masks))
        assert mat_ok, "%s: device matrix differs from the synthetic masks" % name
        r = {k: [] for k in ("h2d_ms", "inflate_ms", "index_ms", "fixed_ms", "parse_ms")}
        for _ in range(args.repeats):
            bx = vcf.load_bgzf(cz.numpy())
            r["h2d_ms"].append(bx.h2d_ms), r["inflate_ms"].append(bx.inflate_ms), r["index_ms"].append(bx.index_ms)
            r["fixed_ms"].append(bx.fixed_ms)
            r["parse_ms"].append(vcf.parse_masks(rows).parse_ms)
        med = {k: spread(v)["median"] for k, v in r.items()}
        ingest = med["h2d_ms"] + med["inflate_ms"] + med["index_ms"] + med["fixed_ms"]
        res[name] = {"compressed_bytes": int(cz.numel()), "ratio": n / cz.numel(), "n_blocks": bx.n_blocks,
                     "host_compress_s": round(comp_s, 1), **{k: spread(v) for k, v in r.items()},
                     "inflate_text_gbs": n / (med["inflate_ms"] * 1e-3) / 1e9, "fixed_bytes": int(bx.fixed_begin[-1]),
                     "upload_inflate_index_fixed_ms": ingest, "over_plain_upload_plus_index": ingest / plain_ms,
                     "text_equals_original": text_ok, "matrix_equals_synth_masks": mat_ok}
        if name != "level6":
            del cz

    # .fasta.gz images: level-6 .vcf.gz -> device matrix, against the plain text -> device matrix
    if gz6 is not None:
        eng = GpuEngine(0)
        eng.set_reference(prot.residues)
        pipe = DevicePipeline(eng, prot, cat, C.default_names(prot), lanes=2)
        digests = {}
        for kind in ("vcf_gz", "plain_text"):
            h = hashlib.sha256()

            def sink(first, k, data, begins):
                h.update(bytes(data))
                return 0

            if kind == "vcf_gz":
                vcf.load_bgzf(gz6.numpy())
            else:
                vcf.load(pinned.numpy())
            mm = vcf.parse_masks(rows)
            pipe.run_masks(mm.ptr, rec.csq_begin, rec.csq_site, shape=mm.shape, chunk_samples=128, gzip=True, sink=sink)
            digests[kind] = h.hexdigest()
        same = digests["vcf_gz"] == digests["plain_text"]
        assert same, ".fasta.gz images from the .vcf.gz differ from those of the plain text"
        res["fasta_gz_same_as_plain"] = same
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
