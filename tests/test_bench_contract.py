"""bench.py keeps its contract: ONE JSON line with the keys the driver reads, on a tiny cohort.
CPU: the reference arm (`--impl reference`).  GPU: our arm, every section switched on, all parity flags true."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
        "dtype", "data", "config", "e2e"}


def run_bench(*args):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, p.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample-haps", "4", "--cpu-seconds", "0.5",
                  "--ref-binary-samples", "2")
    assert BASE <= set(d) and d["impl"] == "reference" and d["metric"] == "generated residues/sec" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["e2e"] == {"value": d["value"], "unit": "residues/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "haplotypes" in cb["sample"]
    assert "workload" in d["config"]


def test_dump_outputs_samples_fixed_windows_of_a_long_tape(tmp_path):
    import torch

    from bench_support import DUMP_BYTES, DUMP_WINDOW, dump_outputs

    n_out = DUMP_BYTES + 3 * DUMP_WINDOW + 5
    tape = torch.from_numpy(np.random.default_rng(1).integers(0, 256, n_out + 64, dtype=np.uint8))
    for d in ("a", "b"):
        dump_outputs(str(tmp_path / d), tape, n_out)
    got = {d: (np.load(tmp_path / d / "result_tape.npy"), np.load(tmp_path / d / "result_tape_window_starts.npy")) for d in "ab"}
    sample, starts = got["a"]
    assert sample.dtype == np.float32 and starts.dtype == np.float64 and sample.nbytes + starts.nbytes <= 64 << 20
    assert np.array_equal(sample, got["b"][0]) and np.array_equal(starts, got["b"][1])  # same positions every run
    s = starts.astype(np.int64)
    assert len(s) == DUMP_BYTES // DUMP_WINDOW and (np.diff(s) >= DUMP_WINDOW).all() and s[-1] + DUMP_WINDOW <= n_out
    want = tape.numpy()[(s[:, None] + np.arange(DUMP_WINDOW)).reshape(-1)]
    assert np.array_equal(sample, want.astype(np.float32))


@pytest.mark.parametrize("args,flag", [(["--steps", "0"], "--steps"),
                                       (["--impl", "reference", "--dump-outputs", "d"], "--dump-outputs"),
                                       (["--only-c3", "--dump-outputs", "d"], "--dump-outputs")])
def test_meaningless_arguments_are_refused(args, flag):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=120)
    assert p.returncode == 2 and flag in p.stderr


@pytest.mark.gpu
def test_our_arm_line_on_a_tiny_cohort(tmp_path):
    d = run_bench("--samples", "24", "--steps", "3", "--warmup", "3", "--e2e-steps", "1", "--e2e-chunk-haps", "16", "--cpu-sample-haps", "8",
                  "--cpu-seconds", "0.5", "--maskdecode-samples", "8", "--gzip-samples", "8", "--pipeline-chunk", "5",
                  "--written-samples", "6", "--c3-samples", "40", "--c3-chunk-samples", "16", "--dropin-haps", "6",
                  "--dump-outputs", str(tmp_path))
    assert BASE <= set(d) and d["n_gpus"] == 1 and d["scaling"] == "weak" and d["dtype"] == "u8" and d["vs_baseline"] is None
    assert d["gpu_launches"] == 7 * d["steps"] and d["warmup"] >= 3  # init, plan x4, copy, status hand-off
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] == d["config"]["result_tape_bytes_per_gpu"]
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["kernel"] == "k_copy_tiles"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert r["dram_frac"] is None or 0 < r["dram_frac"] < 1.2
    assert r["write_only"]["peak_gbs"] == r["write_only"]["ceilings_gbs"]["tma_bulk_store_8k"]
    p = d["parity"]
    assert p["gpu_equals_oracle"] is True and p["e2e_equals_device_path"] is True
    assert p["checked_haplotypes"] == d["config"]["haplotypes_per_gpu"] == p["haplotypes_per_gpu"] and p["all_ranks"] is True
    assert d["dropin"]["gpu_equals_oracle"] is True and d["dropin"]["haplotypes_per_s"] > 0 and d["dropin"]["host_threads"] >= 1
    c3 = d["c3"]
    assert c3["scaling"] == "strong" and c3["samples"] == 40 and c3["value"] > 0 and c3["chunks_this_rank"] == 3
    assert c3["parity"]["gpu_equals_oracle"] is True and c3["parity"]["checked_haplotypes"] == 80 == c3["parity"]["haplotypes"]
    assert d["other_layout"]["records_equal_primary_layout"] is True
    t = d["taskgen"]
    assert t["equals_host_producer"] and t["general_catalogue"]["equals_host_producer"] and t["maskdecode"]["equals_host_lists_and_tasks"]
    assert d["gzip"]["inflates_to_the_image"] is True
    for k in ("fasta", "fasta_gz"):
        assert d["pipeline"][k]["first_and_last_file_equal_oracle_text"] is True
        assert d["pipeline"]["written"][k]["first_file_equals_oracle_text"] is True
    # the dump is the timed step's result tape: the oracle's bytes at the dumped windows
    from bench_support import DUMP_WINDOW, make_workload
    from oracle import cengine

    prot, _, b = make_workload("c2", 24, 0)
    want = np.zeros(b.n_residues, np.uint8)
    assert cengine.batch_execute(b.task_begin, b.tasks, prot.residues, b.alt, b.alt_base, want, b.out_base, threads=4)[0] == 0
    starts = np.load(tmp_path / "result_tape_window_starts.npy").astype(np.int64)
    assert b.n_residues == d["config"]["result_tape_bytes_per_gpu"] and len(starts) > 1
    sample = np.load(tmp_path / "result_tape.npy")
    assert np.array_equal(sample, want[(starts[:, None] + np.arange(DUMP_WINDOW)).reshape(-1)].astype(np.float32))
