#!/usr/bin/env python
"""bench.py -- throughput of the sequence-generation engine (Task-array execution) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c4] [--samples S]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path (validate + plan + copy launch group) over one cohort of synthetic,
device-resident Task arrays: every haplotype's result tape is materialised once.
Workload (config.workload):
  c2  BASELINE.json configs[1]: 2,504 phased samples (5,008 haplotypes) x 20k-transcript proteome,
      missense-dominated csq mix (SURVEY.md 8d C2).  Default.  ~17 GB of residues per step per GPU.
  c4  skewed-segment stress (configs[3] mix, SURVEY 8d C4), same sample count unless --samples is given.
N > 1: every rank owns its own contiguous sample range of the same size (weak scaling, no data-path collective);
value = residues produced by all ranks / max-over-ranks device time.

Prints ONE JSON line (rank 0).  `--impl reference` times the reference-equivalent CPU engine (the oracle's C
restatement of gir.rs:230-234 on UTF-32 tapes, haplotypes spread over all host threads like rayon par_iter,
exec.rs:34-40) on a bounded sample of the same workload; the reference itself is Rust and cannot be rebuilt here
(its prebuilt whole-tool binary is timed beside it when oracle/_ref/vcf2prot is present).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bench_support import (ClockSampler, StreamChecker, alg_bytes, c3_measure, cpu_engine_rate, dropin_measure,  # noqa: E402
                           dump_outputs, gzip_measure, make_workload, pipeline_measure, reference_binary_rate)

FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c4"])
    ap.add_argument("--samples", type=int, default=2504, help="phased samples per GPU (2 haplotypes each)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-chunk-haps", type=int, default=256)
    ap.add_argument("--e2e-depth", type=int, default=2, help="host-pointer chunks in flight (1 = no overlap)")
    ap.add_argument("--cpu-sample-haps", type=int, default=64)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--variant", type=int, default=-1, help="copy-kernel variant (-1: engine's automatic choice)")
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--ref-mode", default="replicas", choices=["replicas", "plain"])
    ap.add_argument("--layout", default="packed", choices=["packed", "aligned"],
                    help="result-tape layout: packed = the reference's own (res_counter, haplotype_instruction.rs:132), "
                         "what a drop-in caller hands over; aligned = transcripts in phase with the proteome tape (<=30 "
                         "'.' pad bytes per transcript, never seen by the consumer) -- measured beside it (other_layout)")
    ap.add_argument("--no-registered-ref", action="store_true",
                    help="pass the proteome with every call (generic register path) instead of registering it once")
    ap.add_argument("--fasta-image", action="store_true",
                    help="emit `>{transcript}_{hap}\\n{seq}\\n` framing as extra copy segments (packed layout only): "
                         "the result tape is the FASTA file image")
    ap.add_argument("--maskdecode-samples", type=int, default=512,
                    help="samples of the cohort whose FORMAT/BCSQ mask matrix is decoded on the device (0 = skip)")
    ap.add_argument("--gzip-samples", type=int, default=256,
                    help="samples whose FASTA file image is gzip-compressed on the device (0 = skip)")
    ap.add_argument("--no-taskgen", action="store_true", help="skip the device-side Task generation measurement")
    ap.add_argument("--pipeline-samples", type=int, default=-1,
                    help="samples run through v2p_pipeline_run_lists (site lists -> .fasta / .fasta.gz images in pinned host "
                         "memory); -1 = the whole cohort, 0 = skip")
    ap.add_argument("--pipeline-chunk", type=int, default=128, help="samples per pipeline chunk")
    ap.add_argument("--written-samples", type=int, default=256,
                    help="samples whose files the pipeline also WRITES, {tmpdir}/{proband}.fasta and .fasta.gz (0 = skip)")
    ap.add_argument("--c3-samples", type=int, default=50000,
                    help="samples of the ONE cohort that is sharded over the ranks and streamed (BASELINE configs[2]); 0 = skip")
    ap.add_argument("--c3-chunk-samples", type=int, default=1024, help="samples per streamed chunk of the c3 section")
    ap.add_argument("--only-c3", action="store_true",
                    help="print only the c3 section (one cohort of --c3-samples samples, sharded over the ranks and streamed): the "
                         "point of the C5 scaling sweep, profiles/dev/c5_sweep.sh")
    ap.add_argument("--no-c3-parity", action="store_true", help="skip the whole-cohort oracle check of the c3 section")
    ap.add_argument("--dropin-haps", type=int, default=32,
                    help="haplotypes driven through v2p_gir_execute from concurrent host threads (the literal drop-in); 0 = skip")
    ap.add_argument("--no-parity", action="store_true", help="skip the whole-cohort oracle check of the timed output")
    ap.add_argument("--ref-binary-samples", type=int, default=0,
                    help="also time the reference's prebuilt whole-tool binary on this many samples (slow)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's result tape of the last step (a fixed, seeded sample of "
                         "it beyond 8 MiB) as float32 DIR/result_tape.npy, its window starts beside it")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.only_c3):
        ap.error("--dump-outputs dumps the timed result tape of --impl ours; --impl reference and --only-c3 have none")
    return args


def ncu_traffic(args, n_res):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture of this configuration
    (profiles/ncu_traffic.json), scaled by residues when the capture is of another cohort size.
    -> (bytes per launch, note, bytes per residue) or (None, None, None)."""
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.isfile(tpath) and not args.fasta_image:
        mode = "plain" if (args.no_registered_ref or args.ref_mode == "plain") else "replicas"
        for ent in json.load(open(tpath)).get("entries", []):
            if (ent["workload"], ent["mode"], ent["layout"]) == (args.workload, mode, args.layout) and ent["dram_bytes_per_launch"]:
                per_res = ent["dram_bytes_per_launch"] / ent["residues"]
                if ent["samples"] == args.samples:
                    return ent["dram_bytes_per_launch"], "ncu --set full capture of this configuration (%s)" % ent["capture"], per_res
                return (int(per_res * n_res), "scaled by residues from the %d-sample ncu --set full capture (%s)" %
                        (ent["samples"], ent["capture"]), per_res)
    return None, None, None


# ------------------------------------------------------------------------------------------------ main
def main():
    args = parse_args()
    if args.fasta_image:
        args.layout = "packed"  # a file image cannot contain pad bytes
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist

    from vcf2prot_b200 import GpuEngine, shard

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.only_c3:  # the C5 sweep point: nothing but the sharded, streamed cohort
        from synth import cohort as C

        prot = C.make_proteome(seed=0x5EED0001)
        eng = GpuEngine(local_rank)
        eng.set_reference(torch.from_numpy(prot.residues).to(dev), args.ref_mode)
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]) if os.path.isfile(
            os.path.join(ROOT, "MEASURED_PEAKS.json")) else FALLBACK_HBM_GBS
        _, _, dram_per_res = ncu_traffic(args, 1)
        line = c3_measure(args, eng, prot, rank, world, local_rank, dev, shard, barrier, peak, dram_per_res)
        if rank == 0:
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return 0

    t_gen = time.perf_counter()
    prot, cat, batch = make_workload(args.workload, args.samples, rank, args.layout, args.fasta_image)
    t_gen = time.perf_counter() - t_gen
    n_hap, n_out, n_tasks = batch.n_hap, batch.n_residues, len(batch.tasks)
    # residues produced: the aligned layout also writes '.' pads and the FASTA image also writes headers -- not counted
    n_res = int((batch.ann_end - batch.ann_start).sum())
    b_alg = alg_bytes(batch)

    to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)
    d_task_begin, d_tasks, d_ref = to_dev(batch.task_begin), to_dev(batch.tasks), to_dev(batch.ref)
    d_alt, d_alt_base, d_out_base = to_dev(batch.alt), to_dev(batch.alt_base), to_dev(batch.out_base)
    d_out = torch.empty(n_out + 64, dtype=torch.uint8, device=dev)

    eng = GpuEngine(local_rank)
    eng.set_tuning(args.variant, args.ctas_per_sm)
    if not args.no_registered_ref:
        eng.set_reference(d_ref, args.ref_mode)  # proteome registered once, as the FASTA is loaded once
        d_ref_arg = None
    else:
        d_ref_arg = d_ref
    side = torch.cuda.Stream(device=dev)
    eng.set_stream(side.cuda_stream)
    dargs = (n_hap, d_task_begin, d_tasks, d_ref_arg, d_alt, d_alt_base, d_out, d_out_base, n_tasks, len(batch.alt), n_out)

    dkw = {"aligned_layout": args.layout == "aligned"}  # the producer's hint (V2P_FLAG_ALIGNED_LAYOUT)
    for _ in range(max(args.warmup, 3)):
        eng.execute_batch_device(*dargs, **dkw)
    barrier()

    sampler = ClockSampler(local_rank if "CUDA_VISIBLE_DEVICES" not in os.environ else
                           int(os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local_rank]))
    if rank == 0:
        sampler.start()
        time.sleep(0.15)
    launches0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    group_ms, copy_ms = [], []
    barrier()
    w0 = time.time()
    with torch.cuda.stream(side):
        ev0.record()
        for _ in range(args.steps):
            group_ms.append(eng.execute_batch_device(*dargs, **dkw))
            copy_ms.append(eng.last_copy_ms)
        ev1.record()
    barrier()
    w1 = time.time()
    launches = eng.launch_count() - launches0
    clocks = sampler.stop(w0, w1) if rank == 0 else None
    dev_ms = ev0.elapsed_time(ev1)  # CUDA events on the launching stream, all K steps
    max_ms = shard.max_over_ranks(dev_ms, dev)  # the slowest rank's device time
    total_res = shard.sum_over_ranks(n_res, dev)  # residues produced by all ranks in one step
    total_haps = shard.sum_over_ranks(n_hap, dev)
    total_alg = shard.sum_over_ranks(b_alg, dev)
    ms_per_step = max_ms / args.steps
    if args.dump_outputs and rank == 0:  # now: the store-ceiling probe below overwrites d_out
        dump_outputs(args.dump_outputs, d_out, n_out)

    # ---- load balance of the copy grid (SURVEY 8d C4): wall time of every warp of the persistent grid, one extra launch
    eng.profile_warps(True)
    eng.execute_batch_device(*dargs, **dkw)
    wns = eng.read_warp_ns().astype(np.float64)
    eng.profile_warps(False)
    skew = None
    if wns.size:
        skew = {"warps": int(wns.size), "warp_ms_max": float(wns.max() / 1e6), "warp_ms_mean": float(wns.mean() / 1e6),
                "warp_ms_min": float(wns.min() / 1e6), "max_over_mean": float(wns.max() / wns.mean()),
                "what": "wall time (%globaltimer) of every warp of k_copy_tiles' persistent grid in one launch: a long segment "
                        "that pinned one worker would show up as max >> mean"}

    # ---- end to end through the C ABI with HOST buffers: per step, every chunk's tasks/alt go H2D from pinned
    #      memory and every result tape comes back D2H into a pinned staging buffer (the FASTA writer's input)
    eng.set_stream(None)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    h_tasks, h_alt, h_ref = pin(batch.tasks), pin(batch.alt), pin(batch.ref)
    h_task_begin, h_alt_base, h_out_base = (np.ascontiguousarray(batch.task_begin), np.ascontiguousarray(batch.alt_base),
                                            np.ascontiguousarray(batch.out_base))
    chunks = [(h0, min(n_hap, h0 + args.e2e_chunk_haps)) for h0 in range(0, n_hap, args.e2e_chunk_haps)]
    max_chunk = max(int(batch.out_base[b] - batch.out_base[a]) for a, b in chunks)
    depth = max(1, min(args.e2e_depth, 3))  # host-pointer batches in flight (engine has 3 staging slots)
    h_outs = [torch.empty(max_chunk + 64, dtype=torch.uint8).pin_memory().numpy() for _ in range(depth)]
    h_out = h_outs[0]
    h2d = sum(int(batch.task_begin[b] - batch.task_begin[a]) * 16 + int(batch.alt_base[b] - batch.alt_base[a]) +
              3 * 8 * (b - a + 1) + (len(batch.ref) if args.no_registered_ref else 0) for a, b in chunks)

    def e2e_step():
        # chunk i's copy-back overlaps chunk i+1's upload + kernels; each in-flight chunk has its own pinned buffer
        pending = []
        for i, (a, b) in enumerate(chunks):
            ev = eng.execute_hap_range(a, b, h_task_begin, h_tasks, None if not args.no_registered_ref else h_ref, h_alt,
                                       h_alt_base, h_out_base, h_outs[i % depth], wait=False, **dkw)
            pending.append(ev)
            if len(pending) >= depth:
                eng.wait_event(pending.pop(0))
        for ev in pending:
            eng.wait_event(ev)

    if args.e2e_steps > 0:
        e2e_step()  # warm-up (allocates the engine's device staging)
    barrier()
    e0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = max(time.perf_counter() - e0, 1e-9)
    e2e_s = shard.max_over_ranks(e2e_s, dev)
    # the last chunk sits in h_out: keep it for the parity spot-check against the device-resident result
    a, b = chunks[-1]
    o0, o1 = int(batch.out_base[a]), int(batch.out_base[b])
    h_last = h_outs[(len(chunks) - 1) % depth]
    e2e_matches_device = bool(np.array_equal(h_last[:o1 - o0], d_out[o0:o1].cpu().numpy())) if args.e2e_steps > 0 else None

    # ---- all of it behind one call: site lists -> .fasta / .fasta.gz images in pinned host memory (every rank its range)
    pipeline_line = None
    if (args.pipeline_samples != 0 and not args.no_registered_ref and not args.fasta_image and
            batch.kept_hap is not None and not args.no_cpu_baseline):
        pipeline_line = pipeline_measure(args, prot, cat, batch, eng, local_rank, barrier, shard, dev)

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    else:
        peak, peak_src = FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"
    traffic, traffic_note, dram_per_res = ncu_traffic(args, n_res)

    # ---- parity of everything that was timed: the WHOLE result tape of every rank against the oracle (gir.rs:230-234)
    parity = None
    if not args.no_parity:
        threads = max(1, (os.cpu_count() or 1) // world)
        ck = StreamChecker(torch, dev, prot.residues, threads)
        ck.check(d_out[:n_out], batch.task_begin, batch.tasks, batch.alt, batch.alt_base, batch.out_base)
        bad_all, haps_all = shard.sum_over_ranks(ck.bad_haps, dev), shard.sum_over_ranks(ck.checked_haps, dev)
        e2e_all = None if e2e_matches_device is None else shard.sum_over_ranks(0 if e2e_matches_device else 1, dev) == 0
        parity = {"checked_haplotypes": haps_all // world, "haplotypes_per_gpu": n_hap, "residues": shard.sum_over_ranks(ck.checked_bytes, dev),
                  "mismatching_haplotypes": bad_all, "gpu_equals_oracle": bad_all == 0 and haps_all == total_haps,
                  "all_ranks": True, "ranks": world, "oracle_threads_per_rank": threads, "seconds": round(ck.seconds, 2),
                  "first_mismatching_haplotype": ck.first_bad, "e2e_equals_device_path": e2e_all,
                  "what": "every rank: the whole device-resident result tape of the timed step, D2H in 1 GiB pieces, "
                          "re-executed haplotype by haplotype by the oracle (ref_batch_check, u8 tapes)"}
        del ck

    # ---- BASELINE configs[2]: ONE 50k-sample cohort, contiguous ranges over the ranks, streamed (strong scaling)
    c3_line = None
    if args.c3_samples > 0 and not args.no_registered_ref and not args.fasta_image and args.layout == "packed":
        c3_line = c3_measure(args, eng, prot, rank, world, local_rank, dev, shard, barrier, peak, dram_per_res)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- CPU baseline (rank 0, N == 1 only): oracle port on a bounded sample of the same cohort
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        nh = min(args.cpu_sample_haps, n_hap)
        rate32, el, reps, nh, nres, _ = cpu_engine_rate(batch, prot, nh, args.cpu_seconds, threads, 4)
        rate8, _, _, _, _, _ = cpu_engine_rate(batch, prot, nh, min(3.0, args.cpu_seconds), threads, 1)
        cpu = {"value": rate32, "unit": "residues/s", "cores": threads, "kind": "port",
               "sample": "first %d haplotypes (%d residues) of the same cohort, UTF-32 tapes like the reference "
                         "(gir.rs:18-22), %d passes in %.1f s, haplotypes over %d threads (exec.rs:34-40)" %
                         (nh, nres, reps, el, threads),
               "value_u8_tapes": rate8}
        rb = reference_binary_rate(prot, cat, batch, args.ref_binary_samples)
        if rb:
            cpu["reference_binary"] = rb

    # ---- SURVEY 8f rank 2: the same cohort's Task arrays generated ON the device from the per-haplotype site lists
    taskgen = None
    other_line = None
    if world == 1 and not args.no_taskgen and not args.fasta_image and batch.kept_hap is not None:
        from synth import cohort as C
        from vcf2prot_b200.taskgen import DeviceCatalogue

        dc = DeviceCatalogue(prot, cat, local_rank)
        dc.generate(batch.kept_hap, batch.kept_site, n_hap, args.layout == "aligned")  # warm-up (allocations)
        g = dc.generate(batch.kept_hap, batch.kept_site, n_hap, args.layout == "aligned")
        same = (g.batch.n_tasks == n_tasks and g.batch.n_out == n_out and
                bool(np.array_equal(dc.read(g.batch.tasks, 4 * min(n_tasks, 1 << 22), np.uint32).reshape(-1, 4),
                                    batch.tasks[: min(n_tasks, 1 << 22)])) and
                bool(np.array_equal(dc.read(g.batch.out_base, n_hap + 1, np.uint64), batch.out_base)))
        if n_tasks > (1 << 22):  # and the tail of the task array
            tail = dc.read(g.batch.tasks + 16 * (n_tasks - (1 << 20)), 4 << 20, np.uint32).reshape(-1, 4)
            same = same and bool(np.array_equal(tail, batch.tasks[n_tasks - (1 << 20):]))
        n_sites = int(len(batch.kept_site))
        taskgen = {"gen_ms": g.gen_ms, "sites": n_sites, "tasks": n_tasks, "tasks_per_s": n_tasks / (g.gen_ms * 1e-3),
                   "h2d_bytes": 4 * n_sites + 8 * (n_hap + 1), "h2d_bytes_if_tasks_were_uploaded": 16 * n_tasks + len(batch.alt),
                   "equals_host_producer": same, "host_producer_seconds": round(t_gen, 1),
                   "what": "v2p_generate_tasks: per-haplotype site lists -> packed Task batch on the GPU (incl. the H2D of the lists)"}
        # ---- the same cohort in the OTHER result-tape layout, generated on the device and executed from there
        other = "aligned" if args.layout == "packed" else "packed"
        from vcf2prot_b200.taskgen import execute_generated

        go = dc.generate(batch.kept_hap, batch.kept_site, n_hap, other == "aligned")
        runs = [execute_generated(eng, go, aligned_layout=(other == "aligned")) for _ in range(3 + min(args.steps, 20))][3:]
        o_group, o_copy = float(np.mean([r[0] for r in runs])), float(np.mean([r[1] for r in runs]))
        # its records must be the primary layout's records (which the oracle checked): first and last haplotype
        rec_ok = True
        o_base = dc.read(go.batch.out_base, n_hap + 1, np.uint64)
        rows_of = lambda h: np.searchsorted(batch.ann_hap, [h, h + 1])
        for h in (0, n_hap - 1):
            lo, hi = rows_of(h)
            o_s = dc.read(go.ann_start + 8 * int(lo), int(hi - lo), np.uint64)
            o_e = dc.read(go.ann_end + 8 * int(lo), int(hi - lo), np.uint64)
            o_tape = dc.read(go.batch.out + int(o_base[h]), int(o_base[h + 1] - o_base[h]), np.uint8)
            p_tape = d_out[int(batch.out_base[h]):int(batch.out_base[h + 1])].cpu().numpy()
            for r in range(int(hi - lo)):
                a, b_ = p_tape[int(batch.ann_start[lo + r]):int(batch.ann_end[lo + r])], o_tape[int(o_s[r]):int(o_e[r])]
                rec_ok = rec_ok and a.shape == b_.shape and bool((a == b_).all())
        n_alg_o = int(go.batch.n_out) + n_res + 16 * int(go.batch.n_tasks)  # written + read + tasks (SURVEY 8d)
        other_line = {"layout": other, "value": n_res / (o_group * 1e-3), "ms_per_step": o_group, "kernel_ms": o_copy,
                      "alg_gbs_kernel": n_alg_o / (o_copy * 1e-3) / 1e9, "result_tape_bytes": int(go.batch.n_out),
                      "records_equal_primary_layout": bool(rec_ok),
                      "what": "same cohort, Task batch generated on the device in the other layout (v2p_generate_tasks) and "
                              "executed in place; per-call CUDA events, %d calls" % len(runs)}
        # ---- the general catalogue (every instruction code; one thread per transcript) on the same lists
        dg = DeviceCatalogue.from_instructions(*C.instruction_arrays(prot, cat), device=local_rank)
        sb_all = np.zeros(n_hap + 1, np.uint64)
        np.cumsum(np.bincount(batch.kept_hap, minlength=n_hap), out=sb_all[1:])
        dg.generate_lists(sb_all, batch.kept_site)  # warm-up (allocations)
        gg = dg.generate_lists(sb_all, batch.kept_site)
        g_same = int(gg.batch.n_tasks) == (n_tasks if args.layout == "packed" else int(go.batch.n_tasks))
        if args.layout == "packed":
            m = min(n_tasks, 1 << 22)
            g_same = (g_same and int(gg.batch.n_out) == n_out and
                      bool(np.array_equal(dg.read(gg.batch.tasks, 4 * m, np.uint32).reshape(-1, 4), batch.tasks[:m])) and
                      bool(np.array_equal(dg.read(gg.batch.tasks + 16 * (n_tasks - m), 4 * m, np.uint32).reshape(-1, 4), batch.tasks[n_tasks - m:])) and
                      bool(np.array_equal(dg.read(gg.batch.out_base, n_hap + 1, np.uint64), batch.out_base)))
        taskgen["general_catalogue"] = {"gen_ms": gg.gen_ms, "tasks_per_s": int(gg.batch.n_tasks) / (gg.gen_ms * 1e-3),
                                        "equals_host_producer": bool(g_same), "skipped_transcripts": int(gg.n_skipped),
                                        "what": "v2p_catalogue_create_ins + v2p_generate_tasks: the reference's Instruction values, "
                                                "all 22 codes' rules, one thread per transcript-on-haplotype (packed layout)"}
        dg.close()
        # ---- SURVEY 8f rank 3: FORMAT/BCSQ bit-mask matrix -> per-haplotype site lists -> Task batch, on the device
        md_samples = min(n_hap // 2, args.maskdecode_samples)
        if md_samples > 0:
            sel = batch.kept_hap < 2 * md_samples
            mh, ms_ = batch.kept_hap[sel], batch.kept_site[sel]
            rec = C.make_records(cat, 0x5EED0009, 1)
            masks = C.encode_masks(rec, md_samples, mh, ms_)
            d_masks = torch.from_numpy(masks.view(np.int32)).to(dev)
            shape = masks.shape
            lst = dc.sites_from_masks(masks, rec.csq_begin, rec.csq_site)  # host matrix: pageable H2D inside decode_ms
            host_ms = lst.decode_ms
            dc.sites_from_masks(d_masks.data_ptr(), rec.csq_begin, rec.csq_site, shape)
            lst = dc.sites_from_masks(d_masks.data_ptr(), rec.csq_begin, rec.csq_site, shape)
            want_begin = np.zeros(2 * md_samples + 1, np.uint64)
            np.cumsum(np.bincount(mh, minlength=2 * md_samples), out=want_begin[1:])
            ok = (lst.n_sites == len(ms_) and bool(np.array_equal(dc.read(lst.sites, lst.n_sites, np.uint32), ms_.astype(np.uint32)))
                  and bool(np.array_equal(dc.read(lst.site_begin, 2 * md_samples + 1, np.uint64), want_begin)))
            g2 = dc.generate_from_lists(lst, args.layout == "aligned")
            n_t2 = int(batch.task_begin[2 * md_samples])
            ok = ok and g2.batch.n_tasks == n_t2 and bool(np.array_equal(
                dc.read(g2.batch.tasks, 4 * min(n_t2, 1 << 20), np.uint32).reshape(-1, 4), batch.tasks[: min(n_t2, 1 << 20)]))
            cells = shape[0] * shape[1]
            taskgen["maskdecode"] = {
                "records": int(shape[0]), "samples": int(md_samples), "words_per_cell": int(shape[2]), "carrier_bits": int(len(ms_)),
                "decode_ms": lst.decode_ms, "cells_per_s": cells / (lst.decode_ms * 1e-3),
                "matrix_gbs": masks.nbytes * 2 / (lst.decode_ms * 1e-3) / 1e9, "decode_ms_from_pageable_host": host_ms,
                "then_generate_ms": g2.gen_ms, "equals_host_lists_and_tasks": ok,
                "what": "v2p_sites_from_masks (matrix resident in HBM; streamed twice) -> v2p_generate_tasks_from_lists"}
            del d_masks
        dc.close()

    # ---- the literal drop-in (gir.rs:236-239 replacement), called like the reference calls it: many threads, one haplotype each
    dropin_line = None
    if world == 1 and args.dropin_haps > 0 and not args.no_cpu_baseline:
        dropin_line = dropin_measure(args, eng, prot, cat, args.dropin_haps)

    # ---- SURVEY 8f rank 4: the -c path.  FASTA image in HBM -> one .fasta.gz per sample, compressed on the device
    gzip_line = None
    if world == 1 and args.gzip_samples > 0 and not args.no_registered_ref:
        gzip_line = gzip_measure(args, prot, cat, eng, dev, local_rank, torch)

    copy_avg_ms = float(np.mean(copy_ms))
    achieved = b_alg / (copy_avg_ms * 1e-3) / 1e9
    # the kernel must WRITE every residue once: this GPU's write-only ceiling, measured live with the repo's own store-only
    # kernels (cudaMemsetAsync; TMA bulk stores of 8 KiB tiles -- the copy kernel's own store) over the result buffer
    from synth import devgen

    torch.cuda.synchronize()
    ceil = devgen.store_ceiling_gbs(local_rank, d_out.data_ptr(), min(n_out, 16 << 30))
    write_peak = ceil["tma_bulk_store_8k"]
    write_rate = n_out / (copy_avg_ms * 1e-3) / 1e9
    value = total_res / (ms_per_step * 1e-3)  # every rank holds its own same-sized sample range (weak scaling)
    line = {
        "metric": "generated residues/sec", "value": value, "unit": "residues/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "%s: %d phased samples/GPU (%d haplotypes) x 20k-transcript proteome (%d residues), "
                               "%s csq mix" % (args.workload, args.samples, n_hap, len(batch.ref),
                                               "missense-dominated" if args.workload == "c2" else "skewed frameshift/insertion"),
                   "haplotypes_per_gpu": n_hap, "tasks_per_gpu": n_tasks, "residues_per_gpu": n_res, "result_tape_bytes_per_gpu": n_out,
                   "mean_task_bytes": n_res / max(n_tasks, 1), "l2_policy": "inputs_larger_than_l2 (output %.1f GB, tasks %.2f GB "
                   "per step; the %.1f MB proteome is L2-resident by design)" % (n_out / 1e9, n_tasks * 16 / 1e9, len(batch.ref) / 1e6),
                   "tile_variant": args.variant, "layout": args.layout,
                   "tile_order": "tape (V2P_FLAG_ALIGNED_LAYOUT)" if args.layout == "aligned" else "haplotype-interleaved", "fasta_image": bool(args.fasta_image), "reference_tape": "caller-supplied per call" if args.no_registered_ref else
                   "registered once (v2p_engine_set_reference, mode %s)" % args.ref_mode, "parallelism": "sample-sharded x%d, no collective" % world},
        "haplotypes_per_s": total_haps / (ms_per_step * 1e-3),
        "alg_gbs": total_alg / (ms_per_step * 1e-3) / 1e9,
        "clocks": clocks,
        "e2e": {"value": total_res * args.e2e_steps / e2e_s, "unit": "residues/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": n_out, "steps": args.e2e_steps, "chunk_haplotypes": args.e2e_chunk_haps,
                "chunks_in_flight": depth,
                "api": "v2p_execute_batch (host pointers, pinned, ASYNC), one call per chunk",
                "what": "raw result tapes: 1 byte per residue must cross PCIe, and one GPU's link delivers 53-56 GB/s to the host "
                        "whatever moves the bytes (profiles/r2/pcie_probe_2gpu.jsonl: copy engine, several streams, write-combined or "
                        "registered huge pages, SM zero-copy stores)",
                "fasta": None if not pipeline_line else {k: pipeline_line["fasta"][k] for k in ("residues_per_s", "h2d_bytes", "d2h_bytes")},
                "fasta_gz": None if not pipeline_line else {k: pipeline_line["fasta_gz"][k] for k in ("residues_per_s", "h2d_bytes", "d2h_bytes")},
                "fasta_note": "the same cohort as .fasta / .fasta.gz FILE IMAGES through v2p_pipeline_run_lists (site lists up, file bytes "
                              "down; the reference's -c flag): compressing on the device is the one lever on a PCIe-bound result"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_note": traffic_note, "kernel": "k_copy_tiles", "peak_source": peak_src,
                     "dram_gbs": None if traffic is None else traffic / (copy_avg_ms * 1e-3) / 1e9,
                     "dram_frac": None if traffic is None else traffic / (copy_avg_ms * 1e-3) / 1e9 / peak,
                     "dram_note": "what DRAM itself moved (ncu dram__bytes_read + dram__bytes_write per launch) / live kernel time / "
                                  "peak: the source tape is L2-resident, so `frac` (algorithmic bytes, SURVEY 8d) counts ~20 GB of "
                                  "L2 hits per launch that never reach DRAM",
                     "alg_bytes_per_launch": b_alg, "kernel_ms": copy_avg_ms, "launch_group_ms": float(np.mean(group_ms)),
                     "kernel_share_of_step": copy_avg_ms / ms_per_step,
                     "write_only": {"achieved_gbs": write_rate, "peak_gbs": write_peak, "frac": write_rate / write_peak,
                                    "ceilings_gbs": ceil,
                                    "note": "result-tape bytes written / kernel time vs a store-only kernel on the same GPU and buffer "
                                            "(TMA bulk stores of 8 KiB tiles, the copy kernel's own store instruction and grid); the hard "
                                            "floor of this path is one DRAM write per residue"}},
        "load_balance": skew, "cpu_baseline": cpu, "parity": parity, "c3": c3_line, "dropin": dropin_line, "other_layout": other_line, "taskgen": taskgen, "gzip": gzip_line, "pipeline": pipeline_line, "gen_seconds": round(t_gen, 1),
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_reference_arm(args):
    """Reference arm: the reference's CPU implementation of the path on this box's host cores."""
    threads = os.cpu_count() or 1
    nh = args.cpu_sample_haps
    prot, cat, batch = make_workload(args.workload, max(1, (nh + 1) // 2), 0)
    steps = max(1, args.steps)
    rates = []
    # each step = one bounded pass budget; keep the whole run within a few minutes
    per_step = min(args.cpu_seconds, max(1.0, 120.0 / (steps + max(args.warmup, 0))))
    for i in range(max(args.warmup, 0) + steps):
        rate, el, reps, nhh, nres, _ = cpu_engine_rate(batch, prot, nh, per_step, threads, 4)
        if i >= args.warmup:
            rates.append(rate)
    value = float(np.mean(rates))
    cpu = {"value": value, "unit": "residues/s", "cores": threads, "kind": "port",
           "sample": "%d haplotypes (%d residues) of the %s cohort, UTF-32 tapes (gir.rs:18-22), haplotypes over %d "
                     "threads (exec.rs:34-40); the Rust reference cannot be compiled in this image" %
                     (nhh, nres, args.workload, threads)}
    rb = reference_binary_rate(prot, cat, batch, args.ref_binary_samples or min(32, batch.n_hap // 2))
    if rb:
        cpu["reference_binary"] = rb
    line = {"impl": "reference", "metric": "generated residues/sec", "value": value, "unit": "residues/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": nres / value * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 (Rust char)",
            "data": "synthetic",
            "config": {"workload": "%s: bounded sample of %d haplotypes of the same synthetic cohort" % (args.workload, nhh)},
            "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": "residues/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
