"""GPU suite (-m gpu): the serial-order path (haplotypes whose tasks are unsorted or overlap) against the oracle.

That path is decided on the host after the plan: plan_one flags the haplotype, k_plan_fix compacts the flagged ones
into a list, and k_serial runs when the call is waited.  Every result here is compared with oracle/ref_engine.c:
whole tapes byte for byte, errors as the whole (status, bad_hap, bad_task) triple.
  A. the contiguity validator (V2P_FLAG_VALIDATE) on unsorted input, through every batch entry and the SoA entry;
  B. device-pointer launches in flight together, with each other, with synchronous calls and with host-pointer calls;
  C. k_serial at span and tile edges, long later-wins chains, strided span loops, thousands of flagged haplotypes,
     neighbour layouts and every source mode (tests/serialgen.py);
  D. the UTF-32 SoA entry over several spans, with and without the '.' fill.
"""
import numpy as np
import pytest

from oracle import cengine
from tests import serialgen as G
from tests.randtasks import random_batch
from tests.test_gpu_parity import gpu_batch, oracle_batch
from vcf2prot_b200 import EngineError, GpuEngine
from vcf2prot_b200 import _lib as L

pytestmark = pytest.mark.gpu

ABI = {cengine.REF_OK: L.V2P_OK, cengine.REF_ERR_RES_OOB: L.ERR_RES_OOB, cengine.REF_ERR_SRC_OOB: L.ERR_SRC_OOB,
       cengine.REF_ERR_BAD_STREAM: L.ERR_BAD_STREAM, cengine.REF_ERR_NOT_CONTIGUOUS: L.ERR_NOT_CONTIGUOUS}


def expected(b, validate):
    st, bh, bi, out = oracle_batch(b, validate=validate)
    return (ABI[st], bh, bi), (out if st == cengine.REF_OK else None)


def triple(fn):
    """(status, bad_hap, bad_task) of a call that returns normally (V2P_OK) or raises EngineError."""
    try:
        fn()
        return (L.V2P_OK, 0, 0)
    except EngineError as e:
        return (e.status, e.bad_hap, e.bad_task)


def with_hap(b, h, rows):
    """b with haplotype h's tasks replaced by `rows` (task_begin follows)."""
    tb = b["task_begin"].astype(np.int64)
    rows = np.asarray(rows, np.uint32).reshape(-1, 4)
    out = dict(b)
    out["tasks"] = np.concatenate([b["tasks"][:tb[h]], rows, b["tasks"][tb[h + 1]:]])
    d = len(rows) - (tb[h + 1] - tb[h])
    out["task_begin"] = np.concatenate([tb[:h + 1], tb[h + 1:] + d]).astype(np.uint64)
    return out


def hap_rows(b, h):
    tb = b["task_begin"]
    return b["tasks"][int(tb[h]):int(tb[h + 1])].copy()


def sub_batch(b, h0, h1):
    """Haplotypes [h0, h1) of b as a batch of their own (bases rebased), for the oracle of a hap-range call."""
    rb = lambda a: (a[h0:h1 + 1] - a[h0]).astype(np.uint64)
    tb = b["task_begin"]
    return dict(task_begin=rb(tb), tasks=b["tasks"][int(tb[h0]):int(tb[h1])], ref=b["ref"],
                alt=b["alt"][int(b["alt_base"][h0]):int(b["alt_base"][h1])], alt_base=rb(b["alt_base"]),
                out_base=rb(b["out_base"]), ref_base=None)


def torch_up(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to("cuda:0")


class Dev:
    """A batch resident on the device, with an output tape prefilled with 'U' (so the '.' fill is checked too)."""

    def __init__(self, b):
        import torch

        self.b = b
        self.d = {k: torch_up(b[k]) for k in ("task_begin", "tasks", "ref", "alt", "alt_base", "out_base")}
        self.n_out = int(b["out_base"][-1])
        self.out = torch.full((self.n_out + 16,), ord("U"), dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()

    def launch(self, eng, wait=True, validate=False):
        d = self.d
        return eng.execute_batch_device(len(self.b["task_begin"]) - 1, d["task_begin"], d["tasks"], d["ref"], d["alt"],
                                        d["alt_base"], self.out, d["out_base"], len(self.b["tasks"]), len(self.b["alt"]),
                                        self.n_out, validate=validate, wait=wait)

    def got(self):
        return self.out[:self.n_out].cpu().numpy()


def run_entries(eng, b, validate, h0=1):
    """The batch through host pointers, a hap-range call over [h0, n_hap) (nonzero origins) and device pointers:
    each gives the oracle's triple, and the oracle's bytes when that is V2P_OK."""
    n_hap = len(b["task_begin"]) - 1
    want, tape = expected(b, validate)
    got = {}
    out = {}
    got["host"] = triple(lambda: out.__setitem__("host", gpu_batch(eng, b, validate=validate)[0]))
    sub = sub_batch(b, h0, n_hap)
    want_sub, tape_sub = expected(sub, validate)
    o0, o1 = int(b["out_base"][h0]), int(b["out_base"][n_hap])
    chunk = np.full(o1 - o0 + 16, ord("U"), np.uint8)
    got["range"] = triple(lambda: eng.execute_hap_range(h0, n_hap, b["task_begin"], b["tasks"], b["ref"], b["alt"],
                                                        b["alt_base"], b["out_base"], chunk, validate=validate))
    dev = Dev(b)
    got["device"] = triple(lambda: dev.launch(eng, validate=validate))
    assert got == {"host": want, "range": want_sub, "device": want}
    if tape is not None:
        assert np.array_equal(out["host"], tape) and np.array_equal(dev.got(), tape)
    if tape_sub is not None:
        assert np.array_equal(chunk[:o1 - o0], tape_sub)
    return want


# ---------------------------------------------------------------------------------------------- A. VALIDATE
BASE_A = dict(seed=1201, n_hap=9, mean_res=30_000)


@pytest.fixture(scope="module")
def base_a():
    b = random_batch(BASE_A["seed"], BASE_A["n_hap"], BASE_A["mean_res"], gap_prob=0.0, empty_hap_prob=0.0,
                     len_mix=(0.4, 0.4, 0.2, 0.0))
    assert expected(b, True)[0] == (L.V2P_OK, 0, 0) and len(G.flagged(b)) == 0
    return b


def _end(r, k):
    return int(r[k, 2]) + int(r[k, 1])


def _pick(r, need_len=3, lo=2):
    """A task index k >= lo whose predecessor has at least need_len bytes and whose own slice can move back."""
    return next(k for k in range(lo, len(r) - 4) if int(r[k - 1, 1]) >= need_len and int(r[k, 1]) >= 1)


def case_overlap1(r, k):
    r[k, 2] -= 1
    return r


def case_duplicate(r, k):
    return np.insert(r, k, r[k - 1], axis=0)


def case_back_to_zero(r, k):
    r[k, 2] = 0
    return r


def case_zero_len_back(r, k):
    return np.insert(r, k, (0, 0, _end(r, k - 1) - 1, 0), axis=0)


def case_contained(r, k):
    p = r[k - 1]
    return np.insert(r, k, (int(p[0]) + 1, int(p[1]) - 2, int(p[2]) + 1, int(p[3])), axis=0)


EDITS = {"overlap_1_byte": case_overlap1, "duplicate": case_duplicate, "back_to_dst_0": case_back_to_zero,
         "zero_length_before_end": case_zero_len_back, "contained_rewrite": case_contained}


@pytest.mark.parametrize("name", list(EDITS))
def test_validate_rejects_every_backward_task(gpu_engine, base_a, name):
    h = 4
    r = hap_rows(base_a, h)
    k = _pick(r)
    b = with_hap(base_a, h, EDITS[name](r, k))
    assert list(G.flagged(b)) == [h]
    assert run_entries(gpu_engine, b, True) == (L.ERR_NOT_CONTIGUOUS, h, k)
    assert run_entries(gpu_engine, b, False)[0] == L.V2P_OK  # without VALIDATE: serial order, the oracle's bytes
    soa_matches_oracle(gpu_engine, b, h)


@pytest.mark.parametrize("lane", [511, 512])
def test_validate_at_a_plan_warp_boundary(gpu_engine, base_a, lane):
    """The disorder at global task 512m - 1 (last lane of a k_plan_tasks warp) or 512m (first lane of the next warp,
    whose predecessor reaches it from the other warp)."""
    tb = base_a["task_begin"].astype(np.int64)
    for g in range(lane, int(tb[-1]), G.PLAN_WARP_TASKS):
        h = int(np.searchsorted(tb, g, side="right") - 1)
        k = g - int(tb[h])
        if h >= 2 and 1 <= k < tb[h + 1] - tb[h] and int(base_a["tasks"][g - 1, 1]) >= 1:
            break
    else:
        pytest.fail("no plan warp boundary inside a haplotype")
    assert (int(tb[h]) + k) % G.PLAN_WARP_TASKS == lane % G.PLAN_WARP_TASKS
    b = with_hap(base_a, h, case_overlap1(hap_rows(base_a, h), k))
    assert run_entries(gpu_engine, b, True) == (L.ERR_NOT_CONTIGUOUS, h, k)
    run_entries(gpu_engine, b, False)


def test_first_task_of_a_haplotype_is_not_judged_against_the_previous_one(gpu_engine, base_a):
    """Haplotype h starts with a 1-byte '.' gap: legal, whatever the previous haplotype's last task covered."""
    h = next(h for h in range(2, BASE_A["n_hap"]) if int(hap_rows(base_a, h)[0, 1]) >= 2)
    r = hap_rows(base_a, h)
    r[0, 2] += 1
    r[0, 1] -= 1
    b = with_hap(base_a, h, r)
    assert len(G.flagged(b)) == 0
    assert run_entries(gpu_engine, b, True) == (L.V2P_OK, 0, 0)


def test_validate_precedence_with_other_findings(gpu_engine, base_a):
    h = 4
    r = hap_rows(base_a, h)
    k = _pick(r)
    # a bad stream code later in the same haplotype: the Task array build panics first
    r1 = case_overlap1(r.copy(), k)
    r1[k + 3, 3] = 2
    assert run_entries(gpu_engine, with_hap(base_a, h, r1), True) == (L.ERR_BAD_STREAM, h, k + 3)
    # a slice error in an earlier haplotype (a source offset: a length would also break contiguity): it fails first
    b = with_hap(base_a, h, case_overlap1(r.copy(), k))
    b["tasks"] = b["tasks"].copy()
    b["tasks"][int(b["task_begin"][h - 1]) + 1, 0] = 0x7FFFFF00
    assert run_entries(gpu_engine, b, True) == (L.ERR_SRC_OOB, h - 1, 1)
    # a forward gap later in the same haplotype: the backward task is the first offender
    r3 = case_overlap1(r.copy(), k)
    j = next(i for i in range(k + 2, len(r3)) if int(r3[i, 1]) >= 1)
    r3[j, 2] += 1  # (task j gives up its first byte: a '.' gap in front of it)
    r3[j, 1] -= 1
    assert run_entries(gpu_engine, with_hap(base_a, h, r3), True) == (L.ERR_NOT_CONTIGUOUS, h, k)
    # a backward task whose own slice is out of range: the validator runs before any slice is taken
    r4 = case_overlap1(r.copy(), k)
    r4[k, 0] = 0x7FFFFF00
    assert run_entries(gpu_engine, with_hap(base_a, h, r4), True) == (L.ERR_NOT_CONTIGUOUS, h, k)
    for rows in (r1, r3, r4):  # the single-haplotype cases through the SoA entry
        soa_matches_oracle(gpu_engine, with_hap(base_a, h, rows), h)


def test_validate_small_literals(gpu_engine):
    """(0,10),(5,3) overlaps at task 1; in (0,10),(3,0),(10,5) the zero-length task is the offender, not the next one."""
    u = lambda *a: np.asarray(a, np.uint64)
    ref = np.frombuffer(b"ABCDEFGHIJKLMNOPQRSTUVWXYZ", np.uint8).copy()
    for rows, want_task in (([(0, 10, 0, 0), (20, 3, 5, 0)], 1), ([(0, 10, 0, 0), (0, 0, 3, 0), (10, 5, 10, 0)], 1)):
        rows = np.asarray(rows, np.uint32)
        n = len(rows)
        # haplotype 0 is sorted, haplotype 1 carries the case (so the hap-range call starts at a nonzero origin)
        b = dict(task_begin=u(0, 1, 1 + n), tasks=np.concatenate([np.asarray([(0, 7, 0, 0)], np.uint32), rows]), ref=ref,
                 alt=np.zeros(0, np.uint8), alt_base=u(0, 0, 0), out_base=u(0, 7, 7 + 15), ref_base=None)
        assert run_entries(gpu_engine, b, True) == (L.ERR_NOT_CONTIGUOUS, 1, want_task)
        run_entries(gpu_engine, b, False)
        soa_matches_oracle(gpu_engine, b, 1)


@pytest.mark.parametrize("where", ["middle", "last"])
@pytest.mark.parametrize("col,value", [(1, 0x7FFFFF00), (2, 0x7FFFFF00)], ids=["bad_source", "bad_result"])
def test_soa_validate_keeps_slice_errors_of_contiguous_tasks(gpu_engine, base_a, where, col, value):
    """A contiguous Task array whose task k has a bad source or result slice: the validator passes, the slice panics
    at k.  (k_soa_pack zeroes a rejected task; the plan must not take that for a contiguity break.)"""
    r = hap_rows(base_a, 4)
    tasks = [[int(t[3]), int(t[0]), int(t[1]), int(t[2])] for t in r]
    k = len(tasks) // 2 if where == "middle" else len(tasks) - 1
    tasks[k][col] = value if col == 1 else tasks[k][1]
    if col == 2:  # a length past the tape's end that keeps the array contiguous: the next task starts behind it
        tasks[k][2] = value
        for t in tasks[k + 1:]:
            t[3] += value - int(r[k, 1])
    ref = base_a["ref"].astype(np.uint32)
    alt = base_a["alt"][int(base_a["alt_base"][4]):int(base_a["alt_base"][5])].astype(np.uint32)
    n_res = int(base_a["out_base"][5] - base_a["out_base"][4])
    st, bad = cengine.gir_execute(tasks, ref, alt, np.zeros(n_res, np.uint32), True, validate=True)
    assert (st, bad) == ({1: cengine.REF_ERR_SRC_OOB, 2: cengine.REF_ERR_RES_OOB}[col], k)
    assert triple(lambda: gpu_engine.execute_soa(tasks, ref, alt, n_res, fill_dot=True, validate=True)) == (ABI[st], 0, k)


def soa_matches_oracle(eng, b, h, validate=True):
    """Haplotype h alone through the SoA entry (v2p_gir_execute): the oracle's (status, index), or its tape."""
    r = hap_rows(b, h)
    tasks = [(int(t[3]), int(t[0]), int(t[1]), int(t[2])) for t in r]
    ref = b["ref"].astype(np.uint32)
    alt = b["alt"][int(b["alt_base"][h]):int(b["alt_base"][h + 1])].astype(np.uint32)
    n_res = int(b["out_base"][h + 1] - b["out_base"][h])
    want = np.zeros(n_res, np.uint32)
    st, bad = cengine.gir_execute(tasks, ref, alt, want, True, validate=validate)
    got = {}
    t = triple(lambda: got.__setitem__("res", eng.execute_soa(tasks, ref, alt, n_res, fill_dot=True, validate=validate)))
    assert (t[0], t[2]) == (ABI[st], bad if st else 0)
    if st == cengine.REF_OK:
        assert np.array_equal(got["res"], want)


# ---------------------------------------------------------------------------------------------- B. in flight
N_B = 24


def unsorted_variant(seed, haps=None, n=3):
    """random_batch with the tasks of some haplotypes reversed (given, or n chosen among those with >= 3 tasks)."""
    b = random_batch(seed, N_B, 8000, empty_hap_prob=0.0)
    b["tasks"] = b["tasks"].copy()
    tb = b["task_begin"]
    if haps is None:
        roomy = [h for h in range(N_B) if int(tb[h + 1] - tb[h]) >= 3]
        haps = sorted(np.random.default_rng(seed).choice(roomy, n, replace=False).tolist())
    for h in haps:
        s, e = int(tb[h]), int(tb[h + 1])
        b["tasks"][s:e] = b["tasks"][s:e][::-1]
    assert list(G.flagged(b)) == list(haps), (seed, haps)
    return b


N_SETS = (2, 4, 3, 5)  # flagged haplotypes per batch: different sets of different sizes


@pytest.fixture(scope="module")
def warm_engine():
    """An engine of its own whose device-pointer scratch already holds more than any batch of group B needs (so
    that a later launch never regrows it: see test_growth_while_in_flight for that)."""
    eng = GpuEngine(0)
    big = random_batch(1299, 4 * N_B, 20_000, empty_hap_prob=0.0)
    Dev(big).launch(eng)
    yield eng
    eng.close()


@pytest.fixture(scope="module")
def batches_b():
    bs = [unsorted_variant(1300 + i, n=n) for i, n in enumerate(N_SETS)]
    return [(b, expected(b, False)[1]) for b in bs]


@pytest.fixture(params=["engine_stream", "caller_stream"])
def stream(request, warm_engine):
    import torch

    if request.param == "caller_stream":
        side = torch.cuda.Stream()
        warm_engine.set_stream(side.cuda_stream)
        yield side
        warm_engine.set_stream(None)
    else:
        yield None


@pytest.mark.parametrize("order", ["launch_order", "reverse_order"])
@pytest.mark.parametrize("n", [2, 3])
def test_device_launches_in_flight(warm_engine, batches_b, stream, n, order):
    devs = [Dev(b) for b, _ in batches_b[:n]]
    evs = [d.launch(warm_engine, wait=False) for d in devs]
    idx = list(range(n)) if order == "launch_order" else list(range(n))[::-1]
    for i in idx:
        warm_engine.wait_event(evs[i])
    for d, (_, want) in zip(devs, batches_b):
        assert np.array_equal(d.got(), want)


def test_async_then_sync_then_wait(warm_engine, batches_b):
    a, s = Dev(batches_b[0][0]), Dev(batches_b[1][0])
    ev = a.launch(warm_engine, wait=False)
    s.launch(warm_engine)
    assert np.array_equal(s.got(), batches_b[1][1])
    warm_engine.wait_event(ev)
    assert np.array_equal(a.got(), batches_b[0][1])


def test_device_and_host_launches_interleaved(warm_engine, batches_b):
    """Device-pointer async launches between host-pointer async hap-range calls on all three staging slots; every
    host chunk needs the serial kernel, so its wait repeats the copy-back."""
    hb = unsorted_variant(1310, (0, 10, 19, 22))
    want = expected(hb, False)[1]
    chunks = [(0, 8), (8, 16), (16, 24)]
    assert all(any(a <= h < z for h in G.flagged(hb)) for a, z in chunks)
    bufs = [np.full(int(hb["out_base"][z] - hb["out_base"][a]) + 16, ord("U"), np.uint8) for a, z in chunks]
    devs = [Dev(b) for b, _ in batches_b[:3]]
    rng_call = lambda i: warm_engine.execute_hap_range(chunks[i][0], chunks[i][1], hb["task_begin"], hb["tasks"], hb["ref"],
                                                       hb["alt"], hb["alt_base"], hb["out_base"], bufs[i], wait=False)
    evs = [("d0", devs[0].launch(warm_engine, wait=False)), ("h0", rng_call(0)), ("d1", devs[1].launch(warm_engine, wait=False)),
           ("h1", rng_call(1)), ("h2", rng_call(2)), ("d2", devs[2].launch(warm_engine, wait=False))]
    for name, ev in evs[::2] + evs[1::2]:
        warm_engine.wait_event(ev)
    for d, (_, w) in zip(devs, batches_b):
        assert np.array_equal(d.got(), w)
    for (a, z), buf in zip(chunks, bufs):
        o0, o1 = int(hb["out_base"][a]), int(hb["out_base"][z])
        assert np.array_equal(buf[:o1 - o0], want[o0:o1]), (a, z)


def test_failing_batch_between_good_ones(warm_engine, batches_b, stream):
    bad = dict(batches_b[1][0])
    h = int(G.flagged(bad)[-1])  # a stream code breaks the last flagged haplotype; the others stay flagged
    bad["tasks"] = bad["tasks"].copy()
    bad["tasks"][int(bad["task_begin"][h]) + 2, 3] = 5
    want_bad, _ = expected(bad, False)
    assert want_bad == (L.ERR_BAD_STREAM, h, 2) and len(G.flagged(bad)) == 4
    devs = [Dev(batches_b[0][0]), Dev(bad), Dev(batches_b[2][0])]
    evs = [d.launch(warm_engine, wait=False) for d in devs]
    warm_engine.wait_event(evs[0])
    assert triple(lambda: warm_engine.wait_event(evs[1])) == want_bad
    warm_engine.wait_event(evs[2])
    assert np.array_equal(devs[0].got(), batches_b[0][1]) and np.array_equal(devs[2].got(), batches_b[2][1])


def test_growth_while_in_flight():
    """A later launch larger than anything the engine ran before (its scratch grows) while the first one still has
    its serial kernel to run at the wait."""
    with GpuEngine(0) as eng:
        small = unsorted_variant(1320, n=2)
        big = random_batch(1321, 16 * N_B, 8000, empty_hap_prob=0.0)
        big["tasks"] = big["tasks"].copy()
        tb = big["task_begin"]
        for h in range(0, 16 * N_B, 5):
            s, e = int(tb[h]), int(tb[h + 1])
            big["tasks"][s:e] = big["tasks"][s:e][::-1]
        assert len(G.flagged(big)) > len(G.flagged(small))
        a, z = Dev(small), Dev(big)
        ev_a = a.launch(eng, wait=False)
        ev_z = z.launch(eng, wait=False)
        eng.wait_event(ev_a)
        eng.wait_event(ev_z)
        assert np.array_equal(a.got(), expected(small, False)[1])
        assert np.array_equal(z.got(), expected(big, False)[1])


# ---------------------------------------------------------------------------------------------- C. k_serial shapes
def bytes_match(eng, b, device=False):
    assert len(b["serial"]) and np.array_equal(G.flagged(b), b["serial"])
    _, want = expected(b, False)
    out, _ = gpu_batch(eng, b)
    assert np.array_equal(out, want)
    if device:
        d = Dev(b)
        d.launch(eng)
        assert np.array_equal(d.got(), want)
    return want


@pytest.fixture
def tuned(gpu_engine):
    yield gpu_engine
    gpu_engine.set_tuning(-1, 0)


def edges_on_launch_edges(b, edge):
    """Every flagged tape starts on a multiple of `edge` of the launch's output (tiles count from there)."""
    assert (b["out_base"][b["serial"]].astype(np.int64) % edge == 0).all()
    return b


def test_span_edges(gpu_engine):
    bytes_match(gpu_engine, edges_on_launch_edges(G.edge_batch(G.SPAN, 1), G.SPAN), device=True)


@pytest.mark.parametrize("tile,variant", [(8192, 8), (4096, 5), (2048, 6)])
def test_tile_edges(tuned, tile, variant):
    tuned.set_tuning(variant, 0)
    bytes_match(tuned, edges_on_launch_edges(G.edge_batch(tile, {8192: 2, 4096: 3, 2048: 4}[tile]), tile))


@pytest.mark.parametrize("variant", [-1, 6, 8])
def test_one_byte_overlaps_keep_array_order(tuned, variant):
    """Without VALIDATE: every task overlaps the one in front of it by exactly one byte, which the later task must win."""
    tuned.set_tuning(variant, 0)
    bytes_match(tuned, G.one_byte_overlap_batch(12), device=True)


def test_task_straddling_a_span_edge_at_every_offset(gpu_engine):
    bytes_match(gpu_engine, G.straddle_batch(5))


def test_later_wins_chain_longer_than_a_window(gpu_engine):
    b = G.chain_batch(6)
    h = int(b["serial"][0])
    assert int(b["task_begin"][h + 1] - b["task_begin"][h]) > 2 * G.SERIAL_THREADS
    bytes_match(gpu_engine, b, device=True)


def test_span_loop_strides_over_the_grid(gpu_engine):
    import torch

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    b = G.strided_batch(7, sms)
    assert int(np.diff(b["out_base"].astype(np.int64)).max()) > 4 * sms * G.SPAN
    bytes_match(gpu_engine, b, device=True)


def test_thousands_of_small_flagged_haplotypes(gpu_engine):
    b = G.many_small_batch(8)
    assert len(b["serial"]) >= 2000
    bytes_match(gpu_engine, b, device=True)


@pytest.mark.parametrize("variant", [-1, 6, 8])
@pytest.mark.parametrize("layout", G.NEIGHBOUR_LAYOUTS)
def test_neighbour_layouts_inside_one_tile(tuned, layout, variant):
    tuned.set_tuning(variant, 0)
    bytes_match(tuned, G.neighbour_batch(layout, 10 + G.NEIGHBOUR_LAYOUTS.index(layout)))


def test_flagged_first_last_and_zero_length_only(gpu_engine):
    b = G.first_last_zero_batch(9)
    assert b["serial"][0] == 0 and b["serial"][-1] == len(b["task_begin"]) - 2
    bytes_match(gpu_engine, b, device=True)


@pytest.mark.parametrize("mode", ["caller_tape", "per_hap", "replicas", "plain"])
def test_every_source_mode(gpu_engine, mode):
    from synth import cohort as C

    prot = C.make_proteome(seed=41, n_tx=300, mu=5.5, sigma=0.7, hi=6000)
    cat = C.make_catalogue(prot, 6000, seed=42, mix=(0.7, 0.06, 0.06, 0.08, 0.04, 0.03, 0.03))
    cat.af[:] = 0.2
    sb = C.synth_batch(prot, cat, 30, 43, ref_mode="per_hap" if mode == "per_hap" else "global")
    b = dict(task_begin=sb.task_begin, tasks=sb.tasks.copy(), ref=sb.ref, alt=sb.alt, alt_base=sb.alt_base,
             out_base=sb.out_base, ref_base=sb.ref_base)
    tb = b["task_begin"]
    for h in (0, 3, 11, 29):
        s, e = int(tb[h]), int(tb[h + 1])
        b["tasks"][s:e] = b["tasks"][s:e][::-1]
    assert set(G.flagged(b)) == {0, 3, 11, 29}
    if mode == "per_hap":
        assert b["ref_base"] is not None and len(np.unique(b["ref_base"])) > 20
    _, want = expected(b, False)
    if mode in ("replicas", "plain"):
        gpu_engine.set_reference(b["ref"], mode)
        out, _ = gpu_engine.execute_batch(b["task_begin"], b["tasks"], None, b["alt"], b["alt_base"], b["out_base"])
    else:
        out, _ = gpu_batch(gpu_engine, b)
    assert np.array_equal(out, want)


# ---------------------------------------------------------------------------------------------- D. UTF-32 SoA
@pytest.mark.parametrize("fill_dot", [True, False])
def test_utf32_soa_unsorted_over_several_spans(gpu_engine, fill_dot):
    """Code points above 0xFF keep 4-byte units on the device: 20,000 residues are 5 spans.  Tasks reversed, with
    '.' gaps between them and rewrites across the span edges (4096 residues apart); without the fill the caller's
    residues in the gaps must survive."""
    rng = np.random.default_rng(77)
    n_res, unit_span = 20_000, G.SPAN // 4
    ref = rng.integers(0x4E00, 0x4F00, size=30_000).astype(np.uint32)
    ref[::5] = rng.integers(65, 91, size=len(ref[::5]))
    alt = rng.integers(0x3B1, 0x3C9, size=3000).astype(np.uint32)
    cuts = sorted({int(x) for x in rng.integers(1, n_res, 300)} | {unit_span * j + d for j in range(1, 5) for d in (-1, 0, 1)})
    edges = [0] + cuts + [n_res]
    tasks = []
    for a, c in zip(edges[:-1], edges[1:]):
        if rng.random() < 0.15:
            continue  # a gap nobody writes
        ln = c - a
        tasks.append((1, int(rng.integers(0, len(alt) - ln)), ln, a) if ln < 500 and rng.random() < 0.4
                     else (0, int(rng.integers(0, len(ref) - ln)), ln, a))
    tasks = tasks[::-1] + [(0, int(rng.integers(0, 20_000)), 40, unit_span * j - 20 + j) for j in range(1, 5)]
    res0 = rng.integers(0x1F300, 0x1F3FF, size=n_res).astype(np.uint32)
    want = np.zeros(n_res, np.uint32) if fill_dot else res0.copy()
    assert cengine.gir_execute(tasks, ref, alt, want, fill_dot)[0] == cengine.REF_OK
    got = gpu_engine.execute_soa(tasks, ref, alt, n_res if fill_dot else res0, fill_dot=fill_dot)
    assert np.array_equal(got, want)
    assert fill_dot or (got == res0).sum() > 100  # gaps kept the caller's residues
