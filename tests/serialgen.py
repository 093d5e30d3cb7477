"""Deterministic batches whose flagged haplotypes take the serial-order kernel (k_serial) at the shapes where it can
go wrong: span and tile edges, long later-wins chains, strided span loops, thousands of small flagged haplotypes,
neighbour layouts inside one tile.  Every builder returns a batch dict in the layout of randtasks.random_batch plus
`serial`, the haplotypes it claims the plan flags; tests/test_serialgen.py checks that claim against `flagged`."""
from __future__ import annotations

import numpy as np

SPAN = 16384          # kSerialSpan: bytes of one k_serial work item
SERIAL_THREADS = 512  # kSerialThreads: tasks judged per window of k_serial
PLAN_WARP_TASKS = 512  # kPlanWarpTasks: consecutive tasks per k_plan_tasks warp
EDGE_OFFSETS = (-17, -16, -1, 0, 1, 15, 16)


def flagged(b) -> np.ndarray:
    """The plan's rule (plan_one) restated: a haplotype takes the serial kernel when one of its tasks starts before
    the previous task of the same haplotype ends.  Returns the flagged haplotype indices."""
    tb = np.asarray(b["task_begin"], np.int64)
    t = np.asarray(b["tasks"], np.int64).reshape(-1, 4)
    early = np.zeros(len(t), bool)
    if len(t) > 1:
        early[1:] = t[1:, 2] < t[:-1, 2] + t[:-1, 1]
    early[tb[:-1][tb[:-1] < tb[1:]]] = False  # a haplotype's first task is not judged against the one in front
    hap = np.searchsorted(tb, np.arange(len(t)), side="right") - 1
    return np.unique(hap[early])


class Builder:
    """Haplotype after haplotype over one shared reference tape; each tape is cut into tasks that cover it."""

    def __init__(self, seed: int, n_ref: int = 70_000, n_alt: int = 4096):
        self.rng = np.random.default_rng(seed)
        self.ref = self.rng.integers(65, 91, size=n_ref, dtype=np.uint8)
        self.n_alt = n_alt
        self.rows, self.tb, self.ob, self.ab, self.alts, self.serial = [], [0], [0], [0], [], []

    @property
    def pos(self) -> int:  # launch-relative start of the next haplotype's tape
        return self.ob[-1]

    def _row(self, dst: int, ln: int):
        if ln <= self.n_alt and self.rng.random() < 0.4:
            return (int(self.rng.integers(0, self.n_alt - ln + 1)), ln, dst, 1)
        return (int(self.rng.integers(0, len(self.ref) - ln + 1)), ln, dst, 0)

    def hap(self, n_res: int, cuts=(), order: str = "sorted", extra=(), zero_back: int = -1, step: int = 3000,
            serial: bool = False) -> int:
        """Tape [0, n_res) cut at `cuts` and at random points (at most `step` apart); tasks in tape order or
        reversed; then `extra` tasks in order: (dst, len) with a random source, or full (src, len, dst, stream) rows.
        zero_back = k inserts a zero-length task at the start of task k behind it (its only disorder).
        `serial` is what the caller claims the plan decides.  Returns the haplotype index."""
        pts = {int(c) for c in cuts if 0 < c < n_res}
        x = 0
        while True:
            x += int(self.rng.integers(1, step))
            if x >= n_res:
                break
            pts.add(x)
        edges = [0] + sorted(pts) + [n_res]
        rows = [self._row(a, c - a) for a, c in zip(edges[:-1], edges[1:])] if n_res else []
        if order == "reversed":
            rows = rows[::-1]
        if zero_back >= 0:
            rows.insert(zero_back + 1, (0, 0, rows[zero_back][2], 0))
        rows += [self._row(*e) if len(e) == 2 else tuple(e) for e in extra]
        return self._push(rows, n_res, serial)

    def empty(self, n_res: int) -> int:
        """A haplotype without tasks: all '.'."""
        return self._push([], n_res, False)

    def _push(self, rows, n_res, serial):
        self.rows += rows
        self.tb.append(self.tb[-1] + len(rows))
        self.ob.append(self.ob[-1] + n_res)
        self.alts.append(self.rng.integers(97, 123, size=self.n_alt, dtype=np.uint8))
        self.ab.append(self.ab[-1] + self.n_alt)
        self.serial.append(serial)
        return len(self.tb) - 2

    def batch(self):
        u = lambda x: np.asarray(x, dtype=np.uint64)
        return dict(task_begin=u(self.tb), tasks=np.asarray(self.rows, np.uint32).reshape(-1, 4), ref=self.ref,
                    alt=np.concatenate(self.alts) if self.alts else np.zeros(0, np.uint8), alt_base=u(self.ab),
                    out_base=u(self.ob), ref_base=None, serial=np.flatnonzero(self.serial))


def edge_batch(edge: int, seed: int):
    """Flagged tapes of edge*k + d bytes (k = 1, 2; d in EDGE_OFFSETS), each starting on a multiple of `edge` of the
    launch's output, tasks reversed with cuts at every edge*j + d: tape ends and task edges on both sides of every
    span (edge = SPAN) or tile edge (tiles are counted from the start of the launch).  A sorted neighbour behind each
    pads the output to the next multiple of `edge`."""
    B = Builder(seed)
    for k in (1, 2):
        for d in EDGE_OFFSETS:
            B.hap(edge * k + d, cuts=[edge * j + dd for j in range(1, k + 1) for dd in EDGE_OFFSETS], order="reversed",
                  serial=True)
            B.hap(-B.pos % edge or edge)
    return B.batch()


def straddle_batch(seed: int):
    """One flagged haplotype per offset s in [-32, 32]: a 64-byte task [SPAN + s - 32, SPAN + s + 32) written over a
    sorted cover, so it straddles the first span edge at every offset of the window (and ends or starts on it)."""
    B = Builder(seed)
    for s in range(-32, 33):
        B.hap(SPAN + 200, extra=[(SPAN + s - 32, 64)], serial=True)
    return B.batch()


def chain_batch(seed: int, n: int = 1500):
    """One flagged haplotype with n > kSerialThreads later-wins overwrites of the same 64 bytes across a span edge,
    each shifted by one (destination cycling over 5 phases, source one further each time), so the array order has
    to hold inside every window of k_serial and from one window to the next."""
    assert n > 2 * SERIAL_THREADS
    B = Builder(seed)
    B.hap(1000)
    B.hap(2 * SPAN + 100, extra=[(i, 64, SPAN - 30 + i % 5, 1) for i in range(n)], serial=True)
    B.hap(1000)
    return B.batch()


def strided_batch(seed: int, sms: int):
    """One flagged haplotype with more spans than the k_serial grid (4 blocks per SM), so every block loops."""
    n_spans = 4 * sms + 37
    B = Builder(seed)
    B.hap(777)
    B.hap(n_spans * SPAN + 123, order="reversed", step=40_000, extra=[(SPAN * j - 5, 10) for j in range(1, n_spans, 97)],
          serial=True)
    return B.batch()


def many_small_batch(seed: int, n: int = 2450):
    """n small haplotypes, all but every 7th flagged (reversed), in one launch."""
    B = Builder(seed)
    for h in range(n):
        n_res = int(B.rng.integers(20, 400))
        if h % 7 == 6:
            B.hap(n_res, step=60)
        else:
            B.hap(n_res, cuts=[n_res // 2], order="reversed", step=60, serial=True)
    return B.batch()


NEIGHBOUR_LAYOUTS = ("flagged|sorted", "sorted|flagged", "flagged|empty", "flagged|flagged")


def neighbour_batch(layout: str, seed: int):
    """Pairs of haplotypes (A|B) whose shared tape edge lies at every 16-byte phase inside one tile (for 2, 4 and
    8 KiB tiles alike: 1008 + 17*ph bytes past a multiple of 8 KiB), and once exactly on a tile edge, where two flagged
    neighbours both write the same lb[] entry in k_plan_fix."""
    first, second = layout.split("|")
    B = Builder(seed)
    offsets = [1008 + 17 * ph for ph in range(16)] + [0]
    for off in offsets:
        target = ((B.pos + 9000 + 8191) // 8192) * 8192 + off
        for kind, n_res in ((first, target - B.pos), (second, int(B.rng.integers(3000, 20_000)))):
            if kind == "empty":
                B.empty(int(B.rng.integers(1, 40)))
            elif kind == "flagged":
                B.hap(n_res, order="reversed", serial=True)
            else:
                B.hap(n_res)
    return B.batch()


def one_byte_overlap_batch(seed: int, n_hap: int = 40):
    """Haplotypes in which every task starts one byte before the previous one ends, at lengths of 2 to 600 bytes and
    every 16-byte phase: each overlap byte must come from the later task."""
    B = Builder(seed)
    for _ in range(n_hap):
        rows, x = [], 0
        n_res = int(B.rng.integers(3000, 40_000))
        while x < n_res - 1:
            ln = min(int(B.rng.choice([int(B.rng.integers(2, 16)), int(B.rng.integers(16, 600))])), n_res - x)
            if ln < 2:
                break
            rows.append(B._row(x, ln))
            x += ln - 1
        B._push(rows, n_res, True)
    return B.batch()


def first_last_zero_batch(seed: int):
    """Flagged haplotypes first and last in the batch, and one in the middle whose only disorder is a zero-length
    task at the start of the task in front of it."""
    B = Builder(seed)
    B.hap(30_000, order="reversed", serial=True)
    B.hap(5000)
    B.hap(20_000, step=2000, zero_back=3, serial=True)
    B.hap(7000)
    B.hap(25_000, order="reversed", serial=True)
    return B.batch()


def cases(sms: int = 148):
    """Every builder, by name, unbuilt (the CPU check of the generators builds one case per test)."""
    out = {"span_edges": lambda: edge_batch(SPAN, 1), "straddle": lambda: straddle_batch(5), "chain": lambda: chain_batch(6),
           "strided": lambda: strided_batch(7, sms), "many_small": lambda: many_small_batch(8),
           "first_last_zero": lambda: first_last_zero_batch(9), "one_byte_overlaps": lambda: one_byte_overlap_batch(12)}
    for tile, seed in ((8192, 2), (4096, 3), (2048, 4)):
        out["tile_edges_%d" % tile] = lambda tile=tile, seed=seed: edge_batch(tile, seed)
    for i, layout in enumerate(NEIGHBOUR_LAYOUTS):
        out["neighbours_" + layout] = lambda layout=layout, i=i: neighbour_batch(layout, 10 + i)
    return out
