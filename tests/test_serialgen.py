"""CPU check of tests/serialgen.py: every generated case flags exactly the haplotypes it claims to, under the plan's
rule restated in numpy, and the oracle executes it."""
import numpy as np
import pytest

from oracle import cengine
from tests import serialgen as G


@pytest.mark.parametrize("name", list(G.cases()))
def test_generated_cases_flag_what_they_claim(name):
    b = G.cases()[name]()
    assert np.array_equal(G.flagged(b), b["serial"]), name
    assert len(b["serial"]) > 0
    out = np.zeros(int(b["out_base"][-1]), np.uint8)
    st, _, _ = cengine.batch_execute(b["task_begin"], b["tasks"], b["ref"], b["alt"], b["alt_base"], out, b["out_base"],
                                     threads=4)
    assert st == cengine.REF_OK


def test_shapes_meet_their_preconditions():
    sms = 148
    b = G.strided_batch(7, sms)
    assert int(np.diff(b["out_base"].astype(np.int64)).max()) > 4 * sms * G.SPAN  # more spans than k_serial blocks
    b = G.chain_batch(6)
    h = int(b["serial"][0])
    assert int(b["task_begin"][h + 1] - b["task_begin"][h]) > 2 * G.SERIAL_THREADS
    assert len(G.many_small_batch(8)["serial"]) >= 2000
    for edge, seed in ((G.SPAN, 1), (8192, 2), (4096, 3), (2048, 4)):  # flagged tapes start on launch-wide edges
        b = G.edge_batch(edge, seed)
        ob = b["out_base"].astype(np.int64)
        starts, lens = ob[b["serial"]], ob[b["serial"] + 1] - ob[b["serial"]]
        assert (starts % edge == 0).all() and sorted(set(lens % edge)) == sorted(d % edge for d in G.EDGE_OFFSETS)
    b = G.one_byte_overlap_batch(12)
    t = b["tasks"].astype(np.int64)
    tb = b["task_begin"].astype(np.int64)
    inner = np.setdiff1d(np.arange(len(t)), tb[:-1])  # every task but a haplotype's first
    assert (t[inner, 2] == t[inner - 1, 2] + t[inner - 1, 1] - 1).all() and len(set(t[:, 2] % 16)) == 16
    for layout in G.NEIGHBOUR_LAYOUTS:  # A|B edges: 16 phases inside a tile, then one on a tile edge
        b = G.neighbour_batch(layout, 1)
        ob = b["out_base"].astype(np.int64)
        edges = ob[1::2]  # (every pair is two haplotypes, the empty kind included)
        assert len(edges) == 17
        assert sorted(edges[:16] % 16) == list(range(16)) and all(1008 <= e % 2048 < 2048 for e in edges[:16])
        assert edges[16] % 8192 == 0


def test_flag_rule_on_small_literals():
    u = lambda *a: np.asarray(a, np.uint64)
    t = lambda rows: np.asarray(rows, np.uint32).reshape(-1, 4)
    # (dst, len) pairs per haplotype; the first task of haplotype 1 starts before haplotype 0's last one ends
    b = dict(task_begin=u(0, 2, 4, 7), tasks=t([(0, 10, 0, 0), (0, 3, 5, 0), (0, 4, 0, 0), (0, 4, 4, 0),
                                               (0, 10, 0, 0), (0, 0, 3, 0), (0, 5, 10, 0)]))
    assert list(G.flagged(b)) == [0, 2]
