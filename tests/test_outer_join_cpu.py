"""Outer joins without a GPU: Spark-semantics restatements of left / right / full outer join (the reference has no
outer joins), pinned on the reference's test_join data (tests/test_pair_rdd.rs:39-82) against hand-written rows, and
a compile check of the C++ example over include/vega_b200.hpp.  tests/test_gpu_outer_join.py checks the device
results against these restatements."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def cogroup_ref(left, right):
    """[(k, (vs, ws))] in union order: the keys of `left` in first-seen order, then the keys only `right` has in
    first-seen order; each value list in input order.  left / right: lists of (k, v)."""
    g = {}
    for k, v in left:
        g.setdefault(k, ([], []))[0].append(v)
    for k, w in right:
        g.setdefault(k, ([], []))[1].append(w)
    return list(g.items())


def outer_join_ref(left, right, how):
    """Spark's left / right / full outer join: per key `for v in vs { for w in ws }`; a key with values on one side
    only keeps them with None on the other side when `how` keeps that side."""
    keep_l, keep_r = how in ("left", "full"), how in ("right", "full")
    out = []
    for k, (vs, ws) in cogroup_ref(left, right):
        if vs and ws:
            out.extend((k, (v, w)) for v in vs for w in ws)
        elif vs and keep_l:
            out.extend((k, (v, None)) for v in vs)
        elif ws and keep_r:
            out.extend((k, (None, w)) for w in ws)
    return out


COL1 = [(1, ("A", "B")), (2, ("C", "D")), (3, ("E", "F")), (4, ("G", "H"))]
COL2 = [(1, "A1"), (1, "A2"), (2, "B1"), (2, "B2"), (3, "C1"), (3, "C2")]
MATCHED = [(1, (("A", "B"), "A1")), (1, (("A", "B"), "A2")), (2, (("C", "D"), "B1")), (2, (("C", "D"), "B2")),
           (3, (("E", "F"), "C1")), (3, (("E", "F"), "C2"))]


def test_left_outer_join_of_test_join_data():
    got = outer_join_ref(COL1, COL2, "left")
    assert got == MATCHED + [(4, (("G", "H"), None))]
    assert [k for k, _ in got].count(4) == 1


def test_right_outer_join_of_test_join_data():
    assert outer_join_ref(COL1, COL2, "right") == MATCHED          # every right key has a left partner
    got = outer_join_ref(COL2, COL1, "right")
    assert got == [(k, (w, v)) for k, (v, w) in MATCHED] + [(4, (None, ("G", "H")))]


def test_full_outer_join_of_test_join_data():
    assert outer_join_ref(COL1, COL2, "full") == MATCHED + [(4, (("G", "H"), None))]
    assert outer_join_ref(COL2, COL1, "full") == [(k, (w, v)) for k, (v, w) in MATCHED] + [(4, (None, ("G", "H")))]


def test_one_sided_and_empty_inputs():
    a = [(5, "x"), (6, "y"), (5, "z")]
    assert outer_join_ref(a, [], "left") == [(5, ("x", None)), (5, ("z", None)), (6, ("y", None))]
    assert outer_join_ref(a, [], "right") == []
    assert outer_join_ref([], a, "full") == [(5, (None, "x")), (5, (None, "z")), (6, (None, "y"))]
    assert outer_join_ref([], [], "full") == []
    assert cogroup_ref(a, [(7, "w"), (5, "v")]) == [(5, (["x", "z"], ["v"])), (6, (["y"], [])), (7, ([], ["w"]))]


def test_outer_join_example_compiles():
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    out = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-I", os.path.join(ROOT, "include"),
                          os.path.join(ROOT, "examples", "outer_join.cpp")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
