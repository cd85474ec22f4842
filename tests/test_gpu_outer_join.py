"""GPU: cogroup (vb_cogroup) and left / right / full outer joins (vb_join_outer) against the reference's golden
vectors, the previous host-side cogroup construction, and the CPU oracle's group_by_key of both sides."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import vega_b200 as vb
from oracle import oracle as O
from tests import outer_ref as X
from vega_b200 import _lib as L

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COL1 = [(1, ("A", "B")), (2, ("C", "D")), (3, ("E", "F")), (4, ("G", "H"))]
COL2 = [(1, "A1"), (1, "A2"), (2, "B1"), (2, "B2"), (3, "C1"), (3, "C2")]


@pytest.fixture(scope="module")
def sc():
    c = vb.Context(0)
    yield c
    c.close()


def _shuffle(sc, keys, vals, M, R):
    """A sealed (lazy) COGROUP shuffle of (keys, vals) over M map slices, R reduce partitions."""
    kc, vc = vb.rdd._Col(keys), vb.rdd._Col(vals, role="value")
    sh = vb.Shuffle(sc, len(vb.slice_starts(kc.n, M)) - 1, R, kc.code, vc.code, L.VB_AGG_COGROUP, key_width=kc.key_width)
    st = vb.slice_starts(kc.n, M)
    for m in range(len(st) - 1):
        sh.map(m, kc, vc, int(st[m]), int(st[m + 1]))
    sh.seal()
    return sh


def _old_cogroup_collect(j):
    """The host-side construction cogroup_collect() used before vb_cogroup: a Python dict over both sides' reduce output."""
    a, b = j._run()
    out = []
    for r in range(j.num_slices):
        ka, oa, va = a.reduce(r)
        kb, ob, vb_ = b.reduce(r)
        g = {}
        for i, k in enumerate(ka.tolist()):
            g[k] = [va[int(oa[i]):int(oa[i + 1])], vb_[:0]]
        for i, k in enumerate(kb.tolist()):
            g.setdefault(k, [va[:0], None])[1] = vb_[int(ob[i]):int(ob[i + 1])]
        out.extend((k, (x[0], x[1])) for k, x in g.items())
    return out


def _assert_same_cogroup_list(got, want):
    assert len(got) == len(want)
    for (kg, (ag, bg)), (kw, (aw, bw)) in zip(got, want):
        assert kg == kw and type(kg) is type(kw)
        for x, y in ((ag, aw), (bg, bw)):
            assert x.dtype == y.dtype and x.shape == y.shape and np.array_equal(x.view(np.uint64), y.view(np.uint64))


# ---- golden vectors ---------------------------------------------------------------------------
def _test_join_rdds(sc):
    r1 = sc.parallelize((np.array([k for k, _ in COL1], dtype=np.int32), np.arange(4, dtype=np.uint64)), 4)
    r2 = sc.parallelize((np.array([k for k, _ in COL2], dtype=np.int32), np.arange(6, dtype=np.uint64)), 4)
    return r1, r2


def test_outer_joins_golden(sc):
    # tests/test_pair_rdd.rs:39-82; payload strings → table indices
    r1, r2 = _test_join_rdds(sc)
    named = lambda rows, t1, t2: sorted((k, (None if v is None else t1[v][1], None if w is None else t2[w][1])) for k, (v, w) in rows)
    matched = [(1, (("A", "B"), "A1")), (1, (("A", "B"), "A2")), (2, (("C", "D"), "B1")), (2, (("C", "D"), "B2")),
               (3, (("E", "F"), "C1")), (3, (("E", "F"), "C2"))]
    assert named(r1.left_outer_join(r2, 4).to_list(), COL1, COL2) == matched + [(4, (("G", "H"), None))]
    assert named(r1.right_outer_join(r2, 4).to_list(), COL1, COL2) == matched
    assert named(r1.full_outer_join(r2, 4).to_list(), COL1, COL2) == matched + [(4, (("G", "H"), None))]
    flip = sorted((k, (w, v)) for k, (v, w) in matched)
    assert named(r2.left_outer_join(r1, 4).to_list(), COL2, COL1) == flip
    assert named(r2.right_outer_join(r1, 4).to_list(), COL2, COL1) == flip + [(4, (None, ("G", "H")))]
    assert named(r2.full_outer_join(r1, 4).to_list(), COL2, COL1) == flip + [(4, (None, ("G", "H")))]
    k, v, w, valid = r1.left_outer_join(r2, 4).collect()
    assert k.dtype == np.int64 and v.dtype == np.uint64 and valid.dtype == np.uint8
    assert k.tolist().count(4) == 1 and valid[k == 4].tolist() == [L.VB_JOIN_HAS_V] and w[k == 4].tolist() == [0]


def test_cogroup_golden(sc):
    # tests/test_rdd.rs:434-456: cogroup of a 4-key RDD with itself → 4 keys, one value per side
    k = np.array([1, 2, 3, 4], dtype=np.int32)
    v = np.arange(4, dtype=np.uint64)
    j = sc.parallelize((k, v), 2).cogroup(sc.parallelize((k, v), 2), 2)
    cg = j.cogroup_collect()
    assert sorted((a, (x.tolist(), y.tolist())) for a, (x, y) in cg) == [(i + 1, ([i], [i])) for i in range(4)]
    _assert_same_cogroup_list(cg, _old_cogroup_collect(j))


@pytest.mark.parametrize("nparts", [3, 2])
def test_cogroup_intersection_subtract_golden(sc, nparts):
    # tests/test_rdd.rs:484-521 (intersection → [3,4,5,13]) and :675-699 (subtract → [0,1,2,10,12,19]) read off the cogroup
    c1 = np.array([1, 2, 3, 4, 5, 10, 12, 13, 19, 0], dtype=np.int32)
    c2 = np.array([3, 4, 5, 6, 7, 8, 11, 13], dtype=np.int32)
    j = sc.parallelize((c1, np.zeros(10, np.uint64)), 2).cogroup(sc.parallelize((c2, np.zeros(8, np.uint64)), 4), nparts)
    cg = j.cogroup_collect()
    assert sorted(a for a, (x, y) in cg if len(x) >= 1 and len(y) >= 1) == [3, 4, 5, 13]
    assert sorted(a for a, (x, y) in cg if len(x) >= 1 and len(y) == 0) == [0, 1, 2, 10, 12, 19]
    assert sorted(a for a, (x, y) in cg if len(x) == 0 and len(y) >= 1) == [6, 7, 8, 11]
    _assert_same_cogroup_list(cg, _old_cogroup_collect(j))


@pytest.mark.parametrize("vdt", ["u64", "f64"])
def test_cogroup_collect_unchanged_on_random_inputs(sc, vdt):
    rng = np.random.default_rng(31)
    ka = rng.integers(0, 3000, 20_000).astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    kb = rng.integers(1500, 5000, 15_000).astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    va = rng.standard_normal(len(ka)) if vdt == "f64" else rng.integers(0, 1 << 60, len(ka)).astype(np.uint64)
    vb_ = rng.integers(-(1 << 40), 1 << 40, len(kb)).astype(np.int64)
    j = sc.parallelize((ka, va), 5).cogroup(sc.parallelize((kb, vb_), 3), 7)
    _assert_same_cogroup_list(j.cogroup_collect(), _old_cogroup_collect(j))


# ---- random differential against the oracle -----------------------------------------------------
def _side(rng, n, universe, vdt):
    keys = universe[rng.integers(0, len(universe), n)] if n and len(universe) else np.zeros(n, universe.dtype)
    if vdt == "f64":
        vals = rng.standard_normal(n)
        vals[::97] = -0.0
        vals[::89] = np.nan
    elif vdt == "i64":
        vals = rng.integers(-(1 << 62), 1 << 62, n).astype(np.int64)
    else:
        vals = rng.integers(0, 2 ** 64 - 1, n, dtype=np.uint64, endpoint=True)
    return keys, vals


def _universes(rng, da, db, overlap, kw):
    """Distinct key sets of sizes da, db sharing round(overlap * min(da, db)) keys."""
    s = int(round(overlap * min(da, db)))
    if kw == 4:
        base = rng.permutation(np.arange(-(1 << 31), (1 << 31) - 1, 977, dtype=np.int64))[: da + db - s]
    else:
        base = np.unique(rng.integers(0, 2 ** 64 - 1, 2 * (da + db) + 8, dtype=np.uint64, endpoint=True))
        base = rng.permutation(base)[: da + db - s]
        base[da - 1 if s else 0] = np.uint64(2 ** 64 - 1)     # the dictionary's spare-slot key, on both sides when s > 0
    return base[:da], base[da - s: da - s + db]


def _check_pair(sc, sa_sh, sb_sh, want_a, want_b, R):
    lib = sc._lib
    for r in range(R):
        got = X.cogroup(lib, sa_sh._h, sb_sh._h, r)
        X.check_cogroup(got, want_a[r], want_b[r], sa_sh.reduce(r)[0], sb_sh.reduce(r)[0])
        keys = got[0]
        inner = X.inner(lib, sa_sh._h, sb_sh._h, r)
        for kind in ("left", "right", "full"):
            k, v, w, valid = X.outer(lib, sa_sh._h, sb_sh._h, r, kind)
            ek, ev, ew, evalid = X.expected_outer(keys, want_a[r], want_b[r], kind)
            # keys in union order, each key's rows contiguous in v-major order: the exact sequence
            assert np.array_equal(k, ek) and np.array_equal(v, ev) and np.array_equal(w, ew) and np.array_equal(valid, evalid), (r, kind)
            m = valid == 3
            assert X.rows_multiset(k[m], v[m], w[m]) == X.rows_multiset(*inner), (r, kind)


GRID = [  # n_a, n_b, M, R, overlap, (left vdt, right vdt), key width
    (0, 0, 1, 1, 0.5, ("u64", "f64"), 8),
    (1, 1, 1, 1, 1.0, ("u64", "f64"), 8),
    (1, 0, 3, 4, 0.5, ("u64", "f64"), 8),
    (0, 1000, 3, 4, 0.5, ("i64", "u64"), 8),
    (1000, 1000, 3, 4, 0.0, ("u64", "f64"), 8),
    (1000, 800, 8, 64, 0.02, ("i64", "u64"), 8),
    (1000, 1000, 1, 1, 1.0, ("u64", "f64"), 8),
    (100_000, 100_000, 8, 4, 0.5, ("i64", "u64"), 8),
    (100_000, 70_000, 3, 64, 0.02, ("u64", "f64"), 8),
    (100_000, 100_000, 8, 64, 1.0, ("i64", "u64"), 8),
    (50_000, 30_000, 4, 4, 0.5, ("u64", "f64"), 4),
    (2_000_000, 2_000_000, 8, 4, 0.5, ("u64", "f64"), 8),
    (2_000_000, 1_000_000, 3, 64, 0.02, ("i64", "u64"), 8),
    (2_000_000, 2_000_000, 1, 1, 0.0, ("u64", "f64"), 8),
]


@pytest.mark.parametrize("na,nb,M,R,overlap,vdts,kw", GRID)
def test_cogroup_and_outer_joins_match_oracle(sc, na, nb, M, R, overlap, vdts, kw):
    rng = np.random.default_rng(na * 7 + nb * 3 + M + R + int(overlap * 100) + kw)
    ua, ub = _universes(rng, max(1, na // 4), max(1, nb // 4), overlap, kw)
    ka, va = _side(rng, na, ua, vdts[0])
    kb, vb_ = _side(rng, nb, ub, vdts[1])
    if kw == 4:
        ka, kb = ka.astype(np.int32), kb.astype(np.int32)
    sa, sb = _shuffle(sc, ka, va, M, R), _shuffle(sc, kb, vb_, M, R)
    want_a = O.shuffle("group", ka.astype(np.int64) if kw == 4 else ka, va, M, R, vdts[0], key_width=kw)
    want_b = O.shuffle("group", kb.astype(np.int64) if kw == 4 else kb, vb_, M, R, vdts[1], key_width=kw)
    _check_pair(sc, sa, sb, want_a, want_b, R)
    sa.free(); sb.free()


def test_self_pair(sc):
    rng = np.random.default_rng(4)
    keys, vals = _side(rng, 30_000, np.append(rng.integers(0, 1 << 62, 4000).astype(np.uint64), np.uint64(2 ** 64 - 1)), "u64")
    sh = _shuffle(sc, keys, vals, 3, 8)
    want = O.shuffle("group", keys, vals, 3, 8)
    _check_pair(sc, sh, sh, want, want, 8)
    sh.free()


def test_inner_join_before_and_after_outer_join_agree(sc):
    rng = np.random.default_rng(12)
    ua, ub = _universes(rng, 5000, 4000, 0.3, 8)
    (ka, va), (kb, vb_) = _side(rng, 40_000, ua, "u64"), _side(rng, 30_000, ub, "u64")
    sa, sb = _shuffle(sc, ka, va, 4, 6), _shuffle(sc, kb, vb_, 3, 6)
    before = [X.rows_multiset(*X.inner(sc._lib, sa._h, sb._h, r)) for r in range(6)]       # both sides lazy: semi-join filter
    for r in range(6):
        X.outer(sc._lib, sa._h, sb._h, r, "full")
    after = [X.rows_multiset(*X.inner(sc._lib, sa._h, sb._h, r)) for r in range(6)]        # both grouped completely
    assert before == after and sum(map(len, before)) > 0
    sa.free(); sb.free()


# ---- outputs and errors -------------------------------------------------------------------------
def test_device_outputs_equal_host_and_valid_may_be_null(sc):
    import torch
    rng = np.random.default_rng(8)
    ua, ub = _universes(rng, 3000, 3000, 0.5, 8)
    (ka, va), (kb, vb_) = _side(rng, 12_000, ua, "u64"), _side(rng, 9_000, ub, "f64")
    sa, sb = _shuffle(sc, ka, va, 3, 4), _shuffle(sc, kb, vb_, 2, 4)
    lib = sc._lib
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None and t.numel() else None
    for r in range(4):
        host = X.cogroup(lib, sa._h, sb._h, r)
        nk, na_, nb_ = len(host[0]), len(host[2]), len(host[4])
        dev = [torch.empty(n, dtype=torch.int64, device="cuda") for n in (nk, nk + 1, na_, nk + 1, nb_)]
        torch.cuda.synchronize()
        L.check(lib.vb_cogroup(sa._h, sb._h, r, *[p(t) for t in dev], L.VB_DEVICE))
        for h, d in zip(host, dev):
            assert np.array_equal(h, d.cpu().numpy().view(np.uint64))
        for kind, code in X.KINDS.items():
            hk, hv, hw, hvalid = X.outer(lib, sa._h, sb._h, r, kind)
            n = len(hk)
            dk, dv, dw = (torch.empty(n, dtype=torch.int64, device="cuda") for _ in range(3))
            dvalid = torch.empty(n, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            L.check(lib.vb_join_outer(sa._h, sb._h, r, code, p(dk), p(dv), p(dw), p(dvalid), L.VB_DEVICE))
            for h, d in ((hk, dk), (hv, dv), (hw, dw)):
                assert np.array_equal(h, d.cpu().numpy().view(np.uint64))
            assert np.array_equal(hvalid, dvalid.cpu().numpy())
            nk2, nv2, nw2, none = X.outer(lib, sa._h, sb._h, r, kind, with_valid=False)   # out_valid = NULL
            assert none is None and np.array_equal(nk2, hk) and np.array_equal(nv2, hv) and np.array_equal(nw2, hw)
    sa.free(); sb.free()


def test_errors(sc):
    lib = sc._lib
    keys = np.arange(1, 200, dtype=np.uint64)
    sa, sb = _shuffle(sc, keys, keys, 2, 4), _shuffle(sc, keys[50:], keys[50:], 2, 4)
    n = ctypes.c_uint64()
    nn = [ctypes.c_uint64() for _ in range(3)]
    refs = [ctypes.byref(x) for x in nn]

    def invalid(rc):
        assert rc == L.VB_ERR_INVALID, rc

    for kind in (0, 4, -1):
        invalid(lib.vb_join_outer_size(sa._h, sb._h, 0, kind, ctypes.byref(n)))
        invalid(lib.vb_join_outer(sa._h, sb._h, 0, kind, None, None, None, None, L.VB_HOST))
    invalid(lib.vb_cogroup_size(sa._h, sb._h, 4, *refs))                              # reduce_id >= n_reduce
    invalid(lib.vb_join_outer_size(sa._h, sb._h, 4, L.VB_JOIN_FULL_OUTER, ctypes.byref(n)))
    other_r = _shuffle(sc, keys, keys, 2, 5)                                          # different n_reduce
    invalid(lib.vb_cogroup_size(sa._h, other_r._h, 0, *refs))
    invalid(lib.vb_join_outer_size(sa._h, other_r._h, 0, L.VB_JOIN_LEFT_OUTER, ctypes.byref(n)))
    narrow = _shuffle(sc, keys.astype(np.uint32), keys, 2, 4)                          # different key width
    invalid(lib.vb_cogroup_size(sa._h, narrow._h, 0, *refs))
    invalid(lib.vb_join_outer_size(narrow._h, sa._h, 0, L.VB_JOIN_RIGHT_OUTER, ctypes.byref(n)))
    red = vb.Shuffle(sc, 1, 4, L.VB_U64, L.VB_U64, L.VB_AGG_SUM)                       # not a group shuffle
    col = vb.rdd._Col(keys)
    red.map(0, col, col, 0, len(keys))
    red.seal()
    invalid(lib.vb_cogroup_size(sa._h, red._h, 0, *refs))
    invalid(lib.vb_join_outer_size(red._h, sa._h, 0, L.VB_JOIN_FULL_OUTER, ctypes.byref(n)))
    r = next(r for r in range(4) if X.cogroup(lib, sa._h, sb._h, r)[0].size)          # NULL outputs with rows to write
    invalid(lib.vb_cogroup(sa._h, sb._h, r, None, None, None, None, None, L.VB_HOST))
    invalid(lib.vb_join_outer(sa._h, sb._h, r, L.VB_JOIN_FULL_OUTER, None, None, None, None, L.VB_HOST))
    invalid(lib.vb_cogroup(sa._h, sb._h, r, None, None, None, None, None, 7))           # bad dst_loc
    # after the errors the pair still gives the right answer
    want_a, want_b = O.shuffle("group", keys, keys, 2, 4), O.shuffle("group", keys[50:], keys[50:], 2, 4)
    _check_pair(sc, sa, sb, want_a, want_b, 4)
    for s in (sa, sb, other_r, narrow, red):
        s.free()


# ---- BASELINE configs[3] per-GPU share ----------------------------------------------------------------
def _big_gpu():
    import torch
    return torch.cuda.get_device_properties(0).total_memory >= 120 * 2 ** 30


_M64 = (1 << 64) - 1


def _splitmix64(x):
    """splitmix64 over a u64 array (the generator's mixing function, vectorised)."""
    z = x + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def _unxorshift(z, s):
    x = z.copy()
    for _ in range(64 // s + 1):
        x = z ^ (x >> np.uint64(s))
    return x


def _splitmix64_inverse(z):
    x = _unxorshift(z, 31) * np.uint64(pow(0x94D049BB133111EB, -1, 1 << 64))
    x = _unxorshift(x, 27) * np.uint64(pow(0xBF58476D1CE4E5B9, -1, 1 << 64))
    return _unxorshift(x, 30) - np.uint64(0x9E3779B97F4A7C15)


def test_outer_joins_at_config4_per_gpu_share(sc):
    """6.25e7 unique keys per side, 1.25e6 of them shared (the inner-join benchmark's shape), every row checked.  The
    generator's keys are splitmix64(rank ^ C), a bijection: inverting it gives each output key's rank, hence which side
    holds it, at which input row, and so its value splitmix64(seed_v + row) & 0xFFFFF — an O(n) check without sorts."""
    import torch
    if not _big_gpu():
        pytest.skip("needs a 180 GB GPU")
    n_side, R = int(5e8) // 8, 8
    shared = n_side // 50
    a = torch.empty((n_side, 2), dtype=torch.int64, device="cuda")
    b = torch.empty((n_side, 2), dtype=torch.int64, device="cuda")
    sc.gen_pairs(out_rows=a, first=0, n=n_side, mode="unique", rank_base=0, seed_v=2)
    sc.gen_pairs(out_rows=b, first=0, n=n_side, mode="unique", rank_base=n_side - shared, seed_v=2)
    probe = np.arange(0, n_side, 999_983, dtype=np.uint64)         # the inverse and the value formula, on sampled input rows
    ha = a[probe.astype(np.int64)].cpu().numpy().view(np.uint64)
    assert np.array_equal(_splitmix64_inverse(ha[:, 0]) ^ np.uint64(0xA5A5A5A5A5A5A5A5), probe)
    assert np.array_equal(ha[:, 1], _splitmix64(probe + np.uint64(2)) & np.uint64(0xFFFFF))
    sa = vb.Shuffle(sc, 8, R, L.VB_U64, L.VB_U64, L.VB_AGG_COGROUP)
    sb = vb.Shuffle(sc, 8, R, L.VB_U64, L.VB_U64, L.VB_AGG_COGROUP)
    for s_, t in ((sa, a), (sb, b)):
        col = vb.rdd._Col(t, allow_rows=True)
        st = vb.slice_starts(col.n, 8)
        for m in range(8):
            s_.map(m, col, None, int(st[m]), int(st[m + 1]))
        s_.seal()
    del a, b
    torch.cuda.empty_cache()
    b0 = np.uint64(n_side - shared)
    for kind, want_rows in (("left", n_side), ("full", 2 * n_side - shared)):
        parts = [X.outer(sc._lib, sa._h, sb._h, r, kind) for r in range(R)]
        k, v, w, valid = (np.concatenate([p[i] for p in parts]) for i in range(4))
        del parts
        assert len(k) == want_rows
        rank = _splitmix64_inverse(k) ^ np.uint64(0xA5A5A5A5A5A5A5A5)
        assert int(rank.max()) < 2 * n_side - shared
        assert (np.bincount(rank.astype(np.int64), minlength=want_rows) == 1).all()   # each key of the kept sides once
        in_a, in_b = rank < np.uint64(n_side), rank >= b0
        assert int((in_a & in_b).sum()) == shared
        assert np.array_equal(valid, (in_a * 1 + in_b * 2).astype(np.uint8))
        assert np.array_equal(v, np.where(in_a, _splitmix64(rank + np.uint64(2)) & np.uint64(0xFFFFF), np.uint64(0)))
        assert np.array_equal(w, np.where(in_b, _splitmix64(rank - b0 + np.uint64(2)) & np.uint64(0xFFFFF), np.uint64(0)))
        if kind == "left":
            assert in_a.all()
    sa.free(); sb.free()


def test_cpp_outer_join_example_runs():
    path = os.path.join(ROOT, "examples", "_build", "outer_join")
    if not os.path.exists(path):
        pytest.skip("examples not built (run __graft_entry__.build())")
    out = subprocess.run([path], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    assert "(4, ((G,H), None))" in out.stdout, out.stdout
