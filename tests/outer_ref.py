"""Cogroup / outer-join helpers of the GPU tests: drive the four C entry points and derive the expected results from
the oracle's group_by_key output of each side (vectorised numpy, so million-row partitions stay cheap)."""
import ctypes

import numpy as np

from vega_b200 import _lib as L

KINDS = {"left": L.VB_JOIN_LEFT_OUTER, "right": L.VB_JOIN_RIGHT_OUTER, "full": L.VB_JOIN_FULL_OUTER}


def _p(x):
    return x.ctypes.data_as(ctypes.c_void_p) if x is not None else None


def cogroup(lib, a, b, r):
    """vb_cogroup of partition r into host arrays, all as u64 bits: (keys, offs_l, vals_l, offs_r, vals_r)."""
    nk, na, nb = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
    L.check(lib.vb_cogroup_size(a, b, r, ctypes.byref(nk), ctypes.byref(na), ctypes.byref(nb)))
    k = np.empty(nk.value, np.uint64)
    ol, orr = np.empty(nk.value + 1, np.uint64), np.empty(nk.value + 1, np.uint64)
    vl, vr = np.empty(na.value, np.uint64), np.empty(nb.value, np.uint64)
    L.check(lib.vb_cogroup(a, b, r, _p(k), _p(ol), _p(vl), _p(orr), _p(vr), L.VB_HOST))
    return k, ol, vl, orr, vr


def outer(lib, a, b, r, kind, with_valid=True):
    """vb_join_outer of partition r into host arrays (u64 bits): (k, v, w, valid or None)."""
    n = ctypes.c_uint64()
    L.check(lib.vb_join_outer_size(a, b, r, KINDS[kind], ctypes.byref(n)))
    k, v, w = (np.empty(n.value, np.uint64) for _ in range(3))
    valid = np.empty(n.value, np.uint8) if with_valid else None
    L.check(lib.vb_join_outer(a, b, r, KINDS[kind], _p(k), _p(v), _p(w), _p(valid), L.VB_HOST))
    return k, v, w, valid


def inner(lib, a, b, r):
    n = ctypes.c_uint64()
    L.check(lib.vb_join_size(a, b, r, ctypes.byref(n)))
    k, v, w = (np.empty(n.value, np.uint64) for _ in range(3))
    L.check(lib.vb_join(a, b, r, _p(k), _p(v), _p(w), L.VB_HOST))
    return k, v, w


def side_lists(keys, side):
    """Per key of `keys`: (start, count) of its value list in the oracle side {"keys", "offsets", "vals"} (count 0 when
    the side lacks the key)."""
    sk = side["keys"].view(np.uint64)
    offs = side["offsets"].astype(np.uint64)
    if len(sk) == 0:
        z = np.zeros(len(keys), np.uint64)
        return z, z.copy()
    order = np.argsort(sk, kind="stable")
    pos = np.minimum(np.searchsorted(sk[order], keys), len(sk) - 1)
    hit = sk[order][pos] == keys
    idx = order[pos]
    start = np.where(hit, offs[idx], 0).astype(np.uint64)
    cnt = np.where(hit, offs[idx + 1] - offs[idx], 0).astype(np.uint64)
    return start, cnt


def _gather(vals, start, cnt):
    """Concatenation of vals[start[i] : start[i] + cnt[i]] over i."""
    n = int(cnt.sum())
    if n == 0:
        return np.empty(0, np.uint64)
    first = np.repeat(np.cumsum(cnt) - cnt, cnt.astype(np.int64))
    local = np.arange(n, dtype=np.uint64) - first
    return vals.view(np.uint64)[(np.repeat(start, cnt.astype(np.int64)) + local).astype(np.int64)]


def check_cogroup(got, sa, sb, left_keys_gpu, right_keys_gpu):
    """got = cogroup(...) of one partition; sa / sb = the oracle's group_by_key partitions of the two sides;
    left_keys_gpu / right_keys_gpu = the keys of each side's own CSR on the device (for the union order)."""
    k, ol, vl, orr, vr = got
    ka, kb = sa["keys"].view(np.uint64), sb["keys"].view(np.uint64)
    assert len(np.unique(k)) == len(k)
    assert np.array_equal(np.sort(k), np.union1d(ka, kb)), "key set"
    nl = len(left_keys_gpu)
    assert np.array_equal(k[:nl], left_keys_gpu.view(np.uint64)), "union order: left keys in left CSR order"
    rk = right_keys_gpu.view(np.uint64)
    assert np.array_equal(k[nl:], rk[~np.isin(rk, ka)]), "union order: right-only keys in right CSR order"
    assert ol[0] == 0 and orr[0] == 0
    for (start, cnt), offs, vals, side in ((side_lists(k, sa), ol, vl, sa), (side_lists(k, sb), orr, vr, sb)):
        assert np.array_equal(np.diff(offs), cnt), "value counts"
        assert np.array_equal(vals, _gather(side["vals"], start, cnt)), "value lists (input order, bit for bit)"


def expected_outer(keys, sa, sb, kind):
    """Rows of an outer join of `kind` over the union keys `keys` (in that order) from the oracle sides:
    per key `for v in vs { for w in ws }`, one-sided keys kept per `kind`, absent values 0.  (k, v, w, valid)."""
    keep_l, keep_r = kind in ("left", "full"), kind in ("right", "full")
    sl, cl = side_lists(keys, sa)
    sr, cr = side_lists(keys, sb)
    both, lonly, ronly = (cl > 0) & (cr > 0), (cl > 0) & (cr == 0), (cl == 0) & (cr > 0)
    n = np.where(both, cl * cr, np.where(lonly & keep_l, cl, np.where(ronly & keep_r, cr, 0))).astype(np.int64)
    total = int(n.sum())
    first = np.repeat(np.cumsum(n) - n, n)
    local = (np.arange(total, dtype=np.int64) - first).astype(np.uint64)
    rb, rl, rr = np.repeat(both, n), np.repeat(lonly, n), np.repeat(ronly, n)
    rcr = np.maximum(np.repeat(cr, n), 1)
    vi = np.where(rb, local // rcr, local)
    wi = np.where(rb, local % rcr, local)
    va = np.append(sa["vals"].view(np.uint64), np.uint64(0))
    wb = np.append(sb["vals"].view(np.uint64), np.uint64(0))
    vidx = np.where(rb | rl, np.repeat(sl, n) + vi, np.uint64(len(va) - 1)).astype(np.int64)
    widx = np.where(rb | rr, np.repeat(sr, n) + wi, np.uint64(len(wb) - 1)).astype(np.int64)
    valid = (rb * 3 + rl * 1 + rr * 2).astype(np.uint8)
    return np.repeat(keys, n), va[vidx], wb[widx], valid


def rows_multiset(k, v, w):
    return sorted(zip(k.view(np.uint64).tolist(), v.view(np.uint64).tolist(), w.view(np.uint64).tolist()))
