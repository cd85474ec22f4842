#!/usr/bin/env python
"""bench_outer_join.py — device-resident timing of cogroup and the outer joins at the BASELINE configs[3] per-GPU
share (8 GPUs): 6.25e7 unique keys per side, 1.25e6 of them on both sides, 8 map and 8 reduce partitions.

One JSON line per operation: inner `join` (the existing path, as the anchor), `cogroup` of every partition through
vb_cogroup, the previous host-side cogroup construction (a Python dict over both sides' group_by_key output; host wall
time, once, over --old-parts partitions), and the left and full outer joins.  Each timed line covers map + seal + the
operation over all partitions into device buffers (CUDA events on the library's stream, median of --reps after one
warm-up), with the per-kernel-class split of vb_shuffle_kernel_time and exact row-count checks.  The GPU's name and
power limit are read in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import vega_b200 as vb
from vega_b200 import _lib as L

ap = argparse.ArgumentParser()
ap.add_argument("--n-side", type=int, default=int(5e8) // 8)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--old-parts", type=int, default=1, help="partitions the host-side dict construction is timed over")
args = ap.parse_args()

assert torch.cuda.is_available(), "bench_outer_join.py measures on the GPU"
N = args.n_side
SHARED = N // 50
M = R = 8


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in out.split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return {"gpu": name, "power_limit": power}


INFO = gpu_info()
sc = vb.Context(0, profile=True)
stream = sc.stream()
a = torch.empty((N, 2), dtype=torch.int64, device="cuda")
b = torch.empty((N, 2), dtype=torch.int64, device="cuda")
sc.gen_pairs(out_rows=a, first=0, n=N, mode="unique", rank_base=0)
sc.gen_pairs(out_rows=b, first=0, n=N, mode="unique", rank_base=N - SHARED)
dptr = lambda t: ctypes.c_void_p(t.data_ptr()) if t.numel() else None


def sides():
    shs = []
    for t in (a, b):
        s_ = vb.Shuffle(sc, M, R, L.VB_U64, L.VB_U64, L.VB_AGG_COGROUP)
        col = vb.rdd._Col(t, allow_rows=True)
        st = vb.slice_starts(col.n, M)
        for m in range(M):
            s_.map(m, col, None, int(st[m]), int(st[m + 1]))
        s_.seal()
        shs.append(s_)
    return shs


def stats_of(sa, sb, rows):
    st, stb = sa.stats(), sb.stats()
    k = {name: round(st["kernels"][name]["ms"] + stb["kernels"][name]["ms"], 3) for name in L.KERNEL_CLASSES}
    return {"kernel_ms": {n: v for n, v in k.items() if v}, "launches": st["kernel_launches"] + stb["kernel_launches"], "rows": rows}


def op_inner(sa, sb):
    tot = 0
    for r in range(R):
        n = ctypes.c_uint64()
        L.check(sc._lib.vb_join_size(sa._h, sb._h, r, ctypes.byref(n)))
        k, v, w = (torch.empty(n.value, dtype=torch.int64, device="cuda") for _ in range(3))
        L.check(sc._lib.vb_join(sa._h, sb._h, r, dptr(k), dptr(v), dptr(w), L.VB_DEVICE))
        tot += n.value
    return tot


def op_cogroup(sa, sb):
    tot = 0
    for r in range(R):
        nk, na, nb = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
        L.check(sc._lib.vb_cogroup_size(sa._h, sb._h, r, ctypes.byref(nk), ctypes.byref(na), ctypes.byref(nb)))
        bufs = [torch.empty(n, dtype=torch.int64, device="cuda") for n in (nk.value, nk.value + 1, na.value, nk.value + 1, nb.value)]
        L.check(sc._lib.vb_cogroup(sa._h, sb._h, r, *[dptr(t) for t in bufs], L.VB_DEVICE))
        tot += nk.value
    return tot


def op_outer(kind):
    def run(sa, sb):
        tot = 0
        for r in range(R):
            n = ctypes.c_uint64()
            L.check(sc._lib.vb_join_outer_size(sa._h, sb._h, r, kind, ctypes.byref(n)))
            k, v, w = (torch.empty(n.value, dtype=torch.int64, device="cuda") for _ in range(3))
            valid = torch.empty(n.value, dtype=torch.uint8, device="cuda")
            L.check(sc._lib.vb_join_outer(sa._h, sb._h, r, kind, dptr(k), dptr(v), dptr(w), dptr(valid), L.VB_DEVICE))
            tot += n.value
        return tot
    return run


def timed(name, op, want_rows):
    res = []
    for rep in range(args.reps + 1):                 # the first pass warms up every shape
        torch.cuda.synchronize(); sc.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        sa, sb = sides()
        rows = op(sa, sb)
        e1.record(stream)
        sc.synchronize(); torch.cuda.synchronize()
        assert rows == want_rows, (name, rows, want_rows)
        st = stats_of(sa, sb, rows)
        sa.free(); sb.free()
        torch.cuda.empty_cache()
        if rep:
            res.append((e0.elapsed_time(e1), st))
    ms = sorted(r[0] for r in res)[len(res) // 2]
    line = {"op": name, "rows_per_side": N, "shared": SHARED, "ms": round(ms, 3), "ms_all": [round(r[0], 3) for r in res]}
    line.update(res[-1][1])
    line.update(INFO)
    print(json.dumps(line), flush=True)


timed("join", op_inner, SHARED)
timed("cogroup", op_cogroup, 2 * N - SHARED)
timed("left_outer_join", op_outer(L.VB_JOIN_LEFT_OUTER), N)
timed("full_outer_join", op_outer(L.VB_JOIN_FULL_OUTER), 2 * N - SHARED)

# the host-side construction cogroup_collect() used before vb_cogroup, once, over the first --old-parts partitions
sa, sb = sides()
sa.reduce_size(0); sb.reduce_size(0)        # group both sides before the clock starts
t0 = time.perf_counter()
keys_out = 0
for r in range(args.old_parts):
    ka, oa, va = sa.reduce(r)
    kb, ob, vb_ = sb.reduce(r)
    g = {}
    for i, k in enumerate(ka.tolist()):
        g[k] = [va[int(oa[i]):int(oa[i + 1])], vb_[:0]]
    for i, k in enumerate(kb.tolist()):
        g.setdefault(k, [va[:0], None])[1] = vb_[int(ob[i]):int(ob[i + 1])]
    keys_out += len(g)
    del g
wall = time.perf_counter() - t0
t0 = time.perf_counter()
new_keys = 0
for r in range(args.old_parts):          # the same partitions through vb_cogroup into host arrays, for the same wall clock
    nk, na, nb = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
    L.check(sc._lib.vb_cogroup_size(sa._h, sb._h, r, ctypes.byref(nk), ctypes.byref(na), ctypes.byref(nb)))
    bufs = [np.empty(n, np.uint64) for n in (nk.value, nk.value + 1, na.value, nk.value + 1, nb.value)]
    L.check(sc._lib.vb_cogroup(sa._h, sb._h, r, *[x.ctypes.data_as(ctypes.c_void_p) for x in bufs], L.VB_HOST))
    new_keys += nk.value
wall_new = time.perf_counter() - t0
assert keys_out == new_keys, (keys_out, new_keys)
line = {"op": "cogroup_collect_python_dict", "partitions": args.old_parts, "keys": keys_out, "host_wall_s": round(wall, 3),
        "vb_cogroup_to_host_wall_s": round(wall_new, 3), "note": "host wall clock after the sides are sealed and grouped"}
line.update(INFO)
print(json.dumps(line), flush=True)
sa.free(); sb.free()
sc.close()
