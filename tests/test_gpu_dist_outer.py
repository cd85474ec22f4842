"""Cogroup and outer joins with two ranks: each rank computes vb_cogroup and vb_join_outer on the reduce partitions it
owns (and gets zero sizes on the others), and the union over ranks must equal the single-process oracle.  With >= 2
GPUs the exchange is the library's own (NCCL or the fused P2P scatter, one rank per GPU); on a 1-GPU box both ranks
share GPU 0 and the all-to-all-v is staged through gloo."""
import os
import pickle
import socket
import sys
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dataset():
    rng = np.random.default_rng(78)
    ka = rng.integers(0, 4000, 60_000).astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(3)
    kb = rng.integers(2000, 7000, 45_000).astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(3)
    va = rng.integers(0, 1 << 50, len(ka)).astype(np.uint64)
    vb_ = rng.integers(0, 1 << 50, len(kb)).astype(np.uint64)
    return ka, va, kb, vb_


def _worker(rank, world, port, Ma, Mb, R, nccl, outdir, p2p):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = rank if nccl else 0
    torch.cuda.set_device(dev)
    if nccl:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{dev}"))
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    import vega_b200 as vb
    from tests import outer_ref as X
    from vega_b200 import _lib as L
    from vega_b200 import dist as vdist
    ka, va, kb, vb_ = _dataset()
    sc = vb.Context(dev)
    if nccl:
        sc.comm_init(rank, world)
    eng = vdist.CudaEngine(sc)
    shs = []
    for keys, vals, M in ((ka, va, Ma), (kb, vb_, Mb)):
        starts = vb.slice_starts(len(keys), M)
        lo, hi = vdist.map_block(rank, world, M)
        maps = [(m, keys[starts[m]:starts[m + 1]], vals[starts[m]:starts[m + 1]]) for m in range(lo, hi)]
        shs.append(vdist.run_shuffle(eng, maps, M, R, 0, 0, L.VB_AGG_COGROUP, rank, world,
                                     exchange_device=None if (nccl or p2p) else "cpu", p2p=p2p))
    sa, sb = shs
    res = {}
    for r in range(R):
        cg = X.cogroup(sc._lib, sa._h, sb._h, r)
        outer = {kind: X.outer(sc._lib, sa._h, sb._h, r, kind) for kind in X.KINDS}
        sides = (sa.reduce(r)[0], sb.reduce(r)[0])
        if r % world != rank:
            assert len(cg[0]) == len(cg[2]) == len(cg[4]) == 0
            assert all(len(o[0]) == 0 for o in outer.values())
        res[r] = (cg, outer, sides)
    with open(os.path.join(outdir, f"o{rank}.pkl"), "wb") as f:
        pickle.dump(res, f)
    sa.free(); sb.free()
    sc.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("Ma,Mb,R,p2p", [(4, 2, 4, False), (3, 5, 6, True), (2, 2, 3, False)])
def test_two_rank_cogroup_and_outer_joins_match_oracle(Ma, Mb, R, p2p):
    from oracle import oracle as O
    from tests import outer_ref as X
    world = 2
    nccl = torch.cuda.device_count() >= 2
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_worker, args=(world, _free_port(), Ma, Mb, R, nccl, d, p2p), nprocs=world, join=True)
        per_rank = [pickle.load(open(os.path.join(d, f"o{r}.pkl"), "rb")) for r in range(world)]
    ka, va, kb, vb_ = _dataset()
    wa, wb = O.shuffle("group", ka, va, Ma, R), O.shuffle("group", kb, vb_, Mb, R)
    inner = O.join(ka, va, Ma, kb, vb_, Mb, R)
    total = {kind: 0 for kind in X.KINDS}
    for r in range(R):
        cg, outer, sides = per_rank[r % world][r]
        X.check_cogroup(cg, wa[r], wb[r], *sides)
        for kind, (k, v, w, valid) in outer.items():
            ek, ev, ew, evalid = X.expected_outer(cg[0], wa[r], wb[r], kind)
            assert np.array_equal(k, ek) and np.array_equal(v, ev) and np.array_equal(w, ew) and np.array_equal(valid, evalid), (r, kind)
            m = valid == 3
            assert X.rows_multiset(k[m], v[m], w[m]) == X.rows_multiset(*inner[r]), (r, kind)
            total[kind] += len(k)
    n_inner = sum(len(x[0]) for x in inner)
    assert n_inner > 0 and min(total.values()) > n_inner
