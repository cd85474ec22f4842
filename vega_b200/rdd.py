"""Host-side mirror of vega's operator API for the shuffle path, above the C ABI.

Same names and argument meaning as the reference for the calls on the path
(src/context.rs `Context::parallelize/make_rdd`, src/rdd/pair_rdd.rs
`group_by_key / reduce_by_key / join / cogroup / partition_by_key`, src/rdd/rdd.rs
`count_by_value / distinct / collect`), so the parity tests read like tests/test_pair_rdd.rs.
Differences forced by the boundary (SURVEY.md F4): rows are 64-bit POD (K,V) arrays
(numpy on the host or torch CUDA tensors), and `reduce_by_key` takes a *named* op
("sum" | "min" | "max") because a closure cannot cross into CUDA.

All compute happens in libvega_b200.so; this module slices the input exactly like
ParallelCollection::slice, drives map tasks → seal → reduce tasks like the scheduler does
(base_scheduler.rs:377-455), and concatenates partitions in order (rdd.rs:420-434).
"""
import ctypes
import itertools
import weakref

import numpy as np

from . import _lib as L

_AGG = {"group": L.VB_AGG_GROUP, "sum": L.VB_AGG_SUM, "min": L.VB_AGG_MIN, "max": L.VB_AGG_MAX,
        "count": L.VB_AGG_COUNT, "cogroup": L.VB_AGG_COGROUP, "sort": L.VB_AGG_SORT}
_NP_OF = {L.VB_U64: np.uint64, L.VB_I64: np.int64, L.VB_F64: np.float64}


def _is_torch(x):
    return hasattr(x, "data_ptr") and hasattr(x, "is_cuda")


def _sync_torch(*tensors):
    """The library runs on its own stream: pending torch work on buffers it is about to touch must be done
    (torch's caching allocator may hand out memory whose previous user is still running on torch's stream)."""
    for t in tensors:
        if t is not None and _is_torch(t) and t.is_cuda:
            import torch
            torch.cuda.current_stream(t.device).synchronize()
            return


class _Col:
    """One 64-bit column (or an (n,2) AoS row block): pointer + location + dtype code."""

    def __init__(self, x, allow_rows=False, role="key"):
        self.key_width = 8
        self.rows = False
        if _is_torch(x):
            import torch
            if not x.is_contiguous():
                x = x.contiguous()
            code = {torch.int64: L.VB_I64, torch.float64: L.VB_F64}.get(x.dtype)
            if code is None and hasattr(torch, "uint64") and x.dtype == torch.uint64:
                code = L.VB_U64
            if code is None:
                raise TypeError(f"unsupported tensor dtype {x.dtype}")
            self.loc = L.VB_DEVICE_BORROWED if x.is_cuda else L.VB_HOST
            if x.is_cuda:
                # the library launches on its own stream: whatever produced this tensor on torch's stream must be done
                torch.cuda.current_stream(x.device).synchronize()
            self.ptr = x.data_ptr()
            shape = tuple(x.shape)
        else:
            x = np.asarray(x)
            if x.dtype in (np.int32, np.uint32):
                self.key_width = 4          # Rust i32/u32 keys hash as 4 LE bytes
                x = x.astype(np.int64 if x.dtype.kind == "i" else np.uint64)
            elif x.dtype in (np.int16, np.uint16, np.int8, np.uint8) or x.dtype.kind == "b":
                # Rust hashes i16 as 2 bytes and i8/u8/bool as 1: the library has 4- and 8-byte key hashes only,
                # so narrow KEYS would be placed differently from the reference's HashPartitioner — refuse them.
                if role == "key":
                    raise TypeError(f"key dtype {x.dtype}: only 32- and 64-bit integer keys hash like the reference's")
                x = x.astype(np.int64 if x.dtype.kind == "i" else np.uint64)
            code = {"u": L.VB_U64, "i": L.VB_I64, "f": L.VB_F64}.get(x.dtype.kind)
            if code is None or x.dtype.itemsize != 8:
                raise TypeError(f"unsupported dtype {x.dtype}")
            x = np.ascontiguousarray(x)
            self.loc = L.VB_HOST
            self.ptr = x.ctypes.data
            shape = x.shape
        if len(shape) == 2 and shape[1] == 2 and allow_rows:
            self.rows = True
        elif len(shape) != 1:
            raise ValueError(f"expected a 1-D column{' or (n,2) rows' if allow_rows else ''}, got shape {shape}")
        self.n = shape[0]
        self.code = code
        self.owner = x

    def at(self, start):
        return ctypes.c_void_p(self.ptr + start * (16 if self.rows else 8)) if self.n else None


def slice_starts(n, num_slices):
    """ParallelCollection::slice boundaries (parallel_collection_rdd.rs:116-145) via the C ABI."""
    buf = np.zeros(min(n, num_slices) + 2, dtype=np.uint64)
    k = L.lib().vb_slice(n, num_slices, buf.ctypes.data)
    if k == 0:
        raise ValueError("Number of slices should be greater than or equal to 1")
    return buf[: k + 1].astype(np.int64)


class Context:
    """vega::Context for the shuffle path (src/context.rs:333-473): owns the device context
    and hands out shuffle ids (`new_shuffle_id`)."""

    def __init__(self, device=0, profile=False):
        self._lib = L.lib()
        h = ctypes.c_void_p()
        L.check(self._lib.vb_ctx_create(device, ctypes.byref(h)))
        self._h = h
        self._ids = itertools.count()
        self._shuffles = weakref.WeakSet()      # live shuffles are freed before the context goes away
        self.comm = None
        if profile:
            self.set_profile(True)

    @staticmethod
    def new(device=0):
        return Context(device)

    def set_profile(self, on):
        L.check(self._lib.vb_ctx_set_profile(self._h, int(bool(on))))

    def new_shuffle_id(self):
        return next(self._ids)

    def synchronize(self):
        L.check(self._lib.vb_ctx_synchronize(self._h))

    def stream(self):
        """The context's CUDA stream as a torch.cuda.ExternalStream (event timing in bench.py)."""
        import torch
        dev = self._lib.vb_ctx_device(self._h)
        return torch.cuda.ExternalStream(self._lib.vb_ctx_stream(self._h), device=f"cuda:{dev}")

    def mem_info(self):
        r, h = ctypes.c_uint64(), ctypes.c_uint64()
        L.check(self._lib.vb_ctx_mem_info(self._h, ctypes.byref(r), ctypes.byref(h)))
        return r.value, h.value

    def parallelize(self, data, num_slices, values=None):
        """`sc.parallelize(vec, num_slices)`.  data: 1-D keys (→ Rdd), (n,2) rows or
        (keys, values) (→ PairRdd)."""
        if values is not None:
            return PairRdd(self, _Col(data), _Col(values, role="value"), num_slices)
        if isinstance(data, tuple) and len(data) == 2:
            return PairRdd(self, _Col(data[0]), _Col(data[1], role="value"), num_slices)
        col = _Col(data, allow_rows=True)
        if col.rows:
            return PairRdd(self, col, None, num_slices)
        return Rdd(self, col, num_slices)

    make_rdd = parallelize

    def range(self, start, end, step, num_slices):
        """`sc.range(start, end, step, num_slices)` (src/context.rs:419-431): (start..=end).step_by(step), generated
        ON the device (vb_range) — a source RDD with no host array and no H2D copy."""
        import torch
        n = self._lib.vb_range_len(start, end, step)
        dev = f"cuda:{self._lib.vb_ctx_device(self._h)}"
        t = torch.empty(n, dtype=torch.int64, device=dev)
        torch.cuda.current_stream(t.device).synchronize()
        L.check(self._lib.vb_range(self._h, ctypes.c_void_p(t.data_ptr()) if n else None, start, end, step))
        col = _Col(t)
        col.code = L.VB_U64
        return Rdd(self, col, num_slices)

    def gen_pairs(self, out_rows=None, out_keys=None, out_vals=None, first=0, n=0, mode="uniform", n_distinct=1,
                  rank_base=0, seed_k=1, seed_v=2, zipf_s=0.0):
        """Fill device buffers (torch CUDA tensors) with the synthetic workload of SURVEY.md §8(d)."""
        m = {"uniform": L.VB_GEN_UNIFORM, "zipf": L.VB_GEN_ZIPF, "unique": L.VB_GEN_UNIQUE}[mode]
        _sync_torch(out_rows, out_keys, out_vals)
        p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        L.check(self._lib.vb_gen_pairs(self._h, p(out_rows), p(out_keys), p(out_vals), first, n, m, n_distinct,
                                       rank_base, seed_k, seed_v, float(zipf_s)))

    def trim(self, keep_bytes=0):
        """Return pool memory beyond keep_bytes to the device."""
        L.check(self._lib.vb_ctx_trim(self._h, keep_bytes))

    # ---- one-process-per-GPU: the NCCL communicator lives inside the library ------------------
    def comm_init(self, rank, world, unique_id=None, group=None):
        """Collective.  unique_id: the 128 bytes from `Context.comm_unique_id()` on rank 0, handed to every
        rank by any host-side bootstrap; if None, torch.distributed (already initialised) broadcasts it —
        torch is then used for this bootstrap only, the exchange itself runs inside libvega_b200."""
        if unique_id is None:
            import torch.distributed as dist
            box = [self.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0, group=group)
            unique_id = box[0]
        buf = (ctypes.c_ubyte * L.VB_UNIQUE_ID_BYTES).from_buffer_copy(unique_id)
        L.check(self._lib.vb_ctx_comm_init(self._h, buf, rank, world))
        self.comm = (rank, world)

    def comm_unique_id(self):
        buf = (ctypes.c_ubyte * L.VB_UNIQUE_ID_BYTES)()
        L.check(self._lib.vb_comm_unique_id(buf))
        return bytes(buf)

    def comm_destroy(self):
        if getattr(self, "comm", None):
            L.check(self._lib.vb_ctx_comm_destroy(self._h))
            self.comm = None

    def close(self):
        if self._h:
            for sh in list(self._shuffles):
                sh.free()
            self._lib.vb_ctx_destroy(self._h)      # collective when a communicator exists
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


class Shuffle:
    """Thin RAII wrapper of one vb_shuf (== one ShuffleDependency / shuffle_id)."""

    def __init__(self, sc, n_map, n_reduce, kcode, vcode, agg, key_width=8, hint=0, rank=0, world=1):
        self.sc, self._lib = sc, sc._lib
        self.n_map, self.n_reduce, self.agg, self.vcode, self.kcode = n_map, n_reduce, agg, vcode, kcode
        self.has_payload = True
        self._keepalive = []      # owners of VB_DEVICE_BORROWED inputs: the library reads them until seal
        h = ctypes.c_void_p()
        part = L.VB_PART_RANGE if agg == L.VB_AGG_SORT else L.VB_PART_HASH_METRO64
        L.check(self._lib.vb_shuffle_create(sc._h, sc.new_shuffle_id(), n_map, n_reduce, kcode, vcode, agg, part, ctypes.byref(h)))
        self._h = h
        sc._shuffles.add(self)
        if key_width != 8:
            L.check(self._lib.vb_shuffle_set_key_width(h, key_width))
        if hint:
            L.check(self._lib.vb_shuffle_set_hint(h, hint))
        if world > 1:
            L.check(self._lib.vb_shuffle_set_dist(h, rank, world))

    def map(self, map_id, keys, vals, start, stop):
        """ShuffleMapTask::run for one map partition = rows [start, stop) of the parent."""
        n = stop - start
        if keys.loc == L.VB_DEVICE_BORROWED:
            self._keepalive.append((keys.owner, vals.owner if vals is not None else None))
        if keys.rows:
            L.check(self._lib.vb_shuffle_map_aos(self._h, map_id, keys.at(start), n, keys.loc))
        else:
            if vals is not None and vals.loc != keys.loc:
                raise ValueError("keys and values must live in the same memory space")
            L.check(self._lib.vb_shuffle_map_soa(self._h, map_id, keys.at(start), vals.at(start) if vals is not None else None, n, keys.loc))

    def exchange(self, mode=L.VB_XCHG_AUTO):
        """The shuffle's exchange step inside the library (collective; needs Context.comm_init)."""
        L.check(self._lib.vb_shuffle_exchange(self._h, mode))

    def exchange_stats(self):
        st = L.vb_xstats()
        L.check(self._lib.vb_shuffle_exchange_stats(self._h, ctypes.byref(st)))
        return {"sent_rows": st.sent_rows, "recv_rows": st.recv_rows, "exchanges": st.exchanges,
                "exchange_ms": st.exchange_ms, "exchange_kind": {0: None, 1: "nccl", 2: "p2p"}[st.kind],
                "prepare_wall_ms": st.prepare_wall_ms, "counts_wall_ms": st.counts_wall_ms, "post_wall_ms": st.post_wall_ms}

    def seal(self):
        L.check(self._lib.vb_shuffle_seal(self._h))
        self._keepalive = []

    def reduce_size(self, r):
        nk, nv = ctypes.c_uint64(), ctypes.c_uint64()
        L.check(self._lib.vb_shuffle_reduce_size(self._h, r, ctypes.byref(nk), ctypes.byref(nv)))
        return nk.value, nv.value

    def reduce(self, r):
        """ShuffledRdd::compute(split r) → host arrays."""
        nk, nv = self.reduce_size(r)
        keys = np.empty(nk, dtype=_NP_OF[self.kcode])
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p) if a is not None else None
        if self.agg in (L.VB_AGG_GROUP, L.VB_AGG_COGROUP):
            offs = np.empty(nk + 1, dtype=np.uint64)
            vals = np.empty(nv, dtype=_NP_OF[self.vcode])
            L.check(self._lib.vb_shuffle_reduce(self._h, r, p(keys), None, p(offs), p(vals), L.VB_HOST))
            return keys, offs, vals
        if self.agg == L.VB_AGG_SORT and not self.has_payload:
            L.check(self._lib.vb_shuffle_reduce(self._h, r, p(keys), None, None, None, L.VB_HOST))
            return keys, None
        out_dt = np.uint64 if self.agg == L.VB_AGG_COUNT else _NP_OF[self.vcode]
        comb = np.empty(nk, dtype=out_dt)
        L.check(self._lib.vb_shuffle_reduce(self._h, r, p(keys), p(comb), None, None, L.VB_HOST))
        return keys, comb

    def reduce_device(self, r, out_keys=None, out_comb=None, out_offs=None, out_vals=None):
        """Same, into caller-provided torch CUDA tensors (any may be None)."""
        _sync_torch(out_keys, out_comb, out_offs, out_vals)
        p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        L.check(self._lib.vb_shuffle_reduce(self._h, r, p(out_keys), p(out_comb), p(out_offs), p(out_vals), L.VB_DEVICE))

    def reduce_blob(self, r):
        """Reduce partition r as the bincode 1.2.1 blob vega stores in SHUFFLE_CACHE (bytes)."""
        n = ctypes.c_uint64()
        L.check(self._lib.vb_shuffle_reduce_blob_size(self._h, r, ctypes.byref(n)))
        buf = np.empty(n.value, dtype=np.uint8)
        L.check(self._lib.vb_shuffle_reduce_blob(self._h, r, buf.ctypes.data_as(ctypes.c_void_p), L.VB_HOST))
        return buf.tobytes()

    def map_blob(self, map_id, blob):
        """Submit one map-side-combined bucket (bincode blob, bytes) as the output of map task `map_id`."""
        buf = np.frombuffer(blob, dtype=np.uint8)
        L.check(self._lib.vb_shuffle_map_blob(self._h, map_id, buf.ctypes.data_as(ctypes.c_void_p), len(buf), L.VB_HOST))

    def stats(self):
        st = L.vb_stats()
        L.check(self._lib.vb_shuffle_stats(self._h, ctypes.byref(st)))
        d = {f: getattr(st, f) for f, _ in st._fields_}
        kt = {}
        for i, name in enumerate(L.KERNEL_CLASSES):
            ms, n = ctypes.c_double(), ctypes.c_uint64()
            L.check(self._lib.vb_shuffle_kernel_time(self._h, i, ctypes.byref(ms), ctypes.byref(n)))
            kt[name] = {"ms": ms.value, "launches": n.value}
        d["kernels"] = kt
        return d

    def free(self):
        if self._h and self.sc._h:
            self._lib.vb_shuffle_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Grouped:
    """Result of group_by_key: CSR over all partitions in partition order.
    `to_list()` gives the reference's Vec<(K, Vec<V>)>."""

    def __init__(self, keys, offsets, vals):
        self.keys, self.offsets, self.vals = keys, offsets, vals

    def to_list(self):
        o = self.offsets
        return [(self.keys[i].item(), self.vals[int(o[i]):int(o[i + 1])]) for i in range(len(self.keys))]

    def to_dict(self):
        return {k: v for k, v in self.to_list()}

    def __len__(self):
        return len(self.keys)


class _Base:
    def number_of_splits(self):
        return self.num_slices


class ShuffledRdd(_Base):
    """ShuffledRdd<K,V,C> (src/rdd/shuffled_rdd.rs): lazy; `collect()` runs the job."""

    def __init__(self, parent, agg_name, num_splits, hint=0):
        if num_splits < 1:
            raise ValueError("num_splits must be >= 1")
        self.parent, self.agg_name, self.num_slices, self.hint = parent, agg_name, num_splits, hint
        self.sc = parent.sc
        self._sh = None

    def _run(self):
        if self._sh is not None:
            return self._sh
        p = self.parent
        starts = slice_starts(p.n, p.num_slices)
        vcode = p.vals.code if p.vals is not None else (p.keys.code if p.keys.rows else L.VB_U64)
        sh = Shuffle(self.sc, len(starts) - 1, self.num_slices, p.keys.code, vcode, _AGG[self.agg_name],
                     key_width=p.keys.key_width, hint=self.hint)
        sh.has_payload = p.vals is not None or p.keys.rows
        for m in range(len(starts) - 1):                    # map stage
            sh.map(m, p.keys, p.vals, int(starts[m]), int(starts[m + 1]))
        sh.seal()                                           # register_map_outputs
        self._sh = sh
        return sh

    def compute(self, split):
        return self._run().reduce(split)

    def collect(self):
        sh = self._run()
        parts = [sh.reduce(r) for r in range(self.num_slices)]     # result stage, partition order
        if self.agg_name in ("group", "cogroup"):
            keys = np.concatenate([p[0] for p in parts])
            vals = np.concatenate([p[2] for p in parts])
            offs, base = [], 0
            for p in parts:
                offs.append(p[1][:-1].astype(np.uint64) + np.uint64(base))
                base += len(p[2])
            offs.append(np.array([base], dtype=np.uint64))
            return Grouped(keys, np.concatenate(offs), vals)
        comb = None if parts[0][1] is None else np.concatenate([p[1] for p in parts])
        return np.concatenate([p[0] for p in parts]), comb

    def stats(self):
        return self._run().stats()


class JoinedRdd(_Base):
    """`a.join(b, num_splits)` (src/rdd/pair_rdd.rs:104-121): cogroup of two Vec-append
    shuffles + per-key cross product, inner join."""

    def __init__(self, left, right, num_splits):
        self.left, self.right, self.num_slices, self.sc = left, right, num_splits, left.sc
        self._shs = None

    def _run(self):
        if self._shs is None:
            a = ShuffledRdd(self.left, "cogroup", self.num_slices)
            b = ShuffledRdd(self.right, "cogroup", self.num_slices)
            if self.left.keys.key_width != self.right.keys.key_width:
                raise TypeError("join sides have different key types")
            self._shs = (a._run(), b._run())
        return self._shs

    def compute(self, split):
        a, b = self._run()
        lib = self.sc._lib
        n = ctypes.c_uint64()
        L.check(lib.vb_join_size(a._h, b._h, split, ctypes.byref(n)))
        k = np.empty(n.value, dtype=_NP_OF[a.kcode])
        v = np.empty(n.value, dtype=_NP_OF[a.vcode])
        w = np.empty(n.value, dtype=_NP_OF[b.vcode])
        p = lambda x: x.ctypes.data_as(ctypes.c_void_p)
        L.check(lib.vb_join(a._h, b._h, split, p(k), p(v), p(w), L.VB_HOST))
        return k, v, w

    def collect(self):
        parts = [self.compute(r) for r in range(self.num_slices)]
        return tuple(np.concatenate([p[i] for p in parts]) for i in range(3))

    def cogroup_partition(self, split):
        """cogroup() of one partition on the device (vb_cogroup): (keys, offs_a, vals_a, offs_b, vals_b).  Keys in union
        order — this side's keys in its CSR order, then the keys only `other` has; each key's values per side in input
        order, an empty list on the side that lacks the key.  Offsets are partition-local CSR (n_keys + 1 entries)."""
        a, b = self._run()
        lib = self.sc._lib
        nk, na, nb = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
        L.check(lib.vb_cogroup_size(a._h, b._h, split, ctypes.byref(nk), ctypes.byref(na), ctypes.byref(nb)))
        keys = np.empty(nk.value, dtype=_NP_OF[a.kcode])
        offs_a = np.empty(nk.value + 1, dtype=np.uint64)
        offs_b = np.empty(nk.value + 1, dtype=np.uint64)
        vals_a = np.empty(na.value, dtype=_NP_OF[a.vcode])
        vals_b = np.empty(nb.value, dtype=_NP_OF[b.vcode])
        p = lambda x: x.ctypes.data_as(ctypes.c_void_p)
        L.check(lib.vb_cogroup(a._h, b._h, split, p(keys), p(offs_a), p(vals_a), p(offs_b), p(vals_b), L.VB_HOST))
        return keys, offs_a, vals_a, offs_b, vals_b

    def cogroup_collect(self):
        """cogroup(): per partition, the union of keys with both value lists (co_grouped_rdd.rs:206-249)."""
        a, b = self._run()
        out = []
        for r in range(self.num_slices):
            keys, oa, va, ob, vb = self.cogroup_partition(r)
            n_left = int(np.count_nonzero(np.diff(oa)))      # union order: every left key has >= 1 left value, the rest none
            ks = keys[:n_left].tolist() + keys[n_left:].view(_NP_OF[b.kcode]).tolist()
            oa, ob = oa.tolist(), ob.tolist()
            out.extend((k, (va[oa[i]:oa[i + 1]], vb[ob[i]:ob[i + 1]])) for i, k in enumerate(ks))
        return out


class OuterJoinedRdd(_Base):
    """`a.left_outer_join(b, n)` / `right_outer_join` / `full_outer_join` (Spark semantics; the reference has no outer
    joins): the cogroup of both sides, keeping keys that have values on one side only.  Rows of a key are contiguous,
    keys in the cogroup's union order, `for v in vs { for w in ws }` per matched key."""

    _KINDS = {"left": L.VB_JOIN_LEFT_OUTER, "right": L.VB_JOIN_RIGHT_OUTER, "full": L.VB_JOIN_FULL_OUTER}

    def __init__(self, left, right, num_splits, how):
        self.joined = JoinedRdd(left, right, num_splits)
        self.kind = self._KINDS[how]
        self.num_slices, self.sc = num_splits, left.sc

    def compute(self, split):
        """(k, v, w, valid): an absent v or w is 0 and its bit (VB_JOIN_HAS_V = 1, VB_JOIN_HAS_W = 2) clear in valid."""
        a, b = self.joined._run()
        lib = self.sc._lib
        n = ctypes.c_uint64()
        L.check(lib.vb_join_outer_size(a._h, b._h, split, self.kind, ctypes.byref(n)))
        k = np.empty(n.value, dtype=_NP_OF[a.kcode])
        v = np.empty(n.value, dtype=_NP_OF[a.vcode])
        w = np.empty(n.value, dtype=_NP_OF[b.vcode])
        valid = np.empty(n.value, dtype=np.uint8)
        p = lambda x: x.ctypes.data_as(ctypes.c_void_p)
        L.check(lib.vb_join_outer(a._h, b._h, split, self.kind, p(k), p(v), p(w), p(valid), L.VB_HOST))
        return k, v, w, valid

    def collect(self):
        parts = [self.compute(r) for r in range(self.num_slices)]
        return tuple(np.concatenate([p[i] for p in parts]) for i in range(4))

    def to_list(self):
        """Spark's shape: [(k, (v or None, w or None))]."""
        k, v, w, valid = self.collect()
        has_v, has_w = (valid & L.VB_JOIN_HAS_V) != 0, (valid & L.VB_JOIN_HAS_W) != 0
        return [(kk, (vv if hv else None, ww if hw else None))
                for kk, vv, ww, hv, hw in zip(k.tolist(), v.tolist(), w.tolist(), has_v.tolist(), has_w.tolist())]


class PairRdd(_Base):
    """PairRdd<K,V> source (ParallelCollection of (K,V)); methods per src/rdd/pair_rdd.rs."""

    def __init__(self, sc, keys, vals, num_slices):
        if num_slices < 1:
            raise ValueError("Number of slices should be greater than or equal to 1")
        if vals is not None and vals.n != keys.n:
            raise ValueError("keys and values differ in length")
        self.sc, self.keys, self.vals, self.num_slices, self.n = sc, keys, vals, num_slices, keys.n

    def group_by_key(self, num_splits):
        return ShuffledRdd(self, "group", num_splits)

    def reduce_by_key(self, op, num_splits, hint=0):
        if op not in ("sum", "min", "max"):
            raise ValueError("reduce_by_key takes a named op: 'sum' | 'min' | 'max' (closures cannot cross the C ABI)")
        return ShuffledRdd(self, op, num_splits, hint)

    def count_by_key(self, num_splits=None, hint=0):
        return ShuffledRdd(self, "count", num_splits or self.num_slices, hint)

    def join(self, other, num_splits):
        return JoinedRdd(self, other, num_splits)

    def cogroup(self, other, num_splits):
        return JoinedRdd(self, other, num_splits)

    def left_outer_join(self, other, num_splits):
        return OuterJoinedRdd(self, other, num_splits, "left")

    def right_outer_join(self, other, num_splits):
        return OuterJoinedRdd(self, other, num_splits, "right")

    def full_outer_join(self, other, num_splits):
        return OuterJoinedRdd(self, other, num_splits, "full")

    def sort_by_key(self, num_splits):
        return ShuffledRdd(self, "sort", num_splits)

    def partition_by_key(self, num_splits):
        """partition_by_key (pair_rdd.rs:157-171): shuffle with the Vec-append aggregator, then
        flatten the values; `glom()` = values per partition."""
        return _Repartitioned(ShuffledRdd(self, "group", num_splits))


class _Repartitioned:
    def __init__(self, sh):
        self.sh = sh

    def glom(self):
        s = self.sh._run()
        return [s.reduce(r)[2] for r in range(self.sh.num_slices)]

    def collect(self):
        return np.concatenate(self.glom()) if self.sh.num_slices else np.empty(0)


class Rdd(_Base):
    """Key-only source RDD: the shuffle-backed ops of src/rdd/rdd.rs."""

    def __init__(self, sc, keys, num_slices):
        if num_slices < 1:
            raise ValueError("Number of slices should be greater than or equal to 1")
        self.sc, self.keys, self.num_slices, self.n = sc, keys, num_slices, keys.n

    def count_by_value(self):
        """rdd.rs:450-459: map(x → (x, 1u64)).reduce_by_key(+, number_of_splits)."""
        n_splits = len(slice_starts(self.n, self.num_slices)) - 1
        return ShuffledRdd(PairRdd(self.sc, self.keys, None, self.num_slices), "count", n_splits)

    def distinct(self, num_partitions=None):
        """rdd.rs:502-522: reduce_by_key on (Some(x), None), keys kept."""
        n_splits = num_partitions or (len(slice_starts(self.n, self.num_slices)) - 1)
        return _Distinct(ShuffledRdd(PairRdd(self.sc, self.keys, None, self.num_slices), "count", n_splits))

    distinct_with_num_partitions = distinct

    def sort(self, num_splits):
        return ShuffledRdd(PairRdd(self.sc, self.keys, None, self.num_slices), "sort", num_splits)

    def intersection(self, other, num_splits=None):
        """rdd.rs:852-946 `intersection` / `intersection_with_num_partitions`: the reference cogroups
        (x, None) of both sides and keeps the keys with `v1.len() >= 1 && v2.len() >= 1` — each key once."""
        return _SetOp(self, other, num_splits or self.number_of_splits_exact(), "and")

    intersection_with_num_partitions = intersection

    def subtract(self, other, num_splits=None):
        """rdd.rs:838-901 `subtract`: keys of self whose cogroup with `other` has exactly one non-empty side
        (`(v1.len() >= 1) ^ (v2.len() >= 1)`), intersected with self — i.e. the distinct keys of self not in other."""
        return _SetOp(self, other, num_splits or self.number_of_splits_exact(), "a_not_b")

    subtract_with_num_partition = subtract

    def group_by(self, func, num_splits=None):
        """rdd.rs:957-990 `group_by(func)`: map(x -> (func(x), x)).group_by_key(num_splits).  `func` is a
        vectorised key function over the item array (numpy / torch), e.g. `lambda x: np.sign(x) + 1`
        — a scalar closure cannot cross into CUDA (SURVEY.md F4), the key column it produces can."""
        owner = self.keys.owner
        k = func(owner)
        if not _is_torch(k):
            k = np.asarray(k)
        return PairRdd(self.sc, _Col(k), _Col(owner, role="value"), self.num_slices).group_by_key(num_splits or self.number_of_splits_exact())

    group_by_with_num_partitions = group_by

    def number_of_splits_exact(self):
        return len(slice_starts(self.n, self.num_slices)) - 1


class _SetOp:
    """intersection / subtract as ONE tagged shuffle: side A rows carry the value 1, side B rows 2^32, the
    map-side combine + merge (hash_agg) sums them, and a key's sum says which sides it occurred on — the same
    information the reference reads off the two Vec lengths of its cogroup (rdd.rs:877-884, :925-932)."""

    def __init__(self, a, b, num_splits, mode):
        if a.keys.key_width != b.keys.key_width or a.keys.code != b.keys.code:
            raise TypeError("both sides must have the same item type")
        self.a, self.b, self.num_slices, self.mode, self.sc = a, b, num_splits, mode, a.sc
        self._sh = None

    @staticmethod
    def _const_like(col, value):
        if _is_torch(col.owner):
            import torch
            t = torch.full((col.n,), value, dtype=torch.int64, device=col.owner.device)
            return _Col(t, role="value")
        return _Col(np.full(col.n, value, dtype=np.uint64), role="value")

    def _run(self):
        if self._sh is not None:
            return self._sh
        sa, sb = slice_starts(self.a.n, self.a.num_slices), slice_starts(self.b.n, self.b.num_slices)
        na, nb = len(sa) - 1, len(sb) - 1
        sh = Shuffle(self.sc, na + nb, self.num_slices, self.a.keys.code, L.VB_U64, L.VB_AGG_SUM, key_width=self.a.keys.key_width)
        ta, tb = self._const_like(self.a.keys, 1), self._const_like(self.b.keys, 1 << 32)
        for m in range(na):
            sh.map(m, self.a.keys, ta, int(sa[m]), int(sa[m + 1]))
        for m in range(nb):
            sh.map(na + m, self.b.keys, tb, int(sb[m]), int(sb[m + 1]))
        sh.seal()
        self._sh = sh
        return sh

    def compute(self, split):
        k, c = self._run().reduce(split)
        c = c.view(np.uint64)
        in_a, in_b = (c & np.uint64(0xFFFFFFFF)) > 0, (c >> np.uint64(32)) > 0
        return k[in_a & in_b] if self.mode == "and" else k[in_a & ~in_b]

    def collect(self):
        parts = [self.compute(r) for r in range(self.num_slices)]
        return np.concatenate(parts) if parts else np.empty(0)


class _Distinct:
    def __init__(self, sh):
        self.sh = sh

    def collect(self):
        return self.sh.collect()[0]
