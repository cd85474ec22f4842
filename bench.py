#!/usr/bin/env python
"""bench.py — headline benchmark of BASELINE.json: reduce_by_key on 1e9 synthetic (u64,u64) pairs,
1e6 distinct keys, sum, 8 map → 8 reduce partitions, on one B200 (configs[1]); N>1 = the same
per-GPU workload on every rank (weak scaling) with the combined rows exchanged by one all-to-all-v.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: create the shuffle, run the M map tasks
(map-side combine: hash_agg_kernel), seal (merge + partition the combined rows).  `value` is
whole-job pairs/s with the input resident in HBM; `e2e` is the same metric through the public API
(vega_b200.Context.parallelize(...).reduce_by_key(...).collect()) with pinned HOST buffers, the
H2D copy of the rows and the D2H copy of the result inside the timed region.
`--impl reference` times the reference's CPU algorithm (oracle port: vega is Rust and cannot be
built here) on the host cores on a bounded sample of the same workload.
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALG_BYTES_PER_PAIR = 16.0       # SURVEY §8(d): 16 B read per pair (+16 B per distinct key written)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", delete=False, suffix=".csv")
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1])); mx.append(float(p[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def cpu_port_run(n_rows, D, M, R, threads, steps, warmup, warm_rows=None):
    """The reference's CPU algorithm (oracle/vega_oracle.c) on `n_rows` rows of the same generator.
    warm_rows: warm-up steps run on this many leading rows (the CPU has no caches to warm at these sizes;
    it keeps a full-size reference run within minutes)."""
    from oracle import oracle as O
    keys, vals = O.gen_uniform(0, n_rows, D, 1, 2)
    times = []
    w = min(warm_rows or n_rows, n_rows)
    for i in range(warmup + steps):
        if i < warmup:
            O.shuffle_timed("sum", keys[:w], vals[:w], M, R, threads=threads)
            continue
        dt, nk = O.shuffle_timed("sum", keys, vals, M, R, threads=threads)
        times.append(dt)
    return times


def bench_config(workload):
    """`config` of the JSON line — the same dict for both arms (the reference arm times the same workload)."""
    return {"workload": workload, "layout": "AoS 16-byte rows resident in HBM", "op": "sum",
            "l2": "inputs (16 GB/GPU) larger than the 126 MB L2; no flush needed",
            "timing": "CUDA events on the library's stream, max over ranks"}


def traffic_lookup(kernel, rows_per_launch, table_slots):
    """Measured DRAM bytes per launch of the dominant kernel from the committed ncu table
    (profiles/traffic_table.json, written from `ncu --set full` captures); None when this exact
    kernel/config has no capture — never a stale constant."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic_table.json")) as f:
            tab = json.load(f)
    except Exception:
        return None, None
    for e in tab.get("entries", []):
        if e["kernel"] == kernel and abs(e["rows_per_launch"] - rows_per_launch) < 1 and e["table_slots"] == table_slots:
            return e["dram_bytes_per_launch"], e["source"]
    return None, None


DUMP_MAX_BYTES = 64 << 20


def u64_halves(a):
    """(n, 2) float64 of [high 32 bits, low 32 bits]: exact, where a cast of a 64-bit key to float64 is not."""
    import numpy as np
    a = a.view(np.uint64)
    return np.stack([(a >> np.uint64(32)).astype(np.float64), (a & np.uint64(0xFFFFFFFF)).astype(np.float64)], axis=1)


def dump_outputs(out_dir, parts, suffix=""):
    """Writes what the caller of the timed path receives from its last step: for each reduce partition this
    rank owns (in order), the (key, sum) rows of Shuffle.reduce(r).  Rows are sorted by key inside each
    partition, since their order there is unspecified, so that two builds compare row for row.
    keys.npy / sums.npy: (n, 2) float64 u64 halves (u64_halves); partition_rows.npy: rows per partition.
    Beyond DUMP_MAX_BYTES a fixed, seeded sample of rows is kept and sample_index.npy names them."""
    import numpy as np
    keys, sums = [], []
    for k, c in parts:
        o = np.argsort(k.view(np.uint64), kind="stable")
        keys.append(k.view(np.uint64)[o])
        sums.append(c.view(np.uint64)[o])
    out = {"partition_rows": np.array([len(k) for k in keys], dtype=np.float64)}
    keys, sums = np.concatenate(keys), np.concatenate(sums)
    # 32 B of keys + sums and 8 B of sample index per row; 4 files with a .npy header of at most 256 B each
    cap = (DUMP_MAX_BYTES - 4 * 256 - out["partition_rows"].nbytes) // 40
    if len(keys) > cap:
        idx = np.sort(np.random.default_rng(0).choice(len(keys), cap, replace=False))
        keys, sums = keys[idx], sums[idx]
        out["sample_index"] = idx.astype(np.float64)
    out["keys"], out["sums"] = u64_halves(keys), u64_halves(sums)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=float, default=1e9, help="pairs per GPU")
    ap.add_argument("--distinct", type=float, default=1e6)
    ap.add_argument("--maps", type=int, default=8, help="map partitions per GPU")
    ap.add_argument("--reduces", type=int, default=8, help="reduce partitions per GPU")
    ap.add_argument("--e2e-rows", type=float, default=None)
    ap.add_argument("--cpu-rows", type=float, default=None, help="rows per CPU step (default: full size for --impl reference if it fits in minutes, 1e8 for the in-run baseline)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's reduce_by_key result to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's result: use it with --impl ours")
    n_gpus = args.gpus
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    N, D, M, R = int(args.rows), int(args.distinct), args.maps, args.reduces
    nproc = os.cpu_count() or 1
    workload = f"reduce_by_key(sum) {N:.0e} (u64,u64) pairs/GPU, {D:.0e} distinct keys, {M} map x {R * max(world, 1)} reduce partitions"

    # ---------------------------------------------------------------- reference arm (CPU port)
    if args.impl == "reference":
        if rank != 0:
            return 0
        threads = min(M, nproc)
        # Full-size steps (the configuration the metric is quoted on) when K of them fit in ~4 minutes at the
        # rate a 1e8-row calibration step shows, else 1e8 rows per step (labelled, not extrapolated).
        from oracle import oracle as O
        n_cal = int(min(1e8, N))
        if args.cpu_rows:
            n_cpu = int(min(args.cpu_rows, N))
            n_cal = min(n_cal, n_cpu)
        else:
            ck, cv = O.gen_uniform(0, n_cal, D, 1, 2)
            cal_dt, _ = O.shuffle_timed("sum", ck, cv, M, R, threads=threads)
            del ck, cv
            est_full = cal_dt * (N / n_cal) * args.steps
            try:
                avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
            except Exception:
                avail = 0
            n_cpu = N if (est_full <= 420.0 and avail > 40 * N) else n_cal
        times = cpu_port_run(n_cpu, D, M, R, threads, args.steps, args.warmup, warm_rows=n_cal)
        tot = sum(times)
        val = n_cpu * len(times) / tot
        line = {
            "impl": "reference", "metric": "reduce_by_key (K,V) pairs/sec", "value": val, "unit": "pairs/s",
            "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": bench_config(workload),
            "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": threads, "kind": "port", "host_cores": nproc,
                             "sample": f"{n_cpu:.0e} pairs per timed step ({'the full configuration' if n_cpu == N else 'bounded sample of the same generator'}; warm-up steps on {n_cal:.0e} pairs), {M}x{R} partitions, C restatement of vega's map-side combine + reduce-side merge (oracle/vega_oracle.c); vega itself is Rust and cannot be built in this image"},
            "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        if nproc > threads:     # informational: the same port with one partition per host core (not this arm's config)
            t2 = cpu_port_run(n_cal, D, nproc, nproc, nproc, 2, 1)
            line["cpu_baseline"]["all_cores"] = {"value": n_cal * len(t2) / sum(t2), "unit": "pairs/s", "cores": nproc,
                                                 "partitions": f"{nproc}x{nproc}", "sample": f"{n_cal:.0e} pairs"}
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------- our arm
    import numpy as np
    import torch

    import vega_b200 as vb
    from vega_b200 import _lib as L
    from vega_b200 import dist as vdist

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    pg = None
    if world > 1:
        import torch.distributed as tdist
        tdist.init_process_group("nccl", device_id=torch.device(dev))
        pg = tdist.group.WORLD

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize()

    sc = vb.Context(local_rank, profile=True)
    if world > 1:
        sc.comm_init(rank, world)      # torch.distributed only bootstraps the NCCL id; the exchange runs inside libvega_b200
    engine = vdist.CudaEngine(sc)
    stream = sc.stream()
    rows = torch.empty((N, 2), dtype=torch.int64, device=dev)       # 16 B/pair resident in HBM
    sc.gen_pairs(out_rows=rows, first=rank * N, n=N, mode="uniform", n_distinct=D, seed_k=1, seed_v=2)
    starts = vb.slice_starts(N, M)
    n_map_global, n_red_global = M * world, R * world
    lo, _ = vdist.map_block(rank, world, n_map_global)
    maps = [(lo + m, rows[int(starts[m]):int(starts[m + 1])], None) for m in range(len(starts) - 1)]

    def step(stats=None):
        sh = vdist.run_shuffle(engine, maps, n_map_global, n_red_global, L.VB_U64, L.VB_U64, L.VB_AGG_SUM, rank, world,
                               group=pg, stats=stats)
        return sh

    for _ in range(args.warmup):
        step().free()
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    agg = {"hot_ms": 0.0, "hot_launches": 0, "hot_rows": 0, "launches": 0, "map_ms": 0.0, "seal_ms": 0.0}
    xstats = {}
    kept = []
    ev0.record(stream)
    t0 = time.perf_counter()
    step_stats = []
    for i in range(args.steps):
        sh = step(xstats)
        step_stats.append(sh.stats())          # reads the event timers of this step
        if i + 1 < args.steps:
            sh.free()                          # steady state: the next step reuses this step's pool memory
        else:
            kept.append(sh)                    # last step's result stays for the parity check below
    ev1.record(stream)
    barrier()
    t1 = time.perf_counter()
    clocks = sampler.stop() if rank == 0 else None
    ms_dev = ev0.elapsed_time(ev1)
    ms_total = max(ms_dev, 0.0)
    n_keys_out = 0
    for st in step_stats:
        agg["hot_ms"] += st["hot_kernel_ms"]; agg["hot_launches"] += st["hot_kernel_launches"]
        agg["hot_rows"] += st["hot_kernel_rows"]; agg["launches"] += st["kernel_launches"]
        agg["map_ms"] += st["map_ms"]; agg["seal_ms"] += st["seal_ms"]
        n_keys_out = st["rows_out"]
    # parity property on the last step (size-independent): every key of the universe present exactly
    # once across this rank's partitions and the sums add up to the sum of all values
    last = kept[-1]
    chk_keys, chk_sum = 0, 0
    last_parts = []
    for r in vdist.owned_partitions(rank, world, n_red_global):
        k, c = last.reduce(r)
        chk_keys += len(k); chk_sum += int(c.sum(dtype=np.uint64))
        last_parts.append((k, c))
    for sh in kept:
        sh.free()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_parts, f"_rank{rank}" if world > 1 else "")
    del last_parts
    if world > 1:
        t = torch.tensor([ms_total, float(chk_keys), float(chk_sum % (1 << 52))], dtype=torch.float64, device=dev)
        tmax = t.clone(); tdist.all_reduce(tmax, op=tdist.ReduceOp.MAX)
        tsum = t.clone(); tdist.all_reduce(tsum, op=tdist.ReduceOp.SUM)
        ms_total = float(tmax[0]); chk_keys = int(tsum[1])
    total_vals = None
    if world == 1:
        total_vals = int(rows[:, 1].sum().item())
        expect_all = N >= 40 * D          # coupon collector: every rank of the key universe occurs
        assert (chk_keys == D if expect_all else chk_keys <= D) and chk_sum == total_vals, \
            f"parity property failed: keys {chk_keys} (D={D}), sum {chk_sum} != {total_vals}"
    ms_per_step = ms_total / args.steps
    value = (N * world) / (ms_per_step * 1e-3)

    out = None
    if rank == 0:
        peak, peak_src = peaks()
        rows_per_launch = agg["hot_rows"] / max(agg["hot_launches"], 1)
        avg_launch_ms = agg["hot_ms"] / max(agg["hot_launches"], 1)
        alg_bytes = rows_per_launch * ALG_BYTES_PER_PAIR + 16.0 * D
        achieved = alg_bytes / (avg_launch_ms * 1e-3) / 1e9 if avg_launch_ms > 0 else 0.0
        variant = step_stats[-1].get("hot_kernel_variant", 0)
        kernel_name = "hash_agg_bulk_kernel<IN_AOS,OPK_ADD_U64>" if variant else "hash_agg_kernel<IN_AOS,OPK_ADD_U64>"
        traffic, traffic_src = traffic_lookup(kernel_name, rows_per_launch, step_stats[-1].get("table_slots", 0))
        out = {
            "metric": "reduce_by_key (K,V) pairs/sec", "value": value, "unit": "pairs/s", "n_gpus": n_gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": bench_config(workload),
            "clocks": clocks,
            "gpu_launches": agg["launches"],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "kernel": kernel_name,
                         "design_roof": {"what": "an exact streaming aggregation into an L2-resident table needs >= 2 L2 requests per row (probe + RED); measured ceilings with no input stream at all (bench_micro/micro_r2.cu, profiles/r2_micro_request_roof.log): random 32 B loads 2.87e11/s (SM L1TEX->XBAR port, 1 request/clk/SM, l1tex__m_l1tex2xbar_req_cycles_active 97 %), 64-bit REDs 1.97e11/s (lts__t_tag_requests-bound), load+RED pairs 1.255e11 rows/s",
                                         "rows_per_s": 1.255e11, "GBps": 1.255e11 * 16 / 1e9, "frac_of_hbm_peak": 1.255e11 * 16 / 1e9 / peak,
                                         "achieved_frac_of_design_roof": achieved / (1.255e11 * 16 / 1e9)},
                         "rows_per_launch": rows_per_launch, "avg_launch_ms": avg_launch_ms, "peak_source": peak_src,
                         "step_share": agg["hot_ms"] / max(ms_total, 1e-9),
                         "whole_step_frac": (N * ALG_BYTES_PER_PAIR + 16.0 * D) / (ms_per_step * 1e-3) / 1e9 / peak},
            "phases_ms_per_step": {"map": agg["map_ms"] / args.steps, "seal": agg["seal_ms"] / args.steps},
            "parity": {"distinct_keys_out": chk_keys, "sum_matches_input": True if world == 1 else None},
        }
        if world > 1:
            sent = xstats.get("sent_rows") or 0
            xms = (xstats.get("exchange_ms") or 0.0) / max(xstats.get("exchanges", 1), 1)
            out["exchange"] = {"collective": "inside libvega_b200 (vb_shuffle_exchange): count all-gather + ONE ncclGroupStart/Send/Recv/GroupEnd carrying both columns of the map-side-combined rows, on the library's stream",
                               "rows_sent_per_rank_per_step": sent, "bytes_sent_per_rank_per_step": 16 * sent,
                               "ms_per_step": xms, "GBps_per_rank": (16 * sent / (xms * 1e-3) / 1e9) if xms > 0 else None,
                               "host_wall_ms_per_step": {k: (xstats.get(k) or 0.0) / max(xstats.get("exchanges", 1), 1)
                                                         for k in ("prepare_wall_ms", "counts_wall_ms", "post_wall_ms")},
                               "note": "latency-bound: map-side combine shrinks 16 GB/rank of rows to <= 16 MB"}

    # ---------------------------------------------------------------- e2e (public API, host buffers)
    if not args.no_e2e:
        n_e2e = int(args.e2e_rows) if args.e2e_rows else N
        host = None
        while host is None and n_e2e >= 1 << 20:
            try:
                host = torch.empty((n_e2e, 2), dtype=torch.int64, pin_memory=True)
            except Exception:
                n_e2e //= 2
        host.copy_(rows[:n_e2e])
        torch.cuda.synchronize()
        sc.set_profile(False)
        hostnp = host.numpy()

        def e2e_step():
            if world == 1:
                k, c = sc.parallelize(hostnp, M).reduce_by_key("sum", R).collect()
                return len(k), 0, 16 * len(k)
            st = vb.slice_starts(n_e2e, M)
            mp = [(lo + m, hostnp[int(st[m]):int(st[m + 1])], None) for m in range(len(st) - 1)]
            sh = vdist.run_shuffle(engine, mp, n_map_global, n_red_global, L.VB_U64, L.VB_U64, L.VB_AGG_SUM, rank, world,
                                   group=pg)
            nk = 0
            for r in vdist.owned_partitions(rank, world, n_red_global):
                k, c = sh.reduce(r)
                nk += len(k)
            sh.free()
            return nk, 0, 16 * nk

        for _ in range(max(1, min(args.warmup, 2))):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        d2h = 0
        e_steps = max(1, min(args.steps, 3))
        for _ in range(e_steps):
            _, _, b = e2e_step()
            d2h = b
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
            dt = float(t[0])
        # the PCIe ceiling of this box for the same bytes: a bare pinned-host -> device copy (no library involved)
        copy_gbps = None
        if world == 1:
            rows[:n_e2e].copy_(host, non_blocking=True); torch.cuda.synchronize()
            tc = time.perf_counter()
            rows[:n_e2e].copy_(host, non_blocking=True); torch.cuda.synchronize()
            copy_gbps = 16 * n_e2e / (time.perf_counter() - tc) / 1e9
        if rank == 0:
            e2e_val = n_e2e * world * e_steps / dt
            out["e2e"] = {"value": e2e_val, "unit": "pairs/s", "h2d_bytes_per_step": 16 * n_e2e,
                          "d2h_bytes_per_step": d2h, "rows_per_gpu": n_e2e, "steps": e_steps,
                          "api": "Context.parallelize(pinned host rows, M).reduce_by_key('sum', R).collect()",
                          "h2d_GBps": 16 * e2e_val / max(world, 1) / 1e9, "pcie_copy_only_GBps": copy_gbps,
                          "frac_of_pcie_copy": (16 * e2e_val / 1e9 / copy_gbps) if copy_gbps else None,
                          "note": "PCIe-bound: the rows cross the host link once; staging is double-buffered on a copy stream, the map-side combine of chunk i runs under the copy of chunk i+1"}
        del host

    # ---------------------------------------------------------------- CPU baseline (rank 0, N=1)
    if rank == 0 and world == 1 and not args.no_cpu:
        n_cpu = int(min(args.cpu_rows or 1e8, N))
        threads = min(M, nproc)
        times = cpu_port_run(n_cpu, D, M, R, threads, 2, 1)
        out["cpu_baseline"] = {"value": n_cpu * len(times) / sum(times), "unit": "pairs/s", "cores": threads, "kind": "port",
                               "host_cores": nproc, "cores_note": "vega runs one task per partition: 8 map then 8 reduce tasks, so 8 threads is all this config can use",
                               "sample": f"first {n_cpu:.0e} pairs of the same generator, {M}x{R} partitions, 2 timed runs; C restatement of vega's algorithm (oracle/vega_oracle.c), not vega itself (Rust, unbuildable here)"}
        if nproc > threads:     # informational: one partition per host core instead of the config's 8
            t2 = cpu_port_run(n_cpu, D, nproc, nproc, nproc, 2, 1)
            out["cpu_baseline"]["all_cores"] = {"value": n_cpu * len(t2) / sum(t2), "unit": "pairs/s", "cores": nproc,
                                                "partitions": f"{nproc}x{nproc}"}
    if rank == 0:
        print(json.dumps(out))
    sc.close()
    if world > 1:
        tdist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
