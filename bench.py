#!/usr/bin/env python
"""bench.py -- the headline benchmark of BASELINE.json: src-dst pairs resolved per second by
iterativelength on an R-MAT scale-22 CSR (4M vertices / 64M edges, int32 on device), 1024 hashed
src-dst pairs per GPU, with the edges-traversed roofline and the reference's CPU operator beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" = one pass of the hot path (pgq_iterativelength) over one batch of P pairs on the resident
CSR.  `value` is timed with the pairs already in HBM (pgq_iterativelength_device on torch's current
stream, CUDA events); `e2e` starts from HOST columns with the copies inside the timed region: at N = 1
the host-pointer C ABI (pgq_iterativelength: pairs H2D + results D2H inside the call), at N > 1
sharding.ShardedLengths (pinned staging, H2D of all pairs, this rank's shard of the searches, one NCCL
all_reduce(MAX) of the result column on the device, D2H).  Prints ONE JSON line on rank 0.

--dump-outputs DIR writes, on rank 0, the result columns of the last timed step as DIR/<name>.npy: `length` (float64,
-1 where there is no path) and `valid` (float32) of the headline, and `c3_*` / `c5_*` of the sub-records.  The
graphs and pairs depend only on the arguments, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from duckpgq_extension_b200 import datagen  # noqa: E402

METRIC = "src-dst pairs/sec (iterativelength, R-MAT CSR)"
UNIT = "pairs/s"
CACHE = os.environ.get("PGQ_CACHE_DIR", "/tmp/duckpgq_b200_cache")


def measured_peak_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            pass
    return local_rank


def load_graph(scale: int, rank: int, world: int, dist):
    """R-MAT edges: rank 0 generates (or finds the cache), the other ranks read the cache."""
    if world > 1:
        if rank == 0:
            g = datagen.rmat_edges_cached(scale, CACHE)
        dist.barrier()
        if rank != 0:
            g = datagen.rmat_edges_cached(scale, CACHE)
        return g
    return datagen.rmat_edges_cached(scale, CACHE)


DUMP_BYTES = 60 << 20  # the arrays of one dump; with the .npy headers well under 64 MB


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """arrays: name -> float32 / float64 array, written as out_dir/<name>.npy.  Above DUMP_BYTES in all, every
    array keeps the same share of its rows, chosen by a fixed seed, so two runs still compare row for row."""
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = max(1, a.size * DUMP_BYTES // total)
            a = a[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU operator on this box's host cores
# ------------------------------------------------------------------------------------------------
def pairs_per_ref_step(total_steps: int) -> int:
    # One 512-lane batch per step.  The reference's batch cost hardly depends on how many of the 512
    # lanes are occupied (4.1 s full vs 3.4 s with 64 lanes at R-MAT-22), so a full batch is its best
    # case per pair and is what it gets whenever the run still ends within a few minutes.
    for limit, s in ((40, 512), (80, 256), (160, 128)):
        if total_steps <= limit:
            return s
    return 64


def run_reference(scale: int, n: int, src, dst, steps: int, warmup: int, pairs_per_step: int):
    """-> (pairs_per_s, info dict).  oracle/_ref (the unmodified reference) when present, else the port.
    The reference gets all the host threads it can use: a step is `chunks_per_step` DataChunks of one 512-lane
    batch each, all steps form ONE statement (the CSR is built once) whose chunks DuckDB deals to its threads
    (oracle/ref_runner.py: time_reference_parallel); enough chunks for two rounds over the threads.  Time = the WALL
    time of the searches."""
    from oracle import ref_runner as rr
    cores = os.cpu_count() or 1
    if rr.reference_available():
        threads = rr.usable_threads(n, cores)
        chunks_per_step = max(1, -(-2 * threads // max(steps, 1)))
        chunks = steps * chunks_per_step
        ps, pd = datagen.hashed_pairs(max((chunks + 1) * pairs_per_step, 1), n)
        db = os.path.join(CACHE, f"rmat{scale}.duckdb")
        rr.prepare_database(db, n, src, dst)
        if warmup > 0:  # (page cache, DuckDB's catalog: one small statement)
            rr.time_reference_parallel(db, n, ps, pd, 1, pairs_per_step, threads)
        r = rr.time_reference_parallel(db, n, ps[pairs_per_step:], pd[pairs_per_step:], chunks, pairs_per_step, threads)
        if r["bfs_s"] is None:
            raise RuntimeError("could not read the statement times from the DuckDB profile")
        info = {"kind": "reference", "cores": threads, "host_cores": cores,
                "sample": f"{steps} x {chunks_per_step} DataChunk(s) of one 512-lane batch of {pairs_per_step} pairs "
                          f"(R-MAT-{scale}) in one statement, reference extension in DuckDB, threads={threads} of "
                          f"{cores} host cores (each running batch holds 3 x n x 64 B); time = wall time of the "
                          f"searches = statement {r['total_s']:.2f} s - the same statement over one chunk of NULL "
                          f"sources {r['csr_s']:.2f} s (CSR build); iterativelength Projection {r['thread_s']:.1f} "
                          f"thread-seconds",
                "bfs_s": r["bfs_s"], "statement_s": r["total_s"], "reachable": r["reachable"],
                "pairs": chunks * pairs_per_step}
        return chunks * pairs_per_step / r["bfs_s"], info
    need = (steps + warmup) * pairs_per_step
    ps, pd = datagen.hashed_pairs(max(need, 1), n)
    from oracle import pgq_oracle as orc
    v, e, _ = orc.csr_build(n, src, dst)
    if warmup > 0:
        rr.time_port_steps(n, v, e, ps, pd, min(warmup, 1), pairs_per_step)
    r = rr.time_port_steps(n, v, e, ps[warmup * pairs_per_step:], pd[warmup * pairs_per_step:], steps, pairs_per_step)
    info = {"kind": "port", "cores": 1, "host_cores": cores,
            "sample": f"{steps} x one 512-lane batch of {pairs_per_step} pairs (R-MAT-{scale}), C restatement "
                      f"oracle/pgq_oracle.c, 1 thread", "bfs_s": r["bfs_s"], "reachable": r["reachable"],
            "pairs": steps * pairs_per_step}
    return steps * pairs_per_step / r["bfs_s"], info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=int, default=22, help="R-MAT scale (22 = BASELINE configs[1])")
    ap.add_argument("--pairs", type=int, default=1024, help="pairs per GPU per step")
    ap.add_argument("--lanes", type=int, default=0)
    ap.add_argument("--direction", type=int, default=0)
    ap.add_argument("--alpha", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the c3 / c5 sub-records (R-MAT-24 / R-MAT-26)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result columns of the last timed step as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the GPU arm (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload = (f"RMAT scale-{args.scale} ({1 << args.scale} v / {(1 << args.scale) * 16} e) int32 CSR, "
                f"{args.pairs} hashed src-dst pairs per GPU, iterativelength")
    config = {"workload": workload, "pairs_per_gpu": args.pairs, "rmat_scale": args.scale,
              "csr": "replicated per GPU", "partition": "searches dealt round-robin over the ranks, all_reduce(MAX) of the result columns", "l2": "inputs_exceed_l2 (CSR 0.5 GB + masks, no reuse across steps)"}

    # ---------------------------------------------------------------- reference arm (CPU only)
    if args.impl == "reference":
        if rank != 0:
            return
        n, src, dst = datagen.rmat_edges_cached(args.scale, CACHE)
        pps = pairs_per_ref_step(args.steps + args.warmup)
        value, info = run_reference(args.scale, n, src, dst, args.steps, min(args.warmup, 1), pps)
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * info["bfs_s"] / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
                "data": "synthetic", "config": config, "gpu_launches": 0,
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": info["cores"], "kind": info["kind"],
                                 "sample": info["sample"]},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ---------------------------------------------------------------- our arm (GPU)
    import torch
    import torch.distributed as dist
    from duckpgq_extension_b200 import pgq, sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    n, src, dst = load_graph(args.scale, rank, world, dist)
    m = int(src.shape[0])
    ctx = pgq.Context(local_rank)
    t0 = time.perf_counter()
    csr = pgq.DeviceCSR.build(ctx, n, src, dst)  # create_csr_vertex/create_csr_edge on the device
    torch.cuda.synchronize()
    csr_build_s = time.perf_counter() - t0
    _, _, csr_bytes = csr.info()
    opts = pgq.Options(args.lanes, args.direction, args.alpha)

    P = args.pairs
    total_pairs = world * P
    nsteps = args.warmup + args.steps
    # weak scaling: world x P pairs per step, a FRESH block of hashed pairs every step.  Every rank holds
    # all of them (16 B per pair) and runs the searches whose ordinal is congruent to its rank
    # (pgq_options.shard_*), so the ranks stay balanced however unevenly the pairs that actually need a
    # search are distributed; one all_reduce(MAX) over the result column assembles the answer -- the only
    # collective, issued on a side stream so that step k+1's searches overlap step k's assembly.
    ps_all, pd_all = datagen.hashed_pairs(total_pairs * nsteps, n)
    ps_all = ps_all.reshape(nsteps, total_pairs)
    pd_all = pd_all.reshape(nsteps, total_pairs)
    opts.shard_index, opts.shard_count = (rank, world) if world > 1 else (0, 0)
    d_src = torch.from_numpy(ps_all).to(dev)
    d_dst = torch.from_numpy(pd_all).to(dev)
    d_len = [torch.empty(total_pairs, dtype=torch.int64, device=dev) for _ in range(2)]
    d_val = torch.empty(total_pairs, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()
    side = torch.cuda.Stream(device=dev)
    reduced = [None, None]  # event: the all_reduce that last used the buffer has finished

    def step_device(i):
        buf = d_len[i & 1]
        if reduced[i & 1] is not None:
            stream.wait_event(reduced[i & 1])
        stt = csr.iterativelength_device(d_src[i].data_ptr(), d_dst[i].data_ptr(), total_pairs, buf.data_ptr(),
                                         d_val.data_ptr(), 0, stream.cuda_stream, opts)
        if world > 1:
            # the one collective: unanswered rows are -1, so MAX assembles the lengths (valid = length >= 0)
            done = torch.cuda.Event()
            done.record(stream)
            side.wait_event(done)
            with torch.cuda.stream(side):
                dist.all_reduce(buf, op=dist.ReduceOp.MAX)
                ev = torch.cuda.Event()
                ev.record(side)
            reduced[i & 1] = ev
        return stt

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # untimed: a call with more searches than one batch holds, so that the second workspace (a call's batches
    # overlap on two streams) exists before the clock starts -- a fresh block of pairs now and then has > 256
    # searching rows, and the first such call would otherwise pay the workspace's cudaMallocs inside the timed loop
    csr.iterativelength(ps_all[0][:P], pd_all[0][:P], None, pgq.Options(args.lanes or 256, args.direction, args.alpha, True))
    for i in range(args.warmup):
        st = step_device(i)
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    # ---- value: K steps, pairs resident in HBM, CUDA events on the launching stream
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    acc = {k: 0 for k in ("kernel_launches", "expand_ms", "edges_traversed", "push_levels", "pull_levels", "pull_ms",
                          "pull_edges", "searches", "pruned", "search_rows", "levels", "batches", "total_ms")}
    for i in range(args.warmup, nsteps):
        st = step_device(i)
        for k in acc:
            acc[k] += st[k]
    if world > 1:
        stream.wait_stream(side)
    ev1.record(stream)
    barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    # per rank: the time its own searches took (sum of the calls' device time) and how many levels they needed --
    # a step ends when the rank with the deepest searches is done
    mine = torch.tensor([acc["total_ms"] / args.steps, acc["levels"] / args.steps, acc["searches"] / args.steps],
                        dtype=torch.float64, device=dev)
    per_rank = [mine.cpu().tolist()]
    if world > 1:
        gathered = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        per_rank = [g.cpu().tolist() for g in gathered]
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    value = total_pairs * args.steps / (ms_total / 1e3)
    last_dev = d_len[(nsteps - 1) & 1].cpu().numpy()
    # (at N > 1 d_val holds this rank's searches only; the assembled column says valid = length >= 0)
    last_valid = d_val.cpu().numpy() if world == 1 else (last_dev >= 0).astype(np.uint8)
    dumps = {"length": last_dev.astype(np.float64), "valid": last_valid.astype(np.float32)}

    # ---- e2e: host buffers through the C ABI (H2D pairs + D2H results inside), result assembly for N > 1
    sharded = sharding.ShardedLengths(csr, dev, pgq.Options(args.lanes, args.direction, args.alpha)) if world > 1 else None

    def step_host(i):
        if world == 1:  # the host-pointer C ABI: pairs H2D + results D2H inside the call
            o, ok, stt = csr.iterativelength(ps_all[i], pd_all[i], None, pgq.Options(args.lanes, args.direction, args.alpha))
            return o, ok, stt
        # one process per GPU: host columns staged through pinned memory, searches sharded, one all_reduce, D2H
        o, ok, stt, (hb, db) = sharded(ps_all[i], pd_all[i])
        stt = dict(stt, h2d_bytes=hb, d2h_bytes=db)
        return o, ok, stt

    for i in range(min(args.warmup, 3)):
        out_h, val_h, st_h = step_host(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    h2d = d2h = 0
    for i in range(args.warmup, nsteps):
        out_h, val_h, st_h = step_host(i)
        h2d += st_h["h2d_bytes"]
        d2h += st_h["d2h_bytes"]
    e1.record(stream)
    barrier()
    ms2 = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = total_pairs * args.steps / (float(ms2.item()) / 1e3)
    clocks = sampler.stop()
    # sanity: the device-resident and the host-pointer runs of the last step agree
    assert np.array_equal(last_dev, np.where(val_h.astype(bool), out_h, -1))
    # outside the timed regions: the last step's pairs with the reference's batch composition (every
    # non-NULL, src != dst row takes a lane), to report its algorithmic work next to the one of the batches we ran
    ref_opts = pgq.Options(st["lanes"], args.direction, args.alpha, True)
    csr.iterativelength(ps_all[-1][:P], pd_all[-1][:P], None, ref_opts)  # untimed: the four-batch call grows the workspaces once
    _, _, st_ref = csr.iterativelength(ps_all[-1][:P], pd_all[-1][:P], None, ref_opts)

    # ---- the north star's other configurations as sub-records (C3: R-MAT-24 / 4096 pairs strong-scaled over
    # the ranks; C5: R-MAT-26, one 512-lane batch per GPU), graphs generated and built on the device
    extra = {}
    if not args.no_extra:
        csr.free()
        del d_src, d_dst
        torch.cuda.empty_cache()
        for name, scale, pairs_total, lanes in (("c3", 24, 4096, 0), ("c5", 26, 512 * world, 512)):
            try:
                extra[name] = run_config(name, scale, pairs_total, lanes, ctx, dev, rank, world, dist, stream, args,
                                         dumps)
            except Exception as ex:  # a sub-record must never cost the headline line
                extra[name] = {"error": f"{type(ex).__name__}: {ex}"[:300]}

    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        steps = args.steps
        W_total, expand_ms = acc["edges_traversed"], acc["expand_ms"]
        expand_launches = acc["push_levels"] + acc["pull_levels"]
        achieved = (W_total * 4.0 / 1e9) / (expand_ms / 1e3) if expand_ms > 0 else 0.0
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")) as f:
                tj = json.load(f)
                traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
        except Exception:
            pass
        pull_l = max(acc["pull_levels"], 1)
        dominant = {"kernel": "k_pull_fused (bottom-up level: expansion + update)", "launches_per_step": acc["pull_levels"] / steps,
                    "ms": acc["pull_ms"] / pull_l, "alg_bytes": acc["pull_edges"] * 4 // pull_l,
                    "achieved": (acc["pull_edges"] * 4.0 / 1e9) / (acc["pull_ms"] / 1e3) if acc["pull_ms"] > 0 else 0.0}
        dominant["frac"] = dominant["achieved"] / peak
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64 lane masks / int32 CSR", "data": "synthetic",
            "config": dict(config, lanes=st["lanes"], direction=args.direction, reachable=int(val_h.sum()),
                           levels_per_step=acc["levels"] / steps, batches_per_step=acc["batches"] / steps,
                           pairs="a fresh block of hashed pairs every step", csr_device_bytes=csr_bytes,
                           csr_build_s=csr_build_s),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d // args.steps,
                    "d2h_bytes_per_step": d2h // args.steps},
            "gpu_launches": acc["kernel_launches"],
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "frontier expansion, all launches of a step (k_pull_fused / k_expand_push*)",
                         "dominant": dominant,
                         "algorithmic_bytes_per_step": W_total * 4 // steps,
                         "edges_traversed_per_step": W_total // steps,
                         "launches_per_step": expand_launches / steps,
                         "searches_per_step": acc["searches"] / steps, "rows_decided_by_degree": acc["pruned"] / steps,
                         "rank0_call_ms_per_step": acc["total_ms"] / steps,
                         "per_rank": {"call_ms_per_step": [round(r[0], 4) for r in per_rank],
                                      "levels_per_step": [round(r[1], 2) for r in per_rank],
                                      "searches_per_step": [round(r[2], 1) for r in per_rank]},
                         "reference_batching": {"edges_traversed_per_step": st_ref["edges_traversed"],
                                                "batches": st_ref["batches"], "levels": st_ref["levels"],
                                                "ms_per_step": st_ref["total_ms"]},
                         "avg_launch_ms": expand_ms / max(expand_launches, 1), "peak_source": peak_src},
        }
        line.update(extra)
        if world == 1 and not args.no_cpu_baseline:
            try:
                cpu_value, info = run_reference(args.scale, n, src, dst, 1, 0, 512)
                line["cpu_baseline"] = {"value": cpu_value, "unit": UNIT, "cores": info["cores"],
                                        "kind": info["kind"], "sample": info["sample"]}
            except Exception as ex:  # the baseline is a reported extra; never lose the GPU line to it
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 1, "kind": "unavailable",
                                        "sample": f"failed: {ex}"[:300]}
                info = None
            # statement level: the SAME statement (CSR CTE + iterativelength over one 512-pair chunk) through DuckDB
            # with the reference extension alone and with the duckpgq_b200 override -- CSR construction included
            try:
                from duckpgq_extension_b200 import duckdb_cli
                db = os.path.join(CACHE, f"rmat{args.scale}.duckdb")
                if info and info.get("kind") == "reference" and duckdb_cli.available() and os.path.exists(db):
                    qs, qd = datagen.hashed_pairs(512, n)
                    cores = os.cpu_count() or 1
                    csr.free()  # the DuckDB process builds its own
                    runs = [duckdb_cli.time_path_statement(db, qs, qd, cores) for _ in range(2)]
                    best = min(runs, key=lambda r: r["statement_s"] or 1e9)
                    line["e2e_query"] = {
                        "statement": f"CSR CTE (create_csr_vertex + create_csr_edge over R-MAT-{args.scale}) + iterativelength "
                                     f"over one 512-pair DataChunk, DuckDB threads={cores}",
                        "reference_statement_s": info.get("statement_s"), "reference_projection_s": info.get("bfs_s"),
                        "b200_statement_s": best["statement_s"], "b200_projection_s": best["projection_s"],
                        "b200_first_run_statement_s": runs[0]["statement_s"], "b200_stats": best["stats"],
                        "same_answer": best["reachable"] == info.get("reachable")}
            except Exception as ex:
                line["e2e_query"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumps)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_config(name, scale, pairs_total, lanes, ctx, dev, rank, world, dist, stream, args, dumps):
    """One of the north star's larger configurations on the same ranks: the graph is generated and built on
    every GPU (replicated CSR), the searches of ONE pair set are dealt over the ranks, all_reduce(MAX)
    assembles the answer.  Timed like the headline: CUDA events, barrier on both sides, max over ranks, --steps
    calls.  The result columns of the last call go to dumps[name + "_length" / "_valid"]."""
    import torch
    from duckpgq_extension_b200 import pgq
    t0 = time.perf_counter()
    n, src, dst = datagen.rmat_edges_device(scale, device=dev)
    m = int(src.numel())
    csr = pgq.DeviceCSR.build_device(ctx, n, m, src.data_ptr(), dst.data_ptr())
    torch.cuda.synchronize()
    del src, dst
    torch.cuda.empty_cache()
    setup_s = time.perf_counter() - t0
    ps, pd = datagen.hashed_pairs(pairs_total, n)
    d_src, d_dst = torch.from_numpy(ps).to(dev), torch.from_numpy(pd).to(dev)
    d_len = torch.empty(pairs_total, dtype=torch.int64, device=dev)
    d_val = torch.empty(pairs_total, dtype=torch.uint8, device=dev)
    opts = pgq.Options(lanes, args.direction, args.alpha, reference_batching=(name == "c5"))
    opts.shard_index, opts.shard_count = (rank, world) if world > 1 else (0, 0)

    def step():
        stt = csr.iterativelength_device(d_src.data_ptr(), d_dst.data_ptr(), pairs_total, d_len.data_ptr(),
                                         d_val.data_ptr(), 0, stream.cuda_stream, opts)
        if world > 1:
            dist.all_reduce(d_len, op=dist.ReduceOp.MAX)
        return stt

    for _ in range(2):
        step()
    reps = args.steps
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        st = step()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1), st["total_ms"]], dtype=torch.float64, device=dev)
    rank_ms = [float(ms[1].item())]
    if world > 1:
        gathered = [torch.zeros_like(ms) for _ in range(world)]
        dist.all_gather(gathered, ms)
        rank_ms = [float(g[1].item()) for g in gathered]
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms[0].item()) / reps
    peak, _ = measured_peak_hbm()
    W, ems = st["edges_traversed"], st["expand_ms"]
    rec = {"workload": f"RMAT scale-{scale} ({n} v / {m} e), {pairs_total} hashed pairs over {world} GPU(s), "
                       f"{'one 512-lane batch per GPU (reference batch composition)' if name == 'c5' else 'default batching'}",
           "value": pairs_total / (total_ms / 1e3), "unit": UNIT, "ms_per_call": total_ms,
           "rank_call_ms": rank_ms, "rank0": {k: st[k] for k in ("lanes", "searches", "batches", "levels", "pull_levels",
                                                                 "push_levels", "edges_traversed", "expand_ms",
                                                                 "pull_ms", "pull_edges")},
           "roofline_frac_rank0": (W * 4.0 / 1e9) / (ems / 1e3) / peak if ems > 0 else None,
           "pull_frac_rank0": (st["pull_edges"] * 4.0 / 1e9) / (st["pull_ms"] / 1e3) / peak if st["pull_ms"] > 0 else None,
           "reachable": int((d_len >= 0).sum().item()), "setup_s": setup_s, "csr_device_bytes": csr.info()[2]}
    last_len = d_len.cpu().numpy()
    dumps[f"{name}_length"] = last_len.astype(np.float64)
    dumps[f"{name}_valid"] = (d_val.cpu().numpy() if world == 1 else last_len >= 0).astype(np.float32)
    csr.free()
    del d_src, d_dst, d_len, d_val
    torch.cuda.empty_cache()
    return rec


if __name__ == "__main__":
    main()
