#!/usr/bin/env python
"""bench.py -- Mchecks/sec of batched CheckPermission (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg3] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (CheckBulkPermissions) over one batch of
synthetic checks of the named workload (SURVEY.md 8d). Prints ONE JSON line.
The device-resident, e2e and (N > 1) sharded legs each time exactly K steps after W (at least 3)
warm-up steps; the sustained leg runs for --sustain-s seconds instead (0 skips it). --impl
reference times K steps after exactly W warm-up steps.

--dump-outputs DIR: after the timed steps, rank 0 writes the answers of the last timed step of every
measured workload as DIR/<workload>_answers.npy (float32 answer codes: 1 no permission, 2 has
permission, 255 error; one per check of the batch, at most 2^20 per workload). With --impl reference
the file holds the oracle's answers to the first checks of the same batch, the sample it times. The
workloads are seeded, so the same arguments give the same inputs on every run and two builds, or a
build and the oracle, can be compared answer for answer.

  value     whole-job Mchecks/s, inputs resident in HBM when the timed region starts
            (zg_check_bulk_device on device buffers, CUDA events on the launch stream,
            max over ranks)
  e2e       the same metric through the reference-facing C ABI call zg_check_bulk with
            pinned HOST buffers: H2D of the 16 B items and D2H of the 1 B answers are
            inside the timed region
  roofline  algorithmic bytes of the check kernel (counted by the instrumented kernel
            variant) / its CUDA-event duration, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the CPU oracle (a port: the reference's engine is a Go module that
            cannot be built here) on a bounded sample, rank 0, N=1

Multi-GPU (--gpus N under torchrun): the store (<= 1.6 GB) is REPLICATED on every GPU
and each rank answers its own batch: no data-path collective, "scaling": "weak".
--impl reference: the oracle on all host threads, rank 0 only.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# bench.py writes nothing under the tree: in a writable tree, importing modules build() does not import
# (workloads, dist) would otherwise leave their bytecode cache there
sys.dont_write_bytecode = True

_REAL_STDOUT = None


def emit(obj):
    """The single JSON line, on the process's original stdout."""
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


METRIC = "Mchecks/sec (batched CheckPermission)"
UNIT = "Mchecks/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="zgpu", choices=["zgpu", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg2", "cfg2-zipf", "cfg3", "cfg4"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (debugging only)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="checks in the CPU-baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--configs", default="cfg2,cfg4",
                    help="other BASELINE configurations reported as sub-results under `configs` ('' = none)")
    ap.add_argument("--no-sharded", action="store_true", help="N > 1: skip the object-hash sharded cfg4 leg")
    ap.add_argument("--sharded-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--sharded-timeout", type=float, default=300.0, help="hard limit of the sharded leg, seconds")
    ap.add_argument("--sustain-s", type=float, default=2.5,
                    help="length of the back-to-back 'sustained' leg of the primary workload (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the answers of the last timed step of each workload as DIR/<workload>_answers.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def host_cores():
    """Threads the CPU arm may really use: the scheduler affinity, not the machine's CPU count."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def workload_config(w, args, world):
    return {
        "workload": f"{w.name}: {w.note}",
        "tuples": w.n_tuples(),
        "batch": w.n_checks(),
        "global_batch": w.n_checks() * world,
        "parallelism": f"replicas x{world} (store replicated, checks sharded, no collective)" if world > 1 else "1 GPU",
        "l2": "L2 flushed (256 MiB write) between timed steps; per-step CUDA events exclude the flush",
        "scale": args.scale,
    }


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload):
    """dram bytes per launch of check_kernel from the committed ncu capture of the same build, if any:
    {"dram_bytes": ..., "kernel_ms": ..., "source": "profiles/..."} (older entries: a bare number)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get(workload)
    return None


class ClockSampler:
    """Samples SM clock and throttle reasons DURING the timed region (NVML, every 5 ms, in a
    thread). B200_PROFILING.md: a run that saw hw_slowdown / hw_thermal_slowdown /
    sw_thermal_slowdown, or clocks stuck far below max with no reason, must be re-measured."""

    def __init__(self, index):
        self.index = index
        self.samples, self.max_mhz, self.reasons = [], None, set()
        self._stop = False
        self._thread = None
        self._err = None

    def _run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {
                "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            }
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
            while not self._stop:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                r = int(get_reasons(h))
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
                time.sleep(0.005)
        except Exception as ex:  # noqa: BLE001  (reported, never fatal for the measurement)
            self._err = repr(ex)

    def start(self):
        import threading

        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop = True
        if self._thread:
            self._thread.join(timeout=5)
        sm = sorted(self.samples)
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "samples": len(sm),
               "reasons": sorted(self.reasons), "source": "NVML, 5 ms period, warm-up through the e2e leg"}
        if self._err:
            out["error"] = self._err
        return out


def cpu_reference_arm(args, rank, world):
    """--impl reference: the oracle port, all host threads, bounded sample per step."""
    if rank != 0:
        return
    import numpy as np

    import zgpu  # noqa: F401  only registers the package so the workload generators import; libzgpu.so is NOT loaded
    from oracle.pyoracle import CHECK_DTYPE, Oracle
    from spicedb_kubeapi_proxy_b200 import workloads

    w = workloads.by_name(args.workload, args.scale)
    o = Oracle(w.schema)
    w.load_into(o)
    items = w.check_items(o, CHECK_DTYPE)
    cores = host_cores()
    o.check_bulk(items[:256])  # builds the index (not timed)
    t = time.perf_counter()
    o.check_bulk(items[:4096], nthreads=cores)
    rate = 4096 / max(time.perf_counter() - t, 1e-6)
    budget_s = 120.0 / max(args.steps + args.warmup, 1)
    n = args.cpu_sample or int(min(items.size, max(2048, rate * min(budget_s, 8.0))))
    sample = items[:n]
    for _ in range(args.warmup):
        o.check_bulk(sample, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        answers = o.check_bulk(sample, nthreads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, f"{w.name}_answers.npy"), answers.astype(np.float32))
    val = n * args.steps / dt / 1e6
    desc = f"first {n} checks of the {w.name} batch per step, {cores} threads"
    emit({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": workload_config(w, args, 1),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc,
                         "note": "C oracle restating SpiceDB v1.47.1 check semantics; the reference's own engine is an "
                                 "un-vendored Go module and no Go toolchain exists on this box",
                         "algorithm": "forward recursive evaluation, no caching (pkg/spicedb/spicedb.go:44-46): ~42 KB of "
                                      "index reads per cfg3 check; the GPU arm is direction-optimised (< 1 KB per check), "
                                      "so most of the ratio between the arms is algorithmic, not hardware"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def bound_from_evidence(dram_frac, frac):
    """Which resource bounds the kernel, from the ncu capture of the same workload: a kernel that moves
    under a quarter of the DRAM peak is not HBM-bound whatever its algorithmic byte rate says."""
    if dram_frac is None:
        return "unknown (no ncu capture committed for this workload)"
    if dram_frac >= 0.25:
        return "hbm"
    return "l2-latency/issue" if (frac or 0) > dram_frac * 2 else "latency/issue"


def measure_workload(name, args, rank, local_rank, world, dist, primary, sampler=None):
    """One workload on this rank's GPU: device-resident value, e2e through the C ABI, algorithmic bytes,
    live parity sample against the CPU oracle (rank 0). Returns the result dict (rank 0) or None."""
    import numpy as np
    import torch

    import zgpu
    from spicedb_kubeapi_proxy_b200 import workloads

    steps, warmup = args.steps, max(args.warmup, 3)
    t_gen = time.perf_counter()
    w = workloads.by_name(name, args.scale)
    eng = zgpu.Engine(w.schema, device=local_rank)
    w.load_into(eng)
    t0 = time.perf_counter()
    eng.publish()
    publish_s = time.perf_counter() - t0
    setup_s = time.perf_counter() - t_gen
    items = w.check_items(eng, zgpu.CHECK_DTYPE)
    if world > 1:  # each rank answers its own batch (weak scaling): rank-specific permutation
        items = items[np.random.default_rng(1000 + rank).permutation(items.size)]
    n = items.size

    d_items = torch.from_numpy(items.view(np.uint8).copy()).cuda()
    d_out = torch.zeros(n, dtype=torch.uint8, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream()

    def step_device():
        eng.check_bulk_device(d_items.data_ptr(), n, d_out.data_ptr(), stream.cuda_stream)

    # algorithmic bytes of one launch, from the instrumented kernel variant (not timed)
    alg_bytes = eng.count_alg_bytes(items)

    for _ in range(warmup):
        flush.zero_()
        step_device()
    torch.cuda.synchronize()
    launches0 = eng.stats()["launches"]
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in evs:
        flush.zero_()  # evict the store and the batch from L2; outside the event pair
        a.record(stream)
        step_device()
        b.record(stream)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    launches = eng.stats()["launches"] - launches0
    last_answers = d_out.cpu().numpy() if (args.dump_outputs and rank == 0) else None
    t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max = float(t.item())
    value = n * world * steps / (dev_ms_max / 1e3) / 1e6

    # ---- sustained: the same step back to back for >= args.sustain_s seconds (clocks settle under
    # load, unlike the 20 x 1 ms timed region); L2 flush between steps, one event pair around all
    sustained = None
    if primary and args.sustain_s > 0:
        per = max(dev_ms_max / steps, 0.05)
        reps = int(min(max(args.sustain_s * 1e3 / (per + 0.08), 50), 200000))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fl = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fl[0].record(stream)
        for _ in range(20):
            flush.zero_()
        fl[1].record(stream)
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        flush_ms = fl[0].elapsed_time(fl[1]) / 20.0
        a.record(stream)
        for _ in range(reps):
            flush.zero_()
            step_device()
        b.record(stream)
        torch.cuda.synchronize()
        tot = a.elapsed_time(b)
        t = torch.tensor([tot], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tot = float(t.item())
        kern = max(tot - reps * flush_ms, 1e-3)
        sustained = {"value": n * world * reps / (kern / 1e3) / 1e6, "unit": UNIT, "steps": reps, "wall_s": tot / 1e3,
                     "note": "back-to-back steps with an L2 flush between them; flush time (measured alone) subtracted"}

    # ---- e2e: the public C ABI call with pinned host buffers, copies inside the timed region
    pin_in = zgpu._lib.PinnedArray(n, zgpu.CHECK_DTYPE)
    pin_out = zgpu._lib.PinnedArray(n, np.uint8)
    pin_in.array[:] = items
    for _ in range(warmup):
        eng.check_bulk_ptr(pin_in.ptr, n, pin_out.ptr)
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        eng.check_bulk_ptr(pin_in.ptr, n, pin_out.ptr)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = n * world * steps / float(t.item()) / 1e6
    clocks = sampler.stop() if (sampler is not None and rank == 0) else None
    host_answers = pin_out.array.copy()
    assert np.array_equal(host_answers, d_out.cpu().numpy()), "host and device entry points disagree"

    # ---- CPU baseline: oracle on a bounded sample (rank 0), also a live parity check of the timed batch
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle.pyoracle import Oracle

        o = Oracle(w.schema)
        w.load_into(o)
        cores = host_cores()
        o.check_bulk(items[:256])  # builds the index (not timed)
        tq = time.perf_counter()
        o.check_bulk(items[:2048], nthreads=cores)
        rate = 2048 / max(time.perf_counter() - tq, 1e-6)
        budget_s = 15.0 if primary else 8.0
        ns = args.cpu_sample or int(min(n, max(50_000 if world == 1 else 8192, rate * budget_s)))
        tq = time.perf_counter()
        want = o.check_bulk(items[:ns], nthreads=cores)
        dt = time.perf_counter() - tq
        mism = int((want != host_answers[:ns]).sum())
        cpu = {"value": ns / dt / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"first {ns} checks of the same batch, {cores} threads, {dt:.1f} s",
               "parity_mismatches_vs_gpu": mism,
               "algorithm": "forward recursive evaluation, no caching (pkg/spicedb/spicedb.go:44-46); the GPU path is "
                            "direction-optimised (reverse rows of the subject), so most of the ratio is algorithmic"}
        if primary:
            # SURVEY 8(d)'s canonical figure: forward evaluation, no short circuit (small sample)
            cpu["canonical_forward_bytes_per_check"] = o.check_bytes(items[:2000]) / 2000.0
        if mism:
            raise SystemExit(f"PARITY FAILURE ({name}): {mism} of {ns} answers differ from the oracle")
        del o

    out = None
    if rank == 0:
        peak, peak_src = measured_peak()
        kernel_ms = dev_ms_max / steps
        achieved = alg_bytes / (kernel_ms / 1e3) / 1e9
        cap = ncu_traffic(w.name) or {}
        traffic = cap.get("dram_bytes") if isinstance(cap, dict) else cap
        cap_ms = cap.get("kernel_ms") if isinstance(cap, dict) else None
        # DRAM rate of the captured launch itself (its own bytes / its own duration), and the same bytes
        # over THIS run's kernel time: they agree when the capture is of the same build
        dram_gbs = traffic / (kernel_ms / 1e3) / 1e9 if traffic else None
        dram_frac = dram_gbs / peak if dram_gbs else None
        out = {
            "value": value, "unit": UNIT, "ms_per_step": kernel_ms,
            "config": workload_config(w, args, world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * 16, "d2h_bytes_per_step": n,
                    "steps": steps, "api": "zg_check_bulk (C ABI, pinned host buffers)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": bound_from_evidence(dram_frac, achieved / peak), "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "dram_gbs": dram_gbs,
                         "dram_frac": dram_frac, "dram_over_algorithmic": (traffic / alg_bytes) if traffic else None,
                         "ncu_capture": cap.get("source") if isinstance(cap, dict) else None,
                         "ncu_capture_kernel_ms": cap_ms,
                         "peak_source": peak_src, "kernel": "zg::check_kernel<false>",
                         "alg_bytes_per_launch": int(alg_bytes), "alg_bytes_per_check": alg_bytes / n,
                         "kernel_ms": kernel_ms,
                         "note": "achieved/frac: bytes the kernel's own loads need (counted by the instrumented variant: "
                                 "16 B item + 1 B answer + 4 B per row offset, probe and edge read, short circuit "
                                 "included) / CUDA-event time. dram_*: ncu dram__bytes_read+write of one launch of the "
                                 "same build / the same time -- the HBM fraction north_star asks for"},
            "cpu_baseline": cpu,
            "has_fraction": float((host_answers == 2).mean()),
            "build": zgpu._lib.lib().zg_build_info().decode(),
            "publish_s": publish_s, "setup_s": setup_s,
        }
        if sustained:
            out["sustained"] = sustained
        if clocks is not None:
            out["clocks"] = clocks
    if last_answers is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, f"{w.name}_answers.npy"), last_answers.astype(np.float32))
    del d_items, d_out, flush, pin_in, pin_out
    eng.close()
    torch.cuda.empty_cache()
    return out


def measure_sharded(args, rank, local_rank, world, dist):
    """cfg4 at full size on an object-hash sharded store: each rank brings 1/N of the 1 M-check batch; the answers
    must equal a replica's bit for bit (checked on rank 0 against an engine holding the whole store)."""
    import numpy as np
    import torch

    import zgpu
    from spicedb_kubeapi_proxy_b200 import dist as zdist
    from spicedb_kubeapi_proxy_b200 import workloads

    def note(msg):
        print(f"[sharded rank {rank} +{time.perf_counter() - t_start:.1f}s] {msg}", file=sys.stderr, flush=True)

    t_start = time.perf_counter()
    w = workloads.by_name("cfg4", args.scale)
    note("workload generated")
    eng = zgpu.Engine(w.schema, device=local_rank, shard_rank=rank, shard_count=world, subquery_capacity=1 << 24)
    w.load_into(eng)  # keeps only the relationships this rank owns
    eng.publish()
    items = w.check_items(eng, zgpu.CHECK_DTYPE)
    lo, hi = zdist.shard_bounds(items.size, rank, world)
    mine = np.ascontiguousarray(items[lo:hi])
    d_items = torch.from_numpy(mine.view(np.uint8).copy()).cuda()
    ck = zdist.DeviceShardedChecker(eng, zdist.TorchDeviceTransport())
    chunk = 1 << 18  # checks per rank per round: bounds the sub-queries a pass may raise (~20 per check, buffer 16 M)
    n_chunks = (hi - lo + chunk - 1) // chunk
    steps, warmup = args.steps, max(args.warmup, 3)

    def one_step():
        outs = []
        for b in range(0, hi - lo, chunk):
            e = min(hi - lo, b + chunk)
            outs.append(ck.check_bulk(d_items[b * 16:e * 16], e - b))
        return torch.cat(outs)

    note(f"shard published: {eng.stats()['tuples']} relationships")
    for i in range(warmup):
        ans = one_step()
        if i == 0:
            note(f"first step done: levels {ck.stats['levels']}, sub-queries sent {ck.stats['subqueries_sent']}")
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        ans = one_step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    note(f"{steps} steps in {dt:.2f} s")
    mism = None
    gathered = [torch.empty(zdist.shard_bounds(items.size, r, world)[1] - zdist.shard_bounds(items.size, r, world)[0],
                            dtype=torch.uint8, device="cuda") for r in range(world)]
    # ragged all-gather of the answers (sizes differ by at most one): pad to the widest
    width = max(g.numel() for g in gathered)
    pad = torch.zeros(width, dtype=torch.uint8, device="cuda")
    pad[: ans.numel()] = ans
    blocks = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(blocks, pad)
    n_tuples_owned = torch.tensor([eng.stats()["tuples"]], dtype=torch.int64, device="cuda")
    dist.all_reduce(n_tuples_owned, op=dist.ReduceOp.SUM)
    st = dict(ck.stats)
    eng.close()
    out = None
    if rank == 0:
        full = np.concatenate([blocks[r][: gathered[r].numel()].cpu().numpy() for r in range(world)])
        rep = zgpu.Engine(w.schema, device=local_rank)
        w.load_into(rep)
        rep.publish()
        want = rep.check_bulk(items)
        mism = int((full != want).sum())
        rep.close()
        passes = warmup + steps  # the checker's counters include the warm-up steps
        out = {"value": items.size * steps / dt / 1e6, "unit": UNIT, "ms_per_step": dt / steps * 1e3, "steps": steps,
               "warmup": warmup, "mismatches_vs_replica": mism, "tuples_over_all_shards": int(n_tuples_owned.item()),
               "levels": st["levels"], "subqueries_per_check": st["subqueries_sent"] / max((hi - lo) * passes, 1),
               "exchanges_per_round": st["exchanges"] / max(passes * n_chunks, 1),
               "bytes_sent_per_rank_per_step": st["bytes_sent"] / passes,
               "limiting": "per-level round trip (kernel pass + count exchange + NCCL all-to-all): latency-bound, "
                           "bytes are far below NVLink",
               "config": {"workload": f"cfg4 object-hash sharded x{world}: {w.note}", "chunk_checks_per_rank": chunk,
                          "global_batch": items.size}}
        if mism:
            out["error"] = f"{mism} answers differ from the replica"
    dist.barrier()
    return out


def run_sharded_leg(args, rank, world, dist):
    """The sharded leg runs in CHILD processes (one per rank, their own process group on another port) under a hard
    timeout: a failure or a hang in the multi-level exchange must never cost the replica numbers of this line."""
    import torch

    torch.cuda.empty_cache()
    out_path = os.path.join(tempfile.gettempdir(), f"zgpu_sharded_{os.environ.get('MASTER_PORT', '0')}.json")
    if rank == 0 and os.path.exists(out_path):
        os.remove(out_path)
    dist.barrier()
    env = dict(os.environ)
    env["MASTER_PORT"] = str(int(os.environ.get("MASTER_PORT", "29500")) + 17)
    # under torchrun the workers use the AGENT's store; the children form their own group: rank 0's child hosts it
    env["TORCHELASTIC_USE_AGENT_STORE"] = "False"
    env["ZGPU_SHARDED_OUT"] = out_path
    cmd = [sys.executable, os.path.abspath(__file__), "--sharded-child", "--gpus", str(world), "--steps", str(args.steps),
           "--warmup", str(args.warmup)]
    err = None
    with tempfile.TemporaryFile() as lf:  # the child's log: relayed to this rank's stderr, its tail into the error
        try:
            r = subprocess.run(cmd, env=env, timeout=args.sharded_timeout, stdout=lf, stderr=subprocess.STDOUT)
            if r.returncode != 0:
                err = f"child rc={r.returncode}"
        except subprocess.TimeoutExpired:
            err = f"child timed out after {args.sharded_timeout} s (raise --sharded-timeout or lower --steps)"
        lf.seek(0)
        log = lf.read().decode(errors="replace")
    sys.stderr.write(log)
    sys.stderr.flush()
    if err:
        err += ": " + log[-300:]
    dist.barrier()
    if rank != 0:
        return None
    if os.path.exists(out_path):
        with open(out_path) as f:
            res = json.load(f)
        os.remove(out_path)
        return res
    return {"error": err or "no result"}


def sharded_child(args):
    import torch
    import torch.distributed as dist

    rank, local_rank, world = dist_env()
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    r = measure_sharded(args, rank, local_rank, world, dist)
    if rank == 0 and r is not None:
        with open(os.environ["ZGPU_SHARDED_OUT"], "w") as f:
            json.dump(r, f)
    dist.destroy_process_group()


def main():
    # stdout must carry exactly ONE JSON line, but libraries print there too (NCCL's version banner
    # under torchrun): point fd 1 at stderr for the whole run and emit the line on the saved fd
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse_args()
    rank, local_rank, world = dist_env()
    if args.impl == "reference":
        cpu_reference_arm(args, rank, world)
        return
    if args.sharded_child:
        sharded_child(args)
        return

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path in libzgpu)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # samples clocks / throttle reasons from the warm-up to the end of the e2e leg
    main_res = measure_workload(args.workload, args, rank, local_rank, world, dist, True, sampler)

    # the other BASELINE configurations as sub-results of the same line (configs[1] and configs[3], the
    # latter at its full 100 M relationships: the regime the HBM-roofline target is quoted on)
    extra = {}
    names = [c for c in args.configs.split(",") if c and c != args.workload] if args.scale == 1.0 else []
    for name in names:
        r = measure_workload(name, args, rank, local_rank, world, dist, False)
        if r is not None:
            extra[name] = r

    # N > 1: north-star's other multi-GPU mode on the configuration it names for it (cfg4, "object-id sharded
    # across 8 GPUs"): every rank owns the relationships whose resource id % N is its rank, checks and raised
    # sub-queries are routed device to device (dist.DeviceShardedChecker: NCCL all-to-all of device buffers per
    # level). A second field of the line, never the headline; a failure is reported, not fatal.
    if world > 1 and args.scale == 1.0 and not args.no_sharded:
        r = run_sharded_leg(args, rank, world, dist)
        if r is not None:
            extra["cfg4_sharded"] = r

    if rank == 0:
        out = {
            "metric": METRIC, "value": main_res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": main_res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic", "impl": "zgpu",
        }
        for k in ("config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks", "sustained", "has_fraction",
                  "publish_s", "setup_s", "build"):
            if k in main_res:
                out[k] = main_res[k]
        if extra:
            out["configs"] = extra
        emit(out)
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
